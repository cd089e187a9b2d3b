"""ORACLE (test infrastructure): tests/golden/reference_checks.npz -- what the REFERENCE'S OWN code returns for the inputs of
the reference checks in the CPU suite, so that those checks run wherever the suite runs, without the reference tree:

  * stage-1: its ``Transformer`` forward (fp32 logits of a 9-token prompt, tiny dims, weight seed 3) and its
    ``generate`` (12 new tokens after ``torch.manual_seed(5)``);
  * speaker encoder: ``SpeakerEncoder.compute_partial_slices`` over a grid of lengths / rates / coverages;
  * adapters: ``FlattenedInterleavedEncodec2Codebook.decode`` and ``TiltedEncodec.decode`` on seeded token lists;
  * stage-2 input: the tensor ``Model.non_causal_sample`` builds for three texts (oracle/make_golden_stage2_input.py).

Needs the reference tree (``MVB_REFERENCE_ROOT``, see oracle/ref_harness.py):  python oracle/make_golden_reference.py
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "metavoice-src_b200"))
from mvb200 import synth  # noqa: E402
from oracle import ref_harness as R  # noqa: E402

SLICE_LENGTHS = (16000, 25601, 102400, 480000, 777777)
SLICE_RATES = ((1.3, 0.75), (2.0, 0.5))
S2_TEXTS = ("a b c", "the quick brown fox", "x")


def stage1(out):
    d = synth.TINY
    sd = synth.stage1_state_dict(d, 3)
    prompt, spk = synth.synthetic_prompt(9, seed=5), synth.synthetic_speaker(seed=2)
    ref = R.build_reference_model(sd, d, torch.float32)
    with torch.no_grad():
        logits = ref(prompt.view(1, -1).repeat(2, 1), spk, torch.arange(9))
    fiu = R.reference_functions()
    ref2 = R.build_reference_model(sd, d, torch.float32)
    kw = dict(temperature=torch.tensor(0.8), top_p=torch.tensor(0.9), guidance_scale=torch.tensor(2.0), top_k=None)
    torch.manual_seed(5)
    y = fiu.generate(ref2, prompt, spk, max_new_tokens=12, end_of_audio_token=9999, **kw)
    out.update(s1_checksum=np.float64(synth.state_dict_checksum(sd)), s1_prompt=prompt.numpy(), s1_spk=spk.numpy(),
               s1_logits=logits.numpy().astype(np.float32), s1_tokens=y.numpy().astype(np.int64))


def speaker_slices(out):
    from fam.quantiser.audio.speaker_encoder.model import SpeakerEncoder
    for n in SLICE_LENGTHS:
        for rate, cov in SLICE_RATES:
            wav_slices, mel_slices = SpeakerEncoder.compute_partial_slices(n, rate, cov)
            out[f"spk_{n}_{rate}_{cov}_wav"] = np.asarray([(s.start, s.stop) for s in wav_slices], np.int64)
            out[f"spk_{n}_{rate}_{cov}_mel"] = np.asarray([(s.start, s.stop) for s in mel_slices], np.int64)


def adapters(out):
    from fam.llm.adapters import FlattenedInterleavedEncodec2Codebook, TiltedEncodec
    g = torch.Generator().manual_seed(0)
    flat = torch.randint(0, 2562, (300,), generator=g).tolist()
    text, cb = FlattenedInterleavedEncodec2Codebook(end_of_audio_token=1024).decode([flat])
    out.update(flat_in=np.asarray(flat, np.int64), flat_text=np.asarray(text, np.int64))
    for i, c in enumerate(cb):
        out[f"flat_cb{i}"] = np.asarray(c, np.int64)
    hier = torch.randint(0, 1100, (8, 200), generator=g).tolist()
    text, codes = TiltedEncodec(end_of_audio_token=1024).decode(hier)
    out.update(hier_in=np.asarray(hier, np.int64), hier_text=np.asarray(text, np.int64), hier_codes=np.asarray(codes, np.int64))


def stage2_input(out):
    from oracle import make_golden_stage2_input as mk
    from mvb200.tokenise import TrainedBPETokeniser
    tok = TrainedBPETokeniser(**synth.synthetic_tokenizer_meta(n_text_tokens=512, offset=1025))
    g = torch.Generator().manual_seed(77)
    codes = [torch.randint(0, 1024, (1, 2, n), generator=g) for n in (10, 300, 255)]
    in_x = mk.reference_in_x(mk.reference_model_class(), tok, list(S2_TEXTS), codes, 256)
    out["s2_texts"] = np.asarray(S2_TEXTS)
    for i, c in enumerate(codes):
        out[f"s2_codes_{i}"] = c[0].numpy().astype(np.int64)
        out[f"s2_in_x_{i}"] = in_x[i].numpy().astype(np.int64)


def main():
    R._import_reference()
    out = {}
    for record in (stage1, speaker_slices, adapters, stage2_input):
        record(out)
    path = os.path.join(ROOT, "tests", "golden", "reference_checks.npz")
    np.savez_compressed(path, **out)
    print(f"{path}: {len(out)} arrays, {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main()
