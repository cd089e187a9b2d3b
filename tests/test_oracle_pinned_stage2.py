"""CPU: stage-2 oracle restatement vs golden vectors from the reference's own GPT, adapters and input builder."""
import numpy as np
import pytest
import torch

from mvb200 import synth
from mvb200.second_stage import build_stage2_input, flattened_interleaved_decode, tilted_decode
from oracle import stage2_port as P


@pytest.mark.parametrize("tag,dims", [("tiny", synth.S2_TINY), ("full", synth.S2_FULL)])
def test_stage2_port_matches_reference_golden(golden_dir, tag, dims):
    g = np.load(f"{golden_dir}/stage2.npz")
    sd = synth.stage2_state_dict(dims, 1)
    assert synth.state_dict_checksum(sd) == pytest.approx(float(g[f"{tag}_checksum"]), abs=1e-9)
    m = P.Stage2Oracle(sd, dims.n_head, dims.rmsnorm_eps)
    idx = torch.from_numpy(g[f"{tag}_idx"]).long()
    logits = m.forward(idx, torch.from_numpy(g[f"{tag}_spk"]))
    keep = g[f"{tag}_keep"]
    got = torch.stack([l[0, keep] for l in logits])
    ref = torch.from_numpy(g[f"{tag}_logits"])
    assert (got - ref).abs().max() / ref.abs().max() < 1e-5
    torch.manual_seed(4242)
    noise = [torch.empty(1, dims.block_size, v).exponential_(1) for v in dims.target_vocab_sizes]
    y = P.non_causal_sample(logits, 1.0, 200, noise)
    assert torch.equal(y[0].int(), torch.from_numpy(g[f"{tag}_tokens"]))


def test_adapters_match_oracle_and_reference_semantics():
    flat = [2100, 2200, 2561, 5, 1030, 7, 1031, 9, 2048]          # text.. EOT a0 b0 a1 b1 a2 EOA  (cb1 one short)
    for fn in (flattened_interleaved_decode, P.flattened_interleaved_decode):
        text, cb = fn(flat)
        assert text == [2100, 2200] and cb == [[5, 7], [6, 7]]
    hier = [[1100, 1537, 3, 4, 5, 1024, 1024], [1024, 1024, 6, 7, 8, 1024, 1024]] + [[9, 9, 1024, 2, 1, 1024, 3]] * 6
    for fn in (tilted_decode, P.tilted_decode):
        text, codes = fn(hier)
        assert text == [1100] and len(codes) == 8 and all(len(c) == 3 for c in codes)
        assert codes[0] == [3, 4, 5] and codes[2] == [9, 9, 2]   # "first-N-valid" truncation (tilted_encodec.py:31-37)


def test_adapters_match_live_reference(golden_dir):
    """What the reference's own FlattenedInterleavedEncodec2Codebook.decode and TiltedEncodec.decode return, as recorded
    by oracle/make_golden_reference.py."""
    g = np.load(f"{golden_dir}/reference_checks.npz")
    flat = g["flat_in"].tolist()
    a = (g["flat_text"].tolist(), [g["flat_cb0"].tolist(), g["flat_cb1"].tolist()])
    assert tuple(a) == tuple(flattened_interleaved_decode(flat))
    hier = g["hier_in"].tolist()
    b = (g["hier_text"].tolist(), g["hier_codes"].tolist())
    assert tuple(b) == tuple(tilted_decode(hier))


def test_input_builder_layout():
    idx = P.build_input([1100, 1537], [1, 2, 3], [4, 5, 6], 8)
    assert idx.tolist() == [[1100, 1537, 1, 2, 3, 1024, 1024, 1024], [1024, 1024, 4, 5, 6, 1024, 1024, 1024]]
    idx = P.build_input([1100, 1537], list(range(10)), list(range(10)), 8)      # truncation to block_size
    assert idx.shape == (2, 8) and idx[0, -1] == 5


@pytest.mark.parametrize("tag", ["tiny", "full"])
def test_product_input_builder_matches_reference_golden(golden_dir, tag):
    """a13: the PRODUCT builder (mvb200.second_stage.build_stage2_input, what SecondStage.build_input calls) against
    the tensor the reference's own Model.non_causal_sample built (oracle/make_golden_stage2_input.py executes
    fam/llm/inference.py:264-306): padded, cut-by-one, truncated and exact-fit cases."""
    g = np.load(f"{golden_dir}/stage2_input.npz")
    bs = int(g[f"{tag}_block"])
    ref = g[f"{tag}_in_x"]
    for i in range(ref.shape[0]):
        got = build_stage2_input(g[f"{tag}_text_{i}"].tolist(), g[f"{tag}_codes_{i}"].tolist(), bs)
        assert got.shape == (2, bs) and got.dtype == torch.int32
        assert np.array_equal(got.numpy(), ref[i]), f"case {i}"
        assert np.array_equal(P.build_input(g[f"{tag}_text_{i}"].tolist(), *g[f"{tag}_codes_{i}"].tolist(), bs).numpy(), ref[i])


def test_product_input_builder_matches_live_reference(golden_dir):
    """The tensor the reference's own Model.non_causal_sample builds for three texts, as recorded by
    oracle/make_golden_reference.py."""
    from mvb200.tokenise import TrainedBPETokeniser
    tok = TrainedBPETokeniser(**synth.synthetic_tokenizer_meta(n_text_tokens=512, offset=1025))
    g = np.load(f"{golden_dir}/reference_checks.npz")
    for i, text in enumerate(g["s2_texts"].tolist()):
        got = build_stage2_input(tok.encode(text), g[f"s2_codes_{i}"].tolist(), 256)
        assert torch.equal(got.long(), torch.from_numpy(g[f"s2_in_x_{i}"]))
