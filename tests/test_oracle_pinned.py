"""CPU: the oracle restatement (oracle/stage1_port.py) against the committed golden vectors that were produced by
the reference's own code (oracle/make_golden.py, oracle/make_golden_reference.py).  If these fail, no GPU parity
claim means anything."""
import numpy as np
import pytest
import torch

from mvb200 import synth
from oracle import stage1_port as P


def _load(golden_dir, name):
    return np.load(f"{golden_dir}/{name}.npz")


def _dims_from(g):
    return synth.Stage1Dims(n_layer=int(g["n_layer"]), n_head=int(g["n_head"]), dim=int(g["dim"]))


def _teacher_forced_logits(model, g, last_step):
    prompt = torch.from_numpy(g["prompt"]); spk = torch.from_numpy(g["spk"]); toks = torch.from_numpy(g["tokens"])
    T = prompt.numel()
    out = [model.forward(prompt.view(1, -1).repeat(2, 1), spk, torch.arange(T))[:, -1]]
    for s in range(1, last_step + 1):
        out.append(model.forward(toks[s - 1].view(1, 1).repeat(2, 1), spk, torch.tensor([T + s - 1]))[:, -1])
    return out


def test_weights_reproducible(golden_dir):
    g = _load(golden_dir, "stage1_tiny")
    sd = synth.stage1_state_dict(_dims_from(g), int(g["weight_seed"]))
    assert synth.state_dict_checksum(sd) == pytest.approx(float(g["weight_checksum"]), rel=0, abs=1e-9)


def test_port_matches_reference_golden_tiny(golden_dir):
    g = _load(golden_dir, "stage1_tiny")
    d = _dims_from(g)
    m = P.Stage1Oracle(synth.stage1_state_dict(d, int(g["weight_seed"])), d.n_head, d.norm_eps, torch.float32)
    m.setup_caches()
    steps = [int(s) for s in g["steps"]]
    lg = _teacher_forced_logits(m, g, max(steps))
    for i, s in enumerate(steps):
        ref = torch.from_numpy(g["logits"][i])
        assert (lg[s] - ref).abs().max() / ref.abs().max() < 1e-5


def test_port_sampler_known_answers(golden_dir):
    g = _load(golden_dir, "sampler")
    for c in range(g["idx"].shape[0]):
        gs, temp, tp, tk = g["params"][c]
        logits = torch.from_numpy(g["logits"][c])[:, None, :]
        idx, probs = P.sample(logits, torch.tensor(gs), torch.tensor(temp), None if tp < 0 else torch.tensor(tp),
                              None if tk == 0 else int(tk), q=torch.from_numpy(g["noise"][c]))
        assert int(idx) == int(g["idx"][c])
        np.testing.assert_allclose(probs.numpy(), g["probs"][c], rtol=1e-6, atol=1e-9)


def test_port_generate_reproduces_reference_tokens(golden_dir):
    """Seeded sampling reproduces the reference's token ids (north_star parity clause), here via the noise the
    reference drew, which the golden file recorded for the kept steps, and via the global generator."""
    g = _load(golden_dir, "stage1_tiny")
    d = _dims_from(g)
    m = P.Stage1Oracle(synth.stage1_state_dict(d, int(g["weight_seed"])), d.n_head, d.norm_eps, torch.float32)
    m.setup_caches()
    torch.manual_seed(1337)
    y = P.generate(m, torch.from_numpy(g["prompt"]), torch.from_numpy(g["spk"]), max_new_tokens=len(g["tokens"]),
                   end_of_audio_token=9999, guidance_scale=float(g["guidance"]), temperature=float(g["temperature"]),
                   top_p=float(g["top_p"]))
    assert y[len(g["prompt"]):].tolist() == g["tokens"].tolist()


def test_port_matches_reference_golden_full_prefill_and_first_steps(golden_dir):
    g = _load(golden_dir, "stage1_full")
    d = _dims_from(g)
    sd = synth.stage1_state_dict(d, int(g["weight_seed"]))
    assert synth.state_dict_checksum(sd) == pytest.approx(float(g["weight_checksum"]), rel=0, abs=1e-9)
    m = P.Stage1Oracle(sd, d.n_head, d.norm_eps, torch.float32, faithful_full_cache=False)
    m.setup_caches()
    lg = _teacher_forced_logits(m, g, 1)
    for i, s in enumerate([int(s) for s in g["steps"]]):
        if s > 1:
            continue
        ref = torch.from_numpy(g["logits"][i])
        assert (lg[s] - ref).abs().max() / ref.abs().max() < 1e-5


def test_prompt_too_long_raises():
    d = synth.TINY
    m = P.Stage1Oracle(synth.stage1_state_dict(d, 0), d.n_head)
    m.setup_caches()
    with pytest.raises(ValueError, match="Prompt is too long"):
        P.generate(m, synth.synthetic_prompt(2048), synth.synthetic_speaker(), guidance_scale=3.0, temperature=1.0)


def test_port_matches_live_reference(golden_dir):
    """The reference's own Transformer forward and generate() on the same weights and inputs, as recorded by
    oracle/make_golden_reference.py."""
    g = _load(golden_dir, "reference_checks")
    d = synth.TINY
    sd = synth.stage1_state_dict(d, 3)
    assert synth.state_dict_checksum(sd) == pytest.approx(float(g["s1_checksum"]), rel=0, abs=1e-9)
    m = P.Stage1Oracle(sd, d.n_head, d.norm_eps, torch.float32); m.setup_caches()
    prompt = torch.from_numpy(g["s1_prompt"]); spk = torch.from_numpy(g["s1_spk"])
    idx = prompt.view(1, -1).repeat(2, 1)
    with torch.no_grad():
        a = torch.from_numpy(g["s1_logits"]); b = m.forward(idx, spk, torch.arange(9))
    assert (a - b).abs().max() < 1e-5
    ya = torch.from_numpy(g["s1_tokens"])
    m2 = P.Stage1Oracle(sd, d.n_head, d.norm_eps, torch.float32); m2.setup_caches()
    torch.manual_seed(5)
    yb = P.generate(m2, prompt, spk, max_new_tokens=12, end_of_audio_token=9999, temperature=0.8, top_p=0.9,
                    guidance_scale=2.0)
    assert ya.tolist() == yb.tolist()
