"""ORACLE (test infrastructure, never the product path): CPU restatement of the reference's stage-2 path.

  * input builder of ``Model.non_causal_sample``            fam/llm/inference.py:264-306
  * ``GPT.forward`` with ``causal=False``                    fam/llm/model.py:195-314
  * ``Block`` / ``SelfAttention`` / ``MLP`` / ``RMSNorm``    fam/llm/layers/combined.py:40-52, attn.py:122-185,
                                                             layers.py:20-72
  * ``_non_causal_sample``                                   fam/llm/mixins/non_causal.py:15-67
  * ``FlattenedInterleavedEncodec2Codebook.decode``          fam/llm/adapters/flattened_encodec.py:8-32
  * ``TiltedEncodec.decode``                                 fam/llm/adapters/tilted_encodec.py:8-39

Pinned by tests/test_oracle_pinned_stage2.py against tests/golden/stage2.npz, produced from the reference's own
``GPT`` by oracle/make_golden_stage2.py.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

PAD = 1024  # _encodec_codes_pad_token / END_OF_AUDIO_TOKEN of the adapters (fast_inference.py:39, inference.py:125)


# ---- adapters (integer, host) ---------------------------------------------------------------------
def flattened_interleaved_decode(tokens: Sequence[int], eoa: int = PAD) -> Tuple[List[int], List[List[int]]]:
    """flattened_encodec.py:8-32: bucket the flat stage-1 stream by VALUE range, not by position."""
    text, cb = [], [[], []]
    for t in tokens:
        if t < eoa:
            cb[0].append(t)
        elif t < 2 * eoa:
            cb[1].append(t - eoa)
        elif t > 2 * eoa:          # t == 2*eoa is the end-of-audio token and is dropped
            text.append(t)
    n = min(len(cb[0]), len(cb[1]))
    return text[:-1], [cb[0][:n], cb[1][:n]]


def tilted_decode(hier: Sequence[Sequence[int]], eoa: int = PAD) -> Tuple[List[int], List[List[int]]]:
    """tilted_encodec.py:8-39: hierarchy 0 also carries text (> eoa); keep codes < eoa, truncate to the shortest."""
    text = [t for t in hier[0] if t > eoa]
    out = [[t for t in hier[0] if t < eoa]] + [[t for t in h if t < eoa] for h in hier[1:]]
    n = min(len(x) for x in out)
    return text[:-1], [x[:n] for x in out]


# ---- input builder --------------------------------------------------------------------------------
def build_input(text_ids: Sequence[int], cb0: Sequence[int], cb1: Sequence[int], block_size: int) -> torch.Tensor:
    """inference.py:283-301: two hierarchies, padded with 1024 / cut to block_size -> int64 [2, block_size]."""
    h0 = list(text_ids) + list(cb0) + [PAD]
    h1 = [PAD] * len(text_ids) + list(cb1) + [PAD]
    rows = []
    for h in (h0, h1):
        h = h + [PAD] * (block_size - len(h)) if len(h) < block_size else h[:block_size]
        rows.append(h)
    return torch.tensor(rows, dtype=torch.long)


class Stage2Oracle:
    def __init__(self, sd: Dict[str, torch.Tensor], n_head: int, eps: float, dtype=torch.float32):
        cv = lambda t: t.to(dtype).contiguous()
        self.n_head, self.eps = n_head, eps
        self.wtes = []
        while f"transformer.wtes.{len(self.wtes)}.weight" in sd:
            self.wtes.append(cv(sd[f"transformer.wtes.{len(self.wtes)}.weight"]))
        self.wpe = cv(sd["transformer.wpe.weight"])
        self.w_spk = cv(sd["speaker_cond_pos.weight"])
        self.ln_f = cv(sd["transformer.ln_f.weight"])
        self.heads = []
        while f"lm_heads.{len(self.heads)}.weight" in sd:
            self.heads.append(cv(sd[f"lm_heads.{len(self.heads)}.weight"]))
        self.layers = []
        while f"transformer.h.{len(self.layers)}.ln_1.weight" in sd:
            p = f"transformer.h.{len(self.layers)}."
            self.layers.append({k: cv(sd[p + n]) for k, n in dict(
                g1="ln_1.weight", g2="ln_2.weight", qkv="attn.c_attn.weight", o="attn.c_proj.weight",
                w1="mlp.swiglu.w1.weight", w3="mlp.swiglu.w3.weight", w2="mlp.c_proj.weight").items()})
        self.block_size = self.wpe.shape[0]

    def _norm(self, x, g):  # layers.py:20-30 (no fp32 upcast in the slow path)
        return x * torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + self.eps) * g

    @torch.no_grad()
    def forward(self, idx: torch.Tensor, spk: Optional[torch.Tensor]) -> List[torch.Tensor]:
        """idx int64 [b, 2, t]; spk [b, 1, spk_dim] -> list of 6 logits [b, t, V_target] (model.py:232-311)."""
        b, nh_in, t = idx.shape
        x = sum(w[idx[:, i]] for i, w in enumerate(self.wtes)) + self.wpe[torch.arange(t)]
        if spk is not None:
            x = x + spk.to(x.dtype) @ self.w_spk.t()                      # spk_emb_on_text=True: all positions
        E = x.shape[-1]
        hs = E // self.n_head
        for L in self.layers:
            n = self._norm(x, L["g1"])
            q, k, v = (n @ L["qkv"].t()).view(b, t, 3, self.n_head, hs).unbind(2)   # attn.py:175,136-140
            q, k, v = (z.transpose(1, 2) for z in (q, k, v))
            att = torch.softmax((q @ k.transpose(-1, -2)) / math.sqrt(hs), dim=-1) @ v   # non-causal, no padding mask
            x = x + att.transpose(1, 2).reshape(b, t, E) @ L["o"].t()
            n = self._norm(x, L["g2"])
            x = x + (F.silu(n @ L["w1"].t()) * (n @ L["w3"].t())) @ L["w2"].t()
        x = self._norm(x, self.ln_f)
        return [x @ h.t() for h in self.heads]


@torch.no_grad()
def non_causal_sample(logits: List[torch.Tensor], temperature: float, top_k: Optional[int],
                      noise: Optional[List[torch.Tensor]] = None) -> torch.Tensor:
    """non_causal.py:36-67.  ``noise[h]`` [b, t, V] replaces the Exp(1) draws torch.multinomial makes internally
    (its n_sample == 1 path is argmax(p / q), q ~ Exp(1)).  Returns int64 [b, 6, t]."""
    outs = []
    for h, lg in enumerate(logits):
        lg = lg / temperature
        if top_k is not None:
            v, _ = torch.topk(lg, min(top_k, lg.size(-1)))
            lg = lg.masked_fill(lg < v[:, :, [-1]], -float("inf"))
        probs = F.softmax(lg, dim=-1)
        rows = []
        for bi in range(probs.shape[0]):
            q = torch.empty_like(probs[bi]).exponential_(1) if noise is None else noise[h][bi]
            rows.append(torch.argmax(probs[bi] / q, dim=-1))
        outs.append(torch.stack(rows))
    return torch.stack(outs, dim=1)
