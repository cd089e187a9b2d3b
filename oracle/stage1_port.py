"""ORACLE (test infrastructure, never the product path): CPU restatement of the reference's
stage-1 causal LM and sampler, in plain torch on the host.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl reference``
legs may import this file.  It follows, function by function:

  * ``fam/llm/fast_model.py:116-167``  Transformer.forward (learned positions, speaker CFG mask)
  * ``fam/llm/fast_model.py:97-113``   KVCache.update (scatter at input_pos, attend to the whole cache)
  * ``fam/llm/fast_model.py:184-227``  Attention.forward (fused wqkv, MHA, SDPA with boolean mask)
  * ``fam/llm/fast_model.py:230-261``  SwiGLU / FeedForward / RMSNorm (fp32 upcast, cast back, then gain)
  * ``fam/llm/fast_inference_utils.py:61-120``   sampler (CFG mix, temperature, top-k, top-p, exp-race)
  * ``fam/llm/fast_inference_utils.py:123-228``  prefill / decode_one_token / decode_n_tokens / generate
  * ``fam/llm/fast_inference_utils.py:246-278``  checkpoint key mapping

Pinning: ``tests/test_oracle_pinned.py`` checks this port against the committed golden vectors produced
by ``oracle/make_golden.py`` and ``oracle/make_golden_reference.py`` from the reference's own code.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn.functional as F


def _strip_prefix(sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    # fast_inference_utils.py:246-249: checkpoints saved from a compiled module carry "_orig_mod."
    return {(k[len("_orig_mod."):] if k.startswith("_orig_mod.") else k): v for k, v in sd.items()}


class Stage1Oracle:
    """Functional restatement of the reference stage-1 model for one utterance (2 CFG rows).

    ``dtype`` selects the arithmetic type of weights/activations/cache (torch.float32 for the
    tier-1 parity oracle, torch.bfloat16 to mimic the reference's production precision).
    """

    def __init__(self, state_dict: Dict[str, torch.Tensor], n_head: int, norm_eps: float = 1e-5,
                 dtype: torch.dtype = torch.float32, faithful_full_cache: bool = True):
        sd = _strip_prefix(state_dict)
        cv = lambda t: t.to(dtype).contiguous()
        self.dtype = dtype
        self.tok_emb = cv(sd["transformer.wtes.0.weight"])      # -> tok_embeddings (utils:250)
        self.pos_emb = cv(sd["transformer.wpe.weight"])         # -> pos_embeddings (utils:251)
        self.w_out = cv(sd["lm_heads.0.weight"])                # -> output         (utils:252)
        self.g_out = cv(sd["transformer.ln_f.weight"])          # -> norm           (utils:253)
        self.w_spk = cv(sd["speaker_cond_pos.weight"])
        self.layers = []
        i = 0
        while f"transformer.h.{i}.ln_1.weight" in sd:
            p = f"transformer.h.{i}."
            self.layers.append(dict(
                g_attn=cv(sd[p + "ln_1.weight"]),                # attention_norm (utils:270-272)
                w_qkv=cv(sd[p + "attn.c_attn.weight"]),          # attention.wqkv (utils:258-260)
                w_o=cv(sd[p + "attn.c_proj.weight"]),            # attention.wo   (utils:261-263)
                g_ffn=cv(sd[p + "ln_2.weight"]),                 # ffn_norm       (utils:273-275)
                w1=cv(sd[p + "mlp.swiglu.w1.weight"]),
                w3=cv(sd[p + "mlp.swiglu.w3.weight"]),
                w2=cv(sd[p + "mlp.c_proj.weight"]),              # feed_forward.w2 (utils:276-278)
            ))
            i += 1
        self.n_layer = len(self.layers)
        self.n_head = n_head
        self.dim = self.tok_emb.shape[1]
        self.head_dim = self.dim // n_head
        self.vocab = self.w_out.shape[0]
        self.block_size = self.pos_emb.shape[0]
        self.eps = norm_eps
        self.faithful_full_cache = faithful_full_cache
        self.max_seq = 0
        self.k_cache: List[torch.Tensor] = []
        self.v_cache: List[torch.Tensor] = []

    # fast_model.py:136-148
    def setup_caches(self, max_batch_size: int = 2, max_seq_length: Optional[int] = None) -> None:
        max_seq_length = max_seq_length or self.block_size
        max_seq_length = (max_seq_length + 7) // 8 * 8  # find_multiple(max_seq_length, 8)
        self.max_seq = max_seq_length
        shape = (max_batch_size, self.n_head, max_seq_length, self.head_dim)
        self.k_cache = [torch.zeros(shape, dtype=self.dtype) for _ in range(self.n_layer)]
        self.v_cache = [torch.zeros(shape, dtype=self.dtype) for _ in range(self.n_layer)]
        self.causal = torch.tril(torch.ones(max_seq_length, max_seq_length, dtype=torch.bool))

    # fast_model.py:250-261
    def _rmsnorm(self, x: torch.Tensor, gain: torch.Tensor) -> torch.Tensor:
        xf = x.float()
        n = xf * torch.rsqrt(torch.mean(xf * xf, dim=-1, keepdim=True) + self.eps)
        return n.to(x.dtype) * gain

    def _attend(self, li: int, q, k, v, input_pos, mask):
        # fast_model.py:104-113: scatter, then attention sees the WHOLE cache through the mask
        self.k_cache[li][:, :, input_pos] = k
        self.v_cache[li][:, :, input_pos] = v
        if self.faithful_full_cache:
            K, V, m = self.k_cache[li], self.v_cache[li], mask
        else:  # identical numerics (masked slots get exactly zero weight), fewer bytes
            hi = int(input_pos.max()) + 1
            K, V, m = self.k_cache[li][:, :, :hi], self.v_cache[li][:, :, :hi], mask[..., :hi]
        # fast_model.py:222: F.scaled_dot_product_attention(q, k, v, attn_mask=mask), default scale
        s = (q @ K.transpose(-1, -2)) * (1.0 / math.sqrt(self.head_dim))
        s = s.masked_fill(~m, float("-inf"))
        return torch.softmax(s, dim=-1) @ V

    # fast_model.py:150-163
    @torch.no_grad()
    def forward(self, idx: torch.Tensor, spk_emb: torch.Tensor, input_pos: torch.Tensor,
                taps: Optional[dict] = None) -> torch.Tensor:
        B, S = idx.shape
        assert B == 2, "the reference fast path is hard-wired to {cond, uncond} rows (fast_model.py:132-134)"
        input_pos = input_pos.long()
        mask = self.causal[None, None, input_pos]                              # [1,1,S,max_seq]
        spk_mask = torch.zeros((2, 1, self.dim), dtype=torch.bool)
        spk_mask[0] = True                                                      # fast_model.py:132-134
        x = (self.tok_emb[idx.long()] + self.pos_emb[input_pos]
             + (spk_emb.to(self.dtype) @ self.w_spk.t()) * spk_mask)
        H, hd = self.n_head, self.head_dim
        for li, L in enumerate(self.layers):
            n = self._rmsnorm(x, L["g_attn"])
            q, k, v = (n @ L["w_qkv"].t()).split([self.dim, self.dim, self.dim], dim=-1)
            q, k, v = (t.view(B, S, H, hd).transpose(1, 2) for t in (q, k, v))
            y = self._attend(li, q, k, v, input_pos, mask)
            y = y.transpose(1, 2).contiguous().view(B, S, self.dim)
            x = x + y @ L["w_o"].t()                                            # fast_model.py:179
            n = self._rmsnorm(x, L["g_ffn"])
            x = x + (F.silu(n @ L["w1"].t()) * (n @ L["w3"].t())) @ L["w2"].t()  # fast_model.py:180
            if taps is not None:
                taps[f"x{li}"] = x.float().clone()
        return self._rmsnorm(x, self.g_out) @ self.w_out.t()                    # fast_model.py:161-163


# ----------------------------------------------------------------------------- sampler
# fast_inference_utils.py:61-65
def exp_race_argmax(probs: torch.Tensor, q: Optional[torch.Tensor] = None) -> torch.Tensor:
    if q is None:
        q = torch.empty_like(probs).exponential_(1)
    return torch.argmax(probs / q, dim=-1, keepdim=True).to(dtype=torch.int)


# fast_inference_utils.py:68-82
def top_p_filter(logits: torch.Tensor, top_p: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    sorted_logits, sorted_indices = torch.sort(logits, descending=False)
    cumulative = sorted_logits.softmax(dim=-1).cumsum(dim=-1)
    drop_sorted = cumulative <= (1 - top_p)
    drop_sorted[-1:] = 0                                   # always keep the most likely token
    drop = drop_sorted.scatter(0, sorted_indices, drop_sorted)
    return logits.masked_fill(drop, -float("Inf")), ~drop


# fast_inference_utils.py:85-104
def logits_to_probs(logits, *, temperature, top_p=None, top_k=None):
    logits = logits / torch.max(temperature, 1e-5 * torch.ones_like(temperature))
    kept = torch.ones_like(logits, dtype=torch.bool)
    if top_k is not None:
        v, _ = torch.topk(logits, min(int(top_k), logits.size(-1)))
        pivot = v.select(-1, -1).unsqueeze(-1)
        kept = kept & ~(logits < pivot)
        logits = torch.where(logits < pivot, -float("Inf"), logits)
    if top_p is not None:
        logits, kp = top_p_filter(logits, top_p)
        kept = kept & kp
    return torch.softmax(logits, dim=-1), kept


# fast_inference_utils.py:107-120
def sample(logits: torch.Tensor, guidance_scale, temperature, top_p=None, top_k=None,
           q: Optional[torch.Tensor] = None, return_kept: bool = False):
    """logits [2, S, V] -> (idx int32 [1], probs [V]); q = optional Exp(1) noise [V]."""
    logits = logits[:, -1]
    cond, uncond = logits.split(logits.size(0) // 2, dim=0)
    mixed = guidance_scale * cond + (1 - guidance_scale) * uncond
    probs, kept = logits_to_probs(mixed[0], temperature=temperature, top_p=top_p, top_k=top_k)
    idx = exp_race_argmax(probs, q)
    if return_kept:
        return idx, probs, kept
    return idx, probs


# fast_inference_utils.py:181-228 (+ :123-174)
@torch.no_grad()
def generate(model: Stage1Oracle, prompt: torch.Tensor, spk_emb: torch.Tensor, *,
             max_new_tokens: Optional[int] = None, end_of_audio_token: int = 2048,
             noise: Optional[torch.Tensor] = None, forced: Optional[torch.Tensor] = None,
             logit_sink: Optional[list] = None, **sampling) -> torch.Tensor:
    """Restatement of ``generate``.  ``noise`` [n_steps, V] replaces the generator draws,
    ``forced`` [n_steps] teacher-forces the fed-back token (the sampled one is still returned
    through ``logit_sink``), both are test hooks that do not exist in the reference."""
    T = prompt.size(0)
    max_seq = model.block_size if max_new_tokens is None else min(T + max_new_tokens, model.block_size)
    max_new = max_seq - T
    if max_new <= 0:
        raise ValueError("Prompt is too long to generate more tokens")
    tp = lambda v: None if v is None else torch.as_tensor(v, dtype=model.dtype)
    sk = dict(guidance_scale=tp(sampling["guidance_scale"]), temperature=tp(sampling["temperature"]),
              top_p=tp(sampling.get("top_p")), top_k=sampling.get("top_k"))
    step = 0

    def one(idx2, pos):
        nonlocal step
        logits = model.forward(idx2, spk_emb, pos)
        q = None if noise is None else noise[step].to(logits.dtype)
        tok, _ = sample(logits, q=q, **sk)
        if logit_sink is not None:
            logit_sink.append((logits[:, -1].float().clone(), int(tok)))
        if forced is not None:
            tok = forced[step].view(1).to(torch.int)
        step += 1
        return tok

    seq = [prompt.to(torch.int)]
    cur = one(prompt.view(1, -1).repeat(2, 1), torch.arange(0, T))             # prefill :211
    seq.append(cur.view(1))
    pos = T
    for _ in range(max_new - 1):                                               # decode_n_tokens :160
        if bool((cur == end_of_audio_token).any()):
            break
        cur = one(cur.view(1, -1).repeat(2, 1), torch.tensor([pos]))
        pos += 1
        seq.append(cur.view(1))
    return torch.cat(seq)
