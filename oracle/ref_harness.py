"""ORACLE (test infrastructure): runs the REFERENCE'S OWN stage-1 code from /root/reference on CPU.

Only usable in the build container (the tree does not exist on the GPU box).  Used to (a) pin
``oracle/stage1_port.py`` and (b) generate the golden fixtures under ``tests/golden/``.

Shims needed to import the reference here (SURVEY.md §0 D6, §8c):
  * ``librosa`` is absent and only imported at ``fam/llm/utils.py:8`` -> empty stub module;
  * ``get_default_dtype()`` returns "float16" without CUDA (``fam/llm/utils.py:83-84``), which makes the
    reference's own KV cache dtype disagree with its weights -> we set ``config.dtype`` before
    ``setup_caches`` (``fam/llm/fast_model.py:144-146``).
"""
from __future__ import annotations

import os
import sys
import types
from typing import Dict

import torch

_VENDORED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def _resolve_root() -> str:
    """/root/reference in the build container; on the GPU box the byte-identical copy oracle/build_ref.py made
    (oracle/_ref, git-ignored, travels with the snapshot)."""
    env = os.environ.get("MVB_REFERENCE_ROOT")
    if env:
        return env
    if os.path.isdir("/root/reference/fam/llm"):
        return "/root/reference"
    return _VENDORED


REFERENCE_ROOT = _resolve_root()


def runnable() -> bool:
    """The reference's code can be imported here (mounted tree or the vendored copy): gates bench.py's reference arm."""
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "fam", "llm"))


def _import_reference():
    if not runnable():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT} (run oracle/build_ref.py in the build container)")
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    if "librosa" not in sys.modules:
        import importlib.machinery
        stub = types.ModuleType("librosa")
        stub.__spec__ = importlib.machinery.ModuleSpec("librosa", None)   # keep importlib.util.find_spec() callers happy
        sys.modules["librosa"] = stub
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import fam.llm.utils as fu
        fu.get_default_dtype = lambda: "bfloat16"
        import fam.llm.fast_model as fm
        fm.get_default_dtype = lambda: "bfloat16"
        import fam.llm.fast_inference_utils as fiu
    return fm, fiu


def rename_to_fast(sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """Apply the reference's own rename rules by calling the same string ops it performs
    (fast_inference_utils.py:246-278) on a copy of the checkpoint dict."""
    out = {}
    table = [(".attn.c_attn.", ".attention.wqkv."), (".attn.c_proj.", ".attention.wo."),
             (".mlp.swiglu.w1.", ".feed_forward.swiglu.w1."), (".mlp.swiglu.w3.", ".feed_forward.swiglu.w3."),
             (".ln_1.", ".attention_norm."), (".ln_2.", ".ffn_norm."), (".mlp.c_proj.", ".feed_forward.w2.")]
    top = {"transformer.wtes.0.weight": "tok_embeddings.weight", "transformer.wpe.weight": "pos_embeddings.weight",
           "lm_heads.0.weight": "output.weight", "transformer.ln_f.weight": "norm.weight"}
    for k, v in sd.items():
        if k.startswith("_orig_mod."):
            k = k[len("_orig_mod."):]
        if k in top:
            out[top[k]] = v
            continue
        k = k.replace("transformer.h.", "layers.")
        for a, b in table:
            k = k.replace(a, b)
        out[k] = v
    return out


def build_reference_model(state_dict: Dict[str, torch.Tensor], dims, dtype: torch.dtype = torch.float32):
    """Instantiate the reference ``Transformer`` with ``dims`` and load the (renamed) weights."""
    fm, _ = _import_reference()
    args = fm.ModelArgs(block_size=dims.block_size, vocab_size=dims.vocab_size, n_layer=dims.n_layer,
                        n_head=dims.n_head, dim=dims.dim, speaker_emb_dim=dims.speaker_emb_dim,
                        norm_eps=dims.norm_eps)
    assert args.intermediate_size == dims.intermediate_size
    with torch.device("meta"):
        model = fm.Transformer(args)
    model.load_state_dict(rename_to_fast(state_dict), assign=True)
    model = model.to(dtype=dtype).eval()
    model.config.dtype = dtype                      # D6: keep the KV cache dtype equal to the weights'
    model.setup_spk_cond_mask()
    model.setup_caches(max_batch_size=2, max_seq_length=args.block_size)
    return model


def reference_functions():
    """The reference's own sampler / generate functions (fast_inference_utils.py)."""
    _, fiu = _import_reference()
    return fiu


def load_model_via_reference_loader(ckpt_path: str):
    """Exercise the reference's own ``_load_model`` key handling on a full-size synthetic checkpoint.
    (The speaker-encoder half of ``_load_model`` needs librosa at call time and is skipped by
    replaying lines 236-281 only.)"""
    fm, _ = _import_reference()
    with torch.device("meta"):
        model = fm.Transformer.from_name("metavoice-1B")
    ckpt = torch.load(ckpt_path, mmap=True, weights_only=False)
    model.load_state_dict(rename_to_fast(ckpt["model"]), assign=True)
    return model.to(dtype=torch.bfloat16).eval(), ckpt
