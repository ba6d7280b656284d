"""ORACLE TOOLING (test infrastructure, NOT product code): import the REAL reference package.

Search order: `oracle/_ref` (the package byte-compiled by oracle/build_ref.py during `__graft_entry__.build()`), then the LightX2V
checkout named by the environment variable LIGHTX2V_REFERENCE; the tests that need the package skip when neither exists.  The
reference needs `DTYPE=BF16` / `ENABLE_GRAPH_MODE=false` in the environment before import (lightx2v/utils/envs.py) and, on a box
WITHOUT a GPU, the two shims of SURVEY.md §8c (torch.cuda.get_device_capability at import time; pin_memory allocations in every
op's load()).  On the GPU box no shim is installed: the reference runs as it ships."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_state = {"done": False, "ok": False, "where": None}


class Cfg(dict):
    """EasyDict stand-in (easydict is not installed): dict with attribute access, as the reference's config objects."""

    __getattr__ = dict.__getitem__


def available() -> bool:
    return _find() is not None


def _find():
    for base in (os.path.join(ROOT, "oracle", "_ref"), os.environ.get("LIGHTX2V_REFERENCE")):
        if base and os.path.isdir(os.path.join(base, "lightx2v")):
            return base
    return None


def import_reference() -> bool:
    """True when `import lightx2v` works afterwards (op registries populated)."""
    if _state["done"]:
        return _state["ok"]
    _state["done"] = True
    base = _find()
    if base is None:
        return False
    os.environ["DTYPE"] = "BF16"
    os.environ.setdefault("ENABLE_GRAPH_MODE", "false")
    import torch

    if not torch.cuda.is_available():
        torch.cuda.get_device_capability = lambda *a, **k: (10, 0)
        _empty = torch.empty

        def empty_nopin(*a, **k):
            k.pop("pin_memory", None)
            return _empty(*a, **k)

        torch.empty = empty_nopin
    if base not in sys.path:
        sys.path.insert(0, base)
    try:
        import lightx2v.common.ops  # noqa: F401  registers MM/ATTN/RMS/LN/TENSOR op classes (common/ops/__init__.py)
        from lightx2v.common.ops import attn, conv, mm, norm, tensor  # noqa: F401
    except Exception as ex:  # noqa
        _state["error"] = repr(ex)
        return False
    _state["ok"], _state["where"] = True, base
    return True


def ref_config(dim, num_heads, ffn_dim, num_layers, task="t2v", mm_type=None, attn_type="flash_attn2"):
    """Config the reference's Wan classes read (configs/wan/*.json + set_config defaults)."""
    return Cfg(task=task, num_layers=num_layers, num_heads=num_heads, dim=dim, ffn_dim=ffn_dim, cpu_offload=False,
               mm_config=({} if mm_type is None else {"mm_type": mm_type}), do_mm_calib=False, self_attn_1_type=attn_type, cross_attn_1_type=attn_type,
               cross_attn_2_type=attn_type, model_cls="wan2.1", freq_dim=256, text_len=512, in_dim=16, out_dim=16, enable_cfg=True,
               attention_type=attn_type, feature_caching="NoCaching", parallel_attn_type=None)
