"""Python front-ends of the hand-written sm_100a kernels (``edl_b200/csrc``).

Dispatch rule: CUDA tensors ALWAYS go to the native extension (and fail loudly if it is missing --
a silent eager fallback on a GPU box would hide that the product path is not running); CPU tensors
use small pure-PyTorch reference implementations so the whole stack is testable without a GPU.
"""
from __future__ import annotations

import importlib
import threading

_lock = threading.Lock()
_C = None
_launches = 0  # number of native kernel launches issued through this module (bench bookkeeping)


def native():
    """Return the compiled extension module, importing it on first use."""
    global _C
    if _C is None:
        with _lock:
            if _C is None:
                try:
                    import torch  # noqa: F401  (must be loaded before the extension)

                    _C = importlib.import_module("edl_b200._C")
                except ImportError as e:  # pragma: no cover - exercised only on broken installs
                    raise RuntimeError(
                        "edl_b200 native extension is not built; run `python -m edl_b200.build_ext` "
                        "(or __graft_entry__.build()). Original error: %r" % (e,)
                    )
    return _C


def native_available() -> bool:
    try:
        native()
        return True
    except RuntimeError:
        return False


def count_launch(n: int = 1) -> None:
    global _launches
    _launches += n


def launches() -> int:
    return _launches


def reset_launches() -> None:
    global _launches
    _launches = 0


# ---- library fallbacks on CUDA tensors: counted and logged, never silent -------------------------------------
# A CUDA tensor that one of our kernels cannot take (a shape the TMA descriptor cannot express, a convolution
# geometry without an own kernel yet) runs on the vendor library (cuBLAS / cuDNN through ATen).  That is a
# correctness safety net, not the product: every such call is counted by reason, logged once per reason, and
# bench.py prints the table as ``library_fallbacks`` (the flagship step must show none it does not name).
_fallbacks = {}


def count_fallback(reason: str, n: int = 1) -> None:
    first = reason not in _fallbacks
    _fallbacks[reason] = _fallbacks.get(reason, 0) + n
    if first:
        import logging

        logging.getLogger("edl_b200").warning("library fallback on a CUDA tensor: %s", reason)
    import os

    if os.environ.get("EDL_STRICT_NATIVE", "0") == "1":
        raise RuntimeError("EDL_STRICT_NATIVE=1: library fallback on a CUDA tensor: " + reason)


def fallbacks() -> dict:
    return dict(_fallbacks)


def reset_fallbacks() -> None:
    _fallbacks.clear()


from .bn import batch_norm_act, BatchNormAct2d, scale_shift_act, bn_stats_into, set_fused_bn, drop_bn_hook  # noqa: E402
from .loss import soft_cross_entropy, topk_accuracy  # noqa: E402
from .pool import max_pool_3x3_s2, avg_pool_2x2, global_avg_pool  # noqa: E402
from .optim import FlatSGDMomentum, FlatAdam, FlatLARS, FlatLAMB  # noqa: E402
from .gemm import stem7_infer, stem7_supported  # noqa: E402
from .gemm import (gemm_bf16, linear_bf16, conv1x1, conv_lib, conv3x3, conv3x3_supported, conv3x3_infer,  # noqa: E402
                   conv3x3_infer_supported, conv3x3_wgrad, conv3x3_wgrad_supported, conv3x3_s2, conv3x3_s2_infer,
                   conv3x3_s2_supported, stem_conv, stem_conv_supported, conv3x3_pair, conv3x3_pair_supported)
from .misc import rope, rope_tables, embedding_bag_mean, normalize_u8, DynamicLossScaler  # noqa: E402

__all__ = [
    "native", "native_available", "launches", "reset_launches", "count_fallback", "fallbacks", "reset_fallbacks",
    "batch_norm_act", "BatchNormAct2d", "scale_shift_act", "bn_stats_into",
    "soft_cross_entropy", "topk_accuracy",
    "max_pool_3x3_s2", "avg_pool_2x2", "global_avg_pool",
    "FlatSGDMomentum", "FlatAdam", "FlatLARS", "FlatLAMB", "gemm_bf16", "linear_bf16", "conv1x1", "conv_lib", "conv3x3",
    "conv3x3_supported", "conv3x3_infer", "conv3x3_infer_supported", "stem7_infer", "stem7_supported",
    "conv3x3_wgrad", "conv3x3_wgrad_supported", "conv3x3_s2", "conv3x3_s2_infer", "conv3x3_s2_supported",
    "stem_conv", "stem_conv_supported", "conv3x3_pair", "conv3x3_pair_supported",
    "rope", "rope_tables", "embedding_bag_mean", "normalize_u8", "DynamicLossScaler", "set_fused_bn", "drop_bn_hook",
]
