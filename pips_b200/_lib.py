"""ctypes binding of libpips_b200.so (the C ABI declared in include/pips_b200.h).

The CUDA library is the product: if it cannot be loaded this module raises -- there is no CPU or
eager-PyTorch fallback for the refinement hot path.
"""
from __future__ import annotations

import ctypes as C
import os

from . import _build

ABI_VERSION = 3            # PIPS_B200_ABI_VERSION of include/pips_b200.h
DEPTH = 12
LEVELS = 4
KPAD = 576
DIM = 512
HIDDEN = 2048
HEAD = 1040
HEAD_PAD = 1280

FEAT_F32, FEAT_BF16 = 0, 1
PREC_F32, PREC_BF16X3, PREC_BF16 = 0, 1, 2
EPI_BIAS, EPI_BIAS_GELU, EPI_BIAS_RESID = 0, 1, 2
SCORE_TILE = 256           # PIPS_SCORE_TILE: the score-loss grid's pixel rows are padded to a multiple of this

PRECISIONS = {"fp32": PREC_F32, "bf16x3": PREC_BF16X3, "bf16": PREC_BF16}
FEAT_DTYPES = {"fp32": FEAT_F32, "bf16": FEAT_BF16}

_p = C.c_void_p
_i = C.c_int
_f = C.c_float


class LayerWeights(C.Structure):
    _fields_ = [(n, _p) for n in (
        "ln1_w", "ln1_b", "tok_w1", "tok_b1", "tok_w2", "tok_b2", "ln2_w", "ln2_b",
        "fc1_b", "fc2_b", "fc1_w_hi", "fc1_w_lo", "fc2_w_hi", "fc2_w_lo", "fc1_w_f32", "fc2_w_f32")]


class Weights(C.Structure):
    _fields_ = ([(n, _p) for n in ("in_w_hi", "in_w_lo", "in_w_f32", "in_b")]
                + [("layer", LayerWeights * DEPTH)]
                + [(n, _p) for n in ("out_ln_w", "out_ln_b", "head_w_hi", "head_w_lo", "head_w_f32", "head_b",
                                     "gn_w", "gn_b", "upd_w", "upd_b", "vis_w", "vis_b")])


class Workspace(C.Structure):
    _fields_ = ([("rows_alloc", _i), ("seqs_alloc", _i)]
                + [(n, _p) for n in ("x0_hi", "x0_lo", "x0_f32", "x", "y_hi", "y_lo", "y_f32",
                                     "h_hi", "h_lo", "h_f32", "p_hi", "p_lo", "p_f32", "delta")])


MAX_PEERS = 16


class PeerOut(C.Structure):
    _fields_ = [("out", _p * MAX_PEERS), ("n_peers", _i), ("n_offset", _i), ("n_total", _i)]


class Problem(C.Structure):
    _fields_ = [("B", _i), ("S", _i), ("N", _i), ("H", _i), ("W", _i), ("feat_dtype", _i), ("precision", _i),
                ("lvl", _p * LEVELS), ("times", _p), ("coords", _p), ("coords0", _p), ("ffeats", _p), ("stride", _f),
                ("frame_base", _p), ("frames_per_batch", _i), ("peer", PeerOut)]


_SIGNATURES = {
    "pips_abi_version": (_i, []),
    "pips_last_error": (C.c_char_p, []),
    "pips_pyramid_build": (_i, [_p, _i, _i, _i, C.POINTER(_p), C.POINTER(_p), _p]),
    "pips_pyramid_build_nhwc": (_i, [_p, _i, _i, _i, C.POINTER(_p), C.POINTER(_p), _p]),
    "pips_init_gather": (_i, [_p, _i, _i, _i, _i, _i, _p, _p, _i, _p, _p, _p]),
    "pips_corr_gather": (_i, [C.POINTER(_p), _i, _i, _i, _i, _i, _i, _p, _p, _p, _p, _i, _p, _p, _p, _i, _p]),
    "pips_peer_alloc": (_i, [C.c_size_t, C.POINTER(_p), C.c_char_p]),
    "pips_peer_open": (_i, [C.c_char_p, C.POINTER(_p)]),
    "pips_peer_close": (_i, [_p]),
    "pips_peer_free": (_i, [_p]),
    "pips_peer_scatter": (_i, [_p, _i, _i, C.POINTER(_p), _i, _i, _i, _p]),
    "pips_peer_barrier": (_i, [C.POINTER(_p), _i, _i, _i, _i, _p]),
    "pips_update_peer": (_i, [_p] * 9 + [_f, _i, _i, _i, C.POINTER(PeerOut), _p]),
    "pips_heatmap_scratch_floats": (C.c_size_t, [_i, _i, _i, _i]),
    "pips_heatmap": (_i, [C.POINTER(_p), _i, _i, _i, _i, _i, _i, _p, _p, _p, _i, _p, _p, C.c_size_t, _p]),
    "pips_gemm_tc": (_i, [_p, _p, _i, _i, _p, _p, _i, _i, _i, _i, _i, _p, _i, _p, _i, _p, _p, _i, _p]),
    "pips_gemm_f32": (_i, [_p, _i, _p, _i, _i, _i, _i, _p, _i, _p, _i, _p]),
    "pips_tokenmix": (_i, [_p, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "pips_tokenmix_tc": (_i, [_p, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "pips_ln_pool": (_i, [_p, _i, _p, _p, _p, _p, _p, _p]),
    "pips_update": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _f, _i, _i, _i, _p]),
    "pips_vis_head": (_i, [_p, _p, _p, _p, _i, _i, _i, _p]),
    "pips_score_grid": (_i, [C.POINTER(_p), _i, _i, _i, _p, _p]),
    "pips_score_loss_scratch_floats": (C.c_size_t, [_i, _i, _i, _i]),
    "pips_score_loss": (_i, [_p, _i, _i, _i, _i, _i, _p, _p, _i, _i, _i, _i, _p, _p]),
    "pips_score_loss_finalize": (_i, [_p, _i, _i, _i, _i, _p, _p, _p]),
    "pips_split_bf16": (_i, [_p, _p, _p, C.c_size_t, _p]),
    "pips_inorm_stats": (_i, [_p, _i, _i, _i, _p, _i, _p, _p]),
    "pips_inorm_apply": (_i, [_p, _p, _p, _p, _i, _i, _p, _p, _i, _i, _i, _i, _p]),
    "pips_resize_split3": (_i, [_p, _i, _i, _i, _i, _p, _i, _i, _i, _i, _p]),
    "pips_inorm_apply_pair": (_i, [_p, _p, _p, _p, _i, _i, _p, _p, _p, _i, _i, _i, _i, _p]),
    "pips_resize_pair": (_i, [_p, _i, _i, _i, _i, _p, _p, _i, _i, _i, _i, _p]),
    "pips_conv_tc": (_i, [_p, _p, _i, _i, _i, _i, _p, _p, _i, _i, _i, _i, _i, _p, _p, _p]),
    "pips_conv_tc_aniso": (_i, [_p, _p, _i, _i, _i, _i, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p]),
    "pips_stem_pack": (_i, [_p, _i, _i, _i, _i, _p, _p, _p]),
    "pips_conv_tc_chunks": (_i, [_i] * 8),
    "pips_conv_tc_stats": (_i, [_p, _p, _i, _i, _i, _i, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p]),
    "pips_conv_rows_chunks": (_i, [_i, _i]),
    "pips_conv_rows": (_i, [_p, _p, _i, _i, _i, _p, _p, _p, _p, _p]),
    "pips_inorm_finalize": (_i, [_p, _i, _i, _i, _i, _p, _p]),
    "pips_mixer_forward": (_i, [C.POINTER(Weights), C.POINTER(Workspace), _i, _i, _p]),
    "pips_refine_iter": (_i, [C.POINTER(Problem), C.POINTER(Weights), C.POINTER(Workspace), _p, _p]),
}

EXPORTS = tuple(_SIGNATURES)

_lib = None


def lib_path() -> str:
    return _build.LIB


def load(build_if_missing: bool = True):
    """Load (building on first use) the shared library and attach prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if _build.is_stale():
        # missing, or built from other sources than the ones on disk (content digest, not mtimes)
        multi = int(os.environ.get("WORLD_SIZE", "1")) > 1           # ranks of one torchrun must not race on the link step
        if build_if_missing and _build.have_nvcc() and not (multi and os.path.exists(path)):
            _build.build()
        elif not os.path.exists(path):
            raise RuntimeError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
        else:
            import warnings
            warnings.warn(f"{path} was built from different sources than pips_b200/csrc now holds; "
                          "rebuild with `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(path)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here == missing export: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.pips_abi_version() != ABI_VERSION:
        raise RuntimeError("libpips_b200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


class PipsCudaError(RuntimeError):
    pass


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().pips_last_error().decode("utf-8", "replace")
        raise PipsCudaError(f"{what or 'libpips_b200'} failed (rc={rc}): {msg}")


def ptr(t) -> int:
    """Device pointer of a torch tensor (None -> NULL)."""
    return 0 if t is None else t.data_ptr()


def ptr_array(tensors):
    arr = (_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = ptr(t)
    return arr
