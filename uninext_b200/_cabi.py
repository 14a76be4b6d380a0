"""ctypes binding of libmsda_b200.so (the C ABI in include/msda_b200.h).

There is NO fallback: if the library is missing or does not export every declared symbol, importing the ops fails
with a RuntimeError that says how to build it. The product never routes through ``oracle/`` or a PyTorch
re-implementation.
"""
from __future__ import annotations

import ctypes
import os

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "lib", "libmsda_b200.so")

_vp, _i, _u64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64
_DIMS = [_i] * 7

# name -> (restype, argtypes); mirrors include/msda_b200.h one to one (tests/test_cabi_symbols.py checks it).
SIGNATURES = {
    "msda_abi_version": (_i, []),
    "msda_strerror": (ctypes.c_char_p, [_i]),
    "msda_uses_fast_path": (_i, [_i, _i, _i, _i]),
    "msda_launch_count": (_u64, []),
    "msda_set_knob": (_i, [_i, _i]),
    "msda_forward_f32": (_i, [_vp] * 5 + _DIMS + [_vp, _vp]),
    "msda_forward_f64": (_i, [_vp] * 5 + _DIMS + [_vp, _vp]),
    "msda_forward_bf16": (_i, [_vp] * 5 + _DIMS + [_vp, _vp]),
    "msda_backward_f32": (_i, [_vp] * 6 + _DIMS + [_vp] * 3 + [_vp]),
    "msda_backward_f64": (_i, [_vp] * 6 + _DIMS + [_vp] * 3 + [_vp]),
    "msda_backward_bf16": (_i, [_vp] * 6 + _DIMS + [_vp] * 4 + [_vp]),
    "msda_backward_det_f32": (_i, [_vp] * 6 + _DIMS + [_vp] * 4 + [_vp]),
    "msda_backward_det_bf16": (_i, [_vp] * 6 + _DIMS + [_vp] * 5 + [_vp]),
    "msda_prologue_forward_f32": (_i, [_vp] * 3 + [ctypes.c_int64, _i, _i, _i, _i] + [_vp] * 3),
    "msda_prologue_backward_f32": (_i, [_vp] * 5 + [ctypes.c_int64, _i, _i, _i, _i] + [_vp] * 2),
    "msda_colsum_f32": (_i, [_vp, ctypes.c_int64, _i, _vp, _vp]),
    "msda_relu_backward_colsum_f32": (_i, [_vp, _vp, ctypes.c_int64, _i, _vp, _vp, _vp]),
    "msda_colsum_det_scratch_bytes": (_i, [ctypes.c_int64, _i, _vp]),
    "msda_layernorm_backward_det_scratch_bytes": (_i, [ctypes.c_int64, _i, _vp]),
    "msda_colsum_det_f32": (_i, [_vp, ctypes.c_int64, _i, _vp, _vp, _vp]),
    "msda_relu_backward_colsum_det_f32": (_i, [_vp, _vp, ctypes.c_int64, _i, _vp, _vp, _vp, _vp]),
    "msda_layernorm_backward_det_f32": (_i, [_vp] * 5 + [ctypes.c_int64, _i] + [_vp] * 5),
    "msda_add_layernorm_forward_f32": (_i, [_vp] * 4 + [ctypes.c_int64, _i, ctypes.c_float] + [_vp] * 5),
    "msda_layernorm_backward_f32": (_i, [_vp] * 5 + [ctypes.c_int64, _i] + [_vp] * 4),
    "msda_linear_tf32": (_i, [_vp] * 3 + [ctypes.c_int64, _i, _i, _vp, _vp]),
    "msda_linear_tf32_ex": (_i, [_vp] * 4 + [ctypes.c_int64, _i, _i, _i, _vp, _vp]),
    "msda_linear_tf32_ws_ok": (_i, [_i, _i]),
    "msda_valid_counts": (_i, [_vp] * 3 + [_i] * 3 + [_vp, _vp]),
    "msda_encoder_ref_points_f32": (_i, [_vp] * 3 + [_i] * 3 + [_vp, _vp]),
    "msda_encoder_proposals_f32": (_i, [_vp] * 4 + [_i] * 3 + [ctypes.c_float, _vp, _vp, _vp]),
    "msda_sine_pos_embed_forward_f32": (_i, [_vp, ctypes.c_int64, _i, _i, ctypes.c_float, _i, _vp, _vp]),
    "msda_sine_pos_embed_backward_f32": (_i, [_vp, _vp, ctypes.c_int64, _i, _i, ctypes.c_float, _i, _vp, _vp]),
    "msda_condinst_forward_f32": (_i, [_vp] * 4 + [_i] * 7 + [_vp, _vp]),
    "msda_condinst_backward_f32": (_i, [_vp] * 5 + [_i] * 7 + [_vp] * 4),
    "msda_condinst_backward_det_scratch_bytes": (_i, [_i] * 5 + [_vp]),
    "msda_condinst_backward_det_f32": (_i, [_vp] * 5 + [_i] * 7 + [_vp] * 5),
    "msda_aligned_bilinear_forward_f32": (_i, [_vp, ctypes.c_int64, _i, _i, _i, _vp, _vp]),
    "msda_aligned_bilinear_backward_f32": (_i, [_vp, ctypes.c_int64, _i, _i, _i, _vp, _vp]),
    "msda_debug_gemm_timeline": (_i, [_vp, _i]),
}
ABI_VERSION = 3
DET_HEADER_WORDS = 4                                                                                  # MSDA_DET_HEADER_WORDS
(KNOB_SLAB, KNOB_BWD_WIN_ROWS, KNOB_BWD_LIST_CAP, KNOB_FWD_SLAB_CTAS, KNOB_F32_VEC8_FWD, KNOB_F32_VEC8_BWD,
 KNOB_BF16_FINE_ROWS, KNOB_BF16_PACKED_FWD, KNOB_ZERO_FILL) = range(9)                                                      # include/msda_b200.h

_lib = None


def scratch_bytes(query, *args) -> int:
    """Bytes of scratch a deterministic entry point needs, from its host-only query function."""
    out = ctypes.c_int64(0)
    check(query(*args, ctypes.byref(out)), query.__name__)
    return out.value


class MSDALibraryError(RuntimeError):
    pass


def load(path: str | None = None):
    """Load (once) and type the library. Raises MSDALibraryError loudly when it is absent or stale."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise MSDALibraryError(
            f"{p} not found: the CUDA extension is not built. Run `python -m uninext_b200.build` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU / PyTorch fallback.")
    try:
        lib = ctypes.CDLL(p)
    except OSError as exc:
        raise MSDALibraryError(f"cannot load {p}: {exc}") from exc
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:
            raise MSDALibraryError(f"{p} does not export `{name}` (stale build? run uninext_b200.build --force)") from exc
        fn.restype, fn.argtypes = res, args
    if lib.msda_abi_version() != ABI_VERSION:
        raise MSDALibraryError(f"{p}: ABI version {lib.msda_abi_version()} != expected {ABI_VERSION}")
    if path is None:
        _lib = lib
    return lib


def check(code: int, what: str) -> None:
    """Turn a non-zero C-ABI return code into a RuntimeError (the reference only printf()s launch failures,
    ms_deform_im2col_cuda.cuh:948-952)."""
    if code != 0:
        msg = load().msda_strerror(code)
        raise RuntimeError(f"{what} failed with code {code}: {msg.decode() if msg else '?'}")
