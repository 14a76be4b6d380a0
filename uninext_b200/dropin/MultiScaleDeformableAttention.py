"""Drop-in for the reference's compiled module ``MultiScaleDeformableAttention``.

The reference builds a pybind11 extension with this name (ops/setup.py:53, ops/src/vision.cpp:13-16) and imports it at
``ops/functions/ms_deform_attn_func.py:18``. Putting this directory on ``sys.path`` (or calling
``uninext_b200.install_dropin()``) makes that import resolve here, so the reference's ``MSDeformAttnFunction``,
``MSDeformAttn`` and both transformer files run unchanged on the sm_100a kernels.

Exports exactly the reference's two functions with the reference's signatures, checks and error type
(``RuntimeError``; ops/src/ms_deform_attn.h:19-62, ops/src/cuda/ms_deform_attn_cuda.cu:28-52,93-116).
Beyond the reference: bfloat16 ``value`` is accepted (sampling locations / attention weights are then taken as fp32),
and the backward honours ``torch.use_deterministic_algorithms(True)`` (``uninext_b200.determinism``): fp32 / bf16 take the
bit-reproducible kernels, fp64 raises (or warns under ``warn_only``) and runs the normal kernels.
"""
from __future__ import annotations

import torch

from uninext_b200 import _cabi, determinism

__all__ = ["ms_deform_attn_forward", "ms_deform_attn_backward"]

_SUFFIX = {torch.float32: "f32", torch.float64: "f64", torch.bfloat16: "bf16"}


def _checks(named, value, im2col_step):
    for name, t in named:
        if not t.is_contiguous():
            raise RuntimeError(f"{name} tensor has to be contiguous")              # cu:28-32, 93-98
        if not t.is_cuda:
            if name == "value":
                raise RuntimeError("Not implemented on the CPU")                  # ms_deform_attn.h:38
            raise RuntimeError(f"{name} must be a CUDA tensor")                    # cu:34-38, 100-105
    if value.dtype not in _SUFFIX:
        raise RuntimeError(f"ms_deform_attn: unsupported dtype {value.dtype}")      # cu:64 dispatches float/double
    batch = value.size(0)
    step = min(batch, int(im2col_step))
    if step <= 0 or batch % step != 0:
        raise RuntimeError(f"batch({batch}) must divide im2col_step({step})")      # cu:52


def _dims(value, spatial_shapes, sampling_loc):
    n, s, m, d = value.shape
    return (n, s, m, d, spatial_shapes.size(0), sampling_loc.size(1), sampling_loc.size(4))


def _aux_dtype(value):
    return torch.float64 if value.dtype == torch.float64 else torch.float32


def _same_dtype(value, *named):
    want = _aux_dtype(value)
    for name, t in named:
        if t.dtype != want:
            raise RuntimeError(f"{name} must be {want} when value is {value.dtype}, got {t.dtype}")


def _check_shapes(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, grad_output=None):
    """The reference reads every size from the tensors and never cross-checks them (cu:40-48): inconsistent shapes are
    out-of-bounds reads / reds there.  Here they are a RuntimeError before anything is launched."""
    if value.dim() != 4:
        raise RuntimeError(f"value must be [N, S, M, D], got {tuple(value.shape)}")
    n, s, m, d = value.shape
    if spatial_shapes.dim() != 2 or spatial_shapes.size(1) != 2:
        raise RuntimeError(f"spatial_shapes must be [L, 2], got {tuple(spatial_shapes.shape)}")
    l = spatial_shapes.size(0)
    if level_start_index.dim() != 1 or level_start_index.size(0) != l:
        raise RuntimeError(f"level_start_index must be [L] = [{l}], got {tuple(level_start_index.shape)}")
    if sampling_loc.dim() != 6 or sampling_loc.size(0) != n or sampling_loc.size(2) != m or sampling_loc.size(3) != l \
            or sampling_loc.size(5) != 2:
        raise RuntimeError(f"sampling_loc must be [N, Lq, M, L, P, 2] = [{n}, Lq, {m}, {l}, P, 2], got "
                           f"{tuple(sampling_loc.shape)}")
    if tuple(attn_weight.shape) != tuple(sampling_loc.shape[:5]):
        raise RuntimeError(f"attn_weight must be [N, Lq, M, L, P] = {tuple(sampling_loc.shape[:5])}, got "
                           f"{tuple(attn_weight.shape)}")
    if grad_output is not None and (grad_output.size(0) != n or grad_output.numel() != n * sampling_loc.size(1) * m * d):
        raise RuntimeError(f"grad_output must be [N, Lq, M*D] = [{n}, {sampling_loc.size(1)}, {m * d}], got "
                           f"{tuple(grad_output.shape)}")


def _level_tensor(t, name):
    if t.dtype != torch.int64:
        raise RuntimeError(f"{name} must be an int64 tensor")                      # cu:67-68 data<int64_t>()
    return t


def ms_deform_attn_forward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, im2col_step):
    """value [N,S,M,D] -> output [N,Lq,M*D]   (reference ms_deform_attn_cuda_forward, cu:20-80)."""
    _checks([("value", value), ("spatial_shapes", spatial_shapes), ("level_start_index", level_start_index),
             ("sampling_loc", sampling_loc), ("attn_weight", attn_weight)], value, im2col_step)
    _same_dtype(value, ("sampling_loc", sampling_loc), ("attn_weight", attn_weight))
    _level_tensor(spatial_shapes, "spatial_shapes"); _level_tensor(level_start_index, "level_start_index")
    _check_shapes(value, spatial_shapes, level_start_index, sampling_loc, attn_weight)
    n, s, m, d, l, lq, p = dims = _dims(value, spatial_shapes, sampling_loc)
    if min(dims) == 0:        # nothing to sample: the reference returns its at::zeros output (cu:54) after a failed empty launch
        return torch.zeros((n, lq, m * d), dtype=value.dtype, device=value.device)
    lib = _cabi.load()
    with torch.cuda.device(value.device):
        out = torch.empty((n, lq, m * d), dtype=value.dtype, device=value.device)
        stream = torch.cuda.current_stream().cuda_stream
        fn = getattr(lib, "msda_forward_" + _SUFFIX[value.dtype])
        code = fn(value.data_ptr(), spatial_shapes.data_ptr(), level_start_index.data_ptr(), sampling_loc.data_ptr(),
                  attn_weight.data_ptr(), *dims, out.data_ptr(), stream)
    _cabi.check(code, "ms_deform_attn_forward")
    return out


def ms_deform_attn_backward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, grad_output,
                            im2col_step, grad_value_dtype=None):
    """-> [grad_value, grad_sampling_loc, grad_attn_weight]   (reference ms_deform_attn_cuda_backward, cu:83-153).
    ``grad_value_dtype=torch.float32`` (bf16 ``value`` only, beyond the reference): hand back the fp32 accumulator
    itself instead of its bf16 rounding -- no conversion pass, no second buffer."""
    _checks([("value", value), ("spatial_shapes", spatial_shapes), ("level_start_index", level_start_index),
             ("sampling_loc", sampling_loc), ("attn_weight", attn_weight), ("grad_output", grad_output)],
            value, im2col_step)
    _same_dtype(value, ("sampling_loc", sampling_loc), ("attn_weight", attn_weight))
    if grad_output.dtype != value.dtype:
        raise RuntimeError(f"grad_output dtype {grad_output.dtype} != value dtype {value.dtype}")
    _level_tensor(spatial_shapes, "spatial_shapes"); _level_tensor(level_start_index, "level_start_index")
    _check_shapes(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, grad_output)
    dims = _dims(value, spatial_shapes, sampling_loc)
    if min(dims) == 0:        # empty problem: the reference's three zeros_like results (cu:121-123)
        gv_dtype = torch.float32 if (value.dtype == torch.bfloat16 and grad_value_dtype == torch.float32) else value.dtype
        return [torch.zeros(value.shape, dtype=gv_dtype, device=value.device), torch.zeros_like(sampling_loc),
                torch.zeros_like(attn_weight)]
    det = determinism.mode() != determinism.OFF
    if det and value.dtype == torch.float64:
        determinism.alert_not_deterministic("ms_deform_attn_backward with float64 value")
        det = False
    lib = _cabi.load()
    with torch.cuda.device(value.device):
        grad_loc = torch.empty_like(sampling_loc)
        grad_attn = torch.empty_like(attn_weight)
        stream = torch.cuda.current_stream().cuda_stream
        common = (grad_output.data_ptr(), value.data_ptr(), spatial_shapes.data_ptr(), level_start_index.data_ptr(),
                  sampling_loc.data_ptr(), attn_weight.data_ptr(), *dims)
        if det:            # bit-reproducible grad_value: 64-bit fixed-point sums in `acc` (zero-filled by the callee)
            acc = torch.empty(_cabi.DET_HEADER_WORDS + value.numel(), dtype=torch.int64, device=value.device)
            if value.dtype == torch.bfloat16:
                buf = torch.empty(value.shape, dtype=torch.float32, device=value.device)
                keep_f32 = grad_value_dtype == torch.float32
                grad_value = buf if keep_f32 else torch.empty_like(value)
                code = lib.msda_backward_det_bf16(*common, acc.data_ptr(), buf.data_ptr(),
                                                  None if keep_f32 else grad_value.data_ptr(), grad_loc.data_ptr(),
                                                  grad_attn.data_ptr(), stream)
            else:
                grad_value = torch.empty_like(value)
                code = lib.msda_backward_det_f32(*common, acc.data_ptr(), grad_value.data_ptr(), grad_loc.data_ptr(),
                                                 grad_attn.data_ptr(), stream)
        elif value.dtype == torch.bfloat16:
            acc = torch.empty(value.shape, dtype=torch.float32, device=value.device)
            keep_f32 = grad_value_dtype == torch.float32
            grad_value = acc if keep_f32 else torch.empty_like(value)
            code = lib.msda_backward_bf16(*common, acc.data_ptr(), None if keep_f32 else grad_value.data_ptr(),
                                          grad_loc.data_ptr(), grad_attn.data_ptr(), stream)
        else:
            grad_value = torch.empty_like(value)          # zero-filled by the callee (cudaMemsetAsync on `stream`)
            fn = getattr(lib, "msda_backward_" + _SUFFIX[value.dtype])
            code = fn(*common, grad_value.data_ptr(), grad_loc.data_ptr(), grad_attn.data_ptr(), stream)
    _cabi.check(code, "ms_deform_attn_backward")
    return [grad_value, grad_loc, grad_attn]
