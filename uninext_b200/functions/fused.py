"""Autograd wrappers of the one-pass kernels around the op (include/msda_b200.h, "callers of the op").

They keep the reference modules' parameters (same tensors, same state_dict) and only change how the arithmetic is
scheduled: the GEMMs stay cuBLAS (torch.addmm / torch.mm), the elementwise / reduction passes around them run as
single hand-written kernels.

* ``sampling_prologue``   -- ms_deform_attn.py:99-112 (two Linears + softmax + location arithmetic) as one GEMM over the
                            concatenated weights + one kernel writing loc/attn in the op's layouts.
* ``linear_colsum``       -- nn.Linear whose bias gradient is one column-sum kernel instead of a generic reduce.
* ``add_layer_norm``      -- ``LayerNorm(a + b)`` (deformable_transformer.py:354-356,359) forward and backward.

These wrappers are conveniences for the callers of the op: when their preconditions do not hold (non-fp32, CPU tensors,
unsupported widths) they hand the same maths to the stock torch ops.  The op itself (MSDeformAttnFunction) has no such
path: it raises without the CUDA library.
"""
from __future__ import annotations

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from uninext_b200 import _cabi, determinism


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _f32c(t):
    return t.contiguous() if t.dtype == torch.float32 else t.float().contiguous()


def _det_scratch(nbytes, device):
    return torch.empty(nbytes // 4, dtype=torch.float32, device=device)


def colsum(x2d: torch.Tensor) -> torch.Tensor:
    """sum over rows of a contiguous fp32 [rows, cols] CUDA tensor (cols % 4 == 0)."""
    rows, cols = x2d.shape
    if cols % 4 or x2d.data_ptr() % 16:
        return x2d.sum(0)
    out = torch.empty(cols, dtype=torch.float32, device=x2d.device)
    lib = _cabi.load()
    with torch.cuda.device(x2d.device):
        if determinism.mode() != determinism.OFF:          # fixed-order sum of per-CTA partial rows
            scratch = _det_scratch(_cabi.scratch_bytes(lib.msda_colsum_det_scratch_bytes, rows, cols), x2d.device)
            _cabi.check(lib.msda_colsum_det_f32(x2d.data_ptr(), rows, cols, scratch.data_ptr(), out.data_ptr(), _stream()),
                        "msda_colsum_det_f32")
        else:
            _cabi.check(lib.msda_colsum_f32(x2d.data_ptr(), rows, cols, out.data_ptr(), _stream()), "msda_colsum_f32")
    return out


def weight_grad(g2: torch.Tensor, x2: torch.Tensor, splits: int = 16) -> torch.Tensor:
    """g2^T @ x2 for a tall-skinny problem ([rows, n]^T @ [rows, c], rows >> n, c).  cuBLAS picks a 16-CTA kernel for the
    un-split product when n*c is small; splitting the reduction into a strided-batched GEMM + a tiny sum fills the GPU."""
    rows, n = g2.shape
    c = x2.shape[1]
    if rows < 8192 or n * c > 256 * 512:
        return torch.mm(g2.t(), x2)
    ch = rows // splits
    kp = ch * splits
    gw = torch.bmm(g2[:kp].view(splits, ch, n).transpose(1, 2), x2[:kp].view(splits, ch, c)).sum(0)
    if kp < rows:
        gw = gw.addmm_(g2[kp:].t(), x2[kp:])
    return gw


def tcgen05_linear_ok(x2: torch.Tensor, weight: torch.Tensor) -> bool:
    """msda_linear_tf32 constraints (include/msda_b200.h): fp32, K % 32 == 0, N % 32 == 0 (N % 64 == 0 above 256), N <= 512."""
    n, k = weight.shape
    return (x2.is_cuda and x2.dtype == torch.float32 and weight.dtype == torch.float32 and k % 32 == 0 and n % 32 == 0
            and n <= 512 and (n <= 256 or n % 64 == 0) and x2.data_ptr() % 16 == 0 and weight.data_ptr() % 16 == 0)


def tcgen05_linear(x2: torch.Tensor, weight: torch.Tensor, bias) -> torch.Tensor:
    """x2 @ weight.T + bias on the hand-written tcgen05 kernel (TF32 MMA, fp32 accumulate in tensor memory)."""
    x2, weight = x2.contiguous(), weight.contiguous()
    m, k = x2.shape
    n = weight.shape[0]
    out = torch.empty((m, n), dtype=torch.float32, device=x2.device)
    with torch.cuda.device(x2.device):
        _cabi.check(_cabi.load().msda_linear_tf32(x2.data_ptr(), weight.data_ptr(),
                                                  bias.data_ptr() if bias is not None else None, m, n, k, out.data_ptr(),
                                                  _stream()), "msda_linear_tf32")
    return out


# "auto" picks the hand-written kernels only where they are the faster choice.  Measured on B200 (profiles/r02*_gemm*.txt):
# cuBLAS TF32 is still ahead on these shapes, so auto resolves to cuBLAS unless MSDA_GEMM_AUTO=tcgen05 is set.
import os as _os
_AUTO_TCGEN05 = _os.environ.get("MSDA_GEMM_AUTO", "cublas") == "tcgen05"
_AUTO_MASKED_TCGEN05 = _os.environ.get("MSDA_GEMM_AUTO_MASKED", "tcgen05") == "tcgen05"     # value_proj + padding mask


def resolve_gemm(gemm: str) -> str:
    """"auto": the hand-written tcgen05 TF32 kernels when the caller has allowed TF32 products
    (``torch.backends.cuda.matmul.allow_tf32`` -- the default of the PyTorch 1.10 stack the reference was trained with), cuBLAS
    fp32 otherwise, so that strict-fp32 runs keep their 1e-4 parity with the reference."""
    if gemm == "auto":
        return "tcgen05" if (torch.backends.cuda.matmul.allow_tf32 and _AUTO_TCGEN05) else "cublas"
    return gemm


def tcgen05_ws_ok(x2: torch.Tensor, weight: torch.Tensor) -> bool:
    """W-stationary kernel with the fused tail (msda_linear_tf32_ex): K <= 256, N <= 256, N % 64 == 0."""
    n, k = weight.shape
    return tcgen05_linear_ok(x2, weight) and bool(_cabi.load().msda_linear_tf32_ws_ok(n, k))


def tcgen05_linear_ex(x2, weight, bias, row_mask=None, relu=False):
    """x2 @ weight.T + bias, rows with ``row_mask`` set written as zeros, optional ReLU -- one kernel (msda_linear_tf32_ex)."""
    x2, weight = x2.contiguous(), weight.contiguous()
    m, k = x2.shape
    n = weight.shape[0]
    out = torch.empty((m, n), dtype=torch.float32, device=x2.device)
    mask8 = None
    if row_mask is not None:
        mask8 = row_mask.reshape(-1).contiguous()
        mask8 = mask8.view(torch.uint8) if mask8.dtype == torch.bool else mask8.to(torch.uint8)       # bool is one byte: no copy
    with torch.cuda.device(x2.device):
        _cabi.check(_cabi.load().msda_linear_tf32_ex(x2.data_ptr(), weight.data_ptr(), bias.data_ptr() if bias is not None else None,
                                                     mask8.data_ptr() if mask8 is not None else None, m, n, k, int(relu),
                                                     out.data_ptr(), _stream()), "msda_linear_tf32_ex")
    return out


def _gemm_bias(x2, weight, bias, gemm):
    if resolve_gemm(gemm) == "tcgen05" and tcgen05_linear_ok(x2, weight):
        return tcgen05_linear(x2, weight, bias)
    return torch.addmm(bias, x2, weight.t())


class _LinearColsum(Function):
    @staticmethod
    def forward(ctx, x, weight, bias, relu, gemm, row_mask):
        x2 = x.reshape(-1, x.shape[-1])
        mask = row_mask.reshape(-1) if row_mask is not None else None
        # "auto" with a row mask: the fused kernel replaces GEMM + masked_fill (21.7 us against 19.2 + 14 us at 44 646 x 256 x 256,
        # profiles/r02ah_gemm_ws2.txt), so it is taken whenever TF32 products are allowed; without a mask cuBLAS stays ahead.
        fused_mask = gemm == "auto" and mask is not None and torch.backends.cuda.matmul.allow_tf32 and _AUTO_MASKED_TCGEN05
        if (resolve_gemm(gemm) == "tcgen05" or fused_mask) and tcgen05_ws_ok(x2, weight):
            y = tcgen05_linear_ex(x2, weight, bias, mask, relu)          # bias, padding-mask zeroing and ReLU in the epilogue
        elif relu:                                           # bias + ReLU in the cuBLASLt epilogue
            y = torch._addmm_activation(bias, x2, weight.t(), use_gelu=False)
            if mask is not None:
                y = y.masked_fill(mask[:, None], 0.0)
        else:
            y = _gemm_bias(x2, weight, bias, gemm)
            if mask is not None:
                y = y.masked_fill(mask[:, None], 0.0)
        ctx.save_for_backward(x2, weight, y if relu else None, mask)
        ctx.xshape, ctx.relu = x.shape, relu
        return y.view(*x.shape[:-1], weight.shape[0])

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        x2, weight, y, mask = ctx.saved_tensors
        g2 = g.reshape(-1, g.shape[-1])
        gb = None
        if ctx.relu and g2.is_cuda and g2.dtype == torch.float32 and g2.shape[1] % 4 == 0 and ctx.needs_input_grad[2]:
            # ReLU backward and the bias gradient in ONE pass over (g, y)  (masked rows have y == 0: zeroed by the same test)
            g2 = g2.contiguous()
            out = torch.empty_like(g2)
            gb = torch.empty(g2.shape[1], dtype=torch.float32, device=g2.device)
            lib = _cabi.load()
            with torch.cuda.device(g2.device):
                if determinism.mode() != determinism.OFF:
                    scratch = _det_scratch(_cabi.scratch_bytes(lib.msda_colsum_det_scratch_bytes, g2.shape[0], g2.shape[1]),
                                           g2.device)
                    _cabi.check(lib.msda_relu_backward_colsum_det_f32(g2.data_ptr(), y.data_ptr(), g2.shape[0], g2.shape[1],
                                                                      out.data_ptr(), scratch.data_ptr(), gb.data_ptr(),
                                                                      _stream()), "msda_relu_backward_colsum_det_f32")
                else:
                    _cabi.check(lib.msda_relu_backward_colsum_f32(g2.data_ptr(), y.data_ptr(), g2.shape[0], g2.shape[1],
                                                                  out.data_ptr(), gb.data_ptr(), _stream()),
                                "msda_relu_backward_colsum_f32")
            g2 = out
        elif ctx.relu:
            g2 = torch.ops.aten.threshold_backward(g2, y, 0.0)          # masked rows have y == 0: already zeroed
        elif mask is not None:
            g2 = g2.masked_fill(mask[:, None], 0.0)
        else:
            g2 = g2.contiguous()
        gx = torch.mm(g2, weight).view(ctx.xshape) if ctx.needs_input_grad[0] else None
        gw = weight_grad(g2, x2) if ctx.needs_input_grad[1] else None
        if gb is None and ctx.needs_input_grad[2]:
            gb = colsum(g2)
        return gx, gw, gb, None, None, None


def linear_colsum(x, linear: torch.nn.Linear, relu: bool = False, gemm: str = "cublas", row_mask=None):
    """``linear(x)`` (optionally followed by ReLU, optionally with the rows of ``row_mask`` zeroed -- the
    ``masked_fill(input_padding_mask)`` after value_proj) with the bias gradient computed by msda_colsum_f32 and the
    weight gradient as a split-K batched GEMM.  ``gemm="tcgen05"`` / ``"auto"`` (under allow_tf32) runs the forward product
    on the hand-written tensor-core kernels, with bias / mask / ReLU fused into their epilogue for K, N <= 256."""
    if (not x.is_cuda) or x.dtype != torch.float32 or linear.bias is None or linear.out_features % 4 or \
            torch.is_autocast_enabled():
        y = linear(x)
        if relu:
            y = torch.relu(y)
        return y if row_mask is None else y.masked_fill(row_mask[..., None], 0.0)
    return _LinearColsum.apply(x, linear.weight, linear.bias, relu, gemm, row_mask)


class _BatchedLinear(Function):
    """y[l] = x2 @ w[l].T + b[l] for l = 0..L-1 as one strided-batched GEMM over a shared A operand."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, x2, w, b):
        L, n, k = w.shape
        y = torch.baddbmm(b[:, None, :], x2.unsqueeze(0).expand(L, -1, -1), w.transpose(1, 2))        # [L, R, n]
        ctx.save_for_backward(x2, w)
        return y

    @staticmethod
    @once_differentiable
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, g):
        x2, w = ctx.saved_tensors
        L = w.shape[0]
        g = g.contiguous()
        gx = None
        if ctx.needs_input_grad[0]:
            gx = torch.mm(g[0], w[0])
            for i in range(1, L):
                gx.addmm_(g[i], w[i])                          # accumulate in place: no [L, R, K] temporary
        gw = torch.stack([weight_grad(g[i], x2) for i in range(L)]) if ctx.needs_input_grad[1] else None
        gb = None
        if ctx.needs_input_grad[2]:
            gb = torch.stack([colsum(g[i]) for i in range(L)]) if g.is_cuda and g.dtype == torch.float32 else g.sum(1)
        return gx, gw, gb


def batched_linear(x2, w, b):
    """x2 [R, K], w [L, N, K], b [L, N] -> [L, R, N]."""
    return _BatchedLinear.apply(x2, w, b)


class _SamplingPrologue(Function):
    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)      # like the reference module (ms_deform_attn.py:78)
    def forward(ctx, query, w_off, b_off, w_attn, b_attn, ref, shapes, n_heads, n_levels, n_points, gemm):
        lib = _cabi.load()
        q2 = query.reshape(-1, query.shape[-1])
        rows = q2.shape[0]
        weight = torch.cat((w_off, w_attn), 0)                    # [M*LP*3, C]: offsets first, logits last
        bias = torch.cat((b_off, b_attn), 0)
        proj = _gemm_bias(q2, weight, bias, gemm)                  # one GEMM instead of two (ms_deform_attn.py:99-100)
        ref_c = _f32c(ref).reshape(rows, n_levels, ref.shape[-1])
        loc = torch.empty((rows, n_heads, n_levels, n_points, 2), dtype=torch.float32, device=query.device)
        attn = torch.empty((rows, n_heads, n_levels, n_points), dtype=torch.float32, device=query.device)
        with torch.cuda.device(query.device):
            _cabi.check(lib.msda_prologue_forward_f32(proj.data_ptr(), ref_c.data_ptr(), shapes.data_ptr(), rows, n_heads,
                                                      n_levels, n_points, ref.shape[-1], loc.data_ptr(), attn.data_ptr(),
                                                      _stream()), "msda_prologue_forward_f32")
        ctx.save_for_backward(q2, weight, attn, ref_c, shapes)
        ctx.dims = (n_heads, n_levels, n_points, ref.shape[-1], w_off.shape[0], query.shape)
        lead = query.shape[:-1]
        return loc.view(*lead, n_heads, n_levels, n_points, 2), attn.view(*lead, n_heads, n_levels, n_points)

    @staticmethod
    @once_differentiable
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, g_loc, g_attn):
        lib = _cabi.load()
        q2, weight, attn, ref_c, shapes = ctx.saved_tensors
        m, l, p, rd, n_off, qshape = ctx.dims
        rows = q2.shape[0]
        g_proj = torch.empty((rows, weight.shape[0]), dtype=torch.float32, device=q2.device)
        g_loc, g_attn = _f32c(g_loc), _f32c(g_attn)
        with torch.cuda.device(q2.device):
            _cabi.check(lib.msda_prologue_backward_f32(g_loc.data_ptr(), g_attn.data_ptr(), attn.data_ptr(), ref_c.data_ptr(),
                                                       shapes.data_ptr(), rows, m, l, p, rd, g_proj.data_ptr(), _stream()),
                        "msda_prologue_backward_f32")
        gq = torch.mm(g_proj, weight).view(qshape) if ctx.needs_input_grad[0] else None
        gw = weight_grad(g_proj, q2)
        gb = colsum(g_proj)
        return gq, gw[:n_off], gb[:n_off], gw[n_off:], gb[n_off:], None, None, None, None, None, None


def sampling_prologue(query, sampling_offsets: torch.nn.Linear, attention_weights: torch.nn.Linear, reference_points,
                      spatial_shapes, n_heads, n_levels, n_points, gemm: str = "cublas"):
    """-> (sampling_locations [.., M, L, P, 2], attention_weights [.., M, L, P]); reference points are constants."""
    return _SamplingPrologue.apply(query, sampling_offsets.weight, sampling_offsets.bias, attention_weights.weight,
                                   attention_weights.bias, reference_points, spatial_shapes, n_heads, n_levels, n_points,
                                   gemm)


class _AddLayerNorm(Function):
    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)      # autocast runs layer_norm in fp32 too
    def forward(ctx, a, b, gamma, beta, eps):
        lib = _cabi.load()
        cols = a.shape[-1]
        a2 = a.reshape(-1, cols).contiguous()
        b2 = b.reshape(-1, cols).contiguous() if b is not None else None
        rows = a2.shape[0]
        y = torch.empty_like(a2)
        z = torch.empty_like(a2) if b2 is not None else a2
        mean = torch.empty(rows, dtype=torch.float32, device=a.device)
        rstd = torch.empty(rows, dtype=torch.float32, device=a.device)
        with torch.cuda.device(a.device):
            _cabi.check(lib.msda_add_layernorm_forward_f32(a2.data_ptr(), b2.data_ptr() if b2 is not None else None,
                                                           gamma.data_ptr(), beta.data_ptr(), rows, cols, float(eps),
                                                           z.data_ptr() if b2 is not None else None, y.data_ptr(),
                                                           mean.data_ptr(), rstd.data_ptr(), _stream()),
                        "msda_add_layernorm_forward_f32")
        ctx.save_for_backward(z, gamma, mean, rstd)
        ctx.has_b = b is not None
        ctx.a_dtype, ctx.b_dtype = a.dtype, (b.dtype if b is not None else None)
        return y.view(a.shape)

    @staticmethod
    @once_differentiable
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, gy):
        lib = _cabi.load()
        z, gamma, mean, rstd = ctx.saved_tensors
        rows, cols = z.shape
        gy2 = _f32c(gy.reshape(rows, cols))
        dz = torch.empty_like(z)
        dgamma = torch.empty_like(gamma)
        dbeta = torch.empty_like(gamma)
        with torch.cuda.device(z.device):
            if determinism.mode() != determinism.OFF:
                scratch = _det_scratch(_cabi.scratch_bytes(lib.msda_layernorm_backward_det_scratch_bytes, rows, cols), z.device)
                _cabi.check(lib.msda_layernorm_backward_det_f32(gy2.data_ptr(), z.data_ptr(), gamma.data_ptr(), mean.data_ptr(),
                                                                rstd.data_ptr(), rows, cols, dz.data_ptr(), scratch.data_ptr(),
                                                                dgamma.data_ptr(), dbeta.data_ptr(), _stream()),
                            "msda_layernorm_backward_det_f32")
            else:
                _cabi.check(lib.msda_layernorm_backward_f32(gy2.data_ptr(), z.data_ptr(), gamma.data_ptr(), mean.data_ptr(),
                                                            rstd.data_ptr(), rows, cols, dz.data_ptr(), dgamma.data_ptr(),
                                                            dbeta.data_ptr(), _stream()), "msda_layernorm_backward_f32")
        dz = dz.view(gy.shape)
        da = dz.to(ctx.a_dtype) if ctx.a_dtype != dz.dtype else dz
        db = (dz.to(ctx.b_dtype) if ctx.b_dtype != dz.dtype else dz) if ctx.has_b else None
        return da, db, dgamma, dbeta, None


def add_layer_norm(a, b, norm: torch.nn.LayerNorm):
    """``norm(a + b)`` (b may be None) as one forward and one backward kernel."""
    cols = a.shape[-1]
    auto = torch.is_autocast_enabled()               # under autocast the inputs are cast to fp32 by custom_fwd
    ok = a.is_cuda and (a.dtype == torch.float32 or auto) and cols in (128, 256, 384, 512) and norm.elementwise_affine \
        and norm.bias is not None and (b is None or b.dtype == torch.float32 or auto) \
        and all(t is None or t.data_ptr() % 16 == 0 for t in (a, b, norm.weight, norm.bias))      # float4 loads in the kernels
    if not ok:
        return norm(a if b is None else a + b)
    return _AddLayerNorm.apply(a, b, norm.weight, norm.bias, norm.eps)
