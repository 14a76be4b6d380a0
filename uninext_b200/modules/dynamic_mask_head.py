"""CondInst dynamic mask head -- the mask branch UNINEXT's instance / video configs add to the deformable transformer
(uninext/models/ddetrs.py; SURVEY.md section 8 f-4, BASELINE.json configs[3] "300 queries + dynamic mask head"):

    controller MLP (ddetrs.py:72-77)        hidden state of every query -> 169 dynamic parameters
    dynamic_mask_with_coords (:508-598)     per selected instance: (rel. coordinates ++ 8 mask-feature channels) ->
                                            conv1x1(10->8) ReLU conv1x1(8->8) ReLU conv1x1(8->1), all weights dynamic
    aligned_bilinear (:921-942)             x (mask_feat_stride / mask_out_stride) up-sampling of the logits

The reference materialises a [1, I*10, H, W] input and runs three grouped convolutions (groups = #instances).  Here the
three layers are one hand-written kernel per direction (uninext_b200/csrc/msda_condinst.cuh) behind the C ABI; this file
is the autograd wrapper and the module with the reference's parameter names (``controller.layers.{0,1,2}``).
"""
from __future__ import annotations

import functools
import math
from typing import List, Sequence, Tuple

import torch
from torch import nn
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from uninext_b200 import _cabi, determinism

from .deformable_transformer import MLP

IN_CHANNELS, DYN_CHANNELS = 8, 8


def dynamic_param_counts(controller_layers: int = 3, rel_coord: bool = True, in_channels: int = IN_CHANNELS,
                         channels: int = DYN_CHANNELS):
    """(weight_nums, bias_nums) of the dynamic head (ddetrs.py:52-70)."""
    weight_nums, bias_nums = [], []
    for l in range(controller_layers):
        if l == 0:
            weight_nums.append((in_channels + (2 if rel_coord else 0)) * channels)
            bias_nums.append(channels)
        elif l == controller_layers - 1:
            weight_nums.append(channels)
            bias_nums.append(1)
        else:
            weight_nums.append(channels * channels)
            bias_nums.append(channels)
    return weight_nums, bias_nums


def _stream():
    return torch.cuda.current_stream().cuda_stream


class _AlignedBilinear(Function):
    @staticmethod
    def forward(ctx, x, factor):
        lib = _cabi.load()
        x = x.contiguous().float()
        *lead, h, w = x.shape
        planes = math.prod(lead) if lead else 1
        out = torch.empty((*lead, h * factor, w * factor), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            _cabi.check(lib.msda_aligned_bilinear_forward_f32(x.data_ptr(), planes, h, w, factor, out.data_ptr(), _stream()),
                        "msda_aligned_bilinear_forward_f32")
        ctx.dims = (planes, h, w, factor, x.shape)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        lib = _cabi.load()
        planes, h, w, factor, shape = ctx.dims
        g = g.contiguous().float()
        gin = torch.empty(shape, dtype=torch.float32, device=g.device)
        with torch.cuda.device(g.device):
            _cabi.check(lib.msda_aligned_bilinear_backward_f32(g.data_ptr(), planes, h, w, factor, gin.data_ptr(), _stream()),
                        "msda_aligned_bilinear_backward_f32")
        return gin, None


def aligned_bilinear(tensor: torch.Tensor, factor: int) -> torch.Tensor:
    """[..., h, w] -> [..., factor*h, factor*w] (ddetrs.py:921-942: replicate pad, align_corners bilinear, shift by factor/2)."""
    assert tensor.dim() >= 2 and factor >= 1 and int(factor) == factor
    if factor == 1:
        return tensor
    if not tensor.is_cuda:
        raise RuntimeError("aligned_bilinear: Not implemented on the CPU")
    return _AlignedBilinear.apply(tensor, int(factor))


class _DynamicMaskHead(Function):
    @staticmethod
    def forward(ctx, feats, params, refs, inst_start, max_inst, stride, rel_coord):
        lib = _cabi.load()
        feats, params, refs = feats.contiguous().float(), params.contiguous().float(), refs.contiguous().float()
        n, c, h, w = feats.shape
        i = params.shape[0]
        logits = torch.empty((i, h, w), dtype=torch.float32, device=feats.device)
        with torch.cuda.device(feats.device):
            _cabi.check(lib.msda_condinst_forward_f32(feats.data_ptr(), params.data_ptr(), refs.data_ptr(), inst_start.data_ptr(),
                                                      n, h, w, i, max_inst, stride, int(rel_coord), logits.data_ptr(),
                                                      _stream()), "msda_condinst_forward_f32")
        ctx.save_for_backward(feats, params, refs, inst_start)
        ctx.cfg = (stride, int(rel_coord), int(max_inst))
        return logits

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        lib = _cabi.load()
        feats, params, refs, inst_start = ctx.saved_tensors
        stride, rel, max_inst = ctx.cfg
        n, c, h, w = feats.shape
        i = params.shape[0]
        g = g.contiguous().float()
        gf, gp, gr = torch.empty_like(feats), torch.empty_like(params), torch.empty_like(refs)
        with torch.cuda.device(feats.device):
            if determinism.mode() != determinism.OFF:      # per-chunk / per-warp partials summed in a fixed order
                nbytes = _cabi.scratch_bytes(lib.msda_condinst_backward_det_scratch_bytes, n, h, w, i, max_inst)
                scratch = torch.empty(max(nbytes // 4, 1), dtype=torch.float32, device=feats.device)
                _cabi.check(lib.msda_condinst_backward_det_f32(g.data_ptr(), feats.data_ptr(), params.data_ptr(),
                                                               refs.data_ptr(), inst_start.data_ptr(), n, h, w, i, max_inst,
                                                               stride, rel, scratch.data_ptr(), gf.data_ptr(), gp.data_ptr(),
                                                               gr.data_ptr(), _stream()), "msda_condinst_backward_det_f32")
            else:
                _cabi.check(lib.msda_condinst_backward_f32(g.data_ptr(), feats.data_ptr(), params.data_ptr(), refs.data_ptr(),
                                                           inst_start.data_ptr(), n, h, w, i, max_inst, stride, rel,
                                                           gf.data_ptr(), gp.data_ptr(), gr.data_ptr(), _stream()),
                            "msda_condinst_backward_f32")
        return gf, gp, gr, None, None, None, None


@functools.lru_cache(maxsize=512)
def _inst_start(num_insts: Tuple[int, ...], device: torch.device) -> torch.Tensor:
    """[N + 1] int32 prefix sums on the device; cached because inference repeats the same counts (one tiny H2D copy per
    distinct tuple instead of per call, and none inside a CUDA-graph capture after the first call)."""
    starts = [0]
    for k in num_insts:
        starts.append(starts[-1] + k)
    return torch.tensor(starts, dtype=torch.int32, device=device)


def dynamic_mask_with_coords(mask_feats: torch.Tensor, reference_points: torch.Tensor, mask_head_params: torch.Tensor,
                             num_insts: Sequence[int], mask_feat_stride: int, rel_coord: bool = True,
                             mask_out_stride: int = 4) -> torch.Tensor:
    """Same contract as the reference method (ddetrs.py:508-598, ``use_raft=False``):
        mask_feats [N, 8, H, W]; reference_points [1, sum(num_insts), 2] in input-image pixels; mask_head_params
        [1, sum(num_insts), 169]; num_insts = instances per image (host ints)  ->  mask logits
        [1, sum(num_insts), H * s, W * s] with s = mask_feat_stride / mask_out_stride."""
    if not mask_feats.is_cuda:
        raise RuntimeError("dynamic_mask_with_coords: Not implemented on the CPU")
    n, c, h, w = mask_feats.shape
    total = int(sum(num_insts))
    w_nums, b_nums = dynamic_param_counts(3, rel_coord)
    if c != IN_CHANNELS or mask_head_params.shape[-1] != sum(w_nums) + sum(b_nums):
        raise RuntimeError(f"dynamic mask head kernels cover {IN_CHANNELS} feature channels and {DYN_CHANNELS} dynamic "
                           f"channels in 3 layers (UNINEXT's configuration); got C={c}, "
                           f"{mask_head_params.shape[-1]} parameters")
    assert mask_feat_stride >= mask_out_stride and mask_feat_stride % mask_out_stride == 0           # ddetrs.py:579-580
    assert len(num_insts) == n and reference_points.shape[1] == total == mask_head_params.shape[1]
    if total == 0:                                                       # ddetrs.py:572-574 keeps the graph connected
        return mask_feats.new_zeros((1, 0, h * (mask_feat_stride // mask_out_stride), w * (mask_feat_stride // mask_out_stride))) \
            + mask_head_params.sum() * 0.0
    params = mask_head_params.reshape(total, -1)
    if not rel_coord:       # 8-channel first layer: embed into the 10-channel kernel layout with zero coordinate weights
        w1 = params[:, :64].reshape(total, 8, 8)
        params = torch.cat((torch.cat((w1.new_zeros(total, 8, 2), w1), -1).reshape(total, 80), params[:, 64:]), -1)
    inst_start = _inst_start(tuple(int(k) for k in num_insts), mask_feats.device)
    logits = _DynamicMaskHead.apply(mask_feats, params, reference_points.reshape(total, 2), inst_start,
                                    int(max(num_insts)), int(mask_feat_stride), bool(rel_coord))
    logits = aligned_bilinear(logits, mask_feat_stride // mask_out_stride)
    return logits.unsqueeze(0)


class CondInstMaskHead(nn.Module):
    """Controller + dynamic mask head.  ``controller`` carries the reference's parameter names
    (``controller.layers.{0,1,2}``, ddetrs.py:72), so the mask-branch weights of a UNINEXT checkpoint load unchanged."""

    def __init__(self, hidden_dim: int = 256, controller_layers: int = 3, rel_coord: bool = True, mask_out_stride: int = 4,
                 mask_feat_stride: int = 8):
        super().__init__()
        if hidden_dim // 32 != IN_CHANNELS or controller_layers != 3:
            raise ValueError("CondInstMaskHead: kernels are built for hidden_dim 256 (8 mask-feature channels) and 3 layers")
        self.rel_coord, self.mask_out_stride, self.mask_feat_stride = rel_coord, mask_out_stride, mask_feat_stride
        self.in_channels, self.dynamic_mask_channels = hidden_dim // 32, DYN_CHANNELS
        self.weight_nums, self.bias_nums = dynamic_param_counts(controller_layers, rel_coord)
        self.num_gen_params = sum(self.weight_nums) + sum(self.bias_nums)
        self.controller = MLP(hidden_dim, hidden_dim, self.num_gen_params, 3)
        for layer in self.controller.layers:                                  # ddetrs.py:74-76
            nn.init.xavier_uniform_(layer.weight)
            nn.init.zeros_(layer.bias)

    def forward(self, hs: torch.Tensor, mask_feats: torch.Tensor, reference_points_px: torch.Tensor,
                selected: List[torch.Tensor]):
        """hs [N, Q, C] decoder states; mask_feats [N, 8, H, W]; reference_points_px [N, Q, 2] (pixels);
        selected[b] = indices of the queries of image b that get a mask (matched / kept instances, ddetrs.py:186-210).
        -> logits [1, sum(len(selected[b])), H * s, W * s]."""
        params = self.controller(hs)
        num_insts = [int(s.numel()) for s in selected]
        p = torch.cat([params[b, s] for b, s in enumerate(selected)], 0).unsqueeze(0)
        r = torch.cat([reference_points_px[b, s] for b, s in enumerate(selected)], 0).unsqueeze(0)
        return dynamic_mask_with_coords(mask_feats, r, p, num_insts, self.mask_feat_stride, self.rel_coord,
                                        self.mask_out_stride)
