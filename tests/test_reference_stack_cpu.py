"""CPU test of bench.py's `frames.reference_stack` wiring (no GPU): the reference's own layer classes (files staged in
oracle/_ref/py by build() from a reference checkout; skipped without one) dropped into run_frames' stack run forward +
backward when ``ms_deform_attn_func.MSDA`` is rebound to a kernels module -- here one built on the reference's CPU function instead of oracle/_ref's CUDA kernels."""
import os
import sys
import warnings

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import refstage  # noqa: E402

pytestmark = pytest.mark.skipif(not refstage.staged(), reason="oracle/_ref/py not staged (no reference checkout at build time)")


class _CpuKernels:
    """ms_deform_attn_forward / _backward of the reference's pybind module, computed with its own CPU function."""
    core = None

    @classmethod
    def ms_deform_attn_forward(cls, value, shapes, lsi, loc, attn, im2col_step):
        with torch.no_grad():
            return cls.core(value, shapes, loc, attn)

    @classmethod
    def ms_deform_attn_backward(cls, value, shapes, lsi, loc, attn, grad_output, im2col_step):
        with torch.enable_grad():
            v, lo, at = (t.detach().clone().requires_grad_(True) for t in (value, loc, attn))
            out = cls.core(v, shapes, lo, at)
            return list(torch.autograd.grad(out, (v, lo, at), grad_output))


def test_reference_layers_run_inside_the_bench_stack():
    import bench
    from uninext_b200.workloads import OpConfig, level_tensors
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        func_mod, _attn, tr_mod, _dino = refstage.import_reference()
    cfg = OpConfig("tiny", 64, 64, 2, 10)
    shapes = cfg.shapes
    model = bench.build_reference_stack(cfg, tr_mod, num_layers=2, d_ffn=64)
    assert type(model.encoder[0]).__module__.startswith("uninext_ref.")          # the reference's classes, not ours
    assert type(model.decoder[0].cross_attn).__module__.startswith("uninext_ref.")
    ss, lsi = level_tensors(shapes, "cpu")
    g = torch.Generator().manual_seed(3)
    src, pos = torch.randn(cfg.batch, cfg.S, 256, generator=g), torch.randn(cfg.batch, cfg.S, 256, generator=g)
    pad = torch.zeros(cfg.batch, cfg.S, dtype=torch.bool)
    _CpuKernels.core = staticmethod(func_mod.ms_deform_attn_core_pytorch)
    was, func_mod.MSDA = func_mod.MSDA, _CpuKernels
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            out = model(src, pos, shapes, ss, lsi, pad)
            out.float().square().mean().backward()
    finally:
        func_mod.MSDA = was
    assert out.shape == (cfg.batch, cfg.dec_queries, 256) and torch.isfinite(out).all()
    missing = [k for k, p in model.named_parameters() if p.grad is None and not k.startswith("level_embed")]
    assert not missing, missing
    # the kernels module bench.py builds has the two entry points the reference file calls (func.py:26,36)
    km = bench.reference_kernels_module(object())
    assert callable(km.ms_deform_attn_forward) and callable(km.ms_deform_attn_backward)
