"""GPU tests (-m gpu): this repo's layers on the sm_100a kernels against what the REFERENCE's own Python classes compute,
and the drop-in module (``import MultiScaleDeformableAttention`` -> uninext_b200/dropin) against the CPU oracle:

  * the drop-in called exactly as the reference's ``MSDeformAttnFunction`` calls its extension (the boundary claim,
    SURVEY.md 8b), checked against the CPU oracle, and
  * this repo's mirrors (``MSDeformAttn``, encoder / decoder layers of both transformer files, the DINO decoder layer with
    its ``attn_masks``, ``DeformableReidHead``, the DINO decoder loop): forward + input gradients + every parameter
    gradient, 2e-4 of scale (fp32), against the reference classes' results on the same weights and inputs
    (tests/reference_cases.py; stored by tests/golden/make_reference_golden.py).
"""
import warnings

import numpy as np
import pytest
import torch

from oracle import msda_oracle
from tests import reference_cases as rc

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from uninext_b200 import _cabi
    from uninext_b200.dropin import MultiScaleDeformableAttention as MSDA
    from uninext_b200.modules import MSDeformAttn
    from uninext_b200.modules.deformable_layers import DeformableTransformerEncoderLayer
    from uninext_b200.modules.deformable_transformer import get_reference_points, valid_ratios_from_masks
    from uninext_b200.workloads import CONFIGS, make_inputs

DEV = "cuda"
TOL = 2e-4
SHAPES = rc.SHAPES


def _rel(got, want):
    return ((got.detach().double() - want.detach().double()).abs().max() /
            want.detach().double().abs().max().clamp_min(1e-30)).item()


def _compare(name, tol=TOL):
    """Runs case `name` of tests/reference_cases.py with this repo's module on the GPU and compares out, input grads and
    every parameter grad with the reference classes' stored results."""
    ours, _, run, inputs = rc.dropin_case(name, DEV)
    want = rc.load("dropin_" + name)
    lib = _cabi.load()
    before = lib.msda_launch_count()
    out, gin, gpar = rc.run_case(ours, run, inputs)
    assert lib.msda_launch_count() > before, "no kernel of libmsda_b200.so ran"
    assert rc.rel_err(out, want, "out") < tol
    for i, g in enumerate(gin):
        assert rc.rel_err(g, want, f"grad_in.{i}") < 5 * tol
    assert set(gpar) == set(want["param_names"].tolist())
    for k, g in gpar.items():
        assert g is not None, k
        assert rc.rel_err(g, want, "grad." + k) < 5 * tol, k


def test_reference_function_on_dropin_matches_oracle():
    """The two extension calls of the reference's MSDeformAttnFunction (func.py:26-37): forward with im2col_step, then
    backward with the saved tensors and grad_output, returning the three input gradients."""
    inp = make_inputs(CONFIGS["cfg1"], "enc", DEV, seed=31, wild_fraction=0.1)
    f64 = lambda t: t.detach().double().cpu().numpy()
    args = (f64(inp["value"]), inp["spatial_shapes"].cpu().numpy(), inp["level_start_index"].cpu().numpy(),
            f64(inp["sampling_locations"]), f64(inp["attention_weights"]))
    out_t = msda_oracle.forward(*args)
    gv_t, gl_t, ga_t = msda_oracle.backward(f64(inp["grad_output"]), *args)
    a = (inp["value"], inp["spatial_shapes"], inp["level_start_index"], inp["sampling_locations"],
         inp["attention_weights"])
    lib = _cabi.load()
    before = lib.msda_launch_count()
    out = MSDA.ms_deform_attn_forward(*a, 64)
    gv, gl, ga = MSDA.ms_deform_attn_backward(*a, inp["grad_output"], 64)
    assert lib.msda_launch_count() - before == 2
    err = lambda g, w: float(np.abs(g.detach().cpu().numpy() - w).max() / max(np.abs(w).max(), 1e-30))
    assert err(out, out_t) < 1e-4 and err(gv, gv_t) < 1e-4 and err(ga, ga_t) < 1e-4
    bad = (np.abs(gl.cpu().numpy() - gl_t) / np.abs(gl_t).max() > 2e-4).sum()
    assert bad <= max(2, 1e-4 * gl_t.size)


def _pyramid_inputs(n, gen, c=256, masked=True):
    return rc.pyramid_inputs(n, gen, DEV, c, masked)


@pytest.mark.parametrize("which", [0, 1])          # 0: deformable_transformer.py, 1: deformable_transformer_dino.py
def test_reference_module_and_encoder_layer_on_dropin(which):
    _compare(f"module_{which}")                    # (a9) the module
    _compare(f"encoder_{which}")                   # (a10) the encoder layer


@pytest.mark.parametrize("which", [0, 1])
def test_reference_decoder_layer_on_dropin(which):
    _compare(f"decoder_{which}")


def test_reference_reid_head_on_dropin():
    _compare("reid")


@pytest.mark.parametrize("batched", [False, True])
@pytest.mark.parametrize("refine", [True, False])
def test_reference_decoder_loop_on_dropin(refine, batched):
    """The whole DINO decoder loop (sine embedding -> ref_point_head -> layer -> box refinement, look_forward_twice),
    reference class against this repo's decoder, which projects the memory for all layers in ONE batched GEMM
    (SURVEY.md section 8 f-2)."""
    from uninext_b200.modules.ms_deform_attn import use_batched_value_proj
    was = use_batched_value_proj()
    use_batched_value_proj(batched)
    try:
        _compare("decoder_loop_refine" if refine else "decoder_loop_plain")
    finally:
        use_batched_value_proj(was)


def test_batched_value_proj_equals_per_layer_projection():
    from uninext_b200.modules.ms_deform_attn import batched_value_proj
    g = torch.Generator().manual_seed(81)
    ss, lsi, masks, flat, src, _ = _pyramid_inputs(2, g)
    torch.manual_seed(7)
    mods = [MSDeformAttn(256, 4, 8, 4).to(DEV) for _ in range(3)]
    x = src.clone().requires_grad_(True)
    vals = batched_value_proj(mods, x, flat)
    want = [m.value_proj(src).masked_fill(flat[..., None], 0.0) for m in mods]
    for a, b in zip(vals, want):
        assert _rel(a, b) < 1e-5
    sum((v * (i + 1)).sum() for i, v in enumerate(vals)).backward()
    gw = [m.value_proj.weight.grad.clone() for m in mods]
    gx = x.grad.clone()
    for m in mods:
        m.zero_grad()
    x2 = src.clone().requires_grad_(True)
    sum((m.value_proj(x2).masked_fill(flat[..., None], 0.0) * (i + 1)).sum() for i, m in enumerate(mods)).backward()
    assert _rel(gx, x2.grad) < 1e-4
    for a, m in zip(gw, mods):
        assert _rel(a, m.value_proj.weight.grad) < 1e-4


def test_layers_run_fp32_under_autocast_like_reference():
    """custom_fwd(cast_inputs=float32) on the reference layers (deformable_transformer.py:351,398): under autocast the
    whole layer, FFN included, computes in fp32 -- ours must give the fp32 result too."""
    g = torch.Generator().manual_seed(70)
    ss, lsi, masks, flat, src, pos = _pyramid_inputs(1, g, masked=False)
    refpts = get_reference_points(SHAPES, valid_ratios_from_masks(masks))
    torch.manual_seed(5)
    layer = DeformableTransformerEncoderLayer(256, 512, 0.0, "relu", 4, 8, 4).to(DEV)
    want = layer(src, pos, refpts, ss, lsi, None)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        got = layer(src.bfloat16(), pos, refpts, ss, lsi, None)
    assert got.dtype == torch.float32
    assert _rel(got, layer(src.bfloat16().float(), pos, refpts, ss, lsi, None)) < 1e-5
    assert _rel(got, want) < 2e-2            # only the bf16 rounding of the input separates them


def test_geometry_kernels_match_reference_functions():
    """f-3 on the GPU: reference points, two-stage proposals and the sine position embedding as single kernels against the
    reference's own functions (deformable_transformer_dino.py:132-171,289-301,612-646; results stored from the same
    inputs)."""
    from uninext_b200.modules.deformable_transformer import gen_encoder_output_proposals, get_sine_pos_embed
    want = rc.load("geometry_gpu")
    g = torch.Generator().manual_seed(90)
    n = 3
    ss, lsi, masks, flat, src, _ = _pyramid_inputs(n, g)
    want_vr = torch.from_numpy(want["valid_ratios"].reshape(tuple(want["valid_ratios.shape"]))).to(DEV)
    lib = _cabi.load()
    n0 = lib.msda_launch_count()
    got = get_reference_points(ss, want_vr)
    assert lib.msda_launch_count() - n0 == 1
    close = lambda got, key, **kw: torch.allclose(
        got.detach().cpu().reshape(-1)[rc.pick(got.numel(), want[key].size)], torch.from_numpy(want[key]), **kw)
    assert tuple(got.shape) == tuple(want["reference_points.shape"]) and close(got, "reference_points", rtol=1e-6, atol=1e-7)

    h = rc.ProposalHolder(256, 91).to(DEV)
    n0 = lib.msda_launch_count()
    prop, keep = gen_encoder_output_proposals(flat, ss)
    assert lib.msda_launch_count() - n0 == 2
    want_prop = torch.from_numpy(want["proposals"]).reshape(tuple(want["proposals.shape"]))
    assert torch.equal(torch.isinf(prop).cpu(), torch.isinf(want_prop))
    fin = ~torch.isinf(want_prop)
    assert torch.allclose(prop.cpu()[fin], want_prop[fin], rtol=1e-5, atol=1e-5)
    got_mem = h.enc_output_norm(h.enc_output(src.masked_fill(~keep, 0.0)))
    assert tuple(got_mem.shape) == tuple(want["memory.shape"]) and close(got_mem, "memory", rtol=1e-4, atol=1e-5)

    pos = torch.rand(2, 19, 4, generator=g).to(DEV)
    a = pos.clone().requires_grad_(True)
    ya = get_sine_pos_embed(a)
    assert tuple(ya.shape) == tuple(want["sine.shape"]) and close(ya, "sine", rtol=0, atol=2e-5)
    go = torch.randn(ya.shape, generator=g).to(DEV)
    ya.backward(go)
    assert rc.rel_err(a.grad, want, "sine_grad") < 1e-4
    assert close(get_sine_pos_embed(pos[..., :2], 64, 20, False), "sine_xy_64_20", atol=2e-5)
