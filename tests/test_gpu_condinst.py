"""GPU tests (-m gpu) of the CondInst dynamic mask head (uninext_b200/modules/dynamic_mask_head.py, kernels in
csrc/msda_condinst.cuh) against the REFERENCE functions themselves -- ``DDETRSegmUni.dynamic_mask_with_coords`` /
``mask_heads_forward`` / ``parse_dynamic_params`` / ``aligned_bilinear`` / ``compute_locations`` of
uninext/models/ddetrs.py, whose fp32 results on the same inputs are stored under tests/golden/reference
(tests/reference_cases.py, tests/golden/make_reference_golden.py): forward and every gradient (mask features, dynamic
parameters, reference points), fp32, 2e-4 of scale."""
import pytest
import torch

from tests import reference_cases as rc

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from uninext_b200 import _cabi
    from uninext_b200.modules.dynamic_mask_head import CondInstMaskHead, aligned_bilinear, dynamic_mask_with_coords

DEV = "cuda"


@pytest.fixture(scope="module")
def aligned_golden():
    return rc.load("condinst_aligned")


@pytest.mark.parametrize("factor", [2, 4])
@pytest.mark.parametrize("shape", [(3, 5, 7), (2, 1, 1), (1, 13, 21), (5, 40, 66)])
def test_aligned_bilinear_matches_reference(aligned_golden, factor, shape):
    x, g = rc.aligned_inputs(shape, DEV)
    a = x.clone().requires_grad_(True)
    got = aligned_bilinear(a, factor)
    cid = rc.aligned_id(factor, shape)
    assert rc.rel_err(got, aligned_golden, cid + "/out") < 1e-6
    go = torch.randn(got.shape, generator=g).to(DEV)
    got.backward(go)
    assert rc.rel_err(a.grad, aligned_golden, cid + "/grad") < 1e-5


@pytest.mark.parametrize("rel_coord", [True, False])
@pytest.mark.parametrize("num_insts,hw,mask_out_stride", [([5, 3], (12, 20), 4), ([0, 7], (9, 11), 4), ([37, 21, 1], (25, 42), 8),
                                                          ([300], (32, 40), 4), ([30, 17], (100, 168), 4), ([3], (7, 9), 2)])
def test_dynamic_mask_head_matches_reference(rel_coord, num_insts, hw, mask_out_stride):
    feats, refs, params, g = rc.dynamic_inputs(rel_coord, num_insts, hw, DEV)
    want = rc.load(rc.dynamic_id(rel_coord, num_insts, hw, mask_out_stride))
    fa, ra, pa = (t.clone().requires_grad_(True) for t in (feats, refs, params))
    lib = _cabi.load()
    before = lib.msda_launch_count()
    got = dynamic_mask_with_coords(fa, ra, pa, num_insts, 8, rel_coord, mask_out_stride)
    assert lib.msda_launch_count() > before
    assert rc.rel_err(got, want, "out") < 2e-4
    go = torch.randn(got.shape, generator=g).to(DEV)
    got.backward(go)
    assert rc.rel_err(fa.grad, want, "grad_feats") < 2e-4
    assert rc.rel_err(pa.grad, want, "grad_params") < 2e-4
    if rel_coord:
        assert rc.rel_err(ra.grad, want, "grad_refs") < 1e-3      # piecewise-linear through two ReLUs: sums of many signed terms


def test_condinst_module_parameter_names_and_forward():
    torch.manual_seed(3)
    head = CondInstMaskHead(256).to(DEV)
    assert set(head.state_dict()) == {f"controller.layers.{i}.{k}" for i in range(3) for k in ("weight", "bias")}
    assert head.num_gen_params == 169 and head.controller.layers[2].out_features == 169
    hs = torch.randn(2, 30, 256, device=DEV)
    feats = torch.randn(2, 8, 10, 16, device=DEV, requires_grad=True)
    refs = torch.rand(2, 30, 2, device=DEV) * 100
    sel = [torch.tensor([1, 5, 7], device=DEV), torch.tensor([0, 29], device=DEV)]
    out = head(hs, feats, refs, sel)
    assert out.shape == (1, 5, 20, 32)
    out.square().mean().backward()
    assert feats.grad is not None and all(p.grad is not None and torch.isfinite(p.grad).all() for p in head.parameters())
