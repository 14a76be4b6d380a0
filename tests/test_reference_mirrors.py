"""CPU tests: the host-side mirrors of the reference's helpers around the op (reference points, proposals, sine position
embedding, MLP) against what the REFERENCE functions themselves compute on the same inputs (stored under
tests/golden/reference by tests/golden/make_reference_golden.py; cases in tests/reference_cases.py)."""
import json
import os

import pytest
import torch

from tests import reference_cases as rc

SHAPES = rc.MIRROR_SHAPES


@pytest.fixture(scope="module")
def want():
    return rc.load("mirrors")


def _stored(want, key):
    return torch.from_numpy(want[key]).reshape(tuple(want[key + ".shape"]))


def test_sine_pos_embed_and_mlp(want):
    from uninext_b200.modules.deformable_transformer import MLP, get_sine_pos_embed
    g = torch.Generator().manual_seed(0)
    pos = torch.rand(2, 7, 4, generator=g)
    for xy in (True, False):
        assert torch.allclose(get_sine_pos_embed(pos, exchange_xy=xy), _stored(want, f"sine_xy{int(xy)}"), rtol=0, atol=1e-6)
    assert torch.allclose(get_sine_pos_embed(pos[..., :2], 64, 20), _stored(want, "sine_64_20"), atol=1e-6)
    torch.manual_seed(1)
    a = MLP(512, 256, 256, 2)
    x = torch.randn(3, 5, 512, generator=g)
    # the reference MLP with these weights, computed once; the same two GEMMs + ReLU agree to rounding on any CPU
    torch.testing.assert_close(a(x), _stored(want, "mlp"), rtol=1e-6, atol=1e-6)


def test_reference_points_and_valid_ratios(want):
    from uninext_b200.modules.deformable_transformer import get_reference_points, valid_ratios_from_masks
    g = torch.Generator().manual_seed(2)
    masks = rc.mirror_masks(3, SHAPES, g)
    vr = valid_ratios_from_masks(masks)
    assert torch.equal(vr, _stored(want, "valid_ratios"))
    ss = torch.as_tensor(SHAPES)
    ref = _stored(want, "reference_points")
    got = get_reference_points(ss, vr)
    assert got.shape == ref.shape and torch.allclose(got, ref, rtol=1e-6, atol=1e-7)
    assert torch.allclose(get_reference_points(SHAPES, vr), ref, rtol=1e-6, atol=1e-7)        # cached grid, list input


def test_encoder_output_proposals(want):
    from uninext_b200.modules.deformable_transformer import gen_encoder_output_proposals
    g = torch.Generator().manual_seed(3)
    masks = rc.mirror_masks(2, SHAPES, g)
    flat = torch.cat([m.flatten(1) for m in masks], 1)
    memory = torch.randn(2, flat.shape[1], 16, generator=g)
    h = rc.ProposalHolder(16, 4)
    want_mem, want_prop = _stored(want, "memory"), _stored(want, "proposals")
    prop, keep = gen_encoder_output_proposals(flat, SHAPES)
    assert torch.equal(torch.isinf(prop), torch.isinf(want_prop))
    fin = ~torch.isinf(want_prop)
    assert torch.allclose(prop[fin], want_prop[fin], rtol=1e-5, atol=1e-6)
    got_mem = h.enc_output_norm(h.enc_output(memory.masked_fill(~keep, 0.0)))
    assert torch.allclose(got_mem, want_mem, rtol=1e-5, atol=1e-6)


def test_layer_signatures_match_reference():
    import inspect
    from uninext_b200.modules.deformable_layers import (DeformableTransformerDecoderLayer,
                                                        DeformableTransformerEncoderLayer)
    from uninext_b200.modules.deformable_transformer import DeformableReidHead
    with open(os.path.join(rc.GOLDEN_REF, "signatures.json")) as fh:
        ref = json.load(fh)
    # positional signature = the reference's; keyword-only extras (projected_value) are this repo's extensions
    names = lambda f: [n for n, p in inspect.signature(f).parameters.items() if p.kind != p.KEYWORD_ONLY][1:]
    assert names(DeformableTransformerEncoderLayer.forward) == ref["DeformableTransformerEncoderLayer.forward"]
    assert names(DeformableTransformerDecoderLayer.forward) == ref["DeformableTransformerDecoderLayer.forward"]
    assert names(DeformableReidHead.forward) == ref["DeformableReidHead.forward"]
    ours = DeformableReidHead(256, DeformableTransformerDecoderLayer(256, 512, 0.0, "relu", 4, 8, 4), 2)
    assert {k: list(v.shape) for k, v in ours.state_dict().items()} == ref["DeformableReidHead.state_dict"]
