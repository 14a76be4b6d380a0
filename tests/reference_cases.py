"""Inputs, weights and stored results of the tests that compare this repo with the REFERENCE's own code.

The reference's Python classes and CUDA kernels are not part of this repository.  tests/golden/make_reference_golden.py
ran them once on the cases defined here and stored what they computed under tests/golden/reference/; the tests rebuild
the same inputs and weights from the same seeds (CPU generators, so every machine gets the same numbers) and compare
this repo's results with the stored ones.  Large tensors are stored as a fixed sample of their elements (``pick``) plus
the maximum magnitude of the whole tensor, so errors stay relative to the scale of the full result.
"""
from __future__ import annotations

import os

import numpy as np
import torch

GOLDEN_REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
SHAPES = [(20, 28), (10, 14), (5, 7), (3, 4)]
FULL = 4096                           # tensors up to this many elements are stored whole


def pick(numel: int, k: int) -> np.ndarray:
    """k distinct, spread-out flat indices of a tensor with `numel` elements (all of them when numel <= k).
    i * 2654435761 mod numel is a permutation of range(numel) because the multiplier is a prime larger than numel."""
    if numel <= k:
        return np.arange(numel, dtype=np.int64)
    return np.sort((np.arange(k, dtype=np.int64) * 2654435761) % numel)


def store(blob: dict, key: str, t, k: int = FULL):
    """Adds tensor `t` (or its sample) to `blob` under `key`, with its shape and scale."""
    a = t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)
    flat = a.reshape(-1)
    blob[key] = flat[pick(flat.size, k)]
    blob[key + ".shape"] = np.asarray(a.shape, dtype=np.int64)
    blob[key + ".scale"] = np.asarray(np.abs(flat).max() if flat.size else 0.0, dtype=np.float64)


def load(name: str) -> dict:
    with np.load(os.path.join(GOLDEN_REF, name + ".npz")) as z:
        return {k: z[k] for k in z.files}


def rel_err(got, blob: dict, key: str) -> float:
    """max |got - stored| over the stored elements, relative to the stored scale of the whole tensor."""
    a = got.detach().double().cpu().numpy() if torch.is_tensor(got) else np.asarray(got, dtype=np.float64)
    assert tuple(a.shape) == tuple(blob[key + ".shape"]), (key, a.shape, blob[key + ".shape"])
    want = blob[key].astype(np.float64)
    flat = a.reshape(-1)[pick(a.size, want.size)]
    return float(np.abs(flat - want).max(initial=0.0) / max(float(blob[key + ".scale"]), 1e-30))


# ---------------------------------------------------------------------------------------------------------------------
# reference layer classes on the drop-in (tests/test_gpu_reference_dropin.py)
# ---------------------------------------------------------------------------------------------------------------------
def pyramid_inputs(n, gen, device, c=256, masked=True):
    from uninext_b200.workloads import level_tensors
    ss, lsi = level_tensors(SHAPES, device)
    s = sum(h * w for h, w in SHAPES)
    masks = []
    for h, w in SHAPES:
        m = torch.zeros(n, h, w, dtype=torch.bool)
        if masked:
            for b in range(n):
                m[b, int(h * (0.7 + 0.3 * b / max(1, n - 1))):, :] = True
                m[b, :, int(w * (0.6 + 0.4 * b / max(1, n - 1))):] = True
        masks.append(m.to(device))
    flat = torch.cat([m.flatten(1) for m in masks], 1)
    src = torch.randn(n, s, c, generator=gen).to(device)
    pos = torch.randn(n, s, c, generator=gen).to(device)
    return ss, lsi, masks, flat, src, pos


def decoder_inputs(n, q, gen, device):
    tgt = torch.randn(n, q, 256, generator=gen).to(device)
    qpos = torch.randn(n, q, 256, generator=gen).to(device)
    boxes = torch.cat((torch.rand(n, q, 2, generator=gen), 0.05 + 0.3 * torch.rand(n, q, 2, generator=gen)), -1).to(device)
    return tgt, qpos, boxes


def _perturb(module, seed):
    """The reference zero-initialises sampling_offsets / attention_weights weights; give them signal (CPU generator)."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in module.named_parameters():
            if name.endswith("sampling_offsets.weight"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
            elif name.endswith("attention_weights.weight"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.05)


DROPIN_CASES = ["module_0", "encoder_0", "module_1", "encoder_1", "decoder_0", "decoder_1", "reid",
                "decoder_loop_refine", "decoder_loop_plain"]


def dropin_case(name, device, ref=None):
    """-> (ours, theirs, run, inputs): this repo's module with seeded weights (built on the CPU, then moved to `device`),
    the reference's class with the same state_dict when `ref` (oracle.refstage.import_reference()) is given, else None;
    run(module, *leaves) -> output; inputs = the leaf tensors whose gradients are compared."""
    from uninext_b200.modules import MSDeformAttn
    from uninext_b200.modules.deformable_layers import (DeformableTransformerDecoderLayer,
                                                        DeformableTransformerEncoderLayer)
    from uninext_b200.modules.deformable_transformer import (MLP, DeformableReidHead, DeformableTransformerDecoder,
                                                             get_reference_points, valid_ratios_from_masks)
    kind, _, arg = name.rpartition("_") if name != "reid" else ("reid", "", "")
    which = int(arg) if arg.isdigit() else 0
    layer_args = (256, 512, 0.0, "relu", 4, 8, 4)
    if kind in ("module", "encoder"):
        g = torch.Generator().manual_seed(40 + which)
        ss, lsi, masks, flat, src, pos = pyramid_inputs(2, g, device)
        refpts = get_reference_points(SHAPES, valid_ratios_from_masks(masks))
        if kind == "module":
            torch.manual_seed(1)
            ours = MSDeformAttn(256, 4, 8, 4)
            make_theirs = lambda: ref[1].MSDeformAttn(256, 4, 8, 4)
            run, inputs = (lambda m, q, x: m(q, refpts, x, ss, lsi, flat)), [src + pos, src]
        else:
            torch.manual_seed(2)
            ours = DeformableTransformerEncoderLayer(*layer_args)
            make_theirs = lambda: ref[2 + which].DeformableTransformerEncoderLayer(*layer_args)
            run, inputs = (lambda m, x: m(x, pos, refpts, ss, lsi, flat)), [src]
        seed = 1 if kind == "module" else 2
    elif kind == "decoder":
        g = torch.Generator().manual_seed(50 + which)
        n, q = 2, 37
        ss, lsi, masks, flat, src, _ = pyramid_inputs(n, g, device)
        vr = valid_ratios_from_masks(masks)
        tgt, qpos, boxes = decoder_inputs(n, q, g, device)
        ref_in = boxes[:, :, None] * torch.cat((vr, vr), -1)[:, None]                  # _dino.py:451-452
        torch.manual_seed(3)
        ours = DeformableTransformerDecoderLayer(*layer_args)
        make_theirs = lambda: ref[2 + which].DeformableTransformerDecoderLayer(*layer_args)
        if which == 0:
            run = lambda m, t, x: m(t, qpos, ref_in, x, ss, lsi, flat)
        else:
            # DINO: denoising groups must not attend to each other (float mask, -inf where blocked; _dino.py:408-412)
            am = torch.zeros(q, q, device=device)
            am[:12, 12:] = float("-inf"); am[12:, :12] = float("-inf")
            run = lambda m, t, x: m(t, qpos, ref_in, x, ss, lsi, flat, am)
        inputs, seed = [tgt, src], 3
    elif kind == "reid":
        g = torch.Generator().manual_seed(60)
        ss, lsi, masks, flat, src, _ = pyramid_inputs(2, g, device)
        vr = valid_ratios_from_masks(masks)
        tgt, _, boxes = decoder_inputs(2, 19, g, device)
        torch.manual_seed(4)
        ours = DeformableReidHead(256, DeformableTransformerDecoderLayer(*layer_args), 2)
        make_theirs = lambda: ref[3].DeformableReidHead(256, ref[3].DeformableTransformerDecoderLayer(*layer_args), 2)
        run, inputs, seed = (lambda m, t, x: m(t, boxes, x, ss, lsi, vr, None, flat, None)), [tgt, src], 4
    elif kind == "decoder_loop":
        refine = arg == "refine"
        g = torch.Generator().manual_seed(80)
        n, q, nl = 2, 23, 3
        ss, lsi, masks, flat, src, _ = pyramid_inputs(n, g, device)
        vr = valid_ratios_from_masks(masks)
        tgt, _, boxes = decoder_inputs(n, q, g, device)
        torch.manual_seed(6)
        ours = DeformableTransformerDecoder(256, DeformableTransformerDecoderLayer(*layer_args), nl,
                                            return_intermediate=True, look_forward_twice=refine)
        if refine:          # the detector attaches the box heads to the decoder (iterative refinement), as the reference does
            ours.bbox_embed = torch.nn.ModuleList(MLP(256, 256, 4, 3) for _ in range(nl))

        def make_theirs():
            dino = ref[3]
            m = dino.DeformableTransformerDecoder(256, dino.DeformableTransformerDecoderLayer(*layer_args), nl,
                                                  return_intermediate=True, look_forward_twice=refine)
            if refine:
                m.bbox_embed = torch.nn.ModuleList(dino.MLP(256, 256, 4, 3) for _ in range(nl))
            return m

        def run(m, t, x):
            hs, refs = m(t, boxes, x, ss, lsi, vr, None, flat, None)
            return torch.cat((hs.flatten(), refs.flatten()))
        inputs, seed = [tgt, src], 6
    else:
        raise ValueError(name)
    _perturb(ours, 100 + seed)
    theirs = None
    if ref is not None:
        theirs = make_theirs()
        theirs.load_state_dict(ours.state_dict(), strict=True)       # this repo's keys load unchanged
        theirs.to(device)
    return ours.to(device), theirs, run, inputs


def run_case(module, run, inputs):
    """Forward + backward of a seeded grad_output -> (out, [input grads], {param name: grad})."""
    import warnings
    leaves = [t.clone().requires_grad_(True) for t in inputs]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        out = run(module, *leaves)
        go = torch.randn(out.shape, generator=torch.Generator().manual_seed(99)).to(out.device)
        out.backward(go)
    return out, [l.grad for l in leaves], {k: p.grad for k, p in module.named_parameters()}


# ---------------------------------------------------------------------------------------------------------------------
# CondInst dynamic mask head (tests/test_gpu_condinst.py)
# ---------------------------------------------------------------------------------------------------------------------
ALIGNED_CASES = [(f, s) for s in [(3, 5, 7), (2, 1, 1), (1, 13, 21), (5, 40, 66)] for f in (2, 4)]
DYNAMIC_CASES = [(r, ni, hw, st) for (ni, hw, st) in [([5, 3], (12, 20), 4), ([0, 7], (9, 11), 4), ([37, 21, 1], (25, 42), 8),
                                                       ([300], (32, 40), 4), ([30, 17], (100, 168), 4), ([3], (7, 9), 2)]
                 for r in (True, False)]


def aligned_id(factor, shape):
    return f"f{factor}_" + "x".join(map(str, shape))


def dynamic_id(rel_coord, num_insts, hw, stride):
    return f"condinst_dynamic_{'rel' if rel_coord else 'abs'}_{'-'.join(map(str, num_insts)) or 'none'}_{hw[0]}x{hw[1]}_s{stride}"


def aligned_inputs(shape, device):
    g = torch.Generator().manual_seed(1)
    x = torch.randn(*shape, generator=g).to(device)
    return x, g


def dynamic_inputs(rel_coord, num_insts, hw, device):
    from uninext_b200.modules.dynamic_mask_head import dynamic_param_counts
    g = torch.Generator().manual_seed(2)
    n, (h, w), total = len(num_insts), hw, sum(num_insts)
    npar = sum(sum(x) for x in dynamic_param_counts(3, rel_coord))
    feats = torch.randn(n, 8, h, w, generator=g).to(device)
    refs = (torch.rand(1, total, 2, generator=g) * torch.tensor([w * 8.0, h * 8.0])).to(device)
    params = (torch.randn(1, total, npar, generator=g) * 0.3).to(device)
    return feats, refs, params, g


# ---------------------------------------------------------------------------------------------------------------------
# geometry helpers (tests/test_reference_mirrors.py on the CPU, test_geometry_kernels_match_reference_functions on the GPU)
# ---------------------------------------------------------------------------------------------------------------------
MIRROR_SHAPES = [(12, 20), (6, 10), (3, 5), (2, 3)]


def mirror_masks(n, shapes, gen):
    """Padding masks the way the reference pads a batch: valid region top-left, padded right / bottom."""
    out = []
    fr = torch.rand(n, 2, generator=gen) * 0.5 + 0.5
    for h, w in shapes:
        m = torch.ones(n, h, w, dtype=torch.bool)
        for b in range(n):
            vh, vw = max(1, int(round(h * fr[b, 0].item()))), max(1, int(round(w * fr[b, 1].item())))
            m[b, :vh, :vw] = False
        out.append(m)
    return out


class ProposalHolder(torch.nn.Module):
    """What the reference's gen_encoder_output_proposals reads from `self`: enc_output / enc_output_norm."""
    def __init__(self, c, seed):
        super().__init__()
        torch.manual_seed(seed)
        self.enc_output = torch.nn.Linear(c, c)
        self.enc_output_norm = torch.nn.LayerNorm(c)
