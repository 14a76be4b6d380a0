"""Golden vectors of the REFERENCE's own code for the cases in tests/reference_cases.py -> tests/golden/reference/.

    python -m oracle.refstage                                   # stage the reference's Python files (oracle/_ref/py)
    python tests/golden/make_reference_golden.py                # CPU: reference layer classes, CondInst, geometry helpers
    python tests/golden/make_reference_golden.py --refcuda      # GPU: the reference's CUDA kernels (oracle/_ref, built by
                                                                #      oracle/build_refcuda.sh) on the parity inputs

CPU part: the reference's classes run unchanged with their MSDeformAttn op computed by the reference's own CPU function
``ms_deform_attn_core_pytorch`` (its CUDA extension is not built here); weights are this repo's modules' seeded weights
loaded into the reference classes (the state_dict keys are the reference's).  Nothing of this repo's compute is on the
reference side.  Only needed when a case changes; the tests read the stored files.
"""
import argparse
import inspect
import json
import os
import sys
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests import reference_cases as rc  # noqa: E402

REFCUDA_CASES = [("cfg1", "enc", "f32"), ("cfg2", "enc", "f32"), ("cfg2", "dec", "f32"), ("cfg1", "dec", "f64")]


def refcuda_id(cfgname, kind, dt):
    return f"refcuda_{cfgname}_{kind}_{dt}"


def _save(out_dir, name, blob):
    path = os.path.join(out_dir, name + ".npz")
    np.savez_compressed(path, **blob)
    print(f"{name}: {os.path.getsize(path) / 1024:.0f} KiB")


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


def cpu_goldens(out_dir):
    from oracle import refpy, refstage
    from uninext_b200.modules.deformable_transformer import MLP
    from uninext_b200.workloads import CONFIGS, make_inputs
    assert refstage.stage() and refpy.stage(), "no reference checkout to stage from"
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = refstage.import_reference()
        ddetrs = refstage.import_ddetrs()
    func_mod, dino = ref[0], ref[3]
    _CpuKernels.core = staticmethod(func_mod.ms_deform_attn_core_pytorch)
    func_mod.MSDA = _CpuKernels

    # reference layer classes (test_gpu_reference_dropin.py)
    for name in rc.DROPIN_CASES:
        _, theirs, run, inputs = rc.dropin_case(name, "cpu", ref)
        out, gin, gpar = rc.run_case(theirs, run, inputs)
        blob = {"param_names": np.array(sorted(gpar))}
        rc.store(blob, "out", out)
        for i, g in enumerate(gin):
            rc.store(blob, f"grad_in.{i}", g)
        for k, g in gpar.items():
            rc.store(blob, "grad." + k, g, k=512)
        _save(out_dir, "dropin_" + name, blob)

    # CondInst (test_gpu_condinst.py)
    blob = {}
    for factor, shape in rc.ALIGNED_CASES:
        x, g = rc.aligned_inputs(shape, "cpu")
        b = x.clone().requires_grad_(True)
        want = ddetrs.aligned_bilinear(b[None], factor)[0]
        want.backward(torch.randn(want.shape, generator=g))
        cid = rc.aligned_id(factor, shape)
        rc.store(blob, cid + "/out", want)
        rc.store(blob, cid + "/grad", b.grad)
    _save(out_dir, "condinst_aligned", blob)
    from uninext_b200.modules.dynamic_mask_head import dynamic_param_counts
    import types
    for rel_coord, num_insts, hw, stride in rc.DYNAMIC_CASES:
        feats, refs, params, g = rc.dynamic_inputs(rel_coord, num_insts, hw, "cpu")
        fb, rb, pb = (t.clone().requires_grad_(True) for t in (feats, refs, params))
        h = types.SimpleNamespace(dynamic_mask_channels=8, mask_out_stride=stride, use_raft=False)   # ddetrs.py:45-70
        h.weight_nums, h.bias_nums = dynamic_param_counts(3, rel_coord)
        h.mask_heads_forward = lambda *a, h=h: ddetrs.DDETRSegmUni.mask_heads_forward(h, *a)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            want = ddetrs.DDETRSegmUni.dynamic_mask_with_coords(h, fb, rb, pb, num_insts=num_insts, mask_feat_stride=8,
                                                                rel_coord=rel_coord)
        want.backward(torch.randn(want.shape, generator=g))
        blob = {}
        rc.store(blob, "out", want)
        rc.store(blob, "grad_feats", fb.grad)
        rc.store(blob, "grad_params", pb.grad)
        if rel_coord:
            rc.store(blob, "grad_refs", rb.grad)
        _save(out_dir, rc.dynamic_id(rel_coord, num_insts, hw, stride), blob)

    # geometry on the GPU (test_geometry_kernels_match_reference_functions)
    g = torch.Generator().manual_seed(90)
    ss, lsi, masks, flat, src, _ = rc.pyramid_inputs(3, g, "cpu")
    holder = dino.DeformableTransformerVLDINO.__new__(dino.DeformableTransformerVLDINO)
    vr = torch.stack([dino.DeformableTransformerVLDINO.get_valid_ratio(holder, m) for m in masks], 1)
    blob = {}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        rc.store(blob, "valid_ratios", vr)
        rc.store(blob, "reference_points", dino.DeformableTransformerEncoderVL.get_reference_points(ss, vr, device="cpu"),
                 k=1 << 20)
        mem, prop = dino.DeformableTransformerVLDINO.gen_encoder_output_proposals(rc.ProposalHolder(256, 91), src, flat, ss)
    rc.store(blob, "proposals", prop, k=1 << 20)
    rc.store(blob, "memory", mem)
    pos = torch.rand(2, 19, 4, generator=g)
    b = pos.clone().requires_grad_(True)
    y = dino.get_sine_pos_embed(b)
    y.backward(torch.randn(y.shape, generator=g))
    rc.store(blob, "sine", y, k=1 << 20)
    rc.store(blob, "sine_grad", b.grad)
    rc.store(blob, "sine_xy_64_20", dino.get_sine_pos_embed(pos[..., :2], 64, 20, False), k=1 << 20)
    _save(out_dir, "geometry_gpu", blob)

    # host-side mirrors (test_reference_mirrors.py)
    blob = {}
    g = torch.Generator().manual_seed(0)
    pos = torch.rand(2, 7, 4, generator=g)
    for xy in (True, False):
        rc.store(blob, f"sine_xy{int(xy)}", dino.get_sine_pos_embed(pos, exchange_xy=xy), k=1 << 20)
    rc.store(blob, "sine_64_20", dino.get_sine_pos_embed(pos[..., :2], 64, 20), k=1 << 20)
    torch.manual_seed(1)
    ours = MLP(512, 256, 256, 2)
    theirs = dino.MLP(512, 256, 256, 2)
    theirs.load_state_dict(ours.state_dict(), strict=True)
    rc.store(blob, "mlp", theirs(torch.randn(3, 5, 512, generator=g)), k=1 << 20)
    g = torch.Generator().manual_seed(2)
    masks = rc.mirror_masks(3, rc.MIRROR_SHAPES, g)
    vr = torch.stack([dino.DeformableTransformerVLDINO.get_valid_ratio(holder, m) for m in masks], 1)
    rc.store(blob, "valid_ratios", vr)
    rc.store(blob, "reference_points", dino.DeformableTransformerEncoderVL.get_reference_points(
        torch.as_tensor(rc.MIRROR_SHAPES), vr, device="cpu"), k=1 << 20)
    g = torch.Generator().manual_seed(3)
    masks = rc.mirror_masks(2, rc.MIRROR_SHAPES, g)
    flat = torch.cat([m.flatten(1) for m in masks], 1)
    memory = torch.randn(2, flat.shape[1], 16, generator=g)
    mem, prop = dino.DeformableTransformerVLDINO.gen_encoder_output_proposals(rc.ProposalHolder(16, 4), memory, flat,
                                                                              torch.as_tensor(rc.MIRROR_SHAPES))
    rc.store(blob, "proposals", prop, k=1 << 20)
    rc.store(blob, "memory", mem, k=1 << 20)
    _save(out_dir, "mirrors", blob)

    # positional signatures and parameter layout of the reference layers (test_layer_signatures_match_reference)
    names = lambda f: [n for n, p in inspect.signature(f).parameters.items() if p.kind != p.KEYWORD_ONLY][1:]
    head = dino.DeformableReidHead(256, dino.DeformableTransformerDecoderLayer(256, 512, 0.0, "relu", 4, 8, 4), 2)
    sig = {"DeformableTransformerEncoderLayer.forward": names(dino.DeformableTransformerEncoderLayer.forward),
           "DeformableTransformerDecoderLayer.forward": names(dino.DeformableTransformerDecoderLayer.forward),
           "DeformableReidHead.forward": names(dino.DeformableReidHead.forward),
           "DeformableReidHead.state_dict": {k: list(v.shape) for k, v in head.state_dict().items()}}
    with open(os.path.join(out_dir, "signatures.json"), "w") as fh:
        json.dump(sig, fh, indent=1, sort_keys=True)
        fh.write("\n")

    # the reference's CPU function itself (test_reference_file_and_port_agree)
    core = refpy.core_pytorch()
    c = make_inputs(CONFIGS["cfg1"], "dec", "cpu", seed=5, wild_fraction=0.1)
    v, lo, at = (c[k].clone().requires_grad_(True) for k in ("value", "sampling_locations", "attention_weights"))
    out = core(v, c["spatial_shapes"], lo, at)
    out.backward(c["grad_output"])
    blob = {}
    for k, t in (("out", out), ("grad_value", v.grad), ("grad_loc", lo.grad), ("grad_attn", at.grad)):
        rc.store(blob, k, t, k=8192)
    _save(out_dir, "core_pytorch_cfg1_dec", blob)


def refcuda_goldens(out_dir):
    from oracle import refcuda
    from uninext_b200.workloads import CONFIGS, make_inputs
    assert refcuda.available(), "oracle/_ref/libmsda_refcuda.so not built"
    for cfgname, kind, dt in REFCUDA_CASES:
        dtype = torch.float32 if dt == "f32" else torch.float64
        inp = make_inputs(CONFIGS[cfgname], kind, "cuda", dtype=dtype, seed=13, wild_fraction=0.05)
        a = (inp["value"], inp["spatial_shapes"], inp["level_start_index"], inp["sampling_locations"],
             inp["attention_weights"])
        out = refcuda.forward(*a)
        gv, gl, ga = refcuda.backward(*a, inp["grad_output"])
        torch.cuda.synchronize()
        blob = {"input_sums": np.array([float(inp[k].double().sum()) for k in
                                        ("value", "sampling_locations", "attention_weights", "grad_output")])}
        for k, t in (("out", out), ("grad_value", gv), ("grad_loc", gl), ("grad_attn", ga)):
            rc.store(blob, k, t, k=8192)
        _save(out_dir, refcuda_id(cfgname, kind, dt), blob)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--refcuda", action="store_true", help="the reference CUDA kernel cases (needs a GPU)")
    ap.add_argument("--out", default=rc.GOLDEN_REF)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    refcuda_goldens(a.out) if a.refcuda else cpu_goldens(a.out)
