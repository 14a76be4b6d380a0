#!/usr/bin/env python
"""CondInst dynamic mask head: this repo's fused kernels vs the REFERENCE function (staged uninext/models/ddetrs.py:
repeat + three grouped convolutions + aligned_bilinear) on the same B200, forward and forward+backward.
    python tools/condinst_bench.py          (needs oracle/_ref/py staged: python -m oracle.refstage)"""
import json
import os
import sys
import types
import warnings

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import refstage  # noqa: E402
from uninext_b200.modules.dynamic_mask_head import dynamic_mask_with_coords, dynamic_param_counts  # noqa: E402

with warnings.catch_warnings():
    warnings.simplefilter("ignore")
    ddetrs = refstage.import_ddetrs()
h = types.SimpleNamespace(dynamic_mask_channels=8, mask_out_stride=4, use_raft=False)
h.weight_nums, h.bias_nums = dynamic_param_counts(3, True)
h.mask_heads_forward = lambda *a: ddetrs.DDETRSegmUni.mask_heads_forward(h, *a)


def timeit(fn, iters=10, warm=3):
    xs = []
    for i in range(warm + iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        if i >= warm:
            xs.append(e0.elapsed_time(e1))
    return sorted(xs)[len(xs) // 2]


for name, num_insts, hw in (("inference, 2 x 300 queries, 100x168", [300, 300], (100, 168)),
                            ("training, 2 x 30 matched instances, 100x168", [30, 30], (100, 168)),
                            ("video clip cfg4, 5 x 300 queries, 48x80", [300] * 5, (48, 80))):
    n, total = len(num_insts), sum(num_insts)
    g = torch.Generator().manual_seed(0)
    feats = torch.randn(n, 8, *hw, generator=g).cuda().requires_grad_(True)
    refs = (torch.rand(1, total, 2, generator=g) * torch.tensor([hw[1] * 8.0, hw[0] * 8.0])).cuda().requires_grad_(True)
    params = (torch.randn(1, total, 169, generator=g) * 0.3).cuda().requires_grad_(True)
    ours = lambda: dynamic_mask_with_coords(feats, refs, params, num_insts, 8, True, 4)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        theirs = lambda: ddetrs.DDETRSegmUni.dynamic_mask_with_coords(h, feats, refs, params, num_insts=num_insts, mask_feat_stride=8,
                                                                      rel_coord=True)
        row = {"case": name}
        for tag, fn in (("ours", ours), ("reference", theirs)):
            with torch.no_grad():
                row[tag + "_fwd_ms"] = round(timeit(fn), 4)

            def fb():
                out = fn()
                out.backward(torch.ones_like(out))
                feats.grad = refs.grad = params.grad = None
            torch.cuda.reset_peak_memory_stats()
            row[tag + "_fwd_bwd_ms"] = round(timeit(fb), 4)
            row[tag + "_peak_MB"] = round(torch.cuda.max_memory_allocated() / 1e6, 1)
        row["speedup_fwd"] = round(row["reference_fwd_ms"] / row["ours_fwd_ms"], 2)
        row["speedup_fwd_bwd"] = round(row["reference_fwd_bwd_ms"] / row["ours_fwd_bwd_ms"], 2)
    print(json.dumps(row), flush=True)
