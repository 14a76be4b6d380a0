#!/usr/bin/env python
"""Cost of the deterministic backward (torch.use_deterministic_algorithms(True) -> msda_backward_det_*).

    python tools/deterministic_bench.py [--iters 30] [--out profiles/det_bench.json]

Per case (cfg2 encoder- / decoder-shaped calls in fp32, cfg3/4/5 in bf16) the drop-in backward is timed with the flag
off and on, alternating in the same process, CUDA events around each call and the L2 overwritten before it (as
tools/opbench.py).  "on" is measured twice: with torch's fill of uninitialised memory
(torch.utils.deterministic.fill_uninitialized_memory, the default under the flag, which also fills the shim's
torch.empty outputs) and without it.  One profiled deterministic call per case splits the device time into the phases
zero-fill / scale / accumulate / convert.  Then the 6+6-layer DeformableStack fwd+bwd step at cfg2 (TF32, eager) is
timed the same way in the same three modes.  Prints one JSON document (GPU name and power limit included)."""
import argparse
import json
import os
import subprocess
import sys

os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")     # torch's own GEMMs under the flag (read at cuBLAS init)

import torch
import torch.utils.deterministic

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from uninext_b200.dropin import MultiScaleDeformableAttention as MSDA  # noqa: E402
from uninext_b200.workloads import CONFIGS, make_inputs  # noqa: E402

CASES = [("cfg2", "enc", torch.float32), ("cfg2", "dec", torch.float32)] + \
        [(c, k, torch.bfloat16) for c in ("cfg3", "cfg4", "cfg5") for k in ("enc", "dec")]
PHASES = (("zero_fill", ("msda_zero_fill", "Memset")), ("scale", ("msda_det_scale", "msda_det_prepare")),
          ("accumulate", ("msda_bwd_tiled", "msda_bwd_generic")), ("convert", ("msda_det_convert",)))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(("name", "power_limit", "max_sm_clock"), (s.strip() for s in q.split(","))))
    except Exception as exc:                 # report, do not guess
        return {"name": torch.cuda.get_device_name(), "error": str(exc)}


def set_mode(mode):
    torch.use_deterministic_algorithms(mode != "off")
    torch.utils.deterministic.fill_uninitialized_memory = mode != "on_nofill"


def phases(call):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    res = {k: 0.0 for k, _ in PHASES}
    res["other"] = 0.0
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = ev.device_time
        for k, keys in PHASES:
            if any(s in ev.name for s in keys):
                res[k] += us
                break
        else:
            res["other"] += us
    return {k: round(v / 1000.0, 4) for k, v in res.items()}


def step_times(iters, warmup, modes):
    from uninext_b200.modules.deformable_layers import DeformableStack
    from uninext_b200.workloads import level_tensors
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = True
    c = CONFIGS["cfg2"]
    torch.manual_seed(1234)
    model = DeformableStack(num_layers=6, num_queries=c.dec_queries).cuda()
    ss, lsi = level_tensors(c.shapes, "cuda")
    g = torch.Generator(device="cuda").manual_seed(77)
    src = torch.randn(c.batch, c.S, 256, device="cuda", generator=g)
    pos = torch.randn(c.batch, c.S, 256, device="cuda", generator=g)
    pad = torch.zeros(c.batch, c.S, dtype=torch.bool, device="cuda")
    times = {m: [] for m in modes}
    for i in range(warmup + iters):
        for m in modes:
            set_mode(m)
            model.zero_grad(set_to_none=True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            model(src, pos, c.shapes, ss, lsi, pad).square().mean().backward()
            e1.record()
            torch.cuda.synchronize()
            if i >= warmup:
                times[m].append(e0.elapsed_time(e1))
    set_mode("off")
    med = {m: sorted(t)[len(t) // 2] for m, t in times.items()}
    return {"step_off": round(med["off"], 3), "step_det": round(med["on"], 3), "step_det_nofill": round(med["on_nofill"], 3),
            "ratio": round(med["on"] / med["off"], 2), "ratio_nofill": round(med["on_nofill"] / med["off"], 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    modes = ("off", "on", "on_nofill")
    result = {"gpu": gpu_info(), "iters": a.iters, "unit": "ms (median)", "cases": []}
    for cfg, kind, dt in CASES:
        inp = make_inputs(CONFIGS[cfg], kind, "cuda", dtype=dt, seed=0)
        args = (inp["value"], inp["spatial_shapes"], inp["level_start_index"], inp["sampling_locations"],
                inp["attention_weights"], inp["grad_output"], 64)
        times = {m: [] for m in modes}
        for i in range(a.warmup + a.iters):
            for m in modes:                    # alternate: the three modes see the same machine state
                set_mode(m)
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                MSDA.ms_deform_attn_backward(*args)
                e1.record()
                torch.cuda.synchronize()
                if i >= a.warmup:
                    times[m].append(e0.elapsed_time(e1))
        med = {m: sorted(t)[len(t) // 2] for m, t in times.items()}
        set_mode("on_nofill")
        ph = phases(lambda: MSDA.ms_deform_attn_backward(*args))
        set_mode("off")
        row = {"config": cfg, "kind": kind, "dtype": str(dt).replace("torch.", ""),
               "bwd_off": round(med["off"], 4), "bwd_det": round(med["on"], 4), "bwd_det_nofill": round(med["on_nofill"], 4),
               "ratio": round(med["on"] / med["off"], 2), "ratio_nofill": round(med["on_nofill"] / med["off"], 2),
               "det_phases_profiled": ph}
        result["cases"].append(row)
        print(json.dumps(row), file=sys.stderr)
    result["step_cfg2_6+6_tf32_eager"] = step_times(a.iters, a.warmup, modes)
    print(json.dumps(result["step_cfg2_6+6_tf32_eager"]), file=sys.stderr)
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
