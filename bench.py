#!/usr/bin/env python
"""bench.py -- MSDeformAttn hot-path benchmark (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps K --warmup W      # the reference's own CPU path on the host cores

One *step* = one pass of the hot path over one batch of the workload (default cfg2 = BASELINE.json configs[1]:
COCO-shape 1333x800, R50 4-level features, 300 queries, 8 heads x 32, 4 levels x 4 points, batch 2, fp32): the
6 encoder-shaped + 6 decoder-shaped MSDeformAttn calls of one transformer pass, each forward AND backward,
through the reference-facing module functions (``MultiScaleDeformableAttention.ms_deform_attn_forward/backward``
-> C ABI).  Every call has its own input tensors (12 distinct sets, ~1 GB > the 126 MB L2), so nothing is served
from a warm cache between steps.

Reported (one JSON line, rank 0):
  value      -- Gsamples/s, whole job (all ranks), device-resident inputs; a sample = one bilinear D-vector tap
                (N*Lq*M*L*P per call), counted once per forward+backward pair.
  e2e        -- same metric with HOST (pinned) inputs and results: H2D of value/loc/attn/grad_out and D2H of
                out/grad_value/grad_loc/grad_attn inside the timed region.
  roofline   -- dominant kernel (encoder-shaped backward: zero-fill + msda_bwd_tiled) against the measured HBM peak.
  cpu_baseline -- the reference's ms_deform_attn_core_pytorch CPU path (its own file, staged in oracle/_ref; the
                  torch port pinned to it when no staged copy exists) on this box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from uninext_b200.workloads import CONFIGS, algorithmic_bytes, make_inputs  # noqa: E402

METRIC = "msdeformattn_fwd_bwd_gsamples_per_s"
UNIT = "Gsamples/s"
N_ENC, N_DEC = 6, 6        # op calls per transformer pass (deformable_transformer.py: 6 encoder + 6 decoder layers)


# ------------------------------------------------------------------------------------------------------------------
def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--dtype", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-frames", action="store_true", help="skip the whole-model frames/s measurement")
    ap.add_argument("--no-reference-cuda", action="store_true", help="skip timing the reference's own CUDA kernels")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config (cfg3/4/5 bf16) kernel table")
    ap.add_argument("--no-reference-stack", action="store_true",
                    help="skip timing the reference's own layer classes on its own CUDA kernels (frames.reference_stack)")
    ap.add_argument("--frames-steps", type=int, default=5)
    ap.add_argument("--cpu-budget-s", type=float, default=25.0, help="target CPU seconds for the cpu_baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0) as DIR/<call>_<name>.npy; see dump_outputs()")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dist_env():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return world, rank, local


def ncu_traffic(tag, key):
    """DRAM bytes per launch from the committed ncu --set full capture (tools/ncu_traffic.py), or None."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(p) as fh:
            return int(json.load(fh)[tag][key]["dram_bytes"])
    except (OSError, KeyError, ValueError):
        return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc, self.thr = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        def pump():
            for ln in self.proc.stdout:
                self.lines.append(ln.strip())
        self.thr = threading.Thread(target=pump, daemon=True)
        self.thr.start()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------------------------
def build_calls(cfg, device, dtype, seed0):
    """12 distinct input sets: 6 encoder-shaped (Lq = S) + 6 decoder-shaped (Lq = dec queries)."""
    calls = []
    for i in range(N_ENC):
        d = make_inputs(cfg, "enc", device, dtype=dtype, seed=seed0 + i)
        d["kind"] = "enc"
        calls.append(d)
    for i in range(N_DEC):
        d = make_inputs(cfg, "dec", device, dtype=dtype, seed=seed0 + 100 + i)
        d["kind"] = "dec"
        calls.append(d)
    return calls


def samples_per_step(cfg):
    return N_ENC * cfg.samples("enc") + N_DEC * cfg.samples("dec")


def run_b200(args):
    world, rank, local = dist_env()
    from uninext_b200 import build as _build
    if local == 0:                       # a clean checkout has no .so (git-ignored): build once per node, like build()
        _build.build()
    else:
        _build.wait_until_built()
    from uninext_b200 import _cabi
    from uninext_b200.dropin import MultiScaleDeformableAttention as MSDA

    world, rank, local = dist_env()
    if args.gpus != world and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if world == 1 and args.gpus > 1:
        raise SystemExit("launch multi-GPU runs with torch.distributed.run (one rank per GPU)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # NCCL prints its version banner on STDOUT: keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=device)
    lib = _cabi.load()
    cfg = CONFIGS[args.config]
    dtype = torch.float32 if args.dtype == "fp32" else torch.bfloat16
    elem = 4 if args.dtype == "fp32" else 2
    calls = build_calls(cfg, device, dtype, seed0=1000 * rank)
    smp_step = samples_per_step(cfg)

    def op_args(c):
        return (c["value"], c["spatial_shapes"], c["level_start_index"], c["sampling_locations"],
                c["attention_weights"])

    def step(ev=None, keep=None):
        for i, c in enumerate(calls):
            a = op_args(c)
            if ev is not None:
                ev[i][0].record()
            out = MSDA.ms_deform_attn_forward(*a, 64)
            if ev is not None:
                ev[i][1].record()
            grads = MSDA.ms_deform_attn_backward(*a, c["grad_output"], 64)
            if ev is not None:
                ev[i][2].record()
            if keep is not None:
                keep.append((out, *grads))
        return out, grads

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    dump = args.dump_outputs is not None and rank == 0
    for _ in range(max(3, args.warmup)):
        step(keep=[] if dump else None)    # when dumping, warm-up holds a step's results too: same allocator pool as the last timed step
    barrier()

    # ---- timed region: exactly K steps, device-resident inputs ----
    K = args.steps
    evs = [[[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in calls] for _ in range(K)]
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    barrier()
    launches0 = lib.msda_launch_count()
    last = [] if dump else None
    t0.record()
    for k in range(K):
        step(evs[k], keep=last if k == K - 1 else None)
    t1.record()
    barrier()
    launches = lib.msda_launch_count() - launches0
    if dump:
        dump_outputs(args.dump_outputs, calls, last)
        del last
    total_ms = t0.elapsed_time(t1)
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([total_ms], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_per_step = total_ms / K
    value = world * smp_step / (ms_per_step * 1e-3) / 1e9

    # per-kernel durations (events on the launching stream), averaged over the timed region
    def avg(kind, a, b):
        xs = [evs[k][i][a].elapsed_time(evs[k][i][b]) for k in range(K) for i, c in enumerate(calls) if c["kind"] == kind]
        return sum(xs) / len(xs)
    kern = {"enc_fwd_ms": avg("enc", 0, 1), "enc_bwd_ms": avg("enc", 1, 2),
            "dec_fwd_ms": avg("dec", 0, 1), "dec_bwd_ms": avg("dec", 1, 2)}
    peak, peak_src = measured_peaks()
    b_bwd = algorithmic_bytes(cfg, "enc", elem, "bwd")
    b_fwd = algorithmic_bytes(cfg, "enc", elem, "fwd")
    ach = b_bwd / (kern["enc_bwd_ms"] * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "encoder-shaped backward: grad_value zero-fill (msda_zero_fill, PDL primary) + msda_bwd_tiled",
                "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                "peak_source": peak_src, "algorithmic_bytes_per_launch": b_bwd,
                "traffic": ncu_traffic(f"{args.config}_enc_{'f32' if args.dtype == 'fp32' else 'bf16'}", "bwd"),
                "traffic_note": "msda_bwd_tiled only (the 45.7 MB grad_value zero-fill is a separate launch); profiles/ncu_traffic.json",
                "binding_ceiling": "backward: each SM's path into the crossbar carries ~25 B/clk of red.global payload (21.8 with all "
                                   "148 SMs active; scales with the SM count, independent of the hot-set size -> it is not the L2 "
                                   "atomic units; profiles/r02b_ubench_smem_rmw_and_egress.txt); the op must add 4 x 128 B per tap "
                                   "(2.5 GB per call) -> 393 us + gathers.  Combining rows inside the SM removes egress one for one "
                                   "but costs 4 shared-memory wavefronts per row on the LSU data pipe the gathers already keep > 50 % "
                                   "busy (slab kernels: -43 % red sectors, +36 % time; profiles/r02c_slab_kernels_ncu.md).  forward: "
                                   "LSU data pipe 66-72 % busy moving 2.93 GB of rows per call (>= 155 k wavefronts per SM)",
                "enc_fwd": {"achieved": round(b_fwd / (kern["enc_fwd_ms"] * 1e-3) / 1e9, 1),
                            "frac": round(b_fwd / (kern["enc_fwd_ms"] * 1e-3) / 1e9 / peak, 4),
                            "algorithmic_bytes_per_launch": b_fwd}}

    # ---- e2e: host (pinned) buffers, copies inside the timed region ----
    e2e, e2e_reps = None, []
    if not args.no_e2e:
        e2e_measure, e2e_result = setup_e2e(MSDA, calls, op_args, world, smp_step, args.e2e_steps, device, barrier)
        e2e_reps.append(e2e_measure())

    frames = None
    if not args.no_frames:
        frames = run_frames(cfg, world, rank, device, args.frames_steps, barrier, lib,
                            reference_stack=not args.no_reference_stack)
    if not args.no_e2e:
        e2e_reps.append(e2e_measure())

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_baseline(cfg, args.cpu_budget_s)

    ref_cuda = None
    if rank == 0 and world == 1 and not args.no_reference_cuda and args.dtype == "fp32":
        ref_cuda = reference_cuda_leg(calls, op_args, kern)

    other_cfgs = None
    if rank == 0 and world == 1 and not args.no_configs:
        other_cfgs = other_configs_leg(MSDA, device, peak)

    if not args.no_e2e:
        e2e_reps.append(e2e_measure())
        e2e = e2e_result(e2e_reps)

    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": K,
            "warmup": max(3, args.warmup), "ms_per_step": round(ms_per_step, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32" if args.dtype == "fp32" else "bf16",
            "data": "synthetic",
            "config": step_config(cfg, world),
            "kernels_ms": {k: round(v, 4) for k, v in kern.items()},
            "gsamples_per_s": {"enc_fwd": round(cfg.samples("enc") / kern["enc_fwd_ms"] / 1e6, 2),
                               "enc_bwd": round(cfg.samples("enc") / kern["enc_bwd_ms"] / 1e6, 2),
                               "dec_fwd": round(cfg.samples("dec") / kern["dec_fwd_ms"] / 1e6, 2),
                               "dec_bwd": round(cfg.samples("dec") / kern["dec_bwd_ms"] / 1e6, 2)},
            "roofline": roofline, "e2e": e2e, "frames": frames, "gpu_launches": int(launches), "clocks": clocks,
            "cpu_baseline": cpu_base, "reference_cuda": ref_cuda, "configs": other_cfgs,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


DUMP_ELEMS = 1 << 18      # per array: 12 calls x 4 arrays x 1 MB (float32) stay below 64 MB


def dump_outputs(path, calls, results):
    """Writes the arrays the timed path returned to its caller in the last timed step: for every call (enc0..enc5,
    dec0..dec5) ``out``, ``grad_value``, ``grad_loc`` and ``grad_attn`` as ``<call>_<name>.npy`` in float32 (bf16 results
    widened).  An array of more than DUMP_ELEMS elements is stored as a fixed sample: the flattened elements at indices
    i * 2654435761 mod numel for i < DUMP_ELEMS, ascending -- the same elements in every run, since the multiplier is a
    prime larger than any array here.  Inputs are seeded, so two builds run with the same arguments compare element for
    element: out, grad_loc and grad_attn repeat bit for bit, grad_value (accumulated with atomics) to rounding."""
    os.makedirs(path, exist_ok=True)
    counts = {"enc": 0, "dec": 0}
    for c, arrays in zip(calls, results):
        call = f"{c['kind']}{counts[c['kind']]}"
        counts[c["kind"]] += 1
        for name, t in zip(("out", "grad_value", "grad_loc", "grad_attn"), arrays):
            flat = t.detach().reshape(-1)
            if flat.numel() > DUMP_ELEMS:
                idx = torch.arange(DUMP_ELEMS, dtype=torch.int64, device=flat.device) * 2654435761 % flat.numel()
                flat = flat[idx.sort().values]
            np.save(os.path.join(path, f"{call}_{name}.npy"), flat.float().cpu().numpy())


def _time_call(fn, iters=10, warm=3):
    """Median CUDA-event time of fn() over `iters` runs, with a 256 MB write between runs to flush the 126 MB L2."""
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    xs = []
    for i in range(warm + iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        if i >= warm:
            xs.append(e0.elapsed_time(e1))
    return statistics.median(xs)


def reference_cuda_leg(calls, op_args, kern):
    """The REAL bar (BASELINE.md 2b): the reference's own CUDA kernels -- ms_deform_im2col_cuda.cuh compiled unmodified
    for sm_100a into oracle/_ref (oracle/build_refcuda.sh) -- timed on the same tensors of the same B200, OUTSIDE the
    timed region of this bench.  oracle/ is used here only as a measured baseline, like cpu_baseline."""
    try:
        from oracle import refcuda
    except Exception as exc:
        return {"unavailable": repr(exc)[:160]}
    if not refcuda.available():
        return {"unavailable": "oracle/_ref/libmsda_refcuda.so not built (needs /root/reference at build time)"}
    res = {"what": "reference kernels ms_deformable_im2col_gpu_kernel / ms_deformable_col2im_gpu_kernel_shm_blocksize_aware_"
                   "reduce_v1<float,32> incl. the reference wrapper's zero-fills (at::zeros, cu:54,121-123); median of 10, L2 "
                   "flushed; not part of `value`"}
    for kind in ("enc", "dec"):
        c = next(x for x in calls if x["kind"] == kind)
        a = op_args(c)
        outs = (torch.empty_like(a[0]), torch.empty_like(a[3]), torch.empty_like(a[4]))
        f = _time_call(lambda: refcuda.forward(*a))
        b = _time_call(lambda: refcuda.backward(*a, c["grad_output"], outs=outs))
        res[kind] = {"ref_fwd_ms": round(f, 4), "ref_bwd_ms": round(b, 4),
                     "ours_fwd_ms": round(kern[f"{kind}_fwd_ms"], 4), "ours_bwd_ms": round(kern[f"{kind}_bwd_ms"], 4),
                     "speedup_fwd": round(f / kern[f"{kind}_fwd_ms"], 2), "speedup_bwd": round(b / kern[f"{kind}_bwd_ms"], 2)}
    return res


def other_configs_leg(MSDA, device, peak):
    """BASELINE.json configs[2..4] (bf16): encoder- and decoder-shaped call times and the HBM-roofline fraction of the
    encoder-shaped ones (algorithmic bytes / time / measured peak).  Parity for these shapes: tests/test_gpu_parity.py."""
    res = {}
    for name in ("cfg3", "cfg4", "cfg5"):
        cfg = CONFIGS[name]
        row = {"workload": cfg.name, "dtype": "bf16"}
        for kind in ("enc", "dec"):
            c = make_inputs(cfg, kind, device, dtype=torch.bfloat16, seed=7)
            a = (c["value"], c["spatial_shapes"], c["level_start_index"], c["sampling_locations"], c["attention_weights"])
            f = _time_call(lambda: MSDA.ms_deform_attn_forward(*a, 64))
            b = _time_call(lambda: MSDA.ms_deform_attn_backward(*a, c["grad_output"], 64))
            smp = cfg.samples(kind)
            row[kind] = {"fwd_ms": round(f, 4), "bwd_ms": round(b, 4),
                         "gsamples_per_s_fwd_bwd": round(smp / (f + b) / 1e6, 2),
                         "frac_fwd": round(algorithmic_bytes(cfg, kind, 2, "fwd") / (f * 1e-3) / 1e9 / peak, 4),
                         "frac_bwd": round(algorithmic_bytes(cfg, kind, 2, "bwd") / (b * 1e-3) / 1e9 / peak, 4)}
            del c, a
        res[name] = row
    return res


def run_frames(cfg, world, rank, device, steps, barrier, lib, reference_stack=True):
    """Whole-model frames/s: one training step of the 6-encoder + 6-decoder-layer deformable transformer (fwd + bwd,
    fp32, d_model 256, d_ffn 2048) on synthetic multi-scale features of the workload's shape; frames sharded over ranks,
    ONE flat NCCL all-reduce of all parameter gradients per step.  Backbone, heads, matcher and losses are excluded."""
    from uninext_b200.dp import FlatGradBucket
    from uninext_b200.modules.deformable_layers import DeformableStack
    from uninext_b200.workloads import level_tensors
    torch.manual_seed(1234)                                   # identical weights on every rank
    model = DeformableStack(num_layers=6, num_queries=cfg.dec_queries).to(device)
    # gradient exchange overlapped with backward: 8 MB slices of the flat buffer are all-reduced from grad hooks as soon as
    # backward has filled them (DDP's behaviour, detectron2/engine/defaults.py:60-79); single GPU: nothing to exchange
    bucket = FlatGradBucket(model.parameters(), overlap=world > 1)
    shapes = cfg.shapes
    ss, lsi = level_tensors(shapes, device)
    g = torch.Generator(device=device).manual_seed(77 + rank)
    src = torch.randn(cfg.batch, cfg.S, 256, device=device, generator=g)
    pos = torch.randn(cfg.batch, cfg.S, 256, device=device, generator=g)
    # the reference always hands MSDeformAttn its padding mask (all-False for unpadded frames, SURVEY.md section 8d), so
    # value_proj is always followed by the masked_fill -- here fused into the GEMM's epilogue when TF32 products are allowed
    pad = torch.zeros(cfg.batch, cfg.S, dtype=torch.bool, device=device)

    def train_step(amp):
        bucket.zero_()
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            out = model(src, pos, shapes, ss, lsi, pad)
        out.float().square().mean().backward()
        bucket.finish()

    def measure(amp):
        for _ in range(3):
            train_step(amp)
        barrier()
        l0 = lib.msda_launch_count()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(steps):
            train_step(amp)
        t1.record()
        barrier()
        ms = t0.elapsed_time(t1)
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        ms /= steps
        return {"frames_per_s": round(world * cfg.batch / (ms * 1e-3), 2), "ms_per_step": round(ms, 3),
                "msda_launches_per_step": int((lib.msda_launch_count() - l0) / steps)}

    res = {"steps": steps, "frames_per_gpu": cfg.batch, "grad_allreduce_bytes": bucket.nbytes,
           "what": "6 enc + 6 dec deformable transformer layers fwd+bwd + one flat gradient all-reduce; synthetic "
                   "features and an all-False padding mask, backbone/heads/losses excluded. fp32 = strict fp32 GEMMs (cfg2's dtype); tf32 = "
                   "torch.backends.cuda.matmul.allow_tf32 (the default of the reference's PyTorch 1.10 stack); "
                   "amp_bf16 = autocast, MSDeformAttn still fp32 as in the reference (custom_fwd cast)"}
    res["fp32"] = measure(False)
    res["frames_per_s"] = res["fp32"]["frames_per_s"]
    res["ms_per_step"] = res["fp32"]["ms_per_step"]
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    res["tf32"] = measure(False)
    torch.backends.cuda.matmul.allow_tf32 = old
    res["amp_bf16"] = measure(True)

    # Whole step captured in a CUDA graph (launch-bound otherwise: ~1000 kernels, 15 ms of device work in a 20 ms step);
    # the gradient all-reduce stays outside the graph and runs after each replay.
    torch.backends.cuda.matmul.allow_tf32 = True
    overlap_was, bucket.overlap = bucket.overlap, False        # no collectives inside the captured graph
    try:
        from uninext_b200.graphs import GraphedStep

        def captured():
            bucket.zero_()
            model(src, pos, shapes, ss, lsi, pad).float().square().mean().backward()
        graph = GraphedStep(captured, warmup=3, device=device)

        def graphed_step(_amp):
            graph.replay()
            bucket.all_reduce_mean()

        train_step_eager = train_step
        train_step = graphed_step          # noqa: F841  (measure() closes over the name below)
        res["tf32_cuda_graph"] = _measure_with(graphed_step, steps, barrier, lib, world, device, cfg)
    except Exception as exc:               # capture is an optimisation; report why it was not available
        res["tf32_cuda_graph"] = {"unavailable": repr(exc)[:200]}
    bucket.overlap = overlap_was
    torch.backends.cuda.matmul.allow_tf32 = old
    if rank == 0 and world == 1 and reference_stack:
        res["reference_stack"] = reference_stack_leg(cfg, device, steps, lib, (src, pos, shapes, ss, lsi, pad), res)
    res["grad_exchange"] = (f"overlapped: {bucket.n_slices} slices all-reduced from grad hooks during backward (eager legs); "
                            "one flat all-reduce after the replay (cuda-graph leg)") if world > 1 else "single GPU: none"
    return res


def reference_kernels_module(refcuda):
    """What the reference's pybind module is to ms_deform_attn_func.py:18, backed by the reference's own kernels
    (oracle/refcuda.py -> oracle/_ref/libmsda_refcuda.so)."""
    class _ReferenceKernels:
        @staticmethod
        def ms_deform_attn_forward(value, shapes, lsi, loc, attn, im2col_step):
            return refcuda.forward(value, shapes, lsi, loc, attn)

        @staticmethod
        def ms_deform_attn_backward(value, shapes, lsi, loc, attn, grad_output, im2col_step):
            return list(refcuda.backward(value, shapes, lsi, loc, attn, grad_output.contiguous()))
    return _ReferenceKernels


def build_reference_stack(cfg, tr_mod, num_layers=6, d_ffn=2048):
    """run_frames' model with the REFERENCE's layer classes (module `tr_mod` = the staged deformable_transformer.py) in
    place of this repo's: same embeddings, reference points, wiring and loss; weights from the same seed."""
    from uninext_b200.modules.deformable_layers import DeformableStack
    torch.manual_seed(1234)
    model = DeformableStack(num_layers=num_layers, num_queries=cfg.dec_queries, d_ffn=d_ffn)
    kw = dict(d_model=256, d_ffn=d_ffn, dropout=0.0, activation="relu", n_levels=len(cfg.shapes), n_heads=cfg.heads,
              n_points=cfg.points)
    model.encoder = torch.nn.ModuleList(tr_mod.DeformableTransformerEncoderLayer(**kw) for _ in range(num_layers))
    model.decoder = torch.nn.ModuleList(tr_mod.DeformableTransformerDecoderLayer(**kw) for _ in range(num_layers))
    return model


def reference_stack_leg(cfg, device, steps, lib, inputs, ours):
    """The anchor for frames/s: the SAME step (6 + 6 layers fwd + bwd, same synthetic features, same loss) run by the
    REFERENCE's GPU stack -- its own Python classes (``DeformableTransformerEncoderLayer`` / ``DecoderLayer`` /
    ``MSDeformAttn`` / ``MSDeformAttnFunction`` of deformable_transformer.py and ops/, unmodified files staged in oracle/_ref/py)
    on its own CUDA kernels (ms_deform_im2col_cuda.cuh compiled unmodified into oracle/_ref/libmsda_refcuda.so).  None of
    this repo's kernels is on that path (checked with the library's launch counter).  Baseline leg only, outside every
    timed region of this repo's numbers, like `reference_cuda`."""
    try:
        from oracle import refcuda, refstage
        if not refstage.staged():
            return {"unavailable": "oracle/_ref/py not staged (needs a reference checkout at build time)"}
        if not refcuda.available():
            return {"unavailable": "oracle/_ref/libmsda_refcuda.so not built (needs /root/reference at build time)"}
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            func_mod, _attn_mod, tr_mod, _dino_mod = refstage.import_reference()

        src, pos, shapes, ss, lsi, pad = inputs
        model = build_reference_stack(cfg, tr_mod).to(device)
        was = func_mod.MSDA
        func_mod.MSDA = reference_kernels_module(refcuda)
        try:
            def step():
                model.zero_grad(set_to_none=True)
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    model(src, pos, shapes, ss, lsi, pad).float().square().mean().backward()

            def measure():
                for _ in range(3):
                    step()
                torch.cuda.synchronize()
                l0 = lib.msda_launch_count()
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                for _ in range(steps):
                    step()
                t1.record()
                torch.cuda.synchronize()
                ms = t0.elapsed_time(t1) / steps
                return {"frames_per_s": round(cfg.batch / (ms * 1e-3), 2), "ms_per_step": round(ms, 3),
                        "msda_b200_launches_per_step": int((lib.msda_launch_count() - l0) / steps)}

            res = {"what": "the reference's own layer classes (deformable_transformer.py:321-416, ops/modules, ops/functions; "
                           "unmodified files, oracle/_ref/py) on the reference's own CUDA kernels (oracle/_ref), eager PyTorch as "
                           "the reference runs them; same step, features and loss as the legs above; single GPU"}
            old = torch.backends.cuda.matmul.allow_tf32
            try:
                torch.backends.cuda.matmul.allow_tf32 = False
                res["fp32"] = measure()
                torch.backends.cuda.matmul.allow_tf32 = True
                res["tf32"] = measure()
            finally:
                torch.backends.cuda.matmul.allow_tf32 = old
        finally:
            func_mod.MSDA = was
        ratio = lambda a, b: round(a / b, 2) if a and b else None
        res["speedup"] = {
            "fp32": ratio(ours.get("fp32", {}).get("frames_per_s"), res["fp32"]["frames_per_s"]),
            "tf32": ratio(ours.get("tf32", {}).get("frames_per_s"), res["tf32"]["frames_per_s"]),
            "tf32_cuda_graph_vs_reference_tf32": ratio(ours.get("tf32_cuda_graph", {}).get("frames_per_s"),
                                                       res["tf32"]["frames_per_s"])}
        del model
        torch.cuda.empty_cache()
        return res
    except Exception as exc:                        # a baseline leg must never take the bench line down
        return {"unavailable": repr(exc)[:300]}



def _measure_with(step_fn, steps, barrier, lib, world, device, cfg):
    for _ in range(3):
        step_fn(False)
    barrier()
    l0 = lib.msda_launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        step_fn(False)
    t1.record()
    barrier()
    ms = t0.elapsed_time(t1)
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms /= steps
    return {"frames_per_s": round(world * cfg.batch / (ms * 1e-3), 2), "ms_per_step": round(ms, 3),
            "msda_launches_per_step_host": int((lib.msda_launch_count() - l0) / steps)}


def bind_to_gpu_numa_node(device):
    """Pin this rank's host threads to the NUMA node its GPU hangs off, so that the pinned e2e buffers it allocates next
    are first-touched on that node: with 8 ranks, buffers on the far socket share one inter-socket link and the PCIe copies
    of every rank slow down together (round 1: 33 % of linear at 8 GPUs).  Best effort; returns what was done."""
    try:
        pr = torch.cuda.get_device_properties(device)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as fh:
            node = int(fh.read().strip())
        if node < 0:
            return {"numa_node": None, "note": "no NUMA information for the GPU"}
        with open(f"/sys/devices/system/node/node{node}/cpulist") as fh:
            cpus = set()
            for part in fh.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except (OSError, ValueError, AttributeError) as exc:
        return {"numa_node": None, "note": repr(exc)[:120]}


def setup_e2e(MSDA, calls, op_args, world, smp_step, steps, device, barrier):
    """Same step, but inputs start in pinned host memory and results end there.  Returns (measure, result):
    measure() times `steps` steps (barrier + synchronize on both sides, max over ranks) and returns ms per step;
    result(reps) builds the JSON object from the repetitions' times (median)."""
    numa = bind_to_gpu_numa_node(device)
    host_in, host_out, dev_in = [], [], []
    h2d = d2h = 0
    for c in calls:
        hin = {k: c[k].cpu().pin_memory() for k in ("value", "sampling_locations", "attention_weights", "grad_output")}
        host_in.append(hin)
        dev_in.append({k: torch.empty_like(c[k]) for k in hin})
        h2d += sum(t.numel() * t.element_size() for t in hin.values())
        n, lq = c["sampling_locations"].shape[:2]
        res = {"out": torch.empty((n, lq, c["value"].shape[2] * c["value"].shape[3]), dtype=c["value"].dtype).pin_memory(),
               "grad_value": torch.empty(c["value"].shape, dtype=c["value"].dtype).pin_memory(),
               "grad_loc": torch.empty(c["sampling_locations"].shape, dtype=c["sampling_locations"].dtype).pin_memory(),
               "grad_attn": torch.empty(c["attention_weights"].shape, dtype=c["attention_weights"].dtype).pin_memory()}
        host_out.append(res)
        d2h += sum(t.numel() * t.element_size() for t in res.values())

    # Three streams: H2D of call i+1 and D2H of call i-1 overlap the kernels of call i (PCIe is full duplex).
    s_in, s_out = torch.cuda.Stream(device=device), torch.cuda.Stream(device=device)
    cur = torch.cuda.current_stream()
    consumed = [None] * len(calls)            # compute-done event per input set: its buffers may be overwritten after it

    def e2e_step():
        for i, (c, hin, din, res) in enumerate(zip(calls, host_in, dev_in, host_out)):
            with torch.cuda.stream(s_in):
                if consumed[i] is not None:
                    s_in.wait_event(consumed[i])
                for k in hin:
                    din[k].copy_(hin[k], non_blocking=True)
                ev_in = torch.cuda.Event()
                ev_in.record(s_in)
            cur.wait_event(ev_in)
            a = (din["value"], c["spatial_shapes"], c["level_start_index"], din["sampling_locations"],
                 din["attention_weights"])
            out = MSDA.ms_deform_attn_forward(*a, 64)
            gv, gl, ga = MSDA.ms_deform_attn_backward(*a, din["grad_output"], 64)
            ev_c = torch.cuda.Event()
            ev_c.record(cur)
            consumed[i] = ev_c
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_c)
                res["out"].copy_(out, non_blocking=True)
                res["grad_value"].copy_(gv, non_blocking=True)
                res["grad_loc"].copy_(gl, non_blocking=True)
                res["grad_attn"].copy_(ga, non_blocking=True)
            for t in (out, gv, gl, ga):
                t.record_stream(s_out)
        ev_out = torch.cuda.Event()
        ev_out.record(s_out)
        cur.wait_event(ev_out)                 # the step ends when its last result has landed in host memory

    def measure():
        e2e_step()                             # warm-up (first repetition: also faults the pinned pages in)
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(steps):
            e2e_step()
        t1.record()
        barrier()
        ms = t0.elapsed_time(t1)
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps

    def result(reps):
        ms = statistics.median(reps)
        return {"value": round(world * smp_step / (ms * 1e-3) / 1e9, 4), "unit": UNIT, "ms_per_step": round(ms, 3),
                "steps": steps, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "reps_ms_per_step": [round(x, 3) for x in reps],
                "policy": f"median of {len(reps)} repetitions of {steps} timed steps each, spread over the run (after the "
                          "device-resident timing, after the frames leg, after the baseline legs): the host side of a shared "
                          "box is bursty -- one run in eight measured a 3x slower PCIe leg on an otherwise normal box "
                          "(profiles/r02zy_zero_fill_ab.txt)",
                "api": "MultiScaleDeformableAttention.ms_deform_attn_forward/backward on pinned-host inputs; "
                       "H2D / kernels / D2H on three streams", "host_numa": numa}

    return measure, result


# ------------------------------------------------------------------------------------------------------------------
# CPU legs: the reference's CPU path (ms_deform_attn_core_pytorch, reference file or port; oracle/ is test infrastructure and
# is imported here ONLY as the measured baseline, never by the product path).
# ------------------------------------------------------------------------------------------------------------------
def cpu_path():
    """-> (fn, kind, description): the reference's own ``ms_deform_attn_core_pytorch`` loaded from the staged copy of the
    reference file (oracle/_ref, put there by build() in the build container; kind "reference"), else the torch port
    that tests/golden pins to it (kind "port")."""
    from oracle import refpy
    fn = refpy.core_pytorch()
    if fn is not None:
        return fn, "reference", ("the reference's own ms_deform_attn_core_pytorch (ops/functions/ms_deform_attn_func.py:43-63, "
                                 "unmodified file staged in oracle/_ref; grid_sample per level) fwd + autograd bwd")
    from oracle.msda_oracle import core_pytorch_port
    return core_pytorch_port, "port", ("torch port of the reference's ms_deform_attn_core_pytorch (no staged copy of the "
                                       "reference file on this box; the port is pinned to it by tests/golden) fwd + autograd bwd")


def step_config(cfg, world):
    """The `config` object of the JSON line -- identical for the product arm and the reference arm."""
    return {"workload": cfg.name, "levels": cfg.shapes, "S": cfg.S, "frames_per_gpu": cfg.batch,
            "heads": cfg.heads, "head_dim": cfg.head_dim, "points": cfg.points,
            "dec_queries": cfg.dec_queries, "calls_per_step": f"{N_ENC} enc + {N_DEC} dec, fwd+bwd",
            "samples_per_step_per_gpu": samples_per_step(cfg), "parallelism": f"dp{world} (frames sharded, no exchange)",
            "l2_policy": "12 distinct input sets per step (~1 GB) > 126 MB L2"}


def cpu_call(port, c):
    v = c["value"].clone().requires_grad_(True)
    lo = c["sampling_locations"].clone().requires_grad_(True)
    at = c["attention_weights"].clone().requires_grad_(True)
    out = port(v, c["spatial_shapes"], lo, at)
    out.backward(c["grad_output"])
    return out


def cpu_sample_calls(cfg, frames, enc_queries=None):
    """One encoder-shaped + one decoder-shaped call on `frames` frames (a 1/6 slice of a step at full batch).
    `enc_queries` keeps only the first q queries of the encoder-shaped call (bounded samples for slow hosts)."""
    import dataclasses
    sub = dataclasses.replace(cfg, batch=frames)
    enc = make_inputs(sub, "enc", "cpu", seed=1)
    smp_enc = sub.samples("enc")
    if enc_queries is not None and enc_queries < enc["sampling_locations"].shape[1]:
        q = int(enc_queries)
        smp_enc = smp_enc * q // enc["sampling_locations"].shape[1]
        for k in ("sampling_locations", "attention_weights", "grad_output"):
            enc[k] = enc[k][:, :q].contiguous()
    return [enc, make_inputs(sub, "dec", "cpu", seed=2)], smp_enc + sub.samples("dec")


def cpu_pick_threads(port, cfg):
    """The reference CPU path is a chain of ATen ops whose OpenMP scaling saturates early; on a 128-core host all
    threads are SLOWER than 16-32.  Time a small slice with a few thread counts and keep the fastest (a stronger
    baseline than 'all cores')."""
    cores = os.cpu_count() or 1
    calls, _ = cpu_sample_calls(cfg, 1, enc_queries=2048)
    best = (None, float("inf"))
    for t in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
        torch.set_num_threads(t)
        cpu_call(port, calls[0])
        t0 = time.perf_counter()
        cpu_call(port, calls[0])
        dt = time.perf_counter() - t0
        if dt < best[1]:
            best = (t, dt)
    torch.set_num_threads(best[0])
    return best[0], cores


def cpu_time_sample(port, cfg, budget_s, max_reps):
    """Times `reps` x (1 enc-shaped + 1 dec-shaped call, fwd + autograd bwd); shrinks the sample (frames, then encoder
    queries) until one repetition fits `budget_s / 3`."""
    frames, enc_q = cfg.batch, None
    calls, smp = cpu_sample_calls(cfg, frames, enc_q)
    t0 = time.perf_counter()
    for c in calls:
        cpu_call(port, c)                                  # warm-up + probe
    probe = time.perf_counter() - t0
    if probe > budget_s / 3 and frames > 1:
        frames = 1
        probe *= 1.0 / cfg.batch
    if probe > budget_s / 3:
        enc_q = max(256, int(cfg.S * (budget_s / 3) / probe))
    if frames != cfg.batch or enc_q is not None:
        calls, smp = cpu_sample_calls(cfg, frames, enc_q)
        t0 = time.perf_counter()
        for c in calls:
            cpu_call(port, c)
        probe = time.perf_counter() - t0
    reps = max(1, min(max_reps, int(budget_s / max(probe, 1e-3)) - 1))
    t0 = time.perf_counter()
    for _ in range(reps):
        for c in calls:
            cpu_call(port, c)
    dt = (time.perf_counter() - t0) / reps
    what = (f"1 encoder-shaped ({'all' if enc_q is None else enc_q} of {cfg.S} queries) + 1 decoder-shaped call on "
            f"{frames} frame(s), fwd + autograd bwd")
    return smp, dt, reps, what


def cpu_baseline(cfg, budget_s):
    fn, kind, desc = cpu_path()
    threads, cores = cpu_pick_threads(fn, cfg)
    smp, dt, reps, what = cpu_time_sample(fn, cfg, budget_s, 10)
    return {"value": round(smp / dt / 1e9, 5), "unit": UNIT, "cores": threads, "host_cores": cores, "kind": kind,
            "impl": desc + "; thread count = fastest of {all, 64, 32, 16, 8}",
            "sample": f"{reps} x ({what})", "seconds_per_sample": round(dt, 3)}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on this box's host cores, same metric.
    Each of the K steps is a bounded sample of the workload, sized so that W + K steps end within a few minutes."""
    world, rank, _ = dist_env()
    if rank != 0:
        return
    cpu_fn, kind, desc = cpu_path()
    cfg = CONFIGS[args.config]
    threads, cores = cpu_pick_threads(cpu_fn, cfg)
    total = max(1, args.steps + args.warmup)
    per_step_budget = min(12.0, 150.0 / total)
    frames, enc_q = cfg.batch, None
    calls, smp = cpu_sample_calls(cfg, frames, enc_q)
    t0 = time.perf_counter()
    for c in calls:
        cpu_call(cpu_fn, c)
    probe = time.perf_counter() - t0
    if probe > per_step_budget and frames > 1:
        frames, probe = 1, probe / cfg.batch
    if probe > per_step_budget:
        enc_q = max(256, int(cfg.S * per_step_budget / probe))
    if frames != cfg.batch or enc_q is not None:
        calls, smp = cpu_sample_calls(cfg, frames, enc_q)
    for _ in range(max(0, args.warmup - 1)):
        for c in calls:
            cpu_call(cpu_fn, c)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for c in calls:
            cpu_call(cpu_fn, c)
    dt = (time.perf_counter() - t0) / args.steps
    val = round(smp / dt / 1e9, 5)
    sample = (f"per step: 1 encoder-shaped ({'all' if enc_q is None else enc_q} of {cfg.S} queries) + 1 decoder-shaped "
              f"call on {frames} frame(s), fwd + autograd bwd")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(dt * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": step_config(cfg, max(1, args.gpus)),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "host_cores": cores, "kind": kind, "sample": sample,
                         "impl": desc + "; thread count = fastest of {all, 64, 32, 16, 8}"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}), flush=True)


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
