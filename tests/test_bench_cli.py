"""Tests of bench.py's command-line contract: the --impl reference arm prints one JSON line with the contract's keys, and
the product arm refuses to run without CUDA instead of falling back (CPU); on a GPU, --dump-outputs writes what the last
timed step returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, env=e,
                          timeout=600)


def test_reference_arm_prints_contract_line():
    p = _run("--impl", "reference", "--config", "cfg1", "--steps", "2", "--warmup", "1")
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "msdeformattn_fwd_bwd_gsamples_per_s"
    for key in ("value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["steps"] == 2 and line["value"] > 0 and line["e2e"]["h2d_bytes_per_step"] == 0
    cb = line["cpu_baseline"]
    sys.path.insert(0, ROOT)
    from oracle import refpy
    assert cb["kind"] == ("reference" if refpy.available() else "port")
    assert cb["value"] == line["value"] and cb["cores"] >= 1 and "sample" in cb
    assert line["config"]["workload"].startswith("cfg1")
    # same `config` object as the product arm prints (the driver compares the two lines)
    import bench
    from uninext_b200.workloads import CONFIGS
    assert line["config"] == json.loads(json.dumps(bench.step_config(CONFIGS["cfg1"], 1)))


def test_reference_file_and_port_agree():
    """The reference's own ms_deform_attn_core_pytorch and the port bench.py falls back to are the same function:
    the port's outputs and autograd gradients on a seeded case match the reference function's, stored under
    tests/golden/reference; so does the staged reference file itself where build() staged it."""
    sys.path.insert(0, ROOT)
    from oracle import refpy
    from oracle.msda_oracle import core_pytorch_port
    from tests import reference_cases as rc
    from uninext_b200.workloads import CONFIGS, make_inputs
    want = rc.load("core_pytorch_cfg1_dec")
    c = make_inputs(CONFIGS["cfg1"], "dec", "cpu", seed=5, wild_fraction=0.1)
    fns = [core_pytorch_port] + ([refpy.core_pytorch()] if refpy.available() else [])
    for fn in fns:
        v = c["value"].clone().requires_grad_(True)
        lo = c["sampling_locations"].clone().requires_grad_(True)
        at = c["attention_weights"].clone().requires_grad_(True)
        out = fn(v, c["spatial_shapes"], lo, at)
        out.backward(c["grad_output"])
        for key, t in (("out", out), ("grad_value", v.grad), ("grad_loc", lo.grad), ("grad_attn", at.grad)):
            assert tuple(t.shape) == tuple(want[key + ".shape"]), key
            got = t.detach().reshape(-1)[torch.from_numpy(rc.pick(t.numel(), want[key].size))]
            torch.testing.assert_close(got, torch.from_numpy(want[key]), rtol=1e-5, atol=1e-6)
    assert "MultiScaleDeformableAttention" not in sys.modules or \
        getattr(sys.modules["MultiScaleDeformableAttention"], "__file__", None) is not None   # the stand-in is gone


def test_reference_arm_non_zero_ranks_exit_quietly():
    p = _run("--impl", "reference", "--config", "cfg1", "--steps", "1", "--warmup", "1", "--gpus", "2",
             env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert p.returncode == 0 and p.stdout.strip() == ""


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU refusal")
def test_product_arm_refuses_without_cuda():
    p = _run("--steps", "1", "--warmup", "1")
    assert p.returncode != 0 and "no CPU fallback" in (p.stderr + p.stdout)


def test_algorithmic_bytes_formula():
    sys.path.insert(0, ROOT)
    from uninext_b200.workloads import CONFIGS, algorithmic_bytes
    c = CONFIGS["cfg2"]
    n, s, m, d, lq = c.batch, c.S, c.heads, c.head_dim, c.S
    taps = c.samples("enc")
    fwd = n * s * m * d * 4 + taps * 8 + taps * 4 + n * lq * m * d * 4
    assert algorithmic_bytes(c, "enc", 4, "fwd") == fwd == 28 * taps
    assert algorithmic_bytes(c, "enc", 4, "bwd") == fwd + 2 * n * s * m * d * 4 + taps * 12 == 56 * taps
    assert algorithmic_bytes(c, "enc", 4, "fwd+bwd") == 84 * taps
    assert algorithmic_bytes(c, "enc", 2, "fwd") == 20 * taps             # bf16 value / out, fp32 loc / attn


@pytest.mark.gpu
def test_dump_outputs_are_what_the_timed_step_returned(tmp_path):
    p = _run("--config", "cfg1", "--steps", "2", "--warmup", "1", "--no-e2e", "--no-cpu-baseline", "--no-frames",
             "--no-reference-cuda", "--no-configs", "--dump-outputs", str(tmp_path))
    assert p.returncode == 0, p.stderr[-2000:]
    assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == 2
    names = {f"{k}{i}_{a}.npy" for k in ("enc", "dec") for i in range(6) for a in ("out", "grad_value", "grad_loc", "grad_attn")}
    assert set(os.listdir(tmp_path)) == names
    arrays = {n: np.load(tmp_path / n) for n in names}
    assert all(a.dtype == np.float32 and a.ndim == 1 for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    # cfg1 decoder-shaped results are small enough to be stored whole: recompute the first call's on its seeded inputs
    sys.path.insert(0, ROOT)
    from uninext_b200.dropin import MultiScaleDeformableAttention as MSDA
    from uninext_b200.workloads import CONFIGS, make_inputs
    c = make_inputs(CONFIGS["cfg1"], "dec", "cuda", seed=100)
    a = (c["value"], c["spatial_shapes"], c["level_start_index"], c["sampling_locations"], c["attention_weights"])
    out = MSDA.ms_deform_attn_forward(*a, 64)
    gv, gl, ga = MSDA.ms_deform_attn_backward(*a, c["grad_output"], 64)
    for name, t in (("out", out), ("grad_loc", gl), ("grad_attn", ga)):
        want = t.reshape(-1).cpu().numpy()
        np.testing.assert_allclose(arrays[f"dec0_{name}.npy"], want, rtol=1e-5, atol=1e-6 * np.abs(want).max())
    assert arrays["dec0_grad_value.npy"].size == 1 << 18 < gv.numel()
