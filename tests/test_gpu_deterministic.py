"""Under torch.use_deterministic_algorithms(True) the op's backward is bit-reproducible: grad_value is accumulated as 64-bit
fixed point (msda_backward_det_*), so it is identical across calls, processes and kernel selections, and still matches
the fp64 truth and the default path within the parity tolerances.  The caller reductions (bias column sums, LayerNorm
backward, CondInst backward) switch to fixed-order kernels, so a whole DeformableStack step repeats bit for bit.  fp64
raises (warns under warn_only), like a torch op without a deterministic implementation."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.conftest import golden_names, load_golden

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

if torch.cuda.is_available():
    from oracle import msda_oracle
    from uninext_b200.dropin import MultiScaleDeformableAttention as MSDA
    from uninext_b200.workloads import CONFIGS, make_inputs


@pytest.fixture
def det():
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(was, warn_only=warn)


def _args(inp):
    return (inp["value"], inp["spatial_shapes"], inp["level_start_index"], inp["sampling_locations"], inp["attention_weights"])


def _ragged(dt, D=32, seed=5):
    """Odd head count, P = 3, pairs not a multiple of a warp's groups, out-of-range taps (as test_gpu_switches.py)."""
    g = torch.Generator().manual_seed(seed)
    ss = torch.tensor([[5, 6], [3, 3]]); lsi = torch.tensor([0, 30])
    v = torch.randn(3, 39, 5, D, generator=g).to("cuda", dt)
    loc = (torch.rand(3, 13, 5, 2, 3, 2, generator=g) * 1.6 - 0.3).cuda()
    at = torch.rand(3, 13, 5, 2, 3, generator=g).cuda()
    go = torch.randn(3, 13, 5 * D, generator=g).to("cuda", dt)
    return dict(value=v, spatial_shapes=ss.cuda(), level_start_index=lsi.cuda(), sampling_locations=loc,
                attention_weights=at, grad_output=go)


def _misaligned(inp):
    """The same data as a contiguous view with a 4-byte storage offset: routed to the generic kernel."""
    v = inp["value"]
    buf = torch.empty(v.numel() + 1, dtype=v.dtype, device=v.device)
    view = buf[1:].view(v.shape)
    view.copy_(v)
    return dict(inp, value=view)


def _cases():
    out = []
    for cfg in ("cfg1", "cfg2"):
        for kind in ("enc", "dec"):
            for dt in (torch.float32, torch.bfloat16):
                out.append((f"{cfg}_{kind}_{dt}", lambda c=cfg, k=kind, d=dt: make_inputs(CONFIGS[c], k, "cuda", dtype=d, seed=3,
                                                                                          wild_fraction=0.1)))
    for dt in (torch.float32, torch.bfloat16):
        out.append((f"ragged_{dt}", lambda d=dt: _ragged(d)))
        for D in (30, 71):
            out.append((f"ragged_D{D}_{dt}", lambda d=dt, D=D: _ragged(d, D)))
        out.append((f"misaligned_{dt}", lambda d=dt: _misaligned(_ragged(d))))
    return out


def _bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


@pytest.mark.parametrize("name,make", _cases(), ids=[c[0] for c in _cases()])
def test_repeatable_across_calls(det, name, make):
    inp = make()
    a = _args(inp)
    ref = None
    for rep in range(4):
        junk = torch.full((inp["value"].numel() * 2 + 64,), 7.0, device="cuda")     # dirty the allocator's blocks
        del junk
        out = MSDA.ms_deform_attn_forward(*a, 64)
        got = [out] + list(MSDA.ms_deform_attn_backward(*a, inp["grad_output"], 64))
        if ref is None:
            ref = [t.clone() for t in got]
        else:
            for i, (t0, t1) in enumerate(zip(ref, got)):
                assert torch.equal(_bits(t0), _bits(t1)), (name, rep, i)


SCRIPT = r"""
import sys, torch
sys.path.insert(0, %r)
from uninext_b200.dropin import MultiScaleDeformableAttention as MSDA
from uninext_b200.workloads import CONFIGS, make_inputs
torch.use_deterministic_algorithms(True)
res = {}
for cfg, kind in (("cfg1", "enc"), ("cfg1", "dec"), ("cfg2", "dec")):
    for dt in (torch.float32, torch.bfloat16):
        inp = make_inputs(CONFIGS[cfg], kind, "cuda", dtype=dt, seed=3, wild_fraction=0.1)
        a = (inp["value"], inp["spatial_shapes"], inp["level_start_index"], inp["sampling_locations"], inp["attention_weights"])
        gv, gl, ga = MSDA.ms_deform_attn_backward(*a, inp["grad_output"], 64)
        v = inp["value"]
        buf = torch.empty(v.numel() + 1, dtype=v.dtype, device="cuda")
        view = buf[1:].view(v.shape); view.copy_(v)                      # same data, generic kernel
        gv_generic = MSDA.ms_deform_attn_backward(view, *a[1:], inp["grad_output"], 64)[0]
        res[(cfg, kind, str(dt))] = (gv.cpu(), gv_generic.cpu(), gl.cpu(), ga.cpu())
torch.save(res, sys.argv[1])
"""


def _run(env, path):
    e = {k: v for k, v in os.environ.items() if not k.startswith("MSDA_")}
    e.update(env)
    subprocess.run([sys.executable, "-c", SCRIPT % ROOT, path], check=True, env=e, timeout=600)
    return torch.load(path)


@pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a GPU")
def test_grad_value_independent_of_kernel_selection_and_process(tmp_path):
    """grad_value is bit-identical across SPLIT on / off, LDG vs TMA taps, patch order, the slab / tensor-memory / VEC8 /
    fine-rows knobs (which the deterministic path does not take), tiled vs generic kernels and separate processes."""
    base = _run({}, str(tmp_path / "base.pt"))
    again = _run({}, str(tmp_path / "again.pt"))
    for key, (gv, gvg, gl, ga) in base.items():
        assert torch.equal(_bits(gv), _bits(gvg)), ("tiled vs generic", key)
        assert all(torch.equal(_bits(x), _bits(y)) for x, y in zip(base[key], again[key])), ("second process", key)
    cases = ({"MSDA_SPLIT": "1"}, {"MSDA_SPLIT": "0"}, {"MSDA_SPLIT": "0", "MSDA_NO_TMA": "1"},
             {"MSDA_SPLIT": "0", "MSDA_PATCHES": "1"},
             {"MSDA_SLAB": "1", "MSDA_F32_VEC8_BWD": "1", "MSDA_BF16_FINE_ROWS": "1"}, {"MSDA_SLAB": "2"})
    for i, env in enumerate(cases):
        other = _run(env, str(tmp_path / f"c{i}.pt"))
        for key in base:
            assert torch.equal(_bits(base[key][0]), _bits(other[key][0])), (env, key)


def _gl_ok(got, want, tol):
    """test_gpu_parity.py's rule: every entry within tol of scale except a <= 1e-4 fraction (at most a handful) of
    cell-boundary taps, whose fp32 coordinate rounds into the neighbouring cell."""
    err = np.abs(got.astype(np.float64) - want) / max(1e-30, float(np.abs(want).max()))
    return float((err > tol).sum()) <= max(2.0, 1e-4 * want.size)


def _maxerr(got, want):
    want = np.asarray(want, dtype=np.float64)
    return float(np.abs(got.detach().double().cpu().numpy() - want).max()) / max(1e-30, float(np.abs(want).max()))


@pytest.mark.parametrize("name", golden_names())
def test_golden_fp32_and_bf16(det, name):
    """The tolerances of test_gpu_parity.py's golden tests (bf16 on the same four cases)."""
    c = load_golden(name)
    t = lambda k, dt: torch.from_numpy(c[k]).to("cuda", dt).contiguous()
    for dt, tol in ((torch.float32, 1e-4), (torch.bfloat16, 1e-2)):
        if dt == torch.bfloat16 and name not in ("prod_small", "prod_small_wide", "prod_small_edges", "d64"):
            continue
        a = (t("value", dt), t("spatial_shapes", torch.int64), t("level_start_index", torch.int64),
             t("sampling_locations", torch.float32), t("attention_weights", torch.float32))
        gv, gl, ga = MSDA.ms_deform_attn_backward(*a, t("grad_output", dt), 64)
        assert _maxerr(gv, c["grad_value"]) < tol, (name, dt)
        assert _maxerr(ga, c["grad_attention_weights"]) < tol, (name, dt)
        assert _gl_ok(gl.cpu().numpy(), c["grad_sampling_locations"], 2 * tol), (name, dt)


@pytest.mark.parametrize("cfg,kind", [("cfg1", "enc"), ("cfg1", "dec"), ("cfg2", "dec")])
def test_matches_oracle_and_default_path(det, cfg, kind):
    for dt, tol in ((torch.float32, 2e-5), (torch.bfloat16, 1e-2)):
        inp = make_inputs(CONFIGS[cfg], kind, "cuda", dtype=dt, seed=7, wild_fraction=0.05)
        a = _args(inp)
        gv = MSDA.ms_deform_attn_backward(*a, inp["grad_output"], 64)[0]
        torch.use_deterministic_algorithms(False)
        gv_default = MSDA.ms_deform_attn_backward(*a, inp["grad_output"], 64)[0]
        torch.use_deterministic_algorithms(True)
        scale = gv_default.double().abs().max().item()
        assert (gv.double() - gv_default.double()).abs().max().item() <= tol * scale, (cfg, kind, dt)
        if cfg == "cfg1" and dt == torch.float32:
            f64 = lambda x: x.detach().double().cpu().numpy()
            want = msda_oracle.backward(f64(inp["grad_output"]), f64(inp["value"]), inp["spatial_shapes"].cpu().numpy(),
                                        inp["level_start_index"].cpu().numpy(), f64(inp["sampling_locations"]),
                                        f64(inp["attention_weights"]))[0]
            assert _maxerr(gv, want) < tol


def test_zero_inputs_give_zeros(det):
    inp = make_inputs(CONFIGS["cfg1"], "dec", "cuda", seed=1)
    a = list(_args(inp))
    gv = MSDA.ms_deform_attn_backward(*a, torch.zeros_like(inp["grad_output"]), 64)[0]
    assert torch.equal(gv, torch.zeros_like(gv))
    a[4] = torch.zeros_like(a[4])
    gv = MSDA.ms_deform_attn_backward(*a, inp["grad_output"], 64)[0]
    assert torch.equal(gv, torch.zeros_like(gv))
    lq0 = inp["sampling_locations"][:, :0].contiguous()
    gv, gl, ga = MSDA.ms_deform_attn_backward(a[0], a[1], a[2], lq0, inp["attention_weights"][:, :0].contiguous(),
                                              inp["grad_output"][:, :0].contiguous(), 64)
    assert torch.equal(gv, torch.zeros_like(gv)) and gl.numel() == 0 and ga.numel() == 0


@pytest.mark.parametrize("mag", [1e-30, 1e30])
def test_extreme_magnitudes_keep_relative_accuracy(det, mag):
    inp = make_inputs(CONFIGS["cfg1"], "enc", "cuda", seed=2, wild_fraction=0.05)
    a = _args(inp)
    want = MSDA.ms_deform_attn_backward(*a, inp["grad_output"], 64)[0].double()
    got = MSDA.ms_deform_attn_backward(*a, inp["grad_output"] * mag, 64)[0].double() / mag
    assert torch.isfinite(got).all()
    assert (got - want).abs().max().item() <= 2e-5 * want.abs().max().item()


def test_non_finite_grad_out_matches_default_pattern(det):
    inp = make_inputs(CONFIGS["cfg1"], "dec", "cuda", seed=4)
    a = _args(inp)
    go = inp["grad_output"].clone()
    go[0, 3, 5] = float("nan")
    go[0, 10, 40] = float("inf")
    go[0, 20, 40] = float("-inf")
    go[0, 30, 77] = float("inf")
    go[0, 31, 77] = float("-inf")
    got = [MSDA.ms_deform_attn_backward(*a, go, 64)[0] for _ in range(3)]
    torch.use_deterministic_algorithms(False)
    want = MSDA.ms_deform_attn_backward(*a, go, 64)[0]
    torch.use_deterministic_algorithms(True)
    for g in got:
        assert torch.equal(torch.isnan(g), torch.isnan(want))
        assert torch.equal(torch.isposinf(g), torch.isposinf(want)) and torch.equal(torch.isneginf(g), torch.isneginf(want))
        assert torch.equal(_bits(g), _bits(got[0]))
    assert torch.isnan(want).any() and torch.isposinf(want).any() and torch.isneginf(want).any()
    fin = torch.isfinite(want)
    scale = want[fin].abs().max().item()
    assert (got[0][fin] - want[fin]).abs().max().item() <= 2e-5 * scale


def test_cuda_graph_replays_eager_result(det):
    inp = make_inputs(CONFIGS["cfg1"], "enc", "cuda", seed=12)
    a = _args(inp)
    want = MSDA.ms_deform_attn_backward(*a, inp["grad_output"], 64)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        got = MSDA.ms_deform_attn_backward(*a, inp["grad_output"], 64)
    for _ in range(3):
        got[0].fill_(3.0)
        g.replay()
    torch.cuda.synchronize()
    for x, y in zip(got, want):
        assert torch.equal(x, y)


def test_fp64_raises_or_warns():
    inp = make_inputs(CONFIGS["cfg1"], "dec", "cuda", dtype=torch.float64, seed=6)
    a = _args(inp)
    want = MSDA.ms_deform_attn_backward(*a, inp["grad_output"], 64)
    try:
        torch.use_deterministic_algorithms(True)
        with pytest.raises(RuntimeError, match="does not have a deterministic implementation, but you set "
                                               "'torch.use_deterministic_algorithms\\(True\\)'"):
            MSDA.ms_deform_attn_backward(*a, inp["grad_output"], 64)
        torch.use_deterministic_algorithms(True, warn_only=True)
        with pytest.warns(UserWarning, match="does not have a deterministic implementation"):
            got = MSDA.ms_deform_attn_backward(*a, inp["grad_output"], 64)
    finally:
        torch.use_deterministic_algorithms(False)
    assert (got[0] - want[0]).abs().max().item() <= 1e-12 * want[0].abs().max().item()
    assert torch.equal(got[1], want[1]) and torch.equal(got[2], want[2])


def test_forward_is_deterministic_without_the_flag():
    inp = make_inputs(CONFIGS["cfg2"], "enc", "cuda", seed=8)
    outs = [MSDA.ms_deform_attn_forward(*_args(inp), 64) for _ in range(3)]
    assert all(torch.equal(o, outs[0]) for o in outs)


def test_caller_reductions_repeatable_and_accurate(det):
    """colsum, the ReLU-backward colsum, the LayerNorm backward and the CondInst backward: torch.equal across repeats
    (allocator dirtied in between) and within the existing tests' tolerances of fp64 / torch references.  warn_only: the
    library's deterministic kernels are taken all the same, while torch's GEMMs only warn about CUBLAS_WORKSPACE_CONFIG."""
    torch.use_deterministic_algorithms(True, warn_only=True)
    from uninext_b200.functions import fused
    from uninext_b200.modules.dynamic_mask_head import _DynamicMaskHead, _inst_start
    g = torch.Generator(device="cuda").manual_seed(3)
    x = torch.randn(44646, 256, device="cuda", generator=g)
    lin = torch.nn.Linear(256, 512).cuda()
    ln = torch.nn.LayerNorm(256).cuda()
    feats = torch.randn(2, 8, 100, 168, device="cuda", generator=g)
    params = torch.randn(600, 169, device="cuda", generator=g) * 0.3
    refs = torch.rand(600, 2, device="cuda", generator=g) * 600
    inst = _inst_start((300, 300), "cuda")
    gl = torch.randn(600, 100, 168, device="cuda", generator=g)

    def run():
        junk = torch.full((1 << 24,), 7.0, device="cuda")
        del junk
        res = [fused.colsum(x)]
        xr = x[:4096].clone().requires_grad_(True)
        y = fused.linear_colsum(xr, lin, relu=True)
        gb, = torch.autograd.grad(y, lin.bias, torch.ones_like(y) * x[:4096, :1])
        res.append(gb)
        a = x[:8192].clone().requires_grad_(True)
        out = fused.add_layer_norm(a, None, ln)
        res += list(torch.autograd.grad(out, (a, ln.weight, ln.bias), x[8192:16384]))
        fe, pa, rf = (t.clone().requires_grad_(True) for t in (feats, params, refs))
        lg = _DynamicMaskHead.apply(fe, pa, rf, inst, 300, 8, True)
        res += list(torch.autograd.grad(lg, (fe, pa, rf), gl))
        return res

    first = run()
    for _ in range(2):
        assert all(torch.equal(a, b) for a, b in zip(first, run()))
    tol = lambda got, want, t: (got.double() - want.double()).abs().max().item() <= t * want.double().abs().max().item()
    assert tol(first[0], x.double().sum(0), 1e-5)
    torch.use_deterministic_algorithms(False)
    default = run()
    for i, (a, b) in enumerate(zip(first, default)):
        assert tol(a, b, 1e-4), i


STACK = r"""
import os, sys, torch
sys.path.insert(0, %r)
torch.use_deterministic_algorithms(True)
from uninext_b200.modules.deformable_layers import DeformableStack
from uninext_b200.workloads import CONFIGS, level_tensors
res = {}
for name, cfg, layers in (("cfg1_2", "cfg1", 2), ("cfg2_6", "cfg2", 6)):
    c = CONFIGS[cfg]
    torch.manual_seed(1234)
    model = DeformableStack(num_layers=layers, num_queries=c.dec_queries).cuda()
    ss, lsi = level_tensors(c.shapes, "cuda")
    g = torch.Generator(device="cuda").manual_seed(77)
    src = torch.randn(c.batch, c.S, 256, device="cuda", generator=g)
    pos = torch.randn(c.batch, c.S, 256, device="cuda", generator=g)
    pad = torch.zeros(c.batch, c.S, dtype=torch.bool, device="cuda")
    model(src, pos, c.shapes, ss, lsi, pad).square().mean().backward()
    res[name] = {k: p.grad.cpu() for k, p in model.named_parameters()}
torch.save(res, sys.argv[1])
from tests import test_gpu_reference_dropin as ref                     # the reference cases through the drop-in, under the flag
for case in ("module_0", "module_1", "encoder_0", "encoder_1", "decoder_0", "decoder_1"):
    ref._compare(case)
"""


@pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a GPU")
def test_whole_stack_gradients_equal_across_processes(tmp_path):
    """DeformableStack (2 layers at cfg1, 6+6 at cfg2) fwd+bwd under the flag in two processes: every parameter gradient is
    torch.equal.  The same processes run the reference cases of tests/reference_cases.py against tests/golden/reference."""
    env = {k: v for k, v in os.environ.items() if not k.startswith("MSDA_")}
    env["CUBLAS_WORKSPACE_CONFIG"] = ":4096:8"                 # torch's own GEMMs under the flag
    runs = []
    for i in range(2):
        path = str(tmp_path / f"stack{i}.pt")
        subprocess.run([sys.executable, "-c", STACK % ROOT, path], check=True, env=env, cwd=ROOT, timeout=900)
        runs.append(torch.load(path))
    for name in runs[0]:
        for k, g in runs[0][name].items():
            assert torch.equal(g, runs[1][name][k]), (name, k)
