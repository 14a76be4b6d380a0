"""CPU tests of the deterministic mode's host side: how torch's flag is read, the PyTorch-worded alert, and the argument
checks of msda_backward_det_* (they return before anything touches the device)."""
import ctypes
import warnings

import pytest
import torch

from uninext_b200 import determinism


@pytest.fixture
def restore_flag():
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    yield
    torch.use_deterministic_algorithms(was, warn_only=warn)


def test_mode_follows_torch_flag(restore_flag):
    torch.use_deterministic_algorithms(False)
    assert determinism.mode() == determinism.OFF
    determinism.alert_not_deterministic("x")                      # off: silent
    torch.use_deterministic_algorithms(True)
    assert determinism.mode() == determinism.ON
    with pytest.raises(RuntimeError, match=r"x does not have a deterministic implementation, but you set "
                                           r"'torch.use_deterministic_algorithms\(True\)'"):
        determinism.alert_not_deterministic("x")
    torch.use_deterministic_algorithms(True, warn_only=True)
    assert determinism.mode() == determinism.WARN
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        determinism.alert_not_deterministic("x")
    assert any("does not have a deterministic implementation" in str(m.message) for m in w)


def test_det_entry_points_reject_bad_arguments():
    from uninext_b200 import _cabi, build
    build.build()
    lib = _cabi.load()
    p = 1 << 20                                                    # never dereferenced: the checks fail first
    dims = (1, 16, 2, 32, 1, 4, 2)
    for fn, extra in ((lib.msda_backward_det_f32, (p, p, p)), (lib.msda_backward_det_bf16, (p, p, p, p))):
        assert fn(p, p, p, p, p, p, *dims, None, *extra, None) == -1                 # no accumulator
        assert fn(p, p, p, p, p, p, *dims, p + 4, *extra, None) == -1                # accumulator not 8-byte aligned
        assert fn(p, p, p, p, p, p, 0, *dims[1:], p, *extra, None) == -1             # non-positive dimension
        assert fn(None, p, p, p, p, p, *dims, p, *extra, None) == -1                 # null input


def test_scratch_size_queries():
    """Host-only scratch sizes of the deterministic caller reductions for the cfg1-cfg5 shapes, MSDA_E_BADARG otherwise."""
    from uninext_b200 import _cabi, build
    from uninext_b200.workloads import CONFIGS
    build.build()
    lib = _cabi.load()
    parts = lambda rows, mult: -(-rows // (-(-max(16, -(-rows // 512)) // mult) * mult))
    for cfg in CONFIGS.values():
        for rows in (cfg.batch * cfg.S, cfg.batch * cfg.dec_queries):
            assert _cabi.scratch_bytes(lib.msda_colsum_det_scratch_bytes, rows, 256) == parts(rows, 1) * 256 * 4
            assert _cabi.scratch_bytes(lib.msda_colsum_det_scratch_bytes, rows, 2048) == parts(rows, 1) * 2048 * 4
            assert _cabi.scratch_bytes(lib.msda_layernorm_backward_det_scratch_bytes, rows, 256) == 2 * parts(rows, 8) * 256 * 4
            assert parts(rows, 1) <= 512
        h, w = cfg.shapes[0][0] * 2, cfg.shapes[0][1] * 2            # mask features at stride 4
        hw = h * w
        want = 4 * (-(-300 // 16) * cfg.batch * 8 * hw + -(-hw // 64) * 300 * cfg.batch * 171)
        assert _cabi.scratch_bytes(lib.msda_condinst_backward_det_scratch_bytes, cfg.batch, h, w, 300 * cfg.batch, 300) == want
    out = ctypes.c_int64(0)
    assert lib.msda_colsum_det_scratch_bytes(0, 256, ctypes.byref(out)) == -1
    assert lib.msda_colsum_det_scratch_bytes(100, 254, ctypes.byref(out)) == -1
    assert lib.msda_colsum_det_scratch_bytes(100, 256, None) == -1
    assert lib.msda_layernorm_backward_det_scratch_bytes(100, 200, ctypes.byref(out)) == -1
    assert lib.msda_condinst_backward_det_scratch_bytes(0, 10, 10, 1, 1, ctypes.byref(out)) == -1
    assert lib.msda_condinst_backward_det_scratch_bytes(1, 10, 10, -1, 1, ctypes.byref(out)) == -1
