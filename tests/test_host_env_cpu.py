"""CPU: the reset entry points of the host step (phc_host_step_submit_reset / phc_host_reset_submit) refuse a NULL
context or NULL arguments, and HostResetBuffers rejects malformed tensors before the library is called (no device is
touched)."""

import ctypes as C
import os

import pytest
import torch

from humanoid_b200 import HostResetBuffers, HostStepBuffers, _cabi


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_cabi.LIB_PATH):
        import __graft_entry__ as g

        g.build()
    return _cabi.load()


def test_null_context_and_arguments_are_refused(lib):
    args, rargs = _cabi.PhcHostStepArgs(), _cabi.PhcHostResetArgs()
    for fn in (lib.phc_host_step_submit_reset, lib.phc_host_reset_submit):
        assert fn(None, 0, C.byref(args), C.byref(rargs), 8) == -1
        assert fn(None, 0, None, None, 8) == -1
        assert fn(None, 0, C.byref(args), None, 8) == -1


def test_reset_args_layout():
    assert C.sizeof(_cabi.PhcHostResetArgs) == 2 * 8 + 2 * 4 + 7 * 8
    assert _cabi.ABI_VERSION == 6


def _bufs(n=12):
    return HostResetBuffers.allocate(n, pinned=False)


def test_buffers_allocate_with_the_header_shapes():
    r = _bufs(12)
    assert r.validate() == 12 and r.validate(12) == 12
    assert tuple(r.root_states.shape) == (12, 13) and tuple(r.dof_pos.shape) == (12, 69)
    assert tuple(r.dof_vel.shape) == (12, 69) and r.phase.dtype == torch.float32
    assert r.env_mask.dtype == torch.uint8 and tuple(r.env_mask.shape) == (12,)
    b = HostStepBuffers.allocate(12, 1, pinned=False)
    a = r._args(b, "start", True)
    assert a.state_init == _cabi.STATE_INIT_START and a.flag_test == 1
    assert a.state_out == b.state.data_ptr() and a.global_offset_out == b.global_offset.data_ptr()
    assert a.motion_start_times_out == b.motion_start_times.data_ptr() and a.root_states == r.root_states.data_ptr()
    assert a.phase == r.phase.data_ptr() and a.env_mask == r.env_mask.data_ptr()
    r.env_mask = None
    assert r.validate() == 12 and r._args(b, "random", False).env_mask is None
    with pytest.raises(ValueError, match="state_init"):
        r._args(b, "sometimes", False)


def test_buffers_validation_rejects_bad_tensors():
    r = _bufs()
    with pytest.raises(ValueError, match="phase"):
        r.validate(13)  # rows of another batch
    r.phase = torch.zeros(12, dtype=torch.float64)
    with pytest.raises(_cabi.PhcError, match="phase"):
        r.validate()
    r = _bufs()
    r.dof_pos = torch.zeros(12, 138)[:, ::2]  # right shape and dtype, strided
    with pytest.raises(_cabi.PhcError, match="contiguous"):
        r.validate()
    r = _bufs()
    r.root_states = torch.zeros(12, 7)
    with pytest.raises(ValueError, match="root_states"):
        r.validate()
    r = _bufs()
    r.env_mask = torch.zeros(12, dtype=torch.int32)
    with pytest.raises(_cabi.PhcError, match="env_mask"):
        r.validate()
    r.env_mask = torch.zeros(12, dtype=torch.bool)
    assert r.validate() == 12


def test_buffers_validation_rejects_a_non_cpu_tensor():
    r = _bufs()
    # a tensor on the meta device stands in for one on the GPU: neither lives in host memory
    r.dof_vel = torch.empty(12, 69, device="meta")
    with pytest.raises(_cabi.PhcError, match="CPU tensor"):
        r.validate()
    if torch.cuda.is_available():
        r.dof_vel = torch.zeros(12, 69, device="cuda")
        with pytest.raises(_cabi.PhcError, match="CPU tensor"):
            r.validate()
