"""CPU: the asynchronous host step's entry points refuse a NULL context, PHC_ERR_BUSY has a message, and
HostStepBuffers rejects malformed tensors before the library is called (no device is touched)."""

import ctypes as C
import os

import pytest
import torch

from humanoid_b200 import HostStepBuffers, _cabi


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_cabi.LIB_PATH):
        import __graft_entry__ as g

        g.build()
    return _cabi.load()


def test_null_context_is_refused(lib):
    args = _cabi.PhcHostStepArgs()
    assert lib.phc_host_step_submit(None, 0, C.byref(args), 8) == -1
    assert lib.phc_host_step_submit(None, 0, None, 8) == -1
    assert lib.phc_host_step_wait(None, 0) == -1


def test_busy_code_has_a_message(lib):
    assert _cabi.PHC_ERR_BUSY == -8 and _cabi.HOST_SLOTS == 2
    msg = lib.phc_strerror(_cabi.PHC_ERR_BUSY)
    assert msg not in (b"ok", b"unknown error") and b"flight" in msg


def _bufs(n=12, T=1):
    return HostStepBuffers.allocate(n, T, pinned=False)


def test_buffers_allocate_with_the_header_shapes():
    b = _bufs(12, 2)
    assert b.validate(2) == 12
    assert tuple(b.state.shape) == (12, 24, 13) and tuple(b.obs_buf.shape) == (12, 358 + 2 * 576)
    assert b.progress_buf.dtype == torch.int16 and b.sampled_motion_ids.dtype == torch.int64
    assert b.reset_buf.dtype == torch.uint8 and tuple(b.reward_raw.shape) == (12, 4)
    args = b._args()
    assert args.state == b.state.data_ptr() and args.terminate_buf == b.terminate_buf.data_ptr()


def test_buffers_validation_rejects_bad_tensors():
    b = _bufs()
    with pytest.raises(ValueError):
        b.validate(2)  # obs rows of T = 1
    b.obs_buf = torch.zeros(12, 934, dtype=torch.float64)
    with pytest.raises(_cabi.PhcError, match="obs_buf"):
        b.validate()
    b = _bufs()
    b.rew_buf = torch.zeros(24)[::2]  # right shape and dtype, strided
    with pytest.raises(_cabi.PhcError, match="contiguous"):
        b.validate()
    b = _bufs()
    b.global_offset = torch.zeros(11, 3)  # n of another batch
    with pytest.raises(ValueError, match="global_offset"):
        b.validate()
    b = _bufs()
    b.reset_buf = torch.zeros(12, dtype=torch.bool)
    with pytest.raises(_cabi.PhcError, match="reset_buf"):
        b.validate()


def test_buffers_validation_rejects_a_cuda_tensor():
    b = _bufs()
    # a tensor on the meta device stands in for one on the GPU: neither lives in host memory
    b.state = torch.empty(12, 24, 13, device="meta")
    with pytest.raises(_cabi.PhcError, match="CPU tensor"):
        b.validate()
    if torch.cuda.is_available():
        b.state = torch.zeros(12, 24, 13, device="cuda")
        with pytest.raises(_cabi.PhcError, match="CPU tensor"):
            b.validate()
