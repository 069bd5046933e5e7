"""CPU: the device-output entry points of the host step (phc_host_step_submit_device / phc_host_reset_submit_device)
refuse a NULL context or NULL arguments, PhcHostDeviceOut matches the header, and HostDeviceOutputs /
HostStepBuffers(host_obs=False) reject malformed tensors before the library is called (no device is touched)."""

import ctypes as C
import os
from types import SimpleNamespace

import pytest
import torch

from humanoid_b200 import HostDeviceOutputs, HostStepBuffers, _cabi

D1 = _cabi.SELF_OBS_DIM + _cabi.TASK_OBS_DIM


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_cabi.LIB_PATH):
        import __graft_entry__ as g

        g.build()
    return _cabi.load()


def test_null_context_and_arguments_are_refused(lib):
    args, rargs, dev = _cabi.PhcHostStepArgs(), _cabi.PhcHostResetArgs(), _cabi.PhcHostDeviceOut()
    for fn in (lib.phc_host_step_submit_device, lib.phc_host_reset_submit_device):
        assert fn(None, 0, C.byref(args), C.byref(rargs), C.byref(dev), 8) == -1
        assert fn(None, 0, None, None, None, 8) == -1
        assert fn(None, 0, C.byref(args), C.byref(rargs), None, 8) == -1
    assert lib.phc_host_reset_submit_device(None, 0, C.byref(args), None, C.byref(dev), 8) == -1


def test_device_out_layout():
    # obs, obs_norm, mean, var | eps, clip | flags + pad | moments | buckets + pad | stream
    assert C.sizeof(_cabi.PhcHostDeviceOut) == 4 * 8 + 2 * 4 + 8 + 8 + 8 + 8
    assert _cabi.PhcHostDeviceOut.stream.offset == 64 and _cabi.PhcHostDeviceOut.obs_moments.offset == 48
    assert _cabi.ABI_VERSION == 6


def _meta(*shape, dtype=torch.float32):
    return torch.empty(*shape, dtype=dtype, device="meta")


def _rn(D=D1, device="meta", clip=10.0):
    return SimpleNamespace(running_mean=torch.empty(1, D, device=device), running_var=torch.empty(1, D, device=device),
                           epsilon=1e-5, clip=clip)  # fmt: skip


def test_host_buffers_without_obs():
    b = HostStepBuffers.allocate(12, 1, pinned=False, host_obs=False)
    assert b.obs_buf is None
    assert b.validate(1, device_out=True) == 12
    assert b._args().obs_buf is None and b._args().state == b.state.data_ptr()
    with pytest.raises(_cabi.PhcError, match="obs_buf must be a CPU tensor"):
        b.validate(1)  # the default still needs the host rows
    b = HostStepBuffers.allocate(12, 1, pinned=False)
    with pytest.raises(_cabi.PhcError, match="obs_buf must be None"):
        b.validate(1, device_out=True)


def test_allocate_needs_the_normalizer_for_obs_norm():
    with pytest.raises(ValueError, match="normalizer"):
        HostDeviceOutputs.allocate(8, 1, device="meta", norm_dtype=torch.bfloat16)


def test_device_outputs_reject_tensors_off_the_gpu():
    # a tensor on the meta device stands in for one that is not on a CUDA device, as a CPU tensor is
    for obs in (torch.zeros(8, D1), _meta(8, D1)):
        with pytest.raises(_cabi.PhcError, match="obs must be a CUDA tensor"):
            HostDeviceOutputs(obs=obs).validate(8)
    with pytest.raises(_cabi.PhcError, match="obs must be a CUDA tensor"):
        HostDeviceOutputs(obs=None).validate(8)


def test_device_outputs_reject_malformed_tensors():
    """dtype, shape and contiguity are checked before the device: every case below fails on its own defect."""
    obs = _meta(8, D1)
    with pytest.raises(ValueError, match="obs has shape"):
        HostDeviceOutputs(obs=obs).validate(9)
    with pytest.raises(ValueError, match="obs has shape"):
        HostDeviceOutputs(obs=obs).validate(8, time_steps=2)
    with pytest.raises(_cabi.PhcError, match="obs must be torch.float32"):
        HostDeviceOutputs(obs=_meta(8, D1, dtype=torch.float64)).validate(8)
    with pytest.raises(_cabi.PhcError, match="obs must be contiguous"):
        HostDeviceOutputs(obs=_meta(8, 2 * D1)[:, ::2]).validate(8)
    with pytest.raises(_cabi.PhcError, match="normalizer"):
        HostDeviceOutputs(obs=obs, obs_norm=_meta(8, D1)).validate(8)
    with pytest.raises(_cabi.PhcError, match="obs_norm must be"):
        HostDeviceOutputs(obs=obs, obs_norm=_meta(8, D1, dtype=torch.float16), normalizer=_rn()).validate(8)
    with pytest.raises(ValueError, match="obs_norm has shape"):
        HostDeviceOutputs(obs=obs, obs_norm=_meta(8, D1 + 1), normalizer=_rn()).validate(8)
    with pytest.raises(_cabi.PhcError, match="obs_norm must be contiguous"):
        HostDeviceOutputs(obs=obs, obs_norm=_meta(D1, 8).t(), normalizer=_rn()).validate(8)
    bad = _rn()
    bad.running_var = _meta(1, D1 + 1)
    with pytest.raises(ValueError, match="running_var has shape"):
        HostDeviceOutputs(obs=obs, obs_norm=_meta(8, D1), normalizer=bad).validate(8)
    with pytest.raises(ValueError, match="clip"):
        HostDeviceOutputs(obs=obs, obs_norm=_meta(8, D1), normalizer=_rn(clip=0.0)).validate(8)
    with pytest.raises(_cabi.PhcError, match="obs_moments must be torch.float64"):
        HostDeviceOutputs(obs=obs, obs_moments=_meta(4, 2 * D1)).validate(8)
    for shape in ((4, D1), (2 * D1,), (4097, 2 * D1)):
        with pytest.raises(ValueError, match="obs_moments"):
            HostDeviceOutputs(obs=obs, obs_moments=_meta(*shape, dtype=torch.float64)).validate(8)
    # well-formed apart from the device: refused for that alone
    ok = HostDeviceOutputs(obs=obs, obs_norm=_meta(8, D1, dtype=torch.bfloat16), normalizer=_rn(),
                           obs_moments=_meta(32, 2 * D1, dtype=torch.float64))  # fmt: skip
    with pytest.raises(_cabi.PhcError, match="obs must be a CUDA tensor"):
        ok.validate(8)


def test_take_obs_moments_needs_moments():
    with pytest.raises(_cabi.PhcError, match="obs_moments"):
        HostDeviceOutputs(obs=_meta(8, D1)).take_obs_moments()
