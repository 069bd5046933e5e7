"""CPU: the env options of the host step (phc_host_step_submit_env / phc_host_reset_submit_env /
phc_host_step_set_initial_state): NULL-context codes, the PhcHostEnvArgs layout, and the Python validation of the new
buffers.  No GPU needed: every call here fails before the library touches a device."""

import ctypes as C

import pytest
import torch

from humanoid_b200 import HostResetBuffers, HostStep, HostStepBuffers, _cabi


@pytest.fixture(scope="module")
def lib():
    return _cabi.load()


def test_null_context_is_refused(lib):
    args, rargs, dev, env = _cabi.PhcHostStepArgs(), _cabi.PhcHostResetArgs(), _cabi.PhcHostDeviceOut(), _cabi.PhcHostEnvArgs()
    for fn in (lib.phc_host_step_submit_env, lib.phc_host_reset_submit_env):
        assert fn(None, 0, C.byref(args), C.byref(rargs), C.byref(dev), C.byref(env), 8) == -1
        assert fn(None, 0, C.byref(args), C.byref(rargs), None, None, 8) == -1
        assert fn(None, 0, None, None, None, None, 8) == -1
    x = (C.c_float * 151)()
    assert lib.phc_host_step_set_initial_state(None, 0, x, x, x, 1) == -1


def test_env_args_layout():
    # dof_force, dof_vel | coef + pad | mpjpe | default_mask
    assert C.sizeof(_cabi.PhcHostEnvArgs) == 5 * 8
    E = _cabi.PhcHostEnvArgs
    assert (E.dof_force.offset, E.dof_vel.offset, E.rew_power_coef.offset, E.mpjpe.offset, E.default_mask.offset) == (
        0, 8, 16, 24, 32)
    # the step args keep their 11 pointers
    assert C.sizeof(_cabi.PhcHostStepArgs) == 11 * 8


def test_allocate_adds_the_option_buffers():
    b = HostStepBuffers.allocate(6, pinned=False)
    assert b.dof_force is None and b.dof_vel is None and b.mpjpe is None and tuple(b.reward_raw.shape) == (6, 4)
    b = HostStepBuffers.allocate(6, pinned=False, power=True, mpjpe=True)
    assert tuple(b.reward_raw.shape) == (6, 5) and tuple(b.dof_force.shape) == (6, 69) and tuple(b.dof_vel.shape) == (6, 69)
    assert tuple(b.mpjpe.shape) == (6,) and b.mpjpe.dtype == torch.float32
    assert b.validate(power=True) == 6
    a = b._args()  # exactly the 11 PhcHostStepArgs pointers, in order
    assert a.reward_raw == b.reward_raw.data_ptr() and a.terminate_buf == b.terminate_buf.data_ptr()
    r = HostResetBuffers.allocate(6, pinned=False, hybrid=True)
    assert r.default_mask.dtype == torch.uint8 and tuple(r.default_mask.shape) == (6,)
    assert HostResetBuffers.allocate(6, pinned=False).default_mask is None


def test_validation_of_the_power_buffers():
    b = HostStepBuffers.allocate(6, pinned=False, power=True)
    with pytest.raises(_cabi.PhcError, match="no power reward"):
        b.validate(power=False)
    b4 = HostStepBuffers.allocate(6, pinned=False)
    with pytest.raises(ValueError, match="reward_raw"):
        b4.validate(power=True)  # width 4 with the power reward
    b4.reward_raw = torch.zeros(6, 5)
    with pytest.raises(_cabi.PhcError, match="needs dof_force"):
        b4.validate(power=True)
    for name, bad, err in (("dof_force", torch.zeros(6, 69, dtype=torch.float64), _cabi.PhcError),
                           ("dof_vel", torch.zeros(6, 68), ValueError),
                           ("dof_force", torch.zeros(69, 6).t(), _cabi.PhcError),
                           ("dof_vel", torch.empty(6, 69, device="meta"), _cabi.PhcError)):  # fmt: skip
        b = HostStepBuffers.allocate(6, pinned=False, power=True)
        setattr(b, name, bad)
        with pytest.raises(err):
            b.validate(power=True)
    for bad, err in ((torch.zeros(6, dtype=torch.float64), _cabi.PhcError), (torch.zeros(5), ValueError),
                     (torch.empty(6, device="meta"), _cabi.PhcError)):  # fmt: skip
        b = HostStepBuffers.allocate(6, pinned=False, mpjpe=True)
        b.mpjpe = bad
        with pytest.raises(err):
            b.validate()


def test_validation_of_the_default_mask():
    r = HostResetBuffers.allocate(6, pinned=False, hybrid=True)
    r.default_mask = torch.ones(6, dtype=torch.bool)
    assert r.validate() == 6
    for bad, err in ((torch.zeros(6), _cabi.PhcError), (torch.zeros(7, dtype=torch.uint8), ValueError),
                     (torch.zeros(6, dtype=torch.uint8, device="meta"), _cabi.PhcError)):  # fmt: skip
        r.default_mask = bad
        with pytest.raises(err):
            r.validate()


def _closed_host_step():
    hs = HostStep.__new__(HostStep)  # no context: every argument check runs before the library is called
    hs._ctx, hs._capi, hs._initial_rows = None, _cabi.load(), [None] * _cabi.HOST_SLOTS
    hs._inflight = hs._inflight_reset = hs._inflight_dev = [None] * _cabi.HOST_SLOTS
    return hs


def test_set_initial_state_arguments():
    hs = _closed_host_step()
    root, dofp, dofv = torch.zeros(5, 13), torch.zeros(5, 69), torch.zeros(5, 69)
    for args, err in (((torch.zeros(5, 13, dtype=torch.float64), dofp, dofv), _cabi.PhcError),
                      ((root, torch.zeros(4, 69), dofv), ValueError),
                      ((root, dofp, torch.zeros(5, 70)), ValueError),
                      ((torch.zeros(5), dofp, dofv), ValueError),
                      ((root, torch.zeros(69, 5).t(), dofv), _cabi.PhcError),
                      ((root, dofp, torch.empty(5, 69, device="meta")), _cabi.PhcError)):  # fmt: skip
        with pytest.raises(err):
            hs.set_initial_state(0, *args)
    with pytest.raises(_cabi.PhcError, match="closed"):
        hs.set_initial_state(0, root, dofp, dofv)  # valid arguments reach the (closed) context


def test_default_init_needs_the_initial_state_and_hybrid_its_mask():
    hs = _closed_host_step()
    hs.use_power_reward, hs.rew_power_coef = False, 0.0005
    b = HostStepBuffers.allocate(6, pinned=False)
    r = HostResetBuffers.allocate(6, pinned=False)
    assert hs._env_args(0, b, r, "random", 6) is None  # no option: the submits without options run
    with pytest.raises(_cabi.PhcError, match="not supported"):
        hs._env_args(1, b, r, "default", 6)
    hs._initial_rows[1] = 6
    assert hs._env_args(1, b, r, "default", 6).default_mask is None
    with pytest.raises(ValueError, match="default_mask"):
        hs._env_args(1, b, r, "hybrid", 6)
    r.default_mask = torch.zeros(6, dtype=torch.bool)
    assert hs._env_args(1, b, r, "hybrid", 6).default_mask == r.default_mask.data_ptr()
