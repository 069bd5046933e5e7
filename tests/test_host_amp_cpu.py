"""CPU: the AMP observations of the host step (phc_host_step_submit_amp / phc_host_reset_submit_amp): the NULL-context
codes, the PhcHostAmp layout, and the Python validation of HostAmpBuffers and of the AMP submits.  No GPU needed: every
call here fails before the library touches a device, and the buffers are built on the meta device where CUDA ones
would be."""

import ctypes as C

import pytest
import torch

from humanoid_b200 import HostAmpBuffers, HostResetBuffers, HostStep, HostStepBuffers, _cabi
from humanoid_b200.host_step import AMP_OBS_PER_STEP


def test_null_context_is_refused():
    lib = _cabi.load()
    args, rargs, dev = _cabi.PhcHostStepArgs(), _cabi.PhcHostResetArgs(), _cabi.PhcHostDeviceOut()
    env, ep, amp = _cabi.PhcHostEnvArgs(), _cabi.PhcHostEpisodeOut(), _cabi.PhcHostAmp()
    step, reset = lib.phc_host_step_submit_amp, lib.phc_host_reset_submit_amp
    assert step(None, 0, C.byref(args), C.byref(rargs), C.byref(dev), C.byref(env), C.byref(ep), C.byref(amp), 8) == -1
    assert step(None, 0, C.byref(args), None, None, None, None, C.byref(amp), 8) == -1
    assert step(None, 0, None, None, None, None, None, None, 8) == -1
    assert reset(None, 0, C.byref(args), C.byref(rargs), C.byref(dev), C.byref(env), C.byref(amp), 8) == -1
    assert reset(None, 0, C.byref(args), C.byref(rargs), None, None, None, 8) == -1


def test_host_amp_layout():
    # dof_pos, dof_vel, amp_obs, amp_obs_demo | num_steps, obs_per_step | key_body_ids[8] | num_key_bodies, num_sel |
    # dof_subset | flags + pad | stream
    A = _cabi.PhcHostAmp
    assert C.sizeof(A) == 104
    offs = tuple(getattr(A, f).offset for f in ("dof_pos", "dof_vel", "amp_obs", "amp_obs_demo", "num_steps",
                                                "obs_per_step", "key_body_ids", "num_key_bodies", "num_sel",
                                                "dof_subset", "flags", "stream"))  # fmt: skip
    assert offs == (0, 8, 16, 24, 32, 36, 40, 72, 76, 80, 88, 96)


def test_allocate_shapes(monkeypatch):
    a = HostAmpBuffers.allocate(10, device="meta")
    assert tuple(a.amp_obs.shape) == (10, 10, 196) and a.amp_obs.dtype == torch.float32 and AMP_OBS_PER_STEP == 196
    assert tuple(a.amp_obs_demo.shape) == (10, 10, 196)
    assert tuple(a.obs.shape) == tuple(a.demo.shape) == (10, 1960)
    assert a.n == 10 and a.num_steps == 10
    assert a.dof_subset.dtype == torch.int64 and tuple(a.dof_subset.shape) == (57,)
    b = HostAmpBuffers.allocate(7, num_steps=1, device="meta", demo=False)
    assert tuple(b.amp_obs.shape) == (7, 1, 196) and b.amp_obs_demo is None and b.demo is None
    # the args carry HumanoidPHC's key bodies (R_Ankle, L_Ankle, R_Wrist, L_Wrist) and flags
    monkeypatch.setattr(_cabi, "stream_ptr", lambda device: 0)  # meta tensors have no stream
    x = b._args(None)
    assert list(x.key_body_ids)[:4] == [7, 3, 22, 17] and x.num_key_bodies == 4 and x.num_sel == 57
    assert x.flags == _cabi.OBS_LOCAL_ROOT | _cabi.OBS_ROOT_HEIGHT | _cabi.OBS_UPRIGHT
    assert x.num_steps == 1 and x.obs_per_step == 196 and not x.dof_pos and not x.amp_obs_demo


def test_step_buffers_with_amp():
    b = HostStepBuffers.allocate(6, pinned=False, amp=True)
    assert tuple(b.dof_pos.shape) == tuple(b.dof_vel.shape) == (6, 69) and b.dof_force is None
    assert b.validate(amp=True) == 6
    assert b.validate() == 6  # AMP buffers also serve steps without AMP
    p = HostStepBuffers.allocate(6, pinned=False, power=True, amp=True)  # one dof_vel, shared with the power reward
    assert p.validate(power=True, amp=True) == 6
    plain = HostStepBuffers.allocate(6, pinned=False)
    with pytest.raises(_cabi.PhcError, match="AMP observations need"):
        plain.validate(amp=True)
    plain.dof_vel = torch.zeros(6, 69)
    with pytest.raises(_cabi.PhcError, match="need dof_pos"):
        plain.validate(amp=True)
    plain.dof_pos, plain.dof_vel = torch.zeros(6, 69), None
    with pytest.raises(_cabi.PhcError, match="need dof_vel"):
        plain.validate(amp=True)
    for name, bad, err in (("dof_pos", torch.zeros(6, 69, dtype=torch.float64), _cabi.PhcError),
                           ("dof_vel", torch.zeros(6, 68), ValueError),
                           ("dof_pos", torch.zeros(69, 6).t(), _cabi.PhcError)):  # fmt: skip
        c = HostStepBuffers.allocate(6, pinned=False, amp=True)
        setattr(c, name, bad)
        with pytest.raises(err):
            c.validate(amp=True)


class _FakeCuda:
    """Patches torch.Tensor so meta tensors pass the CUDA-device check: what follows it is dtype / shape / contiguity."""

    def __enter__(self):
        self.saved = torch.Tensor.device
        meta = torch.device("meta")

        def device(t):
            d = self.saved.__get__(t)
            return torch.device("cuda", 0) if d == meta else d

        torch.Tensor.device = property(device)
        return self

    def __exit__(self, *exc):
        torch.Tensor.device = self.saved


def test_validate_refuses_cpu_tensors():
    a = HostAmpBuffers(amp_obs=torch.zeros(6, 10, 196))
    with pytest.raises(_cabi.PhcError, match="CUDA tensor"):
        a.validate(6)
    with _FakeCuda():
        a = HostAmpBuffers.allocate(6, device="meta")
        a.amp_obs_demo = torch.zeros(6, 10, 196)
        with pytest.raises(_cabi.PhcError, match="CUDA tensor"):
            a.validate(6)


@pytest.mark.parametrize(
    "field, bad, err",
    [
        ("amp_obs", lambda n: torch.zeros(n, 17, 196, device="meta"), ValueError),  # S > 16
        ("amp_obs", lambda n: torch.zeros(n, 0, 196, device="meta"), ValueError),  # S < 1
        ("amp_obs", lambda n: torch.zeros(n, 10, 195, device="meta"), ValueError),  # P
        ("amp_obs", lambda n: torch.zeros(n, 1960, device="meta"), ValueError),  # not [n, S, P]
        ("amp_obs", lambda n: torch.zeros(n + 1, 10, 196, device="meta"), ValueError),  # n
        ("amp_obs", lambda n: torch.zeros(n, 10, 196, dtype=torch.float64, device="meta"), _cabi.PhcError),
        ("amp_obs", lambda n: torch.zeros(n, 196, 10, device="meta").transpose(1, 2), _cabi.PhcError),  # strided
        ("amp_obs_demo", lambda n: torch.zeros(n, 9, 196, device="meta"), ValueError),  # S of amp_obs
        ("amp_obs_demo", lambda n: torch.zeros(n, 10, 196, dtype=torch.bfloat16, device="meta"), _cabi.PhcError),
        ("dof_subset", lambda n: torch.zeros(69, dtype=torch.int64, device="meta"), ValueError),
        ("dof_subset", lambda n: torch.zeros(57, dtype=torch.int32, device="meta"), _cabi.PhcError),
    ],
)
def test_validate_refuses_bad_tensors(field, bad, err):
    n = 10
    with _FakeCuda():
        a = HostAmpBuffers.allocate(n, device="meta")
        a.validate(n)  # the allocated buffers pass
        for S in (1, 16):
            HostAmpBuffers.allocate(n, num_steps=S, device="meta").validate(n)
        setattr(a, field, bad(n))
        with pytest.raises(err):
            a.validate(n)


@pytest.mark.parametrize("state_init", ["default", "hybrid"])
def test_default_and_hybrid_refused_with_amp(state_init):
    """The reference raises NotImplementedError for StateInit.Default / Hybrid with AMP (humanoid_phc.py:795-797): so
    do the AMP submits, before any buffer is checked or the library called."""
    hs = HostStep.__new__(HostStep)  # no context: the refusal comes first
    hs._ctx = None
    b = HostStepBuffers.allocate(4, pinned=False, amp=True)
    r = HostResetBuffers.allocate(4, pinned=False, hybrid=True)
    a = HostAmpBuffers.allocate(4, device="meta")
    with pytest.raises(NotImplementedError):
        hs.submit(0, b, r, state_init=state_init, amp=a)
    with pytest.raises(NotImplementedError):
        hs.reset_submit(0, b, r, state_init=state_init, amp=a)
    with pytest.raises(NotImplementedError):
        hs.reset(b, r, state_init=state_init, amp=a)
