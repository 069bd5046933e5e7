"""GPU: resets on the host-buffer path equal the device path bit for bit.

``HostStep.submit(slot, bufs, reset=...)`` (phc_host_step_submit_reset) against ``HumanoidPHC.step(phase_by_env=...)``
with ``enable_auto_reset()``, and ``HostStep.reset_submit`` (phc_host_reset_submit) against
``HumanoidPHC.reset(env_ids, phase)``, on the same inputs: obs, rewards, reward_raw[:, :4], the step's flags, progress,
the clock, and for the re-posed envs the rigid-body / root / dof rows; every other row of the reset outputs keeps what
it held.  Short clips and clocks near clip ends, so that every step flags envs by clip end and by termination and
spares others; a few envs are pushed away from their reference each step (the stand-in for physics) so that some
terminate in every step."""

import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from humanoid_b200 import HostResetBuffers, HostStep, HostStepBuffers, HumanoidPHC, MotionLib, _cabi, synth
    from util_gpu import DEV

OK, NULL, UNSUPPORTED, BUSY = 0, -1, -4, -8
SENTINEL = 12345.0


def _motion_lib(M=48, seed=601):
    data = synth.make_motion_lib(M, 60, 90, seed=seed, device=DEV)
    return data, MotionLib(data, device=DEV)


class EnvCase:
    """One batch on both paths: host buffers for the host step, a HumanoidPHC with auto-reset on the same inputs."""

    def __init__(self, data, mlib, n, seed, T=1, pinned=True, pinned_reset=None, ids="mod", aligned=True,
                 state_init="random", eval_mode=False, flag_test=False):  # fmt: skip
        clock = synth.make_clock(data, n, seed=seed, ids=ids, aligned=aligned, max_progress=30)
        ref = mlib.get_motion_state(clock.sampled_motion_ids, synth.reward_time(clock, extra_steps=1), clock.global_offset)
        state = synth.make_sim_state(ref, seed=seed + 1)
        env = HumanoidPHC(mlib, n, device=DEV, time_steps=T)
        env.set_sim_state(state)
        env.set_clock(clock)
        env.enable_auto_reset(True)
        env.state_init = state_init
        env.flag_test = flag_test
        if eval_mode:
            env.flag_im_eval = True
            env.set_termination_distances(0.1)
        self.env, self.n, self.T = env, n, T
        self.state_init, self.flag_test = state_init, flag_test
        b = HostStepBuffers.allocate(n, T, pinned=pinned)
        b.state.copy_(state.cpu())
        b.progress_buf.copy_(clock.progress_buf.cpu())
        b.motion_start_times.copy_(clock.motion_start_times.cpu())
        b.motion_start_times_offset.copy_(clock.motion_start_times_offset.cpu())
        b.global_offset.copy_(clock.global_offset.cpu())
        b.sampled_motion_ids.copy_(clock.sampled_motion_ids.cpu())
        self.bufs = b
        self.rb = HostResetBuffers.allocate(n, pinned=pinned if pinned_reset is None else pinned_reset)
        self.gen = torch.Generator().manual_seed(seed + 2)
        self.k = 0

    def host_kwargs(self):
        return dict(state_init=self.state_init, flag_test=self.flag_test)

    def poison(self):
        b, r = self.bufs, self.rb
        for t in (b.obs_buf, b.rew_buf, b.reward_raw):
            t.fill_(float("nan"))
        b.reset_buf.fill_(7)
        b.terminate_buf.fill_(7)
        for t in (r.root_states, r.dof_pos, r.dof_vel):
            t.fill_(SENTINEL)

    def physics(self):
        """The same push on both paths: every body of ~3 % of the envs moves 0.5 m (they terminate), the others a
        little.  fp32 adds of the same operands are exact on both sides."""
        n, k = self.n, self.k
        d = torch.randn(n, 24, 3, generator=self.gen) * 0.01
        far = (torch.arange(n) * 7 + k) % 29 == 0
        d[far, :, 0] += 0.5
        self.bufs.state[..., 0:3] += d
        self.env._rigid_body_state_reshaped[..., 0:3] += d.to(DEV)
        self.k += 1

    def begin(self):
        """Physics, a fresh phase, poisoned outputs; returns the copies the untouched rows are checked against."""
        self.physics()
        self.rb.phase.copy_(torch.rand(self.n, generator=self.gen))
        self.poison()
        b = self.bufs
        return dict(state=b.state.clone(), start=b.motion_start_times.clone(), soff=b.motion_start_times_offset.clone(),
                    goff=b.global_offset.clone())  # fmt: skip

    def advance(self):
        """One auto-reset step of the device path; returns its outputs on the host."""
        e = self.env
        e.step(phase_by_env=self.rb.phase.to(DEV))
        torch.cuda.synchronize()
        return self.snapshot(dict(reset=e.extras["reset"].cpu(), term=e.extras["terminate"].cpu()))

    def snapshot(self, out):
        e = self.env
        out.update(obs=e.obs_buf.cpu(), rew=e.rew_buf.cpu(), raw=e.reward_raw[:, :4].cpu(), prog=e.progress_buf.cpu(),
                   state=e._rigid_body_state_reshaped.cpu(), root=e._humanoid_root_states.cpu(), dofp=e._dof_pos.cpu(),
                   dofv=e._dof_vel.cpu(), start=e._motion_start_times.cpu(), soff=e._motion_start_times_offset.cpu(),
                   goff=e._global_offset.cpu())  # fmt: skip
        return out

    def check_step(self, want, before, what="", terminations=True):
        """``terminations``: whether the step can terminate envs (not right after every env was reset: a termination
        needs progress > 1)."""
        b = self.bufs
        f = want["reset"]
        assert 0 < int(f.sum()) < self.n, f"the case should flag some envs and spare others {what}"
        assert bool((f & ~want["term"]).any()), f"clip end {what}"
        assert bool(want["term"].any()) or not terminations, f"termination {what}"
        assert torch.equal(b.obs_buf, want["obs"]), f"obs {what}"
        assert torch.equal(b.rew_buf, want["rew"]), f"rew {what}"
        assert torch.equal(b.reward_raw, want["raw"]), f"reward_raw {what}"
        assert torch.equal(b.reset_buf.bool(), f) and int(b.reset_buf.max()) <= 1, f"reset {what}"
        assert torch.equal(b.terminate_buf.bool(), want["term"]) and int(b.terminate_buf.max()) <= 1, f"term {what}"
        assert torch.equal(b.progress_buf, want["prog"]), f"progress {what}"
        assert int(b.progress_buf[f].abs().max()) == 0
        self.check_rows(f, want, before, what)

    def check_rows(self, f, want, before, what):
        """Rows of flagged envs equal the device path's; others keep what they held."""
        b, r = self.bufs, self.rb
        for name, got in (("state", b.state), ("start", b.motion_start_times), ("soff", b.motion_start_times_offset),
                          ("goff", b.global_offset)):  # fmt: skip
            assert torch.equal(got[f], want[name][f]), f"{name} of re-posed envs {what}"
            assert torch.equal(got[~f], before[name][~f]), f"{name} of other envs {what}"
        assert float(b.motion_start_times_offset[f].abs().max()) == 0.0 and float(b.global_offset[f].abs().max()) == 0.0
        for name, got in (("root", r.root_states), ("dofp", r.dof_pos), ("dofv", r.dof_vel)):
            assert torch.equal(got[f], want[name][f]), f"{name} of re-posed envs {what}"
            assert bool((got[~f] == SENTINEL).all()), f"{name} of other envs written {what}"


def _set_path(monkeypatch, mode):
    if mode in ("direct", "staged"):
        monkeypatch.setenv("PHC_HOST_PATH", mode)
    else:
        monkeypatch.delenv("PHC_HOST_PATH", raising=False)


def _steps(hs, case, slot, steps, what=""):
    for i in range(steps):
        before = case.begin()
        want = case.advance()
        hs.submit(slot, case.bufs, case.rb, **case.host_kwargs())
        assert hs.wait(slot) is case.bufs
        case.check_step(want, before, f"{what} step {i}")


@pytest.mark.parametrize("slot", [0, 1])
@pytest.mark.parametrize("mode", ["direct", "staged", "pageable", "direct_pageable_reset"])
def test_auto_reset_each_slot_eight_steps_deep(slot, mode, monkeypatch):
    """A ragged batch; the clock, state and progress carried in the host buffers from step to step.  The last mode
    posts the step's outputs into pinned buffers and the reset rows through the slot's staging."""
    _set_path(monkeypatch, "direct" if mode.startswith("direct") else mode)
    data, mlib = _motion_lib()
    case = EnvCase(data, mlib, 2005, 11, pinned=mode != "pageable", pinned_reset=mode in ("direct", "staged"))
    with HostStep(mlib, 2005, num_chunks=3) as hs:
        _steps(hs, case, slot, 8, mode)
        assert hs.path == (2 if mode in ("staged", "pageable") else 1)


@pytest.mark.parametrize("mode", ["direct", "staged"])
def test_auto_reset_two_slots_in_flight_over_different_batches(mode, monkeypatch):
    """Different sizes, clips and clocks (random ids, unaligned start times) on the two slots; B waited before A."""
    _set_path(monkeypatch, mode)
    data, mlib = _motion_lib()
    a = EnvCase(data, mlib, 3001, 21)
    b = EnvCase(data, mlib, 5003, 31, ids="random", aligned=False)
    with HostStep(mlib, 6000, num_chunks=3) as hs:
        for r in range(4):
            ba, bb = a.begin(), b.begin()
            wa, wb = a.advance(), b.advance()
            hs.submit(0, a.bufs, a.rb)
            hs.submit(1, b.bufs, b.rb)
            hs.wait(1)
            hs.wait(0)
            a.check_step(wa, ba, f"A round {r}")
            b.check_step(wb, bb, f"B round {r}")


@pytest.mark.parametrize("mode", ["direct", "staged"])
def test_auto_reset_three_future_steps(mode, monkeypatch):
    """T = 3: the step kernels without the in-kernel reset, followed by phc_reset_envs — on the direct path the
    advanced progress the step mirrored into the caller's buffer must still read 0 for re-posed envs."""
    _set_path(monkeypatch, mode)
    data, mlib = _motion_lib()
    case = EnvCase(data, mlib, 1003, 41, T=3)
    with HostStep(mlib, 1003, time_steps=3, num_chunks=3) as hs:
        _steps(hs, case, 0, 4, mode)


def test_auto_reset_on_the_generic_kernel(monkeypatch):
    """PHC_OPT_FORCE_GENERIC_STEP: the reset is a second launch at T = 1 as well (direct path)."""
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    case = EnvCase(data, mlib, 1003, 45)
    capi = _cabi.load()
    capi.phc_set_option(_cabi.OPT_FORCE_GENERIC_STEP, 1)
    try:
        with HostStep(mlib, 1003, num_chunks=3) as hs:
            _steps(hs, case, 0, 3, "generic")
    finally:
        capi.phc_set_option(_cabi.OPT_FORCE_GENERIC_STEP, 0)


@pytest.mark.parametrize("variant", ["start", "eval", "flag_test"])
def test_auto_reset_state_init_start_eval_mode_and_flag_test(variant, monkeypatch):
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    case = EnvCase(data, mlib, 2005, 51, state_init="start" if variant == "start" else "random",
                   eval_mode=variant == "eval", flag_test=variant == "flag_test")  # fmt: skip
    kw = dict(use_mean=True, termination_distances=0.1) if variant == "eval" else {}
    with HostStep(mlib, 2005, num_chunks=3, **kw) as hs:
        _steps(hs, case, 1, 4, variant)


def test_auto_reset_on_a_staged_chunk_of_more_than_10240_envs(monkeypatch):
    """Three doubling chunks of 24000 envs: the last has 12000, where a step without a reset would take the persistent
    kernel; with the reset it runs K6-fast."""
    _set_path(monkeypatch, "staged")
    data, mlib = _motion_lib(256, 602)
    case = EnvCase(data, mlib, 24000, 61, ids="random")
    with HostStep(mlib, 24000, num_chunks=3) as hs:
        _steps(hs, case, 0, 2, "large")


@pytest.mark.parametrize("pinned", [True, False], ids=["pinned", "pageable"])
def test_host_loop_equals_the_device_loop(pinned, monkeypatch):
    """reset_submit of every env (the first observation), ten steps with auto-reset, then a masked reset_submit of a
    subset: every buffer equals the device loop's reset() + ten auto-reset steps + reset(ids, phase), and the masked
    reset leaves every row of the other envs as it was."""
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    n = 2005
    case = EnvCase(data, mlib, n, 71, pinned=pinned)
    e, b, r = case.env, case.bufs, case.rb
    everyone = torch.ones(n, dtype=torch.bool)
    with HostStep(mlib, n, num_chunks=3) as hs:
        # the first observation: nothing of the state or obs rows is read
        before = case.begin()
        b.state.fill_(float("nan"))
        before["state"] = b.state.clone()
        r.env_mask.fill_(1)
        e.reset(None, r.phase.to(DEV))
        torch.cuda.synchronize()
        want = case.snapshot({})
        hs.reset_submit(1, b, r)
        assert hs.wait(1) is b
        assert torch.equal(b.obs_buf, want["obs"]) and torch.equal(b.progress_buf, want["prog"])
        assert not bool(b.reset_buf.any()) and not bool(b.terminate_buf.any())
        assert bool(torch.isnan(b.rew_buf).all()) and bool(torch.isnan(b.reward_raw).all())  # not touched
        case.check_rows(everyone, want, before, "initial reset")
        r.env_mask.zero_()  # ignored by the step
        for i in range(10):
            before = case.begin()
            want = case.advance()
            hs.submit(i % 2, b, r)
            hs.wait(i % 2)
            case.check_step(want, before, f"loop step {i}", terminations=i > 0)
        # a reset of envs the caller picks
        before = case.begin()
        before.update(obs=b.obs_buf.clone(), prog=b.progress_buf.clone())
        mask = torch.rand(n, generator=case.gen) < 0.3
        ids = mask.nonzero().squeeze(1)
        r.env_mask.copy_(mask)
        e.reset(ids.to(DEV), r.phase[ids].to(DEV))
        torch.cuda.synchronize()
        want = case.snapshot({})
        hs.reset(b, r)
        assert torch.equal(b.obs_buf[mask], want["obs"][mask]) and bool(torch.isnan(b.obs_buf[~mask]).all())
        assert int(b.progress_buf[mask].abs().max()) == 0 and torch.equal(b.progress_buf[~mask], before["prog"][~mask])
        assert int(b.reset_buf[mask].max()) == 0 and int(b.reset_buf[~mask].min()) == 7
        assert int(b.terminate_buf[mask].max()) == 0 and int(b.terminate_buf[~mask].min()) == 7
        assert bool(torch.isnan(b.rew_buf).all()) and bool(torch.isnan(b.reward_raw).all())
        case.check_rows(mask, want, before, "masked reset")


def _plain_step_matches(hs, case, slot):
    """A plain submit after an error: bit-identical to the device path's step without a reset."""
    e = case.env
    e.enable_auto_reset(False)
    case.bufs.progress_buf.copy_(e.progress_buf.cpu())
    e.step()
    torch.cuda.synchronize()
    case.poison()
    hs.submit(slot, case.bufs)
    hs.wait(slot)
    b = case.bufs
    assert torch.equal(b.obs_buf, e.obs_buf.cpu()) and torch.equal(b.rew_buf, e.rew_buf.cpu())
    assert torch.equal(b.reward_raw, e.reward_raw[:, :4].cpu()) and torch.equal(b.progress_buf, e.progress_buf.cpu())
    assert torch.equal(b.reset_buf.bool(), e.reset_buf.cpu()) and torch.equal(b.terminate_buf.bool(), e._terminate_buf.cpu())


def test_invalid_reset_arguments_leave_the_slot_idle(monkeypatch):
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    case = EnvCase(data, mlib, 1003, 81)
    capi = _cabi.load()
    dev_root = torch.zeros(1003, 13, device=DEV)
    with HostStep(mlib, 1003, num_chunks=3) as hs:
        ctx = hs._ctx
        case.poison()
        args = case.bufs._args()
        good = case.rb._args(case.bufs, "random", False)
        for slot in (0, 1):
            for fn in (capi.phc_host_step_submit_reset, capi.phc_host_reset_submit):
                for code in (_cabi.STATE_INIT_DEFAULT, _cabi.STATE_INIT_HYBRID, 7):
                    bad = case.rb._args(case.bufs, "random", False)
                    bad.state_init = code
                    assert fn(ctx, slot, C.byref(args), C.byref(bad), 1003) == UNSUPPORTED
                bad = case.rb._args(case.bufs, "random", False)
                bad.phase = None
                assert fn(ctx, slot, C.byref(args), C.byref(bad), 1003) == NULL
                bad = case.rb._args(case.bufs, "random", False)
                bad.root_states = dev_root.data_ptr()
                assert fn(ctx, slot, C.byref(args), C.byref(bad), 1003) == UNSUPPORTED
                bad = case.rb._args(case.bufs, "random", False)
                bad.dof_vel = None
                assert fn(ctx, slot, C.byref(args), C.byref(bad), 1003) == NULL
                assert fn(ctx, slot, C.byref(args), None, 1003) == NULL
                assert capi.phc_host_step_wait(ctx, slot) == OK
            good.env_mask = None
            assert capi.phc_host_reset_submit(ctx, slot, C.byref(args), C.byref(good), 1003) == NULL
            good.env_mask = case.rb.env_mask.data_ptr()
            assert capi.phc_host_step_wait(ctx, slot) == OK
        assert bool(torch.isnan(case.bufs.obs_buf).all()) and bool((case.rb.root_states == SENTINEL).all())
        with pytest.raises(_cabi.PhcError, match="not supported"):
            hs.submit(0, case.bufs, case.rb, state_init="default")
        for slot in (0, 1):
            _plain_step_matches(hs, case, slot)


def test_busy_slot_and_close_with_resets_in_flight(monkeypatch):
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    a = EnvCase(data, mlib, 2005, 91)
    b = EnvCase(data, mlib, 1999, 95, pinned=False)
    capi = _cabi.load()
    hs = HostStep(mlib, 2005, num_chunks=3)
    ctx = hs._ctx
    # busy: a plain step in flight refuses both reset submits and enqueues nothing for them
    b.poison()
    args_a, args_b = a.bufs._args(), b.bufs._args()
    rargs_b = b.rb._args(b.bufs, "random", False)
    assert capi.phc_host_step_submit(ctx, 0, C.byref(args_a), a.n) == OK
    assert capi.phc_host_step_submit_reset(ctx, 0, C.byref(args_b), C.byref(rargs_b), b.n) == BUSY
    assert capi.phc_host_reset_submit(ctx, 0, C.byref(args_b), C.byref(rargs_b), b.n) == BUSY
    assert capi.phc_host_step_wait(ctx, 0) == OK
    assert bool(torch.isnan(b.bufs.obs_buf).all()) and bool((b.rb.root_states == SENTINEL).all())
    a.bufs.progress_buf.copy_(a.env.progress_buf.cpu())  # the device path did not take that plain step
    # close with a step + reset on pinned buffers and a host reset through staging in flight
    ba = a.begin()
    wa = a.advance()
    before = b.begin()
    b.rb.env_mask.copy_(torch.rand(b.n, generator=b.gen) < 0.5)
    mask = b.rb.env_mask.bool()
    ids = mask.nonzero().squeeze(1)
    b.env.reset(ids.to(DEV), b.rb.phase[ids].to(DEV))
    torch.cuda.synchronize()
    wb = b.snapshot({})
    hs.submit(0, a.bufs, a.rb)
    hs.reset_submit(1, b.bufs, b.rb)
    assert capi.phc_host_step_submit_reset(ctx, 1, C.byref(args_a), C.byref(rargs_b), a.n) == BUSY
    hs.close()
    a.check_step(wa, ba, "close, slot 0")
    assert torch.equal(b.bufs.obs_buf[mask], wb["obs"][mask]) and bool(torch.isnan(b.bufs.obs_buf[~mask]).all())
    b.check_rows(mask, wb, before, "close, slot 1")
