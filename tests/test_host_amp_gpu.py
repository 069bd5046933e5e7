"""GPU: AMP observations on the host step (phc_host_step_submit_amp / phc_host_reset_submit_amp).

1. The reference's recording tests/golden/env_rollout.npz (HumanoidPHC.step / reset with AMP on) replayed unabridged
   through conftest.replay_env_rollout on the host path, with host obs and with device outputs.
2. Bit for bit against HumanoidPHC(use_amp_obs=True) on seeded inputs after every step and reset: amp_obs,
   amp_obs_demo and every other output, over the output paths, chunk counts, slots, state inits, T, the power reward,
   S and the other device tensors of the same submit.
3. Error codes: every refusal leaves the slot idle and the AMP tensors untouched.
4. Ordering against the discriminator's stream, and close() with AMP submits in flight."""

import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from humanoid_b200 import (HostAmpBuffers, HostDeviceOutputs, HostEpisodeBuffers, HostResetBuffers, HostStep,
                               HostStepBuffers, HumanoidPHC, MotionLib, _cabi, synth)  # fmt: skip
    from util_gpu import DEV, DOF_DERIVED_TOL, OBS_TOL, clock_from_golden, lib_from_golden

OK, NULL, SHAPE, UNSUPPORTED, BUSY = 0, -1, -2, -4, -8
SENTINEL = 12345.0
COEF = 0.0005


def _set_path(monkeypatch, mode):
    monkeypatch.setenv("PHC_HOST_PATH", "staged" if mode == "staged" else "direct")


def _same(a, b):
    """Bit equality (NaNs included) of two tensors, wherever they live."""
    a, b = a.detach().cpu(), b.detach().cpu()
    if a.dtype == torch.float32 and b.dtype == torch.float32:
        return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))
    return torch.equal(a, b.to(a.dtype))


# ---------------------------------------------------------------------------------------
# 1. the reference's recording
# ---------------------------------------------------------------------------------------
class _HostUnderReplay:
    """The host path with AMP behind conftest.replay_env_rollout's five calls: write_sim fills the host state, dof rows
    and dof force; step is the host step with the power reward and AMP; reset is the host reset of the recorded envs
    with AMP; read_sim rebuilds [n, 69, 2] from the reset buffers.  PD targets come from the device path's own function
    (the replay checks them)."""

    def __init__(self, g, device_out):
        clock = clock_from_golden(g)
        N = clock.progress_buf.shape[0]
        self.N = N
        mlib = MotionLib(lib_from_golden(g), device=DEV)
        self.pd_env = HumanoidPHC(mlib, N, device=DEV)
        self.pd_env._pd_action_offset.copy_(g.inp("pd_action_offset"))
        self.pd_env._pd_action_scale.copy_(g.inp("pd_action_scale"))
        self.hs = HostStep(mlib, N, num_chunks=3, termination_distances=float(g.inp("termination_distance")),
                           use_power_reward=True, rew_power_coef=float(g.inp("rew_power_coef")))  # fmt: skip
        self.b = b = HostStepBuffers.allocate(N, host_obs=not device_out, power=True, amp=True)
        for name in ("progress_buf", "motion_start_times", "motion_start_times_offset", "global_offset",
                     "sampled_motion_ids"):  # fmt: skip
            getattr(b, name).copy_(getattr(clock, name))
        self.r = HostResetBuffers.allocate(N)
        self.dev = HostDeviceOutputs.allocate(N, device=DEV) if device_out else None
        self.amp = HostAmpBuffers.allocate(N, int(g.inp("num_amp_obs_steps")), DEV)
        assert torch.equal(self.amp.dof_subset.cpu(), g.inp("dof_subset"))

    # the reference's buffer names
    progress_buf = property(lambda self: self.b.progress_buf)
    reset_buf = property(lambda self: self.b.reset_buf)
    _terminate_buf = property(lambda self: self.b.terminate_buf)
    rew_buf = property(lambda self: self.b.rew_buf)
    reward_raw = property(lambda self: self.b.reward_raw)
    _motion_start_times = property(lambda self: self.b.motion_start_times)
    _motion_start_times_offset = property(lambda self: self.b.motion_start_times_offset)
    _global_offset = property(lambda self: self.b.global_offset)
    obs_buf = property(lambda self: self.b.obs_buf if self.dev is None else self.dev.obs)
    _amp_obs_buf = property(lambda self: self.amp.amp_obs)
    _amp_obs_demo_buf = property(lambda self: self.amp.amp_obs_demo)

    def write_sim(self, state, dof_state, dof_force):
        self.b.state.copy_(state)
        self.r.root_states.copy_(state[:, 0])
        self.b.dof_pos.copy_(dof_state[..., 0])
        self.b.dof_vel.copy_(dof_state[..., 1])
        self.r.dof_pos.copy_(dof_state[..., 0])
        self.r.dof_vel.copy_(dof_state[..., 1])
        self.b.dof_force.copy_(dof_force)

    def read_sim(self):
        return self.b.state, self.r.root_states, torch.stack([self.r.dof_pos, self.r.dof_vel], -1)

    def step(self, actions, physics):
        pd = self.pd_env._action_to_pd_targets(actions.to(DEV), freeze_hand=True, freeze_toe=True)
        physics(self)
        self.hs.step(self.b, device_out=self.dev, amp=self.amp)
        return pd

    def reset(self, env_ids, phase):
        if len(env_ids):
            self.r.env_mask.zero_()
            self.r.env_mask[env_ids] = 1
            self.r.phase.zero_()
            self.r.phase[env_ids] = phase
            self.hs.reset(self.b, self.r, device_out=self.dev, amp=self.amp)


@pytest.mark.parametrize("out", ["host_obs", "device_out"])
def test_rollout_vs_reference_recording(golden, out):
    """Every assertion of replay_env_rollout, amp_obs after every step and amp_obs / amp_obs_demo after every reset
    included."""
    from conftest import replay_env_rollout

    g = golden("env_rollout")
    shim = _HostUnderReplay(g, out == "device_out")
    try:
        assert replay_env_rollout(g, shim, read=lambda t: t.cpu(), tol=OBS_TOL, dof_tol=DOF_DERIVED_TOL) > 0
    finally:
        shim.hs.close()


# ---------------------------------------------------------------------------------------
# 2. bit for bit against HumanoidPHC(use_amp_obs=True)
# ---------------------------------------------------------------------------------------
def _motion_lib(M=48, seed=907):
    data = synth.make_motion_lib(M, 60, 90, seed=seed, device=DEV)
    return data, MotionLib(data, device=DEV)


class Case:
    """One batch on both paths with AMP: host buffers, AMP tensors (and device outputs, episode tensors) for the host
    step, a HumanoidPHC(use_amp_obs=True) on the same inputs.  Each step the same physics moves both: the rigid bodies
    are pushed (about 3 % of the envs far enough to terminate) and the dof rows (and dof force) are drawn afresh."""

    def __init__(self, data, mlib, n, seed, T=1, S=10, pinned=True, host_obs=True, power=False, auto_reset=False,
                 state_init="random", flag_test=False, episode=False):  # fmt: skip
        clock = synth.make_clock(data, n, seed=seed, ids="mod", aligned=True, max_progress=30)
        ref = mlib.get_motion_state(clock.sampled_motion_ids, synth.reward_time(clock, extra_steps=1), clock.global_offset)
        state = synth.make_sim_state(ref, seed=seed + 1)
        env = HumanoidPHC(mlib, n, device=DEV, time_steps=T, use_power_reward=power, rew_power_coef=COEF,
                          use_amp_obs=True, num_amp_obs_steps=S)  # fmt: skip
        env.set_sim_state(state)
        env.set_clock(clock)
        env.enable_auto_reset(auto_reset)
        env.state_init = state_init
        env.flag_test = flag_test
        self.env, self.n, self.T, self.S, self.power = env, n, T, S, power
        self.auto_reset, self.state_init, self.flag_test = auto_reset, state_init, flag_test
        self.gen = torch.Generator().manual_seed(seed + 2)
        b = HostStepBuffers.allocate(n, T, pinned=pinned, host_obs=host_obs, power=power, amp=True)
        for name, v in (("state", state), ("progress_buf", clock.progress_buf), ("motion_start_times", clock.motion_start_times),
                        ("motion_start_times_offset", clock.motion_start_times_offset),
                        ("global_offset", clock.global_offset), ("sampled_motion_ids", clock.sampled_motion_ids)):  # fmt: skip
            getattr(b, name).copy_(v.cpu())
        self.bufs = b
        self.rb = HostResetBuffers.allocate(n, pinned=pinned)
        self.dev = None if host_obs else HostDeviceOutputs.allocate(n, T, DEV)
        self.amp = HostAmpBuffers.allocate(n, S, DEV)
        self.ep = HostEpisodeBuffers.allocate(n, 5 if power else 4, DEV) if episode else None
        self.k = 0
        self.flagged = 0

    def host_step(self, mlib, **kw):
        kw.setdefault("num_chunks", 3)
        return HostStep(mlib, self.n, time_steps=self.T, use_power_reward=self.power, rew_power_coef=COEF, **kw)

    def obs(self):
        return self.bufs.obs_buf if self.dev is None else self.dev.obs

    def poison(self):
        b, r = self.bufs, self.rb
        b.rew_buf.fill_(float("nan"))
        b.reward_raw.fill_(float("nan"))
        b.reset_buf.fill_(7)
        b.terminate_buf.fill_(7)
        for t in (r.root_states, r.dof_pos, r.dof_vel, self.obs()):
            t.fill_(SENTINEL)

    def physics(self):
        n, k, env = self.n, self.k, self.env
        d = torch.randn(n, 24, 3, generator=self.gen) * 0.01
        d[(torch.arange(n) * 7 + k) % 29 == 0, :, 0] += 0.5
        self.bufs.state[..., 0:3] += d
        env._rigid_body_state_reshaped[..., 0:3] += d.to(DEV)
        pos, vel = torch.randn(n, 69, generator=self.gen) * 0.5, torch.randn(n, 69, generator=self.gen)
        self.bufs.dof_pos.copy_(pos)
        self.bufs.dof_vel.copy_(vel)
        env._dof_pos.copy_(pos.to(DEV))
        env._dof_vel.copy_(vel.to(DEV))
        if self.power:
            force = torch.randn(n, 69, generator=self.gen) * 50
            self.bufs.dof_force.copy_(force)
            env.dof_force_tensor.copy_(force.to(DEV))
        self.k += 1

    def draw(self):
        self.rb.phase.copy_(torch.rand(self.n, generator=self.gen))

    def advance(self):
        """Physics, fresh draws, poisoned outputs, one step of the device path; returns its outputs."""
        self.physics()
        self.draw()
        self.poison()
        e = self.env
        self.demo_before = self.amp.amp_obs_demo.clone()
        if self.auto_reset:
            e.step(phase_by_env=self.rb.phase.to(DEV))
            flags = (e.extras["reset"].clone(), e.extras["terminate"].clone())
        else:
            e.step()
            flags = (e.reset_buf.clone(), e._terminate_buf.clone())
        torch.cuda.synchronize()
        return self.snapshot(dict(reset=flags[0].cpu(), term=flags[1].cpu()))

    def snapshot(self, out):
        e = self.env
        out.update(obs=e.obs_buf.clone(), rew=e.rew_buf.cpu(), raw=e.reward_raw.cpu(), prog=e.progress_buf.cpu(),
                   root=e._humanoid_root_states.cpu(), dofp=e._dof_pos.cpu(), dofv=e._dof_vel.cpu(),
                   state=e._rigid_body_state_reshaped.cpu(), amp=e._amp_obs_buf.clone(),
                   demo=e._amp_obs_demo_buf.clone())  # fmt: skip
        return out

    def submit(self, hs, slot):
        hs.submit(slot, self.bufs, self.rb if self.auto_reset else None, state_init=self.state_init,
                  flag_test=self.flag_test, device_out=self.dev, episode=self.ep, amp=self.amp)  # fmt: skip

    def check_amp(self, want, what):
        assert _same(self.amp.amp_obs, want["amp"]), f"amp_obs {what}"
        assert _same(self.amp.amp_obs_demo, want["demo"]), f"amp_obs_demo {what}"
        assert self.amp.obs.shape == self.env.amp_obs.shape and _same(self.amp.obs, self.env.amp_obs), what

    def check_step(self, want, what=""):
        b = self.bufs
        f = want["reset"]
        if self.auto_reset:  # over a run some envs are re-posed (flagged), never all of them in one step
            assert int(f.sum()) < self.n, f"the case should spare some envs {what}"
            self.flagged += int(f.sum())
        assert _same(self.obs(), want["obs"]), f"obs {what}"
        assert _same(b.rew_buf, want["rew"]), f"rew {what}"
        assert _same(b.reward_raw, want["raw"][:, : b.reward_raw.shape[1]]), f"reward_raw {what}"
        assert torch.equal(b.reset_buf.bool(), f) and int(b.reset_buf.max()) <= 1, f"reset {what}"
        assert torch.equal(b.terminate_buf.bool(), want["term"]), f"term {what}"
        assert torch.equal(b.progress_buf, want["prog"]), f"progress {what}"
        self.check_amp(want, what)
        if self.auto_reset:
            r = self.rb
            for name, got in (("root", r.root_states), ("dofp", r.dof_pos), ("dofv", r.dof_vel)):
                assert _same(got[f], want[name][f]), f"{name} of re-posed envs {what}"
            assert _same(b.state, want["state"]), f"rigid-body state {what}"
        # the demo rows of the envs not re-posed are untouched
        keep = ~f.to(DEV) if self.auto_reset else torch.ones(self.n, dtype=torch.bool, device=DEV)
        assert _same(self.amp.amp_obs_demo[keep], self.demo_before[keep]), f"demo rows of other envs {what}"
        if self.ep is not None:
            assert _same(self.ep.rewards, want["rew"]), f"episode rewards {what}"

    def reset_masked(self, hs, slot, p=0.4):
        """A masked host reset on both paths (p = 1: every env, how an AMP loop starts)."""
        n = self.n
        mask = torch.rand(n, generator=self.gen) < p if p < 1 else torch.ones(n, dtype=torch.bool)
        ids = mask.nonzero().squeeze(1)
        self.draw()
        self.rb.env_mask.copy_(mask)
        self.poison()
        self.demo_before = self.amp.amp_obs_demo.clone()
        self.env.reset(ids.to(DEV), self.rb.phase[ids].to(DEV))
        torch.cuda.synchronize()
        want = self.snapshot({})
        hs.reset_submit(slot, self.bufs, self.rb, state_init=self.state_init, flag_test=self.flag_test,
                        device_out=self.dev, amp=self.amp)  # fmt: skip
        assert hs.wait(slot) is self.bufs
        m = mask.to(DEV)
        assert _same(self.obs()[m.to(self.obs().device)], want["obs"][m]), "obs of masked envs"
        self.check_amp(want, "after the host reset")
        assert _same(self.amp.amp_obs_demo[~m], self.demo_before[~m]), "demo rows of envs not reset"
        for name, got in (("root", self.rb.root_states), ("dofp", self.rb.dof_pos), ("dofv", self.rb.dof_vel)):
            assert _same(got[mask], want[name][mask]), name
        return mask


def _steps(hs, case, slot, steps, what=""):
    for i in range(steps):
        want = case.advance()
        case.submit(hs, slot)
        assert hs.wait(slot) is case.bufs
        case.check_step(want, f"{what} step {i}")


CONFIGS = {  # id: (path, Case kwargs, HostStep kwargs)
    "direct": ("direct", dict(power=True, auto_reset=True), {}),
    "staged": ("staged", dict(power=True, auto_reset=True), {}),
    "pageable": ("direct", dict(power=True, auto_reset=True, pinned=False), {}),
    "direct-device_out": ("direct", dict(auto_reset=True, host_obs=False), {}),
    "staged-device_out": ("staged", dict(power=True, auto_reset=True, host_obs=False), {}),
    "pageable-device_out": ("direct", dict(auto_reset=True, pinned=False, host_obs=False), {}),
    "chunks1": ("direct", dict(power=True, auto_reset=True), dict(num_chunks=1)),
    "chunks7-ragged1000": ("direct", dict(n=1000, auto_reset=True, host_obs=False), dict(num_chunks=7)),
    "staged-chunks7-ragged1000": ("staged", dict(n=1000, power=True, auto_reset=True), dict(num_chunks=7)),
    "no_reset": ("direct", dict(power=True), {}),
    "no_power-no_reset-staged": ("staged", dict(), {}),
    "start": ("direct", dict(auto_reset=True, state_init="start"), {}),
    "flag_test": ("direct", dict(power=True, auto_reset=True, flag_test=True), {}),
    "T10": ("direct", dict(T=10, auto_reset=True, host_obs=False), {}),
    "T10-staged": ("staged", dict(T=10, power=True, auto_reset=True), {}),
    "S1": ("direct", dict(S=1, auto_reset=True), {}),
    "S16": ("staged", dict(S=16, power=True, auto_reset=True, host_obs=False), {}),
    "device_out-episode": ("direct", dict(power=True, auto_reset=True, host_obs=False, episode=True), {}),
    "staged-episode": ("staged", dict(auto_reset=True, episode=True), {}),
}


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_bit_for_bit_against_device_path(cfg, monkeypatch):
    """A masked host reset of every env (the loop's first AMP observation), four steps on slot 0, a masked host reset
    of 40 % of the envs, four steps on slot 1: after each, every output and the AMP tensors bit for bit."""
    path, kw, hkw = CONFIGS[cfg]
    _set_path(monkeypatch, path)
    data, mlib = _motion_lib()
    n = kw.pop("n", 2005)
    case = Case(data, mlib, n, 11, **kw)
    with case.host_step(mlib, **hkw) as hs:
        case.reset_masked(hs, 0, p=1)
        _steps(hs, case, 0, 4, f"{cfg} slot 0")
        case.reset_masked(hs, 1)
        _steps(hs, case, 1, 4, f"{cfg} slot 1")
        assert bool(case.amp.amp_obs_demo.abs().sum() > 0)
        assert case.flagged > 0 or not case.auto_reset, "no env was re-posed inside a step"
        assert hs.path == (2 if path == "staged" or not kw.get("pinned", True) else 1)


@pytest.mark.parametrize("out", ["host_obs", "device_out"])
@pytest.mark.parametrize("mode", ["direct", "staged"])
def test_two_slots_waited_out_of_order(mode, out, monkeypatch):
    """Two batches of different sizes and S, each on its own slot with its own AMP tensors, submitted back to back and
    waited in reverse order."""
    _set_path(monkeypatch, mode)
    data, mlib = _motion_lib()
    a = Case(data, mlib, 2005, 21, power=True, auto_reset=True, host_obs=out == "host_obs")
    b = Case(data, mlib, 1003, 31, power=True, auto_reset=True, host_obs=out == "host_obs", S=4)
    with a.host_step(mlib) as hs:
        a.reset_masked(hs, 0, p=1)
        b.reset_masked(hs, 1, p=1)
        for r in range(4):
            wa, wb = a.advance(), b.advance()
            a.submit(hs, 0)
            b.submit(hs, 1)
            hs.wait(1)
            hs.wait(0)
            a.check_step(wa, f"A round {r}")
            b.check_step(wb, f"B round {r}")
        assert a.flagged > 0 and b.flagged > 0


# ---------------------------------------------------------------------------------------
# 3. error codes
# ---------------------------------------------------------------------------------------
def test_error_codes_enqueue_nothing(monkeypatch):
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    n = 1003
    case = Case(data, mlib, n, 101, power=True, auto_reset=True)
    capi = _cabi.load()
    amp = case.amp
    amp.amp_obs.fill_(SENTINEL)
    amp.amp_obs_demo.fill_(SENTINEL)
    dev_rows = torch.zeros(n, 69, device=DEV)
    cpu_obs = torch.zeros_like(amp.amp_obs, device="cpu")
    cpu_subset = amp.dof_subset.cpu()
    other_vel = torch.zeros(n, 69).pin_memory()
    with case.host_step(mlib) as hs:
        ctx = hs._ctx
        case.poison()
        args = case.bufs._args()
        env = hs._env_args(0, case.bufs, None, "random", n)

        def A(**fields):
            x = amp._args(case.bufs)
            for k, v in fields.items():
                if k == "key0":
                    x.key_body_ids[0] = v
                else:
                    setattr(x, k, v)
            return C.byref(x)

        def rargs(state_init="random"):
            return C.byref(case.rb._args(case.bufs, state_init, False))

        step_fn, reset_fn = capi.phc_host_step_submit_amp, capi.phc_host_reset_submit_amp
        no_power = _cabi.PhcHostEnvArgs()
        for slot in (0, 1):
            for r in (None, rargs()):
                assert step_fn(ctx, slot, C.byref(args), r, None, C.byref(env), None, None, n) == NULL
                assert step_fn(ctx, slot, C.byref(args), r, None, C.byref(env), None, A(amp_obs=None), n) == NULL
                assert step_fn(ctx, slot, C.byref(args), r, None, C.byref(env), None, A(dof_pos=None), n) == NULL
                # no velocity rows: neither the AMP's nor the power reward's
                assert step_fn(ctx, slot, C.byref(args), r, None, None, None, A(dof_vel=None), n) == NULL
                for bad in (dict(num_steps=0), dict(num_steps=17), dict(obs_per_step=195), dict(key0=24),
                            dict(key0=-1), dict(num_sel=56)):  # fmt: skip
                    assert step_fn(ctx, slot, C.byref(args), r, None, C.byref(env), None, A(**bad), n) == SHAPE, bad
                # two different velocity sources
                assert step_fn(ctx, slot, C.byref(args), r, None, C.byref(env), None,
                               A(dof_vel=other_vel.data_ptr()), n) == SHAPE  # fmt: skip
                for bad in (dict(amp_obs=cpu_obs.data_ptr()), dict(amp_obs_demo=cpu_obs.data_ptr()),
                            dict(dof_subset=cpu_subset.data_ptr()), dict(dof_pos=dev_rows.data_ptr())):  # fmt: skip
                    assert step_fn(ctx, slot, C.byref(args), r, None, C.byref(env), None, A(**bad), n) == UNSUPPORTED
                assert step_fn(ctx, slot, C.byref(args), r, None, C.byref(no_power), None,
                               A(dof_vel=dev_rows.data_ptr()), n) == UNSUPPORTED  # fmt: skip
            assert reset_fn(ctx, slot, C.byref(args), rargs(), None, None, None, n) == NULL
            assert reset_fn(ctx, slot, C.byref(args), rargs(), None, None, A(amp_obs=None), n) == NULL
            assert reset_fn(ctx, slot, C.byref(args), rargs(), None, None, A(num_steps=17), n) == SHAPE
            assert reset_fn(ctx, slot, C.byref(args), rargs(), None, None, A(amp_obs=cpu_obs.data_ptr()), n) == UNSUPPORTED
            # StateInit.Default / Hybrid, on a slot that has its initial rows
            init = (torch.zeros(n, 13), torch.zeros(n, 69), torch.zeros(n, 69))
            hs.set_initial_state(slot, *init)
            hy = _cabi.PhcHostEnvArgs()
            hy.default_mask = case.rb.env_mask.data_ptr()
            penv = hs._env_args(0, case.bufs, None, "random", n)
            penv.default_mask = case.rb.env_mask.data_ptr()
            for si in ("default", "hybrid"):
                assert step_fn(ctx, slot, C.byref(args), rargs(si), None, C.byref(penv), None, A(), n) == UNSUPPORTED
                assert reset_fn(ctx, slot, C.byref(args), rargs(si), None, C.byref(hy), A(), n) == UNSUPPORTED
            assert capi.phc_host_step_wait(ctx, slot) == OK
        torch.cuda.synchronize()
        assert bool((amp.amp_obs == SENTINEL).all()) and bool((amp.amp_obs_demo == SENTINEL).all())
        assert bool(torch.isnan(case.bufs.rew_buf).all()) and bool((case.bufs.obs_buf == SENTINEL).all())
        # busy: the slot in flight refuses both submits, then finishes as before
        amp.amp_obs.zero_()
        amp.amp_obs_demo.zero_()
        case.env._amp_obs_buf.zero_()
        want = case.advance()
        case.submit(hs, 0)
        assert step_fn(ctx, 0, C.byref(args), rargs(), None, C.byref(env), None, A(), n) == BUSY
        assert reset_fn(ctx, 0, C.byref(args), rargs(), None, None, A(), n) == BUSY
        hs.wait(0)
        case.check_step(want, "after the errors")


# ---------------------------------------------------------------------------------------
# 4. ordering and close
# ---------------------------------------------------------------------------------------
def test_ordering_against_the_discriminator_stream(monkeypatch):
    """A read of amp_obs queued on the discriminator's (current) stream behind a long kernel, before the submit, sees
    the history from before the step; after wait, a read on another stream sees the step's rows."""
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    case = Case(data, mlib, 2005, 201, power=True, auto_reset=True, host_obs=False)
    with case.host_step(mlib) as hs:
        case.reset_masked(hs, 0, p=1)
        for i in range(3):
            prev = case.amp.amp_obs.clone()
            want = case.advance()
            torch.cuda._sleep(200_000_000)  # ~0.1 s on the discriminator's (current) stream
            snap = case.amp.amp_obs.clone()
            case.submit(hs, i % 2)
            hs.wait(i % 2)
            torch.cuda.synchronize()
            assert _same(snap, prev), "amp_obs copied before the submit saw the new step"
            assert not _same(prev, want["amp"])
            side = torch.cuda.Stream()
            with torch.cuda.stream(side):
                seen = case.amp.amp_obs.clone()
            side.synchronize()
            assert _same(seen, want["amp"]), "amp_obs after wait, read on another stream"
            case.check_step(want, f"ordering {i}")


def test_close_with_amp_submits_in_flight(monkeypatch):
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    a = Case(data, mlib, 2005, 211, power=True, auto_reset=True)
    b = Case(data, mlib, 1999, 221, power=True, pinned=False, host_obs=False, auto_reset=True)
    hs = a.host_step(mlib)
    a.reset_masked(hs, 0, p=1)
    b.reset_masked(hs, 1, p=1)
    wa, wb = a.advance(), b.advance()
    a.submit(hs, 0)
    b.submit(hs, 1)
    hs.close()
    a.check_step(wa, "close, slot 0")
    b.check_step(wb, "close, slot 1")
