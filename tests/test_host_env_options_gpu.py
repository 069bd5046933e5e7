"""GPU: the env options of the host step — power reward, eval-mode mpjpe, StateInit.Default / Hybrid.

1. Against the reference's own recordings: tests/golden/env_reset_modes.npz (HumanoidPHC.step / reset with
   StateInit.Default / Hybrid and the default power reward) and tests/golden/env_rollout.npz (power reward, random
   init), replayed through the host path with host obs and with device outputs, with the device-path tolerances.
2. Bit for bit against HumanoidPHC(use_power_reward=True) on seeded cases: direct, staged and pageable buffers, both
   slots, auto-reset with every state init, masked host resets, T = 3, the generic kernel, eval-mode mpjpe, and a NaN
   dof force.
3. Error codes: every refusal leaves the slot idle and the outputs untouched."""

import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from conftest import assert_close, assert_equal_exact
    from humanoid_b200 import (HostDeviceOutputs, HostResetBuffers, HostStep, HostStepBuffers, HumanoidPHC, MotionLib,
                               _cabi, synth)  # fmt: skip
    from util_gpu import DEV, DOF_DERIVED_TOL, OBS_TOL, clock_from_golden, lib_from_golden

OK, NULL, SHAPE, UNSUPPORTED, BUSY = 0, -1, -2, -4, -8
SENTINEL = 12345.0
COEF = 0.0005


def _set_path(monkeypatch, mode):
    if mode in ("direct", "staged"):
        monkeypatch.setenv("PHC_HOST_PATH", mode)
    else:
        monkeypatch.delenv("PHC_HOST_PATH", raising=False)
    monkeypatch.delenv("PHC_HOST_STAGED", raising=False)


def _same(a, b):
    """Bit equality (NaNs included) of two tensors, wherever they live."""
    a, b = a.detach().cpu(), b.detach().cpu()
    if a.dtype == torch.float32 and b.dtype == torch.float32:
        return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))
    return torch.equal(a, b.to(a.dtype))


# ---------------------------------------------------------------------------------------
# 1. the reference's recordings
# ---------------------------------------------------------------------------------------
class _HostUnderReplay:
    """The host path behind conftest.replay_env_reset_modes' five calls.  write_sim fills the host state, dof velocity
    and dof force; step is the host step with the power reward; reset is the host reset of an env mask (auto_reset: the
    reset rides inside the step, the replay's reset() only advances the record); read_sim rebuilds [n, 69, 2] from the
    reset buffers.  PD targets come from the device path's own function (the replay checks them)."""

    def __init__(self, g, mode, device_out, auto_reset=False):
        clock = clock_from_golden(g)
        N = clock.progress_buf.shape[0]
        self.g, self.mode, self.N, self.k, self.auto_reset = g, mode, N, 0, auto_reset
        mlib = MotionLib(lib_from_golden(g), device=DEV)
        self.pd_env = HumanoidPHC(mlib, N, device=DEV)
        self.pd_env._pd_action_offset.copy_(g.inp("pd_action_offset"))
        self.pd_env._pd_action_scale.copy_(g.inp("pd_action_scale"))
        self.hs = HostStep(mlib, N, num_chunks=3, termination_distances=float(g.inp("termination_distance")),
                           use_power_reward=True, rew_power_coef=float(g.inp("rew_power_coef")))  # fmt: skip
        self.b = b = HostStepBuffers.allocate(N, host_obs=not device_out, power=True)
        for name in ("progress_buf", "motion_start_times", "motion_start_times_offset", "global_offset",
                     "sampled_motion_ids"):  # fmt: skip
            getattr(b, name).copy_(getattr(clock, name))
        self.r = HostResetBuffers.allocate(N, hybrid=True)
        self.dev = HostDeviceOutputs.allocate(N, device=DEV) if device_out else None
        self.state_init = "random" if mode is None else mode.lower()
        if mode is not None:
            self.hs.set_initial_state(0, *(g.inp(f"initial_{x}").float().contiguous() for x in ("root_states", "dof_pos", "dof_vel")))

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

    def write_sim(self, state, dof_state, dof_force):
        self.b.state.copy_(state)
        self.r.root_states.copy_(state[:, 0])
        self.r.dof_pos.copy_(dof_state[..., 0])
        self.b.dof_vel.copy_(dof_state[..., 1])
        self.r.dof_vel.copy_(dof_state[..., 1])
        self.b.dof_force.copy_(dof_force)

    def read_sim(self):
        return self.b.state, self.r.root_states, torch.stack([self.r.dof_pos, self.r.dof_vel], -1)

    def _draws(self, k):
        """The recorded draws of reset k, by env: env mask, phase, default mask."""
        g, mode, N = self.g, self.mode, self.N
        rows = g.inp(f"{mode}.reset_indices.{k}" if mode else f"reset_indices.{k}")
        emask, dmask, phase = torch.zeros(N, dtype=torch.uint8), torch.zeros(N, dtype=torch.uint8), torch.zeros(N)
        emask[rows] = 1
        if mode == "Default":
            dmask[rows] = 1
        elif mode == "Hybrid":
            ref = g.inp(f"{mode}.ref_mask.{k}")
            dmask[rows] = (~ref).to(torch.uint8)
            phase[rows[ref]] = g.inp(f"{mode}.phase.{k}")
        else:
            phase[rows] = g.inp(f"phase.{k}")
        return emask, phase, dmask

    def _load_draws(self, k):
        emask, phase, dmask = self._draws(k)
        self.r.env_mask.copy_(emask)
        self.r.phase.copy_(phase)
        self.r.default_mask.copy_(dmask)

    def step(self, actions, physics):
        pd = self.pd_env._action_to_pd_targets(actions.to(DEV), freeze_hand=True, freeze_toe=True)
        physics(self)
        if self.auto_reset:
            self._load_draws(self.k)
        self.hs.step(self.b, self.r if self.auto_reset else None, state_init=self.state_init, device_out=self.dev)
        return pd

    def reset(self, env_ids, phase, default_mask=None):
        if not self.auto_reset:
            self._load_draws(self.k)
            if int(self.r.env_mask.sum()):
                self.hs.reset(self.b, self.r, state_init=self.state_init, device_out=self.dev)
        self.k += 1


@pytest.mark.parametrize("out", ["host_obs", "device_out"])
@pytest.mark.parametrize("mode", ["Default", "Hybrid"])
def test_reset_modes_vs_reference_recording(golden, mode, out):
    from conftest import replay_env_reset_modes

    g = golden("env_reset_modes")
    shim = _HostUnderReplay(g, mode, out == "device_out")
    try:
        assert replay_env_reset_modes(g, shim, mode, read=lambda t: t.cpu(), tol=OBS_TOL, dof_tol=DOF_DERIVED_TOL) == 3
    finally:
        shim.hs.close()


@pytest.mark.parametrize("out", ["host_obs", "device_out"])
@pytest.mark.parametrize("mode", ["Default", "Hybrid"])
def test_reset_modes_vs_reference_recording_auto_reset(golden, mode, out):
    """The reset inside the step: the envs not reset match the step record, everything matches the reset record."""
    g = golden("env_reset_modes")
    shim = _HostUnderReplay(g, mode, out == "device_out", auto_reset=True)
    try:
        for k in range(3):
            def physics(e, k=k):
                e.write_sim(g.inp(f"{mode}.state.{k}"), g.inp(f"{mode}.dof_state.{k}"), g.inp(f"{mode}.dof_force.{k}"))

            shim.step(g.inp(f"{mode}.actions.{k}"), physics)
            rows = g.inp(f"{mode}.reset_indices.{k}")
            keep = torch.ones(shim.N, dtype=torch.bool)
            keep[rows] = False
            s = lambda n, k=k: g.out(f"{mode}.step.{k}.{n}")  # noqa: E731
            r = lambda n, k=k: g.out(f"{mode}.reset.{k}.{n}")  # noqa: E731
            assert_equal_exact(shim.reset_buf, s("reset"), f"reset flags[{k}]")
            assert_equal_exact(shim._terminate_buf, s("terminate"), f"terminate flags[{k}]")
            assert_close(shim.rew_buf, s("rew"), what=f"rew[{k}]", **OBS_TOL)
            assert_close(shim.reward_raw, s("reward_raw"), what=f"reward_raw[{k}]", **OBS_TOL)
            assert_close(shim.obs_buf.cpu()[keep], s("obs")[keep], what=f"obs of the envs not reset[{k}]", **OBS_TOL)
            for name in ("progress", "motion_start_times", "global_offset", "motion_start_times_offset"):
                attr = {"progress": "progress_buf"}.get(name, "_" + name)
                assert_equal_exact(getattr(shim, attr), r(name), f"{name} after reset[{k}]")
            sim, root, dof = shim.read_sim()
            assert_close(sim, r("rigid_body_state"), what=f"rigid_body_state after reset[{k}]", **OBS_TOL)
            assert_close(root[rows], r("root_states")[rows], what=f"root_states after reset[{k}]", **OBS_TOL)
            assert_close(dof[rows], r("dof_state")[rows], what=f"dof_state after reset[{k}]", **DOF_DERIVED_TOL)
            assert_close(shim.obs_buf.cpu(), r("obs"), what=f"obs after reset[{k}]", **OBS_TOL)
            shim.k += 1
    finally:
        shim.hs.close()


@pytest.mark.parametrize("out", ["host_obs", "device_out"])
def test_power_rollout_vs_reference_recording(golden, out):
    """env_rollout.npz (the reference's default config: power reward, random init) through the host path: obs, rew,
    all five reward_raw columns, flags and progress after every step; the reset rows and clock after every reset."""
    g = golden("env_rollout")
    shim = _HostUnderReplay(g, None, out == "device_out")
    try:
        K = len([k for k in g.keys() if k.startswith("in.actions.")])
        for k in range(K):
            def physics(e, k=k):
                e.write_sim(g.inp(f"state.{k}"), g.inp(f"dof_state.{k}"), g.inp(f"dof_force.{k}"))

            pd = shim.step(g.inp(f"actions.{k}"), physics)
            assert_equal_exact(pd, g.out(f"pd_target.{k}"), f"pd_target[{k}]")
            o = lambda n, k=k: g.out(f"step.{k}.{n}")  # noqa: E731
            assert_equal_exact(shim.progress_buf, o("progress"), f"progress[{k}]")
            assert_equal_exact(shim.reset_buf, o("reset"), f"reset[{k}]")
            assert_equal_exact(shim._terminate_buf, o("terminate"), f"terminate[{k}]")
            assert_close(shim.obs_buf.cpu(), o("obs"), what=f"obs[{k}]", **OBS_TOL)
            assert_close(shim.rew_buf, o("rew"), what=f"rew[{k}]", **OBS_TOL)
            assert tuple(shim.reward_raw.shape) == tuple(o("reward_raw").shape) == (shim.N, 5)
            assert_close(shim.reward_raw, o("reward_raw"), what=f"reward_raw[{k}]", **OBS_TOL)
            shim.reset(g.inp(f"reset_indices.{k}"), g.inp(f"phase.{k}"))
            o = lambda n, k=k: g.out(f"reset.{k}.{n}")  # noqa: E731
            rows = g.inp(f"reset_indices.{k}")
            for name, attr in (("progress", "progress_buf"), ("reset", "reset_buf"), ("terminate", "_terminate_buf"),
                               ("motion_start_times", "_motion_start_times"), ("global_offset", "_global_offset"),
                               ("motion_start_times_offset", "_motion_start_times_offset")):  # fmt: skip
                assert_equal_exact(getattr(shim, attr), o(name), f"{name} after reset[{k}]")
            sim, root, dof = shim.read_sim()
            assert_close(sim, o("rigid_body_state"), what=f"rigid_body_state after reset[{k}]", **OBS_TOL)
            assert_close(root[rows], o("root_states")[rows], what=f"root_states after reset[{k}]", **OBS_TOL)
            assert_close(dof[rows], o("dof_state")[rows], what=f"dof_state after reset[{k}]", **DOF_DERIVED_TOL)
            assert_close(shim.obs_buf.cpu(), o("obs"), what=f"obs after reset[{k}]", **OBS_TOL)
        assert K > 0
    finally:
        shim.hs.close()


# ---------------------------------------------------------------------------------------
# 2. bit for bit against HumanoidPHC(use_power_reward=True)
# ---------------------------------------------------------------------------------------
def _motion_lib(M=48, seed=901):
    data = synth.make_motion_lib(M, 60, 90, seed=seed, device=DEV)
    return data, MotionLib(data, device=DEV)


class Case:
    """One batch on both paths with the power reward: host buffers (and device outputs) for the host step, a
    HumanoidPHC(use_power_reward=True) on the same inputs.  Each step the same physics moves both: the rigid bodies are
    pushed (about 3 % of the envs far enough to terminate) and the dof force / velocity are drawn afresh."""

    def __init__(self, data, mlib, n, seed, T=1, pinned=True, host_obs=True, auto_reset=False, state_init="random",
                 eval_mode=False, nan_env=None):  # fmt: skip
        clock = synth.make_clock(data, n, seed=seed, ids="mod", aligned=True, max_progress=30)
        ref = mlib.get_motion_state(clock.sampled_motion_ids, synth.reward_time(clock, extra_steps=1), clock.global_offset)
        state = synth.make_sim_state(ref, seed=seed + 1)
        env = HumanoidPHC(mlib, n, device=DEV, time_steps=T, use_power_reward=True, rew_power_coef=COEF)
        env.set_sim_state(state)
        env.set_clock(clock)
        env.enable_auto_reset(auto_reset)
        env.state_init = state_init
        if eval_mode:
            env.flag_im_eval = True
            env.set_termination_distances(0.1)
        self.gen = torch.Generator().manual_seed(seed + 2)
        self.init = (torch.randn(n, 13, generator=self.gen), torch.randn(n, 69, generator=self.gen),
                     torch.randn(n, 69, generator=self.gen))  # fmt: skip
        for t, v in zip((env._initial_humanoid_root_states, env._initial_dof_pos, env._initial_dof_vel), self.init):
            t.copy_(v.to(DEV))
        self.env, self.n, self.T, self.auto_reset, self.state_init = env, n, T, auto_reset, state_init
        self.eval_mode, self.nan_env = eval_mode, nan_env
        b = HostStepBuffers.allocate(n, T, pinned=pinned, host_obs=host_obs, power=True, mpjpe=eval_mode)
        for name, v in (("state", state), ("progress_buf", clock.progress_buf), ("motion_start_times", clock.motion_start_times),
                        ("motion_start_times_offset", clock.motion_start_times_offset),
                        ("global_offset", clock.global_offset), ("sampled_motion_ids", clock.sampled_motion_ids)):  # fmt: skip
            getattr(b, name).copy_(v.cpu())
        self.bufs = b
        self.rb = HostResetBuffers.allocate(n, pinned=pinned, hybrid=True)
        self.dev = None if host_obs else HostDeviceOutputs.allocate(n, T, DEV)
        self.k = 0

    def host_step(self, mlib, **kw):
        kw.setdefault("num_chunks", 3)
        if self.eval_mode:
            kw.update(use_mean=True, termination_distances=0.1)
        return HostStep(mlib, self.n, time_steps=self.T, use_power_reward=True, rew_power_coef=COEF, **kw)

    def set_initial_state(self, hs, slot):
        hs.set_initial_state(slot, *self.init)

    def obs(self):
        return self.bufs.obs_buf if self.dev is None else self.dev.obs

    def poison(self):
        b, r = self.bufs, self.rb
        for t in (b.rew_buf, b.reward_raw) + ((b.mpjpe,) if b.mpjpe is not None else ()):
            t.fill_(float("nan"))
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
        force, vel = torch.randn(n, 69, generator=self.gen) * 50, torch.randn(n, 69, generator=self.gen)
        if self.nan_env is not None:
            force[self.nan_env, 5] = float("nan")
        self.bufs.dof_force.copy_(force)
        self.bufs.dof_vel.copy_(vel)
        env.dof_force_tensor.copy_(force.to(DEV))
        env._dof_vel.copy_(vel.to(DEV))
        self.k += 1

    def draw(self):
        self.rb.phase.copy_(torch.rand(self.n, generator=self.gen))
        self.rb.default_mask.copy_(torch.rand(self.n, generator=self.gen) < 0.5)

    def advance(self):
        """Physics, fresh draws, poisoned outputs, one step of the device path; returns its outputs."""
        self.physics()
        self.draw()
        self.poison()
        e = self.env
        if self.auto_reset:
            e.step(phase_by_env=self.rb.phase.to(DEV), default_mask_by_env=self.rb.default_mask.to(DEV))
            flags = (e.extras["reset"].clone(), e.extras["terminate"].clone())
        else:
            e.step()
            flags = (e.reset_buf.clone(), e._terminate_buf.clone())
        torch.cuda.synchronize()
        return self.snapshot(dict(reset=flags[0].cpu(), term=flags[1].cpu(),
                                  mpjpe=e.extras["mpjpe"].cpu() if self.eval_mode else None))  # fmt: skip

    def snapshot(self, out):
        e = self.env
        out.update(obs=e.obs_buf.clone(), rew=e.rew_buf.cpu(), raw=e.reward_raw.cpu(), prog=e.progress_buf.cpu(),
                   root=e._humanoid_root_states.cpu(), dofp=e._dof_pos.cpu(), dofv=e._dof_vel.cpu(),
                   state=e._rigid_body_state_reshaped.cpu())  # fmt: skip
        return out

    def submit(self, hs, slot):
        hs.submit(slot, self.bufs, self.rb if self.auto_reset else None, state_init=self.state_init, device_out=self.dev)

    def check_step(self, want, what="", first=False):
        b = self.bufs
        f = want["reset"]
        if self.auto_reset:
            assert 0 < int(f.sum()) < self.n, f"the case should flag some envs and spare others {what}"
        if first:  # the power term is zeroed while progress <= 3 and counts after
            assert bool((want["prog"] <= 3).any()) and bool((want["prog"] > 3).any()), f"progress mix {what}"
            assert bool((want["raw"][:, 4] == 0).any()) and bool((want["raw"][:, 4] < 0).any()), f"power mix {what}"
        assert _same(self.obs(), want["obs"]), f"obs {what}"
        assert _same(b.rew_buf, want["rew"]), f"rew {what}"
        assert _same(b.reward_raw, want["raw"]), f"reward_raw {what}"
        assert torch.equal(b.reset_buf.bool(), f) and int(b.reset_buf.max()) <= 1, f"reset {what}"
        assert torch.equal(b.terminate_buf.bool(), want["term"]), f"term {what}"
        assert torch.equal(b.progress_buf, want["prog"]), f"progress {what}"
        if want.get("mpjpe") is not None:
            assert _same(b.mpjpe, want["mpjpe"]), f"mpjpe {what}"
        if self.nan_env is not None:
            assert torch.isnan(b.rew_buf[self.nan_env]) or int(want["prog"][self.nan_env]) <= 3
        if self.auto_reset:
            r = self.rb
            for name, got in (("root", r.root_states), ("dofp", r.dof_pos), ("dofv", r.dof_vel)):
                assert _same(got[f], want[name][f]), f"{name} of re-posed envs {what}"
                assert bool((got[~f] == SENTINEL).all()), f"{name} of other envs written {what}"
            assert _same(b.state, want["state"]), f"rigid-body state {what}"


def _steps(hs, case, slot, steps, what=""):
    for i in range(steps):
        want = case.advance()
        case.submit(hs, slot)
        assert hs.wait(slot) is case.bufs
        case.check_step(want, f"{what} step {i}", first=case.k == 1)


@pytest.mark.parametrize("out", ["host_obs", "device_out"])
@pytest.mark.parametrize("mode", ["direct", "staged", "pageable"])
def test_power_step_each_slot_eight_steps_deep(mode, out, monkeypatch):
    _set_path(monkeypatch, "staged" if mode == "staged" else "direct")
    data, mlib = _motion_lib()
    case = Case(data, mlib, 2005, 11, pinned=mode != "pageable", host_obs=out == "host_obs")
    with case.host_step(mlib) as hs:
        for slot in (0, 1):
            _steps(hs, case, slot, 8, f"{mode} {out} slot {slot}")
        assert hs.path == (1 if mode == "direct" else 2)


@pytest.mark.parametrize("out", ["host_obs", "device_out"])
@pytest.mark.parametrize("mode", ["direct", "staged"])
def test_two_slots_auto_reset_waited_out_of_order(mode, out, monkeypatch):
    """Different initial states on the two slots; each slot carries its own batch, eight steps deep."""
    _set_path(monkeypatch, mode)
    data, mlib = _motion_lib()
    a = Case(data, mlib, 3001, 21, auto_reset=True, state_init="hybrid", host_obs=out == "host_obs")
    b = Case(data, mlib, 2003, 31, auto_reset=True, state_init="default", host_obs=out == "host_obs")
    with HostStep(mlib, 3001, num_chunks=3, use_power_reward=True, rew_power_coef=COEF) as hs:
        a.set_initial_state(hs, 0)
        b.set_initial_state(hs, 1)
        for r in range(8):
            wa, wb = a.advance(), b.advance()
            a.submit(hs, 0)
            b.submit(hs, 1)
            hs.wait(1)
            hs.wait(0)
            a.check_step(wa, f"A round {r}", first=r == 0)
            b.check_step(wb, f"B round {r}", first=r == 0)


@pytest.mark.parametrize("state_init", ["random", "default", "hybrid"])
@pytest.mark.parametrize("out", ["host_obs", "device_out"])
def test_auto_reset_state_init(state_init, out, monkeypatch):
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    case = Case(data, mlib, 2005, 41, auto_reset=True, state_init=state_init, host_obs=out == "host_obs")
    with case.host_step(mlib) as hs:
        case.set_initial_state(hs, 1)
        _steps(hs, case, 1, 4, f"{state_init} {out}")


@pytest.mark.parametrize("variant", ["T3", "generic"])
@pytest.mark.parametrize("mode", ["direct", "staged"])
def test_kernel_variants(variant, mode, monkeypatch):
    """T = 3 and the generic kernel: the step is followed by a separate reset launch (hybrid)."""
    _set_path(monkeypatch, mode)
    data, mlib = _motion_lib()
    T = 3 if variant == "T3" else 1
    case = Case(data, mlib, 1003, 51, T=T, auto_reset=True, state_init="hybrid", host_obs=mode == "direct")
    capi = _cabi.load()
    if variant == "generic":
        capi.phc_set_option(_cabi.OPT_FORCE_GENERIC_STEP, 1)
    try:
        with case.host_step(mlib) as hs:
            case.set_initial_state(hs, 0)
            _steps(hs, case, 0, 3, variant)
    finally:
        capi.phc_set_option(_cabi.OPT_FORCE_GENERIC_STEP, 0)


@pytest.mark.parametrize("mode", ["direct", "staged"])
def test_eval_mode_mpjpe(mode, monkeypatch):
    _set_path(monkeypatch, mode)
    data, mlib = _motion_lib()
    case = Case(data, mlib, 2005, 61, auto_reset=True, eval_mode=True)
    with case.host_step(mlib) as hs:
        _steps(hs, case, 0, 3, f"eval {mode}")


@pytest.mark.parametrize("mode", ["direct", "staged"])
def test_nan_dof_force(mode, monkeypatch):
    """One env with a NaN dof force: its reward is the device path's NaN (once past progress 3), every other env is
    bit-identical."""
    _set_path(monkeypatch, mode)
    data, mlib = _motion_lib()
    n = 1003
    case = Case(data, mlib, n, 71, nan_env=517)
    with case.host_step(mlib) as hs:
        _steps(hs, case, 0, 5, f"nan {mode}")
        assert torch.isnan(case.bufs.rew_buf[517]) and int(torch.isnan(case.bufs.rew_buf).sum()) == 1


@pytest.mark.parametrize("state_init", ["default", "hybrid"])
@pytest.mark.parametrize("out", ["host_obs", "device_out"])
@pytest.mark.parametrize("pinned", [True, False], ids=["pinned", "pageable"])
def test_masked_host_reset(state_init, out, pinned, monkeypatch):
    """Masked envs' obs rows, state and root / dof rows equal HumanoidPHC.reset(env_ids, phase, default_mask); other
    envs keep the sentinel."""
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    n = 2005
    case = Case(data, mlib, n, 81, pinned=pinned, host_obs=out == "host_obs", state_init=state_init)
    b, r = case.bufs, case.rb
    with case.host_step(mlib) as hs:
        case.set_initial_state(hs, 1)
        case.physics()  # a state that differs from any motion frame: a default-path env keeps it
        case.draw()
        mask = torch.rand(n, generator=case.gen) < 0.4
        ids = mask.nonzero().squeeze(1)
        r.env_mask.copy_(mask)
        case.poison()
        prog = b.progress_buf.clone()
        dm = r.default_mask.bool()[ids]
        case.env.reset(ids.to(DEV), r.phase[ids].to(DEV), dm.to(DEV) if state_init == "hybrid" else None)
        torch.cuda.synchronize()
        want = case.snapshot({})
        hs.reset_submit(1, b, r, state_init=state_init, device_out=case.dev)
        assert hs.wait(1) is b
        m = mask.to(case.obs().device)
        assert _same(case.obs()[m], want["obs"][mask.to(DEV)]) and bool((case.obs()[~m] == SENTINEL).all())
        assert _same(b.state, want["state"])
        assert int(b.progress_buf[mask].abs().max()) == 0 and torch.equal(b.progress_buf[~mask], prog[~mask])
        assert int(b.reset_buf[mask].max()) == 0 and int(b.reset_buf[~mask].min()) == 7
        for name, got in (("root", r.root_states), ("dofp", r.dof_pos), ("dofv", r.dof_vel)):
            assert _same(got[mask], want[name][mask]), name
            assert bool((got[~mask] == SENTINEL).all()), name
        defaults = mask & (r.default_mask.bool() if state_init == "hybrid" else torch.ones(n, dtype=torch.bool))
        assert 0 < int(defaults.sum()) and torch.equal(r.root_states[defaults], case.init[0][defaults])


# ---------------------------------------------------------------------------------------
# 3. error codes
# ---------------------------------------------------------------------------------------
def test_error_codes_enqueue_nothing(monkeypatch):
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    n = 1003
    case = Case(data, mlib, n, 101, auto_reset=True, state_init="hybrid", eval_mode=True)
    capi = _cabi.load()
    dev_force = torch.zeros(n, 69, device=DEV)
    dev_mpjpe = torch.zeros(n, device=DEV)
    dev_mask = torch.zeros(n, dtype=torch.uint8, device=DEV)
    with case.host_step(mlib) as hs:
        ctx = hs._ctx
        case.poison()
        args = case.bufs._args()

        def env(**fields):
            e = hs._env_args(0, case.bufs, None, "random", n)
            e.default_mask = case.rb.default_mask.data_ptr()
            for k, v in fields.items():
                setattr(e, k, v)
            return C.byref(e)

        def rargs(state_init="hybrid", **fields):
            r = case.rb._args(case.bufs, state_init, False)
            for k, v in fields.items():
                setattr(r, k, v)
            return C.byref(r)

        step_fn, reset_fn = capi.phc_host_step_submit_env, capi.phc_host_reset_submit_env
        for slot in (0, 1):
            # no initial state on the slot yet
            assert step_fn(ctx, slot, C.byref(args), rargs("default"), None, env(), n) == NULL
            assert reset_fn(ctx, slot, C.byref(args), rargs("hybrid"), None, env(), n) == NULL
            assert step_fn(ctx, slot, C.byref(args), rargs("default"), None, None, n) == NULL
            # the submits without options keep refusing default / hybrid
            assert capi.phc_host_step_submit_reset(ctx, slot, C.byref(args), rargs("default"), n) == UNSUPPORTED
            assert capi.phc_host_reset_submit(ctx, slot, C.byref(args), rargs("hybrid"), n) == UNSUPPORTED
            hs.set_initial_state(slot, *(t[: n - 1].contiguous() for t in case.init))
            assert step_fn(ctx, slot, C.byref(args), rargs("default"), None, env(), n) == SHAPE
            assert reset_fn(ctx, slot, C.byref(args), rargs("hybrid"), None, env(), n) == SHAPE
            case.set_initial_state(hs, slot)
            for fn in (step_fn, reset_fn):
                assert fn(ctx, slot, C.byref(args), rargs(), None, env(default_mask=None), n) == NULL
                assert fn(ctx, slot, C.byref(args), rargs(phase=None), None, env(), n) == NULL
                assert fn(ctx, slot, C.byref(args), rargs(), None, env(default_mask=dev_mask.data_ptr()), n) == UNSUPPORTED
                assert fn(ctx, slot, C.byref(args), rargs(), None, env(), -1 if fn is step_fn else n + 1) == SHAPE
            for r in (None, rargs()):
                assert step_fn(ctx, slot, C.byref(args), r, None, env(dof_vel=None), n) == NULL
                assert step_fn(ctx, slot, C.byref(args), r, None, env(dof_force=None), n) == NULL
                assert step_fn(ctx, slot, C.byref(args), r, None, env(dof_force=dev_force.data_ptr()), n) == UNSUPPORTED
                assert step_fn(ctx, slot, C.byref(args), r, None, env(mpjpe=dev_mpjpe.data_ptr()), n) == UNSUPPORTED
            assert capi.phc_host_step_wait(ctx, slot) == OK
        b = case.bufs
        assert bool(torch.isnan(b.rew_buf).all()) and bool(torch.isnan(b.mpjpe).all())
        assert bool((b.obs_buf == SENTINEL).all()) and bool((case.rb.root_states == SENTINEL).all())
        x = case.init[0]
        assert capi.phc_host_step_set_initial_state(ctx, 2, x.data_ptr(), x.data_ptr(), x.data_ptr(), 1) == SHAPE
        assert capi.phc_host_step_set_initial_state(ctx, 0, x.data_ptr(), x.data_ptr(), x.data_ptr(), n + 1) == SHAPE
        assert capi.phc_host_step_set_initial_state(ctx, 0, None, x.data_ptr(), x.data_ptr(), 1) == NULL
        assert capi.phc_host_step_set_initial_state(ctx, 0, dev_force.data_ptr(), x.data_ptr(), x.data_ptr(), 1) == UNSUPPORTED
        # busy: the slot in flight refuses a new initial state and both submits, then finishes as before
        want = case.advance()
        case.submit(hs, 0)
        i0 = case.init
        assert capi.phc_host_step_set_initial_state(ctx, 0, i0[0].data_ptr(), i0[1].data_ptr(), i0[2].data_ptr(), n) == BUSY
        assert step_fn(ctx, 0, C.byref(args), rargs(), None, env(), n) == BUSY
        assert reset_fn(ctx, 0, C.byref(args), rargs(), None, env(), n) == BUSY
        hs.wait(0)
        case.check_step(want, "after the errors")


def test_close_with_env_submits_in_flight(monkeypatch):
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    a = Case(data, mlib, 2005, 111, auto_reset=True, state_init="hybrid")
    b = Case(data, mlib, 1999, 121, pinned=False, host_obs=False, auto_reset=True, state_init="default")
    hs = HostStep(mlib, 2005, num_chunks=3, use_power_reward=True, rew_power_coef=COEF)
    a.set_initial_state(hs, 0)
    b.set_initial_state(hs, 1)
    wa, wb = a.advance(), b.advance()
    a.submit(hs, 0)
    b.submit(hs, 1)
    hs.close()
    a.check_step(wa, "close, slot 0")
    b.check_step(wb, "close, slot 1")
