"""GPU: the episode bookkeeping of the host step (phc_host_step_submit_episode, HostStep.submit(..., episode=)).

1. Against the oracle, per step: after every wait, oracle.episode_update on the flags, rewards and reward terms the host
   step returned gives the episode tensors bit for bit, over the direct / staged / pageable paths, host obs and device
   outputs, the power reward on and off, auto-reset with every state init, T = 1 and T = 10, several chunks and a ragged
   batch.
2. Against PHCPufferEnv(fused=True) over HumanoidPHC on the same inputs: the per-env tensors bit for bit; at T = 1 with a
   sums row per block the sums and the logged dict bit for bit for 1, 3 and 7 chunks; with 32 rows, and at T = 10,
   within 1e-12.
3. Two batches on two slots, waited out of order: HostEpisodeBuffers.log of both equals mean_and_log over the 2n envs.
4. A NaN reward in an env whose episode ends.
5. Ordering against the learner's stream; error codes; close() with episode submits in flight."""

import ctypes as C
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from humanoid_b200 import (HostDeviceOutputs, HostEpisodeBuffers, HostResetBuffers, HostStep, HostStepBuffers,
                               HumanoidPHC, MotionLib, PHCPufferEnv, RunningNorm, _cabi, synth)  # fmt: skip
    from oracle import phc_oracle as O

DEV = "cuda"
OK, NULL, SHAPE, UNSUPPORTED, BUSY = 0, -1, -2, -4, -8
COEF = 0.0005
EP_FIELDS = ("terminals", "truncations", "masks", "episode_returns", "episode_lengths")


def _same(a, b):
    """Bit equality (NaNs included) of two tensors, wherever they live."""
    a, b = a.detach().cpu(), b.detach().cpu()
    if a.dtype == torch.float32 and b.dtype == torch.float32:
        return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))
    if a.dtype == torch.float64 and b.dtype == torch.float64:
        return a.shape == b.shape and torch.equal(a.view(torch.int64), b.view(torch.int64))
    return a.shape == b.shape and torch.equal(a, b.to(a.dtype))


def _set_path(monkeypatch, path):
    if path in ("direct", "staged"):
        monkeypatch.setenv("PHC_HOST_PATH", path)
    else:
        monkeypatch.delenv("PHC_HOST_PATH", raising=False)


def _motion_lib(M=48, seed=1301):
    data = synth.make_motion_lib(M, 60, 90, seed=seed, device=DEV)
    return data, MotionLib(data, device=DEV)


def _inputs(data, mlib, n, seed):
    clock = synth.make_clock(data, n, seed=seed, ids="mod", aligned=True, max_progress=30)
    ref = mlib.get_motion_state(clock.sampled_motion_ids, synth.reward_time(clock, extra_steps=1), clock.global_offset)
    return clock, synth.make_sim_state(ref, seed=seed + 1)


class World:
    """The seeded physics of N envs, shared by every batch cut from them: each step pushes the rigid bodies (about 3 %
    of the envs far enough to terminate), draws dof force / velocity, reset phases and hybrid masks."""

    def __init__(self, data, mlib, N, seed, nan_env=None):
        self.clock, self.state = _inputs(data, mlib, N, seed)
        self.state = self.state.cpu()
        self.N, self.k, self.nan_env = N, 0, nan_env
        self.gen = torch.Generator().manual_seed(seed + 2)
        self.init = (torch.randn(N, 13, generator=self.gen), torch.randn(N, 69, generator=self.gen),
                     torch.randn(N, 69, generator=self.gen))  # fmt: skip

    def advance(self):
        N, k, g = self.N, self.k, self.gen
        d = torch.randn(N, 24, 3, generator=g) * 0.01
        d[(torch.arange(N) * 7 + k) % 29 == 0, :, 0] += 0.5
        force, vel = torch.randn(N, 69, generator=g) * 50, torch.randn(N, 69, generator=g)
        if self.nan_env is not None:
            force[self.nan_env, 5] = float("nan")
        self.k += 1
        return dict(push=d, force=force, vel=vel, phase=torch.rand(N, generator=g),
                    dmask=(torch.rand(N, generator=g) < 0.5).to(torch.uint8))  # fmt: skip


class Batch:
    """Envs [lo, lo + n) of a World on the host path, with episode buffers (and device outputs)."""

    def __init__(self, world, lo, n, T=1, power=False, pinned=True, device_out=False, reset=None, buckets=None,
                 rewards=True):  # fmt: skip
        self.lo, self.n, self.T, self.power, self.reset = lo, n, T, power, reset
        sl = slice(lo, lo + n)
        b = HostStepBuffers.allocate(n, T, pinned=pinned, host_obs=not device_out, power=power)
        for name in ("progress_buf", "motion_start_times", "motion_start_times_offset", "global_offset",
                     "sampled_motion_ids"):  # fmt: skip
            getattr(b, name).copy_(getattr(world.clock, name)[sl].cpu())
        b.state.copy_(world.state[sl])
        self.bufs = b
        self.rb = HostResetBuffers.allocate(n, pinned=pinned, hybrid=True) if reset else None
        self.dev = None
        if device_out:
            D = _cabi.SELF_OBS_DIM + _cabi.TASK_OBS_DIM * T
            rn = RunningNorm(D, device=DEV)
            rn.running_var.fill_(2.0)
            self.dev = HostDeviceOutputs.allocate(n, T, DEV, norm_dtype=torch.float32, normalizer=rn, moments=True)
        self.ep = HostEpisodeBuffers.allocate(n, 5 if power else 4, device=DEV, buckets=buckets, rewards=rewards)
        self.init = tuple(t[sl].contiguous() for t in world.init)
        self.want = dict(terminals=torch.zeros(n, dtype=torch.bool), truncations=torch.zeros(n, dtype=torch.bool),
                         masks=torch.ones(n, dtype=torch.bool), episode_returns=torch.zeros(n),
                         episode_lengths=torch.zeros(n, dtype=torch.int32), raw_rewards=torch.zeros(5 if power else 4),
                         stats=torch.zeros(4, dtype=torch.float64))  # fmt: skip

    def host_step(self, mlib, **kw):
        kw.setdefault("num_chunks", 3)
        hs = HostStep(mlib, self.n, time_steps=self.T, use_power_reward=self.power, rew_power_coef=COEF, **kw)
        if self.reset in ("default", "hybrid"):
            hs.set_initial_state(0, *self.init)
            hs.set_initial_state(1, *self.init)
        return hs

    def physics(self, p):
        sl = slice(self.lo, self.lo + self.n)
        self.bufs.state[..., 0:3] += p["push"][sl]
        if self.power:
            self.bufs.dof_force.copy_(p["force"][sl])
            self.bufs.dof_vel.copy_(p["vel"][sl])
        if self.rb is not None:
            self.rb.phase.copy_(p["phase"][sl])
            self.rb.default_mask.copy_(p["dmask"][sl])

    def submit(self, hs, slot, episode=True):
        hs.submit(slot, self.bufs, self.rb, state_init=self.reset or "random", device_out=self.dev,
                  episode=self.ep if episode else None)  # fmt: skip

    def oracle(self):
        """oracle.episode_update on what the host step returned (after its wait)."""
        b = self.bufs
        O.episode_update(self.want, b.reset_buf, b.terminate_buf, b.rew_buf, b.reward_raw)

    def check(self, what):
        torch.cuda.synchronize()
        for name in EP_FIELDS:
            assert _same(getattr(self.ep, name), self.want[name]), f"{name} {what}"
        if self.ep.rewards is not None:
            assert _same(self.ep.rewards, self.bufs.rew_buf), f"rewards {what}"


def _run(batch, hs, steps, world, slot=0):
    for i in range(steps):
        batch.physics(world.advance())
        batch.submit(hs, slot)
        hs.wait(slot)
        batch.oracle()
        batch.check(f"step {i}")


# ---------------------------------------------------------------------------------------
# 1. against the oracle, per step
# ---------------------------------------------------------------------------------------
ORACLE_CASES = [  # n, T, path, device_out, power, reset
    (4096, 1, "direct", False, False, None),
    (4096, 1, "direct", True, True, "random"),
    (4096, 1, "staged", False, True, "start"),
    (4096, 1, "pageable", True, False, "default"),
    (1000, 1, "direct", False, True, "hybrid"),
    (1000, 1, "staged", True, False, None),
    (1000, 1, "pageable", False, True, "random"),
    (4096, 1, "direct", True, False, "hybrid"),
    (1000, 10, "direct", False, True, None),
    (1000, 10, "direct", True, False, "random"),
    (1000, 10, "staged", False, False, "hybrid"),
    (1000, 10, "pageable", True, True, "default"),
]


@pytest.mark.parametrize("n, T, path, device_out, power, reset", ORACLE_CASES)
def test_sixteen_steps_against_the_oracle(n, T, path, device_out, power, reset, monkeypatch):
    _set_path(monkeypatch, path)
    data, mlib = _motion_lib()
    world = World(data, mlib, n, 1400 + n + T)
    batch = Batch(world, 0, n, T=T, power=power, pinned=path != "pageable", device_out=device_out, reset=reset)
    with batch.host_step(mlib) as hs:
        _run(batch, hs, 16, world)
    w = batch.want
    assert int(w["stats"][0]) > int(w["stats"][3]) and int(w["stats"][0]) > 0  # terminated episodes among them
    # the logged means: counts and lengths exact, returns and reward terms to fp32 rounding of the block sums
    (got,) = HostEpisodeBuffers.log([batch.ep], 16)
    from humanoid_b200.puffer_env import episode_info

    want, _ = episode_info(w["stats"], w["raw_rewards"], 16)
    assert set(got) == set(want) and len(got) == 3 + (5 if power else 4)
    assert got["episode_length"] == want["episode_length"] and got["truncated_rate"] == want["truncated_rate"]
    for key in want:
        assert math.isclose(got[key], want[key], rel_tol=1e-6, abs_tol=1e-7), key
    assert float(batch.ep.sums.abs().max()) == 0.0  # log zeroes the rows it folds


# ---------------------------------------------------------------------------------------
# 2. against PHCPufferEnv(fused=True) over HumanoidPHC
# ---------------------------------------------------------------------------------------
class Device:
    """The same N envs on the device path under PHCPufferEnv(fused=True) (auto-reset on, as the wrapper sets it)."""

    def __init__(self, mlib, world, T=1, power=False, state_init="random"):
        env = HumanoidPHC(mlib, world.N, device=DEV, time_steps=T, use_power_reward=power, rew_power_coef=COEF)
        env.set_sim_state(world.state.to(DEV))
        env.set_clock(world.clock)
        env.state_init = state_init
        for t, v in zip((env._initial_humanoid_root_states, env._initial_dof_pos, env._initial_dof_vel), world.init):
            t.copy_(v.to(DEV))
        self.env, self.power = env, power
        self.pe = PHCPufferEnv(env, log_interval=16, fused=True)

    def step(self, p):
        e = self.env
        e._rigid_body_state_reshaped[..., 0:3] += p["push"].to(DEV)
        if self.power:
            e.dof_force_tensor.copy_(p["force"].to(DEV))
            e._dof_vel.copy_(p["vel"].to(DEV))
        e.step(phase_by_env=p["phase"].to(DEV), default_mask_by_env=p["dmask"].to(DEV))


def _logs_equal(a, b):
    assert set(a) == set(b)
    for k in a:
        assert (math.isnan(a[k]) and math.isnan(b[k])) or a[k] == b[k], (k, a[k], b[k])


def _against_device(path, n, T, power, chunks, buckets, state_init, monkeypatch, steps=12):
    _set_path(monkeypatch, path)
    data, mlib = _motion_lib()
    world = World(data, mlib, n, 1500 + T)
    dev = Device(mlib, world, T, power, state_init)
    batch = Batch(world, 0, n, T=T, power=power, device_out=True, reset=state_init, buckets=buckets)
    with batch.host_step(mlib, num_chunks=chunks) as hs:
        for i in range(steps):
            p = world.advance()
            dev.step(p)
            batch.physics(p)
            batch.submit(hs, 0)
            hs.wait(0)
            torch.cuda.synchronize()
            for name in EP_FIELDS:
                assert _same(getattr(batch.ep, name), getattr(dev.pe, name)), f"{name} step {i}"
            assert _same(batch.ep.rewards, dev.pe._rew), f"rewards step {i}"
    return dev, batch


@pytest.mark.parametrize("chunks", [1, 3, 7])
@pytest.mark.parametrize("path", ["direct", "staged"])
def test_t1_sums_bit_identical_to_the_device_path_for_any_chunk_count(path, chunks, monkeypatch):
    dev, batch = _against_device(path, 4096, 1, True, chunks, None, "random", monkeypatch)
    assert batch.ep.sums.shape == dev.pe._ep_sums.shape
    assert _same(batch.ep.sums, dev.pe._ep_sums), "bucket rows"
    _logs_equal(HostEpisodeBuffers.log([batch.ep], 16)[0], dev.pe.mean_and_log()[0])


@pytest.mark.parametrize("T, buckets, power", [(1, 32, False), (10, None, True), (10, 32, False)])
def test_sums_within_fp64_rounding_of_the_device_path(T, buckets, power, monkeypatch):
    n = 4096 if T == 1 else 2048
    dev, batch = _against_device("direct", n, T, power, 3, buckets, "hybrid", monkeypatch)
    # the fp64 column sums (episodes, returns, lengths, truncations, reward terms) before the fold
    got_cols, want_cols = batch.ep.sums.sum(0).cpu(), dev.pe._ep_sums.sum(0).cpu()
    assert torch.allclose(got_cols, want_cols, rtol=1e-12, atol=0.0), (got_cols, want_cols)
    got, want = HostEpisodeBuffers.log([batch.ep], 16)[0], dev.pe.mean_and_log()[0]
    # the host path logs the columns of its reward_raw (4, or 5 with the power reward); HumanoidPHC's reward_raw always
    # has the power column, zero when the power reward is off
    assert set(got) == set(want) - ({"rew_power"} if not power else set())
    assert all(want[k] == 0.0 for k in set(want) - set(got))
    assert got["episode_length"] == want["episode_length"] and got["truncated_rate"] == want["truncated_rate"]
    for k in got:  # the reward-term means are fp32: the cast of equal-to-1e-12 sums may round one ulp apart
        assert math.isclose(got[k], want[k], rel_tol=1e-12 if k.startswith("episode") else 2.4e-7), (k, got[k], want[k])


# ---------------------------------------------------------------------------------------
# 3. two batches on two slots
# ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["direct", "staged"])
def test_two_slots_log_equals_one_batch_of_all_envs(path, monkeypatch):
    _set_path(monkeypatch, path)
    data, mlib = _motion_lib()
    n = 2048
    world = World(data, mlib, 2 * n, 1601)
    dev = Device(mlib, world, power=True)
    a = Batch(world, 0, n, power=True, device_out=True, reset="random")
    b = Batch(world, n, n, power=True, device_out=True, reset="random")
    with a.host_step(mlib, num_chunks=3) as hs:
        for i in range(10):
            p = world.advance()
            dev.step(p)
            a.physics(p)
            b.physics(p)
            a.submit(hs, 0)
            b.submit(hs, 1)
            first, second = (1, 0) if i % 2 else (0, 1)
            hs.wait(first)
            hs.wait(second)
            torch.cuda.synchronize()
            for name in EP_FIELDS:
                got = torch.cat([getattr(a.ep, name), getattr(b.ep, name)])
                assert _same(got, getattr(dev.pe, name)), f"{name} step {i}"
    got, want = HostEpisodeBuffers.log([a.ep, b.ep], 16)[0], dev.pe.mean_and_log()[0]
    assert len(got) == 8 and all(k in got for k in ("rew_body_pos", "rew_power"))
    _logs_equal(got, want)


# ---------------------------------------------------------------------------------------
# 4. a NaN reward
# ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["direct", "staged"])
def test_nan_reward_env_whose_episode_ends(path, monkeypatch):
    _set_path(monkeypatch, path)
    data, mlib = _motion_lib()
    n = 1000
    world = World(data, mlib, n, 1701)
    prog = world.clock.progress_buf.cpu()
    # an env the physics pushes over at the 4th step (k = 3) whose power term counts by then
    e = next(i for i in range(n) if (i * 7 + 3) % 29 == 0 and int(prog[i]) > 3)
    world.nan_env = e
    batch = Batch(world, 0, n, power=True, reset="random")
    with batch.host_step(mlib) as hs:
        _run(batch, hs, 5, world)
    w = batch.want
    assert math.isnan(float(w["stats"][1])), "the NaN return was logged"
    assert torch.isfinite(w["stats"][[0, 2, 3]]).all() and torch.isnan(w["raw_rewards"]).any()


# ---------------------------------------------------------------------------------------
# 5. ordering, errors, close
# ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["direct", "staged"])
def test_learner_stream_work_sees_the_previous_step(path, monkeypatch):
    _set_path(monkeypatch, path)
    data, mlib = _motion_lib()
    n = 2005
    world = World(data, mlib, n, 1801)
    batch = Batch(world, 0, n, device_out=True, reset="random")
    with batch.host_step(mlib) as hs:
        _run(batch, hs, 1, world)
        for i in range(3):
            prev = {k: getattr(batch.ep, k).cpu() for k in EP_FIELDS}
            batch.physics(world.advance())
            torch.cuda._sleep(200_000_000)  # ~0.1 s on the learner's (current) stream
            snap = {k: getattr(batch.ep, k).clone() for k in EP_FIELDS}
            batch.submit(hs, i % 2)
            hs.wait(i % 2)
            batch.oracle()
            for k in EP_FIELDS:
                assert _same(snap[k], prev[k]), f"{k} copied before the submit saw the new step"
            assert not _same(prev["terminals"], batch.want["terminals"]) or not _same(prev["episode_lengths"],
                                                                                       batch.want["episode_lengths"])
            side = torch.cuda.Stream()
            with torch.cuda.stream(side):
                seen = {k: getattr(batch.ep, k).clone() for k in EP_FIELDS}
            side.synchronize()
            for k in EP_FIELDS:
                assert _same(seen[k], batch.want[k]), f"{k} after wait, read on another stream"


def _poison(ep):
    ep.terminals.fill_(True)
    ep.truncations.fill_(True)
    ep.masks.fill_(False)
    ep.episode_returns.fill_(12345.0)
    ep.episode_lengths.fill_(777)
    ep.rewards.fill_(float("nan"))
    ep.sums.fill_(0.5)


def _poisoned(ep):
    torch.cuda.synchronize()
    return (bool(ep.terminals.all()) and bool(ep.truncations.all()) and not bool(ep.masks.any())
            and bool((ep.episode_returns == 12345.0).all()) and bool((ep.episode_lengths == 777).all())
            and bool(torch.isnan(ep.rewards).all()) and bool((ep.sums == 0.5).all()))  # fmt: skip


def test_error_codes_enqueue_nothing(monkeypatch):
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    n = 1003
    world = World(data, mlib, n, 1901)
    batch = Batch(world, 0, n, reset="random")
    other = HostEpisodeBuffers.allocate(n, 4, device=DEV)
    capi = _cabi.load()
    host = torch.zeros(n, 12, dtype=torch.float64).pin_memory()
    with batch.host_step(mlib) as hs:
        ctx = hs._ctx
        batch.physics(world.advance())
        _poison(batch.ep)
        batch.bufs.rew_buf.fill_(float("nan"))
        args = batch.bufs._args()
        rargs = batch.rb._args(batch.bufs, "random", False)

        def bad(**fields):
            a = batch.ep._args()
            for k, v in fields.items():
                setattr(a, k, v)
            return a

        cases = [(NULL, None)] + [(NULL, bad(**{f: None})) for f in EP_FIELDS + ("sums",)] + [
            (UNSUPPORTED, bad(terminals=host.data_ptr())), (UNSUPPORTED, bad(sums=host.data_ptr())),
            (UNSUPPORTED, bad(rewards=host.data_ptr())), (SHAPE, bad(buckets=0)), (SHAPE, bad(buckets=4097)),
        ]  # fmt: skip
        for slot in (0, 1):
            for r in (None, C.byref(rargs)):
                for code, a in cases:
                    rc = capi.phc_host_step_submit_episode(ctx, slot, C.byref(args), r, None, None,
                                                           None if a is None else C.byref(a), n)  # fmt: skip
                    assert rc == code, (code, rc)
                assert capi.phc_host_step_wait(ctx, slot) == OK
        assert _poisoned(batch.ep) and bool(torch.isnan(batch.bufs.rew_buf).all())
        # busy: a step in flight refuses a second episode submit on its slot, which writes nothing
        batch.ep.reset()
        for name in ("episode_returns", "episode_lengths"):
            getattr(batch.ep, name).zero_()
        batch.submit(hs, 0)
        _poison(other)
        assert capi.phc_host_step_submit_episode(ctx, 0, C.byref(args), None, None, None, C.byref(other._args()), n) == BUSY
        hs.wait(0)
        assert _poisoned(other)
        batch.oracle()
        batch.check("after the errors")
        batch.physics(world.advance())
        batch.submit(hs, 0)
        hs.wait(0)
        batch.oracle()
        batch.check("the next step")


def test_close_with_episode_submits_in_flight(monkeypatch):
    _set_path(monkeypatch, "direct")
    data, mlib = _motion_lib()
    wa, wb = World(data, mlib, 2005, 2001), World(data, mlib, 1999, 2011)
    a = Batch(wa, 0, 2005, power=True, reset="random")
    b = Batch(wb, 0, 1999, power=True, pinned=False, device_out=True)
    hs = a.host_step(mlib)
    a.physics(wa.advance())
    b.physics(wb.advance())
    a.submit(hs, 0)
    b.submit(hs, 1)
    hs.close()
    for x, what in ((a, "slot 0"), (b, "slot 1")):
        x.oracle()
        x.check(f"close, {what}")
