"""GPU: HumanoidPHC(obs_v=7) — the imitation observation v7 ([d_pos | d_vel | l_pos] per future step) written by the
fused step and the device reset.  Its rows must be the v6 rows' column subset bit for bit, every other output must equal
the v6 env's, and the fused rows must equal the per-function path's."""

import pytest
import torch

from conftest import assert_close

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from humanoid_b200 import HumanoidPHC, MotionLib, RunningNorm, _cabi, synth
    from humanoid_b200.puffer_env import PHCPufferEnv
    from oracle import phc_oracle as O
    from util_gpu import DEV, OBS_TOL, make_case_cpu

SCALAR_BUFFERS = ("rew_buf", "reward_raw", "reset_buf", "_terminate_buf", "progress_buf")
STATE_BUFFERS = ("_rigid_body_state_reshaped", "_humanoid_root_states", "_dof_state", "_motion_start_times",
                 "_motion_start_times_offset", "_global_offset")  # fmt: skip


def cuda(x):
    return x.to(DEV)


def v7_cols(T, selfw=358):
    """Columns of a v6 row that make the v7 row: the self obs, then [d_pos | d_vel | l_pos] of every future step."""
    return torch.cat([torch.arange(selfw), selfw + O.v7_columns(24, T)]).to(DEV)


def _case(N, T=1, seed=777, **env_kw):
    """make(obs_v) -> a fresh env over one library, sim state and clock; envs of both versions start identical."""

    def query(lib_data, ids, times, offset):
        return MotionLib(lib_data, device=DEV).get_motion_state(ids, times, offset)

    lib_data, clock, state = synth.make_case(N, 48, query, seed=seed, device=DEV, max_progress=30, max_frames=90)
    lib = MotionLib(lib_data, device=DEV)

    def make(obs_v, **kw):
        env = HumanoidPHC(lib, N, device=DEV, time_steps=T, obs_v=obs_v, **{**env_kw, **kw})
        env.set_sim_state(state)
        env.set_clock(clock)
        env._dof_state.copy_(torch.randn(env._dof_state.shape, generator=torch.Generator().manual_seed(3)).to(DEV))
        env._humanoid_root_states.fill_(0.5)
        env.dof_force_tensor.copy_(torch.randn(env.dof_force_tensor.shape, generator=torch.Generator().manual_seed(4)).to(DEV))
        return env

    return make


class _Generic:
    def __init__(self, on):
        self.on = on

    def __enter__(self):
        _cabi.load().phc_set_option(_cabi.OPT_FORCE_GENERIC_STEP, 1 if self.on else 0)

    def __exit__(self, *exc):
        _cabi.load().phc_set_option(_cabi.OPT_FORCE_GENERIC_STEP, 0)


def assert_v7_subset(e7, e6, tag="", extra=()):
    T = e7.time_steps
    selfw = e6.num_obs - 576 * T
    assert e7.num_obs == selfw + 216 * T
    assert torch.equal(e7.obs_buf, e6.obs_buf[:, v7_cols(T, selfw)]), f"{tag}: v7 rows are not the v6 subset"
    for name in SCALAR_BUFFERS + tuple(extra):
        assert torch.equal(getattr(e7, name), getattr(e6, name)), f"{tag}: {name}"


# ---------------------------------------------------------------------------------------------------------------
# v7 == the v6 subset, on every kernel v7 can take
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,T,mode", [(4096, 1, "fast"), (1029, 1, "fast"), (1030, 1, "fast"), (3, 1, "fast"),
                                      (12288, 1, "fast"), (1000, 1, "generic"), (515, 3, "fast"), (300, 10, "fast"),
                                      (777, 1, "strided_obs"), (777, 2, "strided_sim")])  # fmt: skip
def test_v7_rows_are_the_v6_columns_bitwise(N, T, mode):
    """1029 / 1030 envs leave tail blocks of one and two envs (float2 stores / bulk store); at 12288 envs the v6 step
    runs the persistent kernel and v7 the single-wave one; T > 1 and strided views take the generic kernel."""
    make = _case(N, T, seed=401 + N)
    e6, e7 = make(6), make(7)
    for e in (e6, e7):
        if mode == "strided_obs":  # rows of a wider tensor: every row ends 6 floats before the next begins
            wide = torch.full((N, e.num_obs + 6), 7.0, device=DEV)
            e.obs_buf = wide[:, : e.num_obs]
            e._wide = wide
        if mode == "strided_sim":  # 16 floats per body: the views are not one AoS-13 tensor
            st = torch.zeros((N, 24, 16), device=DEV)
            st[..., :13] = e._rigid_body_state_reshaped
            e.set_sim_state(st[..., :13], copy=False)
            e._st = st
    with _Generic(mode == "generic"):
        for k in range(3):
            e6.step()
            e7.step()
            torch.cuda.synchronize()
            assert_v7_subset(e7, e6, f"step {k}")
            for e in (e6, e7):
                e.reset_done(cuda(torch.rand(N, generator=torch.Generator().manual_seed(k))))
            assert_v7_subset(e7, e6, f"reset_done {k}", STATE_BUFFERS)
    if mode == "strided_obs":
        assert bool((e7._wide[:, e7.num_obs :] == 7.0).all()), "columns past the row were written"
    if N > 100:
        assert 0 < int(e6._reset_out.sum()) < N


# ---------------------------------------------------------------------------------------------------------------
# fused == per-function path, every self-obs flag set
# ---------------------------------------------------------------------------------------------------------------
FLAG_SETS = [(True, True, True), (False, True, True), (True, False, True), (True, True, False), (False, False, False)]


@pytest.mark.parametrize("flags", FLAG_SETS, ids=lambda f: "local%d_height%d_upright%d" % tuple(map(int, f)))
@pytest.mark.parametrize("kernel", ["fast", "generic", "reset_in_step"])
def test_v7_fused_equals_the_per_function_path(flags, kernel):
    local, height, upright = flags
    N = 1030
    make = _case(N, 1, seed=313, local_root_obs=local, root_height_obs=height, has_upright_start=upright)
    env, ref = make(7), make(7)
    assert env.num_obs == 574 - (0 if height else 1)
    with _Generic(kernel == "generic"):
        if kernel == "reset_in_step":
            env.enable_auto_reset(True)
            phase = cuda(torch.rand(N, generator=torch.Generator().manual_seed(1)))
            env.step(phase_by_env=phase)
            ref.step()
            ref.reset_done(phase)
        else:
            env.step()
            ref.post_physics_step_unfused()
    assert torch.equal(env.obs_buf, ref.obs_buf), "fused rows differ from the per-function / two-launch rows"
    assert torch.equal(env.rew_buf, ref.rew_buf) and torch.equal(env.progress_buf, ref.progress_buf)
    if kernel != "reset_in_step":
        assert torch.equal(env.reward_raw[:, :4], ref.reward_raw[:, :4])
        assert torch.equal(env.reset_buf, ref.reset_buf) and torch.equal(env._terminate_buf, ref._terminate_buf)


# ---------------------------------------------------------------------------------------------------------------
# the per-step options on the v7 single-wave kernel
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("option", ["power", "eval", "res_action", "all"])
def test_v7_options_equal_the_v6_env(option):
    N = 2050
    kw = {}
    if option in ("power", "all"):
        kw["use_power_reward"] = True
    if option in ("res_action", "all"):
        kw["res_action"] = True
    make = _case(N, 1, seed=52, **kw)
    e6, e7 = make(6), make(7)
    rew6, rew7 = torch.zeros(N, device=DEV), torch.zeros(N, device=DEV)
    e6.set_reward_copy(rew6)
    e7.set_reward_copy(rew7)
    for e in (e6, e7):
        if option in ("eval", "all"):
            e.flag_im_eval = True
            e.set_termination_distances(0.1)
    for k in range(3):
        e6.step()
        e7.step()
        extra = ("ref_dof_pos",) if "res_action" in kw else ()
        assert_v7_subset(e7, e6, f"{option} step {k}", extra)
        assert torch.equal(rew6, rew7)
        if option in ("eval", "all"):
            assert torch.equal(e7.extras["mpjpe"], e6.extras["mpjpe"])
        for e in (e6, e7):
            e.reset_done(cuda(torch.rand(N, generator=torch.Generator().manual_seed(k))))
    if "use_power_reward" in kw:
        assert bool((e7.reward_raw[:, 4] != 0).any())


def test_v7_puffer_bookkeeping_equals_the_v6_env():
    N = 4100
    make = _case(N, 1, seed=61)
    p6, p7 = PHCPufferEnv(make(6), fused=True, log_interval=4), PHCPufferEnv(make(7), fused=True, log_interval=4)
    for p in (p6, p7):
        torch.manual_seed(0)  # reset() draws its start times with torch.rand: the same ones for both
        p.reset()
    gen = torch.Generator().manual_seed(8)
    state = p6.env._rigid_body_state_reshaped.clone()
    for k in range(8):
        act = cuda(torch.rand(N, 69, generator=gen) * 2 - 1)
        phase = cuda(torch.rand(N, generator=gen))
        outs = []
        for p in (p6, p7):
            p.env.set_sim_state(state)
            outs.append(p.step(act, phase_by_env=phase))
        (o6, r6, t6, tr6, i6), (o7, r7, t7, tr7, i7) = outs
        assert torch.equal(o7, o6[:, v7_cols(1)]), f"step {k}: observations"
        assert torch.equal(r6, r7) and torch.equal(t6, t7) and torch.equal(tr6, tr7)
        for name in ("masks", "episode_returns", "episode_lengths", "actions"):
            assert torch.equal(getattr(p6, name), getattr(p7, name)), f"step {k}: {name}"
        assert repr(i6) == repr(i7), f"step {k}: logged means"
        assert_v7_subset(p7.env, p6.env, f"step {k}", STATE_BUFFERS)
    assert int(p6.env._reset_out.sum()) > 0


@pytest.mark.parametrize("generic", [False, True], ids=["fast", "generic"])
def test_v7_moments_are_the_column_moments_of_the_rows_written(generic):
    N = 3001
    make = _case(N, 1, seed=207)
    env = make(7, obs_moments=True)
    want = torch.zeros(2 * env.num_obs, dtype=torch.float64, device=DEV)
    with _Generic(generic):
        for k in range(2):
            env.step()
            x = env.obs_buf.double()
            want[: env.num_obs] += x.sum(0)
            want[env.num_obs :] += (x * x).sum(0)
    sums, rows = env.take_obs_moments()
    assert rows == 2 * N and sums.shape == (2 * 574,)
    rel = ((sums - want).abs() / want.abs().clamp_min(1.0)).max()
    assert float(rel) < 1e-11


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("auto", [True, False], ids=["reset_in_step", "reset_done"])
def test_v7_normaliser_and_moments_follow_the_rows_the_policy_saw(auto, dtype):
    """v7 with obs_norm runs on the generic kernel (+ the reset kernel): obs_norm_buf == rn(obs_buf) of the FINAL rows
    and the moments (modes 1 and 2) are those of every row the policy saw."""
    N = 2052
    env = _case(N, 1, seed=991)(7, obs_moments=True)
    rn = RunningNorm(env.num_obs, device=DEV)
    rn.running_mean.normal_(generator=torch.Generator(device=DEV).manual_seed(1))
    rn.running_var.uniform_(0.5, 2.0, generator=torch.Generator(device=DEV).manual_seed(2))
    env.set_obs_normalizer(rn, dtype=dtype)
    env.enable_auto_reset(auto)
    gen = torch.Generator().manual_seed(6)
    env.reset(phase=cuda(torch.rand(N, generator=gen)))
    want = torch.zeros(2 * env.num_obs, dtype=torch.float64, device=DEV)
    rows = 0
    state = env._rigid_body_state_reshaped.clone()

    def check(tag):
        nonlocal rows
        x = env.obs_buf.double()
        want[: env.num_obs] += x.sum(0)
        want[env.num_obs :] += (x * x).sum(0)
        rows += N
        ref = rn(env.obs_buf)
        if dtype == torch.bfloat16:
            assert torch.equal(env.obs_norm_buf, ref.to(torch.bfloat16)) or (
                (env.obs_norm_buf.float() - ref).abs().max() <= 0.0626), tag
        else:
            assert_close(env.obs_norm_buf, ref, what=f"obs_norm_buf {tag}", rtol=1e-6, atol=1e-6)

    check("after reset()")
    flagged = 0
    for k in range(3):
        env.set_sim_state(state)
        phase = cuda(torch.rand(N, generator=gen))
        if auto:
            env.step(phase_by_env=phase)
        else:
            env.step()
            env.reset_done(phase)
        flagged += int(env._reset_out.sum())
        check(f"after step {k}")
    assert flagged > 0
    sums, got_rows = env.take_obs_moments()
    assert got_rows == rows
    assert float(((sums - want).abs() / want.abs().clamp_min(1.0)).max()) < 1e-11


# ---------------------------------------------------------------------------------------------------------------
# resets
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,T,mode", [(4096, 1, "fast"), (1029, 1, "fast_res_action"), (1000, 1, "generic"),
                                      (515, 3, "fast"), (700, 1, "fast_hybrid")])  # fmt: skip
def test_v7_reset_inside_the_step_equals_step_then_reset_bitwise(N, T, mode):
    kw = dict(res_action=True) if "res_action" in mode else {}
    make = _case(N, T, seed=777, **kw)
    a, b, c = make(7), make(7), make(6)
    b.enable_auto_reset(True)
    c.enable_auto_reset(True)
    gen = torch.Generator().manual_seed(4)
    with _Generic(mode == "generic"):
        for k in range(3):
            phase = cuda(torch.rand(N, generator=gen))
            dmask = cuda(torch.rand(N, generator=gen) < 0.5) if "hybrid" in mode else None
            for e in (a, b, c):
                if "hybrid" in mode:
                    e.state_init = "hybrid"
            a.step()
            flags = (a.reset_buf.clone(), a._terminate_buf.clone())
            a.reset_done(phase, dmask)
            b.step(phase_by_env=phase, default_mask_by_env=dmask)
            c.step(phase_by_env=phase, default_mask_by_env=dmask)
            torch.cuda.synchronize()
            assert 0 < int(flags[0].sum()) < N
            for name in ("obs_buf",) + SCALAR_BUFFERS + STATE_BUFFERS:
                assert torch.equal(getattr(a, name), getattr(b, name)), f"step {k}: {name}"
            assert torch.equal(b.extras["reset"], flags[0]) and torch.equal(b.extras["terminate"], flags[1])
            assert_v7_subset(b, c, f"step {k} vs v6", STATE_BUFFERS + (("ref_dof_pos",) if kw else ()))


@pytest.mark.parametrize("state_init", ["random", "start", "default", "hybrid"])
@pytest.mark.parametrize("T", [1, 3])
def test_v7_reset_env_ids_equals_the_v6_subset(state_init, T):
    N = 1500
    make = _case(N, T, seed=123, res_action=True)
    e6, e7 = make(6, obs_moments=True), make(7, obs_moments=True)
    ids = cuda(torch.randperm(N, generator=torch.Generator().manual_seed(5))[:611])
    phase = cuda(torch.rand(611, generator=torch.Generator().manual_seed(6)))
    dmask = cuda(torch.rand(611, generator=torch.Generator().manual_seed(7)) < 0.5)
    for e in (e6, e7):
        e.state_init = state_init
        e._initial_humanoid_root_states.normal_(generator=torch.Generator(device=DEV).manual_seed(8))
        e._initial_dof_pos.normal_(generator=torch.Generator(device=DEV).manual_seed(9))
        e._initial_dof_vel.normal_(generator=torch.Generator(device=DEV).manual_seed(10))
        e.step()
        e.reset(ids, phase=phase, default_mask=dmask if state_init == "hybrid" else None)
    assert_v7_subset(e7, e6, state_init, STATE_BUFFERS + ("ref_dof_pos",))
    # the moments gained the rows reset() rewrote (mode 1): the step's rows plus the reset rows, in fp64 adds whose
    # order the atomics choose
    s6, _ = e6.take_obs_moments()
    s7, _ = e7.take_obs_moments()
    W6 = e6.num_obs
    cols = v7_cols(T)
    want = torch.cat([s6[:W6][cols], s6[W6:][cols]])
    assert float(((s7 - want).abs() / want.abs().clamp_min(1.0)).max()) < 1e-12


def test_v7_rollout_with_auto_reset_replays_in_a_cuda_graph():
    N = 2048
    make = _case(N, 1, seed=205)
    eager, env = make(7), make(7)
    for e in (eager, env):
        e.enable_auto_reset(True)
    phases = cuda(torch.rand(16, N, generator=torch.Generator().manual_seed(11)))
    eager.step(phase_by_env=phases[0])  # the same warm-up step on both
    env.step(phase_by_env=phases[0])
    outs = []
    for k in range(16):
        eager.step(phase_by_env=phases[k])
        outs.append([eager.obs_buf.clone(), eager.rew_buf.clone(), eager._reset_out.clone()])
    phase = phases[0].clone()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        with torch.cuda.graph(graph, stream=stream):
            env.step(phase_by_env=phase)
    torch.cuda.synchronize()
    flagged = 0
    for k in range(16):
        phase.copy_(phases[k])
        graph.replay()
        torch.cuda.synchronize()
        o, r, f = outs[k]
        assert torch.equal(env.obs_buf, o) and torch.equal(env.rew_buf, r) and torch.equal(env._reset_out, f), k
        flagged += int(f.sum())
    for name in SCALAR_BUFFERS + STATE_BUFFERS:
        assert torch.equal(getattr(env, name), getattr(eager, name)), name
    assert flagged > 0


# ---------------------------------------------------------------------------------------------------------------
# against the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [1, 3, 10])
def test_v7_step_vs_oracle(T):
    N = 777
    lib_data, clock, state = make_case_cpu(num_envs=N, num_motions=50, seed=110 + T, max_progress=30)
    prog = clock.progress_buf.clone()
    want = O.step(O.OracleMotionLib(lib_data), state, prog, clock.motion_start_times, clock.motion_start_times_offset,
                  clock.global_offset, clock.sampled_motion_ids, torch.full((24,), 0.25), synth.SIM_DT, time_steps=T)  # fmt: skip
    env = HumanoidPHC(MotionLib(lib_data, device=DEV), N, device=DEV, time_steps=T, obs_v=7)
    env.set_sim_state(cuda(state))
    env.set_clock(clock.to(DEV))
    env.step()
    torch.cuda.synchronize()
    obs = env.obs_buf.cpu()
    assert torch.equal(env.progress_buf.cpu(), prog)
    assert torch.equal(env.reset_buf.cpu(), want[3]) and torch.equal(env._terminate_buf.cpu(), want[4])
    assert_close(env.rew_buf, want[1], what="reward", **OBS_TOL)
    assert_close(obs[:, :358], want[0][:, :358], what="self obs", **OBS_TOL)
    # [N, 216 T]: three 24-body 3-vector groups per step, the groups natural_scale gives a width of 216 k (k != 4 j)
    assert_close(obs[:, 358:], want[0][:, 358 + O.v7_columns(24, T)], what="v7 task obs", **OBS_TOL)


def test_v7_error_codes_through_the_env():
    N = 64
    env = _case(N, 1, seed=3)(7)
    a = env._build_step_args(True)
    lib = _cabi.load()
    import ctypes as C

    a.obs_stride = 573
    assert lib.phc_step_fused(env._motion_lib.handle, C.byref(a), N, _cabi.stream_ptr(env.device)) == -2
    a.obs_stride = 574
    r = env._fill_reset_args(None, None)
    r.obs_flags &= ~_cabi.OBS_TASK_V7
    a.auto_reset = C.pointer(r)
    assert lib.phc_step_fused(env._motion_lib.handle, C.byref(a), N, _cabi.stream_ptr(env.device)) == -2
    torch.cuda.synchronize()
