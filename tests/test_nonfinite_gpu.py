"""GPU: every kernel path on non-finite and degenerate inputs against the oracle, and the RunningNorm kernels at layout
edges against fp64 and IEEE fp32.

A diverged physics step or policy puts NaN, ±inf, zero quaternions or overflowing velocities into the sim state, and a
constant observation column drives var + eps to zero.  The kernels must then give what the reference gives: NaN and
±inf propagate per env, flags follow the reference's comparisons (a NaN distance compares false), and an env next to a
poisoned one in the same block is bit-identical to the same step without the poison."""

import contextlib
import math

import numpy as np
import pytest
import torch

from conftest import assert_equal_exact
from util_cpu import assert_close_strict, poison

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from humanoid_b200 import (
        HumanoidPHC,
        MotionLib,
        PHCPufferEnv,
        RunningNorm,
        _cabi,
        build_amp_observations_smpl,
        compute_humanoid_im_reset,
        compute_humanoid_observations_smpl_max,
        compute_imitation_observations_v6,
        compute_imitation_observations_v7,
        compute_imitation_reward,
        dof_subset_smpl,
        synth,
    )
    from oracle import phc_oracle as O
    from util_gpu import DEV, OBS_TOL, make_case_cpu, oracle_step

NAN, INF = float("nan"), float("inf")
STEP_OUT = ("obs_buf", "rew_buf", "reward_raw", "reset_buf", "_terminate_buf", "progress_buf")


def cuda(x):
    return x.to(DEV)


def _same(x, y):
    """Bit for bit, NaN where NaN."""
    x, y = x.cpu(), y.cpu()
    if x.shape != y.shape or x.dtype != y.dtype:
        return False
    if not x.is_floating_point():
        return torch.equal(x, y)
    return torch.equal(x.isnan(), y.isnan()) and torch.equal(torch.where(x.isnan(), 0, x), torch.where(y.isnan(), 0, y))


_DEFAULTS = dict(FORCE_GENERIC_STEP=0, STEP_PERSIST=1, MULTI_GROUPS=0)


@contextlib.contextmanager
def _options(**kw):
    capi = _cabi.load()
    try:
        for k, v in kw.items():
            assert capi.phc_set_option(getattr(_cabi, "OPT_" + k), v) == 0
        yield
    finally:
        for k in kw:
            capi.phc_set_option(getattr(_cabi, "OPT_" + k), _DEFAULTS[k])


def _case(N, seed=501, ended=False):
    """A seeded case, its clean sim tensors and a poisoned copy.  ``ended``: every other poisoned env sits at the end
    of its clip, so that pass_time flags it and a reset rewrites it."""
    lib_data, clock, state = make_case_cpu(num_envs=N, num_motions=max(4, min(64, N // 8)), seed=seed, max_progress=30)
    g = torch.Generator().manual_seed(seed)
    sim = dict(state=state, dof_force=torch.randn(N, 69, generator=g) * 40, dof_vel=torch.randn(N, 69, generator=g) * 3,
               dof_pos=torch.randn(N, 69, generator=g))  # fmt: skip
    bad, at = poison(sim, N)
    if ended:
        ids = torch.tensor(list(at.values())[::2])
        clock = clock.clone()
        clock.motion_start_times[ids] = lib_data.motion_lengths[clock.sampled_motion_ids[ids]]
        clock.motion_start_times_offset[ids] = 0.0
    return lib_data, clock, sim, bad, at


def _env(lib, clock, sim, T=1, **kw):
    env = HumanoidPHC(lib, sim["state"].shape[0], device=DEV, time_steps=T, use_power_reward=True, **kw)
    env.set_sim_state(cuda(sim["state"]))
    env.set_clock(clock.to(DEV))
    env.dof_force_tensor.copy_(cuda(sim["dof_force"]))
    env._dof_vel.copy_(cuda(sim["dof_vel"]))
    env._dof_pos.copy_(cuda(sim["dof_pos"]))
    return env


def _clean_mask(N, at):
    keep = torch.ones(N, dtype=torch.bool)
    keep[list(at.values())] = False
    return keep


# The kernels' heading rotations keep only the terms a heading quaternion (0, 0, z, w) leaves: the rotated z is the
# input's z, and the rotated x / y mix only x and y.  The reference's full quaternion rotation also multiplies the
# heading's zero x and y by every component, so a NaN or an infinity in one component of a position or velocity turns
# the other rotated components NaN as well (0 * NaN, 0 * inf).  DESIGN.md names this known exception: in these envs the
# kernels' NaN entries must be a subset of the reference's, and the rest is compared as usual.
HEADING_ZERO_TERMS = ("nan_body_pos", "nan_root_pos", "inf_body_vel", "neg_inf_ang_vel")


def _assert_obs(got, want, at, what):
    got, want = got.detach().cpu().double(), want.detach().cpu().double().clone()
    for name in HEADING_ZERO_TERMS:
        e = at[name]
        assert not (torch.isnan(got[e]) & ~torch.isnan(want[e])).any(), f"{what}: NaN in env {e} where the reference has none"
        extra = torch.isnan(want[e]) & ~torch.isnan(got[e])
        want[e] = torch.where(extra, got[e], want[e])
    assert_close_strict(got, want, what=what, **OBS_TOL)


def _ieee_forward(mean, var, x, eps, clip):
    """RunningNorm.forward as the fp32 op sequence with IEEE division and square root (numpy float32).  torch's CPU
    division by the broadcast sqrt is not always the correctly rounded quotient, so it is not the bitwise yardstick."""
    f = lambda t: t.detach().cpu().numpy()  # noqa: E731
    with np.errstate(all="ignore"):
        y = np.clip((f(x) - f(mean)) / np.sqrt(f(var) + np.float32(eps)), np.float32(-clip), np.float32(clip))
    return torch.from_numpy(y)


def _assert_moments(sums, rows, what):
    """fp64 partials against the fp64 column sums of the rows: NaN / ±inf columns exactly where the sums have them,
    finite columns to 1e-12 relative."""
    x = rows.detach().cpu().double()
    want = torch.cat([x.sum(0), (x * x).sum(0)])
    assert_close_strict(sums, want, what=what, rtol=1e-12, atol=1e-12, scale=None)


# ---------------------------------------------------------------------------------------
# the fused step on every kernel
# ---------------------------------------------------------------------------------------
PATHS = {
    "fast": (4099, 1, {}),
    "generic": (1030, 1, dict(FORCE_GENERIC_STEP=1)),
    "persist": (10243, 1, dict(STEP_PERSIST=2)),
    "multi_T3_one_group": (515, 3, dict(MULTI_GROUPS=1)),
    "multi_T3_two_groups": (515, 3, dict(MULTI_GROUPS=2)),
    "multi_T10_one_group": (130, 10, dict(MULTI_GROUPS=1)),
    "multi_T10_two_groups": (130, 10, dict(MULTI_GROUPS=2)),
}


@pytest.mark.parametrize("path", list(PATHS))
def test_poisoned_step_vs_oracle_and_clean_envs_bit_identical(path):
    N, T, opts = PATHS[path]
    lib_data, clock, sim, bad, at = _case(N)
    obs, rew, raw, reset, term, prog = oracle_step(lib_data, clock, bad["state"], time_steps=T, dof_force=bad["dof_force"],
                                                   dof_vel=bad["dof_vel"])  # fmt: skip
    lib = MotionLib(lib_data, device=DEV)
    with _options(**opts):
        a, b = _env(lib, clock, sim, T, obs_moments=True), _env(lib, clock, bad, T, obs_moments=True)
        a.step()
        b.step()
        torch.cuda.synchronize()
    assert (~torch.isfinite(obs[at["nan_root_rot"]])).any() and torch.isnan(rew[at["nan_body_pos"]])
    _assert_obs(b.obs_buf, obs, at, f"{path}: obs")
    assert_close_strict(b.rew_buf, rew, what=f"{path}: reward", **OBS_TOL)
    assert_close_strict(b.reward_raw, raw, what=f"{path}: reward_raw", **OBS_TOL)
    assert_equal_exact(b.reset_buf, reset, f"{path}: reset")
    assert_equal_exact(b._terminate_buf, term, f"{path}: terminate")
    assert_equal_exact(b.progress_buf, prog, f"{path}: progress")
    keep = _clean_mask(N, at)
    for k in STEP_OUT:
        assert _same(getattr(a, k)[cuda(keep)], getattr(b, k)[cuda(keep)]), f"{path}: {k} of a clean env changed"
    sums, rows = b.take_obs_moments()
    assert rows == N
    _assert_moments(sums, b.obs_buf, f"{path}: moments")


# ---------------------------------------------------------------------------------------
# RunningNorm.forward fused into the step, in every epilogue form
# ---------------------------------------------------------------------------------------
def _poisoned_normaliser(W, clean_obs):
    """epsilon = 0, and columns whose statistics are what a NaN row or a constant column leaves behind."""
    rn = RunningNorm(W, epsilon=0.0, device=DEV)
    g = torch.Generator().manual_seed(7)
    mean, var = torch.randn(1, W, generator=g) * 0.3, torch.rand(1, W, generator=g) * 2 + 1e-3
    var[0, 10] = 0.0  # var + eps == 0: ±clip where x != mean ...
    var[0, 11], mean[0, 11] = 0.0, float(clean_obs[1, 11])  # ... and 0 / 0 = NaN where x == mean
    var[0, 12] = 1e-40  # subnormal var + eps
    var[0, 13], mean[0, 13] = 1e-45, float(clean_obs[2, 13])
    var[0, 14] = INF
    var[0, 15] = NAN
    mean[0, 16] = NAN
    mean[0, 17] = INF
    var[0, W - 1] = 0.0
    rn.running_mean.copy_(mean)
    rn.running_var.copy_(var)
    return rn


NORM_FORMS = {  # fast, T = 1, N = 4099: full blocks in place (fp32) / staged (bf16), the partial last block scattered
    "fast_fp32": (4099, 1, {}, torch.float32),
    "fast_bf16": (4099, 1, {}, torch.bfloat16),
    "generic_fp32": (1030, 1, dict(FORCE_GENERIC_STEP=1), torch.float32),
    "generic_bf16": (1030, 1, dict(FORCE_GENERIC_STEP=1), torch.bfloat16),
    "multi_T3_fp32": (515, 3, {}, torch.float32),
}


@pytest.mark.parametrize("form", list(NORM_FORMS))
def test_poisoned_rows_and_statistics_through_the_fused_normaliser(form):
    N, T, opts, dtype = NORM_FORMS[form]
    lib_data, clock, sim, bad, at = _case(N, seed=502)
    lib = MotionLib(lib_data, device=DEV)
    with _options(**opts):
        plain = _env(lib, clock, sim, T)
        plain.step()
        rn = _poisoned_normaliser(plain.num_obs, plain.obs_buf.cpu())
        envs = []
        for s, dt in ((sim, dtype), (bad, dtype), (bad, torch.float32)):
            e = _env(lib, clock, s, T)
            e.set_obs_normalizer(rn, dtype=dt)
            e.step()
            envs.append(e)
        torch.cuda.synchronize()
    a, b, b32 = envs
    assert torch.equal(a.obs_buf, plain.obs_buf)
    y = b.obs_norm_buf
    want = O.running_norm_forward(rn.running_mean.cpu(), rn.running_var.cpu(), b.obs_buf.cpu(), 0.0, rn.clip)
    assert torch.isnan(want[1, 11]) and float(want[2, 13]) == 0.0 and torch.isnan(want[:, 15]).all()
    assert int(torch.isnan(want[list(at.values())]).sum()) > 100
    if dtype == torch.float32:
        assert_close_strict(y, want, what=f"{form}: normalised rows", rtol=1e-5, atol=1e-6, scale=None)
    else:
        assert _same(y, b32.obs_norm_buf.to(torch.bfloat16)), f"{form}: bf16 rows = RN-even rounding of the fp32 rows"
        assert_close_strict(y.float(), want, what=f"{form}: bf16 normalised rows", rtol=2**-8, atol=1e-6, scale=None)
    keep = cuda(_clean_mask(N, at))
    assert _same(a.obs_norm_buf[keep], y[keep]), f"{form}: normalised rows of a clean env changed"


# ---------------------------------------------------------------------------------------
# resets with the normaliser on: the in-step auto-reset and reset_envs (reset_done)
# ---------------------------------------------------------------------------------------
ENV_BUFFERS = ("obs_buf", "rew_buf", "reward_raw", "_rigid_body_state_reshaped", "_humanoid_root_states", "_dof_state",
               "progress_buf", "reset_buf", "_terminate_buf", "_motion_start_times", "_motion_start_times_offset",
               "_global_offset", "obs_norm_buf")  # fmt: skip


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_poisoned_envs_through_resets_with_the_normaliser(dtype):
    N = 1029
    lib_data, clock, sim, bad, at = _case(N, seed=503, ended=True)
    ended = list(at.values())[::2]
    lib = MotionLib(lib_data, device=DEV)
    rn = RunningNorm(934, device=DEV)
    g = torch.Generator().manual_seed(8)
    rn.running_mean.copy_(torch.randn(1, 934, generator=g) * 0.3)
    rn.running_var.copy_(torch.rand(1, 934, generator=g) * 2 + 1e-3)
    rn.running_var[0, 20] = NAN
    a, b = _env(lib, clock, bad), _env(lib, clock, bad)
    for e in (a, b):
        e.set_obs_normalizer(rn, dtype=dtype)
    b.enable_auto_reset(True)
    phase = cuda(torch.rand(N, generator=g))
    a.step()
    flags = a.reset_buf.clone()
    a.reset_done(phase)
    b.step(phase_by_env=phase)
    torch.cuda.synchronize()
    assert bool(flags[ended].all())
    for name in ENV_BUFFERS:
        assert _same(getattr(a, name), getattr(b, name)), name
    assert torch.isfinite(b.obs_buf[ended]).all(), "the reset rewrites the rows of the poisoned envs it re-poses"
    assert not torch.isfinite(b.obs_buf[at["nan_root_pos"]]).all(), "a poisoned env that is not reset keeps its NaN"
    want = O.running_norm_forward(rn.running_mean.cpu(), rn.running_var.cpu(), b.obs_buf.cpu(), rn.epsilon, rn.clip)
    if dtype == torch.float32:
        assert_close_strict(b.obs_norm_buf, want, what="normalised rows after the reset", rtol=1e-5, atol=1e-6, scale=None)
    else:
        assert_close_strict(b.obs_norm_buf.float(), want, what="bf16 normalised rows after the reset", rtol=2**-8,
                            atol=1e-6, scale=None)  # fmt: skip


# ---------------------------------------------------------------------------------------
# the standalone per-function kernels
# ---------------------------------------------------------------------------------------
def test_per_function_kernels_on_the_poisoned_state():
    N = 1029
    lib_data, clock, sim, bad, at = _case(N, seed=504)
    st = bad["state"]
    pos, rot, vel, ang = synth.body_views(st)
    gp, gr, gv, ga = synth.body_views(cuda(st))
    t = synth.reward_time(clock, extra_steps=1)
    ref = O.OracleMotionLib(lib_data).get_motion_state(clock.sampled_motion_ids, t, clock.global_offset)
    rk = [ref[k] for k in ("rg_pos", "rb_rot", "body_vel", "body_ang_vel")]
    grk = [cuda(x) for x in rk]

    got = compute_humanoid_observations_smpl_max(gp, gr, gv, ga, None, None, True, True, True, False, False)
    want = O.self_obs_smpl_max(pos, rot, vel, ang, None, None, True, True, True, False, False)
    _assert_obs(got, want, at, "self obs")
    args = (gp[:, 0], gr[:, 0], gp, gr, gv, ga, *grk, 1, True)
    oargs = (pos[:, 0], rot[:, 0], pos, rot, vel, ang, *rk, 1, True)
    _assert_obs(compute_imitation_observations_v6(*args), O.imitation_obs_v6(*oargs), at, "v6")
    _assert_obs(compute_imitation_observations_v7(*args), O.imitation_obs_v7(*oargs), at, "v7")
    rew, raw = compute_imitation_reward(*args[:10], O.DEFAULT_RWD_SPECS)
    wrew, wraw = O.imitation_reward(*oargs[:10], O.DEFAULT_RWD_SPECS)
    assert_close_strict(rew, wrew, what="reward", **OBS_TOL)
    assert_close_strict(raw, wraw, what="reward_raw", **OBS_TOL)
    assert torch.isnan(wrew[at["nan_root_pos"]]) and float(wraw[at["vel_1e20"], 2]) == 0.0

    g = torch.Generator().manual_seed(9)
    prog = (clock.progress_buf + 1).to(torch.int16)
    pass_time = torch.rand(N, generator=g) < 0.2
    reset_buf = torch.ones(N, dtype=torch.bool)
    for use_mean in (False, True):
        thr = torch.full((24,), 0.25)
        got = compute_humanoid_im_reset(cuda(reset_buf), cuda(prog), None, None, gp, grk[0], cuda(pass_time), True,
                                        cuda(thr), use_mean)  # fmt: skip
        want = O.im_reset(reset_buf, prog, None, None, pos, rk[0], pass_time, True, thr, use_mean)
        assert_equal_exact(got[0], want[0], f"im_reset use_mean={use_mean}: reset")
        assert_equal_exact(got[1], want[1], f"im_reset use_mean={use_mean}: terminated")

    key = torch.tensor([4, 8, 18, 23])
    sub = dof_subset_smpl()
    dp, dv = bad["dof_pos"], bad["dof_vel"]
    got = build_amp_observations_smpl(gp[:, 0], gr[:, 0], gv[:, 0], ga[:, 0], cuda(dp), cuda(dv), gp[:, cuda(key)], None, None,
                                      cuda(sub), True, True, True, False, False, True)  # fmt: skip
    want = O.amp_obs_smpl(pos[:, 0], rot[:, 0], vel[:, 0], ang[:, 0], dp, dv, pos[:, key], None, None, sub, True, True, True,
                          False, False, True)  # fmt: skip
    # exp_map_to_quat keeps the angle only where |angle| > 1e-5, which a NaN angle fails: the reference turns a NaN
    # joint exp map into the identity rotation, and its AMP row stays finite; a NaN dof velocity is copied through
    assert torch.isfinite(want[at["nan_dof_pos"]]).all() and torch.isnan(want[at["nan_dof_vel"]]).any()
    _assert_obs(got, want, at, "AMP obs")


@pytest.mark.parametrize("res_action", [False, True])
def test_pd_targets_propagate_nan_bit_exact(res_action):
    lib = MotionLib(synth.make_motion_lib(4, 6, 9), device=DEV)
    n = 777
    env = HumanoidPHC(lib, n, device=DEV)
    g = torch.Generator().manual_seed(6)
    act = torch.randn(n, 69, generator=g).clamp(-1, 1)
    off, sc = torch.randn(69, generator=g), torch.rand(69, generator=g) * 3
    refp, dofp = torch.randn(n, 69, generator=g), torch.randn(n, 69, generator=g)
    act[3, 5], act[4, 7], act[5, 8] = NAN, INF, -INF
    dofp[6, 12], dofp[7, 13], refp[8, 14] = NAN, INF, NAN  # joints 4 (not frozen)
    env._pd_action_offset.copy_(off)
    env._pd_action_scale.copy_(sc)
    env._dof_pos.copy_(dofp)
    got = env._action_to_pd_targets(cuda(act), res_action=res_action, ref_dof_pos=cuda(refp), freeze_hand=True,
                                    freeze_toe=True)  # fmt: skip
    want = O.action_to_pd_targets(act, off, sc, res_action, refp, dofp, zero_joints=(3, 7, 17, 22))
    assert int(torch.isnan(want).sum()) >= (3 if res_action else 1)
    assert _same(got, want)


# ---------------------------------------------------------------------------------------
# RunningNorm kernels
# ---------------------------------------------------------------------------------------
def test_running_norm_forward_moments_and_update_on_non_finite_columns():
    """Columns: NaN, +inf, -inf, +inf and -inf, values whose square overflows fp32 (the reference's var is inf),
    a constant column (var 0), and ordinary ones.  The forward is the reference's fp32 op sequence: bit-exact."""
    rows, cols = 1000, 9
    g = torch.Generator().manual_seed(10)
    x = torch.randn(rows, cols, generator=g) * 2 + 0.5
    x[5, 0], x[6, 1], x[7, 2], x[8, 3], x[9, 3] = NAN, INF, -INF, INF, -INF
    x[:, 4] = (torch.rand(rows, generator=g) + 1) * 2e20
    x[:, 5] = 7.0
    rn = RunningNorm(cols, device=DEV)
    rn.running_mean.copy_(torch.randn(1, cols, generator=g))
    rn.running_var.copy_(torch.rand(1, cols, generator=g) + 0.5)
    mean, var, count = rn.running_mean.cpu(), rn.running_var.cpu(), rn.count.cpu()
    want = _ieee_forward(mean, var, x, rn.epsilon, rn.clip)
    assert _same(rn(cuda(x)), want)
    assert_close_strict(want, O.running_norm_forward(mean, var, x, rn.epsilon, rn.clip), what="IEEE vs torch", rtol=2e-7,
                        atol=0.0, scale=None)  # fmt: skip
    _assert_moments(rn.moments(cuda(x)), x, "moments")
    rn.update(cuda(x))
    wm, wv, wc = O.running_norm_update(mean, var, count, x)
    assert torch.isnan(wv[0, :4]).all() and wv[0, 4] == INF and wv[0, 5] == 0.0
    assert_close_strict(rn.running_mean, wm, what="running_mean", rtol=1e-6, atol=0.0, scale=None)
    assert_close_strict(rn.running_var, wv, what="running_var", rtol=1e-5, atol=0.0, scale=None)
    assert torch.equal(rn.count.cpu(), wc)
    # forward with the statistics the update left: NaN columns, an infinite variance (x / inf = 0)
    rn.running_mean.copy_(wm)
    rn.running_var.copy_(wv)
    y = torch.randn(64, cols, generator=g)
    assert _same(rn(cuda(y)), _ieee_forward(wm, wv, y, rn.epsilon, rn.clip))


def _ulp_close(a, e):
    a, e = a.cpu(), e.cpu()
    ulp = torch.nextafter(e.abs(), torch.tensor(INF)) - e.abs()
    return bool(((a - e).abs() <= ulp).all())


@pytest.mark.parametrize("cols", [1, 3, 257, 934, 935])
@pytest.mark.parametrize("rows", [1, 7, 8, 9, 8191, 8192, 8193, 70001])
def test_running_norm_kernels_at_layout_edges(rows, cols):
    """The forward is bit-exact against the IEEE fp32 op sequence, the moments agree with fp64 to 1e-12 and the update
    with an fp64 mean / biased variance blended in fp32 to 1 ulp.  Dense rows, a base pointer one float past an 8-byte
    boundary (the one-column-per-thread path), and row / output strides wider than the row; above 8192 rows the
    moments kernel gives each block more rows."""
    g = torch.Generator().manual_seed(rows * 7 + cols)
    base = cuda(torch.randn(rows * (cols + 3) + 2, generator=g) * 2 + 0.5)
    rn = RunningNorm(cols, device=DEV)
    rn.running_mean.copy_(torch.randn(1, cols, generator=g))
    rn.running_var.copy_(torch.rand(1, cols, generator=g) * 2 + 0.01)
    rn.count.fill_(3.0)
    mean, var = rn.running_mean.cpu(), rn.running_var.cpu()
    layouts = {
        "dense": (base[: rows * cols].view(rows, cols), cols),
        "offset": (base[1 : 1 + rows * cols].view(rows, cols), cols),
        "strided": (base[: rows * (cols + 3)].view(rows, cols + 3)[:, :cols], cols + 5),
    }
    for name, (x, out_stride) in layouts.items():
        xc = x.cpu()
        out = torch.full((rows, out_stride), 777.0, device=DEV)
        _cabi.check(_cabi.load().phc_running_norm_forward(
            x.data_ptr(), rows, cols, x.stride(0), rn.running_mean.data_ptr(), rn.running_var.data_ptr(), rn.epsilon,
            rn.clip, out.data_ptr(), out_stride, _cabi.stream_ptr(DEV)), "phc_running_norm_forward")  # fmt: skip
        assert _same(out[:, :cols], _ieee_forward(mean, var, xc, rn.epsilon, rn.clip)), f"{name}: forward"
        assert bool((out[:, cols:] == 777.0).all()), f"{name}: forward wrote past the row"
        sums = rn.moments(x)
        _assert_moments(sums, xc, f"{name}: moments")
    # update: fp64 mean / biased var of the batch, blended in fp32 with weight 1 / count as the kernel does
    x64 = xc.double()
    m, v = x64.mean(0, keepdim=True), x64.var(0, unbiased=False, keepdim=True)
    w = torch.tensor(1.0) / rn.count.cpu()
    want_m = mean * (1.0 - w) + m.float() * w
    want_v = var * (1.0 - w) + v.float() * w
    rn.update_from_moments(sums, rows)
    assert _ulp_close(rn.running_mean, want_m) and _ulp_close(rn.running_var, want_v)


@pytest.mark.parametrize("rows", [8193, 70001])
def test_one_pass_variance_of_a_near_constant_column_stays_within_its_bound(rows):
    """Values a few fp32 ulps apart around 1000: E[x^2] - m^2 cancels almost completely, and the fp64 sums keep the
    error within 4 rows 2^-53 E[x^2] of the two-pass variance (fp32 sums could not)."""
    g = torch.Generator().manual_seed(rows)
    ulp = 2.0**-14  # fp32 ulp at 1000
    x = torch.stack([1000.0 + torch.randint(-3, 4, (rows,), generator=g).float() * ulp,
                     torch.randn(rows, generator=g), torch.full((rows,), 1000.0)], dim=1)  # fmt: skip
    assert x[:, 0].unique().numel() == 7
    rn = RunningNorm(3, device=DEV)
    s = rn.moments(cuda(x)).cpu()
    x64 = x.double()
    v_ref = x64.var(0, unbiased=False)
    v = s[3:] / rows - (s[:3] / rows) ** 2
    bound = 4 * rows * 2.0**-53 * (x64 * x64).mean(0)
    assert bool(((v - v_ref).abs() <= bound).all()), (v, v_ref, bound)
    assert float(v_ref[0]) > 1e-9 and float(v[2]) == 0.0
    rn.update_from_moments(cuda(s), rows)
    got = rn.running_var.cpu().double()[0]
    assert abs(float(got[0]) - float(v_ref[0])) <= float(bound[0]) + 2**-23 * float(v_ref[0])


# ---------------------------------------------------------------------------------------
# episode bookkeeping of PHCPufferEnv.step
# ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("fused", [False, True], ids=["two_launches", "fused"])
def test_episode_bookkeeping_with_a_nan_reward_env_whose_episode_ends(fused):
    N = 1029
    lib_data, clock, sim, bad, at = _case(N, seed=505, ended=True)
    e = at["nan_body_pos"]
    assert e in list(at.values())[::2]  # at its clip's end: reset by the first step
    env = _env(MotionLib(lib_data, device=DEV), clock, bad)
    pe = PHCPufferEnv(env, log_interval=1000, fused=fused)
    want = dict(terminals=torch.zeros(N, dtype=torch.bool), truncations=torch.zeros(N, dtype=torch.bool),
                masks=torch.ones(N, dtype=torch.bool), episode_returns=torch.zeros(N), episode_lengths=torch.zeros(N, dtype=torch.int32),
                raw_rewards=torch.zeros(5), stats=torch.zeros(4, dtype=torch.float64))  # fmt: skip
    g = torch.Generator().manual_seed(11)
    for k in range(3):
        obs, rew, term, trunc, info = pe.step(cuda(torch.rand(N, 69, generator=g) * 4 - 2),
                                              phase_by_env=cuda(torch.rand(N, generator=g)))  # fmt: skip
        if k == 0:
            assert math.isnan(float(rew[e])) and bool(trunc[e] | term[e])
        O.episode_update(want, (term | trunc).cpu(), term.cpu(), rew.cpu(), env.reward_raw.cpu())
    pe._fold()
    torch.cuda.synchronize()
    for key in ("terminals", "truncations", "masks", "episode_lengths"):
        assert_equal_exact(getattr(pe, key), want[key], key)
    assert _same(pe.episode_returns, want["episode_returns"])
    assert math.isnan(want["stats"][1]) and torch.isfinite(want["stats"][[0, 2, 3]]).all()
    assert_close_strict(pe._stats, want["stats"], what="stats", rtol=1e-12, atol=0.0, scale=None)
    assert torch.isnan(want["raw_rewards"]).any() and torch.isfinite(want["raw_rewards"]).any()
    assert_close_strict(pe.raw_rewards, want["raw_rewards"], what="raw_rewards", rtol=1e-6, atol=1e-7, scale=None)
