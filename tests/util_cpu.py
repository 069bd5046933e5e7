"""Helpers shared by the CPU tests."""

import torch

from conftest import assert_close
from humanoid_b200 import synth
from oracle import phc_oracle as O


def assert_close_strict(actual, expected, what="", **tol):
    """``assert_close`` that also tells the non-finite values apart: the NaN, +inf and -inf masks of ``actual`` and
    ``expected`` must be equal (``assert_close`` takes +inf for -inf and 5 for inf, since inf <= inf), then the finite
    entries are compared as ``assert_close`` does, with ``scale="vec"`` unless ``tol`` says otherwise and the vector
    norms taken from ``expected`` with its non-finite entries zeroed."""
    a = torch.as_tensor(actual).detach().cpu().double()
    e = torch.as_tensor(expected).detach().cpu().double()
    assert a.shape == e.shape, f"{what}: shape {tuple(a.shape)} vs {tuple(e.shape)}"
    for name, fa, fe in (("NaN", torch.isnan(a), torch.isnan(e)), ("+inf", a == float("inf"), e == float("inf")),
                         ("-inf", a == float("-inf"), e == float("-inf"))):  # fmt: skip
        if not torch.equal(fa, fe):
            first = (fa != fe).nonzero()[:4].tolist()
            raise AssertionError(f"{what}: {name} pattern differs ({int(fa.sum())} vs {int(fe.sum())}), first at {first}")
    fin = torch.isfinite(e)
    tol.setdefault("scale", "vec")
    assert_close(torch.where(fin, a, 0.0), torch.where(fin, e, 0.0), what=what, **tol)


# What a diverged physics step or policy leaves in the sim state: one kind per env, so that every non-finite output can
# be traced to its input.  `state` is the [N, 24, 13] AoS rigid-body tensor (pos 0:3, quat xyzw 3:7, vel 7:10, ang vel
# 10:13), `dof_*` are [N, 69].
POISONS = (
    "nan_body_pos", "nan_root_pos", "nan_root_rot", "inf_body_vel", "neg_inf_ang_vel", "zero_root_quat", "zero_body_quat",
    "quat_times_3", "vel_1e20", "subnormal_pos", "nan_dof_force", "nan_dof_vel", "nan_dof_pos",
)  # fmt: skip


def poison_envs(n):
    """One env per poison, at the edges of the step kernels' 4-env blocks: env 0, the last env of a block, envs in the
    middle, and the last env (of a partial block where n % 4 != 0)."""
    m = n // 8 * 4
    cand = [0, 3, m, n - 1, m + 3, 4, 7, m - 1, m + 4, n - 2, 8, 11, 12, 15, 16, 19, 20]
    envs = list(dict.fromkeys(e for e in cand if 0 <= e < n))
    assert len(envs) >= len(POISONS), "too few envs for one poison each"
    return dict(zip(POISONS, envs))


def poison(sim, n):
    """A poisoned copy of ``sim`` = dict(state, dof_force, dof_vel, dof_pos); returns (copy, {poison: env})."""
    bad = {k: v.clone() for k, v in sim.items()}
    at = poison_envs(n)
    s = bad["state"]
    nan, inf = float("nan"), float("inf")
    for name, e in at.items():
        if name == "nan_body_pos":
            s[e, 5, 1] = nan
        elif name == "nan_root_pos":
            s[e, 0, 0] = nan
        elif name == "nan_root_rot":
            s[e, 0, 4] = nan
        elif name == "inf_body_vel":
            s[e, 7, 8] = inf
        elif name == "neg_inf_ang_vel":
            s[e, 3, 11] = -inf
        elif name == "zero_root_quat":  # the clamp(min=1e-9) of the norms the heading and tan_norm divide by
            s[e, 0, 3:7] = 0.0
        elif name == "zero_body_quat":
            s[e, 9, 3:7] = 0.0
        elif name == "quat_times_3":
            s[e, 4, 3:7] *= 3.0
        elif name == "vel_1e20":  # its square overflows fp32: the velocity reward term's exp goes to 0
            s[e, 2, 7:10] = 1e20
        elif name == "subnormal_pos":  # every body within subnormal distance of the origin and of the root
            s[e, :, 0:3] = torch.arange(1, 25, dtype=torch.float32)[:, None] * torch.tensor([1e-40, -2e-40, 3e-40])
        elif name == "nan_dof_force":
            bad["dof_force"][e, 10] = nan
        elif name == "nan_dof_vel":
            bad["dof_vel"][e, 20] = nan
        elif name == "nan_dof_pos":
            bad["dof_pos"][e, 30] = nan
    return bad, at


def oracle_env_from_golden(g, use_amp_obs=True):
    lib = O.OracleMotionLib(synth.MotionData(**g.group("in.lib")))
    c = synth.Clock(**g.group("in.clock"))
    if use_amp_obs:
        amp = dict(dof_subset=g.inp("dof_subset"), key_body_ids=g.inp("key_body_ids"),
                   num_amp_obs_steps=int(g.inp("num_amp_obs_steps")))  # fmt: skip
    else:  # the reset-mode fixture runs without the AMP buffers
        amp = dict(dof_subset=torch.arange(69), key_body_ids=torch.zeros(0, dtype=torch.long), num_amp_obs_steps=2,
                   use_amp_obs=False)  # fmt: skip
    env = O.OracleEnv(
        lib, c.progress_buf.shape[0], c.progress_buf, c.motion_start_times, c.motion_start_times_offset,
        c.global_offset, c.sampled_motion_ids, g.inp("pd_action_offset"), g.inp("pd_action_scale"),
        rew_power_coef=float(g.inp("rew_power_coef")), termination_distance=float(g.inp("termination_distance")), **amp,
    )  # fmt: skip

    def write_sim(state, dof_state, dof_force):
        env.state[:], env.dof_state[:], env.dof_force[:] = state, dof_state, dof_force
        env.root_states[:] = state[:, 0]

    env.write_sim = write_sim
    env.read_sim = lambda: (env.state, env.root_states, env.dof_state)
    return env
