"""CPU: the strict comparator, and what the oracle gives on non-finite and degenerate inputs — the values the GPU tests
in test_nonfinite_gpu.py hold the kernels to."""

import math

import numpy as np
import pytest
import torch

from oracle import phc_oracle as O
from util_cpu import POISONS, assert_close_strict, poison
from util_gpu import make_case_cpu, oracle_step

NAN, INF = float("nan"), float("inf")


@pytest.mark.parametrize("got,want", [([INF], [-INF]), ([5.0], [INF]), ([INF], [5.0]), ([-INF], [-1e30]), ([NAN], [1.0]),
                                      ([1.0], [NAN]), ([NAN], [INF]), ([1.0, INF, 2.0], [1.0, 2.0, INF])])  # fmt: skip
def test_strict_comparator_rejects_a_different_non_finite_pattern(got, want):
    with pytest.raises(AssertionError, match="pattern differs"):
        assert_close_strict(torch.tensor(got), torch.tensor(want), what="x")


def test_strict_comparator_accepts_equal_patterns_and_still_compares_the_finite_entries():
    want = torch.tensor([[NAN, INF, -INF, 1.0, 3.0, 4.0]])
    assert_close_strict(torch.tensor([[NAN, INF, -INF, 1.0, 3.0, 4.0 + 1e-6]]), want, what="x", rtol=1e-5, atol=0.0)
    with pytest.raises(AssertionError, match="outside"):
        assert_close_strict(torch.tensor([[NAN, INF, -INF, 1.0, 3.0, 4.1]]), want, what="x", rtol=1e-5, atol=0.0)
    # the vector scale is taken from the finite entries: the 3-vector (INF, 3, 4) is judged against |(0, 3, 4)| = 5
    a, e = torch.tensor([[[INF, 3.0, 4.0001]]]), torch.tensor([[[INF, 3.0, 4.0]]])
    assert_close_strict(a, e, what="x", rtol=2.1e-5, atol=0.0)
    with pytest.raises(AssertionError, match="outside"):
        assert_close_strict(a, e, what="x", rtol=1.9e-5, atol=0.0)


def test_oracle_running_norm_forward_on_non_finite_inputs():
    """RunningNorm.forward = torch.clamp((x - mean) / torch.sqrt(var + eps), -clip, clip) (policies/running_norm.py:15-20):
    clamp keeps NaN, ±inf clamps to ±clip, 0 / 0 is NaN, a subnormal var + eps is an ordinary small divisor."""
    x = torch.tensor([[NAN, INF, -INF, 2.0, 1.0, 1.0, -3.0, 1.0, 5.0, 5.0, 0.5, 0.5]])
    mean = torch.tensor([[0.0, 0.0, 0.0, 1.0, 1.0, 0.0, 0.0, 1.0, NAN, 0.0, INF, 0.0]])
    var = torch.tensor([[1.0, 1.0, 1.0, 0.0, 0.0, 1e-40, 1e-40, 1e-40, 1.0, NAN, 1.0, INF]])
    got = O.running_norm_forward(mean, var, x, epsilon=0.0, clip=10.0)
    want = [NAN, 10.0, -10.0, 10.0, NAN, 10.0, -10.0, 0.0, NAN, NAN, -10.0, 0.0]
    assert torch.equal(torch.isnan(got), torch.isnan(torch.tensor([want])))
    assert torch.equal(torch.nan_to_num(got), torch.nan_to_num(torch.tensor([want])))
    assert got[0, 4] != got[0, 4] and got[0, 3] == 10.0  # var + eps == 0: NaN where x == mean, ±clip elsewhere
    # with the default epsilon a zero variance is an ordinary divisor
    ok = O.running_norm_forward(mean[:, 3:5], var[:, 3:5], x[:, 3:5])
    assert torch.equal(ok, torch.clamp(torch.tensor([[1.0, 0.0]]) / torch.sqrt(torch.tensor(1e-5)), -10.0, 10.0))


def test_oracle_pd_targets_propagate_nan():
    """_action_to_pd_targets (humanoid_phc.py:1218-1228): torch.maximum(torch.minimum(pd, q + pi/2), q - pi/2), where
    minimum / maximum return NaN if either operand is NaN."""
    off, sc = torch.zeros(3), torch.full((3,), 2.0)
    act = torch.tensor([[NAN, 0.5, 0.25]])
    ref = torch.tensor([[0.0, 0.0, 0.0]])
    q = torch.tensor([[0.0, NAN, 0.0]])
    got = O.action_to_pd_targets(act, off, sc, True, ref, q)
    assert math.isnan(got[0, 0]) and math.isnan(got[0, 1])
    assert float(got[0, 2]) == 0.5
    far = O.action_to_pd_targets(torch.tensor([[1.0, -1.0, 0.0]]), off, torch.full((3,), 5.0), True, ref, torch.zeros(1, 3))
    assert far.tolist() == [[np.float32(np.pi / 2), -np.float32(np.pi / 2), 0.0]]
    assert math.isnan(O.action_to_pd_targets(act, off, sc)[0, 0])  # offset + scale * action


def test_oracle_exp_map_to_quat_turns_a_nan_exp_map_into_the_identity():
    """exp_map_to_angle_axis (torch_utils.py:334-350) keeps angle and axis only where |angle| > 1e-5; a NaN angle fails
    that comparison (an infinite one too: atan2(sin inf, cos inf) is NaN), so the AMP observation of a NaN dof_pos is the
    tangent-normal of the identity rotation."""
    q = O.exp_map_to_quat(torch.tensor([[NAN, 0.2, 0.1], [0.3, 0.0, INF]]))
    assert q.tolist() == [[0.0, 0.0, 0.0, 1.0], [0.0, 0.0, 0.0, 1.0]]


def test_oracle_step_confines_each_poison_to_its_env():
    """The oracle's step on the poisoned sim state: every poisoned env differs from the clean step only in its own row,
    each NaN / inf pattern is per env, no poisoned env is flagged by its NaN distance, and the 1e20 velocity sends the
    velocity reward term's exp to 0.  These are the expectations the kernels are held to."""
    N = 64
    lib_data, clock, state = make_case_cpu(num_envs=N, num_motions=16, seed=401, max_progress=30)
    g = torch.Generator().manual_seed(2)
    sim = dict(state=state, dof_force=torch.randn(N, 69, generator=g) * 40, dof_vel=torch.randn(N, 69, generator=g) * 3,
               dof_pos=torch.randn(N, 69, generator=g))  # fmt: skip
    bad, at = poison(sim, N)
    assert list(at) == list(POISONS) and at["nan_body_pos"] == 0 and at["nan_root_pos"] == 3 and at["inf_body_vel"] == N - 1

    def run(s):
        return oracle_step(lib_data, clock, s["state"], dof_force=s["dof_force"], dof_vel=s["dof_vel"])

    clean, dirty = run(sim), run(bad)
    keep = torch.ones(N, dtype=torch.bool)
    keep[list(at.values())] = False
    for a, b in zip(clean, dirty):
        assert torch.equal(a[keep], b[keep])
    obs, rew, raw = dirty[0], dirty[1], dirty[2]
    nonfin = (~torch.isfinite(obs)).sum(1)
    for name in ("nan_body_pos", "nan_root_pos", "nan_root_rot", "inf_body_vel", "neg_inf_ang_vel"):
        assert int(nonfin[at[name]]) >= 6, name
    assert int(nonfin[keep].sum()) == 0
    assert float(raw[at["vel_1e20"], 2]) == 0.0 and torch.isfinite(obs[at["vel_1e20"]]).all()
    for name in ("nan_dof_force", "nan_dof_vel"):  # the power term only, and only once progress > 3
        assert torch.isnan(raw[at[name], 4]) == (clock.progress_buf[at[name]] + 1 > 3)
        assert torch.isfinite(obs[at[name]]).all()
    assert torch.equal(obs[at["nan_dof_pos"]], clean[0][at["nan_dof_pos"]])  # dof_pos is not read by the step
    for name in ("nan_body_pos", "nan_root_pos"):
        assert math.isnan(rew[at[name]]) and not bool(dirty[4][at[name]])
