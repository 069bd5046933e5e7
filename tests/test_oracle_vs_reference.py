"""CPU: the oracle and the loader's host logic against the reference on larger seeded inputs than the step fixtures.

Where the reference's ``puffer_phc`` package can be imported (``oracle.ref_loader``) its functions run live and must
match bit for bit.  Elsewhere the tests compare with ``tests/golden/reference_cases.npz``, the reference's outputs on
the same seeded inputs recorded by ``tests/golden/make_reference_cases.py`` (obs and motion-state rows as a fixed
sample, plus every obs row's sum): flags and indices exactly, floats within TIGHT, as ``test_oracle_golden.py`` does."""

import numpy as np
import pytest
import torch

from conftest import assert_close, assert_equal_exact
from humanoid_b200 import synth
from oracle import phc_oracle as O
from oracle import ref_loader

# same torch build => bit-exact; a tiny tolerance keeps a different host ISA from breaking the recorded pin
TIGHT = dict(rtol=1e-6, atol=1e-7)
RECORDED = "reference_cases"

STEP_CASES = [
    dict(num_envs=256, num_motions=16, seed=1, max_progress=20),  # BASELINE config 1
    dict(num_envs=512, num_motions=512, seed=2, max_frames=90, max_progress=20),  # ids == arange regime
    dict(num_envs=384, num_motions=40, seed=3, ids="random", aligned=False, fps_choices=(30, 60, 120),
         rot_regime="random", max_progress=30),
]  # fmt: skip
MOTION_KEYS = (
    "root_pos", "root_rot", "dof_pos", "root_vel", "root_ang_vel", "dof_vel", "motion_aa",
    "rg_pos", "rb_rot", "body_vel", "body_ang_vel", "motion_bodies", "motion_limb_weights",
)  # fmt: skip
ROW_KEYS = {"obs", *MOTION_KEYS}  # recorded for a fixed seeded sample of env rows only


def _query(lib_data, ids, times, offset):
    """The reference's motion query; the oracle's (bit-identical, tests/golden) to build the inputs without it."""
    if ref_loader.available():
        return ref_loader.make_reference_lib(lib_data).get_motion_state(ids, times, offset)
    return O.OracleMotionLib(lib_data).get_motion_state(ids, times, offset)


def step_case(kw):
    lib_data, clock, state = synth.make_case(query=_query, **kw)
    return lib_data, clock, state, torch.full((24,), 0.25)


def oracle_step(kw):
    lib_data, clock, state, term = step_case(kw)
    obs, reward, raw, reset, terminated = O.step(
        O.OracleMotionLib(lib_data), state, clock.progress_buf.clone(), clock.motion_start_times,
        clock.motion_start_times_offset, clock.global_offset, clock.sampled_motion_ids, term, synth.SIM_DT,
    )  # fmt: skip
    return {"obs": obs, "reward": reward, "reward_raw": raw, "reset": reset, "terminated": terminated}


def reference_step(kw):
    """The post-physics half of HumanoidPHC.step with the reference's own functions (needs the reference)."""
    _, ref_common, _ = ref_loader.load()
    lib_data, clock, state, term = step_case(kw)
    ref_lib = ref_loader.make_reference_lib(lib_data)
    pos, rot, vel, ang = synth.body_views(state)
    dt = synth.SIM_DT
    p = clock.progress_buf.clone()
    p += 1
    t = p * dt + clock.motion_start_times + clock.motion_start_times_offset
    r0 = ref_lib.get_motion_state(clock.sampled_motion_ids, t, clock.global_offset)
    rr, rraw = ref_common.compute_imitation_reward(
        pos[:, 0], rot[:, 0], pos, rot, vel, ang, r0["rg_pos"], r0["rb_rot"], r0["body_vel"], r0["body_ang_vel"],
        O.DEFAULT_RWD_SPECS,
    )  # fmt: skip
    rs, rt = ref_common.compute_humanoid_im_reset(
        torch.ones(state.shape[0], dtype=torch.bool), p, torch.zeros(1), torch.zeros(1), pos.clone(),
        r0["rg_pos"].clone(), t >= ref_lib._motion_lengths[clock.sampled_motion_ids], True, term, False,
    )  # fmt: skip
    t1 = (p + 1) * dt + clock.motion_start_times + clock.motion_start_times_offset
    r1 = ref_lib.get_motion_state(clock.sampled_motion_ids, t1, clock.global_offset)
    so = ref_common.compute_humanoid_observations_smpl_max(pos, rot, vel, ang, None, None, True, True, True, False, False)
    to = ref_common.compute_imitation_observations_v6(
        pos[:, 0], rot[:, 0], pos, rot, vel, ang, r1["rg_pos"], r1["rb_rot"], r1["body_vel"], r1["body_ang_vel"], 1, True
    )  # fmt: skip
    return {"obs": torch.cat([so, to], -1), "reward": rr, "reward_raw": rraw, "reset": rs, "terminated": rt}


def motion_state_case():
    lib_data = synth.make_motion_lib(24, 30, 120, fps_choices=(30, 60), seed=8)
    clock = synth.make_clock(lib_data, 300, seed=9, ids="random", aligned=False)
    t = synth.reward_time(clock) - 0.05  # some negative times
    return lib_data, clock.sampled_motion_ids, t, clock.global_offset


def oracle_motion_state():
    lib_data, ids, t, goff = motion_state_case()
    got = O.OracleMotionLib(lib_data).get_motion_state(ids, t, goff)
    return {k: got[k] for k in MOTION_KEYS}


def reference_motion_state():
    lib_data, ids, t, goff = motion_state_case()
    return ref_loader.make_reference_lib(lib_data).get_motion_state(ids, t, goff)


def sampler_clips(golden):
    g = golden("motion_build")
    nf = g.inp("num_frames").tolist()
    starts = np.concatenate([[0], np.cumsum(nf)])
    clips = {}
    for m in range(len(nf)):
        sl = slice(int(starts[m]), int(starts[m + 1]))
        clips[f"clip{m}"] = {"root_trans_offset": g.inp("root_trans_offset")[sl].clone(), "pose_aa": g.inp("pose_aa")[sl].numpy().copy(),
                             "pose_quat_global": g.inp("pose_quat_global")[sl].numpy().copy(), "beta": np.zeros(16), "fps": int(g.inp("fps")[m])}  # fmt: skip
    return g, clips


FAILED = ["clip3", "clip0"]
SAMPLER_ENVS = 10


def _key_ids(keys):
    return torch.tensor([int(k[len("clip"):]) for k in keys])


def sampler_trace(golden):
    """Host state of the loader (which clips, PMCP weights, batch sampling) along a fixed sequence of calls under fixed
    torch seeds: load_data ordering, load_motions :300-321, update_*_sampling_weight, sample_motions."""
    from humanoid_b200.motion_build import ClipSampler

    _, clips = sampler_clips(golden)
    out = {}
    for im_eval in (False, True):
        e = f"eval{int(im_eval)}"
        mine = ClipSampler()
        mine._init_clips(clips, im_eval=im_eval)
        out[f"{e}.keys"] = _key_ids(mine._motion_data_keys.tolist())
        for step in range(3):
            if step == 1:
                mine.update_soft_sampling_weight(FAILED)
            if step == 2:
                mine.update_hard_sampling_weight(FAILED[:1])
            out[f"{e}.{step}.sampling_prob"] = mine._sampling_prob.clone()
            out[f"{e}.{step}.termination_history"] = mine._termination_history.clone()
            torch.manual_seed(100 + step)
            out[f"{e}.{step}.ids"] = mine.pick_clips(SAMPLER_ENVS, True, 0, None, is_deterministic=False).clone()
            out[f"{e}.{step}.curr_keys"] = _key_ids(mine.curr_motion_keys.tolist())
            out[f"{e}.{step}.batch_prob"] = mine._sampling_batch_prob.clone()
            torch.manual_seed(7)
            out[f"{e}.{step}.sample_motions"] = mine.sample_motions(5).clone()
        # the sequential branch with a start index (evaluation sweep, humanoid_phc.py:1381-1402)
        out[f"{e}.sequential_ids"] = mine.pick_clips(SAMPLER_ENVS, False, 4, None, is_deterministic=False).clone()
        mine.update_soft_sampling_weight([])
        out[f"{e}.final_sampling_prob"] = mine._sampling_prob.clone()
    return out


def reference_sampler_trace(golden):
    """``sampler_trace`` of the reference's MotionLibSMPL (needs the reference)."""
    import types

    _, _, ref_ml = ref_loader.load()
    from puffer_phc.poselib_skeleton import SkeletonTree

    g, clips = sampler_clips(golden)
    nf = g.inp("num_frames").tolist()
    names = [f"b{j}" for j in range(24)]
    N = SAMPLER_ENVS
    trees = [SkeletonTree(names, g.inp("parent_indices").long(), g.inp("local_translation")[e % len(nf)]) for e in range(N)]
    betas = [torch.zeros(17) for _ in range(N)]
    limbs = [np.zeros(10) for _ in range(N)]
    out = {}
    for im_eval in (False, True):
        e = f"eval{int(im_eval)}"
        ref = object.__new__(ref_ml.MotionLibSMPL)
        ref.m_cfg = types.SimpleNamespace(max_length=-1, fix_height=ref_ml.FixHeightMode.no_fix, is_deterministic=False,
                                          im_eval=im_eval, num_thread=1)  # fmt: skip
        ref._device, ref.mesh_parsers = "cpu", None
        # load_data (:192-230) minus joblib.load of a file
        order = sorted(clips.items(), key=lambda kv: len(kv[1]["pose_quat_global"]), reverse=True) if im_eval else clips.items()
        ref._motion_data_list = np.array([v for _, v in order])
        ref._motion_data_keys = np.array([k for k, _ in order])
        ref._num_unique_motions = len(clips)
        ref.setup_constants(fix_height=ref_ml.FixHeightMode.no_fix, num_thread=1)
        out[f"{e}.keys"] = _key_ids(ref._motion_data_keys.tolist())
        for step in range(3):
            if step == 1:
                ref.update_soft_sampling_weight(FAILED)
            if step == 2:
                ref.update_hard_sampling_weight(FAILED[:1])
            out[f"{e}.{step}.sampling_prob"] = ref._sampling_prob.clone()
            out[f"{e}.{step}.termination_history"] = ref._termination_history.clone()
            torch.manual_seed(100 + step)
            np.random.seed(0)
            ref.load_motions(trees, betas, limbs, random_sample=True)
            out[f"{e}.{step}.ids"] = ref._curr_motion_ids.clone()
            out[f"{e}.{step}.curr_keys"] = _key_ids(ref.curr_motion_keys.tolist())
            out[f"{e}.{step}.batch_prob"] = ref._sampling_batch_prob.clone()
            torch.manual_seed(7)
            out[f"{e}.{step}.sample_motions"] = ref.sample_motions(5).clone()
        ref.load_motions(trees, betas, limbs, random_sample=False, start_idx=4)
        out[f"{e}.sequential_ids"] = ref._curr_motion_ids.clone()
        ref.update_soft_sampling_weight([])
        out[f"{e}.final_sampling_prob"] = ref._sampling_prob.clone()
    return out


def recorded(golden, prefix):
    """``{key: tensor}`` of one case of the recording, and the env rows it kept of the ROW_KEYS."""
    got = golden(RECORDED).group(prefix)
    return got, got.pop("rows", None)


def compare(got, want, rows, what):
    """Recorded keys with one row per env (ROW_KEYS) hold only the recording's sampled ``rows``."""
    for k, w in want.items():
        a = got[k][rows] if k in ROW_KEYS else got[k]
        if w.dtype.is_floating_point:
            assert_close(a, w, what=f"{what}: {k}", **TIGHT)
        else:
            assert_equal_exact(a, w, f"{what}: {k}")


@pytest.mark.parametrize("kw", STEP_CASES)
def test_whole_step_bit_exact_vs_reference(kw, golden):
    got = oracle_step(kw)
    assert 0 < got["terminated"].float().mean() < 1
    if ref_loader.available():
        want = reference_step(kw)
        assert torch.equal(got["obs"], want["obs"])
        assert torch.equal(got["reward"], want["reward"]) and torch.equal(got["reward_raw"], want["reward_raw"])
        assert_equal_exact(got["reset"], want["reset"], "reset")
        assert_equal_exact(got["terminated"], want["terminated"], "terminated")
    else:
        want, rows = recorded(golden, f"step{STEP_CASES.index(kw)}")
        row_sum = want.pop("obs_row_sum")
        compare(got, want, rows, "recorded reference step")
        # every row: TIGHT per element, summed over the row
        obs = got["obs"].double()
        tol = TIGHT["rtol"] * obs.abs().sum(1) + TIGHT["atol"] * obs.shape[1]
        assert bool(((obs.sum(1) - row_sum).abs() <= tol).all()), "obs row sums differ from the recording"


def test_motion_state_all_keys_bit_exact_vs_reference(golden):
    got = oracle_motion_state()
    if ref_loader.available():
        for k, v in reference_motion_state().items():
            assert torch.equal(got[k], v), k
    else:
        want, rows = recorded(golden, "motion_state")
        assert set(want) == set(MOTION_KEYS)
        compare(got, want, rows, "recorded reference motion state")


def test_clip_sampler_matches_reference_sampling_state(golden):
    """Host logic of the loader against the reference's MotionLibSMPL under the same torch seeds."""
    got = sampler_trace(golden)
    want = reference_sampler_trace(golden) if ref_loader.available() else recorded(golden, "sampler")[0]
    assert set(got) == set(want)
    for k, w in want.items():
        assert torch.equal(got[k], w.to(got[k].dtype)), k


@pytest.mark.skipif(not ref_loader.available(), reason="reference tree not present")
def test_reference_step_orchestration_equals_the_oracle_step_bit_for_bit():
    """``ref_loader.reference_step`` — what ``bench.py --impl reference`` times (the reference's own functions in the
    env's order) — against ``oracle.step`` on the same inputs, T = 1 and T = 3."""
    for T in (1, 3):
        lib_data, clock, state = synth.make_case(query=_query, num_envs=300, num_motions=24, seed=5 + T, max_progress=20)
        term = torch.full((24,), 0.25)
        p1, p2 = clock.progress_buf.clone(), clock.progress_buf.clone()
        want = O.step(O.OracleMotionLib(lib_data), state, p1, clock.motion_start_times, clock.motion_start_times_offset,
                      clock.global_offset, clock.sampled_motion_ids, term, synth.SIM_DT, time_steps=T)  # fmt: skip
        got = ref_loader.reference_step(ref_loader.make_reference_lib(lib_data), state, p2, clock.motion_start_times,
                                        clock.motion_start_times_offset, clock.global_offset, clock.sampled_motion_ids,
                                        term, synth.SIM_DT, time_steps=T)  # fmt: skip
        assert torch.equal(p1, p2)
        for a, b, nm in zip(got, want, ("obs", "reward", "reward_raw", "reset", "terminated")):
            assert_equal_exact(a, b, f"T={T}: {nm}")
