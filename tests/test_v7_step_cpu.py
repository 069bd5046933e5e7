"""CPU: the imitation observation v7 option of the fused step and the device reset (PHC_OBS_TASK_V7) — the binding's
constant, HumanoidPHC(obs_v=...) validation, and the C-ABI codes that return before anything touches a device."""

import ctypes as C
import os
import re

import pytest

from conftest import ROOT
from humanoid_b200 import _cabi

HEADER = os.path.join(ROOT, "include", "phc_b200.h")
V = _cabi.PhcView
SELF = _cabi.SELF_OBS_DIM


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_cabi.LIB_PATH):
        import __graft_entry__ as g

        g.build()
    return _cabi.load()


@pytest.fixture
def handle(lib):
    d = _cabi.PhcLibDesc()
    for k in ("gts", "grs", "lrs", "gvs", "gavs", "dvs", "motion_lengths", "motion_num_frames", "motion_dt", "length_starts"):
        setattr(d, k, 4096)
    d.total_frames, d.num_motions = 10, 1
    h = C.c_void_p()
    assert lib.phc_lib_create(C.byref(d), C.byref(h)) == 0
    yield h
    lib.phc_lib_destroy(h)


def _body():
    return _cabi.PhcBodyState(V(4096, 312, 13), V(4096 + 12, 312, 13), V(4096 + 28, 312, 13), V(4096 + 40, 312, 13), 24)


def _reset_args(obs_flags, obs_stride, T=1):
    r = _cabi.PhcResetArgs()
    r.body = _body()
    for k in ("progress_buf", "reset_buf", "terminate_buf", "motion_start_times", "motion_start_times_offset",
              "sampled_motion_ids", "obs_buf", "phase"):  # fmt: skip
        setattr(r, k, 4096)
    r.state_init, r.time_steps, r.dt, r.obs_stride, r.obs_flags = _cabi.STATE_INIT_RANDOM, T, 1 / 30, obs_stride, obs_flags
    return r


def _step_args(obs_flags, obs_stride, T=1):
    a = _cabi.PhcStepArgs()
    a.body = _body()
    for k in ("progress_buf", "motion_start_times", "motion_start_times_offset", "sampled_motion_ids",
              "termination_distances", "obs_buf", "rew_buf", "reward_raw", "reset_buf", "terminate_buf"):  # fmt: skip
        setattr(a, k, 4096)
    a.reward_raw_stride, a.time_steps, a.dt, a.obs_stride, a.obs_flags = 5, T, 1 / 30, obs_stride, obs_flags
    # episode bookkeeping with one NULL buffer: PHC_ERR_NULL once the shape checks before it have passed
    a.ep_returns = 4096
    return a


def test_obs_task_v7_matches_the_header():
    m = re.search(r"#define\s+PHC_OBS_TASK_V7\s+(\w+)", open(HEADER).read())
    assert m and int(m.group(1).rstrip("uU"), 0) == _cabi.OBS_TASK_V7 == 8
    # a bit of its own, apart from the self-obs bits and the "given" marker
    assert _cabi.OBS_TASK_V7 & (_cabi.OBS_LOCAL_ROOT | _cabi.OBS_ROOT_HEIGHT | _cabi.OBS_UPRIGHT | _cabi.STEP_OBS_FLAGS_SET) == 0
    assert _cabi.ABI_VERSION == 6


@pytest.mark.parametrize("v", [0, 5, 8, "7", 6.5, None])
def test_obs_v_other_than_6_or_7_raises_before_any_device(v):
    from humanoid_b200 import HumanoidPHC

    with pytest.raises(ValueError, match="obs_v"):
        HumanoidPHC(None, 4, device="cpu", obs_v=v)


@pytest.mark.parametrize("v", [6, 7])
def test_obs_v_6_and_7_pass_validation(v):
    from humanoid_b200 import HumanoidPHC

    with pytest.raises(_cabi.PhcError):  # accepted; the CPU device is what is refused next
        HumanoidPHC(None, 4, device="cpu", obs_v=v)


@pytest.mark.parametrize("flags,T", [(0, 1), (_cabi.STEP_OBS_FLAGS_SET | 7, 1), (_cabi.STEP_OBS_FLAGS_SET | 5, 1), (0, 3)])
def test_step_row_width_follows_the_v7_bit(lib, handle, flags, T):
    """W = selfw + 216 T with the bit (selfw + 576 T without): obs_stride < W is PHC_ERR_SHAPE, W itself passes the
    shape checks (and meets the NULL episode buffer behind them)."""
    selfw = SELF - (1 if flags & _cabi.STEP_OBS_FLAGS_SET and not flags & _cabi.OBS_ROOT_HEIGHT else 0)
    w7, w6 = selfw + 216 * T, selfw + 576 * T
    v7 = flags | _cabi.OBS_TASK_V7
    assert lib.phc_step_fused(handle, C.byref(_step_args(v7, w7 - 1, T)), 8, None) == -2
    assert lib.phc_step_fused(handle, C.byref(_step_args(v7, w7, T)), 8, None) == -1
    assert lib.phc_step_fused(handle, C.byref(_step_args(flags, w7, T)), 8, None) == -2
    assert lib.phc_step_fused(handle, C.byref(_step_args(flags, w6, T)), 8, None) == -1


@pytest.mark.parametrize("T", [1, 10])
def test_reset_row_width_follows_the_v7_bit(lib, handle, T):
    w7 = SELF + 216 * T
    assert lib.phc_reset_envs(handle, C.byref(_reset_args(_cabi.OBS_TASK_V7, w7 - 1, T)), 8, None) == -2
    assert lib.phc_reset_envs(handle, C.byref(_reset_args(_cabi.OBS_TASK_V7, w7, T)), 8, None) == -1  # no env_mask
    assert lib.phc_reset_envs(handle, C.byref(_reset_args(0, w7, T)), 8, None) == -2
    r = _reset_args(_cabi.OBS_TASK_V7, w7, T)
    r.obs_norm, r.norm_mean, r.norm_var, r.norm_clip, r.obs_norm_stride = 4096, 4096, 4096, 10.0, w7 - 1
    assert lib.phc_reset_envs(handle, C.byref(r), 8, None) == -2  # the normalised copy is W wide too


def test_auto_reset_must_agree_with_the_step_on_v7(lib, handle):
    W = SELF + 216
    for step_flags, reset_flags in ((_cabi.OBS_TASK_V7, 0), (0, _cabi.OBS_TASK_V7)):
        a = _step_args(step_flags, SELF + 576)
        r = _reset_args(reset_flags, SELF + 576)
        for k in ("progress_buf", "reset_buf", "terminate_buf", "motion_start_times", "motion_start_times_offset",
                  "sampled_motion_ids", "obs_buf"):  # fmt: skip
            setattr(r, k, getattr(a, k))
        r.body = a.body
        a.auto_reset = C.pointer(r)
        assert lib.phc_step_fused(handle, C.byref(a), 8, None) == -2, (step_flags, reset_flags)
    a = _step_args(_cabi.OBS_TASK_V7, W)
    r = _reset_args(_cabi.OBS_TASK_V7, W)
    r.body = a.body
    a.auto_reset = C.pointer(r)
    assert lib.phc_step_fused(handle, C.byref(a), 8, None) == -1  # agrees: on to the NULL episode buffer
