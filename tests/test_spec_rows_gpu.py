"""GPU: the fast step kernel's speculated frame rows.  Blocks below spec4_blocks (the spare slots of a single-wave grid)
speculate on three candidate query times and copy up to four frame rows; the others copy the rows of two candidates and
fetch the missing rows after validation when progress turns out to have moved by one.  Whichever path a block takes,
and whichever kernel instantiation runs (the plain one, or the one that carries the per-step options), the outputs
are those of the generic kernel, bit for bit."""

import os

import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from humanoid_b200 import HumanoidPHC, MotionLib, _cabi, synth
    from util_gpu import DEV


def _run(lib, clock, state, N, options, steps=3):
    env = HumanoidPHC(lib, N, device=DEV)
    rew_copy = None
    if options:  # a second reward output: the step runs on the instantiation that carries the per-step options
        rew_copy = torch.full((N,), float("nan"), device=DEV)
        env.set_reward_copy(rew_copy)
    env.set_sim_state(state)
    env.set_clock(clock)
    for _ in range(steps):
        env.step()
    torch.cuda.synchronize()
    return env, rew_copy


# 3001 envs: 751 blocks, so a 148-SM B200 at 8 blocks per SM has 433 blocks below spec4_blocks and 318 above it;
# 4096 envs: the headline grid, 160 below and 864 above
@pytest.mark.parametrize("N", [3001, 4096])
@pytest.mark.parametrize("regime", ["aligned30", "mixed_fps_unaligned"])
@pytest.mark.parametrize("kernel", ["plain", "options"])
def test_speculated_rows_on_every_path_equal_generic_kernel_bitwise(N, regime, kernel):
    kw = dict(max_frames=90, max_progress=40)
    if regime != "aligned30":
        kw.update(ids="random", aligned=False, fps_choices=(30, 60, 120), min_frames=60, max_frames=400)
    lib_data, clock, state = synth.make_case(
        N, 257, lambda d, i, t, o: MotionLib(d, device=DEV).get_motion_state(i, t, o), seed=209, device=DEV, **kw
    )
    lib = MotionLib(lib_data, device=DEV)
    capi = _cabi.load()
    options = kernel == "options"
    generic = 1 if os.environ.get("PHC_STEP_GENERIC", "").startswith("1") else 0  # the library's start-up setting
    try:
        assert capi.phc_set_option(_cabi.OPT_FORCE_GENERIC_STEP, 1) == 0
        want, want_copy = _run(lib, clock, state, N, options)
        assert capi.phc_set_option(_cabi.OPT_FORCE_GENERIC_STEP, generic) == 0
        # 1: progress one behind what the block speculated on (the extra-row fetch above spec4_blocks, the fourth
        # speculated row below); 2: start time changed; 4: progress two behind; 8: clip re-assigned; 3: 1 and 2
        for fault in (0, 1, 2, 4, 8, 3):
            assert capi.phc_set_option(_cabi.OPT_TEST_SPEC_FAULT, fault) == 0
            got, got_copy = _run(lib, clock, state, N, options)
            what = f"spec_fault {fault}"
            assert torch.equal(got.obs_buf, want.obs_buf), what
            assert torch.equal(got.rew_buf, want.rew_buf) and torch.equal(got.reward_raw, want.reward_raw), what
            assert torch.equal(got.reset_buf, want.reset_buf), what
            assert torch.equal(got._terminate_buf, want._terminate_buf), what
            assert torch.equal(got.progress_buf, want.progress_buf), what
            if options:
                assert torch.equal(got_copy, want_copy) and torch.equal(got_copy, got.rew_buf), what
    finally:
        capi.phc_set_option(_cabi.OPT_TEST_SPEC_FAULT, 0)
        capi.phc_set_option(_cabi.OPT_FORCE_GENERIC_STEP, generic)
