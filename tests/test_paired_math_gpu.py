"""GPU: the plain fast step kernel blends both query times' reference bodies as the two lanes of fp32x2 instructions
and pairs its observation vectors the same way.  On frames crafted so that the two lanes take different branches or
carry different special values, every output equals the generic kernel's (scalar math) bit for bit, NaN where NaN."""

import os

import pytest
import torch

from util_cpu import assert_close_strict

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from humanoid_b200 import HumanoidPHC, MotionLib, _cabi, synth
    from util_gpu import DEV

OUT = ("obs_buf", "rew_buf", "reward_raw", "reset_buf", "_terminate_buf", "progress_buf")


def _same(x, y):
    if x.dtype != y.dtype or x.shape != y.shape:
        return False
    if not x.is_floating_point():
        return torch.equal(x, y)
    nx, ny = x.isnan(), y.isnan()
    return torch.equal(nx, ny) and torch.equal(torch.where(nx, 0, x).view(torch.int32), torch.where(ny, 0, y).view(torch.int32))


def _craft(lib_data, state, kind, seed):
    """Perturb every third frame of the library (so that an env's two queries, one frame apart, mostly see different
    frames) and, for the signed-zero case, the sim state too."""
    g = torch.Generator().manual_seed(seed)
    lib_data = synth.MotionData(**{k: v.clone() for k, v in lib_data.__dict__.items()})
    state = state.clone()
    F = lib_data.grs.shape[0]
    rows = torch.arange(0, F - 1, 3, device=lib_data.grs.device)
    bodies = torch.randperm(24, generator=g)[:12].to(lib_data.grs.device)
    r, b = rows[:, None], bodies[None, :]
    if kind == "flip":  # q and -q: c < 0 against the neighbouring frame
        lib_data.grs[r, b] = -lib_data.grs[r, b]
    elif kind == "near":  # the next frame a hair away: |sin| < 1e-3, the 0.5 / 0.5 average
        q = lib_data.grs[r, b] + 1e-4 * torch.randn(lib_data.grs[r, b].shape, generator=g).to(lib_data.grs.device)
        lib_data.grs[r + 1, b] = q / q.norm(dim=-1, keepdim=True)
    elif kind == "same":  # the next frame equal, or scaled past 1: c >= 1 selects q0
        lib_data.grs[r + 1, b] = lib_data.grs[r, b] * torch.where(torch.rand(len(rows), 1, 1, generator=g) < 0.5, 1.0, 1.0 + 2e-6).to(lib_data.grs.device)  # fmt: skip
    elif kind == "zeros":  # ±0 and subnormals, in frames and sim state
        for t in (lib_data.gts, lib_data.gvs, lib_data.gavs, lib_data.grs):
            t[r, b, 0] = -0.0
            t[r, b, 1] = 1e-40
        state[::3, :, 7] = -0.0
        state[1::3, :, 8] = -1e-41
        state[2::5, :, 1] = 0.0
    elif kind == "nonfinite":  # NaN / inf in one frame, i.e. in one query of the envs that read it
        lib_data.gts[r, b, 0] = float("nan")
        lib_data.gvs[r, b, 1] = float("inf")
        lib_data.grs[r + 1, b, 2] = float("-inf")
        lib_data.gavs[r, b, 2] = float("nan")
    return lib_data, state


def _run(lib_data, clock, state, N, term):
    env = HumanoidPHC(MotionLib(lib_data, device=DEV), N, device=DEV, termination_distance=term)
    env.set_sim_state(state)
    env.set_clock(clock)
    for _ in range(2):
        env.step()
    torch.cuda.synchronize()
    return env


@pytest.mark.parametrize("N", [1021, 4096])
@pytest.mark.parametrize("kind", ["flip", "near", "same", "zeros", "nonfinite"])
def test_paired_fast_kernel_equals_generic_kernel_bitwise(N, kind):
    lib_data, clock, state = synth.make_case(
        N, 97, lambda d, i, t, o: MotionLib(d, device=DEV).get_motion_state(i, t, o), seed=311, device=DEV,
        max_frames=120, max_progress=60,
    )  # fmt: skip
    lib_data, state = _craft(lib_data, state, kind, seed=17)
    # termination distance at the median body distance: envs on both sides of the threshold
    term = 0.05
    capi = _cabi.load()
    generic = 1 if os.environ.get("PHC_STEP_GENERIC", "").startswith("1") else 0
    try:
        assert capi.phc_set_option(_cabi.OPT_FORCE_GENERIC_STEP, 1) == 0
        want = _run(lib_data, clock, state, N, term)
        assert capi.phc_set_option(_cabi.OPT_FORCE_GENERIC_STEP, 0) == 0
        got = _run(lib_data, clock, state, N, term)
    finally:
        capi.phc_set_option(_cabi.OPT_FORCE_GENERIC_STEP, generic)
    flags = want._terminate_buf.float().mean().item()
    assert kind == "nonfinite" or 0.0 < flags < 1.0, f"termination on one side only ({flags})"
    for name in OUT:
        assert _same(getattr(got, name), getattr(want, name)), f"{kind}: {name}"
    assert_close_strict(got.obs_buf, want.obs_buf, f"{kind}: obs_buf")
    if kind == "nonfinite":
        assert want.obs_buf.isnan().any() and want.obs_buf.isinf().any()
