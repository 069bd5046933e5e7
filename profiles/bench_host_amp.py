"""AMP observations on the host-buffer path (phc_host_step_submit_amp): what HumanoidPHC.step()'s AMP work costs when
the host step does it, against the step without it and against doing it after the step.

The harness of bench_host_episode.py (r7): config 2, two 4096-env batches (bench_host_env.Batch), device obs, direct
path with three chunks, the two-slot async loop, median of --passes loops of --rounds rounds (one round = one step of
batch A and one of B), S = 10.  Legs, alternated in one run:

  a_plain         phc_host_step_submit_device: the step without AMP
  b_amp           phc_host_step_submit_amp: the same step with the AMP roll + slot 0 into device tensors
  b_amp_reset     the same with random auto-reset, early termination off: the ~4 % clip-end envs are re-posed every
                  step and their AMP rows re-initialised (_init_amp_obs)
  b_power_amp     phc_host_step_submit_amp with the power reward (the reference's AMP configuration): one dof velocity
                  upload serves both
  c_workaround    a_plain, then after each wait, on the discriminator's stream: H2D copies of the rigid-body state, the
                  dof rows, the reset flags and the start times, phc_amp_step, and phc_amp_init_ref masked by the envs
                  re-posed (none: a_plain has no auto-reset, so its result can equal b_amp's) — what a host loop had to
                  do before

Floors: the copy engine alone moving 1278 (plain step), 1830 (+ AMP's dof rows) and 2106 B per env (+ the power
reward's dof force).  One host reset of all envs is timed with and without AMP.  The AMP tensors of b_amp and
c_workaround are cleared before every loop and compared bit for bit after the last one; a mismatch fails the run.
Writes r8_host_amp.{json,md} to --out and prints the JSON.

    python profiles/bench_host_amp.py [--rounds 200] [--passes 5] [--out profiles]
"""

from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import torch  # noqa: E402

from bench_host_async import SEED, gpu_card  # noqa: E402
from bench_host_env import Batch  # noqa: E402

LEGS = ("a_plain", "b_amp", "b_amp_reset", "b_power_amp", "c_workaround")
S = 10
COEF = 0.0005
IN_PLAIN, IN_AMP, IN_POWER_AMP = 1278, 1278 + 552, 1278 + 552 + 276


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--num-envs", type=int, default=4096, help="envs per batch")
    ap.add_argument("--rounds", type=int, default=200, help="rounds per timed loop (two batch-steps each)")
    ap.add_argument("--passes", type=int, default=5, help="timed loops per leg (the median is kept)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"), help="directory of r8_host_amp.{json,md}")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"

    import __graft_entry__ as g

    g.build()
    from humanoid_b200 import HostAmpBuffers, HostDeviceOutputs, HostStep, MotionLib, _cabi, synth

    capi = _cabi.load()
    N, R = args.num_envs, args.rounds
    data = synth.make_motion_lib(N, 60, 300, (30,), seed=SEED, device="cuda")
    lib = MotionLib(data, device="cuda")
    A, B = Batch(data, lib, N, SEED + 1), Batch(data, lib, N, SEED + 32)
    gen = torch.Generator().manual_seed(SEED + 77)
    for bt in (A, B):
        b = bt.bufs
        b.dof_pos = (torch.randn(N, 69, generator=gen) * 0.5).pin_memory()
        b.dof_vel = torch.randn(N, 69, generator=gen).pin_memory()
        bt.dof_force = (torch.randn(N, 69, generator=gen) * 50).pin_memory()
        bt.raw5 = torch.zeros(N, 5).pin_memory()
        bt.dargs = b._args()
        bt.dargs.obs_buf = None  # the rows go to the device tensors
        bt.pargs = b._args()
        bt.pargs.obs_buf, bt.pargs.reward_raw = None, bt.raw5.data_ptr()
        bt.dev = HostDeviceOutputs.allocate(N, 1, "cuda")
        bt.reset_rargs = bt.rargs(_cabi.STATE_INIT_RANDOM)
        bt.env_power = _cabi.PhcHostEnvArgs(bt.dof_force.data_ptr(), b.dof_vel.data_ptr(), COEF, None, None)
        bt.amp = {k: HostAmpBuffers.allocate(N, S, "cuda") for k in ("b_amp", "b_amp_reset", "b_power_amp")}
        # c_workaround: the caller's device copies of the state, dof rows, flags and clock, and its own AMP tensors
        bt.amp["c_workaround"] = HostAmpBuffers.allocate(N, S, "cuda")
        bt.d_state = torch.empty(N, 24, 13, device="cuda")
        bt.d_dofp, bt.d_dofv = torch.empty(N, 69, device="cuda"), torch.empty(N, 69, device="cuda")
        bt.d_reset, bt.d_start = torch.empty(N, dtype=torch.uint8, device="cuda"), torch.empty(N, device="cuda")
        bt.d_ids = b.sampled_motion_ids.cuda()
        bt.d_reposed = torch.zeros(N, dtype=torch.uint8, device="cuda")
        body, bt.keep = _cabi.body_state(bt.d_state[..., 0:3], bt.d_state[..., 3:7], bt.d_state[..., 7:10],
                                         bt.d_state[..., 10:13])  # fmt: skip
        w = bt.amp["c_workaround"]
        x = _cabi.PhcAmpEnvArgs()
        x.body = body
        x.dof_pos, x.dof_vel, x.dof_stride, x.dof_elem_stride = bt.d_dofp.data_ptr(), bt.d_dofv.data_ptr(), 69, 1
        h = w._args(None)
        x.key_body_ids, x.num_key_bodies, x.num_sel, x.dof_subset = h.key_body_ids, h.num_key_bodies, h.num_sel, h.dof_subset
        x.flags, x.num_steps, x.obs_per_step = h.flags, h.num_steps, h.obs_per_step
        x.amp_obs_buf, x.amp_obs_demo_buf = w.amp_obs.data_ptr(), w.amp_obs_demo.data_ptr()
        bt.wx = x
        bt.wi = _cabi.PhcAmpEnvArgs.from_buffer_copy(x)
        bt.wi.init_slot0, bt.wi.env_mask = 1, bt.d_reposed.data_ptr()
    torch.cuda.synchronize()

    def submitter(ctx, kind):
        def sub(s, bt):
            r = C.byref(bt.reset_rargs) if kind == "b_amp_reset" else None
            dev = C.byref(bt.dev._args())
            if kind.startswith("b_"):
                power = kind == "b_power_amp"
                a = bt.pargs if power else bt.dargs
                env = C.byref(bt.env_power) if power else None
                rc = capi.phc_host_step_submit_amp(ctx, s, C.byref(a), r, dev, env, None,
                                                   C.byref(bt.amp[kind]._args(bt.bufs)), N)  # fmt: skip
            else:
                rc = capi.phc_host_step_submit_device(ctx, s, C.byref(bt.dargs), r, dev, N)
            _cabi.check(rc, kind)

        return sub

    def after_wait(bt):
        """c_workaround: the state and dof rows back to the device and the standalone AMP launches, on the
        discriminator's stream."""
        b = bt.bufs
        bt.d_state.copy_(b.state, non_blocking=True)
        bt.d_dofp.copy_(b.dof_pos, non_blocking=True)
        bt.d_dofv.copy_(b.dof_vel, non_blocking=True)
        bt.d_reset.copy_(b.reset_buf, non_blocking=True)
        bt.d_start.copy_(b.motion_start_times, non_blocking=True)
        st = _cabi.stream_ptr("cuda")
        _cabi.check(capi.phc_amp_step(C.byref(bt.wx), N, 1, st), "phc_amp_step")
        _cabi.check(capi.phc_amp_init_ref(lib.handle, C.byref(bt.wi), bt.d_ids.data_ptr(), bt.d_start.data_ptr(),
                                          2 * (1.0 / 60.0), N, st), "phc_amp_init_ref")  # fmt: skip

    def async_loop(ctx, kind):
        sub = submitter(ctx, kind)
        work = kind == "c_workaround"

        def loop(r):
            for s, bt in enumerate((A, B)):
                bt.rewind()
                sub(s, bt)
            for i in range(r):
                for s, bt in enumerate((A, B)):
                    _cabi.check(capi.phc_host_step_wait(ctx, s), "wait")
                    if work:
                        after_wait(bt)
                    if i == r - 1:
                        continue
                    bt.rewind()
                    sub(s, bt)
            torch.cuda.synchronize()

        return loop

    def clear():
        for bt in (A, B):
            for a in bt.amp.values():
                a.amp_obs.zero_()
                a.amp_obs_demo.zero_()
        torch.cuda.synchronize()

    os.environ["PHC_HOST_PATH"] = "direct"
    ctxs = {}
    for kind in LEGS:
        hs = HostStep(lib, N, num_chunks=3, enable_early_termination=kind != "b_amp_reset",
                      use_power_reward=kind == "b_power_amp", rew_power_coef=COEF)  # fmt: skip
        ctxs[kind] = (hs, async_loop(hs._ctx, kind))
        ctxs[kind][1](3)  # warm
    runs = {k: [] for k in LEGS}
    failures = []
    for i in range(args.passes):  # the legs alternate: a drift of the host's load spreads over all of them
        for kind in LEGS:
            clear()
            t0 = time.perf_counter()
            ctxs[kind][1](R)
            runs[kind].append(time.perf_counter() - t0)
            if i == args.passes - 1 and kind == "b_amp":
                for bt in (A, B):
                    bt.last = bt.amp["b_amp"].amp_obs.clone()
    # b_amp's last loop and c_workaround's last loop ran the same R steps from cleared tensors
    for name, bt in (("A", A), ("B", B)):
        x, y = bt.last, bt.amp["c_workaround"].amp_obs
        if not torch.equal(x.view(torch.int32), y.view(torch.int32)):
            failures.append(f"batch {name} amp_obs")
    row = {}
    for kind in LEGS:
        row[f"{kind}_async_us"] = statistics.median(runs[kind]) / (2 * R) * 1e6
        row[f"{kind}_async_spread_us"] = [min(runs[kind]) / (2 * R) * 1e6, max(runs[kind]) / (2 * R) * 1e6]
        hs = ctxs[kind][0]
        assert hs.path == 1 and hs.chunks == 3
    # one host reset of every env, with and without AMP (ctx of a_plain), median of 20 after 3 warm
    hs = ctxs["a_plain"][0]
    resets = {}
    for amp_on in (False, True):
        def reset_once():
            A.rb.env_mask.fill_(1)
            _cabi.check(capi.phc_host_reset_submit_amp(hs._ctx, 0, C.byref(A.dargs), C.byref(A.reset_rargs),
                                                       C.byref(A.dev._args()), None,
                                                       C.byref(A.amp["b_amp"]._args(None)), N)
                        if amp_on else
                        capi.phc_host_reset_submit_device(hs._ctx, 0, C.byref(A.dargs), C.byref(A.reset_rargs),
                                                          C.byref(A.dev._args()), N), "reset")  # fmt: skip
            _cabi.check(capi.phc_host_step_wait(hs._ctx, 0), "wait")

        for _ in range(3):
            reset_once()
        ts = []
        for _ in range(20):
            t0 = time.perf_counter()
            reset_once()
            ts.append(time.perf_counter() - t0)
        resets["with_amp" if amp_on else "without_amp"] = statistics.median(ts) * 1e6
    for kind in LEGS:
        ctxs[kind][0].close()
    os.environ.pop("PHC_HOST_PATH", None)
    env = A.device_env(lib, False)
    env.enable_auto_reset(True)
    env.step(phase_by_env=A.phase)
    reposed = float(env.extras["reset"].float().mean())

    # floors: the H2D bytes with the copy engine alone, min over five loops
    s_in = torch.cuda.Stream()
    floors = {}
    for name, per_env in (("h2d_only_1278", IN_PLAIN), ("h2d_only_1830", IN_AMP), ("h2d_only_2106", IN_POWER_AMP)):
        d_in = torch.empty(N * per_env, dtype=torch.uint8, device="cuda")
        p_in = torch.empty(N * per_env, dtype=torch.uint8).pin_memory()

        def floor_loop(n):
            for _ in range(n):
                with torch.cuda.stream(s_in):
                    d_in.copy_(p_in, non_blocking=True)
                s_in.synchronize()

        floor_loop(3)
        fr = []
        for _ in range(5):
            t0 = time.perf_counter()
            floor_loop(2 * R)
            fr.append(time.perf_counter() - t0)
        floors[name] = min(fr) / (2 * R) * 1e6

    out = {"card": gpu_card(), "num_envs_per_batch": N, "amp_steps": S, "rounds_per_loop": R,
           "timing_repeats": args.passes, "path": "direct", "chunks": 3, "legs": row, "floors_us": floors,
           "host_reset_all_envs_us": resets, "reposed_fraction_per_step": reposed,
           "amp_roll_hbm_bytes_per_batch_step": N * S * 196 * 4 * 2}  # fmt: skip
    out["ratios"] = {
        "b_amp_over_a_plain": row["b_amp_async_us"] / row["a_plain_async_us"],
        "c_workaround_over_a_plain": row["c_workaround_async_us"] / row["a_plain_async_us"],
        "b_power_amp_over_its_h2d_floor": row["b_power_amp_async_us"] / floors["h2d_only_2106"],
    }
    out["b_equals_c_bit_for_bit"] = not failures
    out["mismatches"] = failures
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r8_host_amp.json"), "w") as f:
        f.write(json.dumps(out) + "\n")
    lines = [f"# Host-path AMP observations, {out['card']['name']} ({out['card']['power_limit_and_max_sm_clock']})", "",
             f"Two {N}-env config-2 batches, device obs, direct path, three chunks, two-slot async loop, S = {S}; median "
             f"of {args.passes} loops of {R} rounds, legs alternated.  us per batch-step.", "",
             "| leg | us / batch-step | min .. max |", "|---|---|---|"]  # fmt: skip
    for kind in LEGS:
        lo, hi = row[f"{kind}_async_spread_us"]
        lines.append(f"| {kind} | {row[f'{kind}_async_us']:.1f} | {lo:.1f} .. {hi:.1f} |")
    for name, v in floors.items():
        lines.append(f"| {name} (copy engine alone) | {v:.1f} | |")
    lines += ["", f"One host reset of all {N} envs: {resets['without_amp']:.1f} us without AMP, "
              f"{resets['with_amp']:.1f} us with it (median of 20).",
              f"Re-posed fraction per step in b_amp_reset: {reposed:.3f}.",
              f"Ratios: {json.dumps(out['ratios'])}",
              f"b_amp and c_workaround give the same amp_obs bit for bit: {not failures}", ""]  # fmt: skip
    with open(os.path.join(args.out, "r8_host_amp.md"), "w") as f:
        f.write("\n".join(lines))
    print(json.dumps(out), flush=True)
    if failures:
        sys.exit(1)


if __name__ == "__main__":
    main()
