"""Episode bookkeeping on the host-buffer path (phc_host_step_submit_episode): what PHCPufferEnv.step's per-step
bookkeeping costs when the host step does it, against the step without it and against doing it after the step.

The harness of bench_host_env_options.py (r6): config 2, two 4096-env batches (bench_host_env.Batch), device obs, direct
path with three chunks, the two-slot async loop, median of --passes loops of --rounds rounds (one round = one step of
batch A and one of B).  Legs, alternated in one run:

  a_plain          phc_host_step_submit_device: the step without bookkeeping
  b_episode        phc_host_step_submit_episode: the same step with the bookkeeping into device tensors
  a_plain_reset    phc_host_step_submit_device with random auto-reset, early termination off: the ~4 % clip-end envs
                   are re-posed every step (r5 / r6's reset rate)
  b_episode_reset  the same with the bookkeeping
  c_workaround     a_plain, then after each wait: H2D copies of rew_buf / reset_buf / terminate_buf / reward_raw and
                   phc_episode_update on the learner's stream (what a host loop had to do before)

The learner's stream is the current torch stream, the one the device outputs and the episode tensors name; the copies
of c_workaround sit on it, so the next submit's kernels (which wait for that stream) do not overwrite the host rows
before they are read.  Each leg's loop ends with a device synchronise.  The episode tensors of b_episode and
c_workaround are cleared before every loop and compared bit for bit after the last one; a mismatch fails the run.
Writes r7_host_episode.{json,md} to --out and prints the JSON.

    python profiles/bench_host_episode.py [--rounds 200] [--passes 5] [--out profiles]
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

LEGS = ("a_plain", "b_episode", "a_plain_reset", "b_episode_reset", "c_workaround")
EP_FIELDS = ("terminals", "truncations", "masks", "episode_returns", "episode_lengths")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--num-envs", type=int, default=4096, help="envs per batch")
    ap.add_argument("--rounds", type=int, default=200, help="rounds per timed loop (two batch-steps each)")
    ap.add_argument("--passes", type=int, default=5, help="timed loops per leg (the median is kept)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"), help="directory of r7_host_episode.{json,md}")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"

    import __graft_entry__ as g

    g.build()
    from humanoid_b200 import HostDeviceOutputs, HostEpisodeBuffers, HostStep, MotionLib, _cabi, synth

    capi = _cabi.load()
    N, R = args.num_envs, args.rounds
    data = synth.make_motion_lib(N, 60, 300, (30,), seed=SEED, device="cuda")
    lib = MotionLib(data, device="cuda")
    A, B = Batch(data, lib, N, SEED + 1), Batch(data, lib, N, SEED + 32)
    for bt in (A, B):
        bt.dargs = bt.bufs._args()
        bt.dargs.obs_buf = None  # the rows go to the device tensors
        bt.dev = HostDeviceOutputs.allocate(N, 1, "cuda")
        bt.reset_rargs = bt.rargs(_cabi.STATE_INIT_RANDOM)
        bt.ep = {k: HostEpisodeBuffers.allocate(N, 4, "cuda") for k in ("b_episode", "b_episode_reset", "c_workaround")}
        # c_workaround: device copies of the host outputs, and phc_episode_update's own sums
        bt.d_rew, bt.d_raw = torch.empty(N, device="cuda"), torch.empty(N, 4, device="cuda")
        bt.d_reset, bt.d_term = torch.empty(N, dtype=torch.uint8, device="cuda"), torch.empty(N, dtype=torch.uint8, device="cuda")
        bt.stats, bt.raw_rewards = torch.zeros(4, dtype=torch.float64, device="cuda"), torch.zeros(4, device="cuda")
        bt.ws = torch.zeros(16, dtype=torch.float64, device="cuda")  # PHC_EPISODE_WORKSPACE_DOUBLES
        e = bt.ep["c_workaround"]
        a = _cabi.PhcEpisodeArgs()
        a.reset, a.terminate, a.rewards = bt.d_reset.data_ptr(), bt.d_term.data_ptr(), bt.d_rew.data_ptr()
        a.reward_raw, a.reward_raw_stride, a.reward_raw_cols = bt.d_raw.data_ptr(), 4, 4
        a.terminals, a.truncations, a.masks = e.terminals.data_ptr(), e.truncations.data_ptr(), e.masks.data_ptr()
        a.episode_returns, a.episode_lengths = e.episode_returns.data_ptr(), e.episode_lengths.data_ptr()
        a.stats, a.raw_rewards, a.workspace = bt.stats.data_ptr(), bt.raw_rewards.data_ptr(), bt.ws.data_ptr()
        bt.upd = a
    torch.cuda.synchronize()

    def submitter(ctx, kind):
        def sub(s, bt):
            r = C.byref(bt.reset_rargs) if kind.endswith("_reset") else None
            if kind.startswith("b_"):
                rc = capi.phc_host_step_submit_episode(ctx, s, C.byref(bt.dargs), r, C.byref(bt.dev._args()), None,
                                                       C.byref(bt.ep[kind]._args()), N)  # fmt: skip
            else:
                rc = capi.phc_host_step_submit_device(ctx, s, C.byref(bt.dargs), r, C.byref(bt.dev._args()), N)
            _cabi.check(rc, kind)

        return sub

    def after_wait(bt):
        """c_workaround: the host outputs back to the device and the standalone bookkeeping, on the learner's stream."""
        b = bt.bufs
        bt.d_rew.copy_(b.rew_buf, non_blocking=True)
        bt.d_reset.copy_(b.reset_buf, non_blocking=True)
        bt.d_term.copy_(b.terminate_buf, non_blocking=True)
        bt.d_raw.copy_(b.reward_raw, non_blocking=True)
        _cabi.check(capi.phc_episode_update(C.byref(bt.upd), N, _cabi.stream_ptr("cuda")), "phc_episode_update")

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
            for e in bt.ep.values():
                e.reset()
                e.episode_returns.zero_()
                e.episode_lengths.zero_()
            bt.stats.zero_()
            bt.raw_rewards.zero_()
        torch.cuda.synchronize()

    os.environ["PHC_HOST_PATH"] = "direct"
    ctxs = {}
    for kind in LEGS:
        hs = HostStep(lib, N, num_chunks=3, enable_early_termination=not kind.endswith("_reset"))
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
            if i == args.passes - 1 and kind == "b_episode":
                for bt in (A, B):
                    bt.last = {k: v.clone() for k, v in ((f, getattr(bt.ep["b_episode"], f)) for f in EP_FIELDS)}
    # b_episode's last loop and c_workaround's last loop ran the same R steps from cleared tensors
    for name, bt in (("A", A), ("B", B)):
        e = bt.ep["c_workaround"]
        for f in EP_FIELDS:
            x, y = bt.last[f], getattr(e, f)
            same = torch.equal(x.view(torch.int32), y.view(torch.int32)) if x.dtype == torch.float32 else torch.equal(x, y)
            if not same:
                failures.append(f"batch {name} {f}")
    row = {}
    for kind in LEGS:
        row[f"{kind}_async_us"] = statistics.median(runs[kind]) / (2 * R) * 1e6
        row[f"{kind}_async_spread_us"] = [min(runs[kind]) / (2 * R) * 1e6, max(runs[kind]) / (2 * R) * 1e6]
        hs = ctxs[kind][0]
        assert hs.path == 1 and hs.chunks == 3
        hs.close()
    os.environ.pop("PHC_HOST_PATH", None)
    env = A.device_env(lib, False)
    env.enable_auto_reset(True)
    env.step(phase_by_env=A.phase)
    reposed = float(env.extras["reset"].float().mean())

    out = {"card": gpu_card(), "num_envs_per_batch": N, "rounds_per_loop": R, "timing_repeats": args.passes,
           "path": "direct", "chunks": 3, "legs": row, "reposed_fraction_per_step": reposed}  # fmt: skip
    out["ratios"] = {
        "b_episode_over_a_plain": row["b_episode_async_us"] / row["a_plain_async_us"],
        "b_episode_reset_over_a_plain_reset": row["b_episode_reset_async_us"] / row["a_plain_reset_async_us"],
        "c_workaround_over_a_plain": row["c_workaround_async_us"] / row["a_plain_async_us"],
    }
    out["b_equals_c_bit_for_bit"] = not failures
    out["mismatches"] = failures
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r7_host_episode.json"), "w") as f:
        f.write(json.dumps(out) + "\n")
    lines = [f"# Host-path episode bookkeeping, {out['card']['name']} ({out['card']['power_limit_and_max_sm_clock']})", "",
             f"Two {N}-env config-2 batches, device obs, direct path, three chunks, two-slot async loop; median of "
             f"{args.passes} loops of {R} rounds, legs alternated.  us per batch-step.", "",
             "| leg | us / batch-step | min .. max |", "|---|---|---|"]  # fmt: skip
    for kind in LEGS:
        lo, hi = row[f"{kind}_async_spread_us"]
        lines.append(f"| {kind} | {row[f'{kind}_async_us']:.1f} | {lo:.1f} .. {hi:.1f} |")
    lines += ["", f"Re-posed fraction per step in the _reset legs: {reposed:.3f}.",
              f"Ratios: {json.dumps(out['ratios'])}",
              f"b_episode and c_workaround give the same episode tensors bit for bit: {not failures}", ""]  # fmt: skip
    with open(os.path.join(args.out, "r7_host_episode.md"), "w") as f:
        f.write("\n".join(lines))
    print(json.dumps(out), flush=True)
    if failures:
        sys.exit(1)


if __name__ == "__main__":
    main()
