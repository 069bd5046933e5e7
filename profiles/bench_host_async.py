"""The asynchronous host step (phc_host_step_submit / _wait) against the synchronous call, on the headline workload.

Config 2 (one 60-300 frame clip per env, aligned clocks), 4096 envs per batch, built with humanoid_b200.synth as
bench.py builds it.  Legs, each timed with a host clock around loops that end in a wait, median of 5 loops of
--rounds rounds (one round = one step of batch A and one of batch B), after the tuner has settled:

  sync_auto        phc_host_step on batch A alone, schedule tuned by the library (bench.py's `e2e`)
  sync / async     per (output path, chunk count): two batches alternating, synchronously (step A, step B) or over the
                   two slots (submit A, submit B, wait A, submit A, wait B, submit B, ...): us per batch-step
  *_work           the same loops with a fixed host busy-wait (--work-us, a stand-in for policy inference) between a
                   batch's submit and its wait (sync: after each step)
  floor            the same bytes with the copy engines alone (bench.py's method): duplex, D2H only, H2D only

The timed loops call the C ABI through ctypes with prebuilt argument structs, as bench.py does, so the figures are the
library's and not the Python wrapper's.  Every loop rewinds the clocks before each step, and its last outputs are
compared bit for bit with the device path (HumanoidPHC.step) on the same inputs: a mismatch fails the run.  Prints one
JSON line.

    python profiles/bench_host_async.py [--rounds 200] [--work-us 200]
"""

from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SEED = 1234  # bench.py's


def gpu_card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()  # fmt: skip
    except Exception as e:  # the figure is reported as unknown, not guessed
        q = f"unknown ({e})"
    return {"name": name, "power_limit_and_max_sm_clock": q}


class Batch:
    def __init__(self, data, lib, N, seed):
        from humanoid_b200 import HostStepBuffers, HumanoidPHC, synth

        clock = synth.make_clock(data, N, seed=seed, ids="mod", aligned=True, max_progress=30)
        ref = lib.get_motion_state(clock.sampled_motion_ids, synth.reward_time(clock, extra_steps=1), clock.global_offset)
        state = synth.make_sim_state(ref, seed=seed + 1)
        env = HumanoidPHC(lib, N, device="cuda")
        env.set_sim_state(state)
        env.set_clock(clock)
        env.step()
        torch.cuda.synchronize()
        self.want = [env.obs_buf.cpu(), env.rew_buf.cpu(), env.reward_raw[:, :4].cpu(), env.reset_buf.cpu(),
                     env._terminate_buf.cpu(), env.progress_buf.cpu()]  # fmt: skip
        self.prog0 = clock.progress_buf.cpu().pin_memory()
        b = HostStepBuffers.allocate(N, 1, pinned=True)
        for k, v in (("state", state), ("progress_buf", clock.progress_buf), ("motion_start_times", clock.motion_start_times),
                     ("motion_start_times_offset", clock.motion_start_times_offset), ("global_offset", clock.global_offset),
                     ("sampled_motion_ids", clock.sampled_motion_ids)):  # fmt: skip
            getattr(b, k).copy_(v.cpu())
        self.bufs, self.args, self.N = b, b._args(), N

    def rewind(self):
        self.bufs.progress_buf.copy_(self.prog0)

    def matches(self):
        b = self.bufs
        got = [b.obs_buf, b.rew_buf, b.reward_raw, b.reset_buf.bool(), b.terminate_buf.bool(), b.progress_buf]
        return all(torch.equal(g, w) for g, w in zip(got, self.want))


def busy(us):
    if us > 0:
        t = time.perf_counter() + us * 1e-6
        while time.perf_counter() < t:
            pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--num-envs", type=int, default=4096, help="envs per batch")
    ap.add_argument("--rounds", type=int, default=200, help="rounds per timed loop (two batch-steps each)")
    ap.add_argument("--work-us", type=float, default=200.0, help="host work between a batch's submit and its wait")
    ap.add_argument("--chunks", default="2,3,4")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"

    import __graft_entry__ as g

    g.build()
    from humanoid_b200 import HostStep, MotionLib, _cabi, synth

    capi = _cabi.load()
    N, R, W = args.num_envs, args.rounds, args.work_us
    data = synth.make_motion_lib(N, 60, 300, (30,), seed=SEED, device="cuda")
    lib = MotionLib(data, device="cuda")
    A, B = Batch(data, lib, N, SEED + 1), Batch(data, lib, N, SEED + 32)
    torch.cuda.synchronize()
    out = {"card": gpu_card(), "num_envs_per_batch": N, "rounds_per_loop": R, "timing_repeats": 5, "work_us": W}
    failures = []

    def check(what, *batches):
        for bt in batches:
            if not bt.matches():
                failures.append(what)

    def timed(loop, n_steps):
        loop(3)  # warm
        runs = []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            loop(R)
            runs.append(time.perf_counter() - t0)
        return statistics.median(runs) / n_steps * 1e6

    def sync_loop(ctx, batches, work):
        def loop(r):
            for _ in range(r):
                for bt in batches:
                    bt.rewind()
                    _cabi.check(capi.phc_host_step(ctx, C.byref(bt.args), bt.N), "phc_host_step")
                    busy(work)
        return loop

    def async_loop(ctx, work):
        def loop(r):
            for s, bt in enumerate((A, B)):
                bt.rewind()
                _cabi.check(capi.phc_host_step_submit(ctx, s, C.byref(bt.args), bt.N), "submit")
            for i in range(r):
                for s, bt in enumerate((A, B)):
                    _cabi.check(capi.phc_host_step_wait(ctx, s), "wait")
                    if i == r - 1:
                        continue
                    busy(work)  # the policy on this batch's outputs, while the other batch steps
                    bt.rewind()
                    _cabi.check(capi.phc_host_step_submit(ctx, s, C.byref(bt.args), bt.N), "submit")
        return loop

    # ---- 1. the synchronous call, schedule tuned by the library (bench.py's e2e)
    os.environ.pop("PHC_HOST_PATH", None)
    with HostStep(lib, N, num_chunks=0) as hs:
        ctx = hs._ctx
        for _ in range(capi.phc_host_step_tuning_calls(ctx) + 4):
            A.rewind()
            _cabi.check(capi.phc_host_step(ctx, C.byref(A.args), N), "phc_host_step")
        h2d, d2h = int(capi.phc_host_step_h2d_bytes(ctx, N)), int(capi.phc_host_step_d2h_bytes(ctx, N))
        out["sync_auto"] = {"us_per_call": timed(sync_loop(ctx, [A], 0.0), R), "path": hs.path, "chunks": hs.chunks}
        check("sync_auto", A)
        # the async loop on the tuned schedule
        out["async_auto"] = {"us_per_batch_step": timed(async_loop(ctx, 0.0), 2 * R)}
        check("async_auto", A, B)

    # ---- 2. / 3. per output path and chunk count, without and with caller work
    rows = []
    for path in ("direct", "staged"):
        for ch in [int(c) for c in args.chunks.split(",")]:
            os.environ["PHC_HOST_PATH"] = path
            with HostStep(lib, N, num_chunks=ch) as hs:
                ctx = hs._ctx
                row = {"path": path, "chunks": ch}
                for name, loop in (("sync", sync_loop(ctx, [A, B], 0.0)), ("async", async_loop(ctx, 0.0)),
                                   ("sync_work", sync_loop(ctx, [A, B], W)), ("async_work", async_loop(ctx, W))):  # fmt: skip
                    row[name] = timed(loop, 2 * R)
                    check(f"{name} {path} x{ch}", A, B)
                assert hs.path == (1 if path == "direct" else 2) and hs.chunks == ch
                rows.append(row)
    os.environ.pop("PHC_HOST_PATH", None)
    out["per_schedule_us_per_batch_step"] = rows

    # ---- 4. floors for the same bytes (bench.py:632-662): min over five loops
    d_in = torch.empty(h2d, dtype=torch.uint8, device="cuda")
    d_out = torch.empty(d2h, dtype=torch.uint8, device="cuda")
    p_in = torch.empty(h2d, dtype=torch.uint8).pin_memory()
    p_out = torch.empty(d2h, dtype=torch.uint8).pin_memory()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

    def floor_loop(n, both=True, outb=True):
        for _ in range(n):
            if both or not outb:
                with torch.cuda.stream(s_in):
                    d_in.copy_(p_in, non_blocking=True)
            if both or outb:
                with torch.cuda.stream(s_out):
                    p_out.copy_(d_out, non_blocking=True)
            s_in.synchronize()
            s_out.synchronize()

    floors = {}
    for name, kw in (("duplex", {}), ("d2h_only", dict(both=False, outb=True)), ("h2d_only", dict(both=False, outb=False))):
        floor_loop(3, **kw)
        fr = []
        for _ in range(5):
            t0 = time.perf_counter()
            floor_loop(2 * R, **kw)
            fr.append(time.perf_counter() - t0)
        floors[name] = min(fr) / (2 * R) * 1e6
    out["floor_us"] = floors
    out["h2d_bytes_per_batch_step"], out["d2h_bytes_per_batch_step"] = h2d, d2h
    out["matches_device_path"] = not failures
    out["mismatches"] = failures
    print(json.dumps(out), flush=True)
    if failures:
        sys.exit(1)


if __name__ == "__main__":
    main()
