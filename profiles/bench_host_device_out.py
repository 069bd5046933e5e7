"""Host step with device outputs (phc_host_step_submit_device / phc_host_reset_submit_device) against the host-obs step.

Config 2 and the two 4096-env batches of bench_host_env.py (its Batch: 4 % of the envs past their clip end, 30 % far
from their reference).  Legs, each timed with a host clock around loops that end in a wait, median of 5 loops of
--rounds rounds (one round = one step of batch A and one of batch B), async (two slots) and sync (slot 0, one step
at a time):

  host_obs        phc_host_step_submit: obs rows to pinned host memory (the r3 / r4 baseline, re-measured here)
  host_obs_copy   the same plus what a caller with a GPU policy adds today: dev_obs.copy_(obs_buf, non_blocking=True)
                  after each wait, synchronised before that batch's next submit (which rewrites obs_buf)
  dev_obs         phc_host_step_submit_device: obs rows into a CUDA tensor
  dev_norm_mom    dev_obs plus bf16 obs_norm and 32 buckets of moments
  dev_clip_end    dev_obs with auto-reset, early termination off: the 4 % clip-end envs are re-posed each step
  full_reset      phc_host_reset_submit of all 4096 envs of batch A + wait, host obs vs device obs, per call
  schedules       dev_obs on the direct and the staged path at 2 / 3 / 4 chunks

All but the schedules leg run on the direct path with three chunks (the tuner's choice on the B200,
profiles/r3_host_async.md; device-output submits use the settled schedule as the other submits do).  Floors: the
same bytes with the copy engines alone, H2D only (sim state + clock) and D2H only (the scalars a device-out step
returns; also the host-obs step's D2H).  The last outputs of every loop are compared bit for bit with the device path
(HumanoidPHC on the same inputs): a mismatch fails the run.  Bytes per batch-step and direction are computed from the
shapes.  Prints one JSON line.

    python profiles/bench_host_device_out.py [--rounds 200]
    PHC_HOST_TRACE=1 python profiles/bench_host_device_out.py --trace   # per-chunk timeline of dev_obs async (stderr;
                                                                        # direct unless PHC_HOST_PATH says otherwise)
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
from bench_host_env import ROW_BYTES, Batch  # noqa: E402

OUT_BYTES = 4 + 16 + 2 + 1 + 1  # rew | reward_raw[:, :4] | progress | reset | terminate per env


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--num-envs", type=int, default=4096, help="envs per batch")
    ap.add_argument("--rounds", type=int, default=200, help="rounds per timed loop (two batch-steps each)")
    ap.add_argument("--trace", action="store_true", help="only run dev_obs async (with PHC_HOST_TRACE=1 set)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"

    import __graft_entry__ as g

    g.build()
    from humanoid_b200 import HostDeviceOutputs, HostStep, MotionLib, RunningNorm, _cabi, synth

    capi = _cabi.load()
    N, R = args.num_envs, args.rounds
    data = synth.make_motion_lib(N, 60, 300, (30,), seed=SEED, device="cuda")
    lib = MotionLib(data, device="cuda")
    A, B = Batch(data, lib, N, SEED + 1), Batch(data, lib, N, SEED + 32)
    D = _cabi.SELF_OBS_DIM + _cabi.TASK_OBS_DIM
    rn = RunningNorm(D, device="cuda")
    g_ = torch.Generator(device="cuda").manual_seed(SEED)
    rn.running_mean.copy_(torch.randn(1, D, generator=g_, device="cuda") * 0.3)
    rn.running_var.copy_(torch.rand(1, D, generator=g_, device="cuda") * 2 + 0.05)
    for bt in (A, B):
        bt.dargs = bt.bufs._args()
        bt.dargs.obs_buf = None  # the rows go to the device tensors
        bt.dev = HostDeviceOutputs.allocate(N, 1, "cuda")
        bt.dev_nm = HostDeviceOutputs.allocate(N, 1, "cuda", norm_dtype=torch.bfloat16, normalizer=rn, moments=True)
        bt.copy_dst = torch.empty(N, D, device="cuda")
    torch.cuda.synchronize()
    out = {"card": gpu_card(), "num_envs_per_batch": N, "rounds_per_loop": R, "timing_repeats": 5}
    failures = []

    def timed(loop, n_steps):
        loop(3)  # warm
        runs = []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            loop(R)
            runs.append(time.perf_counter() - t0)
        return statistics.median(runs) / n_steps * 1e6

    def submitter(ctx, kind):
        """submit(slot, batch) and the work done after its wait, for one leg."""
        after = lambda bt: None  # noqa: E731
        if kind in ("host_obs", "host_obs_copy"):
            sub = lambda s, bt: _cabi.check(capi.phc_host_step_submit(ctx, s, C.byref(bt.args), bt.N), "submit")  # noqa: E731
            if kind == "host_obs_copy":
                def after(bt):
                    bt.copy_dst.copy_(bt.bufs.obs_buf, non_blocking=True)
                    torch.cuda.current_stream().synchronize()  # the next submit of this batch rewrites obs_buf
            return sub, after
        field = "dev_nm" if kind == "dev_norm_mom" else "dev"
        rargs = {id(bt): bt.rargs(_cabi.STATE_INIT_RANDOM) for bt in (A, B)}

        def sub(s, bt):
            r = C.byref(rargs[id(bt)]) if kind == "dev_clip_end" else None
            d = getattr(bt, field)._args()
            _cabi.check(capi.phc_host_step_submit_device(ctx, s, C.byref(bt.dargs), r, C.byref(d), bt.N), "submit_device")

        return sub, after

    def sync_loop(ctx, kind):
        sub, after = submitter(ctx, kind)

        def loop(r):
            for _ in range(r):
                for bt in (A, B):
                    bt.rewind()
                    sub(0, bt)
                    _cabi.check(capi.phc_host_step_wait(ctx, 0), "wait")
                    after(bt)
        return loop

    def async_loop(ctx, kind):
        sub, after = submitter(ctx, kind)

        def loop(r):
            for s, bt in enumerate((A, B)):
                bt.rewind()
                sub(s, bt)
            for i in range(r):
                for s, bt in enumerate((A, B)):
                    _cabi.check(capi.phc_host_step_wait(ctx, s), "wait")
                    after(bt)
                    if i == r - 1:
                        continue
                    bt.rewind()
                    sub(s, bt)
        return loop

    def matches(bt, kind):
        """The last outputs equal one step (or reset) of the device path on the same inputs."""
        b = bt.bufs
        if kind == "full_reset_dev":
            env = bt.device_env(lib, True)
            env.reset(None, bt.phase)
            torch.cuda.synchronize()
            return torch.equal(bt.dev.obs, env.obs_buf) and int(b.progress_buf.abs().max()) == 0
        env = bt.device_env(lib, kind != "dev_clip_end")
        if kind == "dev_clip_end":
            env.enable_auto_reset(True)
        if kind == "dev_norm_mom":
            env.set_obs_normalizer(rn, torch.bfloat16)
        env.step(phase_by_env=bt.phase)
        flags = (env.extras["reset"], env.extras["terminate"]) if kind == "dev_clip_end" else (env.reset_buf, env._terminate_buf)
        torch.cuda.synchronize()
        obs = {"host_obs": b.obs_buf, "host_obs_copy": bt.copy_dst, "dev_norm_mom": bt.dev_nm.obs}.get(kind, bt.dev.obs)
        ok = torch.equal(obs.to(env.obs_buf.device), env.obs_buf)
        if kind == "dev_norm_mom":
            ok = ok and torch.equal(bt.dev_nm.obs_norm, env.obs_norm_buf)
        ok = ok and torch.equal(b.rew_buf, env.rew_buf.cpu()) and torch.equal(b.reward_raw, env.reward_raw[:, :4].cpu())
        ok = ok and torch.equal(b.reset_buf.bool(), flags[0].cpu()) and torch.equal(b.terminate_buf.bool(), flags[1].cpu())
        return ok and torch.equal(b.progress_buf, env.progress_buf.cpu())

    def leg(ctx, kind, row, modes=("async", "sync")):
        for mode in modes:
            loop = async_loop(ctx, kind) if mode == "async" else sync_loop(ctx, kind)
            row[f"{kind}_{mode}_us"] = timed(loop, 2 * R)
            for name, bt in (("A", A), ("B", B)):
                if not matches(bt, kind):
                    failures.append(f"{kind} {mode} batch {name}")

    if args.trace:
        os.environ.setdefault("PHC_HOST_PATH", "direct")
        with HostStep(lib, N, num_chunks=3) as hs:
            row = {}
            leg(hs._ctx, "dev_obs", row, ("async",))
        print(json.dumps({"trace_run": row, "matches_device_path": not failures}), flush=True)
        sys.exit(1 if failures else 0)

    h2d = N * (24 * 13 * 4 + 8 + 12 + 4 + 4 + 2)
    d2h_host, d2h_dev = N * (D * 4 + OUT_BYTES), N * OUT_BYTES
    main_row = {"path": "direct", "chunks": 3}
    os.environ["PHC_HOST_PATH"] = "direct"
    for kind in ("host_obs", "host_obs_copy", "dev_obs", "dev_norm_mom", "dev_clip_end"):
        with HostStep(lib, N, num_chunks=3, enable_early_termination=kind != "dev_clip_end") as hs:
            assert int(capi.phc_host_step_h2d_bytes(hs._ctx, N)) == h2d
            assert int(capi.phc_host_step_d2h_bytes(hs._ctx, N)) == d2h_host
            leg(hs._ctx, kind, main_row)
            if kind == "dev_clip_end":
                env = A.device_env(lib, False)
                env.enable_auto_reset(True)
                env.step(phase_by_env=A.phase)
                frac = float(env.extras["reset"].float().mean())
                main_row["dev_clip_end_reposed_fraction"] = frac
                main_row["dev_clip_end_d2h_bytes"] = d2h_dev + int(round(frac * N)) * ROW_BYTES
            assert hs.path == 1 and hs.chunks == 3
    # the first observation of a batch: a host reset of every env, host obs vs device obs
    with HostStep(lib, N, num_chunks=3) as hs:
        ctx = hs._ctx
        rargs = A.rargs(_cabi.STATE_INIT_RANDOM)

        def reset_loop(dev):
            def loop(r):
                for _ in range(r):
                    if dev:
                        d = A.dev._args()
                        _cabi.check(capi.phc_host_reset_submit_device(ctx, 0, C.byref(A.dargs), C.byref(rargs), C.byref(d), N),
                                    "reset_submit_device")  # fmt: skip
                    else:
                        _cabi.check(capi.phc_host_reset_submit(ctx, 0, C.byref(A.args), C.byref(rargs), N), "reset_submit")
                    _cabi.check(capi.phc_host_step_wait(ctx, 0), "wait")
            return loop

        main_row["full_reset_host_obs_us"] = timed(reset_loop(False), R)
        main_row["full_reset_dev_obs_us"] = timed(reset_loop(True), R)
        if not matches(A, "full_reset_dev"):
            failures.append("full_reset_dev")
        main_row["full_reset_h2d_bytes"] = N * (8 + 12 + 4 + 4 + 2 + 4 + 1)
        main_row["full_reset_host_obs_d2h_bytes"] = N * (D * 4 + ROW_BYTES + 2)
        main_row["full_reset_dev_obs_d2h_bytes"] = N * (ROW_BYTES + 2)
    out["legs"] = main_row

    sched = []
    for path in ("direct", "staged"):
        os.environ["PHC_HOST_PATH"] = path
        for ch in (2, 3, 4):
            with HostStep(lib, N, num_chunks=ch) as hs:
                row = {"path": path, "chunks": ch}
                leg(hs._ctx, "dev_obs", row)
                assert hs.path == (1 if path == "direct" else 2) and hs.chunks == ch
                sched.append(row)
    os.environ.pop("PHC_HOST_PATH", None)
    out["dev_obs_schedules"] = sched

    # floors for the same bytes with the copy engines alone: min over five loops
    d_in = torch.empty(h2d, dtype=torch.uint8, device="cuda")
    p_in = torch.empty(h2d, dtype=torch.uint8).pin_memory()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    floors = {}
    for name, nbytes, inbound in (("h2d_only", h2d, True), ("d2h_only_dev_out", d2h_dev, False),
                                  ("d2h_only_host_obs", d2h_host, False)):  # fmt: skip
        d_out = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        p_out = torch.empty(nbytes, dtype=torch.uint8).pin_memory()

        def floor_loop(n):
            for _ in range(n):
                if inbound:
                    with torch.cuda.stream(s_in):
                        d_in.copy_(p_in, non_blocking=True)
                    s_in.synchronize()
                else:
                    with torch.cuda.stream(s_out):
                        p_out.copy_(d_out, non_blocking=True)
                    s_out.synchronize()

        floor_loop(3)
        fr = []
        for _ in range(5):
            t0 = time.perf_counter()
            floor_loop(2 * R)
            fr.append(time.perf_counter() - t0)
        floors[name] = min(fr) / (2 * R) * 1e6
    out["floor_us"] = floors
    out["h2d_bytes_per_batch_step"] = h2d
    out["d2h_bytes_per_batch_step"] = {"host_obs": d2h_host, "dev_obs": d2h_dev}
    out["goals"] = {
        "dev_obs_async_over_h2d_floor": main_row["dev_obs_async_us"] / floors["h2d_only"],
        "dev_obs_async_over_host_obs_copy_async": main_row["dev_obs_async_us"] / main_row["host_obs_copy_async_us"],
    }
    out["matches_device_path"] = not failures
    out["mismatches"] = failures
    print(json.dumps(out), flush=True)
    if failures:
        sys.exit(1)


if __name__ == "__main__":
    main()
