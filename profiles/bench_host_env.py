"""Resets on the host-buffer path (phc_host_step_submit_reset / phc_host_reset_submit) against the plain host step.

Config 2 (one 60-300 frame clip per env, aligned clocks) as bench_host_async.py builds it: two batches of 4096 envs
on the two slots, direct path, three chunks (the schedule the tuner keeps on the B200, profiles/r3_host_async.md).
The clocks are set so that 4 % of the envs are past their clip end at the step (every 25th env) and the sim state so
that 30 % are far from their reference (every env with index % 10 < 3, all bodies moved 1 m).  Legs, each timed with
a host clock around loops that end in a wait, median of 5 loops of --rounds rounds (one round = one step of batch A and
one of batch B):

  plain          phc_host_step_submit / wait: no reset (the r3 baseline, re-measured here)
  clip_end       submit with auto-reset, early termination off: the 4 % clip-end envs are re-posed each step
  flag30         submit with auto-reset, early termination on: ~33 % of the envs are re-posed each step
  *_sync         the same steps one at a time (submit + wait on slot 0), batches alternating
  full_reset     phc_host_reset_submit of all 4096 envs of batch A + wait (the first observation), per call

Every loop rewinds the progress before each step, as bench_host_async.py does.  The re-posed envs' state and clock go to
scratch buffers (the C ABI's outs need not alias the inputs), so the inputs, and with them the flagged set, are the
same in every step and the rows cross the link as in a real loop.  The last outputs of every loop are compared bit for
bit with the device path (HumanoidPHC with auto-reset, or HumanoidPHC.reset) on the same inputs: a mismatch fails the
run.  Bytes per call and direction are computed from the shapes.  Prints one JSON line.

    python profiles/bench_host_env.py [--rounds 200]
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

DT = 2 * (1.0 / 60.0)
PROGRESS = 5  # terminations need progress > 1
ROW_BYTES = 24 * 13 * 4 + 13 * 4 + 2 * 69 * 4 + 5 * 4 + 2  # state | root | dof pos, vel | clock | progress of a re-posed env


class Batch:
    def __init__(self, data, lib, N, seed):
        from humanoid_b200 import HostResetBuffers, HostStepBuffers, synth

        self.N = N
        g = torch.Generator(device="cuda").manual_seed(seed)
        ids = torch.arange(N, device="cuda") % data.num_motions
        nf = data.motion_num_frames[ids]
        mlen = data.motion_lengths[ids]
        # start times k / 30 that stay short of the clip end at the reward time, except for every 25th env
        k = (torch.rand(N, generator=g, device="cuda") * (nf - 14).float()).long()
        start = (k * (1 / 30)).to(torch.float32)
        past = torch.arange(N, device="cuda") % 25 == 0
        start[past] = mlen[past]
        goff = torch.randn(N, 3, generator=g, device="cuda")
        goff[:, 2] = 0
        self.clock = synth.Clock(progress_buf=torch.full((N,), PROGRESS, dtype=torch.int16, device="cuda"),
                                 motion_start_times=start, motion_start_times_offset=torch.zeros(N, device="cuda"),
                                 global_offset=goff, sampled_motion_ids=ids)  # fmt: skip
        ref = lib.get_motion_state(ids, synth.reward_time(self.clock, extra_steps=1), goff)
        state = synth.make_sim_state(ref, seed=seed + 1, pos_sigma_lo=0.002, pos_sigma_hi=0.01, rot_sigma=0.01)
        state[(torch.arange(N, device="cuda") % 10) < 3, :, 0] += 1.0
        self.state = state
        self.phase = torch.rand(N, generator=g, device="cuda")
        b = HostStepBuffers.allocate(N, 1, pinned=True)
        for name, v in (("state", state), ("progress_buf", self.clock.progress_buf),
                        ("motion_start_times", start), ("motion_start_times_offset", self.clock.motion_start_times_offset),
                        ("global_offset", goff), ("sampled_motion_ids", ids)):  # fmt: skip
            getattr(b, name).copy_(v.cpu())
        self.prog0 = b.progress_buf.clone().pin_memory()
        r = HostResetBuffers.allocate(N, pinned=True)
        r.phase.copy_(self.phase.cpu())
        r.env_mask.fill_(1)
        self.out = HostStepBuffers.allocate(N, 1, pinned=True)  # scratch for the re-posed envs' state and clock
        self.bufs, self.rb, self.args = b, r, b._args()

    def rargs(self, capi_state_init):
        from humanoid_b200 import _cabi

        o, r = self.out, self.rb
        return _cabi.PhcHostResetArgs(r.phase.data_ptr(), r.env_mask.data_ptr(), capi_state_init, 0, o.state.data_ptr(),
                                      r.root_states.data_ptr(), r.dof_pos.data_ptr(), r.dof_vel.data_ptr(),
                                      o.motion_start_times.data_ptr(), o.motion_start_times_offset.data_ptr(),
                                      o.global_offset.data_ptr())  # fmt: skip

    def rewind(self):
        self.bufs.progress_buf.copy_(self.prog0)

    def device_env(self, lib, early):
        from humanoid_b200 import HumanoidPHC

        env = HumanoidPHC(lib, self.N, device="cuda", enable_early_termination=early)
        env.set_sim_state(self.state)
        env.set_clock(self.clock)
        return env

    def matches(self, lib, kind):
        """The last outputs equal one step (or reset) of the device path on the same inputs."""
        b, o, r = self.bufs, self.out, self.rb
        if kind == "full_reset":
            env = self.device_env(lib, True)
            env.reset(None, self.phase)
            f = torch.ones(self.N, dtype=torch.bool)
            flags = (torch.zeros(self.N, dtype=torch.bool),) * 2
        else:
            env = self.device_env(lib, kind != "clip_end")
            if kind != "plain":
                env.enable_auto_reset(True)
            env.step(phase_by_env=self.phase)
            flags = (env.extras["reset"].cpu(), env.extras["terminate"].cpu())
            f = flags[0]
        torch.cuda.synchronize()
        ok = torch.equal(b.obs_buf, env.obs_buf.cpu()) and torch.equal(b.progress_buf, env.progress_buf.cpu())
        ok = ok and torch.equal(b.reset_buf.bool(), flags[0]) and torch.equal(b.terminate_buf.bool(), flags[1])
        if kind != "full_reset":
            ok = ok and torch.equal(b.rew_buf, env.rew_buf.cpu()) and torch.equal(b.reward_raw, env.reward_raw[:, :4].cpu())
        if kind != "plain":
            for got, want in ((o.state, env._rigid_body_state_reshaped), (r.root_states, env._humanoid_root_states),
                              (r.dof_pos, env._dof_pos), (r.dof_vel, env._dof_vel), (o.motion_start_times, env._motion_start_times),
                              (o.motion_start_times_offset, env._motion_start_times_offset), (o.global_offset, env._global_offset)):  # fmt: skip
                ok = ok and torch.equal(got[f], want.cpu()[f])
        return ok, float(f.float().mean())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--num-envs", type=int, default=4096, help="envs per batch")
    ap.add_argument("--rounds", type=int, default=200, help="rounds per timed loop (two batch-steps each)")
    ap.add_argument("--paths", default="direct:3,staged:3", help="output path:chunk count schedules to time")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"

    import __graft_entry__ as g

    g.build()
    from humanoid_b200 import HostStep, MotionLib, _cabi, synth

    capi = _cabi.load()
    N, R = args.num_envs, args.rounds
    data = synth.make_motion_lib(N, 60, 300, (30,), seed=SEED, device="cuda")
    lib = MotionLib(data, device="cuda")
    A, B = Batch(data, lib, N, SEED + 1), Batch(data, lib, N, SEED + 32)
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
        rargs = {id(bt): bt.rargs(_cabi.STATE_INIT_RANDOM) for bt in (A, B)}
        if kind == "plain":
            return lambda s, bt: _cabi.check(capi.phc_host_step_submit(ctx, s, C.byref(bt.args), bt.N), "submit")
        return lambda s, bt: _cabi.check(
            capi.phc_host_step_submit_reset(ctx, s, C.byref(bt.args), C.byref(rargs[id(bt)]), bt.N), "submit_reset")

    def sync_loop(ctx, submit):
        def loop(r):
            for _ in range(r):
                for bt in (A, B):
                    bt.rewind()
                    submit(0, bt)
                    _cabi.check(capi.phc_host_step_wait(ctx, 0), "wait")
        return loop

    def async_loop(ctx, submit):
        def loop(r):
            for s, bt in enumerate((A, B)):
                bt.rewind()
                submit(s, bt)
            for i in range(r):
                for s, bt in enumerate((A, B)):
                    _cabi.check(capi.phc_host_step_wait(ctx, s), "wait")
                    if i == r - 1:
                        continue
                    bt.rewind()
                    submit(s, bt)
        return loop

    rows = []
    plain_h2d = plain_d2h = 0
    for sched in args.paths.split(","):
        path, ch = sched.split(":")
        os.environ["PHC_HOST_PATH"] = path
        row = {"path": path, "chunks": int(ch)}
        for kind in ("plain", "clip_end", "flag30"):
            with HostStep(lib, N, num_chunks=int(ch), enable_early_termination=kind != "clip_end") as hs:
                ctx = hs._ctx
                plain_h2d, plain_d2h = int(capi.phc_host_step_h2d_bytes(ctx, N)), int(capi.phc_host_step_d2h_bytes(ctx, N))
                sub = submitter(ctx, kind)
                for mode, loop in (("async", async_loop(ctx, sub)), ("sync", sync_loop(ctx, sub))):
                    row[f"{kind}_{mode}_us"] = timed(loop, 2 * R)
                    for name, bt in (("A", A), ("B", B)):
                        ok, frac = bt.matches(lib, kind)
                        if not ok:
                            failures.append(f"{kind} {mode} {path}x{ch} batch {name}")
                    if kind != "plain":
                        row[f"{kind}_reposed_fraction"] = frac
                        row[f"{kind}_h2d_bytes"] = plain_h2d + N * 5
                        row[f"{kind}_d2h_bytes"] = plain_d2h + int(round(frac * N)) * ROW_BYTES
                assert hs.path == (1 if path == "direct" else 2) and hs.chunks == int(ch)
        # the first observation of a batch: a host reset of every env
        with HostStep(lib, N, num_chunks=int(ch)) as hs:
            ctx = hs._ctx
            rargs = A.rargs(_cabi.STATE_INIT_RANDOM)

            def reset_loop(r):
                for _ in range(r):
                    _cabi.check(capi.phc_host_reset_submit(ctx, 0, C.byref(A.args), C.byref(rargs), N), "reset_submit")
                    _cabi.check(capi.phc_host_step_wait(ctx, 0), "wait")

            row["full_reset_us"] = timed(reset_loop, R)
            row["full_reset_h2d_bytes"] = N * (8 + 12 + 4 + 4 + 2 + 4 + 1)
            row["full_reset_d2h_bytes"] = N * (934 * 4 + ROW_BYTES + 2)
            ok, _ = A.matches(lib, "full_reset")
            if not ok:
                failures.append(f"full_reset {path}x{ch}")
        rows.append(row)
    os.environ.pop("PHC_HOST_PATH", None)
    out["per_schedule"] = rows
    out["plain_h2d_bytes"], out["plain_d2h_bytes"] = plain_h2d, plain_d2h
    out["matches_device_path"] = not failures
    out["mismatches"] = failures
    print(json.dumps(out), flush=True)
    if failures:
        sys.exit(1)


if __name__ == "__main__":
    main()
