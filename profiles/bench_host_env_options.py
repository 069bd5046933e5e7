"""Env options on the host-buffer path (phc_host_step_submit_env): what the power reward, StateInit.Hybrid auto-resets
and host obs cost on top of the device-obs step.

The harness of bench_host_device_out.py: config 2, two 4096-env batches (bench_host_env.Batch), direct path with three
chunks, the two-slot async loop, median of 5 loops of --rounds rounds (one round = one step of batch A and one of B).
Legs, alternated in one run (each leg's loops are interleaved with the others', --passes times):

  dev_plain         phc_host_step_submit_device (r5's dev_obs leg)
  dev_power         phc_host_step_submit_env, device obs, power reward
  dev_power_hybrid  the same with StateInit.Hybrid auto-reset and early termination off: the 4 % clip-end envs are
                    re-posed every step, half of them on the default path (r5's reset rate)
  host_power        phc_host_step_submit_env, host obs, power reward

Floors: the copy engines alone moving the H2D bytes of the plain step (1278 B per env) and of the power step (1830 B).
Also timed: the host memcpy of one batch's dof force and velocity rows into pinned staging, which packing them with the
clock (one transfer per chunk instead of three) would put on the caller's thread.  Bytes per batch-step are computed
from the shapes.  Every leg's last outputs are compared bit for bit with HumanoidPHC(use_power_reward=True) on the same
inputs; a mismatch fails the run.  Writes r6_host_env_options.{json,md} to --out and prints the JSON.

    python profiles/bench_host_env_options.py [--rounds 200] [--out profiles]
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

COEF = 0.0005
IN_PLAIN = 24 * 13 * 4 + 8 + 12 + 4 + 4 + 2  # sim state | packed clock per env (1278 B)
IN_POWER = IN_PLAIN + 2 * 69 * 4  # + dof force and dof velocity rows (1830 B)
OUT_DEV = 4 + 16 + 2 + 1 + 1  # rew | reward_raw[:, :4] | progress | reset | terminate
OUT_DEV_POWER = OUT_DEV + 4  # reward_raw[:, 4]
LEGS = ("dev_plain", "dev_power", "dev_power_hybrid", "host_power")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--num-envs", type=int, default=4096, help="envs per batch")
    ap.add_argument("--rounds", type=int, default=200, help="rounds per timed loop (two batch-steps each)")
    ap.add_argument("--passes", type=int, default=5, help="timed loops per leg (the median is kept)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"), help="directory of r6_host_env_options.{json,md}")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"

    import __graft_entry__ as g

    g.build()
    from humanoid_b200 import HostDeviceOutputs, HostStep, HostStepBuffers, HumanoidPHC, MotionLib, _cabi, synth

    capi = _cabi.load()
    N, R = args.num_envs, args.rounds
    data = synth.make_motion_lib(N, 60, 300, (30,), seed=SEED, device="cuda")
    lib = MotionLib(data, device="cuda")
    A, B = Batch(data, lib, N, SEED + 1), Batch(data, lib, N, SEED + 32)
    gen = torch.Generator().manual_seed(SEED)
    for bt in (A, B):
        bt.dargs = bt.bufs._args()
        bt.dargs.obs_buf = None  # the rows go to the device tensors
        bt.dev = HostDeviceOutputs.allocate(N, 1, "cuda")
        p = HostStepBuffers.allocate(N, 1, pinned=True, power=True)  # the power inputs and the five-column reward_raw
        p.dof_force.copy_(torch.randn(N, 69, generator=gen) * 50)
        p.dof_vel.copy_(torch.randn(N, 69, generator=gen))
        bt.power = p
        bt.pargs = bt.bufs._args()
        bt.pargs.reward_raw = p.reward_raw.data_ptr()
        bt.pdargs = bt.bufs._args()
        bt.pdargs.obs_buf, bt.pdargs.reward_raw = None, p.reward_raw.data_ptr()
        bt.env = _cabi.PhcHostEnvArgs(p.dof_force.data_ptr(), p.dof_vel.data_ptr(), COEF, None, None)
        bt.dmask = (torch.rand(N, generator=gen) < 0.5).to(torch.uint8).pin_memory()
        bt.env_hybrid = _cabi.PhcHostEnvArgs(p.dof_force.data_ptr(), p.dof_vel.data_ptr(), COEF, None, bt.dmask.data_ptr())
        bt.init = [torch.randn(N, w, generator=gen) for w in (13, 69, 69)]
        bt.hybrid_rargs = bt.rargs(_cabi.STATE_INIT_HYBRID)
    torch.cuda.synchronize()

    def submitter(ctx, kind):
        def sub(s, bt):
            if kind == "dev_plain":
                rc = capi.phc_host_step_submit_device(ctx, s, C.byref(bt.dargs), None, C.byref(bt.dev._args()), N)
            elif kind == "host_power":
                rc = capi.phc_host_step_submit_env(ctx, s, C.byref(bt.pargs), None, None, C.byref(bt.env), N)
            else:
                hybrid = kind == "dev_power_hybrid"
                rc = capi.phc_host_step_submit_env(ctx, s, C.byref(bt.pdargs), C.byref(bt.hybrid_rargs) if hybrid else None,
                                                   C.byref(bt.dev._args()), C.byref(bt.env_hybrid if hybrid else bt.env), N)  # fmt: skip
            _cabi.check(rc, kind)

        return sub

    def async_loop(ctx, kind):
        sub = submitter(ctx, kind)

        def loop(r):
            for s, bt in enumerate((A, B)):
                bt.rewind()
                sub(s, bt)
            for i in range(r):
                for s, bt in enumerate((A, B)):
                    _cabi.check(capi.phc_host_step_wait(ctx, s), "wait")
                    if i == r - 1:
                        continue
                    bt.rewind()
                    sub(s, bt)

        return loop

    def matches(bt, kind):
        """The last outputs equal one step of HumanoidPHC(use_power_reward=True) on the same inputs."""
        b, p = bt.bufs, bt.power
        hybrid = kind == "dev_power_hybrid"
        env = HumanoidPHC(lib, N, device="cuda", enable_early_termination=not hybrid, use_power_reward=kind != "dev_plain",
                          rew_power_coef=COEF)  # fmt: skip
        env.set_sim_state(bt.state)
        env.set_clock(bt.clock)
        env.dof_force_tensor.copy_(p.dof_force.cuda())
        env._dof_vel.copy_(p.dof_vel.cuda())
        if hybrid:
            env.enable_auto_reset(True)
            env.state_init = "hybrid"
            for t, v in zip((env._initial_humanoid_root_states, env._initial_dof_pos, env._initial_dof_vel), bt.init):
                t.copy_(v.cuda())
        env.step(phase_by_env=bt.phase, default_mask_by_env=bt.dmask.cuda().bool())
        flags = (env.extras["reset"], env.extras["terminate"]) if hybrid else (env.reset_buf, env._terminate_buf)
        torch.cuda.synchronize()
        obs = b.obs_buf if kind == "host_power" else bt.dev.obs
        raw = b.reward_raw if kind == "dev_plain" else p.reward_raw
        want_raw = env.reward_raw[:, : raw.shape[1]].cpu()
        ok = torch.equal(obs.to(env.obs_buf.device), env.obs_buf)
        ok = ok and torch.equal(b.rew_buf, env.rew_buf.cpu()) and torch.equal(raw, want_raw)
        ok = ok and torch.equal(b.reset_buf.bool(), flags[0].cpu()) and torch.equal(b.terminate_buf.bool(), flags[1].cpu())
        return ok and torch.equal(b.progress_buf, env.progress_buf.cpu())

    os.environ["PHC_HOST_PATH"] = "direct"
    ctxs = {}
    for kind in LEGS:
        hs = HostStep(lib, N, num_chunks=3, enable_early_termination=kind != "dev_power_hybrid")
        if kind == "dev_power_hybrid":
            for s, bt in enumerate((A, B)):
                hs.set_initial_state(s, *bt.init)
        ctxs[kind] = (hs, async_loop(hs._ctx, kind))
        ctxs[kind][1](3)  # warm
    runs = {k: [] for k in LEGS}
    failures = []
    for i in range(args.passes):  # the legs alternate: a drift of the host's load spreads over all of them
        for kind in LEGS:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ctxs[kind][1](R)
            runs[kind].append(time.perf_counter() - t0)
            if i == args.passes - 1:  # the legs share the scalar outputs: each is checked before the next runs
                for name, bt in (("A", A), ("B", B)):
                    if not matches(bt, kind):
                        failures.append(f"{kind} batch {name}")
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

    # floors: the H2D bytes with the copy engine alone, min over five loops
    s_in = torch.cuda.Stream()
    floors = {}
    for name, per_env in (("h2d_only_plain", IN_PLAIN), ("h2d_only_power", IN_POWER)):
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
    # what packing the dof rows with the clock would cost the caller's thread per batch-step
    stage = torch.empty(N, 2, 69).pin_memory()
    pk = []
    for _ in range(5):
        t0 = time.perf_counter()
        for _ in range(R):
            stage[:, 0].copy_(A.power.dof_force)
            stage[:, 1].copy_(A.power.dof_vel)
        pk.append(time.perf_counter() - t0)
    pack_us = statistics.median(pk) / R * 1e6

    out = {"card": gpu_card(), "num_envs_per_batch": N, "rounds_per_loop": R, "timing_repeats": args.passes,
           "path": "direct", "chunks": 3, "legs": row, "floor_us": floors,
           "dof_pack_host_memcpy_us_per_batch_step": pack_us, "reposed_fraction_per_step": reposed,
           "h2d_bytes_per_batch_step": {"plain": N * IN_PLAIN, "power": N * IN_POWER},
           "d2h_bytes_per_batch_step": {"dev_plain": N * OUT_DEV, "dev_power": N * OUT_DEV_POWER,
                                        "host_power": N * (OUT_DEV_POWER + (_cabi.SELF_OBS_DIM + _cabi.TASK_OBS_DIM) * 4)}}  # fmt: skip
    out["goals"] = {
        "dev_power_async_over_its_h2d_floor": row["dev_power_async_us"] / floors["h2d_only_power"],
        "dev_plain_async_over_its_h2d_floor": row["dev_plain_async_us"] / floors["h2d_only_plain"],
        "dev_power_over_dev_plain": row["dev_power_async_us"] / row["dev_plain_async_us"],
    }
    out["matches_device_path"] = not failures
    out["mismatches"] = failures
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r6_host_env_options.json"), "w") as f:
        f.write(json.dumps(out) + "\n")
    lines = [f"# Host-path env options, {out['card']}", "",
             f"Two {N}-env config-2 batches, direct path, three chunks, two-slot async loop; median of {args.passes} "
             f"loops of {R} rounds, legs alternated.  us per batch-step.", "",
             "| leg | us / batch-step | min .. max | H2D B | D2H B |", "|---|---|---|---|---|"]  # fmt: skip
    for kind in LEGS:
        h2d = out["h2d_bytes_per_batch_step"]["plain" if kind == "dev_plain" else "power"]
        d2h = out["d2h_bytes_per_batch_step"]["dev_power" if kind == "dev_power_hybrid" else kind]
        lo, hi = row[f"{kind}_async_spread_us"]
        lines.append(f"| {kind} | {row[f'{kind}_async_us']:.1f} | {lo:.1f} .. {hi:.1f} | {h2d} | {d2h} |")
    lines += ["", "| floor | us |", "|---|---|"] + [f"| {k} | {v:.1f} |" for k, v in floors.items()]
    lines += ["", f"Host memcpy of one batch's dof force and velocity into pinned staging: {pack_us:.1f} us.",
              f"Re-posed fraction per step in dev_power_hybrid: {reposed:.3f}.",
              f"Goals: {json.dumps(out['goals'])}", f"Matches the device path bit for bit: {not failures}", ""]  # fmt: skip
    with open(os.path.join(args.out, "r6_host_env_options.md"), "w") as f:
        f.write("\n".join(lines))
    print(json.dumps(out), flush=True)
    if failures:
        sys.exit(1)


if __name__ == "__main__":
    main()
