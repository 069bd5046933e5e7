#!/usr/bin/env python
"""Benchmark of the PHC step path: env-steps/s for the full post-physics step
(motion query @t + reward + reset + motion query @t+dt + self obs + imitation obs v6).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU torch path
    python bench.py --steps K --dump-outputs bench_outputs   # + the last timed step's outputs as <dir>/<name>.npy

One JSON line on stdout (rank 0).  A "step" is one pass of the hot path over one batch of
synthetic sim state.  The headline keys (`value`, `e2e`, `roofline`) are measured on BASELINE.json
configs[1] — num_envs = 4096 per GPU, one 60-300 frame 30 fps clip per env (ids == arange, the
reference regime), frame-aligned start times; weak scaling, envs and their clips partitioned across
ranks, no collective on the step.  The SAME run also measures the other BASELINE configs and reports
them under `configs` in the same line:

    config3  65 536 envs split over the N GPUs (strong scaling, 65 536/N per GPU), plain step and a
             whole 32-step rollout with the RunningNorm moments epilogue + fold + exchange + blend inside
             the timed region
    config4  AMASS-scale library (10 000 clips, ~4 M frames, mixed fps) replicated per GPU, random
             motion ids and unaligned times re-drawn for every ring slot
    config5  T = 10 future reference frames, 16 384 envs split over the N GPUs

`value`  : device-resident inputs; K steps captured in ONE CUDA graph (one kernel per step), timed
           with CUDA events on the launching stream, median over the replays, max over ranks.  Every step
           reads a different sim-state buffer and writes a different obs buffer out of a ring larger than
           the 126 MB L2, so inputs come from HBM and outputs go to HBM.
`e2e`    : the same metric through the C-ABI host pipeline (phc_host_step) with pinned HOST buffers:
           H2D of the sim state + clock, the fused kernel, D2H of obs/reward/flags, all inside the timed
           region; `e2e.floor` is the machine's floor for the same bytes, measured in the same run with all
           ranks copying at once (copy engines, both directions concurrently).
`cpu_baseline` / `--impl reference`: the reference's OWN functions (puffer_phc.envs.common /
           motion_lib / torch_utils, staged under baseline/_ref by __graft_entry__.build(); kind
           "reference") orchestrated as HumanoidPHC.step does, on the box's host cores; falls back to
           oracle/phc_oracle.py (kind "port", bit-identical to the reference) where the staged copy is absent.
`torch_cuda_baseline`: the reference's torch ops eager on this GPU (how the reference itself is
           deployed): the same-box "before".
"""

from __future__ import annotations

import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

NUM_ENVS_PER_GPU = 4096
CONFIG3_TOTAL_ENVS = 65536
CONFIG5_TOTAL_ENVS = 16384
ROLLOUT_STEPS = 32  # batch_size / num_envs = 131072 / 4096 (scripts/phc_train.py; clean_pufferl/core.py:130-182)
BYTES_PER_ENV_STEP = 8804  # SURVEY §8(d) / BASELINE.md §3: T=1, dt-aligned (3 distinct frames)
BYTES_PER_ENV_STEP_T = lambda T: 1248 + 54 + (T + 2) * 1248 + (358 + 576 * T) * 4 + 22  # noqa: E731
METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
SEED = 1234
DUMP_BYTES = 64 * 10**6  # --dump-outputs writes at most this much, .npy headers included
NPY_HEADER = 1024  # bound on one .npy header of these arrays (numpy writes 128 B)


def workload_name(n, workload="config2", clips=0):
    if workload == "config4":
        return (f"PHC SMPL 24-body step compute, num_envs={n} per GPU, AMASS-scale synthetic library ({clips} clips, "
                f"~4 M frames, mixed 30/60/120 fps), random motion ids and unaligned times per step")
    return (f"PHC SMPL 24-body step compute (motion query + smpl_max obs + imitation obs v6 + reward + reset), "
            f"num_envs={n} per GPU, one 60-300 frame 30 fps synthetic clip per env, synthetic sim state")  # fmt: skip


def config_dict(n, world, T, workload="config2", clips=0):
    """The static description of the headline workload — identical for the GPU arm and the reference arm."""
    return {
        "workload": workload_name(n, workload, clips), "num_envs_per_gpu": n, "num_envs_total": n * world,
        "time_steps": T, "motion_clips_per_gpu": clips if workload == "config4" else n,
        "l2": "inputs larger than L2: every step uses the next of a ring of sim-state/obs buffer sets (> 320 MiB), "
              "clock re-seeded each lap",
        "cuda_graph": "the K timed step kernels are one graph", "seed": SEED,
    }  # fmt: skip


def bytes_per_env_step(T, workload):
    if T != 1:
        return BYTES_PER_ENV_STEP_T(T)
    return 10052 if workload == "config4" else BYTES_PER_ENV_STEP  # 4 distinct frames (BASELINE.md §3) / 3


# ---------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md "clocks DURING the timed region")
# ---------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")  # fmt: skip

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )  # fmt: skip
        except OSError:
            self.proc = None
            return self

        def pump():
            for line in self.proc.stdout:
                self.rows.append((time.perf_counter(), line.strip()))

        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()
        return self

    def mark(self):
        return time.perf_counter()

    def summary(self, t0=None, t1=None):
        """Clocks over the samples taken in [t0, t1] (all samples when omitted)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, r in list(self.rows):
            if (t0 is not None and ts < t0) or (t1 is not None and ts > t1):
                continue
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower() == "active":
                    reasons.add(nm)
        return {
            "sm_mhz": statistics.median(sm) if sm else None,
            "sm_max_mhz": max(mx) if mx else None,
            "power_w_max": max(power) if power else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }

    def stop(self):
        if self.proc is None:
            return
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()


# ---------------------------------------------------------------------------------------
# CPU baseline: the reference's own functions (staged copy) or the oracle port, on host cores
# ---------------------------------------------------------------------------------------
def cpu_step_fn(lib_data):
    """(callable(state, prog, clock, term) -> None, kind, description).  The reference's own functions when
    they can be imported (/root/reference in the build container, baseline/_ref on the GPU box), else the port."""
    from humanoid_b200 import synth
    from oracle import ref_loader

    if ref_loader.available():
        # humanoid_phc.py:59-60: the env forces the legacy TorchScript executor
        torch._C._jit_set_profiling_mode(False)
        torch._C._jit_set_profiling_executor(False)
        lib = ref_loader.make_reference_lib(lib_data)

        def fn(state, prog, clock, term):
            ref_loader.reference_step(lib, state, prog, clock.motion_start_times, clock.motion_start_times_offset,
                                      clock.global_offset, clock.sampled_motion_ids, term, synth.SIM_DT)  # fmt: skip

        return fn, "reference", f"the reference's own puffer_phc functions ({ref_loader.where()}), torch CPU fp32"
    from oracle import phc_oracle as O

    lib = O.OracleMotionLib(lib_data)

    def fn(state, prog, clock, term):
        O.step(lib, state, prog, clock.motion_start_times, clock.motion_start_times_offset, clock.global_offset,
               clock.sampled_motion_ids, term, synth.SIM_DT)  # fmt: skip

    return fn, "port", "oracle/phc_oracle.py (torch CPU fp32 restatement, bit-identical to the reference)"


def cpu_rate(lib_data, clock, state, steps, warmup, threads):
    """env-steps/s of the CPU step on CPU copies of the workload."""
    torch.set_num_threads(threads)
    fn, kind, what = cpu_step_fn(lib_data)
    term = torch.full((24,), 0.25)
    n = state.shape[0]
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            prog = clock.progress_buf.clone()
            t0 = time.perf_counter()
            fn(state, prog, clock, term)
            t1 = time.perf_counter()
            if i >= warmup:
                times.append(t1 - t0)
    total = sum(times)
    return n * len(times) / total, 1e3 * total / len(times), kind, what


def run_reference(args):
    """--impl reference: the reference's CPU torch path on this box's host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from humanoid_b200 import synth
    from oracle import phc_oracle as O

    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    n = NUM_ENVS_PER_GPU

    def query(lib_data, ids, times, offset):
        return O.OracleMotionLib(lib_data).get_motion_state(ids, times, offset)

    # a bounded sample: when K is large, shrink the env batch so K steps stay within ~2 minutes
    lib_data, clock, state = synth.make_case(n, n, query, seed=SEED, device="cpu", max_progress=30)
    _, ms, _, _ = cpu_rate(lib_data, clock, state, steps=2, warmup=1, threads=threads)
    budget_ms = 120e3
    n_run = n
    if ms * (args.steps + args.warmup) > budget_ms:
        frac = budget_ms / (ms * (args.steps + args.warmup))
        n_run = max(256, int(n * frac) // 256 * 256)
    sl = slice(0, n_run)
    clock_s = synth.Clock(**{k: v[sl] for k, v in clock.__dict__.items()})
    rate, ms, kind, what = cpu_rate(lib_data, clock_s, state[sl], steps=args.steps, warmup=args.warmup, threads=threads)
    sample = f"{n_run} of {n} envs per step x {args.steps} steps, {what}, {threads} threads"
    line = {
        "impl": "reference",
        "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": config_dict(n, args.gpus, 1),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }  # fmt: skip
    emit(line)


# ---------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------
def load_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic(key):
    """Steady-state DRAM bytes per launch of the step kernel from the committed ncu capture of this config, if any
    (profiles/traffic.json; --cache-control none, taken after >= 20 ring steps)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            d = json.load(f)
        v = d.get(key)
        return int(v) if v is not None else None
    except Exception:
        return None


class Ctx:
    """Per-process plumbing shared by the measurements."""

    def __init__(self, args):
        import torch.distributed as dist

        self.dist = dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        assert self.world == args.gpus or self.world == 1, f"--gpus {args.gpus} but WORLD_SIZE={self.world}"
        self.seed = SEED + 1000 * self.rank  # each rank owns its own envs and their clips
        self.peak, self.peak_src = load_peak()
        self.sampler = ClockSampler(self.local_rank).start() if self.rank == 0 else None
        self.args = args

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


class Ring:
    """A ring of sim-state / obs buffer sets larger than L2 over one motion library, plus the step loop."""

    def __init__(self, ctx, N, T, workload, clips, ring_mb, obs_moments=False, lib_data=None):
        from humanoid_b200 import HumanoidPHC, MotionLib, synth

        dev, seed = ctx.dev, ctx.seed
        self.N, self.T, self.workload = N, T, workload
        self.config4 = workload == "config4"
        obs_dim = 358 + 576 * T
        self.obs_dim = obs_dim
        self.set_bytes = N * (24 * 13 + obs_dim) * 4
        self.R = R = max(4, -(-ring_mb * (1 << 20) // self.set_bytes))  # ring of R buffer sets > L2
        if lib_data is None:
            if self.config4:
                # BASELINE configs[3]: AMASS-scale library (~10k clips, ~4M frames, mixed fps, a few very long
                # clips) replicated per GPU; every ring slot has its OWN clock with random motion ids and
                # unaligned start times, so consecutive steps gather unrelated frames (defeats L2).
                g = torch.Generator(device=dev).manual_seed(seed + 7)
                nf = torch.randint(100, 701, (clips,), generator=g, device=dev)
                nf[: max(1, clips // 500)] = 7000
                lib_data = synth.make_motion_lib(clips, fps_choices=(30, 60, 120), seed=seed, device=dev, frames_per_motion=nf)
            else:
                lib_data = synth.make_motion_lib(N, 60, 300, (30,), seed=seed, device=dev)
        self.lib_data = lib_data
        self.lib = lib = MotionLib(lib_data, device=dev)
        self.envs = []
        clock = None
        first = None
        for r in range(R):
            if self.config4 or clock is None:
                clock = synth.make_clock(lib_data, N, seed=seed + 1 + 31 * r, ids="random" if self.config4 else "mod",
                                         aligned=not self.config4, max_progress=30)  # fmt: skip
            t = synth.reward_time(clock, extra_steps=1 if self.config4 else r + 1)
            ref = lib.get_motion_state(clock.sampled_motion_ids, t, clock.global_offset)
            state = synth.make_sim_state(ref, seed=seed + 2 + r)
            del ref
            env = HumanoidPHC(lib, N, device=dev, time_steps=T, obs_moments=obs_moments and r == 0)
            env.set_sim_state(state, copy=False)
            if first is None or self.config4:
                env.set_clock(clock)
                first = first or env
            else:  # all ring slots share one motion clock
                env.progress_buf = first.progress_buf
                env._motion_start_times = first._motion_start_times
                env._motion_start_times_offset = first._motion_start_times_offset
                env._global_offset = first._global_offset
                env._sampled_motion_ids = first._sampled_motion_ids
                if obs_moments:  # one accumulator for the whole rollout
                    env._obs_moment_buckets = first._obs_moment_buckets
            self.envs.append(env)
        self.first = first
        self.progress0 = first.progress_buf.clone()
        self.prog0_all = [e.progress_buf.clone() for e in self.envs] if self.config4 else None
        torch.cuda.synchronize()

    def rewind(self):
        """Every clock back to where the ring started it."""
        if self.config4:
            for e, p0 in zip(self.envs, self.prog0_all):
                e.progress_buf.copy_(p0)
        else:
            self.first.progress_buf.copy_(self.progress0)

    def run_steps(self, k):
        R = self.R
        for i in range(k):
            if i % R == 0 and (i >= R or not self.config4):  # re-seed the clocks at every lap (config4: from the 2nd)
                self.rewind()
            self.envs[i % R].post_physics_step(True)

    def free(self):
        self.envs, self.first, self.lib, self.lib_data = [], None, None, None
        gc.collect()
        torch.cuda.empty_cache()


def timed_graph(ctx, body, warm, reps, min_seconds=0.0):
    """Capture ``body()`` in ONE CUDA graph and time ``reps`` replays with CUDA events on the launching stream,
    a barrier + synchronize on both sides of every replay.  Returns (median ms of one replay as the max over
    ranks, clocks seen while it ran)."""
    warm()
    torch.cuda.synchronize()
    stream = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        with torch.cuda.graph(graph, stream=stream):
            body()
    torch.cuda.synchronize()
    graph.replay()  # one untimed replay
    torch.cuda.synchronize()
    t_begin = time.perf_counter()
    ms_runs = []
    for _ in range(reps):
        ctx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        graph.replay()
        e1.record()
        ctx.barrier()
        ms_runs.append(e0.elapsed_time(e1))
    ms = ctx.max_over_ranks(statistics.median(ms_runs))
    # keep the GPU under the same load until nvidia-smi (100 ms period) has had a few looks at it; the number of extra
    # replays follows from the max-over-ranks time, so every rank does the same (a replay may hold a peer exchange)
    spent = time.perf_counter() - t_begin
    extra = ctx.max_over_ranks(max(0.0, min_seconds - spent))
    for _ in range(int(extra / max(ms * 1e-3, 1e-5)) if extra > 0 else 0):
        graph.replay()
    torch.cuda.synchronize()
    t_end = time.perf_counter()
    clocks = ctx.sampler.summary(t_begin, t_end) if ctx.sampler is not None else None
    if clocks is not None and not clocks.get("samples"):
        clocks = ctx.sampler.summary()  # too short for a sample of its own: every sample of the run so far
    return ms, clocks, graph


def repeats_for(K, base):
    """A replay of K steps is short when K is small (20 steps = 0.14 ms): take the median over more replays so that
    the max-over-ranks of the timed region reflects the kernel and not one rank's scheduling jitter."""
    return max(base, min(200, -(-1024 // max(K, 1))))


def measure_steps(ctx, ring, K, reps, label):
    """µs per step of K plain fused steps over the ring (one graph), with the roofline fractions."""
    W = max(ctx.args.warmup, 3)
    ms, clocks, graph = timed_graph(ctx, lambda: ring.run_steps(K), lambda: ring.run_steps(max(W, ring.R)), reps,
                                    min_seconds=0.45)  # fmt: skip
    us = ms / K * 1e3
    bpe = bytes_per_env_step(ring.T, ring.workload)
    achieved = bpe * ring.N / (us * 1e-6) / 1e9
    out = {
        "num_envs_per_gpu": ring.N, "num_envs_total": ring.N * ctx.world, "time_steps": ring.T,
        "us_per_step": us, "value": ring.N * ctx.world / (us * 1e-6), "unit": UNIT, "steps": K, "timing_repeats": reps,
        "bytes_per_env_step": bpe, "achieved_gbs": achieved, "frac": achieved / ctx.peak,
        "ring_sets": ring.R, "ring_mib": round(ring.R * ring.set_bytes / 2**20),
        "motion_clips_per_gpu": ring.lib_data.num_motions, "motion_frames_per_gpu": ring.lib_data.total_frames,
        "clocks": clocks,
    }  # fmt: skip
    traffic = load_traffic(f"{label}_T{ring.T}_N{ring.N}")
    if traffic is not None:  # measured steady-state DRAM bytes per launch of this very config
        out["traffic"] = traffic
        out["frac_dram"] = traffic / (us * 1e-6) / 1e9 / ctx.peak
    del graph
    return out


def dump_outputs(ring, K, out_dir):
    """--dump-outputs: what the last of the K timed steps hands its caller — ``obs``, ``reward``, ``reward_raw``,
    ``reset`` and ``terminate`` (HumanoidPHC.step's obs_buf, rew_buf, reward_raw, reset_buf, extras["terminate"]) — as
    float32 ``<name>.npy`` files, so that two builds can be compared output for output.  The K steps are run once more
    from the ring's starting clocks first: config4's clocks move on from one graph replay to the next, so what the
    timing leaves behind would depend on how many replays it took.  (So with config4 the measurements after this one
    start from the ring's starting clocks, not from where the timed replays left them: the frames they gather differ,
    the work per step does not.)  Above DUMP_BYTES in all, a fixed seeded sample of env rows is written, and
    ``env_index.npy`` (float64) names them."""
    import numpy as np

    ring.rewind()
    ring.run_steps(K)
    env = ring.envs[(K - 1) % ring.R]
    outs = {"obs": env.obs_buf, "reward": env.rew_buf, "reward_raw": env.reward_raw, "reset": env.reset_buf,
            "terminate": env._terminate_out}  # fmt: skip
    outs = {k: v.float().cpu() for k, v in outs.items()}
    row_bytes = sum(v[0].numel() for v in outs.values()) * 4
    if ring.N * row_bytes + len(outs) * NPY_HEADER > DUMP_BYTES:
        keep = (DUMP_BYTES - (len(outs) + 1) * NPY_HEADER) // (row_bytes + 8)
        rows = torch.randperm(ring.N, generator=torch.Generator().manual_seed(SEED))[:keep].sort().values
        outs = {k: v[rows] for k, v in outs.items()}
        outs["env_index"] = rows.double()
    os.makedirs(out_dir, exist_ok=True)
    paths = [os.path.join(out_dir, k + ".npy") for k in outs]
    for path, v in zip(paths, outs.values()):
        np.save(path, v.numpy())
    assert sum(os.path.getsize(p) for p in paths) <= DUMP_BYTES, "--dump-outputs exceeded its size bound"


def make_running_norms(ctx, obs_dim):
    """(rn on the fused peer path when world > 1, rn on the NCCL path, note)."""
    from humanoid_b200.running_norm import RunningNorm

    dist, dev = ctx.dist, ctx.dev
    rn = RunningNorm(obs_dim, device=dev)
    rn_nccl = RunningNorm(obs_dim, device=dev)
    note = None
    if ctx.world > 1:
        try:
            rn.enable_peer_reduce(timeout_ms=20000)
            ok = torch.ones(1, device=dev)
        except Exception as exc:  # e.g. no P2P between two of the devices: keep the NCCL path, say so in the line
            note = f"peer path unavailable on rank {ctx.rank}: {exc}"
            ok = torch.zeros(1, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)  # all ranks or none
        if float(ok.item()) == 0.0:
            rn._peers = None
            note = note or "peer path unavailable on another rank"
    return rn, rn_nccl, note


def check_peer_reduce(ctx, rn, rn_nccl, sums_local, rows_local):
    """The fused peer exchange + blend against (a) the NCCL all-reduce + update kernel and (b) a single-process
    update of the all-gathered partials added in rank order.  Every rank checks; the verdicts are AND-ed."""
    from humanoid_b200 import _cabi
    from humanoid_b200.running_norm import RunningNorm

    dist, dev, world = ctx.dist, ctx.dev, ctx.world
    C2 = sums_local.numel()
    for r in (rn, rn_nccl):
        r.running_mean.zero_(), r.running_var.fill_(1.0), r.count.fill_(1.0)
    single = RunningNorm(C2 // 2, device=dev)
    out = {}
    for it in range(2):  # two rollouts: both mailbox slots, count 1 and 2
        local = sums_local * (1.0 + 0.25 * it)
        rn.update_from_moments(local.clone(), rows_local)
        rn_nccl.update_from_moments(local.clone(), rows_local)
        payload = torch.cat([local, torch.tensor([float(rows_local)], dtype=torch.float64, device=dev)])
        gathered = [torch.empty_like(payload) for _ in range(world)]
        dist.all_gather(gathered, payload)
        total = torch.zeros_like(payload)
        for g in gathered:  # rank order, like the peer kernel
            total += g
        _cabi.check(
            _cabi.load().phc_running_norm_update(
                single.running_mean.data_ptr(), single.running_var.data_ptr(), single.count.data_ptr(),
                total.data_ptr(), total[C2:].data_ptr(), C2 // 2, _cabi.stream_ptr(dev)),
            "phc_running_norm_update")  # fmt: skip
    torch.cuda.synchronize()
    if rn._peers is not None:
        rn._peers.status()  # raises if a launch timed out
    bit = bool(torch.equal(rn.running_mean, single.running_mean) and torch.equal(rn.running_var, single.running_var)
               and torch.equal(rn.count, single.count))  # fmt: skip
    close = bool(torch.allclose(rn.running_mean, rn_nccl.running_mean, rtol=1e-6, atol=1e-7)
                 and torch.allclose(rn.running_var, rn_nccl.running_var, rtol=1e-6, atol=1e-7)
                 and torch.equal(rn.count, rn_nccl.count))  # fmt: skip
    # every rank must hold the same statistics: compare with rank 0's
    ref_m, ref_v = rn.running_mean.clone(), rn.running_var.clone()
    dist.broadcast(ref_m, 0)
    dist.broadcast(ref_v, 0)
    same = bool(torch.equal(ref_m, rn.running_mean) and torch.equal(ref_v, rn.running_var))
    verdict = torch.tensor([float(bit), float(close), float(same)], device=dev)
    dist.all_reduce(verdict, op=dist.ReduceOp.MIN)
    v = verdict.tolist()
    out["peer_equals_single_process_bitwise"] = bool(v[0])
    out["peer_equals_nccl"] = bool(v[1])
    out["ranks_bit_identical"] = bool(v[2])
    out["max_abs_diff_vs_nccl"] = ctx.max_over_ranks(float((rn.running_mean - rn_nccl.running_mean).abs().max()))
    return out


def measure_e2e(ctx, ring, K):
    """env-steps/s through phc_host_step with pinned host buffers, plus the concurrent copy-engine floor."""
    import ctypes as C

    from humanoid_b200 import _cabi, synth

    args, dev, N, T = ctx.args, ctx.dev, ring.N, ring.T
    obs_dim = ring.obs_dim

    def pinned(t):
        return t.detach().cpu().contiguous().pin_memory()

    e0 = ring.envs[0]  # the host-buffer leg and the CPU baseline run ring slot 0's inputs
    progress0 = ring.progress0
    h_state = pinned(e0._rigid_body_state_reshaped)
    h_prog0 = pinned(progress0)
    h_prog = h_prog0.clone().pin_memory()
    h_start, h_off = pinned(e0._motion_start_times), pinned(e0._motion_start_times_offset)
    h_goff, h_ids = pinned(e0._global_offset), pinned(e0._sampled_motion_ids)
    h_obs = torch.empty((N, obs_dim), dtype=torch.float32).pin_memory()
    h_rew = torch.empty(N, dtype=torch.float32).pin_memory()
    h_raw = torch.empty((N, 4), dtype=torch.float32).pin_memory()
    h_reset = torch.empty(N, dtype=torch.uint8).pin_memory()
    h_term = torch.empty(N, dtype=torch.uint8).pin_memory()
    capi = _cabi.load()
    hctx = C.c_void_p()
    term_host = (C.c_float * 24)(*([0.25] * 24))
    spec = _cabi.reward_spec(ring.first.rwd_specs)
    _cabi.check(capi.phc_host_step_create(ring.lib.handle, N, T, args.e2e_chunks, term_host, 0xFFFFFF, 0, 1,
                                          synth.SIM_DT, C.byref(spec), C.byref(hctx)), "phc_host_step_create")  # fmt: skip
    hargs = _cabi.PhcHostStepArgs(
        h_state.data_ptr(), h_prog.data_ptr(), h_start.data_ptr(), h_off.data_ptr(), h_goff.data_ptr(),
        h_ids.data_ptr(), h_obs.data_ptr(), h_rew.data_ptr(), h_raw.data_ptr(), h_reset.data_ptr(), h_term.data_ptr(),
    )  # fmt: skip
    Ke = min(K, args.e2e_steps)
    # warm-up, all ranks in step: the library times its two output paths (kernels posting into the mapped host
    # buffers / copy-engine D2H) over these calls, under the load of the other ranks, and keeps the faster one
    ctx.barrier()
    for _ in range(max(12, int(capi.phc_host_step_tuning_calls(hctx)) + 4)):
        h_prog.copy_(h_prog0)
        _cabi.check(capi.phc_host_step(hctx, C.byref(hargs), N), "phc_host_step")
    # the host path must agree with the device path on the same inputs
    e0.progress_buf.copy_(progress0)
    e0.post_physics_step(True)
    torch.cuda.synchronize()
    e2e_ok = bool(torch.equal(e0.obs_buf.cpu(), h_obs) and torch.equal(e0.rew_buf.cpu(), h_rew))
    runs = []
    for _ in range(5):  # median of five timed loops of Ke calls (each call returns with the outputs in host memory)
        ctx.barrier()
        t0 = time.perf_counter()
        for i in range(Ke):
            if i % ring.R == 0:
                h_prog.copy_(h_prog0)
            _cabi.check(capi.phc_host_step(hctx, C.byref(hargs), N), "phc_host_step")
        t1 = time.perf_counter()
        ctx.barrier()
        runs.append(ctx.max_over_ranks(t1 - t0))
    e2e_s = statistics.median(runs)
    h2d = int(capi.phc_host_step_h2d_bytes(hctx, N))
    d2h = int(capi.phc_host_step_d2h_bytes(hctx, N))
    path = {0: "undecided", 1: "direct (kernels post into the mapped host buffers)", 2: "staged (copy-engine D2H)"}.get(
        int(capi.phc_host_step_path(hctx)), "?")
    chunks = int(capi.phc_host_step_chunks(hctx))
    capi.phc_host_step_destroy(hctx)

    # ---- the machine's floor for the same bytes: every rank moves h2d bytes in and d2h bytes out at once, both
    # directions concurrently on the copy engines, pinned memory, one synchronize per "step" like the call above
    d_in = torch.empty(h2d, dtype=torch.uint8, device=dev)
    d_out = torch.empty(d2h, dtype=torch.uint8, device=dev)
    p_in = torch.empty(h2d, dtype=torch.uint8).pin_memory()
    p_out = torch.empty(d2h, dtype=torch.uint8).pin_memory()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

    def floor_loop(n, both=True, out=True):
        for _ in range(n):
            if both or not out:
                with torch.cuda.stream(s_in):
                    d_in.copy_(p_in, non_blocking=True)
            if both or out:
                with torch.cuda.stream(s_out):
                    p_out.copy_(d_out, non_blocking=True)
            s_in.synchronize()
            s_out.synchronize()

    floors = {}
    for name, kw in (("duplex", {}), ("d2h_only", dict(both=False, out=True)), ("h2d_only", dict(both=False, out=False))):
        floor_loop(3, **kw)
        fr = []
        for _ in range(5):  # a floor is the best the machine does: the minimum over five loops (the duplex figure
            ctx.barrier()   # varies by 20 % between loops on some hosts)
            t0 = time.perf_counter()
            floor_loop(Ke, **kw)
            t1 = time.perf_counter()
            ctx.barrier()
            fr.append(ctx.max_over_ranks(t1 - t0))
        floors[name] = min(fr) / Ke * 1e6
    e2e_us = e2e_s / Ke * 1e6
    world = ctx.world
    return {
        "value": N * world * Ke / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
        "steps": Ke, "timing_repeats": 5, "chunks": chunks, "chunks_requested": args.e2e_chunks or "auto", "matches_device_path": e2e_ok,
        "us_per_step": e2e_us, "output_path": path,
        "floor": {
            "what": f"all {world} rank(s) at once: pinned H2D of {h2d} B and D2H of {d2h} B per rank on the copy engines, "
                    "both directions concurrently, one synchronize per step; max over ranks, best of five loops",
            "us_per_step": floors["duplex"], "d2h_only_us": floors["d2h_only"], "h2d_only_us": floors["h2d_only"],
            "value_at_floor": N * world / (floors["duplex"] * 1e-6), "e2e_over_floor": floors["duplex"] / e2e_us,
            "aggregate_gbs": {"d2h": d2h * world / floors["d2h_only"] / 1e3, "h2d": h2d * world / floors["h2d_only"] / 1e3},
        },
    }  # fmt: skip


def measure_rollout(ctx, ring, rn, steps):
    """One rollout as the trainer runs it (scripts/phc_train.py:331-332): `steps` fused steps whose epilogue
    accumulates the RunningNorm moments, then fold + exchange + blend — all inside the timed region, one graph."""
    env0 = ring.first
    N = ring.N
    sums = torch.zeros(2 * ring.obs_dim, dtype=torch.float64, device=ctx.dev)

    def body():
        ring.run_steps(steps)
        env0.take_obs_moments(sums)
        rn.update_from_moments(sums, steps * N)
        if rn._peers is None:  # the NCCL / single-GPU path does not clear the caller's partials
            sums.zero_()

    capturable = ctx.world == 1 or rn._peers is not None
    if capturable:
        ms, clocks, graph = timed_graph(ctx, body, body, max(5, ctx.args.repeats), min_seconds=0.3)
        del graph
    else:  # NCCL exchange: eager launches
        body()
        runs = []
        for _ in range(5):
            ctx.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            body()
            e1.record()
            ctx.barrier()
            runs.append(e0.elapsed_time(e1))
        ms, clocks = ctx.max_over_ranks(statistics.median(runs)), None
    env0.obs_moment_rows = 0
    return {"rollout_steps": steps, "rollout_ms": ms, "us_per_step": ms / steps * 1e3,
            "value": N * ctx.world * steps / (ms * 1e-3), "cuda_graph": capturable, "clocks": clocks,
            "what": "fused steps with the moments epilogue + fold + "
                    + ("one fused peer launch (all-reduce over NVLink peer memory + blend)" if ctx.world > 1 and rn._peers is not None
                       else "NCCL all-reduce + update kernel" if ctx.world > 1 else "update kernel (1 GPU: no exchange)")}  # fmt: skip


def run_gpu(args):
    from humanoid_b200 import synth

    ctx = Ctx(args)
    dist, dev, rank, world = ctx.dist, ctx.dev, ctx.rank, ctx.world
    N, T, K = args.num_envs, args.time_steps, args.steps
    W = max(args.warmup, 3)
    if ctx.sampler is not None:
        time.sleep(0.3)

    # ================= headline: BASELINE configs[1] (or what --num-envs / --workload / --time-steps ask for)
    ring = Ring(ctx, N, T, args.workload, args.clips, args.ring_mb)
    reps = repeats_for(K, args.repeats)
    main = measure_steps(ctx, ring, K, reps, "step_kernel" if args.workload == "config2" else args.workload)
    ms_per_step = main["us_per_step"] * 1e-3
    frac_term = float(ring.envs[(K - 1) % ring.R]._terminate_buf.float().mean().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(ring, K, args.dump_outputs)
    long_run = None
    if K < 256 and not args.no_long_run:  # the same measurement over a longer timed region (512 steps per replay)
        lr = measure_steps(ctx, ring, 512, args.repeats, "step_kernel")
        long_run = {k: lr[k] for k in ("steps", "us_per_step", "value", "frac", "timing_repeats")}

    e2e = measure_e2e(ctx, ring, K)

    # -------- RunningNorm: moments of a rollout + ONE exchange (+ blend), per rollout.
    # The exchange + blend is one launch per rank over NVLink peer memory (phc_running_norm_update_peers);
    # the NCCL all-reduce + update-kernel path is timed beside it and the two are CHECKED against each other.
    obs_dim = ring.obs_dim
    rn, rn_nccl, peer_note = make_running_norms(ctx, obs_dim)
    sums = torch.zeros(2 * obs_dim, dtype=torch.float64, device=dev)
    roll = min(ROLLOUT_STEPS, ring.R)

    def rms_once():
        sums.zero_()
        for r in range(roll):
            rn.moments(ring.envs[r].obs_buf, sums)
        rn.update_from_moments(sums, roll * N)

    def timed_ms(fn, reps=1):
        fn()
        ctx.barrier()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for _ in range(reps):
            fn()
        r1.record()
        ctx.barrier()
        return ctx.max_over_ranks(r0.elapsed_time(r1) / reps)

    rms_ms = timed_ms(rms_once)
    exch_fused_us = timed_ms(lambda: rn.update_from_moments(sums, roll * N), reps=50) * 1e3
    exch_nccl_us = timed_ms(lambda: rn_nccl.update_from_moments(sums, roll * N), reps=50) * 1e3
    if world > 1 and rn._peers is not None:
        try:
            rn._peers.status()  # raises if any launch timed out waiting for a peer
        except Exception as exc:
            peer_note = f"peer launch failed: {exc}"
    fused_on = world > 1 and getattr(rn, "_peers", None) is not None
    rms_check = None
    if fused_on:
        local = torch.zeros(2 * obs_dim, dtype=torch.float64, device=dev)
        for r in range(roll):
            rn.moments(ring.envs[r].obs_buf, local)
        rms_check = check_peer_reduce(ctx, rn, rn_nccl, local, roll * N)

    # -------- CPU baseline and the torch-on-GPU "before", rank 0 at N = 1 only
    cpu_baseline = torch_cuda = None
    if world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        e0 = ring.envs[0]
        lib_cpu = ring.lib_data.to("cpu")
        clock_cpu = synth.Clock(progress_buf=ring.progress0.cpu(), motion_start_times=e0._motion_start_times.cpu(),
                                motion_start_times_offset=e0._motion_start_times_offset.cpu(),
                                global_offset=e0._global_offset.cpu(), sampled_motion_ids=e0._sampled_motion_ids.cpu())  # fmt: skip
        state_cpu = e0._rigid_body_state_reshaped.cpu()
        _, ms1, _, _ = cpu_rate(lib_cpu, clock_cpu, state_cpu, steps=1, warmup=1, threads=threads)
        cs = max(5, min(100, int(15e3 / ms1)))  # about 15 s of CPU work
        rate, msc, kind, what = cpu_rate(lib_cpu, clock_cpu, state_cpu, steps=cs, warmup=3, threads=threads)
        cpu_baseline = {
            "value": rate, "unit": UNIT, "cores": threads, "kind": kind, "ms_per_step": msc,
            "sample": f"{cs} steps of the same {N}-env workload (same tensors copied to host), {what}, {threads} threads",
        }  # fmt: skip
    if world == 1 and not args.no_torch_cuda_baseline:
        # the reference's own deployment: the same torch ops, eager, on this GPU (about 1100 launches per step)
        from oracle import phc_oracle as O

        lib_o = O.OracleMotionLib(ring.lib_data)
        term = torch.full((24,), 0.25, device=dev)
        e0 = ring.envs[0]
        st = e0._rigid_body_state_reshaped

        def torch_step():
            prog = ring.progress0.clone()
            O.step(lib_o, st, prog, e0._motion_start_times, e0._motion_start_times_offset, e0._global_offset,
                   e0._sampled_motion_ids, term, synth.SIM_DT)  # fmt: skip

        with torch.no_grad():
            for _ in range(5):
                torch_step()
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n_rep = 30
            t0.record()
            for _ in range(n_rep):
                torch_step()
            t1.record()
            torch.cuda.synchronize()
        ms = t0.elapsed_time(t1) / n_rep
        torch_cuda = {"value": N / ms * 1e3, "unit": UNIT, "ms_per_step": ms,
                      "what": "the reference's torch ops (oracle/phc_oracle.py restatement, fp32) eager on this GPU, "
                              "~1100 launches per step — how the reference itself runs this path"}  # fmt: skip
    headline_clips = ring.lib_data.num_motions
    ring.free()
    del ring

    # ================= the other BASELINE configs, same run, same line
    configs = {}
    if not args.no_extra_configs:
        # config 3: 65 536 envs over the N GPUs (strong scaling)
        n3 = CONFIG3_TOTAL_ENVS // world
        r3 = Ring(ctx, n3, 1, "config2", 0, args.ring_mb, obs_moments=True)
        buckets = r3.first._obs_moment_buckets
        for e in r3.envs:  # plain step first (no epilogue): the kernel the roofline fraction is quoted on
            e._obs_moment_buckets = None
            e._step_args = None
        c3 = measure_steps(ctx, r3, max(K, 64), args.repeats, "step_kernel")
        for e in r3.envs:
            e._obs_moment_buckets = buckets
            e._step_args = None
        rn3, _, note3 = make_running_norms(ctx, r3.obs_dim)
        c3["rollout"] = measure_rollout(ctx, r3, rn3, ROLLOUT_STEPS)
        c3["scaling"] = "strong"
        c3["what"] = (f"BASELINE configs[2]: {CONFIG3_TOTAL_ENVS} envs env-partitioned over {world} GPU(s), one clip per env; "
                      "`us_per_step` = plain fused step, `rollout` = 32 steps with the RunningNorm moments epilogue + the "
                      "per-rollout exchange and blend inside the timed region")
        if note3:
            c3["note"] = note3
        configs["config3_65536_envs_strong"] = c3
        del rn3
        r3.free()
        del r3

        # config 4: AMASS-scale library, random ids, unaligned times
        r4 = Ring(ctx, NUM_ENVS_PER_GPU, 1, "config4", args.clips, args.ring_mb)
        c4 = measure_steps(ctx, r4, max(K, 64), args.repeats, "config4")
        c4["scaling"] = "weak"
        c4["what"] = ("BASELINE configs[3]: AMASS-scale library replicated per GPU, random motion ids and unaligned times "
                      "re-drawn for every ring slot (4 distinct frames per env-step, no L2 reuse between steps)")
        configs["config4_amass_scale_library"] = c4
        r4.free()
        del r4

        # config 5: T = 10, 16 384 envs over the N GPUs
        n5 = CONFIG5_TOTAL_ENVS // world
        r5 = Ring(ctx, n5, 10, "config2", 0, args.ring_mb)
        c5 = measure_steps(ctx, r5, max(min(K, 128), 32), args.repeats, "step_kernel")
        c5["scaling"] = "strong"
        c5["what"] = f"BASELINE configs[4]: 10 future reference frames per env, {CONFIG5_TOTAL_ENVS} envs over {world} GPU(s)"
        configs["config5_T10_16384_envs"] = c5
        r5.free()
        del r5

    if ctx.sampler is not None:
        ctx.sampler.stop()
    rc = 0
    if rms_check is not None and not (rms_check["peer_equals_single_process_bitwise"] and rms_check["peer_equals_nccl"]
                                      and rms_check["ranks_bit_identical"]):  # fmt: skip
        rc = 3
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        if rc:
            sys.exit(rc)
        return

    bpe = main["bytes_per_env_step"]
    kernel = "phc::step_fast_kernel<4,8,false,false>" if T == 1 else "phc::step_multi2_kernel"
    roofline = {"bound": "hbm", "achieved": main["achieved_gbs"], "peak": ctx.peak, "unit": "GB/s", "frac": main["frac"],
                "traffic": main.get("traffic"), "frac_dram": main.get("frac_dram"), "peak_source": ctx.peak_src,
                "bytes_per_env_step": bpe, "kernel": kernel, "launch_ms": ms_per_step,
                "traffic_source": "profiles/traffic.json: ncu dram__bytes_read.sum + dram__bytes_write.sum of one launch of this "
                                  "config in steady state (--cache-control none, after >= 20 ring steps)"
                                  if main.get("traffic") is not None else None}  # fmt: skip
    line = {
        "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": config_dict(N, world, T, args.workload, headline_clips),
        "workload_stats": {"motion_frames_per_gpu": main["motion_frames_per_gpu"], "ring_sets": main["ring_sets"],
                           "ring_mib": main["ring_mib"], "terminated_frac": round(frac_term, 4),
                           "timing_repeats": main["timing_repeats"]},
        "clocks": main["clocks"],
        "e2e": e2e,
        "gpu_launches": K,
        "roofline": roofline,
        "rms": {"what": f"RunningNorm.update over a {roll}-step rollout: fp64 column moments + "
                        + (f"one fused launch per rank (all-reduce of {(2 * obs_dim + 1) * 8} B over NVLink peer memory + blend)"
                           if fused_on else f"NCCL all-reduce of {(2 * obs_dim + 1) * 8} B + blend" if world > 1
                           else "blend (1 GPU: no exchange)"),
                "ms_per_rollout": rms_ms,
                "exchange_and_blend_us": {"fused_peer_kernel" if fused_on else "update_path": exch_fused_us,
                                          "nccl_all_reduce_plus_update_kernel" if world > 1 else "update_path_again": exch_nccl_us},
                **(rms_check or {}),
                **({"note": peer_note} if peer_note else {})},
    }  # fmt: skip
    if long_run is not None:
        line["long_run"] = long_run
    if cpu_baseline is not None:
        line["cpu_baseline"] = cpu_baseline
    if torch_cuda is not None:
        line["torch_cuda_baseline"] = torch_cuda
    if configs:
        line["configs"] = configs
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    if rc:
        sys.exit(rc)


_JSON_FD = None


def keep_stdout_for_the_json_line():
    """The contract is ONE line on stdout.  Libraries write there too (NCCL prints its version banner from C when
    NCCL_DEBUG is set in the environment), so fd 1 is pointed at stderr for the whole run and the JSON line goes to
    the saved descriptor."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _JSON_FD is None:
        os.write(1, data)
    else:
        os.write(_JSON_FD, data)


def main():
    keep_stdout_for_the_json_line()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=512)
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--num-envs", type=int, default=NUM_ENVS_PER_GPU, help="envs per GPU of the headline measurement")
    ap.add_argument("--time-steps", type=int, default=1, help="future reference frames T of the headline measurement")
    ap.add_argument("--workload", choices=["config2", "config4"], default="config2",
                    help="headline workload. config2: one clip per env, aligned (default, BASELINE configs[1]); config4: "
                         "AMASS-scale library, random ids / unaligned times per step (BASELINE configs[3])")
    ap.add_argument("--clips", type=int, default=10000, help="clips of the config4 library")
    ap.add_argument("--ring-mb", type=int, default=320, help="min size of the sim-state/obs buffer ring (> L2)")
    ap.add_argument("--repeats", type=int, default=5, help="timed graph replays (more when --steps is small); the median is reported")
    ap.add_argument("--e2e-steps", type=int, default=64)
    ap.add_argument("--e2e-chunks", type=int, default=0, help="0 = the library tunes path and chunk count over its first calls")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-torch-cuda-baseline", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true", help="skip BASELINE configs 3 / 4 / 5 (the `configs` key)")
    ap.add_argument("--no-long-run", action="store_true", help="skip the 512-step re-measurement when --steps is small")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline's last timed step (obs, reward, reward_raw, reset, terminate; rank 0) as "
                         "DIR/<name>.npy, at most 64 MB (64e6 bytes)")  # fmt: skip
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; it does not apply to --impl reference")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
