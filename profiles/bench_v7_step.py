"""The fused step with the imitation observation v7 (HumanoidPHC(obs_v=7)) against v6, in one process: CUDA-graph steps
over a ring of sim-state / obs buffer sets larger than L2, v6 and v7 alternated, the card's name and power limit read in
the same run.  Which kernel each side ran is taken from a torch.profiler trace of one eager step.

    python profiles/bench_v7_step.py [--out profiles/r9_v7_step] [--rounds 3] [--steps 256]

Algorithmic bytes per env-step are the DRAM bytes a step cannot avoid: sim rows in (1248 B), clock and flags, frame rows
of the queries, and the obs row out.  v6 moves 8804 B at T = 1 and 40772 B at T = 10; v7 writes 360 fewer floats per
future step, 7364 B and 26372 B.  The copy peak 6456.2 GB/s is the HBM copy rate measured on a B200 (BASELINE.md).
"""

import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from humanoid_b200 import HumanoidPHC, MotionLib, synth  # noqa: E402

COPY_PEAK_GBS = 6456.2
BYTES = {(6, 1): 8804, (7, 1): 7364, (6, 10): 40772, (7, 10): 26372}
SHAPES = [(4096, 1), (16384, 1), (65536, 1), (16384, 10)]
RING_BYTES = 320 << 20  # > 126 MB of L2, several times over


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()  # fmt: skip
    except (OSError, subprocess.TimeoutExpired):
        q = "unavailable"
    return {"name": name, "power_limit_w_and_max_sm_mhz": q}


class Ring:
    """R envs of one obs version over one library, each with its own sim state, clock and obs buffers."""

    def __init__(self, lib, N, T, obs_v, state, clock):
        per_set = N * (24 * 13 * 4 + (358 + (576 if obs_v == 6 else 216) * T) * 4 + 69 * 2 * 4 * 2)
        self.R = max(4, -(-RING_BYTES // per_set))
        self.envs = []
        for _ in range(self.R):
            env = HumanoidPHC(lib, N, device="cuda", time_steps=T, obs_v=obs_v)
            env.set_sim_state(state)
            env.set_clock(clock)
            self.envs.append(env)
        self.clock = clock

    def rewind(self):
        for env in self.envs:
            env.set_clock(self.clock)

    def steps(self, K):
        for k in range(K):
            self.envs[k % self.R].post_physics_step(True)


def kernel_of(ring):
    from torch.profiler import ProfilerActivity, profile

    ring.rewind()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ring.envs[0].post_physics_step(True)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if "step" in e.name and e.device_type.name == "CUDA"]
    n = names[0] if names else "?"
    for short in ("step_persist_kernel", "step_multi2_kernel", "step_multi_kernel", "step_fast_kernel", "step_kernel"):
        if short in n:
            return short, n
    return n, n


def graph_of(ring, K):
    ring.rewind()
    ring.steps(2 * ring.R)  # warm-up: module load, smem attributes, every buffer touched once
    ring.rewind()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            ring.steps(K)
    torch.cuda.synchronize()
    return g, s


def time_graph(ring, g, s, K, reps=5):
    best = float("inf")
    for _ in range(reps):
        ring.rewind()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(s):
            e0.record(s)
            g.replay()
            e1.record(s)
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) * 1e3 / K)
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write <out>.json and <out>.md")
    ap.add_argument("--rounds", type=int, default=3, help="v6 / v7 alternations per shape")
    ap.add_argument("--steps", type=int, default=256, help="steps per graph")
    ap.add_argument("--shapes", default=None, help="N:T,N:T,... (default: the four shapes of the report)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_v7_step.py measures on the GPU; no CUDA device here")
    shapes = [tuple(int(x) for x in s.split(":")) for s in args.shapes.split(",")] if args.shapes else SHAPES
    info = {"card": card(), "steps_per_graph": args.steps, "rounds": args.rounds, "ring_bytes_min": RING_BYTES,
            "copy_peak_gbs": COPY_PEAK_GBS, "shapes": []}  # fmt: skip
    for N, T in shapes:
        clips = min(N, 8192)
        lib_data = synth.make_motion_lib(clips, 60, 300, (30,), seed=1234, device="cuda")
        lib = MotionLib(lib_data, device="cuda")
        clock = synth.make_clock(lib_data, N, seed=1235, max_progress=30)
        ref = lib.get_motion_state(clock.sampled_motion_ids, synth.reward_time(clock, extra_steps=1), clock.global_offset)
        state = synth.make_sim_state(ref, seed=1236)
        rings = {v: Ring(lib, N, T, v, state, clock) for v in (6, 7)}
        kern = {v: kernel_of(rings[v]) for v in (6, 7)}
        graphs = {v: graph_of(rings[v], args.steps) for v in (6, 7)}
        us = {6: [], 7: []}
        for _ in range(args.rounds):
            for v in (6, 7):
                us[v].append(time_graph(rings[v], *graphs[v], args.steps))
        row = {"num_envs": N, "time_steps": T, "ring_sets": {str(v): rings[v].R for v in (6, 7)}}
        for v in (6, 7):
            best = min(us[v])
            bpe = BYTES.get((v, T))
            row[f"v{v}"] = {
                "kernel": kern[v][0], "kernel_symbol": kern[v][1], "us_per_step": us[v], "us_best": best,
                "env_steps_per_s": N / (best * 1e-6), "bytes_per_env_step": bpe,
                "fraction_of_copy_peak": (bpe * N / (best * 1e-6) / 1e9 / COPY_PEAK_GBS) if bpe else None,
            }  # fmt: skip
        info["shapes"].append(row)
        print(json.dumps(row), flush=True)
        del rings, graphs
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out + ".json", "w") as f:
            json.dump(info, f, indent=1)
        lines = [f"# v7 vs v6 fused step — {info['card']['name']}, power limit / max SM clock "
                 f"{info['card']['power_limit_w_and_max_sm_mhz']}", "",
                 f"CUDA graph of {args.steps} steps over a ring of buffer sets > {RING_BYTES >> 20} MiB; best of 5 replays per "
                 f"round, {args.rounds} rounds alternating v6 / v7 (all rounds in the .json).", "",
                 "| envs | T | v6 kernel | v6 us | v7 kernel | v7 us | v6 Menv-steps/s | v7 Menv-steps/s | v6 / v7 of copy peak |",
                 "|---|---|---|---|---|---|---|---|---|"]  # fmt: skip
        for r in info["shapes"]:
            a, b = r["v6"], r["v7"]
            fr = lambda x: "—" if x["fraction_of_copy_peak"] is None else f"{x['fraction_of_copy_peak']:.2f}"  # noqa: E731
            lines.append(f"| {r['num_envs']} | {r['time_steps']} | {a['kernel']} | {a['us_best']:.2f} | {b['kernel']} | "
                         f"{b['us_best']:.2f} | {a['env_steps_per_s'] / 1e6:.1f} | {b['env_steps_per_s'] / 1e6:.1f} | "
                         f"{fr(a)} / {fr(b)} |")  # fmt: skip
        with open(args.out + ".md", "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
