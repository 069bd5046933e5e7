"""Phase timeline of the fast step kernel from per-warp %globaltimer stamps (phc_set_trace_buffer).

    python profiles/trace_step.py [num_envs]
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from humanoid_b200 import HumanoidPHC, MotionLib, _cabi, synth  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
dev = torch.device("cuda", 0)
lib_data = synth.make_motion_lib(N, 60, 300, (30,), seed=1234, device=dev)
lib = MotionLib(lib_data, device=dev)
clock = synth.make_clock(lib_data, N, seed=1235, max_progress=30)
envs = []
for r in range(17):
    ref = lib.get_motion_state(clock.sampled_motion_ids, synth.reward_time(clock, extra_steps=r + 1), clock.global_offset)
    env = HumanoidPHC(lib, N, device=dev)
    env.set_sim_state(synth.make_sim_state(ref, seed=1236 + r), copy=False)
    env.set_clock(clock)
    envs.append(env)
for i in range(20):
    envs[i % 17].post_physics_step(True)
torch.cuda.synchronize()
nw = (N + 3) // 4 * 3
K = 8
buf = torch.zeros(K * nw * 8, dtype=torch.int64, device=dev)
capi = _cabi.load()
for e in envs:
    e._step_args = None
    e.post_physics_step(True)
torch.cuda.synchronize()
# K steps in one CUDA graph, as the bench runs them; each kernel stamps its own slice
capi.phc_set_trace_buffer(buf.data_ptr(), K * nw)
graph = torch.cuda.CUDAGraph()
stream = torch.cuda.Stream()
stream.wait_stream(torch.cuda.current_stream())
with torch.cuda.stream(stream):
    with torch.cuda.graph(graph, stream=stream):
        for k in range(K):
            envs[k].post_physics_step(True)
capi.phc_set_trace_buffer(None, 0)
torch.cuda.synchronize()
graph.replay()
torch.cuda.synchronize()
buf.zero_()
graph.replay()
torch.cuda.synchronize()
T = [b.cpu().numpy().reshape(-1, 3, 8).astype(np.float64) for b in buf.view(K, -1)]
names = ["entry", "tma issued", "dep wait done", "data landed", "phase1 done", "stage written", "past bar3", "exit"]
t00 = T[0][:, :, 0].min()
prev_end = None
for k, t in enumerate(T):
    t = (t - t00) / 1e3
    w0 = t[:, 0, :]
    first, last = t[:, :, 0].min(), t[:, :, 7].max()
    line = f"kernel {k}: first entry {first:7.2f}  last exit {last:7.2f}  span {last - first:5.2f} us"
    if prev_end is not None:
        line += f"  | starts {first - prev_end:+.2f} us vs previous kernel's last exit; period {last - prev_last:5.2f} us"
    print(line)
    if k >= K - 2:
        for j in (0, 2, 1, 3, 4, 5, 6, 7):
            col = w0[:, j] - (prev_end if prev_end is not None else first)
            print(f"    warp0 {names[j]:14s} (rel. prev exit): min {col.min():6.2f}  median {np.median(col):6.2f}  "
                  f"p90 {np.percentile(col, 90):6.2f}  max {col.max():6.2f}")
    prev_end, prev_last = last, last

# straggler analysis of the last kernel: who exits late, and why
t = (T[-1] - t00) / 1e3
w0 = t[:, 0, :]
last_prev = ((T[-2] - t00) / 1e3)[:, :, 7].max()
exit_rel = t[:, :, 7].max(axis=1) - last_prev
post = w0[:, 1] - w0[:, 2]  # dependency resolved -> TMA issued (clock loads, validation, redo)
land = w0[:, 3] - w0[:, 1]  # TMA issued -> data landed
entry_rel = w0[:, 0] - last_prev
print("\nlatest-exiting blocks of the last kernel (us relative to the previous kernel's last exit):")
for i in np.argsort(-exit_rel)[:10]:
    print(f"  block {i:5d}: entry {entry_rel[i]:6.2f}  wait->issued {post[i]:5.2f}  issued->landed {land[i]:5.2f}  "
          f"phase1 {w0[i, 4] - w0[i, 3]:5.2f}  phase2 {w0[i, 5] - w0[i, 4]:5.2f}  exit {exit_rel[i]:5.2f}")
for name, arr in (("wait->issued", post), ("issued->landed", land), ("exit", exit_rel)):
    qs = np.percentile(arr, [50, 90, 99, 100])
    print(f"  {name:15s}: p50 {qs[0]:5.2f}  p90 {qs[1]:5.2f}  p99 {qs[2]:5.2f}  max {qs[3]:5.2f}")

# phase-0 path of each block of the last kernel: warp 1's stamp 1 holds 16 | bit 0 below spec4_blocks | bit 1 extra-row
# fetch | bit 2 redo | bit 3 fresh copies after the wait (nothing speculated), when the kernel records it
code = T[-1][:, 1, 1].astype(np.int64)
if (code & 16).all():
    redo = (code & 4) != 0
    fetch = ((code & 2) != 0) & ~redo
    fresh = ((code & 8) != 0) & ~redo & ~fetch
    hit = ~redo & ~fetch & ~fresh
    spec4 = (code & 1) != 0
    print(f"\nphase-0 paths of the last kernel's {len(code)} blocks ({int(spec4.sum())} below spec4_blocks): "
          f"four-row hit {int((hit & spec4).sum())}, three-row hit {int((hit & ~spec4).sum())}, "
          f"extra-row fetch {int(fetch.sum())}, redo {int(redo.sum())}, no speculation {int(fresh.sum())}")
    for name, sel in (("four-row hit", hit & spec4), ("three-row hit", hit & ~spec4), ("extra-row fetch", fetch)):
        if sel.any():
            print(f"  {name:15s}: median entry {np.median(entry_rel[sel]):6.2f}  issued->landed {np.median(land[sel]):5.2f}"
                  f"  exit {np.median(exit_rel[sel]):5.2f}")
