// Host-buffer entry point around phc_step_fused (the end-to-end call of include/phc_b200.h).
//
// Direct path (all caller buffers pinned, hence mapped into the device address space by UVA): the
// sim state of each chunk is copied in by the host->device copy engine, and the chunk's fused
// kernel writes obs rows, rewards and flags straight into the caller's host buffers with its
// bulk stores (no device->host DMA descriptors, no device staging of outputs), so the two
// directions of the link overlap.  Used whenever cudaPointerGetAttributes says every buffer is
// pinned / managed host memory mapped at its own address (device pointers are rejected: PHC_ERR_UNSUPPORTED).
//
// Staged path (any pageable buffer): chunked copy pipeline, below.
//
// The env batch is cut into chunks; chunk c runs
//     H2D(sim state) + H2D(packed clock)  ->  fused step  ->  D2H(obs) + D2H(packed scalars)
// on stream c % 3, so the host->device copy of one chunk, the kernel of another and the
// device->host copy of a third overlap (PCIe is full duplex; the B200 has copy engines per
// direction).  The five small clock arrays and the five small outputs of a chunk travel as ONE
// transfer each through pinned staging buffers owned by the context (a DMA descriptor costs a
// few microseconds regardless of size; 22 of them per chunk were half of the step time).
//
// Slots.  A context owns PHC_HOST_SLOTS independent pipelines, each with its own device buffers, pinned staging and
// three streams.  phc_host_step_submit enqueues one step on a slot and returns; phc_host_step_wait waits for the
// slot's events and, on the staged path, unpacks the scalar outputs.  With two slots the inbound copy of one batch
// rides under the outbound traffic of the other (the slots' streams do not queue behind each other), and the caller's
// thread is free between submit and wait.  phc_host_step is submit + wait on slot 0.
//
// Resets.  phc_host_step_submit_reset runs each chunk's step with PhcStepArgs.auto_reset over the chunk's own device
// copies (sim state, packed clock, per-slot root / dof scratch); phc_host_reset_submit runs phc_reset_envs over them.
// The uniform numbers and the env mask ride in the chunk's packed clock transfer.  The new state of a re-posed env
// (~1.9 KB) is not in any buffer the plain step sends back, and only a few percent of the envs are re-posed per step:
// one small kernel per chunk (host_export_kernel) writes the rows of those envs alone into the caller's buffers when
// they are pinned, else into the slot's pinned staging, from which wait copies the rows of the flagged envs.
//
// Device outputs.  phc_host_step_submit_device / phc_host_reset_submit_device run the same pipelines with the obs rows
// (and the normalised rows and RunningNorm moments) written by the kernels into the caller's device tensors: no obs
// transfer at all, only the scalars and the reset rows return to the host.  Each chunk's stream waits for an event
// recorded on the caller's stream before its kernel, so the policy's reads of the previous rows come first.
//
// Env options.  phc_host_step_submit_env / phc_host_reset_submit_env run the same pipelines with the power reward (each
// chunk's dof force and dof velocity rows are copied by the copy engine straight from the caller's buffers into the
// slot's device scratch: two transfers per chunk, no CPU copy), mpjpe (posted by the kernel on the direct path, in the
// packed scalars on the staged path) and StateInit.Default / Hybrid (the initial rows are uploaded once per slot by
// phc_host_step_set_initial_state; the hybrid mask rides in the packed clock).  Every other submit is one of these
// with no options.
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include <cuda_runtime.h>

#include "../../include/phc_b200.h"

// phc_kernels.cu: phc_step_fused that also writes the advanced progress to a second address
int step_fused_mirrored(const PhcLib* lib, const PhcStepArgs* args, int64_t n, phc_stream_t stream, int16_t* progress_mirror);
bool lib_has_dof_state(const PhcLib* lib);  // phc_kernels.cu
namespace phc {
int record_cuda_error(int cuda_error);  // phc_kernels.cu; returns PHC_ERR_CUDA
}

namespace {

constexpr int kStreams = 3;
constexpr int kStateFloats = PHC_NUM_BODIES * 13;
// packed clock, per env: ids i64 | goff 3 f32 | start f32 | soff f32 | progress i16  (SoA per chunk)
constexpr size_t kClockBytes = 8 + 12 + 4 + 4 + 2;
// packed scalars out, per env: rew f32 | raw 4 f32 | progress i16 | reset u8 | term u8
// (with the env options: raw 5 f32 with the power reward, mpjpe f32, and default_mask u8 in the clock)
constexpr size_t kOutBytes = 4 + 16 + 2 + 1 + 1;
constexpr int kDof = 69;
constexpr int kMaxChunks = 1024;

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// sub-array offsets inside a chunk's packed regions (each 16-B aligned)
struct Layout {
  size_t ids, goff, start, soff, prog, phase, mask, dmask, clock_bytes;
  size_t rew, raw, mpjpe, oprog, reset, term, out_bytes;
};
// What the env options add to a chunk's packed regions: reward_raw columns (5 with the power reward), mpjpe f32 out,
// the hybrid default_mask u8 in the clock.
struct Extra {
  int raw_cols = 4;
  bool mpjpe = false, dmask = false;
};
// with_reset: the clock also carries phase f32 | env_mask u8 per env
Layout layout(int64_t m, bool with_reset = false, const Extra& x = Extra{}) {
  Layout L;
  size_t o = 0;
  L.ids = o, o = align_up(o + (size_t)m * 8, 16);
  L.goff = o, o = align_up(o + (size_t)m * 12, 16);
  L.start = o, o = align_up(o + (size_t)m * 4, 16);
  L.soff = o, o = align_up(o + (size_t)m * 4, 16);
  L.prog = o, o = align_up(o + (size_t)m * 2, 16);
  L.phase = L.mask = L.dmask = o;
  if (with_reset) {
    L.phase = o, o = align_up(o + (size_t)m * 4, 16);
    L.mask = o, o = align_up(o + (size_t)m, 16);
    L.dmask = o;
    if (x.dmask) o = align_up(o + (size_t)m, 16);
  }
  L.clock_bytes = o;
  o = 0;
  L.rew = o, o = align_up(o + (size_t)m * 4, 16);
  L.raw = o, o = align_up(o + (size_t)m * 4 * x.raw_cols, 16);
  L.mpjpe = o;
  if (x.mpjpe) o = align_up(o + (size_t)m * 4, 16);
  L.oprog = o, o = align_up(o + (size_t)m * 2, 16);
  L.reset = o, o = align_up(o + (size_t)m, 16);
  L.term = o, o = align_up(o + (size_t)m, 16);
  L.out_bytes = o;
  return L;
}

enum Op { kStep, kStepReset, kReset };  // phc_host_step(_submit) / phc_host_step_submit_reset / phc_host_reset_submit

// The per-env host arrays a reset writes (rows of re-posed envs only): the caller's buffers, or the slot's staging.
struct Rows {
  float *state, *root, *dofp, *dofv, *start, *soff, *goff, *obs;
  int16_t* prog;
  uint8_t *rst, *term;
};
Rows rows_at(const Rows& R, int64_t lo, int64_t obs_dim) {
  auto at = [](auto* p, int64_t off) { return p ? p + off : p; };
  return {at(R.state, lo * kStateFloats), at(R.root, lo * 13), at(R.dofp, lo * 69), at(R.dofv, lo * 69),
          at(R.start, lo), at(R.soff, lo), at(R.goff, lo * 3), at(R.obs, lo * obs_dim), at(R.prog, lo),
          at(R.rst, lo), at(R.term, lo)};
}

// The export of one chunk: every array is chunk-local; `out` points into mapped host memory.
struct ExportParams {
  const uint8_t* flag;       // device [m]: env i is exported when set (the step's reset_out, or the reset's env mask)
  const uint8_t* step_term;  // device [m] or NULL: with it, flag / step_term / prog of EVERY env go to out.rst / .term / .prog
  const float *state, *root, *dofp, *dofv, *start, *soff, *goff, *obs;  // device; obs may be NULL
  const int16_t* prog;
  Rows out;                  // out.obs / .prog / .rst / .term may be NULL (not exported)
  int zero_flags;            // the host reset: rst / term of exported envs -> 0
  int64_t obs_dim, m;
};

__device__ __forceinline__ void warp_copy(float* dst, const float* src, int count, int lane) {
  for (int j = lane; j < count; j += 32) dst[j] = src[j];
}

// One warp per env; an env that is not flagged costs one byte read.  A warp's stores are consecutive words, so the
// rows leave as full 128-B posted writes.
constexpr int kExportEnvs = 8;
__global__ void __launch_bounds__(kExportEnvs * 32) host_export_kernel(const ExportParams p) {
  const int lane = threadIdx.x & 31;
  if (p.step_term && threadIdx.x < kExportEnvs) {  // the block's flags and progress as one write each
    const int64_t e = (int64_t)blockIdx.x * kExportEnvs + threadIdx.x;
    if (e < p.m) {
      p.out.rst[e] = p.flag[e];
      p.out.term[e] = p.step_term[e];
      p.out.prog[e] = p.prog[e];
    }
  }
  const int64_t i = (int64_t)blockIdx.x * kExportEnvs + (threadIdx.x >> 5);
  if (i >= p.m || !p.flag[i]) return;
  warp_copy(p.out.state + i * kStateFloats, p.state + i * kStateFloats, kStateFloats, lane);
  warp_copy(p.out.root + i * 13, p.root + i * 13, 13, lane);
  warp_copy(p.out.dofp + i * 69, p.dofp + i * 69, 69, lane);
  warp_copy(p.out.dofv + i * 69, p.dofv + i * 69, 69, lane);
  warp_copy(p.out.goff + i * 3, p.goff + i * 3, 3, lane);
  if (p.out.obs) warp_copy(p.out.obs + i * p.obs_dim, p.obs + i * p.obs_dim, (int)p.obs_dim, lane);
  if (lane == 0) {
    p.out.start[i] = p.start[i];
    p.out.soff[i] = p.soff[i];
    if (p.out.prog && !p.step_term) p.out.prog[i] = p.prog[i];
    if (p.zero_flags) p.out.rst[i] = p.out.term[i] = 0;
  }
}

// One pipeline: what a step in flight uses, and what phc_host_step_wait needs to finish it.
struct Slot {
  bool ready = false;  // buffers, streams and events allocated
  float* d_state = nullptr;
  float* d_obs = nullptr;
  unsigned char* d_clock = nullptr;  // packed clock, device
  unsigned char* d_out = nullptr;    // packed scalar outputs, device
  unsigned char* h_clock = nullptr;  // pinned staging
  unsigned char* h_out = nullptr;    // pinned staging
  cudaStream_t streams[kStreams] = {};
  cudaEvent_t done[kStreams] = {};  // recorded on each stream at the end of an enqueue
  cudaEvent_t dev_ready = nullptr;  // device-output submits: recorded on the caller's stream, waited on before a kernel
  // direct path: verdict cached per set of caller pointers (the 11 of PhcHostStepArgs and PhcHostEnvArgs.mpjpe)
  const void* seen[12] = {};
  int seen_direct = -1;
  // resets, allocated at the first submit that needs them: device root / dof rows of re-posed envs and the flags the
  // reset clears (the caller gets the step's own flags), [max_envs] each; pinned staging of the reset outputs
  unsigned char* d_reset = nullptr;
  float *d_root = nullptr, *d_dofp = nullptr, *d_dofv = nullptr;
  uint8_t *d_kreset = nullptr, *d_kterm = nullptr;
  unsigned char* h_rows = nullptr;
  Rows stage{};
  const void* rseen[9] = {};  // verdict of the reset pointers: the outputs are all pinned and mapped at their address
  int rseen_direct = -1;
  // env options, allocated at first use: the chunk's dof force and dof velocity rows ([max_envs, 2, 69]: per chunk
  // m force rows, then m velocity rows), and the initial root / dof rows of StateInit.Default / Hybrid
  float* d_dof = nullptr;
  float* d_init = nullptr;  // [max_envs] x (13 root | 69 dof pos | 69 dof vel), init_rows of them set
  int64_t init_rows = -1;   // -1: no initial state
  const void* eseen[3] = {};  // the env inputs last found to be host memory
  // the step in flight
  bool busy = false;
  int path = 0;  // 1 direct, 2 staged
  int op = kStep;
  bool rows_staged = false;  // the reset rows go through `stage`, wait copies those of the flagged envs
  int64_t n = 0;
  PhcHostStepArgs args{};
  PhcHostResetArgs rargs{};
  PhcHostEnvArgs env{};
  Extra extra{};
  int nchunks = 0;
  int64_t bounds[kMaxChunks + 2] = {};  // staged path: chunk boundaries, for the unpack in wait
};

}  // namespace

struct PhcHostStep {
  const PhcLib* lib = nullptr;
  int64_t max_envs = 0;
  int32_t T = 1;
  int32_t chunks = 1;
  int64_t obs_dim = 0;
  int device = 0;  // the device current at create: device outputs must live there
  float* term_dist = nullptr;
  uint32_t reset_mask = 0xFFFFFF;
  int32_t use_mean = 0, early = 1;
  float dt = 0.f;
  PhcRewardSpec rwd{};
  size_t pack_capacity = 0;
  Slot slots[PHC_HOST_SLOTS];
  int last_slot = 0;  // the slot of the last submit: phc_host_step_path / _chunks report its verdict
  // which output path pinned callers take: 0 = auto (time both over the first calls, keep the faster), 1 = direct
  // (kernels post into the mapped host buffers), 2 = staged (copy-engine D2H).  PHC_HOST_PATH=auto|direct|staged.
  int mode = 0;
  // the schedule (output path, chunk count) of pinned callers is tuned over the first calls: every candidate is timed
  // kTuneReps times, interleaved, and the fastest mean stays.  num_chunks > 0 at create and PHC_HOST_PATH narrow the
  // candidates (down to one: nothing to tune).
  struct Cand { int path, chunks; double t; int n; };  // t: fastest timed call so far
  Cand cand[8] = {};
  int ncand = 0;
  int chosen = -1;  // index into cand once decided
  int calls = 0;
};
constexpr int kTuneWarm = 2, kTuneReps = 4;

// After the first enqueue an early return must not leave kernels writing into the caller's (mapped) buffers or
// into the staging buffers the next call reuses: every error path drains the slot's three streams first.
static int host_fail(Slot& s, int rc, cudaError_t e) {
  for (auto& st : s.streams)
    if (st) (void)cudaStreamSynchronize(st);
  (void)cudaGetLastError();
  return e != cudaSuccess ? phc::record_cuda_error((int)e) : rc;
}
#define HOST_CUDA(slot, call)                                        \
  do {                                                               \
    cudaError_t e__ = (call);                                        \
    if (e__ != cudaSuccess) return host_fail((slot), PHC_ERR_CUDA, e__); \
  } while (0)

static cudaError_t slot_alloc(const PhcHostStep* c, Slot& s) {
  const size_t n = (size_t)c->max_envs;
  cudaError_t e = cudaSuccess;
  auto dmalloc = [&](void** p, size_t bytes) {
    if (e == cudaSuccess) e = cudaMalloc(p, bytes);
  };
  dmalloc((void**)&s.d_state, n * kStateFloats * sizeof(float));
  dmalloc((void**)&s.d_obs, n * c->obs_dim * sizeof(float));
  dmalloc((void**)&s.d_clock, c->pack_capacity);
  dmalloc((void**)&s.d_out, c->pack_capacity);
  if (e == cudaSuccess) e = cudaMallocHost((void**)&s.h_clock, c->pack_capacity);
  if (e == cudaSuccess) e = cudaMallocHost((void**)&s.h_out, c->pack_capacity);
  for (int i = 0; i < kStreams && e == cudaSuccess; ++i) {
    e = cudaStreamCreateWithFlags(&s.streams[i], cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.done[i], cudaEventDisableTiming);
  }
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.dev_ready, cudaEventDisableTiming);
  s.ready = e == cudaSuccess;
  return e;
}

static void slot_free(Slot& s) {
  for (auto& st : s.streams)
    if (st) (void)cudaStreamSynchronize(st);
  cudaFree(s.d_state);
  cudaFree(s.d_obs);
  cudaFree(s.d_clock);
  cudaFree(s.d_out);
  cudaFree(s.d_reset);
  cudaFree(s.d_dof);
  cudaFree(s.d_init);
  if (s.h_clock) cudaFreeHost(s.h_clock);
  if (s.h_out) cudaFreeHost(s.h_out);
  if (s.h_rows) cudaFreeHost(s.h_rows);
  for (int i = 0; i < kStreams; ++i) {
    if (s.done[i]) cudaEventDestroy(s.done[i]);
    if (s.streams[i]) cudaStreamDestroy(s.streams[i]);
  }
  if (s.dev_ready) cudaEventDestroy(s.dev_ready);
  s = Slot{};
}

// Everything phc_host_step validates, before anything is enqueued; fills the slot's direct-path verdict.  With device
// outputs (dev_out) obs_buf must be NULL: the rows go to the device tensors only.
static int check_args(PhcHostStep* c, Slot& s, const PhcHostStepArgs* a, int64_t n, bool dev_out = false,
                      const float* mpjpe = nullptr) {
  if (n < 0 || n > c->max_envs) return PHC_ERR_SHAPE;
  if (!a->state || !a->progress_buf || !a->motion_start_times || !a->motion_start_times_offset ||
      !a->global_offset || !a->sampled_motion_ids || (!dev_out && !a->obs_buf) || !a->rew_buf || !a->reward_raw ||
      !a->reset_buf || !a->terminate_buf)
    return PHC_ERR_NULL;
  if (dev_out && a->obs_buf) return PHC_ERR_UNSUPPORTED;
  // ---- can the direct path be used: every buffer is pinned / managed host memory mapped at its own address ----------
  const void* ptrs[12] = {a->state, a->progress_buf, a->motion_start_times, a->motion_start_times_offset,
                          a->global_offset, a->sampled_motion_ids, a->obs_buf, a->rew_buf, a->reward_raw,
                          a->reset_buf, a->terminate_buf, mpjpe};
  if (s.seen_direct < 0 || memcmp(ptrs, s.seen, sizeof(ptrs)) != 0) {
    int direct = 1;
    for (int i = 0; i < 12 && direct; ++i) {
      if (!ptrs[i]) continue;  // obs_buf of a device-output submit, mpjpe when not asked for
      cudaPointerAttributes at{};
      if (cudaPointerGetAttributes(&at, ptrs[i]) != cudaSuccess) {
        (void)cudaGetLastError();
        direct = 0;
      } else if (at.type == cudaMemoryTypeDevice) {
        return PHC_ERR_UNSUPPORTED;  // this entry point takes HOST buffers (the clock arrays are memcpy'd by the CPU)
      } else if ((at.type != cudaMemoryTypeHost && at.type != cudaMemoryTypeManaged) || at.devicePointer != ptrs[i]) {
        direct = 0;  // pageable, or mapped at a different device address
      }
    }
    memcpy(s.seen, ptrs, sizeof(ptrs));
    s.seen_direct = direct;
  }
  return PHC_OK;
}

// Everything the two reset submits validate on top of check_args; fills the slot's verdict for the reset outputs.
// env: the env options of an _env submit, NULL for the submits without them (which refuse StateInit.Default / Hybrid).
static int check_reset(const PhcHostStep* c, Slot& s, const PhcHostResetArgs* r, int op, const PhcHostEnvArgs* env,
                       int64_t n) {
  if (!r->state_out || !r->root_states || !r->dof_pos || !r->dof_vel || !r->motion_start_times_out ||
      !r->motion_start_times_offset_out || !r->global_offset_out || (op == kReset && !r->env_mask))
    return PHC_ERR_NULL;
  if (r->state_init < PHC_STATE_INIT_START || r->state_init > (env ? PHC_STATE_INIT_HYBRID : PHC_STATE_INIT_RANDOM))
    return PHC_ERR_UNSUPPORTED;
  if ((r->state_init == PHC_STATE_INIT_RANDOM || r->state_init == PHC_STATE_INIT_HYBRID) && !r->phase)
    return PHC_ERR_NULL;
  // StateInit.Default / Hybrid: the slot's initial rows (phc_host_step_set_initial_state) stand for envs 0..n-1
  if (r->state_init >= PHC_STATE_INIT_DEFAULT) {
    if (s.init_rows < 0 || (r->state_init == PHC_STATE_INIT_HYBRID && !env->default_mask)) return PHC_ERR_NULL;
    if (n > s.init_rows) return PHC_ERR_SHAPE;
  }
  if (!lib_has_dof_state(c->lib)) return PHC_ERR_UNSUPPORTED;
  // outputs first (their verdict), then the two inputs the CPU packs (only refused when on the device)
  const void* ptrs[9] = {r->state_out, r->root_states, r->dof_pos, r->dof_vel, r->motion_start_times_out,
                         r->motion_start_times_offset_out, r->global_offset_out, r->phase, r->env_mask};
  if (s.rseen_direct < 0 || memcmp(ptrs, s.rseen, sizeof(ptrs)) != 0) {
    int direct = 1;
    for (int i = 0; i < 9; ++i) {
      if (!ptrs[i]) continue;
      cudaPointerAttributes at{};
      if (cudaPointerGetAttributes(&at, ptrs[i]) != cudaSuccess) {
        (void)cudaGetLastError();
        if (i < 7) direct = 0;
      } else if (at.type == cudaMemoryTypeDevice) {
        return PHC_ERR_UNSUPPORTED;
      } else if (i < 7 && ((at.type != cudaMemoryTypeHost && at.type != cudaMemoryTypeManaged) || at.devicePointer != ptrs[i])) {
        direct = 0;
      }
    }
    memcpy(s.rseen, ptrs, sizeof(ptrs));
    s.rseen_direct = direct;
  }
  return PHC_OK;
}

// What the device-output submits validate on top of check_args (and check_reset).
static int check_dev(const PhcHostStep* c, const PhcHostDeviceOut* d) {
  if (d->obs_norm && (!d->norm_mean || !d->norm_var)) return PHC_ERR_NULL;
  if (d->flags & ~PHC_STEP_OBS_NORM_BF16) return PHC_ERR_UNSUPPORTED;
  const void* ptrs[5] = {d->obs, d->obs_norm, d->norm_mean, d->norm_var, d->obs_moments};
  for (const void* p : ptrs) {
    if (!p) continue;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
      (void)cudaGetLastError();
      return PHC_ERR_UNSUPPORTED;
    }
    if (at.type != cudaMemoryTypeDevice || at.device != c->device) return PHC_ERR_UNSUPPORTED;
  }
  if ((((uintptr_t)d->obs | (uintptr_t)d->obs_norm) & 15) != 0) return PHC_ERR_ALIGN;
  if (d->obs_moments_buckets < 0 || d->obs_moments_buckets > 4096 || (d->obs_norm && !(d->norm_clip > 0.0f)))
    return PHC_ERR_SHAPE;
  return PHC_OK;
}

// What the env-option submits validate on top of check_args (which takes mpjpe into the direct-path verdict): the power
// inputs come in pairs, and every env field is host memory.  The verdict is cached per set of pointers.
static int check_env(Slot& s, const PhcHostEnvArgs* e) {
  if (!e->dof_force != !e->dof_vel) return PHC_ERR_NULL;
  const void* ptrs[3] = {e->dof_force, e->dof_vel, e->default_mask};
  if (memcmp(ptrs, s.eseen, sizeof(ptrs)) == 0) return PHC_OK;
  for (const void* p : ptrs) {
    if (!p) continue;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
      (void)cudaGetLastError();  // pageable
    } else if (at.type == cudaMemoryTypeDevice) {
      return PHC_ERR_UNSUPPORTED;
    }
  }
  memcpy(s.eseen, ptrs, sizeof(ptrs));
  return PHC_OK;
}

// The power-reward inputs of one chunk: its dof force and dof velocity rows, copied by the copy engine from the caller's
// buffers into the slot's scratch, and the step's power fields pointing there.  Two transfers rather than one through
// staging: packing would first copy 552 B per env on the caller's thread (33 us per 4096-env batch-step on a B200 host,
// profiles/r6_host_env_options.md).  Nothing without a dof force.
static cudaError_t power_inputs(const Slot& s, int64_t lo, int64_t m, cudaStream_t st, PhcStepArgs& k) {
  const PhcHostEnvArgs& e = s.env;
  if (!e.dof_force) return cudaSuccess;
  float* df = s.d_dof + lo * 2 * kDof;
  float* dv = df + m * kDof;
  const size_t bytes = (size_t)m * kDof * sizeof(float);
  cudaError_t err = cudaMemcpyAsync(df, e.dof_force + lo * kDof, bytes, cudaMemcpyHostToDevice, st);
  if (err == cudaSuccess) err = cudaMemcpyAsync(dv, e.dof_vel + lo * kDof, bytes, cudaMemcpyHostToDevice, st);
  k.dof_force = df;
  k.dof_force_stride = kDof;
  k.dof_vel = dv;
  k.dof_vel_stride = kDof;
  k.dof_vel_elem_stride = 1;
  k.rew_power_coef = e.rew_power_coef;
  k.power_col = 4;
  return err;
}

// The chunk's rows in the caller's device tensors.  Chunks start on multiples of 8 envs, so the fp32 and the bf16 rows
// of every chunk start 16-B aligned.
static float* dev_obs(const PhcHostStep* c, const PhcHostDeviceOut* d, int64_t lo) { return d->obs + lo * c->obs_dim; }
static float* dev_obs_norm(const PhcHostStep* c, const PhcHostDeviceOut* d, int64_t lo) {
  if (!d->obs_norm) return nullptr;
  const int64_t bytes = (d->flags & PHC_STEP_OBS_NORM_BF16) ? 2 : 4;
  return (float*)((char*)d->obs_norm + lo * c->obs_dim * bytes);
}
static void dev_step_outputs(const PhcHostStep* c, const PhcHostDeviceOut* d, int64_t lo, PhcStepArgs& k) {
  k.obs_buf = dev_obs(c, d, lo);
  k.obs_norm = dev_obs_norm(c, d, lo);
  k.obs_norm_stride = c->obs_dim;
  k.norm_mean = d->norm_mean;
  k.norm_var = d->norm_var;
  k.norm_epsilon = d->norm_epsilon;
  k.norm_clip = d->norm_clip;
  k.flags |= d->flags;
  k.obs_moments = d->obs_moments;
  k.obs_moments_buckets = d->obs_moments_buckets;
}

// The reset scratch of a slot; the pinned staging only when the rows of this submit go through it.
static cudaError_t reset_alloc(const PhcHostStep* c, Slot& s, bool staging) {
  const size_t n = (size_t)c->max_envs;
  cudaError_t e = cudaSuccess;
  if (!s.d_reset) {
    e = cudaMalloc((void**)&s.d_reset, n * (13 + 69 + 69) * sizeof(float) + 2 * n);
    if (e != cudaSuccess) return e;
    s.d_root = (float*)s.d_reset;
    s.d_dofp = s.d_root + n * 13;
    s.d_dofv = s.d_dofp + n * 69;
    s.d_kreset = (uint8_t*)(s.d_dofv + n * 69);
    s.d_kterm = s.d_kreset + n;
  }
  if (staging && !s.h_rows) {
    const size_t floats[8] = {n * kStateFloats, n * 13, n * 69, n * 69, n, n, n * 3, n * (size_t)c->obs_dim};
    size_t off[8], o = 0;
    for (int i = 0; i < 8; ++i) off[i] = o, o = align_up(o + floats[i] * sizeof(float), 16);
    const size_t prog = o, rst = align_up(prog + n * 2, 16), term = rst + n;
    e = cudaMallocHost((void**)&s.h_rows, term + n);
    if (e != cudaSuccess) return e;
    float* f[8];
    for (int i = 0; i < 8; ++i) f[i] = (float*)(s.h_rows + off[i]);
    s.stage = Rows{f[0], f[1], f[2], f[3], f[4], f[5], f[6], f[7], (int16_t*)(s.h_rows + prog), s.h_rows + rst,
                   s.h_rows + term};
  }
  return e;
}

// The env-option scratch of a slot: the dof rows when this submit has the power reward.
static cudaError_t env_alloc(const PhcHostStep* c, Slot& s) {
  if (!s.env.dof_force || s.d_dof) return cudaSuccess;
  return cudaMalloc((void**)&s.d_dof, (size_t)c->max_envs * 2 * kDof * sizeof(float));
}

// The caller's buffers as export targets
static Rows caller_rows(const PhcHostStepArgs* a, const PhcHostResetArgs* r) {
  return {r->state_out, r->root_states, r->dof_pos, r->dof_vel, r->motion_start_times_out,
          r->motion_start_times_offset_out, r->global_offset_out, a->obs_buf, a->progress_buf, a->reset_buf,
          a->terminate_buf};
}

static PhcBodyState chunk_body(float* st) {
  return PhcBodyState{PhcView{st, kStateFloats, 13}, PhcView{st + 3, kStateFloats, 13}, PhcView{st + 7, kStateFloats, 13},
                      PhcView{st + 10, kStateFloats, 13}, PHC_NUM_BODIES};
}

// Packs a chunk's clock (and, with a reset, its uniform numbers and env mask) into pinned staging.
static void pack_clock(unsigned char* hc, const Layout& L, const PhcHostStepArgs* a, const PhcHostResetArgs* r,
                       const PhcHostEnvArgs& env, int64_t lo, int64_t m) {
  memcpy(hc + L.ids, a->sampled_motion_ids + lo, (size_t)m * 8);
  memcpy(hc + L.goff, a->global_offset + lo * 3, (size_t)m * 12);
  memcpy(hc + L.start, a->motion_start_times + lo, (size_t)m * 4);
  memcpy(hc + L.soff, a->motion_start_times_offset + lo, (size_t)m * 4);
  memcpy(hc + L.prog, a->progress_buf + lo, (size_t)m * 2);
  if (r && r->phase) memcpy(hc + L.phase, r->phase + lo, (size_t)m * 4);
  if (r && r->env_mask) memcpy(hc + L.mask, r->env_mask + lo, (size_t)m);
  if (r && r->state_init == PHC_STATE_INIT_HYBRID) memcpy(hc + L.dmask, env.default_mask + lo, (size_t)m);
}

// The reset over a chunk's device copies.  A step's auto_reset must name the step's own body / clock / flag / obs
// pointers (phc_step_fused checks it), so both are derived from the same chunk offsets.
static PhcResetArgs chunk_reset_args(const PhcHostStep* c, const Slot& s, const PhcHostResetArgs* r, float* st,
                                     unsigned char* dc, const Layout& L, int64_t lo, float* obs) {
  PhcResetArgs ra{};
  ra.body = chunk_body(st);
  ra.humanoid_root_states = s.d_root + lo * 13;
  ra.root_stride = 13;
  ra.dof_pos = s.d_dofp + lo * 69;
  ra.dof_vel = s.d_dofv + lo * 69;
  ra.dof_stride = 69;
  ra.dof_elem_stride = 1;
  ra.progress_buf = (int16_t*)(dc + L.prog);
  ra.reset_buf = s.d_kreset + lo;
  ra.terminate_buf = s.d_kterm + lo;
  ra.motion_start_times = (float*)(dc + L.start);
  ra.motion_start_times_offset = (float*)(dc + L.soff);
  ra.global_offset = (float*)(dc + L.goff);
  ra.sampled_motion_ids = (const int64_t*)(dc + L.ids);
  ra.env_mask = dc + L.mask;
  ra.phase = r->phase ? (const float*)(dc + L.phase) : nullptr;
  ra.state_init = r->state_init;
  ra.flag_test = r->flag_test;
  if (r->state_init >= PHC_STATE_INIT_DEFAULT) {  // the slot's initial rows of the chunk's envs
    const int64_t N = c->max_envs;
    ra.initial_root_states = s.d_init + lo * 13;
    ra.initial_root_stride = 13;
    ra.initial_dof_pos = s.d_init + N * 13 + lo * kDof;
    ra.initial_dof_vel = s.d_init + N * (13 + kDof) + lo * kDof;
    ra.initial_dof_stride = kDof;
    if (r->state_init == PHC_STATE_INIT_HYBRID) ra.default_mask = dc + L.dmask;
  }
  ra.time_steps = c->T;
  ra.dt = c->dt;
  ra.obs_buf = obs;
  ra.obs_stride = c->obs_dim;
  return ra;
}

// The export of the reset rows of one chunk whose device copies `ra` names.
static cudaError_t export_rows(const PhcHostStep* c, const PhcResetArgs& ra, const uint8_t* flag,
                               const uint8_t* step_term, const float* obs, const Rows& out, int zero_flags, int64_t m,
                               cudaStream_t st) {
  ExportParams p{};
  p.flag = flag;
  p.step_term = step_term;
  p.state = ra.body.pos.ptr;
  p.root = ra.humanoid_root_states;
  p.dofp = ra.dof_pos;
  p.dofv = ra.dof_vel;
  p.start = ra.motion_start_times;
  p.soff = ra.motion_start_times_offset;
  p.goff = ra.global_offset;
  p.obs = obs;
  p.prog = ra.progress_buf;
  p.out = out;
  p.zero_flags = zero_flags;
  p.obs_dim = c->obs_dim;
  p.m = m;
  host_export_kernel<<<(unsigned)((m + kExportEnvs - 1) / kExportEnvs), kExportEnvs * 32, 0, st>>>(p);
  return cudaGetLastError();
}

static int direct_enqueue(PhcHostStep* c, Slot& s, const PhcHostStepArgs* a, const PhcHostResetArgs* r,
                          const PhcHostDeviceOut* dev, int64_t n, const int chunks) {
  // Hybrid: everything INBOUND rides the host->device copy engine in a few chunks — the sim
  // rows directly from the caller's buffer, the five small clock arrays packed into one
  // transfer (SM-issued reads of system memory are 32-B PCIe round trips: 6 per block, ~70 us
  // per 4096-env step when the kernel read the clock in place) — while each chunk's kernel
  // WRITES obs rows, rewards and flags straight into the mapped host buffers.  The copy
  // engine pulling chunk c+1 and the kernel pushing chunk c's rows use opposite directions of
  // the link.  The advanced progress is written to the caller's buffer by the kernel as well.
  // equal chunks here: measured, a small first chunk does not help this path (the step is
  // bound by the kernels' posted writes, ~300 us per 4096 envs, plus the first copy)
  const int C = chunks < 1 ? 1 : chunks;
  int64_t per = (n + C - 1) / C;
  per = (per + 7) / 8 * 8;
  size_t coff = 0, ooff = 0;
  int ci = 0;
  // with a reset the step's own flags go to device scratch (the export kernel posts them to the caller with the rows)
  const Rows rows = r ? (s.rows_staged ? s.stage : caller_rows(a, r)) : Rows{};
  static const bool trace_on = getenv("PHC_HOST_TRACE") != nullptr;
  static int trace_calls = 0;
  const bool trace = trace_on && ++trace_calls == 20;
  cudaEvent_t ev0 = nullptr, evh[64], evk[64];
  double host_us[64];
  const auto th0 = std::chrono::steady_clock::now();
  if (trace) {
    cudaEventCreate(&ev0);
    cudaEventRecord(ev0, s.streams[0]);
  }
  for (int64_t lo = 0; lo < n; lo += per, ++ci) {
    const int64_t m = (n - lo) < per ? (n - lo) : per;
    const Layout L = layout(m, r != nullptr, s.extra);
    if (coff + L.clock_bytes > c->pack_capacity || ooff + L.out_bytes > c->pack_capacity)
      return host_fail(s, PHC_ERR_SHAPE, cudaSuccess);
    cudaStream_t st_ = s.streams[ci % kStreams];
    float* st = s.d_state + lo * kStateFloats;
    unsigned char* hc = s.h_clock + coff;
    unsigned char* dc = s.d_clock + coff;
    unsigned char* dout = s.d_out + ooff;
    pack_clock(hc, L, a, r, s.env, lo, m);
    HOST_CUDA(s, cudaMemcpyAsync(dc, hc, L.clock_bytes, cudaMemcpyHostToDevice, st_));
    HOST_CUDA(s, cudaMemcpyAsync(st, a->state + lo * kStateFloats, (size_t)m * kStateFloats * sizeof(float),
                                 cudaMemcpyHostToDevice, st_));
    PhcStepArgs k{};
    if (trace && ci < 64) {
      cudaEventCreate(&evh[ci]);
      cudaEventRecord(evh[ci], st_);
    }
    k.body = chunk_body(st);
    k.progress_buf = (int16_t*)(dc + L.prog);
    k.motion_start_times = (const float*)(dc + L.start);
    k.motion_start_times_offset = (const float*)(dc + L.soff);
    k.global_offset = (const float*)(dc + L.goff);
    k.sampled_motion_ids = (const int64_t*)(dc + L.ids);
    k.termination_distances = c->term_dist;
    k.reset_body_mask = c->reset_mask;
    k.use_mean = c->use_mean;
    k.enable_early_termination = c->early;
    k.advance_progress = 1;
    k.time_steps = c->T;
    k.dt = c->dt;
    k.rwd = c->rwd;
    k.obs_buf = a->obs_buf + lo * c->obs_dim;
    k.obs_stride = c->obs_dim;
    k.rew_buf = a->rew_buf + lo;
    k.reward_raw = a->reward_raw + lo * s.extra.raw_cols;
    k.reward_raw_stride = s.extra.raw_cols;
    k.reset_buf = a->reset_buf + lo;
    k.terminate_buf = a->terminate_buf + lo;
    k.flags = PHC_STEP_MAPPED_HOST_IO;
    k.obs_moments = nullptr;
    k.mpjpe = s.env.mpjpe ? s.env.mpjpe + lo : nullptr;
    HOST_CUDA(s, power_inputs(s, lo, m, st_, k));
    if (dev) dev_step_outputs(c, dev, lo, k);
    PhcResetArgs ra;
    if (r) {
      k.reset_buf = s.d_kreset + lo;
      k.terminate_buf = s.d_kterm + lo;
      k.reset_out = dout + L.reset;
      k.terminate_out = dout + L.term;
      ra = chunk_reset_args(c, s, r, st, dc, L, lo, k.obs_buf);
      k.auto_reset = &ra;
    }
    // the advanced progress goes straight into the caller's buffer too (no device->host copy at the tail).  Not with a
    // reset: where it runs as a second launch (T > 1 here, or the generic kernel) the mirror would keep the advanced
    // progress of the re-posed envs, so the progress leaves with the flags, from the device clock after the reset.
    if (dev) HOST_CUDA(s, cudaStreamWaitEvent(st_, s.dev_ready, 0));
    int rc = step_fused_mirrored(c->lib, &k, m, st_, r ? nullptr : a->progress_buf + lo);
    if (rc) return host_fail(s, rc, cudaSuccess);
    if (r) {
      Rows out = rows_at(rows, lo, c->obs_dim);
      out.obs = nullptr;
      out.prog = a->progress_buf + lo;
      out.rst = a->reset_buf + lo;
      out.term = a->terminate_buf + lo;
      HOST_CUDA(s, export_rows(c, ra, dout + L.reset, dout + L.term, nullptr, out, 0, m, st_));
      ooff += L.out_bytes;
    }
    if (trace && ci < 64) {
      cudaEventCreate(&evk[ci]);
      cudaEventRecord(evk[ci], st_);
      host_us[ci] = std::chrono::duration<double>(std::chrono::steady_clock::now() - th0).count() * 1e6;
    }
    coff += L.clock_bytes;
  }
  if (trace) {
    for (auto st_ : s.streams) HOST_CUDA(s, cudaStreamSynchronize(st_));
    const double tot = std::chrono::duration<double>(std::chrono::steady_clock::now() - th0).count() * 1e6;
    fprintf(stderr, "[phc_host trace] %d chunks of %lld envs, host total %.1f us\n", ci, (long long)per, tot);
    for (int i = 0; i < ci && i < 64; ++i) {
      float a_ms = 0, b_ms = 0;
      cudaEventElapsedTime(&a_ms, ev0, evh[i]);
      cudaEventElapsedTime(&b_ms, ev0, evk[i]);
      fprintf(stderr, "  chunk %d: submitted at %.1f us (host), H2D done %.1f us, kernel done %.1f us\n", i, host_us[i],
              a_ms * 1e3, b_ms * 1e3);
    }
  }
  return PHC_OK;
}

static int staged_enqueue(PhcHostStep* c, Slot& s, const PhcHostStepArgs* a, const PhcHostResetArgs* r,
                          const PhcHostDeviceOut* dev, int64_t n, const int chunks) {
  const cudaMemcpyKind H2D = cudaMemcpyHostToDevice, D2H = cudaMemcpyDeviceToHost;
  // Chunk sizes double (n/2^(C-1), n/2^(C-1), n/2^(C-2), .., n/2): the device->host direction
  // carries 3x the bytes and is the bottleneck, so the first chunk is small to start it early
  // while the later, larger chunks keep the per-transfer overhead low.  Boundaries fall on
  // multiples of 8 envs so every chunk's obs rows start 16-B aligned.
  {
    const int C = chunks < 1 ? 1 : chunks;
    int64_t lo = 0;
    s.nchunks = 0;
    s.bounds[0] = 0;
    for (int i = 0; i < C && lo < n; ++i) {
      const int shift = (i == 0) ? C - 1 : C - i;
      int64_t sz = shift < 62 ? (n >> shift) : 0;
      sz = (sz + 7) / 8 * 8;
      if (sz < 8) sz = 8;
      int64_t hi = (i == C - 1) ? n : (lo + sz < n ? lo + sz : n);
      s.bounds[++s.nchunks] = hi;
      lo = hi;
    }
    s.bounds[s.nchunks] = n;
  }
  const int nchunks = s.nchunks;
  const int64_t* bounds = s.bounds;

  size_t coff = 0, ooff = 0;
  const Rows rows = r ? (s.rows_staged ? s.stage : caller_rows(a, r)) : Rows{};
  static const bool strace_on = getenv("PHC_HOST_TRACE") != nullptr;
  static int strace_calls = 0;
  const bool strace = strace_on && ++strace_calls == 20;
  cudaEvent_t sev0 = nullptr, sevh[16], sevk[16], sevd[16];
  if (strace) {
    cudaEventCreate(&sev0);
    cudaEventRecord(sev0, s.streams[0]);
  }
  for (int ci = 0; ci < nchunks; ++ci) {
    const int64_t lo = bounds[ci], m = bounds[ci + 1] - bounds[ci];
    if (m <= 0) continue;
    const Layout L = layout(m, r != nullptr, s.extra);
    if (coff + L.clock_bytes > c->pack_capacity || ooff + L.out_bytes > c->pack_capacity)
      return host_fail(s, PHC_ERR_SHAPE, cudaSuccess);
    cudaStream_t st_ = s.streams[ci % kStreams];
    // pack the chunk's clock on the host (tens of KB), then ONE transfer
    unsigned char* hc = s.h_clock + coff;
    pack_clock(hc, L, a, r, s.env, lo, m);
    unsigned char* dc = s.d_clock + coff;
    unsigned char* dout = s.d_out + ooff;
    HOST_CUDA(s, cudaMemcpyAsync(s.d_state + lo * kStateFloats, a->state + lo * kStateFloats,
                                 (size_t)m * kStateFloats * sizeof(float), H2D, st_));
    HOST_CUDA(s, cudaMemcpyAsync(dc, hc, L.clock_bytes, H2D, st_));

    PhcStepArgs k{};
    float* st = s.d_state + lo * kStateFloats;
    k.body = chunk_body(st);
    k.progress_buf = (int16_t*)(dc + L.prog);
    k.motion_start_times = (const float*)(dc + L.start);
    k.motion_start_times_offset = (const float*)(dc + L.soff);
    k.global_offset = (const float*)(dc + L.goff);
    k.sampled_motion_ids = (const int64_t*)(dc + L.ids);
    k.termination_distances = c->term_dist;
    k.reset_body_mask = c->reset_mask;
    k.use_mean = c->use_mean;
    k.enable_early_termination = c->early;
    k.advance_progress = 1;
    k.time_steps = c->T;
    k.dt = c->dt;
    k.rwd = c->rwd;
    k.obs_buf = s.d_obs + lo * c->obs_dim;
    k.obs_stride = c->obs_dim;
    k.rew_buf = (float*)(dout + L.rew);
    k.reward_raw = (float*)(dout + L.raw);
    k.reward_raw_stride = s.extra.raw_cols;
    k.reset_buf = dout + L.reset;
    k.terminate_buf = dout + L.term;
    k.obs_moments = nullptr;
    k.mpjpe = s.extra.mpjpe ? (float*)(dout + L.mpjpe) : nullptr;
    HOST_CUDA(s, power_inputs(s, lo, m, st_, k));
    if (dev) dev_step_outputs(c, dev, lo, k);
    PhcResetArgs ra;
    if (r) {  // the step's own flags still leave in the packed scalars
      k.reset_buf = s.d_kreset + lo;
      k.terminate_buf = s.d_kterm + lo;
      k.reset_out = dout + L.reset;
      k.terminate_out = dout + L.term;
      ra = chunk_reset_args(c, s, r, st, dc, L, lo, k.obs_buf);
      k.auto_reset = &ra;
    }
    if (strace && ci < 16) {
      cudaEventCreate(&sevh[ci]);
      cudaEventRecord(sevh[ci], st_);
    }
    if (dev) HOST_CUDA(s, cudaStreamWaitEvent(st_, s.dev_ready, 0));
    int rc = phc_step_fused(c->lib, &k, m, st_);
    if (rc) return host_fail(s, rc, cudaSuccess);
    if (r) {
      Rows out = rows_at(rows, lo, c->obs_dim);
      out.obs = nullptr;
      out.prog = nullptr;
      out.rst = out.term = nullptr;
      HOST_CUDA(s, export_rows(c, ra, dout + L.reset, nullptr, nullptr, out, 0, m, st_));
    }
    if (strace && ci < 16) {
      cudaEventCreate(&sevk[ci]);
      cudaEventRecord(sevk[ci], st_);
    }
    // the advanced progress rides back with the scalar outputs
    HOST_CUDA(s, cudaMemcpyAsync(dout + L.oprog, dc + L.prog, (size_t)m * 2, cudaMemcpyDeviceToDevice, st_));
    if (!dev)
      HOST_CUDA(s, cudaMemcpyAsync(a->obs_buf + lo * c->obs_dim, s.d_obs + lo * c->obs_dim,
                                   (size_t)m * c->obs_dim * sizeof(float), D2H, st_));
    HOST_CUDA(s, cudaMemcpyAsync(s.h_out + ooff, dout, L.out_bytes, D2H, st_));
    if (strace && ci < 16) {
      cudaEventCreate(&sevd[ci]);
      cudaEventRecord(sevd[ci], st_);
    }
    coff += L.clock_bytes;
    ooff += L.out_bytes;
  }
  if (strace) {
    for (auto st_ : s.streams) HOST_CUDA(s, cudaStreamSynchronize(st_));
    fprintf(stderr, "[phc_host trace] staged, %d chunks\n", nchunks);
    for (int i = 0; i < nchunks && i < 16; ++i) {
      float a_ms = 0, b_ms = 0, d_ms = 0;
      cudaEventElapsedTime(&a_ms, sev0, sevh[i]);
      cudaEventElapsedTime(&b_ms, sev0, sevk[i]);
      cudaEventElapsedTime(&d_ms, sev0, sevd[i]);
      fprintf(stderr, "  chunk %d (%lld envs): H2D done %.1f us, kernel done %.1f us, D2H done %.1f us\n", i,
              (long long)(bounds[i + 1] - bounds[i]), a_ms * 1e3, b_ms * 1e3, d_ms * 1e3);
    }
  }
  return PHC_OK;
}

// The host reset: H2D(packed clock + phase + mask) -> phc_reset_envs -> export of the masked envs' rows (obs included)
// on equal chunks.  Nothing else is read or written: no sim state comes in, no whole obs chunk goes out.  With device
// outputs the reset writes the masked envs' obs and normalised rows straight into the caller's tensors and adds them
// to the moments (rows no step has counted, as HumanoidPHC.reset() does); the export then carries no obs.
static int reset_enqueue(PhcHostStep* c, Slot& s, const PhcHostStepArgs* a, const PhcHostResetArgs* r,
                         const PhcHostDeviceOut* dev, int64_t n, const int chunks) {
  const int C = chunks < 1 ? 1 : chunks;
  int64_t per = (n + C - 1) / C;
  per = (per + 7) / 8 * 8;
  const Rows rows = s.rows_staged ? s.stage : caller_rows(a, r);
  size_t coff = 0;
  int ci = 0;
  for (int64_t lo = 0; lo < n; lo += per, ++ci) {
    const int64_t m = (n - lo) < per ? (n - lo) : per;
    const Layout L = layout(m, true, s.extra);
    if (coff + L.clock_bytes > c->pack_capacity) return host_fail(s, PHC_ERR_SHAPE, cudaSuccess);
    cudaStream_t st_ = s.streams[ci % kStreams];
    unsigned char* hc = s.h_clock + coff;
    unsigned char* dc = s.d_clock + coff;
    pack_clock(hc, L, a, r, s.env, lo, m);
    HOST_CUDA(s, cudaMemcpyAsync(dc, hc, L.clock_bytes, cudaMemcpyHostToDevice, st_));
    // a default-path env keeps its rigid-body rows, and its observation is computed from them: the chunk's sim state
    // comes in (read before the export writes state_out, which may alias it)
    if (r->state_init >= PHC_STATE_INIT_DEFAULT)
      HOST_CUDA(s, cudaMemcpyAsync(s.d_state + lo * kStateFloats, a->state + lo * kStateFloats,
                                   (size_t)m * kStateFloats * sizeof(float), cudaMemcpyHostToDevice, st_));
    float* obs = dev ? dev_obs(c, dev, lo) : s.d_obs + lo * c->obs_dim;
    PhcResetArgs ra = chunk_reset_args(c, s, r, s.d_state + lo * kStateFloats, dc, L, lo, obs);
    Rows out = rows_at(rows, lo, c->obs_dim);
    if (dev) {
      ra.obs_norm = dev_obs_norm(c, dev, lo);
      ra.obs_norm_stride = c->obs_dim;
      ra.norm_mean = dev->norm_mean;
      ra.norm_var = dev->norm_var;
      ra.norm_epsilon = dev->norm_epsilon;
      ra.norm_clip = dev->norm_clip;
      ra.obs_norm_bf16 = (dev->flags & PHC_STEP_OBS_NORM_BF16) ? 1 : 0;
      ra.obs_moments_mode = dev->obs_moments ? 1 : 0;
      ra.obs_moments = dev->obs_moments;
      ra.obs_moments_buckets = dev->obs_moments_buckets;
      out.obs = nullptr;
      HOST_CUDA(s, cudaStreamWaitEvent(st_, s.dev_ready, 0));
    }
    const int rc = phc_reset_envs(c->lib, &ra, m, st_);
    if (rc) return host_fail(s, rc, cudaSuccess);
    HOST_CUDA(s, export_rows(c, ra, dc + L.mask, nullptr, dev ? nullptr : obs, out, 1, m, st_));
    coff += L.clock_bytes;
  }
  return PHC_OK;
}

// Enqueues one step (or reset) on a slot (arguments already checked) and marks it in flight.
static int slot_enqueue(PhcHostStep* c, int slot, const PhcHostStepArgs* a, const PhcHostResetArgs* r, int op,
                        int64_t n, const PhcHostStep::Cand& k, const PhcHostDeviceOut* dev = nullptr) {
  Slot& s = c->slots[slot];
  if (dev) HOST_CUDA(s, cudaEventRecord(s.dev_ready, dev->stream));
  // s.env / s.extra were set by the submit (zero for phc_host_step)
  const int rc = op == kReset   ? reset_enqueue(c, s, a, r, dev, n, k.chunks)
                 : k.path == 1 ? direct_enqueue(c, s, a, r, dev, n, k.chunks)
                               : staged_enqueue(c, s, a, r, dev, n, k.chunks);
  if (rc) return rc;
  for (int i = 0; i < kStreams; ++i) HOST_CUDA(s, cudaEventRecord(s.done[i], s.streams[i]));
  s.args = *a;
  s.rargs = r ? *r : PhcHostResetArgs{};
  s.op = op;
  s.n = n;
  s.path = k.path;
  s.busy = true;
  c->last_slot = slot;
  return PHC_OK;
}

// The reset rows of the flagged envs (the step's reset flags, or the reset's env mask), from the slot's staging into
// the caller's buffers.
static void unpack_rows(const PhcHostStep* c, const Slot& s) {
  const Rows src = s.stage, dst = caller_rows(&s.args, &s.rargs);
  const uint8_t* flag = s.op == kReset ? s.rargs.env_mask : s.args.reset_buf;
  const size_t D = (size_t)c->obs_dim;
  for (int64_t i = 0; i < s.n; ++i) {
    if (!flag[i]) continue;
    memcpy(dst.state + i * kStateFloats, src.state + i * kStateFloats, kStateFloats * sizeof(float));
    memcpy(dst.root + i * 13, src.root + i * 13, 13 * sizeof(float));
    memcpy(dst.dofp + i * 69, src.dofp + i * 69, 69 * sizeof(float));
    memcpy(dst.dofv + i * 69, src.dofv + i * 69, 69 * sizeof(float));
    memcpy(dst.goff + i * 3, src.goff + i * 3, 3 * sizeof(float));
    dst.start[i] = src.start[i];
    dst.soff[i] = src.soff[i];
    if (s.op == kReset) {
      if (dst.obs) memcpy(dst.obs + i * D, src.obs + i * D, D * sizeof(float));  // no host obs with device outputs
      dst.prog[i] = src.prog[i];
      dst.rst[i] = src.rst[i];
      dst.term[i] = src.term[i];
    }
  }
}

// Waits for a slot's step; on the staged path unpacks the scalar outputs into the caller's buffers, and the reset rows
// that went through staging.
static int slot_finish(const PhcHostStep* c, Slot& s) {
  if (!s.busy) return PHC_OK;
  s.busy = false;
  cudaError_t err = cudaSuccess;
  for (auto& ev : s.done) {
    const cudaError_t e = cudaEventSynchronize(ev);
    if (err == cudaSuccess) err = e;
  }
  if (err != cudaSuccess) return host_fail(s, PHC_ERR_CUDA, err);
  if (s.path == 2 && s.op != kReset) {
    const PhcHostStepArgs* a = &s.args;
    size_t ooff = 0;
    for (int ci = 0; ci < s.nchunks; ++ci) {
      const int64_t lo = s.bounds[ci], m = s.bounds[ci + 1] - s.bounds[ci];
      if (m <= 0) continue;
      const Layout L = layout(m, s.op != kStep, s.extra);
      const unsigned char* ho = s.h_out + ooff;
      const int W = s.extra.raw_cols;
      memcpy(a->rew_buf + lo, ho + L.rew, (size_t)m * 4);
      memcpy(a->reward_raw + lo * W, ho + L.raw, (size_t)m * 4 * W);
      if (s.extra.mpjpe) memcpy(s.env.mpjpe + lo, ho + L.mpjpe, (size_t)m * 4);
      memcpy(a->progress_buf + lo, ho + L.oprog, (size_t)m * 2);
      memcpy(a->reset_buf + lo, ho + L.reset, (size_t)m);
      memcpy(a->terminate_buf + lo, ho + L.term, (size_t)m);
      ooff += L.out_bytes;
    }
  }
  if (s.op != kStep && s.rows_staged) unpack_rows(c, s);
  return PHC_OK;
}

// The schedule of a step that is not timed by the tuner: pageable callers take the copy-engine path; pinned callers
// the settled schedule, or the first candidate while tuning has not finished.
static PhcHostStep::Cand untimed_schedule(const PhcHostStep* c, const Slot& s) {
  if (s.seen_direct != 1) return {2, c->chunks > 0 ? c->chunks : 3, 0.0, 0};
  return c->cand[c->chosen >= 0 ? c->chosen : 0];
}

static int run_sync(PhcHostStep* c, const PhcHostStepArgs* a, int64_t n, const PhcHostStep::Cand& k) {
  Slot& s = c->slots[0];
  s.env = PhcHostEnvArgs{};
  s.extra = Extra{};
  const int rc = slot_enqueue(c, 0, a, nullptr, kStep, n, k);
  return rc ? rc : slot_finish(c, s);
}

extern "C" {

void phc_host_step_destroy(PhcHostStep* c) {
  if (!c) return;
  for (auto& s : c->slots) {
    (void)slot_finish(c, s);  // a pending DMA or posting kernel must not land in freed memory
    slot_free(s);
  }
  cudaFree(c->term_dist);
  delete c;
}

int phc_host_step_create(const PhcLib* lib, int64_t max_envs, int32_t time_steps, int32_t num_chunks,
                         const float* termination_distances_host, uint32_t reset_body_mask, int32_t use_mean,
                         int32_t enable_early_termination, float dt, const PhcRewardSpec* rwd, PhcHostStep** out) {
  if (!lib || !termination_distances_host || !rwd || !out) return PHC_ERR_NULL;
  if (max_envs <= 0 || time_steps < 1 || time_steps > PHC_MAX_TIME_STEPS || num_chunks < 0 || num_chunks > kMaxChunks)
    return PHC_ERR_SHAPE;
  PhcHostStep* c = new (std::nothrow) PhcHostStep;
  if (!c) return PHC_ERR_ALLOC;
  c->lib = lib;
  c->max_envs = max_envs;
  c->T = time_steps;
  c->chunks = num_chunks;
  c->obs_dim = PHC_SELF_OBS_DIM + (int64_t)PHC_TASK_OBS_DIM * time_steps;
  c->reset_mask = reset_body_mask;
  c->use_mean = use_mean;
  c->early = enable_early_termination;
  c->dt = dt;
  c->rwd = *rwd;
  (void)cudaGetDevice(&c->device);
  if (const char* m = getenv("PHC_HOST_PATH")) c->mode = !strcmp(m, "direct") ? 1 : !strcmp(m, "staged") ? 2 : 0;
  if (getenv("PHC_HOST_STAGED")) c->mode = 2;
  const size_t n = (size_t)max_envs;
  // every chunk's packed region is padded so each sub-array starts 16-B aligned (35 B per env with a reset's clock)
  c->pack_capacity = n * 40 + (size_t)(num_chunks > 8 ? num_chunks : 8) * 8 * 64 + 4096;
  {  // candidates: direct with 2 / 3 / 4 / 6 equal chunks, staged with 3 / 4 doubling chunks
    static const int direct_chunks[] = {3, 4, 2, 6}, staged_chunks[] = {3, 4};
    auto add = [&](int path, int chunks) {
      if (c->mode && c->mode != path) return;
      if (num_chunks > 0 && chunks != num_chunks) return;
      c->cand[c->ncand++] = {path, chunks, 0.0, 0};
    };
    if (num_chunks > 0) {
      add(1, num_chunks);
      add(2, num_chunks);
    } else {
      for (int ch : direct_chunks) add(1, ch);
      for (int ch : staged_chunks) add(2, ch);
    }
    if (c->ncand == 1) c->chosen = 0;
  }
  // slot 0 (the synchronous call's) is allocated here, slot 1 at its first submit
  cudaError_t e = cudaMalloc((void**)&c->term_dist, PHC_NUM_BODIES * sizeof(float));
  if (e == cudaSuccess)
    e = cudaMemcpy(c->term_dist, termination_distances_host, PHC_NUM_BODIES * sizeof(float), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = slot_alloc(c, c->slots[0]);
  if (e != cudaSuccess) {
    phc_host_step_destroy(c);
    return e == cudaErrorMemoryAllocation ? PHC_ERR_ALLOC : PHC_ERR_CUDA;
  }
  *out = c;
  return PHC_OK;
}

int64_t phc_host_step_h2d_bytes(const PhcHostStep* c, int64_t n) {
  (void)c;
  return n * (int64_t)(kStateFloats * sizeof(float) + kClockBytes);
}
int64_t phc_host_step_d2h_bytes(const PhcHostStep* c, int64_t n) {
  return n * (int64_t)(c->obs_dim * sizeof(float) + kOutBytes);
}

int phc_host_step(PhcHostStep* c, const PhcHostStepArgs* a, int64_t n) {
  if (!c || !a) return PHC_ERR_NULL;
  if (c->slots[0].busy) return PHC_ERR_BUSY;
  if (n == 0) return PHC_OK;
  int rc = check_args(c, c->slots[0], a, n);
  if (rc) return rc;

  // ---- which schedule ------------------------------------------------------------------------
  // Only calls made while no slot is in flight are timed: a step of the other slot would share the link.
  if (c->slots[0].seen_direct != 1 || c->chosen >= 0 || c->slots[1].busy)
    return run_sync(c, a, n, untimed_schedule(c, c->slots[0]));
  // Tuning: calls 0-1 warm up, then the candidates take turns (kTuneReps timed calls each) and the fastest mean
  // stays.  What decides is the machine, under whatever load the other GPUs of the box put on the host at that moment:
  // one GPU posts its obs rows into host memory faster than a copy engine drains a staging buffer, eight GPUs posting
  // into one root complex may not (profiles/r2_e2e_floor.md); and on some hosts the inbound copy of the next chunk
  // crawls while a kernel is posting (its read requests queue behind the posted writes), which moves the best chunk
  // count (profiles/r2_host_timeline.md).
  const int k = c->calls++;
  const int which = k < kTuneWarm ? k % c->ncand : (k - kTuneWarm) % c->ncand;
  const auto t0 = std::chrono::steady_clock::now();
  rc = run_sync(c, a, n, c->cand[which]);
  const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  if (rc == PHC_OK && k >= kTuneWarm) {
    // the first timed call of a candidate warms its own launch configuration: not counted.  A candidate's figure is
    // its FASTEST call (what the schedule can do; a mean over three calls carries the host's jitter), and the first
    // candidate — three chunks, direct: the best schedule on most hosts — is only given up for one that is 2 % faster.
    if (k - kTuneWarm >= c->ncand) {
      c->cand[which].t = c->cand[which].n == 0 || dt < c->cand[which].t ? dt : c->cand[which].t;
      c->cand[which].n += 1;
    }
    bool done = true;
    for (int i = 0; i < c->ncand; ++i) done = done && c->cand[i].n >= kTuneReps;
    if (done) {
      int best = 0;
      double best_t = c->cand[0].t * 0.98;
      for (int i = 1; i < c->ncand; ++i)
        if (c->cand[i].t < best_t) best = i, best_t = c->cand[i].t;
      c->chosen = best;
      if (getenv("PHC_HOST_TRACE"))
        for (int i = 0; i < c->ncand; ++i)
          fprintf(stderr, "[phc_host tune] %s, %d chunks: %.1f us%s\n", c->cand[i].path == 1 ? "direct" : "staged",
                  c->cand[i].chunks, c->cand[i].t * 1e6, i == best ? "  <- kept" : "");
    }
  }
  return rc;
}

}  // extern "C"

// The submits: every check before anything is enqueued, then the slot's buffers, then the enqueue.  dev_out: one of
// the device-output submits (dev must then name the device tensors).
// env_entry: one of the _env submits, whose env options (env, NULL for none) may be set; a host reset takes only their
// default_mask.  The other submits have no options and refuse StateInit.Default / Hybrid, as they always did.
static int submit(PhcHostStep* c, int32_t slot, const PhcHostStepArgs* a, const PhcHostResetArgs* r, int op, int64_t n,
                  bool dev_out = false, const PhcHostDeviceOut* dev = nullptr, bool env_entry = false,
                  const PhcHostEnvArgs* env = nullptr) {
  if (!c || !a || (op != kStep && !r) || (dev_out && (!dev || !dev->obs))) return PHC_ERR_NULL;
  if (slot < 0 || slot >= PHC_HOST_SLOTS) return PHC_ERR_SHAPE;
  Slot& s = c->slots[slot];
  if (s.busy) return PHC_ERR_BUSY;
  if (n == 0) return PHC_OK;
  PhcHostEnvArgs ev{};
  if (env && op == kReset) ev.default_mask = env->default_mask;
  else if (env) ev = *env;
  int rc = check_args(c, s, a, n, dev_out, ev.mpjpe);
  if (rc) return rc;
  if ((rc = check_env(s, &ev))) return rc;
  if (op != kStep && (rc = check_reset(c, s, r, op, env_entry ? &ev : nullptr, n))) return rc;
  if (dev_out && (rc = check_dev(c, dev))) return rc;
  s.env = ev;
  s.extra.raw_cols = ev.dof_force ? 5 : 4;
  s.extra.mpjpe = ev.mpjpe != nullptr;
  s.extra.dmask = op != kStep && r->state_init == PHC_STATE_INIT_HYBRID;
  cudaError_t e = cudaSuccess;
  if (!s.ready) {
    e = slot_alloc(c, s);
    if (e != cudaSuccess) slot_free(s);
  }
  if (op != kStep && e == cudaSuccess) {
    // the host reset writes the step buffers' rows too (obs, progress, flags): straight only when they are pinned as well
    s.rows_staged = !s.rseen_direct || (op == kReset && s.seen_direct != 1);
    e = reset_alloc(c, s, s.rows_staged);
  }
  if (e == cudaSuccess) e = env_alloc(c, s);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    return e == cudaErrorMemoryAllocation ? PHC_ERR_ALLOC : phc::record_cuda_error((int)e);
  }
  return slot_enqueue(c, slot, a, r, op, n, untimed_schedule(c, s), dev_out ? dev : nullptr);
}

extern "C" {

int phc_host_step_submit(PhcHostStep* c, int32_t slot, const PhcHostStepArgs* a, int64_t n) {
  return submit(c, slot, a, nullptr, kStep, n);
}

int phc_host_step_submit_reset(PhcHostStep* c, int32_t slot, const PhcHostStepArgs* a, const PhcHostResetArgs* r,
                               int64_t n) {
  return submit(c, slot, a, r, kStepReset, n);
}

int phc_host_reset_submit(PhcHostStep* c, int32_t slot, const PhcHostStepArgs* a, const PhcHostResetArgs* r,
                          int64_t n) {
  return submit(c, slot, a, r, kReset, n);
}

int phc_host_step_submit_device(PhcHostStep* c, int32_t slot, const PhcHostStepArgs* a, const PhcHostResetArgs* r,
                                const PhcHostDeviceOut* dev, int64_t n) {
  return submit(c, slot, a, r, r ? kStepReset : kStep, n, true, dev);
}

int phc_host_reset_submit_device(PhcHostStep* c, int32_t slot, const PhcHostStepArgs* a, const PhcHostResetArgs* r,
                                 const PhcHostDeviceOut* dev, int64_t n) {
  return submit(c, slot, a, r, kReset, n, true, dev);
}

int phc_host_step_submit_env(PhcHostStep* c, int32_t slot, const PhcHostStepArgs* a, const PhcHostResetArgs* r,
                             const PhcHostDeviceOut* dev, const PhcHostEnvArgs* env, int64_t n) {
  return submit(c, slot, a, r, r ? kStepReset : kStep, n, dev != nullptr, dev, true, env);
}

int phc_host_reset_submit_env(PhcHostStep* c, int32_t slot, const PhcHostStepArgs* a, const PhcHostResetArgs* r,
                              const PhcHostDeviceOut* dev, const PhcHostEnvArgs* env, int64_t n) {
  return submit(c, slot, a, r, kReset, n, dev != nullptr, dev, true, env);
}

int phc_host_step_set_initial_state(PhcHostStep* c, int32_t slot, const float* root_states, const float* dof_pos,
                                    const float* dof_vel, int64_t n) {
  if (!c || !root_states || !dof_pos || !dof_vel) return PHC_ERR_NULL;
  if (slot < 0 || slot >= PHC_HOST_SLOTS || n < 0 || n > c->max_envs) return PHC_ERR_SHAPE;
  Slot& s = c->slots[slot];
  if (s.busy) return PHC_ERR_BUSY;
  const float* src[3] = {root_states, dof_pos, dof_vel};
  for (const float* p : src) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) (void)cudaGetLastError();
    else if (at.type == cudaMemoryTypeDevice) return PHC_ERR_UNSUPPORTED;
  }
  const size_t N = (size_t)c->max_envs;
  cudaError_t e = cudaSuccess;
  if (!s.d_init) e = cudaMalloc((void**)&s.d_init, N * (13 + 2 * kDof) * sizeof(float));
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    return e == cudaErrorMemoryAllocation ? PHC_ERR_ALLOC : phc::record_cuda_error((int)e);
  }
  s.init_rows = -1;  // not usable until all three copies have landed
  float* dst[3] = {s.d_init, s.d_init + N * 13, s.d_init + N * (13 + kDof)};
  const size_t row[3] = {13, kDof, kDof};
  for (int i = 0; i < 3 && e == cudaSuccess; ++i)
    e = cudaMemcpy(dst[i], src[i], (size_t)n * row[i] * sizeof(float), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    return phc::record_cuda_error((int)e);
  }
  s.init_rows = n;
  return PHC_OK;
}

int phc_host_step_wait(PhcHostStep* c, int32_t slot) {
  if (!c) return PHC_ERR_NULL;
  if (slot < 0 || slot >= PHC_HOST_SLOTS) return PHC_ERR_SHAPE;
  return slot_finish(c, c->slots[slot]);
}

int phc_host_step_path(const PhcHostStep* c) {
  if (!c) return 0;
  if (c->slots[c->last_slot].seen_direct == 0) return 2;
  return c->chosen >= 0 ? c->cand[c->chosen].path : 0;
}

int phc_host_step_chunks(const PhcHostStep* c) {
  if (!c) return 0;
  if (c->slots[c->last_slot].seen_direct == 0) return c->chunks > 0 ? c->chunks : 3;
  return c->chosen >= 0 ? c->cand[c->chosen].chunks : 0;
}

int phc_host_step_tuning_calls(const PhcHostStep* c) {
  if (!c || c->ncand <= 1) return 0;
  return kTuneWarm + c->ncand * (kTuneReps + 1);
}

}  // extern "C"
