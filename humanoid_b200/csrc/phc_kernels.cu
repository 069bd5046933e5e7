// libphc_b200.so — hand-written sm_100a kernels of the PHC step path behind the C ABI in
// include/phc_b200.h.  No tensor cores (nothing here is a dense contraction): the path is
// gather + stream + per-body quaternion math, bounded by HBM bandwidth and fp32 issue.
//
// Thread mapping everywhere: one thread per (env, body); 24 consecutive threads own one
// env, so an 8-env block is 192 threads = 6 full warps with no idle lanes.  Per-env
// reductions (reward means, termination any/mean) go through shared memory in ATen's CPU
// summation order, so the result does not depend on how envs fall on warps.
//
// Compiled with -fmad=false (see phc_math.cuh).
#include <algorithm>
#include <atomic>
#include <cfloat>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "../../include/phc_b200.h"
#include "phc_math.cuh"

namespace phc {

constexpr int J24 = PHC_NUM_BODIES;
constexpr int SELF_DIM = PHC_SELF_OBS_DIM;
constexpr int TASK_DIM = PHC_TASK_OBS_DIM;
constexpr int TASK_DIM_V7 = 9 * J24;  // 216: [d_pos | d_vel | l_pos] per future step (PHC_OBS_TASK_V7)

static thread_local int g_last_cuda_error = 0;

static inline int cuda_fail(cudaError_t e) {
  g_last_cuda_error = (int)e;
  return PHC_ERR_CUDA;
}
#define PHC_CUDA(call)                              \
  do {                                              \
    cudaError_t e__ = (call);                       \
    if (e__ != cudaSuccess) return cuda_fail(e__);  \
  } while (0)

int record_cuda_error(int cuda_error) { return cuda_fail((cudaError_t)cuda_error); }  // for the other TUs

static inline int launch_status() {
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? PHC_OK : cuda_fail(e);
}

struct LibDev {
  const float *gts, *grs, *lrs, *gvs, *gavs, *dvs, *aa;
  const float *len, *mdt, *bodies, *limb;
  const int64_t *nf, *starts;
  int64_t F, M;
  const float* packed;  // [F][312] = per frame [gts 72 | grs 96 | gvs 72 | gavs 72], owned by PhcLib
};

// ---------------------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ Vec3 ld3(const float* p) { return {p[0], p[1], p[2]}; }
__device__ __forceinline__ Quat ld4(const float* p) { return {p[0], p[1], p[2], p[3]}; }
__device__ __forceinline__ Quat ld4v(const float* p) {  // 16-byte aligned
  float4 v = *reinterpret_cast<const float4*>(p);
  return {v.x, v.y, v.z, v.w};
}
__device__ __forceinline__ void st3(float* p, Vec3 v) {
  p[0] = v.x;
  p[1] = v.y;
  p[2] = v.z;
}
__device__ __forceinline__ void st4(float* p, Quat q) {
  p[0] = q.x;
  p[1] = q.y;
  p[2] = q.z;
  p[3] = q.w;
}
__device__ __forceinline__ void st6_shared(float* p, const float* v) {  // p is 8-byte aligned
  reinterpret_cast<float2*>(p)[0] = make_float2(v[0], v[1]);
  reinterpret_cast<float2*>(p)[1] = make_float2(v[2], v[3]);
  reinterpret_cast<float2*>(p)[2] = make_float2(v[4], v[5]);
}
__device__ __forceinline__ const float* view_at(const PhcView& v, int64_t env, int body) {
  return v.ptr + env * v.stride_env + (int64_t)body * v.stride_body;
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

// ---- TMA bulk copies (cp.async.bulk, SASS UBLKCP) completing on an mbarrier -----------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.shared::cta.b64 st, [%0];\n}\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "PHC_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra PHC_DONE;\n"
      "bra PHC_WAIT;\n"
      "PHC_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// global -> shared, 16-B aligned, size multiple of 16
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                         unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// shared -> global
__device__ __forceinline__ void bulk_s2g(void* gmem_dst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(gmem_dst),
               "r"(smem_u32(smem_src)), "r"(bytes)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

// shared -> global with an fp64 add at the destination (TMA bulk reduction, SASS UBLKRED): the L2 does the adds
__device__ __forceinline__ void bulk_reduce_add_f64(double* gmem_dst, const double* smem_src, uint32_t bytes) {
  asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f64 [%0], [%1], %2;\n" ::"l"(gmem_dst),
               "r"(smem_u32(smem_src)), "r"(bytes)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read_all_but_one() { asm volatile("cp.async.bulk.wait_group.read 1;\n" ::: "memory"); }

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
#define PHC_STAMP(slot)                                                                      \
  do {                                                                                       \
    if (p.trace && (threadIdx.x & 31) == 0)                                                  \
      p.trace[((size_t)blockIdx.x * 3 + (threadIdx.x >> 5)) * 8 + (slot)] = globaltimer_ns(); \
  } while (0)

// per-(query) reference body state
struct RefBody {
  Vec3 pos;
  Quat rot;
  Vec3 vel;
  Vec3 ang;
};

// ---------------------------------------------------------------------------------------
// K0: _calc_frame_blend (motion_lib.py:655-665)
// ---------------------------------------------------------------------------------------
__global__ void frame_blend_kernel(const float* __restrict__ time, const float* __restrict__ len,
                                   const int64_t* __restrict__ nf, const float* __restrict__ dt, int64_t n,
                                   int64_t* __restrict__ i0, int64_t* __restrict__ i1, float* __restrict__ bl) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int64_t a, b;
  float w;
  calc_frame_blend(time[i], len[i], nf[i], dt[i], a, b, w);
  i0[i] = a;
  i1[i] = b;
  bl[i] = w;
}

// ---------------------------------------------------------------------------------------
// Frame packing (one-off, at phc_lib_create): the step kernels read, per frame, the body
// positions, rotations and both velocities — four rows that the reference keeps in four tensors
// (motion_lib.py:407-414).  Interleaving them into one 1248-B row per frame turns four
// gathers into one contiguous 39-sector read and one TMA bulk copy.
// ---------------------------------------------------------------------------------------
__global__ void pack_frames_kernel(LibDev L, float* __restrict__ packed) {
  const int64_t total4 = L.F * 78;  // float4 units
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t f = i / 78;
    const int k = (int)(i - f * 78);
    const float* src;
    if (k < 18)
      src = L.gts + f * 72 + k * 4;
    else if (k < 42)
      src = L.grs + f * 96 + (k - 18) * 4;
    else if (k < 60)
      src = L.gvs + f * 72 + (k - 42) * 4;
    else
      src = L.gavs + f * 72 + (k - 60) * 4;
    reinterpret_cast<float4*>(packed)[i] = *reinterpret_cast<const float4*>(src);
  }
}

// ---------------------------------------------------------------------------------------
// K1: get_motion_state (motion_lib.py:549-626), one thread per (query, body)
// ---------------------------------------------------------------------------------------
constexpr int K1_QPB = 8;  // queries per block

__global__ void __launch_bounds__(K1_QPB* J24)
    motion_state_kernel(LibDev L, const int64_t* __restrict__ ids, const float* __restrict__ times,
                        const float* __restrict__ offset, int64_t n, PhcMotionOut o) {
  const int e = threadIdx.x / J24, b = threadIdx.x % J24;
  const int64_t q = (int64_t)blockIdx.x * K1_QPB + e;
  if (q >= n) return;
  const int64_t id = ids[q];
  int64_t i0, i1;
  float bl;
  calc_frame_blend(times[q], L.len[id], L.nf[id], L.mdt[id], i0, i1, bl);
  const int64_t st = L.starts[id];
  const int64_t f0 = i0 + st, f1 = i1 + st;
  const float om = 1.0f - bl;

  if (b == 0) {
    if (o.frame_idx0) o.frame_idx0[q] = i0;
    if (o.frame_idx1) o.frame_idx1[q] = i1;
    if (o.blend) o.blend[q] = bl;
  }
  // positions (+ offset), velocities
  if (o.rg_pos || (o.root_pos && b == 0)) {
    Vec3 p = lerp3(om, bl, ld3(L.gts + (f0 * J24 + b) * 3), ld3(L.gts + (f1 * J24 + b) * 3));
    if (offset) p = p + ld3(offset + q * 3);
    if (o.rg_pos) st3(o.rg_pos + (q * J24 + b) * 3, p);
    if (o.root_pos && b == 0) st3(o.root_pos + q * 3, p);
  }
  if (o.body_vel || (o.root_vel && b == 0)) {
    Vec3 v = lerp3(om, bl, ld3(L.gvs + (f0 * J24 + b) * 3), ld3(L.gvs + (f1 * J24 + b) * 3));
    if (o.body_vel) st3(o.body_vel + (q * J24 + b) * 3, v);
    if (o.root_vel && b == 0) st3(o.root_vel + q * 3, v);
  }
  if (o.body_ang_vel || (o.root_ang_vel && b == 0)) {
    Vec3 v = lerp3(om, bl, ld3(L.gavs + (f0 * J24 + b) * 3), ld3(L.gavs + (f1 * J24 + b) * 3));
    if (o.body_ang_vel) st3(o.body_ang_vel + (q * J24 + b) * 3, v);
    if (o.root_ang_vel && b == 0) st3(o.root_ang_vel + q * 3, v);
  }
  if (o.rb_rot || (o.root_rot && b == 0)) {
    Quat r = quat_slerp(ld4v(L.grs + (f0 * J24 + b) * 4), ld4v(L.grs + (f1 * J24 + b) * 4), bl);
    if (o.rb_rot) st4(o.rb_rot + (q * J24 + b) * 4, r);
    if (o.root_rot && b == 0) st4(o.root_rot + q * 4, r);
  }
  if (o.dof_pos && b >= 1) {  // _local_rotation_to_dof_smpl, motion_lib.py:670-673
    Quat r = quat_slerp(ld4v(L.lrs + (f0 * J24 + b) * 4), ld4v(L.lrs + (f1 * J24 + b) * 4), bl);
    st3(o.dof_pos + q * 69 + (b - 1) * 3, quat_exp_map(r));
  }
  if (o.dof_vel && b < 23) {
    Vec3 v = lerp3(om, bl, ld3(L.dvs + (f0 * 23 + b) * 3), ld3(L.dvs + (f1 * 23 + b) * 3));
    st3(o.dof_vel + q * 69 + b * 3, v);
  }
  if (o.motion_aa) st3(o.motion_aa + q * 72 + b * 3, ld3(L.aa + f0 * 72 + b * 3));  // frame f0, un-blended
  if (o.motion_bodies && b < 17) o.motion_bodies[q * 17 + b] = L.bodies[id * 17 + b];
  if (o.motion_limb_weights && b < 10) o.motion_limb_weights[q * 10 + b] = L.limb[id * 10 + b];
}

// ---------------------------------------------------------------------------------------
// K2: compute_humanoid_observations_smpl_max (envs/common.py:23-103), thread per (env, body)
// ---------------------------------------------------------------------------------------
__global__ void self_obs_kernel(PhcBodyState s, int64_t n, uint32_t flags, float* __restrict__ out,
                                int64_t out_stride, int epb) {
  const int J = s.num_bodies;
  const int e = threadIdx.x / J, b = threadIdx.x % J;
  const int64_t env = (int64_t)blockIdx.x * epb + e;
  if (e >= epb || env >= n) return;
  const Vec3 root_pos = ld3(view_at(s.pos, env, 0));
  Quat root_rot = ld4(view_at(s.rot, env, 0));
  if (!(flags & PHC_OBS_UPRIGHT)) root_rot = remove_base_rot(root_rot);
  const Heading hi = heading_quat_inv(root_rot);
  const HeadingRot hr = heading_rot(hi);
  float* row = out + env * out_stride;
  int col = 0;
  if (flags & PHC_OBS_ROOT_HEIGHT) {
    if (b == 0) row[0] = root_pos.z;
    col = 1;
  }
  if (b >= 1) st3(row + col + (b - 1) * 3, heading_rotate(hr, ld3(view_at(s.pos, env, b)) - root_pos));
  col += (J - 1) * 3;
  {
    float t6[6];
    if (b == 0 && !(flags & PHC_OBS_LOCAL_ROOT)) {
      // "if not local_root_obs: root_rot_obs = quat_to_tan_norm(root_rot)" (common.py:76-78);
      // root_rot there is the (possibly base-rot-removed) root rotation
      quat_tan_norm(root_rot, t6);
    } else {
      quat_tan_norm(heading_mul_left(hi, ld4(view_at(s.rot, env, b))), t6);
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) row[col + b * 6 + k] = t6[k];
  }
  col += J * 6;
  st3(row + col + b * 3, heading_rotate(hr, ld3(view_at(s.vel, env, b))));
  col += J * 3;
  st3(row + col + b * 3, heading_rotate(hr, ld3(view_at(s.ang_vel, env, b))));
}

// ---------------------------------------------------------------------------------------
// K3: compute_imitation_observations_v6 (envs/common.py:106-176), thread per (env, t, body)
// mode 7 = column subset [d_pos | d_vel | l_pos]
// ---------------------------------------------------------------------------------------
struct TaskObs {  // one body's 24 floats of a v6 block
  Vec3 d_pos;
  float d_rot[6];
  Vec3 d_vel, d_ang, l_pos;
  float l_rot[6];
};

__device__ __forceinline__ void task_obs_body(Heading hi, const HeadingRot& hr, Vec3 root_pos, Vec3 pos, Quat rot, Vec3 vel,
                                              Vec3 ang, const RefBody& r, bool full, TaskObs& o) {
  o.d_pos = heading_rotate(hr, r.pos - pos);
  o.d_vel = heading_rotate(hr, r.vel - vel);
  o.l_pos = heading_rotate(hr, r.pos - root_pos);
  if (full) {
    o.d_ang = heading_rotate(hr, r.ang - ang);
    Quat dg = quat_mul(r.rot, quat_conj(rot));
    Quat dl = heading_mul_right(heading_mul_left(hi, dg), heading_conj(hi));
    quat_tan_norm(dl, o.d_rot);
    quat_tan_norm(heading_mul_left(hi, r.rot), o.l_rot);
  }
}

__global__ void imitation_obs_kernel(const float* __restrict__ root_pos, int64_t rp_stride,
                                     const float* __restrict__ root_rot, int64_t rr_stride, PhcBodyState s,
                                     PhcBodyState ref, int64_t n, int T, int upright, int mode,
                                     float* __restrict__ out, int64_t out_stride) {
  const int J = s.num_bodies;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = n * T * J;
  if (gid >= total) return;
  const int b = (int)(gid % J);
  const int64_t et = gid / J;  // env * T + t
  const int t = (int)(et % T);
  const int64_t env = et / T;
  Quat rr = ld4(root_rot + env * rr_stride);
  if (!upright) rr = remove_base_rot(rr);
  const Heading hi = heading_quat_inv(rr);
  const HeadingRot hr = heading_rot(hi);
  RefBody r;
  r.pos = ld3(view_at(ref.pos, et, b));
  r.rot = ld4(view_at(ref.rot, et, b));
  r.vel = ld3(view_at(ref.vel, et, b));
  r.ang = ld3(view_at(ref.ang_vel, et, b));
  TaskObs o;
  task_obs_body(hi, hr, ld3(root_pos + env * rp_stride), ld3(view_at(s.pos, env, b)), ld4(view_at(s.rot, env, b)),
                ld3(view_at(s.vel, env, b)), ld3(view_at(s.ang_vel, env, b)), r, mode == 6, o);
  if (mode == 6) {
    float* row = out + env * out_stride + (int64_t)t * (24 * J);
    st3(row + b * 3, o.d_pos);
#pragma unroll
    for (int k = 0; k < 6; ++k) row[3 * J + b * 6 + k] = o.d_rot[k];
    st3(row + 9 * J + b * 3, o.d_vel);
    st3(row + 12 * J + b * 3, o.d_ang);
    st3(row + 15 * J + b * 3, o.l_pos);
#pragma unroll
    for (int k = 0; k < 6; ++k) row[18 * J + b * 6 + k] = o.l_rot[k];
  } else {
    float* row = out + env * out_stride + (int64_t)t * (9 * J);
    st3(row + b * 3, o.d_pos);
    st3(row + 3 * J + b * 3, o.d_vel);
    st3(row + 6 * J + b * 3, o.l_pos);
  }
}

// ---------------------------------------------------------------------------------------
// K8: build_amp_observations_smpl (envs/common.py:192-267), 32 threads per env: thread j < nj owns
// joint j of the dof subset (exp map -> quaternion -> tan/norm, and its dof velocities), thread 0
// also the root terms, threads < K the key-body positions.
// ---------------------------------------------------------------------------------------
// One AMP observation row by one warp.  `Src` supplies the inputs: the root state (every lane),
// dof3(d, pos, vel) = position / velocity of three dof indices, key_pos(i) = position of key body i.
template <class Src>
__device__ __forceinline__ void amp_obs_row(const Src& src, int K, const int64_t* __restrict__ dof_subset, int num_sel,
                                            uint32_t flags, int lane, float* __restrict__ row,
                                            float* __restrict__ row2 = nullptr) {  // row2: NULL, or a second copy of the row
  const auto put = [&](int i, float v) {
    row[i] = v;
    if (row2) row2[i] = v;
  };
  const auto put3 = [&](int i, Vec3 v) { put(i, v.x), put(i + 1, v.y), put(i + 2, v.z); };
  const int nj = num_sel / 3;
  const Vec3 root_pos = src.root_pos();
  Quat root_rot = src.root_rot();
  if (!(flags & PHC_OBS_UPRIGHT)) root_rot = remove_base_rot(root_rot);
  const Heading hi = heading_quat_inv(root_rot);
  const HeadingRot hr = heading_rot(hi);
  int col = 0;
  if (flags & PHC_OBS_ROOT_HEIGHT) {
    if (lane == 0) put(0, root_pos.z);
    col = 1;
  }
  if (lane == 0) {
    float t6[6];
    quat_tan_norm((flags & PHC_OBS_LOCAL_ROOT) ? heading_mul_left(hi, root_rot) : root_rot, t6);
#pragma unroll
    for (int k = 0; k < 6; ++k) put(col + k, t6[k]);
    put3(col + 6, heading_rotate(hr, src.root_vel()));
    put3(col + 9, heading_rotate(hr, src.root_ang_vel()));
  }
  col += 12;
  for (int j = lane; j < nj; j += 32) {  // dof_to_obs_smpl (:179-189) + the selected dof velocities
    int64_t d[3];
    float e3[3], v3[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) d[k] = dof_subset ? dof_subset[3 * j + k] : 3 * j + k;
    src.dof3(d, e3, v3);
    float t6[6];
    quat_tan_norm(exp_map_to_quat(Vec3{e3[0], e3[1], e3[2]}), t6);
#pragma unroll
    for (int k = 0; k < 6; ++k) put(col + 6 * j + k, t6[k]);
#pragma unroll
    for (int k = 0; k < 3; ++k) put(col + 6 * nj + 3 * j + k, v3[k]);
  }
  col += 9 * nj;
  if (lane < K) put3(col + 3 * lane, heading_rotate(hr, src.key_pos(lane) - root_pos));
}

struct AmpSrcArrays {  // build_amp_observations_smpl's argument list, row `env`
  const PhcAmpArgs& a;
  int64_t env;
  __device__ Vec3 root_pos() const { return ld3(a.root_pos + env * a.root_pos_stride); }
  __device__ Quat root_rot() const { return ld4(a.root_rot + env * a.root_rot_stride); }
  __device__ Vec3 root_vel() const { return ld3(a.root_vel + env * a.root_vel_stride); }
  __device__ Vec3 root_ang_vel() const { return ld3(a.root_ang_vel + env * a.root_ang_vel_stride); }
  __device__ void dof3(const int64_t* d, float* e3, float* v3) const {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      e3[k] = a.dof_pos[env * a.dof_pos_stride + d[k] * a.dof_pos_elem_stride];
      v3[k] = a.dof_vel[env * a.dof_vel_stride + d[k] * a.dof_vel_elem_stride];
    }
  }
  __device__ Vec3 key_pos(int i) const { return ld3(view_at(a.key_body_pos, env, i)); }
};

__global__ void amp_obs_kernel(PhcAmpArgs a, int64_t n, float* __restrict__ out, int64_t out_stride) {
  const int lane = threadIdx.x & 31;
  const int64_t env = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (env >= n) return;
  amp_obs_row(AmpSrcArrays{a, env}, a.num_key_bodies, a.dof_subset, a.num_sel, a.flags, lane, out + env * out_stride);
}

// ---------------------------------------------------------------------------------------
// K11 / K12: the env's AMP observation buffers (envs/humanoid_phc.py:791-843, 1125-1176, 1341-1350).
//   amp_step_kernel      one warp per env: history roll (slot k+1 <- slot k) + slot 0 from the sim state
//   amp_init_ref_kernel  a block per 8 envs, its warps over the (selected env, slot) pairs: slot 0 from the sim
//                        state (optional), slot k >= 1 from the motion library at motion_time - k*dt, each row
//                        written to the demo buffer as well
// ---------------------------------------------------------------------------------------
constexpr int AMP_MAX_STEPS = 16;
struct AmpEnvParams {
  PhcBodyState body;
  const float* dof_pos;
  const float* dof_vel;
  int64_t dof_stride, dof_estride;
  int key_ids[8];
  int K;
  const int64_t* dof_subset;
  int num_sel;
  uint32_t flags;
  float* buf;
  float* demo;
  int S, P;
  const uint8_t* mask;
  int roll;
  int64_t n;
};

struct AmpSrcSim {  // _compute_amp_observations (:1125-1176): root = body 0 of the sim state
  const AmpEnvParams& p;
  int64_t env;
  __device__ Vec3 root_pos() const { return ld3(view_at(p.body.pos, env, 0)); }
  __device__ Quat root_rot() const { return ld4(view_at(p.body.rot, env, 0)); }
  __device__ Vec3 root_vel() const { return ld3(view_at(p.body.vel, env, 0)); }
  __device__ Vec3 root_ang_vel() const { return ld3(view_at(p.body.ang_vel, env, 0)); }
  __device__ void dof3(const int64_t* d, float* e3, float* v3) const {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      e3[k] = p.dof_pos[env * p.dof_stride + d[k] * p.dof_estride];
      v3[k] = p.dof_vel[env * p.dof_stride + d[k] * p.dof_estride];
    }
  }
  __device__ Vec3 key_pos(int i) const { return ld3(view_at(p.body.pos, env, p.key_ids[i])); }
};

struct AmpSrcLib {  // _get_amp_obs (:821-838): get_motion_state at (id, t) without a global offset
  const LibDev& L;
  const int* key_ids;
  int64_t f0, f1;
  float bl;
  __device__ Vec3 lerp_body(const float* tab, int per_frame, int b) const {
    return lerp3(1.0f - bl, bl, ld3(tab + (f0 * per_frame + b) * 3), ld3(tab + (f1 * per_frame + b) * 3));
  }
  __device__ Vec3 root_pos() const { return lerp_body(L.gts, J24, 0); }
  __device__ Quat root_rot() const { return quat_slerp(ld4v(L.grs + f0 * J24 * 4), ld4v(L.grs + f1 * J24 * 4), bl); }
  __device__ Vec3 root_vel() const { return lerp_body(L.gvs, J24, 0); }
  __device__ Vec3 root_ang_vel() const { return lerp_body(L.gavs, J24, 0); }
  __device__ void dof3(const int64_t* d, float* e3, float* v3) const {
    int last = -1;
    Vec3 em{}, dv{};
#pragma unroll
    for (int k = 0; k < 3; ++k) {  // dof 3j+c belongs to body j+1 (motion_lib.py:670-673), dof velocity row j
      const int j = (int)(d[k] / 3), c = (int)(d[k] % 3);
      if (j != last) {
        em = quat_exp_map(quat_slerp(ld4v(L.lrs + (f0 * J24 + j + 1) * 4), ld4v(L.lrs + (f1 * J24 + j + 1) * 4), bl));
        dv = lerp_body(L.dvs, 23, j);
        last = j;
      }
      e3[k] = c == 0 ? em.x : c == 1 ? em.y : em.z;
      v3[k] = c == 0 ? dv.x : c == 1 ? dv.y : dv.z;
    }
  }
  __device__ Vec3 key_pos(int i) const { return lerp_body(L.gts, J24, key_ids[i]); }
};

__global__ void amp_step_kernel(AmpEnvParams p) {
  const int lane = threadIdx.x & 31;
  const int64_t env = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (env >= p.n || (p.mask && !p.mask[env])) return;
  float* rows = p.buf + env * (int64_t)p.S * p.P;
  if (p.roll) {
    // _update_hist_amp_obs (:1341-1350).  A lane owns column i of every slot, so its loads of the old
    // slots precede its stores in program order; only slot 0 is rewritten by other lanes afterwards.
    if ((p.P & 3) == 0 && ((uintptr_t)rows & 15) == 0) {  // 196 floats per slot = 49 x 16 B: a quarter of the instructions
      float4* rows4 = reinterpret_cast<float4*>(rows);
      const int P4 = p.P >> 2;
      for (int i = lane; i < P4; i += 32) {
        float4 v[AMP_MAX_STEPS - 1];
#pragma unroll
        for (int k = 0; k < AMP_MAX_STEPS - 1; ++k)
          if (k < p.S - 1) v[k] = rows4[k * P4 + i];
#pragma unroll
        for (int k = 0; k < AMP_MAX_STEPS - 1; ++k)
          if (k < p.S - 1) rows4[(k + 1) * P4 + i] = v[k];
      }
    } else {
      for (int i = lane; i < p.P; i += 32) {
        float v[AMP_MAX_STEPS - 1];
#pragma unroll
        for (int k = 0; k < AMP_MAX_STEPS - 1; ++k)
          if (k < p.S - 1) v[k] = rows[k * p.P + i];
#pragma unroll
        for (int k = 0; k < AMP_MAX_STEPS - 1; ++k)
          if (k < p.S - 1) rows[(k + 1) * p.P + i] = v[k];
      }
    }
    __syncwarp();
  }
  amp_obs_row(AmpSrcSim{p, env}, p.K, p.dof_subset, p.num_sel, p.flags, lane, rows);
}

// One block = 8 envs.  Warp 0 lists the block's selected envs (ballot); a block without one leaves after
// reading 8 mask bytes.  The block's warps then walk the (selected env, slot) pairs: slot 0 from the sim state when
// `slot0` (_compute_amp_observations(env_ids), :792), slots >= 1 from the motion library, then the demo copy.
constexpr int AMPI_EPB = 8;

__global__ void __launch_bounds__(1024)
    amp_init_ref_kernel(AmpEnvParams p, LibDev L, const int64_t* __restrict__ motion_ids,
                        const float* __restrict__ motion_times, float dt, int slot0, int epb) {
  __shared__ int s_list[AMPI_EPB];
  __shared__ int s_count;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t env0 = (int64_t)blockIdx.x * epb;
  if (warp == 0) {
    const bool f = lane < epb && env0 + lane < p.n && (!p.mask || p.mask[env0 + lane]);
    const unsigned m = __ballot_sync(0xffffffffu, f);
    if (f) s_list[__popc(m & ((1u << lane) - 1u))] = lane;
    if (lane == 0) s_count = __popc(m);
  }
  __syncthreads();
  const int pairs = s_count * p.S;
  for (int w = warp; w < pairs; w += (int)(blockDim.x >> 5)) {
    const int64_t env = env0 + s_list[w / p.S];
    const int k = w % p.S;
    float* row = p.buf + (env * p.S + k) * (int64_t)p.P;
    // the demo row, _amp_obs_demo_buf[env_ids] = _amp_obs_buf[env_ids] (:819), is written with the row itself
    float* drow = p.demo ? p.demo + (env * p.S + k) * (int64_t)p.P : nullptr;
    if (k > 0) {
      const int64_t id = motion_ids[env];
      // motion_times + (-dt * (arange(S-1) + 1)), both fp32 (:809-810)
      const float t = motion_times[env] + (-dt) * (float)k;
      int64_t i0, i1;
      float bl;
      calc_frame_blend(t, L.len[id], L.nf[id], L.mdt[id], i0, i1, bl);
      const int64_t st = L.starts[id];
      amp_obs_row(AmpSrcLib{L, p.key_ids, i0 + st, i1 + st, bl}, p.K, p.dof_subset, p.num_sel, p.flags, lane, row, drow);
    } else if (slot0) {
      amp_obs_row(AmpSrcSim{p, env}, p.K, p.dof_subset, p.num_sel, p.flags, lane, row, drow);
    } else if (drow) {  // slot 0 was written by an earlier launch
      for (int i = lane; i < p.P; i += 32) drow[i] = row[i];
    }
  }
}

// ---------------------------------------------------------------------------------------
// reward / reset per-body pieces shared by K4, K5 and the fused step
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void reward_partials(Vec3 pos, Quat rot, Vec3 vel, Vec3 ang, const RefBody& r,
                                                float& sp, float& sr, float& sv, float& sa) {
  sp = mean_sq3(r.pos - pos);  // (d**2).mean(-1), common.py:299
  const float a = quat_angle(quat_mul_conj_w(r.rot, rot));
  sr = a * a;
  sv = mean_sq3(r.vel - vel);
  sa = mean_sq3(r.ang - ang);
}

// one env's reward from the four per-body rows (ATen row-sum order), common.py:298-320
__device__ __forceinline__ float reward_term(const float* row, int J, float k) {
  float d = aten_row_sum(row, J) / (float)J;
  return expf((-k) * d);
}

constexpr int GEN_MAX_J = 32;

__global__ void reward_kernel(PhcBodyState s, PhcBodyState ref, int64_t n, PhcRewardSpec spec,
                              float* __restrict__ reward, float* __restrict__ raw, int64_t raw_stride, int epb) {
  extern __shared__ float sm[];  // [epb][4][J] partials, [epb][4] terms
  const int J = s.num_bodies;
  const int e = threadIdx.x / J, b = threadIdx.x % J;
  const int64_t env = (int64_t)blockIdx.x * epb + e;
  const bool valid = e < epb && env < n;
  float* part = sm;
  float* terms = sm + epb * 4 * J;
  if (valid) {
    RefBody r;
    r.pos = ld3(view_at(ref.pos, env, b));
    r.rot = ld4(view_at(ref.rot, env, b));
    r.vel = ld3(view_at(ref.vel, env, b));
    r.ang = ld3(view_at(ref.ang_vel, env, b));
    float sp, sr, sv, sa;
    reward_partials(ld3(view_at(s.pos, env, b)), ld4(view_at(s.rot, env, b)), ld3(view_at(s.vel, env, b)),
                    ld3(view_at(s.ang_vel, env, b)), r, sp, sr, sv, sa);
    part[(e * 4 + 0) * J + b] = sp;
    part[(e * 4 + 1) * J + b] = sr;
    part[(e * 4 + 2) * J + b] = sv;
    part[(e * 4 + 3) * J + b] = sa;
  }
  __syncthreads();
  if (valid && b < 4) {
    const float k = b == 0 ? spec.k_pos : b == 1 ? spec.k_rot : b == 2 ? spec.k_vel : spec.k_ang_vel;
    float t = reward_term(part + (e * 4 + b) * J, J, k);
    terms[e * 4 + b] = t;
    raw[env * raw_stride + b] = t;
  }
  __syncthreads();
  if (valid && b == 0) {
    const float* t = terms + e * 4;
    reward[env] = spec.w_pos * t[0] + spec.w_rot * t[1] + spec.w_vel * t[2] + spec.w_ang_vel * t[3];
  }
}

__global__ void reset_kernel(PhcView pos, PhcView ref, int R, const int16_t* __restrict__ progress,
                             const uint8_t* __restrict__ pass_time, const float* __restrict__ term_dist, int early,
                             int use_mean, int64_t n, uint8_t* __restrict__ reset, uint8_t* __restrict__ terminated,
                             int epb) {
  extern __shared__ float sm[];  // [epb][R] distances
  const int e = threadIdx.x / R, b = threadIdx.x % R;
  const int64_t env = (int64_t)blockIdx.x * epb + e;
  const bool valid = e < epb && env < n;
  if (valid) sm[e * R + b] = norm3(ld3(view_at(pos, env, b)) - ld3(view_at(ref, env, b)));
  __syncthreads();
  if (valid && b == 0) {
    bool fallen = false;
    if (early) {
      const float* d = sm + e * R;
      if (use_mean) {
        fallen = (aten_row_sum(d, R) / (float)R) > term_dist[0];
      } else {
        for (int j = 0; j < R; ++j) fallen = fallen || (d[j] > term_dist[j]);
      }
      fallen = fallen && (progress[env] > 1);
    }
    terminated[env] = fallen ? 1 : 0;
    reset[env] = pass_time[env] ? 1 : (fallen ? 1 : 0);
  }
}

// ---------------------------------------------------------------------------------------
// _action_to_pd_targets (humanoid_phc.py:1218-1228) + the freeze_hand / freeze_toe zeroing of
// step() (:118-127); one thread per (env, dof)
// ---------------------------------------------------------------------------------------
__global__ void pd_targets_kernel(const float* __restrict__ action, const float* __restrict__ offset,
                                  const float* __restrict__ scale, int res_action, const float* __restrict__ ref_dof_pos,
                                  const float* __restrict__ dof_pos, int64_t dp_stride, int64_t dp_estride,
                                  uint32_t zero_mask, int64_t n, int D, float clip, float* __restrict__ actions_out,
                                  float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * D) return;
  const int64_t env = i / D;
  const int d = (int)(i - env * D);
  float a = action[i];
  // np.clip(actions, -1, 1) of the wrapper (clean_pufferl/env.py:110-112); NaN stays NaN as in numpy
  if (clip > 0.0f) a = a < -clip ? -clip : (a > clip ? clip : a);
  if (actions_out) actions_out[i] = a;  // self.actions[:] = ...
  float pd;
  if (res_action) {
    pd = ref_dof_pos[i] + scale[d] * a;
    const float q = dof_pos[env * dp_stride + d * dp_estride];
    const float half_pi = 1.57079637050628662f;  // f32(np.pi / 2)
    // maximum(minimum(pd, upper), lower); torch.minimum / maximum propagate a NaN of either operand, fminf / fmaxf
    // would drop it
    const float upper = q + half_pi, lower = q - half_pi;
    pd = pd < upper || pd != pd ? pd : upper;
    pd = pd > lower || pd != pd ? pd : lower;
  } else {
    pd = offset[d] + scale[d] * a;
  }
  if (zero_mask >> (d / 3) & 1u) pd = 0.0f;
  out[i] = pd;
}

// ---------------------------------------------------------------------------------------
// K7: reference-state-init reset of the envs selected by a mask (humanoid_phc.py:665-778).
// One thread per (env, body).  _sample_ref_state -> get_motion_state (full: local rotations ->
// dof_pos, dof velocities) -> _set_env_state scatter -> clock / buffer resets.  The observation
// of the reset envs is a masked obs-only pass of the step kernel, launched right after.
// ---------------------------------------------------------------------------------------
// what a reset writes besides the observation row (shared by phc_reset_envs and the reset inside the fused step)
struct ResetTargets {
  PhcBodyState body;  // written
  float* root;
  int64_t root_stride;
  float* dof_pos;
  float* dof_vel;
  int64_t dof_stride, dof_estride;
  int16_t* progress;
  uint8_t* reset;
  uint8_t* term;
  float* start;
  float* start_off;
  float* goff;
  const float* phase;
  int state_init, flag_test;
  // StateInit.Default / Hybrid (humanoid_phc.py:688-692, :733-745)
  const float* init_root;
  int64_t init_root_stride;
  const float* init_dof_pos;
  const float* init_dof_vel;
  int64_t init_dof_stride;
  const uint8_t* default_mask;
};

// self-observation variant (compute_humanoid_observations_smpl_max flags, humanoid_phc.py:963-998)
struct ObsFlags {
  int hcol;        // 1: root height column present (root_height_obs)
  int local_root;  // local_root_obs
  int upright;     // upright (False: remove_base_rot before the heading)
  int v7;          // PHC_OBS_TASK_V7: the task block of a future step is [d_pos | d_vel | l_pos]
};
// floats of one future step's task block
__host__ __device__ __forceinline__ int task_width(const ObsFlags& f) { return f.v7 ? TASK_DIM_V7 : TASK_DIM; }

// RunningNorm.forward of the rows a kernel writes (policies/running_norm.py:15-20)
struct NormOut {
  float* out;  // NULL = off
  int64_t stride;
  const float* mean;
  const float* var;
  float eps, clip;
  int bf16;
};

struct ResetParams {
  LibDev L;
  ResetTargets w;
  const int64_t* ids;
  const uint8_t* mask;
  int64_t n;
  float* obs;  // [n, selfw + task_width(of) T]: rows of the reset envs rewritten
  int64_t obs_stride;
  int T;
  float dt;
  ObsFlags of;
  NormOut norm;
  double* moments;  // NULL, or [buckets][2 W]
  int moment_buckets, moments_mode;  // mode 1: add the new rows; 2: replace (subtract the old row first)
  float* ref_dof_pos;  // NULL, or [n, 69]
  int64_t ref_dof_pos_stride;
};

struct ResetEnvOut {  // what the scatter leaves in registers for the observation of the same (env, body)
  Vec3 pos, vel, ang;
  Quat rot;
  float t, len, mdt;
  int64_t nf, st;
  // the clock the env's reference bodies are queried with afterwards: (progress + q) dt + t + soff, posed with g.
  // Reference-state init leaves soff = 0 and g = 0; a default-init env keeps its start time, offset and global offset.
  float soff, g0, g1, g2;
};

constexpr int K7_EPB = 8;

// the reference body b of a just-reset env at (progress + q) dt + start + offset with progress = 0, offset = 0
// (humanoid_phc.py:1063-1067), blended like blend_ref; the global offset is the zero the reset leaves
__device__ __forceinline__ void reset_query_frames(int q, float dt, float t, float len, int64_t nf, float mdt, int64_t st,
                                                   int64_t& f0, int64_t& f1, float& bl, float soff = 0.0f) {
  const float tq = (float)(int16_t)q * dt + t + soff;
  int64_t i0, i1;
  calc_frame_blend(tq, len, nf, mdt, i0, i1, bl);
  f0 = i0 + st, f1 = i1 + st;
}
// the same with a 32-bit frame count (identical results, see calc_frame_blend32): the in-step reset's dependent chain
__device__ __forceinline__ void reset_query_frames32(int q, float dt, float t, float len, int nf, float mdt, int64_t st,
                                                     int64_t& f0, int64_t& f1, float& bl) {
  const float tq = (float)(int16_t)q * dt + t + 0.0f;
  int i0, i1;
  calc_frame_blend32(tq, len, nf, mdt, i0, i1, bl);
  f0 = st + i0, f1 = st + i1;
}
__device__ __forceinline__ RefBody reset_ref_body(const LibDev& L, int q, float dt, float t, float len, int64_t nf, float mdt,
                                                  int64_t st, int b, float soff = 0.0f, float g0 = 0.0f, float g1 = 0.0f,
                                                  float g2 = 0.0f) {
  int64_t f0, f1;
  float bl;
  reset_query_frames(q, dt, t, len, nf, mdt, st, f0, f1, bl, soff);
  const float om = 1.0f - bl;
  RefBody r;
  r.pos = lerp3(om, bl, ld3(L.gts + (f0 * J24 + b) * 3), ld3(L.gts + (f1 * J24 + b) * 3));
  r.pos.x += g0, r.pos.y += g1, r.pos.z += g2;
  r.rot = quat_slerp(ld4v(L.grs + (f0 * J24 + b) * 4), ld4v(L.grs + (f1 * J24 + b) * 4), bl);
  r.vel = lerp3(om, bl, ld3(L.gvs + (f0 * J24 + b) * 3), ld3(L.gvs + (f1 * J24 + b) * 3));
  r.ang = lerp3(om, bl, ld3(L.gavs + (f0 * J24 + b) * 3), ld3(L.gavs + (f1 * J24 + b) * 3));
  return r;
}

// MotionLibBase.sample_time_interval (motion_lib.py:526-535) with the caller's uniform number:
//   ((phase * motion_len) / curr_fps).long() * curr_fps with curr_fps = 1/30; 0 for StateInit.Start / flag_test (:856)
__device__ __forceinline__ float reset_start_time(const ResetTargets& w, int64_t env, float len) {
  if ((w.state_init == PHC_STATE_INIT_RANDOM || w.state_init == PHC_STATE_INIT_HYBRID) && !w.flag_test) {
    const float c30 = (float)(1.0 / 30.0);
    const long long k = (long long)((w.phase[env] * len) / c30);
    return (float)k * c30;
  }
  return 0.0f;
}

// One (env, body) of a reference-state-init reset: get_motion_state at the new start time (motion_lib.py:549-626)
// posed with the OLD global offset (:860), the _set_env_state scatter (humanoid_phc.py:901-931) and, on body 0, the
// clock updates of _reset_ref_state_init (:724-731) and the buffer resets of _reset_env_tensors (:775-778).
// `write_flags`: also clear reset_buf / terminate_buf (the fused step leaves that to the lane that owns the flags).
// the _set_env_state scatter of one (env, body) (humanoid_phc.py:901-931) and, on body 0, the clock updates of
// _reset_ref_state_init (:724-731) and the buffer resets of _reset_env_tensors (:775-778)
__device__ __forceinline__ void reset_store_body(const ResetTargets& w, int64_t env, int b, float t, Vec3 pos, Quat rot,
                                                 Vec3 vel, Vec3 ang, bool write_flags) {
  st3(const_cast<float*>(view_at(w.body.pos, env, b)), pos);
  st4(const_cast<float*>(view_at(w.body.rot, env, b)), rot);
  st3(const_cast<float*>(view_at(w.body.vel, env, b)), vel);
  st3(const_cast<float*>(view_at(w.body.ang_vel, env, b)), ang);
  if (b == 0) {
    if (w.root) {
      float* r = w.root + env * w.root_stride;
      st3(r, pos);
      st4(r + 3, rot);
      st3(r + 7, vel);
      st3(r + 10, ang);
    }
    if (w.goff) {
      w.goff[env * 3 + 0] = 0.0f;
      w.goff[env * 3 + 1] = 0.0f;
      w.goff[env * 3 + 2] = 0.0f;
    }
    w.start[env] = t;
    w.start_off[env] = 0.0f;
    w.progress[env] = 0;
    if (write_flags) {
      w.reset[env] = 0;
      w.term[env] = 0;
    }
  }
}

// dof_pos / dof_vel of one (env, body) from library rows f0, f1: _local_rotation_to_dof_smpl (motion_lib.py:670-673)
// and the dof_vel lerp (:604)
__device__ __forceinline__ void reset_store_dof(const LibDev& L, const ResetTargets& w, int64_t env, int b, int64_t f0,
                                                int64_t f1, float bl) {
  const float om = 1.0f - bl;
  if (w.dof_pos && b >= 1) {
    const Quat lr = quat_slerp(ld4v(L.lrs + (f0 * J24 + b) * 4), ld4v(L.lrs + (f1 * J24 + b) * 4), bl);
    const Vec3 em = quat_exp_map(lr);
    float* d = w.dof_pos + env * w.dof_stride + (int64_t)(b - 1) * 3 * w.dof_estride;
    d[0] = em.x;
    d[w.dof_estride] = em.y;
    d[2 * w.dof_estride] = em.z;
  }
  if (w.dof_vel && b < 23) {
    const Vec3 dv = lerp3(om, bl, ld3(L.dvs + (f0 * 23 + b) * 3), ld3(L.dvs + (f1 * 23 + b) * 3));
    float* d = w.dof_vel + env * w.dof_stride + (int64_t)b * 3 * w.dof_estride;
    d[0] = dv.x;
    d[w.dof_estride] = dv.y;
    d[2 * w.dof_estride] = dv.z;
  }
}

// One (env, body) of a reference-state-init reset: get_motion_state at the new start time (motion_lib.py:549-626)
// posed with the OLD global offset (:860), then the two scatters above.
// `write_flags`: also clear reset_buf / terminate_buf (the fused step leaves that to the lane that owns the flags).
__device__ __forceinline__ void reset_scatter_thread(const LibDev& L, const ResetTargets& w, int64_t env, int b, float t,
                                                     float len, int64_t nf, float mdt, int64_t st, float g0, float g1,
                                                     float g2, bool write_flags, ResetEnvOut& o) {
  int64_t i0, i1;
  float bl;
  calc_frame_blend(t, len, nf, mdt, i0, i1, bl);
  const int64_t f0 = i0 + st, f1 = i1 + st;
  const float om = 1.0f - bl;
  Vec3 pos = lerp3(om, bl, ld3(L.gts + (f0 * J24 + b) * 3), ld3(L.gts + (f1 * J24 + b) * 3));
  pos.x += g0;
  pos.y += g1;
  pos.z += g2;
  const Quat rot = quat_slerp(ld4v(L.grs + (f0 * J24 + b) * 4), ld4v(L.grs + (f1 * J24 + b) * 4), bl);
  const Vec3 vel = lerp3(om, bl, ld3(L.gvs + (f0 * J24 + b) * 3), ld3(L.gvs + (f1 * J24 + b) * 3));
  const Vec3 ang = lerp3(om, bl, ld3(L.gavs + (f0 * J24 + b) * 3), ld3(L.gavs + (f1 * J24 + b) * 3));
  reset_store_body(w, env, b, t, pos, rot, vel, ang, write_flags);
  reset_store_dof(L, w, env, b, f0, f1, bl);
  o.pos = pos, o.rot = rot, o.vel = vel, o.ang = ang;
  o.t = t, o.len = len, o.mdt = mdt, o.nf = nf, o.st = st;
  o.soff = 0.0f, o.g0 = 0.0f, o.g1 = 0.0f, o.g2 = 0.0f;
}

// One (env, body) of a default-init reset (_reset_default, humanoid_phc.py:688-692, then _reset_env_tensors :775-778):
// root / dof state from the initial buffers; the rigid-body tensors, start time, offset and global offset stay; the
// body's CURRENT state goes to the registers the observation of the same launch is computed from.
__device__ __forceinline__ void reset_default_thread(const LibDev& L, const ResetTargets& w, int64_t env, int b, int64_t id,
                                                     float g0, float g1, float g2, ResetEnvOut& o) {
  o.pos = ld3(view_at(w.body.pos, env, b));
  o.rot = ld4(view_at(w.body.rot, env, b));
  o.vel = ld3(view_at(w.body.vel, env, b));
  o.ang = ld3(view_at(w.body.ang_vel, env, b));
  if (b == 0 && w.root) {
    const float* src = w.init_root + env * w.init_root_stride;
    float* r = w.root + env * w.root_stride;
#pragma unroll
    for (int k = 0; k < 13; ++k) r[k] = src[k];
  }
  if (w.dof_pos && b >= 1) {
    const float* src = w.init_dof_pos + env * w.init_dof_stride + (b - 1) * 3;
    float* d = w.dof_pos + env * w.dof_stride + (int64_t)(b - 1) * 3 * w.dof_estride;
    d[0] = src[0], d[w.dof_estride] = src[1], d[2 * w.dof_estride] = src[2];
  }
  if (w.dof_vel && b < 23) {
    const float* src = w.init_dof_vel + env * w.init_dof_stride + b * 3;
    float* d = w.dof_vel + env * w.dof_stride + (int64_t)b * 3 * w.dof_estride;
    d[0] = src[0], d[w.dof_estride] = src[1], d[2 * w.dof_estride] = src[2];
  }
  o.t = w.start[env], o.soff = w.start_off[env];  // the motion clock is not restarted
  o.len = L.len[id], o.mdt = L.mdt[id], o.nf = L.nf[id], o.st = L.starts[id];
  o.g0 = g0, o.g1 = g1, o.g2 = g2;
  if (b == 0) {
    w.progress[env] = 0;
    w.reset[env] = 0;
    w.term[env] = 0;
  }
}

// `act`: this thread's env is in range and selected by the mask (read by the caller, once, before anything is
// written: the mask may be reset_buf itself, which the last lines clear)
__device__ __forceinline__ void reset_scatter_body(const ResetParams& p, const bool act, ResetEnvOut& o) {
  __shared__ float s_goff[K7_EPB][3];
  const int e = threadIdx.x / J24, b = threadIdx.x % J24;
  const int64_t env = (int64_t)blockIdx.x * K7_EPB + e;
  if (act && b < 3) s_goff[e][b] = p.w.goff ? p.w.goff[env * 3 + b] : 0.0f;  // the OLD offset poses the env (:860)
  __syncthreads();
  if (!act) return;
  const int64_t id = p.ids[env];
  if (p.w.state_init == PHC_STATE_INIT_DEFAULT || (p.w.state_init == PHC_STATE_INIT_HYBRID && p.w.default_mask[env])) {
    reset_default_thread(p.L, p.w, env, b, id, s_goff[e][0], s_goff[e][1], s_goff[e][2], o);
    return;
  }
  const float len = p.L.len[id];
  const float t = reset_start_time(p.w, env, len);
  reset_scatter_thread(p.L, p.w, env, b, t, len, p.L.nf[id], p.L.mdt[id], p.L.starts[id], s_goff[e][0], s_goff[e][1],
                       s_goff[e][2], true, o);
}

// ---- the observation row of one (env, body): shared by every step kernel and the reset kernel -----------------
// DEF: the env's default flags (height column, local root, upright) with the 8-byte aligned shared-memory stage of the
// TMA kernels: constant column offsets and float2 stores.  !DEF: any flag combination, any alignment.
template <bool DEF>
__device__ __forceinline__ void put6(float* p, const float* v) {
  if (DEF) {
    st6_shared(p, v);
  } else {
#pragma unroll
    for (int k = 0; k < 6; ++k) p[k] = v[k];
  }
}
// the root rotation the heading is taken from: as is when upright, remove_base_rot first otherwise (common.py:42-47)
__device__ __forceinline__ Quat heading_source(Quat root_rot, int upright) { return upright ? root_rot : remove_base_rot(root_rot); }

// self obs, common.py:23-103: [root_h? | rot(h^-1, p_b - p_root) b >= 1 | tan_norm(h^-1 (x) q_b) | rot(h^-1, v_b) | rot(h^-1, w_b)]
template <bool DEF>
__device__ __forceinline__ void emit_self_obs(float* row, const ObsFlags& of, int b, Vec3 root_pos, Heading hi,
                                              const HeadingRot& hr, Vec3 pos, Quat rot, Vec3 vel, Vec3 ang) {
  const int h = DEF ? 1 : of.hcol;
  if (b == 0) {
    if (h) row[0] = root_pos.z;
  } else {
    st3(row + h + (b - 1) * 3, heading_rotate(hr, pos - root_pos));
  }
  float t6[6];
  if (!DEF && b == 0 && !of.local_root)
    quat_tan_norm(heading_source(rot, of.upright), t6);  // "if not local_root_obs: root_rot_obs = quat_to_tan_norm(root_rot)" (:76-78)
  else
    quat_tan_norm(heading_mul_left(hi, rot), t6);
  put6<DEF>(row + h + 69 + b * 6, t6);
  st3(row + h + 213 + b * 3, heading_rotate(hr, vel));
  st3(row + h + 285 + b * 3, heading_rotate(hr, ang));
}

// one v6 block of 576 floats, common.py:106-176
template <bool DEF>
__device__ __forceinline__ void emit_task_obs(float* tk, int b, Heading hi, const HeadingRot& hr, Vec3 root_pos, Vec3 pos,
                                              Quat rot, Vec3 vel, Vec3 ang, const RefBody& r) {
  TaskObs o;
  task_obs_body(hi, hr, root_pos, pos, rot, vel, ang, r, true, o);
  st3(tk + b * 3, o.d_pos);
  put6<DEF>(tk + 72 + b * 6, o.d_rot);
  st3(tk + 216 + b * 3, o.d_vel);
  st3(tk + 288 + b * 3, o.d_ang);
  st3(tk + 360 + b * 3, o.l_pos);
  put6<DEF>(tk + 432 + b * 6, o.l_rot);
}

// one v7 block of 216 floats: the v6 block's [d_pos | d_vel | l_pos] (its columns 0:72, 216:288, 360:432) from the same
// operations (task_obs_body without the rotation terms, as phc_imitation_obs mode 7)
__device__ __forceinline__ void emit_task_obs_v7(float* tk, int b, Heading hi, const HeadingRot& hr, Vec3 root_pos, Vec3 pos,
                                                 Quat rot, Vec3 vel, Vec3 ang, const RefBody& r) {
  TaskObs o;
  task_obs_body(hi, hr, root_pos, pos, rot, vel, ang, r, false, o);
  st3(tk + b * 3, o.d_pos);
  st3(tk + 72 + b * 3, o.d_vel);
  st3(tk + 144 + b * 3, o.l_pos);
}

// the task block of the layout `v7` selects at run time (generic and reset kernels)
template <bool DEF>
__device__ __forceinline__ void emit_task(bool v7, float* tk, int b, Heading hi, const HeadingRot& hr, Vec3 root_pos,
                                          Vec3 pos, Quat rot, Vec3 vel, Vec3 ang, const RefBody& r) {
  if (v7) emit_task_obs_v7(tk, b, hi, hr, root_pos, pos, rot, vel, ang, r);
  else emit_task_obs<DEF>(tk, b, hi, hr, root_pos, pos, rot, vel, ang, r);
}

// emit_self_obs(row) and emit_task_obs(row + SW) of one body, bit for bit, with the vector work paired into fp32x2
// instructions (phc_math.cuh): the seven heading rotations as (p_b - p_root, v_b) | (d_pos, l_pos) | (d_vel, d_ang)
// and w_b alone, the two heading products and tan-norms of q_b and the reference rotation together.
template <bool DEF>
__device__ __forceinline__ void emit_obs_paired(float* row, int SW, const ObsFlags& of, int b, Vec3 root_pos, Heading hi,
                                                const HeadingRot& hr, Vec3 pos, Quat rot, Vec3 vel, Vec3 ang,
                                                const RefBody& r, float one) {
  const int h = DEF ? 1 : of.hcol;
  float* tk = row + SW;
  const Vec3x2 pv = heading_rotate2(hr, pack3(pos - root_pos, vel));
  const Vec3x2 dl = heading_rotate2(hr, sub3x2(pack3(r.pos, r.pos), pack3(pos, root_pos), one));
  const Vec3x2 dva = heading_rotate2(hr, sub3x2(pack3(r.vel, r.ang), pack3(vel, ang), one));
  if (b == 0) {
    if (h) row[0] = root_pos.z;
  } else {
    st3(row + h + (b - 1) * 3, lane0(pv));
  }
  st3(row + h + 213 + b * 3, lane1(pv));
  st3(row + h + 285 + b * 3, heading_rotate(hr, ang));
  st3(tk + b * 3, lane0(dl));
  st3(tk + 360 + b * 3, lane1(dl));
  st3(tk + 216 + b * 3, lane0(dva));
  st3(tk + 288 + b * 3, lane1(dva));
  Quatx2 hq = heading_mul_left2(hi, pack4(rot, r.rot));
  if (!DEF && b == 0 && !of.local_root) {  // as in emit_self_obs
    const Quat s = heading_source(rot, of.upright);
    hq.x.x = s.x, hq.y.x = s.y, hq.z.x = s.z, hq.w.x = s.w;
  }
  float2 t2[6];
  quat_tan_norm2(hq, one, t2);
  float t6[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) t6[k] = t2[k].x;
  put6<DEF>(row + h + 69 + b * 6, t6);
#pragma unroll
  for (int k = 0; k < 6; ++k) t6[k] = t2[k].y;
  put6<DEF>(tk + 432 + b * 6, t6);
  const Quat dg = quat_mul(r.rot, quat_conj(rot));  // task_obs_body's d_rot
  quat_tan_norm(heading_mul_right(heading_mul_left(hi, dg), heading_conj(hi)), t6);
  put6<DEF>(tk + 72 + b * 6, t6);
}

// emit_self_obs(row) and emit_task_obs_v7(row + SW) of one body, bit for bit, paired as emit_obs_paired does:
// (p_b - p_root, v_b) | (d_pos, l_pos) | (d_vel, w_b).  No reference rotation is read: the tan-norm of q_b stays scalar.
template <bool DEF>
__device__ __forceinline__ void emit_obs_paired_v7(float* row, int SW, const ObsFlags& of, int b, Vec3 root_pos, Heading hi,
                                                   const HeadingRot& hr, Vec3 pos, Quat rot, Vec3 vel, Vec3 ang,
                                                   const RefBody& r, float one) {
  const int h = DEF ? 1 : of.hcol;
  float* tk = row + SW;
  const Vec3x2 pv = heading_rotate2(hr, pack3(pos - root_pos, vel));
  const Vec3x2 dl = heading_rotate2(hr, sub3x2(pack3(r.pos, r.pos), pack3(pos, root_pos), one));
  const Vec3x2 dw = heading_rotate2(hr, pack3(r.vel - vel, ang));
  if (b == 0) {
    if (h) row[0] = root_pos.z;
  } else {
    st3(row + h + (b - 1) * 3, lane0(pv));
  }
  st3(row + h + 213 + b * 3, lane1(pv));
  st3(row + h + 285 + b * 3, lane1(dw));
  st3(tk + b * 3, lane0(dl));
  st3(tk + 72 + b * 3, lane0(dw));
  st3(tk + 144 + b * 3, lane1(dl));
  float t6[6];
  if (!DEF && b == 0 && !of.local_root)
    quat_tan_norm(heading_source(rot, of.upright), t6);
  else
    quat_tan_norm(heading_mul_left(hi, rot), t6);
  put6<DEF>(row + h + 69 + b * 6, t6);
}

// ---------------------------------------------------------------------------------------
// K6: the fused step.  One block = EPB envs x 24 bodies.
//   phase 0  sim tile -> smem (cp.async 16 B when the four views are one 16-B aligned AoS-13
//            tensor; strided scalar loads otherwise); env leaders advance the clock and run
//            the frame-blend for t, t+dt .. t+T*dt
//   phase 1  frames(t) -> smem; per body: lerp/slerp -> reference state, reward partials,
//            distance; smem reductions -> rew_buf / reward_raw / reset_buf / terminate_buf
//   phase 2  for each future step: frames -> smem; reference state; v6 block; the obs row is
//            staged in smem (aliasing the frame buffer) and streamed out with 8-byte stores
// ---------------------------------------------------------------------------------------
constexpr int ROW13 = J24 * 13;              // 312 floats of sim state per env
constexpr int FRAME_FLOATS = J24 * 13;       // pos 72 | rot 96 | vel 72 | ang 72
constexpr int FRAME_F4 = FRAME_FLOATS / 4;   // 78
constexpr int STAGE_FLOATS = SELF_DIM + TASK_DIM;  // 934

constexpr int EP_SUM_COLS = 12;  // 4 episode sums + up to 8 reward_raw column sums (PHC_EPISODE_SUM_COLS)

struct StepParams {
  LibDev L;
  PhcBodyState body;
  int16_t* progress;
  int16_t* progress_mirror;  // NULL, or a second place (mapped host memory) that receives the advanced progress
  const float* start;
  const float* start_off;
  const float* goff;
  const int64_t* ids;
  const float* term_dist;
  uint32_t reset_mask;
  int use_mean, early, advance, T;
  float dt;
  float one;  // 1.0f, the multiplier of the packed add (add2 in phc_math.cuh): a literal would let ptxas fuse it
  PhcRewardSpec rwd;
  float* obs;
  int64_t obs_stride;
  float* rew;
  float* raw;
  int64_t raw_stride;
  uint8_t* reset;
  uint8_t* term;
  double* moments;
  int moment_buckets;  // >= 1: moments is [buckets][2W]; block b adds into bucket b % buckets
  int multi_prefetch;  // K6-multi2: L2-prefetch the frame rows two query iterations ahead
  int moments_bulk;    // the T = 1 kernel hands its partials to TMA bulk reductions instead of issuing atomics
  // episode bookkeeping of the pufferlib wrapper fused into the step (clean_pufferl/env.py:121-159), off when ep_returns is NULL
  uint8_t *ep_terminals, *ep_truncations, *ep_masks;
  float* ep_returns;
  int32_t* ep_lengths;
  double* ep_sums;  // [ep_buckets][EP_SUM_COLS]: {episodes, sum of returns, sum of lengths, truncations, sum of reward_raw[:, c]}
  int ep_buckets, ep_raw_cols;
  int ep_block0;    // the launch's first block in the batch (host chunks): block b adds into bucket (ep_block0 + b) % ep_buckets
  float* mpjpe;     // NULL, or [n]: mean over the 24 bodies of |body_pos - ref_body_pos| (extras["mpjpe"])
  float* obs_norm;  // NULL, or the normalised copy of the obs rows (RunningNorm.forward)
  int64_t obs_norm_stride;
  const float* norm_mean;
  const float* norm_var;
  float norm_eps, norm_clip;
  int norm_bf16;  // obs_norm holds bfloat16 rows (PHC_STEP_OBS_NORM_BF16)
  const float* dof_force;  // power reward inputs (NULL = off)
  int64_t dof_force_stride;
  const float* dof_vel;
  int64_t dof_vel_stride, dof_vel_estride;
  float power_coef;
  int power_col;
  int64_t n;
  int first_wave_blocks;      // blocks that can be resident at once (speculate before the dependency wait)
  int spec4_blocks;           // blocks [0, spec4_blocks) speculate on progress + 3 too (the spare slots of one wave)
  int spec_fault;             // test hook: perturb the speculated clock (PHC_OPT_TEST_SPEC_FAULT)
  unsigned long long* trace;  // NULL, or [grid][8] globaltimer stamps (phc_set_trace_buffer)
  const uint8_t* env_mask;  // NULL, or [n]: only envs with a non-zero byte are processed (generic kernel)
  int obs_only;             // 1: observations only — no reward / reset outputs, clock untouched
  int aos;        // sim state is one AoS-13 tensor, 16-B aligned rows
  int obs_vec2;   // obs rows can be written with 8-byte stores
  float* rew_out;      // NULL, or a second copy of rew_buf (the wrapper's rewards.clone())
  uint8_t* reset_out;  // NULL, or the step's reset flags (kept when the in-step reset clears reset_buf)
  uint8_t* term_out;   // NULL, or extras["terminate"]
  float* ref_dof_pos;  // NULL, or [n, 69]: dof_pos of the query at t + dt (res_action, humanoid_phc.py:1115-1120)
  int64_t ref_dof_pos_stride;
  ObsFlags of;         // self-obs flags; of.hcol && of.local_root && of.upright = the env's defaults
  int selfw;           // 357 + of.hcol
  int reset_on;        // the flagged envs are reset inside the step (PhcStepArgs.auto_reset)
  ResetTargets rw;
  unsigned* tile_counter;  // persistent kernel: [0] next tile to draw, [1] blocks that have left (both 0 between launches)
};

__host__ __device__ __forceinline__ bool default_obs_flags(const ObsFlags& f) { return f.hcol && f.local_root && f.upright; }

// dof_pos of the motion query whose frames are rows f0 / f1 of the library (motion_lib.py:608-610, 670-673): body b >= 1
__device__ __forceinline__ void write_ref_dof_pos(const StepParams& p, int64_t env, int b, int64_t f0, int64_t f1, float bl) {
  if (b < 1) return;
  const Quat lr = quat_slerp(ld4v(p.L.lrs + (f0 * J24 + b) * 4), ld4v(p.L.lrs + (f1 * J24 + b) * 4), bl);
  st3(p.ref_dof_pos + env * p.ref_dof_pos_stride + (b - 1) * 3, quat_exp_map(lr));
}

// RunningNorm.forward of one value (policies/running_norm.py:15-20): clamp((x - mean) / sqrt(var + eps)).
// torch.clamp keeps NaN; fminf / fmaxf would turn it into -clip, so the clamp is two compare-selects.
__device__ __forceinline__ float norm_clamp(float y, float clip) { return y < -clip ? -clip : (y > clip ? clip : y); }
// `sd` = sqrt(var + eps) and `r` ~ 1/sd are per column.  sqrt_faithful needs a normal finite argument (rsqrt.approx.ftz
// flushes a subnormal one, 0 * rsqrt(0) is NaN); 0, subnormals, inf and NaN take IEEE sqrtf.
__device__ __forceinline__ void norm_column(const float* means, const float* vars, float eps, int64_t col, float& mean,
                                            float& sd, float& r) {
  mean = means[col];
  const float v = vars[col] + eps;
  sd = v >= FLT_MIN && v <= FLT_MAX ? sqrt_faithful(v) : sqrtf(v);
  r = rcp_approx(sd);
}
__device__ __forceinline__ void norm_column(const StepParams& p, int64_t col, float& mean, float& sd, float& r) {
  norm_column(p.norm_mean, p.norm_var, p.norm_eps, col, mean, sd, r);
}
// The quotient is within 1 ulp of IEEE division where q = a * r is finite and sd is normal, and the Newton step is then
// finite.  Where the step gives NaN, q already is what IEEE division gives (x or the statistics are inf / NaN, or sd
// is 0 or inf), so q is taken.
__device__ __forceinline__ float norm_value(float x, float mean, float sd, float r, float clip) {
  const float a = x - mean;
  const float y = div_faithful(a, sd, r);
  return norm_clamp(y != y ? a * r : y, clip);
}

// per-body share of power = sum_dof |dof_force * dof_vel| (humanoid_phc.py:1298): body b >= 1 owns
// the 3 dofs of joint b - 1
__device__ __forceinline__ float power_partial(const StepParams& p, int64_t env, int b) {
  if (b == 0) return 0.0f;
  const float* f = p.dof_force + env * p.dof_force_stride + (b - 1) * 3;
  const float* v = p.dof_vel + env * p.dof_vel_stride + (int64_t)(b - 1) * 3 * p.dof_vel_estride;
  return (fabsf(__ldcg(f) * __ldcg(v)) + fabsf(__ldcg(f + 1) * __ldcg(v + p.dof_vel_estride))) +
         fabsf(__ldcg(f + 2) * __ldcg(v + 2 * p.dof_vel_estride));
}
// r = -coef * power, zeroed while progress <= 3 (humanoid_phc.py:1300-1302)
__device__ __forceinline__ float power_reward(const StepParams& p, const float* row24, int prog) {
  const float r = (-p.power_coef) * row_sum24(row24);
  return prog <= 3 ? 0.0f : r;
}

template <int EPB>
struct StepSmem {
  static constexpr int NT = EPB * J24;
  static constexpr int BUF = EPB * (STAGE_FLOATS > 2 * FRAME_FLOATS ? STAGE_FLOATS : 2 * FRAME_FLOATS);
  float sim[EPB * ROW13];
  float buf[BUF];             // frames [EPB][2][312]  /  obs stage [EPB][934]
  float part[6][EPB][J24];    // reward partials x4, distance, power
  float terms[EPB][4];
  float goff[EPB][4];
  float hz[EPB], hw[EPB];
  int64_t f0[PHC_MAX_TIME_STEPS + 1][EPB];
  int64_t f1[PHC_MAX_TIME_STEPS + 1][EPB];
  float bl[PHC_MAX_TIME_STEPS + 1][EPB];
  int prog[EPB];
  int pass[EPB];
  int act[EPB];  // env is in range and selected by env_mask
};

template <int EPB>
__device__ __forceinline__ void load_frames(const LibDev& L, StepSmem<EPB>& S, int q, int e, int b, bool valid) {
  // 24 threads of env e bring its two frames (2 x 78 float4) into S.buf[e][fr][...]
  if (valid) {
    const int64_t fa = S.f0[q][e], fb = S.f1[q][e];
    float* dst_e = S.buf + e * (2 * FRAME_FLOATS);
#pragma unroll
    for (int it = 0; it < (2 * FRAME_F4 + J24 - 1) / J24; ++it) {
      const int i = b + it * J24;
      if (i < 2 * FRAME_F4) {
        const int fr = i >= FRAME_F4;
        const int k = i - fr * FRAME_F4;
        const int64_t f = fr ? fb : fa;
        const float* src;
        if (k < 18)
          src = L.gts + f * 72 + k * 4;
        else if (k < 42)
          src = L.grs + f * 96 + (k - 18) * 4;
        else if (k < 60)
          src = L.gvs + f * 72 + (k - 42) * 4;
        else
          src = L.gavs + f * 72 + (k - 60) * 4;
        cp_async16(dst_e + fr * FRAME_FLOATS + k * 4, src);
      }
    }
  }
  cp_async_commit();
}

template <int EPB>
__device__ __forceinline__ RefBody blend_ref(const StepSmem<EPB>& S, int q, int e, int b) {
  const float* f0 = S.buf + e * (2 * FRAME_FLOATS);
  const float* f1 = f0 + FRAME_FLOATS;
  const float bl = S.bl[q][e];
  const float om = 1.0f - bl;
  RefBody r;
  r.pos = lerp3(om, bl, ld3(f0 + b * 3), ld3(f1 + b * 3));
  r.pos.x += S.goff[e][0];
  r.pos.y += S.goff[e][1];
  r.pos.z += S.goff[e][2];
  r.rot = quat_slerp(ld4v(f0 + 72 + b * 4), ld4v(f1 + 72 + b * 4), bl);
  r.vel = lerp3(om, bl, ld3(f0 + 168 + b * 3), ld3(f1 + 168 + b * 3));
  r.ang = lerp3(om, bl, ld3(f0 + 240 + b * 3), ld3(f1 + 240 + b * 3));
  return r;
}

template <int EPB>
__global__ void __launch_bounds__(EPB* J24) step_kernel(const StepParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  StepSmem<EPB>& S = *reinterpret_cast<StepSmem<EPB>*>(smem_raw);
  constexpr int NT = EPB * J24;
  const int tid = threadIdx.x;
  const int e = tid / J24, b = tid % J24;
  const int64_t env0 = (int64_t)blockIdx.x * EPB;
  const int64_t env = env0 + e;
  const bool valid = env < p.n && (!p.env_mask || p.env_mask[env]);
  const int nvalid = (int)((p.n - env0) < EPB ? (p.n - env0) : EPB);
  const int T = p.T;
  if (b == 0) S.act[e] = valid;  // read after the first barrier

  // ---- phase 0: sim tile + clock ------------------------------------------------------
  if (p.aos) {
    const float* src = p.body.pos.ptr + env0 * p.body.pos.stride_env;
    if (p.body.pos.stride_env == ROW13) {  // envs contiguous: one flat copy
      for (int i = tid; i < nvalid * (ROW13 / 4); i += NT) cp_async16(S.sim + i * 4, src + i * 4);
    } else {
      for (int i = tid; i < nvalid * (ROW13 / 4); i += NT) {
        const int ee = i / (ROW13 / 4), k = i % (ROW13 / 4);
        cp_async16(S.sim + ee * ROW13 + k * 4, src + ee * p.body.pos.stride_env + k * 4);
      }
    }
  } else if (valid) {
    float* d = S.sim + e * ROW13 + b * 13;
    const float* a = view_at(p.body.pos, env, b);
    const float* r = view_at(p.body.rot, env, b);
    const float* v = view_at(p.body.vel, env, b);
    const float* w = view_at(p.body.ang_vel, env, b);
    d[0] = a[0], d[1] = a[1], d[2] = a[2];
    d[3] = r[0], d[4] = r[1], d[5] = r[2], d[6] = r[3];
    d[7] = v[0], d[8] = v[1], d[9] = v[2];
    d[10] = w[0], d[11] = w[1], d[12] = w[2];
  }
  cp_async_commit();

  if (valid && b <= T) {
    // lanes 0..T of the env each run the frame-blend of one query time:
    // q = 0: t = progress*dt + start + offset (humanoid_phc.py:1236); q >= 1: (progress+q)*dt + ..
    // (humanoid_phc.py:1063-1067); progress is already advanced (humanoid_phc.py:138)
    int prog = (int)p.progress[env];
    if (p.advance) prog = (int)(int16_t)(prog + 1);
    const int16_t pq = (int16_t)(prog + b);
    const float t = (float)pq * p.dt + p.start[env] + p.start_off[env];
    const int64_t id = p.ids[env];
    const float len = p.L.len[id];
    int64_t i0, i1;
    float bl;
    calc_frame_blend(t, len, p.L.nf[id], p.L.mdt[id], i0, i1, bl);
    const int64_t st = p.L.starts[id];
    S.f0[b][e] = i0 + st;
    S.f1[b][e] = i1 + st;
    S.bl[b][e] = bl;
    if (b == 0) {
      S.prog[e] = prog;
      S.pass[e] = t >= len;  // _compute_reset, humanoid_phc.py:1317
      S.goff[e][0] = p.goff ? p.goff[env * 3 + 0] : 0.0f;
      S.goff[e][1] = p.goff ? p.goff[env * 3 + 1] : 0.0f;
      S.goff[e][2] = p.goff ? p.goff[env * 3 + 2] : 0.0f;
    }
  }
  __syncthreads();  // frame indices visible
  // progress is written only after every query lane of the env (possibly in another warp) read it
  if (valid && b == 0 && p.advance && !p.obs_only) {
    p.progress[env] = (int16_t)S.prog[e];
    if (p.progress_mirror) p.progress_mirror[env] = (int16_t)S.prog[e];
  }

  // ---- phase 1: reference state at t; reward; reset -------------------------------------
  load_frames<EPB>(p.L, S, 0, e, b, valid);
  cp_async_wait_all();
  __syncthreads();  // sim tile + frames(t) landed

  Vec3 pos, vel, ang;
  Quat rot;
  {
    const float* d = S.sim + e * ROW13 + b * 13;
    pos = {d[0], d[1], d[2]};
    rot = {d[3], d[4], d[5], d[6]};
    vel = {d[7], d[8], d[9]};
    ang = {d[10], d[11], d[12]};
  }
  if (valid) {
    const RefBody r = blend_ref<EPB>(S, 0, e, b);
    float sp, sr, sv, sa;
    reward_partials(pos, rot, vel, ang, r, sp, sr, sv, sa);
    S.part[0][e][b] = sp;
    S.part[1][e][b] = sr;
    S.part[2][e][b] = sv;
    S.part[3][e][b] = sa;
    S.part[4][e][b] = norm3(pos - r.pos);  // torch.norm(rigid_body_pos - ref_body_pos), common.py:343/348
    if (p.dof_force) S.part[5][e][b] = power_partial(p, env, b);
    if (b == 0) {
      const Heading hi = heading_quat_inv(heading_source(rot, p.of.upright));  // common.py:42-47
      S.hz[e] = hi.z;
      S.hw[e] = hi.w;
    }
  }
  __syncthreads();  // partials written; frames(t) no longer needed

  if (T >= 1) load_frames<EPB>(p.L, S, 1, e, b, valid);  // overlap with the reductions below
  if (valid && p.ref_dof_pos && !p.obs_only) write_ref_dof_pos(p, env, b, S.f0[1][e], S.f1[1][e], S.bl[1][e]);

  const bool outs = valid && !p.obs_only;  // obs-only passes leave reward / flags untouched
  if (outs && b < 4) {
    const float k = b == 0 ? p.rwd.k_pos : b == 1 ? p.rwd.k_rot : b == 2 ? p.rwd.k_vel : p.rwd.k_ang_vel;
    const float t = reward_term(&S.part[b][e][0], J24, k);
    S.terms[e][b] = t;
    p.raw[env * p.raw_stride + b] = t;
  } else if (outs && b == 4) {
    bool fallen = false;
    if (p.early) {
      const float* d = &S.part[4][e][0];
      if (p.use_mean) {
        float sel[J24];
        int m = 0;
#pragma unroll
        for (int j = 0; j < J24; ++j)
          if (p.reset_mask >> j & 1u) sel[m++] = d[j];
        // threshold of the first selected body: termination_distance[reset_ids][0] (common.py:343)
        int first = __ffs(p.reset_mask) - 1;
        fallen = m > 0 && (aten_row_sum(sel, m) / (float)m) > p.term_dist[first < 0 ? 0 : first];
      } else {
#pragma unroll
        for (int j = 0; j < J24; ++j)
          if (p.reset_mask >> j & 1u) fallen = fallen || (d[j] > p.term_dist[j]);
      }
      fallen = fallen && (S.prog[e] > 1);  // common.py:353
    }
    const bool rs = S.pass[e] || fallen;  // common.py:362
    p.term[env] = fallen ? 1 : 0;
    p.reset[env] = rs ? 1 : 0;
    if (p.term_out) p.term_out[env] = fallen ? 1 : 0;
    if (p.reset_out) p.reset_out[env] = rs ? 1 : 0;
  } else if (outs && b == 5 && p.mpjpe) {
    p.mpjpe[env] = row_sum24(&S.part[4][e][0]) / 24.0f;  // humanoid_phc.py:167
  }
  __syncwarp();
  if (outs && b == 0) {
    const float* t = S.terms[e];
    float r = p.rwd.w_pos * t[0] + p.rwd.w_rot * t[1] + p.rwd.w_vel * t[2] + p.rwd.w_ang_vel * t[3];
    if (p.dof_force) {
      const float pr = power_reward(p, &S.part[5][e][0], S.prog[e]);
      r += pr;  // rew_buf[:] += power_reward (humanoid_phc.py:1304)
      p.raw[env * p.raw_stride + p.power_col] = pr;
    }
    p.rew[env] = r;
    if (p.rew_out) p.rew_out[env] = r;
  }

  // ---- phase 2: observations -------------------------------------------------------------
  const Vec3 root_pos = {S.sim[e * ROW13 + 0], S.sim[e * ROW13 + 1], S.sim[e * ROW13 + 2]};
  const Heading hi = {S.hz[e], S.hw[e]};
  const HeadingRot hr = heading_rot(hi);
  const int SW = p.selfw;           // 358 with the root height column, 357 without
  const int TW = task_width(p.of);  // 576 (v6) or 216 (v7)
  const int RW = SW + TW;           // floats of a staged row (self obs + one task block)
  const int W = SW + TW * T;

  for (int q = 1; q <= T; ++q) {
    cp_async_wait_all();
    __syncthreads();  // frames(q) landed
    RefBody r;
    if (valid) r = blend_ref<EPB>(S, q, e, b);
    __syncthreads();  // frame buffer dead -> becomes the obs stage

    float* row = S.buf + e * STAGE_FLOATS;  // staged rows keep the 934-float pitch whatever the flags
    if (valid) {
      if (q == 1) emit_self_obs<false>(row, p.of, b, root_pos, hi, hr, pos, rot, vel, ang);
      emit_task<false>(p.of.v7, row + SW, b, hi, hr, root_pos, pos, rot, vel, ang, r);
    }
    __syncthreads();  // stage complete

    // stream the staged columns out: q == 1 -> cols [0, RW), else [SW + TW(q-1), +TW)
    const int s_off = q == 1 ? 0 : SW;
    const int s_len = q == 1 ? RW : TW;
    const int64_t c_off = q == 1 ? 0 : SW + (int64_t)TW * (q - 1);
    if (p.obs_vec2 && (SW & 1) == 0) {
      if (T == 1 && RW == STAGE_FLOATS && p.obs_stride == STAGE_FLOATS && !p.env_mask) {  // rows of the block are one contiguous span
        float2* dst = reinterpret_cast<float2*>(p.obs + env0 * STAGE_FLOATS);
        const float2* src = reinterpret_cast<const float2*>(S.buf);
        for (int i = tid; i < nvalid * (STAGE_FLOATS / 2); i += NT) dst[i] = src[i];
      } else {
        for (int ee = 0; ee < nvalid; ++ee) {
          if (!S.act[ee]) continue;
          float2* dst = reinterpret_cast<float2*>(p.obs + (env0 + ee) * p.obs_stride + c_off);
          const float2* src = reinterpret_cast<const float2*>(S.buf + ee * STAGE_FLOATS + s_off);
          for (int i = tid; i < s_len / 2; i += NT) dst[i] = src[i];
        }
      }
    } else {
      for (int ee = 0; ee < nvalid; ++ee) {
        if (!S.act[ee]) continue;
        float* dst = p.obs + (env0 + ee) * p.obs_stride + c_off;
        const float* src = S.buf + ee * STAGE_FLOATS + s_off;
        for (int i = tid; i < s_len; i += NT) dst[i] = src[i];
      }
    }

    if (p.moments) {  // RunningNorm partials: per-column fp64 sum / sum of squares over the block's envs
      for (int c = tid; c < s_len; c += NT) {
        double s1 = 0.0, s2 = 0.0;
        for (int ee = 0; ee < nvalid; ++ee) {
          if (!S.act[ee]) continue;
          const double x = (double)S.buf[ee * STAGE_FLOATS + s_off + c];
          s1 += x;
          s2 += x * x;
        }
        double* mom = p.moments + (int64_t)(blockIdx.x % p.moment_buckets) * 2 * W;
        atomicAdd(mom + c_off + c, s1);
        atomicAdd(mom + W + c_off + c, s2);
      }
    }
    if (p.obs_norm) {  // RunningNorm.forward of the same staged columns
      for (int c = tid; c < s_len; c += NT) {
        float m, sd, r;
        norm_column(p, c_off + c, m, sd, r);
        for (int ee = 0; ee < nvalid; ++ee) {
          if (!S.act[ee]) continue;
          const float v = norm_value(S.buf[ee * STAGE_FLOATS + s_off + c], m, sd, r, p.norm_clip);
          const int64_t at = (env0 + ee) * p.obs_norm_stride + c_off + c;
          if (p.norm_bf16) reinterpret_cast<__nv_bfloat16*>(p.obs_norm)[at] = __float2bfloat16_rn(v);
          else p.obs_norm[at] = v;
        }
      }
    }

    if (q < T) {
      __syncthreads();  // stage drained before the next frames overwrite it
      load_frames<EPB>(p.L, S, q + 1, e, b, valid);
    }
  }
  cp_async_wait_all();
}

// the columns of an observation row that thread `b` of an env writes: f(first column, count)
template <class F>
__device__ __forceinline__ void for_owned_columns(int b, int hcol, int SW, int T, bool v7, F f) {
  if (b == 0) {
    if (hcol) f(0, 1);
  } else {
    f(hcol + (b - 1) * 3, 3);
  }
  f(hcol + 69 + b * 6, 6);
  f(hcol + 213 + b * 3, 3);
  f(hcol + 285 + b * 3, 3);
  for (int q = 1; q <= T; ++q) {
    if (v7) {
      const int base = SW + TASK_DIM_V7 * (q - 1);
      f(base + b * 3, 3);
      f(base + 72 + b * 3, 3);
      f(base + 144 + b * 3, 3);
      continue;
    }
    const int base = SW + TASK_DIM * (q - 1);
    f(base + b * 3, 3);
    f(base + 72 + b * 6, 6);
    f(base + 216 + b * 3, 3);
    f(base + 288 + b * 3, 3);
    f(base + 360 + b * 3, 3);
    f(base + 432 + b * 6, 6);
  }
}

// Reset of the flagged envs and their observations in ONE launch (phc_reset_envs).  A thread scatters the new state
// of its (env, body) and, with that state still in registers, writes the body's columns of the env's obs row
// (_compute_observations(env_ids), :937-961): the root position and heading come from body 0 through shared memory,
// the reference bodies at t + q dt straight from the motion library.  The arithmetic is the generic step kernel's,
// operand for operand (the clock of a just-reset env: progress 0, offsets 0), so the rows are bit-identical to an
// obs-only pass of step_kernel over the new state; the chain of dependent memory round trips is less than half as
// long.  The mask byte is read once, first, so it may be reset_buf itself; blocks without a flagged env leave at once —
// with nothing flagged the launch reads n mask bytes and nothing else.
// The step's fused epilogues stay consistent with the rewritten rows: the normalised copy of the row is rewritten
// too (norm.out), and the RunningNorm partials either gain the new row (moments_mode 1: rows that were never
// counted) or have the row the step had counted replaced by it (mode 2).
__global__ void __launch_bounds__(K7_EPB* J24) reset_obs_kernel(const ResetParams p) {
  __shared__ float s_root[K7_EPB][5];  // root pos xyz | inverse heading z, w
  const int e = threadIdx.x / J24, b = threadIdx.x % J24;
  const int64_t env = (int64_t)blockIdx.x * K7_EPB + e;
  const bool act = env < p.n && p.mask[env] != 0;
  if (!__syncthreads_or(act)) return;
  ResetEnvOut o;
  reset_scatter_body(p, act, o);
  if (act && b == 0) {
    const Heading h0 = heading_quat_inv(heading_source(o.rot, p.of.upright));  // common.py:42-47
    s_root[e][0] = o.pos.x, s_root[e][1] = o.pos.y, s_root[e][2] = o.pos.z;
    s_root[e][3] = h0.z, s_root[e][4] = h0.w;
  }
  __syncthreads();
  if (!act) return;
  const Vec3 root_pos = {s_root[e][0], s_root[e][1], s_root[e][2]};
  const Heading hi = {s_root[e][3], s_root[e][4]};
  const HeadingRot hr = heading_rot(hi);
  float* row = p.obs + env * p.obs_stride;
  const int SW = 357 + p.of.hcol, TW = task_width(p.of), W = SW + TW * p.T;
  double* mom = p.moments ? p.moments + (int64_t)(blockIdx.x % p.moment_buckets) * 2 * W : nullptr;
  if (mom && p.moments_mode == 2) {  // the step that flagged this env counted the row it wrote: take it out again
    for_owned_columns(b, p.of.hcol, SW, p.T, p.of.v7, [&](int c0, int n) {
      for (int c = c0; c < c0 + n; ++c) {
        const double x = (double)__ldcg(row + c);
        atomicAdd(mom + c, -x);
        atomicAdd(mom + W + c, -(x * x));
      }
    });
  }
  emit_self_obs<false>(row, p.of, b, root_pos, hi, hr, o.pos, o.rot, o.vel, o.ang);
  if (p.ref_dof_pos && b >= 1) {  // self.ref_dof_pos[env_ids] = dof_pos of the query at t + dt (humanoid_phc.py:1115-1120)
    int64_t f0, f1;
    float bl;
    reset_query_frames(1, p.dt, o.t, o.len, o.nf, o.mdt, o.st, f0, f1, bl, o.soff);
    const Quat lr = quat_slerp(ld4v(p.L.lrs + (f0 * J24 + b) * 4), ld4v(p.L.lrs + (f1 * J24 + b) * 4), bl);
    st3(p.ref_dof_pos + env * p.ref_dof_pos_stride + (b - 1) * 3, quat_exp_map(lr));
  }
  for (int q = 1; q <= p.T; ++q) {
    // loading the t + dt frames together with the scatter's (before its stores) was measured: 10 more registers,
    // 3 instead of 4 blocks per SM — 0.6 us faster per loop step at 4 % flagged, 2.5 us slower at 31 %; not kept
    const RefBody r = reset_ref_body(p.L, q, p.dt, o.t, o.len, o.nf, o.mdt, o.st, b, o.soff, o.g0, o.g1, o.g2);
    emit_task<false>(p.of.v7, row + SW + (int64_t)TW * (q - 1), b, hi, hr, root_pos, o.pos, o.rot, o.vel, o.ang, r);
  }
  if (mom || p.norm.out) {  // the thread's own stores above are visible to it
    for_owned_columns(b, p.of.hcol, SW, p.T, p.of.v7, [&](int c0, int n) {
      for (int c = c0; c < c0 + n; ++c) {
        const float v = row[c];
        if (mom) {
          const double x = (double)v;
          atomicAdd(mom + c, x);
          atomicAdd(mom + W + c, x * x);
        }
        if (p.norm.out) {  // policies/running_norm.py:15-20, the step kernels' arithmetic
          float m, sd, r;
          norm_column(p.norm.mean, p.norm.var, p.norm.eps, c, m, sd, r);
          const float y = norm_value(v, m, sd, r, p.norm.clip);
          const int64_t at = env * p.norm.stride + c;
          if (p.norm.bf16) reinterpret_cast<__nv_bfloat16*>(p.norm.out)[at] = __float2bfloat16_rn(y);
          else p.norm.out[at] = y;
        }
      }
    });
  }
}

// ---------------------------------------------------------------------------------------
// K6-fast: the fused step for T == 1 on the AoS sim tensor with a dense obs_buf — the
// configuration the env runs (humanoid_phc.py:1100) and the benchmark measures.
//
//   * launched with programmatic stream serialization; before griddepcontrol.wait warp 0 only
//     speculates on immutable data (frame blends for the candidate progress values, frames copied
//     into shared memory by TMA); after the wait it re-reads the clock, validates, fetches the
//     sim rows and selects (see "phase 0" in the kernel);
//   * all bulk data movement is TMA (cp.async.bulk, SASS UBLKCP) completing on one mbarrier: one
//     copy for the block's sim rows, one per env for its span of packed frame rows;
//   * 24 threads per env do the per-body math out of shared memory; reward means and the
//     termination test are reduced by warp 0 in ATen's summation order, after the store;
//   * the 934-float obs rows of the block are assembled in shared memory (aliasing the frame
//     buffer) and leave with ONE cp.async.bulk shared->global store.
// ---------------------------------------------------------------------------------------
template <int EPB>
struct FastSmem {
  float sim[EPB * ROW13];
  float frames[EPB * 4 * FRAME_FLOATS];  // [env][slot 0..3][312]; later the obs stage [env][934]
  float part[6][EPB][J24];  // reward partials x4, distance, power
  unsigned long long bar;
  float bl[2][EPB];
  int slot[2][2][EPB];
  float goff[EPB][4];
  float hz[EPB], hw[EPB];
  int prog[EPB], pass[EPB], fallen[EPB];
  int parity;  // phase of `bar` the consumers wait for
  // clip metadata of the block's envs (the in-step reset samples a new start time from it) and the library rows of
  // the query at t + dt (ref_dof_pos reads the local rotations of the same two frames)
  float meta_len[EPB], meta_mdt[EPB];
  int meta_nf[EPB];
  int64_t meta_st[EPB];
  int64_t row1[2][EPB];
  int rst[EPB];          // env is reset inside this launch
  float nroot[EPB][5];   // root position and inverse heading of a just-reset env
};

__device__ __forceinline__ RefBody blend_ref3(const float* f0, const float* f1, float bl, float g0, float g1, float g2, int b);
__device__ __forceinline__ RefBody blend_ref2(const float* f0, const float* f1, float bl, const float* goff, int b) {
  return blend_ref3(f0, f1, bl, goff[0], goff[1], goff[2], b);
}
__device__ __forceinline__ RefBody blend_ref3(const float* f0, const float* f1, float bl, float g0, float g1, float g2, int b) {
  const float om = 1.0f - bl;
  RefBody r;
  r.pos = lerp3(om, bl, ld3(f0 + b * 3), ld3(f1 + b * 3));
  r.pos.x += g0;
  r.pos.y += g1;
  r.pos.z += g2;
  r.rot = quat_slerp(ld4v(f0 + 72 + b * 4), ld4v(f1 + 72 + b * 4), bl);
  r.vel = lerp3(om, bl, ld3(f0 + 168 + b * 3), ld3(f1 + 168 + b * 3));
  r.ang = lerp3(om, bl, ld3(f0 + 240 + b * 3), ld3(f1 + 240 + b * 3));
  return r;
}

// blend_ref2 of two queries at once, in fp32x2 instructions: r0 equals blend_ref2(f00, f01, bl.x, goff, b) and r1
// blend_ref2(f10, f11, bl.y, goff, b), bit for bit
__device__ __forceinline__ void blend_ref_pair(const float* f00, const float* f01, const float* f10, const float* f11,
                                               float2 bl, const float* goff, int b, float one, RefBody& r0, RefBody& r1) {
  const float2 om = {1.0f - bl.x, 1.0f - bl.y};
  Vec3x2 pos = lerp3x2(om, bl, pack3(ld3(f00 + b * 3), ld3(f10 + b * 3)), pack3(ld3(f01 + b * 3), ld3(f11 + b * 3)), one);
  pos.x = add2(pos.x, bc2(goff[0]), one);
  pos.y = add2(pos.y, bc2(goff[1]), one);
  pos.z = add2(pos.z, bc2(goff[2]), one);
  const Vec3x2 vel = lerp3x2(om, bl, pack3(ld3(f00 + 168 + b * 3), ld3(f10 + 168 + b * 3)),
                             pack3(ld3(f01 + 168 + b * 3), ld3(f11 + 168 + b * 3)), one);
  const Vec3x2 ang = lerp3x2(om, bl, pack3(ld3(f00 + 240 + b * 3), ld3(f10 + 240 + b * 3)),
                             pack3(ld3(f01 + 240 + b * 3), ld3(f11 + 240 + b * 3)), one);
  quat_slerp_pair(ld4v(f00 + 72 + b * 4), ld4v(f01 + 72 + b * 4), ld4v(f10 + 72 + b * 4), ld4v(f11 + 72 + b * 4), bl,
                  r0.rot, r1.rot);
  r0.pos = lane0(pos), r0.vel = lane0(vel), r0.ang = lane0(ang);
  r1.pos = lane1(pos), r1.vel = lane1(vel), r1.ang = lane1(ang);
}

// The reset of the envs a step flags, inside the step (PhcStepArgs.auto_reset; clean_pufferl/env.py:133-135 ->
// humanoid_phc.py:665-676).  Called by EVERY thread of a block that has a flagged env, once per flagged env, after
// phase 2 (the frame buffer is the stage by now, the threads' own per-body state is dead).  A block with a flagged
// env is what a single-wave step waits for, and its length is a dependent instruction chain, not bandwidth — so the
// work of ONE flagged env is spread over the block's three warps by ROLE, lane = body:
//   warp 0  the env's new state at the start time (get_motion_state, posed with the OLD global offset), the
//           _set_env_state scatter, the clock; publishes the state in the env's (dead) row of the sim tile and the
//           root position / inverse heading; after the block barrier: the self-observation columns of the new row
//   warp 1  the reference body at the new t + dt; after the barrier: the imitation columns (state from the sim tile)
//   warp 2  dof_pos (slerp of the local rotations + exp-map) and dof_vel of the new state; ref_dof_pos if asked for
// Every value is computed by the same functions on the same operands as phc_reset_envs computes it: bit-identical.
// Measured (profiles/r2_step_variants.md, 4096 envs, step with bookkeeping 7.9 us): the env's own 24 threads doing
// all of it one after the other (first version) 16.3 us whatever the fraction flagged; by role 11.7 us at 1 %
// flagged, 18.0 us at 46 % (blocks with several flagged envs take them one after the other; first version 17.1).
// Sharing the tasks of ALL flagged envs of a block out over the warps (state handed over through shared memory
// instead of registers, one barrier per block): 12.4 / 18.7 us, not kept.  The library rows are L2-prefetched
// (reset_prefetch) before phase 2, which covers their latency.
// (Out of line it was a disaster twice over: with the caller's per-body state passed by reference that state lived in
// local memory for the whole kernel, 7.8 -> 46 us per 4096-env step; with the kernel parameters passed by reference,
// 19 us.)
template <int EPB>
__device__ __forceinline__ void reset_prefetch(const StepParams& p, const FastSmem<EPB>& S, int f, int64_t env) {
  // warps 0 / 1, one lane each: both library rows of the state at t / of the reference at t + dt as one L2 prefetch
  // of the packed table; warp 2: the local rotations / dof velocities lane by lane
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float len = S.meta_len[f];
  const float t = reset_start_time(p.rw, env, len);
  int64_t f0, f1;
  float bl;
  reset_query_frames32(w == 1 ? 1 : 0, p.dt, t, len, S.meta_nf[f], S.meta_mdt[f], S.meta_st[f], f0, f1, bl);
  if (w < 2) {
    if (lane == 0) {
      const uint32_t bytes = (uint32_t)(f1 - f0 + 1) * (uint32_t)(FRAME_FLOATS * 4);
      asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;\n" ::"l"(p.L.packed + f0 * FRAME_FLOATS), "r"(bytes) : "memory");
    }
  } else if (lane < J24) {
    asm volatile("prefetch.global.L2 [%0];\n" ::"l"(p.L.lrs + (f0 * J24 + lane) * 4) : "memory");
    asm volatile("prefetch.global.L2 [%0];\n" ::"l"(p.L.lrs + (f1 * J24 + lane) * 4) : "memory");
    if (lane < 23) {
      asm volatile("prefetch.global.L2 [%0];\n" ::"l"(p.L.dvs + (f0 * 23 + lane) * 3) : "memory");
      asm volatile("prefetch.global.L2 [%0];\n" ::"l"(p.L.dvs + (f1 * 23 + lane) * 3) : "memory");
    }
  }
}

__device__ __forceinline__ void put13(float* d, Vec3 pos, Quat rot, Vec3 vel, Vec3 ang) {
  d[0] = pos.x, d[1] = pos.y, d[2] = pos.z;
  d[3] = rot.x, d[4] = rot.y, d[5] = rot.z, d[6] = rot.w;
  d[7] = vel.x, d[8] = vel.y, d[9] = vel.z;
  d[10] = ang.x, d[11] = ang.y, d[12] = ang.z;
}

template <int EPB, bool DEF, bool V7>
__device__ __forceinline__ void reset_in_step(const StepParams& p, FastSmem<EPB>& S, int f, int64_t env) {
  static_assert(EPB * J24 == 96, "three warps, one role each");
  const int w = threadIdx.x >> 5, b = threadIdx.x & 31;
  const bool act = b < J24;
  const float len = S.meta_len[f], mdt = S.meta_mdt[f];
  const int nf = S.meta_nf[f];
  const int64_t st = S.meta_st[f];
  const float t = reset_start_time(p.rw, env, len);
  RefBody own;  // warp 0: the new state; warp 1: the reference at t + dt
  if (act) {
    int64_t f0, f1;
    float bl;
    reset_query_frames32(w == 1 ? 1 : 0, p.dt, t, len, nf, mdt, st, f0, f1, bl);
    if (w < 2) {  // warp 0: posed with the old global offset; warp 1: with the zero the reset leaves
      const bool A = w == 0;
      own = blend_ref3(p.L.packed + f0 * FRAME_FLOATS, p.L.packed + f1 * FRAME_FLOATS, bl, A ? S.goff[f][0] : 0.0f,
                       A ? S.goff[f][1] : 0.0f, A ? S.goff[f][2] : 0.0f, b);
      if (A) {
        reset_store_body(p.rw, env, b, t, own.pos, own.rot, own.vel, own.ang, false);
        put13(S.sim + f * ROW13 + b * 13, own.pos, own.rot, own.vel, own.ang);
        if (b == 0) {
          if (p.progress_mirror) p.progress_mirror[env] = 0;
          const Heading h0 = heading_quat_inv(heading_source(own.rot, p.of.upright));
          S.nroot[f][0] = own.pos.x, S.nroot[f][1] = own.pos.y, S.nroot[f][2] = own.pos.z;
          S.nroot[f][3] = h0.z, S.nroot[f][4] = h0.w;
        }
      }
    } else {
      reset_store_dof(p.L, p.rw, env, b, f0, f1, bl);
      if (p.ref_dof_pos && b >= 1) {  // humanoid_phc.py:1115-1120 on the reset's _compute_task_obs(env_ids)
        int64_t g0, g1;
        float gl;
        reset_query_frames32(1, p.dt, t, len, nf, mdt, st, g0, g1, gl);
        const Quat lr = quat_slerp(ld4v(p.L.lrs + (g0 * J24 + b) * 4), ld4v(p.L.lrs + (g1 * J24 + b) * 4), gl);
        st3(p.ref_dof_pos + env * p.ref_dof_pos_stride + (b - 1) * 3, quat_exp_map(lr));
      }
    }
  }
  __syncthreads();
  if (!act || w == 2) return;
  const int SW = DEF ? SELF_DIM : p.selfw;
  const Vec3 root_pos = {S.nroot[f][0], S.nroot[f][1], S.nroot[f][2]};
  const Heading hi = {S.nroot[f][3], S.nroot[f][4]};
  const HeadingRot hr = heading_rot(hi);
  float* row = S.frames + f * (SW + (V7 ? TASK_DIM_V7 : TASK_DIM));
  if (w == 0) {
    emit_self_obs<DEF>(row, p.of, b, root_pos, hi, hr, own.pos, own.rot, own.vel, own.ang);
  } else {
    const float* d = S.sim + f * ROW13 + b * 13;
    const Vec3 pos{d[0], d[1], d[2]}, vel{d[7], d[8], d[9]}, ang{d[10], d[11], d[12]};
    const Quat rot{d[3], d[4], d[5], d[6]};
    if constexpr (V7) emit_task_obs_v7(row + SW, b, hi, hr, root_pos, pos, rot, vel, ang, own);
    else emit_task_obs<DEF>(row + SW, b, hi, hr, root_pos, pos, rot, vel, ang, own);
  }
}

// NORM: compiled with the RunningNorm.forward epilogue (obs_norm set); the plain instantiation carries none of it
// EP: compiled with the wrapper's episode bookkeeping in the reduction warp (used when ep_returns is set)
// RESET: compiled with the in-step reset of the flagged envs (used when reset_on is set)
// DEF: the env's default self-obs flags (height column, local root, upright): constant columns, 934-float rows
// PLAIN: compiled without the per-step options — power reward, ref_dof_pos, mpjpe, eval mode (use_mean), RunningNorm
// moments, rew_out, progress_mirror — and with goff set: the headline step issues their run-time branches in its
// issue-bound phases, and the eval-mode selection arrays are most of its stack frame
// V7: the v7 task block (PHC_OBS_TASK_V7, 216 floats): rows of SW + 216 floats in the stage, the stores and the moments
template <int EPB, int MINB, bool NORM = false, bool EP = false, bool RESET = false, bool DEF = true, bool PLAIN = false,
          bool V7 = false>
__global__ void __launch_bounds__(EPB* J24, MINB) step_fast_kernel(const __grid_constant__ StepParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  FastSmem<EPB>& S = *reinterpret_cast<FastSmem<EPB>*>(smem_raw);
  constexpr int NT = EPB * J24;
  static_assert(4 * EPB <= 32, "reductions run on one warp");
  static_assert(!NORM || DEF, "the normaliser epilogue is laid out for the default 934-float rows");
  static_assert(!PLAIN || (!NORM && !EP && !RESET && DEF), "the plain step carries none of the epilogues");
  static_assert(!NORM || !V7, "the normaliser epilogue is laid out for v6 rows");
  const bool use_mean = !PLAIN && p.use_mean;
  const bool dof_force = !PLAIN && p.dof_force;
  const bool ref_dof_pos = !PLAIN && p.ref_dof_pos;
  const bool moments = !PLAIN && p.moments;
  const int tid = threadIdx.x;
  const int64_t env0 = (int64_t)blockIdx.x * EPB;
  const int nvalid = p.n <= env0 ? 0 : (int)((p.n - env0) < EPB ? (p.n - env0) : EPB);
  PHC_STAMP(0);

  // ---- phase 0: clock, frame-blend, TMA loads ---------------------------------------------------
  // The kernel is launched with programmatic stream serialization: everything before
  // griddepcontrol.wait overlaps the tail of whatever kernel precedes it in the stream.  That
  // part only SPECULATES, and only on immutable data: 3 lanes per env read the clock as it is
  // now and run the frame blend for progress+1, +2, +3 (this step's two query times, whether or
  // not the previous step's increment has landed yet); when the frames of all three fit the env's
  // four slots they are copied into shared memory right away (frame rows never change).  After
  // the wait the sim rows are fetched at once and the clock is re-read in one round of loads; if
  // motion id, start time and offset are unchanged and progress moved by 0 or 1 the pre-loaded
  // frames and precomputed blends are simply selected, otherwise the env's leader lane redoes
  // its blends and copies.  No caller contract is needed: every dependent read (sim state,
  // progress) and every write happens after the wait.
  // A launch that may not speculate at all (first_wave_blocks == 0: the library was just (re)written on this stream,
  // or the I/O is mapped host memory) releases its dependents only AFTER its own wait: the next step's pre-wait
  // reads of the library are then ordered behind everything this launch was ordered behind.
  if (p.first_wave_blocks > 0) asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
  // blocks beyond the first wave start after the dependency is long resolved: nothing to overlap
  const bool speculate = blockIdx.x < (unsigned)p.first_wave_blocks;
  // only the blocks dispatched into the slots the previous step leaves free run this early enough to find progress not
  // yet advanced; the others enter as the previous step's blocks exit, long after it was written
  const bool spec4 = blockIdx.x < (unsigned)p.spec4_blocks;
  if (tid < 32) {
    static_assert(EPB == 4, "phase 0 maps 8 lanes to each of 4 envs");
    if (tid == 0) mbar_init(&S.bar, 1);
    __syncwarp();
    const int le = tid >> 3, j = tid & 7;
    const bool act = le < nvalid;
    const bool lead = act && j == 0;
    const int64_t env = env0 + (act ? le : 0);
    const int adv = p.advance ? 1 : 0;
    float* fr = S.frames + le * (4 * FRAME_FLOATS);
    // -- speculation (lanes j < 3 of each env)
    int64_t sid = -1, st = 0;
    int nf = 2, sprog = 0;
    float len = 1.0f, mdt = 1.0f, sstart = 0.0f, ssoff = 0.0f;
    int c_f0 = 0, c_f1 = 0;  // clip-local candidate frames for progress + adv + j
    float c_bl = 0.0f, c_t = 0.0f;
    if (speculate && act && j < 3) {
      sid = p.ids[env];
      sprog = (int)p.progress[env];
      sstart = p.start[env];
      ssoff = p.start_off[env];
      if (p.spec_fault) {  // test hook: pretend the clock was different when speculated
        if (p.spec_fault & 1) sprog -= 1;               // previous step's increment not landed yet
        if (p.spec_fault & 2) sstart += 1.0f / 30.0f;   // env was reset in between
        if (p.spec_fault & 4) sprog -= 2;               // progress moved by more than one
        if (p.spec_fault & 8) sid += 1;                 // env was re-assigned a clip
      }
      const int64_t c = sid < 0 ? 0 : (sid >= p.L.M ? p.L.M - 1 : sid);  // stale garbage must not fault
      len = p.L.len[c];
      nf = (int)p.L.nf[c];
      mdt = p.L.mdt[c];
      st = p.L.starts[c];
      c_t = (float)(int16_t)(sprog + adv + j) * p.dt + sstart + ssoff;
      calc_frame_blend32(c_t, len, nf, mdt, c_f0, c_f1, c_bl);
    }
    // Slots hold 4 frames.  Candidates 0..1 serve "progress unchanged since speculation" (the
    // usual case: the previous step wrote progress long before this block started), 1..2 serve
    // "moved by one".  Blocks in spare slots (spec4) copy the frames of all three when they fit;
    // the others copy those of the first two, and fetch the rest after validation if progress
    // moved by one after all (slot = frame - s_lo either way).
    const int hi1 = __shfl_sync(0xffffffffu, c_f1, (tid & ~7) + 1);
    const int hi2 = __shfl_sync(0xffffffffu, c_f1, (tid & ~7) + 2);
    const int s_lo = c_f0;  // on the leader: candidate 0's first frame
    const bool all3 = hi2 - s_lo <= 3 && hi2 >= hi1;
    const int s_hi = all3 && spec4 ? hi2 : hi1;
    const bool spec = speculate && lead && s_hi - s_lo <= 3 && s_hi >= s_lo;
    if (spec) {  // frames of the speculated candidates -> slots 0..(hi-lo)
      const uint32_t bytes = (uint32_t)(s_hi - s_lo + 1) * (uint32_t)(FRAME_FLOATS * 4);
      mbar_expect_tx(&S.bar, bytes);
      bulk_g2s(fr, p.L.packed + (st + s_lo) * FRAME_FLOATS, bytes, &S.bar);
    }
    const bool block_sim = p.body.pos.stride_env == ROW13;  // the block's sim rows are one span
    if (speculate && lead && (block_sim ? le == 0 : true)) {
      // warm L2 with the sim rows: L2 is the point of coherence, so whoever writes them before the
      // dependency resolves updates the same lines
      const uint32_t bytes = (block_sim ? (uint32_t)nvalid : 1u) * (uint32_t)(ROW13 * 4);
      asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;\n" ::"l"(p.body.pos.ptr + env * p.body.pos.stride_env),
                   "r"(bytes)
                   : "memory");
    }
    asm volatile("griddepcontrol.wait;\n" ::: "memory");
    if (p.first_wave_blocks <= 0) asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
    PHC_STAMP(2);
    // -- dependent data: one round of clock loads, the sim rows' copy issued under them
    int prog_in = 0, dd = 0;
    bool ok = false;
    float start = 0.0f, soff = 0.0f, g0 = 0.0f, g1 = 0.0f, g2 = 0.0f;
    int64_t id = 0;
    if (lead) {  // .cg: these addresses may have been read before the wait; never trust L1 for them
      prog_in = (int)__ldcg(p.progress + env);
      id = __ldcg(p.ids + env);
      start = __ldcg(p.start + env);
      soff = __ldcg(p.start_off + env);
      if (PLAIN || p.goff) {
        g0 = __ldcg(p.goff + env * 3 + 0);
        g1 = __ldcg(p.goff + env * 3 + 1);
        g2 = __ldcg(p.goff + env * 3 + 2);
      }
      if (block_sim ? le == 0 : true) {  // sim rows: issued while the clock loads are in flight
        const uint32_t bytes = (block_sim ? (uint32_t)nvalid : 1u) * (uint32_t)(ROW13 * 4);
        mbar_expect_tx(&S.bar, bytes);
        bulk_g2s(S.sim + le * ROW13, p.body.pos.ptr + env * p.body.pos.stride_env, bytes, &S.bar);
      }
      dd = prog_in - sprog;
      ok = speculate && id == sid && __float_as_uint(start) == __float_as_uint(sstart) &&
           __float_as_uint(soff) == __float_as_uint(ssoff) && (dd == 0 || (dd == 1 && all3));
    }
    const int d = (prog_in - sprog) & 1;  // meaningful on leaders with ok
    const int src0 = (tid & ~7) + d, src1 = src0 + 1;
    int a_f0 = __shfl_sync(0xffffffffu, c_f0, src0), a_f1 = __shfl_sync(0xffffffffu, c_f1, src0);
    int b_f0 = __shfl_sync(0xffffffffu, c_f0, src1), b_f1 = __shfl_sync(0xffffffffu, c_f1, src1);
    float a_bl = __shfl_sync(0xffffffffu, c_bl, src0), b_bl = __shfl_sync(0xffffffffu, c_bl, src1);
    float a_t = __shfl_sync(0xffffffffu, c_t, src0);
    // a leader whose pre-loaded frames cannot be used has to wait for them to land before it
    // overwrites the slots: rare, handled with a second phase of the same mbarrier
    const bool redo = lead && spec && !ok;
    const unsigned any_redo = __ballot_sync(0xffffffffu, redo);
    if (any_redo) {
      if (tid == 0) mbar_arrive(&S.bar);
      mbar_wait(&S.bar, 0);
    }
    if (lead) {
      int prog = prog_in;
      if (p.advance) prog = (int)(int16_t)(prog + 1);
      if (!ok) {  // no (usable) speculation: first-wave miss, or a later-wave block
        len = p.L.len[id];
        nf = (int)p.L.nf[id];
        mdt = p.L.mdt[id];
        st = p.L.starts[id];
        // q = 0: t = progress*dt + start + offset (humanoid_phc.py:1236); q = 1: (progress+1)*dt + ..
        // (humanoid_phc.py:1063-1067), progress already advanced (humanoid_phc.py:138)
        a_t = (float)(int16_t)prog * p.dt + start + soff;
        calc_frame_blend32(a_t, len, nf, mdt, a_f0, a_f1, a_bl);
        const float t1 = (float)(int16_t)(prog + 1) * p.dt + start + soff;
        calc_frame_blend32(t1, len, nf, mdt, b_f0, b_f1, b_bl);
      }
      S.bl[0][le] = a_bl;
      S.bl[1][le] = b_bl;
      S.prog[le] = prog;
      S.pass[le] = a_t >= len;  // _compute_reset, humanoid_phc.py:1317
      S.fallen[le] = 0;
      if (p.advance) {
        p.progress[env] = (int16_t)prog;
        if (!PLAIN && p.progress_mirror) p.progress_mirror[env] = (int16_t)prog;
      }
      S.goff[le][0] = g0;
      S.goff[le][1] = g1;
      S.goff[le][2] = g2;
      if (RESET) {
        S.meta_len[le] = len, S.meta_mdt[le] = mdt, S.meta_nf[le] = nf, S.meta_st[le] = st;
      }
      if (ref_dof_pos) S.row1[0][le] = st + b_f0, S.row1[1][le] = st + b_f1;
      if (ok && spec) {  // frames are already (arriving) in the slots
        S.slot[0][0][le] = a_f0 - s_lo;
        S.slot[0][1][le] = a_f1 - s_lo;
        S.slot[1][0][le] = b_f0 - s_lo;
        S.slot[1][1][le] = b_f1 - s_lo;
        if (dd == 1 && s_hi < hi2) {  // moved by one in a block that speculated on two candidates: rows s_hi+1 .. hi2
          const uint32_t bytes = (uint32_t)(hi2 - s_hi) * (uint32_t)(FRAME_FLOATS * 4);
          mbar_expect_tx(&S.bar, bytes);
          bulk_g2s(fr + (s_hi - s_lo + 1) * FRAME_FLOATS, p.L.packed + (st + s_hi + 1) * FRAME_FLOATS, bytes, &S.bar);
        }
      } else {
        // frames of one clip are consecutive rows of the packed table: when the (up to four)
        // frames span <= 4 rows they arrive with ONE copy and slot = frame - first
        const float* tab = p.L.packed + st * FRAME_FLOATS;
        const int lo = a_f0 < b_f0 ? a_f0 : b_f0;
        int hi = a_f1 > b_f1 ? a_f1 : b_f1;
        hi = hi > a_f0 ? hi : a_f0;
        hi = hi > b_f0 ? hi : b_f0;
        if (hi - lo <= 3) {
          S.slot[0][0][le] = a_f0 - lo;
          S.slot[0][1][le] = a_f1 - lo;
          S.slot[1][0][le] = b_f0 - lo;
          S.slot[1][1][le] = b_f1 - lo;
          const uint32_t bytes = (uint32_t)(hi - lo + 1) * (uint32_t)(FRAME_FLOATS * 4);
          mbar_expect_tx(&S.bar, bytes);
          bulk_g2s(fr, tab + (int64_t)lo * FRAME_FLOATS, bytes, &S.bar);
        } else {  // two spans of one or two rows each (idx1 is idx0 or idx0 + 1)
          S.slot[0][0][le] = 0;
          S.slot[0][1][le] = a_f1 - a_f0;
          S.slot[1][0][le] = 2;
          S.slot[1][1][le] = 2 + (b_f1 - b_f0);
          const uint32_t ba = (uint32_t)(a_f1 - a_f0 + 1) * (uint32_t)(FRAME_FLOATS * 4);
          const uint32_t bb = (uint32_t)(b_f1 - b_f0 + 1) * (uint32_t)(FRAME_FLOATS * 4);
          mbar_expect_tx(&S.bar, ba + bb);
          bulk_g2s(fr, tab + (int64_t)a_f0 * FRAME_FLOATS, ba, &S.bar);
          bulk_g2s(fr + 2 * FRAME_FLOATS, tab + (int64_t)b_f0 * FRAME_FLOATS, bb, &S.bar);
        }
      }
    }
    __syncwarp();
    if (p.trace) {  // the block's phase-0 path, in warp 1's unused stamp 1 (profiles/trace_step.py)
      const unsigned fetch = __ballot_sync(0xffffffffu, lead && ok && spec && dd == 1 && s_hi < hi2);
      const unsigned fresh = __ballot_sync(0xffffffffu, lead && !spec);
      if (tid == 0)
        p.trace[((size_t)blockIdx.x * 3 + 1) * 8 + 1] =
            16u | (spec4 ? 1u : 0u) | (fetch ? 2u : 0u) | (any_redo ? 4u : 0u) | (fresh ? 8u : 0u);
    }
    if (tid == 0) {
      S.parity = any_redo ? 1 : 0;
      mbar_arrive(&S.bar);
    }
    PHC_STAMP(1);
  } else {
    asm volatile("griddepcontrol.wait;\n" ::: "memory");
    // warp 1, one lane per env: the heading quaternion straight from the root rotation in global
    // memory (floats 3..6 of the env's sim row), while warp 0 validates the clock
    if (tid >= 32 && tid < 32 + nvalid) {
      const int le = tid - 32;
      const float* rq = p.body.pos.ptr + (env0 + le) * p.body.pos.stride_env + 3;
      const Quat rq4 = Quat{__ldcg(rq), __ldcg(rq + 1), __ldcg(rq + 2), __ldcg(rq + 3)};
      const Heading h0 = heading_quat_inv(DEF ? rq4 : heading_source(rq4, p.of.upright));  // common.py:42-47
      S.hz[le] = h0.z;
      S.hw[le] = h0.w;
    }
  }
  __syncthreads();  // #1: slots / blends / heading / barrier state visible
  mbar_wait(&S.bar, (uint32_t)S.parity);
  PHC_STAMP(3);

  // ---- phase 1: per-body reference states, reward partials, distance ------------------------
  const int e = tid / J24, b = tid % J24;
  const bool valid = e < nvalid;
  Vec3 pos, vel, ang;
  Quat rot;
  RefBody r1;
  if (valid) {
    const float* d = S.sim + e * ROW13 + b * 13;
    pos = {d[0], d[1], d[2]};
    rot = {d[3], d[4], d[5], d[6]};
    vel = {d[7], d[8], d[9]};
    ang = {d[10], d[11], d[12]};
    const float* fr = S.frames + e * (4 * FRAME_FLOATS);
    // the reference bodies of both queries: r0 (t) feeds the reward and the distance, r1 (t + dt) the obs.  Paired
    // into fp32x2 instructions, except in the RESET instantiations, which spill with the paired math at 80 registers.
    RefBody r0;
    const float* f00 = fr + S.slot[0][0][e] * FRAME_FLOATS;
    const float* f01 = fr + S.slot[0][1][e] * FRAME_FLOATS;
    const float* f10 = fr + S.slot[1][0][e] * FRAME_FLOATS;
    const float* f11 = fr + S.slot[1][1][e] * FRAME_FLOATS;
    if constexpr (RESET) {
      r0 = blend_ref2(f00, f01, S.bl[0][e], S.goff[e], b);
      r1 = blend_ref2(f10, f11, S.bl[1][e], S.goff[e], b);
    } else {
      blend_ref_pair(f00, f01, f10, f11, make_float2(S.bl[0][e], S.bl[1][e]), S.goff[e], b, p.one, r0, r1);
    }
    {
      float sp, sr, sv, sa;
      reward_partials(pos, rot, vel, ang, r0, sp, sr, sv, sa);
      S.part[0][e][b] = sp;
      S.part[1][e][b] = sr;
      S.part[2][e][b] = sv;
      S.part[3][e][b] = sa;
      const float dist = norm3(pos - r0.pos);  // torch.norm(rigid_body_pos - ref_body_pos), common.py:343/348
      S.part[4][e][b] = dist;
      if (!use_mean && (p.reset_mask >> b & 1u) && dist > p.term_dist[b]) S.fallen[e] = 1;  // any(), benign race
      if (dof_force) S.part[5][e][b] = power_partial(p, env0 + e, b);
    }
  }
  PHC_STAMP(4);
  __syncthreads();  // #2: partials / heading visible; frame buffer dead -> becomes the obs stage

  // ---- in-step reset of the flagged envs (RESET) -------------------------------------------------
  // Every thread works out which of the block's envs this step flags (the test of the reduction warp below, from
  // the same shared-memory values); a block without one goes straight on.
  bool my_rst = false;
  int rst_mask = 0;  // bit i: env i of the block is reset inside this launch
  if constexpr (RESET) {
    if (p.reset_on) {
      if (p.use_mean) {  // eval mode: the mean needs ATen's row sum — one lane per env, then a block barrier
        if (tid < nvalid) {
          float sel[J24];
          int m = 0;
#pragma unroll
          for (int j = 0; j < J24; ++j)
            if (p.reset_mask >> j & 1u) sel[m++] = S.part[4][tid][j];
          const int first = __ffs(p.reset_mask) - 1;
          bool fallen = p.early && m > 0 && (aten_row_sum(sel, m) / (float)m) > p.term_dist[first < 0 ? 0 : first];
          fallen = fallen && (S.prog[tid] > 1);
          S.rst[tid] = (S.pass[tid] || fallen) ? 1 : 0;
        }
        __syncthreads();
      }
#pragma unroll
      for (int i = 0; i < EPB; ++i) {
        int r = 0;
        if (i < nvalid) r = p.use_mean ? S.rst[i] : ((S.pass[i] || (p.early && S.fallen[i] && S.prog[i] > 1)) ? 1 : 0);
        rst_mask |= r << i;
        if (i == e) my_rst = valid && r;
      }
      // the library rows the reset below will read: into L2 now, phase 2 covers their latency
#pragma unroll
      for (int i = 0; i < EPB; ++i)
        if (rst_mask >> i & 1) reset_prefetch<EPB>(p, S, i, env0 + i);
    }
  }

  // ---- phase 2: observations into the stage ---------------------------------------------------
  const int SW = DEF ? SELF_DIM : p.selfw;  // 358 with the root height column, 357 without
  const int RW = SW + (V7 ? TASK_DIM_V7 : TASK_DIM);  // floats of a staged row
  if (valid && !(RESET && my_rst)) {
    const Vec3 root_pos = {S.sim[e * ROW13 + 0], S.sim[e * ROW13 + 1], S.sim[e * ROW13 + 2]};
    const Heading hi = {S.hz[e], S.hw[e]};
    const HeadingRot hr = heading_rot(hi);
    float* row = S.frames + e * RW;
    if constexpr (RESET) {
      emit_self_obs<DEF>(row, p.of, b, root_pos, hi, hr, pos, rot, vel, ang);  // common.py:23-103
      if constexpr (V7) emit_task_obs_v7(row + SW, b, hi, hr, root_pos, pos, rot, vel, ang, r1);
      else emit_task_obs<DEF>(row + SW, b, hi, hr, root_pos, pos, rot, vel, ang, r1);  // common.py:106-176
    } else if constexpr (V7) {
      emit_obs_paired_v7<DEF>(row, SW, p.of, b, root_pos, hi, hr, pos, rot, vel, ang, r1, p.one);
    } else {
      emit_obs_paired<DEF>(row, SW, p.of, b, root_pos, hi, hr, pos, rot, vel, ang, r1, p.one);  // common.py:23-176
    }
  }
  if constexpr (RESET) {
    if (rst_mask) {  // the rows of the flagged envs, from their new state (one env at a time, the whole block on it)
#pragma unroll 1
      for (int i = 0; i < EPB; ++i)
        if (rst_mask >> i & 1) reset_in_step<EPB, DEF, V7>(p, S, i, env0 + i);
    }
  }
  fence_proxy_async();  // stage writes -> visible to the bulk-store engine
  PHC_STAMP(5);
  __syncthreads();      // #3: stage complete
  PHC_STAMP(6);

  const uint32_t out_bytes = (uint32_t)nvalid * (uint32_t)(RW * 4);
  const bool bulk_ok = (out_bytes & 15u) == 0;
  if (bulk_ok) {
    if (tid == NT - 1 && out_bytes) bulk_s2g(p.obs + env0 * RW, S.frames, out_bytes);
  } else if (DEF || ((nvalid * RW) & 1) == 0) {  // odd tail block: 8-byte stores
    float2* dst = reinterpret_cast<float2*>(p.obs + env0 * RW);
    const float2* src = reinterpret_cast<const float2*>(S.frames);
    for (int i = tid; i < nvalid * RW / 2; i += NT) dst[i] = src[i];
  } else {
    for (int i = tid; i < nvalid * RW; i += NT) p.obs[env0 * RW + i] = S.frames[i];
  }
  if (moments) {
    // RunningNorm partials: per-column fp64 sum / sum of squares of the block's staged rows, added to one of the
    // accumulator buckets: 1868 fp64 adds in L2 per block of four envs (1.9 M per 4096-env step: +3.8 us on a 6.7 us
    // step).  Two ways to cut that were built and measured in round 2 (profiles/r2_step_variants.md):
    //   * p.moments_bulk (PHC_OPT_MOMENTS_BULK, kept as an option): the block writes its 1868 partial sums into shared
    //     memory that is dead by now — the sim tile and the tail of the frame buffer behind the stage, 624 doubles
    //     each — and hands them to the TMA engine as THREE bulk reductions (cp.reduce.async.bulk .add.f64), so no SM
    //     issues an atomic.  10.95 us against 10.47 us for the atomics: the adds themselves, in L2, are the cost, not
    //     their issue.
    //   * a cluster of 8 CTAs pre-reducing over each other's staged rows through distributed shared memory (8x fewer
    //     L2 adds): 16.8 us (cluster of 4: 14.0, of 2: 12.7) — a cluster launch gang-schedules its CTAs and two cluster
    //     barriers sit at the tail of every block of a single-wave grid.  Removed.
    double* mom = p.moments + (int64_t)(blockIdx.x % p.moment_buckets) * 2 * RW;
    if (p.moments_bulk) {
      constexpr int CH = 624;  // doubles per region: min(sizeof sim, sizeof frames - stage) / 8, even
      static_assert(CH * 8 <= (int)sizeof(S.sim) && CH * 8 <= (int)sizeof(S.frames) - EPB * STAGE_FLOATS * 4, "regions");
      double* regA = reinterpret_cast<double*>(S.sim);
      double* regB = reinterpret_cast<double*>(S.frames + EPB * RW);
      const int total = 2 * RW;
      for (int c0 = 0, r = 0; c0 < total; c0 += CH, ++r) {
        double* reg = (r & 1) ? regB : regA;
        const int cnt = total - c0 < CH ? total - c0 : CH;
        if (r >= 2) {  // the region is being read by the reduction issued two rounds ago
          if (tid == 0) bulk_wait_read_all_but_one();
          __syncthreads();
        }
        for (int i = tid; i < cnt; i += NT) {
          const int g = c0 + i;
          const bool sq = g >= RW;
          const int col = sq ? g - RW : g;
          double acc = 0.0;
          for (int ee = 0; ee < nvalid; ++ee) {
            const double x = (double)S.frames[ee * RW + col];
            acc += sq ? x * x : x;
          }
          reg[i] = acc;
        }
        fence_proxy_async();
        __syncthreads();
        if (tid == 0) bulk_reduce_add_f64(mom + c0, reg, (uint32_t)cnt * 8u);
      }
      if (NORM && p.obs_norm) {  // the bf16 staging below reuses both regions
        if (tid == 0) bulk_wait_read();
        __syncthreads();
      }
    } else {
      for (int c = tid; c < RW; c += NT) {
        double s1 = 0.0, s2 = 0.0;
        for (int ee = 0; ee < nvalid; ++ee) {
          const double x = (double)S.frames[ee * RW + c];
          s1 += x;
          s2 += x * x;
        }
        atomicAdd(mom + c, s1);
        atomicAdd(mom + RW + c, s2);
      }
    }
  }
  // res_action: dof_pos of the query at t + dt (humanoid_phc.py:1115-1120), off the critical path; a just-reset env
  // got its row from the reset above
  if (ref_dof_pos && valid && !(RESET && my_rst))
    write_ref_dof_pos(p, env0 + e, b, S.row1[0][e], S.row1[1][e], S.bl[1][e]);
  // RunningNorm.forward, fp32 rows, full blocks: once the raw store has READ the stage, normalise it in place and
  // send it out with a second bulk store instead of 20 scattered 8-byte stores per thread
  const bool norm_inplace = NORM && p.obs_norm && bulk_ok && !p.norm_bf16;
  if (norm_inplace) {
    if (tid == NT - 1) bulk_wait_read();
    __syncthreads();
    float2* st = reinterpret_cast<float2*>(S.frames);
    for (int c2 = tid; c2 < STAGE_FLOATS / 2; c2 += NT) {
      float m0, sd0, r0, m1, sd1, r1;
      norm_column(p, 2 * c2, m0, sd0, r0);
      norm_column(p, 2 * c2 + 1, m1, sd1, r1);
      for (int ee = 0; ee < nvalid; ++ee) {
        const float2 x = st[ee * (STAGE_FLOATS / 2) + c2];
        st[ee * (STAGE_FLOATS / 2) + c2] =
            make_float2(norm_value(x.x, m0, sd0, r0, p.norm_clip), norm_value(x.y, m1, sd1, r1, p.norm_clip));
      }
    }
    fence_proxy_async();
    __syncthreads();
    if (tid == NT - 1) bulk_s2g(p.obs_norm + env0 * STAGE_FLOATS, S.frames, out_bytes);
  }
  // bf16 rows, full blocks: the four rows (7472 B) are packed into shared memory that is dead by now — the sim tile
  // and the tail of the frame buffer behind the stage — so nothing waits for the raw store; the split falls on
  // bf16 element 1864 so that both pieces are multiples of 16 B, and they leave with two bulk stores
  constexpr int NORM16_SPLIT = 932;  // pairs in the first piece: 3728 B, the second holds 936 pairs = 3744 B
  static_assert(EPB != 4 || (NORM16_SPLIT * 4 <= (int)sizeof(S.sim) && (EPB * STAGE_FLOATS / 2 - NORM16_SPLIT) * 4 <=
                                 (int)sizeof(S.frames) - EPB * STAGE_FLOATS * 4), "bf16 staging fits the dead regions");
  const bool norm16_staged =
      NORM && p.obs_norm && bulk_ok && p.norm_bf16 && nvalid == EPB && EPB == 4 && ((uintptr_t)p.obs_norm & 15) == 0;
  if (norm16_staged) {
    __nv_bfloat162* pa = reinterpret_cast<__nv_bfloat162*>(S.sim);
    __nv_bfloat162* pb = reinterpret_cast<__nv_bfloat162*>(S.frames + EPB * STAGE_FLOATS);
    const float2* src = reinterpret_cast<const float2*>(S.frames);
    for (int c2 = tid; c2 < STAGE_FLOATS / 2; c2 += NT) {
      float m0, sd0, r0, m1, sd1, r1;
      norm_column(p, 2 * c2, m0, sd0, r0);
      norm_column(p, 2 * c2 + 1, m1, sd1, r1);
#pragma unroll
      for (int ee = 0; ee < EPB; ++ee) {
        const int i = ee * (STAGE_FLOATS / 2) + c2;
        const float2 x = src[i];
        const __nv_bfloat162 y = __floats2bfloat162_rn(norm_value(x.x, m0, sd0, r0, p.norm_clip),
                                                       norm_value(x.y, m1, sd1, r1, p.norm_clip));
        if (i < NORM16_SPLIT) pa[i] = y;
        else pb[i - NORM16_SPLIT] = y;
      }
    }
    fence_proxy_async();
    __syncthreads();
    if (tid == NT - 1) {
      __nv_bfloat162* dst = reinterpret_cast<__nv_bfloat162*>(p.obs_norm) + env0 * (STAGE_FLOATS / 2);
      bulk_s2g(dst, pa, NORM16_SPLIT * 4);
      bulk_s2g(dst + NORM16_SPLIT, pb, (EPB * STAGE_FLOATS / 2 - NORM16_SPLIT) * 4);
    }
  }
  // ---- reductions and scalar outputs (warp 0), off the critical path: nothing waits for them -------------------------------------------------
  if (tid < 32) {
    const int le = tid >> 2, k = tid & 3;
    const bool act = le < nvalid && tid < 4 * EPB;
    float term_k = 0.0f;
    float ep_ret = 0.0f;  // EP: the env's running return / length, fetched before the reductions below need them
    int32_t ep_len = 0;
    if constexpr (EP) {
      if (p.ep_returns && act && k == 0) {
        ep_ret = p.ep_returns[env0 + le];
        ep_len = p.ep_lengths[env0 + le];
      }
    }
    if (act) {
      const float kk = k == 0 ? p.rwd.k_pos : k == 1 ? p.rwd.k_rot : k == 2 ? p.rwd.k_vel : p.rwd.k_ang_vel;
      term_k = expf((-kk) * (row_sum24(&S.part[k][le][0]) / 24.0f));  // common.py:298-320
      p.raw[(env0 + le) * p.raw_stride + k] = term_k;
    }
    const int base = tid & ~3;
    const float t0 = __shfl_sync(0xffffffffu, term_k, base), t1 = __shfl_sync(0xffffffffu, term_k, base + 1);
    const float t2 = __shfl_sync(0xffffffffu, term_k, base + 2), t3 = __shfl_sync(0xffffffffu, term_k, base + 3);
    float r = 0.0f, pr = 0.0f;  // lanes k == 0: the env's reward and its power term
    int flags = 0;              // lanes k == 1: bit 0 = reset, bit 1 = terminated
    if (act && k == 0) {
      r = p.rwd.w_pos * t0 + p.rwd.w_rot * t1 + p.rwd.w_vel * t2 + p.rwd.w_ang_vel * t3;
      if (dof_force) {
        pr = power_reward(p, &S.part[5][le][0], S.prog[le]);
        r += pr;  // rew_buf[:] += power_reward (humanoid_phc.py:1304)
        p.raw[(env0 + le) * p.raw_stride + p.power_col] = pr;
      }
      p.rew[env0 + le] = r;
      if (!PLAIN && p.rew_out) p.rew_out[env0 + le] = r;
    }
    if (act && k == 1) {
      bool fallen = false;
      if (p.early) {
        if (use_mean) {  // eval mode: mean distance of the selected bodies vs the first one's threshold
          float sel[J24];
          int m = 0;
#pragma unroll
          for (int j = 0; j < J24; ++j)
            if (p.reset_mask >> j & 1u) sel[m++] = S.part[4][le][j];
          const int first = __ffs(p.reset_mask) - 1;
          fallen = m > 0 && (aten_row_sum(sel, m) / (float)m) > p.term_dist[first < 0 ? 0 : first];
        } else {
          fallen = S.fallen[le] != 0;
        }
        fallen = fallen && (S.prog[le] > 1);  // common.py:353
      }
      const bool rs = S.pass[le] || fallen;  // common.py:362
      // with the in-step reset the flagged envs have been reset by now: reset_buf / terminate_buf read 0 afterwards
      // (_reset_env_tensors, humanoid_phc.py:775-778) and the step's flags live on in reset_out / terminate_out
      const bool cleared = RESET && p.reset_on;
      p.term[env0 + le] = (fallen && !cleared) ? 1 : 0;
      p.reset[env0 + le] = (rs && !cleared) ? 1 : 0;
      if (p.term_out) p.term_out[env0 + le] = fallen ? 1 : 0;
      if (p.reset_out) p.reset_out[env0 + le] = rs ? 1 : 0;
      flags = (rs ? 1 : 0) | (fallen ? 2 : 0);
    }
    if (!PLAIN && act && k == 2 && p.mpjpe) p.mpjpe[env0 + le] = row_sum24(&S.part[4][le][0]) / 24.0f;  // humanoid_phc.py:167
    if constexpr (EP) if (p.ep_returns) {
      // PHCPufferEnv.step's bookkeeping (clean_pufferl/env.py:121-159) for the block's envs, on the lanes that hold the
      // reward; the block's sums go to one of ep_buckets fp64 accumulators (atomics on one address serialise).  The sums
      // over the block's four envs are taken in fp32 — counts and lengths are exact there, a four-term sum of returns or
      // reward terms carries 1e-7, below the fp32 means the reference logs — because 24 fp64 shuffle-adds on this warp
      // cost a full microsecond per step at the tail of every block (measured: 8.5 -> 7.5 us per 4096-env step)
      flags = __shfl_sync(0xffffffffu, flags, base + 1);
      float v[EP_SUM_COLS];
#pragma unroll
      for (int i = 0; i < EP_SUM_COLS; ++i) v[i] = 0.0f;
      if (act && k == 0) {
        const int64_t e = env0 + le;
        const bool rs = flags & 1, tm = (flags & 2) != 0, tr = rs && !tm;
        p.ep_terminals[e] = tm ? 1 : 0;
        p.ep_truncations[e] = tr ? 1 : 0;
        p.ep_masks[e] = tr ? 0 : 1;
        float ret = ep_ret;
        int32_t len = ep_len;
        if (rs) {
          v[0] = 1.0f;
          v[1] = ret;
          v[2] = (float)len;
          v[3] = tr ? 1.0f : 0.0f;
          ret = 0.0f;
          len = 0;
        }
        p.ep_returns[e] = ret + r;
        p.ep_lengths[e] = len + 1;
        v[4] = t0, v[5] = t1, v[6] = t2, v[7] = t3;
        if (p.dof_force) {
#pragma unroll
          for (int i = 8; i < EP_SUM_COLS; ++i)
            if (i == 4 + p.power_col) v[i] = pr;
        }
      }
      // the four k == 0 lanes (0, 4, 8, 12) -> lane i keeps the sum of column i, then ONE atomic instruction for the row
      float mine = 0.0f;
#pragma unroll
      for (int i = 0; i < EP_SUM_COLS; ++i) {
        v[i] += __shfl_xor_sync(0xffffffffu, v[i], 4);
        v[i] += __shfl_xor_sync(0xffffffffu, v[i], 8);
        const float tot = __shfl_sync(0xffffffffu, v[i], 0);
        if (tid == i) mine = tot;
      }
      if (tid < 4 + p.ep_raw_cols && mine != 0.0f)
        atomicAdd(p.ep_sums + (int64_t)((p.ep_block0 + blockIdx.x) % p.ep_buckets) * EP_SUM_COLS + tid, (double)mine);
    }
  }

  if (NORM && p.obs_norm && !norm_inplace && !norm16_staged) {
    // RunningNorm.forward fused into the epilogue: the staged rows are read a second time (while the
    // bulk store drains them) and leave normalised with coalesced 8-byte stores; mean / var are 7.5 KB
    // that every block reads from L2
    float2* dst = reinterpret_cast<float2*>(p.obs_norm + env0 * STAGE_FLOATS);
    __nv_bfloat162* dst16 = reinterpret_cast<__nv_bfloat162*>(p.obs_norm) + env0 * (STAGE_FLOATS / 2);
    const float2* src = reinterpret_cast<const float2*>(S.frames);
    for (int c2 = tid; c2 < STAGE_FLOATS / 2; c2 += NT) {
      float m0, sd0, r0, m1, sd1, r1;
      norm_column(p, 2 * c2, m0, sd0, r0);
      norm_column(p, 2 * c2 + 1, m1, sd1, r1);
      for (int ee = 0; ee < nvalid; ++ee) {
        const float2 x = src[ee * (STAGE_FLOATS / 2) + c2];
        const float y0 = norm_value(x.x, m0, sd0, r0, p.norm_clip), y1 = norm_value(x.y, m1, sd1, r1, p.norm_clip);
        if (p.norm_bf16) dst16[ee * (STAGE_FLOATS / 2) + c2] = __floats2bfloat162_rn(y0, y1);  // half the bytes
        else dst[ee * (STAGE_FLOATS / 2) + c2] = make_float2(y0, y1);
      }
    }
  }
  if (bulk_ok && tid == NT - 1) bulk_wait_read();  // shared memory must outlive the store's reads
  if (moments && p.moments_bulk && tid == 0) bulk_wait_read();  // ... and the reductions'
  PHC_STAMP(7);
}

// ---------------------------------------------------------------------------------------
// K6-persist: the T = 1 fused step for grids of more than one wave (BASELINE config 3: 8192 .. 65536 envs per GPU).
//
// K6-fast runs one block per four envs: load -> compute -> store, serially, behind three block barriers, and relies
// on eight co-resident blocks per SM to overlap one block's loads with another's math.  With several waves of blocks
// that leaves the SM's issue slots idle 55-70 % of the time (ncu, round 1): every block spends about half of its life
// in the chain clock -> clip metadata -> frame copy, and the tail of each wave runs under-occupied.  Here a block is
// PERSISTENT and WARP-SPECIALISED:
//
//   * grid = 4 blocks per SM, each 3 consumer warps (4 envs x 24 bodies) + 1 producer warp, looping over env tiles it
//     draws from a device-side counter (the first tile is blockIdx.x), so the SMs finish together whatever the tile
//     count;
//   * the producer warp runs the whole dependent chain of tile k+1 — clock loads, clip metadata gathers, the frame
//     blend in the reference's fp32 order, the TMA copies of the sim rows and the frame span, the heading
//     quaternions — into the second shared-memory stage while the consumers compute tile k; stages are handed over
//     with mbarrier full / empty pairs (the full barrier counts the TMA bytes and the producer's arrival, the empty
//     one is released when the tile's bulk store has read the stage and its reductions are done);
//   * the consumers never touch global memory for input and never wait for a block barrier: two named barriers over
//     the 96 consumer threads per tile (frame buffer -> obs stage hand-over, stage complete), the obs rows leave with
//     one bulk store per tile, reductions and scalar outputs run on consumer warp 0 while warps 1-2 start the next
//     tile.
// Same per-body arithmetic as K6-fast, operand for operand: results are bit-identical (tested against the generic kernel).
// ---------------------------------------------------------------------------------------
constexpr int PS_STAGES = 2;
constexpr int PS_EPB = 4;
constexpr int PS_CONSUMERS = PS_EPB * J24;  // 96
constexpr int PS_THREADS = PS_CONSUMERS + 32;

// SLOTS: frame rows per env held in a stage.  A step needs the rows of two queries, t and t + dt: three consecutive
// rows when the clip's frame time equals the env's dt (the reference's regime: 30 fps clips, dt = 1/30 s), up to
// four otherwise (60 / 120 fps clips, unaligned times).  With SLOTS = 3 a stage is 22.5 KB and FIVE blocks fit an SM
// (15 consumer warps instead of 12: +5 % at 32768 / 65536 envs, 0.93 / 0.98 of the measured HBM peak); an env that
// needs a fourth row reads that one row ("far" row) straight from the packed table, L2-prefetched by the producer.
template <int SLOTS>
struct PersistStage {
  float sim[PS_EPB * ROW13];
  float frames[PS_EPB * SLOTS * FRAME_FLOATS];  // [env][slot][312]; later the obs stage [env][934]
  float part[6][PS_EPB][J24];
  float bl[2][PS_EPB];
  int slot[2][2][PS_EPB];   // slot of (query, frame 0 / 1); == SLOTS: the far row
  int64_t far[PS_EPB];      // packed-table row of the env's far row
  float goff[PS_EPB][4];
  float hz[PS_EPB], hw[PS_EPB];
  int prog[PS_EPB], pass[PS_EPB], fallen[PS_EPB];
  int tile;  // env tile held by the stage, -1: no more tiles
  int pad_[3];
  static_assert(SLOTS * FRAME_FLOATS >= STAGE_FLOATS, "the obs stage aliases the frame buffer");
};
template <int SLOTS>
struct PersistSmem {
  PersistStage<SLOTS> st[PS_STAGES];
  unsigned long long full[PS_STAGES], empty[PS_STAGES];
};
static_assert(sizeof(PersistStage<3>) % 16 == 0 && sizeof(PersistStage<4>) % 16 == 0,
              "stages keep the 16-byte alignment of the TMA destinations");

__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, %0;" ::"r"(PS_CONSUMERS) : "memory"); }

// MOM: the RunningNorm partials of the rows a block writes (obs_moments) stay in REGISTERS across the block's tiles —
// consumer thread i owns columns i, i + 96, ..: ten fp64 sums and ten sums of squares — and reach the accumulator
// buckets once, when the block runs out of tiles: 1868 adds in L2 per BLOCK (592 blocks) instead of per TILE.  In
// K6-fast the same partials cost 1868 adds per four envs, and those adds — 0.6 per ns for the whole chip whatever their
// width or issuer (profiles/r2_moments_modes_experiment.md) — are what its moments epilogue costs.
template <int SLOTS, int BLOCKS_PER_SM, bool MOM = false>
__global__ void __launch_bounds__(PS_THREADS, BLOCKS_PER_SM) step_persist_kernel(const __grid_constant__ StepParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  PersistSmem<SLOTS>& M = *reinterpret_cast<PersistSmem<SLOTS>*>(smem_raw);
  using Stage = PersistStage<SLOTS>;
  const int tid = threadIdx.x;
  const int num_tiles = (int)((p.n + PS_EPB - 1) / PS_EPB);
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < PS_STAGES; ++s) {
      mbar_init(&M.full[s], 1);
      mbar_init(&M.empty[s], MOM ? PS_CONSUMERS / 32 : 1);  // MOM: every consumer warp reads the finished stage
    }
  }
  __syncthreads();

  if (tid >= PS_CONSUMERS) {
    // =========================== producer warp ===========================
    // A tile's inputs sit behind a chain of three dependent memory round trips: clock -> clip metadata -> frame rows.
    // Run one tile at a time that chain is what a block waits for (measured: 4.5 us per tile under load, the whole
    // kernel slower than K6-fast).  The producer is therefore a software pipeline over THREE tiles: in one iteration
    // it issues the clock loads of tile i+2, the metadata gathers of tile i+1 (whose clock it loaded an iteration ago)
    // and — from registers only — blends and copies tile i.  Every load has a whole iteration to land.
    const int lane = tid - PS_CONSUMERS;
    const int le = lane >> 3, j = lane & 7;  // 8 lanes per env of the tile: lane 0 leads, lane 1 does the heading
    // Nothing is read before the dependency wait.  (Copying the frame rows of a block's first two tiles before the wait
    // and validating the clock after it — K6-fast's scheme — was built and measured: 27.59 against 27.59 us at 16384
    // envs, 15.48 against 14.85 at 8192.  What a multi-wave launch loses at its boundaries is the under-filled last
    // tile period and the first tile period in which every block loads at once, not the first tile's round trips.)
    asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
    asm volatile("griddepcontrol.wait;\n" ::: "memory");
    const bool block_sim = p.body.pos.stride_env == ROW13;  // a tile's sim rows are one span
    struct Clock {
      int prog_in;
      int64_t id;
      float start, soff, g0, g1, g2;
    };
    struct Meta {
      float len, mdt;
      int nf;
      int64_t st;
    };
    const auto env_of = [&](int tile) { return (int64_t)tile * PS_EPB + le; };
    const auto live = [&](int tile) { return tile < num_tiles && env_of(tile) < p.n; };
    const auto load_clock = [&](int tile) {  // .cg: the previous step's kernel wrote some of these
      Clock c{0, 0, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
      if (j == 0 && live(tile)) {
        const int64_t env = env_of(tile);
        c.prog_in = (int)__ldcg(p.progress + env);
        c.id = __ldcg(p.ids + env);
        c.start = __ldcg(p.start + env);
        c.soff = __ldcg(p.start_off + env);
        if (p.goff) {
          c.g0 = __ldcg(p.goff + env * 3 + 0);
          c.g1 = __ldcg(p.goff + env * 3 + 1);
          c.g2 = __ldcg(p.goff + env * 3 + 2);
        }
      }
      return c;
    };
    const auto load_rootq = [&](int tile) {  // floats 3..6 of the env's sim row: the root rotation
      Quat q{0.0f, 0.0f, 0.0f, 1.0f};
      if (j == 1 && live(tile)) {
        const float* rq = p.body.pos.ptr + env_of(tile) * p.body.pos.stride_env + 3;
        q = Quat{__ldcg(rq), __ldcg(rq + 1), __ldcg(rq + 2), __ldcg(rq + 3)};
      }
      return q;
    };
    const auto load_meta = [&](int tile, const Clock& c) {
      Meta m{1.0f, 1.0f, 2, 0};
      if (j == 0 && live(tile)) {
        m.len = p.L.len[c.id];
        m.nf = (int)p.L.nf[c.id];
        m.mdt = p.L.mdt[c.id];
        m.st = p.L.starts[c.id];
      }
      return m;
    };
    // a block's first three tiles are static (blockIdx.x, + grid, + 2 grid): nothing to wait for at the start; from the
    // fourth on they are drawn from the counter, which evens out the tail
    const int G = 3 * (int)gridDim.x;
    int tA = (int)blockIdx.x, tB = tA + (int)gridDim.x, tC = tB + (int)gridDim.x;
    Clock cA = load_clock(tA), cB = load_clock(tB);
    Quat qA = load_rootq(tA), qB = load_rootq(tB);
    Meta mA = load_meta(tA, cA);
    for (int it = 0;; ++it) {
      const int s = it % PS_STAGES;
      Stage& S = M.st[s];
      if (tA >= num_tiles) {  // tell the consumers and leave
        if (it >= PS_STAGES) mbar_wait(&M.empty[s], (uint32_t)(((it / PS_STAGES) - 1) & 1));
        if (lane == 0) {
          S.tile = -1;
          mbar_arrive(&M.full[s]);
        }
        break;
      }
      // loads for the tiles behind this one, consumed an iteration from now
      int grab = 0;
      if (lane == 0) grab = G + (int)atomicAdd(p.tile_counter, 1u);
      const Clock cC = load_clock(tC);
      const Quat qC = load_rootq(tC);
      const Meta mB = load_meta(tB, cB);
      // this tile: the stage has to be free
      if (it >= PS_STAGES) mbar_wait(&M.empty[s], (uint32_t)(((it / PS_STAGES) - 1) & 1));
      const int64_t env0 = (int64_t)tA * PS_EPB;
      const int nvalid = (int)((p.n - env0) < PS_EPB ? (p.n - env0) : PS_EPB);
      const bool act = le < nvalid;
      const int64_t env = env0 + (act ? le : 0);
      float* fr = S.frames + le * (SLOTS * FRAME_FLOATS);
      if (act && j == 0) {
        if (block_sim ? le == 0 : true) {  // sim rows
          const uint32_t bytes = (block_sim ? (uint32_t)nvalid : 1u) * (uint32_t)(ROW13 * 4);
          mbar_expect_tx(&M.full[s], bytes);
          bulk_g2s(S.sim + le * ROW13, p.body.pos.ptr + env * p.body.pos.stride_env, bytes, &M.full[s]);
        }
        const float len = mA.len, mdt = mA.mdt;
        const int nf = mA.nf;
        int prog = cA.prog_in;
        if (p.advance) prog = (int)(int16_t)(prog + 1);
        // q = 0: t = progress*dt + start + offset (humanoid_phc.py:1236); q = 1: (progress+1)*dt + ..
        // (humanoid_phc.py:1063-1067), progress already advanced (humanoid_phc.py:138)
        int a_f0, a_f1, b_f0, b_f1;
        float a_bl, b_bl;
        const float a_t = (float)(int16_t)prog * p.dt + cA.start + cA.soff;
        calc_frame_blend32(a_t, len, nf, mdt, a_f0, a_f1, a_bl);
        const float t1 = (float)(int16_t)(prog + 1) * p.dt + cA.start + cA.soff;
        calc_frame_blend32(t1, len, nf, mdt, b_f0, b_f1, b_bl);
        // frames of one clip are consecutive rows of the packed table: when the (up to four) frames span <= SLOTS rows
        // they arrive with ONE copy and slot = frame - first; otherwise the two queries' spans (one or two rows each)
        // are copied one after the other, and a row that does not fit (the fourth of a 3-slot stage) stays in the
        // table as the env's far row
        const float* tab = p.L.packed + mA.st * FRAME_FLOATS;
        const int lo = a_f0 < b_f0 ? a_f0 : b_f0;
        int hi = a_f1 > b_f1 ? a_f1 : b_f1;
        hi = hi > a_f0 ? hi : a_f0;
        hi = hi > b_f0 ? hi : b_f0;
        if (hi - lo <= SLOTS - 1) {
          S.slot[0][0][le] = a_f0 - lo;
          S.slot[0][1][le] = a_f1 - lo;
          S.slot[1][0][le] = b_f0 - lo;
          S.slot[1][1][le] = b_f1 - lo;
          const uint32_t bytes = (uint32_t)(hi - lo + 1) * (uint32_t)(FRAME_FLOATS * 4);
          mbar_expect_tx(&M.full[s], bytes);
          bulk_g2s(fr, tab + (int64_t)lo * FRAME_FLOATS, bytes, &M.full[s]);
        } else {  // spans (a_f0 .. a_f1) and (b_f0 .. b_f1), idx1 is idx0 or idx0 + 1
          const int na = a_f1 - a_f0 + 1;
          int nb = b_f1 - b_f0 + 1;
          S.slot[0][0][le] = 0;
          S.slot[0][1][le] = a_f1 - a_f0;
          S.slot[1][0][le] = na;
          S.slot[1][1][le] = na + (b_f1 - b_f0);
          if (na + nb > SLOTS) {  // SLOTS == 3 and four distinct rows: the last one stays in the table
            nb -= 1;
            S.slot[1][1][le] = SLOTS;
            S.far[le] = mA.st + b_f1;
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;\n" ::"l"(tab + (int64_t)b_f1 * FRAME_FLOATS),
                         "r"((uint32_t)(FRAME_FLOATS * 4))
                         : "memory");
          }
          const uint32_t ba = (uint32_t)na * (uint32_t)(FRAME_FLOATS * 4);
          const uint32_t bb = (uint32_t)nb * (uint32_t)(FRAME_FLOATS * 4);
          mbar_expect_tx(&M.full[s], ba + bb);
          bulk_g2s(fr, tab + (int64_t)a_f0 * FRAME_FLOATS, ba, &M.full[s]);
          bulk_g2s(fr + na * FRAME_FLOATS, tab + (int64_t)b_f0 * FRAME_FLOATS, bb, &M.full[s]);
        }
        S.bl[0][le] = a_bl;
        S.bl[1][le] = b_bl;
        S.prog[le] = prog;
        S.pass[le] = a_t >= len;  // _compute_reset, humanoid_phc.py:1317
        S.fallen[le] = 0;
        if (p.advance) {
          p.progress[env] = (int16_t)prog;
          if (p.progress_mirror) p.progress_mirror[env] = (int16_t)prog;
        }
        S.goff[le][0] = cA.g0;
        S.goff[le][1] = cA.g1;
        S.goff[le][2] = cA.g2;
      } else if (act && j == 1) {
        const Heading h0 = heading_quat_inv(qA);  // upright: root_rot used as is (common.py:42-44)
        S.hz[le] = h0.z;
        S.hw[le] = h0.w;
      }
      __syncwarp();
      if (lane == 0) {
        S.tile = tA;
        mbar_arrive(&M.full[s]);  // release: the stage's scalars are visible to whoever sees the phase complete
      }
      tA = tB, tB = tC, tC = __shfl_sync(0xffffffffu, grab, 0);
      cA = cB, cB = cC, mA = mB, qA = qB, qB = qC;
    }
    // the last block out rewinds the tile counter for the next launch that draws this slot
    if (lane == 0) {
      __threadfence();
      if (atomicAdd(p.tile_counter + 1, 1u) == gridDim.x - 1) {
        p.tile_counter[0] = 0;
        p.tile_counter[1] = 0;
        __threadfence();
      }
    }
    return;
  }

  // =========================== consumer warps ===========================
  const int e = tid / J24, b = tid % J24;
  constexpr int MOM_COLS = (STAGE_FLOATS + PS_CONSUMERS - 1) / PS_CONSUMERS;  // 10 columns per consumer thread
  double ms1[MOM ? MOM_COLS : 1], ms2[MOM ? MOM_COLS : 1];
  if constexpr (MOM) {
#pragma unroll
    for (int k = 0; k < MOM_COLS; ++k) ms1[k] = 0.0, ms2[k] = 0.0;
  }
  for (int it = 0;; ++it) {
    const int s = it % PS_STAGES;
    Stage& S = M.st[s];
    mbar_wait(&M.full[s], (uint32_t)((it / PS_STAGES) & 1));
    const int tile = S.tile;
    if (tile < 0) break;
    const int64_t env0 = (int64_t)tile * PS_EPB;
    const int nvalid = (int)((p.n - env0) < PS_EPB ? (p.n - env0) : PS_EPB);
    const bool valid = e < nvalid;

    // ---- phase 1: per-body reference states, reward partials, distance ------------------------
    Vec3 pos, vel, ang, root_pos;
    Quat rot;
    RefBody r1;
    if (valid) {
      const float* d = S.sim + e * ROW13 + b * 13;
      pos = {d[0], d[1], d[2]};
      rot = {d[3], d[4], d[5], d[6]};
      vel = {d[7], d[8], d[9]};
      ang = {d[10], d[11], d[12]};
      root_pos = {S.sim[e * ROW13 + 0], S.sim[e * ROW13 + 1], S.sim[e * ROW13 + 2]};
      const float* fr = S.frames + e * (SLOTS * FRAME_FLOATS);
      {
        const RefBody r0 = blend_ref2(fr + S.slot[0][0][e] * FRAME_FLOATS, fr + S.slot[0][1][e] * FRAME_FLOATS,
                                      S.bl[0][e], S.goff[e], b);  // the far row, if any, is the second query's
        float sp, sr, sv, sa;
        reward_partials(pos, rot, vel, ang, r0, sp, sr, sv, sa);
        S.part[0][e][b] = sp;
        S.part[1][e][b] = sr;
        S.part[2][e][b] = sv;
        S.part[3][e][b] = sa;
        const float dist = norm3(pos - r0.pos);  // torch.norm(rigid_body_pos - ref_body_pos), common.py:343/348
        S.part[4][e][b] = dist;
        if (!p.use_mean && (p.reset_mask >> b & 1u) && dist > p.term_dist[b]) S.fallen[e] = 1;  // any(), benign race
        if (p.dof_force) S.part[5][e][b] = power_partial(p, env0 + e, b);
      }
      const int s11 = S.slot[1][1][e];
      if (SLOTS >= 4 || s11 < SLOTS)
        r1 = blend_ref2(fr + S.slot[1][0][e] * FRAME_FLOATS, fr + s11 * FRAME_FLOATS, S.bl[1][e], S.goff[e], b);
      else  // the fourth row of a 3-slot stage: read from the packed table (L2: the producer prefetched it)
        r1 = blend_ref2(fr + S.slot[1][0][e] * FRAME_FLOATS, p.L.packed + S.far[e] * FRAME_FLOATS, S.bl[1][e], S.goff[e], b);
    }
    consumer_sync();  // partials visible; frame buffer dead -> becomes the obs stage

    // ---- phase 2: observations into the stage ---------------------------------------------------
    if (valid) {
      const Heading hi = {S.hz[e], S.hw[e]};
      const HeadingRot hr = heading_rot(hi);
      float* row = S.frames + e * STAGE_FLOATS;
      emit_self_obs<true>(row, p.of, b, root_pos, hi, hr, pos, rot, vel, ang);       // common.py:23-103
      emit_task_obs<true>(row + SELF_DIM, b, hi, hr, root_pos, pos, rot, vel, ang, r1);  // common.py:106-176
    }
    fence_proxy_async();  // stage writes -> visible to the bulk-store engine
    consumer_sync();      // stage complete

    const uint32_t out_bytes = (uint32_t)nvalid * (STAGE_FLOATS * 4);
    const bool bulk_ok = (out_bytes & 15u) == 0;
    if (bulk_ok) {
      if (tid == 0) bulk_s2g(p.obs + env0 * STAGE_FLOATS, S.frames, out_bytes);
    } else {  // odd tail tile: 8-byte stores by everyone, and everyone has to be done before the stage is released
      float2* dst = reinterpret_cast<float2*>(p.obs + env0 * STAGE_FLOATS);
      const float2* src = reinterpret_cast<const float2*>(S.frames);
      for (int i = tid; i < nvalid * (STAGE_FLOATS / 2); i += PS_CONSUMERS) dst[i] = src[i];
      consumer_sync();
    }
    if constexpr (MOM) {  // x * x is exact in fp64 for an fp32 x: the fused form equals mul + add bit for bit
#pragma unroll
      for (int k = 0; k < MOM_COLS; ++k) {
        const int c = tid + k * PS_CONSUMERS;
        if (c < STAGE_FLOATS) {
#pragma unroll
          for (int ee = 0; ee < PS_EPB; ++ee) {
            if (ee < nvalid) {
              const double x = (double)S.frames[ee * STAGE_FLOATS + c];
              ms1[k] += x;
              ms2[k] = __fma_rn(x, x, ms2[k]);
            }
          }
        }
      }
      __syncwarp();
      if (tid >= 32 && (tid & 31) == 0) mbar_arrive(&M.empty[s]);  // warps 1-2 are done with the stage; warp 0 below
    }
    // ---- reductions and scalar outputs (consumer warp 0) while warps 1-2 start the next tile ----------
    if (tid < 32) {
      const int le = tid >> 2, k = tid & 3;
      const bool act = le < nvalid && tid < 4 * PS_EPB;
      float term_k = 0.0f;
      if (act) {
        const float kk = k == 0 ? p.rwd.k_pos : k == 1 ? p.rwd.k_rot : k == 2 ? p.rwd.k_vel : p.rwd.k_ang_vel;
        term_k = expf((-kk) * (row_sum24(&S.part[k][le][0]) / 24.0f));  // common.py:298-320
        p.raw[(env0 + le) * p.raw_stride + k] = term_k;
      }
      const int base = tid & ~3;
      const float t0 = __shfl_sync(0xffffffffu, term_k, base), t1 = __shfl_sync(0xffffffffu, term_k, base + 1);
      const float t2 = __shfl_sync(0xffffffffu, term_k, base + 2), t3 = __shfl_sync(0xffffffffu, term_k, base + 3);
      if (act && k == 0) {
        float r = p.rwd.w_pos * t0 + p.rwd.w_rot * t1 + p.rwd.w_vel * t2 + p.rwd.w_ang_vel * t3;
        if (p.dof_force) {
          const float pr = power_reward(p, &S.part[5][le][0], S.prog[le]);
          r += pr;  // rew_buf[:] += power_reward (humanoid_phc.py:1304)
          p.raw[(env0 + le) * p.raw_stride + p.power_col] = pr;
        }
        p.rew[env0 + le] = r;
        if (p.rew_out) p.rew_out[env0 + le] = r;
      }
      if (act && k == 1) {
        bool fallen = false;
        if (p.early) {
          if (p.use_mean) {  // eval mode: mean distance of the selected bodies vs the first one's threshold
            float sel[J24];
            int m = 0;
#pragma unroll
            for (int jj = 0; jj < J24; ++jj)
              if (p.reset_mask >> jj & 1u) sel[m++] = S.part[4][le][jj];
            const int first = __ffs(p.reset_mask) - 1;
            fallen = m > 0 && (aten_row_sum(sel, m) / (float)m) > p.term_dist[first < 0 ? 0 : first];
          } else {
            fallen = S.fallen[le] != 0;
          }
          fallen = fallen && (S.prog[le] > 1);  // common.py:353
        }
        const bool rs = S.pass[le] || fallen;  // common.py:362
        p.term[env0 + le] = fallen ? 1 : 0;
        p.reset[env0 + le] = rs ? 1 : 0;
        if (p.term_out) p.term_out[env0 + le] = fallen ? 1 : 0;
        if (p.reset_out) p.reset_out[env0 + le] = rs ? 1 : 0;
      }
      if (act && k == 2 && p.mpjpe) p.mpjpe[env0 + le] = row_sum24(&S.part[4][le][0]) / 24.0f;  // humanoid_phc.py:167
      __syncwarp();
      if (tid == 0) {  // the stage goes back to the producer once the store has read it and the partials are consumed
        if (bulk_ok) bulk_wait_read();
        mbar_arrive(&M.empty[s]);
      }
    }
  }
  if constexpr (MOM) {
    double* mom = p.moments + (int64_t)(blockIdx.x % p.moment_buckets) * 2 * STAGE_FLOATS;
#pragma unroll
    for (int k = 0; k < MOM_COLS; ++k) {
      const int c = tid + k * PS_CONSUMERS;
      if (c < STAGE_FLOATS) {
        atomicAdd(mom + c, ms1[k]);
        atomicAdd(mom + STAGE_FLOATS + c, ms2[k]);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------
// K6-multi: the fused step for T > 1 future reference frames (BASELINE config 5) on the AoS sim
// tensor and the packed frame table.  Same per-body math as K6-fast; the T+1 motion queries are a
// software pipeline over two half-buffers of two frame rows each:
//
//   q:   wait(half q&1) -> reference state -> (q = 0: reward partials | q >= 1: v6 block -> stage)
//        barrier A      -> warp 0 issues the TMA copy of query q+2 into the half just consumed
//                          while every env's staged 576 (934 for q = 1) floats leave with ONE
//                          cp.async.bulk store (rows of obs_buf alternate between 16-B and 8-B
//                          alignment: a misaligned segment is staged shifted by two floats, its
//                          first and last pair stored by hand)
//        barrier B      -> stage free
//
// so copy latency is hidden one full iteration ahead and there are two block barriers per query
// (the generic kernel has four and exposes every copy).
// ---------------------------------------------------------------------------------------
constexpr int MULTI_EPB = 4;
constexpr int STAGE_STRIDE = 940;  // floats per staged row: 934 + 2 shift, rounded to 16 B

struct MultiSmem {
  float sim[MULTI_EPB * ROW13];
  float frames[MULTI_EPB][4][FRAME_FLOATS];  // [env][half*2 + row][312]
  float stage[MULTI_EPB][STAGE_STRIDE];
  float part[6][MULTI_EPB][J24];
  unsigned long long bar[2];
  int64_t row0[PHC_MAX_TIME_STEPS + 1][MULTI_EPB];  // global row of idx0 of query q
  int two[PHC_MAX_TIME_STEPS + 1][MULTI_EPB];       // idx1 == idx0 + 1
  float bl[PHC_MAX_TIME_STEPS + 1][MULTI_EPB];
  float goff[MULTI_EPB][4];
  float hz[MULTI_EPB], hw[MULTI_EPB];
  int prog[MULTI_EPB], pass[MULTI_EPB], fallen[MULTI_EPB];
};

__global__ void __launch_bounds__(MULTI_EPB* J24, 5) step_multi_kernel(const StepParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  MultiSmem& S = *reinterpret_cast<MultiSmem*>(smem_raw);
  constexpr int EPB = MULTI_EPB, NT = EPB * J24;
  const int tid = threadIdx.x;
  const int64_t env0 = (int64_t)blockIdx.x * EPB;
  const int nvalid = (int)((p.n - env0) < EPB ? (p.n - env0) : EPB);
  const int T = p.T;
  const int W = SELF_DIM + TASK_DIM * T;

  // frames of query q for env le -> half q&1; returns the bytes it expects
  auto issue_frames = [&](int le, int q) {
    const uint32_t bytes = (uint32_t)(1 + S.two[q][le]) * (uint32_t)(FRAME_FLOATS * 4);
    mbar_expect_tx(&S.bar[q & 1], bytes);
    bulk_g2s(&S.frames[le][(q & 1) * 2][0], p.L.packed + S.row0[q][le] * FRAME_FLOATS, bytes, &S.bar[q & 1]);
  };

  // ---- phase 0 ------------------------------------------------------------------------------
  if (tid < 32) {
    if (tid == 0) {
      mbar_init(&S.bar[0], 1);
      mbar_init(&S.bar[1], 1);
    }
    __syncwarp();
    for (int pair = tid; pair < nvalid * (T + 1); pair += 32) {
      const int le = pair / (T + 1), q = pair - le * (T + 1);
      const int64_t env = env0 + le;
      int prog = (int)p.progress[env];
      if (p.advance) prog = (int)(int16_t)(prog + 1);
      // q = 0: t = progress*dt + start + offset (humanoid_phc.py:1236); q >= 1: (progress+q)*dt + ..
      const float t = (float)(int16_t)(prog + q) * p.dt + p.start[env] + p.start_off[env];
      const int64_t id = p.ids[env];
      const float len = p.L.len[id];
      int i0, i1;
      float bl;
      calc_frame_blend32(t, len, (int)p.L.nf[id], p.L.mdt[id], i0, i1, bl);
      S.row0[q][le] = p.L.starts[id] + i0;
      S.two[q][le] = i1 - i0;
      S.bl[q][le] = bl;
      if (q == 0) {
        S.prog[le] = prog;
        S.pass[le] = t >= len;  // _compute_reset, humanoid_phc.py:1317
        S.fallen[le] = 0;
        S.goff[le][0] = p.goff ? p.goff[env * 3 + 0] : 0.0f;
        S.goff[le][1] = p.goff ? p.goff[env * 3 + 1] : 0.0f;
        S.goff[le][2] = p.goff ? p.goff[env * 3 + 2] : 0.0f;
      }
    }
    __syncwarp();
    // progress is written only now: a lane's later (env, q) pair must still read the old value
    if (tid < nvalid && p.advance) p.progress[env0 + tid] = (int16_t)S.prog[tid];
    if (tid < nvalid) {  // sim row + queries 0 and 1 of env `tid`
      mbar_expect_tx(&S.bar[0], ROW13 * 4);
      bulk_g2s(S.sim + tid * ROW13, p.body.pos.ptr + (env0 + tid) * p.body.pos.stride_env, ROW13 * 4, &S.bar[0]);
      issue_frames(tid, 0);
      issue_frames(tid, 1);
    }
    __syncwarp();
    if (tid == 0) {
      mbar_arrive(&S.bar[0]);
      mbar_arrive(&S.bar[1]);
    }
  } else if (tid >= 32 && tid < 32 + nvalid) {  // warp 1: heading quaternions from global memory
    const int le = tid - 32;
    const float* rq = p.body.pos.ptr + (env0 + le) * p.body.pos.stride_env + 3;
    const Heading h0 = heading_quat_inv(Quat{rq[0], rq[1], rq[2], rq[3]});  // upright (common.py:42-44)
    S.hz[le] = h0.z;
    S.hw[le] = h0.w;
  }
  __syncthreads();

  const int e = tid / J24, b = tid % J24;
  const bool valid = e < nvalid;
  const int64_t env = env0 + e;
  Vec3 pos = {}, vel = {}, ang = {}, root_pos = {};
  Quat rot = {};
  Heading hi = {S.hz[valid ? e : 0], S.hw[valid ? e : 0]};
  HeadingRot hr = heading_rot(hi);

  for (int q = 0; q <= T; ++q) {
    mbar_wait(&S.bar[q & 1], (uint32_t)((q >> 1) & 1));
    float* dst = nullptr;   // this env's segment of obs_buf for query q
    int seg = 0, shift = 0;
    if (valid) {
      if (q == 0) {
        const float* d = S.sim + e * ROW13 + b * 13;
        pos = {d[0], d[1], d[2]};
        rot = {d[3], d[4], d[5], d[6]};
        vel = {d[7], d[8], d[9]};
        ang = {d[10], d[11], d[12]};
        root_pos = {S.sim[e * ROW13 + 0], S.sim[e * ROW13 + 1], S.sim[e * ROW13 + 2]};
      }
      const float* f0 = &S.frames[e][(q & 1) * 2][0];
      const RefBody r = blend_ref2(f0, f0 + S.two[q][e] * FRAME_FLOATS, S.bl[q][e], S.goff[e], b);
      if (q == 0) {
        float sp, sr, sv, sa;
        reward_partials(pos, rot, vel, ang, r, sp, sr, sv, sa);
        S.part[0][e][b] = sp;
        S.part[1][e][b] = sr;
        S.part[2][e][b] = sv;
        S.part[3][e][b] = sa;
        const float dist = norm3(pos - r.pos);  // common.py:343/348
        S.part[4][e][b] = dist;
        if (!p.use_mean && (p.reset_mask >> b & 1u) && dist > p.term_dist[b]) S.fallen[e] = 1;
        if (p.dof_force) S.part[5][e][b] = power_partial(p, env, b);
      } else {
        const int64_t c_off = q == 1 ? 0 : SELF_DIM + (int64_t)TASK_DIM * (q - 1);
        seg = q == 1 ? STAGE_FLOATS : TASK_DIM;
        dst = p.obs + env * p.obs_stride + c_off;
        shift = ((uintptr_t)dst & 15) ? 2 : 0;  // 8-B aligned rows: stage shifted so the bulk part is 16-B aligned
        float* row = &S.stage[e][shift];
        float* tk = row;
        if (q == 1) {  // self obs, common.py:23-103 (default flags)
          if (b == 0)
            row[0] = root_pos.z;
          else
            st3(row + 1 + (b - 1) * 3, heading_rotate(hr, pos - root_pos));
          float t6[6];
          quat_tan_norm(heading_mul_left(hi, rot), t6);
          st6_shared(row + 70 + b * 6, t6);
          st3(row + 214 + b * 3, heading_rotate(hr, vel));
          st3(row + 286 + b * 3, heading_rotate(hr, ang));
          tk = row + SELF_DIM;
        }
        TaskObs o;  // task obs v6 block of future step q, common.py:106-176
        task_obs_body(hi, hr, root_pos, pos, rot, vel, ang, r, true, o);
        st3(tk + b * 3, o.d_pos);
        st6_shared(tk + 72 + b * 6, o.d_rot);
        st3(tk + 216 + b * 3, o.d_vel);
        st3(tk + 288 + b * 3, o.d_ang);
        st3(tk + 360 + b * 3, o.l_pos);
        st6_shared(tk + 432 + b * 6, o.l_rot);
      }
    }
    fence_proxy_async();  // stage writes -> bulk store; frame reads -> the copy that refills the half
    __syncthreads();      // A: half (q & 1) consumed, stage complete

    if (q + 2 <= T && tid < 32) {  // prefetch query q + 2 into the half just consumed
      if (tid < nvalid) issue_frames(tid, q + 2);
      __syncwarp();
      if (tid == 0) mbar_arrive(&S.bar[q & 1]);
    }
    if (q >= 1) {
      if (valid && b == 0) {  // one bulk store per env: the 16-B aligned middle of the segment
        const int body4 = (seg - shift) & ~3;  // floats
        bulk_s2g(dst + shift, &S.stage[e][2 * shift], (uint32_t)body4 * 4);
      }
      if (valid && shift && b < 2) dst[b] = S.stage[e][shift + b];  // leading pair
      if (valid && b >= 2 && b < 2 + ((seg - shift) & 3)) {         // trailing pair
        const int c = shift + ((seg - shift) & ~3) + (b - 2);
        dst[c] = S.stage[e][shift + c];
      }
      if (p.moments) {
        const int64_t c_off = q == 1 ? 0 : SELF_DIM + (int64_t)TASK_DIM * (q - 1);
        const int sl = q == 1 ? STAGE_FLOATS : TASK_DIM;
        for (int c = tid; c < sl; c += NT) {
          double s1 = 0.0, s2 = 0.0;
          for (int ee = 0; ee < nvalid; ++ee) {
            const float* d2 = p.obs + (env0 + ee) * p.obs_stride + c_off;
            const double x = (double)S.stage[ee][(((uintptr_t)d2 & 15) ? 2 : 0) + c];
            s1 += x;
            s2 += x * x;
          }
          double* mom = p.moments + (int64_t)(blockIdx.x % p.moment_buckets) * 2 * W;
          atomicAdd(mom + c_off + c, s1);
          atomicAdd(mom + W + c_off + c, s2);
        }
      }
      if (valid && b == 0) bulk_wait_read();
      __syncthreads();  // B: stage free
    }
  }

  // ---- reductions and scalar outputs (warp 0) ---------------------------------------------------
  if (tid < 32) {
    const int le = tid >> 2, k = tid & 3;
    const bool act = le < nvalid && tid < 4 * EPB;
    float term_k = 0.0f;
    if (act) {
      const float kk = k == 0 ? p.rwd.k_pos : k == 1 ? p.rwd.k_rot : k == 2 ? p.rwd.k_vel : p.rwd.k_ang_vel;
      term_k = expf((-kk) * (row_sum24(&S.part[k][le][0]) / 24.0f));  // common.py:298-320
      p.raw[(env0 + le) * p.raw_stride + k] = term_k;
    }
    const int base = tid & ~3;
    const float t0 = __shfl_sync(0xffffffffu, term_k, base), t1 = __shfl_sync(0xffffffffu, term_k, base + 1);
    const float t2 = __shfl_sync(0xffffffffu, term_k, base + 2), t3 = __shfl_sync(0xffffffffu, term_k, base + 3);
    if (act && k == 0) {
      float r = p.rwd.w_pos * t0 + p.rwd.w_rot * t1 + p.rwd.w_vel * t2 + p.rwd.w_ang_vel * t3;
      if (p.dof_force) {
        const float pr = power_reward(p, &S.part[5][le][0], S.prog[le]);
        r += pr;
        p.raw[(env0 + le) * p.raw_stride + p.power_col] = pr;
      }
      p.rew[env0 + le] = r;
      if (p.rew_out) p.rew_out[env0 + le] = r;
    }
    if (act && k == 1) {
      bool fallen = false;
      if (p.early) {
        if (p.use_mean) {
          float sel[J24];
          int m = 0;
#pragma unroll
          for (int j = 0; j < J24; ++j)
            if (p.reset_mask >> j & 1u) sel[m++] = S.part[4][le][j];
          const int first = __ffs(p.reset_mask) - 1;
          fallen = m > 0 && (aten_row_sum(sel, m) / (float)m) > p.term_dist[first < 0 ? 0 : first];
        } else {
          fallen = S.fallen[le] != 0;
        }
        fallen = fallen && (S.prog[le] > 1);  // common.py:353
      }
      const bool rs = S.pass[le] || fallen;  // common.py:362
      p.term[env0 + le] = fallen ? 1 : 0;
      p.reset[env0 + le] = rs ? 1 : 0;
      if (p.term_out) p.term_out[env0 + le] = fallen ? 1 : 0;
      if (p.reset_out) p.reset_out[env0 + le] = rs ? 1 : 0;
    }
    if (act && k == 2 && p.mpjpe) p.mpjpe[env0 + le] = row_sum24(&S.part[4][le][0]) / 24.0f;  // humanoid_phc.py:167
  }
  if (p.ref_dof_pos && tid < EPB * J24 && tid / J24 < nvalid) {  // res_action: dof_pos of the query at t + dt
    const int le = tid / J24;
    write_ref_dof_pos(p, env0 + le, tid % J24, S.row0[1][le], S.row0[1][le] + S.two[1][le], S.bl[1][le]);
  }
}

// ---------------------------------------------------------------------------------------
// K6-multi2: K6-multi with TWO thread groups per block.  Group g (96 threads = 4 envs x 24 bodies)
// owns the queries q = g, g+2, g+4, .. and the frame half g, so consecutive queries of an env are
// worked on at the same time: at small N (config 5 on 8 GPUs: 2048 envs per GPU) a block of K6-multi is
// one warp-serial chain of ~450 dependent instructions per query with 10 warps per SM; here the chain
// per query pair is the same length and the SM holds twice the warps.  Each group synchronises on its
// own named barrier; the groups only meet at the start (sim rows, heading) and never wait for each
// other.  A half is refilled (query q+2) as soon as every thread of its group holds the blended reference
// body, so the copy flies while the observation block is computed, staged and stored.
// ---------------------------------------------------------------------------------------
constexpr int STAGE0_STRIDE = 580;  // group 0 stages task blocks only: 576 + 2 shift, rounded to 16 B

struct Multi2Smem {
  float sim[MULTI_EPB * ROW13];
  float frames[MULTI_EPB][4][FRAME_FLOATS];  // [env][group*2 + row][312]
  float stage1[MULTI_EPB][STAGE_STRIDE];     // group 1: q = 1 stages self obs + first task block
  float stage0[MULTI_EPB][STAGE0_STRIDE];    // group 0: q >= 2
  float part[6][MULTI_EPB][J24];
  unsigned long long bar[2];  // frames of group g
  unsigned long long bar_sim;
  int64_t row0[PHC_MAX_TIME_STEPS + 1][MULTI_EPB];
  int two[PHC_MAX_TIME_STEPS + 1][MULTI_EPB];
  float bl[PHC_MAX_TIME_STEPS + 1][MULTI_EPB];
  float goff[MULTI_EPB][4];
  float hz[MULTI_EPB], hw[MULTI_EPB];
  int prog[MULTI_EPB], pass[MULTI_EPB], fallen[MULTI_EPB];
};

__device__ __forceinline__ void group_sync(int g) {  // named barrier 1 + g over the group's 96 threads
  if (g) asm volatile("bar.sync 2, %0;" ::"r"(MULTI_EPB * J24) : "memory");
  else asm volatile("bar.sync 1, %0;" ::"r"(MULTI_EPB * J24) : "memory");
}

__global__ void __launch_bounds__(2 * MULTI_EPB* J24, 4) step_multi2_kernel(const StepParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Multi2Smem& S = *reinterpret_cast<Multi2Smem*>(smem_raw);
  constexpr int EPB = MULTI_EPB, GT = EPB * J24;
  const int tid = threadIdx.x;
  const int g = tid / GT, lt = tid - g * GT;  // group, thread within the group
  const int64_t env0 = (int64_t)blockIdx.x * EPB;
  const int nvalid = (int)((p.n - env0) < EPB ? (p.n - env0) : EPB);
  const int T = p.T;
  const int W = SELF_DIM + TASK_DIM * T;

  // frames of query q for env le -> the half of group q & 1
  auto issue_frames = [&](int le, int q) {
    const uint32_t bytes = (uint32_t)(1 + S.two[q][le]) * (uint32_t)(FRAME_FLOATS * 4);
    mbar_expect_tx(&S.bar[q & 1], bytes);
    bulk_g2s(&S.frames[le][(q & 1) * 2][0], p.L.packed + S.row0[q][le] * FRAME_FLOATS, bytes, &S.bar[q & 1]);
  };
  // ... and of a query two iterations ahead -> L2: under load a 2.5 KB copy from DRAM takes longer than one query
  // iteration (a sixth of the stall samples sat on the frame mbarrier, profiles/r2s2_multi2_T10_n16384_ncu.md); the copy
  // issued an iteration later then finds its rows in L2
  auto prefetch_frames = [&](int le, int q) {
    if (!p.multi_prefetch) return;
    const uint32_t bytes = (uint32_t)(1 + S.two[q][le]) * (uint32_t)(FRAME_FLOATS * 4);
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;\n" ::"l"(p.L.packed + S.row0[q][le] * FRAME_FLOATS), "r"(bytes)
                 : "memory");
  };

  // ---- phase 0 (whole block) ----------------------------------------------------------------
  if (tid < 64) {  // two warps share the (env, query) pairs: one round of dependent clip-metadata loads for T <= 15
    if (tid == 0) {
      mbar_init(&S.bar[0], 1);
      mbar_init(&S.bar[1], 1);
      mbar_init(&S.bar_sim, 1);
    }
    for (int pair = tid; pair < nvalid * (T + 1); pair += 64) {
      const int le = pair / (T + 1), q = pair - le * (T + 1);
      const int64_t env = env0 + le;
      int prog = (int)p.progress[env];
      if (p.advance) prog = (int)(int16_t)(prog + 1);
      const float t = (float)(int16_t)(prog + q) * p.dt + p.start[env] + p.start_off[env];
      const int64_t id = p.ids[env];
      const float len = p.L.len[id];
      int i0, i1;
      float bl;
      calc_frame_blend32(t, len, (int)p.L.nf[id], p.L.mdt[id], i0, i1, bl);
      S.row0[q][le] = p.L.starts[id] + i0;
      S.two[q][le] = i1 - i0;
      S.bl[q][le] = bl;
      if (q == 0) {
        S.prog[le] = prog;
        S.pass[le] = t >= len;  // _compute_reset, humanoid_phc.py:1317
        S.fallen[le] = 0;
        S.goff[le][0] = p.goff ? p.goff[env * 3 + 0] : 0.0f;
        S.goff[le][1] = p.goff ? p.goff[env * 3 + 1] : 0.0f;
        S.goff[le][2] = p.goff ? p.goff[env * 3 + 2] : 0.0f;
      }
    }
    asm volatile("bar.sync 3, 64;" ::: "memory");  // both warps have read the clock and filled the tables
    // progress is written only now: a lane's later (env, q) pair must still read the old value
    if (tid < nvalid && p.advance) p.progress[env0 + tid] = (int16_t)S.prog[tid];
    if (tid < nvalid) {
      mbar_expect_tx(&S.bar_sim, ROW13 * 4);
      bulk_g2s(S.sim + tid * ROW13, p.body.pos.ptr + (env0 + tid) * p.body.pos.stride_env, ROW13 * 4, &S.bar_sim);
      issue_frames(tid, 0);
      issue_frames(tid, 1);
      if (T >= 2) prefetch_frames(tid, 2);
      if (T >= 3) prefetch_frames(tid, 3);
    }
    if (tid < 32) __syncwarp();
    if (tid == 0) {
      mbar_arrive(&S.bar_sim);
      mbar_arrive(&S.bar[0]);
      mbar_arrive(&S.bar[1]);
    }
  } else if (tid >= 64 && tid < 64 + nvalid) {  // warp 2: heading quaternions from global memory
    const int le = tid - 64;
    const float* rq = p.body.pos.ptr + (env0 + le) * p.body.pos.stride_env + 3;
    const Heading h0 = heading_quat_inv(Quat{rq[0], rq[1], rq[2], rq[3]});  // upright (common.py:42-44)
    S.hz[le] = h0.z;
    S.hw[le] = h0.w;
  }
  __syncthreads();  // the only block-wide barrier

  const int e = lt / J24, b = lt % J24;
  const bool valid = e < nvalid;
  const int64_t env = env0 + e;
  const Heading hi = {S.hz[valid ? e : 0], S.hw[valid ? e : 0]};
  const HeadingRot hr = heading_rot(hi);
  mbar_wait(&S.bar_sim, 0u);  // single phase: both groups read the sim rows
  Vec3 pos = {}, vel = {}, ang = {}, root_pos = {};
  Quat rot = {};
  if (valid) {
    const float* d = S.sim + e * ROW13 + b * 13;
    pos = {d[0], d[1], d[2]};
    rot = {d[3], d[4], d[5], d[6]};
    vel = {d[7], d[8], d[9]};
    ang = {d[10], d[11], d[12]};
    root_pos = {S.sim[e * ROW13 + 0], S.sim[e * ROW13 + 1], S.sim[e * ROW13 + 2]};
  }
  float* const stage_base = g ? &S.stage1[0][0] : &S.stage0[0][0];
  const int stage_stride = g ? STAGE_STRIDE : STAGE0_STRIDE;

  for (int q = g, it = 0; q <= T; q += 2, ++it) {
    mbar_wait(&S.bar[g], (uint32_t)(it & 1));
    float* dst = nullptr;  // this env's segment of obs_buf for query q
    int seg = 0, shift = 0;
    float* row = nullptr;
    RefBody r = {};
    if (valid) {
      const float* f0 = &S.frames[e][g * 2][0];
      r = blend_ref2(f0, f0 + S.two[q][e] * FRAME_FLOATS, S.bl[q][e], S.goff[e], b);
    }
    // the half is dead once every thread of the group holds its reference body: refill it with query q + 2 now, so
    // the copy flies while the observation block is computed, staged and stored
    if (valid && b == 0) bulk_wait_read();  // the previous query's bulk store has read the stage: it may be rewritten
    fence_proxy_async();                    // frame reads -> the copy that refills the half
    group_sync(g);                          // R
    if (q + 2 <= T && lt < 32) {
      if (lt < nvalid) {
        issue_frames(lt, q + 2);
        if (q + 4 <= T) prefetch_frames(lt, q + 4);
      }
      __syncwarp();
      if (lt == 0) mbar_arrive(&S.bar[g]);
    }
    if (valid) {
      if (q == 0) {
        float sp, sr, sv, sa;
        reward_partials(pos, rot, vel, ang, r, sp, sr, sv, sa);
        S.part[0][e][b] = sp;
        S.part[1][e][b] = sr;
        S.part[2][e][b] = sv;
        S.part[3][e][b] = sa;
        const float dist = norm3(pos - r.pos);  // common.py:343/348
        S.part[4][e][b] = dist;
        if (!p.use_mean && (p.reset_mask >> b & 1u) && dist > p.term_dist[b]) S.fallen[e] = 1;
        if (p.dof_force) S.part[5][e][b] = power_partial(p, env, b);
      } else {
        const int64_t c_off = q == 1 ? 0 : SELF_DIM + (int64_t)TASK_DIM * (q - 1);
        seg = q == 1 ? STAGE_FLOATS : TASK_DIM;
        dst = p.obs + env * p.obs_stride + c_off;
        shift = ((uintptr_t)dst & 15) ? 2 : 0;  // 8-B aligned rows: stage shifted so the bulk part is 16-B aligned
        row = stage_base + e * stage_stride + shift;
        float* tk = row;
        if (q == 1) {  // self obs, common.py:23-103 (default flags)
          if (b == 0)
            row[0] = root_pos.z;
          else
            st3(row + 1 + (b - 1) * 3, heading_rotate(hr, pos - root_pos));
          float t6[6];
          quat_tan_norm(heading_mul_left(hi, rot), t6);
          st6_shared(row + 70 + b * 6, t6);
          st3(row + 214 + b * 3, heading_rotate(hr, vel));
          st3(row + 286 + b * 3, heading_rotate(hr, ang));
          tk = row + SELF_DIM;
        }
        TaskObs o;  // task obs v6 block of future step q, common.py:106-176
        task_obs_body(hi, hr, root_pos, pos, rot, vel, ang, r, true, o);
        st3(tk + b * 3, o.d_pos);
        st6_shared(tk + 72 + b * 6, o.d_rot);
        st3(tk + 216 + b * 3, o.d_vel);
        st3(tk + 288 + b * 3, o.d_ang);
        st3(tk + 360 + b * 3, o.l_pos);
        st6_shared(tk + 432 + b * 6, o.l_rot);
      }
    }
    if (q >= 1) {
      fence_proxy_async();  // stage writes -> bulk store
      group_sync(g);        // A: the group's stage complete
      float* srow = stage_base + e * stage_stride;
      if (valid && b == 0) {  // one bulk store per env: the 16-B aligned middle of the segment
        const int body4 = (seg - shift) & ~3;  // floats
        bulk_s2g(dst + shift, srow + 2 * shift, (uint32_t)body4 * 4);
      }
      if (valid && shift && b < 2) dst[b] = srow[shift + b];  // leading pair
      if (valid && b >= 2 && b < 2 + ((seg - shift) & 3)) {   // trailing pair
        const int c = shift + ((seg - shift) & ~3) + (b - 2);
        dst[c] = srow[shift + c];
      }
      if (p.moments) {
        const int64_t c_off = q == 1 ? 0 : SELF_DIM + (int64_t)TASK_DIM * (q - 1);
        const int sl = q == 1 ? STAGE_FLOATS : TASK_DIM;
        for (int c = lt; c < sl; c += GT) {
          double s1 = 0.0, s2 = 0.0;
          for (int ee = 0; ee < nvalid; ++ee) {
            const float* d2 = p.obs + (env0 + ee) * p.obs_stride + c_off;
            const double x = (double)stage_base[ee * stage_stride + (((uintptr_t)d2 & 15) ? 2 : 0) + c];
            s1 += x;
            s2 += x * x;
          }
          double* mom = p.moments + (int64_t)(blockIdx.x % p.moment_buckets) * 2 * W;
          atomicAdd(mom + c_off + c, s1);
          atomicAdd(mom + W + c_off + c, s2);
        }
      }
    }
  }
  if (valid && b == 0) bulk_wait_read();  // shared memory must outlive the last store's reads

  // ---- reductions and scalar outputs (first warp of group 0, which owned q = 0) ------------------
  if (tid < 32) {
    const int le = tid >> 2, k = tid & 3;
    const bool act = le < nvalid && tid < 4 * EPB;
    float term_k = 0.0f;
    if (act) {
      const float kk = k == 0 ? p.rwd.k_pos : k == 1 ? p.rwd.k_rot : k == 2 ? p.rwd.k_vel : p.rwd.k_ang_vel;
      term_k = expf((-kk) * (row_sum24(&S.part[k][le][0]) / 24.0f));  // common.py:298-320
      p.raw[(env0 + le) * p.raw_stride + k] = term_k;
    }
    const int base = tid & ~3;
    const float t0 = __shfl_sync(0xffffffffu, term_k, base), t1 = __shfl_sync(0xffffffffu, term_k, base + 1);
    const float t2 = __shfl_sync(0xffffffffu, term_k, base + 2), t3 = __shfl_sync(0xffffffffu, term_k, base + 3);
    if (act && k == 0) {
      float r = p.rwd.w_pos * t0 + p.rwd.w_rot * t1 + p.rwd.w_vel * t2 + p.rwd.w_ang_vel * t3;
      if (p.dof_force) {
        const float pr = power_reward(p, &S.part[5][le][0], S.prog[le]);
        r += pr;
        p.raw[(env0 + le) * p.raw_stride + p.power_col] = pr;
      }
      p.rew[env0 + le] = r;
      if (p.rew_out) p.rew_out[env0 + le] = r;
    }
    if (act && k == 1) {
      bool fallen = false;
      if (p.early) {
        if (p.use_mean) {
          float sel[J24];
          int m = 0;
#pragma unroll
          for (int j = 0; j < J24; ++j)
            if (p.reset_mask >> j & 1u) sel[m++] = S.part[4][le][j];
          const int first = __ffs(p.reset_mask) - 1;
          fallen = m > 0 && (aten_row_sum(sel, m) / (float)m) > p.term_dist[first < 0 ? 0 : first];
        } else {
          fallen = S.fallen[le] != 0;
        }
        fallen = fallen && (S.prog[le] > 1);  // common.py:353
      }
      const bool rs = S.pass[le] || fallen;  // common.py:362
      p.term[env0 + le] = fallen ? 1 : 0;
      p.reset[env0 + le] = rs ? 1 : 0;
      if (p.term_out) p.term_out[env0 + le] = fallen ? 1 : 0;
      if (p.reset_out) p.reset_out[env0 + le] = rs ? 1 : 0;
    }
    if (act && k == 2 && p.mpjpe) p.mpjpe[env0 + le] = row_sum24(&S.part[4][le][0]) / 24.0f;  // humanoid_phc.py:167
  }
  if (p.ref_dof_pos && tid < EPB * J24 && tid / J24 < nvalid) {  // res_action: dof_pos of the query at t + dt
    const int le = tid / J24;
    write_ref_dof_pos(p, env0 + le, tid % J24, S.row0[1][le], S.row0[1][le] + S.two[1][le], S.bl[1][le]);
  }
}

// ---------------------------------------------------------------------------------------
// RunningNorm kernels (policies/running_norm.py:15-34)
// ---------------------------------------------------------------------------------------
constexpr int MOM_ROWS_PER_BLOCK = 32;
constexpr int MOM_MAX_ROW_BLOCKS = 256;

// grid (ceil(cols / (128*VEC)), ceil(rows / rows_per_block)); a thread owns VEC adjacent columns (coalesced
// across the warp) and walks its rows with 8 independent loads in flight; fp64 partials are merged
// with one atomicAdd per column per block.  fp64 atomics on one address serialise (~30 ns each), so the
// host caps the number of row blocks at MOM_MAX_ROW_BLOCKS by giving each block more rows.
template <int VEC>
__global__ void obs_moments_kernel(const float* __restrict__ x, int64_t rows, int64_t cols, int64_t stride,
                                   int64_t rows_per_block, double* __restrict__ sums) {
  const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_block;
  if (c >= cols) return;
  const int64_t r1 = r0 + rows_per_block < rows ? r0 + rows_per_block : rows;
  double s1[VEC], s2[VEC];
#pragma unroll
  for (int v = 0; v < VEC; ++v) s1[v] = s2[v] = 0.0;
  for (int64_t r = r0; r < r1; r += 8) {
    float vals[8][VEC];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      if (r + u < r1) {
        const float* p = x + (r + u) * stride + c;
        if (VEC == 2) {
          const float2 t = *reinterpret_cast<const float2*>(p);
          vals[u][0] = t.x;
          vals[u][VEC - 1] = t.y;
        } else {
          vals[u][0] = *p;
        }
      } else {
#pragma unroll
        for (int v = 0; v < VEC; ++v) vals[u][v] = 0.0f;
      }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u)
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        const double d = (double)vals[u][v];
        s1[v] += d;
        s2[v] += d * d;
      }
  }
#pragma unroll
  for (int v = 0; v < VEC; ++v)
    if (c + v < cols) {
      atomicAdd(sums + c + v, s1[v]);
      atomicAdd(sums + cols + c + v, s2[v]);
    }
}

// sums[i] += sum_b buckets[b][i] in bucket order; buckets are left zero
__global__ void moments_fold_kernel(double* __restrict__ buckets, int nb, int64_t cols2, double* __restrict__ sums) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cols2) return;
  double acc = sums[i];
  for (int b = 0; b < nb; ++b) {
    acc += buckets[(int64_t)b * cols2 + i];
    buckets[(int64_t)b * cols2 + i] = 0.0;
  }
  sums[i] = acc;
}

__global__ void running_norm_update_kernel(float* __restrict__ mean, float* __restrict__ var,
                                           float* __restrict__ count, const double* __restrict__ sums,
                                           const double* __restrict__ total_rows, int64_t cols) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const double n = *total_rows;
  const float cnt = *count;
  if (c < cols && n > 0) {
    const double m = sums[c] / n;
    double v = sums[cols + c] / n - m * m;  // var(unbiased=False)
    if (v < 0) v = 0;
    const float w = 1.0f / cnt;  // weight = 1 / self.count
    mean[c] = mean[c] * (1.0f - w) + (float)m * w;
    var[c] = var[c] * (1.0f - w) + (float)v * w;
  }
  // count += 1 after every column has read it: done by a second tiny launch
}

__global__ void running_norm_count_kernel(float* count) { *count = *count + 1.0f; }

// one thread per VEC adjacent columns, RN_ROWS rows per block: sqrt once per column, coalesced rows, 8 independent
// loads in flight per thread (the op is 2 x 4 B of traffic per element and nothing else)
constexpr int RN_ROWS = 16;
template <int VEC>
__global__ void running_norm_forward_kernel(const float* __restrict__ x, int64_t rows, int64_t cols, int64_t stride,
                                            const float* __restrict__ mean, const float* __restrict__ var, float eps,
                                            float clip, float* __restrict__ out, int64_t out_stride) {
  const int64_t c = ((int64_t)blockIdx.y * blockDim.x + threadIdx.x) * VEC;
  if (c >= cols) return;
  float m[VEC], sd[VEC];
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    m[v] = mean[c + v];
    sd[v] = sqrtf(var[c + v] + eps);
  }
  const int64_t r0 = (int64_t)blockIdx.x * RN_ROWS;
  const int64_t r1 = r0 + RN_ROWS < rows ? r0 + RN_ROWS : rows;
  for (int64_t r = r0; r < r1; r += 8) {
    float vals[8][VEC];
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if (r + u < r1) {
        const float* p = x + (r + u) * stride + c;
        if (VEC == 2) {
          const float2 t = *reinterpret_cast<const float2*>(p);
          vals[u][0] = t.x;
          vals[u][VEC - 1] = t.y;
        } else {
          vals[u][0] = *p;
        }
      }
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if (r + u < r1) {
        float y[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) y[v] = norm_clamp((vals[u][v] - m[v]) / sd[v], clip);
        float* q = out + (r + u) * out_stride + c;
        if (VEC == 2) *reinterpret_cast<float2*>(q) = make_float2(y[0], y[VEC - 1]);
        else *q = y[0];
      }
  }
}

// -----------------------------------------------------------------------------------------
// K10  episode bookkeeping of the pufferlib wrapper (clean_pufferl/env.py:121-159): one thread
//      per env, ~15 B/env; finished-episode sums and the reward_raw column sums are reduced per
//      block in fp64 and added to a small workspace, the last block folds them into the caller's
//      accumulators and leaves the workspace zero for the next launch.
// -----------------------------------------------------------------------------------------
constexpr int EP_MAX_RAW = 8;
static_assert(PHC_EPISODE_WORKSPACE_DOUBLES >= 13, "workspace layout");  // [0..3] stats, [4..11] reward_raw column sums, [12] block ticket
struct EpisodeParams {
  const uint8_t* reset;
  const uint8_t* terminate;
  const float* rewards;
  const float* reward_raw;
  int64_t raw_stride;
  int raw_cols;
  int64_t n;
  uint8_t* terminals;
  uint8_t* truncations;
  uint8_t* masks;
  float* episode_returns;
  int32_t* episode_lengths;
  double* stats;
  float* raw_rewards;
  double* ws;
};

__global__ void __launch_bounds__(256) episode_update_kernel(EpisodeParams p) {
  double acc[4 + EP_MAX_RAW];
#pragma unroll
  for (int i = 0; i < 4 + EP_MAX_RAW; ++i) acc[i] = 0.0;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < p.n; e += (int64_t)gridDim.x * blockDim.x) {
    const bool rs = p.reset[e] != 0, tm = p.terminate[e] != 0;
    const bool tr = rs && !tm;
    p.terminals[e] = tm ? 1 : 0;
    p.truncations[e] = tr ? 1 : 0;
    p.masks[e] = tr ? 0 : 1;
    float ret = p.episode_returns[e];
    int32_t len = p.episode_lengths[e];
    if (rs) {
      acc[0] += 1.0;
      acc[1] += (double)ret;
      acc[2] += (double)len;
      acc[3] += tr ? 1.0 : 0.0;
      ret = 0.0f;
      len = 0;
    }
    p.episode_returns[e] = ret + p.rewards[e];
    p.episode_lengths[e] = len + 1;
#pragma unroll
    for (int c = 0; c < EP_MAX_RAW; ++c)
      if (c < p.raw_cols) acc[4 + c] += (double)p.reward_raw[e * p.raw_stride + c];
  }
  __shared__ double part[8][4 + EP_MAX_RAW];
  __shared__ bool last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 4 + EP_MAX_RAW; ++i) {
    double v = acc[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) part[warp][i] = v;
  }
  __syncthreads();
  if (threadIdx.x < 4 + p.raw_cols) {
    const int i = threadIdx.x;
    double v = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) v += part[w][i];
    if (v != 0.0) atomicAdd(&p.ws[i], v);
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned long long t = atomicAdd(reinterpret_cast<unsigned long long*>(&p.ws[12]), 1ull);
    last = (t == (unsigned long long)gridDim.x - 1);
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  if (threadIdx.x < 4) {
    p.stats[threadIdx.x] += __ldcg(&p.ws[threadIdx.x]);
    p.ws[threadIdx.x] = 0.0;
  } else if (threadIdx.x < 4 + p.raw_cols) {
    const int c = threadIdx.x - 4;
    p.raw_rewards[c] += (float)(__ldcg(&p.ws[threadIdx.x]) / (double)p.n);
    p.ws[threadIdx.x] = 0.0;
  }
  if (threadIdx.x == 32) *reinterpret_cast<unsigned long long*>(&p.ws[12]) = 0ull;
}

// The same bookkeeping for the step kernels that do not carry it (generic, T > 1): one thread per env after the step,
// block sums into the bucket of the block.  raw_post: NULL, or where the env's reward_raw row (dense, raw_stride
// columns) is posted after it is read from p.raw (the host pipeline's mapped outputs: step_fused_mirrored).
__global__ void __launch_bounds__(256) episode_bucket_kernel(StepParams p, float* raw_post) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  double v[EP_SUM_COLS];
#pragma unroll
  for (int i = 0; i < EP_SUM_COLS; ++i) v[i] = 0.0;
  if (e < p.n) {
    const bool rs = p.reset[e] != 0, tm = p.term[e] != 0, tr = rs && !tm;
    p.ep_terminals[e] = tm ? 1 : 0;
    p.ep_truncations[e] = tr ? 1 : 0;
    p.ep_masks[e] = tr ? 0 : 1;
    float ret = p.ep_returns[e];
    int32_t len = p.ep_lengths[e];
    if (rs) {
      v[0] = 1.0;
      v[1] = (double)ret;
      v[2] = (double)len;
      v[3] = tr ? 1.0 : 0.0;
      ret = 0.0f;
      len = 0;
    }
    p.ep_returns[e] = ret + p.rew[e];
    p.ep_lengths[e] = len + 1;
#pragma unroll
    for (int c = 0; c < EP_SUM_COLS - 4; ++c)
      if (c < p.ep_raw_cols) v[4 + c] = (double)p.raw[e * p.raw_stride + c];
    if (raw_post)
      for (int64_t c = 0; c < p.raw_stride; ++c) raw_post[e * p.raw_stride + c] = p.raw[e * p.raw_stride + c];
  }
  __shared__ double part[8][EP_SUM_COLS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < EP_SUM_COLS; ++i) {
    double x = v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0) part[warp][i] = x;
  }
  __syncthreads();
  if (threadIdx.x < 4 + p.ep_raw_cols) {
    double x = 0.0;
    for (int w = 0; w < 8; ++w) x += part[w][threadIdx.x];
    if (x != 0.0)
      atomicAdd(p.ep_sums + (int64_t)((p.ep_block0 + blockIdx.x) % p.ep_buckets) * EP_SUM_COLS + threadIdx.x, x);
  }
}

// stats[i] += sum_b sums[b][i] (i < 4), raw_rewards[c] += sum_b sums[b][4 + c] / n; the buckets are left zero
__global__ void episode_fold_kernel(double* __restrict__ sums, int nb, int raw_cols, double n, double* __restrict__ stats,
                                    float* __restrict__ raw_rewards) {
  const int i = threadIdx.x;
  if (i >= 4 + raw_cols) return;
  double acc = 0.0;
  for (int b = 0; b < nb; ++b) {
    acc += sums[b * EP_SUM_COLS + i];
    sums[b * EP_SUM_COLS + i] = 0.0;
  }
  if (i < 4) stats[i] += acc;
  else raw_rewards[i - 4] += (float)(acc / n);
}

}  // namespace phc

// =========================================================================================
// C ABI
// =========================================================================================
using namespace phc;

static int g_moments_bulk = -1;  // PHC_OPT_MOMENTS_BULK / env PHC_MOMENTS_BULK=0|1 (default 0: measured no faster than the atomics)
static int g_persist = -1;       // PHC_OPT_STEP_PERSIST / env PHC_STEP_PERSIST: 0 never, 1 from g_persist_min envs on (default), 2 always,
                                 // 3 always and the 4-slot / 4-blocks-per-SM instantiation
static int g_persist_pdl = 1;
static int64_t g_persist_min = 10240;  // measured crossover between 8192 (K6-fast 13.9 us, persistent 15.5) and 10240 (19.95 / 18.49)
static int64_t g_persist_min_moments = 8192;  // with obs_moments: K6-fast pays 1868 L2 adds per four envs

template <typename Kern>
static int launch_step(Kern kern, size_t smem, int epb, const StepParams& p, cudaStream_t stream, bool* attr_set,
                       bool pdl) {
  if (!*attr_set) {
    PHC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    *attr_set = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)((p.n + epb - 1) / epb));
  cfg.blockDim = dim3((unsigned)(epb * J24));
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl ? 1 : 0;
  PHC_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
  return launch_status();
}

struct PhcLib {
  LibDev d;
  float* packed_owned = nullptr;
  // The fast step kernel reads clip metadata and frame rows BEFORE griddepcontrol.wait (it treats the library as
  // immutable).  A launch that (re)writes the library on the same stream — phc_lib_pack, phc_motion_build followed
  // by phc_lib_pack, or the caller's own kernels before phc_lib_create — is only ordered before the step's
  // post-wait reads, so the first fused step after phc_lib_create / phc_lib_pack runs without the speculation.
  mutable std::atomic<int> unspeculated_steps{1};
  // tile counters of the persistent step kernel: every launch draws the next of TILE_SLOTS slots (two words that the
  // launch leaves zero), so launches that overlap on different streams do not share one
  unsigned* tile_counters = nullptr;
  mutable std::atomic<unsigned> tile_seq{0};  // host threads may launch steps of one library concurrently
};
constexpr unsigned TILE_SLOTS = 256;

extern "C" {

const char* phc_strerror(int code) {
  switch (code) {
    case PHC_OK: return "ok";
    case PHC_ERR_NULL: return "required pointer is NULL";
    case PHC_ERR_SHAPE: return "size or count out of range";
    case PHC_ERR_ALIGN: return "pointer or stride not aligned as required";
    case PHC_ERR_UNSUPPORTED: return "not supported by this build";
    case PHC_ERR_CUDA: return "CUDA runtime error";
    case PHC_ERR_ALLOC: return "allocation failed";
    case PHC_PEER_TIMEOUT: return "a peer rank did not publish its partials in time";
    case PHC_ERR_BUSY: return "the host-step slot already has a step in flight";
    default: return "unknown error";
  }
}

int phc_abi_version(void) { return PHC_ABI_VERSION; }
int phc_last_cuda_error(void) { return g_last_cuda_error; }

int phc_lib_create(const PhcLibDesc* desc, PhcLib** out) {
  if (!desc || !out) return PHC_ERR_NULL;
  if (!desc->gts || !desc->grs || !desc->gvs || !desc->gavs || !desc->motion_lengths ||
      !desc->motion_num_frames || !desc->motion_dt || !desc->length_starts)
    return PHC_ERR_NULL;
  if (desc->total_frames <= 0 || desc->num_motions <= 0) return PHC_ERR_SHAPE;
  // frame rows are fetched with 16-byte copies: 288 / 384 B rows keep the alignment of the base
  const uintptr_t a = (uintptr_t)desc->gts | (uintptr_t)desc->grs | (uintptr_t)desc->gvs | (uintptr_t)desc->gavs |
                      (uintptr_t)desc->lrs;
  if (a & 15) return PHC_ERR_ALIGN;
  PhcLib* lib = new (std::nothrow) PhcLib;
  if (!lib) return PHC_ERR_ALLOC;
  lib->d = LibDev{desc->gts,           desc->grs,        desc->lrs,          desc->gvs,
                  desc->gavs,          desc->dvs,        desc->motion_aa,    desc->motion_lengths,
                  desc->motion_dt,     desc->motion_bodies, desc->motion_limb_weights,
                  desc->motion_num_frames, desc->length_starts, desc->total_frames, desc->num_motions, nullptr};
  *out = lib;
  return PHC_OK;
}

int phc_lib_pack(PhcLib* lib, phc_stream_t stream) {
  if (!lib) return PHC_ERR_NULL;
  if (!lib->packed_owned) {
    cudaError_t e = cudaMalloc((void**)&lib->packed_owned, (size_t)lib->d.F * FRAME_FLOATS * sizeof(float));
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      g_last_cuda_error = (int)e;
      return PHC_ERR_ALLOC;
    }
  }
  if (!lib->tile_counters) {
    cudaError_t e = cudaMalloc((void**)&lib->tile_counters, TILE_SLOTS * 2 * sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMemsetAsync(lib->tile_counters, 0, TILE_SLOTS * 2 * sizeof(unsigned), stream);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      g_last_cuda_error = (int)e;
      lib->tile_counters = nullptr;
      return PHC_ERR_ALLOC;
    }
  }
  const int64_t total4 = lib->d.F * 78;
  const unsigned grid = (unsigned)((total4 + 255) / 256 < 148 * 16 ? (total4 + 255) / 256 : 148 * 16);
  pack_frames_kernel<<<grid, 256, 0, stream>>>(lib->d, lib->packed_owned);
  int rc = launch_status();
  if (rc) return rc;
  lib->d.packed = lib->packed_owned;
  lib->unspeculated_steps = 1;  // the next fused step must not read the table before its dependency wait
  return PHC_OK;
}

void phc_lib_destroy(PhcLib* lib) {
  if (!lib) return;
  if (lib->packed_owned) cudaFree(lib->packed_owned);
  if (lib->tile_counters) cudaFree(lib->tile_counters);
  delete lib;
}

int phc_calc_frame_blend(const float* time, const float* len, const int64_t* num_frames, const float* dt,
                         int64_t n, int64_t* frame_idx0, int64_t* frame_idx1, float* blend, phc_stream_t stream) {
  if (n == 0) return PHC_OK;
  if (n < 0) return PHC_ERR_SHAPE;
  if (!time || !len || !num_frames || !dt || !frame_idx0 || !frame_idx1 || !blend) return PHC_ERR_NULL;
  const int bs = 256;
  frame_blend_kernel<<<(unsigned)((n + bs - 1) / bs), bs, 0, stream>>>(time, len, num_frames, dt, n, frame_idx0,
                                                                        frame_idx1, blend);
  return launch_status();
}

int phc_motion_state(const PhcLib* lib, const int64_t* motion_ids, const float* motion_times,
                     const float* offset_or_null, int64_t n, const PhcMotionOut* out, phc_stream_t stream) {
  if (n == 0) return PHC_OK;
  if (n < 0) return PHC_ERR_SHAPE;
  if (!lib || !motion_ids || !motion_times || !out) return PHC_ERR_NULL;
  if (out->dof_pos && !lib->d.lrs) return PHC_ERR_NULL;
  if (out->dof_vel && !lib->d.dvs) return PHC_ERR_NULL;
  if (out->motion_aa && !lib->d.aa) return PHC_ERR_NULL;
  if (out->motion_bodies && !lib->d.bodies) return PHC_ERR_NULL;
  if (out->motion_limb_weights && !lib->d.limb) return PHC_ERR_NULL;
  const unsigned grid = (unsigned)((n + K1_QPB - 1) / K1_QPB);
  motion_state_kernel<<<grid, K1_QPB * J24, 0, stream>>>(lib->d, motion_ids, motion_times, offset_or_null, n, *out);
  return launch_status();
}

static int check_body(const PhcBodyState* s) {
  if (!s) return PHC_ERR_NULL;
  if (!s->pos.ptr || !s->rot.ptr || !s->vel.ptr || !s->ang_vel.ptr) return PHC_ERR_NULL;
  if (s->num_bodies < 1 || s->num_bodies > GEN_MAX_J) return PHC_ERR_SHAPE;
  return PHC_OK;
}

int phc_self_obs_smpl_max(const PhcBodyState* body, int64_t n, uint32_t flags, float* out, int64_t out_stride,
                          phc_stream_t stream) {
  if (n == 0) return PHC_OK;
  if (n < 0) return PHC_ERR_SHAPE;
  int rc = check_body(body);
  if (rc) return rc;
  if (!out) return PHC_ERR_NULL;
  const int J = body->num_bodies;
  const int width = ((flags & PHC_OBS_ROOT_HEIGHT) ? 1 : 0) + 15 * J - 3;
  if (out_stride < width) return PHC_ERR_SHAPE;
  const int epb = 192 / J > 0 ? 192 / J : 1;
  self_obs_kernel<<<(unsigned)((n + epb - 1) / epb), epb * J, 0, stream>>>(*body, n, flags, out, out_stride, epb);
  return launch_status();
}

int phc_imitation_obs(const float* root_pos, int64_t root_pos_stride, const float* root_rot, int64_t root_rot_stride,
                      const PhcBodyState* body, const PhcBodyState* ref, int64_t n, int32_t time_steps,
                      int32_t upright, int32_t mode, float* out, int64_t out_stride, phc_stream_t stream) {
  if (n == 0) return PHC_OK;
  if (n < 0 || time_steps < 1) return PHC_ERR_SHAPE;
  int rc = check_body(body);
  if (rc) return rc;
  rc = check_body(ref);
  if (rc) return rc;
  if (!root_pos || !root_rot || !out) return PHC_ERR_NULL;
  if (ref->num_bodies != body->num_bodies) return PHC_ERR_SHAPE;
  if (mode != 6 && mode != 7) return PHC_ERR_UNSUPPORTED;
  const int J = body->num_bodies;
  const int64_t width = (int64_t)(mode == 6 ? 24 : 9) * J * time_steps;
  if (out_stride < width) return PHC_ERR_SHAPE;
  const int64_t total = n * time_steps * J;
  const int bs = 192;
  imitation_obs_kernel<<<(unsigned)((total + bs - 1) / bs), bs, 0, stream>>>(
      root_pos, root_pos_stride, root_rot, root_rot_stride, *body, *ref, n, time_steps, upright, mode, out, out_stride);
  return launch_status();
}

int phc_amp_obs(const PhcAmpArgs* a, int64_t n, float* out, int64_t out_stride, phc_stream_t stream) {
  if (n == 0) return PHC_OK;
  if (n < 0) return PHC_ERR_SHAPE;
  if (!a || !out || !a->root_pos || !a->root_rot || !a->root_vel || !a->root_ang_vel || !a->dof_pos || !a->dof_vel ||
      !a->key_body_pos.ptr)
    return PHC_ERR_NULL;
  if (a->num_sel < 0 || a->num_sel % 3 != 0 || a->num_sel > 96 || a->num_key_bodies < 0 || a->num_key_bodies > 8)
    return PHC_ERR_SHAPE;
  const int width = ((a->flags & PHC_OBS_ROOT_HEIGHT) ? 1 : 0) + 12 + 3 * a->num_sel + 3 * a->num_key_bodies;
  if (out_stride < width) return PHC_ERR_SHAPE;
  const int epb = 4;
  amp_obs_kernel<<<(unsigned)((n + epb - 1) / epb), epb * 32, 0, stream>>>(*a, n, out, out_stride);
  return launch_status();
}

int phc_imitation_reward(const PhcBodyState* body, const PhcBodyState* ref, int64_t n, const PhcRewardSpec* spec,
                         float* reward, float* reward_raw, int64_t reward_raw_stride, phc_stream_t stream) {
  if (n == 0) return PHC_OK;
  if (n < 0) return PHC_ERR_SHAPE;
  int rc = check_body(body);
  if (rc) return rc;
  rc = check_body(ref);
  if (rc) return rc;
  if (!spec || !reward || !reward_raw) return PHC_ERR_NULL;
  if (ref->num_bodies != body->num_bodies || reward_raw_stride < 4) return PHC_ERR_SHAPE;
  const int J = body->num_bodies;
  const int epb = 192 / J > 0 ? 192 / J : 1;
  const size_t sm = (size_t)epb * 4 * (J + 1) * sizeof(float);
  reward_kernel<<<(unsigned)((n + epb - 1) / epb), epb * J, sm, stream>>>(*body, *ref, n, *spec, reward, reward_raw,
                                                                         reward_raw_stride, epb);
  return launch_status();
}

int phc_im_reset(const PhcView* rigid_body_pos, const PhcView* ref_body_pos, int32_t num_reset_bodies,
                 const int16_t* progress_buf, const uint8_t* pass_time, const float* termination_distance,
                 int32_t enable_early_termination, int32_t use_mean, int64_t n, uint8_t* reset, uint8_t* terminated,
                 phc_stream_t stream) {
  if (n == 0) return PHC_OK;
  if (n < 0 || num_reset_bodies < 1 || num_reset_bodies > GEN_MAX_J) return PHC_ERR_SHAPE;
  if (!rigid_body_pos || !ref_body_pos || !rigid_body_pos->ptr || !ref_body_pos->ptr || !progress_buf || !pass_time ||
      !termination_distance || !reset || !terminated)
    return PHC_ERR_NULL;
  const int R = num_reset_bodies;
  const int epb = 192 / R > 0 ? 192 / R : 1;
  reset_kernel<<<(unsigned)((n + epb - 1) / epb), epb * R, (size_t)epb * R * sizeof(float), stream>>>(
      *rigid_body_pos, *ref_body_pos, R, progress_buf, pass_time, termination_distance, enable_early_termination,
      use_mean, n, reset, terminated, epb);
  return launch_status();
}

// ---- fused step --------------------------------------------------------------------------
constexpr int STEP_EPB = 8;

static int g_spec_fault = 0;  // PHC_OPT_TEST_SPEC_FAULT
static int g_multi_groups = 0;  // PHC_OPT_MULTI_GROUPS: 0 = default (2)
static unsigned long long* g_trace = nullptr;  // phc_set_trace_buffer (profiling only)
static int64_t g_trace_capacity = 0;
static int64_t g_trace_launch = 0;

static ObsFlags obs_flags_from(uint32_t f) {
  ObsFlags of;
  of.v7 = (f & PHC_OBS_TASK_V7) ? 1 : 0;  // whatever the self-obs bits say
  if (!(f & PHC_STEP_OBS_FLAGS_SET) && (f & 7u) == 0) f = PHC_OBS_LOCAL_ROOT | PHC_OBS_ROOT_HEIGHT | PHC_OBS_UPRIGHT;
  of.hcol = (f & PHC_OBS_ROOT_HEIGHT) ? 1 : 0;
  of.local_root = (f & PHC_OBS_LOCAL_ROOT) ? 1 : 0;
  of.upright = (f & PHC_OBS_UPRIGHT) ? 1 : 0;
  return of;
}

static int reset_fill(const PhcLib* lib, const PhcResetArgs* a, int64_t n, ResetParams& r) {
  if (n < 0) return PHC_ERR_SHAPE;
  if (!lib || !a) return PHC_ERR_NULL;
  int rc = check_body(&a->body);
  if (rc) return rc;
  if (a->body.num_bodies != J24) return PHC_ERR_UNSUPPORTED;
  if (!a->progress_buf || !a->reset_buf || !a->terminate_buf || !a->motion_start_times ||
      !a->motion_start_times_offset || !a->sampled_motion_ids || !a->obs_buf)
    return PHC_ERR_NULL;
  if (a->state_init < PHC_STATE_INIT_START || a->state_init > PHC_STATE_INIT_HYBRID) return PHC_ERR_UNSUPPORTED;
  const bool samples = a->state_init == PHC_STATE_INIT_RANDOM || a->state_init == PHC_STATE_INIT_HYBRID;
  if (samples && !a->flag_test && !a->phase) return PHC_ERR_NULL;
  if (a->state_init >= PHC_STATE_INIT_DEFAULT) {
    if (a->state_init == PHC_STATE_INIT_HYBRID && !a->default_mask) return PHC_ERR_NULL;
    if ((a->humanoid_root_states && !a->initial_root_states) || (a->dof_pos && !a->initial_dof_pos) ||
        (a->dof_vel && !a->initial_dof_vel))
      return PHC_ERR_NULL;
    if ((a->humanoid_root_states && a->initial_root_stride < 13) || ((a->dof_pos || a->dof_vel) && a->initial_dof_stride < 69))
      return PHC_ERR_SHAPE;
  }
  if ((a->dof_pos && !lib->d.lrs) || (a->dof_vel && !lib->d.dvs) || (a->ref_dof_pos && !lib->d.lrs)) return PHC_ERR_NULL;
  if (a->time_steps < 1 || a->time_steps > PHC_MAX_TIME_STEPS) return PHC_ERR_SHAPE;
  const ObsFlags of = obs_flags_from(a->obs_flags);
  const int64_t W = 357 + of.hcol + (int64_t)task_width(of) * a->time_steps;
  if (a->obs_stride < W || ((a->dof_pos || a->dof_vel) && a->dof_elem_stride < 1)) return PHC_ERR_SHAPE;
  if (a->obs_norm && (!a->norm_mean || !a->norm_var)) return PHC_ERR_NULL;
  if (a->obs_norm && (a->obs_norm_stride < W || !(a->norm_clip > 0.0f))) return PHC_ERR_SHAPE;
  if (a->obs_moments_mode < 0 || a->obs_moments_mode > 2 || a->obs_moments_buckets < 0 || a->obs_moments_buckets > 4096)
    return PHC_ERR_SHAPE;
  if (a->obs_moments_mode && !a->obs_moments) return PHC_ERR_NULL;
  if (a->ref_dof_pos && a->ref_dof_pos_stride < 69) return PHC_ERR_SHAPE;
  r = ResetParams{};
  r.L = lib->d;
  r.w.body = a->body;
  r.w.root = a->humanoid_root_states;
  r.w.root_stride = a->root_stride;
  r.w.dof_pos = a->dof_pos;
  r.w.dof_vel = a->dof_vel;
  r.w.dof_stride = a->dof_stride;
  r.w.dof_estride = a->dof_elem_stride;
  r.w.progress = a->progress_buf;
  r.w.reset = a->reset_buf;
  r.w.term = a->terminate_buf;
  r.w.start = a->motion_start_times;
  r.w.start_off = a->motion_start_times_offset;
  r.w.goff = a->global_offset;
  r.w.phase = a->phase;
  r.w.state_init = a->state_init;
  r.w.flag_test = a->flag_test;
  r.w.init_root = a->initial_root_states;
  r.w.init_root_stride = a->initial_root_stride;
  r.w.init_dof_pos = a->initial_dof_pos;
  r.w.init_dof_vel = a->initial_dof_vel;
  r.w.init_dof_stride = a->initial_dof_stride;
  r.w.default_mask = a->default_mask;
  r.ids = a->sampled_motion_ids;
  r.mask = a->env_mask;
  r.n = n;
  r.obs = a->obs_buf;  // _compute_observations(env_ids), same launch
  r.obs_stride = a->obs_stride;
  r.T = a->time_steps;
  r.dt = a->dt;
  r.of = of;
  r.norm = NormOut{a->obs_norm, a->obs_norm_stride, a->norm_mean, a->norm_var, a->norm_epsilon, a->norm_clip,
                   a->obs_norm_bf16 ? 1 : 0};
  r.moments = a->obs_moments_mode ? a->obs_moments : nullptr;
  r.moment_buckets = a->obs_moments_buckets > 1 ? a->obs_moments_buckets : 1;
  r.moments_mode = a->obs_moments_mode;
  r.ref_dof_pos = a->ref_dof_pos;
  r.ref_dof_pos_stride = a->ref_dof_pos_stride;
  return PHC_OK;
}

static int reset_launch(const ResetParams& r, cudaStream_t stream) {
  reset_obs_kernel<<<(unsigned)((r.n + K7_EPB - 1) / K7_EPB), K7_EPB * J24, 0, stream>>>(r);
  return launch_status();
}

static int step_fill_params(const PhcLib* lib, const PhcStepArgs* a, int64_t n, StepParams& p) {
  if (!lib || !a) return PHC_ERR_NULL;
  int rc = check_body(&a->body);
  if (rc) return rc;
  if (a->body.num_bodies != J24) return PHC_ERR_UNSUPPORTED;
  if (!a->progress_buf || !a->motion_start_times || !a->motion_start_times_offset || !a->sampled_motion_ids ||
      !a->termination_distances || !a->obs_buf || !a->rew_buf || !a->reward_raw || !a->reset_buf || !a->terminate_buf)
    return PHC_ERR_NULL;
  if (a->time_steps < 1 || a->time_steps > PHC_MAX_TIME_STEPS) return PHC_ERR_SHAPE;
  p.of = obs_flags_from(a->obs_flags);
  p.selfw = 357 + p.of.hcol;
  const int64_t W = p.selfw + (int64_t)task_width(p.of) * a->time_steps;
  if (a->obs_stride < W || a->reward_raw_stride < 4) return PHC_ERR_SHAPE;
  p.rew_out = a->rew_out;
  p.reset_out = a->reset_out;
  p.term_out = a->terminate_out;
  p.ref_dof_pos = a->ref_dof_pos;
  p.ref_dof_pos_stride = a->ref_dof_pos_stride;
  if (a->ref_dof_pos && (!lib->d.lrs || a->ref_dof_pos_stride < 69)) return lib->d.lrs ? PHC_ERR_SHAPE : PHC_ERR_NULL;
  p.reset_on = 0;
  p.rw = ResetTargets{};
  p.tile_counter = nullptr;
  if (a->auto_reset) {
    // the reset rides on the step's own buffers: anything else would not be "the envs this step flags"
    const PhcResetArgs* r = a->auto_reset;
    if (r->body.pos.ptr != a->body.pos.ptr || r->body.rot.ptr != a->body.rot.ptr || r->body.vel.ptr != a->body.vel.ptr ||
        r->body.ang_vel.ptr != a->body.ang_vel.ptr || r->body.pos.stride_env != a->body.pos.stride_env ||
        r->body.pos.stride_body != a->body.pos.stride_body || r->progress_buf != a->progress_buf ||
        r->reset_buf != a->reset_buf || r->terminate_buf != a->terminate_buf || r->obs_buf != a->obs_buf ||
        r->obs_stride != a->obs_stride || r->sampled_motion_ids != a->sampled_motion_ids ||
        r->motion_start_times != a->motion_start_times || r->motion_start_times_offset != a->motion_start_times_offset ||
        r->global_offset != a->global_offset || r->time_steps != a->time_steps || r->dt != a->dt)
      return PHC_ERR_SHAPE;
    const ObsFlags rf = obs_flags_from(r->obs_flags);
    if (rf.hcol != p.of.hcol || rf.local_root != p.of.local_root || rf.upright != p.of.upright || rf.v7 != p.of.v7)
      return PHC_ERR_SHAPE;
    ResetParams rp;
    rc = reset_fill(lib, r, n, rp);
    if (rc) return rc;
    if (r->ref_dof_pos != a->ref_dof_pos) return PHC_ERR_SHAPE;
    p.rw = rp.w;
    p.reset_on = 1;
  }
  p.L = lib->d;
  p.body = a->body;
  p.progress = a->progress_buf;
  p.progress_mirror = nullptr;
  p.start = a->motion_start_times;
  p.start_off = a->motion_start_times_offset;
  p.goff = a->global_offset;
  p.ids = a->sampled_motion_ids;
  p.term_dist = a->termination_distances;
  p.reset_mask = a->reset_body_mask & 0xFFFFFFu;
  p.use_mean = a->use_mean;
  p.early = a->enable_early_termination;
  p.advance = a->advance_progress;
  p.T = a->time_steps;
  p.dt = a->dt;
  p.one = 1.0f;
  p.rwd = a->rwd;
  p.obs = a->obs_buf;
  p.obs_stride = a->obs_stride;
  p.rew = a->rew_buf;
  p.raw = a->reward_raw;
  p.raw_stride = a->reward_raw_stride;
  p.reset = a->reset_buf;
  p.term = a->terminate_buf;
  p.moments = a->obs_moments;
  p.moment_buckets = a->obs_moments_buckets > 1 ? a->obs_moments_buckets : 1;
  p.moments_bulk = 0;
  {
    static int mp = -1;  // env PHC_MULTI_PREFETCH=0|1 (default 1)
    if (mp < 0) {
      const char* w = getenv("PHC_MULTI_PREFETCH");
      mp = (w && w[0] == '0') ? 0 : 1;
    }
    p.multi_prefetch = mp;
  }
  p.ep_terminals = a->ep_terminals;
  p.ep_truncations = a->ep_truncations;
  p.ep_masks = a->ep_masks;
  p.ep_returns = a->ep_returns;
  p.ep_lengths = a->ep_lengths;
  p.ep_sums = a->ep_sums;
  p.ep_buckets = a->ep_buckets;
  p.ep_raw_cols = a->ep_raw_cols;
  p.ep_block0 = 0;
  if (a->ep_returns) {
    if (!a->ep_terminals || !a->ep_truncations || !a->ep_masks || !a->ep_lengths || !a->ep_sums) return PHC_ERR_NULL;
    if (a->ep_buckets < 1 || a->ep_buckets > 4096 || a->ep_raw_cols < 0 || a->ep_raw_cols > EP_SUM_COLS - 4) return PHC_ERR_SHAPE;
  }
  if (a->obs_moments_buckets < 0 || a->obs_moments_buckets > 4096) return PHC_ERR_SHAPE;
  p.mpjpe = a->mpjpe;
  p.obs_norm = a->obs_norm;
  p.obs_norm_stride = a->obs_norm_stride;
  p.norm_mean = a->norm_mean;
  p.norm_var = a->norm_var;
  p.norm_eps = a->norm_epsilon;
  p.norm_clip = a->norm_clip;
  p.norm_bf16 = (a->flags & PHC_STEP_OBS_NORM_BF16) ? 1 : 0;
  if (a->obs_norm) {
    if (!a->norm_mean || !a->norm_var) return PHC_ERR_NULL;
    if (a->obs_norm_stride < W || !(a->norm_clip > 0.0f)) return PHC_ERR_SHAPE;
  }
  p.dof_force = a->dof_force;
  p.dof_force_stride = a->dof_force_stride;
  p.dof_vel = a->dof_vel;
  p.dof_vel_stride = a->dof_vel_stride;
  p.dof_vel_estride = a->dof_vel_elem_stride;
  p.power_coef = a->rew_power_coef;
  p.power_col = a->power_col;
  if (a->dof_force) {
    if (!a->dof_vel) return PHC_ERR_NULL;
    if (a->power_col < 4 || a->power_col >= a->reward_raw_stride || a->dof_force_stride < 69 ||
        a->dof_vel_elem_stride < 1)
      return PHC_ERR_SHAPE;
  }
  p.first_wave_blocks = 0;
  p.spec4_blocks = 0;
  p.spec_fault = g_spec_fault;
  p.env_mask = nullptr;
  p.obs_only = 0;
  {  // profiling only: consecutive launches stamp consecutive slices of the trace buffer
    const int64_t nw = (n + 3) / 4 * 3;
    if (g_trace && (g_trace_launch + 1) * nw <= g_trace_capacity) {
      p.trace = g_trace + g_trace_launch * nw * 8;
      ++g_trace_launch;
    } else {
      p.trace = nullptr;
    }
  }
  p.n = n;
  const PhcBodyState& s = a->body;
  // fast path: the four views are slices of one AoS-13 tensor whose env rows are 16-B aligned
  p.aos = s.rot.ptr == s.pos.ptr + 3 && s.vel.ptr == s.pos.ptr + 7 && s.ang_vel.ptr == s.pos.ptr + 10 &&
          s.pos.stride_body == 13 && s.rot.stride_body == 13 && s.vel.stride_body == 13 &&
          s.ang_vel.stride_body == 13 && s.rot.stride_env == s.pos.stride_env &&
          s.vel.stride_env == s.pos.stride_env && s.ang_vel.stride_env == s.pos.stride_env &&
          ((uintptr_t)s.pos.ptr & 15) == 0 && (s.pos.stride_env % 4) == 0 && s.pos.stride_env >= ROW13;
  p.obs_vec2 = ((uintptr_t)a->obs_buf & 7) == 0 && (a->obs_stride % 2) == 0;
  return PHC_OK;
}

static int g_force_generic = -1;  // PHC_OPT_FORCE_GENERIC_STEP / env PHC_STEP_GENERIC=1
static int g_fast_epb = -1;       // PHC_OPT_STEP_EPB / env PHC_STEP_EPB=4|8
static int g_pdl = -1;            // PHC_OPT_STEP_PDL / env PHC_STEP_PDL=0|1 (default 1)

static void init_options() {
  if (g_force_generic < 0) {
    const char* v = getenv("PHC_STEP_GENERIC");
    g_force_generic = (v && v[0] == '1') ? 1 : 0;
  }
  if (g_fast_epb < 0) {
    const char* w = getenv("PHC_STEP_EPB");
    g_fast_epb = (w && w[0] == '8') ? 8 : 4;
  }
  if (g_pdl < 0) {
    const char* w = getenv("PHC_STEP_PDL");
    g_pdl = (w && w[0] == '0') ? 0 : 1;
  }
  if (g_moments_bulk < 0) {
    const char* w = getenv("PHC_MOMENTS_BULK");
    g_moments_bulk = (w && w[0] == '1') ? 1 : 0;
  }
  if (g_persist < 0) {
    const char* w = getenv("PHC_STEP_PERSIST");
    g_persist = (w && w[0] >= '0' && w[0] <= '3') ? w[0] - '0' : 1;
    g_persist_pdl = g_pdl;
    const char* m = getenv("PHC_STEP_PERSIST_MIN");
    if (m && atoll(m) > 0) g_persist_min = atoll(m);
  }
}

int phc_action_to_pd_targets(const float* action, const float* pd_action_offset, const float* pd_action_scale,
                             int32_t res_action, const float* ref_dof_pos, const float* dof_pos,
                             int64_t dof_pos_stride, int64_t dof_pos_elem_stride, uint32_t zero_mask, int64_t n,
                             int32_t num_dof, float action_clip, float* actions_out, float* out, phc_stream_t stream) {
  if (n == 0) return PHC_OK;
  if (n < 0 || num_dof < 1 || num_dof > 96 || !(action_clip >= 0.0f)) return PHC_ERR_SHAPE;
  if (!action || !pd_action_scale || !out) return PHC_ERR_NULL;
  if (res_action ? (!ref_dof_pos || !dof_pos) : !pd_action_offset) return PHC_ERR_NULL;
  const int64_t total = n * num_dof;
  pd_targets_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(action, pd_action_offset, pd_action_scale,
                                                                         res_action, ref_dof_pos, dof_pos, dof_pos_stride,
                                                                         dof_pos_elem_stride, zero_mask, n, num_dof,
                                                                         action_clip, actions_out, out);
  return launch_status();
}

int phc_reset_envs(const PhcLib* lib, const PhcResetArgs* a, int64_t n, phc_stream_t stream) {
  if (n == 0) return PHC_OK;
  ResetParams r;
  const int rc = reset_fill(lib, a, n, r);
  if (rc) return rc;
  if (!a->env_mask) return PHC_ERR_NULL;
  return reset_launch(r, stream);
}

int phc_set_trace_buffer(uint64_t* device_buf, int64_t capacity_warps) {
  g_trace = (unsigned long long*)device_buf;
  g_trace_capacity = device_buf ? capacity_warps : 0;
  g_trace_launch = 0;
  return PHC_OK;
}

int phc_set_option(int key, int value) {
  init_options();
  switch (key) {
    case PHC_OPT_FORCE_GENERIC_STEP:
      g_force_generic = value ? 1 : 0;
      return PHC_OK;
    case PHC_OPT_STEP_EPB:
      if (value != 4) return PHC_ERR_SHAPE;
      g_fast_epb = value;
      return PHC_OK;
    case PHC_OPT_STEP_PDL:
      g_pdl = value ? 1 : 0;
      g_persist_pdl = g_pdl;
      return PHC_OK;
    case PHC_OPT_TEST_SPEC_FAULT:
      g_spec_fault = value;
      return PHC_OK;
    case PHC_OPT_MULTI_GROUPS:
      if (value < 0 || value > 2) return PHC_ERR_SHAPE;
      g_multi_groups = value;
      return PHC_OK;
    case PHC_OPT_MOMENTS_BULK:
      g_moments_bulk = value ? 1 : 0;
      return PHC_OK;
    case PHC_OPT_STEP_PERSIST:
      if (value < 0 || value > 3) return PHC_ERR_SHAPE;
      g_persist = value;
      return PHC_OK;
    default:
      return PHC_ERR_UNSUPPORTED;
  }
}

}  // extern "C"

// phc_step_fused for one chunk of the host pipeline (phc_host.cu).
//   progress_mirror  NULL, or a second place (the caller's pinned buffer) that receives the advanced progress.
//   env0             the chunk's first env in the batch.  The episode bookkeeping takes its buckets by the block's index
//                    in the batch, so chunks do not pile onto the first rows: the T = 1 kernel's blocks (4 envs, chunks
//                    start on multiples of 8) are the device path's blocks; episode_bucket_kernel's (256 envs) cannot be,
//                    and start at the next row after the previous chunk's.
//   ep_raw           NULL, or device scratch [n, reward_raw_stride] when the step's outputs are mapped host memory and
//                    the episode bookkeeping is on: where the bookkeeping runs after the step it must not read those
//                    back over the link, so the step leaves reward_raw here, the bookkeeping reads it and the step's
//                    device copies rew_out / reset_out / terminate_out (which the caller sets), and posts the raw rows.
int step_fused_mirrored(const PhcLib* lib, const PhcStepArgs* args, int64_t n, phc_stream_t stream,
                        int16_t* progress_mirror, int64_t env0, float* ep_raw) {
  if (n == 0) return PHC_OK;
  if (n < 0 || env0 < 0) return PHC_ERR_SHAPE;
  StepParams p;
  int rc = step_fill_params(lib, args, n, p);
  if (rc) return rc;
  if (!p.ep_returns) ep_raw = nullptr;
  if (ep_raw && (!p.rew_out || !p.reset_out || !p.term_out)) return PHC_ERR_NULL;
  p.progress_mirror = progress_mirror;
  int dev = 0;
  PHC_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return PHC_ERR_UNSUPPORTED;
  init_options();
  // fast path: T == 1, AoS sim tensor (16-B aligned rows), dense 16-B aligned obs_buf.  Any self-obs flag combination
  // runs on it (rows of 933 floats without the height column: four of them are still a multiple of 16 B); the fused
  // normaliser epilogue is laid out for the default 934-float rows only.  v7 rows (574 floats) run on it with the default
  // self-obs flags and without the normaliser; anything else with v7 runs on the generic kernel.
  const bool def = default_obs_flags(p.of);
  const bool v7 = p.of.v7 != 0;
  const int RW = p.selfw + task_width(p.of);
  const bool fast = !g_force_generic && p.T == 1 && p.aos && p.L.packed && p.obs_stride == RW &&
                    ((uintptr_t)p.obs & 15) == 0 && (!v7 || (def && !p.obs_norm)) &&
                    (!p.obs_norm || (def && p.obs_norm_stride == STAGE_FLOATS &&
                                     ((uintptr_t)p.obs_norm & (p.norm_bf16 ? 3 : 15)) == 0));
  static bool attr_gen[64] = {};
  static int first_wave[64] = {};
  // several waves of blocks (BASELINE config 3): the persistent warp-specialised kernel.  It carries the plain step
  // (+ power reward, flag / reward copies); the optional epilogues stay with K6-fast.
  static bool attr_persist[3][64] = {};
  static int sm_count[64] = {};
  const bool persist = fast && def && !v7 && g_persist != 0 &&
                       (g_persist >= 2 || p.n >= (p.moments ? g_persist_min_moments : g_persist_min)) && !p.obs_norm &&
                       !p.ep_returns && !p.reset_on && !p.ref_dof_pos && !p.trace && lib->tile_counters &&
                       !(args->flags & PHC_STEP_MAPPED_HOST_IO);
  if (persist) {
    if (!sm_count[dev]) PHC_CUDA(cudaDeviceGetAttribute(&sm_count[dev], cudaDevAttrMultiProcessorCount, dev));
    // instantiations: 3 frame slots / 5 blocks per SM (default), 4 slots / 4 blocks (tests, comparisons), and with the
    // moments in registers 3 slots / 4 blocks (twenty fp64 accumulators per consumer thread: 128 registers)
    const bool mom = p.moments != nullptr;
    const bool four = !mom && g_persist == 3;
    const int which = mom ? 2 : four ? 1 : 0;
    auto kern = mom ? step_persist_kernel<3, 4, true> : four ? step_persist_kernel<4, 4> : step_persist_kernel<3, 5>;
    const size_t smem = four ? sizeof(PersistSmem<4>) : sizeof(PersistSmem<3>);
    if (!attr_persist[which][dev]) {
      PHC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr_persist[which][dev] = true;
    }
    if (lib->unspeculated_steps > 0) --lib->unspeculated_steps;  // nothing is read before the dependency wait here
    p.tile_counter = lib->tile_counters + 2 * (lib->tile_seq.fetch_add(1u, std::memory_order_relaxed) % TILE_SLOTS);
    const int64_t tiles = (p.n + PS_EPB - 1) / PS_EPB;
    const int64_t resident = (int64_t)sm_count[dev] * (four || mom ? 4 : 5);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(tiles < resident ? tiles : resident));
    cfg.blockDim = dim3(PS_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = g_persist_pdl ? 1 : 0;
    PHC_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
    return launch_status();
  }
  bool reset_after = false;
  if (fast) {
    if (!first_wave[dev]) {
      int sms = 0, per_sm = 0;
      PHC_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
      PHC_CUDA(cudaFuncSetAttribute(step_fast_kernel<4, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)sizeof(FastSmem<4>)));
      PHC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, step_fast_kernel<4, 8>, 4 * J24,
                                                             sizeof(FastSmem<4>)));
      first_wave[dev] = sms * (per_sm > 0 ? per_sm : 1);
    }
    p.first_wave_blocks = (g_pdl && !(args->flags & PHC_STEP_MAPPED_HOST_IO)) ? first_wave[dev] : 0;
    if (lib->unspeculated_steps > 0) {  // library (re)written since the last step: nothing may be read before the wait
      p.first_wave_blocks = 0;
      --lib->unspeculated_steps;
    }
    // a grid smaller than one wave leaves first_wave_blocks - grid slots free: that many blocks enter before the
    // previous step's blocks exit and speculate on a third candidate
    const int64_t grid = (p.n + 3) / 4;
    p.spec4_blocks = p.first_wave_blocks > grid ? (int)(p.first_wave_blocks - grid) : 0;
    // instantiations <EPB, blocks/SM, NORM, EP, RESET, DEF, PLAIN, V7>: <4, 8> carries none of the optional epilogues,
    // the PLAIN one none of the per-step options either; the RESET ones are compiled with the bookkeeping too (both
    // are switched at run time inside); one catch-all for non-default self-obs flags.  v7: a plain one and one with
    // every option, the bookkeeping and the in-step reset switched at run time.
    const bool plain = !p.dof_force && !p.ref_dof_pos && !p.mpjpe && !p.use_mean && !p.moments && !p.rew_out &&
                       !p.progress_mirror && p.goff;
    static bool attr[10][64] = {};
    const bool pdl = g_pdl != 0;
    constexpr size_t SM = sizeof(FastSmem<4>);
    // the moments epilogue leaves as TMA bulk reductions when the accumulators are 16-B aligned
    p.moments_bulk = (p.moments && g_moments_bulk && ((uintptr_t)p.moments & 15) == 0) ? 1 : 0;
    // StateInit.Default / Hybrid resets are not built into the step kernel: the step runs without the in-kernel reset and
    // phc_reset_envs follows it (reset_after below), with the same result
    const bool in_kernel = p.reset_on && p.rw.state_init <= PHC_STATE_INIT_RANDOM;
    reset_after = p.reset_on && !in_kernel;
    StepParams pk = p;
    if (reset_after) pk.reset_on = 0;
    pk.ep_block0 = (int)(env0 / 4);
    if (v7 && plain && !in_kernel && !p.ep_returns)
      rc = launch_step(step_fast_kernel<4, 8, false, false, false, true, true, true>, SM, 4, pk, stream, &attr[8][dev], pdl);
    else if (v7)
      rc = launch_step(step_fast_kernel<4, 8, false, true, true, true, false, true>, SM, 4, pk, stream, &attr[9][dev], pdl);
    else if (!def) rc = launch_step(step_fast_kernel<4, 8, false, true, true, false>, SM, 4, pk, stream, &attr[6][dev], pdl);
    else if (in_kernel) {
      if (p.obs_norm) rc = launch_step(step_fast_kernel<4, 8, true, true, true>, SM, 4, pk, stream, &attr[5][dev], pdl);
      else rc = launch_step(step_fast_kernel<4, 8, false, true, true>, SM, 4, pk, stream, &attr[4][dev], pdl);
    } else if (p.obs_norm && p.ep_returns)
      rc = launch_step(step_fast_kernel<4, 8, true, true>, SM, 4, pk, stream, &attr[3][dev], pdl);
    else if (p.ep_returns) rc = launch_step(step_fast_kernel<4, 8, false, true>, SM, 4, pk, stream, &attr[2][dev], pdl);
    else if (p.obs_norm) rc = launch_step(step_fast_kernel<4, 8, true>, SM, 4, pk, stream, &attr[1][dev], pdl);
    else if (plain)
      rc = launch_step(step_fast_kernel<4, 8, false, false, false, true, true>, SM, 4, pk, stream, &attr[7][dev], pdl);
    else rc = launch_step(step_fast_kernel<4, 8>, SM, 4, pk, stream, &attr[0][dev], pdl);
    if (rc != PHC_OK || !reset_after) return rc;
  } else {
  float* raw_post = nullptr;  // the mapped reward_raw rows, posted by the bookkeeping (ep_raw)
  if (ep_raw) raw_post = p.raw, p.raw = ep_raw;
  // T > 1 on the AoS tensor + packed table: the pipelined TMA kernel
  const bool multi = !g_force_generic && p.T > 1 && p.aos && p.L.packed && p.obs_vec2 && !p.obs_norm && def && !v7 &&
                     !(args->flags & PHC_STEP_MAPPED_HOST_IO);
  static bool attr_multi[64] = {}, attr_multi2[64] = {};
  // two query groups per block (measured: 2048 envs 21.6 -> 18.3 us, 4096 envs 43.7 -> 37.2, 16384 envs 128.2 -> 127.5)
  const int multi_groups = g_multi_groups ? g_multi_groups : 2;
  if (multi && multi_groups == 2) {
    if (!attr_multi2[dev]) {
      PHC_CUDA(cudaFuncSetAttribute(step_multi2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Multi2Smem)));
      attr_multi2[dev] = true;
    }
    step_multi2_kernel<<<(unsigned)((p.n + MULTI_EPB - 1) / MULTI_EPB), 2 * MULTI_EPB * J24, sizeof(Multi2Smem), stream>>>(p);
    rc = launch_status();
  } else if (multi) {
    rc = launch_step(step_multi_kernel, sizeof(MultiSmem), MULTI_EPB, p, stream, &attr_multi[dev], false);
  } else {
    rc = launch_step(step_kernel<STEP_EPB>, sizeof(StepSmem<STEP_EPB>), STEP_EPB, p, stream, &attr_gen[dev], false);
  }
  if (rc == PHC_OK && p.ep_returns) {  // these kernels do not carry the episode bookkeeping: a second, small launch
    StepParams q = p;
    q.ep_block0 = (int)((env0 + 255) / 256);
    if (raw_post) q.rew = p.rew_out, q.reset = p.reset_out, q.term = p.term_out;
    episode_bucket_kernel<<<(unsigned)((p.n + 255) / 256), 256, 0, stream>>>(q, raw_post);
    rc = launch_status();
  }
  reset_after = p.reset_on != 0;  // ... nor the in-step reset
  }
  if (rc == PHC_OK && reset_after) {
    // phc_reset_envs behind the step, reset_buf as its own mask (the step's flags are already
    // in reset_out / terminate_out), the normalised rows and the moments kept consistent with the rewritten rows
    ResetParams r;
    rc = reset_fill(lib, args->auto_reset, n, r);
    if (rc) return rc;
    r.mask = p.reset;
    r.norm = NormOut{p.obs_norm, p.obs_norm_stride, p.norm_mean, p.norm_var, p.norm_eps, p.norm_clip, p.norm_bf16};
    r.moments = p.moments;
    r.moment_buckets = p.moment_buckets;
    r.moments_mode = p.moments ? 2 : 0;
    rc = reset_launch(r, stream);
  }
  return rc;
}

// the host reset path always writes dof_pos / dof_vel: it needs the library's local rotations and dof velocities
bool lib_has_dof_state(const PhcLib* lib) { return lib && lib->d.lrs && lib->d.dvs; }

extern "C" {

int phc_step_fused(const PhcLib* lib, const PhcStepArgs* args, int64_t n, phc_stream_t stream) {
  return step_fused_mirrored(lib, args, n, stream, nullptr, 0, nullptr);
}

// ---- RunningNorm ---------------------------------------------------------------------------
int phc_obs_moments(const float* x, int64_t rows, int64_t cols, int64_t row_stride, double* sums,
                    phc_stream_t stream) {
  if (rows == 0 || cols == 0) return PHC_OK;
  if (rows < 0 || cols < 0 || row_stride < cols) return PHC_ERR_SHAPE;
  if (!x || !sums) return PHC_ERR_NULL;
  int64_t rpb = MOM_ROWS_PER_BLOCK;
  if ((rows + rpb - 1) / rpb > MOM_MAX_ROW_BLOCKS) rpb = ((rows + MOM_MAX_ROW_BLOCKS - 1) / MOM_MAX_ROW_BLOCKS + 7) / 8 * 8;
  const unsigned gy = (unsigned)((rows + rpb - 1) / rpb);
  const bool vec2 = (cols % 2 == 0) && (row_stride % 2 == 0) && (((uintptr_t)x & 7) == 0);
  if (vec2) {
    dim3 grid((unsigned)((cols / 2 + 127) / 128), gy);
    obs_moments_kernel<2><<<grid, 128, 0, stream>>>(x, rows, cols, row_stride, rpb, sums);
  } else {
    dim3 grid((unsigned)((cols + 127) / 128), gy);
    obs_moments_kernel<1><<<grid, 128, 0, stream>>>(x, rows, cols, row_stride, rpb, sums);
  }
  return launch_status();
}

int phc_obs_moments_fold(double* buckets, int32_t num_buckets, int64_t cols2, double* sums, phc_stream_t stream) {
  if (cols2 == 0 || num_buckets == 0) return PHC_OK;
  if (cols2 < 0 || num_buckets < 0) return PHC_ERR_SHAPE;
  if (!buckets || !sums) return PHC_ERR_NULL;
  moments_fold_kernel<<<(unsigned)((cols2 + 127) / 128), 128, 0, stream>>>(buckets, num_buckets, cols2, sums);
  return launch_status();
}

int phc_running_norm_update(float* running_mean, float* running_var, float* count, const double* sums,
                            const double* total_rows, int64_t cols, phc_stream_t stream) {
  if (cols <= 0) return PHC_ERR_SHAPE;
  if (!running_mean || !running_var || !count || !sums || !total_rows) return PHC_ERR_NULL;
  running_norm_update_kernel<<<(unsigned)((cols + 127) / 128), 128, 0, stream>>>(running_mean, running_var, count,
                                                                                 sums, total_rows, cols);
  int rc = launch_status();
  if (rc) return rc;
  running_norm_count_kernel<<<1, 1, 0, stream>>>(count);
  return launch_status();
}

int phc_running_norm_forward(const float* x, int64_t rows, int64_t cols, int64_t row_stride,
                             const float* running_mean, const float* running_var, float epsilon, float clip,
                             float* out, int64_t out_stride, phc_stream_t stream) {
  if (rows == 0 || cols == 0) return PHC_OK;
  if (rows < 0 || cols < 0 || row_stride < cols || out_stride < cols || rows > 0x7fffffff) return PHC_ERR_SHAPE;
  if (!x || !running_mean || !running_var || !out) return PHC_ERR_NULL;
  const bool vec2 = cols % 2 == 0 && row_stride % 2 == 0 && out_stride % 2 == 0 && (((uintptr_t)x | (uintptr_t)out) & 7) == 0;
  if (vec2) {
    dim3 grid((unsigned)((rows + RN_ROWS - 1) / RN_ROWS), (unsigned)((cols / 2 + 127) / 128));
    running_norm_forward_kernel<2><<<grid, 128, 0, stream>>>(x, rows, cols, row_stride, running_mean, running_var, epsilon,
                                                             clip, out, out_stride);
  } else {
    dim3 grid((unsigned)((rows + RN_ROWS - 1) / RN_ROWS), (unsigned)((cols + 127) / 128));
    running_norm_forward_kernel<1><<<grid, 128, 0, stream>>>(x, rows, cols, row_stride, running_mean, running_var, epsilon,
                                                             clip, out, out_stride);
  }
  return launch_status();
}

int phc_episode_fold(double* sums, int32_t num_buckets, int32_t raw_cols, int64_t n, double* stats, float* raw_rewards,
                     phc_stream_t stream) {
  if (!sums || !stats || (raw_cols > 0 && !raw_rewards)) return PHC_ERR_NULL;
  if (num_buckets < 1 || raw_cols < 0 || raw_cols > EP_SUM_COLS - 4 || n < 1) return PHC_ERR_SHAPE;
  episode_fold_kernel<<<1, 32, 0, stream>>>(sums, num_buckets, raw_cols, (double)n, stats, raw_rewards);
  return launch_status();
}

int phc_episode_update(const PhcEpisodeArgs* a, int64_t n, phc_stream_t stream) {
  if (!a) return PHC_ERR_NULL;
  if (n == 0) return PHC_OK;
  if (n < 0 || a->reward_raw_cols < 0 || a->reward_raw_cols > EP_MAX_RAW) return PHC_ERR_SHAPE;
  if (a->reward_raw_cols > 0 && (!a->reward_raw || !a->raw_rewards || a->reward_raw_stride < a->reward_raw_cols))
    return a->reward_raw && a->raw_rewards ? PHC_ERR_SHAPE : PHC_ERR_NULL;
  if (!a->reset || !a->terminate || !a->rewards || !a->terminals || !a->truncations || !a->masks ||
      !a->episode_returns || !a->episode_lengths || !a->stats || !a->workspace)
    return PHC_ERR_NULL;
  EpisodeParams p;
  p.reset = a->reset;
  p.terminate = a->terminate;
  p.rewards = a->rewards;
  p.reward_raw = a->reward_raw;
  p.raw_stride = a->reward_raw_stride;
  p.raw_cols = a->reward_raw_cols;
  p.n = n;
  p.terminals = a->terminals;
  p.truncations = a->truncations;
  p.masks = a->masks;
  p.episode_returns = a->episode_returns;
  p.episode_lengths = a->episode_lengths;
  p.stats = a->stats;
  p.raw_rewards = a->raw_rewards;
  p.ws = a->workspace;
  const int64_t blocks = std::min<int64_t>((n + 255) / 256, 148 * 4);
  episode_update_kernel<<<(unsigned)blocks, 256, 0, stream>>>(p);
  return launch_status();
}

// The shape rule of the AMP buffers: S, P against the flags / key bodies / dof subset, key body ids.  Also what
// phc_host.cu checks before it enqueues anything.
int amp_env_shape(const PhcAmpEnvArgs* a) {
  if (a->num_sel < 0 || a->num_sel % 3 != 0 || a->num_sel > 96 || a->num_key_bodies < 0 || a->num_key_bodies > 8 ||
      a->num_steps < 1 || a->num_steps > AMP_MAX_STEPS)
    return PHC_ERR_SHAPE;
  const int width = ((a->flags & PHC_OBS_ROOT_HEIGHT) ? 1 : 0) + 12 + 3 * a->num_sel + 3 * a->num_key_bodies;
  if (a->obs_per_step != width) return PHC_ERR_SHAPE;
  for (int i = 0; i < a->num_key_bodies; ++i)
    if (a->key_body_ids[i] < 0 || a->key_body_ids[i] >= a->body.num_bodies) return PHC_ERR_SHAPE;
  return PHC_OK;
}

static int amp_env_fill(const PhcAmpEnvArgs* a, int64_t n, AmpEnvParams& p) {
  if (!a) return PHC_ERR_NULL;
  if (n < 0) return PHC_ERR_SHAPE;
  if (!a->amp_obs_buf || !a->body.pos.ptr || !a->body.rot.ptr || !a->body.vel.ptr || !a->body.ang_vel.ptr)
    return PHC_ERR_NULL;
  if (const int rc = amp_env_shape(a)) return rc;
  p.body = a->body;
  p.dof_pos = a->dof_pos;
  p.dof_vel = a->dof_vel;
  p.dof_stride = a->dof_stride;
  p.dof_estride = a->dof_elem_stride;
  for (int i = 0; i < 8; ++i) p.key_ids[i] = a->key_body_ids[i];
  p.K = a->num_key_bodies;
  p.dof_subset = a->dof_subset;
  p.num_sel = a->num_sel;
  p.flags = a->flags;
  p.buf = a->amp_obs_buf;
  p.demo = a->amp_obs_demo_buf;
  p.S = a->num_steps;
  p.P = a->obs_per_step;
  p.mask = a->env_mask;
  p.roll = 0;
  p.n = n;
  return PHC_OK;
}

int phc_amp_step(const PhcAmpEnvArgs* a, int64_t n, int32_t roll_history, phc_stream_t stream) {
  AmpEnvParams p;
  const int rc = amp_env_fill(a, n, p);
  if (rc) return rc;
  if (n == 0) return PHC_OK;
  if (!a->dof_pos || !a->dof_vel) return PHC_ERR_NULL;
  if (a->dof_elem_stride < 1) return PHC_ERR_SHAPE;
  p.roll = roll_history ? 1 : 0;
  const int epb = 4;
  amp_step_kernel<<<(unsigned)((n + epb - 1) / epb), epb * 32, 0, stream>>>(p);
  return launch_status();
}

int phc_amp_init_ref(const PhcLib* lib, const PhcAmpEnvArgs* a, const int64_t* motion_ids, const float* motion_times,
                     float dt, int64_t n, phc_stream_t stream) {
  AmpEnvParams p;
  const int rc = amp_env_fill(a, n, p);
  if (rc) return rc;
  if (n == 0) return PHC_OK;
  if (!lib || !motion_ids || !motion_times) return PHC_ERR_NULL;
  if (!lib->d.lrs || !lib->d.dvs) return PHC_ERR_NULL;  // dof_pos / dof_vel need the local rotations and dof velocities
  for (int i = 0; i < a->num_key_bodies; ++i)
    if (a->key_body_ids[i] >= J24) return PHC_ERR_SHAPE;
  if (a->init_slot0 && (!a->dof_pos || !a->dof_vel)) return PHC_ERR_NULL;
  if (a->init_slot0 && a->dof_elem_stride < 1) return PHC_ERR_SHAPE;
  // measured at 4096 envs x 10 slots (profiles/r1_env_loop.md): 8 envs x 16 warps per block is 2.0 us with nothing
  // flagged and 40 us with 31 % flagged; 2 x 10 is 3.7 / 36 us, 1 x 10 is 6.4 / 35 us — the rows themselves are
  // issue-bound (slerp + exp-map + tan-norm per joint in precise libdevice math), so the default favours the empty case
  static int wpb = 0, epb = 0;
  if (!wpb) {
    const char* v = getenv("PHC_AMPI_WARPS");
    const char* e = getenv("PHC_AMPI_EPB");
    epb = e ? atoi(e) : AMPI_EPB;
    if (epb < 1 || epb > AMPI_EPB) epb = AMPI_EPB;
    wpb = v ? atoi(v) : 16;
    if (wpb < 1 || wpb > 32) wpb = 16;
  }
  amp_init_ref_kernel<<<(unsigned)((n + epb - 1) / epb), wpb * 32, 0, stream>>>(
      p, lib->d, motion_ids, motion_times, dt, a->init_slot0 ? 1 : 0, epb);
  return launch_status();
}

}  // extern "C"
