// dexr_grad.cu -- the backward-pass kernel and the C ABI of libdexr_grad.so (see include/dexr_grad.h).
//
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -shared -Xcompiler -fPIC
// One group of G lanes per frame (G = 16 up to 16 joints, else 32), plain global loads, no atomics: a frame's outputs belong
// to its group, so its gradient does not depend on where in the batch it sits or how large the batch is.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>

#include "dexr_grad_seq_kernels.cuh"

namespace dexr {

struct GradArgs {
  const dexr_table_t* table;
  dexr_params_t prm;
  dexr_grad_frames_t io;
  long long B;
  Dims dm;
  int scratch_off;
};

constexpr int kGradNW = 4;  // warps per CTA

template <int G>
__global__ void __launch_bounds__(kGradNW * 32, 1) dexr_grad_kernel(const GradArgs a) {
  load_shared_table(*reinterpret_cast<SharedTable*>(dsmem), a.table);
  __syncthreads();
  constexpr int GPW = 32 / G;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int gid = warp * GPW + lane / G;
  Solver<G, 0> sv;
  sv.init(a.table, a.dm, (uint32_t)(a.scratch_off + gid * GradScratch<G>::kFloats * 4), a.prm, lane);
  const long long stride = (long long)gridDim.x * kGradNW * GPW;
  for (long long base = ((long long)blockIdx.x * kGradNW + warp) * GPW; base < a.B; base += stride) {
    const long long idx = base + lane / G;
    const bool active = idx < a.B;
    const long long f = active ? idx : base;
    GradInputs in;
    in.kp = a.io.keypoints ? a.io.keypoints + f * 3 * DEXR_NUM_KEYPOINTS : nullptr;
    in.ref = a.io.keypoints ? nullptr : a.io.ref_value + f * 3 * a.dm.n_res;
    in.fixed = a.dm.n_fixed > 0 ? a.io.fixed_qpos + f * a.dm.n_fixed : nullptr;
    in.last = a.io.last_qpos + f * a.dm.n_var;
    in.projected = a.io.projected ? a.io.projected + f * a.dm.len_proj : nullptr;
    in.qpos = a.io.qpos + f * a.dm.n_var;
    in.gq = a.io.grad_qpos + f * a.dm.n_var;
    in.fstatus = a.io.status ? a.io.status[f] : 0;
    GradOutputs out;
    out.gkp = a.io.grad_keypoints ? a.io.grad_keypoints + f * 3 * DEXR_NUM_KEYPOINTS : nullptr;
    out.gref = a.io.grad_ref_value ? a.io.grad_ref_value + f * 3 * a.dm.n_res : nullptr;
    out.glast = a.io.grad_last_qpos ? a.io.grad_last_qpos + f * a.dm.n_var : nullptr;
    const int st = GradFrame<G>::run(sv, in, out, active);
    if (active && sv.l == 0 && a.io.grad_status) a.io.grad_status[f] = st;
  }
}

struct GradSeqArgs {
  const dexr_table_t* table;
  dexr_params_t prm;
  dexr_grad_sequences_t io;
  long long S;
  int T;
  Dims dm;
  int scratch_off;
};

// One group of G lanes per stream, walking its T steps backwards (dexr_grad_seq_kernels.cuh).  Streams are dealt round-robin
// over CTAs (stream = blockIdx + gridDim * slot), as the forward stream kernel deals them: the path is latency bound per stream.
template <int G>
__global__ void __launch_bounds__(kGradNW * 32, 1) dexr_grad_sequences_kernel(const GradSeqArgs a) {
  load_shared_table(*reinterpret_cast<SharedTable*>(dsmem), a.table);
  __syncthreads();
  constexpr int GPW = 32 / G;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int slot = warp * GPW + lane / G;
  Solver<G, 0> sv;
  sv.init(a.table, a.dm, (uint32_t)(a.scratch_off + slot * GradSeqScratch<G>::kFloats * 4), a.prm, lane);
  // (all groups of a warp walk the stream loop together: GradFrame's shift retry is warp-wide)
  for (long long base = 0; base < a.S; base += (long long)gridDim.x * kGradNW * GPW) {
    const long long s = base + (long long)slot * gridDim.x + blockIdx.x;
    const bool active = s < a.S;
    if (!__any_sync(0xffffffffu, active)) break;  // (s only grows: this warp has no stream left)
    GradSeq<G>::run(sv, a.io, active ? s : a.S - 1, a.T, active);
  }
}

// One thread per (stream, joint), serial over the steps; blockDim = (32, kLowpassSPB): a stream's joints share a CTA, so the
// entry filter_init is read by all of them before joint 0 overwrites it.
constexpr int kLowpassSPB = 8;

__global__ void __launch_bounds__(32 * kLowpassSPB) dexr_grad_lowpass_kernel(const float* __restrict__ q, float* __restrict__ y,
                                                                             float* fstate, uint8_t* finit_io, float alpha,
                                                                             long long S, int T, int dof) {
  const long long s = (long long)blockIdx.x * kLowpassSPB + threadIdx.y;
  const int j = threadIdx.x;
  const bool live = s < S && j < dof;
  int finit = 0;
  float fy = 0.f;
  if (live) { finit = finit_io[s]; fy = fstate[s * dof + j]; }
  __syncthreads();
  if (!live) return;
  for (int t = 0; t < T; ++t) {
    const long long e = (s * T + t) * dof + j;
    const float out = q[e];
    fy = finit ? fmaf(alpha, out - fy, fy) : out;  // the expression of dexr_sequences_kernel
    finit = 1;
    y[e] = fy;
  }
  fstate[s * dof + j] = fy;
  if (j == 0) finit_io[s] = (uint8_t)finit;
}

}  // namespace dexr

using namespace dexr;

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

// The caller's current device is restored on every exit path (as libdexr's entry points do).
struct GradDeviceGuard {
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit GradDeviceGuard(int device) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != device) err = cudaSetDevice(device);
    else if (err == cudaSuccess) prev = -1;
  }
  ~GradDeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
  GradDeviceGuard(const GradDeviceGuard&) = delete;
  GradDeviceGuard& operator=(const GradDeviceGuard&) = delete;
};

#define GRAD_CUDA_TRY(expr)                                                                       \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess) return fail(DEXR_E_CUDA, "%s failed: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

static int check_table_params(const dexr_table_t* t, const dexr_params_t* p) {
  if (t->magic != 0x31525844u) return fail(DEXR_E_INVALID, "robot table: bad magic 0x%08x", t->magic);
  if (t->nbytes != sizeof(dexr_table_t))
    return fail(DEXR_E_INVALID, "robot table: size %u does not match library (%zu)", t->nbytes, sizeof(dexr_table_t));
  if (t->dof < 1 || t->dof > DEXR_MAX_LANES) return fail(DEXR_E_INVALID, "robot table: dof %d out of range 1..32", t->dof);
  if (t->n_var < 1 || t->n_var > t->dof) return fail(DEXR_E_INVALID, "robot table: n_var %d out of range", t->n_var);
  if (t->n_res < 1 || t->n_res > DEXR_MAX_RES) return fail(DEXR_E_INVALID, "robot table: n_res %d out of range", t->n_res);
  if (t->loss < 0 || t->loss > 2) return fail(DEXR_E_INVALID, "robot table: loss %d unknown", t->loss);
  if (!(p->huber_delta > 0.f)) return fail(DEXR_E_INVALID, "huber_delta must be > 0");
  if (!(p->norm_delta >= 0.f)) return fail(DEXR_E_INVALID, "norm_delta must be >= 0");
  if (p->preprocess != 0)
    return fail(DEXR_E_INVALID, "preprocess (raw detector landmarks) is not differentiable here: pass pre-processed keypoints");
  return 0;
}

static int check_args(const dexr_table_t* t, const void* table_dev, const dexr_params_t* p, const dexr_grad_frames_t* io) {
  if (!t || !table_dev || !p || !io) return fail(DEXR_E_INVALID, "dexr_grad_frames: null argument");
  if (int e = check_table_params(t, p)) return e;
  if ((io->keypoints == nullptr) == (io->ref_value == nullptr))
    return fail(DEXR_E_INVALID, "give exactly one of keypoints / ref_value");
  if (io->keypoints ? io->grad_ref_value != nullptr : io->grad_keypoints != nullptr)
    return fail(DEXR_E_INVALID, "the input gradient must be of the input given (keypoints -> grad_keypoints, ref_value -> grad_ref_value)");
  if (!io->last_qpos || !io->qpos || !io->grad_qpos) return fail(DEXR_E_INVALID, "last_qpos, qpos and grad_qpos are required");
  if (t->n_fixed > 0 && !io->fixed_qpos) return fail(DEXR_E_INVALID, "the robot has %d fixed joints but fixed_qpos is NULL", t->n_fixed);
  return 0;
}

static int check_seq_args(const dexr_table_t* t, const void* table_dev, const dexr_params_t* p, const dexr_grad_sequences_t* io) {
  if (!t || !table_dev || !p || !io) return fail(DEXR_E_INVALID, "dexr_grad_sequences: null argument");
  if (int e = check_table_params(t, p)) return e;
  if (!io->keypoints || !io->last_qpos || !io->qpos) return fail(DEXR_E_INVALID, "keypoints, last_qpos and qpos are required");
  if (!io->grad_robot_qpos && !io->grad_last_qpos_out && !io->grad_filter_state_out)
    return fail(DEXR_E_INVALID, "no upstream gradient: give grad_robot_qpos, grad_last_qpos_out and / or grad_filter_state_out");
  const bool use_filter = p->lp_alpha >= 0.f && p->lp_alpha <= 1.f;
  if (use_filter && !io->filter_init) return fail(DEXR_E_INVALID, "the low-pass filter is on (lp_alpha in [0,1]): filter_init is required");
  if (t->len_proj > 0 && !io->projected_ws)
    return fail(DEXR_E_INVALID, "DexPilot table (len_proj %d): the flag replay needs projected_ws [S,T,len_proj]", t->len_proj);
  if (t->n_fixed > 0 && !io->fixed_qpos) return fail(DEXR_E_INVALID, "the robot has %d fixed joints but fixed_qpos is NULL", t->n_fixed);
  return 0;
}

static Dims grad_dims(const dexr_table_t& t) {
  Dims d{};
  d.dof = t.dof; d.n_var = t.n_var; d.n_fixed = t.n_fixed; d.n_links = t.n_links; d.n_res = t.n_res; d.loss = t.loss;
  d.n_rounds = t.n_rounds; d.has_mimic = t.has_mimic; d.num_fingers = t.num_fingers; d.len_proj = t.len_proj;
  d.len_s1 = t.len_s1; d.block_width = 0; d.trunk = 0;
  return d;
}

// Selects `device` (restored by the guard) and checks it is an sm_100 part; `sms` its multiprocessor count.
static int open_device(GradDeviceGuard& guard, int device, int& sms) {
  if (guard.err != cudaSuccess) return fail(DEXR_E_CUDA, "selecting device %d failed: %s", device, cudaGetErrorString(guard.err));
  int major = 0;
  GRAD_CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  GRAD_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  if (major < 10) return fail(DEXR_E_NODEVICE, "device %d is sm_%d0; libdexr_grad is built for sm_100a only", device, major);
  return 0;
}

extern "C" {

int dexr_grad_version(void) { return DEXR_GRAD_VERSION; }
#ifndef DEXR_GRAD_BUILD_ID
#define DEXR_GRAD_BUILD_ID "unstamped"
#endif
const char* dexr_grad_build_id(void) { return DEXR_GRAD_BUILD_ID; }
const char* dexr_grad_last_error(void) { return g_err; }
size_t dexr_grad_frames_sizeof(void) { return sizeof(dexr_grad_frames_t); }

int dexr_grad_frames(const dexr_table_t* table_host, const void* table_dev, const dexr_params_t* params,
                     const dexr_grad_frames_t* io, int64_t num_frames, int device, void* cuda_stream) {
  if (int e = check_args(table_host, table_dev, params, io)) return e;
  if (num_frames < 0) return fail(DEXR_E_INVALID, "num_frames < 0");
  if (num_frames == 0) return 0;
  GradDeviceGuard guard(device);
  if (guard.err != cudaSuccess) return fail(DEXR_E_CUDA, "selecting device %d failed: %s", device, cudaGetErrorString(guard.err));
  int major = 0, sms = 0;
  GRAD_CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  GRAD_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  if (major < 10) return fail(DEXR_E_NODEVICE, "device %d is sm_%d0; libdexr_grad is built for sm_100a only", device, major);
  const dexr_table_t& t = *table_host;
  GradArgs a{};
  a.table = static_cast<const dexr_table_t*>(table_dev);
  a.prm = *params;
  a.io = *io;
  a.B = num_frames;
  Dims& d = a.dm;
  d.dof = t.dof; d.n_var = t.n_var; d.n_fixed = t.n_fixed; d.n_links = t.n_links; d.n_res = t.n_res; d.loss = t.loss;
  d.n_rounds = t.n_rounds; d.has_mimic = t.has_mimic; d.num_fingers = t.num_fingers; d.len_proj = t.len_proj;
  d.len_s1 = t.len_s1; d.block_width = 0; d.trunk = 0;
  a.scratch_off = ((int)sizeof(SharedTable) + 15) / 16 * 16;
  cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
  auto launch = [&](auto kern, int gpw, int group_floats) -> int {
    const int smem = a.scratch_off + kGradNW * gpw * group_floats * 4;
    GRAD_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int per_sm = 0;
    GRAD_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kGradNW * 32, smem));
    const long long frames_per_cta = (long long)kGradNW * gpw;
    const long long need = (num_frames + frames_per_cta - 1) / frames_per_cta;
    const int grid = (int)std::max<long long>(1, std::min<long long>(need, (long long)sms * std::max(per_sm, 1)));
    kern<<<grid, kGradNW * 32, smem, stream>>>(a);
    GRAD_CUDA_TRY(cudaGetLastError());
    return 0;
  };
  if (t.dof <= 16) return launch(dexr_grad_kernel<16>, 2, GradScratch<16>::kFloats);
  return launch(dexr_grad_kernel<32>, 1, GradScratch<32>::kFloats);
}

size_t dexr_grad_sequences_sizeof(void) { return sizeof(dexr_grad_sequences_t); }

int dexr_grad_sequences(const dexr_table_t* table_host, const void* table_dev, const dexr_params_t* params,
                        const dexr_grad_sequences_t* io, int64_t num_streams, int64_t num_steps, int device, void* cuda_stream) {
  if (int e = check_seq_args(table_host, table_dev, params, io)) return e;
  if (num_streams < 0 || num_steps < 0 || num_steps > INT32_MAX) return fail(DEXR_E_INVALID, "bad sizes (num_streams / num_steps)");
  if (num_streams == 0 || num_steps == 0) return 0;
  GradDeviceGuard guard(device);
  int sms = 0;
  if (int e = open_device(guard, device, sms)) return e;
  const dexr_table_t& t = *table_host;
  GradSeqArgs a{};
  a.table = static_cast<const dexr_table_t*>(table_dev);
  a.prm = *params;
  a.prm.clip_init = 1;  // the stream recurrence clips every warm start (seq_retarget.py), so the anchor adjoint is masked
  a.io = *io;
  a.S = num_streams;
  a.T = (int)num_steps;
  a.dm = grad_dims(t);
  a.scratch_off = ((int)sizeof(SharedTable) + 15) / 16 * 16;
  cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
  auto launch = [&](auto kern, int gpw, int group_floats) -> int {
    const int smem = a.scratch_off + kGradNW * gpw * group_floats * 4;
    GRAD_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int per_sm = 0;
    GRAD_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kGradNW * 32, smem));
    // one stream per CTA while there are CTAs to spare (a CTA's first slot on every SM before any second slot)
    const int grid = (int)std::max<long long>(1, std::min<long long>(num_streams, (long long)sms * std::max(per_sm, 1)));
    kern<<<grid, kGradNW * 32, smem, stream>>>(a);
    GRAD_CUDA_TRY(cudaGetLastError());
    return 0;
  };
  if (t.dof <= 16) return launch(dexr_grad_sequences_kernel<16>, 2, GradSeqScratch<16>::kFloats);
  return launch(dexr_grad_sequences_kernel<32>, 1, GradSeqScratch<32>::kFloats);
}

int dexr_grad_lowpass(const float* q, float* y, float* filter_state, uint8_t* filter_init, float alpha, int64_t num_streams,
                      int64_t num_steps, int dof, int device, void* cuda_stream) {
  if (!q || !y || !filter_state || !filter_init) return fail(DEXR_E_INVALID, "dexr_grad_lowpass: null argument");
  if (!(alpha >= 0.f && alpha <= 1.f)) return fail(DEXR_E_INVALID, "dexr_grad_lowpass: alpha %g outside [0,1]", (double)alpha);
  if (dof < 1 || dof > DEXR_MAX_LANES) return fail(DEXR_E_INVALID, "dexr_grad_lowpass: dof %d out of range 1..32", dof);
  if (num_streams < 0 || num_steps < 0 || num_steps > INT32_MAX) return fail(DEXR_E_INVALID, "bad sizes (num_streams / num_steps)");
  if (num_streams == 0 || num_steps == 0) return 0;
  GradDeviceGuard guard(device);
  int sms = 0;
  if (int e = open_device(guard, device, sms)) return e;
  const long long grid = (num_streams + kLowpassSPB - 1) / kLowpassSPB;
  if (grid > INT32_MAX) return fail(DEXR_E_INVALID, "dexr_grad_lowpass: too many streams");
  dexr_grad_lowpass_kernel<<<(int)grid, dim3(32, kLowpassSPB), 0, static_cast<cudaStream_t>(cuda_stream)>>>(
      q, y, filter_state, filter_init, alpha, (long long)num_streams, (int)num_steps, dof);
  GRAD_CUDA_TRY(cudaGetLastError());
  return 0;
}

}  // extern "C"
