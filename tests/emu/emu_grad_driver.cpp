// emu_grad_driver.cpp -- TEST INFRASTRUCTURE (see warp_shim.h and emu_driver.cpp).  Runs GradFrame<G>::run from the product's
// dexr_grad_kernels.cuh on the host, laid out like dexr_grad_kernel (dexr_grad.cu): one frame per group of G lanes, G = 16 up to
// 16 joints else 32, the dense Solver<G, 0> for every table.  Scratch is poisoned with NaN before every warp call.
#include "warp_shim.h"

#include <ucontext.h>

#include <cstdio>
#include <vector>

#include "../../dex_retargeting_b200/csrc/dexr_grad_kernels.cuh"

emu_dim3 threadIdx{0, 0, 0}, blockDim{1, 1, 1}, blockIdx{0, 0, 0}, gridDim{1, 1, 1};
namespace dexr {
__attribute__((aligned(16))) unsigned char dsmem[256 * 1024];
}

namespace emu {
constexpr int W = 32;
static ucontext_t main_ctx, ctx[W];
static std::vector<char> stacks[W];
static int cur = -1;
static bool finished[W], arrived[W];
static int arr_op[W];
static uint32_t arr_val[W], snap[W];
static void* arr_site[W];
static char errmsg[512];
static void (*lane_fn)(int);

int lane() { return cur; }

__attribute__((noinline)) const uint32_t* rendezvous(int op, uint32_t value) {
  const int me = cur;
  arr_op[me] = op;
  arr_val[me] = value;
  arr_site[me] = __builtin_return_address(0);
  arrived[me] = true;
  swapcontext(&ctx[me], &main_ctx);
  return snap;
}

static void trampoline(int l) {
  lane_fn(l);
  finished[l] = true;
}

static int run_warp(void (*fn)(int)) {
  lane_fn = fn;
  for (int l = 0; l < W; ++l) {
    finished[l] = arrived[l] = false;
    getcontext(&ctx[l]);
    if (stacks[l].empty()) stacks[l].resize(1 << 20);
    ctx[l].uc_stack.ss_sp = stacks[l].data();
    ctx[l].uc_stack.ss_size = stacks[l].size();
    ctx[l].uc_link = &main_ctx;
    makecontext(&ctx[l], (void (*)())trampoline, 1, l);
  }
  for (;;) {
    for (int l = 0; l < W; ++l)
      if (!finished[l] && !arrived[l]) {
        cur = l;
        swapcontext(&main_ctx, &ctx[l]);
      }
    int nfin = 0, narr = 0;
    for (int l = 0; l < W; ++l) { nfin += finished[l]; narr += arrived[l]; }
    if (nfin == W) return 0;
    if (nfin > 0) {
      snprintf(errmsg, sizeof errmsg, "%d lanes returned while %d wait at a collective (op %d)", nfin, narr, arr_op[0]);
      return -1;
    }
    for (int l = 1; l < W; ++l)
      if (arr_op[l] != arr_op[0] || arr_site[l] != arr_site[0]) {
        snprintf(errmsg, sizeof errmsg, "divergent collectives: lane 0 at op %d site %p, lane %d at op %d site %p", arr_op[0],
                 arr_site[0], l, arr_op[l], arr_site[l]);
        return -1;
      }
    for (int l = 0; l < W; ++l) { snap[l] = arr_val[l]; arrived[l] = false; }
  }
}
}  // namespace emu

using namespace dexr;

namespace {
struct Job {
  const dexr_table_t* tb;
  dexr_params_t prm;
  Dims dm;
  int scratch_off;
  dexr_grad_frames_t io;
  long long B, base;
} job;

template <int G>
void lane_body(int lane) {
  const Job& j = job;
  const int gid = lane / G;
  Solver<G, 0> sv;
  sv.init(j.tb, j.dm, (uint32_t)(j.scratch_off + gid * GradScratch<G>::kFloats * 4), j.prm, lane);
  const long long idx = j.base + gid;
  const bool active = idx < j.B;
  const long long f = active ? idx : j.base;
  const dexr_grad_frames_t& io = j.io;
  GradInputs in;
  in.kp = io.keypoints ? io.keypoints + f * 3 * DEXR_NUM_KEYPOINTS : nullptr;
  in.ref = io.keypoints ? nullptr : io.ref_value + f * 3 * j.dm.n_res;
  in.fixed = j.dm.n_fixed > 0 ? io.fixed_qpos + f * j.dm.n_fixed : nullptr;
  in.last = io.last_qpos + f * j.dm.n_var;
  in.projected = io.projected ? io.projected + f * j.dm.len_proj : nullptr;
  in.qpos = io.qpos + f * j.dm.n_var;
  in.gq = io.grad_qpos + f * j.dm.n_var;
  in.fstatus = io.status ? io.status[f] : 0;
  GradOutputs out;
  out.gkp = io.grad_keypoints ? io.grad_keypoints + f * 3 * DEXR_NUM_KEYPOINTS : nullptr;
  out.gref = io.grad_ref_value ? io.grad_ref_value + f * 3 * j.dm.n_res : nullptr;
  out.glast = io.grad_last_qpos ? io.grad_last_qpos + f * j.dm.n_var : nullptr;
  const int st = GradFrame<G>::run(sv, in, out, active);
  if (active && sv.l == 0 && io.grad_status) io.grad_status[f] = st;
}

template <int G>
int run_all(char* err, int errlen) {
  constexpr int GPW = 32 / G;
  job.scratch_off = ((int)sizeof(SharedTable) + 15) / 16 * 16;
  const int scratch_bytes = GPW * GradScratch<G>::kFloats * 4;
  threadIdx.x = 0; blockDim.x = 1;
  load_shared_table(*reinterpret_cast<SharedTable*>(dsmem), job.tb);
  for (job.base = 0; job.base < job.B; job.base += GPW) {
    uint32_t* sc = reinterpret_cast<uint32_t*>(dsmem + job.scratch_off);
    for (int i = 0; i < scratch_bytes / 4; ++i) sc[i] = 0x7fc00000u;  // NaN poison
    if (emu::run_warp(&lane_body<G>) != 0) {
      snprintf(err, errlen, "frame %lld: %s", job.base, emu::errmsg);
      return -1;
    }
  }
  return 0;
}
}  // namespace

extern "C" int emu_grad_frames(const dexr_table_t* tb, const dexr_params_t* prm, const dexr_grad_frames_t* io, long long B,
                               char* err, int errlen) {
  job = Job{};
  job.tb = tb; job.prm = *prm; job.io = *io; job.B = B;
  Dims& d = job.dm;
  d.dof = tb->dof; d.n_var = tb->n_var; d.n_fixed = tb->n_fixed; d.n_links = tb->n_links; d.n_res = tb->n_res; d.loss = tb->loss;
  d.n_rounds = tb->n_rounds; d.has_mimic = tb->has_mimic; d.num_fingers = tb->num_fingers; d.len_proj = tb->len_proj;
  d.len_s1 = tb->len_s1; d.block_width = 0; d.trunk = 0;
  if (tb->dof <= 16) return run_all<16>(err, errlen);
  return run_all<32>(err, errlen);
}
