// emu_grad_seq_driver.cpp -- TEST INFRASTRUCTURE.  Runs GradSeq<G>::run from the product's dexr_grad_seq_kernels.cuh on the
// host, laid out like dexr_grad_sequences_kernel (dexr_grad.cu): one stream per group of G lanes, G = 16 up to 16 joints else 32.
// Built on emu_grad_driver.cpp (the warp shim's scheduler and emu_grad_frames, so that one library serves both entry points).
#include "emu_grad_driver.cpp"

#include "../../dex_retargeting_b200/csrc/dexr_grad_seq_kernels.cuh"

namespace {
struct SeqJob {
  const dexr_table_t* tb;
  dexr_params_t prm;
  Dims dm;
  int scratch_off;
  dexr_grad_sequences_t io;
  long long S, base;
  int T;
} sjob;

template <int G>
void seq_lane_body(int lane) {
  const SeqJob& j = sjob;
  const int gid = lane / G;
  Solver<G, 0> sv;
  sv.init(j.tb, j.dm, (uint32_t)(j.scratch_off + gid * GradSeqScratch<G>::kFloats * 4), j.prm, lane);
  const long long s = j.base + gid;
  const bool active = s < j.S;
  GradSeq<G>::run(sv, j.io, active ? s : j.S - 1, j.T, active);
}

template <int G>
int seq_run_all(char* err, int errlen) {
  constexpr int GPW = 32 / G;
  sjob.scratch_off = ((int)sizeof(SharedTable) + 15) / 16 * 16;
  const int scratch_bytes = GPW * GradSeqScratch<G>::kFloats * 4;
  threadIdx.x = 0; blockDim.x = 1;
  load_shared_table(*reinterpret_cast<SharedTable*>(dsmem), sjob.tb);
  for (sjob.base = 0; sjob.base < sjob.S; sjob.base += GPW) {
    uint32_t* sc = reinterpret_cast<uint32_t*>(dsmem + sjob.scratch_off);
    for (int i = 0; i < scratch_bytes / 4; ++i) sc[i] = 0x7fc00000u;  // NaN poison
    if (emu::run_warp(&seq_lane_body<G>) != 0) {
      snprintf(err, errlen, "stream %lld: %s", sjob.base, emu::errmsg);
      return -1;
    }
  }
  return 0;
}
}  // namespace

extern "C" int emu_grad_sequences(const dexr_table_t* tb, const dexr_params_t* prm, const dexr_grad_sequences_t* io, long long S,
                                  long long T, char* err, int errlen) {
  sjob = SeqJob{};
  sjob.tb = tb; sjob.prm = *prm; sjob.prm.clip_init = 1; sjob.io = *io; sjob.S = S; sjob.T = (int)T;
  Dims& d = sjob.dm;
  d.dof = tb->dof; d.n_var = tb->n_var; d.n_fixed = tb->n_fixed; d.n_links = tb->n_links; d.n_res = tb->n_res; d.loss = tb->loss;
  d.n_rounds = tb->n_rounds; d.has_mimic = tb->has_mimic; d.num_fingers = tb->num_fingers; d.len_proj = tb->len_proj;
  d.len_s1 = tb->len_s1; d.block_width = 0; d.trunk = 0;
  if (S == 0 || T == 0) return 0;
  if (tb->dof <= 16) return seq_run_all<16>(err, errlen);
  return seq_run_all<32>(err, errlen);
}
