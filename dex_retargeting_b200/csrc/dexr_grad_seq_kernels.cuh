// dexr_grad_seq_kernels.cuh -- backpropagation through time of the stream solver (dexr_sequences_kernel, dexr.cu).
//
// Per stream the forward recurrence is, for t = 0..T-1:
//     a_t  = clip(x*_{t-1})                                   (x*_{-1}: the entry last_qpos)
//     x*_t = argmin F(x; targets(kp_t, flags_t), a_t)
//     q_t  = compose(x*_t)                                    (scatter, fixed joints, mimic)
//     y_t  = finit ? fmaf(alpha, q_t - y_{t-1}, y_{t-1}) : q_t,  finit = 1      (y_t = q_t without the filter)
// and the backward pass walks it in reverse with ybar (filter adjoint, one per joint lane) and carry (anchor adjoint, one per
// variable lane) in registers:
//     ybar += Ybar_t;  qbar_t = alpha ybar, ybar *= 1 - alpha   (filter initialised before step t)
//                      qbar_t = ybar,       ybar  = 0           (step t initialised it)
//     xbar_t = M^T qbar_t + carry                               (mimic fold; fixed joints get nothing)
//     carry  = GradFrame::run(step t, anchor x*_{t-1}, gq = xbar_t)   (anchor adjoint, 0 where the clip moved the warm start)
// After t = 0, carry is dl/d(entry last_qpos) and ybar dl/d(entry filter_state).
//
// The DexPilot flags a frame applied are not in the trace (the forward pass only leaves the final ones), so a first sweep
// replays the hysteresis (prepare_targets: it depends on the keypoints and the previous flags only) from the entry flags into
// the workspace projected_ws[t].  GradFrame<G>::run is reused as it is: it reads the upstream gradient and writes the anchor
// adjoint through per-group shared-memory slots, so a step's arithmetic is exactly dexr_grad_frames'.
#pragma once

#include "dexr_grad_kernels.cuh"

namespace dexr {

// Per-group scratch beyond GradFrame's: the upstream gradient handed to a step, the anchor adjoint it returns, replayed flags.
template <int G>
struct GradSeqScratch {
  static constexpr int kGq = GradScratch<G>::kFloats;     // [MAX_LANES] xbar_t by variable index
  static constexpr int kGlast = kGq + DEXR_MAX_LANES;     // [MAX_LANES] anchor adjoint by variable index
  static constexpr int kFlags = kGlast + DEXR_MAX_LANES;  // DEXR_MAX_RES bytes: DexPilot flags of the replay
  static constexpr int kFloats = ((kFlags + DEXR_MAX_RES / 4 + 3) / 4) * 4;
};

template <int G>
struct GradSeq {
  using SV = Solver<G, 0>;

  // Stream s (every lane of the warp calls it; `active` false: a padding group that computes and writes nothing).
  __device__ __forceinline__ static void run(SV& sv, const dexr_grad_sequences_t& io, long long s, int T, bool active) {
    const Dims& dm = sv.dm;
    const int l = sv.l, var = sv.var, dof = dm.dof, nv = dm.n_var, lp = dm.len_proj;
    constexpr int KP = 3 * DEXR_NUM_KEYPOINTS;
    float* gs = sv.scf();
    float* gq = gs + GradSeqScratch<G>::kGq;
    float* gl = gs + GradSeqScratch<G>::kGlast;
    uint8_t* fl = reinterpret_cast<uint8_t*>(gs + GradSeqScratch<G>::kFlags);

    // ---- replay of the DexPilot hysteresis from the entry flags: projected_ws[t] = the flags frame t applied
    if (lp > 0) {
      if (l < DEXR_MAX_RES) fl[l] = (active && io.projected != nullptr && l < lp) ? io.projected[s * lp + l] : 0;
      __syncwarp();
      for (int t = 0; t < T; ++t) {
        FrameInputs fi;
        fi.kp = io.keypoints + (s * T + t) * KP;
        fi.ref = nullptr; fi.fixed = nullptr; fi.last = nullptr;
        fi.projected = fl;
        sv.prepare_targets(fi, active);
        __syncwarp();
        if (active && l < lp) io.projected_ws[(s * T + t) * lp + l] = fl[l];
        __syncwarp();
      }
    }

    // ---- reverse sweep
    const bool use_filter = sv.prm.lp_alpha >= 0.f && sv.prm.lp_alpha <= 1.f;
    const float alpha = sv.prm.lp_alpha;
    const int finit0 = (active && use_filter) ? io.filter_init[s] : 0;
    float ybar = (active && l < dof && io.grad_filter_state_out != nullptr) ? io.grad_filter_state_out[s * dof + l] : 0.f;
    float carry = (active && var >= 0 && io.grad_last_qpos_out != nullptr) ? io.grad_last_qpos_out[s * nv + var] : 0.f;
    const int gcount = SV::ST().group_count[l];
    for (int t = T - 1; t >= 0; --t) {
      const long long row = s * T + t;
      const float Y = (active && l < dof && io.grad_robot_qpos != nullptr) ? io.grad_robot_qpos[row * dof + l] : 0.f;
      float qbar = Y;
      if (use_filter) {
        ybar += Y;
        if (t > 0 || finit0) { qbar = alpha * ybar; ybar = (1.0f - alpha) * ybar; }
        else { qbar = ybar; ybar = 0.f; }
      }
      // mimic fold M^T: the variable's own lane first, then the joints it drives (GradFrame's g fold)
      float xbar = 0.f;
#pragma unroll
      for (int f = 0; f < DEXR_MAX_GROUP; ++f) {
        const bool v = var >= 0 && f < gcount;
        const float gv = gshfl<G>(qbar, v ? SV::ST().group_lane[l][f] : l);
        if (v) xbar = fmaf(SV::ST().group_mult[l][f], gv, xbar);
      }
      xbar += carry;
      if (var >= 0) gq[var] = xbar;
      __syncwarp();
      GradInputs in;
      in.kp = io.keypoints + row * KP;
      in.ref = nullptr;
      in.fixed = dm.n_fixed > 0 ? io.fixed_qpos + row * dm.n_fixed : nullptr;
      in.last = t > 0 ? io.qpos + (row - 1) * nv : io.last_qpos + s * nv;
      in.projected = lp > 0 ? io.projected_ws + row * lp : nullptr;
      in.qpos = io.qpos + row * nv;
      in.gq = gq;
      in.fstatus = io.status != nullptr ? io.status[row] : 0;
      GradOutputs out;
      out.gkp = io.grad_keypoints != nullptr ? io.grad_keypoints + row * KP : nullptr;
      out.gref = nullptr;
      out.glast = gl;
      const int st = GradFrame<G>::run(sv, in, out, active);
      if (active && l == 0 && io.grad_status != nullptr) io.grad_status[row] = st;
      carry = (active && var >= 0) ? gl[var] : 0.f;
      __syncwarp();
    }
    if (active && var >= 0 && io.grad_last_qpos != nullptr) io.grad_last_qpos[s * nv + var] = carry;
    if (active && l < dof && io.grad_filter_state != nullptr) io.grad_filter_state[s * dof + l] = ybar;
  }
};

}  // namespace dexr
