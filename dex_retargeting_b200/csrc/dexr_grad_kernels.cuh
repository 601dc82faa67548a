// dexr_grad_kernels.cuh -- the implicit-function backward pass of the batched frame solver (libdexr_grad.so).
//
// At the forward solution x* of a frame the solver's minimisation problem
//     F(x; t, a) = sum_k w_k h(r_k(x) - t_k) + norm_delta |x - a|^2     on the box [lower, upper]
// has g = dF/dx = 0 on the free joints and x*_i at a bound on the active ones.  Differentiating that condition, with the upstream
// gradient gbar = dl/dx* and the adjoint v solving H_FF v_F = gbar_F (v = 0 on active joints):
//     tbar_k = w_k d2h(r_k) (J_k v)        effective targets (the ones prepare_targets builds)
//     abar   = 2 norm_delta v              anchor (0 where clip_init moved the warm start)
// and the targets are mapped back to ref_value rows / keypoints by the adjoint of the prelude (scaling, DexPilot projection,
// keypoint gather).  H is the EXACT Hessian at x* (loss curvature through the Jacobian, kinematic curvature, regulariser,
// mimic fold), not the majorisers the forward iteration switches between.
//
// One group of G lanes per frame, lane = joint, exactly like the forward solver: this header reuses Solver<G, 0>'s
// table slice, forward kinematics, link placement, target prelude and collectives from dexr_kernels.cuh, which it includes
// unchanged.  New here: the exact-Hessian assembly, the active set, a Cholesky with a relative pivot floor and a diagonal
// shift retry, the two triangular solves and the target / keypoint / anchor adjoint.  tests/emu compiles this header with g++.
#pragma once

#include "dexr_kernels.cuh"
#include "../../include/dexr_grad.h"

namespace dexr {

// A pivot below this fraction of its original diagonal entry counts as a failed factorisation: fp32 cannot resolve the
// Schur complement below it (condition numbers beyond ~1e6).
constexpr float kGradPivotFloor = 1e-6f;
// Diagonal shifts mu diag|H_FF| tried after a failed factorisation: 1e-6, 1e-5, ..., 1e-1.
constexpr int kGradShifts = 6;

// Per-group scratch beyond Solver's: adjoint of the effective targets per residual, and the frame's DexPilot flags (a private
// copy: prepare_targets writes the flags it applies, the caller's post-forward flags are never touched).
template <int G>
struct GradScratch {
  static constexpr int kTbar = Scratch<G>::kFloats;             // [MAX_RES][4] ref_value-row adjoint of residual k
  static constexpr int kFlags = kTbar + DEXR_MAX_RES * 4;       // DEXR_MAX_RES bytes
  static constexpr int kFloats = kFlags + DEXR_MAX_RES / 4;
};

struct GradInputs {
  const float* kp;        // 63 floats (keypoints mode) or nullptr
  const float* ref;       // m*3 floats (ref mode) or nullptr
  const float* fixed;     // n_fixed floats or nullptr
  const float* last;      // n_var floats
  const uint8_t* projected;  // len_proj post-forward flags or nullptr
  const float* qpos;      // n_var floats: x*
  const float* gq;        // n_var floats: upstream gradient
  int fstatus;            // forward status word (0 if unknown)
};

struct GradOutputs {
  float* gkp;    // 63 floats or nullptr
  float* gref;   // m*3 floats or nullptr
  float* glast;  // n_var floats or nullptr
};

template <int G>
struct GradFrame {
  using SV = Solver<G, 0>;
  static constexpr int NP = G;

  // Returns the grad status word (DEXR_GRAD_STATUS_*); writes the outputs when `active`.  Every lane of the warp must call it.
  __device__ __forceinline__ static int run(SV& sv, const GradInputs& in, const GradOutputs& out, bool active) {
    const Dims& dm = sv.dm;
    const int l = sv.l, lane = sv.lane, var = sv.var;
    const int dof = dm.dof, m = dm.n_res, loss = dm.loss;
    const float nd = sv.prm.norm_delta, beta = sv.prm.huber_delta, inv_beta = sv.inv_beta;
    float* gs = sv.scf();
    float4* tbar_buf = reinterpret_cast<float4*>(gs + GradScratch<G>::kTbar);
    uint8_t* flags = reinterpret_cast<uint8_t*>(gs + GradScratch<G>::kFlags);
    int gstatus = 0;

    // ---- inputs: anchor (clipped warm start), x*, fixed joints, upstream gradient, targets
    float xin = 0.f, xs = 0.f, gbar = 0.f;
    if (active && var >= 0) { xin = in.last[var]; xs = in.qpos[var]; gbar = in.gq[var]; }
    bool anchor_live = true;  // d anchor / d last_qpos = 1 unless clip_init moved this coordinate
    if (sv.prm.clip_init && var >= 0) {
      const float c = fminf(fmaxf(xin, SV::ST().clip_lo[l]), SV::ST().clip_hi[l]);
      anchor_live = c == xin;
      xin = c;
    }
    sv.x0 = xin;
    sv.x = xs;
    const int fixedi = SV::ST().fixed_index[l];
    sv.qfix = (active && fixedi >= 0) ? in.fixed[fixedi] : 0.f;
    if (l < DEXR_MAX_RES) flags[l] = (active && in.projected != nullptr && l < dm.len_proj) ? in.projected[l] : 0;
    __syncwarp();
    FrameInputs fi;
    fi.kp = in.kp; fi.ref = in.ref; fi.fixed = in.fixed; fi.last = in.last;
    fi.projected = flags;  // (zeros when the caller has none: the same flags the forward derived from the distances alone)
    bool finite = isfinite(xin) && isfinite(xs) && isfinite(gbar) && isfinite(sv.qfix);
    const bool ok_targets = sv.prepare_targets(fi, active);
    finite = !gany<G>(!finite, lane) && ok_targets;
    __syncwarp();
    if (in.fstatus & (DEXR_STATUS_MAXITER | DEXR_STATUS_NONFINITE)) gstatus |= DEXR_GRAD_STATUS_SKIPPED;
    if (!finite) gstatus |= DEXR_GRAD_STATUS_NONFINITE;
    const bool live = active && gstatus == 0;
    if (!live) { sv.x = 0.f; sv.x0 = 0.f; sv.qfix = 0.f; gbar = 0.f; }

    // ---- kinematics at x*
    sv.q = sv.compose_q(sv.x);
    {
      float R[9];
      sv.fk(sv.q, R, sv.p);
      sv.write_world_links();
      sv.write_links(R, sv.p, 0);
      sv.set_world_axis(R);
    }
    __syncwarp();

    // ---- exact gradient and Hessian at x* (joint space), one residual at a time
    float H[NP];
#pragma unroll
    for (int i = 0; i < NP; ++i) H[i] = 0.f;
    float g = 0.f, t0 = 0.f, t1 = 0.f, t2 = 0.f;
    const bool rev = sv.jtype == 0;
    const float4* lpc = sv.lp(0);
    for (int k = 0; k < m; ++k) {
      float j0, j1, j2, rx, ry, rz;
      jacobian_column(sv, k, lpc, j0, j1, j2, rx, ry, rz);
      const float4 T = sv.fr()[k];
      float gx, gy, gz, y0, y1, y2;
      loss_terms(loss, T.w, beta, inv_beta, rx, ry, rz, j0, j1, j2, gx, gy, gz, y0, y1, y2);
      g = fmaf(j0, gx, fmaf(j1, gy, fmaf(j2, gz, g)));
      t0 += j1 * gz - j2 * gy; t1 += j2 * gx - j0 * gz; t2 += j0 * gy - j1 * gx;
      sv.jbuf(0, 0)[l] = j0; sv.jbuf(0, 1)[l] = j1; sv.jbuf(0, 2)[l] = j2;
      __syncwarp();
#pragma unroll
      for (int i = 0; i < NP; ++i)
        H[i] = fmaf(sv.jbuf(0, 0)[i], y0, fmaf(sv.jbuf(0, 1)[i], y1, fmaf(sv.jbuf(0, 2)[i], y2, H[i])));
      __syncwarp();
    }
    // kinematic curvature: H[l][i] += a_i . t_l (i ancestor-or-self of l), a_l . t_i (i descendant of l), revolute axes only
    {
      const float ar0 = rev ? sv.a[0] : 0.f, ar1 = rev ? sv.a[1] : 0.f, ar2 = rev ? sv.a[2] : 0.f;
      sv.at_a(l) = make_float4(ar0, ar1, ar2, 0.f);
      sv.at_t(l) = make_float4(t0, t1, t2, 0.f);
      __syncwarp();
#pragma unroll
      for (int i = 0; i < NP; ++i) {
        const float4 ai = sv.at_a(i);
        const float4 ti = sv.at_t(i);
        const float vu = fmaf(ai.x, t0, fmaf(ai.y, t1, ai.z * t2));
        const float vd = fmaf(ar0, ti.x, fmaf(ar1, ti.y, ar2 * ti.z));
        H[i] += ((sv.anc >> i) & 1u) ? vu : (((sv.desc >> i) & 1u) ? vd : 0.f);
      }
      __syncwarp();
    }
    // ---- mimic fold: H_x = M^T H_q M, g_x = M^T g_q (the forward solver's fold, restated)
    if (dm.has_mimic) {
      const float ml = var >= 0 ? 1.0f : (sv.msrc >= 0 ? sv.mmult : 0.f);
      float* hbuf = sv.hb();
#pragma unroll
      for (int i = 0; i < NP; ++i) hbuf[i * NP + l] = ml * H[i];
      __syncwarp();
#pragma unroll
      for (int i = 0; i < NP; ++i) H[i] = 0.f;
      const int gcount = SV::ST().group_count[l];
      for (int f = 0; f < DEXR_MAX_GROUP; ++f) {
        if (var >= 0 && f < gcount) {
          const int cl = SV::ST().group_lane[l][f];
#pragma unroll
          for (int i = 0; i < NP; ++i) H[i] += hbuf[i * NP + cl];
        }
      }
      __syncwarp();
#pragma unroll
      for (int i = 0; i < NP; ++i) hbuf[i * NP + l] = H[i];
      __syncwarp();
      float* hrow = sv.lcol();
      for (int s = 0; s < dof; ++s) {
        float acc = 0.f;
        const int cnt = SV::ST().group_count[s];
        for (int f = 0; f < cnt; ++f) acc = fmaf(SV::ST().group_mult[s][f], hbuf[SV::ST().group_lane[s][f] * NP + l], acc);
        hrow[s * NP + l] = acc;
      }
      __syncwarp();
#pragma unroll
      for (int s = 0; s < NP; ++s) H[s] = (s < dof) ? hrow[s * NP + l] : 0.f;
      float gx_ = 0.f;
#pragma unroll
      for (int f = 0; f < DEXR_MAX_GROUP; ++f) {
        const bool v = var >= 0 && f < gcount;
        const float gv = gshfl<G>(g, v ? SV::ST().group_lane[l][f] : l);
        if (v) gx_ = fmaf(SV::ST().group_mult[l][f], gv, gx_);
      }
      g = gx_;
      __syncwarp();
    }

    // ---- regulariser, active set (the rule of the float64 polish: at a bound with the gradient pointing outward)
    const bool isvar = var >= 0;
    g = isvar ? fmaf(2.0f * nd, sv.x - sv.x0, g) : 0.f;
    const bool act = isvar && ((sv.x <= sv.lo && g > 0.f) || (sv.x >= sv.hi && g < 0.f));
    const bool free_ = isvar && !act;
    const unsigned fmask = gballot<G>(free_, lane);
    if (act) gstatus |= DEXR_GRAD_STATUS_ACTIVE;  // (made group-wide below)
    // reduced system: rows / columns of frozen lanes become identity, regulariser on the free diagonal
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      const bool keep = free_ && ((fmask >> j) & 1u);
      float v = keep ? H[j] : 0.f;
      if (j == l) v = free_ ? v + 2.0f * nd : (l < dof ? 1.0f : 0.f);
      H[j] = v;
    }
    float* hbuf = sv.hb();
#pragma unroll
    for (int i = 0; i < NP; ++i) hbuf[i * NP + l] = H[i];
    __syncwarp();
    const float D = l < dof ? fabsf(hbuf[l * NP + l]) : 0.f;  // diag|H_FF| (1 on frozen lanes)
    const float rhs = free_ ? gbar : 0.f;

    // ---- Cholesky H_FF + mu diag|H_FF| = L L^T with the forward solver's rotating-row layout, then the two triangular
    // solves.  mu = 0 first; after a failure (or a pivot below the relative floor) the smallest working shift of the ladder.
    float v = 0.f;
    bool solved = false;
    int shifts = 0;
    for (int att = 0; att <= kGradShifts; ++att) {
      if (!gany<32>(!solved, lane)) break;  // (warp-uniform: the two groups of a 16-lane warp retry together)
      float mu = 0.f;
      if (att > 0) { mu = 1e-6f; for (int e = 1; e < att; ++e) mu *= 10.f; }
      if (att > 0) {
#pragma unroll
        for (int i = 0; i < NP; ++i) H[i] = hbuf[i * NP + l];
      }
      float y = rhs, myinv = 1.0f;
      bool bad = false;
      float* Lr = sv.lrow();
      float* Lc = sv.lcol();
      __syncwarp();
      for (int k = 0; k < dof; ++k) {
        float hk = H[0];
        if (k == l) hk = fmaf(mu, D, hk);
        const float dkk = gshfl<G>(hk, k);
        const float Dk = gshfl<G>(D, k);
        bad = bad || !(dkk > kGradPivotFloor * Dk) || !(dkk > 1e-30f);
        const float inv = 1.0f / sqrtf(fmaxf(dkk, 1e-30f));
        const float lik = hk * inv;
        const float yk = gshfl<G>(y, k) * inv;
        if (l == k) { myinv = inv; y = yk; }
        if (l > k) y = fmaf(-lik, yk, y);
        float* row = Lr + (k & 1) * NP;
        row[(l - k - 1) & (NP - 1)] = lik;
        Lc[k * (NP + 1) + l] = lik;
        __syncwarp();
        const int live = dof - k - 1;  // columns right of the pivot; the registers beyond stand for no joint
#pragma unroll
        for (int j = 0; j < NP; ++j) H[j] = fmaf(-lik, j < live ? row[j] : 0.f, j + 1 < NP ? H[j + 1] : 0.f);
        __syncwarp();
      }
      for (int k = dof - 1; k >= 0; --k) {
        const float xk = gshfl<G>(y * myinv, k);
        if (l == k) y = xk;
        if (l < k) y = fmaf(-Lc[l * (NP + 1) + k], xk, y);
      }
      bad = gany<G>(bad || !isfinite(y), lane);
      if (!solved && !bad) {
        v = free_ ? y : 0.f;
        solved = true;
        shifts = att;
      }
      __syncwarp();
    }
    if (!solved && live) gstatus |= DEXR_GRAD_STATUS_SINGULAR;
    if (shifts > 0) gstatus |= DEXR_GRAD_STATUS_SHIFTED;
    gstatus |= gany<G>((gstatus & DEXR_GRAD_STATUS_ACTIVE) != 0, lane) ? DEXR_GRAD_STATUS_ACTIVE : 0;
    const bool zero = (gstatus & (DEXR_GRAD_STATUS_SKIPPED | DEXR_GRAD_STATUS_NONFINITE | DEXR_GRAD_STATUS_SINGULAR)) != 0;
    if (zero || !live) v = 0.f;

    // ---- anchor adjoint
    if (active && out.glast != nullptr && var >= 0) out.glast[var] = anchor_live ? 2.0f * nd * v : 0.f;

    // ---- target adjoint: tbar_k = w_k d2h(r_k) J_k v, with J_k v = sum over joints of J_k[:, c] (M v)_c
    float vq = var >= 0 ? v : 0.f;
    {
      const float src = gshfl<G>(v, sv.msrc >= 0 ? sv.msrc : l);
      if (var < 0 && sv.msrc >= 0) vq = sv.mmult * src;
    }
    for (int k = 0; k < m; ++k) {
      float j0, j1, j2, rx, ry, rz;
      jacobian_column(sv, k, lpc, j0, j1, j2, rx, ry, rz);
      const float jv0 = gsum<G>(j0 * vq), jv1 = gsum<G>(j1 * vq), jv2 = gsum<G>(j2 * vq);
      if (l == k) {
        const float4 T = sv.fr()[k];
        float tb0, tb1, tb2;
        if (loss == DEXR_LOSS_POSITION) {
          tb0 = fabsf(rx) < beta ? T.w * inv_beta * jv0 : 0.f;
          tb1 = fabsf(ry) < beta ? T.w * inv_beta * jv1 : 0.f;
          tb2 = fabsf(rz) < beta ? T.w * inv_beta * jv2 : 0.f;
        } else {
          const float d = sqrtf(fmaf(rx, rx, fmaf(ry, ry, rz * rz)));
          if (d < beta) {
            tb0 = T.w * inv_beta * jv0; tb1 = T.w * inv_beta * jv1; tb2 = T.w * inv_beta * jv2;
          } else {
            const float invd = 1.0f / d;
            const float ux = rx * invd, uy = ry * invd, uz = rz * invd;
            const float uj = fmaf(ux, jv0, fmaf(uy, jv1, uz * jv2));
            const float s = T.w * invd;
            tb0 = s * fmaf(-uj, ux, jv0); tb1 = s * fmaf(-uj, uy, jv1); tb2 = s * fmaf(-uj, uz, jv2);
          }
        }
        // (a zeroed frame may have non-finite targets: store exact zeros, not 0 * NaN)
        tbar_buf[k] = (zero || !live) ? make_float4(0.f, 0.f, 0.f, 0.f) : ref_row_adjoint(sv, in, k, flags, tb0, tb1, tb2);
      }
    }
    __syncwarp();
    if (active && out.gref != nullptr) {
      for (int e = l; e < 3 * m; e += G) {
        const float4 r = tbar_buf[e / 3];
        out.gref[e] = (e % 3 == 0) ? r.x : (e % 3 == 1 ? r.y : r.z);
      }
    }
    // ---- keypoint adjoint: the gather rho_k = kp[task_k] - kp[origin_k] (or kp[idx_k]) transposed, one keypoint per lane
    if (active && out.gkp != nullptr) {
      for (int c = l; c < DEXR_NUM_KEYPOINTS; c += G) {
        float a0 = 0.f, a1 = 0.f, a2 = 0.f;
        for (int k = 0; k < m; ++k) {
          const float4 r = tbar_buf[k];
          if (SV::ST().res_ht[k] == c) { a0 += r.x; a1 += r.y; a2 += r.z; }
          if (SV::ST().res_ho[k] == c) { a0 -= r.x; a1 -= r.y; a2 -= r.z; }
        }
        out.gkp[3 * c] = a0; out.gkp[3 * c + 1] = a1; out.gkp[3 * c + 2] = a2;
      }
    }
    __syncwarp();
    return gstatus;
  }

  // Jacobian column of lane l for residual k (task minus origin link) and the residual r_k = p_task - p_origin - t_k.
  __device__ __forceinline__ static void jacobian_column(const SV& sv, int k, const float4* lpc, float& j0, float& j1, float& j2,
                                                         float& rx, float& ry, float& rz) {
    const int l = sv.l;
    const int ti = SV::ST().res_task[k], oi = SV::ST().res_origin[k];
    const float4 T = sv.fr()[k];
    const float4 pt = lpc[ti];
    const uint32_t mt = SV::ST().link_anc[ti];
    const bool rev = sv.jtype == 0;
    rx = pt.x - T.x; ry = pt.y - T.y; rz = pt.z - T.z;
    j0 = 0.f; j1 = 0.f; j2 = 0.f;
    if ((mt >> l) & 1u) {
      if (rev) {
        const float dx = pt.x - sv.p[0], dy = pt.y - sv.p[1], dz = pt.z - sv.p[2];
        j0 = sv.a[1] * dz - sv.a[2] * dy; j1 = sv.a[2] * dx - sv.a[0] * dz; j2 = sv.a[0] * dy - sv.a[1] * dx;
      } else { j0 = sv.a[0]; j1 = sv.a[1]; j2 = sv.a[2]; }
    }
    if (oi >= 0) {
      const float4 po = lpc[oi];
      const uint32_t mo = SV::ST().link_anc[oi];
      rx -= po.x; ry -= po.y; rz -= po.z;
      if ((mo >> l) & 1u) {
        if (rev) {
          const float dx = po.x - sv.p[0], dy = po.y - sv.p[1], dz = po.z - sv.p[2];
          j0 -= sv.a[1] * dz - sv.a[2] * dy; j1 -= sv.a[2] * dx - sv.a[0] * dz; j2 -= sv.a[0] * dy - sv.a[1] * dx;
        } else { j0 -= sv.a[0]; j1 -= sv.a[1]; j2 -= sv.a[2]; }
      }
    }
  }

  // Loss gradient w.r.t. the residual (gx, gy, gz) and the exact loss curvature applied to the Jacobian column (y0, y1, y2).
  __device__ __forceinline__ static void loss_terms(int loss, float w, float beta, float inv_beta, float rx, float ry, float rz,
                                                    float j0, float j1, float j2, float& gx, float& gy, float& gz, float& y0,
                                                    float& y1, float& y2) {
    if (loss == DEXR_LOSS_POSITION) {  // per-coordinate Huber: curvature 1/beta inside, 0 outside
      const bool qx = fabsf(rx) < beta, qy = fabsf(ry) < beta, qz = fabsf(rz) < beta;
      gx = w * (qx ? rx * inv_beta : copysignf(1.f, rx));
      gy = w * (qy ? ry * inv_beta : copysignf(1.f, ry));
      gz = w * (qz ? rz * inv_beta : copysignf(1.f, rz));
      y0 = qx ? w * inv_beta * j0 : 0.f; y1 = qy ? w * inv_beta * j1 : 0.f; y2 = qz ? w * inv_beta * j2 : 0.f;
    } else {  // norm Huber: I / beta inside, (I - u u^T) / |r| outside
      const float d = sqrtf(fmaf(rx, rx, fmaf(ry, ry, rz * rz)));
      const bool quad = d < beta;
      const float invd = d > 1e-30f ? 1.0f / d : 0.f;
      const float ux = rx * invd, uy = ry * invd, uz = rz * invd;
      const float hp = quad ? d * inv_beta : 1.0f;
      gx = w * hp * ux; gy = w * hp * uy; gz = w * hp * uz;
      const float s_iso = w * (quad ? inv_beta : invd);
      const float s_rad = quad ? 0.f : w * invd;
      const float uj = s_rad * fmaf(ux, j0, fmaf(uy, j1, uz * j2));
      y0 = fmaf(s_iso, j0, -uj * ux); y1 = fmaf(s_iso, j1, -uj * uy); y2 = fmaf(s_iso, j2, -uj * uz);
    }
  }

  // Adjoint of the prelude's map from the ref_value row rho_k (= the keypoint difference) to the effective target t_k:
  // scaling, or the DexPilot projection t = eta rho / (|rho| + 1e-6) on rows whose flag is set.
  __device__ __forceinline__ static float4 ref_row_adjoint(const SV& sv, const GradInputs& in, int k, const uint8_t* flags,
                                                           float tb0, float tb1, float tb2) {
    const Dims& dm = sv.dm;
    if (dm.loss == DEXR_LOSS_POSITION) return make_float4(tb0, tb1, tb2, 0.f);
    const float s = sv.prm.scaling;
    if (dm.loss == DEXR_LOSS_DEXPILOT && k < dm.len_proj && flags[k]) {
      float px, py, pz;
      if (in.kp != nullptr) {
        const int ht = SV::ST().res_ht[k], ho = SV::ST().res_ho[k];
        px = in.kp[3 * ht]; py = in.kp[3 * ht + 1]; pz = in.kp[3 * ht + 2];
        if (ho >= 0) { px -= in.kp[3 * ho]; py -= in.kp[3 * ho + 1]; pz -= in.kp[3 * ho + 2]; }
      } else {
        px = in.ref[3 * k]; py = in.ref[3 * k + 1]; pz = in.ref[3 * k + 2];
      }
      const float eta = k < dm.len_s1 ? sv.prm.eta1 : sv.prm.eta2;
      const float n = sqrtf(fmaf(px, px, fmaf(py, py, pz * pz)));
      const float c = eta / (n + 1e-6f);
      // d t / d rho = c (I - rho rho^T / (|rho| (|rho| + 1e-6))), symmetric
      const float pr = n > 0.f ? fmaf(px, tb0, fmaf(py, tb1, pz * tb2)) / (n * (n + 1e-6f)) : 0.f;
      return make_float4(c * fmaf(-pr, px, tb0), c * fmaf(-pr, py, tb1), c * fmaf(-pr, pz, tb2), 0.f);
    }
    return make_float4(s * tb0, s * tb1, s * tb2, 0.f);
  }
};

}  // namespace dexr
