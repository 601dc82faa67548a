/*
 * dexr_grad.h -- C ABI of libdexr_grad.so, the backward pass of dexr_solve_frames (include/dexr.h).
 *
 * A frame's forward solution x* minimises F(x; t, a) = sum_k w_k h(r_k(x) - t_k) + norm_delta |x - a|^2 over the box
 * [lower, upper]; t are the effective targets built from keypoints / ref_value, a is the (clipped) warm start.  Given the
 * upstream gradient dl/dx*, one call returns dl/dkeypoints (or dl/dref_value) and dl/dlast_qpos of every frame by implicit
 * differentiation at x*: one exact-Hessian build, one Cholesky factorisation and two triangular solves per frame.  Joints held
 * at a bound (x* on the bound with the gradient pointing outward) do not move with the inputs; the warm start's role as the
 * starting point is not differentiable and gets no gradient.
 *
 * A separate library so that libdexr.so stays the binary its profiles were taken on.  It needs no link to it: the device
 * table argument is the one dexr_robot_device_table() returns for the forward handle.
 * Return convention as in dexr.h: 0 on success, negative DEXR_E_* on failure, dexr_grad_last_error() for the message.
 */
#ifndef DEXR_GRAD_H_
#define DEXR_GRAD_H_

#include "dexr.h"

#ifdef __cplusplus
extern "C" {
#endif

#define DEXR_GRAD_VERSION 1

/* Per-frame status word of the backward call (grad_status).  Bits 0-1 are informational; bits 2-4 mean the frame's
 * gradient was set to zero. */
#define DEXR_GRAD_STATUS_ACTIVE (1 << 0)    /* some joints sit at an active bound (their adjoint is 0)                   */
#define DEXR_GRAD_STATUS_SHIFTED (1 << 1)   /* H_FF needed a diagonal shift mu diag|H_FF| (mu = 1e-6 * 10^j) to factorise */
#define DEXR_GRAD_STATUS_SINGULAR (1 << 2)  /* no shift up to 0.1 worked: zero gradient                                  */
#define DEXR_GRAD_STATUS_SKIPPED (1 << 3)   /* the forward status has DEXR_STATUS_MAXITER or _NONFINITE: zero gradient    */
#define DEXR_GRAD_STATUS_NONFINITE (1 << 4) /* a non-finite input or upstream gradient: zero gradient                     */

/* Buffers of one backward call.  DEVICE pointers, rows contiguous; the inputs are those of the forward call. */
typedef struct dexr_grad_frames {
  const float* keypoints;   /* [B,21,3]: exactly one of keypoints / ref_value, as in the forward call             */
  const float* ref_value;   /* [B,m,3]                                                                            */
  const float* fixed_qpos;  /* [B,n_fixed] or NULL when n_fixed == 0                                              */
  const float* last_qpos;   /* [B,n_var] the forward call's warm start / anchor                                   */
  const uint8_t* projected; /* [B,len_proj] DexPilot flags AFTER the forward call, or NULL; never written          */
  const float* qpos;        /* [B,n_var] forward solution x*                                                      */
  const int32_t* status;    /* [B] forward status words, or NULL                                                  */
  const float* grad_qpos;   /* [B,n_var] upstream gradient dl/dx*                                                 */
  float* grad_keypoints;    /* [B,21,3] or NULL (keypoints mode): overwritten; keypoints no residual reads get 0  */
  float* grad_ref_value;    /* [B,m,3] or NULL (ref_value mode): overwritten                                      */
  float* grad_last_qpos;    /* [B,n_var] or NULL: overwritten                                                     */
  int32_t* grad_status;     /* [B] or NULL: DEXR_GRAD_STATUS_* words                                              */
} dexr_grad_frames_t;

/* Buffers of one backward call through S streams of T frames (dexr_solve_sequences).  DEVICE pointers, rows contiguous.
 * The trace is the forward pass's unfiltered solution of every step; `last_qpos`, `projected` and `filter_init` are the state
 * the streams ENTERED the forward call with.  Upstream gradients: of the (filtered) robot qpos of every step, of the exit
 * last_qpos (= x*_{T-1}) and of the exit filter_state (= y_{T-1}); NULL stands for zero. */
typedef struct dexr_grad_sequences {
  /* inputs */
  const float* keypoints;             /* [S,T,21,3]                                                                  */
  const float* fixed_qpos;            /* [S,T,n_fixed] or NULL when n_fixed == 0                                     */
  const float* last_qpos;             /* [S,n_var] entry warm start / anchor of step 0                               */
  const uint8_t* projected;           /* [S,len_proj] entry DexPilot flags, or NULL (all cleared)                     */
  const uint8_t* filter_init;         /* [S] entry filter_init; required when the filter is on (params lp_alpha)     */
  const float* qpos;                  /* [S,T,n_var] trace: forward solution x*_t of every step                      */
  const int32_t* status;              /* [S,T] forward status words, or NULL                                         */
  const float* grad_robot_qpos;       /* [S,T,dof] dl/dy_t, or NULL                                                  */
  const float* grad_last_qpos_out;    /* [S,n_var] dl/d(exit last_qpos), or NULL                                     */
  const float* grad_filter_state_out; /* [S,dof] dl/d(exit filter_state), or NULL                                    */
  /* workspace */
  uint8_t* projected_ws;              /* [S,T,len_proj] the flags each step applied (replayed); required if len_proj  */
  /* outputs (overwritten) */
  float* grad_keypoints;              /* [S,T,21,3] or NULL                                                          */
  float* grad_last_qpos;              /* [S,n_var] dl/d(entry last_qpos), or NULL                                    */
  float* grad_filter_state;           /* [S,dof] dl/d(entry filter_state), or NULL                                   */
  int32_t* grad_status;               /* [S,T] DEXR_GRAD_STATUS_* words, or NULL                                     */
} dexr_grad_sequences_t;

int dexr_grad_version(void);
/* 16 hex digits: sha256 over the sources this library was compiled from (csrc/dexr_grad.cu, csrc/dexr_grad_kernels.cuh,
 * csrc/dexr_grad_seq_kernels.cuh, csrc/dexr_kernels.cuh, include/dexr_grad.h, include/dexr.h), stamped by
 * dex_retargeting_b200/build.py. */
const char* dexr_grad_build_id(void);
const char* dexr_grad_last_error(void);
size_t dexr_grad_frames_sizeof(void);
/* Enqueue the backward pass of num_frames frames on `cuda_stream` (asynchronous).  `table_host` is the host table the
 * forward handle was created from (launch dimensions, validation), `table_dev` its device copy (dexr_robot_device_table),
 * `params` the forward call's parameters; `preprocess` (raw detector landmarks) is not supported. */
int dexr_grad_frames(const dexr_table_t* table_host, const void* table_dev, const dexr_params_t* params,
                     const dexr_grad_frames_t* io, int64_t num_frames, int device, void* cuda_stream);

size_t dexr_grad_sequences_sizeof(void);
/* Enqueue the backward pass of S streams x T steps of dexr_solve_sequences (one group of lanes walks a stream backwards).
 * `params`: the forward call's (lp_alpha selects the filter; the warm-start clip is always on, as in the forward recurrence).
 * A step whose forward status is flagged, or whose backward is singular / non-finite, gets a zero gradient, and its zero
 * anchor adjoint stops the carry to earlier steps.  DexPilot flags get no gradient. */
int dexr_grad_sequences(const dexr_table_t* table_host, const void* table_dev, const dexr_params_t* params,
                        const dexr_grad_sequences_t* io, int64_t num_streams, int64_t num_steps, int device, void* cuda_stream);
/* The stream solver's low-pass filter on its own: y_t = finit ? fmaf(alpha, q_t - y_{t-1}, y_{t-1}) : q_t, then finit = 1,
 * over q [S,T,dof] -> y [S,T,dof], with filter_state [S,dof] / filter_init [S] read at entry and updated at exit exactly as
 * dexr_solve_sequences updates them.  With the solver run unfiltered (lp_alpha < 0) this gives the filtered call's bits. */
int dexr_grad_lowpass(const float* q, float* y, float* filter_state, uint8_t* filter_init, float alpha, int64_t num_streams,
                      int64_t num_steps, int dof, int device, void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* DEXR_GRAD_H_ */
