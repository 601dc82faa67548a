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

int dexr_grad_version(void);
/* 16 hex digits: sha256 over the sources this library was compiled from (csrc/dexr_grad.cu, csrc/dexr_grad_kernels.cuh,
 * csrc/dexr_kernels.cuh, include/dexr_grad.h, include/dexr.h), stamped by dex_retargeting_b200/build.py. */
const char* dexr_grad_build_id(void);
const char* dexr_grad_last_error(void);
size_t dexr_grad_frames_sizeof(void);
/* Enqueue the backward pass of num_frames frames on `cuda_stream` (asynchronous).  `table_host` is the host table the
 * forward handle was created from (launch dimensions, validation), `table_dev` its device copy (dexr_robot_device_table),
 * `params` the forward call's parameters; `preprocess` (raw detector landmarks) is not supported. */
int dexr_grad_frames(const dexr_table_t* table_host, const void* table_dev, const dexr_params_t* params,
                     const dexr_grad_frames_t* io, int64_t num_frames, int device, void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* DEXR_GRAD_H_ */
