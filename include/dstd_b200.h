/*
 * dstd_b200.h — C ABI of libdstd_b200.so: the B200 (sm_100a) DSTD-GC hot path.
 *
 * The reference (Jaakk0F/DSTD-GCN) has no FFI: its hot path is Python calling
 * ATen.  Each entry point below replaces a group of ATen call sites (file:line
 * into /root/reference) and is what a maintainer's ctypes stub binds
 * (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - plain pointers + sizes, no torch types; every buffer (outputs, saved
 *     tensors, workspace, gradients) is owned by the caller; the library never
 *     allocates, frees or synchronises; all work is enqueued on `stream`.
 *   - all tensors are fp32 device memory; element strides (not bytes).
 *   - return 0 on success, a negative dstd_status otherwise;
 *     dstd_last_error() gives a thread-local message.
 *   - no global mutable state except the per-thread error string and one-time
 *     cudaFuncSetAttribute calls; entry points are re-entrant and may be called
 *     from autograd worker threads (they do not change the current device).
 *
 * Unit coordinates.  One DSTD-GC "unit" works on x[n, c, p, k]:
 *     spatial  unit: p = frame t (P = T), k = joint v (K = V)
 *     temporal unit: p = joint v (P = V), k = frame t (K = T)
 *   so a [N,C,T,V] tensor is passed with (sp,sk) = (V,1) to a spatial unit and
 *   (1,V) to a temporal unit; the fast variant's [N,T,V,C] tensor uses sc = 1.
 */
#ifndef DSTD_B200_H
#define DSTD_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* dstd_stream_t; /* cudaStream_t */

typedef enum {
  DSTD_OK = 0,
  DSTD_ERR_BAD_ARG = -1,      /* null pointer / non-positive dim / inconsistent args */
  DSTD_ERR_UNSUPPORTED = -2,  /* shape outside the compiled tile limits */
  DSTD_ERR_WORKSPACE = -3,    /* workspace smaller than dstd_*_workspace_bytes() */
  DSTD_ERR_CUDA = -4          /* CUDA runtime error at launch */
} dstd_status;

/* strided fp32 view addressed by (n, c, p, k) */
typedef struct {
  float* ptr;
  long long sn, sc, sp, sk;
} dstd_view;

#define DSTD_MAX_BRANCH 2

/* flags */
#define DSTD_FLAG_ADJ_T 1  /* fast variant (dstdgcn_fast.py:125,145): the dynamic adjacency is applied transposed */

/* weights of one DSTD-GC branch (model/dstdgcn.py:66-71).  Cin/Cout/P as in the args struct. */
typedef struct {
  const float *w_m1, *b_m1; /* conv_m1  [2,Cin] [2] */
  const float *w_m2, *b_m2; /* conv_m2  [2,Cin] [2] */
  const float *w_rm, *b_rm; /* conv_rm  [P,2P]  [P] */
  const float *w_f, *b_f;   /* conv_f   [Cout,Cin] [Cout] */
  const float *adj;         /* static adjacency [K,K]           (A_s[i] / A_t[i]) */
  const float *adj_w;       /* optional elementwise weight [K,K] (W_s[i]); NULL => 1 */
  const float *adj_r;       /* optional additive term [K,K]      (R_s[i] / R_t[i]); NULL => 0 */
} dstd_branch;

/* gradients of the above; any pointer may be NULL (not wanted).  Written, not accumulated. */
typedef struct {
  float *w_m1, *b_m1, *w_m2, *b_m2, *w_rm, *b_rm, *w_f, *b_f;
  float *adj_eff; /* d/d(adj*adj_w + adj_r) [K,K]  (= dR_s / dR_t; fast variant: dA_s)  (dstdgcn.py:149,160) */
  float *adj_w;   /* d/d adj_w = adj * adj_eff [K,K] (dW_s); only written when the branch has adj_w */
} dstd_branch_grad;

/* ---------------------------------------------------------------------------------------------
 * DSTD-GC unit: sum over nb branches of DSTDGC.forward (model/dstdgcn.py:80-94, called from
 * DSTDGCB.forward :145-150 / :157-161; fast: dstdgcn_fast.py:108-155).
 *   m [n,b,j,p,k]   = W{m1,m2}_b x + b            j = 0,1: conv_m1 rows; 2,3: conv_m2 rows
 *   pd[n,b,p,v,w]   = sum_{r,p'} Wrm_b[p, r*P+p'] tanh(m[n,b,r,p',v] - m[n,b,2+r,p',w]) + brm_b[p]
 *   xm              = alpha * pd + (adj*adj_w + adj_r)
 *   xa[n,b,c,p,w]   = sum_v x[n,c,p,v] xm[n,b,p,v,w]   (row c = Cin: x := 1, i.e. column sums of xm)
 *   out[n,o,p,w]    = sum_b ( sum_c Wf_b[o,c] xa[n,b,c,p,w] + bf_b[o] xa[n,b,Cin,p,w] ) (+ skip)
 * With DSTD_FLAG_ADJ_T the aggregation uses xm[n,b,p,w,v] instead (fast variant).
 * m, pd (and xa, see dstd_gc_needs_xa) are written and must be kept for the backward call.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int N, Cin, Cout, P, K, nb, flags;
  dstd_view x;           /* [N,Cin,P,K] */
  dstd_view out;         /* [N,Cout,P,K] */
  dstd_view skip;        /* optional (ptr NULL => none): added to out (ST_GCNN_layer skip, dstdgcn.py:248) */
  const float* alpha;    /* device scalar (alpha_sm / alpha_tm); NULL => 1 */
  dstd_branch br[DSTD_MAX_BRANCH];
  float* m;              /* [N,nb,4,P,K] */
  float* pd;             /* [N,nb,P,K,K] */
  float* xa;             /* [N,nb,Cin+1,P,K]; NULL allowed when !dstd_gc_needs_xa() */
  void* ws;              /* workspace, dstd_gc_fwd_workspace_bytes() */
  size_t ws_bytes;
} dstd_gc_fwd_args;

typedef struct {
  int N, Cin, Cout, P, K, nb, flags;
  dstd_view x;           /* forward input */
  dstd_view gout;        /* gradient of out; (the gradient of skip is gout itself) */
  dstd_view gx;          /* gradient of x, written */
  const float* alpha;
  dstd_branch br[DSTD_MAX_BRANCH];
  const float* m;        /* saved by forward */
  const float* pd;
  const float* xa;
  dstd_branch_grad gbr[DSTD_MAX_BRANCH];
  float* galpha;         /* [1], written; NULL => not wanted */
  void* ws;              /* dstd_gc_bwd_workspace_bytes() */
  size_t ws_bytes;
  dstd_view gx_add;      /* optional (ptr may be NULL): gx = d(out)/d(x)^T gout + gx_add, i.e. another gradient of x
                            (in DSTDGCB the block input also feeds the BN residual, model/dstdgcn.py:145,153) summed
                            in the pass that writes gx instead of by a separate add */
} dstd_gc_bwd_args;

/* 1 when dstd_gc_backward for this shape reads the saved `xa` (unfused fallback); 0 when the fused backward recomputes
 * it on chip, in which case `xa` may be NULL in both calls. */
int dstd_gc_needs_xa(int Cin, int Cout, int P, int K, int nb);
size_t dstd_gc_fwd_workspace_bytes(int N, int Cin, int Cout, int P, int K, int nb);
size_t dstd_gc_bwd_workspace_bytes(int N, int Cin, int Cout, int P, int K, int nb);
int dstd_gc_forward(const dstd_gc_fwd_args* a, dstd_stream_t stream);
int dstd_gc_backward(const dstd_gc_bwd_args* a, dstd_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Fused BatchNorm(C*V channels, statistics over N,T) + residual add + PReLU + dropout mask:
 *   out = mask * prelu( gamma * (y - mean) * invstd + beta + r )
 * replaces BatchNorm.forward (model/dstdgcn.py:44-50; fast dstdgcn_fast.py:50-56), `x += r`,
 * `self.prelu(x)` (:152-154), bn_in/prelu/do_in (:306-308) and encoders[i][1:3] (:283-284).
 * Views are addressed (n,c,t,v) -> (n,c,p,k).  BN parameter index is c*V+v, or v*C+c when vc_order.
 * training: batch statistics (biased variance), running stats updated with `momentum`
 * (unbiased variance), *num_batches_tracked += 1.  eval: running statistics.
 * Shapes: V <= 128 joints and T*V <= 4096 positions.  Planes of 4097 .. 8192 positions run only
 * when V > 32 and the bulk-copy kernels take the call: no mask, dense 16-byte aligned channel
 * slabs, the channel count a multiple of the slab's (1, 2 or 4 channels, at most 2 above 4096
 * positions), DSTD_BN_FAST not 0.  Otherwise DSTD_ERR_UNSUPPORTED.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int N, C, T, V;
  int vc_order;
  int training;
  float eps, momentum;
  dstd_view y;
  dstd_view r;                 /* optional */
  dstd_view out;
  const float *gamma, *beta;   /* [C*V] */
  float *running_mean, *running_var;     /* [C*V]; may be NULL in training (no tracking) */
  long long* num_batches_tracked;        /* device int64 scalar; may be NULL */
  const float* prelu;          /* device scalar slope; NULL => no activation */
  const float* mask;           /* optional, contiguous, same element order as `out` is WRITTEN
                                  logically: index ((n*C+c)*T+t)*V+v */
  float *save_mean, *save_invstd;        /* [C*V], written (needed by backward) */
  void* ws;
  size_t ws_bytes;
} dstd_bn_act_fwd_args;

typedef struct {
  int N, C, T, V;
  int vc_order;
  int training;
  dstd_view y;
  dstd_view r;                 /* optional, as in forward */
  dstd_view gout;
  dstd_view gy;                /* written */
  dstd_view gr;                /* written when ptr != NULL (requires r) */
  const float *gamma, *beta;
  const float* prelu;
  const float* mask;
  const float *save_mean, *save_invstd;
  float *ggamma, *gbeta;       /* [C*V], written */
  float* gprelu;               /* [1], written when prelu != NULL and ptr != NULL */
  void* ws;
  size_t ws_bytes;
  dstd_view gr_add;            /* optional (ptr may be NULL; requires gr): gr = d(pre-activation) + gr_add.  Lets the
                                  caller fold another gradient of the same tensor into this pass -- in DSTDGCB the
                                  block input is both the BN residual (model/dstdgcn.py:153) and the layer skip
                                  (:248), and autograd would otherwise sum the two with a separate strided add */
} dstd_bn_act_bwd_args;

size_t dstd_bn_act_workspace_bytes(int N, int C, int T, int V);
int dstd_bn_act_forward(const dstd_bn_act_fwd_args* a, dstd_stream_t stream);
int dstd_bn_act_backward(const dstd_bn_act_bwd_args* a, dstd_stream_t stream);

/* Synchronised BatchNorm (data parallel: statistics over the batches of all ranks).  Each direction of a
 * training-mode call (training = 1, else DSTD_ERR_BAD_ARG) runs as two phases; between them the caller all-gathers
 * one fp64 buffer of dstd_bn_sync_buffer_doubles(C, V) = 3*C*V doubles per rank, in rank order, into
 * `all` = double[world][3][C*V] (BN parameter order c*V+v, or v*C+c when vc_order).
 *   forward  local : writes `mine` = (count, mean, M2) of this rank's batch; no outputs (of the tensors only y and
 *                    the workspace are used).
 *   forward  global: merges the rows in rank order (Chan), writes save_mean / save_invstd, the running statistics
 *                    (global count, unbiased variance), num_batches_tracked += 1, and `out`.
 *   backward local : writes this rank's ggamma / gbeta / gprelu (sums over this rank's batch only: they are summed
 *                    over ranks with the other parameter gradients) and `mine` = (count, sum g', sum g' xhat), where
 *                    g' is the gradient of the pre-activation and save_mean / save_invstd hold the global statistics.
 *   backward global: writes gy (and gr) from the rank-order fp64 sums of the gathered rows over the global count.
 * The global phases use no workspace (ws may be NULL) and the global backward no ggamma / gbeta / gprelu (may be
 * NULL).  The local backward does not write gy / gr but needs them (their layouts pick the same kernels as the plain
 * call); the caller passes the buffers the global backward will write.  Identical `all` buffers give bit-identical
 * results on every rank. */
size_t dstd_bn_sync_buffer_doubles(int C, int V);
int dstd_bn_act_forward_local(const dstd_bn_act_fwd_args* a, double* mine, dstd_stream_t stream);
int dstd_bn_act_forward_global(const dstd_bn_act_fwd_args* a, const double* all, int world, dstd_stream_t stream);
int dstd_bn_act_backward_local(const dstd_bn_act_bwd_args* a, double* mine, dstd_stream_t stream);
int dstd_bn_act_backward_global(const dstd_bn_act_bwd_args* a, const double* all, int world, dstd_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * 1x1 channel mix  out[n,o,p,k] = sum_c w[o,c] x[n,c,p,k] + b[o]
 * replaces DSTDGCB.residual[0] (nn.Conv2d 1x1, model/dstdgcn.py:118; nn.Linear in fast :183-186)
 * and ST_GCNN_layer.residual conv (:228).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int N, Cin, Cout, P, K;
  dstd_view x, out;
  const float *w, *b;          /* [Cout,Cin], [Cout] (b may be NULL) */
} dstd_chmix_fwd_args;

typedef struct {
  int N, Cin, Cout, P, K;
  dstd_view x, gout, gx;       /* gx.ptr may be NULL */
  const float* w;
  float *gw, *gb;              /* written; may be NULL */
  void* ws;
  size_t ws_bytes;
} dstd_chmix_bwd_args;

size_t dstd_chmix_bwd_workspace_bytes(int N, int Cin, int Cout, int P, int K);
int dstd_chmix_forward(const dstd_chmix_fwd_args* a, dstd_stream_t stream);
int dstd_chmix_backward(const dstd_chmix_bwd_args* a, dstd_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Model head / tail (DSTDGCN.forward, model/dstdgcn.py:298-303 and :314-315; fast :553-557,:611).
 *   prep  : h[n,c,t,v] = x[n,t,v,c]                     c < 3
 *           h[n,c,t,v] = x[n,t,v,c-3] - x[n,T-1,v,c-3]  3 <= c < 6
 *   finish: y[n,t,v,c] = z[n,c,t,v] + x[n,T-1,v,c]
 * x, y, gx, gy are contiguous [N,T,V,3].
 * ------------------------------------------------------------------------------------------- */
int dstd_prep_forward(const float* x, dstd_view h, int N, int T, int V, dstd_stream_t stream);
int dstd_prep_backward(dstd_view gh, float* gx, int N, int T, int V, dstd_stream_t stream);
int dstd_finish_forward(dstd_view z, const float* x, float* y, int N, int T, int V, dstd_stream_t stream);
/* gz[n,c,t,v] = gy[n,t,v,c]; gx[n,t,v,c] = (t == T-1) ? sum_t' gy[n,t',v,c] : 0 (gx may be NULL) */
int dstd_finish_backward(const float* gy, dstd_view gz, float* gx, int N, int T, int V, dstd_stream_t stream);
/* The same four for D coordinates per joint, 1 <= D <= 32 (DSTDGCN(input_channels = 2*D)): x, y, gx, gy are contiguous
 * [N,T,V,D], h / gh have 2*D channels, z / gz have D.  D = 3 computes the bits of the calls above.  D outside 1..32:
 * DSTD_ERR_UNSUPPORTED. */
int dstd_prep_forward_d(const float* x, dstd_view h, int N, int T, int V, int D, dstd_stream_t stream);
int dstd_prep_backward_d(dstd_view gh, float* gx, int N, int T, int V, int D, dstd_stream_t stream);
int dstd_finish_forward_d(dstd_view z, const float* x, float* y, int N, int T, int V, int D, dstd_stream_t stream);
int dstd_finish_backward_d(const float* gy, dstd_view gz, float* gx, int N, int T, int V, int D, dstd_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Engine glue on device (engine/prediction.py:253-258,290-294; engine/utils/loss.py:52-65):
 *   mpjpe : loss = mean_j || pred[j,:] - target[j,:] ||_2 over J 3-vectors; writes the loss scalar
 *           (accumulating `scale * loss` into *loss_out when accumulate != 0) and
 *           gpred = scale * d loss / d pred.
 *   adam  : torch.optim.Adam semantics (no amsgrad, no weight decay unless wd != 0, coupled L2) on a
 *           flat parameter bucket; `step` is the 1-based step count; grad is multiplied by grad_scale
 *           first (1/world_size after an all-reduce(sum)).  When `lr_dev` / `step_dev` are non-NULL the kernel reads
 *           the learning rate / step count from device memory instead (so that a CUDA graph of the whole training
 *           step stays valid across steps and StepLR updates).
 * ------------------------------------------------------------------------------------------- */
size_t dstd_mpjpe_workspace_bytes(long long J);
int dstd_mpjpe_forward_backward(const float* pred, const float* target, long long J, float scale, int accumulate,
                                float* loss_out, float* gpred, void* ws, size_t ws_bytes, dstd_stream_t stream);
/* pose error: mpjpe over J D-vectors, 1 <= D <= 32 (pred, target, gpred contiguous [J,D]); same deterministic
 * two-kernel reduction, accumulate and scale; D = 3 computes the bits of dstd_mpjpe_forward_backward.  D outside
 * 1..32: DSTD_ERR_UNSUPPORTED. */
size_t dstd_pose_error_workspace_bytes(long long J);
int dstd_pose_error_forward_backward(const float* pred, const float* target, long long J, int D, float scale,
                                     int accumulate, float* loss_out, float* gpred, void* ws, size_t ws_bytes,
                                     dstd_stream_t stream);
int dstd_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                   float beta1, float beta2, float eps, float weight_decay, float grad_scale, int step,
                   const float* lr_dev, const int* step_dev, dstd_stream_t stream);

/* misc */
const char* dstd_last_error(void);
const char* dstd_version(void);      /* "dstd_b200 <ver> sm_100a" */
int dstd_kernel_launch_count(void);  /* kernels launched by this library in this process (monotonic) */
/* Device-side failures.  A tensor-core pipeline whose completion barrier times out cannot return a status (nothing here
 * synchronises), so the kernel poisons its outputs with NaN and writes a code into a host-mapped word; every later
 * dstd_gc_* call then fails with DSTD_ERR_CUDA until the word is cleared.  dstd_device_error returns the word (0 = none)
 * and clears it when `clear` != 0; dstd_debug_raise_device_error sets it from a kernel on `stream` (test hook). */
int dstd_device_error(int clear);
int dstd_debug_raise_device_error(int code, dstd_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DSTD_B200_H */
