// Fused BatchNorm(C*V channels, statistics over N,T) + residual + PReLU + dropout mask, forward and backward
// (model/dstdgcn.py:44-50 BatchNorm.forward, :152-154 `x = bn(x); x += r; x = prelu(x)`, :306-308, :283-284).
//
// Kernel families:
//  * generic (bn_stats, bn_apply, bn_bwd_reduce, bn_bwd_apply): any strides, dropout mask.  CTA = (channel c, batch
//    split s); a thread owns up to BN_MAXJ fixed (t,v) positions of the T x V plane and walks the samples of its
//    split, so the per-(c,v) BN parameters are per-thread constants and every access to a [T x V] plane is one
//    contiguous, coalesced sweep.  When the producer and the consumer keep the plane in different memory orders
//    (T-major vs V-major: this op is where the block switches between the spatial and the temporal unit layout) the
//    plane is transposed through shared memory.
//  * fast (bnf_apply, bnf_bwd_reduce, bnf_bwd_apply): dense CH-channel slabs staged by bulk copies ("fast path"
//    below); bit-identical to the generic kernels.
//  * synchronised BatchNorm: bn_sync_fold_fwd / bn_sync_fold_bwd (this rank's exchange rows) and bn_sync_merge_fwd
//    (the ranks' rows merged) around the all-gather.
// Twins of a kernel carry the same body with a compile-time flag and are named by suffix, in this order:
// `_add` stages gr_add and sums it into gr, `_sync` is the global phase of the synchronised backward (k1, k2 from the
// gathered rows), `_wide` sizes the per-(c, v) shared tables for V = 33 .. BN_MAXV.  Every V <= 32 kernel is the
// kernel of a 32-joint build.
//
// Statistics use shifted sums (shift = y[0,c,0,v]) accumulated in fp32 per thread and combined in fp64, so the
// E[x^2]-E[x]^2 cancellation does not bite on millimetre-scale poses.
#include <initializer_list>
#include <type_traits>

#include "kernels.cuh"
#include "umma.cuh"

namespace dstd {

constexpr int BN_THREADS_MAX = 512;
constexpr int BN_MAXJ = 8;       // positions per thread  -> T*V <= 4096
// Joints.  The per-(c, v) shared tables of the kernels are sized for one warp of joints (V <= 32); the `_wide_`
// instantiations size them for BN_MAXV and run V = 33 .. BN_MAXV, so the V <= 32 kernels are those of a 32-joint
// build.  Every block of the generic kernels has at least min(T*V, 257) threads and the fast plan gives the wide
// kernels at least V, so "one thread per v" loops need no stride.
constexpr int BN_MAXV = 128;
__host__ __device__ constexpr int bn_table_v(bool wide) { return wide ? BN_MAXV : 32; }
// samples per pipeline stage: the largest of 4/2/1 not above `cap` whose `planes_per_u` staged planes fit `budget`
static int bn_pick_u(size_t plane_bytes, int planes_per_u, int cap, size_t budget) {
  int u = 4;
  while (u > 1 && (u > cap || (size_t)u * planes_per_u * plane_bytes > budget)) u >>= 1;
  return u;
}
static const size_t BN_SMEM_BUDGET = 111 * 1024;   // two CTAs per SM (9 planes of 4 samples at H3.6M = 110.9 KB)

// per_cta: Switches::bn_samples_per_cta.  The default 32 is measured best on B200: 16 was best with one stream, with the
// two-stream step 32-64 is (+2 %)
static int bn_act_splits(int N, int per_cta) {
  int s = (N + per_cta - 1) / per_cta;
  if (s > 128) s = 128;
  if (s < 1) s = 1;
  return s;
}

struct BnGeom {
  int threads, nj;
};
static BnGeom bn_geom(int T, int V) {
  int tv = T * V;
  BnGeom g;
  int nj = cdiv(tv, BN_THREADS_MAX);
  g.nj = nj <= 1 ? 1 : nj <= 2 ? 2 : nj <= 4 ? 4 : 8;
  g.threads = cdiv(cdiv(tv, g.nj), 32) * 32;
  return g;
}

// position j (0..TV) in the memory order of view `v` -> logical (t, v)
__host__ __device__ __forceinline__ bool t_fastest(const View4& vw) { return !(vw.sk == 1 || vw.sp != 1); }
__device__ __forceinline__ void decode_pos(const View4& vw, int j, int T, int V, int& t, int& v) {
  if (!t_fastest(vw)) {   // V fastest (or generic): j = t*V + v
    t = j / V;
    v = j - t * V;
  } else {                // T fastest: j = v*T + t
    v = j / T;
    t = j - v * T;
  }
}
__device__ __forceinline__ bool same_order(const View4& a, const View4& b) { return t_fastest(a) == t_fastest(b); }
__device__ __forceinline__ int bn_pidx(int c, int v, int C, int V, int vc_order) { return vc_order ? v * C + c : c * V + v; }
__device__ __forceinline__ long long pos_off(const View4& vw, int t, int v) {
  return (long long)t * vw.sp + (long long)v * vw.sk;
}

struct BnFwdP {
  int N, C, T, V, vc_order, training, S;
  float eps, momentum;
  View4 y, r, out;
  const float *gamma, *beta;
  float *running_mean, *running_var;
  long long* nbt;
  const float* prelu;
  const float* mask;
  float *save_mean, *save_invstd;
  float* part;   // [S][C][V][2]
};

// Per-thread position table, built once per CTA: the integer divisions of decode_pos and the 64-bit stride products
// stay out of the per-sample loop (they were most of the instruction stream: 112 warp instructions per 32 elements
// in bn_apply before, profiles/r01_ncu_full_bn_before.md).  Positions are enumerated in the memory order of `order`
// (so that a warp's accesses to it are one contiguous sweep) and addressed in `addr`.
template <int NJ>
struct PosTab {
  const float* base;    // addr.p + n0*sn + c*sc (uniform over the CTA)
  int off[NJ];          // in-plane element offset of this thread's i-th position in `addr` (a plane spans < 2^31)
  int idx[NJ];          // logical slot t*V+v, -1 = no position
  int v[NJ];
};
template <int NJ>
__device__ __forceinline__ void tab_init(PosTab<NJ>& tb, const View4& order, const View4& addr, int c, int n0, int T,
                                         int V, int TV) {
  tb.base = addr.p + (long long)n0 * addr.sn + (long long)c * addr.sc;
#pragma unroll
  for (int i = 0; i < NJ; ++i) {
    const int j = threadIdx.x + i * blockDim.x;
    tb.idx[i] = -1;
    tb.v[i] = 0;
    tb.off[i] = 0;
    if (j < TV) {
      int t, v;
      decode_pos(order, j, T, V, t, v);
      tb.idx[i] = t * V + v;
      tb.v[i] = v;
      tb.off[i] = (int)pos_off(addr, t, v);
    }
  }
}
// ---- the three streaming kernels (apply, backward reduce, backward apply).
// Inputs are staged into shared memory as LINEAR copies of each tensor's [T x V] plane in that tensor's own memory
// order (8-byte cp.async when the plane is dense and 8-byte aligned: one instruction per two elements), double
// buffered; the consumer, which walks positions in the OUTPUT's memory order, picks its element at the slot the
// tensor's order implies (v*T+t or t*V+v), so a layout switch costs a strided shared-memory read and nothing else.
// A thread keeps per owned position only the packed logical (t, v) under the two enumeration orders; addresses and
// slots are re-derived with a few integer ops per U samples.  (Per-tensor offset tables in registers pushed these
// kernels past 100 registers, and capped at 64 the compiler rematerialised whole address chains per element:
// profiles/r01_ncu_full_bn_before.md.)
template <int NJ>
struct Pos2 {
  int tf[NJ], vf[NJ];   // (t << 8) | v of position j = tid + i*blockDim in the T-fastest / V-fastest enumeration; -1 none
};
template <int NJ>
__device__ __forceinline__ void pos_init(Pos2<NJ>& ps, int T, int V, int TV) {
#pragma unroll
  for (int i = 0; i < NJ; ++i) {
    const int j = threadIdx.x + i * blockDim.x;
    ps.tf[i] = ps.vf[i] = -1;
    if (j < TV) {
      int a = j / T;                 // T fastest: j = v*T + t
      ps.tf[i] = ((j - a * T) << 8) | a;
      a = j / V;                     // V fastest: j = t*V + v
      ps.vf[i] = (a << 8) | (j - a * V);
    }
  }
}
__device__ __forceinline__ void cp_async4_s(unsigned sdst, const float* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(sdst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async8_s(unsigned sdst, const float* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sdst), "l"(gsrc) : "memory");
}
// the [T x V] planes of `w` are dense in w's memory order
__host__ __device__ __forceinline__ bool plane_dense(const View4& w, int T, int V) {
  return t_fastest(w) ? (w.sp == 1 && w.sk == T) : (w.sk == 1 && w.sp == V);
}
// how a [T x V] plane of `w` can be copied: 2 = dense and every plane 8-byte aligned, 1 = dense, 0 = generic strides
__device__ __forceinline__ int plane_mode(const View4& w, int T, int V) {
  if (!plane_dense(w, T, V)) return 0;
  const bool al8 = ((reinterpret_cast<unsigned long long>(w.p) & 7ull) == 0) && !((w.sn | w.sc) & 1ll) && !((T * V) & 1);
  return al8 ? 2 : 1;
}
// slot of logical (t, v) in a plane staged in w's memory order
__device__ __forceinline__ int slot_of(bool tfast, int t, int v, int T, int V) { return tfast ? v * T + t : t * V + v; }

// cp.async samples n .. n+U-1 (`left` of them exist) of channel plane c of `w` into the [U][T*V] region at shared
// address `sdst`, each plane in w's own memory order.
// The forward passes `mode` = plane_mode(w, T, V), hoisted out of its sample loop, and, since the launch geometry
// gives NJ * blockDim >= T*V, leaves the pair loop after one pair for NJ <= 2.  BWD: the backward kernels' form, which
// derives `mode` here at every call (the argument is ignored) and has no single-pair break: they sit at the
// 64-register cap and measured slower with the hoisted mode / single-pair form.
template <int NJ, int U, bool FULL, bool BWD>
__device__ __forceinline__ void stage_async(const Pos2<NJ>& ps, const View4& w, int mode, int c, int n, int left,
                                            unsigned sdst, int T, int V) {
  const int TV = T * V;
  if (BWD) mode = plane_mode(w, T, V);
  const float* base = w.p + (long long)n * w.sn + (long long)c * w.sc;
  if (mode == 2) {
    for (int j = 2 * threadIdx.x; j < TV; j += 2 * blockDim.x) {
      const float* p = base + j;
      unsigned d = sdst + (unsigned)j * 4u;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (FULL || u < left) cp_async8_s(d, p);
        p += w.sn;
        d += (unsigned)TV * 4u;
      }
      if (!BWD && NJ <= 2) break;
    }
  } else {
    const bool tfast = t_fastest(w);
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
      const int pk = tfast ? ps.tf[i] : ps.vf[i];
      if (pk >= 0) {
        const int j = threadIdx.x + i * blockDim.x;
        const float* p = base + (mode ? (long long)j : (long long)(pk >> 8) * w.sp + (long long)(pk & 255) * w.sk);
        unsigned d = sdst + (unsigned)j * 4u;
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (FULL || u < left) cp_async4_s(d, p);
          p += w.sn;
          d += (unsigned)TV * 4u;
        }
      }
    }
  }
}

// Split s's partial pair of channel c for every v: the per-position sums in sh[0 .. T*V) and sh[T*V .. 2*T*V)
// (logical slots t*V+v) summed over t in order, in fp64, into part[s][c][v][0..1]
__device__ __forceinline__ void bn_store_partials(const float* sh, float* part, int s, int C, int c, int T, int V) {
  if (threadIdx.x < V) {
    const int v = threadIdx.x, TV = T * V;
    double s1 = 0., s2 = 0.;
    for (int t = 0; t < T; ++t) {
      s1 += sh[t * V + v];
      s2 += sh[TV + t * V + v];
    }
    float* dst = part + (((long long)s * C + c) * V + v) * 2;
    dst[0] = (float)s1;
    dst[1] = (float)s2;
  }
}

// ------------------------------------------------------------------------------------------ forward: statistics
template <int NJ>
__device__ __forceinline__ void bn_stats_body(const BnFwdP& q) {
  extern __shared__ float sh[];   // [2][T*V]
  constexpr int SU = 8;
  const int c = blockIdx.x, s = blockIdx.y, T = q.T, V = q.V, TV = T * V;
  const int n0 = (int)((long long)q.N * s / q.S), n1 = (int)((long long)q.N * (s + 1) / q.S), cnt = n1 - n0;
  const long long sn = q.y.sn;
  if (plane_mode(q.y, T, V) == 2) {
    // dense, 8-byte aligned planes: two adjacent positions per thread, LDG.64, SU samples in flight
    const bool tfast = t_fastest(q.y);
    const float* base = q.y.p + (long long)n0 * sn + (long long)c * q.y.sc;
    for (int j = 2 * threadIdx.x; j < TV; j += 2 * blockDim.x) {
      int t0, v0, t1, v1;
      decode_pos(q.y, j, T, V, t0, v0);
      decode_pos(q.y, j + 1, T, V, t1, v1);
      const float* sp0 = q.y.p + (long long)c * q.y.sc;   // shift = y[0, c, 0, v]
      const float sh0 = __ldg(sp0 + (tfast ? (long long)v0 * T : (long long)v0));
      const float sh1 = __ldg(sp0 + (tfast ? (long long)v1 * T : (long long)v1));
      float a1x = 0.f, a2x = 0.f, a1y = 0.f, a2y = 0.f;
      const float* p = base + j;
      for (int nn = 0; nn < cnt; nn += SU) {
        const int left = cnt - nn;
        float2 d[SU];
#pragma unroll
        for (int u = 0; u < SU; ++u) {
          d[u] = (u < left) ? __ldg(reinterpret_cast<const float2*>(p)) : make_float2(sh0, sh1);
          p += sn;
        }
#pragma unroll
        for (int u = 0; u < SU; ++u) {
          const float dx = d[u].x - sh0, dy = d[u].y - sh1;
          a1x += dx;
          a2x = fmaf(dx, dx, a2x);
          a1y += dy;
          a2y = fmaf(dy, dy, a2y);
        }
      }
      sh[t0 * V + v0] = a1x;
      sh[TV + t0 * V + v0] = a2x;
      sh[t1 * V + v1] = a1y;
      sh[TV + t1 * V + v1] = a2y;
    }
  } else {
    PosTab<NJ> ty;
    tab_init<NJ>(ty, q.y, q.y, c, n0, T, V, TV);
    float a1[NJ], a2[NJ], shift[NJ];
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
      a1[i] = a2[i] = 0.f;
      shift[i] = ty.idx[i] >= 0 ? __ldg(q.y.p + (long long)c * q.y.sc + (long long)ty.v[i] * q.y.sk) : 0.f;
    }
    for (int nn = 0; nn < cnt; nn += SU) {
      const int left = cnt - nn;
      float d[NJ][SU];
#pragma unroll
      for (int i = 0; i < NJ; ++i) {
        const float* p = ty.base + (long long)nn * sn + ty.off[i];
#pragma unroll
        for (int u = 0; u < SU; ++u, p += sn) d[i][u] = (ty.idx[i] >= 0 && u < left) ? __ldg(p) - shift[i] : 0.f;
      }
#pragma unroll
      for (int i = 0; i < NJ; ++i) {
#pragma unroll
        for (int u = 0; u < SU; ++u) {
          a1[i] += d[i][u];
          a2[i] = fmaf(d[i][u], d[i][u], a2[i]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < NJ; ++i)
      if (ty.idx[i] >= 0) {
        sh[ty.idx[i]] = a1[i];
        sh[TV + ty.idx[i]] = a2[i];
      }
  }
  __syncthreads();
  bn_store_partials(sh, q.part, s, q.C, c, T, V);
}

template <int NJ>
__global__ void __launch_bounds__(BN_THREADS_MAX) bn_stats_kernel(BnFwdP q) {
  bn_stats_body<NJ>(q);
}
// planes of 4097 .. 8192 positions, whose apply and backward passes run the BIG fast kernels (V > 32 only)
__global__ void __launch_bounds__(2 * BN_THREADS_MAX) bn_stats_big_kernel(BnFwdP q) {
  bn_stats_body<BN_MAXJ>(q);
}

// Sum the per-split partial pairs of channel c for every v, in a fixed order (so that every CTA of the channel gets
// bit-identical totals): 8 lanes per v, strided over the splits, combined with a butterfly.  Called by all threads;
// the totals land in tot[v][0..1].  This replaces a separate "finalize" launch between the reduction and the apply
// pass (9 us each, 76 of them per training step).
__device__ __forceinline__ void sum_partials(const float* part, int S, int C, int c, int V, double (*tot)[2]) {
  const int lim = (V * 8 + 31) & ~31;
  for (int idx = threadIdx.x; idx < lim; idx += blockDim.x) {
    const int v = idx >> 3, k = idx & 7;
    double s1 = 0., s2 = 0.;
    if (v < V)
      for (int ss = k; ss < S; ss += 8) {
        const float* p = part + (((long long)ss * C + c) * V + v) * 2;
        s1 += p[0];
        s2 += p[1];
      }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if (k == 0 && v < V) {
      tot[v][0] = s1;
      tot[v][1] = s2;
    }
  }
}

__global__ void bn_eval_stats_kernel(BnFwdP q) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= q.C * q.V) return;
  q.save_mean[idx] = q.running_mean[idx];
  q.save_invstd[idx] = rsqrtf(q.running_var[idx] + q.eps);
}

// ------------------------------------------------------------------------------------------ forward: apply
// Positions are walked in the memory order of `out`.  Consumer state hoisted out of the sample loop: per position the
// running output pointer and the shared-memory slots of y and r.
template <int NJ, int U, bool FULL, bool MASK>
__device__ __forceinline__ void bn_apply_consume(const BnFwdP& q, const float* stage, float* (&op)[NJ],
                                                 const int (&sy)[NJ], const int (&sr)[NJ], const int (&me)[NJ], int c,
                                                 int n, int left, const float (&sm)[NJ], const float (&sc)[NJ],
                                                 const float (&sf)[NJ], float slope, bool has_r) {
  const int TV = q.T * q.V;
  const long long osn = q.out.sn;
#pragma unroll
  for (int i = 0; i < NJ; ++i) {
    if (sy[i] >= 0) {
      const float* py = stage + sy[i];
      const float* pr = stage + U * TV + sr[i];
      float* o = op[i];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (FULL || u < left) {
          float pre = fmaf(*py - sm[i], sc[i], sf[i]);
          if (has_r) pre += *pr;
          float a = pre > 0.f ? pre : slope * pre;
          if (MASK) a *= __ldg(q.mask + ((long long)(n + u) * q.C + c) * TV + me[i]);
          *o = a;
        }
        o += osn;
        py += TV;
        pr += TV;
      }
      op[i] = o;
    }
  }
}

template <int NJ, int U, bool WIDE>
__device__ __forceinline__ void bn_apply_body(const BnFwdP& q) {
  extern __shared__ float sh[];   // [2 stages][nst = 1 (y) or 2 (y, r)][U][T*V]
  constexpr int VW = bn_table_v(WIDE);
  const int c = blockIdx.x, s = blockIdx.y, T = q.T, V = q.V, TV = T * V;
  const int n0 = (int)((long long)q.N * s / q.S), n1 = (int)((long long)q.N * (s + 1) / q.S), cnt = n1 - n0;
  const bool has_r = q.r.p != nullptr;
  const float slope = q.prelu ? __ldg(q.prelu) : 1.f;
  const int stage_f = (has_r ? 2 : 1) * U * TV, iters = (cnt + U - 1) / U;
  const unsigned sbase = (unsigned)__cvta_generic_to_shared(sh);
  Pos2<NJ> ps;
  pos_init<NJ>(ps, T, V, TV);
  const int mode_y = plane_mode(q.y, T, V), mode_r = has_r ? plane_mode(q.r, T, V) : 0;
  auto issue = [&](int it) {
    const unsigned d = sbase + (unsigned)((it & 1) * stage_f) * 4u;
    const int n = n0 + it * U, left = n1 - n;
    if (left >= U) {
      stage_async<NJ, U, true, false>(ps, q.y, mode_y, c, n, left, d, T, V);
      if (has_r) stage_async<NJ, U, true, false>(ps, q.r, mode_r, c, n, left, d + (unsigned)(U * TV) * 4u, T, V);
    } else {
      stage_async<NJ, U, false, false>(ps, q.y, mode_y, c, n, left, d, T, V);
      if (has_r) stage_async<NJ, U, false, false>(ps, q.r, mode_r, c, n, left, d + (unsigned)(U * TV) * 4u, T, V);
    }
  };
  if (iters > 0) issue(0);
  cp_async_commit();
  __shared__ double tot[VW][2];
  __shared__ float st_mean[VW], st_is[VW];
  if (q.training) {   // batch statistics from the split partials; the s == 0 CTA of the channel publishes them
    sum_partials(q.part, q.S, q.C, c, V, tot);
    __syncthreads();
    if (threadIdx.x < V) {
      const int v = threadIdx.x;
      const double cntd = (double)q.N * q.T;
      const double shift = __ldg(q.y.p + vix(q.y, 0, c, 0, v));
      const double dm = tot[v][0] / cntd;
      double var = tot[v][1] / cntd - dm * dm;
      if (var < 0.) var = 0.;
      const double mean = shift + dm;
      const float fm = (float)mean, fi = (float)(1.0 / sqrt(var + (double)q.eps));
      st_mean[v] = fm;
      st_is[v] = fi;
      if (s == 0) {
        const int pi = bn_pidx(c, v, q.C, V, q.vc_order);
        q.save_mean[pi] = fm;
        q.save_invstd[pi] = fi;
        if (q.running_mean) {
          const double unb = cntd > 1. ? var * cntd / (cntd - 1.) : var;
          q.running_mean[pi] = (float)((1.0 - q.momentum) * q.running_mean[pi] + q.momentum * mean);
          q.running_var[pi] = (float)((1.0 - q.momentum) * q.running_var[pi] + q.momentum * unb);
        }
        if (c == 0 && v == 0 && q.nbt) *q.nbt += 1;
      }
    }
    __syncthreads();
  }
  float sc[NJ], sf[NJ], sm[NJ];   // out = (y - mean) * (gamma * invstd) + beta  (centred first: no cancellation)
  float* op[NJ];
  int sy[NJ], sr[NJ], me[NJ];
  {
    const bool tfast = t_fastest(q.out), tf_y = t_fastest(q.y), tf_r = has_r && t_fastest(q.r);
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
      sc[i] = sf[i] = sm[i] = 0.f;
      op[i] = nullptr;
      sy[i] = -1;
      sr[i] = me[i] = 0;
      const int pk = tfast ? ps.tf[i] : ps.vf[i];
      if (pk >= 0) {
        const int t = pk >> 8, v = pk & 255;
        const int pi = bn_pidx(c, v, q.C, V, q.vc_order);
        const float g = __ldg(q.gamma + pi), is = q.training ? st_is[v] : q.save_invstd[pi];
        sm[i] = q.training ? st_mean[v] : q.save_mean[pi];
        sc[i] = g * is;
        sf[i] = __ldg(q.beta + pi);
        op[i] = q.out.p + vix(q.out, n0, c, t, v);
        sy[i] = slot_of(tf_y, t, v, T, V);
        sr[i] = slot_of(tf_r, t, v, T, V);
        me[i] = t * V + v;
      }
    }
  }
  for (int it = 0; it < iters; ++it) {
    if (it + 1 < iters) issue(it + 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const int n = n0 + it * U, left = n1 - n;
    const float* stage = sh + (it & 1) * stage_f;
    if (q.mask) bn_apply_consume<NJ, U, false, true>(q, stage, op, sy, sr, me, c, n, left, sm, sc, sf, slope, has_r);
    else if (left >= U) bn_apply_consume<NJ, U, true, false>(q, stage, op, sy, sr, me, c, n, left, sm, sc, sf, slope, has_r);
    else bn_apply_consume<NJ, U, false, false>(q, stage, op, sy, sr, me, c, n, left, sm, sc, sf, slope, has_r);
    __syncthreads();   // the buffer is refilled by the prefetch of the next iteration
  }
}

template <int NJ, int U>
__global__ void __launch_bounds__(BN_THREADS_MAX, 2) bn_apply_kernel(BnFwdP q) {
  bn_apply_body<NJ, U, false>(q);
}
template <int NJ, int U>
__global__ void __launch_bounds__(BN_THREADS_MAX, 2) bn_apply_wide_kernel(BnFwdP q) {
  bn_apply_body<NJ, U, true>(q);
}

// ------------------------------------------------------------------------------------------ backward
struct BnBwdP {
  int N, C, T, V, vc_order, training, S;
  View4 y, r, gout, gy, gr, gadd;
  const float *gamma, *beta, *prelu, *mask, *save_mean, *save_invstd;
  float *ggamma, *gbeta, *gprelu;
  float* part;    // [S][C][V][2]
  float* part_p;  // [S][C]
};

// gprelu = the np slope partials of pass 1 summed in a fixed order; called by all threads of one CTA
__device__ __forceinline__ void bn_sum_slope_partials(const BnBwdP& q, int np, float* red) {
  float a = 0.f;
  for (int i = threadIdx.x; i < np; i += blockDim.x) a += q.part_p[i];
  const float t = block_sum(a, red);
  if (threadIdx.x == 0) q.gprelu[0] = t;
}

// d(pre-activation) at one element; also returns xhat and the PReLU-slope contribution
__device__ __forceinline__ float bn_gpre(bool has_prelu, float yv, float rv, float gv, float mv, float mu, float is,
                                         float g, float b, float slope, float& xhat, float& gslope) {
  xhat = (yv - mu) * is;
  gv *= mv;
  gslope = 0.f;
  if (has_prelu) {
    const float pre = fmaf(xhat, g, b) + rv;
    if (pre <= 0.f) {
      gslope = gv * pre;
      gv *= slope;
    }
  }
  return gv;
}

// pass 1: per-(c,v) sums of gpre and gpre*xhat, PReLU slope gradient.  Positions in gout's memory order; gout, y
// and r come through shared memory (cp.async, double-buffered) like in the forward.
template <int NJ, int U, bool FULL, bool MASK>
__device__ __forceinline__ void bn_bwd_reduce_consume(const BnBwdP& q, const float* stage, const int (&sg)[NJ],
                                                      const int (&sy)[NJ], const int (&sr)[NJ], const int (&me)[NJ],
                                                      int c, int n, int left, const float (&mu)[NJ],
                                                      const float (&is)[NJ], const float (&g)[NJ],
                                                      const float (&b)[NJ], float slope, bool has_prelu, bool use_r,
                                                      float (&a1)[NJ], float (&a2)[NJ], float& gsl) {
  const int TV = q.T * q.V;
#pragma unroll
  for (int i = 0; i < NJ; ++i) {
    if (sg[i] >= 0) {
      const float* pg = stage + sg[i];
      const float* py = stage + U * TV + sy[i];
      const float* pr = stage + 2 * U * TV + sr[i];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (FULL || u < left) {
          const float rv = use_r ? *pr : 0.f;
          const float mv = MASK ? __ldg(q.mask + ((long long)(n + u) * q.C + c) * TV + me[i]) : 1.f;
          float xhat, gs;
          const float gp = bn_gpre(has_prelu, *py, rv, *pg, mv, mu[i], is[i], g[i], b[i], slope, xhat, gs);
          a1[i] += gp;
          a2[i] = fmaf(gp, xhat, a2[i]);
          gsl += gs;
        }
        pg += TV;
        py += TV;
        pr += TV;
      }
    }
  }
}

template <int NJ, int U>
__global__ void __launch_bounds__(BN_THREADS_MAX, 2) bn_bwd_reduce_kernel(BnBwdP q) {
  extern __shared__ float sh[];   // [2 stages][nst = 2 (gout, y) or 3 (+ r)][U][T*V]
  __shared__ float red[32];
  const int c = blockIdx.x, s = blockIdx.y, T = q.T, V = q.V, TV = T * V;
  const int n0 = (int)((long long)q.N * s / q.S), n1 = (int)((long long)q.N * (s + 1) / q.S), cnt = n1 - n0;
  const bool has_prelu = q.prelu != nullptr;
  const bool use_r = q.r.p && has_prelu;
  const float slope = has_prelu ? __ldg(q.prelu) : 1.f;
  const int stage_f = (use_r ? 3 : 2) * U * TV, iters = (cnt + U - 1) / U;
  const unsigned sbase = (unsigned)__cvta_generic_to_shared(sh);
  Pos2<NJ> ps;
  pos_init<NJ>(ps, T, V, TV);
  auto issue = [&](int it) {
    const unsigned d = sbase + (unsigned)((it & 1) * stage_f) * 4u, du = (unsigned)(U * TV) * 4u;
    const int n = n0 + it * U, left = n1 - n;
    if (left >= U) {
      stage_async<NJ, U, true, true>(ps, q.gout, 0, c, n, left, d, T, V);
      stage_async<NJ, U, true, true>(ps, q.y, 0, c, n, left, d + du, T, V);
      if (use_r) stage_async<NJ, U, true, true>(ps, q.r, 0, c, n, left, d + 2 * du, T, V);
    } else {
      stage_async<NJ, U, false, true>(ps, q.gout, 0, c, n, left, d, T, V);
      stage_async<NJ, U, false, true>(ps, q.y, 0, c, n, left, d + du, T, V);
      if (use_r) stage_async<NJ, U, false, true>(ps, q.r, 0, c, n, left, d + 2 * du, T, V);
    }
  };
  if (iters > 0) issue(0);
  cp_async_commit();
  float mu[NJ], is[NJ], g[NJ], b[NJ], a1[NJ], a2[NJ];
  int sg[NJ], sy[NJ], sr[NJ], me[NJ];
  float gsl = 0.f;
  {
    const bool tfast = t_fastest(q.gout), tf_y = t_fastest(q.y), tf_r = use_r && t_fastest(q.r);
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
      mu[i] = is[i] = g[i] = b[i] = a1[i] = a2[i] = 0.f;
      sg[i] = -1;
      sy[i] = sr[i] = me[i] = 0;
      const int pk = tfast ? ps.tf[i] : ps.vf[i];
      if (pk >= 0) {
        const int t = pk >> 8, v = pk & 255;
        const int pi = bn_pidx(c, v, q.C, V, q.vc_order);
        mu[i] = __ldg(q.save_mean + pi);
        is[i] = __ldg(q.save_invstd + pi);
        g[i] = __ldg(q.gamma + pi);
        b[i] = __ldg(q.beta + pi);
        sg[i] = slot_of(tfast, t, v, T, V);
        sy[i] = slot_of(tf_y, t, v, T, V);
        sr[i] = slot_of(tf_r, t, v, T, V);
        me[i] = t * V + v;
      }
    }
  }
  for (int it = 0; it < iters; ++it) {
    if (it + 1 < iters) issue(it + 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const int n = n0 + it * U, left = n1 - n;
    const float* stage = sh + (it & 1) * stage_f;
    if (q.mask)
      bn_bwd_reduce_consume<NJ, U, false, true>(q, stage, sg, sy, sr, me, c, n, left, mu, is, g, b, slope, has_prelu,
                                                use_r, a1, a2, gsl);
    else if (left >= U)
      bn_bwd_reduce_consume<NJ, U, true, false>(q, stage, sg, sy, sr, me, c, n, left, mu, is, g, b, slope, has_prelu,
                                                use_r, a1, a2, gsl);
    else
      bn_bwd_reduce_consume<NJ, U, false, false>(q, stage, sg, sy, sr, me, c, n, left, mu, is, g, b, slope, has_prelu,
                                                 use_r, a1, a2, gsl);
    __syncthreads();
  }
  cp_async_wait<0>();
  __syncthreads();
#pragma unroll
  for (int i = 0; i < NJ; ++i) {
    if (sg[i] >= 0) {
      sh[me[i]] = a1[i];
      sh[TV + me[i]] = a2[i];
    }
  }
  __syncthreads();
  bn_store_partials(sh, q.part, s, q.C, c, T, V);
  float tot = block_sum(gsl, red);
  if (threadIdx.x == 0) q.part_p[(long long)s * q.C + c] = tot;
}

// pass 2: gy (and gr).  Positions in gy's memory order; y, gout and r come through shared memory (cp.async,
// double-buffered), gr leaves through it.
template <int NJ, int U, bool FULL, bool MASK, bool ADD>
__device__ __forceinline__ void bn_bwd_apply_consume(const BnBwdP& q, const float* stage, float* sho, float* (&gyp)[NJ],
                                                     const int (&sg)[NJ], const int (&sy)[NJ], const int (&sr)[NJ],
                                                     const int (&so)[NJ], const int (&sa)[NJ], int add_region,
                                                     const int (&me)[NJ], int c, int n, int left,
                                                     const float (&mu)[NJ], const float (&is)[NJ],
                                                     const float (&g)[NJ], const float (&b)[NJ],
                                                     const float (&gi)[NJ], const float (&k1)[NJ],
                                                     const float (&k2)[NJ], float slope, bool has_prelu, bool use_r,
                                                     bool has_gr) {
  const int TV = q.T * q.V;
  const long long gysn = q.gy.sn;
#pragma unroll
  for (int i = 0; i < NJ; ++i) {
    if (sg[i] >= 0) {
      const float* pg = stage + sg[i];
      const float* py = stage + U * TV + sy[i];
      const float* pr = stage + 2 * U * TV + sr[i];
      const float* pa = ADD ? stage + add_region * U * TV + sa[i] : stage;
      float* po = sho + so[i];
      float* o = gyp[i];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (FULL || u < left) {
          const float rv = use_r ? *pr : 0.f;
          const float mv = MASK ? __ldg(q.mask + ((long long)(n + u) * q.C + c) * TV + me[i]) : 1.f;
          float xhat, gs;
          const float gp = bn_gpre(has_prelu, *py, rv, *pg, mv, mu[i], is[i], g[i], b[i], slope, xhat, gs);
          *o = gi[i] * (gp - k1[i] - xhat * k2[i]);
          if (has_gr) *po = ADD ? gp + *pa : gp;
        }
        o += gysn;
        pg += TV;
        py += TV;
        pr += TV;
        if (ADD) pa += TV;
        po += TV;
      }
      gyp[i] = o;
    }
  }
}

// Synchronised BatchNorm (dstd_bn_act_backward_global): k1 = sum(g') / n and k2 = sum(g' xhat) / n over the global
// batch, from the gathered exchange rows (count, sum g', sum g' xhat) of the `world` ranks, summed in rank order in
// fp64.  tot[v] of channel c receives (k1, k2).
__device__ __forceinline__ void sync_bwd_totals(const double* all, int world, int C, int V, int c, int vc_order,
                                                double (*tot)[2]) {
  const long long cv = (long long)C * V;
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    const int pi = bn_pidx(c, v, C, V, vc_order);
    double n = 0., s1 = 0., s2 = 0.;
    for (int r = 0; r < world; ++r) {
      const double* row = all + 3 * cv * r + pi;
      n += row[0];
      s1 += row[cv];
      s2 += row[2 * cv];
    }
    tot[v][0] = s1 / n;
    tot[v][1] = s2 / n;
  }
}

// SYNC: the global phase of the synchronised backward.  k1 / k2 come from the gathered rows (`all`, `world`) instead
// of the split partials, and the parameter gradients are not written (the local phase wrote this rank's share).
template <int NJ, int U, bool ADD, bool SYNC, bool WIDE>
__device__ __forceinline__ void bn_bwd_apply_body(const BnBwdP& q, const double* all, int world) {
  extern __shared__ float sh[];   // [2 stages][nst = 2 (gout, y), + r, + gr_add][U][T*V], then [U][T*V] for gr
  constexpr int VW = bn_table_v(WIDE);
  const int c = blockIdx.x, s = blockIdx.y, T = q.T, V = q.V, TV = T * V;
  const int n0 = (int)((long long)q.N * s / q.S), n1 = (int)((long long)q.N * (s + 1) / q.S), cnt = n1 - n0;
  const bool has_prelu = q.prelu != nullptr;
  const bool use_r = q.r.p && has_prelu;
  const bool has_gr = q.gr.p != nullptr;
  const float slope = has_prelu ? __ldg(q.prelu) : 1.f;
  const float icnt = 1.0f / ((float)q.N * (float)T);
  const bool has_add = ADD;       // the host launches the ADD instantiation only with gr and gr_add present
  const int add_region = has_add ? (use_r ? 3 : 2) : 0;           // staged planes: gout, y, (r), (gr_add); 0: unused
  const int stage_f = ((use_r ? 3 : 2) + (has_add ? 1 : 0)) * U * TV, iters = (cnt + U - 1) / U;
  const unsigned sbase = (unsigned)__cvta_generic_to_shared(sh);
  float* sho = sh + 2 * stage_f;                       // gr hand-over, each plane in gr's memory order
  const int gr_mode = has_gr ? plane_mode(q.gr, T, V) : 0;
  const bool tfast_gr = has_gr && t_fastest(q.gr);
  Pos2<NJ> ps;
  pos_init<NJ>(ps, T, V, TV);
  auto issue = [&](int it) {
    const unsigned d = sbase + (unsigned)((it & 1) * stage_f) * 4u, du = (unsigned)(U * TV) * 4u;
    const int n = n0 + it * U, left = n1 - n;
    if (left >= U) {
      stage_async<NJ, U, true, true>(ps, q.gout, 0, c, n, left, d, T, V);
      stage_async<NJ, U, true, true>(ps, q.y, 0, c, n, left, d + du, T, V);
      if (use_r) stage_async<NJ, U, true, true>(ps, q.r, 0, c, n, left, d + 2 * du, T, V);
      if (has_add) stage_async<NJ, U, true, true>(ps, q.gadd, 0, c, n, left, d + add_region * du, T, V);
    } else {
      stage_async<NJ, U, false, true>(ps, q.gout, 0, c, n, left, d, T, V);
      stage_async<NJ, U, false, true>(ps, q.y, 0, c, n, left, d + du, T, V);
      if (use_r) stage_async<NJ, U, false, true>(ps, q.r, 0, c, n, left, d + 2 * du, T, V);
      if (has_add) stage_async<NJ, U, false, true>(ps, q.gadd, 0, c, n, left, d + add_region * du, T, V);
    }
  };
  if (iters > 0) issue(0);
  cp_async_commit();
  // sums of pass 1 over the splits; the s == 0 CTA of the channel publishes the parameter gradients
  __shared__ double tot[VW][2];
  __shared__ float red[32];
  if (SYNC) {
    sync_bwd_totals(all, world, q.C, V, c, q.vc_order, tot);
    __syncthreads();
  } else {
    sum_partials(q.part, q.S, q.C, c, V, tot);
    if (c == 0 && s == 0 && q.gprelu) bn_sum_slope_partials(q, q.S * q.C, red);
    __syncthreads();
    if (s == 0 && threadIdx.x < V) {
      const int pi = bn_pidx(c, threadIdx.x, q.C, V, q.vc_order);
      q.gbeta[pi] = (float)tot[threadIdx.x][0];
      q.ggamma[pi] = (float)tot[threadIdx.x][1];
    }
  }
  // per position: xhat = (y - mu) * is;  gy = gi * (gp - k1 - xhat * k2)
  float mu[NJ], is[NJ], g[NJ], b[NJ], gi[NJ], k1[NJ], k2[NJ];
  float* gyp[NJ];
  int sg[NJ], sy[NJ], sr[NJ], so[NJ], sa[NJ], me[NJ];
  {
    const bool tfast = t_fastest(q.gy), tf_g = t_fastest(q.gout), tf_y = t_fastest(q.y), tf_r = use_r && t_fastest(q.r),
               tf_a = ADD && t_fastest(q.gadd);
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
      mu[i] = is[i] = g[i] = b[i] = gi[i] = k1[i] = k2[i] = 0.f;
      gyp[i] = nullptr;
      sg[i] = -1;
      sy[i] = sr[i] = so[i] = sa[i] = me[i] = 0;
      const int pk = tfast ? ps.tf[i] : ps.vf[i];
      if (pk >= 0) {
        const int t = pk >> 8, v = pk & 255;
        const int pi = bn_pidx(c, v, q.C, V, q.vc_order);
        mu[i] = __ldg(q.save_mean + pi);
        is[i] = __ldg(q.save_invstd + pi);
        g[i] = __ldg(q.gamma + pi);
        b[i] = __ldg(q.beta + pi);
        gi[i] = g[i] * is[i];
        if (SYNC) {
          k1[i] = (float)tot[v][0];
          k2[i] = (float)tot[v][1];
        } else if (q.training) {
          k1[i] = (float)tot[v][0] * icnt;
          k2[i] = (float)tot[v][1] * icnt;
        }
        gyp[i] = q.gy.p + vix(q.gy, n0, c, t, v);
        sg[i] = slot_of(tf_g, t, v, T, V);
        sy[i] = slot_of(tf_y, t, v, T, V);
        sr[i] = slot_of(tf_r, t, v, T, V);
        so[i] = slot_of(tfast_gr, t, v, T, V);
        if (ADD) sa[i] = slot_of(tf_a, t, v, T, V);
        me[i] = t * V + v;
      }
    }
  }
  for (int it = 0; it < iters; ++it) {
    if (it + 1 < iters) issue(it + 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const int n = n0 + it * U, left = n1 - n;
    const float* stage = sh + (it & 1) * stage_f;
    if (q.mask)
      bn_bwd_apply_consume<NJ, U, false, true, ADD>(q, stage, sho, gyp, sg, sy, sr, so, sa, add_region, me, c, n, left, mu, is, g, b, gi, k1,
                                               k2, slope, has_prelu, use_r, has_gr);
    else if (left >= U)
      bn_bwd_apply_consume<NJ, U, true, false, ADD>(q, stage, sho, gyp, sg, sy, sr, so, sa, add_region, me, c, n, left, mu, is, g, b, gi, k1,
                                               k2, slope, has_prelu, use_r, has_gr);
    else
      bn_bwd_apply_consume<NJ, U, false, false, ADD>(q, stage, sho, gyp, sg, sy, sr, so, sa, add_region, me, c, n, left, mu, is, g, b, gi,
                                                k1, k2, slope, has_prelu, use_r, has_gr);
    if (has_gr) {
      __syncthreads();
      float* grbase = q.gr.p + (long long)n * q.gr.sn + (long long)c * q.gr.sc;
      if (gr_mode == 2) {
        for (int j = 2 * threadIdx.x; j < TV; j += 2 * blockDim.x) {
          float* grp = grbase + j;
          const float* po = sho + j;
#pragma unroll
          for (int u = 0; u < U; ++u) {
            if (u < left) *reinterpret_cast<float2*>(grp) = *reinterpret_cast<const float2*>(po);
            grp += q.gr.sn;
            po += TV;
          }
        }
      } else {
#pragma unroll
        for (int i = 0; i < NJ; ++i) {
          const int pk = tfast_gr ? ps.tf[i] : ps.vf[i];
          if (pk >= 0) {
            const int j = threadIdx.x + i * blockDim.x;
            float* grp = grbase + (gr_mode ? (long long)j : (long long)(pk >> 8) * q.gr.sp + (long long)(pk & 255) * q.gr.sk);
            const float* po = sho + j;
#pragma unroll
            for (int u = 0; u < U; ++u) {
              if (u < left) *grp = *po;
              grp += q.gr.sn;
              po += TV;
            }
          }
        }
      }
    }
    __syncthreads();
  }
}

template <int NJ, int U>
__global__ void __launch_bounds__(BN_THREADS_MAX, 2) bn_bwd_apply_kernel(BnBwdP q) {
  bn_bwd_apply_body<NJ, U, false, false, false>(q, nullptr, 0);
}
// same with a fourth staged tensor, gr_add, summed into gr (separate instantiation: the plain kernel sits at the
// 64-register cap and pays ~13 % for the extra slots)
template <int NJ, int U>
__global__ void __launch_bounds__(BN_THREADS_MAX, 2) bn_bwd_apply_add_kernel(BnBwdP q) {
  bn_bwd_apply_body<NJ, U, true, false, false>(q, nullptr, 0);
}
// the global phase of the synchronised backward (k1, k2 from the gathered rows)
template <int NJ, int U>
__global__ void __launch_bounds__(BN_THREADS_MAX, 2) bn_bwd_apply_sync_kernel(BnBwdP q, const double* all, int world) {
  bn_bwd_apply_body<NJ, U, false, true, false>(q, all, world);
}
template <int NJ, int U>
__global__ void __launch_bounds__(BN_THREADS_MAX, 2) bn_bwd_apply_add_sync_kernel(BnBwdP q, const double* all, int world) {
  bn_bwd_apply_body<NJ, U, true, true, false>(q, all, world);
}
// V = 33 .. BN_MAXV
template <int NJ, int U>
__global__ void __launch_bounds__(BN_THREADS_MAX, 2) bn_bwd_apply_wide_kernel(BnBwdP q) {
  bn_bwd_apply_body<NJ, U, false, false, true>(q, nullptr, 0);
}
template <int NJ, int U>
__global__ void __launch_bounds__(BN_THREADS_MAX, 2) bn_bwd_apply_add_wide_kernel(BnBwdP q) {
  bn_bwd_apply_body<NJ, U, true, false, true>(q, nullptr, 0);
}
template <int NJ, int U>
__global__ void __launch_bounds__(BN_THREADS_MAX, 2) bn_bwd_apply_sync_wide_kernel(BnBwdP q, const double* all, int world) {
  bn_bwd_apply_body<NJ, U, false, true, true>(q, all, world);
}
template <int NJ, int U>
__global__ void __launch_bounds__(BN_THREADS_MAX, 2) bn_bwd_apply_add_sync_wide_kernel(BnBwdP q, const double* all,
                                                                                       int world) {
  bn_bwd_apply_body<NJ, U, true, true, true>(q, all, world);
}

// ================================================================================================ fast path
// The same three streaming passes for the case every BatchNorm of the model but the masked input one is in: no dropout
// mask, every tensor a dense [N][C][plane] array whose CH-channel slabs (CH = 1, 2 or 4: the smallest count that makes
// CH * T*V * 4 bytes a multiple of 16) are 16-byte aligned.  Differences from the generic kernels above:
//  * a CTA owns CH adjacent channels and one batch split; a slab of every staged tensor arrives by ONE bulk-async copy
//    (cp.async.bulk + mbarrier expect_tx, issued by thread 0), double buffered - the other threads spend no
//    instruction on staging (the generic kernels spend ~20 on address arithmetic per 8-byte cp.async);
//  * a thread keeps per owned position one packed word of shared-memory slots; the per-(c,v) constants live in a
//    shared-memory table, outputs are walked linearly (position j of the slab in the output's own memory order);
//  * per-element arithmetic and the order of every sum are those of the generic kernels: outputs and statistics are
//    bit-identical (tests/test_gpu_parity.py::test_bn_fast_path_equals_generic), the PReLU-slope partial is summed
//    over a different thread mapping (equal to rounding).
constexpr int BNF_MAXCH = 4;
// BIG instantiations: slabs of 4097 .. 8192 positions (the stress configuration: two channels x T*V = 2750) with up to
// 1024 threads, one CTA per SM, 13-bit slots (two channels at most, so the constant index still fits the word)
constexpr int BNF_THREADS_BIG = 1024;
// Position word: the slots in the low 2 SB bits, the constant-table index ch * VW + v from bit KS.  The wide tables
// (VW = BN_MAXV rows per channel) need a 64-bit word.
template <bool BIG, bool WIDE = false> struct BnfBits {
  static constexpr int SB = BIG ? 13 : 12;
  static constexpr uint32_t SM = (1u << SB) - 1u;
  static constexpr int VW = bn_table_v(WIDE), KS = WIDE ? 32 : 2 * SB;
  using Pk = typename std::conditional<WIDE, unsigned long long, uint32_t>::type;
  // slot of slab position (ch, t, v) in a slab staged in memory order tf_a | the same in order tf_b << SB
  __device__ __forceinline__ static uint32_t slots(int ch, int t, int v, int T, int V, int TV, bool tf_a, bool tf_b) {
    return (uint32_t)(ch * TV + slot_of(tf_a, t, v, T, V)) | ((uint32_t)(ch * TV + slot_of(tf_b, t, v, T, V)) << SB);
  }
  // the position word: slots(...) | (ch * VW + v) << KS
  __device__ __forceinline__ static Pk pack(int ch, int t, int v, int T, int V, int TV, bool tf_a, bool tf_b) {
    return slots(ch, t, v, T, V, TV, tf_a, tf_b) | ((Pk)(ch * VW + v) << KS);
  }
};

__device__ __forceinline__ void bnf_decode(bool tfast, int j, int T, int V, int TV, int& ch, int& t, int& v) {
  ch = j / TV;
  const int jj = j - ch * TV;
  if (tfast) {
    v = jj / T;
    t = jj - v * T;
  } else {
    t = jj / V;
    v = jj - t * V;
  }
}
__device__ __forceinline__ void bnf_timeout(int* err) {
  if (err) *(volatile int*)err = 2;
}
// the two stage mbarriers, initialised by thread 0 (the caller synchronises the block before their first use)
__device__ __forceinline__ void bnf_mbar_init(uint64_t* mbar) {
  if (threadIdx.x == 0) {
    umma::mbar_init(&mbar[0], 1);
    umma::mbar_init(&mbar[1], 1);
    umma::mbar_init_fence();
  }
}
// the per-(ch, v) constant table of the CH channels at c0 from the BN parameters: ctab[ch * VW + v] = f(pi), pi the
// parameter index of (c0 + ch, v)
template <bool WIDE, class F>
__device__ __forceinline__ void bnf_fill_ctab(float4* ctab, int CH, int c0, int C, int V, int vc_order, F f) {
  constexpr int VW = bn_table_v(WIDE);
  if (WIDE) {
    for (int ix = threadIdx.x; ix < CH * VW; ix += blockDim.x)
      if (ix % VW < V) ctab[ix] = f(bn_pidx(c0 + ix / VW, ix % VW, C, V, vc_order));
  } else if (threadIdx.x < CH * 32 && (threadIdx.x & 31) < V) {
    ctab[threadIdx.x] = f(bn_pidx(c0 + (threadIdx.x >> 5), threadIdx.x & 31, C, V, vc_order));
  }
}

// ---- forward apply: positions in out's memory order
template <int NJ, int U, bool HAS_R, bool FULL, bool BIG, bool WIDE>
__device__ __forceinline__ void bnf_apply_consume(const float* st, const float4* ctab,
                                                  const typename BnfBits<BIG, WIDE>::Pk (&pk)[NJ], float* ob,
                                                  long long osn, int CHTV, int left, float slope) {
#pragma unroll
  for (int i = 0; i < NJ; ++i) {
    if ((int)(threadIdx.x + i * blockDim.x) < CHTV) {
      constexpr int SB = BnfBits<BIG, WIDE>::SB, KS = BnfBits<BIG, WIDE>::KS;
      constexpr uint32_t SM = BnfBits<BIG, WIDE>::SM;
      const uint32_t lo = (uint32_t)pk[i];
      const float4 k = ctab[(uint32_t)(pk[i] >> KS)];
      const float* py = st + (lo & SM);
      const float* pr = st + U * CHTV + ((lo >> SB) & SM);
      float* o = ob + i * blockDim.x;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (FULL || u < left) {
          float pre = fmaf(py[u * CHTV] - k.x, k.y, k.z);
          if (HAS_R) pre += pr[u * CHTV];
          o[u * osn] = pre > 0.f ? pre : slope * pre;
        }
      }
    }
  }
}

template <int NJ, int U, bool HAS_R, bool BIG, bool WIDE>
__device__ __forceinline__ void bnf_apply_body(const BnFwdP& q, int CH, int* err) {
  constexpr int VW = BnfBits<BIG, WIDE>::VW;
  extern __shared__ __align__(16) float sh[];   // [2 stages][y (, r)][U][CH * T*V]
  __shared__ __align__(16) float4 ctab[BNF_MAXCH * VW];     // per (ch, v): mean, gamma * invstd, beta
  __shared__ double tot[VW][2];
  __shared__ __align__(8) uint64_t mbar[2];
  const int c0 = blockIdx.x * CH, s = blockIdx.y, T = q.T, V = q.V, TV = T * V, CHTV = CH * TV;
  const int n0 = (int)((long long)q.N * s / gridDim.y), n1 = (int)((long long)q.N * (s + 1) / gridDim.y), cnt = n1 - n0;
  constexpr int NST = HAS_R ? 2 : 1;
  const int stage_f = NST * U * CHTV, iters = (cnt + U - 1) / U;
  const float slope = q.prelu ? __ldg(q.prelu) : 1.f;
  bnf_mbar_init(mbar);
  __syncthreads();
  auto issue = [&](int it) {   // thread 0: one bulk copy per sample and tensor
    const int n = n0 + it * U, cu = min(U, n1 - n);
    float* d = sh + (it & 1) * stage_f;
    uint64_t* mb = &mbar[it & 1];
    umma::mbar_expect_tx(mb, (uint32_t)(NST * cu * CHTV) * 4u);
    const float* gy = q.y.p + (long long)n * q.y.sn + (long long)c0 * q.y.sc;
    for (int u = 0; u < cu; ++u) umma::bulk_g2s(d + u * CHTV, gy + u * q.y.sn, (uint32_t)CHTV * 4u, mb);
    if (HAS_R) {
      const float* gr = q.r.p + (long long)n * q.r.sn + (long long)c0 * q.r.sc;
      for (int u = 0; u < cu; ++u) umma::bulk_g2s(d + (U + u) * CHTV, gr + u * q.r.sn, (uint32_t)CHTV * 4u, mb);
    }
  };
  if (threadIdx.x == 0 && iters > 0) issue(0);
  if (q.training) {   // batch statistics from the split partials (same arithmetic as bn_apply_kernel)
    for (int ch = 0; ch < CH; ++ch) {
      const int c = c0 + ch;
      sum_partials(q.part, q.S, q.C, c, V, tot);
      __syncthreads();
      if (threadIdx.x < V) {
        const int v = threadIdx.x;
        const double cntd = (double)q.N * q.T;
        const double shift = __ldg(q.y.p + vix(q.y, 0, c, 0, v));
        const double dm = tot[v][0] / cntd;
        double var = tot[v][1] / cntd - dm * dm;
        if (var < 0.) var = 0.;
        const double mean = shift + dm;
        const float fm = (float)mean, fi = (float)(1.0 / sqrt(var + (double)q.eps));
        const int pi = bn_pidx(c, v, q.C, V, q.vc_order);
        ctab[ch * VW + v] = make_float4(fm, __ldg(q.gamma + pi) * fi, __ldg(q.beta + pi), 0.f);
        if (s == 0) {
          q.save_mean[pi] = fm;
          q.save_invstd[pi] = fi;
          if (q.running_mean) {
            const double unb = cntd > 1. ? var * cntd / (cntd - 1.) : var;
            q.running_mean[pi] = (float)((1.0 - q.momentum) * q.running_mean[pi] + q.momentum * mean);
            q.running_var[pi] = (float)((1.0 - q.momentum) * q.running_var[pi] + q.momentum * unb);
          }
          if (c == 0 && v == 0 && q.nbt) *q.nbt += 1;
        }
      }
      __syncthreads();
    }
  } else {
    bnf_fill_ctab<WIDE>(ctab, CH, c0, q.C, V, q.vc_order, [&](int pi) {
      return make_float4(q.save_mean[pi], __ldg(q.gamma + pi) * q.save_invstd[pi], __ldg(q.beta + pi), 0.f);
    });
    __syncthreads();
  }
  typename BnfBits<BIG, WIDE>::Pk pk[NJ];   // slot in y's slab | slot in r's slab << SB | (ch * VW + v) << KS   (valid iff j < CHTV)
  {
    const bool tf_o = t_fastest(q.out), tf_y = t_fastest(q.y), tf_r = HAS_R && t_fastest(q.r);
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
      const int j = threadIdx.x + i * blockDim.x;
      pk[i] = 0u;
      if (j < CHTV) {
        int ch, t, v;
        bnf_decode(tf_o, j, T, V, TV, ch, t, v);
        pk[i] = BnfBits<BIG, WIDE>::pack(ch, t, v, T, V, TV, tf_y, tf_r);
      }
    }
  }
  float* ob = q.out.p + (long long)n0 * q.out.sn + (long long)c0 * q.out.sc + threadIdx.x;
  const long long osn = q.out.sn;
  for (int it = 0; it < iters; ++it) {
    if (threadIdx.x == 0 && it + 1 < iters) issue(it + 1);   // that buffer was released by the barrier ending it - 1
    if (!umma::mbar_wait(&mbar[it & 1], (uint32_t)(it >> 1) & 1u)) bnf_timeout(err);
    const float* st = sh + (it & 1) * stage_f;
    const int left = n1 - (n0 + it * U);
    if (left >= U) bnf_apply_consume<NJ, U, HAS_R, true, BIG, WIDE>(st, ctab, pk, ob, osn, CHTV, left, slope);
    else bnf_apply_consume<NJ, U, HAS_R, false, BIG, WIDE>(st, ctab, pk, ob, osn, CHTV, left, slope);
    ob += U * osn;
    __syncthreads();
  }
}

template <int NJ, int U, bool HAS_R, bool BIG>
__global__ void __launch_bounds__(BIG ? BNF_THREADS_BIG : BN_THREADS_MAX, BIG ? 1 : 2) bnf_apply_kernel(BnFwdP q, int CH, int* err) {
  bnf_apply_body<NJ, U, HAS_R, BIG, false>(q, CH, err);
}
template <int NJ, int U, bool HAS_R, bool BIG>
__global__ void __launch_bounds__(BIG ? BNF_THREADS_BIG : BN_THREADS_MAX, BIG ? 1 : 2) bnf_apply_wide_kernel(BnFwdP q, int CH, int* err) {
  bnf_apply_body<NJ, U, HAS_R, BIG, true>(q, CH, err);
}

// ---- backward pass 1: positions in y's memory order
template <int NJ, int U, bool USE_R, bool FULL, bool BIG, bool WIDE>
__device__ __forceinline__ void bnf_reduce_consume(const float* st, const float4* ctab,
                                                   const typename BnfBits<BIG, WIDE>::Pk (&pk)[NJ], int CHTV,
                                                   int left, float slope, bool has_prelu, float (&a1)[NJ],
                                                   float (&a2)[NJ], float& gsl) {
#pragma unroll
  for (int i = 0; i < NJ; ++i) {
    if ((int)(threadIdx.x + i * blockDim.x) < CHTV) {
      constexpr int SB = BnfBits<BIG, WIDE>::SB, KS = BnfBits<BIG, WIDE>::KS;
      constexpr uint32_t SM = BnfBits<BIG, WIDE>::SM;
      const uint32_t lo = (uint32_t)pk[i];
      const float4 k = ctab[(uint32_t)(pk[i] >> KS)];
      const float* pg = st + (lo & SM);
      const float* py = st + U * CHTV + threadIdx.x + i * blockDim.x;
      const float* pr = st + 2 * U * CHTV + ((lo >> SB) & SM);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (FULL || u < left) {
          float xhat, gs;
          const float gp = bn_gpre(has_prelu, py[u * CHTV], USE_R ? pr[u * CHTV] : 0.f, pg[u * CHTV], 1.f, k.x, k.y, k.z,
                                   k.w, slope, xhat, gs);
          a1[i] += gp;
          a2[i] = fmaf(gp, xhat, a2[i]);
          gsl += gs;
        }
      }
    }
  }
}

template <int NJ, int U, bool USE_R, bool BIG, bool WIDE>
__device__ __forceinline__ void bnf_bwd_reduce_body(const BnBwdP& q, int CH, int* err) {
  constexpr int VW = BnfBits<BIG, WIDE>::VW;
  extern __shared__ __align__(16) float sh[];   // [2 stages][gout, y (, r)][U][CH * T*V]
  __shared__ __align__(16) float4 ctab[BNF_MAXCH * VW];     // per (ch, v): mean, invstd, gamma, beta
  __shared__ float red[32];
  __shared__ __align__(8) uint64_t mbar[2];
  const int c0 = blockIdx.x * CH, s = blockIdx.y, T = q.T, V = q.V, TV = T * V, CHTV = CH * TV;
  const int n0 = (int)((long long)q.N * s / gridDim.y), n1 = (int)((long long)q.N * (s + 1) / gridDim.y), cnt = n1 - n0;
  constexpr int NST = USE_R ? 3 : 2;
  const int stage_f = NST * U * CHTV, iters = (cnt + U - 1) / U;
  const bool has_prelu = q.prelu != nullptr;
  const float slope = has_prelu ? __ldg(q.prelu) : 1.f;
  bnf_mbar_init(mbar);
  bnf_fill_ctab<WIDE>(ctab, CH, c0, q.C, V, q.vc_order, [&](int pi) {
    return make_float4(__ldg(q.save_mean + pi), __ldg(q.save_invstd + pi), __ldg(q.gamma + pi), __ldg(q.beta + pi));
  });
  __syncthreads();
  auto issue = [&](int it) {
    const int n = n0 + it * U, cu = min(U, n1 - n);
    float* d = sh + (it & 1) * stage_f;
    uint64_t* mb = &mbar[it & 1];
    umma::mbar_expect_tx(mb, (uint32_t)(NST * cu * CHTV) * 4u);
    const float* g0 = q.gout.p + (long long)n * q.gout.sn + (long long)c0 * q.gout.sc;
    const float* g1 = q.y.p + (long long)n * q.y.sn + (long long)c0 * q.y.sc;
    for (int u = 0; u < cu; ++u) umma::bulk_g2s(d + u * CHTV, g0 + u * q.gout.sn, (uint32_t)CHTV * 4u, mb);
    for (int u = 0; u < cu; ++u) umma::bulk_g2s(d + (U + u) * CHTV, g1 + u * q.y.sn, (uint32_t)CHTV * 4u, mb);
    if (USE_R) {
      const float* g2 = q.r.p + (long long)n * q.r.sn + (long long)c0 * q.r.sc;
      for (int u = 0; u < cu; ++u) umma::bulk_g2s(d + (2 * U + u) * CHTV, g2 + u * q.r.sn, (uint32_t)CHTV * 4u, mb);
    }
  };
  if (threadIdx.x == 0 && iters > 0) issue(0);
  typename BnfBits<BIG, WIDE>::Pk pk[NJ];   // slot in gout's slab | slot in r's slab << SB | (ch * VW + v) << KS;  y is read at j itself
  float a1[NJ], a2[NJ], gsl = 0.f;
  const bool tf_y = t_fastest(q.y);
  {
    const bool tf_g = t_fastest(q.gout), tf_r = USE_R && t_fastest(q.r);
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
      const int j = threadIdx.x + i * blockDim.x;
      pk[i] = 0u;
      a1[i] = a2[i] = 0.f;
      if (j < CHTV) {
        int ch, t, v;
        bnf_decode(tf_y, j, T, V, TV, ch, t, v);
        pk[i] = BnfBits<BIG, WIDE>::pack(ch, t, v, T, V, TV, tf_g, tf_r);
      }
    }
  }
  for (int it = 0; it < iters; ++it) {
    if (threadIdx.x == 0 && it + 1 < iters) issue(it + 1);
    if (!umma::mbar_wait(&mbar[it & 1], (uint32_t)(it >> 1) & 1u)) bnf_timeout(err);
    const float* st = sh + (it & 1) * stage_f;
    const int left = n1 - (n0 + it * U);
    if (left >= U) bnf_reduce_consume<NJ, U, USE_R, true, BIG, WIDE>(st, ctab, pk, CHTV, left, slope, has_prelu, a1, a2, gsl);
    else bnf_reduce_consume<NJ, U, USE_R, false, BIG, WIDE>(st, ctab, pk, CHTV, left, slope, has_prelu, a1, a2, gsl);
    __syncthreads();
  }
  // per-(c,v) totals: positions to their logical slot, then one thread per (ch, v) sums over t in order (fp64)
#pragma unroll
  for (int i = 0; i < NJ; ++i) {
    const int j = threadIdx.x + i * blockDim.x;
    if (j < CHTV) {
      int ch, t, v;
      bnf_decode(tf_y, j, T, V, TV, ch, t, v);
      sh[ch * TV + t * V + v] = a1[i];
      sh[CHTV + ch * TV + t * V + v] = a2[i];
    }
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < CH * V; idx += blockDim.x) {
    const int ch = idx / V, v = idx - ch * V;
    double s1 = 0., s2 = 0.;
    for (int t = 0; t < T; ++t) {
      s1 += sh[ch * TV + t * V + v];
      s2 += sh[CHTV + ch * TV + t * V + v];
    }
    float* dst = q.part + (((long long)s * q.C + c0 + ch) * V + v) * 2;
    dst[0] = (float)s1;
    dst[1] = (float)s2;
  }
  const float totp = block_sum(gsl, red);
  if (threadIdx.x == 0) q.part_p[(long long)s * gridDim.x + blockIdx.x] = totp;
}

template <int NJ, int U, bool USE_R, bool BIG>
__global__ void __launch_bounds__(BIG ? BNF_THREADS_BIG : BN_THREADS_MAX, BIG ? 1 : 2) bnf_bwd_reduce_kernel(BnBwdP q, int CH, int* err) {
  bnf_bwd_reduce_body<NJ, U, USE_R, BIG, false>(q, CH, err);
}
template <int NJ, int U, bool USE_R, bool BIG>
__global__ void __launch_bounds__(BIG ? BNF_THREADS_BIG : BN_THREADS_MAX, BIG ? 1 : 2) bnf_bwd_reduce_wide_kernel(BnBwdP q, int CH, int* err) {
  bnf_bwd_reduce_body<NJ, U, USE_R, BIG, true>(q, CH, err);
}

// ---- backward pass 2: positions in gy's memory order; gr (same order as gy) is stored straight from registers
template <int NJ, int U, bool USE_R, bool HAS_GR, bool ADD, bool FULL, bool BIG, bool WIDE>
__device__ __forceinline__ void bnf_bwd_apply_consume(const float* st, const float4* ctab, const float4* ctab2,
                                                      const typename BnfBits<BIG, WIDE>::Pk (&pk)[NJ],
                                                      const uint32_t (&pk2)[NJ], float* gyb, float* grb,
                                                      long long gysn, long long grsn, int CHTV, int left, float slope,
                                                      bool has_prelu) {
  constexpr int ADD_REGION = USE_R ? 3 : 2;
#pragma unroll
  for (int i = 0; i < NJ; ++i) {
    if ((int)(threadIdx.x + i * blockDim.x) < CHTV) {
      constexpr int SB = BnfBits<BIG, WIDE>::SB, KS = BnfBits<BIG, WIDE>::KS;
      constexpr uint32_t SM = BnfBits<BIG, WIDE>::SM;
      const uint32_t lo = (uint32_t)pk[i];
      const float4 k = ctab[(uint32_t)(pk[i] >> KS)], k2 = ctab2[(uint32_t)(pk[i] >> KS)];
      const float* pg = st + (lo & SM);
      const float* py = st + U * CHTV + ((lo >> SB) & SM);
      const float* pr = st + 2 * U * CHTV + (pk2[i] & SM);
      const float* pa = st + ADD_REGION * U * CHTV + ((pk2[i] >> SB) & SM);
      float* o = gyb + i * blockDim.x;
      float* o2 = grb + i * blockDim.x;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (FULL || u < left) {
          float xhat, gs;
          const float gp = bn_gpre(has_prelu, py[u * CHTV], USE_R ? pr[u * CHTV] : 0.f, pg[u * CHTV], 1.f, k.x, k.y, k.z,
                                   k.w, slope, xhat, gs);
          o[u * gysn] = k2.x * (gp - k2.y - xhat * k2.z);
          if (HAS_GR) o2[u * grsn] = ADD ? gp + pa[u * CHTV] : gp;
        }
      }
    }
  }
}

// SYNC: global phase of the synchronised backward, as in bn_bwd_apply_body
template <int NJ, int U, bool USE_R, bool HAS_GR, bool ADD, bool BIG, bool SYNC, bool WIDE>
__device__ __forceinline__ void bnf_bwd_apply_body(const BnBwdP& q, int CH, int NP, int* err, const double* all, int world) {
  constexpr int VW = BnfBits<BIG, WIDE>::VW;
  extern __shared__ __align__(16) float sh[];   // [2 stages][gout, y (, r) (, gr_add)][U][CH * T*V]
  __shared__ __align__(16) float4 ctab[BNF_MAXCH * VW];     // mean, invstd, gamma, beta
  __shared__ __align__(16) float4 ctab2[BNF_MAXCH * VW];    // gamma * invstd, k1, k2
  __shared__ double tot[VW][2];
  __shared__ float red[32];
  __shared__ __align__(8) uint64_t mbar[2];
  const int c0 = blockIdx.x * CH, s = blockIdx.y, T = q.T, V = q.V, TV = T * V, CHTV = CH * TV;
  const int n0 = (int)((long long)q.N * s / gridDim.y), n1 = (int)((long long)q.N * (s + 1) / gridDim.y), cnt = n1 - n0;
  constexpr int NST = 2 + (USE_R ? 1 : 0) + (ADD ? 1 : 0), ADD_REGION = USE_R ? 3 : 2;
  const int stage_f = NST * U * CHTV, iters = (cnt + U - 1) / U;
  const bool has_prelu = q.prelu != nullptr;
  const float slope = has_prelu ? __ldg(q.prelu) : 1.f;
  const float icnt = 1.0f / ((float)q.N * (float)T);
  bnf_mbar_init(mbar);
  __syncthreads();
  auto issue = [&](int it) {
    const int n = n0 + it * U, cu = min(U, n1 - n);
    float* d = sh + (it & 1) * stage_f;
    uint64_t* mb = &mbar[it & 1];
    umma::mbar_expect_tx(mb, (uint32_t)(NST * cu * CHTV) * 4u);
    const float* g0 = q.gout.p + (long long)n * q.gout.sn + (long long)c0 * q.gout.sc;
    const float* g1 = q.y.p + (long long)n * q.y.sn + (long long)c0 * q.y.sc;
    for (int u = 0; u < cu; ++u) umma::bulk_g2s(d + u * CHTV, g0 + u * q.gout.sn, (uint32_t)CHTV * 4u, mb);
    for (int u = 0; u < cu; ++u) umma::bulk_g2s(d + (U + u) * CHTV, g1 + u * q.y.sn, (uint32_t)CHTV * 4u, mb);
    if (USE_R) {
      const float* g2 = q.r.p + (long long)n * q.r.sn + (long long)c0 * q.r.sc;
      for (int u = 0; u < cu; ++u) umma::bulk_g2s(d + (2 * U + u) * CHTV, g2 + u * q.r.sn, (uint32_t)CHTV * 4u, mb);
    }
    if (ADD) {
      const float* g3 = q.gadd.p + (long long)n * q.gadd.sn + (long long)c0 * q.gadd.sc;
      for (int u = 0; u < cu; ++u) umma::bulk_g2s(d + (ADD_REGION * U + u) * CHTV, g3 + u * q.gadd.sn, (uint32_t)CHTV * 4u, mb);
    }
  };
  if (threadIdx.x == 0 && iters > 0) issue(0);
  // sums of pass 1 over the splits; the s == 0 CTA publishes the parameter gradients of its channels
  if (!SYNC && blockIdx.x == 0 && s == 0 && q.gprelu) bn_sum_slope_partials(q, NP, red);
  for (int ch = 0; ch < CH; ++ch) {
    const int c = c0 + ch;
    if (SYNC) sync_bwd_totals(all, world, q.C, V, c, q.vc_order, tot);
    else sum_partials(q.part, q.S, q.C, c, V, tot);
    __syncthreads();
    if (threadIdx.x < V) {
      const int v = threadIdx.x, pi = bn_pidx(c, v, q.C, V, q.vc_order);
      const float mu = __ldg(q.save_mean + pi), is = __ldg(q.save_invstd + pi), g = __ldg(q.gamma + pi);
      ctab[ch * VW + v] = make_float4(mu, is, g, __ldg(q.beta + pi));
      if (SYNC) {
        ctab2[ch * VW + v] = make_float4(g * is, (float)tot[v][0], (float)tot[v][1], 0.f);
      } else {
        ctab2[ch * VW + v] = make_float4(g * is, q.training ? (float)tot[v][0] * icnt : 0.f,
                                         q.training ? (float)tot[v][1] * icnt : 0.f, 0.f);
        if (s == 0) {
          q.gbeta[pi] = (float)tot[v][0];
          q.ggamma[pi] = (float)tot[v][1];
        }
      }
    }
    __syncthreads();
  }
  typename BnfBits<BIG, WIDE>::Pk pk[NJ];   // gout slot | y slot << SB | (ch * VW + v) << KS
  uint32_t pk2[NJ];                         // r slot | gr_add slot << SB
  {
    const bool tf_o = t_fastest(q.gy), tf_g = t_fastest(q.gout), tf_y = t_fastest(q.y), tf_r = USE_R && t_fastest(q.r),
               tf_a = ADD && t_fastest(q.gadd);
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
      const int j = threadIdx.x + i * blockDim.x;
      pk[i] = 0u;
      pk2[i] = 0u;
      if (j < CHTV) {
        int ch, t, v;
        bnf_decode(tf_o, j, T, V, TV, ch, t, v);
        pk[i] = BnfBits<BIG, WIDE>::pack(ch, t, v, T, V, TV, tf_g, tf_y);
        pk2[i] = BnfBits<BIG, WIDE>::slots(ch, t, v, T, V, TV, tf_r, tf_a);
      }
    }
  }
  float* gyb = q.gy.p + (long long)n0 * q.gy.sn + (long long)c0 * q.gy.sc + threadIdx.x;
  float* grb = HAS_GR ? q.gr.p + (long long)n0 * q.gr.sn + (long long)c0 * q.gr.sc + threadIdx.x : nullptr;
  const long long gysn = q.gy.sn, grsn = HAS_GR ? q.gr.sn : 0;
  for (int it = 0; it < iters; ++it) {
    if (threadIdx.x == 0 && it + 1 < iters) issue(it + 1);
    if (!umma::mbar_wait(&mbar[it & 1], (uint32_t)(it >> 1) & 1u)) bnf_timeout(err);
    const float* st = sh + (it & 1) * stage_f;
    const int left = n1 - (n0 + it * U);
    if (left >= U)
      bnf_bwd_apply_consume<NJ, U, USE_R, HAS_GR, ADD, true, BIG, WIDE>(st, ctab, ctab2, pk, pk2, gyb, grb, gysn, grsn, CHTV, left, slope, has_prelu);
    else
      bnf_bwd_apply_consume<NJ, U, USE_R, HAS_GR, ADD, false, BIG, WIDE>(st, ctab, ctab2, pk, pk2, gyb, grb, gysn, grsn, CHTV, left, slope, has_prelu);
    gyb += U * gysn;
    if (HAS_GR) grb += U * grsn;
    __syncthreads();
  }
}

template <int NJ, int U, bool USE_R, bool HAS_GR, bool ADD, bool BIG>
__global__ void __launch_bounds__(BIG ? BNF_THREADS_BIG : BN_THREADS_MAX, BIG ? 1 : 2) bnf_bwd_apply_kernel(BnBwdP q, int CH, int NP, int* err) {
  bnf_bwd_apply_body<NJ, U, USE_R, HAS_GR, ADD, BIG, false, false>(q, CH, NP, err, nullptr, 0);
}
template <int NJ, int U, bool USE_R, bool HAS_GR, bool ADD, bool BIG>
__global__ void __launch_bounds__(BIG ? BNF_THREADS_BIG : BN_THREADS_MAX, BIG ? 1 : 2) bnf_bwd_apply_sync_kernel(BnBwdP q, int CH, int* err, const double* all, int world) {
  bnf_bwd_apply_body<NJ, U, USE_R, HAS_GR, ADD, BIG, true, false>(q, CH, 0, err, all, world);
}
template <int NJ, int U, bool USE_R, bool HAS_GR, bool ADD, bool BIG>
__global__ void __launch_bounds__(BIG ? BNF_THREADS_BIG : BN_THREADS_MAX, BIG ? 1 : 2) bnf_bwd_apply_wide_kernel(BnBwdP q, int CH, int NP, int* err) {
  bnf_bwd_apply_body<NJ, U, USE_R, HAS_GR, ADD, BIG, false, true>(q, CH, NP, err, nullptr, 0);
}
template <int NJ, int U, bool USE_R, bool HAS_GR, bool ADD, bool BIG>
__global__ void __launch_bounds__(BIG ? BNF_THREADS_BIG : BN_THREADS_MAX, BIG ? 1 : 2) bnf_bwd_apply_sync_wide_kernel(BnBwdP q, int CH, int* err, const double* all, int world) {
  bnf_bwd_apply_body<NJ, U, USE_R, HAS_GR, ADD, BIG, true, true>(q, CH, 0, err, all, world);
}

// ---- synchronised BatchNorm: fold and merge kernels around the exchange of per-rank rows
// Exchange rows of one rank, fp64, in BN parameter order: [3][C*V] = (count, mean, M2) in the forward,
// (count, sum g', sum g' xhat) in the backward.  One CTA per channel (fold), one thread per parameter index (merge).

// forward, local phase: this rank's split partials (shifted sums) -> (count, mean_r, M2_r)
template <bool WIDE>
__device__ __forceinline__ void bn_sync_fold_fwd_body(const BnFwdP& q, double* mine) {
  __shared__ double tot[bn_table_v(WIDE)][2];
  const int c = blockIdx.x, V = q.V;
  const long long cv = (long long)q.C * V;
  sum_partials(q.part, q.S, q.C, c, V, tot);
  __syncthreads();
  if (threadIdx.x < V) {
    const int v = threadIdx.x, pi = bn_pidx(c, v, q.C, V, q.vc_order);
    const double cntd = (double)q.N * q.T;
    const double shift = __ldg(q.y.p + vix(q.y, 0, c, 0, v));
    const double dm = tot[v][0] / cntd;
    double m2 = tot[v][1] - tot[v][0] * dm;
    if (m2 < 0.) m2 = 0.;
    mine[pi] = cntd;
    mine[cv + pi] = shift + dm;
    mine[2 * cv + pi] = m2;
  }
}
__global__ void bn_sync_fold_fwd_kernel(BnFwdP q, double* mine) { bn_sync_fold_fwd_body<false>(q, mine); }
__global__ void bn_sync_fold_fwd_wide_kernel(BnFwdP q, double* mine) { bn_sync_fold_fwd_body<true>(q, mine); }

// forward, global phase: Chan's merge of the `world` rows in rank order -> save_mean / save_invstd, running statistics
// (global count, unbiased variance), num_batches_tracked
__global__ void bn_sync_merge_fwd_kernel(BnFwdP q, const double* all, int world) {
  const long long cv = (long long)q.C * q.V;
  const int pi = blockIdx.x * blockDim.x + threadIdx.x;
  if (pi >= cv) return;
  double n = 0., s = 0.;
  for (int r = 0; r < world; ++r) {
    const double nr = all[3 * cv * r + pi];
    n += nr;
    s += nr * all[3 * cv * r + cv + pi];
  }
  const double mean = s / n;
  double m2 = 0.;
  for (int r = 0; r < world; ++r) {
    const double* row = all + 3 * cv * r + pi;
    const double d = row[cv] - mean;
    m2 += row[2 * cv] + row[0] * d * d;
  }
  const double var = m2 / n;
  q.save_mean[pi] = (float)mean;
  q.save_invstd[pi] = (float)(1.0 / sqrt(var + (double)q.eps));
  if (q.running_mean) {
    const double unb = n > 1. ? m2 / (n - 1.) : var;
    q.running_mean[pi] = (float)((1.0 - q.momentum) * q.running_mean[pi] + q.momentum * mean);
    q.running_var[pi] = (float)((1.0 - q.momentum) * q.running_var[pi] + q.momentum * unb);
  }
  if (pi == 0 && q.nbt) *q.nbt += 1;
}

// backward, local phase: this rank's parameter gradients (the sums and the order of bn_bwd_apply / bnf_bwd_apply:
// launched with the block size of the apply kernel the plain call would run, over its NP slope partials) and its
// exchange rows (count, sum g', sum g' xhat)
template <bool WIDE>
__device__ __forceinline__ void bn_sync_fold_bwd_body(const BnBwdP& q, int NP, double* mine) {
  __shared__ double tot[bn_table_v(WIDE)][2];
  __shared__ float red[32];
  const int c = blockIdx.x, V = q.V;
  const long long cv = (long long)q.C * V;
  sum_partials(q.part, q.S, q.C, c, V, tot);
  if (c == 0 && q.gprelu) bn_sum_slope_partials(q, NP, red);
  __syncthreads();
  if (threadIdx.x < V) {
    const int v = threadIdx.x, pi = bn_pidx(c, v, q.C, V, q.vc_order);
    q.gbeta[pi] = (float)tot[v][0];
    q.ggamma[pi] = (float)tot[v][1];
    mine[pi] = (double)q.N * q.T;
    mine[cv + pi] = tot[v][0];
    mine[2 * cv + pi] = tot[v][1];
  }
}
__global__ void bn_sync_fold_bwd_kernel(BnBwdP q, int NP, double* mine) { bn_sync_fold_bwd_body<false>(q, NP, mine); }
__global__ void bn_sync_fold_bwd_wide_kernel(BnBwdP q, int NP, double* mine) { bn_sync_fold_bwd_body<true>(q, NP, mine); }

// host side of the fast path
struct BnFastPlan {
  bool ok;
  int ch, nj, threads;
  bool big;     // slab of 4097 .. 8192 positions: BIG instantiations (<= 1024 threads, one CTA per SM)
  bool wide;    // V > 32: the _wide_ instantiations
};
static bool bnf_slab_ok(const View4& w, int T, int V) {
  if (!w.p) return true;
  return plane_dense(w, T, V) && w.sc == (long long)T * V && (reinterpret_cast<unsigned long long>(w.p) & 15ull) == 0 &&
         (w.sn & 3ll) == 0;
}
static BnFastPlan bnf_plan(bool fast, int C, int T, int V, const float* mask, std::initializer_list<const View4*> ws) {
  BnFastPlan pl{false, 0, 0, 0, false, V > 32};
  if (!fast || mask || V > BN_MAXV) return pl;
  const int TV = T * V;
  pl.ch = (TV % 4 == 0) ? 1 : (TV % 2 == 0) ? 2 : 4;
  const int chtv = pl.ch * TV;
  pl.big = chtv > 4096;
  if (C % pl.ch || chtv > 8 * BNF_THREADS_BIG || (pl.big && pl.ch > 2)) return pl;
  for (const View4* w : ws)
    if (!bnf_slab_ok(*w, T, V)) return pl;
  pl.nj = chtv <= 4 * BN_THREADS_MAX ? 4 : 8;
  pl.threads = cdiv(cdiv(chtv, pl.nj), 32) * 32;
  if (pl.wide && pl.threads < V) pl.threads = cdiv(V, 32) * 32;   // one thread per v in the per-channel steps
  pl.ok = true;
  return pl;
}
// The per-(c, v) tables of the wide fast kernels take up to 13.5 KB more static shared memory (bnf_bwd_apply: two
// float4 tables of BNF_MAXCH * BN_MAXV rows and the fp64 totals) than the 32-joint ones; it comes off the budget.
constexpr size_t BNF_WIDE_TABLES = (size_t)(2 * BNF_MAXCH * 16 + 16) * (BN_MAXV - 32);
// samples per stage: the largest of 4/2/1 whose two stages of `nst` slabs fit two CTAs per SM; 0 = none
static int bnf_pick_u(size_t slab_bytes, int nst, bool big = false, bool wide = false) {
  const size_t budget = (big ? (size_t)220 * 1024 : BN_SMEM_BUDGET) - (wide ? BNF_WIDE_TABLES : 0);   // BIG: one CTA per SM
  for (int u = big ? 2 : 4; u >= 1; u >>= 1)
    if ((size_t)2 * nst * u * slab_bytes <= budget) return u;
  return 0;
}

// Kernel dispatch: call f with std::integral_constant arguments naming a compiled instantiation.
template <int K> using IntC = std::integral_constant<int, K>;
// samples per pipeline stage: 4, 2, or 1 for any other value
template <class F> static int with_u(int u, F&& f) {
  if (u == 4) return f(IntC<4>{});
  if (u == 2) return f(IntC<2>{});
  return f(IntC<1>{});
}
// positions per thread of the generic kernels: 1, 2, 4, or 8 for any other value
template <class F> static int with_nj(int nj, F&& f) {
  if (nj == 1) return f(IntC<1>{});
  if (nj == 2) return f(IntC<2>{});
  if (nj == 4) return f(IntC<4>{});
  return f(IntC<8>{});
}
// fast path f(NJ, U, BIG): BIG slabs run 8 positions per thread and 2 or 1 samples per stage, the others NJ = plan.nj
// (4, or 8 for any other value) and U as with_u
template <class F> static int with_bnf(const BnFastPlan& plan, int u, F&& f) {
  if (plan.big) return u == 2 ? f(IntC<8>{}, IntC<2>{}, std::true_type{}) : f(IntC<8>{}, IntC<1>{}, std::true_type{});
  return with_u(u, [&](auto U) {
    return plan.nj == 4 ? f(IntC<4>{}, U, std::false_type{}) : f(IntC<8>{}, U, std::false_type{});
  });
}

// one launch of a streaming pass: the largest shared-memory carve-out for the kernel, then the launch
template <class... P, class... A>
static int bn_launch(void (*kernel)(P...), dim3 grid, int threads, size_t smem, cudaStream_t st, const char* name,
                     const A&... args) {
  prefer_smem_carveout((const void*)kernel, true);
  kernel<<<grid, threads, smem, st>>>(args...);
  count_launch();
  DSTD_LAUNCH_CHECK(name);
  return DSTD_OK;
}

}  // namespace dstd

// =========================================================================================== C ABI
using namespace dstd;

extern "C" size_t dstd_bn_act_workspace_bytes(int N, int C, int T, int V) {
  int S = N > 128 ? 128 : N;   // upper bound of bn_act_splits
  if (S < 1) S = 1;
  return arena_need({(size_t)S * C * V * 2 * sizeof(float), (size_t)S * C * sizeof(float)});
}

// Which call an argument check serves: the plain one, or the local / global phase of a synchronised one.  The local
// forward reads y only (and the workspace); the global phases read no workspace; the global backward writes no
// parameter gradients.
enum BnPhase { BN_PLAIN, BN_LOCAL, BN_GLOBAL };

// T*V above BN_MAXJ * BN_THREADS_MAX: only V > 32 on the fast path (`fast`: it takes every pass of the call)
static int bn_check_positions(int T, int V, bool fast) {
  DSTD_REQUIRE(T * V <= BN_MAXJ * BN_THREADS_MAX || (V > 32 && fast), DSTD_ERR_UNSUPPORTED,
               "bn_act: T*V=%d outside the compiled limits: the generic kernels (dropout mask, layouts the fast path "
               "does not take, V <= 32) run up to %d positions, the fast path for V > 32 slabs of up to %d",
               T * V, BN_MAXJ * BN_THREADS_MAX, 8 * BNF_THREADS_BIG);
  return DSTD_OK;
}

// fast-path samples per stage of the forward apply pass; 0 = the generic kernel
static int bn_fwd_fast_u(const BnFwdP& q, const Switches& sw, BnFastPlan* out = nullptr) {
  const BnFastPlan fp = bnf_plan(sw.bn_fast, q.C, q.T, q.V, q.mask, {&q.y, &q.r, &q.out});
  if (out) *out = fp;
  return fp.ok ? bnf_pick_u((size_t)fp.ch * q.T * q.V * sizeof(float), q.r.p ? 2 : 1, fp.big, fp.wide) : 0;
}

// ---- forward: argument checks and kernel parameters shared by the plain call and the two synchronised phases
static int bn_fwd_setup(const dstd_bn_act_fwd_args* a, const Switches& sw, BnFwdP& q, BnPhase ph = BN_PLAIN) {
  DSTD_REQUIRE(a, DSTD_ERR_BAD_ARG, "bn_act_forward: null args");
  DSTD_REQUIRE(a->N > 0 && a->C > 0 && a->T > 0 && a->V > 0, DSTD_ERR_BAD_ARG, "bn_act_forward: bad dims");
  DSTD_REQUIRE(a->y.ptr && (ph == BN_LOCAL || (a->out.ptr && a->gamma && a->beta && a->save_mean && a->save_invstd)),
               DSTD_ERR_BAD_ARG, "bn_act_forward: null tensor");
  DSTD_REQUIRE(a->V <= BN_MAXV, DSTD_ERR_UNSUPPORTED, "bn_act: V=%d joints (max %d) outside the compiled limits",
               a->V, BN_MAXV);
  DSTD_REQUIRE(a->training || (a->running_mean && a->running_var), DSTD_ERR_BAD_ARG,
               "bn_act_forward: eval mode needs running statistics");
  DSTD_REQUIRE(ph == BN_GLOBAL || (a->ws_bytes >= dstd_bn_act_workspace_bytes(a->N, a->C, a->T, a->V) && a->ws),
               DSTD_ERR_WORKSPACE, "bn_act_forward: workspace too small");
  q.N = a->N; q.C = a->C; q.T = a->T; q.V = a->V;
  q.vc_order = a->vc_order; q.training = a->training;
  q.S = bn_act_splits(a->N, sw.bn_samples_per_cta);
  q.eps = a->eps; q.momentum = a->momentum;
  q.y = mk(a->y); q.r = mk(a->r); q.out = mk(a->out);
  q.gamma = a->gamma; q.beta = a->beta;
  q.running_mean = a->running_mean; q.running_var = a->running_var;
  q.nbt = a->num_batches_tracked;
  q.prelu = a->prelu; q.mask = a->mask;
  q.save_mean = a->save_mean; q.save_invstd = a->save_invstd;
  q.part = nullptr;
  if (ph != BN_GLOBAL) {
    Arena ar(a->ws, a->ws_bytes);
    q.part = ar.take<float>((size_t)q.S * q.C * q.V * 2);
  }
  return bn_check_positions(q.T, q.V, q.T * q.V <= BN_MAXJ * BN_THREADS_MAX || bn_fwd_fast_u(q, sw) > 0);
}

static int bn_fwd_stats(const BnFwdP& q, cudaStream_t st) {
  const BnGeom g = bn_geom(q.T, q.V);
  const size_t smem = 2 * (size_t)q.T * q.V * sizeof(float);
  if (q.T * q.V > BN_MAXJ * BN_THREADS_MAX)
    return bn_launch(bn_stats_big_kernel, dim3(q.C, q.S), g.threads, smem, st, "bn_stats", q);
  with_nj(g.nj, [&](auto NJ) {
    bn_stats_kernel<NJ><<<dim3(q.C, q.S), g.threads, smem, st>>>(q);
    return 0;
  });
  count_launch();
  DSTD_LAUNCH_CHECK("bn_stats");
  return DSTD_OK;
}

// the apply pass: bulk-copy staged kernel when the layouts allow it (see "fast path"), the generic one otherwise
static int bn_fwd_apply(const BnFwdP& q, const Switches& sw, cudaStream_t st) {
  const size_t tvb = (size_t)q.T * q.V * sizeof(float);
  const int nst = q.r.p ? 2 : 1;                       // staged tensors: y (, r); two pipeline stages
  BnFastPlan fp;
  const int fu = bn_fwd_fast_u(q, sw, &fp);
  if (fu) {
    const dim3 grid(q.C / fp.ch, q.S);
    const size_t smem = (size_t)2 * nst * fu * fp.ch * tvb;
    int* err = device_error_word();
    return with_bnf(fp, fu, [&](auto NJ, auto U, auto BIG) {
      const auto k = q.r.p ? (fp.wide ? bnf_apply_wide_kernel<NJ, U, true, BIG> : bnf_apply_kernel<NJ, U, true, BIG>)
                           : (fp.wide ? bnf_apply_wide_kernel<NJ, U, false, BIG> : bnf_apply_kernel<NJ, U, false, BIG>);
      return bn_launch(k, grid, fp.threads, smem, st, "bnf_apply", q, fp.ch, err);
    });
  }
  const BnGeom g = bn_geom(q.T, q.V);
  const int u = bn_pick_u(tvb, 2 * nst, 4, BN_SMEM_BUDGET);
  const size_t smu = (size_t)2 * nst * u * tvb;
  return with_nj(g.nj, [&](auto NJ) {
    return with_u(u, [&](auto U) {
      const auto k = q.V > 32 ? bn_apply_wide_kernel<NJ, U> : bn_apply_kernel<NJ, U>;
      return bn_launch(k, dim3(q.C, q.S), g.threads, smu, st, "bn_apply", q);
    });
  });
}

extern "C" int dstd_bn_act_forward(const dstd_bn_act_fwd_args* a, dstd_stream_t stream) {
  const Switches sw = read_switches();
  cudaStream_t st = (cudaStream_t)stream;
  BnFwdP q;
  int rc = bn_fwd_setup(a, sw, q);
  if (rc != DSTD_OK) return rc;
  if (q.training) {
    rc = bn_fwd_stats(q, st);
    if (rc != DSTD_OK) return rc;
  } else {
    bn_eval_stats_kernel<<<cdiv(q.C * q.V, 128), 128, 0, st>>>(q);
    count_launch();
    DSTD_LAUNCH_CHECK("bn_eval_stats");
  }
  return bn_fwd_apply(q, sw, st);
}

extern "C" size_t dstd_bn_sync_buffer_doubles(int C, int V) { return (size_t)3 * C * V; }

extern "C" int dstd_bn_act_forward_local(const dstd_bn_act_fwd_args* a, double* mine, dstd_stream_t stream) {
  DSTD_REQUIRE(a && a->training == 1, DSTD_ERR_BAD_ARG, "bn_act_forward_local: needs training = 1");
  DSTD_REQUIRE(mine, DSTD_ERR_BAD_ARG, "bn_act_forward_local: null exchange buffer");
  const Switches sw = read_switches();
  cudaStream_t st = (cudaStream_t)stream;
  BnFwdP q;
  int rc = bn_fwd_setup(a, sw, q, BN_LOCAL);
  if (rc != DSTD_OK) return rc;
  rc = bn_fwd_stats(q, st);
  if (rc != DSTD_OK) return rc;
  if (q.V > 32) bn_sync_fold_fwd_wide_kernel<<<q.C, 256, 0, st>>>(q, mine);
  else bn_sync_fold_fwd_kernel<<<q.C, 256, 0, st>>>(q, mine);
  count_launch();
  DSTD_LAUNCH_CHECK("bn_sync_fold_fwd");
  return DSTD_OK;
}

extern "C" int dstd_bn_act_forward_global(const dstd_bn_act_fwd_args* a, const double* all, int world,
                                          dstd_stream_t stream) {
  DSTD_REQUIRE(a && a->training == 1, DSTD_ERR_BAD_ARG, "bn_act_forward_global: needs training = 1");
  DSTD_REQUIRE(all && world >= 1, DSTD_ERR_BAD_ARG, "bn_act_forward_global: null exchange buffer or world < 1");
  const Switches sw = read_switches();
  cudaStream_t st = (cudaStream_t)stream;
  BnFwdP q;
  int rc = bn_fwd_setup(a, sw, q, BN_GLOBAL);
  if (rc != DSTD_OK) return rc;
  bn_sync_merge_fwd_kernel<<<cdiv(q.C * q.V, 128), 128, 0, st>>>(q, all, world);
  count_launch();
  DSTD_LAUNCH_CHECK("bn_sync_merge_fwd");
  q.training = 0;          // the apply kernels' eval branch: normalise with save_mean / save_invstd as given
  return bn_fwd_apply(q, sw, st);
}

// ---- backward: shared argument checks, kernel parameters and the kernel plan
struct BnBwdPlan {
  BnFastPlan fp;
  int u1, u2;        // fast path: samples per stage of the reduce / apply pass (both nonzero = fast path taken)
  int ub, ub2;       // generic path: the same
  int nst, nst2;     // staged tensors of the reduce / apply pass
  bool use_r, add;
  BnGeom g;
  bool fast() const { return u1 && u2; }
};

static BnBwdPlan bn_bwd_plan(const BnBwdP& q, const Switches& sw);

// (the local phase takes gy / gr as well: it does not write them, but their layouts pick the kernels, as in the plain
// call)
static int bn_bwd_setup(const dstd_bn_act_bwd_args* a, const Switches& sw, BnBwdP& q, BnPhase ph = BN_PLAIN) {
  DSTD_REQUIRE(a, DSTD_ERR_BAD_ARG, "bn_act_backward: null args");
  DSTD_REQUIRE(a->N > 0 && a->C > 0 && a->T > 0 && a->V > 0, DSTD_ERR_BAD_ARG, "bn_act_backward: bad dims");
  DSTD_REQUIRE(a->y.ptr && a->gout.ptr && a->gy.ptr && a->gamma && a->beta && a->save_mean && a->save_invstd &&
                   (ph == BN_GLOBAL || (a->ggamma && a->gbeta)),
               DSTD_ERR_BAD_ARG, "bn_act_backward: null tensor");
  DSTD_REQUIRE(!a->gr.ptr || a->r.ptr, DSTD_ERR_BAD_ARG, "bn_act_backward: gr requested without r");
  DSTD_REQUIRE(!a->gr_add.ptr || a->gr.ptr, DSTD_ERR_BAD_ARG, "bn_act_backward: gr_add given without gr");
  DSTD_REQUIRE(a->V <= BN_MAXV, DSTD_ERR_UNSUPPORTED, "bn_act: V=%d joints (max %d) outside the compiled limits",
               a->V, BN_MAXV);
  DSTD_REQUIRE(ph == BN_GLOBAL || (a->ws_bytes >= dstd_bn_act_workspace_bytes(a->N, a->C, a->T, a->V) && a->ws),
               DSTD_ERR_WORKSPACE, "bn_act_backward: workspace too small");
  q.N = a->N; q.C = a->C; q.T = a->T; q.V = a->V;
  q.vc_order = a->vc_order; q.training = a->training;
  q.S = bn_act_splits(a->N, sw.bn_samples_per_cta);
  q.y = mk(a->y); q.r = mk(a->r); q.gout = mk(a->gout); q.gy = mk(a->gy); q.gr = mk(a->gr); q.gadd = mk(a->gr_add);
  q.gamma = a->gamma; q.beta = a->beta; q.prelu = a->prelu; q.mask = a->mask;
  q.save_mean = a->save_mean; q.save_invstd = a->save_invstd;
  q.ggamma = a->ggamma; q.gbeta = a->gbeta; q.gprelu = a->prelu ? a->gprelu : nullptr;
  q.part = q.part_p = nullptr;
  if (ph != BN_GLOBAL) {
    Arena ar(a->ws, a->ws_bytes);
    q.part = ar.take<float>((size_t)q.S * q.C * q.V * 2);
    q.part_p = ar.take<float>((size_t)q.S * q.C);
  }
  return bn_check_positions(q.T, q.V, q.T * q.V <= BN_MAXJ * BN_THREADS_MAX || bn_bwd_plan(q, sw).fast());
}

static BnBwdPlan bn_bwd_plan(const BnBwdP& q, const Switches& sw) {
  BnBwdPlan p;
  const size_t tv = (size_t)q.T * q.V * sizeof(float);
  p.g = bn_geom(q.T, q.V);
  p.use_r = q.r.p && q.prelu;
  p.add = q.gadd.p != nullptr;
  p.nst = p.use_r ? 3 : 2;                             // staged tensors: gout, y (, r); two pipeline stages
  p.nst2 = p.nst + (p.add ? 1 : 0);                    // pass 2 also stages gr_add
  const bool has_gr = q.gr.p != nullptr;
  const bool combo = p.use_r ? has_gr : (!has_gr && !p.add);     // the instantiations the model uses
  const bool gr_same = !has_gr || t_fastest(q.gr) == t_fastest(q.gy);
  p.fp = (combo && gr_same) ? bnf_plan(sw.bn_fast, q.C, q.T, q.V, q.mask, {&q.y, &q.r, &q.gout, &q.gy, &q.gr, &q.gadd})
                            : BnFastPlan{false, 0, 0, 0, false, false};
  p.u1 = p.fp.ok ? bnf_pick_u((size_t)p.fp.ch * tv, p.nst, p.fp.big, p.fp.wide) : 0;
  p.u2 = p.fp.ok ? bnf_pick_u((size_t)p.fp.ch * tv, p.nst2, p.fp.big, p.fp.wide) : 0;
  p.ub = bn_pick_u(tv, 2 * p.nst + 1, 4, BN_SMEM_BUDGET);
  p.ub2 = bn_pick_u(tv, 2 * p.nst2 + 1, p.ub, BN_SMEM_BUDGET);
  return p;
}

// pass 1 (per-split partial sums); the fast path's or the generic kernel, as planned
static int bn_bwd_reduce(const BnBwdP& q, const BnBwdPlan& p, cudaStream_t st) {
  const size_t tv = (size_t)q.T * q.V * sizeof(float);
  if (p.fast()) {
    const dim3 grid(q.C / p.fp.ch, q.S);
    int* err = device_error_word();
    const size_t smem = (size_t)2 * p.nst * p.u1 * p.fp.ch * tv;
    return with_bnf(p.fp, p.u1, [&](auto NJ, auto U, auto BIG) {
      const auto k = p.use_r ? (p.fp.wide ? bnf_bwd_reduce_wide_kernel<NJ, U, true, BIG> : bnf_bwd_reduce_kernel<NJ, U, true, BIG>)
                             : (p.fp.wide ? bnf_bwd_reduce_wide_kernel<NJ, U, false, BIG> : bnf_bwd_reduce_kernel<NJ, U, false, BIG>);
      return bn_launch(k, grid, p.fp.threads, smem, st, "bnf_bwd_reduce", q, p.fp.ch, err);
    });
  }
  size_t sm_red = (size_t)2 * p.nst * p.ub * tv;
  if (sm_red < 2 * tv) sm_red = 2 * tv;
  return with_nj(p.g.nj, [&](auto NJ) {   // any V
    return with_u(p.ub, [&](auto U) {
      return bn_launch(bn_bwd_reduce_kernel<NJ, U>, dim3(q.C, q.S), p.g.threads, sm_red, st, "bn_bwd_reduce", q);
    });
  });
}

// pass 2 (gy, gr; the plain call also the parameter gradients).  all == nullptr: the plain kernels, k1 / k2 from this
// call's own partial sums; otherwise the synchronised twins, k1 / k2 from the `world` gathered exchange rows.
static int bn_bwd_apply(const BnBwdP& q, const BnBwdPlan& p, const double* all, int world, cudaStream_t st) {
  const size_t tv = (size_t)q.T * q.V * sizeof(float);
  if (p.fast()) {
    const dim3 grid(q.C / p.fp.ch, q.S);
    int* err = device_error_word();
    const int np = (int)(grid.x * grid.y);
    const size_t smem2 = (size_t)2 * p.nst2 * p.u2 * p.fp.ch * tv;
    // the instantiations the model uses: (USE_R, HAS_GR, ADD) = (1, 1, 1), (1, 1, 0) or (0, 0, 0)
    return with_bnf(p.fp, p.u2, [&](auto NJ, auto U, auto BIG) {
      if (!all) {
        const auto k = p.use_r && p.add ? (p.fp.wide ? bnf_bwd_apply_wide_kernel<NJ, U, true, true, true, BIG>
                                                     : bnf_bwd_apply_kernel<NJ, U, true, true, true, BIG>)
                       : p.use_r        ? (p.fp.wide ? bnf_bwd_apply_wide_kernel<NJ, U, true, true, false, BIG>
                                                     : bnf_bwd_apply_kernel<NJ, U, true, true, false, BIG>)
                                        : (p.fp.wide ? bnf_bwd_apply_wide_kernel<NJ, U, false, false, false, BIG>
                                                     : bnf_bwd_apply_kernel<NJ, U, false, false, false, BIG>);
        return bn_launch(k, grid, p.fp.threads, smem2, st, "bnf_bwd_apply", q, p.fp.ch, np, err);
      }
      const auto k = p.use_r && p.add ? (p.fp.wide ? bnf_bwd_apply_sync_wide_kernel<NJ, U, true, true, true, BIG>
                                                   : bnf_bwd_apply_sync_kernel<NJ, U, true, true, true, BIG>)
                     : p.use_r        ? (p.fp.wide ? bnf_bwd_apply_sync_wide_kernel<NJ, U, true, true, false, BIG>
                                                   : bnf_bwd_apply_sync_kernel<NJ, U, true, true, false, BIG>)
                                      : (p.fp.wide ? bnf_bwd_apply_sync_wide_kernel<NJ, U, false, false, false, BIG>
                                                   : bnf_bwd_apply_sync_kernel<NJ, U, false, false, false, BIG>);
      return bn_launch(k, grid, p.fp.threads, smem2, st, "bnf_bwd_apply", q, p.fp.ch, err, all, world);
    });
  }
  const size_t sm2 = (size_t)(2 * p.nst2 + 1) * p.ub2 * tv;
  const dim3 grid(q.C, q.S);
  const bool wide = q.V > 32, add = q.gadd.p != nullptr;
  return with_nj(p.g.nj, [&](auto NJ) {
    return with_u(p.ub2, [&](auto U) {
      if (!all) {
        const auto k = add ? (wide ? bn_bwd_apply_add_wide_kernel<NJ, U> : bn_bwd_apply_add_kernel<NJ, U>)
                           : (wide ? bn_bwd_apply_wide_kernel<NJ, U> : bn_bwd_apply_kernel<NJ, U>);
        return bn_launch(k, grid, p.g.threads, sm2, st, "bn_bwd_apply", q);
      }
      const auto k = add ? (wide ? bn_bwd_apply_add_sync_wide_kernel<NJ, U> : bn_bwd_apply_add_sync_kernel<NJ, U>)
                         : (wide ? bn_bwd_apply_sync_wide_kernel<NJ, U> : bn_bwd_apply_sync_kernel<NJ, U>);
      return bn_launch(k, grid, p.g.threads, sm2, st, "bn_bwd_apply", q, all, world);
    });
  });
}

extern "C" int dstd_bn_act_backward(const dstd_bn_act_bwd_args* a, dstd_stream_t stream) {
  const Switches sw = read_switches();
  cudaStream_t st = (cudaStream_t)stream;
  BnBwdP q;
  int rc = bn_bwd_setup(a, sw, q);
  if (rc != DSTD_OK) return rc;
  const BnBwdPlan p = bn_bwd_plan(q, sw);
  rc = bn_bwd_reduce(q, p, st);
  if (rc != DSTD_OK) return rc;
  return bn_bwd_apply(q, p, nullptr, 0, st);
}

extern "C" int dstd_bn_act_backward_local(const dstd_bn_act_bwd_args* a, double* mine, dstd_stream_t stream) {
  DSTD_REQUIRE(a && a->training == 1, DSTD_ERR_BAD_ARG, "bn_act_backward_local: needs training = 1");
  DSTD_REQUIRE(mine, DSTD_ERR_BAD_ARG, "bn_act_backward_local: null exchange buffer");
  const Switches sw = read_switches();
  cudaStream_t st = (cudaStream_t)stream;
  BnBwdP q;
  int rc = bn_bwd_setup(a, sw, q, BN_LOCAL);
  if (rc != DSTD_OK) return rc;
  const BnBwdPlan p = bn_bwd_plan(q, sw);
  rc = bn_bwd_reduce(q, p, st);
  if (rc != DSTD_OK) return rc;
  // the block size and slope-partial count of the apply kernel the plain call would run: same gprelu summation order
  const int threads = p.fast() ? p.fp.threads : p.g.threads;
  const int np = p.fast() ? (q.C / p.fp.ch) * q.S : q.S * q.C;
  if (q.V > 32) bn_sync_fold_bwd_wide_kernel<<<q.C, threads, 0, st>>>(q, np, mine);
  else bn_sync_fold_bwd_kernel<<<q.C, threads, 0, st>>>(q, np, mine);
  count_launch();
  DSTD_LAUNCH_CHECK("bn_sync_fold_bwd");
  return DSTD_OK;
}

extern "C" int dstd_bn_act_backward_global(const dstd_bn_act_bwd_args* a, const double* all, int world,
                                           dstd_stream_t stream) {
  DSTD_REQUIRE(a && a->training == 1, DSTD_ERR_BAD_ARG, "bn_act_backward_global: needs training = 1");
  DSTD_REQUIRE(all && world >= 1, DSTD_ERR_BAD_ARG, "bn_act_backward_global: null exchange buffer or world < 1");
  const Switches sw = read_switches();
  cudaStream_t st = (cudaStream_t)stream;
  BnBwdP q;
  int rc = bn_bwd_setup(a, sw, q, BN_GLOBAL);
  if (rc != DSTD_OK) return rc;
  return bn_bwd_apply(q, bn_bwd_plan(q, sw), all, world, st);
}
