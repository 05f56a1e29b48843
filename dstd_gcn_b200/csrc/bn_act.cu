// Fused BatchNorm(C*V channels, statistics over N,T) + residual + PReLU + dropout mask, forward and backward
// (model/dstdgcn.py:44-50 BatchNorm.forward, :152-154 `x = bn(x); x += r; x = prelu(x)`, :306-308, :283-284).
//
// Work decomposition shared by all four kernels: CTA = (channel c, batch split s); a thread owns up to MAXJ fixed
// (t,v) positions of the T x V plane and walks the samples of its split, so the per-(c,v) BN parameters are
// per-thread constants and every access to a [T x V] plane is one contiguous, coalesced sweep.  When the producer and
// the consumer keep the plane in different memory orders (T-major vs V-major: this op is where the block switches
// between the spatial and the temporal unit layout) the plane is transposed through shared memory.
//
// Statistics use shifted sums (shift = y[0,c,0,v]) accumulated in fp32 per thread and combined in fp64, so the
// E[x^2]-E[x]^2 cancellation does not bite on millimetre-scale poses.
#include <initializer_list>

#include "kernels.cuh"
#include "umma.cuh"

namespace dstd {

constexpr int BN_THREADS_MAX = 512;
constexpr int BN_MAXJ = 8;       // positions per thread  -> T*V <= 4096
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
__device__ __forceinline__ bool t_fastest(const View4& vw) { return !(vw.sk == 1 || vw.sp != 1); }
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
// how a [T x V] plane of `w` can be copied: 2 = dense and every plane 8-byte aligned, 1 = dense, 0 = generic strides
__device__ __forceinline__ int plane_mode(const View4& w, int T, int V) {
  const bool dense = t_fastest(w) ? (w.sp == 1 && w.sk == T) : (w.sk == 1 && w.sp == V);
  if (!dense) return 0;
  const bool al8 = ((reinterpret_cast<unsigned long long>(w.p) & 7ull) == 0) && !((w.sn | w.sc) & 1ll) && !((T * V) & 1);
  return al8 ? 2 : 1;
}
// slot of logical (t, v) in a plane staged in w's memory order
__device__ __forceinline__ int slot_of(bool tfast, int t, int v, int T, int V) { return tfast ? v * T + t : t * V + v; }

// cp.async samples n .. n+U-1 (`left` of them exist) of channel plane c of `w` into the [U][T*V] region at shared
// address `sdst`, each plane in w's own memory order
template <int NJ, int U, bool FULL>
__device__ __forceinline__ void stage_async(const Pos2<NJ>& ps, const View4& w, int mode, int c, int n, int left,
                                            unsigned sdst, int T, int V) {
  const int TV = T * V;
  const float* base = w.p + (long long)n * w.sn + (long long)c * w.sc;
  if (mode == 2) {
    // the launch geometry gives NJ * blockDim >= T*V, so for NJ <= 2 a thread owns at most one pair of positions
    for (int j = 2 * threadIdx.x; j < TV; j += 2 * blockDim.x) {
      const float* p = base + j;
      unsigned d = sdst + (unsigned)j * 4u;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (FULL || u < left) cp_async8_s(d, p);
        p += w.sn;
        d += (unsigned)TV * 4u;
      }
      if (NJ <= 2) break;
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

// backward kernels: same copy, plane mode derived at the call (they sit at the 64-register cap and measured slower
// with the hoisted mode / single-pair form of the forward)
template <int NJ, int U, bool FULL>
__device__ __forceinline__ void stage_async_b(const Pos2<NJ>& ps, const View4& w, int c, int n, int left, unsigned sdst,
                                              int T, int V) {
  const int TV = T * V, mode = plane_mode(w, T, V);
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

// ------------------------------------------------------------------------------------------ forward: statistics
template <int NJ>
__global__ void __launch_bounds__(BN_THREADS_MAX) bn_stats_kernel(BnFwdP q) {
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
  if (threadIdx.x < V) {
    int v = threadIdx.x;
    double s1 = 0., s2 = 0.;
    for (int t = 0; t < T; ++t) {
      s1 += sh[t * V + v];
      s2 += sh[TV + t * V + v];
    }
    float* dst = q.part + (((long long)s * q.C + c) * V + v) * 2;
    dst[0] = (float)s1;
    dst[1] = (float)s2;
  }
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

template <int NJ, int U>
__global__ void __launch_bounds__(BN_THREADS_MAX, 2) bn_apply_kernel(BnFwdP q) {
  extern __shared__ float sh[];   // [2 stages][nst = 1 (y) or 2 (y, r)][U][T*V]
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
      stage_async<NJ, U, true>(ps, q.y, mode_y, c, n, left, d, T, V);
      if (has_r) stage_async<NJ, U, true>(ps, q.r, mode_r, c, n, left, d + (unsigned)(U * TV) * 4u, T, V);
    } else {
      stage_async<NJ, U, false>(ps, q.y, mode_y, c, n, left, d, T, V);
      if (has_r) stage_async<NJ, U, false>(ps, q.r, mode_r, c, n, left, d + (unsigned)(U * TV) * 4u, T, V);
    }
  };
  if (iters > 0) issue(0);
  cp_async_commit();
  __shared__ double tot[32][2];
  __shared__ float st_mean[32], st_is[32];
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

// ------------------------------------------------------------------------------------------ backward
struct BnBwdP {
  int N, C, T, V, vc_order, training, S;
  View4 y, r, gout, gy, gr, gadd;
  const float *gamma, *beta, *prelu, *mask, *save_mean, *save_invstd;
  float *ggamma, *gbeta, *gprelu;
  float* part;    // [S][C][V][2]
  float* part_p;  // [S][C]
};

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
      stage_async_b<NJ, U, true>(ps, q.gout, c, n, left, d, T, V);
      stage_async_b<NJ, U, true>(ps, q.y, c, n, left, d + du, T, V);
      if (use_r) stage_async_b<NJ, U, true>(ps, q.r, c, n, left, d + 2 * du, T, V);
    } else {
      stage_async_b<NJ, U, false>(ps, q.gout, c, n, left, d, T, V);
      stage_async_b<NJ, U, false>(ps, q.y, c, n, left, d + du, T, V);
      if (use_r) stage_async_b<NJ, U, false>(ps, q.r, c, n, left, d + 2 * du, T, V);
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
  if (threadIdx.x < V) {
    int v = threadIdx.x;
    double s1 = 0., s2 = 0.;
    for (int t = 0; t < T; ++t) {
      s1 += sh[t * V + v];
      s2 += sh[TV + t * V + v];
    }
    float* dst = q.part + (((long long)s * q.C + c) * V + v) * 2;
    dst[0] = (float)s1;
    dst[1] = (float)s2;
  }
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

template <int NJ, int U, bool ADD>
__device__ __forceinline__ void bn_bwd_apply_body(const BnBwdP& q) {
  extern __shared__ float sh[];   // [2 stages][nst = 2 (gout, y), + r, + gr_add][U][T*V], then [U][T*V] for gr
  const int c = blockIdx.x, s = blockIdx.y, T = q.T, V = q.V, TV = T * V;
  const int n0 = (int)((long long)q.N * s / q.S), n1 = (int)((long long)q.N * (s + 1) / q.S), cnt = n1 - n0;
  const bool has_prelu = q.prelu != nullptr;
  const bool use_r = q.r.p && has_prelu;
  const bool has_gr = q.gr.p != nullptr;
  const float slope = has_prelu ? __ldg(q.prelu) : 1.f;
  const float icnt = 1.0f / ((float)q.N * (float)T);
  const bool has_add = ADD;       // the host launches the ADD instantiation only with gr and gr_add present
  const int add_region = has_add ? (use_r ? 3 : 2) : -1;          // staged planes: gout, y, (r), (gr_add)
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
      stage_async_b<NJ, U, true>(ps, q.gout, c, n, left, d, T, V);
      stage_async_b<NJ, U, true>(ps, q.y, c, n, left, d + du, T, V);
      if (use_r) stage_async_b<NJ, U, true>(ps, q.r, c, n, left, d + 2 * du, T, V);
      if (has_add) stage_async_b<NJ, U, true>(ps, q.gadd, c, n, left, d + add_region * du, T, V);
    } else {
      stage_async_b<NJ, U, false>(ps, q.gout, c, n, left, d, T, V);
      stage_async_b<NJ, U, false>(ps, q.y, c, n, left, d + du, T, V);
      if (use_r) stage_async_b<NJ, U, false>(ps, q.r, c, n, left, d + 2 * du, T, V);
      if (has_add) stage_async_b<NJ, U, false>(ps, q.gadd, c, n, left, d + add_region * du, T, V);
    }
  };
  if (iters > 0) issue(0);
  cp_async_commit();
  // sums of pass 1 over the splits; the s == 0 CTA of the channel publishes the parameter gradients
  __shared__ double tot[32][2];
  __shared__ float red[32];
  sum_partials(q.part, q.S, q.C, c, V, tot);
  if (c == 0 && s == 0 && q.gprelu) {   // fixed-order sum of the slope partials
    float a = 0.f;
    for (int i = threadIdx.x; i < q.S * q.C; i += blockDim.x) a += q.part_p[i];
    const float t = block_sum(a, red);
    if (threadIdx.x == 0) q.gprelu[0] = t;
  }
  __syncthreads();
  if (s == 0 && threadIdx.x < V) {
    const int pi = bn_pidx(c, threadIdx.x, q.C, V, q.vc_order);
    q.gbeta[pi] = (float)tot[threadIdx.x][0];
    q.ggamma[pi] = (float)tot[threadIdx.x][1];
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
        if (q.training) {
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
  bn_bwd_apply_body<NJ, U, false>(q);
}
// same with a fourth staged tensor, gr_add, summed into gr (separate instantiation: the plain kernel sits at the
// 64-register cap and pays ~13 % for the extra slots)
template <int NJ, int U>
__global__ void __launch_bounds__(BN_THREADS_MAX, 2) bn_bwd_apply_add_kernel(BnBwdP q) {
  bn_bwd_apply_body<NJ, U, true>(q);
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
template <bool BIG> struct BnfBits { static constexpr int SB = BIG ? 13 : 12; static constexpr uint32_t SM = (1u << SB) - 1u; };

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

// ---- forward apply: positions in out's memory order
template <int NJ, int U, bool HAS_R, bool FULL, bool BIG>
__device__ __forceinline__ void bnf_apply_consume(const float* st, const float4* ctab, const uint32_t (&pk)[NJ], float* ob,
                                                  long long osn, int CHTV, int left, float slope) {
#pragma unroll
  for (int i = 0; i < NJ; ++i) {
    if ((int)(threadIdx.x + i * blockDim.x) < CHTV) {
      constexpr int SB = BnfBits<BIG>::SB;
      constexpr uint32_t SM = BnfBits<BIG>::SM;
      const float4 k = ctab[pk[i] >> (2 * SB)];
      const float* py = st + (pk[i] & SM);
      const float* pr = st + U * CHTV + ((pk[i] >> SB) & SM);
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

template <int NJ, int U, bool HAS_R, bool BIG>
__global__ void __launch_bounds__(BIG ? BNF_THREADS_BIG : BN_THREADS_MAX, BIG ? 1 : 2) bnf_apply_kernel(BnFwdP q, int CH, int* err) {
  extern __shared__ __align__(16) float sh[];   // [2 stages][y (, r)][U][CH * T*V]
  __shared__ __align__(16) float4 ctab[BNF_MAXCH * 32];     // per (ch, v): mean, gamma * invstd, beta
  __shared__ double tot[32][2];
  __shared__ __align__(8) uint64_t mbar[2];
  const int c0 = blockIdx.x * CH, s = blockIdx.y, T = q.T, V = q.V, TV = T * V, CHTV = CH * TV;
  const int n0 = (int)((long long)q.N * s / gridDim.y), n1 = (int)((long long)q.N * (s + 1) / gridDim.y), cnt = n1 - n0;
  constexpr int NST = HAS_R ? 2 : 1;
  const int stage_f = NST * U * CHTV, iters = (cnt + U - 1) / U;
  const float slope = q.prelu ? __ldg(q.prelu) : 1.f;
  if (threadIdx.x == 0) {
    umma::mbar_init(&mbar[0], 1);
    umma::mbar_init(&mbar[1], 1);
    umma::mbar_init_fence();
  }
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
        ctab[ch * 32 + v] = make_float4(fm, __ldg(q.gamma + pi) * fi, __ldg(q.beta + pi), 0.f);
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
    if (threadIdx.x < CH * 32 && (threadIdx.x & 31) < V) {
      const int pi = bn_pidx(c0 + (threadIdx.x >> 5), threadIdx.x & 31, q.C, V, q.vc_order);
      ctab[threadIdx.x] = make_float4(q.save_mean[pi], __ldg(q.gamma + pi) * q.save_invstd[pi], __ldg(q.beta + pi), 0.f);
    }
    __syncthreads();
  }
  uint32_t pk[NJ];   // slot in y's slab | slot in r's slab << SB | (ch * 32 + v) << 2 SB   (valid iff j < CHTV)
  {
    constexpr int SB = BnfBits<BIG>::SB;
    const bool tf_o = t_fastest(q.out), tf_y = t_fastest(q.y), tf_r = HAS_R && t_fastest(q.r);
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
      const int j = threadIdx.x + i * blockDim.x;
      pk[i] = 0u;
      if (j < CHTV) {
        int ch, t, v;
        bnf_decode(tf_o, j, T, V, TV, ch, t, v);
        pk[i] = (uint32_t)(ch * TV + slot_of(tf_y, t, v, T, V)) | ((uint32_t)(ch * TV + slot_of(tf_r, t, v, T, V)) << SB) |
                ((uint32_t)(ch * 32 + v) << (2 * SB));
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
    if (left >= U) bnf_apply_consume<NJ, U, HAS_R, true, BIG>(st, ctab, pk, ob, osn, CHTV, left, slope);
    else bnf_apply_consume<NJ, U, HAS_R, false, BIG>(st, ctab, pk, ob, osn, CHTV, left, slope);
    ob += U * osn;
    __syncthreads();
  }
}

// ---- backward pass 1: positions in y's memory order
template <int NJ, int U, bool USE_R, bool FULL, bool BIG>
__device__ __forceinline__ void bnf_reduce_consume(const float* st, const float4* ctab, const uint32_t (&pk)[NJ], int CHTV,
                                                   int left, float slope, bool has_prelu, float (&a1)[NJ],
                                                   float (&a2)[NJ], float& gsl) {
#pragma unroll
  for (int i = 0; i < NJ; ++i) {
    if ((int)(threadIdx.x + i * blockDim.x) < CHTV) {
      constexpr int SB = BnfBits<BIG>::SB;
      constexpr uint32_t SM = BnfBits<BIG>::SM;
      const float4 k = ctab[pk[i] >> (2 * SB)];
      const float* pg = st + (pk[i] & SM);
      const float* py = st + U * CHTV + threadIdx.x + i * blockDim.x;
      const float* pr = st + 2 * U * CHTV + ((pk[i] >> SB) & SM);
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

template <int NJ, int U, bool USE_R, bool BIG>
__global__ void __launch_bounds__(BIG ? BNF_THREADS_BIG : BN_THREADS_MAX, BIG ? 1 : 2) bnf_bwd_reduce_kernel(BnBwdP q, int CH, int* err) {
  extern __shared__ __align__(16) float sh[];   // [2 stages][gout, y (, r)][U][CH * T*V]
  __shared__ __align__(16) float4 ctab[BNF_MAXCH * 32];     // per (ch, v): mean, invstd, gamma, beta
  __shared__ float red[32];
  __shared__ __align__(8) uint64_t mbar[2];
  const int c0 = blockIdx.x * CH, s = blockIdx.y, T = q.T, V = q.V, TV = T * V, CHTV = CH * TV;
  const int n0 = (int)((long long)q.N * s / gridDim.y), n1 = (int)((long long)q.N * (s + 1) / gridDim.y), cnt = n1 - n0;
  constexpr int NST = USE_R ? 3 : 2;
  const int stage_f = NST * U * CHTV, iters = (cnt + U - 1) / U;
  const bool has_prelu = q.prelu != nullptr;
  const float slope = has_prelu ? __ldg(q.prelu) : 1.f;
  if (threadIdx.x == 0) {
    umma::mbar_init(&mbar[0], 1);
    umma::mbar_init(&mbar[1], 1);
    umma::mbar_init_fence();
  }
  if (threadIdx.x < CH * 32 && (threadIdx.x & 31) < V) {
    const int pi = bn_pidx(c0 + (threadIdx.x >> 5), threadIdx.x & 31, q.C, V, q.vc_order);
    ctab[threadIdx.x] = make_float4(__ldg(q.save_mean + pi), __ldg(q.save_invstd + pi), __ldg(q.gamma + pi), __ldg(q.beta + pi));
  }
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
  uint32_t pk[NJ];   // slot in gout's slab | slot in r's slab << SB | (ch * 32 + v) << 2 SB;  y is read at j itself
  float a1[NJ], a2[NJ], gsl = 0.f;
  const bool tf_y = t_fastest(q.y);
  {
    constexpr int SB = BnfBits<BIG>::SB;
    const bool tf_g = t_fastest(q.gout), tf_r = USE_R && t_fastest(q.r);
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
      const int j = threadIdx.x + i * blockDim.x;
      pk[i] = 0u;
      a1[i] = a2[i] = 0.f;
      if (j < CHTV) {
        int ch, t, v;
        bnf_decode(tf_y, j, T, V, TV, ch, t, v);
        pk[i] = (uint32_t)(ch * TV + slot_of(tf_g, t, v, T, V)) | ((uint32_t)(ch * TV + slot_of(tf_r, t, v, T, V)) << SB) |
                ((uint32_t)(ch * 32 + v) << (2 * SB));
      }
    }
  }
  for (int it = 0; it < iters; ++it) {
    if (threadIdx.x == 0 && it + 1 < iters) issue(it + 1);
    if (!umma::mbar_wait(&mbar[it & 1], (uint32_t)(it >> 1) & 1u)) bnf_timeout(err);
    const float* st = sh + (it & 1) * stage_f;
    const int left = n1 - (n0 + it * U);
    if (left >= U) bnf_reduce_consume<NJ, U, USE_R, true, BIG>(st, ctab, pk, CHTV, left, slope, has_prelu, a1, a2, gsl);
    else bnf_reduce_consume<NJ, U, USE_R, false, BIG>(st, ctab, pk, CHTV, left, slope, has_prelu, a1, a2, gsl);
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

// ---- backward pass 2: positions in gy's memory order; gr (same order as gy) is stored straight from registers
template <int NJ, int U, bool USE_R, bool HAS_GR, bool ADD, bool FULL, bool BIG>
__device__ __forceinline__ void bnf_bwd_apply_consume(const float* st, const float4* ctab, const float4* ctab2,
                                                      const uint32_t (&pk)[NJ], const uint32_t (&pk2)[NJ], float* gyb, float* grb,
                                                      long long gysn, long long grsn, int CHTV, int left, float slope,
                                                      bool has_prelu) {
  constexpr int ADD_REGION = USE_R ? 3 : 2;
#pragma unroll
  for (int i = 0; i < NJ; ++i) {
    if ((int)(threadIdx.x + i * blockDim.x) < CHTV) {
      constexpr int SB = BnfBits<BIG>::SB;
      constexpr uint32_t SM = BnfBits<BIG>::SM;
      const float4 k = ctab[pk[i] >> (2 * SB)], k2 = ctab2[pk[i] >> (2 * SB)];
      const float* pg = st + (pk[i] & SM);
      const float* py = st + U * CHTV + ((pk[i] >> SB) & SM);
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

template <int NJ, int U, bool USE_R, bool HAS_GR, bool ADD, bool BIG>
__global__ void __launch_bounds__(BIG ? BNF_THREADS_BIG : BN_THREADS_MAX, BIG ? 1 : 2) bnf_bwd_apply_kernel(BnBwdP q, int CH, int NP, int* err) {
  extern __shared__ __align__(16) float sh[];   // [2 stages][gout, y (, r) (, gr_add)][U][CH * T*V]
  __shared__ __align__(16) float4 ctab[BNF_MAXCH * 32];     // mean, invstd, gamma, beta
  __shared__ __align__(16) float4 ctab2[BNF_MAXCH * 32];    // gamma * invstd, k1, k2
  __shared__ double tot[32][2];
  __shared__ float red[32];
  __shared__ __align__(8) uint64_t mbar[2];
  const int c0 = blockIdx.x * CH, s = blockIdx.y, T = q.T, V = q.V, TV = T * V, CHTV = CH * TV;
  const int n0 = (int)((long long)q.N * s / gridDim.y), n1 = (int)((long long)q.N * (s + 1) / gridDim.y), cnt = n1 - n0;
  constexpr int NST = 2 + (USE_R ? 1 : 0) + (ADD ? 1 : 0), ADD_REGION = USE_R ? 3 : 2;
  const int stage_f = NST * U * CHTV, iters = (cnt + U - 1) / U;
  const bool has_prelu = q.prelu != nullptr;
  const float slope = has_prelu ? __ldg(q.prelu) : 1.f;
  const float icnt = 1.0f / ((float)q.N * (float)T);
  if (threadIdx.x == 0) {
    umma::mbar_init(&mbar[0], 1);
    umma::mbar_init(&mbar[1], 1);
    umma::mbar_init_fence();
  }
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
  if (blockIdx.x == 0 && s == 0 && q.gprelu) {   // fixed-order sum of the slope partials
    float a = 0.f;
    for (int i = threadIdx.x; i < NP; i += blockDim.x) a += q.part_p[i];
    const float t = block_sum(a, red);
    if (threadIdx.x == 0) q.gprelu[0] = t;
  }
  for (int ch = 0; ch < CH; ++ch) {
    const int c = c0 + ch;
    sum_partials(q.part, q.S, q.C, c, V, tot);
    __syncthreads();
    if (threadIdx.x < V) {
      const int v = threadIdx.x, pi = bn_pidx(c, v, q.C, V, q.vc_order);
      const float mu = __ldg(q.save_mean + pi), is = __ldg(q.save_invstd + pi), g = __ldg(q.gamma + pi);
      ctab[ch * 32 + v] = make_float4(mu, is, g, __ldg(q.beta + pi));
      ctab2[ch * 32 + v] = make_float4(g * is, q.training ? (float)tot[v][0] * icnt : 0.f,
                                       q.training ? (float)tot[v][1] * icnt : 0.f, 0.f);
      if (s == 0) {
        q.gbeta[pi] = (float)tot[v][0];
        q.ggamma[pi] = (float)tot[v][1];
      }
    }
    __syncthreads();
  }
  uint32_t pk[NJ], pk2[NJ];   // gout slot | y slot << SB | (ch*32+v) << 2 SB;   r slot | gr_add slot << SB
  {
    constexpr int SB = BnfBits<BIG>::SB;
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
        pk[i] = (uint32_t)(ch * TV + slot_of(tf_g, t, v, T, V)) | ((uint32_t)(ch * TV + slot_of(tf_y, t, v, T, V)) << SB) |
                ((uint32_t)(ch * 32 + v) << (2 * SB));
        pk2[i] = (uint32_t)(ch * TV + slot_of(tf_r, t, v, T, V)) | ((uint32_t)(ch * TV + slot_of(tf_a, t, v, T, V)) << SB);
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
      bnf_bwd_apply_consume<NJ, U, USE_R, HAS_GR, ADD, true, BIG>(st, ctab, ctab2, pk, pk2, gyb, grb, gysn, grsn, CHTV, left, slope, has_prelu);
    else
      bnf_bwd_apply_consume<NJ, U, USE_R, HAS_GR, ADD, false, BIG>(st, ctab, ctab2, pk, pk2, gyb, grb, gysn, grsn, CHTV, left, slope, has_prelu);
    gyb += U * gysn;
    if (HAS_GR) grb += U * grsn;
    __syncthreads();
  }
}

// host side of the fast path
struct BnFastPlan {
  bool ok;
  int ch, nj, threads;
  bool big;     // slab of 4097 .. 8192 positions: BIG instantiations (<= 1024 threads, one CTA per SM)
};
static bool bnf_tfast(const View4& w) { return !(w.sk == 1 || w.sp != 1); }
static bool bnf_slab_ok(const View4& w, int T, int V) {
  if (!w.p) return true;
  const bool dense = bnf_tfast(w) ? (w.sp == 1 && w.sk == T) : (w.sk == 1 && w.sp == V);
  return dense && w.sc == (long long)T * V && (reinterpret_cast<unsigned long long>(w.p) & 15ull) == 0 && (w.sn & 3ll) == 0;
}
static BnFastPlan bnf_plan(bool fast, int C, int T, int V, const float* mask, std::initializer_list<const View4*> ws) {
  BnFastPlan pl{false, 0, 0, 0, false};
  if (!fast || mask || V > 32) return pl;
  const int TV = T * V;
  pl.ch = (TV % 4 == 0) ? 1 : (TV % 2 == 0) ? 2 : 4;
  const int chtv = pl.ch * TV;
  pl.big = chtv > 4096;
  if (C % pl.ch || chtv > 8 * BNF_THREADS_BIG || (pl.big && pl.ch > 2)) return pl;
  for (const View4* w : ws)
    if (!bnf_slab_ok(*w, T, V)) return pl;
  pl.nj = chtv <= 4 * BN_THREADS_MAX ? 4 : 8;
  pl.threads = cdiv(cdiv(chtv, pl.nj), 32) * 32;
  pl.ok = true;
  return pl;
}
// samples per stage: the largest of 4/2/1 whose two stages of `nst` slabs fit two CTAs per SM; 0 = none
static int bnf_pick_u(size_t slab_bytes, int nst, bool big = false) {
  const size_t budget = big ? (size_t)220 * 1024 : BN_SMEM_BUDGET;   // BIG: one CTA per SM
  for (int u = big ? 2 : 4; u >= 1; u >>= 1)
    if ((size_t)2 * nst * u * slab_bytes <= budget) return u;
  return 0;
}

#define DSTD_BNF_ONE(KERN, NJ_, U_, BIG_, grid, threads, smem, st, ...)                               \
  do {                                                                                                \
    prefer_smem_carveout((const void*)KERN(NJ_, U_, BIG_), true);                                     \
    KERN(NJ_, U_, BIG_)<<<grid, threads, smem, st>>>(__VA_ARGS__);                                    \
  } while (0)
#define DSTD_BNF_U(KERN, NJ_, u, grid, threads, smem, st, ...)                                        \
  do {                                                                                                \
    switch (u) {                                                                                      \
      case 4: DSTD_BNF_ONE(KERN, NJ_, 4, false, grid, threads, smem, st, __VA_ARGS__); break;         \
      case 2: DSTD_BNF_ONE(KERN, NJ_, 2, false, grid, threads, smem, st, __VA_ARGS__); break;         \
      default: DSTD_BNF_ONE(KERN, NJ_, 1, false, grid, threads, smem, st, __VA_ARGS__); break;        \
    }                                                                                                 \
  } while (0)
// plan: {nj, big}; BIG slabs always run 8 positions per thread, 2 or 1 samples per stage
#define DSTD_BNF(KERN, plan, u, grid, threads, smem, st, ...)                                         \
  do {                                                                                                \
    if ((plan).big) {                                                                                 \
      if ((u) == 2) DSTD_BNF_ONE(KERN, 8, 2, true, grid, threads, smem, st, __VA_ARGS__);             \
      else DSTD_BNF_ONE(KERN, 8, 1, true, grid, threads, smem, st, __VA_ARGS__);                      \
    } else if ((plan).nj == 4) DSTD_BNF_U(KERN, 4, u, grid, threads, smem, st, __VA_ARGS__);          \
    else DSTD_BNF_U(KERN, 8, u, grid, threads, smem, st, __VA_ARGS__);                                \
  } while (0)

// U (samples per pipeline stage) is a launch-time choice among the compiled instantiations
#define DSTD_BN_CASE(kern, NJ_, u, grid, threads, smem, st, q)                       \
  do {                                                                                \
    switch (u) {                                                                      \
      case 4:                                                                         \
        prefer_smem_carveout((const void*)kern<NJ_, 4>, true);                        \
        kern<NJ_, 4><<<grid, threads, smem, st>>>(q);                                 \
        break;                                                                        \
      case 2:                                                                         \
        prefer_smem_carveout((const void*)kern<NJ_, 2>, true);                        \
        kern<NJ_, 2><<<grid, threads, smem, st>>>(q);                                 \
        break;                                                                        \
      default:                                                                        \
        prefer_smem_carveout((const void*)kern<NJ_, 1>, true);                        \
        kern<NJ_, 1><<<grid, threads, smem, st>>>(q);                                 \
        break;                                                                        \
    }                                                                                 \
  } while (0)
#define DSTD_BN_DISPATCH_U(kern, nj, u, grid, threads, smem, st, q)                  \
  do {                                                                                \
    switch (nj) {                                                                     \
      case 1: DSTD_BN_CASE(kern, 1, u, grid, threads, smem, st, q); break;            \
      case 2: DSTD_BN_CASE(kern, 2, u, grid, threads, smem, st, q); break;            \
      case 4: DSTD_BN_CASE(kern, 4, u, grid, threads, smem, st, q); break;            \
      default: DSTD_BN_CASE(kern, 8, u, grid, threads, smem, st, q); break;           \
    }                                                                                 \
  } while (0)

#define DSTD_BN_DISPATCH(kern, nj, grid, threads, smem, st, q)          \
  do {                                                                  \
    switch (nj) {                                                       \
      case 1: kern<1><<<grid, threads, smem, st>>>(q); break;           \
      case 2: kern<2><<<grid, threads, smem, st>>>(q); break;           \
      case 4: kern<4><<<grid, threads, smem, st>>>(q); break;           \
      default: kern<8><<<grid, threads, smem, st>>>(q); break;          \
    }                                                                   \
  } while (0)

}  // namespace dstd

// =========================================================================================== C ABI
using namespace dstd;

extern "C" size_t dstd_bn_act_workspace_bytes(int N, int C, int T, int V) {
  int S = N > 128 ? 128 : N;   // upper bound of bn_act_splits
  if (S < 1) S = 1;
  return arena_need({(size_t)S * C * V * 2 * sizeof(float), (size_t)S * C * sizeof(float)});
}

extern "C" int dstd_bn_act_forward(const dstd_bn_act_fwd_args* a, dstd_stream_t stream) {
  DSTD_REQUIRE(a, DSTD_ERR_BAD_ARG, "bn_act_forward: null args");
  DSTD_REQUIRE(a->N > 0 && a->C > 0 && a->T > 0 && a->V > 0, DSTD_ERR_BAD_ARG, "bn_act_forward: bad dims");
  DSTD_REQUIRE(a->y.ptr && a->out.ptr && a->gamma && a->beta && a->save_mean && a->save_invstd, DSTD_ERR_BAD_ARG,
               "bn_act_forward: null tensor");
  DSTD_REQUIRE(a->T * a->V <= BN_MAXJ * BN_THREADS_MAX && a->V <= 32, DSTD_ERR_UNSUPPORTED,
               "bn_act: T*V=%d (max %d) or V=%d (max 32) outside the compiled limits", a->T * a->V,
               BN_MAXJ * BN_THREADS_MAX, a->V);
  DSTD_REQUIRE(a->training || (a->running_mean && a->running_var), DSTD_ERR_BAD_ARG,
               "bn_act_forward: eval mode needs running statistics");
  DSTD_REQUIRE(a->ws_bytes >= dstd_bn_act_workspace_bytes(a->N, a->C, a->T, a->V) && a->ws, DSTD_ERR_WORKSPACE,
               "bn_act_forward: workspace too small");
  const Switches sw = read_switches();
  cudaStream_t st = (cudaStream_t)stream;
  BnFwdP q;
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
  Arena ar(a->ws, a->ws_bytes);
  q.part = ar.take<float>((size_t)q.S * q.C * q.V * 2);
  BnGeom g = bn_geom(q.T, q.V);
  const size_t tvb = (size_t)q.T * q.V * sizeof(float);
  const size_t sm2 = 2 * tvb;
  const int nst = q.r.p ? 2 : 1;                       // staged tensors: y (, r); two pipeline stages
  const int u = bn_pick_u(tvb, 2 * nst, 4, BN_SMEM_BUDGET);
  const size_t smu = (size_t)2 * nst * u * tvb;
  const int cv = q.C * q.V;
  if (q.training) {
    DSTD_BN_DISPATCH(bn_stats_kernel, g.nj, dim3(q.C, q.S), g.threads, sm2, st, q);
    count_launch();
    DSTD_LAUNCH_CHECK("bn_stats");
  } else {
    bn_eval_stats_kernel<<<cdiv(cv, 128), 128, 0, st>>>(q);
    count_launch();
    DSTD_LAUNCH_CHECK("bn_eval_stats");
  }
  const BnFastPlan fp = bnf_plan(sw.bn_fast, q.C, q.T, q.V, q.mask, {&q.y, &q.r, &q.out});
  const int fu = fp.ok ? bnf_pick_u((size_t)fp.ch * tvb, nst, fp.big) : 0;
  if (fu) {   // bulk-copy staged kernel (see "fast path")
    const dim3 grid(q.C / fp.ch, q.S);
    const size_t smem = (size_t)2 * nst * fu * fp.ch * tvb;
    int* err = device_error_word();
#define DSTD_K_APPLY_R(NJ_, U_, B_) bnf_apply_kernel<NJ_, U_, true, B_>
#define DSTD_K_APPLY(NJ_, U_, B_) bnf_apply_kernel<NJ_, U_, false, B_>
    if (q.r.p) DSTD_BNF(DSTD_K_APPLY_R, fp, fu, grid, fp.threads, smem, st, q, fp.ch, err);
    else DSTD_BNF(DSTD_K_APPLY, fp, fu, grid, fp.threads, smem, st, q, fp.ch, err);
#undef DSTD_K_APPLY_R
#undef DSTD_K_APPLY
    count_launch();
    DSTD_LAUNCH_CHECK("bnf_apply");
    return DSTD_OK;
  }
  DSTD_BN_DISPATCH_U(bn_apply_kernel, g.nj, u, dim3(q.C, q.S), g.threads, smu, st, q);
  count_launch();
  DSTD_LAUNCH_CHECK("bn_apply");
  return DSTD_OK;
}

extern "C" int dstd_bn_act_backward(const dstd_bn_act_bwd_args* a, dstd_stream_t stream) {
  DSTD_REQUIRE(a, DSTD_ERR_BAD_ARG, "bn_act_backward: null args");
  DSTD_REQUIRE(a->N > 0 && a->C > 0 && a->T > 0 && a->V > 0, DSTD_ERR_BAD_ARG, "bn_act_backward: bad dims");
  DSTD_REQUIRE(a->y.ptr && a->gout.ptr && a->gy.ptr && a->gamma && a->beta && a->save_mean && a->save_invstd &&
                   a->ggamma && a->gbeta,
               DSTD_ERR_BAD_ARG, "bn_act_backward: null tensor");
  DSTD_REQUIRE(!a->gr.ptr || a->r.ptr, DSTD_ERR_BAD_ARG, "bn_act_backward: gr requested without r");
  DSTD_REQUIRE(!a->gr_add.ptr || a->gr.ptr, DSTD_ERR_BAD_ARG, "bn_act_backward: gr_add given without gr");
  DSTD_REQUIRE(a->T * a->V <= BN_MAXJ * BN_THREADS_MAX && a->V <= 32, DSTD_ERR_UNSUPPORTED,
               "bn_act: T*V=%d or V=%d outside the compiled limits", a->T * a->V, a->V);
  DSTD_REQUIRE(a->ws_bytes >= dstd_bn_act_workspace_bytes(a->N, a->C, a->T, a->V) && a->ws, DSTD_ERR_WORKSPACE,
               "bn_act_backward: workspace too small");
  const Switches sw = read_switches();
  cudaStream_t st = (cudaStream_t)stream;
  BnBwdP q;
  q.N = a->N; q.C = a->C; q.T = a->T; q.V = a->V;
  q.vc_order = a->vc_order; q.training = a->training;
  q.S = bn_act_splits(a->N, sw.bn_samples_per_cta);
  q.y = mk(a->y); q.r = mk(a->r); q.gout = mk(a->gout); q.gy = mk(a->gy); q.gr = mk(a->gr); q.gadd = mk(a->gr_add);
  q.gamma = a->gamma; q.beta = a->beta; q.prelu = a->prelu; q.mask = a->mask;
  q.save_mean = a->save_mean; q.save_invstd = a->save_invstd;
  q.ggamma = a->ggamma; q.gbeta = a->gbeta; q.gprelu = a->prelu ? a->gprelu : nullptr;
  Arena ar(a->ws, a->ws_bytes);
  q.part = ar.take<float>((size_t)q.S * q.C * q.V * 2);
  q.part_p = ar.take<float>((size_t)q.S * q.C);
  BnGeom g = bn_geom(q.T, q.V);
  const size_t tv = (size_t)q.T * q.V * sizeof(float);
  const int nst = (q.r.p && q.prelu) ? 3 : 2;          // staged tensors: gout, y (, r); two pipeline stages
  {
    const bool use_r = q.r.p && q.prelu, has_gr = q.gr.p != nullptr, add = q.gadd.p != nullptr;
    const bool combo = use_r ? has_gr : (!has_gr && !add);     // the instantiations the model uses
    const bool gr_same = !has_gr || bnf_tfast(q.gr) == bnf_tfast(q.gy);
    const BnFastPlan fp = (combo && gr_same) ? bnf_plan(sw.bn_fast, q.C, q.T, q.V, q.mask, {&q.y, &q.r, &q.gout, &q.gy, &q.gr, &q.gadd})
                                             : BnFastPlan{false, 0, 0, 0, false};
    const int u1 = fp.ok ? bnf_pick_u((size_t)fp.ch * tv, nst, fp.big) : 0;
    const int u2 = fp.ok ? bnf_pick_u((size_t)fp.ch * tv, nst + (add ? 1 : 0), fp.big) : 0;
    if (u1 && u2) {
      const dim3 grid(q.C / fp.ch, q.S);
      int* err = device_error_word();
#define DSTD_K_RED_R(NJ_, U_, B_) bnf_bwd_reduce_kernel<NJ_, U_, true, B_>
#define DSTD_K_RED(NJ_, U_, B_) bnf_bwd_reduce_kernel<NJ_, U_, false, B_>
      if (use_r) DSTD_BNF(DSTD_K_RED_R, fp, u1, grid, fp.threads, (size_t)2 * nst * u1 * fp.ch * tv, st, q, fp.ch, err);
      else DSTD_BNF(DSTD_K_RED, fp, u1, grid, fp.threads, (size_t)2 * nst * u1 * fp.ch * tv, st, q, fp.ch, err);
#undef DSTD_K_RED_R
#undef DSTD_K_RED
      count_launch();
      DSTD_LAUNCH_CHECK("bnf_bwd_reduce");
      const int np = (int)(grid.x * grid.y);
      const size_t smem2 = (size_t)2 * (nst + (add ? 1 : 0)) * u2 * fp.ch * tv;
#define DSTD_K_APP_RA(NJ_, U_, B_) bnf_bwd_apply_kernel<NJ_, U_, true, true, true, B_>
#define DSTD_K_APP_R(NJ_, U_, B_) bnf_bwd_apply_kernel<NJ_, U_, true, true, false, B_>
#define DSTD_K_APP(NJ_, U_, B_) bnf_bwd_apply_kernel<NJ_, U_, false, false, false, B_>
      if (use_r && add) DSTD_BNF(DSTD_K_APP_RA, fp, u2, grid, fp.threads, smem2, st, q, fp.ch, np, err);
      else if (use_r) DSTD_BNF(DSTD_K_APP_R, fp, u2, grid, fp.threads, smem2, st, q, fp.ch, np, err);
      else DSTD_BNF(DSTD_K_APP, fp, u2, grid, fp.threads, smem2, st, q, fp.ch, np, err);
#undef DSTD_K_APP_RA
#undef DSTD_K_APP_R
#undef DSTD_K_APP
      count_launch();
      DSTD_LAUNCH_CHECK("bnf_bwd_apply");
      return DSTD_OK;
    }
  }
  const int ub = bn_pick_u(tv, 2 * nst + 1, 4, BN_SMEM_BUDGET);
  size_t sm_red = (size_t)2 * nst * ub * tv;
  if (sm_red < 2 * tv) sm_red = 2 * tv;
  DSTD_BN_DISPATCH_U(bn_bwd_reduce_kernel, g.nj, ub, dim3(q.C, q.S), g.threads, sm_red, st, q);
  count_launch();
  DSTD_LAUNCH_CHECK("bn_bwd_reduce");
  const int nst2 = nst + (q.gadd.p ? 1 : 0);           // pass 2 also stages gr_add
  const int ub2 = bn_pick_u(tv, 2 * nst2 + 1, ub, BN_SMEM_BUDGET);
  if (q.gadd.p) {
    DSTD_BN_DISPATCH_U(bn_bwd_apply_add_kernel, g.nj, ub2, dim3(q.C, q.S), g.threads, (size_t)(2 * nst2 + 1) * ub2 * tv, st, q);
  } else {
    DSTD_BN_DISPATCH_U(bn_bwd_apply_kernel, g.nj, ub2, dim3(q.C, q.S), g.threads, (size_t)(2 * nst2 + 1) * ub2 * tv, st, q);
  }
  count_launch();
  DSTD_LAUNCH_CHECK("bn_bwd_apply");
  return DSTD_OK;
}
