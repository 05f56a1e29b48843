// Shape-generic kernels of the DSTD-GC unit for shapes outside the tile limits of the specialised kernels (P or K > 40):
// the stress configuration of BASELINE.json (T = 125 frames, 256 channels: spatial unit P = 125, K = 22; temporal unit
// P = 22, K = 125).  Same maths and the same buffers as dynadj.cu / aggregate.cu (model/dstdgcn.py:82-93 and its
// autograd, SURVEY.md Appendix A), CUDA cores, tiled through shared memory, every reduction in a fixed order
// (deterministic).  The pairwise tanh tensor D (2750 KB per sample at the stress shape) is produced and consumed in
// (k', pair) tiles and never leaves the SM; the channel contraction of these shapes runs in bgemm / wgrad (gemm.cu).
//   limits: P <= 128, K <= 128.
#include "kernels.cuh"

namespace dstd {

constexpr int GEN_MAX = 128;

bool generic_supported(int P, int K) { return P >= 1 && K >= 1 && P <= GEN_MAX && K <= GEN_MAX; }

// ------------------------------------------------------------------------------------------ dynamic adjacency, forward
//   pd[n,b,p,e] = brm[p] + sum_{k'=(r,p')} Wrm[p][k'] tanh(m[n,b,r,p',v] - m[n,b,2+r,p',w]),  e = v*K + w
// CTA = (128-pair tile, b, n).  Per chunk of 16 reduction rows k' the m rows are staged in shared memory, the pairwise tanh
// tile D[k'][e] is produced once (one pair per thread and row: the (v, w) decode is per-thread constant), and the
// contraction runs on register tiles: thread = 4 consecutive pairs x RP rows p, per k' one float4 of D and RP/4 float4 of
// Wrm for 4 RP FMAs.
constexpr int DG_TP = 128, DG_KC = 16;

template <int RP>    // rows per thread: 8 row groups x RP >= P
__global__ void __launch_bounds__(256) dynadj_fwd_gen_kernel(DynAdjFwdParams q) {
  __shared__ __align__(16) float Ds[DG_KC][DG_TP];
  __shared__ __align__(16) float Ws[DG_KC][8 * RP];
  __shared__ float m1c[DG_KC][GEN_MAX], m2c[DG_KC][GEN_MAX];
  const int P = q.P, K = q.K, KK = K * K, P2 = 2 * P;
  const int tid = threadIdx.x, eg = tid & 31, rg = tid >> 5;      // pairs 4 eg .. 4 eg + 3, rows rg RP .. rg RP + RP - 1
  const int b = blockIdx.y, n = blockIdx.z, e0 = blockIdx.x * DG_TP;
  const float* mb = q.m + (long long)(n * q.nb + b) * 4 * P * K;
  const float* wrm = q.w_rm[b];
  // the pair this thread produces in the D tile (rows tid / 128 + 2 j of the chunk)
  const int de = tid & (DG_TP - 1), dk0 = tid >> 7;
  const int e_d = e0 + de, dv = e_d < KK ? e_d / K : 0, dw = e_d < KK ? e_d - dv * K : 0;
  float acc[RP][4];
#pragma unroll
  for (int j = 0; j < RP; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
  for (int k0 = 0; k0 < P2; k0 += DG_KC) {
    __syncthreads();          // the previous chunk's tiles are consumed
    for (int i = tid; i < DG_KC * K; i += 256) {
      const int kk = i / K, x = i - kk * K, kp = k0 + kk;
      float a = 0.f, c = 0.f;
      if (kp < P2) {
        const int r = kp / P, pp = kp - r * P;
        a = __ldg(mb + (r * P + pp) * K + x);
        c = __ldg(mb + ((2 + r) * P + pp) * K + x);
      }
      m1c[kk][x] = a;
      m2c[kk][x] = c;
    }
    for (int i = tid; i < DG_KC * 8 * RP; i += 256) {
      const int kk = i / (8 * RP), p = i - kk * (8 * RP);
      Ws[kk][p] = (k0 + kk < P2 && p < P) ? __ldg(wrm + (long long)p * P2 + k0 + kk) : 0.f;
    }
    __syncthreads();
#pragma unroll 4
    for (int j = 0; j < DG_KC / 2; ++j) {
      const int kk = dk0 + 2 * j;
      Ds[kk][de] = (k0 + kk < P2 && e_d < KK) ? fast_tanh(m1c[kk][dv] - m2c[kk][dw]) : 0.f;
    }
    __syncthreads();
#pragma unroll 2
    for (int kk = 0; kk < DG_KC; ++kk) {
      const float4 d = *reinterpret_cast<const float4*>(&Ds[kk][4 * eg]);
#pragma unroll
      for (int j4 = 0; j4 < RP; j4 += 4) {
        const float4 w = *reinterpret_cast<const float4*>(&Ws[kk][rg * RP + j4]);
#define DSTD_DG_ROW(U, WV)                                 \
  acc[j4 + U][0] = fmaf(WV, d.x, acc[j4 + U][0]);          \
  acc[j4 + U][1] = fmaf(WV, d.y, acc[j4 + U][1]);          \
  acc[j4 + U][2] = fmaf(WV, d.z, acc[j4 + U][2]);          \
  acc[j4 + U][3] = fmaf(WV, d.w, acc[j4 + U][3]);
        DSTD_DG_ROW(0, w.x) DSTD_DG_ROW(1, w.y) DSTD_DG_ROW(2, w.z) DSTD_DG_ROW(3, w.w)
#undef DSTD_DG_ROW
      }
    }
  }
  float* dst = q.pd + (long long)(n * q.nb + b) * P * KK;
#pragma unroll
  for (int j = 0; j < RP; ++j) {
    const int p = rg * RP + j;
    if (p < P) {
      const float bv = __ldg(q.b_rm[b] + p);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = e0 + 4 * eg + u;
        if (e < KK) dst[(long long)p * KK + e] = acc[j][u] + bv;
      }
    }
  }
}

int launch_dynadj_fwd_gen(const DynAdjFwdParams& q, cudaStream_t st) {
  DSTD_REQUIRE(generic_supported(q.P, q.K), DSTD_ERR_UNSUPPORTED, "dynadj_fwd_gen: P=%d K=%d outside limits (<= %d)", q.P, q.K, GEN_MAX);
  dim3 grid(cdiv(q.K * q.K, DG_TP), q.nb, q.N);
  if (q.P <= 32) dynadj_fwd_gen_kernel<4><<<grid, 256, 0, st>>>(q);
  else if (q.P <= 64) dynadj_fwd_gen_kernel<8><<<grid, 256, 0, st>>>(q);
  else dynadj_fwd_gen_kernel<16><<<grid, 256, 0, st>>>(q);
  count_launch();
  return check_launch("dynadj_fwd_gen");
}

// ------------------------------------------------------------------------------------------ dynamic adjacency, backward
// CTA = (b, n, tile of VT whole rows v with all their w).  With gP = alpha * gxm:
//   gD[k'][e] = sum_p Wrm[p][k'] gP[p][e] ;  gS = gD (1 - D^2)
//   gm1[r,p',v] = sum_w gS[(r,p'),v,w]                                       complete inside the tile -> gm
//   gm2[r,p',w] = - sum_v gS[(r,p'),v,w]                                     partial per tile -> gm2_part, summed below
//   gWrm[p][k'] = sum_e gP[p][e] D[k'][e]   gbrm[p] = sum_e gP[p][e]         -> partial slot (n, tile) (already x alpha)
//   gA_eff[e]   = sum_p gxm[p][e]                                            -> slot n (the tiles own disjoint e ranges)
//   galpha      = sum gxm pd                                                 -> partial slot (n, tile)
constexpr int DB_KC = 16, DB_TP = 128, DB_GLD = DB_TP + 4;   // GLD % 4 == 0: float4 reads along the pairs

int dynadj_gen_tiles(int K) {
  const int VT = DB_TP / K > 0 ? DB_TP / K : 1;
  return (K + VT - 1) / VT;
}

// Register-tiled: the two contractions of a chunk of 16 reduction rows k' run on 4 x 2 (pairs x rows, step c) and
// 2 x 4 (output rows x reduction rows, step d) thread tiles with float4 shared-memory reads; Wrm and the m rows of the
// chunk are staged in shared memory (the first version read Wrm from global memory inside the FMA loop).
__global__ void __launch_bounds__(256) dynadj_bwd_gen_kernel(DynAdjBwdParams q, float* __restrict__ gm2_part, int NT) {
  extern __shared__ __align__(16) float smem[];
  const int P = q.P, K = q.K, KK = K * K, P2 = 2 * P, P21 = P2 + 1;
  const int VT = max(1, DB_TP / K);                       // K <= 128: at least one row per tile
  float* gPs = smem;                         // [P][DB_GLD]   alpha * gxm, columns >= tp zero
  float* Wc = gPs + P * DB_GLD;              // [P][DB_KC]    Wrm[p][k0 + kk]
  float* Ds = Wc + ((P * DB_KC + 3) & ~3);   // [DB_KC][DB_TP]
  float* Gs = Ds + DB_KC * DB_TP;            // [DB_KC][DB_TP]
  float* m1c = Gs + DB_KC * DB_TP;           // [DB_KC][DB_TP]  m1 rows at v0 .. v0 + vt - 1
  float* m2c = m1c + DB_KC * DB_TP;          // [DB_KC][DB_TP]  m2 rows, all w
  float* red = m2c + DB_KC * DB_TP;          // [32]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.x, n = blockIdx.y, tile = blockIdx.z;
  const int v0 = tile * VT, vt = min(VT, K - v0), tp = vt * K, e0 = v0 * K;
  const float alpha = q.alpha ? __ldg(q.alpha) : 1.0f;
  const float* mb = q.m + (long long)(n * q.nb + b) * 4 * P * K;
  const float* gx = q.gxm + (long long)(n * q.nb + b) * P * KK;
  const float* pdb = q.pd + (long long)(n * q.nb + b) * P * KK;
  const float* wrm = q.w_rm[b];
  float* gmb = q.gm + (long long)(n * q.nb + b) * 4 * P * K;
  const long long slot = ((long long)n * NT + tile) * q.nb + b;
  float* pw = q.part_wrm + slot * P * P21;
  float* pa = q.part_adj + ((long long)n * q.nb + b) * KK;
  float* g2 = gm2_part + (((long long)(n * q.nb + b)) * NT + tile) * P2 * K;
  float ga = 0.f;

  // a. gP tile (zero beyond tp), alpha gradient
  for (int i = tid; i < P * DB_TP; i += 256) {
    const int p = i / DB_TP, e = i - p * DB_TP;
    float v = 0.f;
    if (e < tp) {
      const float g = __ldg(gx + (long long)p * KK + e0 + e);
      ga = fmaf(g, __ldg(pdb + (long long)p * KK + e0 + e), ga);
      v = alpha * g;
    }
    gPs[p * DB_GLD + e] = v;
  }
  __syncthreads();
  for (int e = tid; e < tp; e += 256) {          // static-adjacency gradient: the raw sum (alpha may be 0)
    float s = 0.f;
    for (int p = 0; p < P; ++p) s += __ldg(gx + (long long)p * KK + e0 + e);
    pa[e0 + e] = s;
  }
  for (int p = warp; p < P; p += 8) {            // conv_rm bias gradient: row sums (fixed order: lanes then butterfly)
    float s = 0.f;
    for (int e = lane; e < tp; e += 32) s += gPs[p * DB_GLD + e];
    s = warp_sum(s);
    if (lane == 0) pw[(long long)p * P21 + P2] = s;
  }
  // thread-constant decodes
  const int de = tid & (DB_TP - 1), dk0 = tid >> 7;                    // D tile: pair de, rows dk0 + 2 j
  const int dvl = de < tp ? de / K : 0, dw = de < tp ? de - dvl * K : 0;
  const int ceg = tid & 31, ckg = tid >> 5;                            // step c: pairs 4 ceg .., rows 2 ckg, 2 ckg + 1
  const int dkq = tid & 3, dpg = tid >> 2;                             // step d: rows 4 dkq .., outputs p = 2 dpg, 2 dpg + 1
  for (int k0 = 0; k0 < P2; k0 += DB_KC) {
    // stage the m rows and the Wrm columns of this chunk
    for (int i = tid; i < DB_KC * DB_TP; i += 256) {
      const int kk = i >> 7, x = i & (DB_TP - 1), kp = k0 + kk;
      float a = 0.f, c = 0.f;
      if (kp < P2) {
        const int r = kp / P, pp = kp - r * P;
        if (x < vt) a = __ldg(mb + (r * P + pp) * K + v0 + x);
        if (x < K) c = __ldg(mb + ((2 + r) * P + pp) * K + x);
      }
      m1c[i] = a;
      m2c[i] = c;
    }
    for (int i = tid; i < P * DB_KC; i += 256) {
      const int p = i / DB_KC, kk = i - p * DB_KC;
      Wc[i] = (k0 + kk < P2) ? __ldg(wrm + (long long)p * P2 + k0 + kk) : 0.f;
    }
    __syncthreads();
    // b. D chunk
#pragma unroll
    for (int j = 0; j < DB_KC / 2; ++j) {
      const int kk = dk0 + 2 * j;
      Ds[kk * DB_TP + de] = (k0 + kk < P2 && de < tp) ? fast_tanh(m1c[kk * DB_TP + dvl] - m2c[kk * DB_TP + dw]) : 0.f;
    }
    __syncthreads();
    // c. gS = (Wrm^T gP) (1 - D^2)
    {
      float a0[4] = {0.f, 0.f, 0.f, 0.f}, a1[4] = {0.f, 0.f, 0.f, 0.f};
      const float* gp = gPs + 4 * ceg;
      const float* wc = Wc + 2 * ckg;
#pragma unroll 4
      for (int p = 0; p < P; ++p) {
        const float4 g = *reinterpret_cast<const float4*>(gp + p * DB_GLD);
        const float2 w = *reinterpret_cast<const float2*>(wc + p * DB_KC);
        a0[0] = fmaf(w.x, g.x, a0[0]); a0[1] = fmaf(w.x, g.y, a0[1]); a0[2] = fmaf(w.x, g.z, a0[2]); a0[3] = fmaf(w.x, g.w, a0[3]);
        a1[0] = fmaf(w.y, g.x, a1[0]); a1[1] = fmaf(w.y, g.y, a1[1]); a1[2] = fmaf(w.y, g.z, a1[2]); a1[3] = fmaf(w.y, g.w, a1[3]);
      }
      const float4 d0 = *reinterpret_cast<const float4*>(Ds + (2 * ckg) * DB_TP + 4 * ceg);
      const float4 d1 = *reinterpret_cast<const float4*>(Ds + (2 * ckg + 1) * DB_TP + 4 * ceg);
      *reinterpret_cast<float4*>(Gs + (2 * ckg) * DB_TP + 4 * ceg) =
          make_float4(a0[0] * (1.f - d0.x * d0.x), a0[1] * (1.f - d0.y * d0.y), a0[2] * (1.f - d0.z * d0.z), a0[3] * (1.f - d0.w * d0.w));
      *reinterpret_cast<float4*>(Gs + (2 * ckg + 1) * DB_TP + 4 * ceg) =
          make_float4(a1[0] * (1.f - d1.x * d1.x), a1[1] * (1.f - d1.y * d1.y), a1[2] * (1.f - d1.z * d1.z), a1[3] * (1.f - d1.w * d1.w));
    }
    // d. gWrm[p][k'] = sum_e gP[p][e] D[k'][e]
    if (2 * dpg < P) {
      float a[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
      const float* g0 = gPs + (2 * dpg) * DB_GLD;
      const float* g1 = gPs + (2 * dpg + 1 < P ? 2 * dpg + 1 : 2 * dpg) * DB_GLD;
      const float* dr = Ds + (4 * dkq) * DB_TP;
      const int tp4 = (tp + 3) & ~3;
      for (int e4 = 0; e4 < tp4; e4 += 4) {
        const float4 x0 = *reinterpret_cast<const float4*>(g0 + e4);
        const float4 x1 = *reinterpret_cast<const float4*>(g1 + e4);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float4 d = *reinterpret_cast<const float4*>(dr + u * DB_TP + e4);
          a[0][u] = fmaf(x0.x, d.x, fmaf(x0.y, d.y, fmaf(x0.z, d.z, fmaf(x0.w, d.w, a[0][u]))));
          a[1][u] = fmaf(x1.x, d.x, fmaf(x1.y, d.y, fmaf(x1.z, d.z, fmaf(x1.w, d.w, a[1][u]))));
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int kp = k0 + 4 * dkq + u;
        if (kp < P2) {
          pw[(long long)(2 * dpg) * P21 + kp] = a[0][u];
          if (2 * dpg + 1 < P) pw[(long long)(2 * dpg + 1) * P21 + kp] = a[1][u];
        }
      }
    }
    __syncthreads();
    // e. row sums (warp per (k', v): lanes over w, fixed butterfly) and column sums of gS
    for (int o = warp; o < DB_KC * vt; o += 8) {
      const int kk = o / vt, vl = o - kk * vt, kp = k0 + kk;
      float s = 0.f;
      for (int w = lane; w < K; w += 32) s += Gs[kk * DB_TP + vl * K + w];
      s = warp_sum(s);
      if (lane == 0 && kp < P2) {
        const int r = kp / P, pp = kp - r * P;
        gmb[(r * P + pp) * K + v0 + vl] = s;
      }
    }
    for (int i = tid; i < DB_KC * K; i += 256) {
      const int kk = i / K, w = i - kk * K, kp = k0 + kk;
      if (kp < P2) {
        float s = 0.f;
        for (int vl = 0; vl < vt; ++vl) s += Gs[kk * DB_TP + vl * K + w];
        g2[kp * K + w] = s;
      }
    }
    __syncthreads();
  }
  ga = block_sum(ga, red);
  if (tid == 0) q.part_alpha[slot] = ga;
}

// gm2[n,b,r,p',w] = - sum over the v tiles of the partial column sums (fixed order)
__global__ void gm2_reduce_kernel(const float* __restrict__ gm2_part, float* __restrict__ gm, int NB, int NT, int P, int K) {
  const long long per = (long long)2 * P * K, total = (long long)NB * per;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long nb_ = i / per, r = i - nb_ * per;
    const float* src = gm2_part + nb_ * NT * per + r;
    float s = 0.f;
    for (int t = 0; t < NT; ++t) s += src[t * per];
    gm[nb_ * 2 * per + per + r] = -s;
  }
}

size_t dynadj_bwd_gen_ws_floats(int N, int nb, int P, int K) { return (size_t)N * nb * dynadj_gen_tiles(K) * 2 * P * K; }

int launch_dynadj_bwd_gen(const DynAdjBwdParams& q, float* gm2_part, cudaStream_t st) {
  DSTD_REQUIRE(generic_supported(q.P, q.K), DSTD_ERR_UNSUPPORTED, "dynadj_bwd_gen: P=%d K=%d outside limits (<= %d)", q.P, q.K, GEN_MAX);
  const int NT = dynadj_gen_tiles(q.K);
  DSTD_REQUIRE(q.S == q.N * NT && gm2_part, DSTD_ERR_BAD_ARG, "dynadj_bwd_gen: one partial slot per (sample, tile) expected");
  const size_t smem = ((size_t)q.P * DB_GLD + ((q.P * DB_KC + 3) & ~3) + 4 * DB_KC * DB_TP + 32) * sizeof(float);
  ensure_max_smem((const void*)dynadj_bwd_gen_kernel);
  dim3 grid(q.nb, q.N, NT);
  dynadj_bwd_gen_kernel<<<grid, 256, smem, st>>>(q, gm2_part, NT);
  count_launch();
  DSTD_LAUNCH_CHECK("dynadj_bwd_gen");
  const long long total = (long long)q.N * q.nb * 2 * q.P * q.K;
  gm2_reduce_kernel<<<cdiv(total, 256) < 1184 ? cdiv(total, 256) : 1184, 256, 0, st>>>(gm2_part, q.gm, q.N * q.nb, NT, q.P, q.K);
  count_launch();
  return check_launch("gm2_reduce");
}

// ------------------------------------------------------------------------------------------ aggregation, forward
//   xa[n,b,c,p,w] = sum_v x[n,c,p,v] xmu_b[p,v,w]  (c < Cin; row Cin: x := 1)
// CTA = (p, n); the K x K adjacency of (n, b, p) sits in shared memory (rows / columns beyond K are zero, so the inner
// loops carry no guards); warp = 8 channels x 128 columns (4 per lane) register tile: per four v the warp reads
// 8 broadcast float4 of x and 16 row segments of xmu for 128 FMAs per lane.
constexpr int AG_CW = 8;                                      // channels per warp tile
__host__ __device__ inline int ag_kp4(int K) { return (K + 3) & ~3; }
__host__ __device__ inline int ag_kl(int K) { return ((K + 31) & ~31) + 1; }   // odd row stride >= 32-multiple + 1

// xmu_b[v][w] = alpha pd[n,b,p][v][w] + (A .* W + R)[v][w] (transposed when adj_t) into xm[KP4][KL], zero padded
__device__ __forceinline__ void ag_build_xm(const AggParams& q, int n, int b, int p, float alpha, float* xm, int KP4, int KL) {
  const int K = q.K, KK = K * K;
  for (int i = threadIdx.x; i < KP4 * KL; i += blockDim.x) xm[i] = 0.f;
  __syncthreads();
  const float* pdp = q.pd + ((long long)(n * q.nb + b) * q.P + p) * KK;
  for (int i = threadIdx.x; i < KK; i += blockDim.x) {
    const int r = i / K, c = i - r * K;
    float a = __ldg(q.adj[b] + i);
    if (q.adj_w[b]) a *= __ldg(q.adj_w[b] + i);
    if (q.adj_r[b]) a += __ldg(q.adj_r[b] + i);
    const float val = fmaf(alpha, __ldg(pdp + i), a);
    if (q.adj_t) xm[c * KL + r] = val; else xm[r * KL + c] = val;
  }
}

template <int NI>   // 32-column groups per lane: ceil(K / 32)
__global__ void __launch_bounds__(256) aggregate_fwd_gen_kernel(AggParams q) {
  extern __shared__ __align__(16) float smem[];
  const int K = q.K, P = q.P, Cin = q.Cin, C1 = Cin + 1, KP4 = ag_kp4(K), KL = ag_kl(K);
  float* xm = smem;                          // [KP4][KL]   xmu[v][w]
  float* xs = xm + ((KP4 * KL + 3) & ~3);    // [8 warps][AG_CW][KP4]   input rows of the warp's channels
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int p = blockIdx.x, n = blockIdx.y;
  const float alpha = q.alpha ? __ldg(q.alpha) : 1.0f;
  float* xw = xs + warp * AG_CW * KP4;
  const float* xb = q.x.p + vix(q.x, n, 0, p, 0);
  for (int b = 0; b < q.nb; ++b) {
    __syncthreads();                         // every warp is done with the previous branch's xm
    ag_build_xm(q, n, b, p, alpha, xm, KP4, KL);
    __syncthreads();
    for (int c0 = warp * AG_CW; c0 < C1; c0 += 8 * AG_CW) {
      // the warp's AG_CW rows: all loads of a lane issued before the first store (one exposed latency per tile)
      float stg[AG_CW][NI];
#pragma unroll
      for (int cl = 0; cl < AG_CW; ++cl) {
        const int c = c0 + cl;
#pragma unroll
        for (int i = 0; i < NI; ++i) {
          const int v = lane + 32 * i;
          stg[cl][i] = v < K ? (c < Cin ? __ldg(xb + (long long)c * q.x.sc + (long long)v * q.x.sk) : (c == Cin ? 1.0f : 0.f)) : 0.f;
        }
      }
#pragma unroll
      for (int cl = 0; cl < AG_CW; ++cl)
#pragma unroll
        for (int i = 0; i < NI; ++i)
          if (lane + 32 * i < KP4) xw[cl * KP4 + lane + 32 * i] = stg[cl][i];
      __syncwarp();
      float acc[AG_CW][NI];
#pragma unroll
      for (int cl = 0; cl < AG_CW; ++cl)
#pragma unroll
        for (int i = 0; i < NI; ++i) acc[cl][i] = 0.f;
      for (int v4 = 0; v4 < KP4; v4 += 4) {
        float4 xv[AG_CW];
#pragma unroll
        for (int cl = 0; cl < AG_CW; ++cl) xv[cl] = *reinterpret_cast<const float4*>(xw + cl * KP4 + v4);
#pragma unroll
        for (int vv = 0; vv < 4; ++vv) {
          const float* row = xm + (v4 + vv) * KL + lane;
          float m[NI];
#pragma unroll
          for (int i = 0; i < NI; ++i) m[i] = row[32 * i];      // KL - 1 >= 32 NI: in bounds, zero beyond K
#pragma unroll
          for (int cl = 0; cl < AG_CW; ++cl) {
            const float xe = vv == 0 ? xv[cl].x : vv == 1 ? xv[cl].y : vv == 2 ? xv[cl].z : xv[cl].w;
#pragma unroll
            for (int i = 0; i < NI; ++i) acc[cl][i] = fmaf(xe, m[i], acc[cl][i]);
          }
        }
      }
#pragma unroll
      for (int cl = 0; cl < AG_CW; ++cl) {
        const int c = c0 + cl;
        if (c < C1) {
          float* dst = q.xa + (((long long)(n * q.nb + b) * C1 + c) * P + p) * K;
#pragma unroll
          for (int i = 0; i < NI; ++i)
            if (lane + 32 * i < K) dst[lane + 32 * i] = acc[cl][i];
        }
      }
      __syncwarp();
    }
  }
}

// ---- tensor-path forward aggregation (mma.sync m16n8k8 TF32 with 3xTF32 compensation), K >= 48.
// The CUDA-core kernel above is bound by shared-memory wavefronts: every warp re-reads the whole K x K adjacency (four
// wavefronts per v) for 32 FFMAs, 24 wavefronts per 128 FFMAs against the 16 FFMAs per wavefront that four schedulers
// need (measured 29 % FMA utilisation).  Here a warp owns a 16-channel tile x all w columns (C fragments), the A
// fragments (x) come straight from global memory in fragment layout (a quad reads 16 contiguous bytes of a channel row,
// the k + 4 half is the other half of the same sector), the B fragments (xm) from shared memory with a row stride of
// 8 (mod 32) floats: one B fragment feeds 3 MMAs = 2048 MACs per two shared-memory loads.
__device__ __forceinline__ void ag_split(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}
__device__ __forceinline__ void ag_mma(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
__host__ __device__ inline int agm_kld(int K) { return ((K + 31) & ~31) + 8; }   // == 8 (mod 32): conflict-free B fragments

template <int NT>   // 8-column tiles of w: 8 NT >= K
__global__ void __launch_bounds__(256) aggregate_fwd_gen_mma_kernel(AggParams q) {
  extern __shared__ __align__(16) float smem[];
  const int K = q.K, P = q.P, Cin = q.Cin, C1 = Cin + 1, KP8 = (K + 7) & ~7, KLD = agm_kld(K);
  float* xm = smem;                          // [KP8][KLD]   xmu[v][w], zero padded
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, fg = lane >> 2, ft = lane & 3;
  const int p = blockIdx.x, n = blockIdx.y;
  const float alpha = q.alpha ? __ldg(q.alpha) : 1.0f;
  const float* xb = q.x.p + vix(q.x, n, 0, p, 0);
  const int mtiles = (C1 + 15) >> 4;
  for (int b = 0; b < q.nb; ++b) {
    __syncthreads();                         // every warp is done with the previous branch's xm
    ag_build_xm(q, n, b, p, alpha, xm, KP8, KLD);
    __syncthreads();
    for (int mt = warp; mt < mtiles; mt += 8) {
      const int c0 = mt * 16 + fg, c1 = c0 + 8;
      // row sources of this lane: a channel row of x, the ones row (c == Cin) or nothing
      const float* r0 = c0 < Cin ? xb + (long long)c0 * q.x.sc : nullptr;
      const float* r1 = c1 < Cin ? xb + (long long)c1 * q.x.sc : nullptr;
      const float one0 = c0 == Cin ? 1.f : 0.f, one1 = c1 == Cin ? 1.f : 0.f;
      float acc[NT][4];
#pragma unroll
      for (int i = 0; i < NT; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
      auto lda = [&](int k0, float (&a)[4]) {
        const int v0 = k0 + ft, v1 = v0 + 4;
        a[0] = v0 < K ? (r0 ? __ldg(r0 + (long long)v0 * q.x.sk) : one0) : 0.f;
        a[1] = v0 < K ? (r1 ? __ldg(r1 + (long long)v0 * q.x.sk) : one1) : 0.f;
        a[2] = v1 < K ? (r0 ? __ldg(r0 + (long long)v1 * q.x.sk) : one0) : 0.f;
        a[3] = v1 < K ? (r1 ? __ldg(r1 + (long long)v1 * q.x.sk) : one1) : 0.f;
      };
      float an[4];
      lda(0, an);
      for (int k0 = 0; k0 < KP8; k0 += 8) {
        uint32_t ah[4], al[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) ag_split(an[e], ah[e], al[e]);
        if (k0 + 8 < KP8) lda(k0 + 8, an);   // next k-step's fragment in flight during this one's MMAs
        const float* br = xm + (k0 + ft) * KLD + fg;
#pragma unroll
        for (int i = 0; i < NT; ++i) {
          uint32_t bh[2], bl[2];
          ag_split(br[i * 8], bh[0], bl[0]);
          ag_split(br[4 * KLD + i * 8], bh[1], bl[1]);
          ag_mma(acc[i], al, bh);
          ag_mma(acc[i], ah, bl);
          ag_mma(acc[i], ah, bh);
        }
      }
      float* d0 = q.xa + (((long long)(n * q.nb + b) * C1 + c0) * P + p) * K;
      float* d1 = q.xa + (((long long)(n * q.nb + b) * C1 + c1) * P + p) * K;
#pragma unroll
      for (int i = 0; i < NT; ++i) {
        const int w = i * 8 + 2 * ft;
        if (c0 < C1) {
          if (w < K) d0[w] = acc[i][0];
          if (w + 1 < K) d0[w + 1] = acc[i][1];
        }
        if (c1 < C1) {
          if (w < K) d1[w] = acc[i][2];
          if (w + 1 < K) d1[w + 1] = acc[i][3];
        }
      }
    }
  }
}

int launch_aggregate_fwd_gen(const AggParams& q, bool mma, cudaStream_t st) {
  DSTD_REQUIRE(generic_supported(q.P, q.K), DSTD_ERR_UNSUPPORTED, "aggregate_fwd_gen: P=%d K=%d outside limits", q.P, q.K);
  if (mma && q.K >= 48) {
    const int KP8 = (q.K + 7) & ~7, KLD = agm_kld(q.K);
    const size_t sm = (size_t)KP8 * KLD * sizeof(float);
    dim3 grid(q.P, q.N);
#define DSTD_AGM(NT_)                                                         \
  {                                                                           \
    ensure_max_smem((const void*)aggregate_fwd_gen_mma_kernel<NT_>);          \
    aggregate_fwd_gen_mma_kernel<NT_><<<grid, 256, sm, st>>>(q);              \
  }
    const int nt = (q.K + 7) / 8;
    if (nt <= 8) DSTD_AGM(8) else if (nt <= 12) DSTD_AGM(12) else DSTD_AGM(16)
#undef DSTD_AGM
    count_launch();
    return check_launch("aggregate_fwd_gen_mma");
  }
  const int KP4 = ag_kp4(q.K), KL = ag_kl(q.K);
  const size_t smem = ((size_t)((KP4 * KL + 3) & ~3) + (size_t)8 * AG_CW * KP4) * sizeof(float);
  dim3 grid(q.P, q.N);
#define DSTD_AGF(NI_)                                                     \
  {                                                                       \
    ensure_max_smem((const void*)aggregate_fwd_gen_kernel<NI_>);          \
    aggregate_fwd_gen_kernel<NI_><<<grid, 256, smem, st>>>(q);            \
  }
  switch ((q.K + 31) / 32) {
    case 1: DSTD_AGF(1) break;
    case 2: DSTD_AGF(2) break;
    case 3: DSTD_AGF(3) break;
    default: DSTD_AGF(4) break;
  }
#undef DSTD_AGF
  count_launch();
  return check_launch("aggregate_fwd_gen");
}

// ------------------------------------------------------------------------------------------ aggregation, backward
//   gx[n,c,p,v]      = sum_b sum_w gxa_b[c,p,w] xmu_b[p,v,w]
//   gxmu_b[p,v,w]    = sum_{c <= Cin} xaug[c,p,v] gxa_b[c,p,w]
// CTA = (p, n), channels in chunks of CC (a multiple of 32, ~16 KB per staged tensor) through shared memory, every global
// load of a chunk issued before the first store.  gx: warp = 4 channels x 32 NI rows v, the odd row stride of xmu makes
// the lane = v reads conflict free.  gxmu: 4 x 4 (v, w) register tiles kept for the whole channel loop (two float4
// reads per 16 FMAs).  K > 44: up to four tiles per thread, all channels.  Small K (at most 128 tiles): G = 256 / tiles
// thread groups split the channels of a chunk and their tiles are summed in group order at the end (deterministic).
// gx accumulates over the branches in global memory (same thread, same address).
template <int NI, bool SMALL>
__global__ void __launch_bounds__(256) aggregate_bwd_gen_kernel(AggParams q, int CC, int G) {
  extern __shared__ __align__(16) float smem[];
  const int K = q.K, P = q.P, KK = K * K, Cin = q.Cin, C1 = Cin + 1, KP4 = ag_kp4(K), KL = ag_kl(K);
  float* xm = smem;                          // [KP4][KL]   xmu_b[v][w]
  float* xs = xm + ((KP4 * KL + 3) & ~3);    // [CC][KP4]  x rows (ones row included), zero padded
  float* gs = xs + CC * KP4;                 // [CC][KP4]  gxa_b rows, zero padded
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int p = blockIdx.x, n = blockIdx.y;
  const float alpha = q.alpha ? __ldg(q.alpha) : 1.0f;
  const int TW = KP4 >> 2, ntile = TW * TW;  // 4 x 4 tiles of the (v, w) grid
  constexpr int NT = SMALL ? 1 : 4;          // tiles per thread: SMALL (tid % ntile, channel group tid / ntile), else tid + 256 j
  const int grp = SMALL ? tid / ntile : 0, tsm = SMALL ? tid - grp * ntile : 0;
  const bool act_sm = SMALL && grp < G;
  const float* xb = q.x.p + vix(q.x, n, 0, p, 0);
  const int chunk_e = CC * KP4;
  for (int b = 0; b < q.nb; ++b) {
    __syncthreads();
    ag_build_xm(q, n, b, p, alpha, xm, KP4, KL);
    float tacc[NT][16];
#pragma unroll
    for (int j = 0; j < NT; ++j)
#pragma unroll
      for (int e = 0; e < 16; ++e) tacc[j][e] = 0.f;
    const float* gb = q.gxa + ((long long)(n * q.nb + b) * C1 * P + p) * K;
    for (int c0 = 0; c0 < C1; c0 += CC) {
      __syncthreads();
      for (int base = 0; base < chunk_e; base += 256 * 8) {
        float xa_[8], ga_[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int i = base + tid + 256 * u;
          const int cl = i / KP4, k = i - cl * KP4, c = c0 + cl;
          const bool in = i < chunk_e && k < K;
          xa_[u] = in ? (c < Cin ? __ldg(xb + (long long)c * q.x.sc + (long long)k * q.x.sk) : (c == Cin ? 1.0f : 0.f)) : 0.f;
          ga_[u] = (in && c < C1) ? __ldg(gb + (long long)c * P * K + k) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int i = base + tid + 256 * u;
          if (i < chunk_e) {
            xs[i] = xa_[u];
            gs[i] = ga_[u];
          }
        }
      }
      __syncthreads();
      // gx rows of this chunk: warp = CC/8 channels in groups of 4, lane = rows v = lane + 32 i
      for (int cg = 0; cg < CC / 8; cg += 4) {
        const int clb = warp * (CC / 8) + cg;
        if (c0 + clb >= Cin) break;
        float acc[4][NI];
#pragma unroll
        for (int cl = 0; cl < 4; ++cl)
#pragma unroll
          for (int i = 0; i < NI; ++i) acc[cl][i] = 0.f;
        for (int w4 = 0; w4 < KP4; w4 += 4) {
          float4 gv[4];
#pragma unroll
          for (int cl = 0; cl < 4; ++cl) gv[cl] = *reinterpret_cast<const float4*>(gs + (clb + cl) * KP4 + w4);
#pragma unroll
          for (int i = 0; i < NI; ++i) {
            const int v = lane + 32 * i;
            if (v < KP4) {                      // rows K .. KP4-1 of xm are zero
              const float* row = xm + v * KL + w4;
              const float m0 = row[0], m1 = row[1], m2 = row[2], m3 = row[3];
#pragma unroll
              for (int cl = 0; cl < 4; ++cl)
                acc[cl][i] = fmaf(gv[cl].x, m0, fmaf(gv[cl].y, m1, fmaf(gv[cl].z, m2, fmaf(gv[cl].w, m3, acc[cl][i]))));
            }
          }
        }
#pragma unroll
        for (int cl = 0; cl < 4; ++cl) {
          const int c = c0 + clb + cl;
          if (c < Cin) {
#pragma unroll
            for (int i = 0; i < NI; ++i) {
              const int v = lane + 32 * i;
              if (v < K) {
                float* d = q.gx.p + vix(q.gx, n, c, p, v);
                *d = (b > 0 ? *d : 0.f) + acc[cl][i];
              }
            }
          }
        }
      }
      // gxmu tiles += xs^T gs over the chunk
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        const int t = SMALL ? tsm : tid + 256 * j;
        if (SMALL ? act_sm : t < ntile) {
          const int tv = t / TW, tw = t - tv * TW;
          const float* xr = xs + 4 * tv;
          const float* gr = gs + 4 * tw;
          const int cstep = SMALL ? G : 1;
#pragma unroll 4
          for (int cl = SMALL ? grp : 0; cl < CC; cl += cstep) {
            const float4 a = *reinterpret_cast<const float4*>(xr + cl * KP4);
            const float4 g = *reinterpret_cast<const float4*>(gr + cl * KP4);
            tacc[j][0] = fmaf(a.x, g.x, tacc[j][0]); tacc[j][1] = fmaf(a.x, g.y, tacc[j][1]);
            tacc[j][2] = fmaf(a.x, g.z, tacc[j][2]); tacc[j][3] = fmaf(a.x, g.w, tacc[j][3]);
            tacc[j][4] = fmaf(a.y, g.x, tacc[j][4]); tacc[j][5] = fmaf(a.y, g.y, tacc[j][5]);
            tacc[j][6] = fmaf(a.y, g.z, tacc[j][6]); tacc[j][7] = fmaf(a.y, g.w, tacc[j][7]);
            tacc[j][8] = fmaf(a.z, g.x, tacc[j][8]); tacc[j][9] = fmaf(a.z, g.y, tacc[j][9]);
            tacc[j][10] = fmaf(a.z, g.z, tacc[j][10]); tacc[j][11] = fmaf(a.z, g.w, tacc[j][11]);
            tacc[j][12] = fmaf(a.w, g.x, tacc[j][12]); tacc[j][13] = fmaf(a.w, g.y, tacc[j][13]);
            tacc[j][14] = fmaf(a.w, g.z, tacc[j][14]); tacc[j][15] = fmaf(a.w, g.w, tacc[j][15]);
          }
        }
      }
    }
    float* dst = q.gxm + ((long long)(n * q.nb + b) * P + p) * KK;
    if (SMALL) {
      // group partials through the (now free) chunk buffers, summed in group order
      __syncthreads();
      float* scr = xs;                         // [G][KP4][KP4]  (host checks that it fits in the two chunk buffers)
      if (act_sm) {
        const int tv = tsm / TW, tw = tsm - tv * TW;
#pragma unroll
        for (int e = 0; e < 16; ++e) scr[(grp * KP4 + 4 * tv + (e >> 2)) * KP4 + 4 * tw + (e & 3)] = tacc[0][e];
      }
      __syncthreads();
      for (int i = tid; i < KK; i += 256) {
        const int v = i / K, w = i - v * K;
        float sres = 0.f;
        for (int g = 0; g < G; ++g) sres += scr[(g * KP4 + v) * KP4 + w];
        dst[q.adj_t ? (w * K + v) : i] = sres;
      }
    } else {
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        const int t = tid + 256 * j;
        if (t < ntile) {
          const int tv = t / TW, tw = t - tv * TW;
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            const int v = 4 * tv + (e >> 2), w = 4 * tw + (e & 3);
            if (v < K && w < K) dst[q.adj_t ? (w * K + v) : (v * K + w)] = tacc[j][e];
          }
        }
      }
    }
  }
}

int launch_aggregate_bwd_gen(const AggParams& q, cudaStream_t st) {
  DSTD_REQUIRE(generic_supported(q.P, q.K), DSTD_ERR_UNSUPPORTED, "aggregate_bwd_gen: P=%d K=%d outside limits", q.P, q.K);
  const int KP4 = ag_kp4(q.K), KL = ag_kl(q.K), ntile = (KP4 / 4) * (KP4 / 4);
  int CC = 4096 / KP4 / 32 * 32;
  const int c1r = (q.Cin + 1 + 31) / 32 * 32;
  if (CC > c1r) CC = c1r;
  if (CC > 256) CC = 256;
  if (CC < 32) CC = 32;
  const bool small = ntile <= 128;
  int G = small ? 256 / ntile : 1;
  while (small && G > 1 && (size_t)G * KP4 * KP4 > (size_t)2 * CC * KP4) --G;   // partials must fit in the chunk buffers
  const size_t smem = ((size_t)((KP4 * KL + 3) & ~3) + (size_t)2 * CC * KP4) * sizeof(float);
  dim3 grid(q.P, q.N);
#define DSTD_AGB(NI_, SM_)                                                      \
  {                                                                             \
    ensure_max_smem((const void*)aggregate_bwd_gen_kernel<NI_, SM_>);           \
    aggregate_bwd_gen_kernel<NI_, SM_><<<grid, 256, smem, st>>>(q, CC, G);      \
  }
  const int ni = (q.K + 31) / 32;
  if (small) {
    if (ni == 1) DSTD_AGB(1, true) else DSTD_AGB(2, true)       // ntile <= 128 means K <= 44
  } else {
    switch (ni) {
      case 2: DSTD_AGB(2, false) break;
      case 3: DSTD_AGB(3, false) break;
      default: DSTD_AGB(4, false) break;
    }
  }
#undef DSTD_AGB
  count_launch();
  return check_launch("aggregate_bwd_gen");
}

}  // namespace dstd
