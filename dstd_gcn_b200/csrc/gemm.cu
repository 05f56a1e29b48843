// Generic channel-contraction kernels (fp32 SIMT, register-blocked, shared-memory staged):
//   bgemm : Out[n,i,p,k] = sum_c W(c,i) In[n,c,p,k] (+ bias[i]) (+ Add[n,i,p,k])      "1x1 conv" family
//   wgrad : G[i,c]       = sum_{n,p,k} A[n,i,p,k] B[n,c,p,k]                           weight gradients
//   reduce_segments : sum split partials and scatter sub-matrices into parameter-gradient tensors
// Columns g = (n,p,k) are flattened across the batch so tiles never straddle padding.
#include "kernels.cuh"

namespace dstd {

// ================================================================================= bgemm
template <int BM, int BN, int TM, int TN>
__global__ void __launch_bounds__((BM / TM) * (BN / TN)) bgemm_kernel(BgemmParams q) {
  constexpr int KC = 16;
  constexpr int NT = (BM / TM) * (BN / TN);
  __shared__ __align__(16) float Ws[KC][BM];
  __shared__ __align__(16) float Is[KC][BN];
  __shared__ long long col_in[BN], col_out[BN], col_add[BN];

  const int tid = threadIdx.x;
  const int tx = tid % (BN / TN), ty = tid / (BN / TN);
  const long long g0 = (long long)blockIdx.x * BN;
  const int row0 = q.m0 + blockIdx.y * BM;
  const int PK = q.P * q.K;

  for (int c = tid; c < BN; c += NT) {
    long long g = g0 + c;
    if (g < q.G) {
      int n = (int)(g / PK);
      int j = (int)(g - (long long)n * PK);
      int p = j / q.K, k = j - p * q.K;
      col_in[c] = vix(q.in, n, 0, p, k);
      col_out[c] = vix(q.out, n, 0, p, k);
      col_add[c] = q.add.p ? vix(q.add, n, 0, p, k) : 0;
    } else {
      col_in[c] = -1;
      col_out[c] = -1;
      col_add[c] = 0;
    }
  }
  __syncthreads();

  float acc[TM][TN];
#pragma unroll
  for (int a = 0; a < TM; ++a)
#pragma unroll
    for (int b = 0; b < TN; ++b) acc[a][b] = 0.f;

  for (int kc0 = 0; kc0 < q.Kd; kc0 += KC) {
    for (int idx = tid; idx < KC * BM; idx += NT) {
      int kk = idx / BM, i = idx - kk * BM;
      int c = kc0 + kk, row = row0 + i;
      float v = 0.f;
      if (c < q.Kd && row < q.m1) v = __ldg(q.w + (long long)c * q.wsc + (long long)row * q.wsi);
      Ws[kk][i] = v;
    }
    for (int idx = tid; idx < KC * BN; idx += NT) {
      int kk = idx / BN, col = idx - kk * BN;
      int c = kc0 + kk;
      long long off = col_in[col];
      float v = 0.f;
      if (c < q.Kd && off >= 0) v = (c == q.ones_row) ? 1.0f : __ldg(q.in.p + off + (long long)c * q.in.sc);
      Is[kk][col] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < KC; ++kk) {
      float a[TM], b[TN];
#pragma unroll
      for (int i = 0; i < TM; i += 4) {
        float4 t = *reinterpret_cast<const float4*>(&Ws[kk][ty * TM + i]);
        a[i] = t.x; a[i + 1] = t.y; a[i + 2] = t.z; a[i + 3] = t.w;
      }
#pragma unroll
      for (int j = 0; j < TN; j += 4) {
        float4 t = *reinterpret_cast<const float4*>(&Is[kk][tx * TN + j]);
        b[j] = t.x; b[j + 1] = t.y; b[j + 2] = t.z; b[j + 3] = t.w;
      }
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < TM; ++i) {
    int row = row0 + ty * TM + i;
    if (row >= q.m1) continue;
    float bv = q.bias ? __ldg(q.bias + row) : 0.f;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      int col = tx * TN + j;
      long long off = col_out[col];
      if (off < 0) continue;
      float v = acc[i][j] + bv;
      if (q.add.p) v += q.add.p[col_add[col] + (long long)row * q.add.sc];
      q.out.p[off + (long long)row * q.out.sc] = v;
    }
  }
}

int launch_bgemm(BgemmParams q, cudaStream_t st) {
  if (q.G <= 0 || q.M <= 0) return 0;
  if (q.tc_ws && bgemm_tc_supported(q.M, q.Kd)) return launch_bgemm_tc(q, q.tc_ws, st);   // tcgen05 path (bgemm_tc.cu)
  // full 64-row tiles on the wide kernel, a remainder of <= 16 rows on the skinny one
  int full = (q.M / 64) * 64;
  int rem = q.M - full;
  if (rem > 16) { full = q.M; rem = 0; }
  if (full > 0) {
    BgemmParams p = q;
    p.m0 = 0;
    p.m1 = full;
    dim3 grid(cdiv(q.G, 128), cdiv(full, 64));
    bgemm_kernel<64, 128, 8, 4><<<grid, 256, 0, st>>>(p);
    count_launch();
  }
  if (rem > 0) {
    BgemmParams p = q;
    p.m0 = full;
    p.m1 = q.M;
    dim3 grid(cdiv(q.G, 256), 1);
    bgemm_kernel<16, 256, 4, 4><<<grid, 256, 0, st>>>(p);
    count_launch();
  }
  return check_launch("bgemm");
}

// ================================================================================= wgrad
// G[i,c] = sum_g A[i,g] B[c,g].  Both operands are contiguous along the reduction index g, so tiles are staged
// untransposed ([row][32 g] with a 36-float pitch: float4 reads along g are bank-conflict free for 32 lanes on
// consecutive rows) and each thread owns rows {ty*TM+a} x columns {lane + 32 b}.
template <int TM, int TN>
__global__ void __launch_bounds__(256) wgrad_kernel(WgradParams q) {
  constexpr int KC = 32, PITCH = 36;
  constexpr int BM = 8 * TM, BC = 32 * TN;
  constexpr int NA = BM * KC / 256, NB = BC * KC / 256;   // values of a tile each thread stages (its column = lane)
  __shared__ __align__(16) float As[BM][PITCH];
  __shared__ __align__(16) float Bs[BC][PITCH];

  const int tid = threadIdx.x, lane = tid & 31, ty = tid >> 5;
  const int i0 = blockIdx.y * BM, c0 = blockIdx.z * BC;
  const int PK = q.P * q.K;
  long long gbeg = (long long)blockIdx.x * q.cols_per_split;
  long long gend = gbeg + q.cols_per_split;
  if (gend > q.G) gend = q.G;

  float acc[TM][TN];
#pragma unroll
  for (int a = 0; a < TM; ++a)
#pragma unroll
    for (int b = 0; b < TN; ++b) acc[a][b] = 0.f;

  // software pipeline: the next tile's values are loaded into registers while the current tile is multiplied, so
  // the global-load latency is paid once per CTA instead of once per 32 columns
  float ra[NA], rb[NB];
  auto load_tile = [&](long long gc) {
    const long long g = gc + lane;
    long long aoff = -1, boff = -1;
    if (g < gend) {
      const int n = (int)(g / PK);
      const int j = (int)(g - (long long)n * PK);
      const int p = j / q.K, k = j - p * q.K;
      aoff = vix(q.a, n, 0, p, k);
      boff = vix(q.b, n, 0, p, k);
    }
#pragma unroll
    for (int u = 0; u < NA; ++u) {
      const int i = i0 + ty + 8 * u;
      ra[u] = (aoff >= 0 && i < q.M) ? __ldg(q.a.p + aoff + (long long)i * q.a.sc) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < NB; ++u) {
      const int cc = c0 + ty + 8 * u;
      rb[u] = (boff >= 0 && cc < q.Cd) ? ((cc == q.b_ones_row) ? 1.0f : __ldg(q.b.p + boff + (long long)cc * q.b.sc)) : 0.f;
    }
  };
  if (gbeg < gend) load_tile(gbeg);
  for (long long gc = gbeg; gc < gend; gc += KC) {
#pragma unroll
    for (int u = 0; u < NA; ++u) As[ty + 8 * u][lane] = ra[u];
#pragma unroll
    for (int u = 0; u < NB; ++u) Bs[ty + 8 * u][lane] = rb[u];
    __syncthreads();
    if (gc + KC < gend) load_tile(gc + KC);
#pragma unroll
    for (int k4 = 0; k4 < KC; k4 += 4) {
      float4 a4[TM], b4[TN];
#pragma unroll
      for (int a = 0; a < TM; ++a) a4[a] = *reinterpret_cast<const float4*>(&As[ty * TM + a][k4]);
#pragma unroll
      for (int b = 0; b < TN; ++b) b4[b] = *reinterpret_cast<const float4*>(&Bs[lane + 32 * b][k4]);
#pragma unroll
      for (int a = 0; a < TM; ++a)
#pragma unroll
        for (int b = 0; b < TN; ++b) {
          acc[a][b] = fmaf(a4[a].x, b4[b].x, acc[a][b]);
          acc[a][b] = fmaf(a4[a].y, b4[b].y, acc[a][b]);
          acc[a][b] = fmaf(a4[a].z, b4[b].z, acc[a][b]);
          acc[a][b] = fmaf(a4[a].w, b4[b].w, acc[a][b]);
        }
    }
    __syncthreads();
  }
  float* dst = q.partial + (long long)blockIdx.x * q.M * q.Cd;
#pragma unroll
  for (int a = 0; a < TM; ++a) {
    int i = i0 + ty * TM + a;
    if (i >= q.M) continue;
#pragma unroll
    for (int b = 0; b < TN; ++b) {
      int c = c0 + lane + 32 * b;
      if (c < q.Cd) dst[(long long)i * q.Cd + c] = acc[a][b];
    }
  }
}

int wgrad_splits(long long G) {
  long long s = (G + 511) / 512;
  if (s > 592) s = 592;
  if (s < 1) s = 1;
  return (int)s;
}

template <int TM>
static void wgrad_dispatch_tn(const WgradParams& q, int tn, dim3 grid, cudaStream_t st) {
  switch (tn) {
    case 1: wgrad_kernel<TM, 1><<<grid, 256, 0, st>>>(q); break;
    case 2: wgrad_kernel<TM, 2><<<grid, 256, 0, st>>>(q); break;
    case 3: wgrad_kernel<TM, 3><<<grid, 256, 0, st>>>(q); break;
    case 4: wgrad_kernel<TM, 4><<<grid, 256, 0, st>>>(q); break;
    default: wgrad_kernel<TM, 5><<<grid, 256, 0, st>>>(q); break;
  }
}

// partial must hold wgrad_splits(G) * M * Cd floats
int launch_wgrad(WgradParams& q, bool tc, cudaStream_t st) {
  if (tc && wgrad_tc_supported(q.M, q.Cd)) return launch_wgrad_tc(q, st);     // tcgen05 path (bgemm_tc.cu)
  q.S = wgrad_splits(q.G);
  long long per = (q.G + q.S - 1) / q.S;
  q.cols_per_split = (per + 31) / 32 * 32;
  q.S = cdiv(q.G, q.cols_per_split);
  int tn = cdiv(q.Cd, 32);
  if (tn > 5) tn = (q.Cd % 128 == 0 || q.Cd > 160) ? 4 : 5;
  if (q.M <= 8) {
    dim3 grid(q.S, cdiv(q.M, 8), cdiv(q.Cd, 32 * tn));
    wgrad_dispatch_tn<1>(q, tn, grid, st);
  } else {
    dim3 grid(q.S, cdiv(q.M, 64), cdiv(q.Cd, 32 * tn));
    wgrad_dispatch_tn<8>(q, tn, grid, st);
  }
  count_launch();
  return check_launch("wgrad");
}

// ================================================================================= reduce + scatter
// block = 8 warps: warp w sums the w-th eighth of the S partials for 32 consecutive outputs (coalesced 128-byte
// loads, 4 in flight), the eight sub-sums are combined in a fixed order through shared memory (deterministic).  A
// single thread per output walking all S partials was a chain of ~S/8 dependent L2 round trips (22-25 us per call).
__global__ void __launch_bounds__(256) reduce_segments_kernel(ReduceParams q) {
  __shared__ float part[8][32];
  const ReduceSeg& s = q.seg[blockIdx.y];
  const int total = s.rows * s.cols, lane = threadIdx.x & 31, ch = threadIdx.x >> 5;
  const int per = (s.S + 7) / 8, k0 = ch * per, k1 = min(s.S, k0 + per);
  for (int base = blockIdx.x * 32; base < total; base += gridDim.x * 32) {
    const int idx = base + lane;
    const int r = idx / s.cols, c = idx - r * s.cols;
    float v = 0.f;
    if (idx < total) {
      const float* src = s.src + (long long)r * s.src_ld + c;
      float a[4] = {0.f, 0.f, 0.f, 0.f};
      int k = k0;
      for (; k + 4 <= k1; k += 4) {
#pragma unroll
        for (int u = 0; u < 4; ++u) a[u] += src[(long long)(k + u) * s.sstride];
      }
      for (int u = 0; k < k1; ++k, ++u) a[u] += src[(long long)k * s.sstride];
      v = (a[0] + a[1]) + (a[2] + a[3]);
    }
    part[ch][lane] = v;
    __syncthreads();
    if (ch == 0 && idx < total) {
      float t = part[0][lane];
#pragma unroll
      for (int j = 1; j < 8; ++j) t += part[j][lane];
      t *= s.scale;
      if (s.dst) s.dst[(long long)r * s.dst_ld + c] = t;
      if (s.dst2) s.dst2[(long long)r * s.dst_ld + c] = t * __ldg(s.mul + (long long)r * s.dst_ld + c);
    }
    __syncthreads();
  }
}

int launch_reduce(const ReduceParams& q, cudaStream_t st) {
  if (q.nseg == 0) return 0;
  int maxe = 1;
  for (int i = 0; i < q.nseg; ++i) maxe = max(maxe, q.seg[i].rows * q.seg[i].cols);
  dim3 grid(min(cdiv(maxe, 32), 128), q.nseg);
  reduce_segments_kernel<<<grid, 256, 0, st>>>(q);
  count_launch();
  return check_launch("reduce_segments");
}

}  // namespace dstd

// ================================================================================= mproj backward
// Backward of the 4*nb-row reduction convs (conv_m1 / conv_m2 of every branch, model/dstdgcn.py:82) in one pass over x:
//   gx[c][g]  += sum_j wm[j][c] gm[j][g]                  (read-modify-write of the aggregation part of gx)
//   gwm[j][c] += sum_g gm[j][g] [x;1][c][g]               (register accumulators, one partial per CTA)
// Memory bound by design: x and gm are read once, gx is read and written once.
namespace dstd {

constexpr int MP_TP = 256;        // columns per tile (one per thread)
constexpr int MP_LD = MP_TP + 4;  // (LD/4) odd: float4 reads along g with lane = channel are conflict free
constexpr int MP_CG = 5;          // channel groups of 64 -> Cin + 1 <= 320

__global__ void __launch_bounds__(256, 2) mproj_bwd_kernel(MprojBwdParams q) {
  extern __shared__ __align__(16) float smem[];
  const int Cin = q.Cin, C1 = Cin + 1, J = q.J, PK = q.P * q.K;
  float* xs = smem;                    // [C1][MP_LD]
  float* gms = xs + C1 * MP_LD;        // [8][MP_LD]
  float* wmT = gms + 8 * MP_LD;        // [Cin][8]   wm transposed, zero padded to 8 rows
  const int tid = threadIdx.x;
  for (int i = tid; i < Cin * 8; i += 256) {
    int c = i >> 3, j = i & 7;
    wmT[i] = j < J ? __ldg(q.wm + (long long)j * C1 + c) : 0.f;
  }
  float acc[MP_CG][2];
#pragma unroll
  for (int a = 0; a < MP_CG; ++a) acc[a][0] = acc[a][1] = 0.f;
  const int cl = tid & 63, jg = tid >> 6;   // phase 2: channel (+64 a), rows (2 jg, 2 jg + 1)
  const long long ntiles = (q.G + MP_TP - 1) / MP_TP;

  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long g = tile * MP_TP + tid;
    const bool ok = g < q.G;
    long long ox = 0, og = 0, om = 0, oa = 0;
    if (ok) {
      const int n = (int)(g / PK);
      const int rem = (int)(g - (long long)n * PK);
      const int p = rem / q.K, k = rem - p * q.K;
      ox = vix(q.x, n, 0, p, k);
      og = vix(q.gx, n, 0, p, k);
      if (q.gx_add.p) oa = vix(q.gx_add, n, 0, p, k);
      om = (long long)n * J * PK + rem;
    }
    float gm[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) gm[j] = (ok && j < J) ? __ldg(q.gm + om + (long long)j * PK) : 0.f;
    __syncthreads();   // previous tile's phase 2 done (also orders the wmT staging)
#pragma unroll
    for (int j = 0; j < 8; ++j) gms[j * MP_LD + tid] = gm[j];
    // phase 1: x tile straight into shared memory with cp.async (all Cin copies of the thread in flight, no
    // registers), overlapped with the gx read-modify-write, 16 channels in flight
    for (int c = 0; c < Cin; ++c) cp_async4(xs + c * MP_LD + tid, q.x.p + ox + (long long)c * q.x.sc, ok);
    for (int c0 = 0; c0 < Cin; c0 += 16) {
      float gv[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) gv[u] = (ok && c0 + u < Cin) ? q.gx.p[og + (long long)(c0 + u) * q.gx.sc] : 0.f;
      if (q.gx_add.p) {
#pragma unroll
        for (int u = 0; u < 16; ++u)
          if (ok && c0 + u < Cin) gv[u] += __ldg(q.gx_add.p + oa + (long long)(c0 + u) * q.gx_add.sc);
      }
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        if (c0 + u < Cin) {
          const float4 wa = *reinterpret_cast<const float4*>(wmT + (c0 + u) * 8);
          const float4 wb = *reinterpret_cast<const float4*>(wmT + (c0 + u) * 8 + 4);
          float s = gv[u];
          s = fmaf(wa.x, gm[0], s); s = fmaf(wa.y, gm[1], s); s = fmaf(wa.z, gm[2], s); s = fmaf(wa.w, gm[3], s);
          s = fmaf(wb.x, gm[4], s); s = fmaf(wb.y, gm[5], s); s = fmaf(wb.z, gm[6], s); s = fmaf(wb.w, gm[7], s);
          if (ok) q.gx.p[og + (long long)(c0 + u) * q.gx.sc] = s;
        }
      }
    }
    cp_async_wait_all();
    xs[Cin * MP_LD + tid] = ok ? 1.0f : 0.f;   // ones row (bias gradients)
    __syncthreads();
    // phase 2: gwm[j][c] += sum_g gm[j][g] x[c][g]
#pragma unroll
    for (int a = 0; a < MP_CG; ++a) {
      const int c = cl + 64 * a;
      if (c < C1) {
        const float* xr = xs + c * MP_LD;
        const float* g0 = gms + (2 * jg) * MP_LD;
        const float* g1 = g0 + MP_LD;
        float s0 = 0.f, s1 = 0.f;
#pragma unroll 4
        for (int g4 = 0; g4 < MP_TP; g4 += 4) {
          const float4 xv = *reinterpret_cast<const float4*>(xr + g4);
          const float4 a0 = *reinterpret_cast<const float4*>(g0 + g4);
          const float4 a1 = *reinterpret_cast<const float4*>(g1 + g4);
          s0 = fmaf(a0.x, xv.x, s0); s0 = fmaf(a0.y, xv.y, s0); s0 = fmaf(a0.z, xv.z, s0); s0 = fmaf(a0.w, xv.w, s0);
          s1 = fmaf(a1.x, xv.x, s1); s1 = fmaf(a1.y, xv.y, s1); s1 = fmaf(a1.z, xv.z, s1); s1 = fmaf(a1.w, xv.w, s1);
        }
        acc[a][0] += s0;
        acc[a][1] += s1;
      }
    }
  }
  float* dst = q.partial + (long long)blockIdx.x * J * C1;
#pragma unroll
  for (int a = 0; a < MP_CG; ++a) {
    const int c = cl + 64 * a;
    if (c < C1) {
      if (2 * jg < J) dst[(long long)(2 * jg) * C1 + c] = acc[a][0];
      if (2 * jg + 1 < J) dst[(long long)(2 * jg + 1) * C1 + c] = acc[a][1];
    }
  }
}

bool mproj_bwd_supported(int Cin, int J) {
  return J <= 8 && Cin + 1 <= 64 * MP_CG &&
         ((size_t)(Cin + 1 + 8) * MP_LD + (size_t)Cin * 8) * sizeof(float) <= (size_t)MAX_DYN_SMEM;
}

int mproj_bwd_ctas(long long G) {
  long long t = (G + MP_TP - 1) / MP_TP;
  const int cap = 2 * num_sms();
  return (int)(t < cap ? t : cap);
}

int launch_mproj_bwd(const MprojBwdParams& q, cudaStream_t st) {
  DSTD_REQUIRE(mproj_bwd_supported(q.Cin, q.J), DSTD_ERR_UNSUPPORTED, "mproj_bwd: Cin=%d J=%d outside limits", q.Cin, q.J);
  size_t smem = ((size_t)(q.Cin + 1 + 8) * MP_LD + (size_t)q.Cin * 8) * sizeof(float);
  if (smem > 48 * 1024) ensure_max_smem((const void*)mproj_bwd_kernel);
  mproj_bwd_kernel<<<mproj_bwd_ctas(q.G), 256, smem, st>>>(q);
  count_launch();
  return check_launch("mproj_bwd");
}

}  // namespace dstd

// ================================================================================= mproj forward
// m[n,j,p,k] = sum_c wm[j][c] x[n,c,p,k] + wm[j][Cin]   for the J = 4*nb reduction rows (conv_m1 / conv_m2 of every
// branch, model/dstdgcn.py:82) in one streaming pass over x: thread = column, 8 channels in flight, weights broadcast
// from shared memory.  HBM bound: reads the tile once, writes J/C of a tile.
namespace dstd {

__global__ void __launch_bounds__(256) mproj_fwd_kernel(MprojFwdParams q) {
  extern __shared__ __align__(16) float wmT[];   // [Cin+1][8]
  const int Cin = q.Cin, C1 = Cin + 1, J = q.J, PK = q.P * q.K;
  for (int i = threadIdx.x; i < C1 * 8; i += 256) {
    const int c = i >> 3, j = i & 7;
    wmT[i] = j < J ? __ldg(q.wm + (long long)j * C1 + c) : 0.f;
  }
  __syncthreads();
  const long long g = (long long)blockIdx.x * 256 + threadIdx.x;
  if (g >= q.G) return;
  const int n = (int)(g / PK);
  const int rem = (int)(g - (long long)n * PK);
  const int p = rem / q.K, k = rem - p * q.K;
  const float* xp = q.x.p + vix(q.x, n, 0, p, k);
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = wmT[Cin * 8 + j];
  for (int c0 = 0; c0 < Cin; c0 += 8) {
    float xv[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) xv[u] = (c0 + u < Cin) ? __ldg(xp + (long long)(c0 + u) * q.x.sc) : 0.f;
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      if (c0 + u < Cin) {
        const float4 wa = *reinterpret_cast<const float4*>(wmT + (c0 + u) * 8);
        const float4 wb = *reinterpret_cast<const float4*>(wmT + (c0 + u) * 8 + 4);
        acc[0] = fmaf(wa.x, xv[u], acc[0]); acc[1] = fmaf(wa.y, xv[u], acc[1]);
        acc[2] = fmaf(wa.z, xv[u], acc[2]); acc[3] = fmaf(wa.w, xv[u], acc[3]);
        acc[4] = fmaf(wb.x, xv[u], acc[4]); acc[5] = fmaf(wb.y, xv[u], acc[5]);
        acc[6] = fmaf(wb.z, xv[u], acc[6]); acc[7] = fmaf(wb.w, xv[u], acc[7]);
      }
    }
  }
  float* mp = q.m + (long long)n * J * PK + rem;
#pragma unroll
  for (int j = 0; j < 8; ++j)
    if (j < J) mp[(long long)j * PK] = acc[j];
}

int launch_mproj_fwd(const MprojFwdParams& q, cudaStream_t st) {
  DSTD_REQUIRE(q.J <= 8, DSTD_ERR_UNSUPPORTED, "mproj_fwd: J=%d > 8", q.J);
  const size_t smem = (size_t)(q.Cin + 1) * 8 * sizeof(float);
  mproj_fwd_kernel<<<cdiv(q.G, 256), 256, smem, st>>>(q);
  count_launch();
  return check_launch("mproj_fwd");
}

}  // namespace dstd
