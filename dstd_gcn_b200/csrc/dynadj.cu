// Dynamic adjacency construction of one DSTD-GC (model/dstdgcn.py:85-86 / :91-92) and its backward.
//
//   pd[p,v,w] = sum_{r,q} Wrm[p, r*P+q] * tanh(m1[r,q,v] - m2[r,q,w]) + brm[p]
//
// Both directions run on mma.sync m16n8k8 TF32 with 3xTF32 compensation (hi*hi + hi*lo + lo*hi), and the pairwise
// tanh tensor D [2P,K,K] (135-216 KB/sample in the reference) never leaves the SM:
//   forward : pd = Wrm D + brm, CTA = (sample, branch); the B fragments (D values) are computed in registers in
//             fragment layout, the A fragments (Wrm) come from shared memory.
//   backward: persistent CTAs over batch splits; per pair row v, gD = Wrm^T gxm, D evaluated in the accumulator
//             layout of gD, gS = alpha gD (1 - D^2) and its row/column sums (gm1 / gm2), and gWrm += gxm D^T kept in
//             registers across the split.
//   limits: P <= 40, K <= 40 (larger shapes run generic.cu).
#include "kernels.cuh"

namespace dstd {

// ================================================================================= forward
// pd[p][e] = sum_k Wrm[p][k] D[k][e] + brm[p] as mma.sync m16n8k8 TF32 (3xTF32) with the B fragments (the pairwise
// tanh values) COMPUTED IN REGISTERS in fragment layout: every D element is evaluated by exactly one lane, never stored,
// and feeds all 16-row tiles of p; the A fragments (Wrm) come from shared memory.  A CUDA-core version with a register
// tile of p was limited by the shared-memory return path (one broadcast weight delivery per FMA; DESIGN.md section 3).
__device__ __forceinline__ void fsplit3(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}
__device__ __forceinline__ void fmma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

template <int MT>
__global__ void __launch_bounds__(256) dynadj_fwd_mma_kernel(DynAdjFwdParams q, int WS) {
  extern __shared__ __align__(16) float smem[];
  const int P = q.P, K = q.K, PK = P * K, KK = K * K, P2 = 2 * P;
  float* ms = smem;                        // [4][PK]
  float* wsm = ms + ((4 * PK + 3) & ~3);   // [MT*16][WS]  Wrm, zero beyond P rows / 2P columns
  float* bs = wsm + MT * 16 * WS;          // [MT*16]
  const int n = blockIdx.x, b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int fg = lane >> 2, ft = lane & 3;
  const float* mg = q.m + ((long long)(n * q.nb + b) * 4) * PK;
  const float* wrm = q.w_rm[b];
  float* pdg = q.pd + (long long)(n * q.nb + b) * P * KK;
  for (int i = tid; i < 4 * PK; i += 256) ms[i] = __ldg(mg + i);
  for (int i = tid; i < MT * 16 * WS; i += 256) {
    const int p = i / WS, k = i - p * WS;
    wsm[i] = (p < P && k < P2) ? __ldg(wrm + (long long)p * P2 + k) : 0.f;
  }
  for (int i = tid; i < MT * 16; i += 256) bs[i] = i < P ? __ldg(q.b_rm[b] + i) : 0.f;
  __syncthreads();

  const int NT = (KK + 7) >> 3, ntask = (NT + 1) >> 1;
  const int ksteps = (P2 + 7) >> 3;
  for (int task = warp; task < ntask; task += 8) {
    int vi[2], wi[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int e = min((2 * task + i) * 8 + fg, KK - 1);
      vi[i] = e / K;
      wi[i] = e - vi[i] * K;
    }
    float acc[MT][2][4];
#pragma unroll
    for (int m = 0; m < MT; ++m)
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        acc[m][i][0] = acc[m][i][1] = bs[m * 16 + fg];
        acc[m][i][2] = acc[m][i][3] = bs[m * 16 + fg + 8];
      }
    for (int ks = 0; ks < ksteps; ++ks) {
      const int ka = ks * 8 + ft, kb = ka + 4;
      uint32_t bh[2][2], bl[2][2];
      {
        const int ra = ka >= P ? 1 : 0, rb = kb >= P ? 1 : 0;
        const float* m1a = ms + ra * PK + (ka - ra * P) * K;
        const float* m1b = ms + rb * PK + (kb - rb * P) * K;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const float da = ka < P2 ? fast_tanh(m1a[vi[i]] - m1a[2 * PK + wi[i]]) : 0.f;
          const float db = kb < P2 ? fast_tanh(m1b[vi[i]] - m1b[2 * PK + wi[i]]) : 0.f;
          fsplit3(da, bh[i][0], bl[i][0]);
          fsplit3(db, bh[i][1], bl[i][1]);
        }
      }
#pragma unroll
      for (int m = 0; m < MT; ++m) {
        const float* wr = wsm + (m * 16 + fg) * WS + ks * 8 + ft;
        uint32_t ah[4], al[4];
        fsplit3(wr[0], ah[0], al[0]);
        fsplit3(wr[8 * WS], ah[1], al[1]);
        fsplit3(wr[4], ah[2], al[2]);
        fsplit3(wr[8 * WS + 4], ah[3], al[3]);
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          fmma_tf32(acc[m][i], ah, bh[i]);
          fmma_tf32(acc[m][i], ah, bl[i]);
          fmma_tf32(acc[m][i], al, bh[i]);
        }
      }
    }
#pragma unroll
    for (int m = 0; m < MT; ++m)
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int e = (2 * task + i) * 8 + 2 * ft;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int p = m * 16 + fg + 8 * h;
          if (p < P) {
            if (e < KK) pdg[(long long)p * KK + e] = acc[m][i][2 * h];
            if (e + 1 < KK) pdg[(long long)p * KK + e + 1] = acc[m][i][2 * h + 1];
          }
        }
      }
  }
}

template <int MT>
static int dynadj_fwd_mma_launch(const DynAdjFwdParams& q, cudaStream_t st) {
  int WS = (2 * q.P + 7) / 8 * 8;
  while ((WS / 4) % 2 == 0) WS += 4;          // WS/4 odd: conflict-free A-fragment loads
  const size_t smem = ((size_t)((4 * q.P * q.K + 3) & ~3) + (size_t)MT * 16 * WS + MT * 16) * sizeof(float);
  auto kern = dynadj_fwd_mma_kernel<MT>;
  if (smem > 48 * 1024) ensure_max_smem((const void*)kern);
  kern<<<dim3(q.N, q.nb), 256, smem, st>>>(q, WS);
  count_launch();
  return check_launch("dynadj_fwd_mma");
}

bool dynadj_supported(int P, int K) { return P >= 1 && P <= 40 && K >= 1 && K <= 40; }

int launch_dynadj_fwd(const DynAdjFwdParams& q, cudaStream_t st) {
  DSTD_REQUIRE(dynadj_supported(q.P, q.K), DSTD_ERR_UNSUPPORTED,
               "dynadj_fwd: P=%d K=%d outside the compiled tile limits (P, K <= 40)", q.P, q.K);
  if (q.P <= 16) return dynadj_fwd_mma_launch<1>(q, st);
  if (q.P <= 32) return dynadj_fwd_mma_launch<2>(q, st);
  return dynadj_fwd_mma_launch<3>(q, st);
}

// ================================================================================= backward

// batch splits = persistent CTAs per branch: one CTA per SM in total (the tensor-path kernel keeps its gWrm tile in
// registers across its samples, so fewer, longer CTAs amortise the prologue and the partial write-out)
int dynadj_bwd_splits(int N, int nb) {
  int s = num_sms() / (nb < 1 ? 1 : nb);
  if (s < 1) s = 1;
  return N < s ? N : s;
}

// ---- tensor-path backward.  Per (sample, branch) and per row v of the pair grid, with channels k = 0..2P-1:
//   (i)   gD[k][w]  = sum_p Wrm[p][k] gxm[p][v][w]            m16n8k8, A = Wrm^T (register fragments, pre-split),
//                                                             B = gxm chunk (shared memory)
//   (ii)  D[k][w]   = tanh(m1[k][v] - m2[k][w]) evaluated IN THE ACCUMULATOR LAYOUT of (i): the lane that holds
//         gD[k][w] also computes D[k][w], so gS = alpha gD (1 - D^2) and its row/column sums (gm1 / gm2) are register
//         work (quad shuffles for the row sums; the column sums stay in registers over the warp's v rows)
//   (iii) gWrm[p][k] += sum_w gxm[p][v][w] D[k][w]             m16n8k8 with the SAME D registers as B fragments (the
//         k-slot permutation slot t <-> pair 2t, slot t+4 <-> pair 2t+1 makes the C layout of (i) a B layout) and
//         A = gxm chunk rows; accumulators live in registers across the whole batch split.
// A warp owns one 16-channel tile (kt) and every VS-th row v.  All products are 3xTF32 (hi*hi + hi*lo + lo*hi); every
// cross-warp sum is done in a fixed order (no atomics), so results are run-to-run identical.  A CUDA-core version that
// rebuilt D in shared memory was limited by the shared-memory return path (DESIGN.md section 3).
template <int KSTEPS, int WT>
__global__ void __launch_bounds__(384) dynadj_bwd_mma_kernel(DynAdjBwdParams q, int KT, int VS) {
  constexpr int MTP = (KSTEPS + 1) / 2;   // 16-row tiles of p
  constexpr int PR = MTP * 16;            // chunk rows (>= KSTEPS * 8), rows >= P stay zero
  constexpr int CS = 40;                  // chunk row stride: 8 mod 32 -> conflict-free fragment loads; cols >= K zero
  constexpr int WC = WT * 8;
  extern __shared__ __align__(16) float smem[];
  const int P = q.P, K = q.K, PK = P * K, KK = K * K, P2 = 2 * P, P21 = P2 + 1;
  const int pk4 = (4 * PK + 3) & ~3;
  float* ms = smem;                                // [4][PK]
  float* gm1s = ms + pk4;                          // [2][PK]   gm1 rows of the current sample
  float* chunk = gm1s + ((2 * PK + 3) & ~3);       // [2][VS][PR][CS]
  float* gA = chunk + 2 * VS * PR * CS;            // [KK]
  float* wfin = gA + ((KK + 3) & ~3);              // [VS][P][2P+1]  per-v-split partials of gWrm (+ bias column)
  float* csb = wfin + ((VS * P * P21 + 3) & ~3);   // [VS][KT*16][WC]  per-v-split column sums of gS
  float* red = csb + VS * KT * 16 * WC;            // [32]
  const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int fg = lane >> 2, ft = lane & 3;
  const int kt = warp % KT, vs = warp / KT;
  const int b = blockIdx.y;
  const float alpha = q.alpha ? __ldg(q.alpha) : 1.0f;
  const float* wrm = q.w_rm[b];

  for (int i = tid; i < 2 * VS * PR * CS; i += nthr) chunk[i] = 0.f;
  for (int i = tid; i < KK; i += nthr) gA[i] = 0.f;
  for (int i = tid; i < VS * P * P21; i += nthr) wfin[i] = 0.f;

  // channels of this lane's two accumulator rows, and where their m rows start (-1: beyond 2P)
  const int kc0 = kt * 16 + fg, kc1 = kc0 + 8;
  const int r0 = kc0 >= P ? 1 : 0, r1 = kc1 >= P ? 1 : 0;
  const int mo0 = kc0 < P2 ? r0 * PK + (kc0 - r0 * P) * K : -1;   // m1 row; the m2 row is 2*PK further
  const int mo1 = kc1 < P2 ? r1 * PK + (kc1 - r1 * P) * K : -1;

  // Two spare (padding) channel rows of the last tile, when there are any, turn the two plain reductions of gxm into
  // by-products of the MMAs: row 2P of D is all ones, so column 2P of (iii) is the bias gradient sum_e gxm[p][e];
  // row 2P+1 of Wrm^T is all ones, so that row of (i) is the static-adjacency gradient sum_p gxm[p][v][w].
  const bool spare = P2 + 2 <= KT * 16;
  const int kb = spare ? P2 : -1, ka = spare ? P2 + 1 : -1;

  // A fragments of (i): Wrm^T tile, split once
  uint32_t wah[KSTEPS][4], wal[KSTEPS][4];
#pragma unroll
  for (int ks = 0; ks < KSTEPS; ++ks) {
    const int p0 = ks * 8 + ft, p1 = p0 + 4;
    const float o0 = (kc0 == ka) ? 1.f : 0.f, o1 = (kc1 == ka) ? 1.f : 0.f;
    const float a0 = p0 < P ? (kc0 < P2 ? __ldg(wrm + (long long)p0 * P2 + kc0) : o0) : 0.f;
    const float a1 = p0 < P ? (kc1 < P2 ? __ldg(wrm + (long long)p0 * P2 + kc1) : o1) : 0.f;
    const float a2 = p1 < P ? (kc0 < P2 ? __ldg(wrm + (long long)p1 * P2 + kc0) : o0) : 0.f;
    const float a3 = p1 < P ? (kc1 < P2 ? __ldg(wrm + (long long)p1 * P2 + kc1) : o1) : 0.f;
    fsplit3(a0, wah[ks][0], wal[ks][0]);
    fsplit3(a1, wah[ks][1], wal[ks][1]);
    fsplit3(a2, wah[ks][2], wal[ks][2]);
    fsplit3(a3, wah[ks][3], wal[ks][3]);
  }
  float accW[MTP][2][4];
#pragma unroll
  for (int m = 0; m < MTP; ++m)
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) accW[m][nt][i] = 0.f;
  float galpha = 0.f, gbias = 0.f;          // gbias (no spare rows only): row sum of gxm for the (j, p) row this thread owns
  const int hb_j = tid / P, hb_p = tid - hb_j * P;

  const int nsteps_v = (K + VS - 1) / VS;
  const int nsamp = (q.N - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const long long total = (long long)nsamp * nsteps_v;

  auto prefetch = [&](long long st) {
    const int n = (int)blockIdx.x + (int)(st / nsteps_v) * (int)gridDim.x;
    const int v0 = (int)(st % nsteps_v) * VS;
    const float* src = q.gxm + ((long long)n * q.nb + b) * P * KK;
    float* dst = chunk + (st & 1) * VS * PR * CS;
    for (int j = 0; j < VS; ++j) {
      const int v = v0 + j;
      if (v >= K) break;
      for (int i = tid; i < PK; i += nthr) {
        const int p = i / K, w = i - p * K;
        cp_async4(dst + (j * PR + p) * CS + w, src + (long long)p * KK + v * K + w, true);
      }
    }
  };
  if (total > 0) prefetch(0);

  float mbv[WT][4], cs[WT][4];
  for (long long st = 0; st < total; ++st) {
    const int n = (int)blockIdx.x + (int)(st / nsteps_v) * (int)gridDim.x;
    const int si = (int)(st % nsteps_v), v0 = si * VS;
    const long long nb_ = (long long)n * q.nb + b;
    if (si == 0) {   // new sample: its reduction rows
      __syncthreads();
      const float* mg = q.m + nb_ * 4 * PK;
      for (int i = tid; i < 4 * PK; i += nthr) ms[i] = __ldg(mg + i);
    }
    cp_async_wait_all();
    __syncthreads();                       // chunk st landed (and ms); everyone is done with the other buffer
    if (st + 1 < total) prefetch(st + 1);
    if (si == 0) {
#pragma unroll
      for (int wt = 0; wt < WT; ++wt) {
        const int w = wt * 8 + 2 * ft;
        mbv[wt][0] = (mo0 >= 0 && w < K) ? ms[mo0 + 2 * PK + w] : 0.f;
        mbv[wt][1] = (mo0 >= 0 && w + 1 < K) ? ms[mo0 + 2 * PK + w + 1] : 0.f;
        mbv[wt][2] = (mo1 >= 0 && w < K) ? ms[mo1 + 2 * PK + w] : 0.f;
        mbv[wt][3] = (mo1 >= 0 && w + 1 < K) ? ms[mo1 + 2 * PK + w + 1] : 0.f;
        cs[wt][0] = cs[wt][1] = cs[wt][2] = cs[wt][3] = 0.f;
      }
    }
    const float* cbuf = chunk + (st & 1) * VS * PR * CS;
    const int v = v0 + vs;
    if (v < K) {
      const float* ch = cbuf + vs * PR * CS;
      const float ma0 = mo0 >= 0 ? ms[mo0 + v] : 0.f, ma1 = mo1 >= 0 ? ms[mo1 + v] : 0.f;
      float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
      for (int wt = 0; wt < WT; ++wt) {   // tiles beyond K (only when K <= 8 (WT - 1)) see zero chunks: no guard, so
        {                                   // that the scheduler can interleave the tiles' instruction streams
          // (i) gD tile: three independent accumulation chains (hi*hi, hi*lo, lo*hi)
          float gd[4] = {0.f, 0.f, 0.f, 0.f}, gd1[4] = {0.f, 0.f, 0.f, 0.f}, gd2[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int ks = 0; ks < KSTEPS; ++ks) {
            const float* bp = ch + (ks * 8 + ft) * CS + wt * 8 + fg;
            uint32_t bh[2], bl[2];
            fsplit3(bp[0], bh[0], bl[0]);
            fsplit3(bp[4 * CS], bh[1], bl[1]);
            fmma_tf32(gd, wah[ks], bh);
            fmma_tf32(gd1, wah[ks], bl);
            fmma_tf32(gd2, wal[ks], bh);
          }
          // (ii) D in the accumulator layout, gS and its sums
          float d[4];
          d[0] = fast_tanh(ma0 - mbv[wt][0]);
          d[1] = fast_tanh(ma0 - mbv[wt][1]);
          d[2] = fast_tanh(ma1 - mbv[wt][2]);
          d[3] = fast_tanh(ma1 - mbv[wt][3]);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            gd[i] += gd1[i] + gd2[i];
            const float gs = alpha * gd[i] * (1.0f - d[i] * d[i]);
            cs[wt][i] += gs;
            if (i < 2) rs0 += gs;
            else rs1 += gs;
          }
          if (spare) {                       // warp-uniform except for the two lanes rows that own kb / ka
            if (kc0 == kb) d[0] = d[1] = 1.f;
            if (kc1 == kb) d[2] = d[3] = 1.f;
            const int w = wt * 8 + 2 * ft;
            if (kc0 == ka) {
              if (w < K) gA[v * K + w] += gd[0];
              if (w + 1 < K) gA[v * K + w + 1] += gd[1];
            }
            if (kc1 == ka) {
              if (w < K) gA[v * K + w] += gd[2];
              if (w + 1 < K) gA[v * K + w + 1] += gd[3];
            }
          }
          // (iii) gWrm tile: B = D (two channel n-tiles), A = gxm rows
          uint32_t dh[2][2], dl[2][2];
          fsplit3(d[0], dh[0][0], dl[0][0]);
          fsplit3(d[1], dh[0][1], dl[0][1]);
          fsplit3(d[2], dh[1][0], dl[1][0]);
          fsplit3(d[3], dh[1][1], dl[1][1]);
#pragma unroll
          for (int m = 0; m < MTP; ++m) {
            const float2 x0 = *reinterpret_cast<const float2*>(ch + (m * 16 + fg) * CS + wt * 8 + 2 * ft);
            const float2 x1 = *reinterpret_cast<const float2*>(ch + (m * 16 + fg + 8) * CS + wt * 8 + 2 * ft);
            uint32_t ah[4], al[4];
            fsplit3(x0.x, ah[0], al[0]);
            fsplit3(x1.x, ah[1], al[1]);
            fsplit3(x0.y, ah[2], al[2]);
            fsplit3(x1.y, ah[3], al[3]);
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
              fmma_tf32(accW[m][nt], ah, dh[nt]);
              fmma_tf32(accW[m][nt], ah, dl[nt]);
              fmma_tf32(accW[m][nt], al, dh[nt]);
            }
          }
        }
      }
      // gm1[k][v]: sum over w = over the quad's columns; this warp is the only writer of (k, v)
      rs0 += __shfl_xor_sync(0xffffffffu, rs0, 1);
      rs0 += __shfl_xor_sync(0xffffffffu, rs0, 2);
      rs1 += __shfl_xor_sync(0xffffffffu, rs1, 1);
      rs1 += __shfl_xor_sync(0xffffffffu, rs1, 2);
      if (ft == 0) {
        if (mo0 >= 0) gm1s[mo0 + v] = rs0;
        if (mo1 >= 0) gm1s[mo1 + v] = rs1;
      }
    }
    // without spare rows (2P a multiple of 16): bias gradient (row sums) and static-adjacency gradient (column sums)
    // as plain reductions over the chunks of this step
    if (!spare) {
      if (tid < VS * P && v0 + hb_j < K) {
        const float* row = cbuf + (hb_j * PR + hb_p) * CS;
        float sacc = 0.f;
        for (int w = 0; w < K; ++w) sacc += row[w];
        gbias += sacc;
      }
      for (int i = tid; i < VS * K; i += nthr) {
        const int j = i / K, w = i - j * K, vv = v0 + j;
        if (vv < K) {
          const float* col = cbuf + j * PR * CS + w;
          float sacc = 0.f;
          for (int p = 0; p < P; ++p) sacc += col[p * CS];
          gA[vv * K + w] += sacc;
        }
      }
    }
    if (si == nsteps_v - 1) {   // sample finished: column sums of the v-splits -> gm2 (fixed order); gm rows go out
      float* cw = csb + (vs * KT + kt) * 16 * WC;
#pragma unroll
      for (int wt = 0; wt < WT; ++wt) {
        const int w = wt * 8 + 2 * ft;
        cw[fg * WC + w] = cs[wt][0];
        cw[fg * WC + w + 1] = cs[wt][1];
        cw[(fg + 8) * WC + w] = cs[wt][2];
        cw[(fg + 8) * WC + w + 1] = cs[wt][3];
      }
      __syncthreads();
      float* gmg = q.gm + nb_ * 4 * PK;
      for (int i = tid; i < 2 * PK; i += nthr) {
        gmg[i] = gm1s[i];                                       // gm1 rows
        const int k = i / K, w = i - k * K;                     // gm2[k][w] = -sum_v gS
        float sacc = 0.f;
        for (int j = 0; j < VS; ++j) sacc += csb[(j * KT * 16 + k) * WC + w];
        gmg[2 * PK + i] = -sacc;
      }
    }
  }

  // per-split partials: the gWrm tiles of the v-split warps (+ bias column) are summed in a fixed order
  __syncthreads();
  {
    float* wv = wfin + vs * P * P21;
#pragma unroll
    for (int m = 0; m < MTP; ++m)
#pragma unroll
      for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int pp = m * 16 + fg + 8 * (i >> 1), kk = kt * 16 + nt * 8 + 2 * ft + (i & 1);
          if (pp < P && (kk < P2 || kk == kb)) wv[pp * P21 + kk] = accW[m][nt][i];
        }
    if (!spare && tid < VS * P) wfin[(hb_j * P + hb_p) * P21 + P2] = gbias;
  }
  __syncthreads();
  // alpha gradient sum gxm . pd without reading pd: pd = Wrm D + brm, so it equals <Wrm, gWrm> + <brm, gbrm> (unscaled)
  const long long sb = (long long)blockIdx.x * q.nb + b;
  float* pw = q.part_wrm + sb * P * P21;
  const float* brm = q.b_rm[b];
  for (int i = tid; i < P * P21; i += nthr) {
    float sacc = 0.f;
    for (int j = 0; j < VS; ++j) sacc += wfin[j * P * P21 + i];
    pw[i] = alpha * sacc;
    const int pp = i / P21, kk = i - pp * P21;
    galpha = fmaf(sacc, kk < P2 ? __ldg(wrm + (long long)pp * P2 + kk) : __ldg(brm + pp), galpha);
  }
  float* pa = q.part_adj + sb * KK;
  for (int i = tid; i < KK; i += nthr) pa[i] = gA[i];
  const float ga = block_sum(galpha, red);
  if (tid == 0) q.part_alpha[sb] = ga;
}

template <int KSTEPS, int WT>
static int dynadj_bwd_mma_launch(const DynAdjBwdParams& q, cudaStream_t st) {
  constexpr int MTP = (KSTEPS + 1) / 2, PR = MTP * 16, CS = 40;
  const int P = q.P, K = q.K;
  const int KT = (2 * P + 15) / 16;
  int VS = 12 / KT;
  if (VS > 4) VS = 4;
  if (VS < 1) VS = 1;
  const size_t fl = (size_t)((4 * P * K + 3) & ~3) + ((2 * P * K + 3) & ~3) + (size_t)2 * VS * PR * CS +
                    ((K * K + 3) & ~3) + ((VS * P * (2 * P + 1) + 3) & ~3) + (size_t)VS * KT * 16 * WT * 8 + 32;
  const size_t smem = fl * sizeof(float);
  auto kern = dynadj_bwd_mma_kernel<KSTEPS, WT>;
  if (smem > 48 * 1024) ensure_max_smem((const void*)kern);
  kern<<<dim3(q.S, q.nb), KT * VS * 32, smem, st>>>(q, KT, VS);
  count_launch();
  return check_launch("dynadj_bwd_mma");
}

int launch_dynadj_bwd(const DynAdjBwdParams& q, cudaStream_t st) {
  DSTD_REQUIRE(dynadj_supported(q.P, q.K), DSTD_ERR_UNSUPPORTED,
               "dynadj_bwd: P=%d K=%d outside the compiled tile limits (P, K <= 40)", q.P, q.K);
  const int ks = q.P <= 24 ? 3 : 5, wt = q.K <= 24 ? 3 : q.K <= 32 ? 4 : 5;
  if (ks == 3 && wt == 3) return dynadj_bwd_mma_launch<3, 3>(q, st);
  if (ks == 3 && wt == 4) return dynadj_bwd_mma_launch<3, 4>(q, st);
  if (ks == 3 && wt == 5) return dynadj_bwd_mma_launch<3, 5>(q, st);
  if (ks == 5 && wt == 3) return dynadj_bwd_mma_launch<5, 3>(q, st);
  if (ks == 5 && wt == 4) return dynadj_bwd_mma_launch<5, 4>(q, st);
  return dynadj_bwd_mma_launch<5, 5>(q, st);
}

}  // namespace dstd
