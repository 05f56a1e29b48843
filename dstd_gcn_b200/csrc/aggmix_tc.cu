// Fused adjacency aggregation + channel mix, forward, with the channel contraction on the 5th-generation tensor cores
// (tcgen05.mma kind::tf32, accumulators in TMEM) -- the sm_100a path of model/dstdgcn.py:81 + :87/:93 (+ :150/:161/:248).
//
// Persistent CTAs (one per SM).  The conv_f weights of every branch stay resident in shared memory for the life of the
// CTA, already split into TF32 "hi" and "lo" parts and laid out as UMMA K-major core matrices by the pack kernel.
// Per work item (sample n, chunk of PCH frames):
//   1. cp.async staging of the x chunk and the raw dynamic adjacency; xm = alpha*pd + A_eff formed in shared memory
//   2. per branch b: CUDA-core aggregation  xa_b[c][pos] = sum_v x[c][l,v] xm_b[l][v][w]  written straight into the UMMA
//      A-operand tile (positions = M rows, channels = K, hi/lo split on the fly), then ONE elected thread issues
//      3 x (KD/8) tcgen05.mma (hi*hi + hi*lo + lo*hi: split-TF32 error compensation, needed for the 1e-4
//      parity budget) accumulating D[pos][o] over both branches in TMEM; completion through tcgen05.commit -> mbarrier
//   3. epilogue: tcgen05.ld (32 lanes x 32 columns per warp) -> (+ skip) -> coalesced stores of out[o][pos]
// Tile format (validated in isolation by tools/umma_test.cu): K-major, no swizzle, 8 x 16 B core matrices,
//   element (row r, k) at (r/8)*SBO + (k/4)*LBO + (r%8)*16 + (k%4)*4 bytes with LBO = 144 B (not 128: the 16-byte skew
//   makes the lane = channel stores of the aggregation bank-conflict free) and SBO = (KD/4)*LBO.
#include "kernels.cuh"
#include "umma.cuh"

namespace dstd {

constexpr int TC_LBO_F = 36;   // floats between K-adjacent core matrices (144 B)

__host__ __device__ __forceinline__ int tc_off(int r, int k, int sbo_f) {
  return (r >> 3) * sbo_f + (k >> 2) * TC_LBO_F + ((r & 7) << 2) + (k & 3);
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint64_t tc_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;   // descriptor version (sm_100)
  return d;                 // layout type 0: no swizzle
}

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc),
      "r"(acc)
      : "memory");
}

// bounded wait (a malformed pipeline must fail loudly, not hang the GPU)
__device__ __forceinline__ bool mbar_wait(uint32_t mbar, uint32_t parity) {
  uint32_t done = 0;
  for (int it = 0; it < (1 << 22) && !done; ++it) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}\n"
        : "=r"(done)
        : "r"(mbar), "r"(parity)
        : "memory");
  }
  return done != 0;
}

__device__ __forceinline__ void mma_tf32_sync(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
  // truncation split on the full-rate logic pipe (cvt.rna.tf32 is quarter rate): |lo| < 2^-10 |x|, x == hi + lo exactly
  hi = __uint_as_float(__float_as_uint(x) & 0xffffe000u);
  lo = x - hi;
}

constexpr int TC_NT = 512;   // 16 warps per persistent CTA

template <int WH>
__global__ void __launch_bounds__(TC_NT, 1) aggmix_fwd_tc_kernel(AggMixParams q, int KD, int NP, int tmem_cols, int* err_flag) {
  extern __shared__ __align__(16) float smem[];
  constexpr int KP = 2 * WH;
  const int K = q.K, P = q.P, KK = K * K, Cin = q.Cin, Cout = q.Cout, nb = q.nb, PCH = q.PCH;
  const int sbo_f = (KD / 4) * TC_LBO_F;
  // rows (positions) actually written; the M = 128 descriptor reads on into the following buffers for the unused rows,
  // which only produces D rows nobody loads
  const int a_tile_f = ((PCH * K + 7) / 8) * sbo_f;
  const int b_tile_f = (NP / 8) * sbo_f;             // NP rows (output channels, padded to 16)
  const int npos_max = PCH * K;
  const int XS_LD = ((npos_max + 3) / 8) * 8 + 4;    // == 4 (mod 8): the A-fragment loads (rows fg, columns ft) hit 32 banks
  float* a_hi = smem;                                // UMMA A operand tiles
  float* a_lo = a_hi + a_tile_f;
  float* b_img = a_lo + a_tile_f;                    // [nb][hi|lo][b_tile_f]   resident weights
  float* xs = b_img + nb * 2 * b_tile_f;             // [Cin][XS_LD]
  float* xms = xs + ((Cin * XS_LD + 3) & ~3);        // [nb][PCH][K][KP]
  float* aeff = xms + nb * PCH * K * KP;             // [nb][K*K]
  float* pdr = aeff + ((nb * KK + 3) & ~3);          // [nb][PCH][K*K]
  // layer-skip chunk [Cout][XS_LD] (only when a skip is fused): staged with the lanes walking the SKIP tensor's own
  // contiguous direction, because the skip is kept in the other memory order (it is the block input)
  int* rowtab = reinterpret_cast<int*>(pdr + ((nb * PCH * KK + 3) & ~3));   // [nb*PCH*K]  (b*PCH + l) << 8 | v per row
  float* csum = reinterpret_cast<float*>(rowtab + ((nb * PCH * K + 3) & ~3));   // [nb*PCH*K]  column sums of xm (the bias row)
  float* sks = csum + ((nb * PCH * K + 3) & ~3);
  uint64_t* mbar = reinterpret_cast<uint64_t*>(sks + (q.skip.p ? ((Cout * XS_LD + 3) & ~3) : 0));
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mbar + 1);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float alpha = q.alpha ? __ldg(q.alpha) : 1.0f;
  const int nchunk = (P + PCH - 1) / PCH;
  const long long nitems = (long long)q.N * nchunk;

  // TMA bulk copies (cp.async.bulk): the weight image once per CTA, the raw dynamic adjacency of every item (one
  // contiguous block per branch) when K*K*4 is a multiple of 16; otherwise 4-byte cp.async per element
  __shared__ uint64_t pd_bar;
  const bool pd_bulk = (KK & 3) == 0 && (reinterpret_cast<uintptr_t>(q.pd) & 15) == 0;
  uint32_t pd_phase = 0;
  // ---- once per CTA: resident weights, static adjacency, zeroed A tiles (pad rows of K must read as 0), TMEM, mbarrier
  {
    if (tid == 0) {
      umma::mbar_init(&pd_bar, 1);
      umma::mbar_init_fence();
      umma::mbar_expect_tx(&pd_bar, (uint32_t)(nb * 2 * b_tile_f * 4));
      umma::bulk_g2s(b_img, q.wtc, (uint32_t)(nb * 2 * b_tile_f * 4), &pd_bar);
    }
    for (int i = tid; i < 2 * a_tile_f; i += TC_NT) a_hi[i] = 0.f;
    for (int i = tid; i < nb * KK; i += TC_NT) {
      const int b = i / KK, e = i - b * KK;
      float a = __ldg(q.adj[b] + e);
      if (q.adj_w[b]) a *= __ldg(q.adj_w[b] + e);
      if (q.adj_r[b]) a += __ldg(q.adj_r[b] + e);
      aeff[i] = a;
    }
    if (tid == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(mbar)));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int i = tid; i < nb * PCH * K; i += TC_NT) rowtab[i] = ((i / K) << 8) | (i % K);
    __syncthreads();               // the barrier initialisation is visible to every waiter
    umma::mbar_wait(&pd_bar, pd_phase);
    pd_phase ^= 1;
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  }
  const uint32_t tmem_d = *tmem_slot;
  const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(NP >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  const uint32_t lbo_b = TC_LBO_F * 4, sbo_b = (uint32_t)sbo_f * 4;
  uint32_t phase = 0;
  bool ok = true;

  // optional per-phase cycle counters (-DDSTD_PHASE_TIMING, printed by CTA 0)
#ifdef DSTD_PHASE_TIMING
  long long tph[6] = {0, 0, 0, 0, 0, 0}, tlast = clock64();
#define TPH(i) do { long long _t = clock64(); tph[i] += _t - tlast; tlast = _t; } while (0)
#else
#define TPH(i) do {} while (0)
#endif
  for (long long item = blockIdx.x; item < nitems; item += gridDim.x) {
    const int n = (int)(item / nchunk), p0 = (int)(item - (long long)n * nchunk) * PCH;
    const int pv = min(PCH, P - p0);
    const int npos = pv * K;

    // ---- 1. stage x chunk + raw dynamic adjacency
    {
      constexpr int TNS = 4;   // 128 position slots
      int poff[TNS];
#pragma unroll
      for (int i = 0; i < TNS; ++i) {
        const int j = lane + 32 * i;
        const int l = j / K, k = j - l * K;
        poff[i] = j < npos ? (int)(l * q.x.sp + k * q.x.sk) : -1;
      }
      const float* xb = q.x.p + (long long)n * q.x.sn + (long long)p0 * q.x.sp;
      for (int c = warp; c < Cin; c += TC_NT / 32) {
#pragma unroll
        for (int i = 0; i < TNS; ++i)
          if (poff[i] >= 0) cp_async4(xs + c * XS_LD + lane + 32 * i, xb + (long long)c * q.x.sc + poff[i], true);
      }
      if (pd_bulk) {
        if (tid == 0) {
          umma::mbar_expect_tx(&pd_bar, (uint32_t)(nb * pv * KK * 4));
          for (int b = 0; b < nb; ++b)
            umma::bulk_g2s(pdr + b * PCH * KK, q.pd + ((long long)(n * nb + b) * P + p0) * KK, (uint32_t)(pv * KK * 4), &pd_bar);
        }
      } else {
        for (int b = 0; b < nb; ++b) {
          const float* pdl = q.pd + ((long long)(n * nb + b) * P + p0) * KK;
          for (int i = tid; i < pv * KK; i += TC_NT) cp_async4(pdr + b * PCH * KK + i, pdl + i, true);
        }
      }
      if (q.skip.p) {
        // lane order (k major, l minor) when the skip is contiguous along p, else the position order
        const bool p_fast = q.skip.sp == 1 && q.skip.sk != 1;
        int soff[TNS], sdst[TNS];
#pragma unroll
        for (int i = 0; i < TNS; ++i) {
          const int j = lane + 32 * i;
          int l, k;
          if (p_fast) { k = j / pv; l = j - k * pv; } else { l = j / K; k = j - l * K; }
          soff[i] = j < npos ? (int)(l * q.skip.sp + k * q.skip.sk) : -1;
          sdst[i] = l * K + k;
        }
        const float* sb = q.skip.p + (long long)n * q.skip.sn + (long long)p0 * q.skip.sp;
        for (int o = warp; o < Cout; o += TC_NT / 32) {
#pragma unroll
          for (int i = 0; i < TNS; ++i)
            if (soff[i] >= 0) cp_async4(sks + o * XS_LD + sdst[i], sb + (long long)o * q.skip.sc + soff[i], true);
        }
      }
      cp_async_wait_all();
      if (pd_bulk) {
        umma::mbar_wait(&pd_bar, pd_phase);
        pd_phase ^= 1;
      }
      __syncthreads();
      TPH(0);   // staging
      // element-parallel; the row decode comes from a table built once per CTA (no runtime division in the loop)
      for (int i = tid; i < nb * PCH * K * KP; i += TC_NT) {
        const int row = i / KP, w = i - row * KP;
        const int info = rowtab[row], bl = info >> 8, v = info & 255;   // bl = b * PCH + l
        const int b = bl >= PCH ? 1 : 0, l = bl - b * PCH;
        float val = 0.f;
        if (w < K && l < pv) {
          const int e = q.adj_t ? (w * K + v) : (v * K + w);
          val = fmaf(alpha, pdr[bl * KK + e], aeff[b * KK + e]);
        }
        xms[i] = val;
      }
      __syncthreads();
      // column sums of xm (they carry the conv_f bias through the ones row of the A tile) for every (branch, frame) at
      // once: one thread per column, off the per-branch critical path (they were computed by four warps inside the
      // branch loop, a 22-long dependent chain in front of every MMA issue)
      for (int i = tid; i < nb * PCH * K; i += TC_NT) {
        const int bl = i / K, w = i - bl * K;
        const float* xm_l = xms + (bl * K) * KP + w;
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;     // four independent chains: the loads overlap
        int v = 0;
        for (; v + 4 <= K; v += 4) {
          s0 += xm_l[v * KP];
          s1 += xm_l[(v + 1) * KP];
          s2 += xm_l[(v + 2) * KP];
          s3 += xm_l[(v + 3) * KP];
        }
        for (; v < K; ++v) s0 += xm_l[v * KP];
        csum[i] = (s0 + s1) + (s2 + s3);
      }
      // The tiles leave no room for a second staging buffer: pull the next item's chunk into L2 while this one computes,
      // so that its cp.async staging pays L2 instead of HBM latency
      {
        const long long nxt = item + gridDim.x;
        if (nxt < nitems) {
          const int n2 = (int)(nxt / nchunk), q0 = (int)(nxt - (long long)n2 * nchunk) * PCH;
          const int pv2 = min(PCH, P - q0);
          auto pf_rows = [&](const float* base, long long row_stride, int rows, int run) {   // rows of `run` floats
            const int lines = (run * 4 + 127) / 128 + 1;
            for (int i = tid; i < rows * lines; i += TC_NT) {
              const int r = i / lines, li = i - r * lines;
              const float* a = base + (long long)r * row_stride + min(li * 32, run - 1);
              asm volatile("prefetch.global.L2 [%0];" ::"l"(a));
            }
          };
          if (q.x.sk == 1 && q.x.sp == K) pf_rows(q.x.p + (long long)n2 * q.x.sn + (long long)q0 * q.x.sp, q.x.sc, Cin, pv2 * K);
          pf_rows(q.pd + ((long long)n2 * nb * P + q0) * KK, (long long)P * KK, nb, pv2 * KK);
        }
      }
      __syncthreads();   // csum visible to the branch loop
      TPH(1);   // adjacency transform
    }

    // ---- 2. per branch: aggregation into the UMMA A tile, then the tensor-core channel mix
    for (int b = 0; b < nb; ++b) {
      // aggregation xa[c][l,w] = sum_v x[c][l,v] xm_b[l][v][w] on mma.sync (3xTF32, register fragments), written
      // straight into the UMMA A tile (hi / lo).  warp = (frame, 16-channel tile), all w tiles; K = v masked at K
      {
        constexpr int NTW = KP / 8;
        const int fg = lane >> 2, ft = lane & 3;
        const int MTc = (Cin + 15) >> 4;
        for (int grp = warp; grp < pv * MTc; grp += TC_NT / 32) {
          const int l = grp / MTc, m0 = (grp % MTc) * 16;
          float acc[NTW][4];
#pragma unroll
          for (int i = 0; i < NTW; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
          const float* ar = xs + min(m0 + fg, Cin - 1) * XS_LD + l * K + ft;
          const float* ar8 = xs + min(m0 + fg + 8, Cin - 1) * XS_LD + l * K + ft;
          const float* br = xms + ((b * PCH + l) * K + ft) * KP + fg;
          for (int k0 = 0; k0 < K; k0 += 8) {
            const bool k_lo = k0 + ft < K, k_hi = k0 + ft + 4 < K;
            uint32_t ah[4], al[4];
            float h_, l_;
            split_tf32(k_lo ? ar[k0] : 0.f, h_, l_);       ah[0] = __float_as_uint(h_); al[0] = __float_as_uint(l_);
            split_tf32(k_lo ? ar8[k0] : 0.f, h_, l_);      ah[1] = __float_as_uint(h_); al[1] = __float_as_uint(l_);
            split_tf32(k_hi ? ar[k0 + 4] : 0.f, h_, l_);   ah[2] = __float_as_uint(h_); al[2] = __float_as_uint(l_);
            split_tf32(k_hi ? ar8[k0 + 4] : 0.f, h_, l_);  ah[3] = __float_as_uint(h_); al[3] = __float_as_uint(l_);
#pragma unroll
            for (int i = 0; i < NTW; ++i) {
              uint32_t bh[2], bl[2];
              split_tf32(k_lo ? br[k0 * KP + i * 8] : 0.f, h_, l_);        bh[0] = __float_as_uint(h_); bl[0] = __float_as_uint(l_);
              split_tf32(k_hi ? br[(k0 + 4) * KP + i * 8] : 0.f, h_, l_);  bh[1] = __float_as_uint(h_); bl[1] = __float_as_uint(l_);
              mma_tf32_sync(acc[i], ah, bh);
              mma_tf32_sync(acc[i], ah, bl);
              mma_tf32_sync(acc[i], al, bh);
            }
          }
          // tile offset = position part + channel part (tc_off): the channel part of this lane's two rows (c, c + 8) is
          // computed once per tile, the position part once per column pair
          {
            const int c0 = m0 + fg;
            const int cp0 = (c0 >> 2) * TC_LBO_F + (c0 & 3), cp1 = cp0 + 2 * TC_LBO_F;
            const bool cok0 = c0 < Cin, cok1 = c0 + 8 < Cin;
#pragma unroll
            for (int i = 0; i < NTW; ++i) {
              const int w0 = i * 8 + 2 * ft, r0 = l * K + w0, r1 = r0 + 1;
              const int pp0 = (r0 >> 3) * sbo_f + ((r0 & 7) << 2), pp1 = (r1 >> 3) * sbo_f + ((r1 & 7) << 2);
              const bool wok0 = w0 < K, wok1 = w0 + 1 < K;
              float hi, lo;
              if (cok0 && wok0) { split_tf32(acc[i][0], hi, lo); a_hi[pp0 + cp0] = hi; a_lo[pp0 + cp0] = lo; }
              if (cok0 && wok1) { split_tf32(acc[i][1], hi, lo); a_hi[pp1 + cp0] = hi; a_lo[pp1 + cp0] = lo; }
              if (cok1 && wok0) { split_tf32(acc[i][2], hi, lo); a_hi[pp0 + cp1] = hi; a_lo[pp0 + cp1] = lo; }
              if (cok1 && wok1) { split_tf32(acc[i][3], hi, lo); a_hi[pp1 + cp1] = hi; a_lo[pp1 + cp1] = lo; }
            }
          }
        }
        // ones row (K index Cin): the precomputed column sums of xm
        for (int i = tid; i < pv * K; i += TC_NT) {
          float hi, lo;
          split_tf32(csum[b * PCH * K + i], hi, lo);
          const int o = tc_off(i, Cin, sbo_f);
          a_hi[o] = hi;
          a_lo[o] = lo;
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> tensor-core (async proxy) reads
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncthreads();
      TPH(2);   // aggregation + tile writes (+ fence, barrier)
      if (warp == 0) {
        // Warp-uniform issue: every lane of warp 0 runs the descriptor arithmetic (32-bit, on values made provably
        // uniform by broadcast shuffles), one elected lane issues.  Issuing from `if (tid == 0)` kept the descriptors in
        // vector registers and paid a chain of R2UR moves in front of each of the 27 small MMAs of a branch, with
        // every other warp of the CTA waiting for the commit behind them.
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t ua = __shfl_sync(0xffffffffu, smem_u32(a_hi), 0);
        const uint32_t ub = __shfl_sync(0xffffffffu, smem_u32(b_img + (b * 2) * b_tile_f), 0);
        const uint32_t tm = __shfl_sync(0xffffffffu, tmem_d, 0);
        const uint32_t lof = (lbo_b >> 4) << 16, hiw = (sbo_b >> 4) | (1u << 14);
        const uint32_t dah = ((ua & 0x3FFFFu) >> 4) | lof, dal = (((ua + (uint32_t)a_tile_f * 4u) & 0x3FFFFu) >> 4) | lof;
        const uint32_t dbh = ((ub & 0x3FFFFu) >> 4) | lof, dbl = (((ub + (uint32_t)b_tile_f * 4u) & 0x3FFFFu) >> 4) | lof;
        uint32_t leader;
        asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}\n" : "=r"(leader));
        const int nks = KD / 8;
#pragma unroll
        for (int ks = 0; ks < 9; ++ks) {       // KD <= 72 (Cin <= 64)
          if (ks < nks) {
            const uint32_t adv = (uint32_t)ks * ((2u * lbo_b) >> 4);   // 8 K-elements = two core matrices
            umma::mma_tf32_lohi(tm, dah + adv, hiw, dbh + adv, hiw, idesc, (b > 0 || ks > 0) ? 1u : 0u, leader);
            umma::mma_tf32_lohi(tm, dah + adv, hiw, dbl + adv, hiw, idesc, 1u, leader);
            umma::mma_tf32_lohi(tm, dal + adv, hiw, dbh + adv, hiw, idesc, 1u, leader);   // lo*lo (2^-22 relative) is dropped
          }
        }
        umma::commit_elect(mbar);
      }
      // the A tile is rewritten by the next branch / item and TMEM is read by the epilogue only after the MMAs retire.
      // Only the issuing warp polls the mbarrier; the other 15 sleep at a block barrier (512 threads spinning on
      // try_wait compete with the tensor core for shared-memory bandwidth and issue slots)
      if (warp == 0) ok = mbar_wait(smem_u32(mbar), phase) && ok;
      ok = __syncthreads_and(ok);
      phase ^= 1;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      TPH(3);   // MMA issue + wait for the commit
    }

    // ---- 3. epilogue: TMEM -> registers -> out (+ skip).  warp w: lanes 32 (w%4) .. +31 (positions), columns 16 (w/4) ..
    {
      const int pos = (warp & 3) * 32 + lane;
      const int l = pos / K, k = pos - l * K;
      const bool pok = pos < npos;
      const long long off_o = (long long)n * q.out.sn + (long long)(p0 + l) * q.out.sp + (long long)k * q.out.sk;
      for (int col0 = (warp >> 2) * 16; col0 < NP; col0 += 64) {
        uint32_t r[16];
        const uint32_t taddr = tmem_d + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)col0;
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
              "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
            : "r"(taddr)
            : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (pok) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int o = col0 + j;
            if (o < Cout) {
              float v = ok ? __uint_as_float(r[j]) : __int_as_float(0x7fc00000);   // a stalled pipeline must be loud
              if (q.skip.p) v += sks[o * XS_LD + pos];
              q.out.p[off_o + (long long)o * q.out.sc] = v;
            }
          }
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncthreads();   // TMEM drained and xs / xms / pdr free before the next item
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      TPH(4);   // epilogue
    }
  }
#ifdef DSTD_PHASE_TIMING
  if (blockIdx.x == 0 && tid == 0)
    printf("aggmix_fwd_tc phases (cycles, CTA 0): stage %lld transform %lld aggregate %lld mma+wait %lld epilogue %lld\n", tph[0],
           tph[1], tph[2], tph[3], tph[4]);
#endif
  if (!ok && tid == 0 && err_flag) {
    *(volatile int*)err_flag = 1;
    __threadfence_system();
  }
  __syncthreads();
  if (warp == 0)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(tmem_cols) : "memory");
}

// ------------------------------------------------------------------------------------------ weight image for the tensor path
// wtc[b][hi|lo][tc_off(o, j)]: conv_f weights (+ bias in K row Cin) of branch b as UMMA K-major core matrices, TF32 split
// One pass over the padded image (NP output rows x KD reduction rows per branch): out-of-range rows are written as
// zeros, so no separate clear is needed (the 16-byte gaps between core matrices are never read by the MMA).
__global__ void pack_tc_kernel(PackParams q, float* wtc, int KD, int NP) {
  const int sbo_f = (KD / 4) * TC_LBO_F, tile = (NP / 8) * sbo_f;
  const int total = q.nb * NP * KD;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int j = i % KD;
    int t = i / KD;
    const int o = t % NP, b = t / NP;
    float w = 0.f;
    if (o < q.Cout && j <= q.Cin) w = j < q.Cin ? __ldg(q.w_f[b] + (long long)o * q.Cin + j) : __ldg(q.b_f[b] + o);
    uint32_t h;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(w));
    const float hi = __uint_as_float(h);
    const int off = tc_off(o, j, sbo_f);
    wtc[(b * 2 + 0) * tile + off] = hi;
    wtc[(b * 2 + 1) * tile + off] = w - hi;
  }
}

// ------------------------------------------------------------------------------------------ geometry / launch
struct TcGeom {
  int WH, PCH, KD, NP, tmem_cols;
  size_t smem, wtc_floats;
};

static bool tc_geom(int Cin, int Cout, int P, int K, int nb, TcGeom& g, bool with_skip = true) {
  if (K > 40 || K < 1 || Cin > 64 || Cout > 64) return false;
  g.WH = K <= 24 ? 12 : K <= 32 ? 16 : 20;
  g.KD = (Cin + 1 + 7) / 8 * 8;
  g.NP = (Cout + 15) / 16 * 16;
  g.tmem_cols = g.NP <= 32 ? 32 : 64;
  const int KP = 2 * g.WH, sbo_f = (g.KD / 4) * TC_LBO_F;
  g.wtc_floats = (size_t)nb * 2 * (g.NP / 8) * sbo_f;
  for (int pch = (128 / K >= 4 ? 4 : 128 / K); pch >= 1; --pch) {   // 4 frames = 16 aggregation items = 16 warps
    if (pch > P && pch > 1) continue;
    const int XS_LD = ((pch * K + 3) / 8) * 8 + 4;
    size_t f = (size_t)2 * ((pch * K + 7) / 8) * sbo_f + g.wtc_floats + (size_t)((Cin * XS_LD + 3) & ~3) + (size_t)nb * pch * K * KP +
               (size_t)((nb * K * K + 3) & ~3) + (size_t)((nb * pch * K * K + 3) & ~3) + (size_t)2 * ((nb * pch * K + 3) & ~3) + 8 +
               (with_skip ? (size_t)((Cout * XS_LD + 3) & ~3) : 0);
    // the M = 128 descriptors read 16 row groups from each A tile: keep that window inside the allocation
    const size_t a_window = (size_t)((pch * K + 7) / 8) * sbo_f + (size_t)16 * sbo_f + 64;
    if (f < a_window) f = a_window;
    if (f * sizeof(float) <= (size_t)MAX_DYN_SMEM - 256) {
      g.PCH = pch;
      g.smem = f * sizeof(float);
      return true;
    }
  }
  return false;
}

bool aggmix_tc_supported(int Cin, int Cout, int P, int K, int nb) {
  TcGeom g;
  return tc_geom(Cin, Cout, P, K, nb, g);
}

size_t aggmix_tc_ws_floats(int Cin, int Cout, int P, int K, int nb) {
  TcGeom g;
  if (!tc_geom(Cin, Cout, P, K, nb, g)) return 0;
  return g.wtc_floats + 4;   // + error flag
}

int launch_aggmix_fwd_tc(AggMixParams q, const PackParams& pk, float* wtc_ws, cudaStream_t st) {
  TcGeom g;
  DSTD_REQUIRE(tc_geom(q.Cin, q.Cout, q.P, q.K, q.nb, g, q.skip.p != nullptr), DSTD_ERR_UNSUPPORTED,
               "aggmix_fwd_tc: shape outside limits");
  int* err_flag = device_error_word();     // host-mapped: the next entry point reports a timed-out pipeline
  pack_tc_kernel<<<min(cdiv(q.nb * g.NP * g.KD, 256), 64), 256, 0, st>>>(pk, wtc_ws, g.KD, g.NP);
  count_launch();
  DSTD_LAUNCH_CHECK("pack_tc");
  q.PCH = g.PCH;
  q.CoutP = g.NP;
  q.wtc = wtc_ws;
  const long long items = (long long)q.N * cdiv(q.P, g.PCH);
  const int ctas = (int)(items < num_sms() ? items : num_sms());
#define DSTD_AMTC(WH_)                                                                      \
  if (g.WH == WH_) {                                                                        \
    auto kern = aggmix_fwd_tc_kernel<WH_>;                                                  \
    ensure_max_smem((const void*)kern);                                                     \
    kern<<<ctas, TC_NT, g.smem, st>>>(q, g.KD, g.NP, g.tmem_cols, err_flag);                  \
  }
  DSTD_AMTC(12) DSTD_AMTC(16) DSTD_AMTC(20)
#undef DSTD_AMTC
  count_launch();
  return check_launch("aggmix_fwd_tc");
}

}  // namespace dstd
