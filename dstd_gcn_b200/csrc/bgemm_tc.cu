// Channel-mix GEMM of the unfused path (C > 64: the stress configuration, BASELINE.json configs[4]) on the 5th-generation
// tensor cores:   Out[n, i, p, k] = sum_c W(c, i) In[n, c, p, k] (+ bias[i]) (+ Add[n, i, p, k])        (model/dstdgcn.py:81 and
// its data gradient, with 256 channels and up to 771 reduction rows).  Same contract as bgemm (gemm.cu), which runs the
// shapes this kernel does not take.
//
//   D[i (M, tiles of 128)][g (N = NP positions)] += A[i][c] B[c][g]      tcgen05.mma kind::f16, bf16 operands, fp32 in TMEM
//
// fp32 parity comes from the three-way bf16 split x = h + m + l and six products per k-step (hh, hm, mh, mm, hl, lh: the
// same error as 3xTF32, DESIGN.md section 7); tf32 operands are not an option because the activations are
// position-contiguous, i.e. an MN-major B operand, and tf32 has no swizzle-free MN-major form (profiles/r02_umma_probe_*).
//   A: the weights, split and laid out as K-major 16-bit row images per K chunk by a pack kernel, brought in by ONE TMA
//      bulk copy per chunk (cp.async.bulk + mbarrier expect_tx), double buffered;
//   B: the activation chunk [KC rows][NP positions], loaded by all threads (position pairs, coalesced), split on the
//      CUDA cores and stored as a 16-bit row image read through the MN-major view, double buffered, the loads of chunk
//      c + 1 in flight (registers) while chunk c is converted;
//   MMAs of chunk c are issued by warp 0 (descriptor arithmetic warp-uniform, one elected lane) and retire onto the
//      mbarrier that frees the two buffers of that stage (tcgen05.commit), so the conversion of chunk c + 1 and the bulk
//      copy of its weights overlap the tensor work of chunk c;
//   epilogue: tcgen05.ld (lane = output row) -> fp32 staging in the freed buffers -> coalesced stores along positions.
#include "kernels.cuh"
#include "umma.cuh"

namespace dstd {

struct BgemmTcGeom {
  int mtiles, np, kc, nchunk, tmem_cols;
  uint32_t a_sbo, a_plane, a_chunk, b_sbo, b_plane, b_chunk;
  size_t smem;
};

static __host__ __device__ inline BgemmTcGeom tc_geom(int M, int Kd) {
  BgemmTcGeom g;
  g.mtiles = (M + 127) / 128;
  g.np = g.mtiles <= 4 ? 128 : 96;     // TMEM: mtiles * np <= 512 columns
  g.kc = 16;   // two CTAs per SM for up to two M tiles (86 KB, 256 TMEM columns each): their phases interleave
  g.nchunk = (Kd + g.kc - 1) / g.kc;
  int cols = g.mtiles * g.np, pw = 32;
  while (pw < cols) pw <<= 1;
  g.tmem_cols = pw;
  g.a_sbo = (uint32_t)umma::img16_sbo_b(g.kc);                 // K-major image [128 mtiles rows][kc]
  g.a_plane = (uint32_t)(g.mtiles * 16) * g.a_sbo;
  g.a_chunk = 3u * g.a_plane;
  g.b_sbo = (uint32_t)umma::img16_sbo_b(g.np);                 // row image [kc rows][np positions]
  g.b_plane = (uint32_t)(g.kc / 8) * g.b_sbo;
  g.b_chunk = 3u * g.b_plane;
  g.smem = (size_t)2 * (g.a_chunk + g.b_chunk) + (size_t)3 * g.np * sizeof(long long) + 64;
  return g;
}

__device__ __forceinline__ uint32_t dlo(uint32_t saddr, uint32_t lbo_b) { return ((saddr & 0x3FFFFu) >> 4) | ((lbo_b >> 4) << 16); }
__device__ __forceinline__ uint32_t dhi(uint32_t sbo_b) { return (sbo_b >> 4) | (1u << 14); }
__device__ __forceinline__ uint32_t elect_lane() {    // the lane tcgen05.commit's elect.sync picks as well
  uint32_t p;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}\n" : "=r"(p));
  return p;
}

// weights -> [chunk][plane h/m/l][K-major row image of (mtiles*128) x kc], zero padded
__global__ void bgemm_tc_pack_kernel(const float* __restrict__ w, long long wsc, long long wsi, int M, int Kd, BgemmTcGeom g,
                                     unsigned char* __restrict__ img) {
  const int rows = g.mtiles * 128, kp = g.kc / 2;
  const long long total = (long long)g.nchunk * rows * kp;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int kq = (int)(i % kp) * 2;
    const int m = (int)((i / kp) % rows), c = (int)(i / ((long long)kp * rows));
    const int k0 = c * g.kc + kq;
    const float v0 = (m < M && k0 < Kd) ? __ldg(w + (long long)k0 * wsc + (long long)m * wsi) : 0.f;
    const float v1 = (m < M && k0 + 1 < Kd) ? __ldg(w + (long long)(k0 + 1) * wsc + (long long)m * wsi) : 0.f;
    uint32_t h0, m0, l0, h1, m1, l1;
    umma::split_bf16x3(v0, h0, m0, l0);
    umma::split_bf16x3(v1, h1, m1, l1);
    unsigned char* dst = img + (size_t)c * g.a_chunk + umma::img16_off_b(m, kq, (int)g.a_sbo);
    *reinterpret_cast<uint32_t*>(dst) = umma::pack_bf16(h0, h1);
    *reinterpret_cast<uint32_t*>(dst + g.a_plane) = umma::pack_bf16(m0, m1);
    *reinterpret_cast<uint32_t*>(dst + 2 * g.a_plane) = umma::pack_bf16(l0, l1);
  }
}

constexpr int BT_NT = 256;

template <int NP, int KC>
__global__ void __launch_bounds__(BT_NT, 2) bgemm_tc_kernel(BgemmParams q, BgemmTcGeom g, const unsigned char* __restrict__ wimg,
                                                            int* err) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr int PAIRS = NP / 2, RSTEP = BT_NT / PAIRS, PP = (KC + RSTEP - 1) / RSTEP;   // rows r0 + RSTEP j (< KC), j < PP, per thread
  unsigned char* abuf = smem;                                   // [2][a_chunk]
  unsigned char* bbuf = abuf + 2 * g.a_chunk;                   // [2][b_chunk]
  long long* col_in = reinterpret_cast<long long*>(bbuf + 2 * g.b_chunk);
  long long* col_out = col_in + NP;
  long long* col_add = col_out + NP;
  uint64_t* bar = reinterpret_cast<uint64_t*>(col_add + NP);   // [0..1] weights landed, [2..3] stage free
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bar + 4);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int PK = q.P * q.K;
  const long long g0 = (long long)blockIdx.x * NP;

  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) umma::mbar_init(&bar[i], 1);
    umma::mbar_init_fence();
  }
  if (warp == 0) umma::tmem_alloc(tslot, (uint32_t)g.tmem_cols);
  for (int c = tid; c < NP; c += BT_NT) {
    const long long gg = g0 + c;
    if (gg < q.G) {
      const int n = (int)(gg / PK);
      const int j = (int)(gg - (long long)n * PK);
      const int p = j / q.K, k = j - p * q.K;
      col_in[c] = vix(q.in, n, 0, p, k);
      col_out[c] = vix(q.out, n, 0, p, k);
      col_add[c] = q.add.p ? vix(q.add, n, 0, p, k) : 0;
    } else {
      col_in[c] = -1;
      col_out[c] = -1;
      col_add[c] = 0;
    }
  }
  umma::fence_before();
  __syncthreads();
  umma::fence_after();
  const uint32_t tmem = __shfl_sync(0xffffffffu, *reinterpret_cast<volatile uint32_t*>(tslot), 0);

  // this thread's position pair and first row of the B chunk
  const int pi = tid % PAIRS, r0 = tid / PAIRS;
  const bool conv = r0 < RSTEP;                    // NP = 96: 240 of the 256 threads convert
  const long long off0 = conv ? col_in[2 * pi] : -1, off1 = conv ? col_in[2 * pi + 1] : -1;
  const bool vec = off0 >= 0 && off1 == off0 + 1 && !((off0 | q.in.sc) & 1) && !(reinterpret_cast<uintptr_t>(q.in.p) & 7);
  float pv[PP][2];
  const long long rstep = (long long)RSTEP * q.in.sc;
  auto load_chunk = [&](int c) {
    const int kd0 = c * KC + r0;
    uint32_t jm = 0;                                   // rows of this thread that exist in this chunk
#pragma unroll
    for (int j = 0; j < PP; ++j)
      if (conv && kd0 + RSTEP * j < q.Kd && r0 + RSTEP * j < KC) jm |= 1u << j;
    if (vec) {                                         // the common case: one predicated 8-byte load per row
      const float* bp = q.in.p + off0 + (long long)kd0 * q.in.sc;
#pragma unroll
      for (int j = 0; j < PP; ++j) {
        float2 t = make_float2(0.f, 0.f);
        if ((jm >> j) & 1u) t = __ldg(reinterpret_cast<const float2*>(bp + j * rstep));
        pv[j][0] = t.x;
        pv[j][1] = t.y;
      }
    } else {
#pragma unroll
      for (int j = 0; j < PP; ++j) {
        const long long ro = (long long)(kd0 + RSTEP * j) * q.in.sc;
        pv[j][0] = (((jm >> j) & 1u) && off0 >= 0) ? __ldg(q.in.p + off0 + ro) : 0.f;
        pv[j][1] = (((jm >> j) & 1u) && off1 >= 0) ? __ldg(q.in.p + off1 + ro) : 0.f;
      }
    }
    if (q.ones_row >= 0) {
#pragma unroll
      for (int j = 0; j < PP; ++j)
        if (((jm >> j) & 1u) && kd0 + RSTEP * j == q.ones_row) {
          pv[j][0] = off0 >= 0 ? 1.f : 0.f;
          pv[j][1] = off1 >= 0 ? 1.f : 0.f;
        }
    }
  };
  load_chunk(0);
  auto issue_w = [&](int c) {     // thread 0: one bulk copy brings the weight images of chunk c
    umma::mbar_expect_tx(&bar[c & 1], g.a_chunk);
    umma::bulk_g2s(abuf + (size_t)(c & 1) * g.a_chunk, wimg + (size_t)c * g.a_chunk, g.a_chunk, &bar[c & 1]);
  };
  if (tid == 0) {
    issue_w(0);
    if (g.nchunk > 1) issue_w(1);
  }

  const uint32_t abase = umma::smem_u32(abuf), bbase = umma::smem_u32(bbuf);
  const uint32_t idesc = umma::idesc_bf16(128, NP, 0, 1);
  const int NC = g.nchunk;
  bool ok = true;
  for (int c = 0; c < NC; ++c) {
    const int buf = c & 1, use = c >> 1;
    if (c >= 2) ok &= umma::mbar_wait(&bar[2 + buf], (uint32_t)(use - 1) & 1u);   // the MMAs of chunk c - 2 retired
    unsigned char* bdst = bbuf + (size_t)buf * g.b_chunk;
#pragma unroll
    for (int j = 0; j < PP; ++j) {
      const int r = r0 + RSTEP * j;
      if (!conv || r >= KC) continue;
      uint32_t h0, m0, l0, h1, m1, l1;
      umma::split_bf16x3(pv[j][0], h0, m0, l0);
      umma::split_bf16x3(pv[j][1], h1, m1, l1);
      unsigned char* d = bdst + umma::img16_off_b(r, 2 * pi, (int)g.b_sbo);
      *reinterpret_cast<uint32_t*>(d) = umma::pack_bf16(h0, h1);
      *reinterpret_cast<uint32_t*>(d + g.b_plane) = umma::pack_bf16(m0, m1);
      *reinterpret_cast<uint32_t*>(d + 2 * g.b_plane) = umma::pack_bf16(l0, l1);
    }
    umma::fence_async_smem();     // the generic-proxy stores above become visible to the tensor core (async proxy)
    umma::fence_before();
    __syncthreads();
    if (c + 1 < NC) load_chunk(c + 1);     // issued after the proxy fence: in flight during the MMAs of this chunk
    if (warp == 0) {
      ok &= umma::mbar_wait(&bar[buf], (uint32_t)use & 1u);    // weights of this chunk landed
      umma::fence_after();
      // broadcast shuffles: ptxas then knows the stage bases are warp-uniform and keeps every descriptor word on the
      // uniform datapath (without them: four R2UR moves in front of each MMA)
      const uint32_t a0 = __shfl_sync(0xffffffffu, abase + (uint32_t)buf * g.a_chunk, 0);
      const uint32_t b0 = __shfl_sync(0xffffffffu, bbase + (uint32_t)buf * g.b_chunk, 0);
      const uint32_t ahi = dhi(g.a_sbo), bhi = dhi(umma::IMG16_LBO_B);     // MN-major view: fields swapped
      const uint32_t leader = elect_lane();
      // consecutive instructions go to different accumulators (M tiles); small terms first: l*h, h*l, m*m, m*h, h*m, h*h
#pragma unroll
      for (int s = 0; s < KC / 16; ++s) {
#pragma unroll
        for (int t = 0; t < 6; ++t) {
          const uint32_t pa = (t == 0) ? 2u : (t == 2 || t == 3) ? 1u : 0u;      // plane of A: 0 = h, 1 = m, 2 = l
          const uint32_t pb = (t == 1) ? 2u : (t == 2 || t == 4) ? 1u : 0u;      // plane of B
          const uint32_t first = (c == 0 && s == 0 && t == 0) ? 0u : 1u;
          // fully unrolled over the (at most five) M tiles with a uniform guard: a run-time loop here makes ptxas carry
          // the descriptor words in vector registers and pay ~9 R2UR moves in front of every MMA
#pragma unroll
          for (int mt = 0; mt < 5; ++mt) {
            if (mt < g.mtiles) {
              const uint32_t as = a0 + pa * g.a_plane + (uint32_t)(mt * 16) * g.a_sbo + (uint32_t)s * 2u * umma::IMG16_LBO_B;
              const uint32_t bs = b0 + pb * g.b_plane + (uint32_t)s * 2u * g.b_sbo;
              umma::mma_f16_lohi(tmem + (uint32_t)(mt * NP), dlo(as, umma::IMG16_LBO_B), ahi, dlo(bs, g.b_sbo), bhi, idesc, first,
                                 leader);
            }
          }
        }
      }
      umma::commit_elect(&bar[2 + buf]);
      // weights of chunk c + 1 (c >= 1; chunks 0 and 1 were requested up front): their buffer is free once the MMAs of
      // chunk c - 1, issued one iteration ago, have retired; the copy then lands under the tensor work of chunk c
      if (c >= 1 && c + 1 < NC) {
        ok &= umma::mbar_wait(&bar[2 + (buf ^ 1)], (uint32_t)((c - 1) >> 1) & 1u);
        if (lane == 0) issue_w(c + 1);
      }
    }
  }
  // every MMA retired: the last commit covers all earlier ones
  {
    const int lb = (NC - 1) & 1, lu = (NC - 1) >> 1;
    ok &= umma::mbar_wait(&bar[2 + lb], (uint32_t)lu & 1u);
    umma::fence_after();
  }
  if (!ok && tid == 0 && err) *(volatile int*)err = 3;

  // ---- epilogue: one M tile at a time through fp32 staging [128][NP + 4] in the freed weight buffers
  float* stage = reinterpret_cast<float*>(abuf);
  constexpr int SLD = NP + 4;
  const int lq = warp & 3, chalf = warp >> 2;
  for (int mt = 0; mt < g.mtiles; ++mt) {
    const uint32_t trow = tmem + ((uint32_t)(lq * 32) << 16) + (uint32_t)(mt * NP + chalf * (NP / 2));
    float* srow = stage + (lq * 32 + lane) * SLD + chalf * (NP / 2);
#pragma unroll
    for (int c8 = 0; c8 < NP / 2; c8 += 16) {
      uint32_t v0[8], v1[8];
      umma::tmem_ld8(trow + c8, v0);
      umma::tmem_ld8(trow + c8 + 8, v1);
      umma::tmem_ld_wait();
      *reinterpret_cast<uint4*>(srow + c8) = make_uint4(v0[0], v0[1], v0[2], v0[3]);
      *reinterpret_cast<uint4*>(srow + c8 + 4) = make_uint4(v0[4], v0[5], v0[6], v0[7]);
      *reinterpret_cast<uint4*>(srow + c8 + 8) = make_uint4(v1[0], v1[1], v1[2], v1[3]);
      *reinterpret_cast<uint4*>(srow + c8 + 12) = make_uint4(v1[4], v1[5], v1[6], v1[7]);
    }
    __syncthreads();
    for (int idx = tid; idx < 128 * NP; idx += BT_NT) {
      const int row = idx / NP, col = idx - row * NP, i = mt * 128 + row;
      const long long off = col_out[col];
      if (i < q.M && off >= 0) {
        float v = stage[row * SLD + col];
        if (q.bias) v += __ldg(q.bias + i);
        if (q.add.p) v += q.add.p[col_add[col] + (long long)i * q.add.sc];
        q.out.p[off + (long long)i * q.out.sc] = v;
      }
    }
    __syncthreads();
  }
  umma::fence_before();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tmem, (uint32_t)g.tmem_cols);
}

// ================================================================================= weight gradient on tcgen05
//   G[i][c] = sum_g A[i][g] B[c][g]      (A = gout [M rows], B = xa [Cd rows], g = the N*P*K positions: split-K)
// Both operands are position-contiguous, i.e. K-major row images [rows][32 positions] for the tensor core.  CTA = (split
// of the positions, 128-row tile of A, column block of B of NBW <= 256 rows): per chunk of 32 positions all threads load
// position pairs (coalesced), split them three ways and store the images; warp 0 issues 2 k-steps x 6 products into ONE
// TMEM accumulator [128 x NBW]; tcgen05.commit -> mbarrier releases the (single) stage, the loads of the next chunk are
// already in registers; two CTAs per SM interleave their convert / MMA phases.  Epilogue: tcgen05.ld -> the split's
// partial [M][Cd] (summed by reduce_segments in a fixed order, like the CUDA-core wgrad).
constexpr int WT_KC = 32;

struct WgradTcGeom {
  int mtiles, nblocks, nbw, tmem_cols, S;
  long long cols_per_split;
  uint32_t sbo, a_plane, b_plane;
  size_t smem;
};
static WgradTcGeom wgrad_tc_geom(int M, int Cd, long long G, int S_max) {
  WgradTcGeom g;
  g.mtiles = (M + 127) / 128;
  g.nblocks = (Cd + 255) / 256;
  g.nbw = ((Cd + g.nblocks - 1) / g.nblocks + 15) / 16 * 16;
  int pw = 32;
  while (pw < g.nbw) pw <<= 1;
  g.tmem_cols = pw;
  int S = (2 * num_sms() + g.mtiles * g.nblocks - 1) / (g.mtiles * g.nblocks);
  if (S > S_max) S = S_max;
  if (S < 1) S = 1;
  long long per = (G + S - 1) / S;
  g.cols_per_split = (per + WT_KC - 1) / WT_KC * WT_KC;
  g.S = (int)((G + g.cols_per_split - 1) / g.cols_per_split);
  g.sbo = (uint32_t)umma::img16_sbo_b(WT_KC);
  g.a_plane = 16u * g.sbo;
  g.b_plane = (uint32_t)(g.nbw / 8) * g.sbo;
  g.smem = (size_t)3 * (g.a_plane + g.b_plane) + 64;
  return g;
}

__global__ void __launch_bounds__(BT_NT, 2) wgrad_tc_kernel(WgradParams q, WgradTcGeom g, int* err) {
  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* aimg = smem;                         // [3 planes][128 rows][32 positions]
  unsigned char* bimg = aimg + 3 * g.a_plane;         // [3 planes][nbw rows][32 positions]
  uint64_t* bar = reinterpret_cast<uint64_t*>(bimg + 3 * g.b_plane);
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bar + 1);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int mt = blockIdx.y / g.nblocks, nbk = blockIdx.y - mt * g.nblocks;
  const int i0 = mt * 128, c0 = nbk * g.nbw, NBJ = g.nbw / 16;
  const int PK = q.P * q.K;
  const long long gbeg = (long long)blockIdx.x * g.cols_per_split;
  long long gend = gbeg + g.cols_per_split;
  if (gend > q.G) gend = q.G;

  if (tid == 0) {
    umma::mbar_init(&bar[0], 1);
    umma::mbar_init_fence();
  }
  if (warp == 0) umma::tmem_alloc(tslot, (uint32_t)g.tmem_cols);
  umma::fence_before();
  __syncthreads();
  umma::fence_after();
  const uint32_t tmem = __shfl_sync(0xffffffffu, *reinterpret_cast<volatile uint32_t*>(tslot), 0);

  // position pair of the chunk and rows rl + 16 j.  A warp holds rows r and r + 4: with the 144-byte group pitch the
  // two rows' 16-byte groups then fall on disjoint banks (rows r and r + 1 collide two-way)
  const int pi = tid & 15, rl = (warp & 3) + 4 * ((tid >> 4) & 1) + 8 * (warp >> 2);
  float pa[8][2], pb[16][2];
  // per-thread constants of the conversion: which of its rows exist, where the ones row sits, image offsets
  uint32_t amask = 0, bmask = 0;
  int onesj = -1;
#pragma unroll
  for (int j = 0; j < 8; ++j)
    if (i0 + rl + 16 * j < q.M) amask |= 1u << j;
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const int cc = c0 + rl + 16 * j;
    if (j < NBJ && cc < q.Cd) {
      if (cc == q.b_ones_row) onesj = j;
      else bmask |= 1u << j;
    }
  }
  const uint32_t soff0 = (uint32_t)umma::img16_off_b(rl, 2 * pi, (int)g.sbo), sstep = 2u * g.sbo;   // rows + 16
  const bool al_a = !(q.a.sc & 1) && !(reinterpret_cast<uintptr_t>(q.a.p) & 7);
  const bool al_b = !(q.b.sc & 1) && !(reinterpret_cast<uintptr_t>(q.b.p) & 7);
  const long long astep = 16 * q.a.sc, bstep = 16 * q.b.sc;
  // (sample, in-sample position) of this thread's first position, advanced by 32 per chunk: no 64-bit division in the loop
  int pn, prem;
  {
    const long long gg = gbeg + 2 * pi;
    pn = (int)(gg / PK);
    prem = (int)(gg - (long long)pn * PK);
  }
  auto load_chunk = [&](long long gc) {
    const long long gg = gc + 2 * pi;
    long long a0 = -1, a1 = -1, b0 = -1, b1 = -1;
    if (gg < gend) {
      const int p = prem / q.K, k = prem - p * q.K;
      a0 = vix(q.a, pn, 0, p, k);
      b0 = vix(q.b, pn, 0, p, k);
      if (gg + 1 < gend) {
        int n1 = pn, p1 = p, k1 = k + 1;
        if (k1 == q.K) {
          k1 = 0;
          if (++p1 == q.P) {
            p1 = 0;
            ++n1;
          }
        }
        a1 = vix(q.a, n1, 0, p1, k1);
        b1 = vix(q.b, n1, 0, p1, k1);
      }
    }
    prem += WT_KC;
    while (prem >= PK) {
      prem -= PK;
      ++pn;
    }
    if (al_a && a1 == a0 + 1 && !(a0 & 1)) {        // the common case: one 8-byte load per row, predicated, no branches
      const float* ap = q.a.p + a0 + (long long)(i0 + rl) * q.a.sc;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float2 t = make_float2(0.f, 0.f);
        if ((amask >> j) & 1u) t = __ldg(reinterpret_cast<const float2*>(ap + j * astep));
        pa[j][0] = t.x;
        pa[j][1] = t.y;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const long long ro = (long long)(i0 + rl + 16 * j) * q.a.sc;
        pa[j][0] = (((amask >> j) & 1u) && a0 >= 0) ? __ldg(q.a.p + a0 + ro) : 0.f;
        pa[j][1] = (((amask >> j) & 1u) && a1 >= 0) ? __ldg(q.a.p + a1 + ro) : 0.f;
      }
    }
    if (al_b && b1 == b0 + 1 && !(b0 & 1)) {
      const float* bp = q.b.p + b0 + (long long)(c0 + rl) * q.b.sc;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        float2 t = make_float2(0.f, 0.f);
        if ((bmask >> j) & 1u) t = __ldg(reinterpret_cast<const float2*>(bp + j * bstep));
        pb[j][0] = t.x;
        pb[j][1] = t.y;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const long long ro = (long long)(c0 + rl + 16 * j) * q.b.sc;
        pb[j][0] = (((bmask >> j) & 1u) && b0 >= 0) ? __ldg(q.b.p + b0 + ro) : 0.f;
        pb[j][1] = (((bmask >> j) & 1u) && b1 >= 0) ? __ldg(q.b.p + b1 + ro) : 0.f;
      }
    }
    if (onesj >= 0) {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (j == onesj) {
          pb[j][0] = b0 >= 0 ? 1.f : 0.f;
          pb[j][1] = b1 >= 0 ? 1.f : 0.f;
        }
    }
  };
  if (gbeg < gend) load_chunk(gbeg);

  const uint32_t abase = __shfl_sync(0xffffffffu, umma::smem_u32(aimg), 0), bbase = __shfl_sync(0xffffffffu, umma::smem_u32(bimg), 0);
  const uint32_t idesc = umma::idesc_bf16(128, g.nbw, 0, 0);
  const uint32_t hi = dhi(g.sbo);
  bool ok = true;
  int it = 0;
  for (long long gc = gbeg; gc < gend; gc += WT_KC, ++it) {
    if (it > 0) ok &= umma::mbar_wait(&bar[0], (uint32_t)(it - 1) & 1u);     // the MMAs of the previous chunk read the images
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      uint32_t h0, m0, l0, h1, m1, l1;
      umma::split_bf16x3(pa[j][0], h0, m0, l0);
      umma::split_bf16x3(pa[j][1], h1, m1, l1);
      unsigned char* d = aimg + soff0 + (uint32_t)j * sstep;
      *reinterpret_cast<uint32_t*>(d) = umma::pack_bf16(h0, h1);
      *reinterpret_cast<uint32_t*>(d + g.a_plane) = umma::pack_bf16(m0, m1);
      *reinterpret_cast<uint32_t*>(d + 2 * g.a_plane) = umma::pack_bf16(l0, l1);
    }
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      if (j < NBJ) {
        uint32_t h0, m0, l0, h1, m1, l1;
        umma::split_bf16x3(pb[j][0], h0, m0, l0);
        umma::split_bf16x3(pb[j][1], h1, m1, l1);
        unsigned char* d = bimg + soff0 + (uint32_t)j * sstep;
        *reinterpret_cast<uint32_t*>(d) = umma::pack_bf16(h0, h1);
        *reinterpret_cast<uint32_t*>(d + g.b_plane) = umma::pack_bf16(m0, m1);
        *reinterpret_cast<uint32_t*>(d + 2 * g.b_plane) = umma::pack_bf16(l0, l1);
      }
    }
    umma::fence_async_smem();
    umma::fence_before();
    __syncthreads();
    if (gc + WT_KC < gend) load_chunk(gc + WT_KC);
    if (warp == 0) {
      umma::fence_after();
      const uint32_t leader = elect_lane();
#pragma unroll
      for (int s = 0; s < WT_KC / 16; ++s) {
#pragma unroll
        for (int t = 0; t < 6; ++t) {
          const uint32_t pla = (t == 0) ? 2u : (t == 2 || t == 3) ? 1u : 0u;
          const uint32_t plb = (t == 1) ? 2u : (t == 2 || t == 4) ? 1u : 0u;
          const uint32_t as = abase + pla * g.a_plane + (uint32_t)s * 2u * umma::IMG16_LBO_B;
          const uint32_t bs = bbase + plb * g.b_plane + (uint32_t)s * 2u * umma::IMG16_LBO_B;
          umma::mma_f16_lohi(tmem, dlo(as, umma::IMG16_LBO_B), hi, dlo(bs, umma::IMG16_LBO_B), hi, idesc,
                             (it == 0 && s == 0 && t == 0) ? 0u : 1u, leader);
        }
      }
      umma::commit_elect(&bar[0]);
    }
  }
  if (it > 0) {
    ok &= umma::mbar_wait(&bar[0], (uint32_t)(it - 1) & 1u);
    umma::fence_after();
  }
  if (!ok && tid == 0 && err) *(volatile int*)err = 4;

  // epilogue: lane = row of the tile, columns in two halves -> this split's partial
  {
    const int lq = warp & 3, chalf = warp >> 2, half = g.nbw / 2, i = i0 + lq * 32 + lane;
    float* dst = q.partial + ((long long)blockIdx.x * q.M + i) * q.Cd + c0;
    for (int c8 = 0; c8 < half; c8 += 8) {
      uint32_t v[8];
      const int col = chalf * half + c8;
      if (it > 0) {
        umma::tmem_ld8(tmem + ((uint32_t)(lq * 32) << 16) + (uint32_t)col, v);
        umma::tmem_ld_wait();
      } else {
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = 0u;
      }
      if (i < q.M) {
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (c0 + col + u < q.Cd) dst[col + u] = __uint_as_float(v[u]);
      }
    }
  }
  umma::fence_before();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tmem, (uint32_t)g.tmem_cols);
}

bool wgrad_tc_supported(int M, int Cd) { return M >= 128 && Cd >= 128; }

// partial must hold wgrad_splits(G) * M * Cd floats (the split count used here never exceeds it); fills q.S
int launch_wgrad_tc(WgradParams& q, cudaStream_t st) {
  const WgradTcGeom g = wgrad_tc_geom(q.M, q.Cd, q.G, wgrad_splits(q.G));
  q.S = g.S;
  q.cols_per_split = g.cols_per_split;
  int* err = device_error_word();
  ensure_max_smem((const void*)wgrad_tc_kernel);
  wgrad_tc_kernel<<<dim3(g.S, g.mtiles * g.nblocks), BT_NT, g.smem, st>>>(q, g, err);
  count_launch();
  return check_launch("wgrad_tc");
}

bool bgemm_tc_supported(int M, int Kd) {
  if (M < 128 || Kd < 64) return false;               // small products stay on the CUDA-core kernel
  const BgemmTcGeom g = tc_geom(M, Kd);
  return g.mtiles <= 5 && g.smem <= (size_t)MAX_DYN_SMEM;
}

size_t bgemm_tc_ws_bytes(int M, int Kd) {
  if (M < 128 || Kd < 64) return 0;
  const BgemmTcGeom g = tc_geom(M, Kd);
  return g.mtiles <= 5 ? (size_t)g.nchunk * g.a_chunk : 0;
}

int launch_bgemm_tc(const BgemmParams& q, void* ws, cudaStream_t st) {
  const BgemmTcGeom g = tc_geom(q.M, q.Kd);
  unsigned char* img = reinterpret_cast<unsigned char*>(ws);
  DSTD_REQUIRE((reinterpret_cast<uintptr_t>(img) & 15) == 0, DSTD_ERR_BAD_ARG, "bgemm_tc: workspace must be 16-byte aligned");
  const long long total = (long long)g.nchunk * g.mtiles * 128 * (g.kc / 2);
  bgemm_tc_pack_kernel<<<(int)((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184), 256, 0, st>>>(q.w, q.wsc, q.wsi, q.M,
                                                                                                         q.Kd, g, img);
  count_launch();
  DSTD_LAUNCH_CHECK("bgemm_tc_pack");
  int* err = device_error_word();
  const int tiles = cdiv(q.G, g.np);
#define DSTD_BT(NP_, KC_)                                                                \
  {                                                                                      \
    ensure_max_smem((const void*)bgemm_tc_kernel<NP_, KC_>);                             \
    bgemm_tc_kernel<NP_, KC_><<<tiles, BT_NT, g.smem, st>>>(q, g, img, err);             \
  }
  if (g.np == 128) DSTD_BT(128, 16)
  else DSTD_BT(96, 16)
#undef DSTD_BT
  count_launch();
  return check_launch("bgemm_tc");
}

}  // namespace dstd
