// Fused adjacency aggregation + channel mix of one DSTD-GC unit with EVERY contraction on the 5th-generation tensor
// cores (tcgen05.mma, accumulators in TMEM), forward and backward: the sm_100a path of model/dstdgcn.py:81 + :87/:93
// (+ :150/:161/:248) and of its autograd (SURVEY.md Appendix A).
//
// Formulation ("mix first", the reference's own order).  Per work item = (sample n, F consecutive frames p), with
// xmu_b[l][v][w] = alpha*pd_b[l][v][w] + A_eff_b[v][w] (transposed for the fast variant):
//   forward    xf_b[o][l,v]  = sum_c Wf_b[o][c] x[c][l,v] + bf_b[o]                       (F1: K = c)
//              out[o][l,w]   = sum_b sum_v xf_b[o][l,v] xmu_b[l][v][w]  (+ skip)           (F2: per frame, K = v)
//   backward   xf_b recomputed as above                                                    (B1)
//              h_b[o][l,v]   = sum_w gout[o][l,w] xmu_b[l][v][w]                           (B2: per frame, K = w)
//              gxmu_b[l][v][w] = sum_o xf_b[o][l,v] gout[o][l,w]            -> HBM (gxm)   (B3: per frame, K = o)
//              gx[c][l,v]    = sum_b sum_o Wf_b[o][c] h_b[o][l,v]                          (B4: K = o)
//              gWf_b[o][c]  += sum_{l,v} h_b[o][l,v] x[c][l,v];  gbf_b[o] += sum h_b       (B5: K = position; TMEM-resident
//                                                                                           for the life of the CTA)
// Every activation tile takes part in contractions over channels AND over positions, i.e. the tensor core has to read it
// in both orientations.  tf32 operands have no MN-major form without swizzle (profiles/r02_umma_probe_tf32.txt), so
// each tile would need two shared-memory images per hi/lo part and nothing fits.  16-bit operands do: ONE "row image"
// ([channel rows][positions], 8-row x 16-byte core matrices, csrc/umma.cuh) is read as a K-major operand (K = position)
// or as an MN-major operand (K = channel) by swapping the descriptor's LBO/SBO fields (validated on a B200:
// profiles/r02_umma_probe_bf16x3.txt).  fp32 accuracy comes from the three-way bf16 split x = h + m + l and the six
// products hh + hm + mh + mm + hl + lh (relative error ~2^-21, the same as 3xTF32, and the same tensor time because
// kind::f16 contracts K = 16 per instruction).
// All accumulators are M = 64 (channels on the TMEM lanes); results return through tcgen05.ld with thread = channel row,
// which is exactly the order in which the next row image is written (16-byte stores, bank-conflict free).
#include "kernels.cuh"
#include "umma.cuh"

namespace dstd {

using namespace umma;

constexpr int UT_NT = 512;          // 16 warps; warp w drains TMEM lane quarter w % 4, column groups w / 4 (mod 4)
constexpr int UT_WP_B = 8 * 8 * IMG16_LBO_B;   // bytes of one [64][64] weight plane

// optional per-phase cycle counters (-DDSTD_PHASE_TIMING, printed by CTA 0)
#ifdef DSTD_PHASE_TIMING
#define UT_PH_DECL long long tph[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, tlast = clock64()
#define UT_PH(i) do { long long _t = clock64(); tph[i] += _t - tlast; tlast = _t; } while (0)
#else
#define UT_PH_DECL do {} while (0)
#define UT_PH(i) do {} while (0)
#endif

struct UnitGeom {
  int F, KQ, KW, NPOS, NG, Q, QG;      // frames per item; frame pitch (K up to 8); window (K up to 16); F*KQ; NPOS/8; image width; Q/8
  int CinK, CoutK, CinN;               // contraction lengths (multiples of 16), N of the weight-gradient GEMM
  int N16;                             // NPOS rounded up to 16 (N of the M = 128 chains)
  int plane_b, sbo_b;                  // [64][Q] plane
  int xr, xq, xplane_b, xsbo_b;        // xmu images [xr][xq]
  int tmem_cols;
  int terms;                           // split products per k-step: 6 (fp32 parity), 3 or 1 (DSTD_PRECISION, stated tolerance)
  int o_x0, o_g1, o_s, o_w, o_xmu, o_aeff, o_bias, o_etab, o_gst, o_pst, o_pout, o_pskip, o_bar;   // shared-memory byte offsets
  int smem;
};

// ------------------------------------------------------------------------------------------ device helpers
__device__ __forceinline__ void store_split8(unsigned char* pl0, int plane_b, int off_b, const float (&v)[8]) {
  uint32_t h[8], m[8], l[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) split_bf16x3(v[e], h[e], m[e], l[e]);
  *reinterpret_cast<uint4*>(pl0 + off_b) =
      make_uint4(pack_bf16(h[0], h[1]), pack_bf16(h[2], h[3]), pack_bf16(h[4], h[5]), pack_bf16(h[6], h[7]));
  *reinterpret_cast<uint4*>(pl0 + plane_b + off_b) =
      make_uint4(pack_bf16(m[0], m[1]), pack_bf16(m[2], m[3]), pack_bf16(m[4], m[5]), pack_bf16(m[6], m[7]));
  *reinterpret_cast<uint4*>(pl0 + 2 * plane_b + off_b) =
      make_uint4(pack_bf16(l[0], l[1]), pack_bf16(l[2], l[3]), pack_bf16(l[4], l[5]), pack_bf16(l[6], l[7]));
}
__device__ __forceinline__ void store_zero8(unsigned char* pl0, int plane_b, int off_b) {
  const uint4 z = make_uint4(0u, 0u, 0u, 0u);
  *reinterpret_cast<uint4*>(pl0 + off_b) = z;
  *reinterpret_cast<uint4*>(pl0 + plane_b + off_b) = z;
  *reinterpret_cast<uint4*>(pl0 + 2 * plane_b + off_b) = z;
}

// Frame chunk of a [N,C,P,K] tensor -> row image [64][Q].  Warp w owns rows w, w + 16, w + 32, w + 48; lane i owns the
// column pairs 2 i, 2 i + 1 and 64 + 2 i, 65 + 2 i of each, so consecutive lanes read consecutive addresses of a
// channel's contiguous (l, k) run (the loads of a warp coalesce; an 8-positions-per-thread mapping made every load
// touch 8 cache lines).  A thread's columns, and with them its frame / position offsets, never change.
// The 16 floats of the NEXT item are loaded into registers right after the current ones are stored, which hides the
// global latency behind the whole item; every element of the image is rewritten per item (zeros outside the data), so
// the region may serve as scratch in between.
struct ImgThread {
  int goff[2];           // l * sp + k * sk of column 2 (lane + 32 j), or -1 for padding / beyond the data
  int l[2], k[2];        // frame / position of that column
  int soff[2];           // byte offset of the column pair inside row 0 of a plane, -1 beyond the image
  int sk;
};
__device__ __forceinline__ ImgThread img_thread(const UnitGeom& g, const View4& t, int lane) {
  ImgThread it;
  it.sk = (int)t.sk;
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int q = 2 * (lane + 32 * j), l = q / g.KQ, k = q - l * g.KQ;       // KQ is even: a pair never straddles frames
    it.l[j] = l;
    it.k[j] = k;
    it.goff[j] = q < g.NPOS ? (int)(l * t.sp + k * t.sk) : -1;
    it.soff[j] = q < g.Q ? img16_off_b(0, q, g.sbo_b) : -1;
  }
  return it;
}
__device__ __forceinline__ void img_load(float (&v)[4][4], const ImgThread& it, const View4& t, int n, int p0, int pv, int C,
                                         int K, int warp) {
  const float* base = t.p + (long long)n * t.sn + (long long)p0 * t.sp;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = warp + 16 * i;
    const float* src = base + (long long)c * t.sc;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const bool ok = c < C && it.goff[j] >= 0 && it.l[j] < pv;
      v[i][2 * j] = (ok && it.k[j] < K) ? __ldg(src + it.goff[j]) : 0.f;
      v[i][2 * j + 1] = (ok && it.k[j] + 1 < K) ? __ldg(src + it.goff[j] + it.sk) : 0.f;
    }
  }
}
__device__ __forceinline__ void img_store(unsigned char* img, const float (&v)[4][4], const ImgThread& it, const UnitGeom& g,
                                          int warp) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = warp + 16 * i;
    unsigned char* row = img + (c >> 3) * g.sbo_b + ((c & 7) << 4);
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      if (it.soff[j] >= 0) {        // one 32-bit store per plane: the pair of bf16 (16-bit scattered stores were 3-4x slower)
        uint32_t h0, m0, l0, h1, m1, l1;
        split_bf16x3(v[i][2 * j], h0, m0, l0);
        split_bf16x3(v[i][2 * j + 1], h1, m1, l1);
        unsigned char* d = row + it.soff[j];
        *reinterpret_cast<uint32_t*>(d) = pack_bf16(h0, h1);
        *reinterpret_cast<uint32_t*>(d + g.plane_b) = pack_bf16(m0, m1);
        *reinterpret_cast<uint32_t*>(d + 2 * g.plane_b) = pack_bf16(l0, l1);
      }
    }
  }
}

// xmu_b[l][v][w] images of the item from the raw dynamic adjacency (alpha * pd + A_eff; transposed when adj_t).  Work unit =
// a pair of image elements (v, 2 i), (v, 2 i + 1): two loads, one 32-bit store per plane.  ptab[u] = first source element
// | image byte offset << 16 of pair u (u < K * ceil(K / 2)); the second source element is `estep` further (1, or K when
// the adjacency is used transposed) and exists when bit 15 of the low half is clear.  All loads of a thread are issued
// before the first value is used (one L2 round trip per item instead of one per frame).
struct XmuThread {       // the (at most two) image pairs of this thread: constant for the life of the CTA
  uint32_t t[2];         // ptab entries; 0xffffffff = none
  int grp, ngrp;         // with few pairs per frame the CTA splits into ngrp thread groups that take frames grp, grp + ngrp, ..
};
__device__ __forceinline__ XmuThread xmu_thread(const uint32_t* ptab, int npair, int tid) {
  XmuThread x;
  int shift = 5;
  while ((1 << shift) < npair && shift < 9) ++shift;
  x.ngrp = UT_NT >> shift;                   // 1 when npair > 256
  x.grp = tid >> shift;
  const int u = tid & ((1 << shift) - 1);
  x.t[0] = u < npair ? ptab[u] : 0xffffffffu;
  x.t[1] = (x.ngrp == 1 && u + UT_NT < npair) ? ptab[u + UT_NT] : 0xffffffffu;
  return x;
}
__device__ __forceinline__ void build_xmu(unsigned char* xmu, const UnitGeom& g, const float* __restrict__ pd,
                                          const float* aeff, const XmuThread& xt, int estep, float alpha, int n, int p0, int pv,
                                          int P, int KK, int nb, int tid) {
  constexpr int FB = 3;                                // frames in flight
  for (int b = 0; b < nb; ++b) {
    const float* src = pd + ((long long)(n * nb + b) * P + p0) * KK;
    unsigned char* im = xmu + (size_t)b * g.F * 3 * g.xplane_b;
    float ae[2][2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const uint32_t t = xt.t[k];
      ae[k][0] = t != 0xffffffffu ? aeff[b * KK + (t & 0x7fffu)] : 0.f;
      ae[k][1] = (t != 0xffffffffu && !(t & 0x8000u)) ? aeff[b * KK + (t & 0x7fffu) + estep] : 0.f;
    }
    for (int l0 = xt.grp; l0 < pv; l0 += FB * xt.ngrp) {
      float pr[FB][2][2];
#pragma unroll
      for (int j = 0; j < FB; ++j)
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const uint32_t t = xt.t[k];
          const bool on = l0 + j * xt.ngrp < pv && t != 0xffffffffu;
          const float* e = src + (l0 + j * xt.ngrp) * KK + (t & 0x7fffu);
          pr[j][k][0] = on ? __ldg(e) : 0.f;
          pr[j][k][1] = (on && !(t & 0x8000u)) ? __ldg(e + estep) : 0.f;
        }
#pragma unroll
      for (int j = 0; j < FB; ++j)
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const uint32_t t = xt.t[k];
          if (l0 + j * xt.ngrp < pv && t != 0xffffffffu) {
            const float v0 = fmaf(alpha, pr[j][k][0], ae[k][0]);
            const float v1 = (t & 0x8000u) ? 0.f : fmaf(alpha, pr[j][k][1], ae[k][1]);
            uint32_t h0, m0, q0, h1, m1, q1;
            split_bf16x3(v0, h0, m0, q0);
            split_bf16x3(v1, h1, m1, q1);
            unsigned char* d = im + (size_t)(l0 + j * xt.ngrp) * 3 * g.xplane_b + (t >> 16);
            *reinterpret_cast<uint32_t*>(d) = pack_bf16(h0, h1);
            *reinterpret_cast<uint32_t*>(d + g.xplane_b) = pack_bf16(m0, m1);
            *reinterpret_cast<uint32_t*>(d + 2 * g.xplane_b) = pack_bf16(q0, q1);
          }
        }
    }
  }
  if (pv < g.F) {        // frames beyond the tensor: their products must vanish
    for (int b = 0; b < nb; ++b) {
      const int words = (g.F - pv) * 3 * g.xplane_b / 4;
      uint32_t* z = reinterpret_cast<uint32_t*>(xmu + (size_t)(b * g.F + pv) * 3 * g.xplane_b);
      for (int i = tid; i < words; i += UT_NT) z[i] = 0u;
    }
  }
}

struct OpView {          // one operand of a six-term MMA chain: a row image seen K-major or MN-major
  uint32_t start, lbo_b, sbo_b, kstep_b, plane_b;
};
__device__ __forceinline__ OpView view_k(uint32_t img, int sbo_b, int plane_b, int q0) {     // rows = M/N, K = position
  return OpView{img + (uint32_t)(q0 >> 3) * IMG16_LBO_B, (uint32_t)IMG16_LBO_B, (uint32_t)sbo_b, 2u * IMG16_LBO_B, (uint32_t)plane_b};
}
__device__ __forceinline__ OpView view_mn(uint32_t img, int sbo_b, int plane_b, int q0) {    // M/N = position, K = rows
  return OpView{img + (uint32_t)(q0 >> 3) * IMG16_LBO_B, (uint32_t)sbo_b, (uint32_t)IMG16_LBO_B, 2u * (uint32_t)sbo_b, (uint32_t)plane_b};
}
__device__ __forceinline__ bool elect_one() {
  uint32_t p;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}\n" : "=r"(p));
  return p != 0;
}
// A family of `nrep` MMA chains  D_r (+)= A_r B_r^T  (r = frame of the item: accumulator, A window and B image advance
// linearly), each `ksteps` x 16 long with the six split products hh hm mh mm hl lh per k-step.
// Issue order matters: a product that accumulates into the accumulator of the previous instruction waits for it (small
// MMAs then cost their full ~46-cycle latency each: measured), so step i of EVERY chain is issued before step i + 1, and
// two families that do not depend on each other are interleaved (issue2).  All of this is run by ALL lanes of the
// issuing warp: the descriptor arithmetic stays on the uniform datapath (issuing from inside `if (tid == 0)` cost
// ~90 cycles per instruction in R2UR moves) and only the elected lane fires the instructions.
struct Fam {
  uint32_t d, a_lo, b_lo, a_hi, b_hi;      // first chain: accumulator, descriptor halves of the h planes at k-step 0
  uint32_t a_ks, b_ks, a_pl, b_pl;         // 16-byte units: per k-step, per split plane
  uint32_t d_inc, a_inc, b_inc;            // per chain (TMEM columns, 16-byte units)
  uint32_t idesc;
  int nrep, ksteps, terms;
  bool acc;
};
__device__ __forceinline__ Fam make_fam(int terms, uint32_t tmem_d, const OpView& a, const OpView& b, int ksteps, uint32_t idesc,
                                        bool acc, int nrep = 1, uint32_t d_inc = 0, uint32_t a_inc_b = 0, uint32_t b_inc_b = 0) {
  Fam f;
  f.terms = terms;
  f.d = tmem_d;
  f.a_hi = (a.sbo_b >> 4) | (1u << 14);
  f.b_hi = (b.sbo_b >> 4) | (1u << 14);
  f.a_lo = ((a.start & 0x3FFFFu) >> 4) | ((a.lbo_b >> 4) << 16);
  f.b_lo = ((b.start & 0x3FFFFu) >> 4) | ((b.lbo_b >> 4) << 16);
  f.a_ks = a.kstep_b >> 4; f.b_ks = b.kstep_b >> 4;
  f.a_pl = a.plane_b >> 4; f.b_pl = b.plane_b >> 4;
  f.d_inc = d_inc; f.a_inc = a_inc_b >> 4; f.b_inc = b_inc_b >> 4;
  f.idesc = idesc;
  f.nrep = nrep; f.ksteps = ksteps;
  f.acc = acc;
  return f;
}
// one split product (planes ta of A, tb of B) of every chain of the family at k-step offsets (al0, bl0)
__device__ __forceinline__ void fam_product(const Fam& f, uint32_t al0, uint32_t bl0, uint32_t ta, uint32_t tb, uint32_t acc,
                                            bool leader) {
  const uint32_t al = al0 + ta * f.a_pl, bl = bl0 + tb * f.b_pl;
  for (int r = 0; r < f.nrep; ++r) {
    const uint32_t d = f.d + r * f.d_inc, alr = al + r * f.a_inc, blr = bl + r * f.b_inc;
    mma_f16_lohi(d, alr, f.a_hi, blr, f.b_hi, f.idesc, acc, leader);
  }
}
template <bool TWO>
__device__ __forceinline__ void issue_fams(const Fam& x, const Fam& y) {
  const bool leader = elect_one();
  const int kmax = TWO ? max(x.ksteps, y.ksteps) : x.ksteps;
  uint32_t xa = x.a_lo, xb = x.b_lo, ya = y.a_lo, yb = y.b_lo;
  for (int ks = 0; ks < kmax; ++ks, xa += x.a_ks, xb += x.b_ks, ya += y.a_ks, yb += y.b_ks) {
#pragma unroll
    for (int t = 0; t < 6; ++t) {            // hh hm mh mm hl lh
      const uint32_t ta = (t == 2 || t == 3) ? 1u : (t == 5 ? 2u : 0u), tb = (t == 1 || t == 3) ? 1u : (t == 4 ? 2u : 0u);
      if (ks < x.ksteps && t < x.terms) fam_product(x, xa, xb, ta, tb, (x.acc || ks > 0 || t > 0) ? 1u : 0u, leader);
      if (TWO && ks < y.ksteps && t < y.terms) fam_product(y, ya, yb, ta, tb, (y.acc || ks > 0 || t > 0) ? 1u : 0u, leader);
    }
  }
}
__device__ __forceinline__ void issue1(const Fam& x) { issue_fams<false>(x, x); }
__device__ __forceinline__ void issue2(const Fam& x, const Fam& y) { issue_fams<true>(x, y); }

// Which accumulator rows a warp drains.  M = 64 accumulators keep row m on TMEM lane (m % 16) + 32 (m / 16): the lower half
// of every warp's lane quarter; M = 128 accumulators keep row m on lane m (rows 64 b .. 64 b + 63 = branch b).
struct RowMap {
  int qd;            // TMEM lane quarter of this warp (always warp % 4)
  int row;           // image row of this lane
  bool active;       // this lane holds a row
  bool part;         // this warp takes part at all
  int g0, gstep;     // column groups g0, g0 + gstep, ...
};
__device__ __forceinline__ RowMap rows_m64(int warp, int lane) {
  return RowMap{warp & 3, 16 * (warp & 3) + lane, lane < 16, true, warp >> 2, 4};
}
__device__ __forceinline__ RowMap rows_m128_branch(int warp, int lane, int b) {
  const int qd = warp & 3;
  return RowMap{qd, 32 * (qd & 1) + lane, true, (qd >> 1) == b, warp >> 2, 4};
}

// accumulator [64 rows][NG * 8 columns] at TMEM column `col` -> row image (thread = row).  bias[row] is added, the sum of the
// stored values is returned (row sums of h = bias gradient), groups NG .. QG-1 are written as zeros.
__device__ __forceinline__ float drain_to_image(uint32_t tmem_base, int col, unsigned char* img, const UnitGeom& g,
                                                const float* bias, const RowMap& rm) {
  float rs = 0.f;
  if (!rm.part) return rs;
  const uint32_t tl = tmem_base + ((uint32_t)(32 * rm.qd) << 16) + (uint32_t)col;
  const float bv = (bias && rm.active) ? bias[rm.row] : 0.f;
  for (int gi = rm.g0; gi < g.QG; gi += 2 * rm.gstep) {
    const int gj = gi + rm.gstep;
    uint32_t v0[8], v1[8];
    if (gi < g.NG) tmem_ld8(tl + 8 * gi, v0);
    if (gj < g.NG) tmem_ld8(tl + 8 * gj, v1);
    tmem_ld_wait();
    if (rm.active) {
      float f[8];
      if (gi < g.NG) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          f[e] = __uint_as_float(v0[e]) + bv;
          rs += f[e];
        }
        store_split8(img, g.plane_b, img16_off_b(rm.row, 8 * gi, g.sbo_b), f);
      } else {
        store_zero8(img, g.plane_b, img16_off_b(rm.row, 8 * gi, g.sbo_b));
      }
      if (gj < g.NG) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          f[e] = __uint_as_float(v1[e]) + bv;
          rs += f[e];
        }
        store_split8(img, g.plane_b, img16_off_b(rm.row, 8 * gj, g.sbo_b), f);
      } else if (gj < g.QG) {
        store_zero8(img, g.plane_b, img16_off_b(rm.row, 8 * gj, g.sbo_b));
      }
    }
  }
  return rs;
}

// accumulator [rows < nrows][ng * 8 columns] -> fp32 staging tile st[row][ld]
__device__ __forceinline__ void drain_to_stage(uint32_t tmem_base, int col, float* st, int ld, int ng, int nrows,
                                               const RowMap& rm) {
  if (!rm.part) return;
  const uint32_t tl = tmem_base + ((uint32_t)(32 * rm.qd) << 16) + (uint32_t)col;
  for (int gi = rm.g0; gi < ng; gi += rm.gstep) {
    uint32_t v[8];
    tmem_ld8(tl + 8 * gi, v);
    tmem_ld_wait();
    if (rm.active && rm.row < nrows) {
      float4* d = reinterpret_cast<float4*>(st + rm.row * ld + 8 * gi);
      d[0] = make_float4(__uint_as_float(v[0]), __uint_as_float(v[1]), __uint_as_float(v[2]), __uint_as_float(v[3]));
      d[1] = make_float4(__uint_as_float(v[4]), __uint_as_float(v[5]), __uint_as_float(v[6]), __uint_as_float(v[7]));
    }
  }
}

// fp32 staging tile [rows][ld] -> tensor chunk, coalesced along each channel's (l, k) run.  pst[j] / pgo[j]: staging
// column and global offset of position j = l * K + k (tables built once per CTA: no divisions here)
__device__ __forceinline__ void stage_to_global(const float* st, int ld, float* gb, long long sc, const unsigned short* pst,
                                                const int* pgo, const float* sb, long long ssc, const int* psk, int rows,
                                                int npos, bool ok, int warp, int lane) {
  const float nanv = __int_as_float(0x7fc00000);      // a stalled pipeline must be loud
  for (int o = warp; o < rows; o += UT_NT / 32) {
    const float* sr = st + o * ld;
    float* gr = gb + (long long)o * sc;
    const float* kr = sb ? sb + (long long)o * ssc : nullptr;
    for (int j = lane; j < npos; j += 32) {
      float v = ok ? sr[pst[j]] : nanv;
      if (kr) v += __ldg(kr + psk[j]);
      gr[pgo[j]] = v;
    }
  }
}

// once per CTA: weight images, biases, effective static adjacency, index tables, TMEM, mbarrier
template <typename Q>
__device__ __forceinline__ uint32_t unit_setup(const Q& q, const UnitGeom& g, unsigned char* smem, const unsigned char* wimg,
                                               const View4& outv, const View4* skipv, int tid, int warp) {
  float* aeff = reinterpret_cast<float*>(smem + g.o_aeff);
  float* bias = reinterpret_cast<float*>(smem + g.o_bias);
  uint32_t* etab = reinterpret_cast<uint32_t*>(smem + g.o_etab);
  unsigned short* gst = reinterpret_cast<unsigned short*>(smem + g.o_gst);
  unsigned short* pst = reinterpret_cast<unsigned short*>(smem + g.o_pst);
  int* pout = reinterpret_cast<int*>(smem + g.o_pout);
  int* pskip = reinterpret_cast<int*>(smem + g.o_pskip);
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem + g.o_bar);
  uint32_t* slot = reinterpret_cast<uint32_t*>(mbar + 1);
  const int K = q.K, KK = K * K;
  for (int i = tid; i < q.nb * KK; i += UT_NT) {
    const int b = i / KK, e = i - b * KK;
    float a = __ldg(q.adj[b] + e);
    if (q.adj_w[b]) a *= __ldg(q.adj_w[b] + e);
    if (q.adj_r[b]) a += __ldg(q.adj_r[b] + e);
    aeff[i] = a;
  }
  for (int i = tid; i < q.nb * 64; i += UT_NT) bias[i] = (i & 63) < q.Cout ? __ldg(q.b_f[i >> 6] + (i & 63)) : 0.f;
  for (int e = tid; e < KK; e += UT_NT) {
    const int r = e / K, c = e - r * K;
    const int v = q.adj_t ? c : r, w = q.adj_t ? r : c;
    gst[e] = (unsigned short)(v * g.KQ + w);          // pd element e in a [KQ][KQ] fp32 staging tile of xmu / gxmu
  }
  {
    const int hk = (K + 1) / 2;
    for (int u = tid; u < K * hk; u += UT_NT) {         // image pair (v, 2 i), (v, 2 i + 1)
      const int v = u / hk, i = u - v * hk, w = 2 * i;
      const uint32_t e0 = (uint32_t)(q.adj_t ? w * K + v : v * K + w);
      etab[u] = e0 | (w + 1 < K ? 0u : 0x8000u) | ((uint32_t)img16_off_b(v, w, g.xsbo_b) << 16);
    }
  }
  for (int j = tid; j < g.F * K; j += UT_NT) {
    const int l = j / K, k = j - l * K;
    pst[j] = (unsigned short)(l * g.KQ + k);
    pout[j] = (int)(l * outv.sp + k * outv.sk);
    if (skipv) pskip[j] = (int)(l * skipv->sp + k * skipv->sk);
  }
  {   // xmu images: the padding rows / columns stay zero for the life of the CTA
    uint32_t* z = reinterpret_cast<uint32_t*>(smem + g.o_xmu);
    for (int i = tid; i < q.nb * g.F * 3 * g.xplane_b / 4; i += UT_NT) z[i] = 0u;
  }
  if (tid == 0) {         // weight images: one TMA bulk copy (cp.async.bulk) counted on the MMA barrier's first phase
    mbar_init(mbar, 1);
    mbar_init_fence();
    mbar_expect_tx(mbar, (uint32_t)(q.nb * 3 * UT_WP_B));
    bulk_g2s(smem + g.o_w, wimg, (uint32_t)(q.nb * 3 * UT_WP_B), mbar);
  }
  if (warp == 0) tmem_alloc(slot, (uint32_t)g.tmem_cols);
  fence_async_smem();
  fence_before();
  __syncthreads();
  fence_after();
  mbar_wait(mbar, 0);     // phase 0 is spent on the weights: the MMA phases of the kernels start at parity 1
  return *slot;
}

// ------------------------------------------------------------------------------------------ forward
struct UnitFwdParams {
  int N, Cin, Cout, P, K, nb, adj_t;
  View4 x, out, skip;
  const float* pd;
  const float* alpha;
  const float* adj[DSTD_MAX_BRANCH];
  const float* adj_w[DSTD_MAX_BRANCH];
  const float* adj_r[DSTD_MAX_BRANCH];
  const float* b_f[DSTD_MAX_BRANCH];
  const unsigned char* wimg;
  int* err_flag;
};

__global__ void __launch_bounds__(UT_NT, 1) unit_fwd_tc_kernel(UnitFwdParams q, UnitGeom g) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned char* x0 = smem + g.o_x0;
  unsigned char* s = smem + g.o_s;
  unsigned char* xmu = smem + g.o_xmu;
  const float* aeff = reinterpret_cast<const float*>(smem + g.o_aeff);
  const float* bias = reinterpret_cast<const float*>(smem + g.o_bias);
  const uint32_t* etab = reinterpret_cast<const uint32_t*>(smem + g.o_etab);
  const unsigned short* pst = reinterpret_cast<const unsigned short*>(smem + g.o_pst);
  const int* pout = reinterpret_cast<const int*>(smem + g.o_pout);
  const int* pskip = reinterpret_cast<const int*>(smem + g.o_pskip);
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem + g.o_bar);
  // the broadcast shuffle tells the compiler that the TMEM base is warp-uniform (it was read from shared memory)
  const uint32_t tm = __shfl_sync(0xffffffffu, unit_setup(q, g, smem, q.wimg, q.out, q.skip.p ? &q.skip : nullptr, tid, warp), 0);
  const float alpha = q.alpha ? __ldg(q.alpha) : 1.0f;
  const int K = q.K, KK = K * K, P = q.P, nb = q.nb;
  const int nchunk = (P + g.F - 1) / g.F;
  const long long nitems = (long long)q.N * nchunk;
  // TMEM: D1 = xf of every branch (nb == 2: ONE M = 128 accumulator, rows 64 b .. = branch b) | Dout
  const uint32_t d1 = tm, dout = tm + (uint32_t)g.N16;
  const bool stacked = nb == 2;
  // the xf chain is split into two independent column halves when that keeps N a multiple of 16 (M = 128) / 8 (M = 64)
  const int f1_full = stacked ? g.N16 : g.NPOS;
  const int f1_rep = 1, f1_n = f1_full;     // (two column halves re-read A twice: the chains are shared-memory bound)
  const uint32_t id_f1 = idesc_bf16(stacked ? 128 : 64, f1_n, 0, 1), id_f2 = idesc_bf16(64, g.KQ, 0, 1);
  const uint32_t sx0 = smem_u32(x0), ss = smem_u32(s), sw = smem_u32(smem + g.o_w), sxm = smem_u32(xmu);
  const int ST_LD = g.NPOS + 4;
  float* stage = reinterpret_cast<float*>(s);          // the scratch image is free again when the epilogue runs
  const ImgThread itx = img_thread(g, q.x, lane);
  const XmuThread xth = xmu_thread(etab, K * ((K + 1) / 2), tid);
  float xv[4][4];
  uint32_t phase = 1;
  bool ok = true;
  if ((long long)blockIdx.x < nitems) {
    const int n = (int)(blockIdx.x / nchunk), p0 = (int)(blockIdx.x - (long long)n * nchunk) * g.F;
    img_load(xv, itx, q.x, n, p0, min(g.F, P - p0), q.Cin, K, warp);
  }

  UT_PH_DECL;
  for (long long item = blockIdx.x; item < nitems; item += gridDim.x) {
    const int n = (int)(item / nchunk), p0 = (int)(item - (long long)n * nchunk) * g.F;
    const int pv = min(g.F, P - p0);
    img_store(x0, xv, itx, g, warp);
    UT_PH(0);
    build_xmu(xmu, g, q.pd, aeff, xth, q.adj_t ? K : 1, alpha, n, p0, pv, P, KK, nb, tid);
    UT_PH(1);
    fence_async_smem();
    UT_PH(8);
    fence_before();
    __syncthreads();
    UT_PH(9);
    if (warp == 0) {      // F1: xf = [Wf_0; Wf_1] x (one M = 128 chain for both branches)
      fence_after();
      issue1(make_fam(g.terms, d1, view_k(sw, 8 * IMG16_LBO_B, nb * UT_WP_B, 0), view_mn(sx0, g.sbo_b, g.plane_b, 0), g.CinK / 16, id_f1,
                      false, f1_rep, f1_n, 0, (uint32_t)(f1_n >> 3) * IMG16_LBO_B));
      commit_elect(mbar);
      __syncwarp();
      ok = mbar_wait(mbar, phase) && ok;
    }
    UT_PH(2);
    ok = __syncthreads_and(ok);
    phase ^= 1;
    fence_after();
    UT_PH(3);
    for (int b = 0; b < nb; ++b) {
      drain_to_image(tm, 0, s, g, bias + b * 64, stacked ? rows_m128_branch(warp, lane, b) : rows_m64(warp, lane));   // X1_b = split(xf_b + bf_b)
      fence_async_smem();
      fence_before();
      __syncthreads();
      UT_PH(4);
      if (warp == 0) {    // F2: out[:, frame l] += xf_b[:, frame l] xmu_b[l]
        fence_after();
        issue1(make_fam(g.terms, dout, view_k(ss, g.sbo_b, g.plane_b, 0), view_mn(sxm + (uint32_t)(b * g.F) * 3 * g.xplane_b, g.xsbo_b, g.xplane_b, 0),
                        g.KW / 16, id_f2, b > 0, g.F, g.KQ, (uint32_t)(g.KQ >> 3) * IMG16_LBO_B, 3u * g.xplane_b));
        commit_elect(mbar);
        __syncwarp();
      }
      if (b == nb - 1) {
        // the next item's x chunk travels during the last MMA phase and the epilogue.  (Issued here, after the last
        // proxy fence of the item: a fence waits for ALL outstanding memory operations of the thread, loads included.)
        const long long nx = item + gridDim.x;
        if (nx < nitems) {
          const int n2 = (int)(nx / nchunk), q0 = (int)(nx - (long long)n2 * nchunk) * g.F;
          img_load(xv, itx, q.x, n2, q0, min(g.F, P - q0), q.Cin, K, warp);
        }
      }
      if (warp == 0) ok = mbar_wait(mbar, phase) && ok;
      UT_PH(5);
      ok = __syncthreads_and(ok);      // the scratch image is rewritten by the next branch / used as staging
      phase ^= 1;
      fence_after();
      UT_PH(6);
    }
    // epilogue: TMEM -> fp32 staging -> (+ skip) -> out, coalesced along each channel's contiguous (l, k) run
    drain_to_stage(tm, g.N16, stage, ST_LD, g.NG, q.Cout, rows_m64(warp, lane));
    fence_before();
    __syncthreads();
    stage_to_global(stage, ST_LD, q.out.p + (long long)n * q.out.sn + (long long)p0 * q.out.sp, q.out.sc, pst, pout,
                    q.skip.p ? q.skip.p + (long long)n * q.skip.sn + (long long)p0 * q.skip.sp : nullptr, q.skip.sc, pskip,
                    q.Cout, pv * K, ok, warp, lane);
    __syncthreads();      // staging / TMEM free before the next item
    fence_after();
    UT_PH(7);
  }
#ifdef DSTD_PHASE_TIMING
  if (blockIdx.x == 0 && tid == 0)
    printf("unit_fwd_tc phases (cycles, CTA 0, F=%d): build_x %lld build_xmu+sync %lld issueF1 %lld waitF1 %lld drainX1 %lld "
           "issueF2 %lld waitF2 %lld epilogue %lld | proxy fence %lld sync %lld\n", g.F, tph[0], tph[1], tph[2], tph[3], tph[4], tph[5], tph[6], tph[7], tph[8], tph[9]);
#endif
  if (!ok && tid == 0 && q.err_flag) {
    *(volatile int*)q.err_flag = 1;
    __threadfence_system();
  }
  fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tm, (uint32_t)g.tmem_cols);
}

// ------------------------------------------------------------------------------------------ backward
struct UnitBwdParams {
  int N, Cin, Cout, P, K, nb, adj_t;
  View4 x, gout, gx;
  const float* pd;
  const float* alpha;
  const float* adj[DSTD_MAX_BRANCH];
  const float* adj_w[DSTD_MAX_BRANCH];
  const float* adj_r[DSTD_MAX_BRANCH];
  const float* b_f[DSTD_MAX_BRANCH];
  const unsigned char* wimg;
  float* gxm;          // [N,nb,P,K,K]
  float* part_w;       // [ctas][nb][Cout][Cin]
  float* part_b;       // [ctas][nb][Cout]
  int* err_flag;
};

__global__ void __launch_bounds__(UT_NT, 1) unit_bwd_tc_kernel(UnitBwdParams q, UnitGeom g) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned char* x0 = smem + g.o_x0;
  unsigned char* g1 = smem + g.o_g1;
  unsigned char* s = smem + g.o_s;
  unsigned char* xmu = smem + g.o_xmu;
  const float* aeff = reinterpret_cast<const float*>(smem + g.o_aeff);
  const float* bias = reinterpret_cast<const float*>(smem + g.o_bias);
  const uint32_t* etab = reinterpret_cast<const uint32_t*>(smem + g.o_etab);
  const unsigned short* gst = reinterpret_cast<const unsigned short*>(smem + g.o_gst);
  const unsigned short* pst = reinterpret_cast<const unsigned short*>(smem + g.o_pst);
  const int* pout = reinterpret_cast<const int*>(smem + g.o_pout);
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem + g.o_bar);
  const uint32_t tm = __shfl_sync(0xffffffffu, unit_setup(q, g, smem, q.wimg, q.gx, nullptr, tid, warp), 0);   // warp-uniform
  const float alpha = q.alpha ? __ldg(q.alpha) : 1.0f;
  const int K = q.K, KK = K * K, P = q.P, nb = q.nb;
  const int nchunk = (P + g.F - 1) / g.F;
  const long long nitems = (long long)q.N * nchunk;
  // TMEM columns: D1 (xf; nb == 2: one M = 128 accumulator for both branches) | D2 (h_b) | D3 (gxmu_b: M = 128, all frame
  // pairs, the diagonal blocks are kept) | D4 (gx) | D5_b (gWf_b, resident for the life of the CTA)
  const int c_d2 = g.N16, c_d3 = g.N16 + g.NPOS, c_d4 = 2 * g.N16 + g.NPOS, c_d5 = 2 * g.N16 + 2 * g.NPOS;
  const uint32_t d1 = tm, d2 = tm + c_d2, d3 = tm + c_d3, d4 = tm + c_d4, d5 = tm + c_d5;
  const bool stacked = nb == 2;
  // long chains are split into two independent column halves when that keeps N a multiple of 16 (M = 128) / 8 (M = 64)
  const int b1_full = stacked ? g.N16 : g.NPOS;
  const int b1_rep = 1, b1_n = b1_full;     // (two column halves re-read A twice: the chains are shared-memory bound)
  const int b3_rep = 1, b3_n = g.N16;
  const uint32_t id_b1 = idesc_bf16(stacked ? 128 : 64, b1_n, 0, 1), id_b2 = idesc_bf16(64, g.KQ, 0, 0),
                 id_b3 = idesc_bf16(128, b3_n, 1, 1), id_b4 = idesc_bf16(64, g.NPOS, 1, 1), id_b5 = idesc_bf16(64, g.CinN, 0, 0);
  const uint32_t sx0 = smem_u32(x0), sg1 = smem_u32(g1), ss = smem_u32(s), sw = smem_u32(smem + g.o_w), sxm = smem_u32(xmu);
  const int ST_LD = g.NPOS + 4;
  float* stage_gx = reinterpret_cast<float*>(g1);      // gout image is dead when the gx epilogue runs
  float* stage_gxm = reinterpret_cast<float*>(s);      // [F][KQ rows v][KQ] between B3 and the h drain
  const ImgThread itx = img_thread(g, q.x, lane), itg = img_thread(g, q.gout, lane);
  const XmuThread xth = xmu_thread(etab, K * ((K + 1) / 2), tid);
  float xv[4][4], gv[4][4];
  float accb[DSTD_MAX_BRANCH] = {0.f, 0.f};
  uint32_t phase = 1;
  bool ok = true;
  if ((long long)blockIdx.x < nitems) {
    const int n = (int)(blockIdx.x / nchunk), p0 = (int)(blockIdx.x - (long long)n * nchunk) * g.F;
    img_load(xv, itx, q.x, n, p0, min(g.F, P - p0), q.Cin, K, warp);
    img_load(gv, itg, q.gout, n, p0, min(g.F, P - p0), q.Cout, K, warp);
  }

  UT_PH_DECL;
  for (long long item = blockIdx.x; item < nitems; item += gridDim.x) {
    const int n = (int)(item / nchunk), p0 = (int)(item - (long long)n * nchunk) * g.F;
    const int pv = min(g.F, P - p0);
    const bool first = item == (long long)blockIdx.x;
    img_store(x0, xv, itx, g, warp);
    img_store(g1, gv, itg, g, warp);
    UT_PH(0);
    build_xmu(xmu, g, q.pd, aeff, xth, q.adj_t ? K : 1, alpha, n, p0, pv, P, KK, nb, tid);
    fence_async_smem();
    fence_before();
    __syncthreads();
    UT_PH(1);
#pragma unroll
    for (int b = 0; b < DSTD_MAX_BRANCH; ++b) {
      if (b >= nb) break;
      const uint32_t swb = sw + b * UT_WP_B;
      if (warp == 0) {    // B1: xf = [Wf_0; Wf_1] x (once per item) ; B2: h_b[:, frame l] = gout[:, frame l] xmu_b[l]^T
        fence_after();
        Fam f1 = make_fam(g.terms, d1, view_k(sw, 8 * IMG16_LBO_B, nb * UT_WP_B, 0), view_mn(sx0, g.sbo_b, g.plane_b, 0), g.CinK / 16, id_b1,
                          false, b1_rep, b1_n, 0, (uint32_t)(b1_n >> 3) * IMG16_LBO_B);
        if (b > 0) f1.ksteps = 0;
        issue2(f1, make_fam(g.terms, d2, view_k(sg1, g.sbo_b, g.plane_b, 0), view_k(sxm + (uint32_t)(b * g.F) * 3 * g.xplane_b, g.xsbo_b, g.xplane_b, 0),
                            g.KW / 16, id_b2, false, g.F, g.KQ, (uint32_t)(g.KQ >> 3) * IMG16_LBO_B, 3u * g.xplane_b));
        commit_elect(mbar);
        __syncwarp();
        ok = mbar_wait(mbar, phase) && ok;
      }
      ok = __syncthreads_and(ok);
      phase ^= 1;
      fence_after();
      UT_PH(2);
      drain_to_image(tm, 0, s, g, bias + b * 64, stacked ? rows_m128_branch(warp, lane, b) : rows_m64(warp, lane));   // X1_b = split(xf_b + bf_b)
      fence_async_smem();
      fence_before();
      __syncthreads();
      UT_PH(3);
      if (warp == 0) {    // B3: G[(l,v)][(l',w)] = sum_o xf_b[o][l,v] gout[o][l',w]: ONE M = 128 chain over all frame pairs (the
        fence_after();    // per-frame M = 64, N = KQ products cost ~46 cycles each however small); gxmu_b[l] = block (l, l)
        issue1(make_fam(g.terms, d3, view_mn(ss, g.sbo_b, g.plane_b, 0), view_mn(sg1, g.sbo_b, g.plane_b, 0), g.CoutK / 16, id_b3, false,
                        b3_rep, b3_n, 0, (uint32_t)(b3_n >> 3) * IMG16_LBO_B));
        commit_elect(mbar);
        __syncwarp();
        ok = mbar_wait(mbar, phase) && ok;
      }
      ok = __syncthreads_and(ok);
      phase ^= 1;
      fence_after();
      UT_PH(4);
      // gxmu -> staging [l][v][KQ] (the X1 image is dead) -> HBM in the layout of pd
      {   // lane = position (l, v) of lane quarter warp % 4; it keeps the KQ columns of its own frame
        const int qd = warp & 3, pos = 32 * qd + lane, lf = pos / g.KQ;
        const int l_lo = (32 * qd) / g.KQ, l_hi = min(g.F - 1, (32 * qd + 31) / g.KQ);
        for (int l = l_lo; l <= l_hi; ++l)
          for (int gi = warp >> 2; gi < g.KQ / 8; gi += 4) {
            uint32_t v[8];
            tmem_ld8(tm + ((uint32_t)(32 * qd) << 16) + (uint32_t)(c_d3 + l * g.KQ + 8 * gi), v);
            tmem_ld_wait();
            if (lf == l && pos - l * g.KQ < K) {
              float4* d = reinterpret_cast<float4*>(stage_gxm + pos * g.KQ + 8 * gi);
              d[0] = make_float4(__uint_as_float(v[0]), __uint_as_float(v[1]), __uint_as_float(v[2]), __uint_as_float(v[3]));
              d[1] = make_float4(__uint_as_float(v[4]), __uint_as_float(v[5]), __uint_as_float(v[6]), __uint_as_float(v[7]));
            }
          }
      }
      fence_before();
      __syncthreads();
      {
        float* dst = q.gxm + ((long long)(n * nb + b) * P + p0) * KK;
        const float nanv = __int_as_float(0x7fc00000);
        for (int l = 0; l < pv; ++l)
          for (int e = tid; e < KK; e += UT_NT) dst[l * KK + e] = ok ? stage_gxm[l * g.KQ * g.KQ + gst[e]] : nanv;
      }
      __syncthreads();
      fence_after();
      UT_PH(5);
      accb[b] += drain_to_image(tm, c_d2, s, g, nullptr, rows_m64(warp, lane));        // H1_b = split(h_b); row sums = bias gradient
      fence_async_smem();
      fence_before();
      __syncthreads();
      UT_PH(6);
      if (warp == 0) {    // B4: gx += Wf_b^T h_b ; B5: gWf_b += h_b x^T
        fence_after();
        issue2(make_fam(g.terms, d4, view_mn(swb, 8 * IMG16_LBO_B, nb * UT_WP_B, 0), view_mn(ss, g.sbo_b, g.plane_b, 0), g.CoutK / 16, id_b4, b > 0),
               make_fam(g.terms, d5 + b * g.CinN, view_k(ss, g.sbo_b, g.plane_b, 0), view_k(sx0, g.sbo_b, g.plane_b, 0), g.Q / 16, id_b5, !first));
        commit_elect(mbar);
        __syncwarp();
      }
      if (b == nb - 1) {
        // the next item's x / gout chunks travel during the last MMA phase and the gx epilogue.  (Issued here, after the
        // last proxy fence of the item: a fence waits for ALL outstanding memory operations of the thread, loads included.)
        const long long nx = item + gridDim.x;
        if (nx < nitems) {
          const int n2 = (int)(nx / nchunk), q0 = (int)(nx - (long long)n2 * nchunk) * g.F;
          img_load(xv, itx, q.x, n2, q0, min(g.F, P - q0), q.Cin, K, warp);
          img_load(gv, itg, q.gout, n2, q0, min(g.F, P - q0), q.Cout, K, warp);
        }
      }
      if (warp == 0) ok = mbar_wait(mbar, phase) && ok;
      ok = __syncthreads_and(ok);      // the scratch image / D1..D3 are reused by the next branch
      phase ^= 1;
      fence_after();
      UT_PH(7);
    }
    // gx chunk: TMEM -> fp32 staging -> HBM, coalesced along each channel's contiguous (l, k) run
    drain_to_stage(tm, c_d4, stage_gx, ST_LD, g.NG, q.Cin, rows_m64(warp, lane));
    fence_before();
    __syncthreads();
    stage_to_global(stage_gx, ST_LD, q.gx.p + (long long)n * q.gx.sn + (long long)p0 * q.gx.sp, q.gx.sc, pst, pout, nullptr, 0,
                    nullptr, q.Cin, pv * K, ok, warp, lane);
    __syncthreads();
    fence_after();
    UT_PH(8);
  }
#ifdef DSTD_PHASE_TIMING
  if (blockIdx.x == 0 && tid == 0)
    printf("unit_bwd_tc phases (cycles, CTA 0, F=%d): build_x_g %lld build_xmu+sync %lld B1B2 %lld drainX1 %lld B3 %lld "
           "gxm_out %lld drainH1 %lld B4B5 %lld gx_out %lld\n", g.F, tph[0], tph[1], tph[2], tph[3], tph[4], tph[5], tph[6],
           tph[7], tph[8]);
#endif

  // ---- per-CTA partials of the conv_f gradients: D5_b -> part_w, row sums -> part_b (fixed-order combine of the four
  //      column-group warps of a lane quarter)
  {
    const bool any = (long long)blockIdx.x < nitems;
    float* red = reinterpret_cast<float*>(s);             // [nb][4 wq][64]
    const int qd = warp & 3, wq = warp >> 2, r = 16 * qd + lane;
    if (lane < 16)
      for (int b = 0; b < nb; ++b) red[(b * 4 + wq) * 64 + r] = accb[b];
    float* pw = q.part_w + (long long)blockIdx.x * nb * q.Cout * q.Cin;
    if (!any) {           // this CTA had no item: D5 was never written
      for (int i = tid; i < nb * q.Cout * q.Cin; i += UT_NT) pw[i] = 0.f;
    } else {
      for (int b = 0; b < nb; ++b) {
        const uint32_t tl = tm + ((uint32_t)(32 * qd) << 16) + c_d5 + b * g.CinN;
        for (int c0 = 8 * wq; c0 < g.CinN; c0 += 32) {
          uint32_t v[8];
          tmem_ld8(tl + c0, v);
          tmem_ld_wait();
          if (lane < 16 && r < q.Cout) {
#pragma unroll
            for (int e = 0; e < 8; ++e)
              if (c0 + e < q.Cin) pw[((long long)b * q.Cout + r) * q.Cin + c0 + e] = ok ? __uint_as_float(v[e]) : __int_as_float(0x7fc00000);
          }
        }
      }
    }
    __syncthreads();
    float* pb = q.part_b + (long long)blockIdx.x * nb * q.Cout;
    for (int i = tid; i < nb * q.Cout; i += UT_NT) {
      const int b = i / q.Cout, o = i - b * q.Cout;
      const float* rr = red + b * 4 * 64 + o;
      pb[i] = (rr[0] + rr[64]) + (rr[128] + rr[192]);
    }
  }
  if (!ok && tid == 0 && q.err_flag) {
    *(volatile int*)q.err_flag = 1;
    __threadfence_system();
  }
  fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tm, (uint32_t)g.tmem_cols);
}

// ------------------------------------------------------------------------------------------ weight images
// wimg[plane h|m|l][b][row image [64][64]]: conv_f weights of branch b (rows = output channel, columns = input channel),
// zero outside [Cout][Cin]; the branches of a plane are contiguous so that both read as ONE [128][64] K-major operand
__global__ void pack_w16_kernel(PackParams q, unsigned char* wimg) {
  const int total = q.nb * 64 * 8;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int b = i >> 9, o = (i >> 3) & 63, c0 = (i & 7) * 8;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = (o < q.Cout && c0 + e < q.Cin) ? __ldg(q.w_f[b] + (long long)o * q.Cin + c0 + e) : 0.f;
    uint32_t h[8], m[8], l[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) split_bf16x3(v[e], h[e], m[e], l[e]);
    unsigned char* d = wimg + (size_t)b * UT_WP_B + img16_off_b(o, c0, 8 * IMG16_LBO_B);     // [plane][branch][row image]
    const size_t ps = (size_t)q.nb * UT_WP_B;
    *reinterpret_cast<uint4*>(d) = make_uint4(pack_bf16(h[0], h[1]), pack_bf16(h[2], h[3]), pack_bf16(h[4], h[5]), pack_bf16(h[6], h[7]));
    *reinterpret_cast<uint4*>(d + ps) =
        make_uint4(pack_bf16(m[0], m[1]), pack_bf16(m[2], m[3]), pack_bf16(m[4], m[5]), pack_bf16(m[6], m[7]));
    *reinterpret_cast<uint4*>(d + 2 * ps) =
        make_uint4(pack_bf16(l[0], l[1]), pack_bf16(l[2], l[3]), pack_bf16(l[4], l[5]), pack_bf16(l[6], l[7]));
  }
}

// ------------------------------------------------------------------------------------------ geometry / launch
static int round_up(int x, int m) { return (x + m - 1) / m * m; }

// bwd: X0, G1 and scratch images; fwd: X0 and scratch.  The largest F (frames per item) that fits 227 KB wins.  The
// product count `terms` does not change the geometry.
static bool unit_geom(int Cin, int Cout, int P, int K, int nb, bool bwd, int terms, UnitGeom& g) {
  if (K < 1 || K > 40 || K * ((K + 1) / 2) > 2 * UT_NT || Cin < 1 || Cin > 64 || Cout < 1 || Cout > 64 || nb < 1 || nb > DSTD_MAX_BRANCH) return false;
  g.KQ = round_up(K, 8);
  g.terms = terms;
  g.KW = round_up(K, 16);
  g.CinK = round_up(Cin, 16);
  g.CoutK = round_up(Cout, 16);
  g.CinN = round_up(Cin, 8);
  // xmu images: bwd reads them K-major (rows v = N <= KQ, K = w < KW), fwd MN-major (K = rows v < KW, N = w <= KQ)
  g.xr = bwd ? g.KQ : g.KW;
  g.xq = bwd ? g.KW : g.KQ;
  g.xsbo_b = img16_sbo_b(g.xq);
  g.xplane_b = img16_bytes(g.xr, g.xq);
  for (int F = 128 / g.KQ; F >= 1; --F) {
    if (F > P && F > 1) continue;
    g.F = F;
    g.NPOS = F * g.KQ;
    g.NG = g.NPOS / 8;
    g.Q = round_up((F - 1) * g.KQ + g.KW, 16);
    g.QG = g.Q / 8;
    if (g.NG > 16 || g.QG > 16) continue;          // image builder: four columns per lane
    g.sbo_b = img16_sbo_b(g.Q);
    g.plane_b = img16_bytes(64, g.Q);
    g.N16 = round_up(g.NPOS, 16);
    const int cols = bwd ? 2 * g.N16 + 2 * g.NPOS + nb * g.CinN : g.N16 + g.NPOS;
    if (cols > 512) continue;
    g.tmem_cols = cols <= 32 ? 32 : cols <= 64 ? 64 : cols <= 128 ? 128 : cols <= 256 ? 256 : 512;
    int o = 0;
    auto take = [&](int bytes) { int r = o; o += (bytes + 127) & ~127; return r; };
    g.o_x0 = take(3 * g.plane_b);
    g.o_g1 = bwd ? take(3 * g.plane_b) : 0;
    g.o_s = take(3 * g.plane_b);
    g.o_w = take(nb * 3 * UT_WP_B);                // MN-major windows of the scratch image may run on into the weights
    g.o_xmu = take(nb * F * 3 * g.xplane_b);
    g.o_aeff = take(nb * K * K * 4);
    g.o_bias = take(nb * 64 * 4);
    g.o_etab = take(K * ((K + 1) / 2) * 4);
    g.o_gst = take(K * K * 2);
    g.o_pst = take(F * K * 2);
    g.o_pout = take(F * K * 4);
    g.o_pskip = take(F * K * 4);
    g.o_bar = take(64);
    g.smem = o + 2048;                             // slack: M = 64 operand windows of the last image may read past it
    // fp32 staging tiles alias whole images
    if ((size_t)64 * (g.NPOS + 4) * 4 > (size_t)3 * g.plane_b) continue;
    if (bwd && (size_t)F * g.KQ * g.KQ * 4 > (size_t)3 * g.plane_b) continue;
    if (g.smem <= MAX_DYN_SMEM - 1024) return true;
  }
  return false;
}

// Opt-in (DSTD_UNIT_TC=1): measured on B200 at the H3.6M encoder shape, batch 256, the all-tcgen05 kernels are at parity
// with the mma.sync / tcgen05-mix forward (unit forward 0.358 vs 0.353 ms) and 20 % behind the mma.sync backward
// (0.82 vs 0.68 ms; 8.3 k vs 9.6 k samples/s for the whole step): the six-term bf16 chains re-read every operand from
// shared memory per instruction and M = 64 accumulators run at half rate (DESIGN.md section 3).
// DSTD_PRECISION (secondary, stated-tolerance modes; the default "fp32" is the parity path): "bf16x2" keeps the products
// hh + hm + mh (relative error ~2^-15), "bf16" only hh (plain bf16 operands, fp32 accumulate, ~2^-8).  Both run on these
// kernels (there is no other reduced-precision implementation), so they imply DSTD_UNIT_TC=1 (read_switches, api.cu).
bool unit_tc_supported(int Cin, int Cout, int P, int K, int nb) {
  UnitGeom g;
  return unit_geom(Cin, Cout, P, K, nb, true, 6, g) && unit_geom(Cin, Cout, P, K, nb, false, 6, g);
}

size_t unit_tc_ws_bytes(int nb) { return (size_t)nb * 3 * UT_WP_B + 256; }

int unit_bwd_tc_ctas(int N, int Cin, int Cout, int P, int K, int nb) {
  UnitGeom g;
  if (!unit_geom(Cin, Cout, P, K, nb, true, 6, g)) return 0;
  const long long items = (long long)N * cdiv(P, g.F);
  const int sms = num_sms();
  return (int)(items < sms ? items : sms);
}

static int pack_w16(const PackParams& pk, unsigned char* ws, int** err_flag, cudaStream_t st) {
  *err_flag = device_error_word();
  pack_w16_kernel<<<cdiv(pk.nb * 512, 256), 256, 0, st>>>(pk, ws);
  count_launch();
  return check_launch("pack_w16");
}

int launch_unit_fwd_tc(const AggMixParams& a, const PackParams& pk, void* ws, int terms, cudaStream_t st) {
  UnitGeom g;
  DSTD_REQUIRE(unit_geom(a.Cin, a.Cout, a.P, a.K, a.nb, false, terms, g), DSTD_ERR_UNSUPPORTED, "unit_fwd_tc: shape outside limits");
  int* err_flag;
  int rc = pack_w16(pk, (unsigned char*)ws, &err_flag, st);
  if (rc) return rc;
  UnitFwdParams q;
  q.N = a.N; q.Cin = a.Cin; q.Cout = a.Cout; q.P = a.P; q.K = a.K; q.nb = a.nb; q.adj_t = a.adj_t;
  q.x = a.x; q.out = a.out; q.skip = a.skip; q.pd = a.pd; q.alpha = a.alpha;
  for (int b = 0; b < DSTD_MAX_BRANCH; ++b) {
    q.adj[b] = a.adj[b]; q.adj_w[b] = a.adj_w[b]; q.adj_r[b] = a.adj_r[b]; q.b_f[b] = pk.b_f[b];
  }
  q.wimg = (const unsigned char*)ws;
  q.err_flag = err_flag;
  const long long items = (long long)a.N * cdiv(a.P, g.F);
  const int sms = num_sms();
  const int ctas = (int)(items < sms ? items : sms);
  ensure_max_smem((const void*)unit_fwd_tc_kernel);
  unit_fwd_tc_kernel<<<ctas, UT_NT, g.smem, st>>>(q, g);
  count_launch();
  return check_launch("unit_fwd_tc");
}

int launch_unit_bwd_tc(const AggMixBwdParams& a, const PackParams& pk, void* ws, int terms, cudaStream_t st) {
  UnitGeom g;
  DSTD_REQUIRE(unit_geom(a.Cin, a.Cout, a.P, a.K, a.nb, true, terms, g), DSTD_ERR_UNSUPPORTED, "unit_bwd_tc: shape outside limits");
  int* err_flag;
  int rc = pack_w16(pk, (unsigned char*)ws, &err_flag, st);
  if (rc) return rc;
  UnitBwdParams q;
  q.N = a.N; q.Cin = a.Cin; q.Cout = a.Cout; q.P = a.P; q.K = a.K; q.nb = a.nb; q.adj_t = a.adj_t;
  q.x = a.x; q.gout = a.gout; q.gx = a.gx; q.pd = a.pd; q.alpha = a.alpha;
  for (int b = 0; b < DSTD_MAX_BRANCH; ++b) {
    q.adj[b] = a.adj[b]; q.adj_w[b] = a.adj_w[b]; q.adj_r[b] = a.adj_r[b]; q.b_f[b] = a.b_f[b];
  }
  q.wimg = (const unsigned char*)ws;
  q.gxm = a.gxm; q.part_w = a.part_w; q.part_b = a.part_b;
  q.err_flag = err_flag;
  const int ctas = unit_bwd_tc_ctas(a.N, a.Cin, a.Cout, a.P, a.K, a.nb);
  ensure_max_smem((const void*)unit_bwd_tc_kernel);
  unit_bwd_tc_kernel<<<ctas, UT_NT, g.smem, st>>>(q, g);
  count_launch();
  return check_launch("unit_bwd_tc");
}

}  // namespace dstd
