// Internal launcher interface between api.cu and the kernel translation units.
#pragma once
#include <initializer_list>

#include "common.cuh"

namespace dstd {

// ------------------------------------------------------------------ gemm.cu
struct BgemmParams {
  int M, Kd;           // output rows, reduction length
  long long G;         // columns = N*P*K
  int P, K;
  const float* w;      // weight element (c, i) at w[c*wsc + i*wsi]
  long long wsc, wsi;
  const float* bias;   // [M] or null
  View4 in;            // row c at in.p + c*in.sc
  int ones_row;        // row index that reads as 1.0 (or -1)
  View4 out;
  View4 add;           // optional (p == null)
  int m0, m1;          // filled by the launcher
  void* tc_ws = nullptr;   // optional: bgemm_tc_ws_bytes(M, Kd) of workspace enables the tcgen05 kernel (bgemm_tc.cu)
};
int launch_bgemm(BgemmParams q, cudaStream_t st);
bool bgemm_tc_supported(int M, int Kd);
size_t bgemm_tc_ws_bytes(int M, int Kd);
int launch_bgemm_tc(const BgemmParams& q, void* ws, cudaStream_t st);

struct WgradParams {
  int M, Cd;
  long long G;
  int P, K;
  View4 a;             // [*, M, P, K]
  View4 b;             // [*, Cd, P, K]
  int b_ones_row;      // row of B that reads as 1.0 (or -1)
  float* partial;      // [S][M][Cd]
  int S;               // filled by the launcher
  long long cols_per_split;
};
int wgrad_splits(long long G);
int launch_wgrad(WgradParams& q, bool tc, cudaStream_t st);   // fills q.S (partials written); tc: tcgen05 allowed
bool wgrad_tc_supported(int M, int Cd);
int launch_wgrad_tc(WgradParams& q, cudaStream_t st);   // tcgen05 version (bgemm_tc.cu), same contract

struct MprojBwdParams {
  int Cin, J, P, K;    // J = 4 * nb rows of [conv_m1; conv_m2] per branch
  long long G;         // columns = N*P*K
  View4 x;             // [N,Cin,P,K]
  View4 gx;            // [N,Cin,P,K] read-modify-write
  View4 gx_add;        // optional: added into gx in the same pass
  const float* gm;     // dense [N,J,P,K]
  const float* wm;     // [J][Cin+1]
  float* partial;      // [ctas][J][Cin+1]
};
struct MprojFwdParams {
  int Cin, J, P, K;
  long long G;
  View4 x;             // [N,Cin,P,K]
  const float* wm;     // [J][Cin+1]  (bias in column Cin)
  float* m;            // dense [N,J,P,K]
};
int launch_mproj_fwd(const MprojFwdParams& q, cudaStream_t st);
bool mproj_bwd_supported(int Cin, int J);
int mproj_bwd_ctas(long long G);
int launch_mproj_bwd(const MprojBwdParams& q, cudaStream_t st);

struct ReduceSeg {
  const float* src;    // partial k, element (r, c) at src[k*sstride + r*src_ld + c]
  int S;
  long long sstride;
  int rows, cols, src_ld;
  float* dst;          // dense [rows][dst_ld]; may be null
  int dst_ld;
  const float* mul;    // optional: dst2 = value * mul (same indexing as dst)
  float* dst2;
  float scale;
};
struct ReduceParams {
  ReduceSeg seg[24];
  int nseg;
};
int launch_reduce(const ReduceParams& q, cudaStream_t st);

// ------------------------------------------------------------------ dynadj.cu
struct DynAdjFwdParams {
  int N, P, K, nb;
  const float* m;      // [N,nb,4,P,K]
  const float* w_rm[DSTD_MAX_BRANCH];
  const float* b_rm[DSTD_MAX_BRANCH];
  float* pd;           // [N,nb,P,K,K]
};
int launch_dynadj_fwd(const DynAdjFwdParams& q, cudaStream_t st);

struct DynAdjBwdParams {
  int N, P, K, nb;
  const float* m;      // [N,nb,4,P,K]
  const float* pd;     // [N,nb,P,K,K]
  const float* gxm;    // [N,nb,P,K,K]
  const float* w_rm[DSTD_MAX_BRANCH];
  const float* b_rm[DSTD_MAX_BRANCH];
  const float* alpha;  // device scalar or null (=1)
  float* gm;           // [N,nb,4,P,K]
  int S;               // number of batch splits
  float* part_wrm;     // [S][nb][P][2P+1]   (already scaled by alpha)
  float* part_adj;     // [S][nb][K*K]
  float* part_alpha;   // [S][nb]
};
int dynadj_bwd_splits(int N, int nb);
int launch_dynadj_bwd(const DynAdjBwdParams& q, cudaStream_t st);
bool dynadj_supported(int P, int K);

// ------------------------------------------------------------------ aggregate.cu
struct AggParams {
  int N, Cin, P, K, nb, adj_t;
  View4 x;             // [N,Cin,P,K]
  const float* pd;     // [N,nb,P,K,K]
  const float* alpha;
  const float* adj[DSTD_MAX_BRANCH];
  const float* adj_w[DSTD_MAX_BRANCH];
  const float* adj_r[DSTD_MAX_BRANCH];
  float* xa;           // fwd out: [N,nb,Cin+1,P,K]
  // backward only
  const float* gxa;    // [N,nb,Cin+1,P,K]
  View4 gx;            // [N,Cin,P,K] written
  float* gxm;          // [N,nb,P,K,K] written
};
int launch_aggregate_fwd(const AggParams& q, cudaStream_t st);
int launch_aggregate_bwd(const AggParams& q, cudaStream_t st);
bool aggregate_supported(int Cin, int P, int K);

// ------------------------------------------------------------------ generic.cu (P or K > 40: the stress configuration)
bool generic_supported(int P, int K);
int launch_dynadj_fwd_gen(const DynAdjFwdParams& q, cudaStream_t st);
int dynadj_gen_tiles(int K);                                               // v tiles per (sample, branch)
size_t dynadj_bwd_gen_ws_floats(int N, int nb, int P, int K);              // gm2 partials
int launch_dynadj_bwd_gen(const DynAdjBwdParams& q, float* gm2_part, cudaStream_t st);   // q.S == N * tiles slots; part_adj: N slots
int launch_aggregate_fwd_gen(const AggParams& q, bool mma, cudaStream_t st);   // mma: mma.sync kernel for K >= 48
int launch_aggregate_bwd_gen(const AggParams& q, cudaStream_t st);

// ------------------------------------------------------------------ aggmix.cu
struct AggMixParams {
  int N, Cin, Cout, P, K, nb, adj_t;
  int PCH, CoutP;      // filled by the launcher
  View4 x;             // [N,Cin,P,K]
  View4 out;           // [N,Cout,P,K]
  View4 skip;          // optional
  const float* pd;     // [N,nb,P,K,K]
  const float* alpha;
  const float* adj[DSTD_MAX_BRANCH];
  const float* adj_w[DSTD_MAX_BRANCH];
  const float* adj_r[DSTD_MAX_BRANCH];
  const float* wcatT;  // [nb*(Cin+1)][CoutP] from the pack kernel
  const float* wtc;    // tensor-core path: UMMA weight image (filled by launch_aggmix_fwd_tc)
  float* xa;           // optional [N,nb,Cin+1,P,K]
};
int launch_aggmix_fwd(AggMixParams q, cudaStream_t st);
bool aggmix_supported(int Cin, int Cout, int P, int K, int nb);
// tcgen05 variant (aggmix_tc.cu)
struct PackParams;
bool aggmix_tc_supported(int Cin, int Cout, int P, int K, int nb);
size_t aggmix_tc_ws_floats(int Cin, int Cout, int P, int K, int nb);
int launch_aggmix_fwd_tc(AggMixParams q, const PackParams& pk, float* wtc_ws, cudaStream_t st);

// ------------------------------------------------------------------ aggmix_bwd.cu
struct AggMixBwdParams {
  int N, Cin, Cout, P, K, nb, adj_t;
  int PCH, LD, CinP, WS;   // filled by the launcher
  View4 x;             // [N,Cin,P,K]
  View4 gout;          // [N,Cout,P,K]
  View4 gx;            // [N,Cin,P,K] written (aggregation part of the input gradient)
  const float* pd;     // [N,nb,P,K,K]
  const float* alpha;
  const float* adj[DSTD_MAX_BRANCH];
  const float* adj_w[DSTD_MAX_BRANCH];
  const float* adj_r[DSTD_MAX_BRANCH];
  const float* w_f[DSTD_MAX_BRANCH];   // [Cout][Cin]
  const float* b_f[DSTD_MAX_BRANCH];   // [Cout]
  float* gxm;          // [N,nb,P,K,K] written
  float* part_w;       // [ctas][nb][Cout][Cin]
  float* part_b;       // [ctas][nb][Cout]
};
int launch_aggmix_bwd(AggMixBwdParams q, cudaStream_t st);
bool aggmix_bwd_supported(int Cin, int Cout, int P, int K, int nb);
int aggmix_bwd_ctas(int N, int P, int K, int Cin, int Cout, int nb);

// ------------------------------------------------------------------ unit_tc.cu (all contractions on tcgen05, bf16x3 operands)
bool unit_tc_supported(int Cin, int Cout, int P, int K, int nb);
size_t unit_tc_ws_bytes(int nb);
int unit_bwd_tc_ctas(int N, int Cin, int Cout, int P, int K, int nb);
// terms: split products per k-step (Switches::unit_terms)
int launch_unit_fwd_tc(const AggMixParams& q, const PackParams& pk, void* ws, int terms, cudaStream_t st);
int launch_unit_bwd_tc(const AggMixBwdParams& q, const PackParams& pk, void* ws, int terms, cudaStream_t st);

// ------------------------------------------------------------------ misc.cu
struct PackParams {
  int Cin, Cout, nb;
  const float* w_f[DSTD_MAX_BRANCH];
  const float* b_f[DSTD_MAX_BRANCH];
  const float* w_m1[DSTD_MAX_BRANCH];
  const float* b_m1[DSTD_MAX_BRANCH];
  const float* w_m2[DSTD_MAX_BRANCH];
  const float* b_m2[DSTD_MAX_BRANCH];
  float* wcat;         // [Cout][nb*(Cin+1)]
  float* wm;           // [4*nb][Cin+1]
  float* wcatT;        // optional [nb*(Cin+1)][CoutP], CoutP = Cout rounded up to 8, zero padded
};
int launch_pack(const PackParams& q, cudaStream_t st);

}  // namespace dstd
