// C ABI of libdstd_b200 (include/dstd_b200.h): argument validation, workspace carving and the kernel schedule of
// the DSTD-GC unit (model/dstdgcn.py:80-94 as called from DSTDGCB.forward :145-150 / :157-161) and the 1x1 channel mix.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <map>
#include <mutex>
#include <set>
#include <utility>

#include "kernels.cuh"

namespace dstd {

static thread_local char g_err[512] = "";
static std::atomic<int> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return DSTD_ERR_CUDA;
  }
  return DSTD_OK;
}

// the 227 KB per-CTA limit covers static + dynamic shared memory
static int max_dyn_for(const void* kernel) {
  cudaFuncAttributes fa;
  if (cudaFuncGetAttributes(&fa, kernel) != cudaSuccess) return MAX_DYN_SMEM;
  return MAX_DYN_SMEM - (int)fa.sharedSizeBytes;
}

static int current_device() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess) { cudaGetLastError(); return -1; }
  return d;
}

int num_sms() {
  static std::mutex mu;
  static std::map<int, int> cache;
  const int d = current_device();
  if (d < 0) return 148;
  std::lock_guard<std::mutex> lk(mu);
  auto it = cache.find(d);
  if (it != cache.end()) return it->second;
  int n = 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, d) != cudaSuccess || n < 1) { cudaGetLastError(); n = 148; }
  cache[d] = n;
  return n;
}

// cudaFuncSetAttribute applies to the current device only: remember (device, kernel) pairs
void ensure_max_smem(const void* kernel) {
  static std::mutex mu;
  static std::set<std::pair<int, const void*>> done;
  const int d = current_device();
  std::lock_guard<std::mutex> lk(mu);
  if (done.count({d, kernel})) return;
  cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn_for(kernel));
  done.insert({d, kernel});
}

// Streaming kernels with modest dynamic shared memory: without a preference the driver picks the smallest carve-out
// that fits ONE CTA (measured: bn_bwd_apply ran 1 CTA/SM), so ask for the largest shared-memory partition once.
void prefer_smem_carveout(const void* kernel, bool need_max) {
  static std::mutex mu;
  static std::set<std::pair<int, const void*>> done;
  const int d = current_device();
  std::lock_guard<std::mutex> lk(mu);
  if (done.count({d, kernel})) return;
  if (need_max) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn_for(kernel));
  cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  done.insert({d, kernel});
}

// ---- device-side error word (host-mapped, so that reading it never synchronises)
static int* g_err_host = nullptr;
static int* g_err_dev = nullptr;
static std::mutex g_err_mu;

int* device_error_word() {
  std::lock_guard<std::mutex> lk(g_err_mu);
  if (g_err_dev) return g_err_dev;
  int* h = nullptr;
  if (cudaHostAlloc((void**)&h, sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError();     // e.g. called for the first time under stream capture: the kernel then runs without the word
    return nullptr;
  }
  *h = 0;
  int* d = nullptr;
  if (cudaHostGetDevicePointer((void**)&d, h, 0) != cudaSuccess) {
    cudaGetLastError();
    cudaFreeHost(h);
    return nullptr;
  }
  g_err_host = h;
  g_err_dev = d;
  return g_err_dev;
}

int poll_device_error(const char* fn) {
  const int* h = g_err_host;
  if (h && *(volatile const int*)h != 0) {
    set_error("%s: an earlier kernel of this library reported a device-side failure (code %d: tensor-core pipeline "
              "timeout); its outputs are invalid.  dstd_device_error(1) clears the condition", fn, *(volatile const int*)h);
    return DSTD_ERR_CUDA;
  }
  return DSTD_OK;
}

__global__ void raise_device_error_kernel(int* word, int code) {
  *(volatile int*)word = code;
  __threadfence_system();
}

Switches read_switches() {
  auto value = [](const char* name) -> const char* {   // unset or empty: the default
    const char* e = getenv(name);
    return e && e[0] ? e : nullptr;
  };
  auto flag = [&](const char* name, bool dflt) {
    const char* e = value(name);
    return e ? strcmp(e, "0") != 0 : dflt;
  };
  Switches sw;
  const char* p = value("DSTD_PRECISION");
  sw.unit_terms = (p && strncmp(p, "bf16", 4) == 0) ? (strncmp(p + 4, "x2", 2) == 0 ? 3 : 1) : 6;
  sw.unit_tc = flag("DSTD_UNIT_TC", false) || sw.unit_terms != 6;
  sw.aggmix_tc = !flag("DSTD_DISABLE_TC", false);
  sw.bgemm_tc = flag("DSTD_BGEMM_TC", true);
  sw.agg_gen_mma = flag("DSTD_AGG_GEN_MMA", false);
  sw.bn_fast = flag("DSTD_BN_FAST", true);
  const char* spc = value("DSTD_BN_SAMPLES_PER_CTA");
  sw.bn_samples_per_cta = spc ? std::max(1, atoi(spc)) : 32;
  return sw;
}

// ---------------------------------------------------------------------------------------------- DSTD-GC plan
// shapes beyond the specialised tiles (P or K > 40) run the shape-generic kernels of generic.cu
static bool use_generic(int Cin, int P, int K) { return !(dynadj_supported(P, K) && aggregate_supported(Cin, P, K)); }

enum class GcFwd { unit_tc, aggmix_tc, aggmix, unfused };   // unit_tc.cu / aggmix_tc.cu / aggmix.cu / aggregate + bgemm
enum class GcBwd { unit_tc, aggmix, unfused };              // unit_tc.cu / aggmix_bwd.cu / bgemm + wgrad + aggregate

// Every kernel-path and workspace decision of one DSTD-GC call: the forward, the backward, the workspace queries and
// dstd_gc_needs_xa all read it, so that they cannot disagree.
struct GcPlan {
  int N, Cin, Cout, P, K, nb, C1;
  long long G;        // positions N * P * K
  bool generic;
  GcFwd fwd;
  GcBwd bwd;
  bool needs_xa;      // the backward reads the xa the forward keeps (the unfused path on either side)
  int terms;          // split products per k-step of the unit kernels
  int S1, S2;         // splits of the channel weight gradient / of the dynamic-adjacency backward
  size_t slots;       // per-CTA partial slots of the persistent kernels (two per SM)
};

// have_xa: the caller passes an xa buffer to the forward.  The unit and tcgen05 forwards do not write it, so the
// CUDA-core fused forward runs instead.
static GcPlan gc_plan(int N, int Cin, int Cout, int P, int K, int nb, const Switches& sw, bool have_xa = false) {
  GcPlan pl;
  pl.N = N; pl.Cin = Cin; pl.Cout = Cout; pl.P = P; pl.K = K; pl.nb = nb; pl.C1 = Cin + 1;
  pl.G = (long long)N * P * K;
  pl.generic = use_generic(Cin, P, K);
  const bool unit = !pl.generic && sw.unit_tc && unit_tc_supported(Cin, Cout, P, K, nb);
  const bool aggmix = !pl.generic && aggmix_supported(Cin, Cout, P, K, nb);
  const bool aggmix_bwd = !pl.generic && aggmix_bwd_supported(Cin, Cout, P, K, nb);
  if (unit && !have_xa) pl.fwd = GcFwd::unit_tc;
  else if (aggmix && !have_xa && sw.aggmix_tc && aggmix_tc_supported(Cin, Cout, P, K, nb)) pl.fwd = GcFwd::aggmix_tc;
  else pl.fwd = aggmix ? GcFwd::aggmix : GcFwd::unfused;
  pl.bwd = unit ? GcBwd::unit_tc : aggmix_bwd ? GcBwd::aggmix : GcBwd::unfused;
  pl.needs_xa = !(unit || aggmix) || pl.bwd == GcBwd::unfused;
  pl.terms = sw.unit_terms;
  pl.S1 = wgrad_splits(pl.G);
  pl.S2 = pl.generic ? N * dynadj_gen_tiles(K) : dynadj_bwd_splits(N, nb);
  pl.slots = (size_t)2 * num_sms();
  return pl;
}

// Workspace carving: over the caller's workspace it hands out the buffers, over a null base it sizes them (gc_*_ws).
struct GcFwdWs {
  float *wcat, *wm, *wcatT, *wtc;   // packed weights: [Cout][nb*C1], [4*nb][C1], transposed for aggmix, aggmix_tc image
  void *wunit, *wbt;                // unit_tc weight images, bgemm_tc weight images
};
static GcFwdWs carve_fwd(const GcPlan& pl, Arena& ar) {
  GcFwdWs w;
  w.wcat = ar.take<float>((size_t)pl.Cout * pl.nb * pl.C1);
  w.wm = ar.take<float>((size_t)4 * pl.nb * pl.C1);
  w.wcatT = ar.take<float>((size_t)pl.nb * pl.C1 * ((pl.Cout + 7) / 8 * 8));
  w.wtc = ar.take<float>(aggmix_tc_ws_floats(pl.Cin, pl.Cout, pl.P, pl.K, pl.nb));
  w.wunit = ar.take<char>(unit_tc_ws_bytes(pl.nb));
  w.wbt = ar.take<char>(bgemm_tc_ws_bytes(pl.Cout, pl.nb * pl.C1));
  return w;
}
static size_t gc_fwd_ws(const GcPlan& pl) {
  Arena ar(nullptr, 0);
  carve_fwd(pl, ar);
  return ar.need();
}

struct GcBwdWs {
  float *wcat, *wm;                          // packed weights
  float *gxa, *gxm, *gm;                     // intermediates (gxa: unfused path only)
  float *p_wcat, *p_wm, *p_wrm, *p_adj, *p_alpha, *p_wf, *p_bf;   // split / per-CTA partials of the parameter gradients
  void *wunit, *wbt;
  float* gm2_part;                           // generic dynamic-adjacency backward
};
static GcBwdWs carve_bwd(const GcPlan& pl, Arena& ar) {
  const size_t G = pl.G, nb = pl.nb, C1 = pl.C1, P = pl.P, K = pl.K, S1 = pl.S1, S2 = pl.S2, ps = pl.slots;
  const bool unf = pl.bwd == GcBwd::unfused;
  GcBwdWs w;
  w.wcat = ar.take<float>(pl.Cout * nb * C1);
  w.wm = ar.take<float>(4 * nb * C1);
  w.gxa = ar.take<float>(unf ? G * nb * C1 : 0);
  w.gxm = ar.take<float>(G * nb * K);
  w.gm = ar.take<float>(G * nb * 4);
  w.p_wcat = ar.take<float>(unf ? S1 * pl.Cout * nb * C1 : 0);
  w.p_wm = ar.take<float>((S1 > ps ? S1 : ps) * 4 * nb * C1);
  w.p_wrm = ar.take<float>(S2 * nb * P * (2 * P + 1));
  w.p_adj = ar.take<float>(S2 * nb * K * K);
  w.p_alpha = ar.take<float>(S2 * nb);
  w.p_wf = ar.take<float>(ps * nb * pl.Cout * pl.Cin);
  w.p_bf = ar.take<float>(ps * nb * pl.Cout);
  w.wunit = ar.take<char>(unit_tc_ws_bytes(pl.nb));
  w.wbt = ar.take<char>(bgemm_tc_ws_bytes(pl.nb * pl.C1, pl.Cout));
  w.gm2_part = ar.take<float>(pl.generic ? dynadj_bwd_gen_ws_floats(pl.N, pl.nb, pl.P, pl.K) : 0);
  return w;
}
static size_t gc_bwd_ws(const GcPlan& pl) {
  Arena ar(nullptr, 0);
  carve_bwd(pl, ar);
  return ar.need();
}

static int gc_check_common(int N, int Cin, int Cout, int P, int K, int nb, const dstd_branch* br, const char* fn) {
  DSTD_REQUIRE(N > 0 && Cin > 0 && Cout > 0 && P > 0 && K > 0, DSTD_ERR_BAD_ARG, "%s: non-positive dimension", fn);
  DSTD_REQUIRE(nb >= 1 && nb <= DSTD_MAX_BRANCH, DSTD_ERR_BAD_ARG, "%s: nb=%d outside [1,%d]", fn, nb, DSTD_MAX_BRANCH);
  for (int b = 0; b < nb; ++b)
    DSTD_REQUIRE(br[b].w_m1 && br[b].b_m1 && br[b].w_m2 && br[b].b_m2 && br[b].w_rm && br[b].b_rm && br[b].w_f &&
                     br[b].b_f && br[b].adj,
                 DSTD_ERR_BAD_ARG, "%s: branch %d has a null weight", fn, b);
  DSTD_REQUIRE(!use_generic(Cin, P, K) || generic_supported(P, K), DSTD_ERR_UNSUPPORTED,
               "%s: unit shape P=%d K=%d outside the compiled tile limits (P<=128, K<=128)", fn, P, K);
  return DSTD_OK;
}

// Per-branch pointers of the kernel parameter blocks; the slots beyond nb repeat branch 0.
template <typename Q>
static void fill_adj(Q& q, int nb, const dstd_branch* br) {
  for (int b = 0; b < DSTD_MAX_BRANCH; ++b) {
    const dstd_branch& s = br[b < nb ? b : 0];
    q.adj[b] = s.adj; q.adj_w[b] = s.adj_w; q.adj_r[b] = s.adj_r;
  }
}
template <typename Q>
static void fill_rm(Q& q, int nb, const dstd_branch* br) {
  for (int b = 0; b < DSTD_MAX_BRANCH; ++b) {
    q.w_rm[b] = br[b < nb ? b : 0].w_rm;
    q.b_rm[b] = br[b < nb ? b : 0].b_rm;
  }
}

static void fill_pack(PackParams& pk, int Cin, int Cout, int nb, const dstd_branch* br, float* wcat, float* wm,
                      float* wcatT = nullptr) {
  pk.wcatT = wcatT;
  pk.Cin = Cin; pk.Cout = Cout; pk.nb = nb;
  for (int b = 0; b < DSTD_MAX_BRANCH; ++b) {
    const dstd_branch& s = br[b < nb ? b : 0];
    pk.w_f[b] = s.w_f; pk.b_f[b] = s.b_f;
    pk.w_m1[b] = s.w_m1; pk.b_m1[b] = s.b_m1;
    pk.w_m2[b] = s.w_m2; pk.b_m2[b] = s.b_m2;
  }
  pk.wcat = wcat; pk.wm = wm;
}

static void fill_agg(AggParams& ag, int N, int Cin, int P, int K, int nb, int flags, const dstd_view& x,
                     const float* pd, const float* alpha, const dstd_branch* br) {
  ag.N = N; ag.Cin = Cin; ag.P = P; ag.K = K; ag.nb = nb;
  ag.adj_t = (flags & DSTD_FLAG_ADJ_T) ? 1 : 0;
  ag.x = mk(x);
  ag.pd = pd;
  ag.alpha = alpha;
  fill_adj(ag, nb, br);
  ag.xa = nullptr; ag.gxa = nullptr; ag.gxm = nullptr;
  ag.gx = View4{nullptr, 0, 0, 0, 0};
}

// one reduction of split partials into a parameter gradient (skipped when nothing is requested)
static void add_seg(ReduceParams& rp, const float* src, int S, long long sstride, int rows, int cols, int src_ld,
                    float* dst, int dst_ld, const float* mul = nullptr, float* dst2 = nullptr) {
  if (!dst && !dst2) return;
  ReduceSeg& s = rp.seg[rp.nseg++];
  s.src = src; s.S = S; s.sstride = sstride; s.rows = rows; s.cols = cols; s.src_ld = src_ld;
  s.dst = dst; s.dst_ld = dst_ld; s.mul = mul; s.dst2 = dst2; s.scale = 1.0f;
}

}  // namespace dstd

using namespace dstd;

extern "C" const char* dstd_last_error(void) { return g_err; }
extern "C" const char* dstd_version(void) { return "dstd_b200 0.1 sm_100a"; }
extern "C" int dstd_kernel_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
extern "C" int dstd_device_error(int clear) {
  device_error_word();
  int v = 0;
  if (g_err_host) {
    v = *(volatile int*)g_err_host;
    if (clear) *(volatile int*)g_err_host = 0;
  }
  return v;
}
extern "C" int dstd_debug_raise_device_error(int code, dstd_stream_t stream) {
  int* w = device_error_word();
  DSTD_REQUIRE(w, DSTD_ERR_CUDA, "debug_raise_device_error: the error word is unavailable");
  raise_device_error_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(w, code);
  count_launch();
  return check_launch("raise_device_error");
}

extern "C" int dstd_gc_needs_xa(int Cin, int Cout, int P, int K, int nb) {
  return gc_plan(1, Cin, Cout, P, K, nb, read_switches()).needs_xa ? 1 : 0;
}
extern "C" size_t dstd_gc_fwd_workspace_bytes(int N, int Cin, int Cout, int P, int K, int nb) {
  return gc_fwd_ws(gc_plan(N, Cin, Cout, P, K, nb, read_switches()));
}
extern "C" size_t dstd_gc_bwd_workspace_bytes(int N, int Cin, int Cout, int P, int K, int nb) {
  return gc_bwd_ws(gc_plan(N, Cin, Cout, P, K, nb, read_switches()));
}

// ---------------------------------------------------------------------------------------------- DSTD-GC forward
extern "C" int dstd_gc_forward(const dstd_gc_fwd_args* a, dstd_stream_t stream) {
  DSTD_REQUIRE(a, DSTD_ERR_BAD_ARG, "gc_forward: null args");
  int rc = poll_device_error("gc_forward");
  if (rc) return rc;
  rc = gc_check_common(a->N, a->Cin, a->Cout, a->P, a->K, a->nb, a->br, "gc_forward");
  if (rc) return rc;
  DSTD_REQUIRE(a->x.ptr && a->out.ptr && a->m && a->pd, DSTD_ERR_BAD_ARG, "gc_forward: null tensor");
  const Switches sw = read_switches();
  const GcPlan pl = gc_plan(a->N, a->Cin, a->Cout, a->P, a->K, a->nb, sw, a->xa != nullptr);
  const size_t need = gc_fwd_ws(pl);
  DSTD_REQUIRE(a->ws && a->ws_bytes >= need, DSTD_ERR_WORKSPACE, "gc_forward: workspace too small (%zu < %zu)",
               a->ws_bytes, need);
  cudaStream_t st = (cudaStream_t)stream;
  const int N = a->N, Cin = a->Cin, Cout = a->Cout, P = a->P, K = a->K, nb = a->nb, C1 = pl.C1;
  Arena ar(a->ws, a->ws_bytes);
  const GcFwdWs w = carve_fwd(pl, ar);
  const bool fused = pl.fwd != GcFwd::unfused;

  PackParams pk;
  fill_pack(pk, Cin, Cout, nb, a->br, w.wcat, w.wm, fused ? w.wcatT : nullptr);
  if ((rc = launch_pack(pk, st))) return rc;

  // 1. m = [conv_m1; conv_m2] x + b        (all branches in one streaming pass over x)
  {
    MprojFwdParams mp;
    mp.Cin = Cin; mp.J = 4 * nb; mp.P = P; mp.K = K; mp.G = pl.G;
    mp.x = mk(a->x); mp.wm = w.wm; mp.m = a->m;
    if ((rc = launch_mproj_fwd(mp, st))) return rc;
  }

  // 2. pd = conv_rm(tanh(m1 - m2))         (pairwise tensor stays on chip)
  DynAdjFwdParams dp;
  dp.N = N; dp.P = P; dp.K = K; dp.nb = nb; dp.m = a->m; dp.pd = a->pd;
  fill_rm(dp, nb, a->br);
  if ((rc = pl.generic ? launch_dynadj_fwd_gen(dp, st) : launch_dynadj_fwd(dp, st))) return rc;

  // 3+4 fused: out = wcat ([x;1] (alpha pd + A)) (+ skip); the aggregated tile stays in shared memory
  if (fused) {
    AggMixParams am;
    am.N = N; am.Cin = Cin; am.Cout = Cout; am.P = P; am.K = K; am.nb = nb;
    am.adj_t = (a->flags & DSTD_FLAG_ADJ_T) ? 1 : 0;
    am.PCH = 0; am.CoutP = 0;
    am.x = mk(a->x); am.out = mk(a->out); am.skip = mk(a->skip);
    am.pd = a->pd; am.alpha = a->alpha;
    fill_adj(am, nb, a->br);
    am.wcatT = w.wcatT;
    am.wtc = nullptr;
    am.xa = a->xa;
    if (pl.fwd == GcFwd::unit_tc) return launch_unit_fwd_tc(am, pk, w.wunit, pl.terms, st);
    if (pl.fwd == GcFwd::aggmix_tc) return launch_aggmix_fwd_tc(am, pk, w.wtc, st);
    return launch_aggmix_fwd(am, st);
  }
  DSTD_REQUIRE(a->xa, DSTD_ERR_BAD_ARG, "gc_forward: the unfused path needs the xa buffer");

  // 3. xa = [x;1] (alpha pd + A)           (aggregation before the channel mix)
  AggParams ag;
  fill_agg(ag, N, Cin, P, K, nb, a->flags, a->x, a->pd, a->alpha, a->br);
  ag.xa = a->xa;
  if ((rc = pl.generic ? launch_aggregate_fwd_gen(ag, sw.agg_gen_mma, st) : launch_aggregate_fwd(ag, st))) return rc;

  // 4. out = [Wf_0 bf_0 | Wf_1 bf_1] xa (+ skip)
  BgemmParams g2;
  g2.M = Cout; g2.Kd = nb * C1; g2.G = pl.G; g2.P = P; g2.K = K;
  g2.w = w.wcat; g2.wsc = 1; g2.wsi = nb * C1; g2.bias = nullptr;
  g2.in = dense_view(a->xa, nb * C1, P, K); g2.ones_row = -1;
  g2.out = mk(a->out);
  g2.add = mk(a->skip);
  g2.tc_ws = sw.bgemm_tc && bgemm_tc_ws_bytes(Cout, nb * C1) ? w.wbt : nullptr;
  return launch_bgemm(g2, st);
}

// ---------------------------------------------------------------------------------------------- DSTD-GC backward
extern "C" int dstd_gc_backward(const dstd_gc_bwd_args* a, dstd_stream_t stream) {
  DSTD_REQUIRE(a, DSTD_ERR_BAD_ARG, "gc_backward: null args");
  int rc = poll_device_error("gc_backward");
  if (rc) return rc;
  rc = gc_check_common(a->N, a->Cin, a->Cout, a->P, a->K, a->nb, a->br, "gc_backward");
  if (rc) return rc;
  DSTD_REQUIRE(a->x.ptr && a->gout.ptr && a->gx.ptr && a->m && a->pd, DSTD_ERR_BAD_ARG, "gc_backward: null tensor");
  const Switches sw = read_switches();
  const GcPlan pl = gc_plan(a->N, a->Cin, a->Cout, a->P, a->K, a->nb, sw);
  const size_t need = gc_bwd_ws(pl);
  DSTD_REQUIRE(a->ws && a->ws_bytes >= need, DSTD_ERR_WORKSPACE, "gc_backward: workspace too small (%zu < %zu)",
               a->ws_bytes, need);
  cudaStream_t st = (cudaStream_t)stream;
  const int N = a->N, Cin = a->Cin, Cout = a->Cout, P = a->P, K = a->K, nb = a->nb, C1 = pl.C1;
  const long long G = pl.G;
  Arena ar(a->ws, a->ws_bytes);
  const GcBwdWs w = carve_bwd(pl, ar);
  const bool fused = pl.bwd != GcBwd::unfused;

  PackParams pk;
  fill_pack(pk, Cin, Cout, nb, a->br, w.wcat, w.wm);
  if ((rc = launch_pack(pk, st))) return rc;

  int S1a = 0, n_wf = 0;
  if (fused) {
    // 1-3 fused: gxa, xa (recomputed), g(wcat), gx (aggregation part), gxm without leaving the SM
    AggMixBwdParams am;
    am.N = N; am.Cin = Cin; am.Cout = Cout; am.P = P; am.K = K; am.nb = nb;
    am.adj_t = (a->flags & DSTD_FLAG_ADJ_T) ? 1 : 0;
    am.PCH = am.LD = am.CinP = am.WS = 0;
    am.x = mk(a->x); am.gout = mk(a->gout); am.gx = mk(a->gx);
    am.pd = a->pd; am.alpha = a->alpha;
    fill_adj(am, nb, a->br);
    for (int b = 0; b < DSTD_MAX_BRANCH; ++b) {
      am.w_f[b] = pk.w_f[b]; am.b_f[b] = pk.b_f[b];
    }
    am.gxm = w.gxm; am.part_w = w.p_wf; am.part_b = w.p_bf;
    if (pl.bwd == GcBwd::unit_tc) {
      if ((rc = launch_unit_bwd_tc(am, pk, w.wunit, pl.terms, st))) return rc;
      n_wf = unit_bwd_tc_ctas(N, Cin, Cout, P, K, nb);
    } else {
      if ((rc = launch_aggmix_bwd(am, st))) return rc;
      n_wf = aggmix_bwd_ctas(N, P, K, Cin, Cout, nb);
    }
  } else {
  DSTD_REQUIRE(a->xa, DSTD_ERR_BAD_ARG, "gc_backward: the unfused path needs the saved xa buffer");

  // 1. gxa = wcat^T gout
  BgemmParams g1;
  g1.M = nb * C1; g1.Kd = Cout; g1.G = G; g1.P = P; g1.K = K;
  g1.w = w.wcat; g1.wsc = nb * C1; g1.wsi = 1; g1.bias = nullptr;
  g1.in = mk(a->gout); g1.ones_row = -1;
  g1.out = dense_view(w.gxa, nb * C1, P, K);
  g1.add = View4{nullptr, 0, 0, 0, 0};
  g1.tc_ws = sw.bgemm_tc && bgemm_tc_ws_bytes(nb * C1, Cout) ? w.wbt : nullptr;
  if ((rc = launch_bgemm(g1, st))) return rc;

  // 2. g(wcat)[o, j] = sum gout[o] xa[j]
  WgradParams w1;
  w1.M = Cout; w1.Cd = nb * C1; w1.G = G; w1.P = P; w1.K = K;
  w1.a = mk(a->gout);
  w1.b = dense_view(const_cast<float*>(a->xa), nb * C1, P, K);
  w1.b_ones_row = -1;
  w1.partial = w.p_wcat;
  if ((rc = launch_wgrad(w1, sw.bgemm_tc, st))) return rc;
  S1a = w1.S;

  // 3. aggregation backward: gx (first contribution), gxm
  AggParams ag;
  fill_agg(ag, N, Cin, P, K, nb, a->flags, a->x, a->pd, a->alpha, a->br);
  ag.gxa = w.gxa;
  ag.gx = mk(a->gx);
  ag.gxm = w.gxm;
  if ((rc = pl.generic ? launch_aggregate_bwd_gen(ag, st) : launch_aggregate_bwd(ag, st))) return rc;
  }

  // 4. dynamic adjacency backward: gm, partial gWrm/gbrm, gA_eff, galpha
  DynAdjBwdParams db;
  db.N = N; db.P = P; db.K = K; db.nb = nb;
  db.m = a->m; db.pd = a->pd; db.gxm = w.gxm; db.alpha = a->alpha; db.gm = w.gm;
  fill_rm(db, nb, a->br);
  db.S = pl.S2; db.part_wrm = w.p_wrm; db.part_adj = w.p_adj; db.part_alpha = w.p_alpha;
  if ((rc = pl.generic ? launch_dynadj_bwd_gen(db, w.gm2_part, st) : launch_dynadj_bwd(db, st))) return rc;

  // 5+6. gx += wm^T gm ; g(wm)[j, c] = sum gm[j] [x;1][c]   (one pass over x)
  int S1b = 0;
  if (mproj_bwd_supported(Cin, 4 * nb)) {
    MprojBwdParams mp;
    mp.Cin = Cin; mp.J = 4 * nb; mp.P = P; mp.K = K; mp.G = G;
    mp.x = mk(a->x); mp.gx = mk(a->gx); mp.gx_add = mk(a->gx_add); mp.gm = w.gm; mp.wm = w.wm; mp.partial = w.p_wm;
    if ((rc = launch_mproj_bwd(mp, st))) return rc;
    S1b = mproj_bwd_ctas(G);
  } else {
    DSTD_REQUIRE(!a->gx_add.ptr, DSTD_ERR_UNSUPPORTED, "gc_backward: gx_add needs the fused m-projection backward (Cin <= 320)");
    BgemmParams g2;
    g2.M = Cin; g2.Kd = 4 * nb; g2.G = G; g2.P = P; g2.K = K;
    g2.w = w.wm; g2.wsc = C1; g2.wsi = 1; g2.bias = nullptr;
    g2.in = dense_view(w.gm, 4 * nb, P, K); g2.ones_row = -1;
    g2.out = mk(a->gx);
    g2.add = mk(a->gx);
    if ((rc = launch_bgemm(g2, st))) return rc;
    WgradParams w2;
    w2.M = 4 * nb; w2.Cd = C1; w2.G = G; w2.P = P; w2.K = K;
    w2.a = dense_view(w.gm, 4 * nb, P, K);
    w2.b = mk(a->x);
    w2.b_ones_row = Cin;
    w2.partial = w.p_wm;
    if ((rc = launch_wgrad(w2, sw.bgemm_tc, st))) return rc;
    S1b = w2.S;
  }

  // 7. reduce the split partials and scatter them into the parameter gradients
  ReduceParams rp;
  rp.nseg = 0;
  const long long st_wcat = (long long)Cout * nb * C1, st_wm = (long long)4 * nb * C1;
  const int P21 = 2 * P + 1, S2 = pl.S2;
  for (int b = 0; b < nb; ++b) {
    const dstd_branch_grad& g = a->gbr[b];
    if (fused) {
      add_seg(rp, w.p_wf + (long long)b * Cout * Cin, n_wf, (long long)nb * Cout * Cin, Cout, Cin, Cin, g.w_f, Cin);
      add_seg(rp, w.p_bf + (long long)b * Cout, n_wf, (long long)nb * Cout, Cout, 1, 1, g.b_f, 1);
    } else {
      add_seg(rp, w.p_wcat + b * C1, S1a, st_wcat, Cout, Cin, nb * C1, g.w_f, Cin);
      add_seg(rp, w.p_wcat + b * C1 + Cin, S1a, st_wcat, Cout, 1, nb * C1, g.b_f, 1);
    }
    add_seg(rp, w.p_wm + (b * 4 + 0) * C1, S1b, st_wm, 2, Cin, C1, g.w_m1, Cin);
    add_seg(rp, w.p_wm + (b * 4 + 0) * C1 + Cin, S1b, st_wm, 2, 1, C1, g.b_m1, 1);
    add_seg(rp, w.p_wm + (b * 4 + 2) * C1, S1b, st_wm, 2, Cin, C1, g.w_m2, Cin);
    add_seg(rp, w.p_wm + (b * 4 + 2) * C1 + Cin, S1b, st_wm, 2, 1, C1, g.b_m2, 1);
    add_seg(rp, w.p_wrm + (long long)b * P * P21, S2, (long long)nb * P * P21, P, 2 * P, P21, g.w_rm, 2 * P);
    add_seg(rp, w.p_wrm + (long long)b * P * P21 + 2 * P, S2, (long long)nb * P * P21, P, 1, P21, g.b_rm, 1);
    float* gadjw = a->br[b].adj_w ? g.adj_w : nullptr;
    add_seg(rp, w.p_adj + (long long)b * K * K, pl.generic ? N : S2, (long long)nb * K * K, K, K, K, g.adj_eff, K,
            a->br[b].adj, gadjw);
  }
  add_seg(rp, w.p_alpha, S2 * nb, 1, 1, 1, 1, a->alpha ? a->galpha : nullptr, 1);
  return launch_reduce(rp, st);
}

// ---------------------------------------------------------------------------------------------- 1x1 channel mix
extern "C" size_t dstd_chmix_bwd_workspace_bytes(int N, int Cin, int Cout, int P, int K) {
  const long long G = (long long)N * P * K;
  return arena_need({(size_t)wgrad_splits(G) * Cout * (Cin + 1) * 4});
}

extern "C" int dstd_chmix_forward(const dstd_chmix_fwd_args* a, dstd_stream_t stream) {
  DSTD_REQUIRE(a && a->x.ptr && a->out.ptr && a->w, DSTD_ERR_BAD_ARG, "chmix_forward: null argument");
  DSTD_REQUIRE(a->N > 0 && a->Cin > 0 && a->Cout > 0 && a->P > 0 && a->K > 0, DSTD_ERR_BAD_ARG,
               "chmix_forward: non-positive dimension");
  BgemmParams g;
  g.M = a->Cout; g.Kd = a->Cin; g.G = (long long)a->N * a->P * a->K; g.P = a->P; g.K = a->K;
  g.w = a->w; g.wsc = 1; g.wsi = a->Cin; g.bias = a->b;
  g.in = mk(a->x); g.ones_row = -1;
  g.out = mk(a->out);
  g.add = View4{nullptr, 0, 0, 0, 0};
  return launch_bgemm(g, (cudaStream_t)stream);
}

extern "C" int dstd_chmix_backward(const dstd_chmix_bwd_args* a, dstd_stream_t stream) {
  DSTD_REQUIRE(a && a->x.ptr && a->gout.ptr && a->w, DSTD_ERR_BAD_ARG, "chmix_backward: null argument");
  DSTD_REQUIRE(a->N > 0 && a->Cin > 0 && a->Cout > 0 && a->P > 0 && a->K > 0, DSTD_ERR_BAD_ARG,
               "chmix_backward: non-positive dimension");
  const Switches sw = read_switches();
  cudaStream_t st = (cudaStream_t)stream;
  const int Cin = a->Cin, Cout = a->Cout, C1 = Cin + 1;
  const long long G = (long long)a->N * a->P * a->K;
  int rc;
  if (a->gx.ptr) {
    BgemmParams g;
    g.M = Cin; g.Kd = Cout; g.G = G; g.P = a->P; g.K = a->K;
    g.w = a->w; g.wsc = Cin; g.wsi = 1; g.bias = nullptr;
    g.in = mk(a->gout); g.ones_row = -1;
    g.out = mk(a->gx);
    g.add = View4{nullptr, 0, 0, 0, 0};
    if ((rc = launch_bgemm(g, st))) return rc;
  }
  if (a->gw || a->gb) {
    DSTD_REQUIRE(a->ws && a->ws_bytes >= dstd_chmix_bwd_workspace_bytes(a->N, Cin, Cout, a->P, a->K),
                 DSTD_ERR_WORKSPACE, "chmix_backward: workspace too small");
    Arena ar(a->ws, a->ws_bytes);
    const int S = wgrad_splits(G);
    float* part = ar.take<float>((size_t)S * Cout * C1);
    WgradParams w;
    w.M = Cout; w.Cd = C1; w.G = G; w.P = a->P; w.K = a->K;
    w.a = mk(a->gout);
    w.b = mk(a->x);
    w.b_ones_row = Cin;
    w.partial = part;
    if ((rc = launch_wgrad(w, sw.bgemm_tc, st))) return rc;
    ReduceParams rp;
    rp.nseg = 0;
    add_seg(rp, part, w.S, (long long)Cout * C1, Cout, Cin, C1, a->gw, Cin);
    add_seg(rp, part + Cin, w.S, (long long)Cout * C1, Cout, 1, C1, a->gb, 1);
    return launch_reduce(rp, st);
  }
  return DSTD_OK;
}
