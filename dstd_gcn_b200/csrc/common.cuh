// Shared device/host helpers for libdstd_b200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/dstd_b200.h"

namespace dstd {

// ----------------------------------------------------------------------------- host side
void set_error(const char* fmt, ...);
void count_launch(int n = 1);
int check_launch(const char* what);  // cudaGetLastError -> status (+message)
void prefer_smem_carveout(const void* kernel, bool need_max);  // largest smem carve-out (+227 KB opt-in if need_max)
void ensure_max_smem(const void* kernel);  // one-time (per device) opt-in to 227 KB dynamic shared memory
constexpr int MAX_DYN_SMEM = 227 * 1024;
int num_sms();              // multiprocessors of the current device (148 on B200; also the answer when no device is present)
// Device-side failures (a tensor-core pipeline whose mbarrier wait timed out) are written to one host-mapped word by
// the kernel and surfaced by the NEXT entry point as DSTD_ERR_CUDA (sticky until dstd_device_error(1) clears it).
int* device_error_word();   // device pointer to the word (nullptr when it cannot be set up, e.g. under stream capture)
int poll_device_error(const char* fn);

// The library's environment switches (README.md, "Environment switches").  An entry point that depends on one calls
// read_switches() once at its start, so a switch flipped between calls takes effect on the next call.  A flag that is
// unset or empty takes its default, "0" turns it off and any other value turns it on.
struct Switches {
  bool unit_tc;           // DSTD_UNIT_TC (off); also on when DSTD_PRECISION selects a reduced mode
  int unit_terms;         // DSTD_PRECISION: 6 split products per k-step (fp32 parity), 3 (bf16x2) or 1 (bf16)
  bool aggmix_tc;         // tcgen05 fused forward; off with DSTD_DISABLE_TC
  bool bgemm_tc;          // DSTD_BGEMM_TC (on): channel GEMMs and weight gradients on tcgen05 where the shape allows
  bool agg_gen_mma;       // DSTD_AGG_GEN_MMA (off): mma.sync forward aggregation of the shape-generic path
  bool bn_fast;           // DSTD_BN_FAST (on)
  int bn_samples_per_cta; // DSTD_BN_SAMPLES_PER_CTA (32)
};
Switches read_switches();

#define DSTD_REQUIRE(cond, code, ...)      \
  do {                                     \
    if (!(cond)) {                         \
      ::dstd::set_error(__VA_ARGS__);      \
      return (code);                       \
    }                                      \
  } while (0)

#define DSTD_LAUNCH_CHECK(what)                     \
  do {                                              \
    int _rc = ::dstd::check_launch(what);           \
    if (_rc != 0) return _rc;                       \
  } while (0)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// bump allocator over the caller's workspace; over a null base it only counts: need() is then the workspace size that
// the same sequence of take() calls requires (arena_need of their byte counts)
struct Arena {
  uintptr_t base;
  size_t cap, off;
  Arena(void* p, size_t n) : base((uintptr_t)p), cap(n), off(0) {}
  template <typename T>
  T* take(size_t count) {
    size_t o = align_up(off, 256);
    off = o + count * sizeof(T);
    return (T*)(base + o);
  }
  bool ok() const { return off <= cap; }
  size_t need() const { return align_up(off, 256) + 256; }
};
static inline size_t arena_need(std::initializer_list<size_t> bytes) {
  size_t o = 0;
  for (size_t b : bytes) o = align_up(o, 256) + b;
  return align_up(o, 256) + 256;
}

// ----------------------------------------------------------------------------- device side
struct View4 {
  float* p;
  long long sn, sc, sp, sk;
};
static inline View4 mk(const dstd_view& v) { return View4{v.ptr, v.sn, v.sc, v.sp, v.sk}; }
static inline View4 dense_view(float* p, long long C, long long P, long long K) {
  return View4{p, C * P * K, P * K, K, 1};
}

__device__ __forceinline__ long long vix(const View4& v, int n, int c, int p, int k) {
  return (long long)n * v.sn + (long long)c * v.sc + (long long)p * v.sp + (long long)k * v.sk;
}

// tanh of the pairwise differences.  Default: CUDA's tanhf (polynomial below 0.55, ex2/rcp above; <= 2 ulp), measured
// at 7.0 results/clk/SM on B200 against 7.9 for the bare ex2+rcp form (tools/microbench.cu).  The bare form
// 1 - 2/(exp(2x)+1) has a ~1.2e-7 ABSOLUTE error, i.e. a large relative error on the small differences that dominate
// here; on the full-depth model that error, amplified by the cancellation in bias-like gradients, cost 3-5x in gradient
// parity (tools/diag_fullsize.py), so it is opt-in (-DDSTD_FAST_TANH).  tanh.approx.f32 (5e-4 relative) is out of the
// question for the 1e-4 parity budget.
__device__ __forceinline__ float fast_tanh(float x) {
#ifdef DSTD_FAST_TANH
  float e = exp2f(x * 2.885390081777927f);  // exp(2x); ex2.approx, saturates to inf / 0
  return 1.0f - __fdividef(2.0f, e + 1.0f);
#else
  return tanhf(x);
#endif
}

// ---- cp.async (LDGSTS): fire-and-forget global -> shared copies; a staging loop issues all of them back to back, so the
// memory-level parallelism is the number of copies per thread, not 1.  valid == false zero-fills the destination.
__device__ __forceinline__ void cp_async4(float* smem_dst, const float* gsrc, bool valid) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int sz = valid ? 4 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(d), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {   // all but the N most recent groups have landed
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// block-wide sum; `red` is >= 32 floats of shared memory; result valid in every thread
__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  float r = (threadIdx.x < (blockDim.x + 31) / 32) ? red[threadIdx.x] : 0.f;
  if (w == 0) r = warp_sum(r);
  if (threadIdx.x == 0) red[0] = r;
  __syncthreads();
  r = red[0];
  return r;
}

}  // namespace dstd
