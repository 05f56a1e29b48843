// Small kernels around the DSTD-GC units: weight packing, model head/tail (DSTDGCN.forward, model/dstdgcn.py:298-303
// and :314-315), and the engine glue on device (mpjpe_error_3d engine/utils/loss.py:52-65, Adam engine/prediction.py:188).
#include "kernels.cuh"

namespace dstd {

// ------------------------------------------------------------------------------------------ weight packing
// wcat[o][b*(Cin+1)+c] = c<Cin ? w_f_b[o][c] : b_f_b[o]      (channel mix applied after the aggregation; the bias
//                                                             multiplies the "ones" row = column sums of the adjacency)
// wm[b*4+j][c]         = rows of conv_m1 (j=0,1) / conv_m2 (j=2,3), bias in column Cin
__global__ void pack_kernel(PackParams q) {
  const int C1 = q.Cin + 1, ld = q.nb * C1;
  const int n1 = q.Cout * ld, n2 = 4 * q.nb * C1;
  const int CoutP = (q.Cout + 7) / 8 * 8;
  const int n3 = q.wcatT ? ld * CoutP : 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n1 + n2 + n3; i += gridDim.x * blockDim.x) {
    if (i >= n1 + n2) {
      int k = i - n1 - n2;
      int j = k / CoutP, o = k - j * CoutP;
      int b = j / C1, c = j - b * C1;
      float v = 0.f;
      if (o < q.Cout) v = c < q.Cin ? __ldg(q.w_f[b] + (long long)o * q.Cin + c) : __ldg(q.b_f[b] + o);
      q.wcatT[k] = v;
    } else if (i < n1) {
      int o = i / ld, rem = i - o * ld;
      int b = rem / C1, c = rem - b * C1;
      q.wcat[i] = c < q.Cin ? __ldg(q.w_f[b] + (long long)o * q.Cin + c) : __ldg(q.b_f[b] + o);
    } else {
      int k = i - n1;
      int row = k / C1, c = k - row * C1;
      int b = row >> 2, j = row & 3;
      const float* w = j < 2 ? q.w_m1[b] : q.w_m2[b];
      const float* bb = j < 2 ? q.b_m1[b] : q.b_m2[b];
      int jj = j & 1;
      q.wm[k] = c < q.Cin ? __ldg(w + (long long)jj * q.Cin + c) : __ldg(bb + jj);
    }
  }
}

int launch_pack(const PackParams& q, cudaStream_t st) {
  int total = q.Cout * q.nb * (q.Cin + 1) + 4 * q.nb * (q.Cin + 1);
  if (q.wcatT) total += q.nb * (q.Cin + 1) * ((q.Cout + 7) / 8 * 8);
  pack_kernel<<<min(cdiv(total, 256), 64), 256, 0, st>>>(q);
  count_launch();
  return check_launch("pack");
}

// ------------------------------------------------------------------------------------------ head / tail
__global__ void prep_fwd_kernel(const float* __restrict__ x, View4 h, int N, int T, int V) {
  const long long total = (long long)N * T * V;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int v = (int)(i % V);
    long long r = i / V;
    int t = (int)(r % T), n = (int)(r / T);
    const float* xp = x + i * 3;
    const float* lp = x + (((long long)n * T + (T - 1)) * V + v) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float a = __ldg(xp + c);
      h.p[vix(h, n, c, t, v)] = a;
      h.p[vix(h, n, c + 3, t, v)] = a - __ldg(lp + c);
    }
  }
}

// gx[n,t,v,c] = gh[n,c,t,v] + gh[n,3+c,t,v] - (t == T-1) * sum_t' gh[n,3+c,t',v]
__global__ void prep_bwd_kernel(View4 gh, float* __restrict__ gx, int N, int T, int V) {
  const long long total = (long long)N * T * V;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int v = (int)(i % V);
    long long r = i / V;
    int t = (int)(r % T), n = (int)(r / T);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float g = gh.p[vix(gh, n, c, t, v)] + gh.p[vix(gh, n, c + 3, t, v)];
      if (t == T - 1) {
        float s = 0.f;
        for (int u = 0; u < T; ++u) s += gh.p[vix(gh, n, c + 3, u, v)];
        g -= s;
      }
      gx[i * 3 + c] = g;
    }
  }
}

__global__ void finish_fwd_kernel(View4 z, const float* __restrict__ x, float* __restrict__ y, int N, int T, int V) {
  const long long total = (long long)N * T * V;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int v = (int)(i % V);
    long long r = i / V;
    int t = (int)(r % T), n = (int)(r / T);
    const float* lp = x + (((long long)n * T + (T - 1)) * V + v) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) y[i * 3 + c] = z.p[vix(z, n, c, t, v)] + __ldg(lp + c);
  }
}

__global__ void finish_bwd_kernel(const float* __restrict__ gy, View4 gz, float* __restrict__ gx, int N, int T, int V) {
  const long long total = (long long)N * T * V;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int v = (int)(i % V);
    long long r = i / V;
    int t = (int)(r % T), n = (int)(r / T);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      gz.p[vix(gz, n, c, t, v)] = __ldg(gy + i * 3 + c);
      if (gx) {
        float s = 0.f;
        if (t == T - 1)
          for (int u = 0; u < T; ++u) s += __ldg(gy + (((long long)n * T + u) * V + v) * 3 + c);
        gx[i * 3 + c] = s;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------ MPJPE
constexpr int MPJPE_BLOCKS = 296, MPJPE_THREADS = 256;

__global__ void __launch_bounds__(MPJPE_THREADS) mpjpe_kernel(const float* __restrict__ pred,
                                                              const float* __restrict__ target, long long J,
                                                              float gscale, float* __restrict__ gpred,
                                                              float* __restrict__ partial) {
  __shared__ float red[32];
  float acc = 0.f;
  for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < J; j += (long long)gridDim.x * blockDim.x) {
    float dx = pred[j * 3] - target[j * 3], dy = pred[j * 3 + 1] - target[j * 3 + 1],
          dz = pred[j * 3 + 2] - target[j * 3 + 2];
    float nrm = sqrtf(dx * dx + dy * dy + dz * dz);
    acc += nrm;
    float inv = nrm > 0.f ? gscale / nrm : 0.f;
    gpred[j * 3] = dx * inv;
    gpred[j * 3 + 1] = dy * inv;
    gpred[j * 3 + 2] = dz * inv;
  }
  float tot = block_sum(acc, red);
  if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}

__global__ void mpjpe_finish_kernel(const float* __restrict__ partial, int nblk, float lscale, int accumulate,
                                    float* loss) {
  __shared__ double red[32];
  double a = 0.;
  for (int i = threadIdx.x; i < nblk; i += blockDim.x) a += partial[i];
  a = warp_sum(a);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
    float l = (float)(t * lscale);
    *loss = accumulate ? *loss + l : l;
  }
}

// ------------------------------------------------------------------------------------------ any coordinate count D
// The same head, tail and loss for x [N,T,V,D], 1 <= D <= MAX_COORDS (DSTDGCN(input_channels = 2D)).  The kernels above
// keep serving D = 3.  Coalescing: every [N,T,V,D] array (x, y, gx, gy, pred, target, gpred) is walked one float per
// thread in memory order, so a warp reads or writes 32 consecutive floats whatever D is; no thread steps through a
// D-float row.  The [N,C,T,V] side goes through the caller's view: consecutive threads touch D channel planes, each at
// consecutive joints.  Each element's arithmetic, and its order, is that of the D = 3 kernels, so D = 3 gives their bits.
constexpr int MAX_COORDS = 32;

// flat element e of a contiguous [N,T,V,D] array -> (n, t, v, c) and the element of the same (n, v, c) at t = T-1
struct PoseElem {
  int n, t, v, c;
  long long last;
};

__device__ __forceinline__ PoseElem pose_elem(long long e, int T, int V, int D) {
  PoseElem p;
  const long long i = e / D;
  p.c = (int)(e - i * D);
  p.v = (int)(i % V);
  const long long r = i / V;
  p.t = (int)(r % T);
  p.n = (int)(r / T);
  p.last = (((long long)p.n * T + (T - 1)) * V + p.v) * D + p.c;
  return p;
}

__global__ void prep_fwd_d_kernel(const float* __restrict__ x, View4 h, int N, int T, int V, int D) {
  const long long total = (long long)N * T * V * D;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const PoseElem p = pose_elem(e, T, V, D);
    const float a = __ldg(x + e);
    h.p[vix(h, p.n, p.c, p.t, p.v)] = a;
    h.p[vix(h, p.n, p.c + D, p.t, p.v)] = a - __ldg(x + p.last);
  }
}

// gx[n,t,v,c] = gh[n,c,t,v] + gh[n,D+c,t,v] - (t == T-1) * sum_t' gh[n,D+c,t',v]
__global__ void prep_bwd_d_kernel(View4 gh, float* __restrict__ gx, int N, int T, int V, int D) {
  const long long total = (long long)N * T * V * D;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const PoseElem p = pose_elem(e, T, V, D);
    float g = gh.p[vix(gh, p.n, p.c, p.t, p.v)] + gh.p[vix(gh, p.n, p.c + D, p.t, p.v)];
    if (p.t == T - 1) {
      float s = 0.f;
      for (int u = 0; u < T; ++u) s += gh.p[vix(gh, p.n, p.c + D, u, p.v)];
      g -= s;
    }
    gx[e] = g;
  }
}

__global__ void finish_fwd_d_kernel(View4 z, const float* __restrict__ x, float* __restrict__ y, int N, int T, int V,
                                    int D) {
  const long long total = (long long)N * T * V * D;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const PoseElem p = pose_elem(e, T, V, D);
    y[e] = z.p[vix(z, p.n, p.c, p.t, p.v)] + __ldg(x + p.last);
  }
}

// the t = T-1 column sum reads gy at stride V*D per frame, but the threads of a warp read consecutive floats each frame
__global__ void finish_bwd_d_kernel(const float* __restrict__ gy, View4 gz, float* __restrict__ gx, int N, int T, int V,
                                    int D) {
  const long long total = (long long)N * T * V * D;
  const long long frame = (long long)V * D;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const PoseElem p = pose_elem(e, T, V, D);
    gz.p[vix(gz, p.n, p.c, p.t, p.v)] = __ldg(gy + e);
    if (gx) {
      float s = 0.f;
      if (p.t == T - 1)
        for (int u = 0; u < T; ++u) s += __ldg(gy + p.last - (long long)(T - 1 - u) * frame);
      gx[e] = s;
    }
  }
}

// Pose error over J D-vectors.  Thread j of a block owns joint j of the block's current tile of MPJPE_THREADS joints, as
// in mpjpe_kernel (same joints per thread, same order, same block sum, so the partials and the loss are deterministic
// and at D = 3 equal mpjpe_kernel's).  The tile's pred - target is staged through shared memory with coalesced loads, the
// gradient leaves the same way.  Rows are padded to an odd stride so that the per-joint row reads hit 32 banks.
__global__ void __launch_bounds__(MPJPE_THREADS) pose_error_kernel(const float* __restrict__ pred,
                                                                   const float* __restrict__ target, long long J, int D,
                                                                   float gscale, float* __restrict__ gpred,
                                                                   float* __restrict__ partial) {
  extern __shared__ float tile[];   // [MPJPE_THREADS][D | 1]
  __shared__ float red[32];
  const int ld = D | 1;
  float acc = 0.f;
  for (long long j0 = blockIdx.x * (long long)MPJPE_THREADS; j0 < J; j0 += (long long)gridDim.x * MPJPE_THREADS) {
    const int nj = (int)min((long long)MPJPE_THREADS, J - j0);
    const long long off = j0 * D;
    for (int e = threadIdx.x; e < nj * D; e += MPJPE_THREADS) {
      const int r = e / D;
      tile[r * ld + (e - r * D)] = pred[off + e] - target[off + e];
    }
    __syncthreads();
    if (threadIdx.x < nj) {
      float* d = tile + threadIdx.x * ld;
      // the contraction mpjpe_kernel's dx*dx + dy*dy + dz*dz compiles to
      float ss = D == 1 ? d[0] * d[0] : fmaf(d[0], d[0], d[1] * d[1]);
      for (int c = 2; c < D; ++c) ss = fmaf(d[c], d[c], ss);
      const float nrm = sqrtf(ss);
      acc += nrm;
      const float inv = nrm > 0.f ? gscale / nrm : 0.f;
      for (int c = 0; c < D; ++c) d[c] *= inv;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < nj * D; e += MPJPE_THREADS) {
      const int r = e / D;
      gpred[off + e] = tile[r * ld + (e - r * D)];
    }
    __syncthreads();
  }
  float tot = block_sum(acc, red);
  if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}

// ------------------------------------------------------------------------------------------ Adam
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, long long n, float lr, float b1, float b2, float eps, float wd,
                            float gs, float bc1, float bc2_sqrt, const float* __restrict__ lr_dev,
                            const int* __restrict__ step_dev) {
  if (lr_dev) lr = __ldg(lr_dev);
  if (step_dev) {
    const float s = (float)__ldg(step_dev);
    bc1 = -expm1f(s * log1pf(b1 - 1.f));          // 1 - b1^s without cancellation
    bc2_sqrt = sqrtf(-expm1f(s * log1pf(b2 - 1.f)));
  }
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float gi = g[i] * gs;
    float pi = p[i];
    if (wd != 0.f) gi = fmaf(wd, pi, gi);
    float mi = b1 * m[i] + (1.f - b1) * gi;
    float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = pi - (lr / bc1) * (mi / denom);
  }
}

}  // namespace dstd

// =========================================================================================== C ABI
using namespace dstd;

static int grid_for(long long total, int threads) {
  long long b = (total + threads - 1) / threads;
  if (b > num_sms() * 16) b = num_sms() * 16;
  if (b < 1) b = 1;
  return (int)b;
}

extern "C" int dstd_prep_forward(const float* x, dstd_view h, int N, int T, int V, dstd_stream_t stream) {
  DSTD_REQUIRE(x && h.ptr && N > 0 && T > 0 && V > 0, DSTD_ERR_BAD_ARG, "prep_forward: bad args");
  prep_fwd_kernel<<<grid_for((long long)N * T * V, 256), 256, 0, (cudaStream_t)stream>>>(x, mk(h), N, T, V);
  count_launch();
  return check_launch("prep_fwd");
}

extern "C" int dstd_prep_backward(dstd_view gh, float* gx, int N, int T, int V, dstd_stream_t stream) {
  DSTD_REQUIRE(gx && gh.ptr && N > 0 && T > 0 && V > 0, DSTD_ERR_BAD_ARG, "prep_backward: bad args");
  prep_bwd_kernel<<<grid_for((long long)N * T * V, 256), 256, 0, (cudaStream_t)stream>>>(mk(gh), gx, N, T, V);
  count_launch();
  return check_launch("prep_bwd");
}

extern "C" int dstd_finish_forward(dstd_view z, const float* x, float* y, int N, int T, int V, dstd_stream_t stream) {
  DSTD_REQUIRE(x && y && z.ptr && N > 0 && T > 0 && V > 0, DSTD_ERR_BAD_ARG, "finish_forward: bad args");
  finish_fwd_kernel<<<grid_for((long long)N * T * V, 256), 256, 0, (cudaStream_t)stream>>>(mk(z), x, y, N, T, V);
  count_launch();
  return check_launch("finish_fwd");
}

extern "C" int dstd_finish_backward(const float* gy, dstd_view gz, float* gx, int N, int T, int V,
                                    dstd_stream_t stream) {
  DSTD_REQUIRE(gy && gz.ptr && N > 0 && T > 0 && V > 0, DSTD_ERR_BAD_ARG, "finish_backward: bad args");
  finish_bwd_kernel<<<grid_for((long long)N * T * V, 256), 256, 0, (cudaStream_t)stream>>>(gy, mk(gz), gx, N, T, V);
  count_launch();
  return check_launch("finish_bwd");
}

extern "C" size_t dstd_mpjpe_workspace_bytes(long long J) {
  (void)J;
  return arena_need({(size_t)MPJPE_BLOCKS * sizeof(float)});
}

extern "C" int dstd_mpjpe_forward_backward(const float* pred, const float* target, long long J, float scale,
                                           int accumulate, float* loss_out, float* gpred, void* ws, size_t ws_bytes,
                                           dstd_stream_t stream) {
  DSTD_REQUIRE(pred && target && loss_out && gpred && J > 0, DSTD_ERR_BAD_ARG, "mpjpe: bad args");
  DSTD_REQUIRE(ws && ws_bytes >= dstd_mpjpe_workspace_bytes(J), DSTD_ERR_WORKSPACE, "mpjpe: workspace too small");
  Arena ar(ws, ws_bytes);
  float* partial = ar.take<float>(MPJPE_BLOCKS);
  int nblk = (int)((J + MPJPE_THREADS - 1) / MPJPE_THREADS);
  if (nblk > MPJPE_BLOCKS) nblk = MPJPE_BLOCKS;
  cudaStream_t st = (cudaStream_t)stream;
  mpjpe_kernel<<<nblk, MPJPE_THREADS, 0, st>>>(pred, target, J, scale / (float)J, gpred, partial);
  count_launch();
  DSTD_LAUNCH_CHECK("mpjpe");
  mpjpe_finish_kernel<<<1, 256, 0, st>>>(partial, nblk, scale / (float)J, accumulate, loss_out);
  count_launch();
  return check_launch("mpjpe_finish");
}

#define REQUIRE_COORDS(what, D)                                                                                    \
  DSTD_REQUIRE((D) >= 1 && (D) <= MAX_COORDS, DSTD_ERR_UNSUPPORTED,                                                \
               what ": D=%d coordinates per joint outside the supported 1..%d", (D), MAX_COORDS)

extern "C" int dstd_prep_forward_d(const float* x, dstd_view h, int N, int T, int V, int D, dstd_stream_t stream) {
  DSTD_REQUIRE(x && h.ptr && N > 0 && T > 0 && V > 0, DSTD_ERR_BAD_ARG, "prep_forward_d: bad args");
  REQUIRE_COORDS("prep_forward_d", D);
  prep_fwd_d_kernel<<<grid_for((long long)N * T * V * D, 256), 256, 0, (cudaStream_t)stream>>>(x, mk(h), N, T, V, D);
  count_launch();
  return check_launch("prep_fwd_d");
}

extern "C" int dstd_prep_backward_d(dstd_view gh, float* gx, int N, int T, int V, int D, dstd_stream_t stream) {
  DSTD_REQUIRE(gx && gh.ptr && N > 0 && T > 0 && V > 0, DSTD_ERR_BAD_ARG, "prep_backward_d: bad args");
  REQUIRE_COORDS("prep_backward_d", D);
  prep_bwd_d_kernel<<<grid_for((long long)N * T * V * D, 256), 256, 0, (cudaStream_t)stream>>>(mk(gh), gx, N, T, V, D);
  count_launch();
  return check_launch("prep_bwd_d");
}

extern "C" int dstd_finish_forward_d(dstd_view z, const float* x, float* y, int N, int T, int V, int D,
                                     dstd_stream_t stream) {
  DSTD_REQUIRE(x && y && z.ptr && N > 0 && T > 0 && V > 0, DSTD_ERR_BAD_ARG, "finish_forward_d: bad args");
  REQUIRE_COORDS("finish_forward_d", D);
  finish_fwd_d_kernel<<<grid_for((long long)N * T * V * D, 256), 256, 0, (cudaStream_t)stream>>>(mk(z), x, y, N, T, V,
                                                                                                 D);
  count_launch();
  return check_launch("finish_fwd_d");
}

extern "C" int dstd_finish_backward_d(const float* gy, dstd_view gz, float* gx, int N, int T, int V, int D,
                                      dstd_stream_t stream) {
  DSTD_REQUIRE(gy && gz.ptr && N > 0 && T > 0 && V > 0, DSTD_ERR_BAD_ARG, "finish_backward_d: bad args");
  REQUIRE_COORDS("finish_backward_d", D);
  finish_bwd_d_kernel<<<grid_for((long long)N * T * V * D, 256), 256, 0, (cudaStream_t)stream>>>(gy, mk(gz), gx, N, T,
                                                                                                 V, D);
  count_launch();
  return check_launch("finish_bwd_d");
}

extern "C" size_t dstd_pose_error_workspace_bytes(long long J) {
  (void)J;
  return arena_need({(size_t)MPJPE_BLOCKS * sizeof(float)});
}

extern "C" int dstd_pose_error_forward_backward(const float* pred, const float* target, long long J, int D, float scale,
                                                int accumulate, float* loss_out, float* gpred, void* ws,
                                                size_t ws_bytes, dstd_stream_t stream) {
  DSTD_REQUIRE(pred && target && loss_out && gpred && J > 0, DSTD_ERR_BAD_ARG, "pose_error: bad args");
  REQUIRE_COORDS("pose_error", D);
  DSTD_REQUIRE(ws && ws_bytes >= dstd_pose_error_workspace_bytes(J), DSTD_ERR_WORKSPACE,
               "pose_error: workspace too small");
  Arena ar(ws, ws_bytes);
  float* partial = ar.take<float>(MPJPE_BLOCKS);
  int nblk = (int)((J + MPJPE_THREADS - 1) / MPJPE_THREADS);
  if (nblk > MPJPE_BLOCKS) nblk = MPJPE_BLOCKS;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t smem = (size_t)MPJPE_THREADS * (D | 1) * sizeof(float);   // <= 33 KB at D = 32
  pose_error_kernel<<<nblk, MPJPE_THREADS, smem, st>>>(pred, target, J, D, scale / (float)J, gpred, partial);
  count_launch();
  DSTD_LAUNCH_CHECK("pose_error");
  mpjpe_finish_kernel<<<1, 256, 0, st>>>(partial, nblk, scale / (float)J, accumulate, loss_out);
  count_launch();
  return check_launch("pose_error_finish");
}

extern "C" int dstd_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                              float beta1, float beta2, float eps, float weight_decay, float grad_scale, int step,
                              const float* lr_dev, const int* step_dev, dstd_stream_t stream) {
  DSTD_REQUIRE(param && grad && exp_avg && exp_avg_sq && n > 0 && (step > 0 || step_dev), DSTD_ERR_BAD_ARG,
               "adam_step: bad args");
  if (step <= 0) step = 1;
  double bc1 = 1.0 - pow((double)beta1, (double)step);
  double bc2 = 1.0 - pow((double)beta2, (double)step);
  adam_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2,
                                                                  eps, weight_decay, grad_scale, (float)bc1,
                                                                  (float)sqrt(bc2), lr_dev, step_dev);
  count_launch();
  return check_launch("adam");
}
