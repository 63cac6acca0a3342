// Device kernels of the C API's graph executor (csrc/runtime/device_exec.h) for the operators the fused training kernels do not cover:
// windowed pooling with any kernel / stride / padding, elementwise activations, broadcast binary arithmetic with reduce-to-shape gradients,
// strided copies (Concat), counter-based dropout, softmax over (outer, C, inner) and the SoftmaxOutput gradient, BatchNorm's gradient with
// running statistics, and the rows <-> NCHW transposes around convolution GEMMs.  Every backward kernel ADDS into its gradient buffer: the
// executor zeroes gradients once per Backward and fan-out accumulates, as in the host executor (train_exec.h).
//
// The gx_rt_* functions give the C API (compiled with g++, without CUDA headers, loading this library with dlopen) the few runtime calls it
// needs: device count, current device, one stream per device, streams of its own (one per native predictor), copies (peer copies
// included), memset, stream synchronisation, stream-to-stream joins, page-locked host staging and the capture / replay of a stream's work
// as a CUDA graph.
#include <cuda_runtime.h>

#include <mutex>
#include <vector>

#include "common.cuh"

namespace {

using gx::launch_pdl;
using gx::pdl_wait;

constexpr int kThreads = 256;
inline unsigned blocks_for(long long n, long long cap = 148LL * 32) {
  long long b = (n + kThreads - 1) / kThreads;
  return (unsigned)(b < 1 ? 1 : b > cap ? cap : b);
}
#define GRID_STRIDE(i, n) for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < (n); i += (long long)gridDim.x * blockDim.x)

// ------------------------------------------------------------------------------------------------ small elementwise helpers
__global__ void axpy_kernel(float* __restrict__ y, const float* __restrict__ x, float a, long long n) {
  pdl_wait();
  GRID_STRIDE(i, n) y[i] += a * x[i];
}
__global__ void add_scalar_kernel(float* __restrict__ y, float c, long long n) {
  pdl_wait();
  GRID_STRIDE(i, n) y[i] += c;
}
__global__ void mul_add_kernel(float* __restrict__ y, const float* __restrict__ a, const float* __restrict__ b, long long n) {
  pdl_wait();
  GRID_STRIDE(i, n) y[i] += a[i] * b[i];
}
// y[n, c, p] (+)= rows[(n * HW + p) * ld + c]
__global__ void rows_to_nchw_kernel(const float* __restrict__ rows, float* __restrict__ y, int N, int C, int HW, long long ld, int accumulate) {
  pdl_wait();
  const long long total = (long long)N * C * HW;
  GRID_STRIDE(i, total) {
    const long long p = i % HW, c = (i / HW) % C, n = i / ((long long)HW * C);
    const float v = rows[(n * HW + p) * ld + c];
    y[i] = accumulate ? y[i] + v : v;
  }
}

// ------------------------------------------------------------------------------------------------ activations
// kind: 0 relu, 1 sigmoid, 2 tanh, 3 softrelu, 4 softsign, 5 leaky (slope)
__device__ __forceinline__ float act_f(int k, float v, float slope) {
  switch (k) {
    case 0: return v > 0.f ? v : 0.f;
    case 1: return 1.f / (1.f + expf(-v));
    case 2: return tanhf(v);
    case 3: return v > 20.f ? v : log1pf(expf(v));
    case 4: return v / (1.f + fabsf(v));
    default: return v > 0.f ? v : slope * v;
  }
}
__device__ __forceinline__ float act_g(int k, float x, float y, float slope) {
  switch (k) {
    case 0: return x > 0.f ? 1.f : 0.f;
    case 1: return y * (1.f - y);
    case 2: return 1.f - y * y;
    case 3: return 1.f / (1.f + expf(-x));
    case 4: { const float d = 1.f + fabsf(x); return 1.f / (d * d); }
    default: return x > 0.f ? 1.f : slope;
  }
}
__global__ void act_fwd_kernel(int kind, const float* __restrict__ x, float* __restrict__ y, long long n, float slope) {
  pdl_wait();
  GRID_STRIDE(i, n) y[i] = act_f(kind, x[i], slope);
}
__global__ void act_bwd_kernel(int kind, const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ dy, float* __restrict__ dx,
                               long long n, float slope) {
  pdl_wait();
  GRID_STRIDE(i, n) dx[i] += dy[i] * act_g(kind, x[i], y[i], slope);
}

// ------------------------------------------------------------------------------------------------ pooling (NCHW, any window)
struct PoolGeom { int H, W, OH, OW, kh, kw, sh, sw, ph, pw, type, count_pad; };   // type 0 max, 1 avg, 2 sum

__device__ __forceinline__ float pool_divisor(const PoolGeom& g, int y0, int x0, int ya, int yb, int xa, int xb) {
  if (g.type != 1) return 1.f;
  if (g.count_pad) return (float)((min(y0 + g.kh, g.H + g.ph) - y0) * (min(x0 + g.kw, g.W + g.pw) - x0));
  const int cnt = (yb - ya) * (xb - xa);
  return (float)(cnt > 1 ? cnt : 1);
}
__global__ void pool_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int* __restrict__ idx, long long NC, PoolGeom g) {
  pdl_wait();
  const long long total = NC * g.OH * g.OW;
  GRID_STRIDE(o, total) {
    const int ox = (int)(o % g.OW), oy = (int)((o / g.OW) % g.OH);
    const long long c = o / ((long long)g.OW * g.OH);
    const int y0 = oy * g.sh - g.ph, x0 = ox * g.sw - g.pw;
    const int ya = max(y0, 0), yb = min(y0 + g.kh, g.H), xa = max(x0, 0), xb = min(x0 + g.kw, g.W);
    const float* src = x + c * g.H * g.W;
    if (g.type == 0) {
      float best = -INFINITY; int bi = -1;
      for (int iy = ya; iy < yb; ++iy)
        for (int ix = xa; ix < xb; ++ix) { const float v = src[iy * g.W + ix]; if (v > best) { best = v; bi = iy * g.W + ix; } }
      y[o] = bi < 0 ? 0.f : best; idx[o] = bi;
    } else {
      float acc = 0.f;
      for (int iy = ya; iy < yb; ++iy)
        for (int ix = xa; ix < xb; ++ix) acc += src[iy * g.W + ix];
      y[o] = acc / pool_divisor(g, y0, x0, ya, yb, xa, xb);
    }
  }
}
// windows overlap when stride < kernel: scatter with atomics
__global__ void pool_bwd_kernel(const float* __restrict__ dy, const int* __restrict__ idx, float* __restrict__ dx, long long NC, PoolGeom g) {
  pdl_wait();
  const long long total = NC * g.OH * g.OW;
  GRID_STRIDE(o, total) {
    const long long c = o / ((long long)g.OW * g.OH);
    float* dst = dx + c * g.H * g.W;
    if (g.type == 0) { if (idx[o] >= 0) atomicAdd(dst + idx[o], dy[o]); continue; }
    const int ox = (int)(o % g.OW), oy = (int)((o / g.OW) % g.OH);
    const int y0 = oy * g.sh - g.ph, x0 = ox * g.sw - g.pw;
    const int ya = max(y0, 0), yb = min(y0 + g.kh, g.H), xa = max(x0, 0), xb = min(x0 + g.kw, g.W);
    const float v = dy[o] / pool_divisor(g, y0, x0, ya, yb, xa, xb);
    for (int iy = ya; iy < yb; ++iy)
      for (int ix = xa; ix < xb; ++ix) atomicAdd(dst + iy * g.W + ix, v);
  }
}

// ------------------------------------------------------------------------------------------------ broadcast binary (add / sub / mul / div / max / min)
constexpr int kMaxDims = 8;
struct Bcast { int ndim; long long dims[kMaxDims], ls[kMaxDims], rs[kMaxDims]; };   // output extents; operand strides (0 on broadcast axes)

__device__ __forceinline__ void bcast_offsets(const Bcast& b, long long f, long long* li, long long* ri) {
  long long l = 0, r = 0;
  for (int d = b.ndim - 1; d >= 0; --d) { const long long c = f % b.dims[d]; f /= b.dims[d]; l += c * b.ls[d]; r += c * b.rs[d]; }
  *li = l; *ri = r;
}
// 3 div, 4 maximum, 5 minimum (forward only; the operands' order in 4 / 5 is std::max / std::min's)
__device__ __forceinline__ float bin_f(int k, float l, float r) {
  switch (k) {
    case 0: return l + r;
    case 1: return l - r;
    case 2: return l * r;
    case 3: return l / r;
    case 4: return l < r ? r : l;
    default: return r < l ? r : l;
  }
}

__global__ void binary_fwd_kernel(int kind, const float* __restrict__ l, const float* __restrict__ r, float* __restrict__ y, long long n, Bcast b) {
  pdl_wait();
  GRID_STRIDE(i, n) { long long li, ri; bcast_offsets(b, i, &li, &ri); y[i] = bin_f(kind, l[li], r[ri]); }
}
// gradients reduced to each operand's shape; atomics only where an operand is broadcast
__global__ void binary_bwd_kernel(int kind, const float* __restrict__ l, const float* __restrict__ r, const float* __restrict__ dy, float* dl, float* dr,
                                  long long n, Bcast b, int l_bcast, int r_bcast) {
  pdl_wait();
  GRID_STRIDE(i, n) {
    long long li, ri; bcast_offsets(b, i, &li, &ri);
    const float g = dy[i];
    const float gl = kind == 2 ? g * r[ri] : g;
    const float gr = kind == 0 ? g : kind == 1 ? -g : g * l[li];
    if (dl) { if (l_bcast) atomicAdd(dl + li, gl); else dl[li] += gl; }
    if (dr) { if (r_bcast) atomicAdd(dr + ri, gr); else dr[ri] += gr; }
  }
}

// ------------------------------------------------------------------------------------------------ strided block copy (Concat)
// dst[o * dst_stride + k] (+)= src[o * src_stride + k]  for o < outer, k < len
__global__ void strided_copy_kernel(const float* __restrict__ src, float* __restrict__ dst, long long outer, long long len, long long src_stride,
                                    long long dst_stride, int accumulate) {
  pdl_wait();
  const long long total = outer * len;
  GRID_STRIDE(i, total) {
    const long long o = i / len, k = i % len;
    const float v = src[o * src_stride + k];
    float* d = dst + o * dst_stride + k;
    *d = accumulate ? *d + v : v;
  }
}

// ------------------------------------------------------------------------------------------------ dropout
// Philox-4x32-10 keyed by (seed, step) over the element index: the mask depends only on the seed, the forward count and the element, never
// on the launch shape
__device__ __forceinline__ uint32_t philox_uniform_bits(uint32_t seed, uint32_t step, uint64_t i) {
  uint32_t c0 = (uint32_t)i, c1 = (uint32_t)(i >> 32), c2 = step, c3 = 0u, k0 = seed, k1 = 0x5bd1e995u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t lo0 = 0xD2511F53u * c0, hi0 = __umulhi(0xD2511F53u, c0);
    const uint32_t lo1 = 0xCD9E8D57u * c2, hi1 = __umulhi(0xCD9E8D57u, c2);
    c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return c0;
}
__global__ void dropout_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, float* __restrict__ mask, long long n, float p, uint32_t seed,
                                   uint32_t step) {
  pdl_wait();
  const float scale = 1.f / (1.f - p);
  GRID_STRIDE(i, n) {
    const float u = (philox_uniform_bits(seed, step, (uint64_t)i) >> 8) * (1.f / 16777216.f);     // [0, 1) with 24 bits
    const float m = u >= p ? scale : 0.f;
    mask[i] = m; y[i] = x[i] * m;
  }
}

// ------------------------------------------------------------------------------------------------ softmax over (outer, C, inner)
// one warp per (outer, inner) row
__global__ void softmax_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, long long outer, int C, long long inner, int log_out) {
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const long long rows = outer * inner;
  for (long long row = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5; row < rows; row += ((long long)gridDim.x * blockDim.x) >> 5) {
    const long long o = row / inner, i = row % inner;
    const float* xs = x + o * C * inner + i; float* ys = y + o * C * inner + i;
    float m = -INFINITY;
    for (int k = lane; k < C; k += 32) m = fmaxf(m, xs[k * inner]);
    for (int s = 16; s; s >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, s));
    float z = 0.f;
    for (int k = lane; k < C; k += 32) z += expf(xs[k * inner] - m);
    for (int s = 16; s; s >>= 1) z += __shfl_xor_sync(0xffffffffu, z, s);
    const float lz = logf(z);
    for (int k = lane; k < C; k += 32) ys[k * inner] = log_out ? xs[k * inner] - m - lz : expf(xs[k * inner] - m) / z;
  }
}
__global__ void softmax_bwd_kernel(const float* __restrict__ y, const float* __restrict__ dy, float* __restrict__ dx, long long outer, int C, long long inner,
                                   int log_out) {
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const long long rows = outer * inner;
  for (long long row = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5; row < rows; row += ((long long)gridDim.x * blockDim.x) >> 5) {
    const long long base = (row / inner) * C * inner + row % inner;
    float dot = 0.f;
    for (int k = lane; k < C; k += 32) dot += log_out ? dy[base + k * inner] : dy[base + k * inner] * y[base + k * inner];
    for (int s = 16; s; s >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, s);
    for (int k = lane; k < C; k += 32) {
      const long long at = base + k * inner;
      dx[at] += log_out ? dy[at] - expf(y[at]) * dot : y[at] * (dy[at] - dot);
    }
  }
}
// SoftmaxOutput's gradient: (p - onehot(label)) * grad_scale / norm, rows with the ignored label skipped.  norm: 0 null, 1 batch (outer),
// 2 valid (rows not ignored; every block counts them itself, so there is no second launch)
__global__ void softmax_output_bwd_kernel(const float* __restrict__ y, const float* __restrict__ label, float* __restrict__ dx, long long outer, int C,
                                          long long inner, float grad_scale, int use_ignore, float ignore, int norm) {
  pdl_wait();
  __shared__ float s_valid[32];
  const long long rows = outer * inner;
  float scale = grad_scale;
  if (norm == 1) scale /= (float)outer;
  else if (norm == 2) {
    float v = 0.f;
    for (long long t = threadIdx.x; t < rows; t += blockDim.x) v += (use_ignore && label[t] == ignore) ? 0.f : 1.f;
    for (int s = 16; s; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
    if ((threadIdx.x & 31) == 0) s_valid[threadIdx.x >> 5] = v;
    __syncthreads();
    float tot = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += s_valid[w];
    scale /= fmaxf(tot, 1.f);
  }
  const long long total = rows * C;
  GRID_STRIDE(e, total) {
    const long long o = e / ((long long)C * inner), k = (e / inner) % C, i = e % inner;
    const float l = label[o * inner + i];
    if (use_ignore && l == ignore) continue;
    dx[e] += (y[e] - ((long long)l == k ? 1.f : 0.f)) * scale;
  }
}

// ------------------------------------------------------------------------------------------------ BatchNorm backward with fixed statistics
// use_global_stats (or a backward after an inference forward): y = (x - mean) * rsqrt(var + eps) * gamma + beta with mean / var constants.
// One block per channel.  gamma == nullptr means fix_gamma (gamma = 1, no gamma gradient).
__global__ void bn_global_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy, const float* __restrict__ gamma, const float* __restrict__ mean,
                                     const float* __restrict__ var, float eps, float* dx, float* dgamma, float* dbeta, int N, int C, int HW) {
  pdl_wait();
  __shared__ float s_a[32], s_b[32];
  const int c = blockIdx.x;
  const float mu = mean[c], inv = rsqrtf(var[c] + eps), g = gamma ? gamma[c] : 1.f;
  float sdy = 0.f, sdyx = 0.f;
  const long long cnt = (long long)N * HW;
  for (long long t = threadIdx.x; t < cnt; t += blockDim.x) {
    const long long at = ((t / HW) * C + c) * HW + t % HW;
    const float d = dy[at];
    sdy += d; sdyx += d * (x[at] - mu) * inv;
    if (dx) dx[at] += d * g * inv;
  }
  for (int s = 16; s; s >>= 1) { sdy += __shfl_xor_sync(0xffffffffu, sdy, s); sdyx += __shfl_xor_sync(0xffffffffu, sdyx, s); }
  if ((threadIdx.x & 31) == 0) { s_a[threadIdx.x >> 5] = sdy; s_b[threadIdx.x >> 5] = sdyx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { a += s_a[w]; b += s_b[w]; }
    if (dbeta) dbeta[c] += a;
    if (dgamma && gamma) dgamma[c] += b;
  }
}

// ------------------------------------------------------------------------------------------------ per-device streams
std::mutex g_stream_mu;
std::vector<cudaStream_t> g_streams;

}  // namespace

// ================================================================================================ runtime calls for the C API
GX_API int gx_rt_device_count(int* out) {
  *out = 0;
  const cudaError_t e = cudaGetDeviceCount(out);
  if (e != cudaSuccess) { cudaGetLastError(); *out = 0; }
  return (int)e;
}
GX_API int gx_rt_set_device(int dev) { return (int)cudaSetDevice(dev); }
// the library's stream of `dev`, created on first use (non-blocking: it does not serialise against the legacy default stream)
GX_API void* gx_rt_stream(int dev) {
  std::lock_guard<std::mutex> lk(g_stream_mu);
  if (dev < 0) return nullptr;
  if ((size_t)dev >= g_streams.size()) g_streams.resize(dev + 1, nullptr);
  if (!g_streams[dev]) {
    int cur = 0; cudaGetDevice(&cur);
    if (cudaSetDevice(dev) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    cudaStream_t s = nullptr;
    if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); s = nullptr; }
    cudaSetDevice(cur);
    g_streams[dev] = s;
  }
  return g_streams[dev];
}
// kind: 1 host -> device, 2 device -> host, 3 device -> device, 4 inferred from the pointers (cudaMemcpyDefault); ordered on `stream`
GX_API int gx_rt_memcpy(void* dst, const void* src, unsigned long long bytes, int kind, void* stream) {
  const cudaMemcpyKind k = kind == 1 ? cudaMemcpyHostToDevice : kind == 2 ? cudaMemcpyDeviceToHost : kind == 4 ? cudaMemcpyDefault : cudaMemcpyDeviceToDevice;
  if (bytes == 0) return 0;
  return (int)cudaMemcpyAsync(dst, src, bytes, k, static_cast<cudaStream_t>(stream));
}
GX_API int gx_rt_memset(void* dst, int value, unsigned long long bytes, void* stream) {
  if (bytes == 0) return 0;
  return (int)cudaMemsetAsync(dst, value, bytes, static_cast<cudaStream_t>(stream));
}
GX_API int gx_rt_stream_sync(void* stream) { return (int)cudaStreamSynchronize(static_cast<cudaStream_t>(stream)); }
GX_API const char* gx_rt_error_string(int code) { return cudaGetErrorString(static_cast<cudaError_t>(code)); }
// a non-blocking stream on `dev` owned by the caller (the current device is left as it was)
GX_API int gx_rt_stream_create(int dev, void** out) {
  *out = nullptr;
  int cur = 0;
  cudaGetDevice(&cur);
  cudaError_t e = cudaSetDevice(dev);
  cudaStream_t s = nullptr;
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
  cudaSetDevice(cur);
  if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
  *out = s;
  return 0;
}
GX_API int gx_rt_stream_destroy(void* stream) { return stream ? (int)cudaStreamDestroy(static_cast<cudaStream_t>(stream)) : 0; }
// CUDA graphs of one stream's work.  Capture is thread-local: allocations and other calls made meanwhile by other threads (another
// predictor's create, the pool's cudaMalloc) neither join nor invalidate it.
GX_API int gx_rt_graph_begin(void* stream) { return (int)cudaStreamBeginCapture(static_cast<cudaStream_t>(stream), cudaStreamCaptureModeThreadLocal); }
// ends the capture and instantiates it; on failure *out is null and the capture is over
GX_API int gx_rt_graph_end(void* stream, void** out) {
  *out = nullptr;
  cudaGraph_t g = nullptr;
  cudaError_t e = cudaStreamEndCapture(static_cast<cudaStream_t>(stream), &g);
  if (e != cudaSuccess) { cudaGetLastError(); if (g) cudaGraphDestroy(g); return (int)e; }
  cudaGraphExec_t x = nullptr;
  e = cudaGraphInstantiateWithFlags(&x, g, 0);
  cudaGraphDestroy(g);
  if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
  *out = x;
  return 0;
}
GX_API int gx_rt_graph_launch(void* exec, void* stream) { return (int)cudaGraphLaunch(static_cast<cudaGraphExec_t>(exec), static_cast<cudaStream_t>(stream)); }
GX_API int gx_rt_graph_destroy(void* exec) { return exec ? (int)cudaGraphExecDestroy(static_cast<cudaGraphExec_t>(exec)) : 0; }
// copy between the memory of two devices (directly over NVLink / PCIe when peer access is possible, staged by the driver otherwise),
// ordered on `stream`
GX_API int gx_rt_memcpy_peer(void* dst, int dst_dev, const void* src, int src_dev, unsigned long long bytes, void* stream) {
  if (bytes == 0) return 0;
  return (int)cudaMemcpyPeerAsync(dst, dst_dev, src, src_dev, bytes, static_cast<cudaStream_t>(stream));
}
// makes `waiter` wait for the work queued so far on `signaller` (a stream of device signaller_dev) without blocking the host: an event of
// the library, one per signalling stream, is recorded there and waited on.  Re-recording it later does not affect waits already enqueued.
GX_API int gx_rt_stream_join(void* waiter, void* signaller, int signaller_dev) {
  if (waiter == signaller) return 0;
  static std::mutex mu;
  static std::vector<std::pair<void*, cudaEvent_t>> events;
  std::lock_guard<std::mutex> lk(mu);
  cudaEvent_t ev = nullptr;
  for (auto& e : events) if (e.first == signaller) ev = e.second;
  int cur = 0;
  cudaGetDevice(&cur);
  cudaError_t e = cudaSetDevice(signaller_dev);
  if (e == cudaSuccess && !ev) {
    e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (e == cudaSuccess) events.emplace_back(signaller, ev);
  }
  if (e == cudaSuccess) e = cudaEventRecord(ev, static_cast<cudaStream_t>(signaller));
  if (e == cudaSuccess) e = cudaStreamWaitEvent(static_cast<cudaStream_t>(waiter), ev, 0);
  cudaSetDevice(cur);
  if (e != cudaSuccess) cudaGetLastError();
  return (int)e;
}
// page-locked host memory (portable: usable by every device's copies), for staging buffers whose copies must stay asynchronous
GX_API int gx_rt_host_alloc(unsigned long long bytes, void** out) {
  *out = nullptr;
  const cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable);
  if (e != cudaSuccess) { cudaGetLastError(); *out = nullptr; }
  return (int)e;
}
GX_API int gx_rt_host_free(void* p) { return p ? (int)cudaFreeHost(p) : 0; }

// ================================================================================================ graph operator kernels
GX_API int gx_axpy(float* y, const float* x, float a, long long n, cudaStream_t s) {
  if (n <= 0) return 0;
  return launch_pdl(axpy_kernel, dim3(blocks_for(n)), dim3(kThreads), 0, s, y, x, a, n);
}
GX_API int gx_add_scalar(float* y, float c, long long n, cudaStream_t s) {
  if (n <= 0) return 0;
  return launch_pdl(add_scalar_kernel, dim3(blocks_for(n)), dim3(kThreads), 0, s, y, c, n);
}
GX_API int gx_mul_add(float* y, const float* a, const float* b, long long n, cudaStream_t s) {
  if (n <= 0) return 0;
  return launch_pdl(mul_add_kernel, dim3(blocks_for(n)), dim3(kThreads), 0, s, y, a, b, n);
}
GX_API int gx_rows_to_nchw(const float* rows, float* y, int N, int C, int HW, long long ld, int accumulate, cudaStream_t s) {
  return launch_pdl(rows_to_nchw_kernel, dim3(blocks_for((long long)N * C * HW)), dim3(kThreads), 0, s, rows, y, N, C, HW, ld, accumulate);
}
GX_API int gx_act_fwd(int kind, const float* x, float* y, long long n, float slope, cudaStream_t s) {
  if (kind < 0 || kind > 5) return -1;
  return launch_pdl(act_fwd_kernel, dim3(blocks_for(n)), dim3(kThreads), 0, s, kind, x, y, n, slope);
}
GX_API int gx_act_bwd(int kind, const float* x, const float* y, const float* dy, float* dx, long long n, float slope, cudaStream_t s) {
  if (kind < 0 || kind > 5) return -1;
  return launch_pdl(act_bwd_kernel, dim3(blocks_for(n)), dim3(kThreads), 0, s, kind, x, y, dy, dx, n, slope);
}
// type 0 max (idx receives the arg-max offset in its plane, -1 for an empty window), 1 avg, 2 sum
GX_API int gx_pool_fwd(int type, const float* x, float* y, int* idx, long long NC, int H, int W, int OH, int OW, int kh, int kw, int sh, int sw, int ph,
                       int pw, int count_pad, cudaStream_t s) {
  if (type < 0 || type > 2 || (type == 0 && !idx)) return -1;
  const PoolGeom g{H, W, OH, OW, kh, kw, sh, sw, ph, pw, type, count_pad};
  return launch_pdl(pool_fwd_kernel, dim3(blocks_for(NC * OH * OW)), dim3(kThreads), 0, s, x, y, idx, NC, g);
}
GX_API int gx_pool_bwd(int type, const float* dy, const int* idx, float* dx, long long NC, int H, int W, int OH, int OW, int kh, int kw, int sh, int sw,
                       int ph, int pw, int count_pad, cudaStream_t s) {
  if (type < 0 || type > 2 || (type == 0 && !idx)) return -1;
  const PoolGeom g{H, W, OH, OW, kh, kw, sh, sw, ph, pw, type, count_pad};
  return launch_pdl(pool_bwd_kernel, dim3(blocks_for(NC * OH * OW)), dim3(kThreads), 0, s, dy, idx, dx, NC, g);
}
// kind 0 add, 1 sub, 2 mul, 3 div, 4 maximum, 5 minimum (gx_binary_bwd: 0-2).  out_dims: the output extents (ndim <= 8); ls / rs: element
// strides of each operand, 0 on broadcast axes
GX_API int gx_binary_fwd(int kind, const float* l, const float* r, float* y, int ndim, const long long* out_dims, const long long* ls, const long long* rs,
                         cudaStream_t s) {
  if (kind < 0 || kind > 5 || ndim < 1 || ndim > kMaxDims) return -1;
  Bcast b; b.ndim = ndim;
  long long n = 1;
  for (int d = 0; d < ndim; ++d) { b.dims[d] = out_dims[d]; b.ls[d] = ls[d]; b.rs[d] = rs[d]; n *= out_dims[d]; }
  return launch_pdl(binary_fwd_kernel, dim3(blocks_for(n)), dim3(kThreads), 0, s, kind, l, r, y, n, b);
}
GX_API int gx_binary_bwd(int kind, const float* l, const float* r, const float* dy, float* dl, float* dr, int ndim, const long long* out_dims,
                         const long long* ls, const long long* rs, cudaStream_t s) {
  if (kind < 0 || kind > 2 || ndim < 1 || ndim > kMaxDims) return -1;
  Bcast b; b.ndim = ndim;
  long long n = 1;
  int lb = 0, rb = 0;
  for (int d = 0; d < ndim; ++d) {
    b.dims[d] = out_dims[d]; b.ls[d] = ls[d]; b.rs[d] = rs[d]; n *= out_dims[d];
    if (out_dims[d] > 1 && ls[d] == 0) lb = 1;
    if (out_dims[d] > 1 && rs[d] == 0) rb = 1;
  }
  return launch_pdl(binary_bwd_kernel, dim3(blocks_for(n)), dim3(kThreads), 0, s, kind, l, r, dy, dl, dr, n, b, lb, rb);
}
GX_API int gx_strided_copy(const float* src, float* dst, long long outer, long long len, long long src_stride, long long dst_stride, int accumulate,
                           cudaStream_t s) {
  if (outer <= 0 || len <= 0) return 0;
  return launch_pdl(strided_copy_kernel, dim3(blocks_for(outer * len)), dim3(kThreads), 0, s, src, dst, outer, len, src_stride, dst_stride, accumulate);
}
// mask receives 1/(1-p) for kept elements and 0 for dropped ones; backward is gx_mul_add(dx, dy, mask)
GX_API int gx_dropout_fwd(const float* x, float* y, float* mask, long long n, float p, unsigned int seed, unsigned int step, cudaStream_t s) {
  if (!(p > 0.f && p < 1.f)) return -1;
  return launch_pdl(dropout_fwd_kernel, dim3(blocks_for(n)), dim3(kThreads), 0, s, x, y, mask, n, p, seed, step);
}
GX_API int gx_softmax_fwd(const float* x, float* y, long long outer, int C, long long inner, int log_out, cudaStream_t s) {
  return launch_pdl(softmax_fwd_kernel, dim3(blocks_for(outer * inner * 32)), dim3(kThreads), 0, s, x, y, outer, C, inner, log_out);
}
GX_API int gx_softmax_bwd(const float* y, const float* dy, float* dx, long long outer, int C, long long inner, int log_out, cudaStream_t s) {
  return launch_pdl(softmax_bwd_kernel, dim3(blocks_for(outer * inner * 32)), dim3(kThreads), 0, s, y, dy, dx, outer, C, inner, log_out);
}
GX_API int gx_softmax_output_bwd(const float* y, const float* label, float* dx, long long outer, int C, long long inner, float grad_scale, int use_ignore,
                                 float ignore, int norm, cudaStream_t s) {
  return launch_pdl(softmax_output_bwd_kernel, dim3(blocks_for(outer * inner * C, 148LL * 4)), dim3(kThreads), 0, s, y, label, dx, outer, C, inner, grad_scale,
                    use_ignore, ignore, norm);
}
GX_API int gx_bn_global_bwd(const float* x, const float* dy, const float* gamma, const float* mean, const float* var, float eps, float* dx, float* dgamma,
                            float* dbeta, int N, int C, int HW, cudaStream_t s) {
  return launch_pdl(bn_global_bwd_kernel, dim3(C), dim3(kThreads), 0, s, x, dy, gamma, mean, var, eps, dx, dgamma, dbeta, N, C, HW);
}
