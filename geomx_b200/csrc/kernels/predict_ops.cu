// Device kernels of the native predictor (csrc/runtime/predict_device.h) for the operators the graph executor's kernels (graph_ops.cu) do
// not cover: one elementwise map for the unary / activation / scalar / clip family, the per-channel affine of BatchNorm at inference on any
// axis, transpose of up to 8 axes, the Embedding gather and a dilated im2col.  Every kernel starts with pdl_wait() and is launched with
// launch_pdl(), so a captured forward keeps programmatic dependencies between consecutive operators.
#include <cuda_runtime.h>

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

// ------------------------------------------------------------------------------------------------ elementwise map
// kind  0..10: relu, sigmoid, tanh, exp, log, sqrt, abs, negative, square, softsign, softrelu (predict.h UnaryKind order)
//      11: leaky (a = slope), 12: elu (a = slope), 13: clip to [a, b]
//      14..19: x + a, x - a, x * a, x / a, a - x, a / x (predict.h ScalarKind order)
// x and y may be the same buffer: the planner runs these operators in place.
__device__ __forceinline__ float map_f(int k, float v, float a, float b) {
  switch (k) {
    case 0: return v > 0.f ? v : 0.f;
    case 1: return 1.f / (1.f + expf(-v));
    case 2: return tanhf(v);
    case 3: return expf(v);
    case 4: return logf(v);
    case 5: return sqrtf(v);
    case 6: return fabsf(v);
    case 7: return -v;
    case 8: return v * v;
    case 9: return v / (1.f + fabsf(v));
    case 10: return v > 20.f ? v : log1pf(expf(v));
    case 11: return v > 0.f ? v : a * v;
    case 12: return v > 0.f ? v : a * (expf(v) - 1.f);
    case 13: { const float lo = v < a ? a : v; return b < lo ? b : lo; }       // std::min(std::max(v, a), b)
    case 14: return v + a;
    case 15: return v - a;
    case 16: return v * a;
    case 17: return v / a;
    case 18: return a - v;
    default: return a / v;
  }
}
__global__ void map_kernel(int kind, const float* x, float* y, long long n, float a, float b) {
  pdl_wait();
  GRID_STRIDE(i, n) y[i] = map_f(kind, x[i], a, b);
}

// ------------------------------------------------------------------------------------------------ per-channel affine over (outer, C, inner)
// y = x * scale[c] + shift[c]: BatchNorm at inference with scale / shift folded on the host.  In place allowed.
__global__ void channel_affine_kernel(const float* x, float* y, const float* __restrict__ scale, const float* __restrict__ shift, long long n, int C,
                                      long long inner) {
  pdl_wait();
  GRID_STRIDE(i, n) {
    const int c = (int)((i / inner) % C);
    y[i] = x[i] * scale[c] + shift[c];
  }
}

// ------------------------------------------------------------------------------------------------ transpose
constexpr int kMaxDims = 8;
struct Perm {
  int ndim;
  long long out_dims[kMaxDims];     // output extents
  long long in_step[kMaxDims];      // input element stride of each output axis
};
// the innermost axis stays innermost: output-order gather, reads of consecutive threads are contiguous along that axis
__global__ void transpose_gather_kernel(const float* __restrict__ x, float* __restrict__ y, long long n, Perm p) {
  pdl_wait();
  GRID_STRIDE(i, n) {
    long long f = i, src = 0;
    for (int d = p.ndim - 1; d >= 0; --d) { const long long c = f % p.out_dims[d]; f /= p.out_dims[d]; src += c * p.in_step[d]; }
    y[i] = x[src];
  }
}
// the innermost axis moves: a batch of 2-D transposes between the input's innermost axis (extent X, output stride ox) and the input axis
// that becomes the output's innermost (extent Y, input stride iy).  A 32 x 32 tile goes through shared memory so that reads run along the
// input's innermost axis and writes along the output's.  The other axes (at most 6) enumerate the batch.
struct Tile2D {
  long long X, Y, iy, ox, batch;
  int nb;
  long long b_dims[kMaxDims], b_in[kMaxDims], b_out[kMaxDims];
};
__global__ void __launch_bounds__(256) transpose_tiled_kernel(const float* __restrict__ x, float* __restrict__ y, Tile2D t) {
  pdl_wait();
  __shared__ float tile[32][33];
  const long long x0 = (long long)blockIdx.x * 32, y0 = (long long)blockIdx.y * 32;
  for (long long b = blockIdx.z; b < t.batch; b += gridDim.z) {
    long long f = b, in_base = 0, out_base = 0;
    for (int d = t.nb - 1; d >= 0; --d) { const long long c = f % t.b_dims[d]; f /= t.b_dims[d]; in_base += c * t.b_in[d]; out_base += c * t.b_out[d]; }
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
      const long long yy = y0 + r, xx = x0 + threadIdx.x;
      if (yy < t.Y && xx < t.X) tile[r][threadIdx.x] = x[in_base + yy * t.iy + xx];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
      const long long xx = x0 + r, yy = y0 + threadIdx.x;
      if (xx < t.X && yy < t.Y) y[out_base + xx * t.ox + yy] = tile[threadIdx.x][r];
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------ Embedding
// y[r, :] = w[clamp(trunc(idx[r]), 0, V - 1), :]
__global__ void embedding_kernel(const float* __restrict__ idx, const float* __restrict__ w, float* __restrict__ y, long long rows, long long V, long long D) {
  pdl_wait();
  const long long n = rows * D;
  GRID_STRIDE(i, n) {
    const long long r = i / D, j = i - r * D;
    const float f = idx[r];
    const long long k = f >= (float)(V - 1) ? V - 1 : f < 1.f ? 0 : (long long)f;
    y[i] = w[k * D + j];
  }
}

// ------------------------------------------------------------------------------------------------ dilated im2col
// col[(n * OH + oh) * OW + ow][(c * KH + kh) * KW + kw] (row stride ldc, columns K..ldc zero) = x[n, c, oh*sh - ph + kh*dh, ow*sw - pw + kw*dw]
__global__ void __launch_bounds__(256) im2col_dilated_kernel(const float* __restrict__ x, float* __restrict__ col, int C, int H, int W, int KH, int KW,
                                                             int OH, int OW, int sh, int sw, int ph, int pw, int dh, int dw, int K, int ldc, long long total) {
  pdl_wait();
  GRID_STRIDE(i, total) {
    const int k = (int)(i % ldc);
    const long long row = i / ldc;
    float v = 0.f;
    if (k < K) {
      const int kw = k % KW, kh = (k / KW) % KH, c = k / (KW * KH);
      const int ow = (int)(row % OW), oh = (int)((row / OW) % OH);
      const long long n = row / ((long long)OW * OH);
      const int h = oh * sh - ph + kh * dh, w = ow * sw - pw + kw * dw;
      if (h >= 0 && h < H && w >= 0 && w < W) v = __ldg(x + ((n * C + c) * H + h) * W + w);
    }
    col[i] = v;
  }
}

}  // namespace

// ================================================================================================ entry points
GX_API int gx_map_fwd(int kind, const float* x, float* y, long long n, float a, float b, cudaStream_t s) {
  if (kind < 0 || kind > 19) return -1;
  if (n <= 0) return 0;
  return launch_pdl(map_kernel, dim3(blocks_for(n)), dim3(kThreads), 0, s, kind, x, y, n, a, b);
}
GX_API int gx_channel_affine(const float* x, float* y, const float* scale, const float* shift, long long outer, int C, long long inner, cudaStream_t s) {
  const long long n = outer * C * inner;
  if (C < 1 || inner < 1) return -1;
  if (n <= 0) return 0;
  return launch_pdl(channel_affine_kernel, dim3(blocks_for(n)), dim3(kThreads), 0, s, x, y, scale, shift, n, C, inner);
}
// y = x.transpose(axes): in_dims are the input extents, axes[d] the input axis that becomes output axis d (a permutation of 0..ndim-1)
GX_API int gx_transpose(const float* x, float* y, int ndim, const long long* in_dims, const int* axes, cudaStream_t s) {
  if (ndim < 1 || ndim > kMaxDims) return -1;
  long long in_stride[kMaxDims], out_dims[kMaxDims], out_stride[kMaxDims];
  int seen[kMaxDims] = {0};
  long long n = 1;
  for (int d = ndim - 1; d >= 0; --d) { in_stride[d] = n; n *= in_dims[d]; }
  for (int d = 0; d < ndim; ++d) {
    if (axes[d] < 0 || axes[d] >= ndim || seen[axes[d]]) return -1;
    seen[axes[d]] = 1; out_dims[d] = in_dims[axes[d]];
  }
  if (n <= 0) return 0;
  long long acc = 1;
  for (int d = ndim - 1; d >= 0; --d) { out_stride[d] = acc; acc *= out_dims[d]; }
  const int last = ndim - 1;
  if (axes[last] == last || in_dims[last] == 1 || (out_dims[last] + 31) / 32 > 65535) {
    Perm p; p.ndim = ndim;
    for (int d = 0; d < ndim; ++d) { p.out_dims[d] = out_dims[d]; p.in_step[d] = in_stride[axes[d]]; }
    return launch_pdl(transpose_gather_kernel, dim3(blocks_for(n)), dim3(kThreads), 0, s, x, y, n, p);
  }
  Tile2D t;
  int jo = 0;                                                  // output position of the input's innermost axis
  for (int d = 0; d < ndim; ++d) if (axes[d] == last) jo = d;
  t.X = in_dims[last]; t.Y = out_dims[last]; t.iy = in_stride[axes[last]]; t.ox = out_stride[jo];
  t.nb = 0; t.batch = 1;
  for (int d = 0; d < ndim; ++d) {
    if (d == jo || d == last) continue;
    t.b_dims[t.nb] = out_dims[d]; t.b_in[t.nb] = in_stride[axes[d]]; t.b_out[t.nb] = out_stride[d]; ++t.nb;
    t.batch *= out_dims[d];
  }
  const long long gz = t.batch < 65535 ? t.batch : 65535;
  return launch_pdl(transpose_tiled_kernel, dim3((unsigned)((t.X + 31) / 32), (unsigned)((t.Y + 31) / 32), (unsigned)gz), dim3(32, 8), 0, s, x, y, t);
}
GX_API int gx_embedding_fwd(const float* idx, const float* w, float* y, long long rows, long long V, long long D, cudaStream_t s) {
  if (V < 1 || D < 1) return -1;
  if (rows <= 0) return 0;
  return launch_pdl(embedding_kernel, dim3(blocks_for(rows * D)), dim3(kThreads), 0, s, idx, w, y, rows, V, D);
}
// gx_im2col with a dilation (dh, dw); the column layout is gx_im2col's
GX_API int gx_im2col_dilated(const float* x, float* col, int N, int C, int H, int W, int KH, int KW, int sh, int sw, int ph, int pw, int dh, int dw, int ldc,
                             cudaStream_t s) {
  const int OH = (H + 2 * ph - dh * (KH - 1) - 1) / sh + 1, OW = (W + 2 * pw - dw * (KW - 1) - 1) / sw + 1;
  const int K = C * KH * KW;
  if (OH < 1 || OW < 1 || ldc < K) return -1;
  const long long total = (long long)N * OH * OW * ldc;
  return launch_pdl(im2col_dilated_kernel, dim3(blocks_for(total, 148LL * 16)), dim3(kThreads), 0, s, x, col, C, H, W, KH, KW, OH, OW, sh, sw, ph, pw, dh,
                    dw, K, ldc, total);
}
