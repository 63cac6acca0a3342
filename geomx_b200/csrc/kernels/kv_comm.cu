// Reduction kernels of the C API's in-process KVStores (csrc/runtime/kvstore_nd.h) for sm_100a.
//
// gx_kv_sum_quantize sums up to 8 fp32 arrays left to right, acc = ((in0 + in1) + in2) + ..., the order the host reduction uses, so a device
// store and a host store agree bit for bit.  With thr > 0 the same launch adds the residual and emits 2-bit words with the bit layout of
// hips/gradient_compression.h Quantize2Bit and compress.cu gx_quantize_2bit (value j of a word in byte j>>2, bit pair 6-2*(j&3)).
// gx_kv_dequant_sum is the receiving side of the reference's compressed inter-GPU reduce (src/kvstore/comm.h:545-589): it dequantises up to
// 8 word arrays and sums them, again left to right, in one launch.  Callers chain longer lists: the output of one launch is input 0 of the
// next (sum) or accumulated into (dequant), which keeps the order.
//
// One thread owns one 16-value group, i.e. one output word: it reads each input with four 128-bit loads when the group is whole and every
// pointer is 16-byte aligned, and element by element otherwise (the tail, odd offsets).
#include "common.cuh"

namespace {

constexpr int kMaxIn = 8;
constexpr int kThreads = 256;

struct SumArgs {
  const float* in[kMaxIn];
  int cnt;
};
struct WordArgs {
  const uint32_t* in[kMaxIn];
  int cnt;
};

__device__ __forceinline__ int word_shift(int j) { return ((j >> 2) << 3) + (6 - 2 * (j & 3)); }

__device__ __forceinline__ uint32_t quantize_one(float v, float* res, float thr, int j) {
  float r = *res + v;
  uint32_t code = 0;
  if (r >= thr) { code = 3; r -= thr; }
  else if (r <= -thr) { code = 2; r += thr; }
  *res = r;
  return code << word_shift(j);
}

// out may be null (quantise only) and may alias in[0]; residual / words are used when thr > 0
__global__ void __launch_bounds__(kThreads) kv_sum_quantize_kernel(SumArgs a, float* out, float* residual, uint32_t* words, long long n, float thr,
                                                                   int vec) {
  gx::pdl_wait();
  const long long groups = (n + 15) / 16;
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < groups; g += (long long)gridDim.x * blockDim.x) {
    const long long base = g * 16;
    float acc[16];
    if (vec && base + 16 <= n) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 v = reinterpret_cast<const float4*>(a.in[0] + base)[q];
        acc[4 * q] = v.x; acc[4 * q + 1] = v.y; acc[4 * q + 2] = v.z; acc[4 * q + 3] = v.w;
      }
#pragma unroll
      for (int s = 1; s < kMaxIn; ++s) {
        if (s >= a.cnt) break;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 v = reinterpret_cast<const float4*>(a.in[s] + base)[q];
          acc[4 * q] += v.x; acc[4 * q + 1] += v.y; acc[4 * q + 2] += v.z; acc[4 * q + 3] += v.w;
        }
      }
      if (out) {
#pragma unroll
        for (int q = 0; q < 4; ++q) reinterpret_cast<float4*>(out + base)[q] = make_float4(acc[4 * q], acc[4 * q + 1], acc[4 * q + 2], acc[4 * q + 3]);
      }
      if (thr > 0.f) {
        float4 r[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) r[q] = reinterpret_cast<const float4*>(residual + base)[q];
        float* rf = reinterpret_cast<float*>(r);
        uint32_t word = 0;
#pragma unroll
        for (int j = 0; j < 16; ++j) word |= quantize_one(acc[j], rf + j, thr, j);
#pragma unroll
        for (int q = 0; q < 4; ++q) reinterpret_cast<float4*>(residual + base)[q] = r[q];
        words[g] = word;
      }
    } else {
      const int m = (int)(n - base < 16 ? n - base : 16);
      uint32_t word = 0;
      for (int j = 0; j < m; ++j) {
        float v = a.in[0][base + j];
#pragma unroll
        for (int s = 1; s < kMaxIn; ++s) {
          if (s >= a.cnt) break;
          v += a.in[s][base + j];
        }
        if (out) out[base + j] = v;
        if (thr > 0.f) word |= quantize_one(v, residual + base + j, thr, j);
      }
      if (thr > 0.f) words[g] = word;
    }
  }
}

__global__ void __launch_bounds__(kThreads) kv_dequant_sum_kernel(WordArgs a, float* __restrict__ out, long long n, float thr, int accumulate, int vec) {
  gx::pdl_wait();
  const long long groups = (n + 15) / 16;
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < groups; g += (long long)gridDim.x * blockDim.x) {
    const long long base = g * 16;
    float acc[16];
    const bool whole = vec && base + 16 <= n;
    if (accumulate) {
      if (whole) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 v = reinterpret_cast<const float4*>(out + base)[q];
          acc[4 * q] = v.x; acc[4 * q + 1] = v.y; acc[4 * q + 2] = v.z; acc[4 * q + 3] = v.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[j] = base + j < n ? out[base + j] : 0.f;
      }
    }
#pragma unroll
    for (int s = 0; s < kMaxIn; ++s) {
      if (s >= a.cnt) break;
      const uint32_t w = a.in[s][g];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const uint32_t code = (w >> word_shift(j)) & 3u;
        const float v = code == 3 ? thr : (code == 2 ? -thr : 0.f);
        acc[j] = (s == 0 && !accumulate) ? v : acc[j] + v;
      }
    }
    if (whole) {
#pragma unroll
      for (int q = 0; q < 4; ++q) reinterpret_cast<float4*>(out + base)[q] = make_float4(acc[4 * q], acc[4 * q + 1], acc[4 * q + 2], acc[4 * q + 3]);
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j) if (base + j < n) out[base + j] = acc[j];
    }
  }
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline unsigned grid_for_groups(long long n) {
  const long long g = (n + 15) / 16;
  const long long b = (g + kThreads - 1) / kThreads;
  return (unsigned)(b < 1 ? 1 : b > 148LL * 16 ? 148LL * 16 : b);
}

}  // namespace

// out[i] = in[0][i] + in[1][i] + ... (left to right), 1 <= cnt <= 8.  thr > 0: also r = residual[i] + out[i], 2-bit code of r into words
// (ceil(n/16) uint32), residual[i] = r minus the transmitted value.  out may be null when only the words are wanted, and may equal inputs[0].
GX_API int gx_kv_sum_quantize(float* out, const float* const* inputs, int cnt, long long n, float* residual, void* words, float thr, cudaStream_t s) {
  if (cnt < 1 || cnt > kMaxIn || n < 0 || (thr > 0.f && (!residual || !words)) || (!(thr > 0.f) && !out)) return -1;
  if (n == 0) return 0;
  SumArgs a{};
  bool vec = out == nullptr || aligned16(out);
  for (int i = 0; i < cnt; ++i) { a.in[i] = inputs[i]; vec = vec && aligned16(inputs[i]); }
  a.cnt = cnt;
  if (thr > 0.f) vec = vec && aligned16(residual);
  return gx::launch_pdl(kv_sum_quantize_kernel, dim3(grid_for_groups(n)), dim3(kThreads), 0, s, a, out, residual, reinterpret_cast<uint32_t*>(words), n,
                        thr > 0.f ? thr : 0.f, vec ? 1 : 0);
}
// out[i] (+)= deq(words[0])[i] + deq(words[1])[i] + ... (left to right), 1 <= cnt <= 8; deq maps the codes 3 / 2 / 0 to thr / -thr / 0
GX_API int gx_kv_dequant_sum(float* out, const void* const* words, int cnt, long long n, float thr, int accumulate, cudaStream_t s) {
  if (cnt < 1 || cnt > kMaxIn || n < 0 || !out) return -1;
  if (n == 0) return 0;
  WordArgs a{};
  for (int i = 0; i < cnt; ++i) a.in[i] = static_cast<const uint32_t*>(words[i]);
  a.cnt = cnt;
  return gx::launch_pdl(kv_dequant_sum_kernel, dim3(grid_for_groups(n)), dim3(kThreads), 0, s, a, out, n, thr, accumulate, aligned16(out) ? 1 : 0);
}
