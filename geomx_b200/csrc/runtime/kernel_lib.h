// The sm_100a kernel library (lib/libgeomx_kernels.so) as seen from the C API.  The C API links neither libcudart nor the kernel library, so
// that it loads on machines without CUDA: the first device request dlopen()s the kernel library that sits next to the C API's own binary
// (libgeomx_capi.so and _C*.so both live in geomx_b200/lib/) and resolves the gx_* entry points below into one table.  Streams are opaque
// pointers here; no CUDA header is included.
#pragma once
#include <dlfcn.h>

#include <cstdint>
#include <mutex>
#include <stdexcept>
#include <string>

namespace gxrt {
namespace kern {

using Stream = void*;

struct Lib {
  // runtime (graph_ops.cu)
  int (*device_count)(int*);
  int (*set_device)(int);
  void* (*stream)(int);
  int (*memcpy)(void*, const void*, unsigned long long, int, void*);
  int (*memset)(void*, int, unsigned long long, void*);
  int (*stream_sync)(void*);
  const char* (*error_string)(int);
  int (*stream_create)(int, void**);
  int (*stream_destroy)(void*);
  int (*graph_begin)(void*);
  int (*graph_end)(void*, void**);
  int (*graph_launch)(void*, void*);
  int (*graph_destroy)(void*);
  int (*memcpy_peer)(void*, int, const void*, int, unsigned long long, void*);
  int (*stream_join)(void*, void*, int);
  int (*host_alloc)(unsigned long long, void**);
  int (*host_free)(void*);
  // device memory pool (storage_gpu.cu)
  void* (*pool_alloc)(int, uint64_t, void*);
  int (*pool_free)(int, void*, void*);
  // existing kernels
  int (*gemm_tf32)(const float*, long long, int, const float*, long long, int, int, int, int, float*, long long, const float*, const float*, long long,
                   float*, int, int, int, int, float, int, Stream);
  int (*gemm_simt)(const float*, long long, int, const float*, long long, int, int, int, int, float*, long long, const float*, const float*, long long,
                   float*, int, int, int, int, float, Stream);
  int (*im2col)(const float*, float*, int, int, int, int, int, int, int, int, int, int, int, Stream);
  int (*col2im)(const float*, float*, int, int, int, int, int, int, int, int, int, int, int, Stream);
  int (*nchw_to_rows)(const float*, float*, int, int, int, Stream);
  int (*colsum)(const float*, float*, long long, int, long long, int, Stream);
  int (*bn_fwd)(const float*, const float*, const float*, float*, float*, float*, float*, float*, int, int, int, int, float, float, Stream);
  int (*bn_bwd)(const float*, const float*, const float*, const float*, const float*, float*, float*, float*, int, int, int, Stream);
  int (*depthwise_fwd)(const float*, const float*, const float*, float*, int, int, int, int, int, int, int, int, int, int, int, Stream);
  int (*depthwise_dgrad)(const float*, const float*, float*, int, int, int, int, int, int, int, int, int, int, Stream);
  int (*depthwise_wgrad)(const float*, const float*, float*, float*, int, int, int, int, int, int, int, int, int, int, Stream);
  int (*single_opt)(int, float*, const float*, float*, float*, long long, float, float, float, float, float, float, float, float, float, Stream);
  int (*nary_sum)(float*, const float* const*, int, long long, Stream);
  // graph operator kernels (graph_ops.cu)
  int (*axpy)(float*, const float*, float, long long, Stream);
  int (*add_scalar)(float*, float, long long, Stream);
  int (*mul_add)(float*, const float*, const float*, long long, Stream);
  int (*rows_to_nchw)(const float*, float*, int, int, int, long long, int, Stream);
  int (*act_fwd)(int, const float*, float*, long long, float, Stream);
  int (*act_bwd)(int, const float*, const float*, const float*, float*, long long, float, Stream);
  int (*pool_fwd)(int, const float*, float*, int*, long long, int, int, int, int, int, int, int, int, int, int, int, Stream);
  int (*pool_bwd)(int, const float*, const int*, float*, long long, int, int, int, int, int, int, int, int, int, int, int, Stream);
  int (*binary_fwd)(int, const float*, const float*, float*, int, const long long*, const long long*, const long long*, Stream);
  int (*binary_bwd)(int, const float*, const float*, const float*, float*, float*, int, const long long*, const long long*, const long long*, Stream);
  int (*strided_copy)(const float*, float*, long long, long long, long long, long long, int, Stream);
  int (*dropout_fwd)(const float*, float*, float*, long long, float, unsigned, unsigned, Stream);
  int (*softmax_fwd)(const float*, float*, long long, int, long long, int, Stream);
  int (*softmax_bwd)(const float*, const float*, float*, long long, int, long long, int, Stream);
  int (*softmax_output_bwd)(const float*, const float*, float*, long long, int, long long, float, int, float, int, Stream);
  int (*bn_global_bwd)(const float*, const float*, const float*, const float*, const float*, float, float*, float*, float*, int, int, int, Stream);
  // native predictor kernels (predict_ops.cu)
  int (*map_fwd)(int, const float*, float*, long long, float, float, Stream);
  int (*channel_affine)(const float*, float*, const float*, const float*, long long, int, long long, Stream);
  int (*transpose)(const float*, float*, int, const long long*, const int*, Stream);
  int (*embedding_fwd)(const float*, const float*, float*, long long, long long, long long, Stream);
  int (*im2col_dilated)(const float*, float*, int, int, int, int, int, int, int, int, int, int, int, int, int, Stream);
  // KVStore reductions (kv_comm.cu)
  int (*kv_sum_quantize)(float*, const float* const*, int, long long, float*, void*, float, Stream);
  int (*kv_dequant_sum)(float*, const void* const*, int, long long, float, int, Stream);
};

namespace detail {
inline void KernLibAnchor() {}        // dladdr target: any symbol of the binary this header is compiled into

template <typename T>
void Resolve(void* h, const char* name, T* slot) {
  void* p = dlsym(h, name);
  if (!p) throw std::runtime_error(std::string("the kernel library lacks ") + name + " (rebuild with python -m geomx_b200.build)");
  *slot = reinterpret_cast<T>(p);
}

inline Lib LoadLib() {
  Dl_info info{};
  if (!dladdr(reinterpret_cast<void*>(&KernLibAnchor), &info) || !info.dli_fname) throw std::runtime_error("cannot locate the C API library on disk");
  std::string dir = info.dli_fname;
  const size_t slash = dir.rfind('/');
  dir = slash == std::string::npos ? "." : dir.substr(0, slash);
  const std::string path = dir + "/libgeomx_kernels.so";
  void* h = dlopen(path.c_str(), RTLD_NOW | RTLD_LOCAL);
  if (!h) {
    const char* e = dlerror();
    throw std::runtime_error("cannot load the kernel library " + path + ": " + (e ? e : "unknown error"));
  }
  Lib L{};
  Resolve(h, "gx_rt_device_count", &L.device_count);
  Resolve(h, "gx_rt_set_device", &L.set_device);
  Resolve(h, "gx_rt_stream", &L.stream);
  Resolve(h, "gx_rt_memcpy", &L.memcpy);
  Resolve(h, "gx_rt_memset", &L.memset);
  Resolve(h, "gx_rt_stream_sync", &L.stream_sync);
  Resolve(h, "gx_rt_error_string", &L.error_string);
  Resolve(h, "gx_rt_stream_create", &L.stream_create);
  Resolve(h, "gx_rt_stream_destroy", &L.stream_destroy);
  Resolve(h, "gx_rt_graph_begin", &L.graph_begin);
  Resolve(h, "gx_rt_graph_end", &L.graph_end);
  Resolve(h, "gx_rt_graph_launch", &L.graph_launch);
  Resolve(h, "gx_rt_graph_destroy", &L.graph_destroy);
  Resolve(h, "gx_rt_memcpy_peer", &L.memcpy_peer);
  Resolve(h, "gx_rt_stream_join", &L.stream_join);
  Resolve(h, "gx_rt_host_alloc", &L.host_alloc);
  Resolve(h, "gx_rt_host_free", &L.host_free);
  Resolve(h, "gx_gpu_pool_alloc", &L.pool_alloc);
  Resolve(h, "gx_gpu_pool_free", &L.pool_free);
  Resolve(h, "gx_gemm_tf32", &L.gemm_tf32);
  Resolve(h, "gx_gemm_simt", &L.gemm_simt);
  Resolve(h, "gx_im2col", &L.im2col);
  Resolve(h, "gx_col2im", &L.col2im);
  Resolve(h, "gx_nchw_to_rows", &L.nchw_to_rows);
  Resolve(h, "gx_colsum", &L.colsum);
  Resolve(h, "gx_bn_fwd", &L.bn_fwd);
  Resolve(h, "gx_bn_bwd", &L.bn_bwd);
  Resolve(h, "gx_depthwise_fwd", &L.depthwise_fwd);
  Resolve(h, "gx_depthwise_dgrad", &L.depthwise_dgrad);
  Resolve(h, "gx_depthwise_wgrad", &L.depthwise_wgrad);
  Resolve(h, "gx_single_opt", &L.single_opt);
  Resolve(h, "gx_nary_sum", &L.nary_sum);
  Resolve(h, "gx_axpy", &L.axpy);
  Resolve(h, "gx_add_scalar", &L.add_scalar);
  Resolve(h, "gx_mul_add", &L.mul_add);
  Resolve(h, "gx_rows_to_nchw", &L.rows_to_nchw);
  Resolve(h, "gx_act_fwd", &L.act_fwd);
  Resolve(h, "gx_act_bwd", &L.act_bwd);
  Resolve(h, "gx_pool_fwd", &L.pool_fwd);
  Resolve(h, "gx_pool_bwd", &L.pool_bwd);
  Resolve(h, "gx_binary_fwd", &L.binary_fwd);
  Resolve(h, "gx_binary_bwd", &L.binary_bwd);
  Resolve(h, "gx_strided_copy", &L.strided_copy);
  Resolve(h, "gx_dropout_fwd", &L.dropout_fwd);
  Resolve(h, "gx_softmax_fwd", &L.softmax_fwd);
  Resolve(h, "gx_softmax_bwd", &L.softmax_bwd);
  Resolve(h, "gx_softmax_output_bwd", &L.softmax_output_bwd);
  Resolve(h, "gx_bn_global_bwd", &L.bn_global_bwd);
  Resolve(h, "gx_map_fwd", &L.map_fwd);
  Resolve(h, "gx_channel_affine", &L.channel_affine);
  Resolve(h, "gx_transpose", &L.transpose);
  Resolve(h, "gx_embedding_fwd", &L.embedding_fwd);
  Resolve(h, "gx_im2col_dilated", &L.im2col_dilated);
  Resolve(h, "gx_kv_sum_quantize", &L.kv_sum_quantize);
  Resolve(h, "gx_kv_dequant_sum", &L.kv_dequant_sum);
  return L;
}
}  // namespace detail

// the loaded table; throws (with the cause) when the library cannot be loaded.  A failed load is retried on the next call.
inline const Lib& Get() {
  static std::mutex mu;
  static bool loaded = false;
  static Lib lib;
  std::lock_guard<std::mutex> lk(mu);
  if (!loaded) { lib = detail::LoadLib(); loaded = true; }
  return lib;
}

// a CUDA status of the library -> exception naming the call
inline void Check(int rc, const char* what) {
  if (rc == 0) return;
  const char* msg = rc > 0 ? Get().error_string(rc) : "invalid arguments";
  throw std::runtime_error(std::string(what) + ": " + (msg ? msg : "CUDA error") + " (" + std::to_string(rc) + ")");
}

// the library's stream of `dev`, after checking that the device exists
inline Stream DeviceStream(int dev, const char* what) {
  const Lib& L = Get();
  int n = 0;
  L.device_count(&n);
  if (dev < 0 || dev >= n) throw std::runtime_error(std::string(what) + ": no CUDA device " + std::to_string(dev) + " (" + std::to_string(n) + " visible)");
  Stream s = L.stream(dev);
  if (!s) throw std::runtime_error(std::string(what) + ": cannot create a stream on device " + std::to_string(dev));
  return s;
}

}  // namespace kern
}  // namespace gxrt
