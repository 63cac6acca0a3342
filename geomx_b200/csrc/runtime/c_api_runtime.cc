// Plain C API of the native runtime for non-Python front ends: host NDArray handles with the byte-exact `.params` serializer, the profiler,
// the dependency engine and the pooled host storage.  Together with csrc/hips/c_api.cc (GXKVStore*) this is the flat C ABI of the framework.
//
// Parity (names follow the reference with the GX prefix): include/mxnet/c_api.h
//   NDArray   MXNDArrayCreateEx / Free / GetShape / GetDType / GetData / SyncCopyFromCPU / SyncCopyToCPU / Save / Load   (:540-1010)
//   Profiler  MXSetProfilerConfig / MXSetProfilerState / MXDumpProfile / MXProfilePause / MXProfileSetMarker            (src/c_api/c_api_profile.cc:264-560)
//   Engine    the push/wait contract of include/mxnet/engine.h:115-314 (NewVariable / PushAsync / WaitForVar / WaitForAll) for C callbacks
//   Storage   include/mxnet/storage.h Alloc / Free of the pooled host manager (src/storage/pooled_storage_manager.h:52-172)
// An NDArray handle owns host memory (GXNDArrayCreate) or float32 device memory from the native pool (GXNDArrayCreateEx, dev_type 2).  Work
// on device arrays is ordered on one stream per device inside the kernel library: copies, executor passes and imperative operators are
// enqueued in call order, and SyncCopyToCPU / WaitToRead / WaitToWrite / WaitAll synchronise that stream.  Every function returns 0 on
// success and -1 on failure; GXRTGetLastError() describes the failure of the calling thread.
#include <cstdint>
#include <cstring>
#include <fstream>
#include <map>
#include <set>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "engine.h"
#include "host_array.h"
#include "kernel_lib.h"
#include "params_io.h"
#include "profiler.h"
#include "storage.h"

#define GX_CAPI extern "C" __attribute__((visibility("default")))

namespace {
thread_local std::string rt_error;
template <typename F>
int Guard(F&& f) {
  try { f(); return 0; }
  catch (const std::exception& e) { rt_error = e.what(); return -1; }
  catch (...) { rt_error = "unknown error"; return -1; }
}
using gxrt::capi::HostArray;
using gxrt::capi::ND;
// results of the last GXNDArrayLoad of this thread (the reference returns pointers into thread-local storage as well, c_api.cc MXNDArrayLoad)
thread_local std::vector<void*> load_handles;
thread_local std::vector<std::string> load_names;
thread_local std::vector<const char*> load_name_ptrs;

gx_rt::PooledHostStorage& HostPool() { static gx_rt::PooledHostStorage pool; return pool; }
std::mutex engine_mu;
std::unique_ptr<gxrt::Engine> engine;
gxrt::Engine* Eng() {
  std::lock_guard<std::mutex> lk(engine_mu);
  if (!engine) engine.reset(new gxrt::Engine(4, false));
  return engine.get();
}
}  // namespace

GX_CAPI const char* GXRTGetLastError() { return rt_error.c_str(); }
void GXRTSetLastError(const std::string& msg) { rt_error = msg; }       // for the other translation units of the C ABI (c_predict_api.cc)

// ------------------------------------------------------------------------------------------------ device arrays
namespace {
std::mutex dev_mu;
std::map<uintptr_t, size_t> dev_buffers;                                 // live device allocations: start -> bytes
std::set<int> devices_used;
}  // namespace
namespace gxrt {
namespace capi {
size_t HostArray::Bytes() const { return device() ? static_cast<size_t>(gxrt::Prod(rec.shape)) * 4 : rec.data.size(); }
HostArray* NewDeviceArray(const std::vector<int64_t>& shape, int dev) {
  namespace K = gxrt::kern;
  K::Stream s = K::DeviceStream(dev, "GXNDArrayCreateEx");
  const K::Lib& L = K::Get();
  auto a = std::make_unique<HostArray>();
  a->rec.dtype = 0; a->rec.shape = shape; a->dev_id = dev;
  const size_t bytes = static_cast<size_t>(gxrt::Prod(shape)) * 4;
  K::Check(L.set_device(dev), "GXNDArrayCreateEx");
  a->dptr = static_cast<float*>(L.pool_alloc(dev, bytes ? bytes : 4, s));
  if (!a->dptr) throw std::runtime_error("GXNDArrayCreateEx: out of device memory on device " + std::to_string(dev) + " (" + std::to_string(bytes) + " bytes)");
  a->owns_dptr = true;
  { std::lock_guard<std::mutex> lk(dev_mu); dev_buffers[reinterpret_cast<uintptr_t>(a->dptr)] = bytes; devices_used.insert(dev); }
  K::Check(L.memset(a->dptr, 0, bytes, s), "GXNDArrayCreateEx");
  return a.release();
}
void ReleaseDevice(HostArray* a) {
  if (!a->device() || !a->owns_dptr || !a->dptr) return;
  { std::lock_guard<std::mutex> lk(dev_mu); dev_buffers.erase(reinterpret_cast<uintptr_t>(a->dptr)); }
  const gxrt::kern::Lib& L = gxrt::kern::Get();
  L.pool_free(a->dev_id, a->dptr, L.stream(a->dev_id));
  a->dptr = nullptr;
}
gxrt::NDRec HostCopy(const HostArray* a) {
  if (!a->device()) return a->rec;
  namespace K = gxrt::kern;
  gxrt::NDRec r;
  r.dtype = a->rec.dtype; r.shape = a->rec.shape;
  r.data.assign(a->Bytes(), '\0');
  K::Stream s = K::Get().stream(a->dev_id);
  K::Check(K::Get().memcpy(&r.data[0], a->dptr, r.data.size(), 2, s), "device -> host copy");
  K::Check(K::Get().stream_sync(s), "device -> host copy");
  return r;
}
void SyncDevice(int dev) {
  namespace K = gxrt::kern;
  K::Check(K::Get().stream_sync(K::Get().stream(dev)), "device synchronise");
}
void SyncAllDevices() {
  std::set<int> devs;
  { std::lock_guard<std::mutex> lk(dev_mu); devs = devices_used; }
  for (int d : devs) SyncDevice(d);
}
bool IsDeviceBuffer(const void* p) {
  const uintptr_t u = reinterpret_cast<uintptr_t>(p);
  std::lock_guard<std::mutex> lk(dev_mu);
  auto it = dev_buffers.upper_bound(u);
  if (it == dev_buffers.begin()) return false;
  --it;
  return u < it->first + std::max<size_t>(it->second, 1);
}
}  // namespace capi
}  // namespace gxrt

// ------------------------------------------------------------------------------------------------ NDArray (host)
// dtype: mshadow flags (0 f32, 1 f64, 2 f16, 3 u8, 4 i32, 5 i8, 6 i64)
GX_CAPI int GXNDArrayCreate(const uint32_t* shape, uint32_t ndim, int dtype, void** out) {
  return Guard([&] {
    auto a = std::make_unique<HostArray>();
    a->rec.dtype = dtype;
    a->rec.shape.assign(shape, shape + ndim);
    a->rec.data.assign(static_cast<size_t>(gxrt::Prod(a->rec.shape)) * gxrt::FlagSize(dtype), '\0');
    *out = a.release();
  });
}
// dev_type 1 (CPU): GXNDArrayCreate.  dev_type 2 (GPU): float32 device memory on dev_id from the native pool, zero-filled.  delay_alloc is
// accepted for the reference's signature; memory is always allocated here.
GX_CAPI int GXNDArrayCreateEx(const uint32_t* shape, uint32_t ndim, int dev_type, int dev_id, int delay_alloc, int dtype, void** out) {
  (void)delay_alloc;
  if (dev_type == 1) return GXNDArrayCreate(shape, ndim, dtype, out);
  return Guard([&] {
    if (dev_type != 2) throw std::runtime_error("GXNDArrayCreateEx: dev_type " + std::to_string(dev_type) + " is not supported (1 CPU, 2 GPU)");
    if (dtype != 0) throw std::runtime_error("GXNDArrayCreateEx: device arrays are float32 (dtype flag 0), got dtype flag " + std::to_string(dtype));
    *out = gxrt::capi::NewDeviceArray(std::vector<int64_t>(shape, shape + ndim), dev_id);
  });
}
GX_CAPI int GXNDArrayFree(void* h) { return Guard([&] { delete ND(h); }); }
GX_CAPI int GXNDArrayGetShape(void* h, uint32_t* out_ndim, const uint32_t** out_shape) {
  return Guard([&] {
    HostArray* a = ND(h);
    a->shape32.assign(a->rec.shape.begin(), a->rec.shape.end());
    *out_ndim = static_cast<uint32_t>(a->shape32.size());
    *out_shape = a->shape32.data();
  });
}
GX_CAPI int GXNDArrayGetDType(void* h, int* out) { return Guard([&] { *out = ND(h)->rec.dtype; }); }
// device arrays: the device pointer (for the caller's own CUDA code; work queued on the library stream may still be writing it — WaitToRead)
GX_CAPI int GXNDArrayGetData(void* h, void** out) {
  return Guard([&] { HostArray* a = ND(h); *out = a->device() ? static_cast<void*>(a->dptr) : static_cast<void*>(&a->rec.data[0]); });
}
GX_CAPI int GXNDArraySyncCopyFromCPU(void* h, const void* data, size_t size_elems) {
  return Guard([&] {
    HostArray* a = ND(h);
    const size_t bytes = size_elems * gxrt::FlagSize(a->rec.dtype);
    if (bytes != a->Bytes()) throw std::runtime_error("SyncCopyFromCPU: size does not match the array");
    if (a->device()) {
      // pageable source: the copy has left `data` when cudaMemcpyAsync returns, so the caller may reuse its buffer at once
      namespace K = gxrt::kern;
      K::Check(K::Get().memcpy(a->dptr, data, bytes, 1, K::Get().stream(a->dev_id)), "SyncCopyFromCPU");
      return;
    }
    memcpy(&a->rec.data[0], data, bytes);
  });
}
GX_CAPI int GXNDArraySyncCopyToCPU(void* h, void* data, size_t size_elems) {
  return Guard([&] {
    HostArray* a = ND(h);
    const size_t bytes = size_elems * gxrt::FlagSize(a->rec.dtype);
    if (bytes != a->Bytes()) throw std::runtime_error("SyncCopyToCPU: size does not match the array");
    if (a->device()) {
      namespace K = gxrt::kern;
      K::Stream s = K::Get().stream(a->dev_id);
      K::Check(K::Get().memcpy(data, a->dptr, bytes, 2, s), "SyncCopyToCPU");
      K::Check(K::Get().stream_sync(s), "SyncCopyToCPU");
      return;
    }
    memcpy(data, a->rec.data.data(), bytes);
  });
}
// `.params` / NDArray-list file, byte-compatible with NDArray::Save (src/ndarray/ndarray.cc:1583-1811); keys may be null (unnamed list)
GX_CAPI int GXNDArraySave(const char* fname, uint32_t num, void** handles, const char** keys) {
  return Guard([&] {
    std::vector<gxrt::NDRec> recs;
    std::vector<std::string> names;
    for (uint32_t i = 0; i < num; ++i) { recs.push_back(gxrt::capi::HostCopy(ND(handles[i]))); if (keys) names.emplace_back(keys[i]); }
    const std::string blob = gxrt::WriteList(recs, names);
    std::ofstream f(fname, std::ios::binary);
    if (!f) throw std::runtime_error(std::string("cannot open ") + fname);
    f.write(blob.data(), static_cast<std::streamsize>(blob.size()));
  });
}
GX_CAPI int GXNDArrayLoad(const char* fname, uint32_t* out_size, void*** out_handles, uint32_t* out_name_size, const char*** out_names) {
  return Guard([&] {
    std::ifstream f(fname, std::ios::binary);
    if (!f) throw std::runtime_error(std::string("cannot open ") + fname);
    std::string s((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    gxrt::BufReader r(s.data(), s.size());
    if (r.Get<uint64_t>() != gxrt::kListMagic) throw std::runtime_error("Invalid NDArray file format");
    r.Get<uint64_t>();
    const uint64_t n = r.Get<uint64_t>();
    load_handles.clear(); load_names.clear(); load_name_ptrs.clear();
    for (uint64_t i = 0; i < n; ++i) { auto a = std::make_unique<HostArray>(); a->rec = gxrt::ReadArray(r); load_handles.push_back(a.release()); }
    const uint64_t m = r.Get<uint64_t>();
    for (uint64_t i = 0; i < m; ++i) { const uint64_t l = r.Get<uint64_t>(); load_names.push_back(r.Raw(l)); }
    for (auto& nm : load_names) load_name_ptrs.push_back(nm.c_str());
    *out_size = static_cast<uint32_t>(load_handles.size()); *out_handles = load_handles.data();
    *out_name_size = static_cast<uint32_t>(load_name_ptrs.size()); *out_names = load_name_ptrs.data();
  });
}

// ------------------------------------------------------------------------------------------------ profiler
// keys: filename, aggregate_stats, continuous_dump, dump_period (the subset of MXSetProfilerConfig this profiler has knobs for)
GX_CAPI int GXSetProfilerConfig(int num, const char* const* keys, const char* const* vals) {
  return Guard([&] {
    std::string fn = "profile.json"; bool agg = false, cont = false; double period = 1.0;
    for (int i = 0; i < num; ++i) {
      const std::string k = keys[i], v = vals[i];
      if (k == "filename") fn = v;
      else if (k == "aggregate_stats") agg = (v == "1" || v == "true" || v == "True");
      else if (k == "continuous_dump") cont = (v == "1" || v == "true" || v == "True");
      else if (k == "dump_period") period = std::stod(v);
    }
    hips::Profiler::Get()->SetConfig(fn, agg, cont, period);
  });
}
GX_CAPI int GXSetProfilerState(int state) { return Guard([&] { hips::Profiler::Get()->SetState(state != 0); }); }
GX_CAPI int GXProfilePause(int paused) { return Guard([&] { hips::Profiler::Get()->Pause(paused != 0); }); }
GX_CAPI int GXDumpProfile(int finished) { return Guard([&] { hips::Profiler::Get()->Dump(finished != 0); }); }
// instant marker / duration event from a non-Python front end (MXProfileSetMarker, MXProfileDurationStart/Stop collapsed into one call)
GX_CAPI int GXProfileSetMarker(const char* name, const char* category) {
  return Guard([&] { hips::Profiler::Get()->Add(name, category ? category : "marker", 'i', hips::Profiler::NowUs()); });
}
GX_CAPI int GXProfileAddDuration(const char* name, const char* category, double start_us, double dur_us) {
  return Guard([&] { hips::Profiler::Get()->Add(name, category ? category : "operator", 'X', start_us, dur_us); });
}
GX_CAPI double GXProfileNowUs() { return hips::Profiler::NowUs(); }

// ------------------------------------------------------------------------------------------------ dependency engine
typedef void (*GXEngineFn)(void* arg);
GX_CAPI int GXEngineNewVariable(int* out) { return Guard([&] { *out = Eng()->NewVariable(); }); }
// fn(arg) runs once every earlier writer of the const vars and every earlier reader/writer of the mutable vars has completed
GX_CAPI int GXEnginePushAsync(GXEngineFn fn, void* arg, const int* const_vars, int num_const, const int* mutable_vars, int num_mutable, int priority,
                              const char* name) {
  return Guard([&] {
    Eng()->Push([fn, arg] { fn(arg); }, std::vector<int>(const_vars, const_vars + num_const), std::vector<int>(mutable_vars, mutable_vars + num_mutable),
                priority, name ? name : "c_api_op");
  });
}
// same, on the worker pool of `device` (-1: CPU) chosen by `prop` (0 normal / compute, 1 copy, 2 priority) — engine.h FnProperty + exec_ctx
GX_CAPI int GXEnginePushAsyncEx(GXEngineFn fn, void* arg, const int* const_vars, int num_const, const int* mutable_vars, int num_mutable, int priority,
                                const char* name, int device, int prop) {
  return Guard([&] {
    Eng()->Push([fn, arg] { fn(arg); }, std::vector<int>(const_vars, const_vars + num_const), std::vector<int>(mutable_vars, mutable_vars + num_mutable),
                priority, name ? name : "c_api_op", device, static_cast<gxrt::FnProperty>(prop < 0 || prop > 2 ? 0 : prop));
  });
}
GX_CAPI int GXEngineDeleteVariable(int var) { return Guard([&] { Eng()->DeleteVariable(var); }); }
GX_CAPI int GXEngineWaitForVar(int var) { return Guard([&] { Eng()->WaitForVar(var); }); }
GX_CAPI int GXEngineWaitAll() { return Guard([&] { Eng()->WaitForAll(); }); }

// ------------------------------------------------------------------------------------------------ storage
GX_CAPI int GXStorageAlloc(size_t nbytes, void** out) {
  return Guard([&] { *out = HostPool().Alloc(nbytes); if (*out == nullptr) throw std::runtime_error("out of host memory"); });
}
GX_CAPI int GXStorageFree(void* p) { return Guard([&] { HostPool().Free(p); }); }
