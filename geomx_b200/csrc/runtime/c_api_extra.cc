// Remaining small groups of the flat C ABI: NDArray views / raw-bytes serialisation / synchronisation, profiler objects, process-level knobs.
//
// Parity: include/mxnet/c_api.h
//   :560-760    MXNDArrayCreateNone / Slice / At / Reshape / GetContext / GetStorageType / WaitToRead / WaitToWrite / WaitAll /
//               SaveRawBytes / LoadFromRawBytes   (host arrays are synchronous; for device arrays the wait functions synchronise the
//               library stream of the array's device, WaitAll every device stream and the C engine)
//   :280-420    MXProfileCreateDomain / CreateTask / CreateFrame / CreateEvent / CreateCounter / DestroyHandle / DurationStart / DurationStop /
//               SetCounter / AdjustCounter        (src/c_api/c_api_profile.cc:300-560)
//   :190-260    MXSetNumOMPThreads / MXEngineSetBulkSize / MXGetGPUCount / MXNotifyShutdown
#include <dlfcn.h>

#include <atomic>
#include <cstdint>
#include <cstring>
#include <memory>
#include <string>

#include "host_array.h"
#include "params_io.h"
#include "profiler.h"

#define GX_CAPI extern "C" __attribute__((visibility("default")))

void GXRTSetLastError(const std::string& msg);
extern "C" int GXEngineWaitAll();

namespace {
using gxrt::capi::HostArray;
using gxrt::capi::ND;

template <typename F>
int Guard(F&& f) {
  try { f(); return 0; }
  catch (const std::exception& e) { GXRTSetLastError(e.what()); return -1; }
  catch (...) { GXRTSetLastError("unknown error"); return -1; }
}

thread_local std::string raw_bytes;

struct ProfObject {
  enum Kind { kDomain, kTask, kFrame, kEvent, kCounter } kind;
  std::string name, domain;
  double t0 = -1;
  std::atomic<int64_t> value{0};
};
ProfObject* PO(void* h) { if (!h) throw std::runtime_error("null profile handle"); return static_cast<ProfObject*>(h); }
const char* KindName(ProfObject::Kind k) { switch (k) { case ProfObject::kTask: return "task"; case ProfObject::kFrame: return "frame"; case ProfObject::kEvent: return "event"; default: return "counter"; } }
void* MakeObject(ProfObject::Kind kind, void* domain, const char* name) {
  auto o = std::make_unique<ProfObject>();
  o->kind = kind; o->name = name ? name : "";
  if (domain) { if (PO(domain)->kind != ProfObject::kDomain) throw std::runtime_error("not a profile domain handle"); o->domain = PO(domain)->name; }
  return o.release();
}
std::atomic<int> omp_threads{0}, bulk_size{15};
}  // namespace

// ================================================================================================ NDArray
GX_CAPI int GXNDArrayCreateNone(void** out) { return Guard([&] { *out = new HostArray(); }); }
// rows [begin, end) of the first axis, as a copy (host arrays of this ABI do not alias; write back with SyncCopyFromCPU on the parent's data)
GX_CAPI int GXNDArraySlice(void* h, uint32_t begin, uint32_t end, void** out) {
  return Guard([&] {
    HostArray* a = ND(h);
    const std::string& data = gxrt::capi::HostBytes(a, "GXNDArraySlice");
    if (a->rec.shape.empty() || begin > end || end > static_cast<uint32_t>(a->rec.shape[0])) throw std::runtime_error("Slice: range out of bounds");
    const size_t row = data.size() / static_cast<size_t>(std::max<int64_t>(a->rec.shape[0], 1));
    auto s = std::make_unique<HostArray>();
    s->rec.dtype = a->rec.dtype; s->rec.shape = a->rec.shape; s->rec.shape[0] = end - begin;
    s->rec.data.assign(data.data() + begin * row, (end - begin) * row);
    *out = s.release();
  });
}
GX_CAPI int GXNDArrayAt(void* h, uint32_t idx, void** out) {
  return Guard([&] {
    HostArray* a = ND(h);
    const std::string& data = gxrt::capi::HostBytes(a, "GXNDArrayAt");
    if (a->rec.shape.empty() || idx >= static_cast<uint32_t>(a->rec.shape[0])) throw std::runtime_error("At: index out of bounds");
    const size_t row = data.size() / static_cast<size_t>(a->rec.shape[0]);
    auto s = std::make_unique<HostArray>();
    s->rec.dtype = a->rec.dtype; s->rec.shape.assign(a->rec.shape.begin() + 1, a->rec.shape.end());
    if (s->rec.shape.empty()) s->rec.shape.push_back(1);
    s->rec.data.assign(data.data() + idx * row, row);
    *out = s.release();
  });
}
// dims: positive extents, one -1 is inferred, 0 copies the input extent at that position
GX_CAPI int GXNDArrayReshape(void* h, int ndim, const int* dims, void** out) {
  return Guard([&] {
    HostArray* a = ND(h);
    const std::string& data = gxrt::capi::HostBytes(a, "GXNDArrayReshape");
    const int64_t total = gxrt::Prod(a->rec.shape);
    std::vector<int64_t> shp; int infer = -1; int64_t known = 1;
    for (int i = 0; i < ndim; ++i) {
      int64_t d = dims[i];
      if (d == 0) { if (static_cast<size_t>(i) >= a->rec.shape.size()) throw std::runtime_error("Reshape: 0 past the input rank"); d = a->rec.shape[i]; }
      if (d == -1) { if (infer >= 0) throw std::runtime_error("Reshape: more than one -1"); infer = i; shp.push_back(1); continue; }
      if (d < 0) throw std::runtime_error("Reshape: negative extent");
      shp.push_back(d); known *= d;
    }
    if (infer >= 0) { if (known == 0 || total % known) throw std::runtime_error("Reshape: cannot infer -1"); shp[infer] = total / known; known *= shp[infer]; }
    if (known != total) throw std::runtime_error("Reshape: size changes from " + std::to_string(total) + " to " + std::to_string(known));
    auto s = std::make_unique<HostArray>();
    s->rec.dtype = a->rec.dtype; s->rec.shape = shp; s->rec.data = data;
    *out = s.release();
  });
}
// (1, 0) kCPU for host arrays, (2, dev_id) kGPU for device arrays
GX_CAPI int GXNDArrayGetContext(void* h, int* out_dev_type, int* out_dev_id) {
  return Guard([&] { HostArray* a = ND(h); *out_dev_type = a->device() ? 2 : 1; *out_dev_id = a->device() ? a->dev_id : 0; });
}
GX_CAPI int GXNDArrayGetStorageType(void* h, int* out) { return Guard([&] { *out = ND(h)->rec.shape.empty() ? -1 : 0; }); }                           // kDefaultStorage
GX_CAPI int GXNDArrayWaitToRead(void* h) { return Guard([&] { HostArray* a = ND(h); if (a->device()) gxrt::capi::SyncDevice(a->dev_id); }); }
GX_CAPI int GXNDArrayWaitToWrite(void* h) { return Guard([&] { HostArray* a = ND(h); if (a->device()) gxrt::capi::SyncDevice(a->dev_id); }); }
GX_CAPI int GXNDArrayWaitAll() {
  if (Guard([&] { gxrt::capi::SyncAllDevices(); }) != 0) return -1;
  return GXEngineWaitAll();
}
// one array in NDArray::Save's layout (src/ndarray/ndarray.cc:1583-1660); the buffer is thread-local
GX_CAPI int GXNDArraySaveRawBytes(void* h, size_t* out_size, const char** out_buf) {
  return Guard([&] {
    const std::string list = gxrt::WriteList({gxrt::capi::HostCopy(ND(h))}, {});
    raw_bytes = list.substr(24, list.size() - 24 - 8);          // strip the list header (magic, reserved, count) and the empty name table
    *out_size = raw_bytes.size(); *out_buf = raw_bytes.data();
  });
}
GX_CAPI int GXNDArrayLoadFromRawBytes(const void* buf, size_t size, void** out) {
  return Guard([&] {
    gxrt::BufReader r(static_cast<const char*>(buf), size);
    auto a = std::make_unique<HostArray>();
    a->rec = gxrt::ReadArray(r);
    *out = a.release();
  });
}

// ================================================================================================ profiler objects
GX_CAPI int GXProfileCreateDomain(const char* domain, void** out) { return Guard([&] { *out = MakeObject(ProfObject::kDomain, nullptr, domain); }); }
GX_CAPI int GXProfileCreateTask(void* domain, const char* name, void** out) { return Guard([&] { *out = MakeObject(ProfObject::kTask, domain, name); }); }
GX_CAPI int GXProfileCreateFrame(void* domain, const char* name, void** out) { return Guard([&] { *out = MakeObject(ProfObject::kFrame, domain, name); }); }
GX_CAPI int GXProfileCreateEvent(const char* name, void** out) { return Guard([&] { *out = MakeObject(ProfObject::kEvent, nullptr, name); }); }
GX_CAPI int GXProfileCreateCounter(void* domain, const char* name, void** out) { return Guard([&] { *out = MakeObject(ProfObject::kCounter, domain, name); }); }
GX_CAPI int GXProfileDestroyHandle(void* h) { return Guard([&] { delete PO(h); }); }
GX_CAPI int GXProfileDurationStart(void* h) { return Guard([&] { PO(h)->t0 = hips::Profiler::NowUs(); }); }
GX_CAPI int GXProfileDurationStop(void* h) {
  return Guard([&] {
    ProfObject* o = PO(h);
    if (o->t0 < 0) throw std::runtime_error("DurationStop without DurationStart");
    const std::string cat = o->domain.empty() ? KindName(o->kind) : o->domain;
    if (hips::Profiler::Get()->active()) hips::Profiler::Get()->Add(o->name, cat, 'X', o->t0, hips::Profiler::NowUs() - o->t0);
    o->t0 = -1;
  });
}
GX_CAPI int GXProfileSetCounter(void* h, uint64_t value) {
  return Guard([&] {
    ProfObject* o = PO(h);
    o->value = static_cast<int64_t>(value);
    if (hips::Profiler::Get()->active()) hips::Profiler::Get()->Add(o->name, o->domain.empty() ? "counter" : o->domain, 'C', hips::Profiler::NowUs(), 0, 0, 0, static_cast<double>(value));
  });
}
GX_CAPI int GXProfileAdjustCounter(void* h, int64_t delta) {
  return Guard([&] {
    ProfObject* o = PO(h);
    const int64_t v = (o->value += delta);
    if (hips::Profiler::Get()->active()) hips::Profiler::Get()->Add(o->name, o->domain.empty() ? "counter" : o->domain, 'C', hips::Profiler::NowUs(), 0, 0, 0, static_cast<double>(v));
  });
}

// ================================================================================================ process-level knobs
GX_CAPI int GXSetNumOMPThreads(int n) { return Guard([&] { if (n < 0) throw std::runtime_error("thread count must be non-negative"); omp_threads = n; }); }
GX_CAPI int GXGetNumOMPThreads(int* out) { return Guard([&] { *out = omp_threads; }); }
GX_CAPI int GXEngineSetBulkSize(int size, int* prev) { return Guard([&] { if (prev) *prev = bulk_size; bulk_size = size; }); }
// devices visible to the CUDA driver (0 without a driver): dlopen so the C library itself links no CUDA
GX_CAPI int GXGetGPUCount(int* out) {
  return Guard([&] {
    *out = 0;
    void* lib = dlopen("libcuda.so.1", RTLD_LAZY | RTLD_LOCAL);
    if (!lib) return;
    auto init = reinterpret_cast<int (*)(unsigned)>(dlsym(lib, "cuInit"));
    auto count = reinterpret_cast<int (*)(int*)>(dlsym(lib, "cuDeviceGetCount"));
    int n = 0;
    if (init && count && init(0) == 0 && count(&n) == 0) *out = n;
    dlclose(lib);
  });
}
GX_CAPI int GXNotifyShutdown() { return Guard([&] { GXEngineWaitAll(); if (hips::Profiler::Get()->active()) hips::Profiler::Get()->Dump(true); }); }
