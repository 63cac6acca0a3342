// Plain C API of the HiPS runtime (parameter-server client, server loop, environment) for non-Python front ends.
//
// Parity: the KVStore part of MXNet's C API — include/mxnet/c_api.h MXKVStoreCreate / Free / Init / Push / Pull / Barrier / GetRank /
// GetGroupSize / IsWorkerNode / IsServerNode / IsSchedulerNode / RunServer / SendCommmandToServers / SetGradientCompression /
// GetNumDeadNode / MXInitPSEnv / MXGetLastError (src/c_api/c_api.cc:1021-1320) — with raw host buffers instead of NDArray handles
// (tensors belong to PyTorch in this design).  Every function returns 0 on success and -1 on failure; GXGetLastError() describes it.
// The symbols live in the same shared object as the Python bindings (geomx_b200/lib/_C*.so) with default visibility.
#include <cstring>
#include <string>

#include "env.h"
#include "kvstore_dist.h"

#define GX_CAPI extern "C" __attribute__((visibility("default")))

namespace gxrt { namespace capi { bool IsDeviceBuffer(const void* p); } }    // runtime/c_api_runtime.cc

namespace {
// buffers of device NDArrays (GXNDArrayGetData) are refused: the parameter-server plane reads and writes host memory
void HostOnly(const void* p, const char* fn) {
  if (p && gxrt::capi::IsDeviceBuffer(p)) throw std::runtime_error(std::string(fn) + ": device array (the KVStore group works on host buffers only)");
}
thread_local std::string last_error;
template <typename F>
int Guard(F&& f) {
  try { f(); return 0; }
  catch (const std::exception& e) { last_error = e.what(); return -1; }
  catch (...) { last_error = "unknown error"; return -1; }
}
hips::KVStoreDist* KV(void* h) {
  if (h == nullptr) throw hips::Error("null KVStore handle");
  return static_cast<hips::KVStoreDist*>(h);
}
}  // namespace

GX_CAPI const char* GXGetLastError() { return last_error.c_str(); }

GX_CAPI int GXInitPSEnv(int num, const char** keys, const char** vals) {
  return Guard([&] { for (int i = 0; i < num; ++i) hips::Environment::Get()->Set(keys[i], vals[i]); });
}
GX_CAPI int GXKVStoreIsWorkerNode(int* out) { return Guard([&] { hips::Postoffice::Get()->InitEnvironment(); *out = hips::Postoffice::Get()->is_worker(); }); }
GX_CAPI int GXKVStoreIsServerNode(int* out) { return Guard([&] { hips::Postoffice::Get()->InitEnvironment(); *out = hips::Postoffice::Get()->is_server(); }); }
GX_CAPI int GXKVStoreIsSchedulerNode(int* out) {
  return Guard([&] { hips::Postoffice::Get()->InitEnvironment(); *out = hips::Postoffice::Get()->is_scheduler() || hips::Postoffice::Get()->is_global_scheduler(); });
}

GX_CAPI int GXKVStoreCreate(const char* type, void** out) { return Guard([&] { *out = new hips::KVStoreDist(type ? type : "dist_sync"); }); }
GX_CAPI int GXKVStoreFree(void* h) { return Guard([&] { delete KV(h); }); }
GX_CAPI int GXKVStoreGetRank(void* h, int* out) { return Guard([&] { *out = KV(h)->rank(); }); }
GX_CAPI int GXKVStoreGetGroupSize(void* h, int* out) { return Guard([&] { *out = KV(h)->num_workers(); }); }
GX_CAPI int GXKVStoreGetNumAllWorkers(void* h, int* out) { return Guard([&] { *out = KV(h)->num_all_workers(); }); }
GX_CAPI int GXKVStoreIsMasterWorker(void* h, int* out) { return Guard([&] { *out = KV(h)->is_master_worker(); }); }

// dtype: mshadow flags (0 f32, 1 f64, 2 f16, 3 u8, 4 i32, 5 i8, 6 i64, 12 bf16).  The caller keeps `data` alive until the handle was waited.
GX_CAPI int GXKVStoreInit(void* h, int key, const void* data, size_t elems, int dtype) { return Guard([&] { HostOnly(data, "GXKVStoreInit"); KV(h)->Init(key, data, elems, dtype); }); }
GX_CAPI int GXKVStorePush(void* h, int key, const void* data, size_t elems, int dtype, int priority, int* handle) {
  return Guard([&] { HostOnly(data, "GXKVStorePush"); const int r = KV(h)->Push(key, data, elems, dtype, priority); if (handle) *handle = r; });
}
GX_CAPI int GXKVStorePull(void* h, int key, void* out, size_t elems, int dtype, int priority, int* handle) {
  return Guard([&] { HostOnly(out, "GXKVStorePull"); const int r = KV(h)->Pull(key, out, elems, dtype, priority); if (handle) *handle = r; });
}
GX_CAPI int GXKVStorePushRowSparse(void* h, int key, const int64_t* row_ids, size_t nrows, const float* rows, size_t row_len, int priority, int* handle) {
  return Guard([&] { HostOnly(rows, "GXKVStorePushRowSparse"); const int r = KV(h)->PushRows(key, row_ids, nrows, rows, row_len, priority); if (handle) *handle = r; });
}
GX_CAPI int GXKVStorePullRowSparse(void* h, int key, const int64_t* row_ids, size_t nrows, float* out, size_t row_len, int priority, int* handle) {
  return Guard([&] { HostOnly(out, "GXKVStorePullRowSparse"); const int r = KV(h)->PullRows(key, row_ids, nrows, out, row_len, priority); if (handle) *handle = r; });
}
GX_CAPI int GXKVStoreWait(void* h, int handle) { return Guard([&] { KV(h)->Wait(handle); }); }
GX_CAPI int GXKVStoreWaitAll(void* h) { return Guard([&] { KV(h)->WaitAll(); }); }
GX_CAPI int GXKVStoreBarrier(void* h) { return Guard([&] { KV(h)->Barrier(); }); }
GX_CAPI int GXKVStoreSendCommmandToServers(void* h, int head, const char* body) {   // (sic) the reference spells it with three m's
  return Guard([&] { KV(h)->SendCommandToServers(head, body ? body : ""); });
}
GX_CAPI int GXKVStoreSetGradientCompression(void* h, const char* type, float threshold) {
  return Guard([&] { KV(h)->SetGradientCompression(type ? type : "none", threshold); });
}
GX_CAPI int GXKVStoreGetNumDeadNode(void* h, int node_id, int timeout_sec, int* out) { return Guard([&] { *out = KV(h)->num_dead_node(node_id, timeout_sec); }); }
// server / scheduler processes: blocks until the job ends.  Optimizers arrive as declarative specs (command 7) and run natively.
GX_CAPI int GXKVStoreGetType(void* h, const char** out) { return Guard([&] { *out = KV(h)->type().c_str(); }); }
// MXKVStoreRunServer(handle, controller, controller_handle) + MXKVStoreSetUpdater(handle, updater, updater_handle) in one call for server
// processes: controller(head, body, arg) receives the commands workers send with SendCommmandToServers; updater(key, grad, weight, n, arg)
// replaces the built-in optimizer when not null (fp32 host buffers, update `weight` in place).
typedef void (*GXKVController)(int head, const char* body, void* arg);
typedef void (*GXKVUpdater)(int key, const float* grad, float* weight, size_t n, void* arg);
GX_CAPI int GXKVStoreRunServerEx(void* h, GXKVController controller, void* controller_arg, GXKVUpdater updater, void* updater_arg) {
  return Guard([&] {
    hips::KVStoreDistServer::Controller c = nullptr; hips::KVStoreDistServer::Updater u = nullptr;
    if (controller) c = [controller, controller_arg](int head, const std::string& body) { controller(head, body.c_str(), controller_arg); };
    if (updater) u = [updater, updater_arg](int key, const float* g, float* w, size_t n) { updater(key, g, w, n, updater_arg); };
    KV(h)->RunServer(c, u, nullptr);
  });
}
GX_CAPI int GXKVStoreRunServer(void* h) { return Guard([&] { KV(h)->RunServer(nullptr, nullptr, nullptr); }); }
GX_CAPI int GXKVStoreShutdown(void* h) { return Guard([&] { KV(h)->Shutdown(); }); }
