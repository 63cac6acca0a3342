// Plain C API of the HiPS runtime (parameter-server client, server loop, environment) and of the in-process KVStores for non-Python front
// ends.
//
// Parity: the KVStore part of MXNet's C API — include/mxnet/c_api.h MXKVStoreCreate / Free / Init / Push / Pull / SetUpdater / Barrier /
// GetRank / GetGroupSize / IsWorkerNode / IsServerNode / IsSchedulerNode / RunServer / SendCommmandToServers / SetGradientCompression /
// GetNumDeadNode / MXInitPSEnv / MXGetLastError (src/c_api/c_api.cc:1021-1320).  Two forms of the data calls: GXKVStoreInit / Push / Pull
// take raw host buffers (dist stores only); GXKVStoreInitND / PushND / PullND take NDArray handles, host or device, on every store type
// (csrc/runtime/kvstore_nd.h).  `local`, `local_update_cpu` and `local_allreduce_cpu` create an in-process store that reduces on the host;
// `device` and `local_allreduce_device` one that keeps each key on a GPU; every other type is the parameter-server worker (KVStoreDist).
// Every function returns 0 on success and -1 on failure; GXGetLastError() describes it.  The symbols live in the same shared object as the
// Python bindings (geomx_b200/lib/_C*.so) with default visibility.
#include <cstring>
#include <memory>
#include <string>

#include "env.h"
#include "kvstore_dist.h"
#include "runtime/kvstore_nd.h"

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

// a KVStore handle: the parameter-server worker (with the NDArray forms on top) or an in-process store
struct KVHandle {
  std::string type;
  std::unique_ptr<hips::KVStoreDist> dist;
  std::unique_ptr<gxrt::kvnd::DistND> dist_nd;
  std::unique_ptr<gxrt::kvnd::LocalStore> local;
};
KVHandle* KV(void* h) {
  if (h == nullptr) throw hips::Error("null KVStore handle");
  return static_cast<KVHandle*>(h);
}
// the worker endpoint; `nd` names the NDArray form an in-process store offers instead (or null when it has none)
hips::KVStoreDist* Dist(void* h, const char* fn, const char* nd = nullptr) {
  KVHandle* k = KV(h);
  if (k->dist) return k->dist.get();
  throw std::runtime_error(std::string(fn) + ": a '" + k->type + "' store is in-process and works on NDArray handles" +
                           (nd ? std::string("; use ") + nd : std::string(" (this function needs a dist store)")));
}
bool IsLocalType(const std::string& t) { return t == "local" || t == "local_update_cpu" || t == "local_allreduce_cpu"; }
bool IsDeviceType(const std::string& t) { return t == "device" || t == "local_allreduce_device"; }
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

GX_CAPI int GXKVStoreCreate(const char* type, void** out) {
  return Guard([&] {
    auto k = std::make_unique<KVHandle>();
    k->type = type ? type : "dist_sync";
    if (IsLocalType(k->type) || IsDeviceType(k->type)) {
      k->local.reset(new gxrt::kvnd::LocalStore(k->type, IsDeviceType(k->type)));
    } else {
      k->dist.reset(new hips::KVStoreDist(k->type));
      k->dist_nd.reset(new gxrt::kvnd::DistND(k->dist.get()));
    }
    *out = k.release();
  });
}
GX_CAPI int GXKVStoreFree(void* h) {
  return Guard([&] {
    std::unique_ptr<KVHandle> k(KV(h));
    if (k->dist) k->dist->Shutdown();            // outstanding pushes still read the staging buffers of dist_nd
    k->dist_nd.reset();
  });
}
GX_CAPI int GXKVStoreGetRank(void* h, int* out) { return Guard([&] { KVHandle* k = KV(h); *out = k->dist ? k->dist->rank() : 0; }); }
GX_CAPI int GXKVStoreGetGroupSize(void* h, int* out) { return Guard([&] { KVHandle* k = KV(h); *out = k->dist ? k->dist->num_workers() : 1; }); }
GX_CAPI int GXKVStoreGetNumAllWorkers(void* h, int* out) { return Guard([&] { KVHandle* k = KV(h); *out = k->dist ? k->dist->num_all_workers() : 1; }); }
GX_CAPI int GXKVStoreIsMasterWorker(void* h, int* out) { return Guard([&] { KVHandle* k = KV(h); *out = k->dist ? k->dist->is_master_worker() : 0; }); }

// dtype: mshadow flags (0 f32, 1 f64, 2 f16, 3 u8, 4 i32, 5 i8, 6 i64, 12 bf16).  The caller keeps `data` alive until the handle was waited.
GX_CAPI int GXKVStoreInit(void* h, int key, const void* data, size_t elems, int dtype) {
  return Guard([&] {
    HostOnly(data, "GXKVStoreInit");
    Dist(h, "GXKVStoreInit", "GXKVStoreInitND")->Init(key, data, elems, dtype);
    KV(h)->dist_nd->NoteRawInit(key, elems, dtype);
  });
}
GX_CAPI int GXKVStorePush(void* h, int key, const void* data, size_t elems, int dtype, int priority, int* handle) {
  return Guard([&] {
    HostOnly(data, "GXKVStorePush");
    const int r = Dist(h, "GXKVStorePush", "GXKVStorePushND")->Push(key, data, elems, dtype, priority);
    if (handle) *handle = r;
  });
}
GX_CAPI int GXKVStorePull(void* h, int key, void* out, size_t elems, int dtype, int priority, int* handle) {
  return Guard([&] {
    HostOnly(out, "GXKVStorePull");
    const int r = Dist(h, "GXKVStorePull", "GXKVStorePullND")->Pull(key, out, elems, dtype, priority);
    if (handle) *handle = r;
  });
}
GX_CAPI int GXKVStorePushRowSparse(void* h, int key, const int64_t* row_ids, size_t nrows, const float* rows, size_t row_len, int priority, int* handle) {
  return Guard([&] {
    HostOnly(rows, "GXKVStorePushRowSparse");
    const int r = Dist(h, "GXKVStorePushRowSparse")->PushRows(key, row_ids, nrows, rows, row_len, priority);
    if (handle) *handle = r;
  });
}
GX_CAPI int GXKVStorePullRowSparse(void* h, int key, const int64_t* row_ids, size_t nrows, float* out, size_t row_len, int priority, int* handle) {
  return Guard([&] {
    HostOnly(out, "GXKVStorePullRowSparse");
    const int r = Dist(h, "GXKVStorePullRowSparse")->PullRows(key, row_ids, nrows, out, row_len, priority);
    if (handle) *handle = r;
  });
}

// NDArray forms (MXKVStoreInit / Push / Pull argument order): a key listed k times in one push is k values summed left to right; listed k
// times in one pull, k outputs.  Host or device arrays on every store type; the device path never blocks on a local or device store.
GX_CAPI int GXKVStoreInitND(void* h, uint32_t num, const int* keys, void** vals) {
  return Guard([&] { KVHandle* k = KV(h); if (k->local) k->local->Init(num, keys, vals); else k->dist_nd->Init(num, keys, vals); });
}
GX_CAPI int GXKVStorePushND(void* h, uint32_t num, const int* keys, void** vals, int priority) {
  return Guard([&] { KVHandle* k = KV(h); if (k->local) k->local->Push(num, keys, vals); else k->dist_nd->Push(num, keys, vals, priority); });
}
GX_CAPI int GXKVStorePullND(void* h, uint32_t num, const int* keys, void** vals, int priority) {
  return Guard([&] { KVHandle* k = KV(h); if (k->local) k->local->Pull(num, keys, vals); else k->dist_nd->Pull(num, keys, vals, priority); });
}
// updater(key, recv, local, arg) replaces the assignment of a push on local / device stores: recv holds the reduced sum and local the stored
// value, both on the key's home (host or GPU); both handles belong to the store and live for the duration of the call
typedef void (*GXKVStoreUpdater)(int key, void* recv, void* local, void* arg);
GX_CAPI int GXKVStoreSetUpdater(void* h, GXKVStoreUpdater updater, void* arg) {
  return Guard([&] {
    KVHandle* k = KV(h);
    if (!k->local)
      throw std::runtime_error("GXKVStoreSetUpdater: a '" + k->type + "' store updates on its servers; send the optimizer with GXKVStoreSendCommmandToServers "
                               "(command 7) or run the servers with an updater through GXKVStoreRunServerEx");
    k->local->SetUpdater(updater, arg);
  });
}
GX_CAPI int GXKVStoreWait(void* h, int handle) { return Guard([&] { KVHandle* k = KV(h); if (k->dist) k->dist->Wait(handle); }); }
GX_CAPI int GXKVStoreWaitAll(void* h) { return Guard([&] { KVHandle* k = KV(h); if (k->dist) k->dist->WaitAll(); }); }
GX_CAPI int GXKVStoreBarrier(void* h) { return Guard([&] { KVHandle* k = KV(h); if (k->dist) k->dist->Barrier(); }); }
GX_CAPI int GXKVStoreSendCommmandToServers(void* h, int head, const char* body) {   // (sic) the reference spells it with three m's
  return Guard([&] { KVHandle* k = KV(h); if (k->dist) k->dist->SendCommandToServers(head, body ? body : ""); });
}
GX_CAPI int GXKVStoreSetGradientCompression(void* h, const char* type, float threshold) {
  return Guard([&] {
    KVHandle* k = KV(h);
    if (k->local) k->local->SetGradientCompression(type ? type : "none", threshold);
    else k->dist->SetGradientCompression(type ? type : "none", threshold);
  });
}
GX_CAPI int GXKVStoreGetNumDeadNode(void* h, int node_id, int timeout_sec, int* out) {
  return Guard([&] { KVHandle* k = KV(h); *out = k->dist ? k->dist->num_dead_node(node_id, timeout_sec) : 0; });
}
// server / scheduler processes: blocks until the job ends.  Optimizers arrive as declarative specs (command 7) and run natively.
GX_CAPI int GXKVStoreGetType(void* h, const char** out) { return Guard([&] { *out = KV(h)->type.c_str(); }); }
// MXKVStoreRunServer(handle, controller, controller_handle) + MXKVStoreSetUpdater(handle, updater, updater_handle) in one call for server
// processes: controller(head, body, arg) receives the commands workers send with SendCommmandToServers; updater(key, grad, weight, n, arg)
// replaces the built-in optimizer when not null (fp32 host buffers, update `weight` in place).
typedef void (*GXKVController)(int head, const char* body, void* arg);
typedef void (*GXKVUpdater)(int key, const float* grad, float* weight, size_t n, void* arg);
GX_CAPI int GXKVStoreRunServerEx(void* h, GXKVController controller, void* controller_arg, GXKVUpdater updater, void* updater_arg) {
  return Guard([&] {
    hips::KVStoreDist* kv = Dist(h, "GXKVStoreRunServerEx");
    hips::KVStoreDistServer::Controller c = nullptr; hips::KVStoreDistServer::Updater u = nullptr;
    if (controller) c = [controller, controller_arg](int head, const std::string& body) { controller(head, body.c_str(), controller_arg); };
    if (updater) u = [updater, updater_arg](int key, const float* g, float* w, size_t n) { updater(key, g, w, n, updater_arg); };
    kv->RunServer(c, u, nullptr);
  });
}
GX_CAPI int GXKVStoreRunServer(void* h) { return Guard([&] { Dist(h, "GXKVStoreRunServer")->RunServer(nullptr, nullptr, nullptr); }); }
GX_CAPI int GXKVStoreShutdown(void* h) { return Guard([&] { KVHandle* k = KV(h); if (k->dist) k->dist->Shutdown(); }); }
