// KVStore on NDArray handles for the flat C ABI (GXKVStoreInitND / PushND / PullND / SetUpdater in csrc/hips/c_api.cc).
//
// Parity: MXKVStoreInit / Push / Pull / SetUpdater (include/mxnet/c_api.h) over KVStoreLocal (src/kvstore/kvstore_local.h: grouping of
// repeated keys, updater vs. assign) with CommCPU / CommDevice (src/kvstore/comm.h: host reduce, reduce on one GPU, the compressed inter-GPU
// reduce of :545-589), and the device-array side of KVStoreDist (src/kvstore/kvstore_dist.h).  The Python twin is kvstore/local.py.
//
// Semantics shared by every store type:
//   * a key listed k times in one push is k values (one per device); they are summed left to right in the order given, then pushed once;
//   * a key listed k times in one pull writes the stored value into all k outputs;
//   * a key repeated in one init, or initialised twice, is an error; so are an unknown key, a shape or dtype that differs from the init
//     value, and a key whose values in one call mix host and device arrays.  Messages name the C function and the key.
//
// LocalStore ("local" and the "device" family).  A key lives on its home: the host for `local`, and for `device` the GPU of the value given
// to Init (a host init value keeps the key on the host).  Device values of a host key travel through page-locked staging and are summed on
// the host, which makes `local` the oracle of `device`.  Device values of a device key are gathered to the home GPU with peer copies issued
// on each source's stream (so each copy follows the work already queued there) and summed there by one gx_kv_sum_quantize launch per 8
// values.  With 2-bit compression (device store, more than one value) each value is quantised on its own GPU with a residual per
// (key, position), only the words travel, and gx_kv_dequant_sum adds them up on the home GPU.  Pulls copy the stored value into each output on
// the output device's stream.  Nothing synchronises with the host on the device path: streams wait for each other through events, so work
// issued later on any device in call order sees the result.
//
// DistND (every other type).  Host values are summed on the host and sent with the bytes the raw-buffer GXKVStorePush sends.  Device values
// are summed on their home GPU (the device of the init value, else of the first value pushed); under 2-bit compression the sum is quantised
// in the same launch with a per-key residual kept on that GPU.  The sum or the words go to a page-locked buffer of the key, the home stream is
// synchronised once and the push leaves asynchronously.  A pull issues the requests of all keys of the call, waits for all of them, then
// enqueues one host-to-device copy per key and the copies to the remaining outputs — so the keys of one PullND share their round trips, and
// unlike the reference's engine-scheduled pull the call returns after the network part is done.
#pragma once
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <set>
#include <stdexcept>
#include <string>
#include <vector>

#include "hips/kvstore_dist.h"
#include "host_array.h"
#include "kernel_lib.h"
#include "params_io.h"

namespace gxrt {
namespace kvnd {

namespace K = gxrt::kern;
using capi::HostArray;

typedef void (*Updater)(int key, void* recv, void* local, void* arg);

[[noreturn]] inline void Fail(const char* fn, int key, const std::string& what) {
  throw std::runtime_error(std::string(fn) + ": key " + std::to_string(key) + ": " + what);
}

inline std::string ShapeStr(const std::vector<int64_t>& s) {
  std::string r = "(";
  for (size_t i = 0; i < s.size(); ++i) r += (i ? "," : "") + std::to_string(s[i]);
  return r + ")";
}

// the values (or outputs) of one key within one call, keys in order of first appearance
struct Group {
  int key;
  std::vector<HostArray*> vals;
  bool device() const { return vals[0]->device(); }
};
inline std::vector<Group> GroupByKey(const char* fn, uint32_t num, const int* keys, void** vals) {
  std::vector<Group> out;
  std::map<int, size_t> at;
  for (uint32_t i = 0; i < num; ++i) {
    HostArray* a = capi::ND(vals[i]);
    auto it = at.find(keys[i]);
    if (it == at.end()) { at[keys[i]] = out.size(); out.push_back(Group{keys[i], {a}}); continue; }
    Group& g = out[it->second];
    if (g.vals[0]->device() != a->device()) Fail(fn, keys[i], "mixes host and device arrays (all values of one key must be of one kind)");
    g.vals.push_back(a);
  }
  return out;
}

// page-locked host memory of the kernel library
struct Pinned {
  void* p = nullptr;
  size_t bytes = 0;
  Pinned() = default;
  Pinned(const Pinned&) = delete;
  Pinned& operator=(const Pinned&) = delete;
  ~Pinned() { Free(); }
  void* Reserve(size_t b) {
    if (b > bytes) { Free(); K::Check(K::Get().host_alloc(b, &p), "page-locked host allocation"); bytes = b; }
    return p;
  }
  void Free() { if (p) K::Get().host_free(p); p = nullptr; bytes = 0; }
};

// device memory from the native pool; (re)allocation zero-fills
struct DevBuf {
  int dev = -1;
  void* p = nullptr;
  size_t bytes = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : dev(o.dev), p(o.p), bytes(o.bytes) { o.p = nullptr; o.bytes = 0; }
  ~DevBuf() { Free(); }
  template <typename T = void>
  T* Reserve(int d, size_t b) {
    if (d != dev || b > bytes) {
      Free();
      const K::Lib& L = K::Get();
      K::Stream s = K::DeviceStream(d, "KVStore");
      K::Check(L.set_device(d), "KVStore");
      p = L.pool_alloc(d, b ? b : 4, s);
      if (!p) throw std::runtime_error("KVStore: out of device memory on device " + std::to_string(d) + " (" + std::to_string(b) + " bytes)");
      dev = d; bytes = b;
      K::Check(L.memset(p, 0, b, s), "KVStore");
    }
    return static_cast<T*>(p);
  }
  void Free() {
    if (p) { const K::Lib& L = K::Get(); L.pool_free(dev, p, L.stream(dev)); }
    p = nullptr; bytes = 0;
  }
};

inline K::Stream Str(int dev) { return K::DeviceStream(dev, "KVStore"); }
inline void Join(int waiter_dev, int signaller_dev) {
  if (waiter_dev == signaller_dev) return;
  K::Check(K::Get().stream_join(Str(waiter_dev), Str(signaller_dev), signaller_dev), "KVStore stream join");
}

// dst = src[0] + src[1] + ... elementwise on the host, left to right (dst may be src[0])
template <typename T>
void SumT(const std::vector<const void*>& src, void* dst, size_t n) {
  T* d = static_cast<T*>(dst);
  if (d != src[0]) std::memcpy(d, src[0], n * sizeof(T));
  for (size_t j = 1; j < src.size(); ++j) {
    const T* s = static_cast<const T*>(src[j]);
    for (size_t i = 0; i < n; ++i) d[i] = static_cast<T>(d[i] + s[i]);
  }
}
inline void HostSum(const char* fn, int key, int dtype, const std::vector<const void*>& src, void* dst, size_t n) {
  if (src.size() == 1) { if (dst != src[0]) std::memcpy(dst, src[0], n * gxrt::FlagSize(dtype)); return; }
  switch (dtype) {
    case 0: SumT<float>(src, dst, n); break;
    case 1: SumT<double>(src, dst, n); break;
    case 3: SumT<uint8_t>(src, dst, n); break;
    case 4: SumT<int32_t>(src, dst, n); break;
    case 5: SumT<int8_t>(src, dst, n); break;
    case 6: SumT<int64_t>(src, dst, n); break;
    default: Fail(fn, key, "cannot sum values of dtype flag " + std::to_string(dtype) + " on the host");
  }
}

// gathers the device values of `g` onto `home` (peer copies on each source's stream into `stage`) and returns the pointers to sum there
inline std::vector<const float*> Gather(const Group& g, int home, size_t n, std::vector<DevBuf>& stage) {
  const K::Lib& L = K::Get();
  if (stage.size() < g.vals.size()) stage.resize(g.vals.size());
  std::vector<const float*> ptrs;
  for (size_t i = 0; i < g.vals.size(); ++i) {
    const HostArray* v = g.vals[i];
    if (v->dev_id == home) { ptrs.push_back(v->dptr); continue; }
    float* dst = stage[i].Reserve<float>(home, n * 4);
    Join(v->dev_id, home);                                 // the previous reduce on home has read this staging buffer
    K::Check(L.memcpy_peer(dst, home, v->dptr, v->dev_id, n * 4, Str(v->dev_id)), "KVStore peer copy");
    Join(home, v->dev_id);
    ptrs.push_back(dst);
  }
  return ptrs;
}

// out = ptrs[0] + ptrs[1] + ... on `home`, 8 values per launch; with thr > 0 the last launch also quantises (residual / words on home)
inline void DeviceSum(int home, const std::vector<const float*>& ptrs, float* out, size_t n, float thr, float* residual, void* words) {
  const K::Lib& L = K::Get();
  K::Stream s = Str(home);
  K::Check(L.set_device(home), "KVStore");
  size_t i = 0;
  std::vector<const float*> chunk;
  while (i < ptrs.size()) {
    chunk.clear();
    if (i > 0) chunk.push_back(out);
    while (chunk.size() < 8 && i < ptrs.size()) chunk.push_back(ptrs[i++]);
    const bool last = i == ptrs.size();
    K::Check(L.kv_sum_quantize(out, chunk.data(), static_cast<int>(chunk.size()), static_cast<long long>(n), last ? residual : nullptr,
                               last ? words : nullptr, last ? thr : 0.f, s),
             "gx_kv_sum_quantize");
  }
}

// ================================================================================================ in-process stores
class LocalStore {
 public:
  LocalStore(const std::string& type, bool device) : type_(type), device_(device) {}
  bool device_store() const { return device_; }

  void SetUpdater(Updater u, void* arg) { std::lock_guard<std::recursive_mutex> lk(mu_); updater_ = u; updater_arg_ = arg; }
  void SetGradientCompression(const std::string& type, float thr) {
    std::lock_guard<std::recursive_mutex> lk(mu_);
    if (type == "none") { thr_ = 0.f; return; }
    if (type != "2bit") throw std::runtime_error("GXKVStoreSetGradientCompression: unknown type '" + type + "' for a '" + type_ + "' store (none | 2bit)");
    if (!device_) throw std::runtime_error("GXKVStoreSetGradientCompression: gradient compression is not supported for a '" + type_ + "' store (use 'device')");
    if (!(thr > 0.f)) throw std::runtime_error("GXKVStoreSetGradientCompression: threshold must be greater than 0");
    thr_ = thr;
  }

  void Init(uint32_t num, const int* keys, void** vals) {
    const char* fn = "GXKVStoreInitND";
    std::lock_guard<std::recursive_mutex> lk(mu_);
    std::vector<Group> gs = GroupByKey(fn, num, keys, vals);
    for (const Group& g : gs) {
      if (g.vals.size() > 1) Fail(fn, g.key, "repeated in one init");
      if (store_.count(g.key)) Fail(fn, g.key, "already initialised");
    }
    for (const Group& g : gs) {
      const HostArray* v = g.vals[0];
      auto e = std::make_unique<Entry>();
      e->shape = v->rec.shape; e->dtype = v->rec.dtype; e->n = static_cast<size_t>(gxrt::Prod(v->rec.shape));
      if (device_ && v->device()) {
        e->home = v->dev_id;
        e->stored.reset(capi::NewDeviceArray(e->shape, e->home));
        K::Check(K::Get().memcpy(e->stored->dptr, v->dptr, e->n * 4, 3, Str(e->home)), fn);
      } else {
        e->stored.reset(new HostArray());
        e->stored->rec = capi::HostCopy(v);
      }
      store_[g.key] = std::move(e);
    }
  }

  void Push(uint32_t num, const int* keys, void** vals) {
    const char* fn = "GXKVStorePushND";
    std::lock_guard<std::recursive_mutex> lk(mu_);
    std::vector<Group> gs = GroupByKey(fn, num, keys, vals);
    for (const Group& g : gs) Check(fn, g);
    for (const Group& g : gs) {
      Entry& e = *store_[g.key];
      HostArray* target = updater_ ? Recv(e) : e.stored.get();
      if (e.home < 0) ReduceToHost(fn, g, e, target);
      else if (g.device()) ReduceOnDevice(g, e, target);
      else {
        std::vector<const void*> src;
        for (const HostArray* v : g.vals) src.push_back(v->rec.data.data());
        e.host_scratch.resize(e.n * 4);
        HostSum(fn, g.key, 0, src, &e.host_scratch[0], e.n);
        K::Check(K::Get().memcpy(target->dptr, e.host_scratch.data(), e.n * 4, 1, Str(e.home)), fn);   // pageable: staged before return
      }
      if (updater_) updater_(g.key, e.recv.get(), e.stored.get(), updater_arg_);
    }
  }

  void Pull(uint32_t num, const int* keys, void** outs) {
    const char* fn = "GXKVStorePullND";
    std::lock_guard<std::recursive_mutex> lk(mu_);
    std::vector<Group> gs = GroupByKey(fn, num, keys, outs);
    for (const Group& g : gs) Check(fn, g);
    const K::Lib* L = nullptr;
    for (const Group& g : gs) {
      Entry& e = *store_[g.key];
      for (HostArray* o : g.vals) {
        if (o == e.stored.get()) continue;
        if (e.home < 0) {
          if (!o->device()) { std::memcpy(&o->rec.data[0], e.stored->rec.data.data(), e.stored->rec.data.size()); continue; }
          L = &K::Get();
          K::Check(L->memcpy(o->dptr, e.stored->rec.data.data(), e.n * 4, 1, Str(o->dev_id)), fn);
        } else if (!o->device()) {
          L = &K::Get();
          K::Check(L->memcpy(&o->rec.data[0], e.stored->dptr, e.n * 4, 2, Str(e.home)), fn);
          K::Check(L->stream_sync(Str(e.home)), fn);
        } else {
          L = &K::Get();
          Join(o->dev_id, e.home);
          if (o->dev_id == e.home) K::Check(L->memcpy(o->dptr, e.stored->dptr, e.n * 4, 3, Str(e.home)), fn);
          else K::Check(L->memcpy_peer(o->dptr, o->dev_id, e.stored->dptr, e.home, e.n * 4, Str(o->dev_id)), fn);
          Join(e.home, o->dev_id);                            // a later push rewrites the stored value after this copy has read it
        }
      }
    }
  }

  // the stored value's home: -1 host, else the CUDA device (tests and tools)
  int Home(int key) {
    std::lock_guard<std::recursive_mutex> lk(mu_);
    auto it = store_.find(key);
    if (it == store_.end()) Fail("GXKVStoreGetHome", key, "not initialised");
    return it->second->home;
  }

 private:
  struct Entry {
    std::vector<int64_t> shape;
    int dtype = 0;
    size_t n = 0;
    int home = -1;                                  // -1: the host
    std::unique_ptr<HostArray> stored, recv;        // recv: the reduced sum handed to the updater
    std::vector<DevBuf> stage;                      // per position: a value (or its words) copied to the home GPU
    std::vector<DevBuf> residual, words;            // per position, on the value's GPU (2-bit)
    std::vector<Pinned> pinned;                     // per position: a device value on its way to a host reduce
    std::string host_scratch;
  };

  void Check(const char* fn, const Group& g) {
    auto it = store_.find(g.key);
    if (it == store_.end()) Fail(fn, g.key, "not initialised");
    const Entry& e = *it->second;
    for (const HostArray* v : g.vals) {
      if (v->rec.shape != e.shape) Fail(fn, g.key, "shape " + ShapeStr(v->rec.shape) + " does not match the stored " + ShapeStr(e.shape));
      if (v->rec.dtype != e.dtype) Fail(fn, g.key, "dtype flag " + std::to_string(v->rec.dtype) + " does not match the stored " + std::to_string(e.dtype));
    }
  }

  HostArray* Recv(Entry& e) {
    if (!e.recv) {
      if (e.home >= 0) e.recv.reset(capi::NewDeviceArray(e.shape, e.home));
      else { e.recv.reset(new HostArray()); e.recv->rec = e.stored->rec; }
    }
    return e.recv.get();
  }

  void ReduceToHost(const char* fn, const Group& g, Entry& e, HostArray* target) {
    std::vector<const void*> src;
    if (!g.device()) {
      for (const HostArray* v : g.vals) src.push_back(v->rec.data.data());
    } else {
      const K::Lib& L = K::Get();
      if (e.pinned.size() < g.vals.size()) e.pinned = std::vector<Pinned>(g.vals.size());
      std::set<int> devs;
      for (size_t i = 0; i < g.vals.size(); ++i) {
        const HostArray* v = g.vals[i];
        void* p = e.pinned[i].Reserve(e.n * 4);
        K::Check(L.memcpy(p, v->dptr, e.n * 4, 2, Str(v->dev_id)), fn);
        devs.insert(v->dev_id);
        src.push_back(p);
      }
      for (int d : devs) K::Check(L.stream_sync(Str(d)), fn);
    }
    HostSum(fn, g.key, e.dtype, src, &target->rec.data[0], e.n);
  }

  void ReduceOnDevice(const Group& g, Entry& e, HostArray* target) {
    const K::Lib& L = K::Get();
    const size_t k = g.vals.size();
    if (!(thr_ > 0.f) || k == 1) {
      DeviceSum(e.home, Gather(g, e.home, e.n, e.stage), target->dptr, e.n, 0.f, nullptr, nullptr);
      return;
    }
    // 2-bit (comm.h:545-589): quantise each value on its own GPU, move the words, dequantise + sum on home
    const size_t nwords = static_cast<size_t>(hips::GradientCompression::CompressedSize2Bit(static_cast<int64_t>(e.n)));
    if (e.residual.size() < k) { e.residual.resize(k); e.words.resize(k); }
    if (e.stage.size() < k) e.stage.resize(k);
    std::vector<const void*> ptrs;
    for (size_t i = 0; i < k; ++i) {
      const HostArray* v = g.vals[i];
      const int d = v->dev_id;
      float* res = e.residual[i].Reserve<float>(d, e.n * 4);
      void* w = e.words[i].Reserve(d, nwords * 4);
      if (d != e.home) Join(d, e.home);                     // the previous dequantise has read these words
      K::Check(L.set_device(d), "KVStore");
      const float* in = v->dptr;
      K::Check(L.kv_sum_quantize(nullptr, &in, 1, static_cast<long long>(e.n), res, w, thr_, Str(d)), "gx_kv_sum_quantize");
      if (d == e.home) { ptrs.push_back(w); continue; }
      void* dst = e.stage[i].Reserve(e.home, nwords * 4);
      K::Check(L.memcpy_peer(dst, e.home, w, d, nwords * 4, Str(d)), "KVStore peer copy");
      Join(e.home, d);
      ptrs.push_back(dst);
    }
    K::Check(L.set_device(e.home), "KVStore");
    for (size_t i = 0; i < k; i += 8) {
      const int cnt = static_cast<int>(std::min<size_t>(8, k - i));
      K::Check(L.kv_dequant_sum(target->dptr, ptrs.data() + i, cnt, static_cast<long long>(e.n), thr_, i > 0 ? 1 : 0, Str(e.home)), "gx_kv_dequant_sum");
    }
  }

  std::string type_;
  bool device_;
  float thr_ = 0.f;
  Updater updater_ = nullptr;
  void* updater_arg_ = nullptr;
  std::recursive_mutex mu_;
  std::map<int, std::unique_ptr<Entry>> store_;
};

// ================================================================================================ NDArray forms on the parameter-server plane
class DistND {
 public:
  explicit DistND(hips::KVStoreDist* kv) : kv_(kv) {}

  // the raw-buffer GXKVStoreInit of `key`: later NDArray calls check against it
  void NoteRawInit(int key, size_t elems, int dtype) {
    std::lock_guard<std::mutex> lk(mu_);
    auto& e = store_[key];
    if (!e) { e.reset(new Entry()); e->n = elems; e->dtype = dtype; e->raw = true; }
  }

  void Init(uint32_t num, const int* keys, void** vals) {
    const char* fn = "GXKVStoreInitND";
    std::vector<Group> gs = GroupByKey(fn, num, keys, vals);
    {
      std::lock_guard<std::mutex> lk(mu_);
      for (const Group& g : gs) {
        if (g.vals.size() > 1) Fail(fn, g.key, "repeated in one init");
        if (store_.count(g.key)) Fail(fn, g.key, "already initialised");
      }
    }
    for (const Group& g : gs) {
      const HostArray* v = g.vals[0];
      auto e = std::make_unique<Entry>();
      e->shape = v->rec.shape; e->dtype = v->rec.dtype; e->n = static_cast<size_t>(gxrt::Prod(v->rec.shape));
      e->home = v->device() ? v->dev_id : -1;
      const gxrt::NDRec rec = capi::HostCopy(v);
      kv_->Init(g.key, rec.data.data(), e->n, e->dtype);
      std::lock_guard<std::mutex> lk(mu_);
      store_[g.key] = std::move(e);
    }
  }

  void Push(uint32_t num, const int* keys, void** vals, int priority) {
    const char* fn = "GXKVStorePushND";
    std::vector<Group> gs = GroupByKey(fn, num, keys, vals);
    std::vector<Entry*> es = Lookup(fn, gs);
    for (size_t gi = 0; gi < gs.size(); ++gi) {
      const Group& g = gs[gi];
      Entry& e = *es[gi];
      if (e.push_handle >= 0) { kv_->Wait(e.push_handle); e.push_handle = -1; }   // its staging buffer is about to be rewritten
      if (!g.device()) {
        std::vector<const void*> src;
        for (const HostArray* v : g.vals) src.push_back(v->rec.data.data());
        e.host_stage.resize(e.n * gxrt::FlagSize(e.dtype));
        HostSum(fn, g.key, e.dtype, src, &e.host_stage[0], e.n);
        e.push_handle = kv_->Push(g.key, e.host_stage.data(), e.n, e.dtype, priority);
        continue;
      }
      if (e.dtype != 0) Fail(fn, g.key, "device values need a float32 key");
      const K::Lib& L = K::Get();
      if (e.home < 0) e.home = g.vals[0]->dev_id;
      const int home = e.home;
      const bool two_bit = kv_->gradient_compression().type() == hips::CompressionType::kTwoBit;
      std::vector<const float*> ptrs = Gather(g, home, e.n, e.stage);
      if (two_bit) {
        const size_t nwords = static_cast<size_t>(hips::GradientCompression::CompressedSize2Bit(static_cast<int64_t>(e.n)));
        float* res = e.residual.Reserve<float>(home, e.n * 4);
        void* w = e.words.Reserve(home, nwords * 4);
        float* sum = ptrs.size() > 1 ? e.merge.Reserve<float>(home, e.n * 4) : nullptr;
        if (sum) DeviceSum(home, ptrs, sum, e.n, kv_->gradient_compression().threshold(), res, w);
        else {
          K::Check(L.set_device(home), "KVStore");
          K::Check(L.kv_sum_quantize(nullptr, ptrs.data(), 1, static_cast<long long>(e.n), res, w, kv_->gradient_compression().threshold(), Str(home)),
                   "gx_kv_sum_quantize");
        }
        void* pin = e.push_pin.Reserve(nwords * 4);
        K::Check(L.memcpy(pin, w, nwords * 4, 2, Str(home)), fn);
        K::Check(L.stream_sync(Str(home)), fn);
        e.push_handle = kv_->PushPacked2Bit(g.key, static_cast<const uint32_t*>(pin), e.n, priority);
      } else {
        const float* src = ptrs[0];
        if (ptrs.size() > 1) { float* sum = e.merge.Reserve<float>(home, e.n * 4); DeviceSum(home, ptrs, sum, e.n, 0.f, nullptr, nullptr); src = sum; }
        void* pin = e.push_pin.Reserve(e.n * 4);
        K::Check(L.memcpy(pin, src, e.n * 4, 2, Str(home)), fn);
        K::Check(L.stream_sync(Str(home)), fn);
        e.push_handle = kv_->Push(g.key, pin, e.n, 0, priority);
      }
    }
  }

  void Pull(uint32_t num, const int* keys, void** outs, int priority) {
    const char* fn = "GXKVStorePullND";
    std::vector<Group> gs = GroupByKey(fn, num, keys, outs);
    std::vector<Entry*> es = Lookup(fn, gs);
    std::vector<int> handles;
    for (size_t gi = 0; gi < gs.size(); ++gi) {
      const Group& g = gs[gi];
      Entry& e = *es[gi];
      void* dst;
      if (g.device()) {
        if (e.dtype != 0) Fail(fn, g.key, "device outputs need a float32 key");
        if (e.pull_dev >= 0) K::Check(K::Get().stream_sync(Str(e.pull_dev)), fn);     // the previous host-to-device copy has left the buffer
        e.pull_dev = -1;
        dst = e.pull_pin.Reserve(e.n * 4);
      } else {
        dst = &g.vals[0]->rec.data[0];
      }
      handles.push_back(kv_->Pull(g.key, dst, e.n, e.dtype, priority));
    }
    for (int h : handles) kv_->Wait(h);
    for (size_t gi = 0; gi < gs.size(); ++gi) {
      const Group& g = gs[gi];
      Entry& e = *es[gi];
      HostArray* first = g.vals[0];
      if (!g.device()) {
        for (size_t i = 1; i < g.vals.size(); ++i)
          if (g.vals[i] != first) std::memcpy(&g.vals[i]->rec.data[0], first->rec.data.data(), first->rec.data.size());
        continue;
      }
      const K::Lib& L = K::Get();
      K::Check(L.memcpy(first->dptr, e.pull_pin.p, e.n * 4, 1, Str(first->dev_id)), fn);
      e.pull_dev = first->dev_id;
      for (size_t i = 1; i < g.vals.size(); ++i) {
        HostArray* o = g.vals[i];
        if (o == first) continue;
        Join(o->dev_id, first->dev_id);
        if (o->dev_id == first->dev_id) K::Check(L.memcpy(o->dptr, first->dptr, e.n * 4, 3, Str(o->dev_id)), fn);
        else K::Check(L.memcpy_peer(o->dptr, o->dev_id, first->dptr, first->dev_id, e.n * 4, Str(o->dev_id)), fn);
        Join(first->dev_id, o->dev_id);
      }
    }
  }

 private:
  struct Entry {
    std::vector<int64_t> shape;                     // empty for keys initialised through the raw-buffer form (checked by size)
    size_t n = 0;
    int dtype = 0;
    bool raw = false;
    int home = -1;                                  // GPU that reduces device values
    int push_handle = -1, pull_dev = -1;
    std::string host_stage;
    Pinned push_pin, pull_pin;
    DevBuf merge, residual, words;
    std::vector<DevBuf> stage;
  };

  std::vector<Entry*> Lookup(const char* fn, const std::vector<Group>& gs) {
    std::lock_guard<std::mutex> lk(mu_);
    std::vector<Entry*> es;
    for (const Group& g : gs) {
      auto it = store_.find(g.key);
      if (it == store_.end()) Fail(fn, g.key, "not initialised");
      Entry* e = it->second.get();
      for (const HostArray* v : g.vals) {
        const size_t n = static_cast<size_t>(gxrt::Prod(v->rec.shape));
        if (e->raw ? n != e->n : v->rec.shape != e->shape)
          Fail(fn, g.key, "shape " + ShapeStr(v->rec.shape) + " does not match the initialised " + (e->raw ? std::to_string(e->n) + " elements" : ShapeStr(e->shape)));
        if (v->rec.dtype != e->dtype) Fail(fn, g.key, "dtype flag " + std::to_string(v->rec.dtype) + " does not match the initialised " + std::to_string(e->dtype));
      }
      es.push_back(e);
    }
    return es;
  }

  hips::KVStoreDist* kv_;
  std::mutex mu_;
  std::map<int, std::unique_ptr<Entry>> store_;
};

}  // namespace kvnd
}  // namespace gxrt
