// KVStoreDist — worker endpoint of the local PS (and process bootstrap for every role).
//
// Parity: src/kvstore/kvstore_dist.h — ctor/dtor (:52-88: ps::StartAsync, barrier, kStopServer from rank 0 on shutdown), InitImpl
// (:308-322: rank 0 pushes the initial value, then Barrier), Push_/PushDefault (:460-625: key -> server sharding, ZPush), PushCompressed
// (:530-563: 2-bit with residual), EncodeP3Key + P3_ZPush (:763-799, :565-601: priority slices, the response carries the parameters and
// pull becomes a no-op), PullImpl (:330-418), SetGradientCompression (:192-198), Barrier (:207-210: workers only), SendCommandToServers
// (:212-215), get_num_dead_node (:225-234), RunServer (:236-257).  KVStore::Create (src/kvstore/kvstore.cc:41-82): the rank-0 worker of
// every party sends kSyncMode to its servers; with a `_sync` type the master worker also sends kSyncGlobalMode.
//
// Buffers are raw host pointers owned by the caller (Python keeps pinned staging tensors alive until Wait); all calls are thread-safe.
#pragma once
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "gradient_compression.h"
#include "key_codec.h"
#include "kv_app.h"
#include "kvstore_dist_server.h"

namespace hips {

class KVStoreDist {
 public:
  explicit KVStoreDist(const std::string& type) : type_(type) {
    Postoffice* po = Postoffice::Get();
    po->InitEnvironment();
    Environment* env = Environment::Get();
    bigarray_bound_ = static_cast<size_t>(env->GetFloat("MXNET_KVSTORE_BIGARRAY_BOUND", 1000000));
    size_lower_bound_ = static_cast<size_t>(env->GetFloat("MXNET_KVSTORE_SIZE_LOWER_BOUND", 200000));
    enable_p3_ = env->GetInt("ENABLE_P3", 0) != 0;
    if (po->is_worker()) {
      ps_worker_.reset(new KVWorker(0, 0));
      po->Start(0, true);
      started_ = true;
      // KVStore::Create: rank-0 worker configures the party's servers (a recovered worker finds them configured)
      if (po->is_recovery()) return;
      if (type.find("dist") != std::string::npos && rank() == 0) SendCommandToServers(static_cast<int>(CommandType::kSyncMode), "");
      if (type.find("_sync") != std::string::npos && po->is_master_worker()) SendCommandToServers(static_cast<int>(CommandType::kSyncGlobalMode), "");
    }
  }
  ~KVStoreDist() { Shutdown(); }

  void Shutdown() {
    if (!started_) return;
    started_ = false;
    Postoffice* po = Postoffice::Get();
    if (po->is_worker()) {
      WaitAll();
      Barrier();
      if (rank() == 0 && !po->is_master_worker()) SendCommandToServers(static_cast<int>(CommandType::kStopServer), "");
      po->set_finalizing();
      ps_worker_.reset();
    }
    po->Finalize(0, true);
  }

  // ---- roles / sizes ------------------------------------------------------------------------------------------------
  const std::string& type() const { return type_; }
  int rank() { return Postoffice::Get()->my_rank(kLocal); }
  int num_workers() { return Postoffice::Get()->num_workers(); }
  int num_all_workers() { return Postoffice::Get()->num_all_workers(); }
  bool is_master_worker() { return Postoffice::Get()->is_master_worker(); }
  bool is_recovery() { return Postoffice::Get()->is_recovery(); }
  int num_dead_node(int node_id, int timeout) {
    int n = 0;
    for (int r : Postoffice::Get()->GetDeadNodes(timeout, kLocal)) if (r & node_id) ++n;
    return n;
  }

  // ---- server / scheduler processes -----------------------------------------------------------------------------------
  // blocks until the job ends.  controller(head, body) / updater(key, grad, weight, n) are foreign (Python) callbacks.
  void RunServer(const KVStoreDistServer::Controller& controller, const KVStoreDistServer::Updater& updater,
                 const std::function<void(KVStoreDistServer*)>& on_ready = nullptr) {
    Postoffice* po = Postoffice::Get();
    if (po->is_server()) {
      server_.reset(new KVStoreDistServer());
      server_->set_controller(controller);
      if (updater) server_->set_updater(updater);
    }
    po->Start(0, true);
    started_ = true;
    if (server_) {
      if (on_ready) on_ready(server_.get());
      server_->Run();
    }
    po->set_finalizing();
    po->Finalize(0, true);
    started_ = false;
    server_.reset();
  }
  KVStoreDistServer* server() { return server_.get(); }

  // ---- data -----------------------------------------------------------------------------------------------------------
  void Init(int key, const void* data, size_t elems, int dtype) {
    { std::lock_guard<std::mutex> lk(mu_); info_[key] = KeyInfo{elems, dtype}; }
    if (Postoffice::Get()->is_recovery()) return;   // the key already lives on the servers; the others are past this barrier (kvstore_dist.h:321)
    if (rank() == 0) {
      const int h = PushImpl(key, data, elems, dtype, 0, /*allow_compress=*/false);
      Wait(h);
    }
    Barrier();
  }
  // returns a handle for Wait()
  int Push(int key, const void* data, size_t elems, int dtype, int priority) { return PushImpl(key, data, elems, dtype, priority, true); }
  // a float32 push of `elems` values that the caller already quantised to 2-bit words (with its own residual, e.g. on a GPU): the same
  // message as Push sends under 2-bit compression.  The caller keeps `words` alive until the handle was waited.
  int PushPacked2Bit(int key, const uint32_t* words, size_t elems, int priority) {
    HIPS_CHECK_MSG(gc_.type() == CompressionType::kTwoBit, "PushPacked2Bit needs 2-bit compression");
    const int h = Track({ZPushWords(key, words, static_cast<size_t>(GradientCompression::CompressedSize2Bit(static_cast<int64_t>(elems))), priority, nullptr)});
    { std::lock_guard<std::mutex> lk(mu_); last_push_[key] = h; }
    return h;
  }
  const GradientCompression& gradient_compression() const { return gc_; }

  int Pull(int key, void* out, size_t elems, int dtype, int priority) {
    // ordering: a pull of `key` observes the effect of this worker's previous push of `key` (reference: shared comm_buf_ engine var)
    int pending = -1;
    {
      std::lock_guard<std::mutex> lk(mu_);
      auto it = last_push_.find(key);
      if (it != last_push_.end()) { pending = it->second; last_push_.erase(it); }
    }
    if (pending >= 0) Wait(pending);
    if (TSNode* t = ps_worker_->ts()) {
      // intra-party TSEngine: after the first synchronisation round the parameters arrive through the relay broadcast — wait (in Wait())
      // for the version that contains this worker's latest push instead of sending a pull request
      int version = 0;
      { std::lock_guard<std::mutex> lk(mu_); auto it = ts_push_count_.find(key); if (it != ts_push_count_.end()) version = it->second; }
      if (version > 0) {
        (void)t;
        std::lock_guard<std::mutex> lk(mu_);
        const int h = next_handle_++;
        handles_[h] = {};
        relay_waits_[h] = RelayWait{key, version, out, elems * static_cast<size_t>(DTypeSize(dtype))};
        return h;
      }
    }
    if (enable_p3_) {  // P3: the push response already carried the parameters (filled by the push callback before Wait returned)
      std::lock_guard<std::mutex> lk(mu_);
      auto pt = p3_buf_.find(key);
      if (pt != p3_buf_.end()) {
        HIPS_CHECK(pt->second.size() == elems * DTypeSize(dtype));
        memcpy(out, pt->second.data(), pt->second.size());
        p3_buf_.erase(pt);
        const int h = next_handle_++;
        handles_[h] = {};
        return h;
      }
    }
    const int bytes = DTypeSize(dtype);
    PSKVPlan plan = EncodeKeyPlan(kLocal, key, elems, bytes, bigarray_bound_, Pinned(elems, dtype));
    SArray<Key> keys;
    for (Key k : plan.keys) keys.push_back(k);
    auto vals = std::make_shared<SArray<char>>(static_cast<char*>(out), elems * bytes, false);
    auto lens = std::make_shared<SArray<int>>();
    const int cmd = GetCommandType(RequestType::kDefaultPushPull, dtype);
    const int ts = ps_worker_->ZPull(keys, vals.get(), lens.get(), cmd, [vals, lens]() {}, priority, key);
    return Track({ts});
  }

  // ---- row_sparse (reference PushRowSparse :628-657, PullRowSparse_ :660-702): only the listed rows travel.  Payload layout:
  //      int64 nrows, int64 row_len, int64 ids[nrows], then (push only) float rows[nrows][row_len]
  int PushRows(int key, const int64_t* ids, size_t nrows, const float* rows, size_t row_len, int priority) {
    auto buf = std::make_shared<std::vector<char>>((2 + nrows) * sizeof(int64_t) + nrows * row_len * sizeof(float));
    int64_t* hdr = reinterpret_cast<int64_t*>(buf->data());
    hdr[0] = static_cast<int64_t>(nrows); hdr[1] = static_cast<int64_t>(row_len);
    if (nrows) { memcpy(hdr + 2, ids, nrows * sizeof(int64_t)); memcpy(hdr + 2 + nrows, rows, nrows * row_len * sizeof(float)); }
    const auto& krs = Postoffice::Get()->GetServerKeyRanges(kLocal);
    SArray<Key> keys; keys.push_back(krs[(key * 9973) % krs.size()].begin() + static_cast<Key>(key));
    SArray<char> vals(buf->data(), buf->size(), false);
    SArray<int> lens; lens.push_back(static_cast<int>(buf->size()));
    const int cmd = GetCommandType(RequestType::kRowSparsePushPull, kFloat32);
    const int h = Track({ps_worker_->ZPush(keys, vals, lens, cmd, [buf]() {}, priority, key)});
    { std::lock_guard<std::mutex> lk(mu_); last_push_[key] = h; }
    return h;
  }
  int PullRows(int key, const int64_t* ids, size_t nrows, float* out, size_t row_len, int priority) {
    int pending = -1;
    { std::lock_guard<std::mutex> lk(mu_); auto it = last_push_.find(key); if (it != last_push_.end()) { pending = it->second; last_push_.erase(it); } }
    if (pending >= 0) Wait(pending);
    auto req = std::make_shared<std::vector<char>>((2 + nrows) * sizeof(int64_t));
    int64_t* hdr = reinterpret_cast<int64_t*>(req->data());
    hdr[0] = static_cast<int64_t>(nrows); hdr[1] = static_cast<int64_t>(row_len);
    if (nrows) memcpy(hdr + 2, ids, nrows * sizeof(int64_t));
    const auto& krs = Postoffice::Get()->GetServerKeyRanges(kLocal);
    SArray<Key> keys; keys.push_back(krs[(key * 9973) % krs.size()].begin() + static_cast<Key>(key));
    auto vals = std::make_shared<SArray<char>>(reinterpret_cast<char*>(out), nrows * row_len * sizeof(float), false);
    auto lens = std::make_shared<SArray<int>>();
    SArray<char> payload(req->data(), req->size(), false);
    const int cmd = GetCommandType(RequestType::kRowSparsePushPull, kFloat32);
    return Track({ps_worker_->ZPull(keys, vals.get(), lens.get(), cmd, [vals, lens, req]() {}, priority, key, &payload)});
  }

  void Wait(int handle) {
    std::vector<int> tss;
    RelayWait rw;
    {
      std::lock_guard<std::mutex> lk(mu_);
      auto it = handles_.find(handle);
      if (it == handles_.end()) return;
      tss = it->second;
      handles_.erase(it);
      auto rt = relay_waits_.find(handle);
      if (rt != relay_waits_.end()) { rw = rt->second; relay_waits_.erase(rt); }
    }
    for (int ts : tss) ps_worker_->Wait(ts);
    if (rw.out != nullptr) ps_worker_->ts()->WaitRelayed(rw.key, rw.version, rw.out, rw.nbytes);
  }
  // (peer merges received, relay transfers sent) by this worker's TSEngine node — 0,0 when the overlay is off
  std::pair<long, long> ts_stats() {
    TSNode* t = ps_worker_ ? ps_worker_->ts() : nullptr;
    return t ? std::make_pair(t->merges_received(), t->relays_sent()) : std::make_pair(0L, 0L);
  }
  void WaitAll() {
    std::vector<int> hs;
    { std::lock_guard<std::mutex> lk(mu_); for (auto& kv : handles_) hs.push_back(kv.first); }
    for (int h : hs) Wait(h);
  }

  void SetGradientCompression(const std::string& type, float threshold) {
    {
      // the key -> server plan depends on the compression type, so it has to be fixed before the first key exists (the reference makes the
      // same demand: "Gradient compression must be set before init", kvstore.py set_gradient_compression)
      std::lock_guard<std::mutex> lk(mu_);
      HIPS_CHECK_MSG(info_.empty(), "set_gradient_compression must be called before the first kv.init");
    }
    gc_.SetParams(type, threshold);
    // master worker: tell the global servers (rank 0 relays to the parties' servers); ordinary rank-0 worker: tell the local server
    if (rank() == 0 || is_master_worker()) SendCommandToServers(static_cast<int>(CommandType::kSetGradientCompression), gc_.EncodeParams());
  }
  void Barrier() { Postoffice::Get()->Barrier(0, kWorkerGroup, kLocal); }
  void SendCommandToServers(int head, const std::string& body) {
    const int ts = ps_worker_->Request(head, body, kServerGroup, kLocal);
    ps_worker_->Wait(ts);
  }
  size_t send_bytes() { return Postoffice::Get()->van(kLocal)->send_bytes(); }
  size_t recv_bytes() { return Postoffice::Get()->van(kLocal)->recv_bytes(); }

 private:
  struct KeyInfo { size_t elems; int dtype; };
  struct RelayWait { int key = 0, version = 0; void* out = nullptr; size_t nbytes = 0; };
  int Track(const std::vector<int>& tss) {
    std::lock_guard<std::mutex> lk(mu_);
    const int h = next_handle_++;
    handles_[h] = tss;
    return h;
  }
  int NewDoneHandle() { return Track({}); }
  // compressed keys live un-partitioned on their hashed server (key_codec.h CompressionPinsKey): init, push and pull agree on ONE plan
  bool Pinned(size_t elems, int dtype) const { return CompressionPinsKey(static_cast<int>(gc_.type()), elems, dtype, size_lower_bound_); }

  // the 2-bit wire message of `key`: `nwords` packed words on its hashed server; `keep` holds the words alive until the send is done
  int ZPushWords(int key, const uint32_t* words, size_t nwords, int priority, const std::function<void()>& keep) {
    const auto& krs = Postoffice::Get()->GetServerKeyRanges(kLocal);
    SArray<Key> keys; keys.push_back(krs[(key * 9973) % krs.size()].begin() + static_cast<Key>(key));
    SArray<char> vals(reinterpret_cast<char*>(const_cast<uint32_t*>(words)), nwords * 4, false);
    SArray<int> lens; lens.push_back(static_cast<int>(nwords * 4));
    const int cmd = GetCommandType(RequestType::kCompressedPushPull, kFloat32);
    return ps_worker_->ZPush(keys, vals, lens, cmd, keep, priority, key);
  }

  int PushImpl(int key, const void* data, size_t elems, int dtype, int priority, bool allow_compress) {
    const int bytes = DTypeSize(dtype);
    std::vector<int> tss;
    if (allow_compress && gc_.type() == CompressionType::kTwoBit && dtype == kFloat32) {
      // worker -> local server 2-bit path (reference PushCompressed): quantise with the per-key residual, 16x smaller payload
      std::vector<float>* res;
      { std::lock_guard<std::mutex> lk(mu_); res = &residual_[key]; if (res->size() != elems) res->assign(elems, 0.f); }
      auto words = std::make_shared<std::vector<uint32_t>>(GradientCompression::CompressedSize2Bit(static_cast<int64_t>(elems)));
      gc_.Quantize2Bit(static_cast<const float*>(data), res->data(), words->data(), static_cast<int64_t>(elems));
      tss.push_back(ZPushWords(key, words->data(), words->size(), priority, [words]() {}));
    } else if (enable_p3_ && allow_compress) {
      // P3: the response of the push carries the updated parameters; keep them for the following pull
      auto buf = std::make_shared<std::vector<char>>(static_cast<const char*>(data), static_cast<const char*>(data) + elems * bytes);
      PSKVPlan plan = EncodeKeyPlan(kLocal, key, elems, bytes, bigarray_bound_, Pinned(elems, dtype));
      SArray<Key> keys; for (Key k : plan.keys) keys.push_back(k);
      SArray<int> lens; for (int l : plan.lens) lens.push_back(l);
      SArray<char> vals(buf->data(), buf->size(), false);
      const int cmd = GetCommandType(RequestType::kDefaultPushPull, dtype);
      tss.push_back(ps_worker_->P3_ZPush(keys, vals, lens, cmd, [this, key, buf]() { std::lock_guard<std::mutex> lk(mu_); p3_buf_[key] = *buf; }, priority, key));
    } else {
      PSKVPlan plan = EncodeKeyPlan(kLocal, key, elems, bytes, bigarray_bound_, Pinned(elems, dtype));
      SArray<Key> keys; for (Key k : plan.keys) keys.push_back(k);
      SArray<int> lens; for (int l : plan.lens) lens.push_back(l);
      SArray<char> vals(static_cast<char*>(const_cast<void*>(data)), elems * bytes, false);
      const int cmd = GetCommandType(RequestType::kDefaultPushPull, dtype);
      const bool via_ts = allow_compress && ps_worker_->ts() != nullptr && keys.size() == 1;
      tss.push_back(ps_worker_->ZPush(keys, vals, lens, cmd, nullptr, priority, key, via_ts));
      if (via_ts) { std::lock_guard<std::mutex> lk(mu_); ++ts_push_count_[key]; }
    }
    const int h = Track(tss);
    { std::lock_guard<std::mutex> lk(mu_); last_push_[key] = h; }
    return h;
  }

  std::string type_;
  std::unique_ptr<KVWorker> ps_worker_;
  std::unique_ptr<KVStoreDistServer> server_;
  GradientCompression gc_;
  std::mutex mu_;
  std::unordered_map<int, KeyInfo> info_;
  std::unordered_map<int, std::vector<int>> handles_;
  std::unordered_map<int, int> last_push_;
  std::unordered_map<int, int> ts_push_count_;            // TSEngine: rounds this worker contributed to, per key (= expected relay version)
  std::unordered_map<int, RelayWait> relay_waits_;
  std::unordered_map<int, std::vector<float>> residual_;
  std::unordered_map<int, std::vector<char>> p3_buf_;
  int next_handle_ = 1;
  size_t bigarray_bound_ = 1000000, size_lower_bound_ = 200000;
  bool enable_p3_ = false, started_ = false;
};

}  // namespace hips
