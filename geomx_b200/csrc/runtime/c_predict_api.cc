// C predict API: a minimal, Python-free interface to run inference from a symbol JSON and a `.params` blob (predict.h is the runtime).
//
// Parity (GX prefix, same argument lists): include/mxnet/c_predict_api.h
//   MXPredCreate :78, MXPredCreatePartialOut :111, MXPredCreateMultiThread :144, MXPredReshape :170, MXPredGetOutputShape :185,
//   MXPredSetInput :198, MXPredForward :207, MXPredPartialForward :224, MXPredGetOutput :233, MXPredFree :242, MXNDList{Create,Get,Free} :252-277.
// dev_type 1 (cpu) runs on the host: the planned predictor (predict.h), or the general executor for graphs outside its operator set.
// dev_type 2 (gpu) runs the planned predictor on device dev_id with sm_100a kernels (predict_device.h); there is no host fallback, and a
// graph the device runner cannot serve is refused at create.
// Errors: -1 + GXRTGetLastError() (shared with c_api_runtime.cc, thread-local).
#include <cstdint>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "host_array.h"
#include "predict.h"
#include "predict_device.h"
#include "train_exec.h"

#define GX_CAPI extern "C" __attribute__((visibility("default")))

extern "C" const char* GXRTGetLastError();
void GXRTSetLastError(const std::string& msg);          // c_api_runtime.cc

namespace {
using gxrt::predict::DevicePredictor;
using gxrt::predict::NDList;
using gxrt::predict::Predictor;
using gxrt::predict::Shape;

template <typename F>
int Guard(F&& f) {
  try { f(); return 0; }
  catch (const std::exception& e) { GXRTSetLastError(e.what()); return -1; }
  catch (...) { GXRTSetLastError("unknown error"); return -1; }
}
// Second engine behind the same ABI: graphs that use operators outside the planned predictor's set (predict.h: ~35 layer / elementwise
// operators, single outputs) run on the host executor of the graph runtime in inference mode (train_exec.h: the full operator table incl.
// multi-output nodes).  It keeps every activation (no arena reuse) — the price of generality; GXPredGetPlan reports that size.
class GraphPredictor {
 public:
  using ParamMap = std::map<std::string, std::pair<Shape, std::vector<float>>>;
  GraphPredictor(const std::string& json, const char* params, size_t param_size, const std::vector<std::string>& in_keys, const std::vector<Shape>& in_shapes,
                 const std::vector<std::string>& out_keys) {
    namespace G = gxrt::graph;
    sym_ = G::FromJSON(json);
    if (!out_keys.empty()) {                 // internal outputs by name ("fc1" or "fc1_output")
      const G::Symbol internals = G::GetInternals(sym_);
      G::Symbol picked;
      for (auto& k : out_keys) {
        bool found = false;
        for (auto& e : internals.outputs) if (e.node->name == k || G::OutputName(e) == k) { picked.outputs.push_back(e); found = true; break; }
        if (!found) throw std::runtime_error("output " + k + " is not a node of the graph");
      }
      sym_ = picked;
    }
    params_ = std::make_shared<ParamMap>();
    if (params != nullptr && param_size > 0) {
      gxrt::BufReader r(params, param_size);
      if (r.Get<uint64_t>() != gxrt::kListMagic) throw std::runtime_error("parameter blob: not an NDArray list");
      r.Get<uint64_t>();
      const uint64_t n = r.Get<uint64_t>();
      if (n > (1u << 24)) throw std::runtime_error("parameter blob: implausible array count");
      std::vector<gxrt::NDRec> recs;
      for (uint64_t i = 0; i < n; ++i) recs.push_back(gxrt::ReadArray(r));
      const uint64_t m = r.Get<uint64_t>();
      if (m != n) throw std::runtime_error("parameter blob: arrays are not named");
      for (uint64_t i = 0; i < m; ++i) {
        const uint64_t l = r.Get<uint64_t>();
        std::string name = r.Raw(l);
        if (name.compare(0, 4, "arg:") == 0 || name.compare(0, 4, "aux:") == 0) name = name.substr(4);
        (*params_)[name] = {recs[i].shape, gxrt::predict::ToFloat(recs[i])};
      }
    }
    for (size_t i = 0; i < in_keys.size(); ++i) input_shapes_[in_keys[i]] = in_shapes[i];
    Bind();
  }
  std::unique_ptr<GraphPredictor> Clone(const std::map<std::string, Shape>* new_shapes) const {
    std::unique_ptr<GraphPredictor> p(new GraphPredictor(*this));
    if (new_shapes) for (auto& kv : *new_shapes) {
      if (!p->input_shapes_.count(kv.first)) throw std::runtime_error("reshape: " + kv.first + " is not an input of this predictor");
      p->input_shapes_[kv.first] = kv.second;
    }
    p->Bind();
    return p;
  }
  void SetInput(const std::string& key, const float* data, size_t size) {
    auto it = inputs_.find(key);
    if (it == inputs_.end() || !input_shapes_.count(key)) throw std::runtime_error("SetInput: unknown input " + key);
    if (size != it->second.size()) throw std::runtime_error("SetInput: " + key + " expects " + std::to_string(it->second.size()) + " values, got " + std::to_string(size));
    memcpy(it->second.data(), data, size * sizeof(float));
  }
  void Forward() { ex_->Forward(false); }
  void PartialForward(int step, int* step_left) { if (step == 0) Forward(); *step_left = 0; }      // one step: this engine does not expose single operators
  size_t NumOutputs() const { return ex_->NumOutputs(); }
  const Shape& OutputShape(size_t i) const { if (i >= ex_->NumOutputs()) throw std::runtime_error("output index out of range"); return ex_->OutputShape(i); }
  void GetOutput(size_t i, float* out, size_t size) const {
    const Shape& s = OutputShape(i);
    if (size != static_cast<size_t>(gxrt::predict::Numel(s))) throw std::runtime_error("GetOutput: output " + std::to_string(i) + " has " + std::to_string(gxrt::predict::Numel(s)) + " values, buffer holds " + std::to_string(size));
    memcpy(out, ex_->OutputData(i), size * sizeof(float));
  }
  size_t ArenaBytes() const { return activation_bytes_; }
  size_t NumOps() const { return num_ops_; }

 private:
  GraphPredictor(const GraphPredictor& o) : sym_(o.sym_), params_(o.params_), input_shapes_(o.input_shapes_) {}
  void Bind() {
    namespace G = gxrt::graph;
    std::map<std::string, Shape> known = input_shapes_;
    const auto arg_names = G::ListArguments(sym_), aux_names = G::ListAuxiliaryStates(sym_);
    for (auto& n : arg_names) { auto p = params_->find(n); if (p != params_->end() && !known.count(n)) known[n] = p->second.first; }
    for (auto& n : aux_names) { auto p = params_->find(n); if (p != params_->end()) known[n] = p->second.first; }
    for (auto& kv : input_shapes_) if (std::find(arg_names.begin(), arg_names.end(), kv.first) == arg_names.end()) throw std::runtime_error("input " + kv.first + " is not an argument of the graph");
    const G::ShapeResult sr = G::InferShapes(sym_, known, false);
    std::map<std::string, Shape> by_name;
    for (auto& kv : sr.shape) if (kv.first->op == "null") by_name[kv.first->name] = kv.second;
    inputs_.clear();
    std::vector<gxrt::exec::Tensor> args, grads, aux;
    std::vector<int> reqs;
    auto bind = [&](const std::string& n, bool is_input) -> gxrt::exec::Tensor {
      auto p = params_->find(n);
      if (!is_input && p != params_->end()) {
        if (p->second.first != by_name.at(n)) throw std::runtime_error("parameter " + n + " has shape " + gxrt::predict::ShapeStr(p->second.first) + ", the graph needs " + gxrt::predict::ShapeStr(by_name.at(n)));
        return {p->second.second.data(), p->second.first};
      }
      auto& buf = inputs_[n];                      // inputs, and arguments that are in neither list (labels): zero-filled, never read in inference
      buf.assign(static_cast<size_t>(gxrt::predict::Numel(by_name.at(n))), 0.f);
      return {buf.data(), by_name.at(n)};
    };
    for (auto& n : arg_names) { args.push_back(bind(n, input_shapes_.count(n) > 0)); grads.push_back({nullptr, {}}); reqs.push_back(gxrt::exec::kNullOp); }
    for (auto& n : aux_names) {
      if (!params_->count(n)) throw std::runtime_error("auxiliary state " + n + " is not in the parameter file");
      aux.push_back(bind(n, false));
    }
    ex_.reset(new gxrt::exec::Executor(sym_, args, grads, reqs, aux));
    activation_bytes_ = 0; num_ops_ = 0;
    for (auto& kv : sr.shape) if (kv.first->op != "null") { activation_bytes_ += static_cast<size_t>(gxrt::predict::Numel(kv.second)) * G::NumOutputs(*kv.first) * sizeof(float); ++num_ops_; }
  }
  gxrt::graph::Symbol sym_;
  std::shared_ptr<ParamMap> params_;                 // shared between clones; inference never writes parameters (BatchNorm uses the running statistics)
  std::map<std::string, Shape> input_shapes_;
  std::map<std::string, std::vector<float>> inputs_;
  std::unique_ptr<gxrt::exec::Executor> ex_;
  size_t activation_bytes_ = 0, num_ops_ = 0;
};

struct Handle {
  std::unique_ptr<Predictor> pred;       // the planned predictor (predict.h) ...
  std::unique_ptr<GraphPredictor> gen;   // ... or the general executor, when the graph needs operators the planned one does not have ...
  std::unique_ptr<DevicePredictor> dev;  // ... or the planned predictor on a GPU (dev_type 2)
  std::vector<uint32_t> shape_out;       // GetOutputShape hands out a pointer that stays valid until the next call on this handle
  const gxrt::predict::GraphPlan& plan() const { if (dev) return *dev; if (pred) return *pred; throw std::logic_error("no planned predictor"); }
};
Handle* H(void* h) { if (!h) throw std::runtime_error("null predictor handle"); return static_cast<Handle*>(h); }
// a device handle makes its device current before anything else
Handle* HD(void* h, const char* fn) { Handle* x = H(h); if (x->dev) x->dev->SetDevice(fn); return x; }
// a create: every error on a GPU also says where graphs the native device runner cannot serve can go instead
template <typename F>
int CreateGuard(int dev_type, F&& f) {
  return Guard([&] {
    try { f(); }
    catch (const std::exception& e) {
      if (dev_type != 2) throw;
      throw std::runtime_error(e.what() + std::string("; geomx_b200.predictor.Predictor(dev_type='gpu') serves graphs on the Python Executor"));
    }
  });
}

std::vector<Shape> Shapes(uint32_t n, const uint32_t* indptr, const uint32_t* data) {
  std::vector<Shape> out(n);
  for (uint32_t i = 0; i < n; ++i) {
    if (indptr[i + 1] < indptr[i] || indptr[i + 1] - indptr[i] > 8) throw std::runtime_error("input_shape_indptr is not a valid index pointer");
    out[i].assign(data + indptr[i], data + indptr[i + 1]);
  }
  return out;
}
void Make(Handle* h, const char* json, const void* params, int param_size, int dev_type, int dev_id, uint32_t n_in, const char** keys,
          const uint32_t* indptr, const uint32_t* shape_data, uint32_t n_out, const char** out_keys) {
  if (dev_type != 1 && dev_type != 2) throw std::runtime_error("dev_type " + std::to_string(dev_type) + " is not supported (1 CPU, 2 GPU)");
  if (json == nullptr) throw std::runtime_error("null symbol JSON");
  if (param_size < 0) throw std::runtime_error("negative param_size");
  std::vector<std::string> ik, ok;
  for (uint32_t i = 0; i < n_in; ++i) ik.emplace_back(keys[i]);
  for (uint32_t i = 0; i < n_out; ++i) ok.emplace_back(out_keys[i]);
  const auto shapes = Shapes(n_in, indptr, shape_data);
  if (dev_type == 2) {
    h->dev = std::make_unique<DevicePredictor>(std::string(json), static_cast<const char*>(params), static_cast<size_t>(param_size), ik, shapes, ok, dev_id);
    return;
  }
  try {
    h->pred = std::make_unique<Predictor>(std::string(json), static_cast<const char*>(params), static_cast<size_t>(param_size), ik, shapes, ok);
  } catch (const std::runtime_error& e) {
    const std::string msg = e.what();
    const bool unsupported = msg.find("is not supported by the native predictor") != std::string::npos || msg.find("secondary") != std::string::npos ||
                             msg.find("are supported by the native predictor") != std::string::npos || msg.find("is not a node of the graph") != std::string::npos;
    if (!unsupported) throw;
    try { h->gen = std::make_unique<GraphPredictor>(std::string(json), static_cast<const char*>(params), static_cast<size_t>(param_size), ik, shapes, ok); }
    catch (const std::exception& e2) { throw std::runtime_error(msg + "; the general executor could not run the graph either: " + e2.what()); }
  }
}
}  // namespace

GX_CAPI int GXPredCreate(const char* symbol_json, const void* param_bytes, int param_size, int dev_type, int dev_id, uint32_t num_input_nodes,
                         const char** input_keys, const uint32_t* input_shape_indptr, const uint32_t* input_shape_data, void** out) {
  return CreateGuard(dev_type, [&] {
    auto h = std::make_unique<Handle>();
    Make(h.get(), symbol_json, param_bytes, param_size, dev_type, dev_id, num_input_nodes, input_keys, input_shape_indptr, input_shape_data, 0, nullptr);
    *out = h.release();
  });
}
GX_CAPI int GXPredCreatePartialOut(const char* symbol_json, const void* param_bytes, int param_size, int dev_type, int dev_id, uint32_t num_input_nodes,
                                   const char** input_keys, const uint32_t* input_shape_indptr, const uint32_t* input_shape_data,
                                   uint32_t num_output_nodes, const char** output_keys, void** out) {
  return CreateGuard(dev_type, [&] {
    auto h = std::make_unique<Handle>();
    Make(h.get(), symbol_json, param_bytes, param_size, dev_type, dev_id, num_input_nodes, input_keys, input_shape_indptr, input_shape_data, num_output_nodes,
         output_keys);
    *out = h.release();
  });
}
// num_threads predictors over ONE copy of the graph and the parameters, each with its own inputs and activation arena (and, on a GPU, its
// own stream: the handles may serve from different threads at once)
GX_CAPI int GXPredCreateMultiThread(const char* symbol_json, const void* param_bytes, int param_size, int dev_type, int dev_id, uint32_t num_input_nodes,
                                    const char** input_keys, const uint32_t* input_shape_indptr, const uint32_t* input_shape_data, int num_threads, void** out) {
  return CreateGuard(dev_type, [&] {
    if (num_threads < 1) throw std::runtime_error("num_threads must be positive");
    std::vector<std::unique_ptr<Handle>> hs;
    hs.push_back(std::make_unique<Handle>());
    Make(hs[0].get(), symbol_json, param_bytes, param_size, dev_type, dev_id, num_input_nodes, input_keys, input_shape_indptr, input_shape_data, 0, nullptr);
    for (int i = 1; i < num_threads; ++i) {
      hs.push_back(std::make_unique<Handle>());
      if (hs[0]->dev) hs[i]->dev = hs[0]->dev->Clone(nullptr);
      else if (hs[0]->pred) hs[i]->pred = hs[0]->pred->Clone(nullptr);
      else hs[i]->gen = hs[0]->gen->Clone(nullptr);
    }
    for (int i = 0; i < num_threads; ++i) out[i] = hs[i].release();
  });
}
// a NEW handle with other input shapes that shares the parameters of `handle` (which stays valid)
GX_CAPI int GXPredReshape(uint32_t num_input_nodes, const char** input_keys, const uint32_t* input_shape_indptr, const uint32_t* input_shape_data, void* handle, void** out) {
  return Guard([&] {
    std::map<std::string, Shape> shapes;
    const auto list = Shapes(num_input_nodes, input_shape_indptr, input_shape_data);
    for (uint32_t i = 0; i < num_input_nodes; ++i) shapes[input_keys[i]] = list[i];
    auto h = std::make_unique<Handle>();
    Handle* src = HD(handle, "GXPredReshape");
    if (src->dev) h->dev = src->dev->Clone(&shapes);
    else if (src->pred) h->pred = src->pred->Clone(&shapes);
    else h->gen = src->gen->Clone(&shapes);
    *out = h.release();
  });
}
GX_CAPI int GXPredGetOutputShape(void* handle, uint32_t index, uint32_t** shape_data, uint32_t* shape_ndim) {
  return Guard([&] {
    Handle* h = HD(handle, "GXPredGetOutputShape");
    const Shape& s = h->gen ? h->gen->OutputShape(index) : h->plan().OutputShape(index);
    h->shape_out.assign(s.begin(), s.end());
    *shape_data = h->shape_out.data();
    *shape_ndim = static_cast<uint32_t>(h->shape_out.size());
  });
}
GX_CAPI int GXPredGetNumOutputs(void* handle, uint32_t* out) {
  return Guard([&] { Handle* h = HD(handle, "GXPredGetNumOutputs"); *out = static_cast<uint32_t>(h->gen ? h->gen->NumOutputs() : h->plan().NumOutputs()); });
}
// host handles read host memory only; device handles (dev_type 2) read host or device memory
GX_CAPI int GXPredSetInput(void* handle, const char* key, const float* data, uint32_t size) {
  return Guard([&] {
    if ((!handle || !H(handle)->dev) && gxrt::capi::IsDeviceBuffer(data))
      throw std::runtime_error("GXPredSetInput: device array (the predictor reads host memory; serve device data through GXExecutorForward)");
    Handle* h = HD(handle, "GXPredSetInput");
    if (h->dev) h->dev->SetInput(key, data, size); else if (h->pred) h->pred->SetInput(key, data, size); else h->gen->SetInput(key, data, size);
  });
}
// on a device handle: asynchronous, the first call runs eagerly, later calls replay one captured CUDA graph
GX_CAPI int GXPredForward(void* handle) {
  return Guard([&] { Handle* h = HD(handle, "GXPredForward"); if (h->dev) h->dev->Forward(); else if (h->pred) h->pred->Forward(); else h->gen->Forward(); });
}
GX_CAPI int GXPredPartialForward(void* handle, int step, int* step_left) {
  return Guard([&] {
    Handle* h = HD(handle, "GXPredPartialForward");
    if (h->dev) h->dev->PartialForward(step, step_left); else if (h->pred) h->pred->PartialForward(step, step_left); else h->gen->PartialForward(step, step_left);
  });
}
// on a device handle: waits for the handle's stream; `data` may be host or device memory
GX_CAPI int GXPredGetOutput(void* handle, uint32_t index, float* data, uint32_t size) {
  return Guard([&] {
    if ((!handle || !H(handle)->dev) && gxrt::capi::IsDeviceBuffer(data))
      throw std::runtime_error("GXPredGetOutput: device array (the predictor writes host memory)");
    Handle* h = HD(handle, "GXPredGetOutput");
    if (h->dev) h->dev->GetOutput(index, data, size); else if (h->pred) h->pred->GetOutput(index, data, size); else h->gen->GetOutput(index, data, size);
  });
}
// 1: the planned predictor (predict.h) runs this graph on the host, 2: the general executor (train_exec.h) does, 3: the planned predictor
// runs it on a GPU (predict_device.h)
GX_CAPI int GXPredGetEngine(void* handle, int* out) { return Guard([&] { Handle* h = H(handle); *out = h->dev ? 3 : h->pred ? 1 : 2; }); }
// planner statistics: bytes of the activation arena and the number of operators that run
GX_CAPI int GXPredGetPlan(void* handle, uint64_t* arena_bytes, uint32_t* num_ops) {
  return Guard([&] {
    Handle* h = H(handle);
    *arena_bytes = h->gen ? h->gen->ArenaBytes() : h->plan().ArenaBytes();
    *num_ops = static_cast<uint32_t>(h->gen ? h->gen->NumOps() : h->plan().NumOps());
  });
}
// a device handle waits for its stream before its memory goes back to the pool
GX_CAPI int GXPredFree(void* handle) { return Guard([&] { delete HD(handle, "GXPredFree"); }); }

GX_CAPI int GXNDListCreate(const char* nd_file_bytes, int nd_file_size, void** out, uint32_t* out_length) {
  return Guard([&] {
    if (nd_file_size < 0) throw std::runtime_error("negative nd_file_size");
    auto l = std::make_unique<NDList>(nd_file_bytes, static_cast<size_t>(nd_file_size));
    *out_length = static_cast<uint32_t>(l->data.size());
    *out = l.release();
  });
}
GX_CAPI int GXNDListGet(void* handle, uint32_t index, const char** out_key, const float** out_data, const uint32_t** out_shape, uint32_t* out_ndim) {
  return Guard([&] {
    if (!handle) throw std::runtime_error("null list handle");
    NDList* l = static_cast<NDList*>(handle);
    if (index >= l->data.size()) throw std::runtime_error("list index out of range");
    *out_key = l->names[index].c_str(); *out_data = l->data[index].data();
    *out_shape = l->shapes[index].data(); *out_ndim = static_cast<uint32_t>(l->shapes[index].size());
  });
}
GX_CAPI int GXNDListFree(void* handle) { return Guard([&] { delete static_cast<NDList*>(handle); }); }
