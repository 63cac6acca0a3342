// Symbol / Executor / imperative-invoke / autograd groups of the flat C ABI, on the native graph (graph.h) and the host training executor
// (train_exec.h).  With c_api_runtime.cc (NDArray, profiler, engine, storage), c_api_io.cc (RecordIO, data iterators), c_predict_api.cc and
// csrc/hips/c_api.cc (KVStore) this completes the function groups of the reference's C API for a front end that links no Python.
//
// Parity (GX prefix instead of MX, same argument order unless stated): include/mxnet/c_api.h
//   :1040-1530  MXSymbolListAtomicSymbolCreators / GetAtomicSymbolName / GetAtomicSymbolInfo / CreateAtomicSymbol / CreateVariable / CreateGroup /
//               CreateFromFile / CreateFromJSON / SaveToFile / SaveToJSON / Free / Copy / Print / GetName / GetAttr / SetAttr / ListAttr /
//               ListAttrShallow / ListArguments / ListOutputs / ListAuxiliaryStates / GetInternals / GetChildren / GetOutput / GetNumOutputs /
//               Compose / InferShape / InferShapePartial / InferType, MXListAllOpNames
//   :1530-1760  MXExecutorBind(X/EX) / SimpleBind / Forward / Backward(Ex) / Outputs / Print / Free
//   :1010-1040  MXImperativeInvoke;  :880-1010  MXAutogradSetIsRecording / SetIsTraining / IsRecording / IsTraining / MarkVariables / Backward(Ex) /
//               ComputeGradient / GetSymbol, MXNDArrayGetGrad / Detach
// Returned string / array pointers live in thread-local storage and stay valid until the next call of the same function group on the same
// thread (the reference's MXAPIThreadLocalEntry contract, src/c_api/c_api_common.h:60-100).
#include <cstdint>
#include <cstring>
#include <fstream>
#include <memory>
#include <string>
#include <vector>

#include "device_exec.h"
#include "graph.h"
#include "host_array.h"
#include "train_exec.h"

#define GX_CAPI extern "C" __attribute__((visibility("default")))

void GXRTSetLastError(const std::string& msg);

namespace gxrt {
namespace capi {

// ------------------------------------------------------------------------------------------------ autograd history
struct AGNode {
  // leaf: a marked variable
  HostArray* var = nullptr;                           // nulled when the handle is freed
  // operator: one recorded invocation
  std::unique_ptr<exec::Executor> ex;
  graph::Symbol sym;                                  // the one-node graph (inputs are variables in0, in1, ...)
  std::vector<std::vector<float>> in_copy;            // inputs as they were at invocation time (the caller may overwrite or free its arrays)
  std::vector<std::vector<float>> in_grad;
  std::vector<std::shared_ptr<AGNode>> in_node;       // history of each input (null: not tracked)
  std::vector<int> in_out;                            // ... and which output of that producer the input is
  int num_outputs = 1;
  std::string op;
  graph::AttrMap attrs;
  bool released = false;
};

HostArray::~HostArray() {
  if (ag && ag->var == this) ag->var = nullptr;
  try { ReleaseDevice(this); } catch (...) {}
}

}  // namespace capi
}  // namespace gxrt

namespace {
using gxrt::capi::AGNode;
using gxrt::capi::HostArray;
using gxrt::capi::ND;
using gxrt::graph::AttrMap;
using gxrt::graph::OpDef;
using gxrt::graph::Symbol;
using gxrt::predict::Numel;
using gxrt::predict::Shape;
namespace G = gxrt::graph;
namespace E = gxrt::exec;

template <typename F>
int Guard(F&& f) {
  try { f(); return 0; }
  catch (const std::exception& e) { GXRTSetLastError(e.what()); return -1; }
  catch (...) { GXRTSetLastError("unknown error"); return -1; }
}

Symbol* SYM(void* h) { if (!h) throw std::runtime_error("null Symbol handle"); return static_cast<Symbol*>(h); }

// thread-local return storage
struct Ret {
  std::string str;
  std::vector<std::string> strs;
  std::vector<const char*> ptrs;
  std::vector<void*> handles;
  const char** Strings(std::vector<std::string> v) { strs = std::move(v); ptrs.clear(); for (auto& s : strs) ptrs.push_back(s.c_str()); return ptrs.data(); }
};
thread_local Ret ret_sym, ret_info, ret_exec, ret_inv;
struct ShapeRet {
  std::vector<Shape> shapes[3];
  std::vector<uint32_t> ndim[3];
  std::vector<std::vector<uint32_t>> data[3];
  std::vector<const uint32_t*> ptr[3];
  std::vector<int> types[3];
};
thread_local ShapeRet ret_shape;

float* F32(HostArray* a, const char* what) {
  std::string& bytes = gxrt::capi::HostBytes(a, what);
  if (a->rec.dtype != 0) throw std::runtime_error(std::string(what) + ": the native executor computes in float32 (dtype flag 0), got dtype flag " + std::to_string(a->rec.dtype));
  return reinterpret_cast<float*>(&bytes[0]);
}
Shape ShapeOf(const HostArray* a) { return Shape(a->rec.shape.begin(), a->rec.shape.end()); }
HostArray* NewArray(const Shape& s) {
  auto a = std::make_unique<HostArray>();
  a->rec.dtype = 0;
  a->rec.shape.assign(s.begin(), s.end());
  a->rec.data.assign(static_cast<size_t>(Numel(s)) * 4, '\0');
  return a.release();
}
AttrMap Attrs(uint32_t n, const char** keys, const char** vals) {
  AttrMap m;
  for (uint32_t i = 0; i < n; ++i) { if (!keys[i] || !vals[i]) throw std::runtime_error("null attribute key / value"); m[keys[i]] = vals[i]; }
  return m;
}

// ---- executor handle: the executor + the arrays it hands out
struct ExecHandle {
  std::unique_ptr<E::Executor> ex;
  std::unique_ptr<E::DeviceExecutor> dex;                // set instead of ex for graphs bound to device arrays; outputs are views of its memory
  std::vector<std::unique_ptr<HostArray>> outputs;
  std::vector<std::unique_ptr<HostArray>> owned;        // SimpleBind: arguments / gradients / auxiliary states allocated here
  std::string printed;
};
ExecHandle* EX(void* h) { if (!h) throw std::runtime_error("null Executor handle"); return static_cast<ExecHandle*>(h); }

ExecHandle* BindImpl(Symbol* sym, const std::vector<HostArray*>& args, const std::vector<HostArray*>& grads, const std::vector<int>& reqs,
                     const std::vector<HostArray*>& aux) {
  std::vector<E::Tensor> ta, tg, tx;
  for (auto* a : args) ta.push_back({F32(a, "Bind argument"), ShapeOf(a)});
  for (size_t i = 0; i < args.size(); ++i) {
    HostArray* g = i < grads.size() ? grads[i] : nullptr;
    if (g && i < reqs.size() && reqs[i] != E::kNullOp) tg.push_back({F32(g, "Bind gradient"), ShapeOf(g)}); else tg.push_back({nullptr, {}});
  }
  for (auto* a : aux) tx.push_back({F32(a, "Bind auxiliary state"), ShapeOf(a)});
  auto h = std::make_unique<ExecHandle>();
  h->ex.reset(new E::Executor(*sym, ta, tg, reqs, tx));
  for (size_t i = 0; i < h->ex->NumOutputs(); ++i) h->outputs.emplace_back(NewArray(h->ex->OutputShape(i)));
  return h.release();
}
// all arrays on device dev: the device executor; outputs are device arrays that view the executor's output buffers
ExecHandle* BindDeviceImpl(Symbol* sym, int dev, const std::vector<HostArray*>& args, const std::vector<HostArray*>& grads, const std::vector<int>& reqs,
                           const std::vector<HostArray*>& aux) {
  std::vector<E::Tensor> ta, tg, tx;
  for (auto* a : args) ta.push_back({a->dptr, ShapeOf(a)});
  for (size_t i = 0; i < args.size(); ++i) {
    HostArray* g = i < grads.size() ? grads[i] : nullptr;
    if (g && i < reqs.size() && reqs[i] != E::kNullOp) tg.push_back({g->dptr, ShapeOf(g)}); else tg.push_back({nullptr, {}});
  }
  for (auto* a : aux) tx.push_back({a->dptr, ShapeOf(a)});
  auto h = std::make_unique<ExecHandle>();
  h->dex.reset(new E::DeviceExecutor(*sym, dev, ta, tg, reqs, tx));
  for (size_t i = 0; i < h->dex->NumOutputs(); ++i) {
    auto o = std::make_unique<HostArray>();
    const Shape& s = h->dex->OutputShape(i);
    o->rec.dtype = 0; o->rec.shape.assign(s.begin(), s.end()); o->dev_id = dev; o->dptr = h->dex->OutputData(i); o->owns_dptr = false;
    h->outputs.push_back(std::move(o));
  }
  return h.release();
}
// where the arrays of a bind live: -1 all on the host, d >= 0 all on device d; a mix or several devices is an error
int BindDevice(const char* fn, const std::vector<HostArray*>& arrays) {
  int dev = -2;
  for (HostArray* a : arrays) {
    if (!a) continue;
    const int d = a->device() ? a->dev_id : -1;
    if (dev == -2) dev = d;
    else if (d != dev) throw std::runtime_error(std::string(fn) + ": arrays on " + (dev < 0 ? std::string("the host") : "gpu(" + std::to_string(dev) + ")") + " and " +
                                                (d < 0 ? std::string("the host") : "gpu(" + std::to_string(d) + ")") + " cannot be bound together");
  }
  return dev == -2 ? -1 : dev;
}
void PublishOutputs(ExecHandle* h) {
  for (size_t i = 0; i < h->outputs.size(); ++i) memcpy(&h->outputs[i]->rec.data[0], h->ex->OutputData(i), h->outputs[i]->rec.data.size());
}

// ---- autograd state
thread_local bool ag_recording = false, ag_training = false;

void CollectTopo(const std::shared_ptr<AGNode>& n, std::set<AGNode*>* seen, std::vector<std::shared_ptr<AGNode>>* order) {
  if (!n || !seen->insert(n.get()).second) return;
  for (auto& i : n->in_node) CollectTopo(i, seen, order);
  order->push_back(n);
}

void BackwardImpl(uint32_t num, void** outs, void** ograds, bool retain) {
  std::vector<std::shared_ptr<AGNode>> order;
  std::set<AGNode*> seen;
  std::map<AGNode*, std::vector<std::vector<float>>> grad;          // per history node: one gradient buffer per output (empty = no gradient arrived)
  auto slot = [&](AGNode* n, int out, size_t size) -> std::vector<float>& {
    auto& v = grad[n];
    if (v.empty()) v.resize(static_cast<size_t>(std::max(n->num_outputs, 1)));
    if (v[out].empty()) v[out].assign(size, 0.f);
    return v[out];
  };
  for (uint32_t i = 0; i < num; ++i) {
    HostArray* o = ND(outs[i]);
    if (o->device()) throw std::runtime_error("GXAutogradBackward: device array (autograd records host arrays only)");
    if (!o->ag) throw std::runtime_error("Backward: output " + std::to_string(i) + " was not computed while recording (or its graph was already freed)");
    CollectTopo(o->ag, &seen, &order);
    const size_t n = o->rec.data.size() / 4;
    auto& g = slot(o->ag.get(), o->ag_out, n);
    if (ograds && ograds[i]) {
      HostArray* og = ND(ograds[i]);
      const float* p = F32(og, "GXAutogradBackward");
      if (og->rec.data.size() != o->rec.data.size()) throw std::runtime_error("Backward: head gradient " + std::to_string(i) + " does not match its output");
      for (size_t k = 0; k < n; ++k) g[k] += p[k];
    } else for (auto& v : g) v += 1.f;
  }
  for (size_t k = order.size(); k-- > 0;) {
    AGNode* n = order[k].get();
    auto it = grad.find(n);
    if (it == grad.end()) continue;
    if (n->op.empty()) {                    // leaf
      const std::vector<float>& g = it->second[0];
      if (n->var && n->var->grad && n->var->grad_req != E::kNullOp && !g.empty()) {
        float* dst = F32(n->var->grad, "gradient buffer");
        if (n->var->grad->rec.data.size() / 4 != g.size()) throw std::runtime_error("Backward: a gradient buffer does not match its variable");
        if (n->var->grad_req == E::kAddTo) for (size_t i = 0; i < g.size(); ++i) dst[i] += g[i];
        else memcpy(dst, g.data(), g.size() * 4);
      }
      continue;
    }
    if (n->released) throw std::runtime_error("Backward: the graph was already freed by an earlier backward pass (retain_graph = 0)");
    std::vector<const float*> heads;
    for (int o = 0; o < n->num_outputs; ++o) {           // outputs nobody differentiated through contribute zeros
      auto& g = it->second[o];
      if (g.empty()) g.assign(static_cast<size_t>(Numel(n->ex->OutputShape(o))), 0.f);
      heads.push_back(g.data());
    }
    n->ex->Backward(heads);
    for (size_t i = 0; i < n->in_node.size(); ++i) {
      if (!n->in_node[i]) continue;
      auto& g = slot(n->in_node[i].get(), n->in_out[i], n->in_grad[i].size());
      for (size_t e = 0; e < g.size(); ++e) g[e] += n->in_grad[i][e];
    }
  }
  if (!retain) for (auto& n : order) if (n->ex) { n->ex.reset(); n->in_copy.clear(); n->in_grad.clear(); n->released = true; }
}

}  // namespace

// ================================================================================================ Symbol
GX_CAPI int GXListAllOpNames(uint32_t* out_size, const char*** out_array) {
  return Guard([&] {
    std::vector<std::string> v;
    for (auto& d : G::OpTable()) v.push_back(d.name);
    *out_array = ret_info.Strings(std::move(v)); *out_size = static_cast<uint32_t>(ret_info.strs.size());
  });
}
GX_CAPI int GXSymbolListAtomicSymbolCreators(uint32_t* out_size, void*** out_array) {
  return Guard([&] {
    ret_info.handles.clear();
    for (auto& d : G::OpTable()) ret_info.handles.push_back(const_cast<OpDef*>(&d));
    *out_size = static_cast<uint32_t>(ret_info.handles.size()); *out_array = ret_info.handles.data();
  });
}
GX_CAPI int GXSymbolGetAtomicSymbolName(void* creator, const char** name) { return Guard([&] { if (!creator) throw std::runtime_error("null creator"); *name = static_cast<OpDef*>(creator)->name; }); }
GX_CAPI int GXSymbolGetAtomicSymbolInfo(void* creator, const char** name, const char** description, uint32_t* num_args, const char*** arg_names,
                                        const char*** arg_type_infos, const char*** arg_descriptions, const char** key_var_num_args, const char** return_type) {
  return Guard([&] {
    if (!creator) throw std::runtime_error("null creator");
    const OpDef* d = static_cast<OpDef*>(creator);
    static thread_local std::vector<const char*> names, types, docs;
    names.clear(); types.clear(); docs.clear();
    for (auto& p : d->params) { names.push_back(p.name); types.push_back(p.type); docs.push_back(p.doc); }
    *name = d->name; *description = d->doc; *num_args = static_cast<uint32_t>(names.size());
    *arg_names = names.data(); *arg_type_infos = types.data(); *arg_descriptions = docs.data();
    *key_var_num_args = d->key_var_num_args;
    if (return_type) *return_type = "Symbol";
  });
}
GX_CAPI int GXSymbolCreateAtomicSymbol(void* creator, uint32_t num_param, const char** keys, const char** vals, void** out) {
  return Guard([&] {
    if (!creator) throw std::runtime_error("null creator");
    *out = new Symbol(G::CreateAtomic(static_cast<OpDef*>(creator)->name, Attrs(num_param, keys, vals)));
  });
}
// convenience over the creator table: by operator name
GX_CAPI int GXSymbolCreateAtomicSymbolByName(const char* op, uint32_t num_param, const char** keys, const char** vals, void** out) {
  return Guard([&] { *out = new Symbol(G::CreateAtomic(op, Attrs(num_param, keys, vals))); });
}
GX_CAPI int GXSymbolCreateVariable(const char* name, void** out) { return Guard([&] { *out = new Symbol(G::Variable(name)); }); }
GX_CAPI int GXSymbolCreateGroup(uint32_t num, void** symbols, void** out) {
  return Guard([&] { std::vector<Symbol> v; for (uint32_t i = 0; i < num; ++i) v.push_back(*SYM(symbols[i])); *out = new Symbol(G::Group(v)); });
}
GX_CAPI int GXSymbolCreateFromJSON(const char* json, void** out) { return Guard([&] { *out = new Symbol(G::FromJSON(json)); }); }
GX_CAPI int GXSymbolCreateFromFile(const char* fname, void** out) {
  return Guard([&] {
    std::ifstream f(fname, std::ios::binary);
    if (!f) throw std::runtime_error(std::string("cannot open ") + fname);
    const std::string s((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    *out = new Symbol(G::FromJSON(s));
  });
}
GX_CAPI int GXSymbolSaveToJSON(void* sym, const char** out_json) { return Guard([&] { ret_sym.str = G::ToJSON(*SYM(sym)); *out_json = ret_sym.str.c_str(); }); }
GX_CAPI int GXSymbolSaveToFile(void* sym, const char* fname) {
  return Guard([&] {
    const std::string s = G::ToJSON(*SYM(sym));
    std::ofstream f(fname, std::ios::binary);
    if (!f) throw std::runtime_error(std::string("cannot open ") + fname);
    f.write(s.data(), static_cast<std::streamsize>(s.size()));
  });
}
GX_CAPI int GXSymbolFree(void* sym) { return Guard([&] { delete SYM(sym); }); }
GX_CAPI int GXSymbolCopy(void* sym, void** out) { return Guard([&] { *out = new Symbol(G::Copy(*SYM(sym))); }); }
GX_CAPI int GXSymbolPrint(void* sym, const char** out_str) {
  return Guard([&] {
    std::string o;
    const Symbol& s = *SYM(sym);
    o += "Symbol Outputs:\n";
    for (size_t i = 0; i < s.outputs.size(); ++i) o += "\toutput[" + std::to_string(i) + "]=" + G::OutputName(s.outputs[i]) + "(" + std::to_string(s.outputs[i].index) + ")\n";
    for (G::Node* n : G::Topo(s)) {
      if (n->op == "null") { o += "Variable:" + n->name + "\n"; continue; }
      o += "--------------------\nOp:" + n->op + ", Name=" + n->name + "\nInputs:\n";
      for (size_t i = 0; i < n->inputs.size(); ++i) o += "\targ[" + std::to_string(i) + "]=" + n->inputs[i].node->name + "(" + std::to_string(n->inputs[i].index) + ")\n";
      if (!n->attrs.empty()) { o += "Attrs:\n"; for (auto& kv : n->attrs) o += "\t" + kv.first + "=" + kv.second + "\n"; }
    }
    ret_sym.str = o; *out_str = ret_sym.str.c_str();
  });
}
GX_CAPI int GXSymbolGetName(void* sym, const char** out, int* success) {
  return Guard([&] {
    const Symbol& s = *SYM(sym);
    if (s.outputs.size() == 1) { ret_sym.str = s.outputs[0].node->name; *out = ret_sym.str.c_str(); *success = 1; } else { *out = nullptr; *success = 0; }
  });
}
GX_CAPI int GXSymbolGetAttr(void* sym, const char* key, const char** out, int* success) {
  return Guard([&] {
    const Symbol& s = *SYM(sym);
    *success = 0; *out = nullptr;
    if (s.outputs.size() != 1) return;
    const AttrMap& a = s.outputs[0].node->attrs;
    auto it = a.find(key);
    if (it == a.end()) it = a.find(std::string("__") + key + "__");      // the front ends store user attributes with dunder names
    if (it != a.end()) { ret_sym.str = it->second; *out = ret_sym.str.c_str(); *success = 1; }
  });
}
GX_CAPI int GXSymbolSetAttr(void* sym, const char* key, const char* value) {
  return Guard([&] {
    Symbol& s = *SYM(sym);
    if (s.outputs.size() != 1) throw std::runtime_error("SetAttr: needs a single-output symbol");
    s.outputs[0].node->attrs[key] = value;
  });
}
// pairs (key, value); recursive form prefixes keys with "<node>$"
GX_CAPI int GXSymbolListAttr(void* sym, uint32_t* out_size, const char*** out) {
  return Guard([&] {
    std::vector<std::string> v;
    for (G::Node* n : G::Topo(*SYM(sym))) for (auto& kv : n->attrs) { v.push_back(n->name + "$" + kv.first); v.push_back(kv.second); }
    *out = ret_sym.Strings(std::move(v)); *out_size = static_cast<uint32_t>(ret_sym.strs.size() / 2);
  });
}
GX_CAPI int GXSymbolListAttrShallow(void* sym, uint32_t* out_size, const char*** out) {
  return Guard([&] {
    const Symbol& s = *SYM(sym);
    std::vector<std::string> v;
    if (s.outputs.size() == 1) for (auto& kv : s.outputs[0].node->attrs) { v.push_back(kv.first); v.push_back(kv.second); }
    *out = ret_sym.Strings(std::move(v)); *out_size = static_cast<uint32_t>(ret_sym.strs.size() / 2);
  });
}
GX_CAPI int GXSymbolListArguments(void* sym, uint32_t* out_size, const char*** out) {
  return Guard([&] { *out = ret_sym.Strings(G::ListArguments(*SYM(sym))); *out_size = static_cast<uint32_t>(ret_sym.strs.size()); });
}
GX_CAPI int GXSymbolListOutputs(void* sym, uint32_t* out_size, const char*** out) {
  return Guard([&] { *out = ret_sym.Strings(G::ListOutputs(*SYM(sym))); *out_size = static_cast<uint32_t>(ret_sym.strs.size()); });
}
GX_CAPI int GXSymbolListAuxiliaryStates(void* sym, uint32_t* out_size, const char*** out) {
  return Guard([&] { *out = ret_sym.Strings(G::ListAuxiliaryStates(*SYM(sym))); *out_size = static_cast<uint32_t>(ret_sym.strs.size()); });
}
GX_CAPI int GXSymbolGetNumOutputs(void* sym, uint32_t* out) { return Guard([&] { *out = static_cast<uint32_t>(SYM(sym)->outputs.size()); }); }
GX_CAPI int GXSymbolGetInternals(void* sym, void** out) { return Guard([&] { *out = new Symbol(G::GetInternals(*SYM(sym))); }); }
GX_CAPI int GXSymbolGetChildren(void* sym, void** out) { return Guard([&] { *out = new Symbol(G::GetChildren(*SYM(sym))); }); }
GX_CAPI int GXSymbolGetOutput(void* sym, uint32_t index, void** out) {
  return Guard([&] {
    const Symbol& s = *SYM(sym);
    if (index >= s.outputs.size()) throw std::runtime_error("GetOutput: index " + std::to_string(index) + " out of range");
    *out = new Symbol(Symbol{{s.outputs[index]}});
  });
}
// keys == nullptr: positional inputs; otherwise keyword inputs
GX_CAPI int GXSymbolCompose(void* sym, const char* name, uint32_t num_args, const char** keys, void** args) {
  return Guard([&] {
    std::vector<Symbol> pos; std::vector<std::pair<std::string, Symbol>> kw;
    for (uint32_t i = 0; i < num_args; ++i) { if (keys && keys[i]) kw.emplace_back(keys[i], *SYM(args[i])); else pos.push_back(*SYM(args[i])); }
    G::Compose(SYM(sym), name ? name : "", pos, kw);
  });
}

namespace {
int InferShapeImpl(void* sym, uint32_t num_args, const char** keys, const uint32_t* ind_ptr, const uint32_t* shape_data, uint32_t* in_size, const uint32_t** in_ndim,
                   const uint32_t*** in_data, uint32_t* out_size, const uint32_t** out_ndim, const uint32_t*** out_data, uint32_t* aux_size,
                   const uint32_t** aux_ndim, const uint32_t*** aux_data, int* complete, bool partial) {
  return Guard([&] {
    const Symbol& s = *SYM(sym);
    const auto arg_names = G::ListArguments(s);
    std::map<std::string, Shape> known;
    for (uint32_t i = 0; i < num_args; ++i) {
      Shape sh(shape_data + ind_ptr[i], shape_data + ind_ptr[i + 1]);
      if (sh.empty() || std::any_of(sh.begin(), sh.end(), [](int64_t d) { return d == 0; })) continue;      // 0 = unknown in the reference's convention
      if (keys) known[keys[i]] = sh;
      else { if (i >= arg_names.size()) throw std::runtime_error("InferShape: more positional shapes than arguments"); known[arg_names[i]] = sh; }
    }
    const G::ShapeResult r = G::InferShapes(s, known, partial);
    std::map<std::string, Shape> by_name;
    for (auto& kv : r.shape) if (kv.first->op == "null") by_name[kv.first->name] = kv.second;
    ShapeRet& R = ret_shape;
    for (int g = 0; g < 3; ++g) R.shapes[g].clear();
    for (auto& n : arg_names) R.shapes[0].push_back(by_name.count(n) ? by_name[n] : Shape{});
    for (auto& e : s.outputs) { auto it = r.shape.find(e.node.get()); R.shapes[1].push_back(it == r.shape.end() ? Shape{} : it->second); }
    for (auto& n : G::ListAuxiliaryStates(s)) R.shapes[2].push_back(by_name.count(n) ? by_name[n] : Shape{});
    for (int g = 0; g < 3; ++g) {
      R.ndim[g].clear(); R.data[g].clear(); R.ptr[g].clear();
      for (auto& sh : R.shapes[g]) { R.ndim[g].push_back(static_cast<uint32_t>(sh.size())); R.data[g].emplace_back(sh.begin(), sh.end()); }
      for (auto& d : R.data[g]) R.ptr[g].push_back(d.data());
    }
    *in_size = static_cast<uint32_t>(R.shapes[0].size()); *in_ndim = R.ndim[0].data(); *in_data = R.ptr[0].data();
    *out_size = static_cast<uint32_t>(R.shapes[1].size()); *out_ndim = R.ndim[1].data(); *out_data = R.ptr[1].data();
    *aux_size = static_cast<uint32_t>(R.shapes[2].size()); *aux_ndim = R.ndim[2].data(); *aux_data = R.ptr[2].data();
    *complete = r.complete ? 1 : 0;
  });
}
}  // namespace
// shapes arrive CSR-packed: argument i has dims shape_data[ind_ptr[i] .. ind_ptr[i+1]); keys == nullptr means positional (ListArguments order)
GX_CAPI int GXSymbolInferShape(void* sym, uint32_t num_args, const char** keys, const uint32_t* ind_ptr, const uint32_t* shape_data, uint32_t* in_size,
                               const uint32_t** in_ndim, const uint32_t*** in_data, uint32_t* out_size, const uint32_t** out_ndim, const uint32_t*** out_data,
                               uint32_t* aux_size, const uint32_t** aux_ndim, const uint32_t*** aux_data, int* complete) {
  return InferShapeImpl(sym, num_args, keys, ind_ptr, shape_data, in_size, in_ndim, in_data, out_size, out_ndim, out_data, aux_size, aux_ndim, aux_data, complete, false);
}
GX_CAPI int GXSymbolInferShapePartial(void* sym, uint32_t num_args, const char** keys, const uint32_t* ind_ptr, const uint32_t* shape_data, uint32_t* in_size,
                                      const uint32_t** in_ndim, const uint32_t*** in_data, uint32_t* out_size, const uint32_t** out_ndim,
                                      const uint32_t*** out_data, uint32_t* aux_size, const uint32_t** aux_ndim, const uint32_t*** aux_data, int* complete) {
  return InferShapeImpl(sym, num_args, keys, ind_ptr, shape_data, in_size, in_ndim, in_data, out_size, out_ndim, out_data, aux_size, aux_ndim, aux_data, complete, true);
}
// dtype flags (mshadow: 0 f32, 1 f64, 2 f16, ...; -1 unknown).  Every operator of the native table keeps the type of its first known input.
GX_CAPI int GXSymbolInferType(void* sym, uint32_t num_args, const char** keys, const int* arg_type_data, uint32_t* in_size, const int** in_data, uint32_t* out_size,
                              const int** out_data, uint32_t* aux_size, const int** aux_data, int* complete) {
  return Guard([&] {
    const Symbol& s = *SYM(sym);
    const auto arg_names = G::ListArguments(s);
    int t = -1;
    std::map<std::string, int> given;
    for (uint32_t i = 0; i < num_args; ++i) {
      if (arg_type_data[i] < 0) continue;
      const std::string nm = keys ? keys[i] : (i < arg_names.size() ? arg_names[i] : std::string());
      given[nm] = arg_type_data[i];
      if (t >= 0 && t != arg_type_data[i]) throw std::runtime_error("InferType: arguments with different dtypes (" + std::to_string(t) + " vs " + std::to_string(arg_type_data[i]) + "); the native operators do not mix precisions");
      t = arg_type_data[i];
    }
    ShapeRet& R = ret_shape;
    R.types[0].assign(arg_names.size(), t); R.types[1].assign(s.outputs.size(), t); R.types[2].assign(G::ListAuxiliaryStates(s).size(), t);
    *in_size = static_cast<uint32_t>(R.types[0].size()); *in_data = R.types[0].data();
    *out_size = static_cast<uint32_t>(R.types[1].size()); *out_data = R.types[1].data();
    *aux_size = static_cast<uint32_t>(R.types[2].size()); *aux_data = R.types[2].data();
    *complete = t >= 0;
  });
}

// ================================================================================================ Executor
// Host arrays bind the host executor (dev_type / dev_id are then accepted for signature parity only).  Device arrays, all on gpu(dev_id) with
// dev_type 2, bind the device executor (device_exec.h); mixing host and device arrays, or devices, is an error.
// grad_req_type: 0 null, 1 write, 3 add (include/mxnet/op_attr_types.h OpReqType).
GX_CAPI int GXExecutorBind(void* sym, int dev_type, int dev_id, uint32_t len, void** in_args, void** arg_grad_store, const uint32_t* grad_req_type,
                           uint32_t aux_states_len, void** aux_states, void** out) {
  return Guard([&] {
    std::vector<HostArray*> args, grads, aux; std::vector<int> reqs;
    for (uint32_t i = 0; i < len; ++i) {
      args.push_back(ND(in_args[i]));
      grads.push_back(arg_grad_store && arg_grad_store[i] ? ND(arg_grad_store[i]) : nullptr);
      reqs.push_back(grad_req_type && grads.back() ? static_cast<int>(grad_req_type[i]) : E::kNullOp);
    }
    for (uint32_t i = 0; i < aux_states_len; ++i) aux.push_back(ND(aux_states[i]));
    std::vector<HostArray*> all = args;
    all.insert(all.end(), grads.begin(), grads.end()); all.insert(all.end(), aux.begin(), aux.end());
    const int dev = BindDevice("GXExecutorBind", all);
    if (dev < 0) { *out = BindImpl(SYM(sym), args, grads, reqs, aux); return; }
    if (dev_type != 2 || dev_id != dev)
      throw std::runtime_error("GXExecutorBind: the arrays live on gpu(" + std::to_string(dev) + "), the bind asks for dev_type " + std::to_string(dev_type) + " dev_id " + std::to_string(dev_id));
    *out = BindDeviceImpl(SYM(sym), dev, args, grads, reqs, aux);
  });
}
// Allocates every argument, gradient and auxiliary array from the given input shapes (role of MXExecutorSimpleBind, c_api.h:1640; the
// signature is reduced to what a host executor needs).  grad_req: "null" | "write" | "add" for all arguments except those named in
// `no_grad_keys` (typically data and label).  The arrays come back in ListArguments / ListAuxiliaryStates order and belong to the executor.
// dev_type 1: host arrays and the host executor (GXExecutorSimpleBind).  dev_type 2: zero-filled device arrays on gpu(dev_id) and the device
// executor.  The device's position follows the reference's MXExecutorSimpleBind (c_api.h:1640).
GX_CAPI int GXExecutorSimpleBindEx(void* sym, int dev_type, int dev_id, uint32_t num_shapes, const char** keys, const uint32_t* ind_ptr, const uint32_t* shape_data,
                                   const char* grad_req, uint32_t num_no_grad, const char** no_grad_keys, void** out, uint32_t* num_args, void*** in_args,
                                   void*** arg_grads, uint32_t* num_aux, void*** aux_states) {
  return Guard([&] {
    if (dev_type != 1 && dev_type != 2) throw std::runtime_error("GXExecutorSimpleBindEx: dev_type " + std::to_string(dev_type) + " is not supported (1 CPU, 2 GPU)");
    const bool on_dev = dev_type == 2;
    auto make = [&](const Shape& sh) { return on_dev ? gxrt::capi::NewDeviceArray(std::vector<int64_t>(sh.begin(), sh.end()), dev_id) : NewArray(sh); };
    Symbol* s = SYM(sym);
    std::map<std::string, Shape> known;
    for (uint32_t i = 0; i < num_shapes; ++i) known[keys[i]] = Shape(shape_data + ind_ptr[i], shape_data + ind_ptr[i + 1]);
    const G::ShapeResult r = G::InferShapes(*s, known, false);
    std::map<std::string, Shape> by_name;
    for (auto& kv : r.shape) if (kv.first->op == "null") by_name[kv.first->name] = kv.second;
    const std::string req = grad_req ? grad_req : "write";
    const int rq = req == "null" ? E::kNullOp : req == "add" ? E::kAddTo : req == "write" ? E::kWriteTo : -1;
    if (rq < 0) throw std::runtime_error("SimpleBind: grad_req must be null, write or add");
    std::set<std::string> no_grad;
    for (uint32_t i = 0; i < num_no_grad; ++i) no_grad.insert(no_grad_keys[i]);
    std::vector<std::unique_ptr<HostArray>> owned;
    std::vector<HostArray*> args, grads, aux; std::vector<int> reqs;
    for (auto& n : G::ListArguments(*s)) {
      owned.emplace_back(make(by_name.at(n))); args.push_back(owned.back().get());
      const int q = no_grad.count(n) ? E::kNullOp : rq;
      reqs.push_back(q);
      if (q != E::kNullOp) { owned.emplace_back(make(by_name.at(n))); grads.push_back(owned.back().get()); } else grads.push_back(nullptr);
    }
    for (auto& n : G::ListAuxiliaryStates(*s)) { owned.emplace_back(make(by_name.at(n))); aux.push_back(owned.back().get()); }
    ExecHandle* h = on_dev ? BindDeviceImpl(s, dev_id, args, grads, reqs, aux) : BindImpl(s, args, grads, reqs, aux);
    h->owned = std::move(owned);
    static thread_local std::vector<void*> ra, rg, rx;
    ra.assign(args.begin(), args.end()); rg.assign(grads.begin(), grads.end()); rx.assign(aux.begin(), aux.end());
    *out = h; *num_args = static_cast<uint32_t>(ra.size()); *in_args = ra.data(); *arg_grads = rg.data();
    *num_aux = static_cast<uint32_t>(rx.size()); *aux_states = rx.data();
  });
}
GX_CAPI int GXExecutorSimpleBind(void* sym, uint32_t num_shapes, const char** keys, const uint32_t* ind_ptr, const uint32_t* shape_data, const char* grad_req,
                                 uint32_t num_no_grad, const char** no_grad_keys, void** out, uint32_t* num_args, void*** in_args, void*** arg_grads,
                                 uint32_t* num_aux, void*** aux_states) {
  return GXExecutorSimpleBindEx(sym, 1, 0, num_shapes, keys, ind_ptr, shape_data, grad_req, num_no_grad, no_grad_keys, out, num_args, in_args, arg_grads, num_aux,
                                aux_states);
}
GX_CAPI int GXExecutorForward(void* h, int is_train) {
  return Guard([&] {
    ExecHandle* e = EX(h);
    if (e->dex) { e->dex->Forward(is_train != 0); return; }
    e->ex->Forward(is_train != 0); PublishOutputs(e);
  });
}
// head_grads may be null / len 0 for loss heads
GX_CAPI int GXExecutorBackward(void* h, uint32_t len, void** head_grads) {
  return Guard([&] {
    ExecHandle* e = EX(h);
    std::vector<const float*> hg;
    for (uint32_t i = 0; i < len; ++i) {
      if (!head_grads || !head_grads[i]) { hg.push_back(nullptr); continue; }
      HostArray* g = ND(head_grads[i]);
      if (e->dex) {
        if (!g->device() || g->dev_id != e->dex->device()) throw std::runtime_error("GXExecutorBackward: head gradient " + std::to_string(i) + " must be a device array on gpu(" + std::to_string(e->dex->device()) + ")");
        if (i < e->outputs.size() && g->Bytes() != e->outputs[i]->Bytes()) throw std::runtime_error("Backward: head gradient " + std::to_string(i) + " does not match its output");
        hg.push_back(g->dptr);
        continue;
      }
      if (i < e->outputs.size() && g->rec.data.size() != e->outputs[i]->rec.data.size()) throw std::runtime_error("Backward: head gradient " + std::to_string(i) + " does not match its output");
      hg.push_back(F32(g, "GXExecutorBackward"));
    }
    if (e->dex) e->dex->Backward(hg); else e->ex->Backward(hg);
  });
}
GX_CAPI int GXExecutorBackwardEx(void* h, uint32_t len, void** head_grads, int is_train) { (void)is_train; return GXExecutorBackward(h, len, head_grads); }
// the handles stay valid until the executor is freed; their contents are refreshed by every Forward
GX_CAPI int GXExecutorOutputs(void* h, uint32_t* out_size, void*** out) {
  return Guard([&] {
    ExecHandle* e = EX(h);
    static thread_local std::vector<void*> r;
    r.clear(); for (auto& o : e->outputs) r.push_back(o.get());
    *out_size = static_cast<uint32_t>(r.size()); *out = r.data();
  });
}
GX_CAPI int GXExecutorPrint(void* h, const char** out_str) {
  return Guard([&] { ExecHandle* e = EX(h); e->printed = e->dex ? e->dex->Print() : e->ex->Print(); *out_str = e->printed.c_str(); });
}
GX_CAPI int GXExecutorFree(void* h) { return Guard([&] { delete EX(h); }); }

// ================================================================================================ imperative invoke + autograd
GX_CAPI int GXAutogradSetIsRecording(int is_recording, int* prev) { return Guard([&] { if (prev) *prev = ag_recording; ag_recording = is_recording != 0; }); }
GX_CAPI int GXAutogradSetIsTraining(int is_training, int* prev) { return Guard([&] { if (prev) *prev = ag_training; ag_training = is_training != 0; }); }
GX_CAPI int GXAutogradIsRecording(bool* curr) { return Guard([&] { *curr = ag_recording; }); }
GX_CAPI int GXAutogradIsTraining(bool* curr) { return Guard([&] { *curr = ag_training; }); }
GX_CAPI int GXAutogradMarkVariables(uint32_t num_var, void** var_handles, const uint32_t* reqs_array, void** grad_handles) {
  return Guard([&] {
    for (uint32_t i = 0; i < num_var; ++i) {
      HostArray* v = ND(var_handles[i]); HostArray* g = ND(grad_handles[i]);
      F32(v, "GXAutogradMarkVariables"); F32(g, "GXAutogradMarkVariables");
      if (g->rec.data.size() != v->rec.data.size()) throw std::runtime_error("MarkVariables: gradient " + std::to_string(i) + " does not match its variable");
      v->ag = std::make_shared<AGNode>(); v->ag->var = v;
      v->grad = g; v->grad_req = static_cast<int>(reqs_array[i]);
    }
  });
}
GX_CAPI int GXNDArrayGetGrad(void* handle, void** out) { return Guard([&] { *out = ND(handle)->grad; }); }
// a new handle with the same contents and no history
GX_CAPI int GXNDArrayDetach(void* handle, void** out) {
  return Guard([&] {
    HostArray* a = ND(handle);
    auto c = std::make_unique<HostArray>();
    c->rec.dtype = a->rec.dtype; c->rec.shape = a->rec.shape; c->rec.data = gxrt::capi::HostBytes(a, "GXNDArrayDetach");
    *out = c.release();
  });
}

// One operator on device arrays through a one-node device executor, on the library stream of their device.  Trailing auxiliary inputs
// (BatchNorm's running statistics, optimizer states) are bound in place; given output arrays may alias an input, since the result is copied
// out of the executor's own buffers.
void InvokeDevice(const OpDef* d, const Symbol& sym, int num_inputs, void** inputs, int* num_outputs, void*** outputs) {
  std::vector<HostArray*> in;
  for (int i = 0; i < num_inputs; ++i) in.push_back(ND(inputs[i]));
  const int dev = BindDevice("GXImperativeInvoke", in);
  const int n_arg = num_inputs - d->num_aux;
  std::vector<E::Tensor> ta, tg, tx; std::vector<int> reqs;
  for (int i = 0; i < num_inputs; ++i) {
    if (in[i]->rec.dtype != 0) throw std::runtime_error("GXImperativeInvoke: device arrays are float32");
    (i < n_arg ? ta : tx).push_back({in[i]->dptr, ShapeOf(in[i])});
    if (i < n_arg) { tg.push_back({nullptr, {}}); reqs.push_back(E::kNullOp); }
  }
  E::DeviceExecutor ex(sym, dev, ta, tg, reqs, tx);
  ex.Forward(ag_training);
  const int nout = static_cast<int>(ex.NumOutputs());
  const bool given = *num_outputs > 0 && outputs && *outputs;
  if (given && *num_outputs != nout) throw std::runtime_error(std::string(d->name) + ": " + std::to_string(*num_outputs) + " output arrays given, the operator produces " + std::to_string(nout));
  std::vector<HostArray*> outs;
  for (int o = 0; o < nout; ++o) {
    const Shape& os = ex.OutputShape(o);
    const std::vector<int64_t> shp(os.begin(), os.end());
    HostArray* out = nullptr;
    if (given) {
      out = ND((*outputs)[o]);
      if (!out->device() || out->dev_id != dev) throw std::runtime_error("GXImperativeInvoke: output " + std::to_string(o) + " must be a device array on gpu(" + std::to_string(dev) + ")");
      if (out->rec.shape != shp || !out->owns_dptr) {
        std::unique_ptr<HostArray> fresh(gxrt::capi::NewDeviceArray(shp, dev));
        gxrt::capi::ReleaseDevice(out);
        out->dptr = fresh->dptr; out->owns_dptr = true; out->rec.shape = shp; out->rec.dtype = 0;
        fresh->owns_dptr = false;
      }
    } else {
      out = gxrt::capi::NewDeviceArray(shp, dev);
    }
    outs.push_back(out);
  }
  for (int o = 0; o < nout; ++o) {
    const gxrt::kern::Lib& L = gxrt::kern::Get();
    gxrt::kern::Check(L.memcpy(outs[o]->dptr, ex.OutputData(o), outs[o]->Bytes(), 3, L.stream(dev)), "GXImperativeInvoke");
  }
  if (!given) { ret_inv.handles.assign(outs.begin(), outs.end()); *outputs = ret_inv.handles.data(); }
  *num_outputs = nout;
}

// One operator on host arrays (device arrays: InvokeDevice).  *num_outputs == 0 (or *outputs == nullptr): the output array is created and returned through thread-local
// storage (the caller owns the handle, GXNDArrayFree); otherwise the given array is overwritten (resized when necessary).  While recording,
// the invocation is kept — with a snapshot of its inputs and its forward state — so GXAutogradBackward can differentiate through it.
GX_CAPI int GXImperativeInvoke(void* creator, int num_inputs, void** inputs, int* num_outputs, void*** outputs, int num_params, const char** param_keys,
                               const char** param_vals) {
  return Guard([&] {
    if (!creator) throw std::runtime_error("null creator");
    const OpDef* d = static_cast<OpDef*>(creator);
    AttrMap attrs = Attrs(static_cast<uint32_t>(num_params), param_keys, param_vals);
    if (*d->key_var_num_args && !attrs.count(d->key_var_num_args)) attrs[d->key_var_num_args] = std::to_string(num_inputs);
    Symbol sym = G::CreateAtomic(d->name, attrs);
    const size_t want = d->inputs(G::AttrView(attrs)).size();
    if (static_cast<size_t>(num_inputs) != want) throw std::runtime_error(std::string(d->name) + ": " + std::to_string(num_inputs) + " inputs given, the operator takes " + std::to_string(want));
    std::vector<Symbol> vars;
    for (int i = 0; i < num_inputs; ++i) vars.push_back(G::Variable("in" + std::to_string(i)));
    G::Compose(&sym, "op", vars, {});
    bool on_device = false;
    for (int i = 0; i < num_inputs; ++i) on_device = on_device || ND(inputs[i])->device();
    if (on_device) {
      if (ag_recording) throw std::runtime_error("GXImperativeInvoke: device inputs while autograd is recording (autograd records host arrays only)");
      InvokeDevice(d, sym, num_inputs, inputs, num_outputs, outputs);
      return;
    }
    auto node = std::make_shared<AGNode>();
    node->sym = sym; node->op = d->name; node->attrs = attrs;
    const int n_aux = d->num_aux, n_arg = num_inputs - n_aux;
    bool tracked = false;
    std::vector<HostArray*> in;
    for (int i = 0; i < num_inputs; ++i) {
      HostArray* a = ND(inputs[i]);
      const float* p = F32(a, "GXImperativeInvoke");
      in.push_back(a);
      node->in_copy.emplace_back(p, p + a->rec.data.size() / 4);
      node->in_node.push_back(i < n_arg && ag_recording ? a->ag : nullptr);
      node->in_out.push_back(a->ag_out);
      if (node->in_node.back()) tracked = true;
    }
    std::vector<E::Tensor> ta, tg, tx; std::vector<int> reqs;
    node->in_grad.resize(num_inputs);
    for (int i = 0; i < n_arg; ++i) {
      ta.push_back({node->in_copy[i].data(), ShapeOf(in[i])});
      if (node->in_node[i]) { node->in_grad[i].assign(node->in_copy[i].size(), 0.f); tg.push_back({node->in_grad[i].data(), ShapeOf(in[i])}); reqs.push_back(E::kWriteTo); }
      else { tg.push_back({nullptr, {}}); reqs.push_back(E::kNullOp); }
    }
    for (int i = n_arg; i < num_inputs; ++i) tx.push_back({node->in_copy[i].data(), ShapeOf(in[i])});
    node->ex.reset(new E::Executor(sym, ta, tg, reqs, tx));
    node->ex->Forward(ag_training);
    for (int i = n_arg; i < num_inputs; ++i) memcpy(&in[i]->rec.data[0], node->in_copy[i].data(), in[i]->rec.data.size());      // running statistics are updated in place
    const int nout = static_cast<int>(node->ex->NumOutputs());
    node->num_outputs = nout;
    const bool given = *num_outputs > 0 && outputs && *outputs;
    if (given && *num_outputs != nout) throw std::runtime_error(std::string(d->name) + ": " + std::to_string(*num_outputs) + " output arrays given, the operator produces " + std::to_string(nout));
    if (!given) ret_inv.handles.clear();
    for (int o = 0; o < nout; ++o) {
      const Shape& os = node->ex->OutputShape(o);
      HostArray* out = nullptr;
      if (given) {
        out = ND((*outputs)[o]);
        out->rec.dtype = 0; out->rec.shape.assign(os.begin(), os.end()); out->rec.data.assign(static_cast<size_t>(Numel(os)) * 4, '\0');
      } else {
        out = NewArray(os);
        ret_inv.handles.push_back(out);
      }
      memcpy(&out->rec.data[0], node->ex->OutputData(o), out->rec.data.size());
      if (tracked) { out->ag = node; out->ag_out = o; } else { out->ag.reset(); out->ag_out = 0; }
    }
    if (!given) *outputs = ret_inv.handles.data();
    *num_outputs = nout;
  });
}
GX_CAPI int GXImperativeInvokeByName(const char* op, int num_inputs, void** inputs, int* num_outputs, void*** outputs, int num_params, const char** param_keys,
                                     const char** param_vals) {
  const OpDef* d = G::FindOp(op ? op : "");
  if (!d) { GXRTSetLastError(std::string("operator ") + (op ? op : "(null)") + " is not registered in the native graph runtime"); return -1; }
  return GXImperativeInvoke(const_cast<OpDef*>(d), num_inputs, inputs, num_outputs, outputs, num_params, param_keys, param_vals);
}
GX_CAPI int GXAutogradBackward(uint32_t num_output, void** output_handles, void** ograd_handles, int retain_graph) {
  return Guard([&] { BackwardImpl(num_output, output_handles, ograd_handles, retain_graph != 0); });
}
GX_CAPI int GXAutogradBackwardEx(uint32_t num_output, void** output_handles, void** ograd_handles, int retain_graph, int is_train) {
  (void)is_train;
  return GXAutogradBackward(num_output, output_handles, ograd_handles, retain_graph);
}
GX_CAPI int GXAutogradComputeGradient(uint32_t num_output, void** output_handles) { return GXAutogradBackward(num_output, output_handles, nullptr, 0); }
// the recorded history of an array as a Symbol: marked variables become var0, var1, ... in first-visit order, untracked inputs const0, ...
GX_CAPI int GXAutogradGetSymbol(void* handle, void** out) {
  return Guard([&] {
    HostArray* a = ND(handle);
    if (!a->ag) throw std::runtime_error("GetSymbol: the array has no recorded history");
    std::map<AGNode*, Symbol> built;
    int nvar = 0, nconst = 0, nop = 0;
    std::function<Symbol(const std::shared_ptr<AGNode>&)> build = [&](const std::shared_ptr<AGNode>& n) -> Symbol {
      auto it = built.find(n.get());
      if (it != built.end()) return it->second;
      Symbol s;
      if (n->op.empty()) s = G::Variable("var" + std::to_string(nvar++));
      else {
        s = G::CreateAtomic(n->op, n->attrs);
        std::vector<Symbol> ins;
        for (size_t k = 0; k < n->in_node.size(); ++k) {
          if (!n->in_node[k]) { ins.push_back(G::Variable("const" + std::to_string(nconst++))); continue; }
          const Symbol src = build(n->in_node[k]);
          ins.push_back(Symbol{{src.outputs.at(static_cast<size_t>(n->in_out[k]))}});
        }
        G::Compose(&s, n->op + std::to_string(nop++), ins, {});
      }
      built[n.get()] = s;
      return s;
    };
    *out = new Symbol(Symbol{{build(a->ag).outputs.at(static_cast<size_t>(a->ag_out))}});
  });
}

// ================================================================================================ misc
GX_CAPI int GXGetVersion(int* out) { return Guard([&] { *out = 10400; }); }
GX_CAPI int GXRandomSeed(int seed) { return Guard([&] { E::Executor::GlobalSeed().store(static_cast<uint32_t>(seed)); }); }
