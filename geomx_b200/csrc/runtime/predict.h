// Native inference runtime behind the C predict API (c_predict_api.cc): loads a symbol JSON + a `.params` blob, infers every shape once, plans
// ONE activation arena with liveness-based block reuse (views and in-place elementwise ops share storage), and runs the graph on the host in fp32.
//
// Parity: include/mxnet/c_predict_api.h:60-277 / src/c_api/c_predict_api.cc (MXPredCreate* / Reshape / SetInput / Forward / PartialForward /
// GetOutputShape / GetOutput / Free, MXNDList*).  The reference binds a full Executor; a deployment library that links no Python and no
// framework wants exactly the opposite, so this is a self-contained interpreter: its own JSON reader, its own operator set (the layers
// that symbol.py builds structurally + the elementwise family), its own memory planner (role of src/executor/graph_executor.cc
// InitDataEntryMemory / nnvm PlanMemory).  Both graph dialects load: this framework's `geomx_b200-symbol-1` and the reference's nnvm JSON
// (string-valued attrs, `[node, index, version]` input triples, BatchNorm statistics as inputs 3/4), so `-symbol.json` + `.params`
// checkpoints written by either side can be served.  GraphPlan holds everything that does not depend on the device; Predictor runs it on
// the host, predict_device.h::DevicePredictor runs the same plan on a GPU.
#pragma once
#include <algorithm>
#include <cctype>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <functional>
#include <limits>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "params_io.h"

namespace gxrt {
namespace predict {

// ------------------------------------------------------------------------------------------------ JSON
struct JValue {
  enum Kind { kNull, kBool, kNum, kStr, kArr, kObj } kind = kNull;
  bool b = false;
  double num = 0;
  std::string str;
  std::vector<JValue> arr;
  std::vector<std::pair<std::string, JValue>> obj;
  const JValue* Find(const std::string& k) const {
    if (kind != kObj) return nullptr;
    for (auto& kv : obj) if (kv.first == k) return &kv.second;
    return nullptr;
  }
};

class JParser {
 public:
  JParser(const char* p, size_t n) : p_(p), n_(n) {}
  JValue Parse() { JValue v = Value(0); Skip(); if (o_ != n_) Fail("trailing characters"); return v; }
 private:
  static constexpr int kMaxDepth = 64;
  const char* p_; size_t n_, o_ = 0;
  [[noreturn]] void Fail(const char* what) const { throw std::runtime_error(std::string("symbol JSON: ") + what + " at offset " + std::to_string(o_)); }
  void Skip() { while (o_ < n_ && (p_[o_] == ' ' || p_[o_] == '\n' || p_[o_] == '\t' || p_[o_] == '\r')) ++o_; }
  char Peek() { Skip(); if (o_ >= n_) Fail("unexpected end"); return p_[o_]; }
  void Expect(char c) { if (Peek() != c) Fail("unexpected character"); ++o_; }
  bool Lit(const char* s) { const size_t l = strlen(s); if (o_ + l <= n_ && memcmp(p_ + o_, s, l) == 0) { o_ += l; return true; } return false; }
  std::string String() {
    Expect('"');
    std::string s;
    while (true) {
      if (o_ >= n_) Fail("unterminated string");
      char c = p_[o_++];
      if (c == '"') break;
      if (c != '\\') { s.push_back(c); continue; }
      if (o_ >= n_) Fail("unterminated escape");
      c = p_[o_++];
      switch (c) {
        case 'n': s.push_back('\n'); break; case 't': s.push_back('\t'); break; case 'r': s.push_back('\r'); break;
        case 'b': s.push_back('\b'); break; case 'f': s.push_back('\f'); break;
        case 'u': {
          if (o_ + 4 > n_) Fail("short \\u escape");
          unsigned cp = 0;
          for (int i = 0; i < 4; ++i) {
            const char h = p_[o_++];
            cp = cp * 16 + (h >= '0' && h <= '9' ? h - '0' : h >= 'a' && h <= 'f' ? h - 'a' + 10 : h >= 'A' && h <= 'F' ? h - 'A' + 10 : (Fail("bad \\u escape"), 0));
          }
          if (cp >= 0xD800 && cp < 0xDC00 && o_ + 6 <= n_ && p_[o_] == '\\' && p_[o_ + 1] == 'u') {     // surrogate pair -> one code point
            unsigned lo = 0; bool ok = true;
            for (int i = 0; i < 4; ++i) {
              const char h = p_[o_ + 2 + i];
              const int dgt = h >= '0' && h <= '9' ? h - '0' : h >= 'a' && h <= 'f' ? h - 'a' + 10 : h >= 'A' && h <= 'F' ? h - 'A' + 10 : -1;
              if (dgt < 0) { ok = false; break; }
              lo = lo * 16 + static_cast<unsigned>(dgt);
            }
            if (ok && lo >= 0xDC00 && lo < 0xE000) { cp = 0x10000 + ((cp - 0xD800) << 10) + (lo - 0xDC00); o_ += 6; }
          }
          if (cp >= 0xD800 && cp < 0xE000) cp = 0xFFFD;                      // a lone surrogate is not encodable
          if (cp >= 0x10000) {
            s.push_back(static_cast<char>(0xF0 | (cp >> 18))); s.push_back(static_cast<char>(0x80 | ((cp >> 12) & 0x3F)));
            s.push_back(static_cast<char>(0x80 | ((cp >> 6) & 0x3F))); s.push_back(static_cast<char>(0x80 | (cp & 0x3F)));
          } else if (cp < 0x80) s.push_back(static_cast<char>(cp));
          else if (cp < 0x800) { s.push_back(static_cast<char>(0xC0 | (cp >> 6))); s.push_back(static_cast<char>(0x80 | (cp & 0x3F))); }
          else { s.push_back(static_cast<char>(0xE0 | (cp >> 12))); s.push_back(static_cast<char>(0x80 | ((cp >> 6) & 0x3F))); s.push_back(static_cast<char>(0x80 | (cp & 0x3F))); }
          break;
        }
        default: s.push_back(c);
      }
    }
    return s;
  }
  JValue Value(int depth) {
    if (depth > kMaxDepth) Fail("nesting too deep");
    JValue v;
    const char c = Peek();
    if (c == '{') {
      ++o_; v.kind = JValue::kObj;
      if (Peek() == '}') { ++o_; return v; }
      while (true) {
        std::string k = (Skip(), String());
        Expect(':');
        v.obj.emplace_back(std::move(k), Value(depth + 1));
        const char d = Peek(); ++o_;
        if (d == '}') break;
        if (d != ',') Fail("expected , or }");
      }
    } else if (c == '[') {
      ++o_; v.kind = JValue::kArr;
      if (Peek() == ']') { ++o_; return v; }
      while (true) {
        v.arr.push_back(Value(depth + 1));
        const char d = Peek(); ++o_;
        if (d == ']') break;
        if (d != ',') Fail("expected , or ]");
      }
    } else if (c == '"') {
      v.kind = JValue::kStr; v.str = String();
    } else if (Lit("true")) { v.kind = JValue::kBool; v.b = true;
    } else if (Lit("false")) { v.kind = JValue::kBool; v.b = false;
    } else if (Lit("null")) { v.kind = JValue::kNull;
    } else if (Lit("NaN")) { v.kind = JValue::kNum; v.num = std::nan("");
    } else if (Lit("Infinity")) { v.kind = JValue::kNum; v.num = std::numeric_limits<double>::infinity();
    } else if (Lit("-Infinity")) { v.kind = JValue::kNum; v.num = -std::numeric_limits<double>::infinity();
    } else {
      const size_t s = o_;
      while (o_ < n_ && (std::isdigit(static_cast<unsigned char>(p_[o_])) || p_[o_] == '-' || p_[o_] == '+' || p_[o_] == '.' || p_[o_] == 'e' || p_[o_] == 'E')) ++o_;
      if (o_ == s) Fail("unexpected token");
      try { v.num = std::stod(std::string(p_ + s, o_ - s)); } catch (...) { Fail("bad number"); }
      v.kind = JValue::kNum;
    }
    return v;
  }
};

// attribute access that is indifferent to the dialect: typed JSON values (ours) or python-repr strings (nnvm: "(5, 5)", "True", "20")
class Attrs {
 public:
  Attrs() = default;
  explicit Attrs(const JValue* o) : o_(o) {}
  const JValue* Raw(const std::string& k) const { const JValue* v = o_ ? o_->Find(k) : nullptr; return (v && v->kind != JValue::kNull && !(v->kind == JValue::kStr && v->str == "None")) ? v : nullptr; }
  bool Has(const std::string& k) const { return Raw(k) != nullptr; }
  double Float(const std::string& k, double def) const {
    const JValue* v = Raw(k);
    if (!v) return def;
    if (v->kind == JValue::kNum) return v->num;
    if (v->kind == JValue::kBool) return v->b;
    if (v->kind == JValue::kStr) { try { return std::stod(v->str); } catch (...) {} }
    throw std::runtime_error("attribute " + k + " is not a number");
  }
  int64_t Int(const std::string& k, int64_t def) const { return static_cast<int64_t>(std::llround(Float(k, static_cast<double>(def)))); }
  bool Bool(const std::string& k, bool def) const {
    const JValue* v = Raw(k);
    if (!v) return def;
    if (v->kind == JValue::kBool) return v->b;
    if (v->kind == JValue::kNum) return v->num != 0;
    if (v->kind == JValue::kStr) return v->str == "True" || v->str == "true" || v->str == "1";
    return def;
  }
  std::string Str(const std::string& k, const std::string& def) const {
    const JValue* v = Raw(k);
    return (v && v->kind == JValue::kStr) ? v->str : def;
  }
  std::vector<int64_t> Tuple(const std::string& k, std::vector<int64_t> def) const {
    const JValue* v = Raw(k);
    if (!v) return def;
    std::vector<int64_t> out;
    if (v->kind == JValue::kArr) { for (auto& e : v->arr) out.push_back(static_cast<int64_t>(std::llround(e.num))); return out; }
    if (v->kind == JValue::kNum) return {static_cast<int64_t>(std::llround(v->num))};
    if (v->kind == JValue::kStr) {
      const std::string& s = v->str;
      size_t i = 0;
      while (i < s.size()) {
        if (std::isdigit(static_cast<unsigned char>(s[i])) || s[i] == '-') {
          size_t j = i + 1;
          while (j < s.size() && std::isdigit(static_cast<unsigned char>(s[j]))) ++j;
          out.push_back(std::stoll(s.substr(i, j - i)));
          i = j;
        } else { ++i; }
      }
      return out.empty() ? def : out;
    }
    return def;
  }
 private:
  const JValue* o_ = nullptr;
};

// ------------------------------------------------------------------------------------------------ helpers
using Shape = std::vector<int64_t>;
inline int64_t Numel(const Shape& s) { int64_t p = 1; for (auto d : s) p *= d; return p; }
inline std::string ShapeStr(const Shape& s) { std::string o = "("; for (size_t i = 0; i < s.size(); ++i) o += (i ? ", " : "") + std::to_string(s[i]); return o + ")"; }

inline float HalfToFloat(uint16_t h) {
  const uint32_t sign = (h & 0x8000u) << 16, exp = (h >> 10) & 0x1F, man = h & 0x3FF;
  uint32_t bits;
  if (exp == 0) {
    if (man == 0) bits = sign;
    else { int e = -1; uint32_t m = man; do { ++e; m <<= 1; } while ((m & 0x400) == 0); bits = sign | ((127 - 15 - e) << 23) | ((m & 0x3FF) << 13); }
  } else if (exp == 31) bits = sign | 0x7F800000u | (man << 13);
  else bits = sign | ((exp + 112) << 23) | (man << 13);
  float f; memcpy(&f, &bits, 4); return f;
}

inline std::vector<float> ToFloat(const NDRec& r) {
  const int64_t n = Numel(r.shape);
  std::vector<float> out(static_cast<size_t>(n));
  const char* p = r.data.data();
  if (r.data.size() != static_cast<size_t>(n) * FlagSize(r.dtype)) throw std::runtime_error("parameter blob: size does not match its shape");
  switch (r.dtype) {
    case 0: memcpy(out.data(), p, n * 4); break;
    case 1: for (int64_t i = 0; i < n; ++i) { double d; memcpy(&d, p + 8 * i, 8); out[i] = static_cast<float>(d); } break;
    case 2: for (int64_t i = 0; i < n; ++i) { uint16_t h; memcpy(&h, p + 2 * i, 2); out[i] = HalfToFloat(h); } break;
    case 3: for (int64_t i = 0; i < n; ++i) out[i] = static_cast<uint8_t>(p[i]); break;
    case 4: for (int64_t i = 0; i < n; ++i) { int32_t d; memcpy(&d, p + 4 * i, 4); out[i] = static_cast<float>(d); } break;
    case 5: for (int64_t i = 0; i < n; ++i) out[i] = static_cast<int8_t>(p[i]); break;
    case 6: for (int64_t i = 0; i < n; ++i) { int64_t d; memcpy(&d, p + 8 * i, 8); out[i] = static_cast<float>(d); } break;
    default: throw std::runtime_error("parameter blob: unknown dtype flag");
  }
  return out;
}

// splits [0, n) over a few threads when the loop is worth it (cost = rough number of multiply-adds)
template <typename F>
void ParallelFor(int64_t n, double cost, F&& fn) {
  static const int kMax = std::max(1, std::min(16, static_cast<int>(std::thread::hardware_concurrency())));
  const int t = static_cast<int>(std::min<int64_t>(std::min<int64_t>(kMax, n), static_cast<int64_t>(cost / 2e6) + 1));
  if (t <= 1) { fn(0, n); return; }
  std::vector<std::thread> th;
  const int64_t per = (n + t - 1) / t;
  for (int i = 1; i < t; ++i) { const int64_t a = i * per, b = std::min(n, a + per); if (a < b) th.emplace_back([&fn, a, b] { fn(a, b); }); }
  fn(0, std::min(n, per));
  for (auto& x : th) x.join();
}

// C[m, n] (+)= A[m, k] . B[n, k]^T, row-major; the inner reduction keeps 8 partial sums so it vectorises without -ffast-math
inline void GemmNT(const float* A, const float* B, float* C, int64_t M, int64_t N, int64_t K, const float* bias) {
  ParallelFor(M * N, static_cast<double>(M) * N * K, [&](int64_t lo, int64_t hi) {
    for (int64_t idx = lo; idx < hi; ++idx) {
      const int64_t i = idx / N, j = idx % N;
      const float* a = A + i * K; const float* b = B + j * K;
      float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      int64_t k = 0;
      for (; k + 8 <= K; k += 8) for (int u = 0; u < 8; ++u) acc[u] += a[k + u] * b[k + u];
      float s = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
      for (; k < K; ++k) s += a[k] * b[k];
      C[idx] = s + (bias ? bias[j] : 0.f);
    }
  });
}

// ------------------------------------------------------------------------------------------------ graph
struct Entry { int node = -1; int index = 0; };
struct Node {
  std::string op, name;
  Attrs attrs;
  std::vector<Entry> inputs;
  bool nnvm = false;                 // dialect: decides the defaults of absent attributes (Pooling stride, BatchNorm fix_gamma / eps)
  Shape shape;                       // output 0 (every supported op has one visible output)
  int storage = -1;
  bool known = false;                // shape inferred
};

struct Storage {
  bool external = false;             // parameter / input buffer owned outside the arena
  int block = -1;
  int64_t size = 0;
  int ref = 0;
  float* ptr = nullptr;
};

// Everything about a predictor that does not depend on where it runs: the graph (both dialects), the parameters, the input shapes, shape
// inference, reachability and the liveness plan of the activation arena.  The host Predictor below and the device runner of
// predict_device.h both execute this plan: order_ lists the operators that run, nodes_[i].storage names the storage each output lives in,
// storages_ are either external (an input or a parameter) or a block of the arena at block_offset_[block] floats, and the arena holds
// arena_floats_ floats.
class GraphPlan {
 public:
  GraphPlan(const std::string& json, const char* params, size_t param_size, const std::vector<std::string>& input_keys,
            const std::vector<Shape>& input_shapes, const std::vector<std::string>& output_keys) {
    doc_ = std::make_shared<JValue>(JParser(json.data(), json.size()).Parse());
    BuildGraph(output_keys);
    LoadParams(params, param_size);
    for (size_t i = 0; i < input_keys.size(); ++i) input_shapes_[input_keys[i]] = input_shapes[i];
    Plan();
  }
  // the same graph and parameters with other input shapes (those not named keep theirs), planned anew
  void Replan(const std::map<std::string, Shape>* new_shapes) {
    if (new_shapes) for (auto& kv : *new_shapes) {
      if (!input_shapes_.count(kv.first)) throw std::runtime_error("reshape: " + kv.first + " is not an input of this predictor");
      input_shapes_[kv.first] = kv.second;
    }
    Plan();
  }
  size_t NumOutputs() const { return heads_.size(); }
  const Shape& OutputShape(size_t i) const { return nodes_[Head(i)].shape; }
  size_t ArenaBytes() const { return static_cast<size_t>(arena_floats_) * sizeof(float); }
  size_t NumOps() const { return order_.size(); }

 protected:
  GraphPlan(const GraphPlan&) = default;
  std::shared_ptr<JValue> doc_;
  std::vector<Node> nodes_;
  std::vector<Entry> heads_;
  std::shared_ptr<std::map<std::string, std::pair<Shape, std::vector<float>>>> params_;
  std::map<std::string, Shape> input_shapes_;
  std::vector<int> order_;
  std::vector<Storage> storages_;
  std::vector<int64_t> block_offset_;
  int64_t arena_floats_ = 0;

  int Head(size_t i) const { if (i >= heads_.size()) throw std::runtime_error("output index out of range"); return heads_[i].node; }
  bool IsInput(const Node& nd) const { return nd.op == "null" && input_shapes_.count(nd.name) > 0; }

  // ---- graph construction (both dialects)
  void BuildGraph(const std::vector<std::string>& output_keys) {
    const JValue* jn = doc_->Find("nodes");
    if (!jn || jn->kind != JValue::kArr) throw std::runtime_error("symbol JSON: no \"nodes\" array");
    const bool nnvm = doc_->Find("arg_nodes") != nullptr || (doc_->Find("format") == nullptr);
    const int n = static_cast<int>(jn->arr.size());
    nodes_.resize(n);
    auto entry = [&](const JValue& e, int self) {
      Entry en;
      if (e.kind == JValue::kNum) en.node = static_cast<int>(e.num);
      else if (e.kind == JValue::kArr && !e.arr.empty()) { en.node = static_cast<int>(e.arr[0].num); en.index = e.arr.size() > 1 ? static_cast<int>(e.arr[1].num) : 0; }
      else throw std::runtime_error("symbol JSON: malformed input reference");
      if (en.node < 0 || en.node >= self) throw std::runtime_error("symbol JSON: node inputs must refer to earlier nodes");
      return en;
    };
    for (int i = 0; i < n; ++i) {
      const JValue& j = jn->arr[i];
      Node& nd = nodes_[i];
      const JValue* op = j.Find("op"); const JValue* name = j.Find("name");
      if (!op || op->kind != JValue::kStr) throw std::runtime_error("symbol JSON: node without op");
      nd.op = op->str; nd.name = name && name->kind == JValue::kStr ? name->str : ("node" + std::to_string(i));
      nd.nnvm = nnvm;
      const JValue* at = j.Find("attrs"); if (!at) at = j.Find("param"); if (!at) at = j.Find("attr");     // pre-1.0 files: "param" = operator arguments, "attr" = user annotations
      nd.attrs = Attrs(at);
      if (const JValue* in = j.Find("inputs")) for (auto& e : in->arr) nd.inputs.push_back(entry(e, i));
      if (const JValue* aux = j.Find("aux")) for (auto& e : aux->arr) nd.inputs.push_back(entry(e, i));   // ours: statistics after the inputs = nnvm order
      if (nd.op == "_nd") {             // generic imperative-op node of symbol.py: the function name is the operator, kwargs are the attributes
        const std::string fn = nd.attrs.Str("fn", "");
        const size_t dot = fn.rfind('.');
        nd.op = dot == std::string::npos ? fn : fn.substr(dot + 1);
        if (static_cast<size_t>(nd.attrs.Int("npos", static_cast<int64_t>(nd.inputs.size()))) != nd.inputs.size())
          throw std::runtime_error(nd.name + ": tensor keyword arguments are not supported by the native predictor");
        nd.attrs = Attrs(at ? at->Find("kwargs") : nullptr);
      }
    }
    const JValue* heads = doc_->Find("heads");
    if (!heads || heads->kind != JValue::kArr || heads->arr.empty()) throw std::runtime_error("symbol JSON: no heads");
    for (auto& h : heads->arr) {
      Entry e = entry(h, n);
      if (nodes_[e.node].op == "_group") for (auto& g : nodes_[e.node].inputs) heads_.push_back(g);
      else heads_.push_back(e);
    }
    if (!output_keys.empty()) {        // MXPredCreatePartialOut: internal outputs by name ("fc1" or "fc1_output")
      heads_.clear();
      for (auto& k : output_keys) {
        int found = -1;
        for (int i = 0; i < n; ++i) if (nodes_[i].name == k || nodes_[i].name + "_output" == k) found = i;
        if (found < 0) throw std::runtime_error("output " + k + " is not a node of the graph");
        heads_.push_back(Entry{found, 0});
      }
    }
    for (auto& h : heads_)
      if (h.index != 0) throw std::runtime_error(nodes_[h.node].name + " (" + nodes_[h.node].op + "): secondary operator outputs cannot be predictor outputs");
  }

  void LoadParams(const char* blob, size_t size) {
    params_ = std::make_shared<std::map<std::string, std::pair<Shape, std::vector<float>>>>();
    if (blob == nullptr || size == 0) return;
    BufReader r(blob, size);
    if (r.Get<uint64_t>() != kListMagic) throw std::runtime_error("parameter blob: not an NDArray list");
    r.Get<uint64_t>();
    const uint64_t n = r.Get<uint64_t>();
    if (n > (1u << 24)) throw std::runtime_error("parameter blob: implausible array count");
    std::vector<NDRec> recs;
    for (uint64_t i = 0; i < n; ++i) recs.push_back(ReadArray(r));
    const uint64_t m = r.Get<uint64_t>();
    if (m != n) throw std::runtime_error("parameter blob: arrays are not named");
    for (uint64_t i = 0; i < m; ++i) {
      const uint64_t l = r.Get<uint64_t>();
      std::string name = r.Raw(l);
      if (name.compare(0, 4, "arg:") == 0 || name.compare(0, 4, "aux:") == 0) name = name.substr(4);
      (*params_)[name] = {recs[i].shape, ToFloat(recs[i])};
    }
  }

  // ---- shape inference + memory plan + parameter binding
  static bool IsView(const std::string& op) {
    return op == "Flatten" || op == "flatten" || op == "Reshape" || op == "reshape" || op == "Dropout" || op == "identity" || op == "_copy" ||
           op == "BlockGrad" || op == "stop_gradient" || op == "LinearRegressionOutput" || op == "MAERegressionOutput" || op == "expand_dims";
  }
  static bool IsInplace(const std::string& op) {
    static const char* k[] = {"Activation", "LeakyReLU", "relu", "sigmoid", "tanh", "exp", "log", "sqrt", "abs", "negative", "square", "softsign",
                              "clip", "_plus_scalar", "_minus_scalar", "_mul_scalar", "_div_scalar", "_rminus_scalar", "_rdiv_scalar",
                              "_PlusScalar", "_MinusScalar", "_MulScalar", "_DivScalar", "_RMinusScalar", "_RDivScalar", "LogisticRegressionOutput"};
    for (auto s : k) if (op == s) return true;
    return false;
  }

  void Plan() {
    const int n = static_cast<int>(nodes_.size());
    // reachability from the heads: only those nodes run
    std::vector<char> need(n, 0);
    std::vector<int> stack;
    for (auto& h : heads_) stack.push_back(h.node);
    while (!stack.empty()) { const int i = stack.back(); stack.pop_back(); if (need[i]) continue; need[i] = 1; for (auto& e : nodes_[i].inputs) stack.push_back(e.node); }
    std::vector<int> consumers(n, 0);
    for (int i = 0; i < n; ++i) if (need[i]) for (auto& e : nodes_[i].inputs) ++consumers[e.node];
    for (auto& h : heads_) consumers[h.node] += 1 << 20;          // outputs stay alive

    storages_.clear(); order_.clear();
    for (auto& nd : nodes_) { nd.known = false; nd.storage = -1; nd.shape.clear(); }
    std::vector<int64_t> block_size;
    std::vector<int> free_blocks;
    auto release = [&](int sid) {
      Storage& s = storages_[sid];
      if (--s.ref == 0 && !s.external) free_blocks.push_back(s.block);
    };
    for (int i = 0; i < n; ++i) {
      if (!need[i]) continue;
      Node& nd = nodes_[i];
      if (nd.op == "null") {
        Storage s; s.external = true; s.ref = consumers[i];
        auto in = input_shapes_.find(nd.name);
        if (in != input_shapes_.end()) {
          nd.shape = in->second; nd.known = true;
        } else {
          auto p = params_->find(nd.name);
          if (p != params_->end()) { nd.shape = p->second.first; nd.known = true; }
          // else: a label (or an unused variable) — resolved by the consumer, which must not read it
        }
        if (nd.known) for (auto d : nd.shape) if (d < 1) throw std::runtime_error(nd.name + ": empty tensors are not supported, shape " + ShapeStr(nd.shape));
        s.size = nd.known ? Numel(nd.shape) : 0;
        nd.storage = static_cast<int>(storages_.size()); storages_.push_back(s);
        continue;
      }
      for (auto& e : nd.inputs) if (e.index != 0) throw std::runtime_error(nd.name + ": reads a secondary output, which the native predictor does not produce");
      InferShape(nd);
      const int64_t numel = Numel(nd.shape);
      const Node* src = nd.inputs.empty() ? nullptr : &nodes_[nd.inputs[0].node];
      if (IsView(nd.op) && src->known) {
        nd.storage = src->storage;
        storages_[nd.storage].ref += consumers[i];
      } else if (IsInplace(nd.op) && !storages_[src->storage].external && storages_[src->storage].ref == 1 && consumers[i] > 0) {
        nd.storage = src->storage;
        storages_[nd.storage].ref += consumers[i];
      } else {
        int best = -1;
        for (size_t f = 0; f < free_blocks.size(); ++f) {
          const int b = free_blocks[f];
          if (block_size[b] >= numel && (best < 0 || block_size[b] < block_size[free_blocks[best]])) best = static_cast<int>(f);
        }
        int blk;
        if (best >= 0) { blk = free_blocks[best]; free_blocks.erase(free_blocks.begin() + best); }
        else if (!free_blocks.empty()) {         // grow the largest free block instead of opening a new one
          size_t g = 0;
          for (size_t f = 1; f < free_blocks.size(); ++f) if (block_size[free_blocks[f]] > block_size[free_blocks[g]]) g = f;
          blk = free_blocks[g]; free_blocks.erase(free_blocks.begin() + g); block_size[blk] = numel;
        } else { blk = static_cast<int>(block_size.size()); block_size.push_back(numel); }
        Storage s; s.block = blk; s.size = numel; s.ref = std::max(consumers[i], 1);
        nd.storage = static_cast<int>(storages_.size()); storages_.push_back(s);
        if (consumers[i] == 0) release(nd.storage);
      }
      order_.push_back(i);
      for (auto& e : nd.inputs) if (nodes_[e.node].storage >= 0) release(nodes_[e.node].storage);
    }
    block_offset_.assign(block_size.size(), 0);
    arena_floats_ = 0;
    for (size_t b = 0; b < block_size.size(); ++b) { block_offset_[b] = arena_floats_; arena_floats_ += (block_size[b] + 15) / 16 * 16; }
    for (auto& h : heads_) if (!nodes_[h.node].known) throw std::runtime_error("output " + nodes_[h.node].name + " has no shape");
  }

  const Node& In(const Node& nd, size_t i) const {
    if (i >= nd.inputs.size()) throw std::runtime_error(nd.name + " (" + nd.op + "): missing input " + std::to_string(i));
    return nodes_[nd.inputs[i].node];
  }
  const Shape& InShape(const Node& nd, size_t i) const {
    const Node& s = In(nd, i);
    if (!s.known) throw std::runtime_error(nd.name + " (" + nd.op + "): input " + s.name + " has no value — not an input key and not in the parameter file");
    return s.shape;
  }
  void Need(const Node& nd, size_t i, const Shape& want) const {
    if (InShape(nd, i) != want) throw std::runtime_error(nd.name + ": " + In(nd, i).name + " has shape " + ShapeStr(InShape(nd, i)) + ", expected " + ShapeStr(want));
  }
  static int64_t Axis(int64_t a, size_t nd) { if (a < 0) a += static_cast<int64_t>(nd); if (a < 0 || a >= static_cast<int64_t>(nd)) throw std::runtime_error("axis out of range"); return a; }

  struct Conv { int64_t kh, kw, sh, sw, ph, pw, dh, dw, groups; };
  Conv ConvAttrs(const Node& nd) const {
    const auto k = nd.attrs.Tuple("kernel", {});
    if (k.size() != 2) throw std::runtime_error(nd.name + ": only 2-D convolution / pooling windows are supported by the native predictor");
    auto two = [&](const char* key, int64_t def) { auto v = nd.attrs.Tuple(key, {}); if (v.empty()) v = {def, def}; if (v.size() == 1) v.push_back(v[0]); return v; };
    const auto s = two("stride", 1), p = two("pad", 0), d = two("dilate", 1);
    if (k[0] < 1 || k[1] < 1 || s[0] < 1 || s[1] < 1 || d[0] < 1 || d[1] < 1 || p[0] < 0 || p[1] < 0 || k[0] > 4096 || k[1] > 4096 || p[0] > 4096 || p[1] > 4096)
      throw std::runtime_error(nd.name + ": kernel / stride / dilate must be positive and pad non-negative");
    return Conv{k[0], k[1], s[0], s[1], p[0], p[1], d[0], d[1], nd.attrs.Int("num_group", 1)};
  }
  struct Pool { int64_t kh, kw, sh, sw, ph, pw; bool global, full; int type; bool count_pad; };
  Pool PoolAttrs(const Node& nd, const Shape& x) const {
    Pool p{};
    p.global = nd.attrs.Bool("global_pool", false);
    const std::string t = nd.attrs.Str("pool_type", "max");
    p.type = t == "max" ? 0 : t == "avg" ? 1 : t == "sum" ? 2 : -1;
    if (p.type < 0) throw std::runtime_error(nd.name + ": pool_type " + t + " is not supported");
    p.full = nd.attrs.Str("pooling_convention", "valid") == "full";
    p.count_pad = nd.attrs.Bool("count_include_pad", true);
    if (p.global) { p.kh = x[2]; p.kw = x[3]; p.sh = p.sw = 1; p.ph = p.pw = 0; return p; }
    auto k = nd.attrs.Tuple("kernel", {});
    if (k.size() == 1) k.push_back(k[0]);
    if (k.size() != 2) throw std::runtime_error(nd.name + ": only 2-D pooling is supported");
    auto s = nd.attrs.Tuple("stride", {});
    if (s.empty()) s = nd.nnvm ? Shape{1, 1} : k;            // symbol.py: an absent stride means the window; nnvm: 1
    if (s.size() == 1) s.push_back(s[0]);
    auto pd = nd.attrs.Tuple("pad", {0, 0});
    if (pd.empty()) pd = {0, 0};
    if (pd.size() == 1) pd.push_back(pd[0]);
    p.kh = k[0]; p.kw = k[1]; p.sh = s[0]; p.sw = s[1]; p.ph = pd[0]; p.pw = pd[1];
    if (p.kh < 1 || p.kw < 1 || p.sh < 1 || p.sw < 1 || p.ph < 0 || p.pw < 0 || p.ph >= p.kh || p.pw >= p.kw)
      throw std::runtime_error(nd.name + ": pooling needs kernel >= 1, stride >= 1 and 0 <= pad < kernel");
    return p;
  }
  static int64_t PoolOut(int64_t in, int64_t k, int64_t s, int64_t p, bool full) {
    const int64_t span = in + 2 * p - k;
    if (span < 0) throw std::runtime_error("pooling window larger than the padded input");
    return (full ? (span + s - 1) / s : span / s) + 1;
  }

  static Shape Broadcast(const Shape& a, const Shape& b, const std::string& who) {
    const size_t n = std::max(a.size(), b.size());
    Shape out(n);
    for (size_t i = 0; i < n; ++i) {
      const int64_t x = i + a.size() >= n ? a[i + a.size() - n] : 1, y = i + b.size() >= n ? b[i + b.size() - n] : 1;
      if (x != y && x != 1 && y != 1) throw std::runtime_error(who + ": shapes " + ShapeStr(a) + " and " + ShapeStr(b) + " do not broadcast");
      out[i] = std::max(x, y);
    }
    return out;
  }
  static int BinaryKind(const std::string& op) {
    static const std::pair<const char*, int> k[] = {
      {"_plus", 0}, {"_Plus", 0}, {"elemwise_add", 0}, {"broadcast_add", 0}, {"broadcast_plus", 0}, {"_add", 0}, {"add", 0},
      {"_minus", 1}, {"_Minus", 1}, {"elemwise_sub", 1}, {"broadcast_sub", 1}, {"broadcast_minus", 1}, {"_sub", 1}, {"subtract", 1},
      {"_mul", 2}, {"_Mul", 2}, {"elemwise_mul", 2}, {"broadcast_mul", 2}, {"multiply", 2},
      {"_div", 3}, {"_Div", 3}, {"elemwise_div", 3}, {"broadcast_div", 3}, {"divide", 3},
      {"broadcast_maximum", 4}, {"_maximum", 4}, {"maximum", 4}, {"broadcast_minimum", 5}, {"_minimum", 5}, {"minimum", 5}};
    for (auto& e : k) if (op == e.first) return e.second;
    return -1;
  }
  static int ScalarKind(const std::string& op) {
    static const std::pair<const char*, int> k[] = {{"_plus_scalar", 0}, {"_PlusScalar", 0}, {"_minus_scalar", 1}, {"_MinusScalar", 1}, {"_mul_scalar", 2}, {"_MulScalar", 2},
                                                     {"_div_scalar", 3}, {"_DivScalar", 3}, {"_rminus_scalar", 4}, {"_RMinusScalar", 4}, {"_rdiv_scalar", 5}, {"_RDivScalar", 5}};
    for (auto& e : k) if (op == e.first) return e.second;
    return -1;
  }
  static int UnaryKind(const std::string& op) {
    static const std::pair<const char*, int> k[] = {{"relu", 0}, {"sigmoid", 1}, {"tanh", 2}, {"exp", 3}, {"log", 4}, {"sqrt", 5}, {"abs", 6}, {"negative", 7}, {"square", 8},
                                                     {"softsign", 9}, {"softrelu", 10}};
    for (auto& e : k) if (op == e.first) return e.second;
    return -1;
  }

  void InferShape(Node& nd) {
    const std::string& op = nd.op;
    const Attrs& a = nd.attrs;
    if (op == "FullyConnected") {
      const Shape& x = InShape(nd, 0);
      const int64_t h = a.Int("num_hidden", 0);
      const bool flat = a.Bool("flatten", true);
      if (x.empty()) throw std::runtime_error(nd.name + ": scalar input");
      const int64_t k = flat ? Numel(x) / x[0] : x.back();
      Need(nd, 1, {h, k});
      if (!a.Bool("no_bias", false)) Need(nd, 2, {h});
      if (flat) nd.shape = {x[0], h}; else { nd.shape = x; nd.shape.back() = h; }
    } else if (op == "Convolution") {
      const Shape& x = InShape(nd, 0);
      if (x.size() != 4) throw std::runtime_error(nd.name + ": convolution input must be NCHW, got " + ShapeStr(x));
      const Conv c = ConvAttrs(nd);
      const int64_t f = a.Int("num_filter", 0);
      if (c.groups < 1 || x[1] % c.groups || f % c.groups) throw std::runtime_error(nd.name + ": channels are not divisible by num_group");
      Need(nd, 1, {f, x[1] / c.groups, c.kh, c.kw});
      if (!a.Bool("no_bias", false)) Need(nd, 2, {f});
      const int64_t oh = (x[2] + 2 * c.ph - c.dh * (c.kh - 1) - 1) / c.sh + 1, ow = (x[3] + 2 * c.pw - c.dw * (c.kw - 1) - 1) / c.sw + 1;
      if (oh <= 0 || ow <= 0) throw std::runtime_error(nd.name + ": kernel larger than the padded input");
      nd.shape = {x[0], f, oh, ow};
    } else if (op == "Pooling") {
      const Shape& x = InShape(nd, 0);
      if (x.size() != 4) throw std::runtime_error(nd.name + ": pooling input must be NCHW");
      const Pool p = PoolAttrs(nd, x);
      nd.shape = {x[0], x[1], p.global ? 1 : PoolOut(x[2], p.kh, p.sh, p.ph, p.full), p.global ? 1 : PoolOut(x[3], p.kw, p.sw, p.pw, p.full)};
    } else if (op == "Flatten" || op == "flatten") {
      const Shape& x = InShape(nd, 0);
      nd.shape = {x.empty() ? 1 : x[0], x.empty() ? 1 : Numel(x) / std::max<int64_t>(x[0], 1)};
    } else if (op == "Reshape" || op == "reshape") {
      const Shape& x = InShape(nd, 0);
      const auto spec = a.Tuple("shape", {});
      Shape out; size_t src = 0; int infer = -1;
      for (size_t i = 0; i < spec.size(); ++i) {
        const int64_t d = spec[i];
        if (d > 0) { out.push_back(d); ++src; }
        else if (d == 0) { if (src >= x.size()) throw std::runtime_error(nd.name + ": reshape code 0 past the input rank"); out.push_back(x[src++]); }
        else if (d == -1) { if (infer >= 0) throw std::runtime_error(nd.name + ": two -1 in reshape"); infer = static_cast<int>(out.size()); out.push_back(1); ++src; }
        else if (d == -2) { while (src < x.size()) out.push_back(x[src++]); }
        else if (d == -3) { if (src + 1 >= x.size()) throw std::runtime_error(nd.name + ": reshape code -3 past the input rank"); out.push_back(x[src] * x[src + 1]); src += 2; }
        else throw std::runtime_error(nd.name + ": reshape code " + std::to_string(d) + " is not supported");
      }
      if (infer >= 0) { const int64_t rest = Numel(out); if (rest == 0 || Numel(x) % rest) throw std::runtime_error(nd.name + ": cannot infer -1"); out[infer] = Numel(x) / rest; }
      if (Numel(out) != Numel(x)) throw std::runtime_error(nd.name + ": reshape " + ShapeStr(x) + " -> " + ShapeStr(out) + " changes the size");
      nd.shape = out;
    } else if (op == "expand_dims") {
      Shape x = InShape(nd, 0);
      int64_t ax = a.Int("axis", 0); if (ax < 0) ax += static_cast<int64_t>(x.size()) + 1;
      if (ax < 0 || ax > static_cast<int64_t>(x.size())) throw std::runtime_error(nd.name + ": axis out of range");
      x.insert(x.begin() + ax, 1); nd.shape = x;
    } else if (op == "BatchNorm") {
      const Shape& x = InShape(nd, 0);
      const int64_t ax = Axis(a.Int("axis", 1), x.size());
      for (size_t i = 1; i <= 4; ++i) Need(nd, i, {x[ax]});
      nd.shape = x;
    } else if (op == "Concat" || op == "concat") {
      Shape out = InShape(nd, 0);
      const int64_t ax = Axis(a.Int("dim", 1), out.size());
      for (size_t i = 1; i < nd.inputs.size(); ++i) {
        const Shape& s = InShape(nd, i);
        if (s.size() != out.size()) throw std::runtime_error(nd.name + ": concat inputs differ in rank");
        for (size_t d = 0; d < s.size(); ++d) if (static_cast<int64_t>(d) != ax && s[d] != out[d]) throw std::runtime_error(nd.name + ": concat inputs differ outside the axis");
        out[ax] += s[ax];
      }
      nd.shape = out;
    } else if (op == "transpose") {
      const Shape& x = InShape(nd, 0);
      auto axes = a.Tuple("axes", {});
      if (axes.empty()) for (size_t i = 0; i < x.size(); ++i) axes.push_back(static_cast<int64_t>(x.size() - 1 - i));
      if (axes.size() != x.size()) throw std::runtime_error(nd.name + ": axes do not match the input rank");
      std::vector<char> seen(x.size(), 0);
      nd.shape.resize(x.size());
      for (size_t i = 0; i < x.size(); ++i) { const int64_t ax = Axis(axes[i], x.size()); if (seen[ax]) throw std::runtime_error(nd.name + ": repeated axis"); seen[ax] = 1; nd.shape[i] = x[ax]; }
    } else if (op == "Embedding") {
      const Shape& x = InShape(nd, 0);
      const Shape& w = InShape(nd, 1);
      if (w.size() != 2) throw std::runtime_error(nd.name + ": embedding weight must be 2-D");
      nd.shape = x; nd.shape.push_back(w[1]);
    } else if (BinaryKind(op) >= 0) {
      nd.shape = Broadcast(InShape(nd, 0), InShape(nd, 1), nd.name);
    } else if (op == "add_n" || op == "ElementWiseSum") {
      nd.shape = InShape(nd, 0);
      for (size_t i = 1; i < nd.inputs.size(); ++i) Need(nd, i, nd.shape);
    } else if (op == "Activation" || op == "LeakyReLU" || op == "Dropout" || op == "softmax" || op == "log_softmax" || op == "SoftmaxOutput" || op == "Softmax" ||
               op == "SoftmaxActivation" || op == "LinearRegressionOutput" || op == "MAERegressionOutput" || op == "LogisticRegressionOutput" || op == "identity" ||
               op == "_copy" || op == "BlockGrad" || op == "stop_gradient" || op == "clip" || ScalarKind(op) >= 0 || UnaryKind(op) >= 0) {
      nd.shape = InShape(nd, 0);
    } else {
      throw std::runtime_error("operator " + op + " (node " + nd.name + ") is not supported by the native predictor");
    }
    nd.known = true;
  }
};

// the host runner of a GraphPlan: fp32 on the CPU, the arena and the input buffers in host memory, parameters read in place
class Predictor : public GraphPlan {
 public:
  Predictor(const std::string& json, const char* params, size_t param_size, const std::vector<std::string>& input_keys,
            const std::vector<Shape>& input_shapes, const std::vector<std::string>& output_keys)
      : GraphPlan(json, params, param_size, input_keys, input_shapes, output_keys) {
    Bind();
  }
  // another predictor over the same graph and parameters with its own inputs and arena (MXPredCreateMultiThread / MXPredReshape)
  std::unique_ptr<Predictor> Clone(const std::map<std::string, Shape>* new_shapes) const {
    std::unique_ptr<Predictor> p(new Predictor(*this));
    p->Replan(new_shapes);
    p->Bind();
    return p;
  }

  void SetInput(const std::string& key, const float* data, size_t size) {
    auto it = inputs_.find(key);
    if (it == inputs_.end()) throw std::runtime_error("SetInput: unknown input " + key);
    if (size != it->second.size()) throw std::runtime_error("SetInput: " + key + " expects " + std::to_string(it->second.size()) + " values, got " + std::to_string(size));
    memcpy(it->second.data(), data, size * sizeof(float));
  }
  void Forward() { for (size_t i = 0; i < order_.size(); ++i) Run(order_[i]); }
  // one operator per call (MXPredPartialForward): step counts executed operators, step_left reaches 0 after the last one
  void PartialForward(int step, int* step_left) {
    if (step < 0 || step >= static_cast<int>(order_.size())) { *step_left = 0; return; }
    Run(order_[step]);
    *step_left = static_cast<int>(order_.size()) - step - 1;
  }
  void GetOutput(size_t i, float* out, size_t size) const {
    const Node& n = nodes_[Head(i)];
    if (size != static_cast<size_t>(Numel(n.shape))) throw std::runtime_error("GetOutput: output " + std::to_string(i) + " has " + std::to_string(Numel(n.shape)) + " values, buffer holds " + std::to_string(size));
    memcpy(out, storages_[n.storage].ptr, size * sizeof(float));
  }

 private:
  Predictor(const Predictor&) = default;
  std::map<std::string, std::vector<float>> inputs_;
  std::vector<float> arena_;

  // host memory behind the plan: zeroed input buffers, parameters in place, one arena for every other storage
  void Bind() {
    inputs_.clear();
    for (auto& nd : nodes_) {
      if (nd.op != "null" || nd.storage < 0) continue;
      Storage& s = storages_[nd.storage];
      if (IsInput(nd)) { auto& buf = inputs_[nd.name]; buf.assign(static_cast<size_t>(Numel(nd.shape)), 0.f); s.ptr = buf.data(); }
      else if (nd.known) s.ptr = params_->at(nd.name).second.data();
    }
    arena_.assign(static_cast<size_t>(arena_floats_), 0.f);
    for (auto& s : storages_) if (!s.external) s.ptr = arena_.data() + block_offset_[s.block];
  }
  const float* InPtr(const Node& nd, size_t i) const { return storages_[In(nd, i).storage].ptr; }

  // ---- execution
  static float Act(int kind, float v) {
    switch (kind) {
      case 0: return v > 0 ? v : 0.f;
      case 1: return 1.f / (1.f + std::exp(-v));
      case 2: return std::tanh(v);
      case 3: return std::exp(v);
      case 4: return std::log(v);
      case 5: return std::sqrt(v);
      case 6: return std::fabs(v);
      case 7: return -v;
      case 8: return v * v;
      case 9: return v / (1.f + std::fabs(v));
      default: return v > 20.f ? v : std::log1p(std::exp(v));      // softrelu
    }
  }
  static void Map(int kind, const float* x, float* y, int64_t n) { for (int64_t i = 0; i < n; ++i) y[i] = Act(kind, x[i]); }

  void Softmax(const Node& nd, const float* x, float* y, int64_t axis, bool log) const {
    const Shape& s = nd.shape;
    const int64_t ax = Axis(axis, s.size()), C = s[ax];
    int64_t inner = 1; for (size_t i = ax + 1; i < s.size(); ++i) inner *= s[i];
    const int64_t outer = Numel(s) / (C * inner);
    for (int64_t o = 0; o < outer; ++o) for (int64_t in = 0; in < inner; ++in) {
      const float* px = x + o * C * inner + in; float* py = y + o * C * inner + in;
      float m = -std::numeric_limits<float>::infinity();
      for (int64_t c = 0; c < C; ++c) m = std::max(m, px[c * inner]);
      double sum = 0;
      for (int64_t c = 0; c < C; ++c) sum += std::exp(static_cast<double>(px[c * inner] - m));
      const float lse = static_cast<float>(std::log(sum));
      for (int64_t c = 0; c < C; ++c) { const float v = px[c * inner] - m - lse; py[c * inner] = log ? v : std::exp(v); }
    }
  }

  void Run(int id) {
    Node& nd = nodes_[id];
    const std::string& op = nd.op;
    const Attrs& a = nd.attrs;
    float* y = storages_[nd.storage].ptr;
    const int64_t n = Numel(nd.shape);
    if (IsView(op)) return;
    const float* x = InPtr(nd, 0);
    const Shape& xs = In(nd, 0).shape;
    int k;
    if (op == "FullyConnected") {
      const Shape& w = In(nd, 1).shape;
      GemmNT(x, InPtr(nd, 1), y, n / w[0], w[0], w[1], a.Bool("no_bias", false) ? nullptr : InPtr(nd, 2));
    } else if (op == "Convolution") {
      RunConv(nd, x, xs, y);
    } else if (op == "Pooling") {
      RunPool(nd, x, xs, y);
    } else if (op == "Activation") {
      const std::string t = a.Str("act_type", "relu");
      k = UnaryKind(t);
      if (k < 0) throw std::runtime_error(nd.name + ": act_type " + t + " is not supported");
      Map(k, x, y, n);
    } else if (op == "LeakyReLU") {
      const std::string t = a.Str("act_type", "leaky");
      const float slope = static_cast<float>(a.Float("slope", 0.25));
      if (t == "leaky") for (int64_t i = 0; i < n; ++i) y[i] = x[i] > 0 ? x[i] : slope * x[i];
      else if (t == "elu") for (int64_t i = 0; i < n; ++i) y[i] = x[i] > 0 ? x[i] : slope * (std::exp(x[i]) - 1.f);
      else throw std::runtime_error(nd.name + ": LeakyReLU act_type " + t + " is not supported");
    } else if ((k = UnaryKind(op)) >= 0) {
      Map(k, x, y, n);
    } else if (op == "clip") {
      const float lo = static_cast<float>(a.Float("a_min", -std::numeric_limits<float>::infinity())), hi = static_cast<float>(a.Float("a_max", std::numeric_limits<float>::infinity()));
      for (int64_t i = 0; i < n; ++i) y[i] = std::min(std::max(x[i], lo), hi);
    } else if (op == "LogisticRegressionOutput") {
      Map(1, x, y, n);
    } else if (op == "BatchNorm") {
      const int64_t ax = Axis(a.Int("axis", 1), xs.size()), C = xs[ax];
      int64_t inner = 1; for (size_t i = ax + 1; i < xs.size(); ++i) inner *= xs[i];
      const float eps = static_cast<float>(a.Float("eps", 1e-3));
      const bool fix_gamma = a.Bool("fix_gamma", nd.nnvm);
      const float *g = InPtr(nd, 1), *b = InPtr(nd, 2), *mean = InPtr(nd, 3), *var = InPtr(nd, 4);
      std::vector<float> scale(C), shift(C);
      for (int64_t c = 0; c < C; ++c) { scale[c] = (fix_gamma ? 1.f : g[c]) / std::sqrt(var[c] + eps); shift[c] = b[c] - mean[c] * scale[c]; }
      for (int64_t i = 0; i < n; ++i) { const int64_t c = (i / inner) % C; y[i] = x[i] * scale[c] + shift[c]; }
    } else if (op == "Concat" || op == "concat") {
      const int64_t ax = Axis(a.Int("dim", 1), nd.shape.size());
      int64_t inner = 1; for (size_t i = ax + 1; i < nd.shape.size(); ++i) inner *= nd.shape[i];
      const int64_t outer = n / (nd.shape[ax] * inner);
      int64_t at = 0;
      for (size_t j = 0; j < nd.inputs.size(); ++j) {
        const int64_t c = In(nd, j).shape[ax];
        const float* p = InPtr(nd, j);
        for (int64_t o = 0; o < outer; ++o) memcpy(y + (o * nd.shape[ax] + at) * inner, p + o * c * inner, static_cast<size_t>(c * inner) * sizeof(float));
        at += c;
      }
    } else if (op == "softmax" || op == "log_softmax") {
      Softmax(nd, x, y, a.Int("axis", -1), op == "log_softmax");
    } else if (op == "SoftmaxOutput" || op == "Softmax") {
      Softmax(nd, x, y, nd.shape.size() < 2 ? 0 : (a.Bool("preserve_shape", false) ? -1 : 1), false);
    } else if (op == "SoftmaxActivation") {
      if (a.Str("mode", "instance") == "channel" || nd.shape.size() <= 2) Softmax(nd, x, y, nd.shape.size() < 2 ? 0 : 1, false);
      else { Node flat; flat.shape = {nd.shape[0], n / nd.shape[0]}; Softmax(flat, x, y, 1, false); }     // instance: over everything but the batch axis
    } else if (op == "transpose") {
      auto axes = a.Tuple("axes", {});
      const size_t r = xs.size();
      if (axes.empty()) for (size_t i = 0; i < r; ++i) axes.push_back(static_cast<int64_t>(r - 1 - i));
      std::vector<int64_t> xstride(r, 1), step(r);
      for (int i = static_cast<int>(r) - 2; i >= 0; --i) xstride[i] = xstride[i + 1] * xs[i + 1];
      for (size_t i = 0; i < r; ++i) step[i] = xstride[Axis(axes[i], r)];
      std::vector<int64_t> idx(r, 0);
      int64_t src = 0;
      for (int64_t i = 0; i < n; ++i) {
        y[i] = x[src];
        for (int d = static_cast<int>(r) - 1; d >= 0; --d) {
          src += step[d];
          if (++idx[d] < nd.shape[d]) break;
          src -= step[d] * nd.shape[d]; idx[d] = 0;
        }
      }
    } else if (op == "Embedding") {
      const Shape& w = In(nd, 1).shape;
      const float* wp = InPtr(nd, 1);
      const int64_t rows = Numel(xs);
      for (int64_t i = 0; i < rows; ++i) {
        int64_t r = static_cast<int64_t>(x[i]);
        r = std::min(std::max<int64_t>(r, 0), w[0] - 1);
        memcpy(y + i * w[1], wp + r * w[1], static_cast<size_t>(w[1]) * sizeof(float));
      }
    } else if ((k = BinaryKind(op)) >= 0) {
      RunBinary(nd, k, x, InPtr(nd, 1), y);
    } else if ((k = ScalarKind(op)) >= 0) {
      const float s = static_cast<float>(a.Float("scalar", 0.0));
      switch (k) {
        case 0: for (int64_t i = 0; i < n; ++i) y[i] = x[i] + s; break;
        case 1: for (int64_t i = 0; i < n; ++i) y[i] = x[i] - s; break;
        case 2: for (int64_t i = 0; i < n; ++i) y[i] = x[i] * s; break;
        case 3: for (int64_t i = 0; i < n; ++i) y[i] = x[i] / s; break;
        case 4: for (int64_t i = 0; i < n; ++i) y[i] = s - x[i]; break;
        default: for (int64_t i = 0; i < n; ++i) y[i] = s / x[i]; break;
      }
    } else if (op == "add_n" || op == "ElementWiseSum") {
      for (int64_t i = 0; i < n; ++i) y[i] = x[i];
      for (size_t j = 1; j < nd.inputs.size(); ++j) { const float* p = InPtr(nd, j); for (int64_t i = 0; i < n; ++i) y[i] += p[i]; }
    } else {
      throw std::runtime_error("operator " + op + " has no native kernel");
    }
  }

  static float Bin(int k, float p, float q) {
    switch (k) { case 0: return p + q; case 1: return p - q; case 2: return p * q; case 3: return p / q; case 4: return std::max(p, q); default: return std::min(p, q); }
  }
  void RunBinary(const Node& nd, int k, const float* p, const float* q, float* y) const {
    const Shape& ps = In(nd, 0).shape; const Shape& qs = In(nd, 1).shape;
    const int64_t n = Numel(nd.shape);
    if (ps == qs) { for (int64_t i = 0; i < n; ++i) y[i] = Bin(k, p[i], q[i]); return; }
    const size_t r = nd.shape.size();
    std::vector<int64_t> sp(r, 0), sq(r, 0), idx(r, 0);
    auto strides = [&](const Shape& s, std::vector<int64_t>& out) {
      int64_t st = 1;
      for (int i = static_cast<int>(s.size()) - 1; i >= 0; --i) { out[i + r - s.size()] = s[i] == 1 ? 0 : st; st *= s[i]; }
    };
    strides(ps, sp); strides(qs, sq);
    int64_t ip = 0, iq = 0;
    for (int64_t i = 0; i < n; ++i) {
      y[i] = Bin(k, p[ip], q[iq]);
      for (int d = static_cast<int>(r) - 1; d >= 0; --d) {
        ip += sp[d]; iq += sq[d];
        if (++idx[d] < nd.shape[d]) break;
        ip -= sp[d] * nd.shape[d]; iq -= sq[d] * nd.shape[d]; idx[d] = 0;
      }
    }
  }

  // convolution = per-image im2col + weight-row x column-matrix accumulation (i-k-j order: the inner loop runs over output pixels)
  void RunConv(const Node& nd, const float* x, const Shape& xs, float* y) {
    const Conv c = ConvAttrs(nd);
    const float* w = InPtr(nd, 1);
    const float* bias = nd.attrs.Bool("no_bias", false) ? nullptr : InPtr(nd, 2);
    const int64_t B = xs[0], C = xs[1], H = xs[2], W = xs[3], F = nd.shape[1], OH = nd.shape[2], OW = nd.shape[3];
    const int64_t cg = C / c.groups, fg = F / c.groups, K = cg * c.kh * c.kw, P = OH * OW;
    const bool pointwise = c.kh == 1 && c.kw == 1 && c.sh == 1 && c.sw == 1 && c.ph == 0 && c.pw == 0;
    ParallelFor(B, static_cast<double>(B) * F * K * P, [&](int64_t lo, int64_t hi) {
      std::vector<float> col(pointwise ? 0 : static_cast<size_t>(K * P));
      for (int64_t b = lo; b < hi; ++b) for (int64_t g = 0; g < c.groups; ++g) {
        const float* xg = x + (b * C + g * cg) * H * W;
        const float* cm = xg;
        if (!pointwise) {
          for (int64_t ci = 0; ci < cg; ++ci) for (int64_t i = 0; i < c.kh; ++i) for (int64_t j = 0; j < c.kw; ++j) {
            float* dst = col.data() + ((ci * c.kh + i) * c.kw + j) * P;
            for (int64_t oh = 0; oh < OH; ++oh) {
              const int64_t ih = oh * c.sh - c.ph + i * c.dh;
              if (ih < 0 || ih >= H) { for (int64_t ow = 0; ow < OW; ++ow) dst[oh * OW + ow] = 0.f; continue; }
              const float* src = xg + (ci * H + ih) * W;
              for (int64_t ow = 0; ow < OW; ++ow) { const int64_t iw = ow * c.sw - c.pw + j * c.dw; dst[oh * OW + ow] = (iw >= 0 && iw < W) ? src[iw] : 0.f; }
            }
          }
          cm = col.data();
        }
        for (int64_t f = 0; f < fg; ++f) {
          float* out = y + ((b * F + g * fg + f) * P);
          const float b0 = bias ? bias[g * fg + f] : 0.f;
          for (int64_t p = 0; p < P; ++p) out[p] = b0;
          const float* wr = w + (g * fg + f) * K;
          for (int64_t kk = 0; kk < K; ++kk) { const float wv = wr[kk]; const float* cr = cm + kk * P; for (int64_t p = 0; p < P; ++p) out[p] += wv * cr[p]; }
        }
      }
    });
  }

  void RunPool(const Node& nd, const float* x, const Shape& xs, float* y) const {
    const Pool p = PoolAttrs(nd, xs);
    const int64_t planes = xs[0] * xs[1], H = xs[2], W = xs[3], OH = nd.shape[2], OW = nd.shape[3];
    ParallelFor(planes, static_cast<double>(planes) * OH * OW * p.kh * p.kw, [&](int64_t lo, int64_t hi) {
      for (int64_t pl = lo; pl < hi; ++pl) {
        const float* src = x + pl * H * W; float* dst = y + pl * OH * OW;
        for (int64_t oh = 0; oh < OH; ++oh) for (int64_t ow = 0; ow < OW; ++ow) {
          const int64_t h0 = oh * p.sh - p.ph, w0 = ow * p.sw - p.pw;
          const int64_t h1 = std::min(h0 + p.kh, H + p.ph), w1 = std::min(w0 + p.kw, W + p.pw);     // window clipped to the padded plane
          const int64_t hs = std::max<int64_t>(h0, 0), ws = std::max<int64_t>(w0, 0), he = std::min(h1, H), we = std::min(w1, W);
          float acc = p.type == 0 ? -std::numeric_limits<float>::infinity() : 0.f;
          for (int64_t h = hs; h < he; ++h) for (int64_t w = ws; w < we; ++w) { const float v = src[h * W + w]; acc = p.type == 0 ? std::max(acc, v) : acc + v; }
          if (p.type == 1) { const int64_t cnt = p.count_pad ? (h1 - h0) * (w1 - w0) : (he - hs) * (we - ws); acc /= static_cast<float>(std::max<int64_t>(cnt, 1)); }
          if (p.type == 0 && (he <= hs || we <= ws)) acc = 0.f;
          dst[oh * OW + ow] = acc;
        }
      }
    });
  }
};

// MXNDList*: a parsed NDArray-list file handed out as float arrays
struct NDList {
  std::vector<std::string> names;
  std::vector<std::vector<float>> data;
  std::vector<std::vector<uint32_t>> shapes;
  NDList(const char* blob, size_t size) {
    BufReader r(blob, size);
    if (r.Get<uint64_t>() != kListMagic) throw std::runtime_error("not an NDArray list");
    r.Get<uint64_t>();
    const uint64_t n = r.Get<uint64_t>();
    if (n > (1u << 24)) throw std::runtime_error("implausible array count");
    for (uint64_t i = 0; i < n; ++i) {
      NDRec a = ReadArray(r);
      data.push_back(ToFloat(a));
      shapes.emplace_back(a.shape.begin(), a.shape.end());
    }
    const uint64_t m = r.Get<uint64_t>();
    if (m != 0 && m != n) throw std::runtime_error("name count does not match the array count");
    for (uint64_t i = 0; i < m; ++i) { const uint64_t l = r.Get<uint64_t>(); names.push_back(r.Raw(l)); }
    names.resize(n);
  }
};

}  // namespace predict
}  // namespace gxrt
