// Host training executor over the native graph (graph.h): binds argument / gradient / auxiliary arrays, runs forward (training or inference
// mode) and backward in fp32 on the CPU.  It is what GXExecutor* and the GXAutograd* / GXImperativeInvoke C API run on (c_api_graph.cc), i.e.
// the path a non-Python front end uses to TRAIN through this framework without PyTorch in the process.
//
// Parity: include/mxnet/c_api.h:1530-1760 (MXExecutorBind / BindX / BindEX / SimpleBind, Forward, Backward(Ex), Outputs, Print, Free) over
// src/executor/graph_executor.cc (Init / InitArguments / Forward / Backward / RunOps) and the operator gradients registered with FGradient
// (src/operator/nn/*.cc, src/operator/softmax_output-inl.h, regression_output-inl.h).  The reference builds a separate backward graph with
// nnvm::pass::Gradient and plans memory for both; here the forward activations are kept per node and the backward pass is a reverse sweep
// that calls one gradient routine per operator — on the host the simplicity is worth more than the reuse (the device path's equivalents are
// the fused sm_100a kernels and the CUDA-graph executor of models/cnn.py, DESIGN.md §1).  Its device twin for graphs bound to device arrays
// of the C API is device_exec.h::DeviceExecutor: same slot layout and gradient-flow rules, sm_100a kernels per node.
#pragma once
#include <atomic>
#include <cstring>
#include <mutex>
#include <random>

#include "graph.h"

namespace gxrt {
namespace exec {

using graph::AttrView;
using graph::Entry;
using graph::Node;
using graph::Symbol;
using predict::Numel;
using predict::ParallelFor;
using predict::Shape;
using predict::ShapeStr;

enum GradReq { kNullOp = 0, kWriteTo = 1, kWriteInplace = 2, kAddTo = 3 };

// ------------------------------------------------------------------------------------------------ dense kernels
// serial C[M,N] (+)= op(A) . op(B); the j-inner loops vectorise.  A is [M,K] (ta = false) or [K,M]; B is [K,N] (tb = false) or [N,K].
inline void GemmSerial(bool ta, bool tb, int64_t M, int64_t N, int64_t K, const float* A, const float* B, float* C, bool accumulate) {
  if (!accumulate) std::fill(C, C + M * N, 0.f);
  if (!tb) {
    for (int64_t i = 0; i < M; ++i) {
      float* c = C + i * N;
      for (int64_t k = 0; k < K; ++k) {
        const float a = ta ? A[k * M + i] : A[i * K + k];
        if (a == 0.f) continue;
        const float* b = B + k * N;
        for (int64_t j = 0; j < N; ++j) c[j] += a * b[j];
      }
    }
  } else if (!ta) {
    for (int64_t i = 0; i < M; ++i) for (int64_t j = 0; j < N; ++j) {
      const float* a = A + i * K; const float* b = B + j * K;
      float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      int64_t k = 0;
      for (; k + 8 <= K; k += 8) for (int u = 0; u < 8; ++u) acc[u] += a[k + u] * b[k + u];
      float s = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
      for (; k < K; ++k) s += a[k] * b[k];
      C[i * N + j] += s;
    }
  } else {
    for (int64_t i = 0; i < M; ++i) for (int64_t j = 0; j < N; ++j) {
      float s = 0;
      for (int64_t k = 0; k < K; ++k) s += A[k * M + i] * B[j * K + k];
      C[i * N + j] += s;
    }
  }
}
// rows of C split over threads
inline void Gemm(bool ta, bool tb, int64_t M, int64_t N, int64_t K, const float* A, const float* B, float* C, bool accumulate) {
  ParallelFor(M, static_cast<double>(M) * N * K, [&](int64_t lo, int64_t hi) {
    if (!ta) GemmSerial(false, tb, hi - lo, N, K, A + lo * K, B, C + lo * N, accumulate);
    else {
      // A^T rows lo..hi are columns of A: walk them in place
      for (int64_t i = lo; i < hi; ++i) {
        float* c = C + i * N;
        if (!accumulate) std::fill(c, c + N, 0.f);
        for (int64_t k = 0; k < K; ++k) {
          const float a = A[k * M + i];
          if (a == 0.f) continue;
          if (!tb) { const float* b = B + k * N; for (int64_t j = 0; j < N; ++j) c[j] += a * b[j]; }
          else for (int64_t j = 0; j < N; ++j) c[j] += a * B[j * K + k];
        }
      }
    }
  });
}

struct Win { int64_t kh, kw, sh, sw, ph, pw, dh, dw; };

inline void Im2Col(const float* x, int64_t C, int64_t H, int64_t W, const Win& w, int64_t OH, int64_t OW, float* col) {
  for (int64_t c = 0; c < C; ++c) for (int64_t r = 0; r < w.kh; ++r) for (int64_t s = 0; s < w.kw; ++s) {
    float* row = col + ((c * w.kh + r) * w.kw + s) * OH * OW;
    for (int64_t oy = 0; oy < OH; ++oy) {
      const int64_t iy = oy * w.sh - w.ph + r * w.dh;
      if (iy < 0 || iy >= H) { std::fill(row + oy * OW, row + (oy + 1) * OW, 0.f); continue; }
      for (int64_t ox = 0; ox < OW; ++ox) {
        const int64_t ix = ox * w.sw - w.pw + s * w.dw;
        row[oy * OW + ox] = (ix >= 0 && ix < W) ? x[(c * H + iy) * W + ix] : 0.f;
      }
    }
  }
}
inline void Col2Im(const float* col, int64_t C, int64_t H, int64_t W, const Win& w, int64_t OH, int64_t OW, float* dx) {
  for (int64_t c = 0; c < C; ++c) for (int64_t r = 0; r < w.kh; ++r) for (int64_t s = 0; s < w.kw; ++s) {
    const float* row = col + ((c * w.kh + r) * w.kw + s) * OH * OW;
    for (int64_t oy = 0; oy < OH; ++oy) {
      const int64_t iy = oy * w.sh - w.ph + r * w.dh;
      if (iy < 0 || iy >= H) continue;
      for (int64_t ox = 0; ox < OW; ++ox) {
        const int64_t ix = ox * w.sw - w.pw + s * w.dw;
        if (ix >= 0 && ix < W) dx[(c * H + iy) * W + ix] += row[oy * OW + ox];
      }
    }
  }
}

inline float ActF(int kind, float v) {
  switch (kind) {
    case 0: return v > 0 ? v : 0;
    case 1: return 1.f / (1.f + std::exp(-v));
    case 2: return std::tanh(v);
    case 3: return v > 20.f ? v : std::log1p(std::exp(v));      // softrelu
    case 4: return v / (1.f + std::fabs(v));                    // softsign
    default: return v;
  }
}
// derivative from input x and output y
inline float ActG(int kind, float x, float y) {
  switch (kind) {
    case 0: return x > 0 ? 1.f : 0.f;
    case 1: return y * (1.f - y);
    case 2: return 1.f - y * y;
    case 3: return 1.f / (1.f + std::exp(-x));
    case 4: { const float d = 1.f + std::fabs(x); return 1.f / (d * d); }
    default: return 1.f;
  }
}
inline int ActKind(const std::string& t, const std::string& who) {
  static const char* names[] = {"relu", "sigmoid", "tanh", "softrelu", "softsign"};
  for (int i = 0; i < 5; ++i) if (t == names[i]) return i;
  throw std::runtime_error(who + ": activation " + t + " is not supported");
}

// index helper for broadcasting: maps a flat index of `out` to the flat index of an operand with (possibly) size-1 axes
struct Bcast {
  std::vector<int64_t> out_dims, stride;
  Bcast(const Shape& out, const Shape& in) {
    out_dims = out; stride.assign(out.size(), 0);
    int64_t st = 1;
    for (int i = static_cast<int>(in.size()) - 1, o = static_cast<int>(out.size()) - 1; o >= 0; --i, --o) {
      const int64_t d = i >= 0 ? in[i] : 1;
      stride[o] = d == 1 ? 0 : st;
      st *= d;
    }
  }
  int64_t At(int64_t flat) const {
    int64_t off = 0;
    for (int o = static_cast<int>(out_dims.size()) - 1; o >= 0; --o) { off += (flat % out_dims[o]) * stride[o]; flat /= out_dims[o]; }
    return off;
  }
};

// ------------------------------------------------------------------------------------------------ executor
struct Tensor {                         // a bound array: external float storage + shape
  float* data = nullptr;
  Shape shape;
};

class Executor {
 public:
  // args / grads / aux in ListArguments / ListAuxiliaryStates order; grads[i].data may be null when reqs[i] == kNullOp
  Executor(const Symbol& sym, const std::vector<Tensor>& args, const std::vector<Tensor>& grads, const std::vector<int>& reqs, const std::vector<Tensor>& aux)
      : sym_(sym) {
    order_ = graph::Topo(sym_);
    const auto aux_nodes = graph::AuxNodes(order_);
    std::map<std::string, Shape> known;
    size_t ai = 0, xi = 0;
    for (Node* n : order_) {
      index_[n] = static_cast<int>(slots_.size());
      slots_.emplace_back();
      slots_.back().node = n;
      if (n->op != "null") {
        // outputs 1.. of a multi-output node live in sibling slots right behind the node's own slot: consumers address (node, j) as slot + j
        for (int j = 1, k = graph::NumOutputs(*n); j < k; ++j) { slots_.emplace_back(); slots_.back().node = n; slots_.back().sibling_of = index_[n]; }
        continue;
      }
      Slot& s = slots_.back();
      if (aux_nodes.count(n)) {
        if (xi >= aux.size()) throw std::runtime_error("Bind: " + std::to_string(aux.size()) + " auxiliary states given, the symbol has more (missing " + n->name + ")");
        s.ext = aux[xi].data; s.shape = aux[xi].shape; s.is_aux = true; ++xi;
      } else {
        if (ai >= args.size()) throw std::runtime_error("Bind: " + std::to_string(args.size()) + " arguments given, the symbol has more (missing " + n->name + ")");
        s.ext = args[ai].data; s.shape = args[ai].shape;
        s.req = ai < reqs.size() ? reqs[ai] : kNullOp;
        if (s.req != kNullOp) {
          if (ai >= grads.size() || grads[ai].data == nullptr) throw std::runtime_error("Bind: argument " + n->name + " has grad_req != null but no gradient array");
          if (grads[ai].shape != s.shape) throw std::runtime_error("Bind: gradient of " + n->name + " has shape " + ShapeStr(grads[ai].shape) + ", the argument " + ShapeStr(s.shape));
          s.ext_grad = grads[ai].data;
        }
        arg_slots_.push_back(index_[n]);
        ++ai;
      }
      if (s.ext == nullptr) throw std::runtime_error("Bind: null array for " + n->name);
      known[n->name] = s.shape;
    }
    if (ai != args.size()) throw std::runtime_error("Bind: " + std::to_string(args.size()) + " arguments given, the symbol takes " + std::to_string(ai));
    if (xi != aux.size()) throw std::runtime_error("Bind: " + std::to_string(aux.size()) + " auxiliary states given, the symbol takes " + std::to_string(xi));
    const graph::ShapeResult sr = graph::InferShapes(sym_, known, false);
    for (auto& s : slots_) {
      s.shape = sr.shape.at(s.node);
      if (s.node->op != "null") { s.own.assign(static_cast<size_t>(Numel(s.shape)), 0.f); }
      if (s.sibling_of < 0) for (auto& e : s.node->inputs) s.in.push_back(index_.at(e.node.get()) + e.index);
    }
    // gradient flow: a node needs a gradient when any input does; BlockGrad cuts it
    for (auto& s : slots_) {
      if (s.node->op == "null") { s.need_grad = s.req != kNullOp; continue; }
      if (s.node->op == "BlockGrad") continue;
      if (s.sibling_of >= 0) { s.need_grad = slots_[s.sibling_of].need_grad; continue; }
      for (int i : s.in) if (slots_[i].need_grad) s.need_grad = true;
    }
    for (auto& h : sym_.outputs) heads_.push_back(index_.at(h.node.get()) + h.index);
    rng_.seed(GlobalSeed().fetch_add(1) * 2654435761u + 12345u);
  }

  static std::atomic<uint32_t>& GlobalSeed() { static std::atomic<uint32_t> s{0}; return s; }

  size_t NumOutputs() const { return heads_.size(); }
  const Shape& OutputShape(size_t i) const { return slots_[heads_.at(i)].shape; }
  const float* OutputData(size_t i) const { const Slot& s = slots_[heads_.at(i)]; return s.node->op == "null" ? s.ext : s.own.data(); }

  void Forward(bool is_train) {
    is_train_ = is_train;
    for (auto& s : slots_) if (s.node->op != "null" && s.sibling_of < 0) Run(s);
    forwarded_ = true;
  }

  // head_grads[i] may be null: loss heads (SoftmaxOutput, *RegressionOutput, MakeLoss) ignore it, other heads get ones (MXExecutorBackward with
  // no head gradient on a non-loss head is an error in the reference; autograd's default of ones is the useful convention for a C front end)
  void Backward(const std::vector<const float*>& head_grads) {
    if (!forwarded_) throw std::runtime_error("Backward: call Forward(is_train=1) first");
    if (!head_grads.empty() && head_grads.size() != heads_.size()) throw std::runtime_error("Backward: " + std::to_string(head_grads.size()) + " head gradients for " + std::to_string(heads_.size()) + " outputs");
    for (auto& s : slots_) if (s.need_grad) s.grad.assign(static_cast<size_t>(Numel(s.shape)), 0.f); else s.grad.clear();
    for (size_t i = 0; i < heads_.size(); ++i) {
      Slot& s = slots_[heads_[i]];
      if (!s.need_grad) continue;
      const float* g = head_grads.empty() ? nullptr : head_grads[i];
      if (g) for (size_t k = 0; k < s.grad.size(); ++k) s.grad[k] += g[k];
      else for (auto& v : s.grad) v += 1.f;
    }
    for (size_t k = slots_.size(); k-- > 0;) {
      Slot& s = slots_[k];
      if (s.node->op == "null" || !s.need_grad || s.sibling_of >= 0) continue;       // a sibling's gradient is consumed by its node's own slot, visited later in this sweep
      Grad(s);
      std::vector<float>().swap(s.grad);                   // activations' gradients are dead once propagated
    }
    for (int i : arg_slots_) {
      Slot& s = slots_[i];
      if (s.req == kNullOp) continue;
      if (s.req == kAddTo) for (size_t k = 0; k < s.grad.size(); ++k) s.ext_grad[k] += s.grad[k];
      else memcpy(s.ext_grad, s.grad.data(), s.grad.size() * sizeof(float));
    }
  }

  std::string Print() const {
    std::string o;
    int64_t act = 0;
    for (auto& s : slots_) {
      if (s.sibling_of >= 0) continue;
      if (s.node->op == "null") { o += "Variable:" + s.node->name + " " + ShapeStr(s.shape) + (s.is_aux ? " aux" : s.req != kNullOp ? " grad" : "") + "\n"; continue; }
      o += "Op:" + s.node->op + ", Name=" + s.node->name + " -> " + ShapeStr(s.shape) + "\n";
      for (int i : s.in) o += "  arg: " + slots_[i].node->name + "\n";
      act += Numel(s.shape);
    }
    o += "Total " + std::to_string(act * 4 / 1024) + " KB allocated for activations\n";
    return o;
  }

 private:
  struct Slot {
    Node* node = nullptr;
    Shape shape;
    std::vector<int> in;
    float* ext = nullptr;              // variables: the bound array
    float* ext_grad = nullptr;
    int req = kNullOp;
    bool is_aux = false, need_grad = false;
    int sibling_of = -1;               // >= 0: this slot is output (index - sibling_of) of the multi-output node in slot sibling_of
    std::vector<float> own, grad;
    std::vector<int32_t> idx;          // Pooling(max): winning input offset per output
    std::vector<float> saved;          // Dropout mask / BatchNorm batch mean + inverse std / LayerNorm statistics / LRN scale / softmax probabilities
    std::vector<int64_t> map;          // gather-style operators: source element of every output element (-1 = constant fill)
  };
  Symbol sym_;
  std::vector<Node*> order_;
  std::unordered_map<Node*, int> index_;
  std::vector<Slot> slots_;
  std::vector<int> arg_slots_, heads_;
  bool is_train_ = false, forwarded_ = false;
  std::mt19937 rng_;

  const float* Val(int i) const { const Slot& s = slots_[i]; return s.node->op == "null" ? s.ext : s.own.data(); }
  float* AuxPtr(int i) { return slots_[i].ext; }
  static Win WinOf(const graph::detail::Win& w) { return Win{w.kh, w.kw, w.sh, w.sw, w.ph, w.pw, w.dh, w.dw}; }

  // softmax over the middle axis of (outer, c, inner)
  static void SoftmaxFwd(const float* x, float* y, int64_t outer, int64_t c, int64_t inner, bool log) {
    ParallelFor(outer * inner, static_cast<double>(outer) * inner * c * 8, [&](int64_t lo, int64_t hi) {
      for (int64_t t = lo; t < hi; ++t) {
        const int64_t o = t / inner, i = t % inner;
        const float* xs = x + o * c * inner + i; float* ys = y + o * c * inner + i;
        float m = xs[0];
        for (int64_t k = 1; k < c; ++k) m = std::max(m, xs[k * inner]);
        float z = 0;
        for (int64_t k = 0; k < c; ++k) z += std::exp(xs[k * inner] - m);
        const float lz = std::log(z);
        for (int64_t k = 0; k < c; ++k) ys[k * inner] = log ? xs[k * inner] - m - lz : std::exp(xs[k * inner] - m) / z;
      }
    });
  }
  static void SplitAxis(const Shape& s, int64_t ax, int64_t* outer, int64_t* c, int64_t* inner) {
    *outer = 1; *inner = 1; *c = s[ax];
    for (int64_t i = 0; i < ax; ++i) *outer *= s[i];
    for (size_t i = ax + 1; i < s.size(); ++i) *inner *= s[i];
  }

  // ---- forward
  void Run(Slot& s) {
    const Node& n = *s.node;
    const std::string& op = n.op;
    AttrView a(n.attrs);
    float* y = s.own.data();
    const int64_t ny = Numel(s.shape);
    const float* x = Val(s.in[0]);
    const Shape& xs = slots_[s.in[0]].shape;
    const int64_t nx = Numel(xs);
    if (op == "FullyConnected") {
      const int64_t h = s.shape.back(), k = slots_[s.in[1]].shape[1], m = nx / k;
      const float* b = s.in.size() > 2 ? Val(s.in[2]) : nullptr;
      predict::GemmNT(x, Val(s.in[1]), y, m, h, k, b);
    } else if (op == "Convolution") {
      const Win w = WinOf(graph::detail::Window(n, false, xs));
      const int64_t N = xs[0], C = xs[1], H = xs[2], W = xs[3], F = s.shape[1], OH = s.shape[2], OW = s.shape[3], G = a.Int("num_group", 1);
      const int64_t Cg = C / G, Fg = F / G, K = Cg * w.kh * w.kw, P = OH * OW;
      const float* wt = Val(s.in[1]); const float* b = s.in.size() > 2 ? Val(s.in[2]) : nullptr;
      ParallelFor(N, static_cast<double>(N) * F * K * P, [&](int64_t lo, int64_t hi) {
        std::vector<float> col(static_cast<size_t>(K * P));
        for (int64_t i = lo; i < hi; ++i) for (int64_t g = 0; g < G; ++g) {
          Im2Col(x + (i * C + g * Cg) * H * W, Cg, H, W, w, OH, OW, col.data());
          float* out = y + (i * F + g * Fg) * P;
          GemmSerial(false, false, Fg, P, K, wt + g * Fg * K, col.data(), out, false);
          if (b) for (int64_t f = 0; f < Fg; ++f) { const float bv = b[g * Fg + f]; float* o = out + f * P; for (int64_t p = 0; p < P; ++p) o[p] += bv; }
        }
      });
    } else if (op == "Pooling") {
      const Win w = WinOf(graph::detail::Window(n, true, xs));
      const std::string t = a.Str("pool_type", "max");
      const int type = t == "max" ? 0 : t == "avg" ? 1 : t == "sum" ? 2 : -1;
      if (type < 0) throw std::runtime_error(n.name + ": pool_type " + t + " is not supported");
      const bool count_pad = a.Bool("count_include_pad", true);
      const int64_t NC = xs[0] * xs[1], H = xs[2], W = xs[3], OH = s.shape[2], OW = s.shape[3];
      if (type == 0) s.idx.assign(static_cast<size_t>(ny), -1);
      ParallelFor(NC, static_cast<double>(ny) * w.kh * w.kw * 4, [&](int64_t lo, int64_t hi) {
        for (int64_t c = lo; c < hi; ++c) for (int64_t oy = 0; oy < OH; ++oy) for (int64_t ox = 0; ox < OW; ++ox) {
          const int64_t y0 = oy * w.sh - w.ph, x0 = ox * w.sw - w.pw;
          const int64_t ya = std::max<int64_t>(y0, 0), yb = std::min(y0 + w.kh, H), xa = std::max<int64_t>(x0, 0), xb = std::min(x0 + w.kw, W);
          const float* src = x + c * H * W;
          const int64_t o = (c * OH + oy) * OW + ox;
          if (type == 0) {
            float best = -std::numeric_limits<float>::infinity(); int32_t bi = -1;
            for (int64_t iy = ya; iy < yb; ++iy) for (int64_t ix = xa; ix < xb; ++ix) if (src[iy * W + ix] > best) { best = src[iy * W + ix]; bi = static_cast<int32_t>(iy * W + ix); }
            y[o] = bi < 0 ? 0.f : best; s.idx[o] = bi;
          } else {
            float acc = 0;
            for (int64_t iy = ya; iy < yb; ++iy) for (int64_t ix = xa; ix < xb; ++ix) acc += src[iy * W + ix];
            if (type == 1) {
              const int64_t full = (std::min(y0 + w.kh, H + w.ph) - y0) * (std::min(x0 + w.kw, W + w.pw) - x0);
              acc /= static_cast<float>(count_pad ? full : std::max<int64_t>((yb - ya) * (xb - xa), 1));
            }
            y[o] = acc;
          }
        }
      });
    } else if (op == "Activation") {
      const int k = ActKind(a.Str("act_type", "relu"), n.name);
      for (int64_t i = 0; i < ny; ++i) y[i] = ActF(k, x[i]);
    } else if (op == "LeakyReLU") {
      const std::string t = a.Str("act_type", "leaky");
      const float slope = static_cast<float>(a.Float("slope", 0.25));
      if (t == "leaky") for (int64_t i = 0; i < ny; ++i) y[i] = x[i] > 0 ? x[i] : slope * x[i];
      else if (t == "elu") for (int64_t i = 0; i < ny; ++i) y[i] = x[i] > 0 ? x[i] : slope * (std::exp(x[i]) - 1.f);
      else throw std::runtime_error(n.name + ": LeakyReLU act_type " + t + " is not supported");
    } else if (op == "BatchNorm") {
      const int64_t ax = graph::detail::AxisOf(a.Int("axis", 1), xs.size(), n.name);
      int64_t outer, C, inner; SplitAxis(xs, ax, &outer, &C, &inner);
      const float eps = static_cast<float>(a.Float("eps", 1e-3)), mom = static_cast<float>(a.Float("momentum", 0.9));
      const bool fix_gamma = a.Bool("fix_gamma", true), global = a.Bool("use_global_stats", false) || !is_train_;
      const float* gamma = Val(s.in[1]); const float* beta = Val(s.in[2]);
      float* mm = AuxPtr(s.in[3]); float* mv = AuxPtr(s.in[4]);
      s.saved.assign(static_cast<size_t>(2 * C), 0.f);
      const int64_t cnt = outer * inner;
      ParallelFor(C, static_cast<double>(nx) * 6, [&](int64_t lo, int64_t hi) {
        for (int64_t c = lo; c < hi; ++c) {
          float mean, var;
          if (global) { mean = mm[c]; var = mv[c]; }
          else {
            double sm = 0, sq = 0;
            for (int64_t o = 0; o < outer; ++o) { const float* p = x + (o * C + c) * inner; for (int64_t i = 0; i < inner; ++i) sm += p[i]; }
            mean = static_cast<float>(sm / cnt);
            for (int64_t o = 0; o < outer; ++o) { const float* p = x + (o * C + c) * inner; for (int64_t i = 0; i < inner; ++i) { const double d = p[i] - mean; sq += d * d; } }
            var = static_cast<float>(sq / cnt);
            mm[c] = mm[c] * mom + mean * (1.f - mom);
            mv[c] = mv[c] * mom + var * (1.f - mom);
          }
          const float inv = 1.f / std::sqrt(var + eps), g = fix_gamma ? 1.f : gamma[c];
          s.saved[c] = mean; s.saved[C + c] = inv;
          for (int64_t o = 0; o < outer; ++o) {
            const float* p = x + (o * C + c) * inner; float* q = y + (o * C + c) * inner;
            for (int64_t i = 0; i < inner; ++i) q[i] = (p[i] - mean) * inv * g + beta[c];
          }
        }
      });
    } else if (op == "Dropout") {
      const float p = static_cast<float>(a.Float("p", 0.5));
      if (!is_train_ || p <= 0.f) { s.saved.clear(); memcpy(y, x, ny * sizeof(float)); }
      else {
        if (p >= 1.f) throw std::runtime_error(n.name + ": drop probability must be < 1");
        s.saved.resize(static_cast<size_t>(ny));
        std::bernoulli_distribution keep(1.0 - p);
        const float scale = 1.f / (1.f - p);
        for (int64_t i = 0; i < ny; ++i) { s.saved[i] = keep(rng_) ? scale : 0.f; y[i] = x[i] * s.saved[i]; }
      }
    } else if (op == "Flatten" || op == "Reshape" || op == "expand_dims" || op == "identity" || op == "BlockGrad" || op == "MakeLoss" ||
               op == "LinearRegressionOutput" || op == "MAERegressionOutput") {
      memcpy(y, x, ny * sizeof(float));
    } else if (op == "LogisticRegressionOutput") {
      for (int64_t i = 0; i < ny; ++i) y[i] = ActF(1, x[i]);
    } else if (op == "transpose") {
      auto axes = a.Tuple("axes", {});
      const size_t r = xs.size();
      if (axes.empty()) for (size_t i = 0; i < r; ++i) axes.push_back(static_cast<int64_t>(r - 1 - i));
      std::vector<int64_t> xstride(r, 1);
      for (int i = static_cast<int>(r) - 2; i >= 0; --i) xstride[i] = xstride[i + 1] * xs[i + 1];
      for (int64_t f = 0; f < ny; ++f) {
        int64_t rem = f, off = 0;
        for (int i = static_cast<int>(r) - 1; i >= 0; --i) { off += (rem % s.shape[i]) * xstride[graph::detail::AxisOf(axes[i], r, n.name)]; rem /= s.shape[i]; }
        y[f] = x[off];
      }
    } else if (op == "Concat") {
      const int64_t ax = graph::detail::AxisOf(a.Int("dim", 1), s.shape.size(), n.name);
      int64_t outer, C, inner; SplitAxis(s.shape, ax, &outer, &C, &inner);
      int64_t at = 0;
      for (int i : s.in) {
        const int64_t ci = slots_[i].shape[ax]; const float* src = Val(i);
        for (int64_t o = 0; o < outer; ++o) memcpy(y + (o * C + at) * inner, src + o * ci * inner, ci * inner * sizeof(float));
        at += ci;
      }
    } else if (op == "add_n") {
      memcpy(y, x, ny * sizeof(float));
      for (size_t k = 1; k < s.in.size(); ++k) { const float* v = Val(s.in[k]); for (int64_t i = 0; i < ny; ++i) y[i] += v[i]; }
    } else if (op == "sgd_update" || op == "sgd_mom_update" || op == "adam_update") {
      // ndarray/op_lib.py: g = clip(rescale * grad) + wd * w; the states (trailing auxiliary inputs) are updated in place
      const float lr = static_cast<float>(a.Float("lr", 0)), wd = static_cast<float>(a.Float("wd", 0)), rescale = static_cast<float>(a.Float("rescale_grad", 1)),
                  clip = static_cast<float>(a.Float("clip_gradient", -1));
      const float* g = Val(s.in[1]);
      auto prep = [&](int64_t i) { float v = g[i] * rescale; if (clip >= 0.f) v = std::min(std::max(v, -clip), clip); return v + wd * x[i]; };
      if (op == "sgd_update") for (int64_t i = 0; i < ny; ++i) y[i] = x[i] - lr * prep(i);
      else if (op == "sgd_mom_update") {
        const float mom = static_cast<float>(a.Float("momentum", 0));
        float* m = AuxPtr(s.in[2]);
        for (int64_t i = 0; i < ny; ++i) { m[i] = m[i] * mom - lr * prep(i); y[i] = x[i] + m[i]; }
      } else {
        const float b1 = static_cast<float>(a.Float("beta1", 0.9)), b2 = static_cast<float>(a.Float("beta2", 0.999)), eps = static_cast<float>(a.Float("epsilon", 1e-8));
        float* m = AuxPtr(s.in[2]); float* v = AuxPtr(s.in[3]);
        for (int64_t i = 0; i < ny; ++i) {
          const float gg = prep(i);
          m[i] = m[i] * b1 + gg * (1.f - b1); v[i] = v[i] * b2 + gg * gg * (1.f - b2);
          y[i] = x[i] - lr * m[i] / (std::sqrt(v[i]) + eps);
        }
      }
    } else if (op == "Embedding") {
      const float* w = Val(s.in[1]);
      const int64_t V = slots_[s.in[1]].shape[0], D = slots_[s.in[1]].shape[1];
      for (int64_t i = 0; i < nx; ++i) {
        const int64_t r = std::min<int64_t>(std::max<int64_t>(static_cast<int64_t>(x[i]), 0), V - 1);
        memcpy(y + i * D, w + r * D, D * sizeof(float));
      }
    } else if (op == "SoftmaxOutput" || op == "SoftmaxActivation") {
      int64_t outer, C, inner; SplitAxis(xs, 1, &outer, &C, &inner);
      if (op == "SoftmaxOutput" && !a.Bool("multi_output", false) && xs.size() > 2) { C = nx / xs[0]; inner = 1; outer = xs[0]; }
      SoftmaxFwd(x, y, outer, C, inner, false);
    } else if (op == "softmax" || op == "log_softmax") {
      int64_t outer, C, inner; SplitAxis(xs, graph::detail::AxisOf(a.Int("axis", -1), xs.size(), n.name), &outer, &C, &inner);
      SoftmaxFwd(x, y, outer, C, inner, op == "log_softmax");
    } else if (op == "clip") {
      const float lo = static_cast<float>(a.Float("a_min", -std::numeric_limits<float>::infinity())), hi = static_cast<float>(a.Float("a_max", std::numeric_limits<float>::infinity()));
      for (int64_t i = 0; i < ny; ++i) y[i] = std::min(std::max(x[i], lo), hi);
    } else if (op == "SliceChannel") {
      const int64_t k = graph::NumOutputs(n);
      int64_t outer, C, inner; SplitAxis(xs, graph::detail::AxisOf(a.Int("axis", 1), xs.size(), n.name), &outer, &C, &inner);
      const int64_t Ck = C / k, self = &s - slots_.data();
      for (int64_t j = 0; j < k; ++j) {
        float* dst = slots_[self + j].own.data();
        for (int64_t o = 0; o < outer; ++o) memcpy(dst + o * Ck * inner, x + (o * C + j * Ck) * inner, Ck * inner * sizeof(float));
      }
    } else if (IsGather(op)) {
      BuildMap(s);
      const float fill = op == "Pad" ? static_cast<float>(a.Float("constant_value", 0)) : 0.f;
      for (int64_t i = 0; i < ny; ++i) y[i] = s.map[i] < 0 ? fill : x[s.map[i]];
    } else if (op == "squeeze" || op == "Cast") {
      memcpy(y, x, ny * sizeof(float));
    } else if (op == "where") {
      const float* t = Val(s.in[1]); const float* f = Val(s.in[2]);
      for (int64_t i = 0; i < ny; ++i) y[i] = x[i] != 0.f ? t[i] : f[i];
    } else if (op == "one_hot") {
      const int64_t D = s.shape.back();
      const float on = static_cast<float>(a.Float("on_value", 1)), off = static_cast<float>(a.Float("off_value", 0));
      for (int64_t i = 0; i < nx; ++i) for (int64_t k = 0; k < D; ++k) y[i * D + k] = static_cast<int64_t>(x[i]) == k ? on : off;
    } else if (op == "argmax" || op == "argmin") {
      int64_t outer, C, inner; SplitAxis(xs, graph::detail::AxisOf(a.Int("axis", 0), xs.size(), n.name), &outer, &C, &inner);
      const bool mx = op == "argmax";
      for (int64_t o = 0; o < outer; ++o) for (int64_t i = 0; i < inner; ++i) {
        const float* p = x + o * C * inner + i; int64_t best = 0;
        for (int64_t k = 1; k < C; ++k) if (mx ? p[k * inner] > p[best * inner] : p[k * inner] < p[best * inner]) best = k;
        y[o * inner + i] = static_cast<float>(best);
      }
    } else if (op == "max" || op == "min" || op == "prod" || op == "norm") {
      const auto red = ReducedAxes(s, xs);
      const int kind = op == "max" ? 0 : op == "min" ? 1 : op == "prod" ? 2 : 3;
      std::vector<double> acc(static_cast<size_t>(ny), kind == 0 ? -std::numeric_limits<double>::infinity() : kind == 1 ? std::numeric_limits<double>::infinity() : kind == 2 ? 1.0 : 0.0);
      for (int64_t f = 0; f < nx; ++f) {
        double& v = acc[ReducedIndex(f, xs, red)];
        if (kind == 0) v = std::max<double>(v, x[f]); else if (kind == 1) v = std::min<double>(v, x[f]); else if (kind == 2) v *= x[f]; else v += static_cast<double>(x[f]) * x[f];
      }
      for (int64_t i = 0; i < ny; ++i) y[i] = static_cast<float>(kind == 3 ? std::sqrt(acc[i]) : acc[i]);
    } else if (op == "LayerNorm" || op == "InstanceNorm") {
      int64_t outer, C, inner; NormGroups(s, xs, &outer, &C, &inner);
      const bool layer = op == "LayerNorm";
      const float eps = static_cast<float>(a.Float("eps", layer ? 1e-5 : 1e-3));
      const float* gamma = Val(s.in[1]); const float* beta = Val(s.in[2]);
      // LayerNorm: statistics over the middle axis C per (outer, inner), scale indexed by c.  InstanceNorm: statistics over inner per (n, c), scale indexed by c.
      const int64_t groups = layer ? outer * inner : outer * C, len = layer ? C : inner;
      s.saved.assign(static_cast<size_t>(2 * groups), 0.f);
      for (int64_t g = 0; g < groups; ++g) {
        const int64_t base = layer ? (g / inner) * C * inner + g % inner : g * inner, stride = layer ? inner : 1;
        double sm = 0, sq = 0;
        for (int64_t k = 0; k < len; ++k) sm += x[base + k * stride];
        const float mean = static_cast<float>(sm / len);
        for (int64_t k = 0; k < len; ++k) { const double d = x[base + k * stride] - mean; sq += d * d; }
        const float inv = 1.f / std::sqrt(static_cast<float>(sq / len) + eps);
        s.saved[2 * g] = mean; s.saved[2 * g + 1] = inv;
        for (int64_t k = 0; k < len; ++k) { const int64_t c = layer ? k : g % C; y[base + k * stride] = (x[base + k * stride] - mean) * inv * gamma[c] + beta[c]; }
      }
    } else if (op == "L2Normalization") {
      int64_t outer, C, inner; NormGroups(s, xs, &outer, &C, &inner);
      const float eps = static_cast<float>(a.Float("eps", 1e-10));
      s.saved.assign(static_cast<size_t>(outer * inner), 0.f);
      for (int64_t o = 0; o < outer; ++o) for (int64_t i = 0; i < inner; ++i) {
        const float* p = x + o * C * inner + i; float* q = y + o * C * inner + i;
        double sq = 0;
        for (int64_t k = 0; k < C; ++k) sq += static_cast<double>(p[k * inner]) * p[k * inner];
        const float nrm = std::sqrt(static_cast<float>(sq) + eps);
        s.saved[o * inner + i] = nrm;
        for (int64_t k = 0; k < C; ++k) q[k * inner] = p[k * inner] / nrm;
      }
    } else if (op == "LRN") {
      const int64_t N = xs[0], C = xs[1], P = xs[2] * xs[3], half = a.Int("nsize", 1) / 2;
      const float alpha = static_cast<float>(a.Float("alpha", 1e-4)) / static_cast<float>(a.Int("nsize", 1)), beta = static_cast<float>(a.Float("beta", 0.75)), knorm = static_cast<float>(a.Float("knorm", 2));
      s.saved.assign(static_cast<size_t>(nx), 0.f);
      for (int64_t b = 0; b < N; ++b) for (int64_t c = 0; c < C; ++c) for (int64_t p = 0; p < P; ++p) {
        float sq = 0;
        for (int64_t k = std::max<int64_t>(c - half, 0); k <= std::min(c + half, C - 1); ++k) { const float v = x[(b * C + k) * P + p]; sq += v * v; }
        const int64_t at = (b * C + c) * P + p;
        s.saved[at] = knorm + alpha * sq;
        y[at] = x[at] * std::pow(s.saved[at], -beta);
      }
    } else if (op == "Deconvolution") {
      const Win w = WinOf(graph::detail::Window(n, false, xs));
      const int64_t N = xs[0], C = xs[1], H = xs[2], W = xs[3], F = s.shape[1], OH = s.shape[2], OW = s.shape[3], G = a.Int("num_group", 1);
      const int64_t Cg = C / G, Fg = F / G, K = Fg * w.kh * w.kw, P = H * W;
      const float* wt = Val(s.in[1]); const float* b = s.in.size() > 2 ? Val(s.in[2]) : nullptr;
      std::fill(y, y + ny, 0.f);
      ParallelFor(N, static_cast<double>(N) * C * K * P, [&](int64_t lo, int64_t hi) {
        std::vector<float> col(static_cast<size_t>(K * P));
        for (int64_t i = lo; i < hi; ++i) for (int64_t g = 0; g < G; ++g) {
          GemmSerial(true, false, K, P, Cg, wt + g * Cg * K, x + (i * C + g * Cg) * P, col.data(), false);      // col = W_g^T . x_g
          Col2Im(col.data(), Fg, OH, OW, w, H, W, y + (i * F + g * Fg) * OH * OW);
        }
        if (b) for (int64_t i = lo; i < hi; ++i) for (int64_t f = 0; f < F; ++f) { float* o = y + (i * F + f) * OH * OW; for (int64_t p = 0; p < OH * OW; ++p) o[p] += b[f]; }
      });
    } else if (op == "smooth_l1") {
      const float s2 = static_cast<float>(a.Float("scalar", 1)) * static_cast<float>(a.Float("scalar", 1));
      for (int64_t i = 0; i < ny; ++i) { const float v = std::fabs(x[i]); y[i] = v < 1.f / s2 ? 0.5f * s2 * v * v : v - 0.5f / s2; }
    } else if (op == "softmax_cross_entropy") {
      const int64_t N = xs[0], C = xs[1];
      const float* label = Val(s.in[1]);
      s.saved.resize(static_cast<size_t>(nx));
      SoftmaxFwd(x, s.saved.data(), N, C, 1, false);
      double loss = 0;
      for (int64_t i = 0; i < N; ++i) loss -= std::log(std::max(s.saved[i * C + std::min<int64_t>(std::max<int64_t>(static_cast<int64_t>(label[i]), 0), C - 1)], 1e-30f));
      y[0] = static_cast<float>(loss);
    } else if (op == "sum" || op == "mean") {
      ReduceFwd(s, x, xs, y, op == "mean");
    } else if (op == "dot") {
      const bool ta = a.Bool("transpose_a", false), tb = a.Bool("transpose_b", false);
      const int64_t M = s.shape[0], N = s.shape[1], K = ta ? xs[0] : xs[1];
      Gemm(ta, tb, M, N, K, x, Val(s.in[1]), y, false);
    } else if (s.in.size() == 2) {
      const int kind = BinaryKind(op);
      const float* r = Val(s.in[1]);
      const Shape& rs = slots_[s.in[1]].shape;
      if (xs == s.shape && rs == s.shape) for (int64_t i = 0; i < ny; ++i) y[i] = Bin(kind, x[i], r[i]);
      else { const Bcast bl(s.shape, xs), br(s.shape, rs); for (int64_t i = 0; i < ny; ++i) y[i] = Bin(kind, x[bl.At(i)], r[br.At(i)]); }
    } else if (op[0] == '_') {
      const float c = static_cast<float>(a.Float("scalar", 0));
      const int k = ScalarKind(op);
      for (int64_t i = 0; i < ny; ++i) y[i] = Sc(k, x[i], c);
    } else {
      const int k = UnaryKind(op);
      if (k < 0) throw std::runtime_error("operator " + op + " has no host kernel");
      for (int64_t i = 0; i < ny; ++i) y[i] = Un(k, x[i]);
    }
  }

  static int BinaryKind(const std::string& op) {
    static const std::pair<const char*, int> names[] = {
        {"elemwise_add", 0}, {"broadcast_add", 0}, {"elemwise_sub", 1}, {"broadcast_sub", 1}, {"elemwise_mul", 2}, {"broadcast_mul", 2}, {"elemwise_div", 3},
        {"broadcast_div", 3}, {"broadcast_maximum", 4}, {"broadcast_minimum", 5}, {"broadcast_power", 6}, {"broadcast_equal", 7}, {"broadcast_not_equal", 8},
        {"broadcast_greater", 9}, {"broadcast_greater_equal", 10}, {"broadcast_lesser", 11}, {"broadcast_lesser_equal", 12}};
    for (auto& e : names) if (op == e.first) return e.second;
    throw std::runtime_error("operator " + op + " has no host kernel");
  }
  static float Bin(int k, float l, float r) {
    switch (k) {
      case 0: return l + r; case 1: return l - r; case 2: return l * r; case 3: return l / r; case 4: return std::max(l, r); case 5: return std::min(l, r);
      case 6: return std::pow(l, r); case 7: return l == r; case 8: return l != r; case 9: return l > r; case 10: return l >= r; case 11: return l < r; default: return l <= r;
    }
  }
  static int ScalarKind(const std::string& op) {
    static const char* names[] = {"_plus_scalar", "_minus_scalar", "_rminus_scalar", "_mul_scalar", "_div_scalar", "_rdiv_scalar", "_power_scalar", "_maximum_scalar",
                                  "_minimum_scalar", "_rpower_scalar"};
    for (int i = 0; i < 10; ++i) if (op == names[i]) return i;
    throw std::runtime_error("operator " + op + " has no host kernel");
  }
  static float Sc(int k, float x, float c) {
    switch (k) {
      case 0: return x + c; case 1: return x - c; case 2: return c - x; case 3: return x * c; case 4: return x / c; case 5: return c / x; case 6: return std::pow(x, c);
      case 7: return std::max(x, c); case 8: return std::min(x, c); default: return std::pow(c, x);
    }
  }
  static float ScG(int k, float x, float c, float y) {
    switch (k) {
      case 0: case 1: return 1.f; case 2: return -1.f; case 3: return c; case 4: return 1.f / c; case 5: return -c / (x * x); case 6: return c * std::pow(x, c - 1.f);
      case 7: return x >= c ? 1.f : 0.f; case 8: return x <= c ? 1.f : 0.f; default: return y * std::log(c);
    }
  }
  static int UnaryKind(const std::string& op) {
    static const char* names[] = {"relu", "sigmoid", "tanh", "exp", "log", "sqrt", "abs", "negative", "square", "softsign", "sin", "cos", "tan", "arcsin", "arccos", "arctan",
                                  "sinh", "cosh", "log1p", "expm1", "log2", "log10", "rsqrt", "reciprocal", "cbrt", "erf", "floor", "ceil", "round", "sign"};
    for (int i = 0; i < 30; ++i) if (op == names[i]) return i;
    return -1;
  }
  static float Un(int k, float v) {
    switch (k) {
      case 0: return v > 0 ? v : 0; case 1: return 1.f / (1.f + std::exp(-v)); case 2: return std::tanh(v); case 3: return std::exp(v); case 4: return std::log(v);
      case 5: return std::sqrt(v); case 6: return std::fabs(v); case 7: return -v; case 8: return v * v; case 9: return v / (1.f + std::fabs(v));
      case 10: return std::sin(v); case 11: return std::cos(v); case 12: return std::tan(v); case 13: return std::asin(v); case 14: return std::acos(v); case 15: return std::atan(v);
      case 16: return std::sinh(v); case 17: return std::cosh(v); case 18: return std::log1p(v); case 19: return std::expm1(v); case 20: return std::log2(v);
      case 21: return std::log10(v); case 22: return 1.f / std::sqrt(v); case 23: return 1.f / v; case 24: return std::cbrt(v); case 25: return std::erf(v);
      case 26: return std::floor(v); case 27: return std::ceil(v); case 28: return std::round(v); default: return v > 0 ? 1.f : v < 0 ? -1.f : 0.f;
    }
  }
  // d out / d in for unary kinds, from input x and output y
  static float UnG(int k, float x, float y) {
    switch (k) {
      case 0: return x > 0 ? 1.f : 0.f; case 1: return y * (1.f - y); case 2: return 1.f - y * y; case 3: return y; case 4: return 1.f / x;
      case 5: return 0.5f / y; case 6: return x > 0 ? 1.f : x < 0 ? -1.f : 0.f; case 7: return -1.f; case 8: return 2.f * x;
      case 9: { const float d = 1.f + std::fabs(x); return 1.f / (d * d); }
      case 10: return std::cos(x); case 11: return -std::sin(x); case 12: return 1.f + y * y; case 13: return 1.f / std::sqrt(1.f - x * x); case 14: return -1.f / std::sqrt(1.f - x * x);
      case 15: return 1.f / (1.f + x * x); case 16: return std::cosh(x); case 17: return std::sinh(x); case 18: return 1.f / (1.f + x); case 19: return y + 1.f;
      case 20: return 1.f / (x * 0.6931471805599453f); case 21: return 1.f / (x * 2.302585092994046f); case 22: return -0.5f * y / x; case 23: return -y * y;
      case 24: return y / (3.f * x); case 25: return 1.1283791670955126f * std::exp(-x * x);
      default: return 0.f;                // floor / ceil / round / sign
    }
  }

  static bool IsGather(const std::string& op) {
    static const char* names[] = {"slice_axis", "slice", "SwapAxis", "tile", "repeat", "Pad", "reverse", "broadcast_to", "broadcast_axis", "UpSampling", "take", "pick"};
    for (auto nme : names) if (op == nme) return true;
    return false;
  }
  // source element of every output element for the gather-style operators; rebuilt every forward (take / pick depend on index values)
  void BuildMap(Slot& s) {
    const Node& n = *s.node;
    const std::string& op = n.op;
    AttrView a(n.attrs);
    const Shape& xs = slots_[s.in[0]].shape;
    const Shape& os = s.shape;
    const int64_t ny = Numel(os);
    s.map.assign(static_cast<size_t>(ny), 0);
    if (op == "take" || op == "pick") {
      const float* idx = Val(s.in[1]);
      const int64_t ax = graph::detail::AxisOf(a.Int("axis", op == "take" ? 0 : -1), xs.size(), n.name);
      int64_t outer, C, inner; SplitAxis(xs, ax, &outer, &C, &inner);
      if (op == "take") {
        const int64_t ni = Numel(slots_[s.in[1]].shape);
        for (int64_t o = 0; o < outer; ++o) for (int64_t j = 0; j < ni; ++j) {
          const int64_t r = std::min<int64_t>(std::max<int64_t>(static_cast<int64_t>(idx[j]), 0), C - 1);
          for (int64_t i = 0; i < inner; ++i) s.map[(o * ni + j) * inner + i] = (o * C + r) * inner + i;
        }
      } else {
        for (int64_t o = 0; o < outer; ++o) for (int64_t i = 0; i < inner; ++i) {
          const int64_t r = std::min<int64_t>(std::max<int64_t>(static_cast<int64_t>(idx[o * inner + i]), 0), C - 1);
          s.map[o * inner + i] = (o * C + r) * inner + i;
        }
      }
      return;
    }
    // per-axis affine / modular index rules: the input may have a lower rank than the output (tile)
    const size_t r = os.size();
    Shape in = xs; while (in.size() < r) in.insert(in.begin(), 1);
    std::vector<int64_t> stride(r, 1);
    for (int i = static_cast<int>(r) - 2; i >= 0; --i) stride[i] = stride[i + 1] * in[i + 1];
    std::vector<int64_t> off(r, 0), div(r, 1), perm(r);
    std::vector<char> wrap(r, 0), flip(r, 0), bcast(r, 0);
    for (size_t i = 0; i < r; ++i) perm[i] = static_cast<int64_t>(i);
    std::vector<int64_t> before(r, 0);
    int pad_mode = -1;
    if (op == "slice_axis") {
      const int64_t ax = graph::detail::AxisOf(a.Int("axis", 0), r, n.name);
      int64_t lo, hi; graph::detail::SliceRange(a.Has("begin"), a.Int("begin", 0), a.Has("end"), a.Int("end", 0), in[ax], n.name, &lo, &hi);
      off[ax] = lo;
    } else if (op == "slice") {
      const auto b = graph::detail::TupleOpt(a, "begin"), e = graph::detail::TupleOpt(a, "end");
      for (size_t i = 0; i < b.size(); ++i) { int64_t lo, hi; graph::detail::SliceRange(b[i].first, b[i].second, e[i].first, e[i].second, in[i], n.name, &lo, &hi); off[i] = lo; }
    } else if (op == "SwapAxis") {
      std::swap(perm[graph::detail::AxisOf(a.Int("dim1", 0), r, n.name)], perm[graph::detail::AxisOf(a.Int("dim2", 0), r, n.name)]);
    } else if (op == "tile") {
      for (size_t i = 0; i < r; ++i) wrap[i] = 1;
    } else if (op == "repeat") {
      div[graph::detail::AxisOf(a.Int("axis", 0), r, n.name)] = a.Int("repeats", 1);
    } else if (op == "UpSampling") {
      div[2] = div[3] = a.Int("scale", 1);
    } else if (op == "reverse") {
      for (auto ax : a.Tuple("axis", {})) flip[graph::detail::AxisOf(ax, r, n.name)] = 1;
    } else if (op == "broadcast_to" || op == "broadcast_axis") {
      for (size_t i = 0; i < r; ++i) bcast[i] = in[i] == 1 && os[i] != 1;
    } else if (op == "Pad") {
      const auto pw = a.Tuple("pad_width", {});
      for (size_t i = 0; i < r; ++i) before[i] = pw[2 * i];
      const std::string mode = a.Str("mode", "constant");
      pad_mode = mode == "constant" ? 0 : mode == "edge" ? 1 : 2;
    }
    std::vector<int64_t> idx(r);
    for (int64_t f = 0; f < ny; ++f) {
      int64_t rem = f;
      for (int i = static_cast<int>(r) - 1; i >= 0; --i) { idx[i] = rem % os[i]; rem /= os[i]; }
      int64_t src = 0; bool constant = false;
      for (size_t i = 0; i < r; ++i) {
        int64_t v = idx[i];
        const size_t d = static_cast<size_t>(perm[i]);           // SwapAxis: output axis i reads input axis perm[i]
        if (pad_mode >= 0) {
          v -= before[i];
          if (v < 0 || v >= in[i]) {
            if (pad_mode == 0) { constant = true; break; }
            v = pad_mode == 1 ? std::min(std::max<int64_t>(v, 0), in[i] - 1) : (v < 0 ? -v : 2 * (in[i] - 1) - v);
          }
        }
        v = v / div[i] + off[i];
        if (wrap[i]) v %= in[i];
        if (flip[i]) v = in[i] - 1 - v;
        if (bcast[i]) v = 0;
        src += v * stride[d];
      }
      s.map[f] = constant ? -1 : src;
    }
  }
  // (outer, C, inner) view for the normalisation operators
  void NormGroups(const Slot& s, const Shape& xs, int64_t* outer, int64_t* C, int64_t* inner) const {
    const Node& n = *s.node;
    AttrView a(n.attrs);
    if (n.op == "LayerNorm") { SplitAxis(xs, graph::detail::AxisOf(a.Int("axis", -1), xs.size(), n.name), outer, C, inner); return; }
    if (n.op == "InstanceNorm") { *outer = xs[0]; *C = xs[1]; *inner = Numel(xs) / (xs[0] * xs[1]); return; }
    const std::string mode = a.Str("mode", "instance");
    const int64_t total = Numel(xs);
    if (mode == "instance") { *outer = xs[0]; *C = total / xs[0]; *inner = 1; }
    else if (mode == "channel") { if (xs.size() < 2) throw std::runtime_error(n.name + ": channel mode needs at least 2 axes"); *outer = xs[0]; *C = xs[1]; *inner = total / (xs[0] * xs[1]); }
    else if (mode == "spatial") { if (xs.size() < 3) throw std::runtime_error(n.name + ": spatial mode needs at least 3 axes"); *outer = xs[0] * xs[1]; *C = total / (xs[0] * xs[1]); *inner = 1; }
    else throw std::runtime_error(n.name + ": L2Normalization mode " + mode + " is not supported");
  }

  std::vector<char> ReducedAxes(const Slot& s, const Shape& xs) const {
    auto axes = AttrView(s.node->attrs).Tuple("axis", {});
    std::vector<char> red(xs.size(), axes.empty());
    for (auto ax : axes) red[graph::detail::AxisOf(ax, xs.size(), s.node->name)] = 1;
    return red;
  }
  // flat index of the reduced output that input element `f` contributes to
  static int64_t ReducedIndex(int64_t f, const Shape& xs, const std::vector<char>& red) {
    int64_t off = 0, st = 1;
    for (int i = static_cast<int>(xs.size()) - 1; i >= 0; --i) { const int64_t c = f % xs[i]; f /= xs[i]; if (!red[i]) { off += c * st; st *= xs[i]; } }
    return off;
  }
  void ReduceFwd(Slot& s, const float* x, const Shape& xs, float* y, bool mean) const {
    const auto red = ReducedAxes(s, xs);
    const int64_t nx = Numel(xs), ny = Numel(s.shape);
    std::vector<double> acc(static_cast<size_t>(ny), 0.0);
    for (int64_t f = 0; f < nx; ++f) acc[ReducedIndex(f, xs, red)] += x[f];
    const double div = mean ? static_cast<double>(nx / ny) : 1.0;
    for (int64_t i = 0; i < ny; ++i) y[i] = static_cast<float>(acc[i] / div);
  }

  // ---- backward: s.grad holds d loss / d output; adds into the inputs' grad buffers (only where need_grad)
  float* GradOf(int i) { Slot& s = slots_[i]; return s.need_grad ? s.grad.data() : nullptr; }

  void Grad(Slot& s) {
    const Node& n = *s.node;
    const std::string& op = n.op;
    AttrView a(n.attrs);
    const float* dy = s.grad.data();
    const float* y = s.own.data();
    const int64_t ny = Numel(s.shape);
    const float* x = Val(s.in[0]);
    const Shape& xs = slots_[s.in[0]].shape;
    const int64_t nx = Numel(xs);
    float* dx = GradOf(s.in[0]);
    if (op == "FullyConnected") {
      const int64_t h = s.shape.back(), k = slots_[s.in[1]].shape[1], m = nx / k;
      if (dx) Gemm(false, false, m, k, h, dy, Val(s.in[1]), dx, true);                              // dX += dY . W
      if (float* dw = GradOf(s.in[1])) Gemm(true, false, h, k, m, dy, x, dw, true);                  // dW += dY^T . X
      if (s.in.size() > 2) if (float* db = GradOf(s.in[2])) for (int64_t i = 0; i < m; ++i) for (int64_t j = 0; j < h; ++j) db[j] += dy[i * h + j];
    } else if (op == "Convolution") {
      const Win w = WinOf(graph::detail::Window(n, false, xs));
      const int64_t N = xs[0], C = xs[1], H = xs[2], W = xs[3], F = s.shape[1], OH = s.shape[2], OW = s.shape[3], G = a.Int("num_group", 1);
      const int64_t Cg = C / G, Fg = F / G, K = Cg * w.kh * w.kw, P = OH * OW;
      const float* wt = Val(s.in[1]);
      float* dw = GradOf(s.in[1]);
      float* db = s.in.size() > 2 ? GradOf(s.in[2]) : nullptr;
      std::mutex mu;
      std::map<int64_t, std::pair<std::vector<float>, std::vector<float>>> parts;      // per chunk of images, keyed by its first image: summed in key order below
      ParallelFor(N, static_cast<double>(N) * F * K * P * 2, [&](int64_t lo, int64_t hi) {
        std::vector<float> col(static_cast<size_t>(K * P)), dcol(dx ? static_cast<size_t>(K * P) : 0);
        std::vector<float> dw_local(dw ? static_cast<size_t>(F * K) : 0, 0.f), db_local(db ? static_cast<size_t>(F) : 0, 0.f);
        for (int64_t i = lo; i < hi; ++i) for (int64_t g = 0; g < G; ++g) {
          const float* dout = dy + (i * F + g * Fg) * P;
          if (dw) {
            Im2Col(x + (i * C + g * Cg) * H * W, Cg, H, W, w, OH, OW, col.data());
            GemmSerial(false, true, Fg, K, P, dout, col.data(), dw_local.data() + g * Fg * K, true);    // dW += dOut . col^T
          }
          if (db) for (int64_t f = 0; f < Fg; ++f) { float sm = 0; for (int64_t p = 0; p < P; ++p) sm += dout[f * P + p]; db_local[g * Fg + f] += sm; }
          if (dx) {
            GemmSerial(true, false, K, P, Fg, wt + g * Fg * K, dout, dcol.data(), false);               // dcol = W^T . dOut
            Col2Im(dcol.data(), Cg, H, W, w, OH, OW, dx + (i * C + g * Cg) * H * W);
          }
        }
        std::lock_guard<std::mutex> lk(mu);
        parts[lo] = {std::move(dw_local), std::move(db_local)};
      });
      // a fixed summation order: the weight gradient does not depend on which thread finished first (bitwise reproducible runs)
      for (auto& kv : parts) {
        if (dw) for (size_t k = 0; k < kv.second.first.size(); ++k) dw[k] += kv.second.first[k];
        if (db) for (size_t k = 0; k < kv.second.second.size(); ++k) db[k] += kv.second.second[k];
      }
    } else if (op == "Pooling") {
      if (!dx) return;
      const Win w = WinOf(graph::detail::Window(n, true, xs));
      const std::string t = a.Str("pool_type", "max");
      const bool count_pad = a.Bool("count_include_pad", true);
      const int64_t NC = xs[0] * xs[1], H = xs[2], W = xs[3], OH = s.shape[2], OW = s.shape[3];
      for (int64_t c = 0; c < NC; ++c) for (int64_t oy = 0; oy < OH; ++oy) for (int64_t ox = 0; ox < OW; ++ox) {
        const int64_t o = (c * OH + oy) * OW + ox;
        float* dst = dx + c * H * W;
        if (t == "max") { if (s.idx[o] >= 0) dst[s.idx[o]] += dy[o]; continue; }
        const int64_t y0 = oy * w.sh - w.ph, x0 = ox * w.sw - w.pw;
        const int64_t ya = std::max<int64_t>(y0, 0), yb = std::min(y0 + w.kh, H), xa = std::max<int64_t>(x0, 0), xb = std::min(x0 + w.kw, W);
        float g = dy[o];
        if (t == "avg") {
          const int64_t full = (std::min(y0 + w.kh, H + w.ph) - y0) * (std::min(x0 + w.kw, W + w.pw) - x0);
          g /= static_cast<float>(count_pad ? full : std::max<int64_t>((yb - ya) * (xb - xa), 1));
        }
        for (int64_t iy = ya; iy < yb; ++iy) for (int64_t ix = xa; ix < xb; ++ix) dst[iy * W + ix] += g;
      }
    } else if (op == "Activation") {
      if (!dx) return;
      const int k = ActKind(a.Str("act_type", "relu"), n.name);
      for (int64_t i = 0; i < ny; ++i) dx[i] += dy[i] * ActG(k, x[i], y[i]);
    } else if (op == "LeakyReLU") {
      if (!dx) return;
      const float slope = static_cast<float>(a.Float("slope", 0.25));
      const bool elu = a.Str("act_type", "leaky") == "elu";
      for (int64_t i = 0; i < ny; ++i) dx[i] += dy[i] * (x[i] > 0 ? 1.f : elu ? y[i] + slope : slope);
    } else if (op == "BatchNorm") {
      const int64_t ax = graph::detail::AxisOf(a.Int("axis", 1), xs.size(), n.name);
      int64_t outer, C, inner; SplitAxis(xs, ax, &outer, &C, &inner);
      const bool fix_gamma = a.Bool("fix_gamma", true), global = a.Bool("use_global_stats", false) || !is_train_;
      const float* gamma = Val(s.in[1]);
      float* dg = GradOf(s.in[1]); float* dbeta = GradOf(s.in[2]);
      const int64_t cnt = outer * inner;
      for (int64_t c = 0; c < C; ++c) {
        const float mean = s.saved[c], inv = s.saved[C + c], g = fix_gamma ? 1.f : gamma[c];
        double sdy = 0, sdyx = 0;
        for (int64_t o = 0; o < outer; ++o) {
          const float* p = x + (o * C + c) * inner; const float* q = dy + (o * C + c) * inner;
          for (int64_t i = 0; i < inner; ++i) { sdy += q[i]; sdyx += q[i] * (p[i] - mean) * inv; }
        }
        if (dg && !fix_gamma) dg[c] += static_cast<float>(sdyx);
        if (dbeta) dbeta[c] += static_cast<float>(sdy);
        if (!dx) continue;
        const float msdy = static_cast<float>(sdy / cnt), msdyx = static_cast<float>(sdyx / cnt);
        for (int64_t o = 0; o < outer; ++o) {
          const float* p = x + (o * C + c) * inner; const float* q = dy + (o * C + c) * inner; float* d = dx + (o * C + c) * inner;
          if (global) for (int64_t i = 0; i < inner; ++i) d[i] += q[i] * g * inv;
          else for (int64_t i = 0; i < inner; ++i) d[i] += g * inv * (q[i] - msdy - (p[i] - mean) * inv * msdyx);
        }
      }
    } else if (op == "Dropout") {
      if (!dx) return;
      if (s.saved.empty()) for (int64_t i = 0; i < ny; ++i) dx[i] += dy[i];
      else for (int64_t i = 0; i < ny; ++i) dx[i] += dy[i] * s.saved[i];
    } else if (op == "Flatten" || op == "Reshape" || op == "expand_dims" || op == "identity") {
      if (dx) for (int64_t i = 0; i < ny; ++i) dx[i] += dy[i];
    } else if (op == "BlockGrad") {
    } else if (op == "MakeLoss") {
      if (dx) { const float gs = static_cast<float>(a.Float("grad_scale", 1.0)); for (int64_t i = 0; i < ny; ++i) dx[i] += gs; }
    } else if (op == "transpose") {
      if (!dx) return;
      auto axes = a.Tuple("axes", {});
      const size_t r = xs.size();
      if (axes.empty()) for (size_t i = 0; i < r; ++i) axes.push_back(static_cast<int64_t>(r - 1 - i));
      std::vector<int64_t> xstride(r, 1);
      for (int i = static_cast<int>(r) - 2; i >= 0; --i) xstride[i] = xstride[i + 1] * xs[i + 1];
      for (int64_t f = 0; f < ny; ++f) {
        int64_t rem = f, off = 0;
        for (int i = static_cast<int>(r) - 1; i >= 0; --i) { off += (rem % s.shape[i]) * xstride[graph::detail::AxisOf(axes[i], r, n.name)]; rem /= s.shape[i]; }
        dx[off] += dy[f];
      }
    } else if (op == "Concat") {
      const int64_t ax = graph::detail::AxisOf(a.Int("dim", 1), s.shape.size(), n.name);
      int64_t outer, C, inner; SplitAxis(s.shape, ax, &outer, &C, &inner);
      int64_t at = 0;
      for (int i : s.in) {
        const int64_t ci = slots_[i].shape[ax];
        if (float* d = GradOf(i)) for (int64_t o = 0; o < outer; ++o) { const float* q = dy + (o * C + at) * inner; float* dd = d + o * ci * inner; for (int64_t k = 0; k < ci * inner; ++k) dd[k] += q[k]; }
        at += ci;
      }
    } else if (op == "add_n") {
      for (int i : s.in) if (float* d = GradOf(i)) for (int64_t k = 0; k < ny; ++k) d[k] += dy[k];
    } else if (op == "Embedding") {
      if (float* dw = GradOf(s.in[1])) {
        const int64_t V = slots_[s.in[1]].shape[0], D = slots_[s.in[1]].shape[1];
        for (int64_t i = 0; i < nx; ++i) {
          const int64_t r = std::min<int64_t>(std::max<int64_t>(static_cast<int64_t>(x[i]), 0), V - 1);
          for (int64_t d = 0; d < D; ++d) dw[r * D + d] += dy[i * D + d];
        }
      }
    } else if (op == "SoftmaxOutput") {
      if (!dx) return;
      const float* label = Val(s.in[1]);
      const Shape& ls = slots_[s.in[1]].shape;
      const float gs = static_cast<float>(a.Float("grad_scale", 1.0));
      if (ls == xs) { for (int64_t i = 0; i < ny; ++i) dx[i] += (y[i] - label[i]) * gs; return; }      // probability labels
      int64_t outer, C, inner; SplitAxis(xs, 1, &outer, &C, &inner);
      if (!a.Bool("multi_output", false) && xs.size() > 2) { C = nx / xs[0]; inner = 1; outer = xs[0]; }
      if (Numel(ls) != outer * inner) throw std::runtime_error(n.name + ": label shape " + ShapeStr(ls) + " does not match the prediction " + ShapeStr(xs));
      const bool use_ignore = a.Bool("use_ignore", false);
      const float ignore = static_cast<float>(a.Float("ignore_label", -1));
      const std::string norm = a.Str("normalization", "null");
      int64_t valid = 0;
      for (int64_t t = 0; t < outer * inner; ++t) if (!(use_ignore && label[t] == ignore)) ++valid;
      const float scale = gs / (norm == "batch" ? static_cast<float>(outer) : norm == "valid" ? static_cast<float>(std::max<int64_t>(valid, 1)) : 1.f);
      for (int64_t o = 0; o < outer; ++o) for (int64_t i = 0; i < inner; ++i) {
        const float l = label[o * inner + i];
        if (use_ignore && l == ignore) continue;
        const int64_t cls = static_cast<int64_t>(l);
        for (int64_t k = 0; k < C; ++k) dx[(o * C + k) * inner + i] += (y[(o * C + k) * inner + i] - (k == cls ? 1.f : 0.f)) * scale;
      }
    } else if (op == "LinearRegressionOutput" || op == "LogisticRegressionOutput" || op == "MAERegressionOutput") {
      if (!dx) return;
      const float* label = Val(s.in[1]);
      if (Numel(slots_[s.in[1]].shape) != ny) throw std::runtime_error(n.name + ": label size does not match the prediction");
      const float scale = static_cast<float>(a.Float("grad_scale", 1.0)) / static_cast<float>(std::max<int64_t>(ny / std::max<int64_t>(xs[0], 1), 1));
      if (op == "MAERegressionOutput") for (int64_t i = 0; i < ny; ++i) dx[i] += (y[i] > label[i] ? 1.f : y[i] < label[i] ? -1.f : 0.f) * scale;
      else for (int64_t i = 0; i < ny; ++i) dx[i] += (y[i] - label[i]) * scale;
    } else if (op == "SoftmaxActivation" || op == "softmax" || op == "log_softmax") {
      if (!dx) return;
      int64_t outer, C, inner;
      SplitAxis(xs, op == "SoftmaxActivation" ? 1 : graph::detail::AxisOf(a.Int("axis", -1), xs.size(), n.name), &outer, &C, &inner);
      const bool lg = op == "log_softmax";
      for (int64_t o = 0; o < outer; ++o) for (int64_t i = 0; i < inner; ++i) {
        const float* ys = y + o * C * inner + i; const float* gs = dy + o * C * inner + i; float* ds = dx + o * C * inner + i;
        float dot = 0;
        for (int64_t k = 0; k < C; ++k) dot += lg ? gs[k * inner] : gs[k * inner] * ys[k * inner];
        for (int64_t k = 0; k < C; ++k) ds[k * inner] += lg ? gs[k * inner] - std::exp(ys[k * inner]) * dot : ys[k * inner] * (gs[k * inner] - dot);
      }
    } else if (op == "clip") {
      if (!dx) return;
      const float lo = static_cast<float>(a.Float("a_min", -std::numeric_limits<float>::infinity())), hi = static_cast<float>(a.Float("a_max", std::numeric_limits<float>::infinity()));
      for (int64_t i = 0; i < ny; ++i) if (x[i] >= lo && x[i] <= hi) dx[i] += dy[i];
    } else if (op == "SliceChannel") {
      if (!dx) return;
      const int64_t k = graph::NumOutputs(n);
      int64_t outer, C, inner; SplitAxis(xs, graph::detail::AxisOf(a.Int("axis", 1), xs.size(), n.name), &outer, &C, &inner);
      const int64_t Ck = C / k, self = &s - slots_.data();
      for (int64_t j = 0; j < k; ++j) {
        const float* g = slots_[self + j].grad.data();
        for (int64_t o = 0; o < outer; ++o) for (int64_t e = 0; e < Ck * inner; ++e) dx[(o * C + j * Ck) * inner + e] += g[o * Ck * inner + e];
      }
      for (int64_t j = 1; j < k; ++j) std::vector<float>().swap(slots_[self + j].grad);
    } else if (IsGather(op)) {
      if (dx) for (int64_t i = 0; i < ny; ++i) if (s.map[i] >= 0) dx[s.map[i]] += dy[i];
    } else if (op == "squeeze" || op == "Cast") {
      if (dx) for (int64_t i = 0; i < ny; ++i) dx[i] += dy[i];
    } else if (op == "where") {
      float* dt = GradOf(s.in[1]); float* df = GradOf(s.in[2]);
      for (int64_t i = 0; i < ny; ++i) { if (x[i] != 0.f) { if (dt) dt[i] += dy[i]; } else if (df) df[i] += dy[i]; }
    } else if (op == "one_hot" || op == "argmax" || op == "argmin" || op == "sgd_update" || op == "sgd_mom_update" || op == "adam_update") {
    } else if (op == "max" || op == "min" || op == "prod" || op == "norm") {
      if (!dx) return;
      const auto red = ReducedAxes(s, xs);
      for (int64_t f = 0; f < nx; ++f) {
        const int64_t o = ReducedIndex(f, xs, red);
        if (op == "prod") dx[f] += dy[o] * y[o] / x[f];
        else if (op == "norm") dx[f] += y[o] > 0 ? dy[o] * x[f] / y[o] : 0.f;
        else if (x[f] == y[o]) dx[f] += dy[o];
      }
    } else if (op == "LayerNorm" || op == "InstanceNorm") {
      int64_t outer, C, inner; NormGroups(s, xs, &outer, &C, &inner);
      const bool layer = op == "LayerNorm";
      const float* gamma = Val(s.in[1]);
      float* dg = GradOf(s.in[1]); float* db = GradOf(s.in[2]);
      const int64_t groups = layer ? outer * inner : outer * C, len = layer ? C : inner;
      for (int64_t g = 0; g < groups; ++g) {
        const int64_t base = layer ? (g / inner) * C * inner + g % inner : g * inner, stride = layer ? inner : 1;
        const float mean = s.saved[2 * g], inv = s.saved[2 * g + 1];
        double sg = 0, sgx = 0;
        for (int64_t k = 0; k < len; ++k) {
          const int64_t c = layer ? k : g % C, at = base + k * stride;
          const float xh = (x[at] - mean) * inv, gy = dy[at] * gamma[c];
          sg += gy; sgx += gy * xh;
          if (dg) dg[c] += dy[at] * xh;
          if (db) db[c] += dy[at];
        }
        if (!dx) continue;
        const float msg = static_cast<float>(sg / len), msgx = static_cast<float>(sgx / len);
        for (int64_t k = 0; k < len; ++k) {
          const int64_t c = layer ? k : g % C, at = base + k * stride;
          dx[at] += inv * (dy[at] * gamma[c] - msg - (x[at] - mean) * inv * msgx);
        }
      }
    } else if (op == "L2Normalization") {
      if (!dx) return;
      int64_t outer, C, inner; NormGroups(s, xs, &outer, &C, &inner);
      for (int64_t o = 0; o < outer; ++o) for (int64_t i = 0; i < inner; ++i) {
        const int64_t base = o * C * inner + i;
        const float nrm = s.saved[o * inner + i];
        double dot = 0;
        for (int64_t k = 0; k < C; ++k) dot += static_cast<double>(dy[base + k * inner]) * y[base + k * inner];
        for (int64_t k = 0; k < C; ++k) dx[base + k * inner] += (dy[base + k * inner] - y[base + k * inner] * static_cast<float>(dot)) / nrm;
      }
    } else if (op == "LRN") {
      if (!dx) return;
      const int64_t N = xs[0], C = xs[1], P = xs[2] * xs[3], half = a.Int("nsize", 1) / 2;
      const float alpha = static_cast<float>(a.Float("alpha", 1e-4)) / static_cast<float>(a.Int("nsize", 1)), beta = static_cast<float>(a.Float("beta", 0.75));
      for (int64_t b = 0; b < N; ++b) for (int64_t c = 0; c < C; ++c) for (int64_t p = 0; p < P; ++p) {
        const int64_t at = (b * C + c) * P + p;
        float acc = 0;
        for (int64_t k = std::max<int64_t>(c - half, 0); k <= std::min(c + half, C - 1); ++k) { const int64_t o = (b * C + k) * P + p; acc += dy[o] * y[o] / s.saved[o]; }
        dx[at] += dy[at] * std::pow(s.saved[at], -beta) - 2.f * alpha * beta * x[at] * acc;
      }
    } else if (op == "Deconvolution") {
      const Win w = WinOf(graph::detail::Window(n, false, xs));
      const int64_t N = xs[0], C = xs[1], H = xs[2], W = xs[3], F = s.shape[1], OH = s.shape[2], OW = s.shape[3], G = a.Int("num_group", 1);
      const int64_t Cg = C / G, Fg = F / G, K = Fg * w.kh * w.kw, P = H * W;
      const float* wt = Val(s.in[1]);
      float* dw = GradOf(s.in[1]);
      float* db = s.in.size() > 2 ? GradOf(s.in[2]) : nullptr;
      std::vector<float> col(static_cast<size_t>(K * P));
      for (int64_t i = 0; i < N; ++i) for (int64_t g = 0; g < G; ++g) {
        Im2Col(dy + (i * F + g * Fg) * OH * OW, Fg, OH, OW, w, H, W, col.data());                               // col(dY): [K, H*W]
        if (dx) GemmSerial(false, false, Cg, P, K, wt + g * Cg * K, col.data(), dx + (i * C + g * Cg) * P, true);   // dX_g += W_g . col
        if (dw) GemmSerial(false, true, Cg, K, P, x + (i * C + g * Cg) * P, col.data(), dw + g * Cg * K, true);     // dW_g += X_g . col^T
      }
      if (db) for (int64_t i = 0; i < N; ++i) for (int64_t f = 0; f < F; ++f) { const float* o = dy + (i * F + f) * OH * OW; float sm = 0; for (int64_t p = 0; p < OH * OW; ++p) sm += o[p]; db[f] += sm; }
    } else if (op == "smooth_l1") {
      if (!dx) return;
      const float s2 = static_cast<float>(a.Float("scalar", 1)) * static_cast<float>(a.Float("scalar", 1));
      for (int64_t i = 0; i < ny; ++i) dx[i] += dy[i] * (std::fabs(x[i]) < 1.f / s2 ? s2 * x[i] : (x[i] > 0 ? 1.f : -1.f));
    } else if (op == "softmax_cross_entropy") {
      if (!dx) return;
      const int64_t N = xs[0], C = xs[1];
      const float* label = Val(s.in[1]);
      for (int64_t i = 0; i < N; ++i) {
        const int64_t cls = std::min<int64_t>(std::max<int64_t>(static_cast<int64_t>(label[i]), 0), C - 1);
        for (int64_t k = 0; k < C; ++k) dx[i * C + k] += dy[0] * (s.saved[i * C + k] - (k == cls ? 1.f : 0.f));
      }
    } else if (op == "sum" || op == "mean") {
      if (!dx) return;
      const auto red = ReducedAxes(s, xs);
      const float div = op == "mean" ? static_cast<float>(nx / ny) : 1.f;
      for (int64_t f = 0; f < nx; ++f) dx[f] += dy[ReducedIndex(f, xs, red)] / div;
    } else if (op == "dot") {
      const bool ta = a.Bool("transpose_a", false), tb = a.Bool("transpose_b", false);
      const float* r = Val(s.in[1]);
      const Shape& rs = slots_[s.in[1]].shape;
      const int64_t M = s.shape[0], N = s.shape[1], K = ta ? xs[0] : xs[1];
      // Y = op(A) op(B):  d op(A) = dY op(B)^T,  d op(B) = op(A)^T dY;  a transposed operand receives the transpose of that
      if (dx) { if (!ta) Gemm(false, !tb, M, K, N, dy, r, dx, true); else Gemm(tb, true, K, M, N, r, dy, dx, true); }
      if (float* dr = GradOf(s.in[1])) { if (!tb) Gemm(!ta, false, K, N, M, x, dy, dr, true); else Gemm(true, ta, N, K, M, dy, x, dr, true); }
      (void)rs;
    } else if (s.in.size() == 2) {
      const int kind = BinaryKind(op);
      const float* r = Val(s.in[1]);
      const Shape& rs = slots_[s.in[1]].shape;
      float* dr = GradOf(s.in[1]);
      const Bcast bl(s.shape, xs), br(s.shape, rs);
      const bool same = xs == s.shape && rs == s.shape;
      for (int64_t i = 0; i < ny; ++i) {
        const int64_t li = same ? i : bl.At(i), ri = same ? i : br.At(i);
        const float l = x[li], rv = r[ri], g = dy[i];
        float gl, gr;
        switch (kind) {
          case 0: gl = g; gr = g; break;
          case 1: gl = g; gr = -g; break;
          case 2: gl = g * rv; gr = g * l; break;
          case 3: gl = g / rv; gr = -g * l / (rv * rv); break;
          case 4: gl = l >= rv ? g : 0.f; gr = l >= rv ? 0.f : g; break;
          case 5: gl = l <= rv ? g : 0.f; gr = l <= rv ? 0.f : g; break;
          case 6: gl = g * rv * std::pow(l, rv - 1.f); gr = g * y[i] * std::log(l); break;
          default: gl = 0.f; gr = 0.f; break;               // comparisons
        }
        if (dx) dx[li] += gl;
        if (dr) dr[ri] += gr;
      }
    } else if (op[0] == '_') {
      if (!dx) return;
      const float c = static_cast<float>(a.Float("scalar", 0));
      const int k = ScalarKind(op);
      for (int64_t i = 0; i < ny; ++i) dx[i] += dy[i] * ScG(k, x[i], c, y[i]);
    } else {
      if (!dx) return;
      const int k = UnaryKind(op);
      for (int64_t i = 0; i < ny; ++i) dx[i] += dy[i] * UnG(k, x[i], y[i]);
    }
  }
};

}  // namespace exec
}  // namespace gxrt
