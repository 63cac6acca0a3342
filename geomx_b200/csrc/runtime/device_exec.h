// Device training executor of the C API: the twin of train_exec.h::Executor for graphs bound to device arrays (GXExecutorSimpleBindEx /
// GXExecutorBind with dev_type 2, and GXImperativeInvoke on device inputs).  Same slot layout, same gradient-flow rules (BlockGrad cuts the
// gradient, fan-out accumulates) and the same kNullOp / kWriteTo / kAddTo handling; the difference is that every activation, gradient and
// operator workspace is a device allocation made at bind time, and every node runs sm_100a kernels of libgeomx_kernels.so on the library's
// stream of the executor's device.  Forward and Backward allocate nothing and never synchronise with the host.
//
// Operators: FullyConnected, Convolution (2-D, groups, depthwise), BatchNorm (axis 1), Pooling (max / avg / sum), Activation and relu,
// LeakyReLU (leaky), elemwise / broadcast add / sub / mul, add_n, Concat, Flatten, Reshape, identity, BlockGrad, MakeLoss, Dropout, SoftmaxOutput,
// softmax, log_softmax and the update operators sgd_update / sgd_mom_update / adam_update.  Anything else — another operator, a dilated
// convolution, BatchNorm on another axis — is refused at bind with the node's name; nothing runs on the host instead.
#pragma once
#include <cstring>
#include <string>
#include <vector>

#include "graph.h"
#include "kernel_lib.h"
#include "train_exec.h"

namespace gxrt {
namespace exec {

class DeviceExecutor {
 public:
  // args / grads / aux: device pointers in ListArguments / ListAuxiliaryStates order; grads[i].data may be null when reqs[i] == kNullOp
  DeviceExecutor(const Symbol& sym, int dev, const std::vector<Tensor>& args, const std::vector<Tensor>& grads, const std::vector<int>& reqs,
                 const std::vector<Tensor>& aux)
      : sym_(sym), dev_(dev), L_(kern::Get()) {
    stream_ = kern::DeviceStream(dev, "Bind");
    kern::Check(L_.set_device(dev_), "Bind");
    order_ = graph::Topo(sym_);
    for (Node* n : order_) if (n->op != "null") CheckSupported(*n);
    const auto aux_nodes = graph::AuxNodes(order_);
    std::map<std::string, Shape> known;
    size_t ai = 0, xi = 0;
    for (Node* n : order_) {
      index_[n] = static_cast<int>(slots_.size());
      slots_.emplace_back();
      Slot& s = slots_.back();
      s.node = n;
      if (n->op != "null") continue;
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
      for (auto& e : s.node->inputs) s.in.push_back(index_.at(e.node.get()) + e.index);
    }
    for (auto& s : slots_) {
      if (s.node->op == "null") { s.need_grad = s.req != kNullOp; continue; }
      if (s.node->op == "BlockGrad" || IsUpdate(s.node->op)) continue;
      for (int i : s.in) if (slots_[i].need_grad) s.need_grad = true;
    }
    for (auto& h : sym_.outputs) heads_.push_back(index_.at(h.node.get()) + h.index);
    seed_ = Executor::GlobalSeed().fetch_add(1) * 2654435761u + 12345u;
    // device memory: activations and per-node state, one gradient arena (zeroed by one memset per Backward), one shared workspace
    size_t grad_elems = 0, scratch = 0;
    for (auto& s : slots_) {
      if (s.need_grad) grad_elems += Pad(Numel(s.shape));
      if (s.node->op == "null") continue;
      s.own = Alloc(Numel(s.shape));
      Plan(s, &scratch);
    }
    if (grad_elems) {
      grad_arena_ = Alloc(static_cast<int64_t>(grad_elems)); grad_bytes_ = grad_elems * 4;
      size_t at = 0;
      for (auto& s : slots_) if (s.need_grad) { s.grad = grad_arena_ + at; at += Pad(Numel(s.shape)); }
    }
    if (scratch) scratch_ = Alloc(static_cast<int64_t>(scratch));
  }
  ~DeviceExecutor() { for (void* p : allocs_) L_.pool_free(dev_, p, stream_); }
  DeviceExecutor(const DeviceExecutor&) = delete;
  DeviceExecutor& operator=(const DeviceExecutor&) = delete;

  int device() const { return dev_; }
  size_t NumOutputs() const { return heads_.size(); }
  const Shape& OutputShape(size_t i) const { return slots_[heads_.at(i)].shape; }
  float* OutputData(size_t i) const { return Val(heads_.at(i)); }

  void Forward(bool is_train) {
    kern::Check(L_.set_device(dev_), "Forward");
    is_train_ = is_train;
    for (auto& s : slots_) if (s.node->op != "null") Run(s);
    ++step_;
    forwarded_ = true;
  }

  // head_grads: device pointers, or empty / null entries (loss heads ignore them, other heads get ones)
  void Backward(const std::vector<const float*>& head_grads) {
    if (!forwarded_) throw std::runtime_error("Backward: call Forward(is_train=1) first");
    if (!head_grads.empty() && head_grads.size() != heads_.size()) throw std::runtime_error("Backward: " + std::to_string(head_grads.size()) + " head gradients for " + std::to_string(heads_.size()) + " outputs");
    kern::Check(L_.set_device(dev_), "Backward");
    if (grad_bytes_) K(L_.memset(grad_arena_, 0, grad_bytes_, stream_), "zero gradients");
    for (size_t i = 0; i < heads_.size(); ++i) {
      Slot& s = slots_[heads_[i]];
      if (!s.need_grad) continue;
      const float* g = head_grads.empty() ? nullptr : head_grads[i];
      if (g) K(L_.axpy(s.grad, g, 1.f, Numel(s.shape), stream_), "head gradient");
      else K(L_.add_scalar(s.grad, 1.f, Numel(s.shape), stream_), "head gradient");
    }
    for (size_t k = slots_.size(); k-- > 0;) {
      Slot& s = slots_[k];
      if (s.node->op == "null" || !s.need_grad) continue;
      Grad(s);
    }
    for (int i : arg_slots_) {
      Slot& s = slots_[i];
      if (s.req == kNullOp) continue;
      const int64_t n = Numel(s.shape);
      if (s.req == kAddTo) K(L_.axpy(s.ext_grad, s.grad, 1.f, n, stream_), "gradient accumulation");
      else K(L_.memcpy(s.ext_grad, s.grad, static_cast<unsigned long long>(n) * 4, 3, stream_), "gradient copy");
    }
  }

  std::string Print() const {
    std::string o;
    int64_t act = 0;
    for (auto& s : slots_) {
      if (s.node->op == "null") { o += "Variable:" + s.node->name + " " + ShapeStr(s.shape) + (s.is_aux ? " aux" : s.req != kNullOp ? " grad" : "") + "\n"; continue; }
      o += "Op:" + s.node->op + ", Name=" + s.node->name + " -> " + ShapeStr(s.shape) + "\n";
      for (int i : s.in) o += "  arg: " + slots_[i].node->name + "\n";
      act += Numel(s.shape);
    }
    o += "Total " + std::to_string(act * 4 / 1024) + " KB allocated for activations on gpu(" + std::to_string(dev_) + ")\n";
    return o;
  }

 private:
  struct Slot {
    Node* node = nullptr;
    Shape shape;
    std::vector<int> in;
    float* ext = nullptr;               // variables: the bound device array
    float* ext_grad = nullptr;
    int req = kNullOp;
    bool is_aux = false, need_grad = false;
    float* own = nullptr;               // operators: the output
    float* grad = nullptr;              // d loss / d output (inside the gradient arena)
    float* saved = nullptr;             // BatchNorm: mean, inverse std, ones (fix_gamma); Dropout: mask; Convolution: im2col matrix
    int* idx = nullptr;                 // Pooling(max): arg-max offsets
    bool dropped = false;               // Dropout: the last forward applied a mask
    bool depthwise = false;             // Convolution: num_group == C == F through the depthwise kernels
    int64_t ldc = 0;                    // Convolution: row stride of the im2col matrix (a multiple of 4 for the TMA GEMM)
  };
  Symbol sym_;
  int dev_;
  const kern::Lib& L_;
  kern::Stream stream_ = nullptr;
  std::vector<Node*> order_;
  std::unordered_map<Node*, int> index_;
  std::vector<Slot> slots_;
  std::vector<int> arg_slots_, heads_;
  std::vector<void*> allocs_;
  float* grad_arena_ = nullptr;
  size_t grad_bytes_ = 0;
  float* scratch_ = nullptr;
  bool is_train_ = false, forwarded_ = false;
  uint32_t seed_ = 0, step_ = 0;

  static size_t Pad(int64_t n) { return static_cast<size_t>((n + 63) / 64 * 64); }        // 256-byte aligned sub-buffers
  static bool IsUpdate(const std::string& op) { return op == "sgd_update" || op == "sgd_mom_update" || op == "adam_update"; }
  static bool IsCopy(const std::string& op) { return op == "Flatten" || op == "Reshape" || op == "identity" || op == "BlockGrad" || op == "MakeLoss"; }
  static int BinKind(const std::string& op) {
    if (op == "elemwise_add" || op == "broadcast_add") return 0;
    if (op == "elemwise_sub" || op == "broadcast_sub") return 1;
    if (op == "elemwise_mul" || op == "broadcast_mul") return 2;
    return -1;
  }
  void K(int rc, const char* what) const { kern::Check(rc, what); }
  float* Alloc(int64_t n) {
    const size_t bytes = static_cast<size_t>(std::max<int64_t>(n, 1)) * 4;
    void* p = L_.pool_alloc(dev_, bytes, stream_);
    if (!p) throw std::runtime_error("Bind: out of device memory on gpu(" + std::to_string(dev_) + ") (" + std::to_string(bytes) + " bytes)");
    allocs_.push_back(p);
    K(L_.memset(p, 0, bytes, stream_), "Bind");
    return static_cast<float*>(p);
  }
  float* Val(int i) const { const Slot& s = slots_[i]; return s.node->op == "null" ? s.ext : s.own; }
  float* GradOf(int i) { Slot& s = slots_[i]; return s.need_grad ? s.grad : nullptr; }
  const Shape& ShapeOfSlot(int i) const { return slots_[i].shape; }

  void CheckSupported(const Node& n) const {
    const std::string& op = n.op;
    AttrView a(n.attrs);
    auto refuse = [&](const std::string& why) { throw std::runtime_error("Bind: node " + n.name + " (" + op + "): " + why); };
    if (graph::NumOutputs(n) != 1) refuse("multi-output operators are not supported by the device executor");
    if (op == "Convolution") {
      const auto d = a.Tuple("dilate", {});
      for (auto v : d) if (v != 1) refuse("dilated convolution is not supported by the device executor");
      if (a.Tuple("kernel", {}).size() != 2) refuse("only 2-D convolution is supported by the device executor");
    } else if (op == "Pooling") {
      const std::string t = a.Str("pool_type", "max");
      if (t != "max" && t != "avg" && t != "sum") refuse("pool_type " + t + " is not supported by the device executor");
    } else if (op == "Activation") {
      ActKind(a.Str("act_type", "relu"), n.name);
    } else if (op == "relu") {
    } else if (op == "LeakyReLU") {
      if (a.Str("act_type", "leaky") != "leaky") refuse("act_type " + a.Str("act_type", "leaky") + " is not supported by the device executor");
    } else if (op == "BatchNorm") {
      if (a.Int("axis", 1) != 1) refuse("only axis=1 is supported by the device executor");
    } else if (op == "FullyConnected" || op == "Concat" || op == "add_n" || op == "Dropout" || op == "SoftmaxOutput" || op == "softmax" ||
               op == "log_softmax" || IsCopy(op) || IsUpdate(op) || BinKind(op) >= 0) {
    } else {
      refuse("operator is not supported by the device executor");
    }
  }

  // per-node device state and the node's workspace need (floats) at bind
  void Plan(Slot& s, size_t* scratch) {
    const Node& n = *s.node;
    const std::string& op = n.op;
    AttrView a(n.attrs);
    const Shape& xs = slots_[s.in[0]].shape;
    if (op == "Convolution") {
      if (xs.size() != 4) throw std::runtime_error("Bind: node " + n.name + " (Convolution): input must be NCHW");
      const Win w = WinOf(graph::detail::Window(n, false, xs));
      const int64_t N = xs[0], C = xs[1], H = xs[2], W = xs[3], F = s.shape[1], P = s.shape[2] * s.shape[3], G = a.Int("num_group", 1);
      const size_t plane_in = static_cast<size_t>(H * W + w.kh * w.kw) * 4, plane_out = static_cast<size_t>(P + w.kh * w.kw) * 4,
                   plane_w = static_cast<size_t>(H * W + P) * 4;
      s.depthwise = G == C && G == F && G > 1 && plane_in <= 200 * 1024 && plane_out <= 200 * 1024 && plane_w <= 200 * 1024;
      if (s.depthwise) { *scratch = std::max(*scratch, static_cast<size_t>(N * C * H * W + F * w.kh * w.kw + F)); return; }
      s.ldc = (C * w.kh * w.kw + 3) / 4 * 4;
      s.saved = Alloc(N * P * s.ldc);
      *scratch = std::max(*scratch, static_cast<size_t>(N * P * F + N * P * s.ldc + N * C * H * W));
    } else if (op == "BatchNorm") {
      const int64_t C = xs[1];
      s.saved = Alloc(3 * C);
      std::vector<float> ones(static_cast<size_t>(C), 1.f);
      K(L_.memcpy(s.saved + 2 * C, ones.data(), static_cast<unsigned long long>(C) * 4, 1, stream_), "Bind");
      *scratch = std::max(*scratch, static_cast<size_t>(Numel(xs) + 2 * C));
    } else if (op == "Pooling") {
      if (a.Str("pool_type", "max") == "max") s.idx = reinterpret_cast<int*>(Alloc(Numel(s.shape)));
    } else if (op == "Dropout") {
      s.saved = Alloc(Numel(s.shape));
    } else if (op == "SoftmaxOutput") {
      const Shape& ls = slots_[s.in[1]].shape;
      int64_t outer, C, inner; SoftmaxOutputSplit(s, &outer, &C, &inner);
      if (ls != xs && Numel(ls) != outer * inner) throw std::runtime_error("Bind: node " + n.name + " (SoftmaxOutput): label shape " + ShapeStr(ls) + " does not match the prediction " + ShapeStr(xs));
    }
  }

  static Win WinOf(const graph::detail::Win& w) { return Win{w.kh, w.kw, w.sh, w.sw, w.ph, w.pw, w.dh, w.dw}; }
  static void SplitAxis(const Shape& s, int64_t ax, int64_t* outer, int64_t* c, int64_t* inner) {
    *outer = 1; *inner = 1; *c = s[ax];
    for (int64_t i = 0; i < ax; ++i) *outer *= s[i];
    for (size_t i = ax + 1; i < s.size(); ++i) *inner *= s[i];
  }
  void SoftmaxOutputSplit(const Slot& s, int64_t* outer, int64_t* C, int64_t* inner) const {
    const Shape& xs = slots_[s.in[0]].shape;
    SplitAxis(xs, 1, outer, C, inner);
    if (!AttrView(s.node->attrs).Bool("multi_output", false) && xs.size() > 2) { *C = Numel(xs) / xs[0]; *inner = 1; *outer = xs[0]; }
  }

  // D (+)= op(A) . op(B) on the tcgen05 GEMM (3xTF32 by default); operands that miss the TMA alignment go to the CUDA-core GEMM
  void Gemm(const float* A, int64_t lda, int a_mn, const float* B, int64_t ldb, int b_mn, int64_t M, int64_t N, int64_t Kd, float* D, int64_t ldd,
            const float* bias, int accumulate) {
    int rc = L_.gemm_tf32(A, lda, a_mn, B, ldb, b_mn, static_cast<int>(M), static_cast<int>(N), static_cast<int>(Kd), D, ldd, bias, nullptr, 0, nullptr, 0,
                          accumulate, 0, 0, 1.f, 1, stream_);
    if (rc < 0) rc = L_.gemm_simt(A, lda, a_mn, B, ldb, b_mn, static_cast<int>(M), static_cast<int>(N), static_cast<int>(Kd), D, ldd, bias, nullptr, 0,
                                  nullptr, 0, accumulate, 0, 0, 1.f, stream_);
    K(rc, "GEMM");
  }
  void Copy(float* dst, const float* src, int64_t n) { K(L_.memcpy(dst, src, static_cast<unsigned long long>(n) * 4, 3, stream_), "device copy"); }
  // operand strides of a broadcast binary operator over the output's axes
  static void BcastStrides(const Shape& out, const Shape& in, long long* st) {
    long long acc = 1;
    for (int i = static_cast<int>(in.size()) - 1, o = static_cast<int>(out.size()) - 1; o >= 0; --i, --o) {
      const int64_t d = i >= 0 ? in[i] : 1;
      st[o] = d == 1 ? 0 : acc;
      acc *= d;
    }
  }

  // ---- forward
  void Run(Slot& s) {
    const Node& n = *s.node;
    const std::string& op = n.op;
    AttrView a(n.attrs);
    float* y = s.own;
    const int64_t ny = Numel(s.shape);
    const float* x = Val(s.in[0]);
    const Shape& xs = slots_[s.in[0]].shape;
    if (op == "FullyConnected") {
      const int64_t h = s.shape.back(), k = slots_[s.in[1]].shape[1], m = Numel(xs) / k;
      Gemm(x, k, 0, Val(s.in[1]), k, 0, m, h, k, y, h, s.in.size() > 2 ? Val(s.in[2]) : nullptr, 0);
    } else if (op == "Convolution") {
      const Win w = WinOf(graph::detail::Window(n, false, xs));
      const int64_t N = xs[0], C = xs[1], H = xs[2], W = xs[3], F = s.shape[1], P = s.shape[2] * s.shape[3], G = a.Int("num_group", 1);
      const float* wt = Val(s.in[1]); const float* b = s.in.size() > 2 ? Val(s.in[2]) : nullptr;
      if (s.depthwise) {
        K(L_.depthwise_fwd(x, wt, b, y, (int)N, (int)C, (int)H, (int)W, (int)w.kh, (int)w.kw, (int)w.sh, (int)w.sw, (int)w.ph, (int)w.pw, 0, stream_), "depthwise convolution");
        return;
      }
      const int64_t Cg = C / G, Fg = F / G, Kg = Cg * w.kh * w.kw;
      float* col = s.saved; float* rows = scratch_;
      K(L_.im2col(x, col, (int)N, (int)C, (int)H, (int)W, (int)w.kh, (int)w.kw, (int)w.sh, (int)w.sw, (int)w.ph, (int)w.pw, (int)s.ldc, stream_), "im2col");
      for (int64_t g = 0; g < G; ++g) Gemm(col + g * Kg, s.ldc, 0, wt + g * Fg * Kg, Kg, 0, N * P, Fg, Kg, rows + g * Fg, F, b ? b + g * Fg : nullptr, 0);
      K(L_.rows_to_nchw(rows, y, (int)N, (int)F, (int)P, F, 0, stream_), "rows to NCHW");
    } else if (op == "BatchNorm") {
      const int64_t N = xs[0], C = xs[1], HW = Numel(xs) / (xs[0] * xs[1]);
      const float eps = static_cast<float>(a.Float("eps", 1e-3)), mom = static_cast<float>(a.Float("momentum", 0.9));
      const bool fix_gamma = a.Bool("fix_gamma", true), global = a.Bool("use_global_stats", false) || !is_train_;
      const float* gamma = fix_gamma ? s.saved + 2 * C : Val(s.in[1]);
      K(L_.bn_fwd(x, gamma, Val(s.in[2]), Val(s.in[3]), Val(s.in[4]), y, s.saved, s.saved + C, (int)N, (int)C, (int)HW, global ? 0 : 1, mom, eps, stream_), "BatchNorm");
    } else if (op == "Pooling") {
      const Win w = WinOf(graph::detail::Window(n, true, xs));
      const std::string t = a.Str("pool_type", "max");
      K(L_.pool_fwd(t == "max" ? 0 : t == "avg" ? 1 : 2, x, y, s.idx, xs[0] * xs[1], (int)xs[2], (int)xs[3], (int)s.shape[2], (int)s.shape[3], (int)w.kh, (int)w.kw,
                    (int)w.sh, (int)w.sw, (int)w.ph, (int)w.pw, a.Bool("count_include_pad", true) ? 1 : 0, stream_), "Pooling");
    } else if (op == "Activation" || op == "relu") {
      K(L_.act_fwd(op == "relu" ? 0 : ActKind(a.Str("act_type", "relu"), n.name), x, y, ny, 0.f, stream_), op.c_str());
    } else if (op == "LeakyReLU") {
      K(L_.act_fwd(5, x, y, ny, static_cast<float>(a.Float("slope", 0.25)), stream_), "LeakyReLU");
    } else if (BinKind(op) >= 0) {
      long long dims[8], ls[8], rs[8];
      for (size_t d = 0; d < s.shape.size(); ++d) dims[d] = s.shape[d];
      BcastStrides(s.shape, xs, ls); BcastStrides(s.shape, slots_[s.in[1]].shape, rs);
      K(L_.binary_fwd(BinKind(op), x, Val(s.in[1]), y, static_cast<int>(s.shape.size()), dims, ls, rs, stream_), op.c_str());
    } else if (op == "add_n") {
      std::vector<const float*> ins;
      for (int i : s.in) ins.push_back(Val(i));
      if (ins.size() <= 8) { K(L_.nary_sum(y, ins.data(), static_cast<int>(ins.size()), ny, stream_), "add_n"); return; }
      Copy(y, ins[0], ny);
      for (size_t i = 1; i < ins.size(); ++i) K(L_.axpy(y, ins[i], 1.f, ny, stream_), "add_n");
    } else if (op == "Concat") {
      const int64_t ax = graph::detail::AxisOf(a.Int("dim", 1), s.shape.size(), n.name);
      int64_t outer, C, inner; SplitAxis(s.shape, ax, &outer, &C, &inner);
      int64_t at = 0;
      for (int i : s.in) {
        const int64_t ci = slots_[i].shape[ax];
        K(L_.strided_copy(Val(i), y + at * inner, outer, ci * inner, ci * inner, C * inner, 0, stream_), "Concat");
        at += ci;
      }
    } else if (IsCopy(op)) {
      Copy(y, x, ny);
    } else if (op == "Dropout") {
      const float p = static_cast<float>(a.Float("p", 0.5));
      s.dropped = is_train_ && p > 0.f;
      if (!s.dropped) { Copy(y, x, ny); return; }
      if (p >= 1.f) throw std::runtime_error(n.name + ": drop probability must be < 1");
      K(L_.dropout_fwd(x, y, s.saved, ny, p, seed_, step_, stream_), "Dropout");
    } else if (op == "SoftmaxOutput") {
      int64_t outer, C, inner; SoftmaxOutputSplit(s, &outer, &C, &inner);
      K(L_.softmax_fwd(x, y, outer, (int)C, inner, 0, stream_), "SoftmaxOutput");
    } else if (op == "softmax" || op == "log_softmax") {
      int64_t outer, C, inner; SplitAxis(xs, graph::detail::AxisOf(a.Int("axis", -1), xs.size(), n.name), &outer, &C, &inner);
      K(L_.softmax_fwd(x, y, outer, (int)C, inner, op == "log_softmax" ? 1 : 0, stream_), op.c_str());
    } else if (IsUpdate(op)) {
      // the new weight goes to the output; optimizer states (trailing auxiliary inputs) are updated in place
      Copy(y, x, ny);
      const float lr = static_cast<float>(a.Float("lr", 0)), wd = static_cast<float>(a.Float("wd", 0)), rescale = static_cast<float>(a.Float("rescale_grad", 1)),
                  clip = static_cast<float>(a.Float("clip_gradient", -1));
      const float* g = Val(s.in[1]);
      if (op == "adam_update")
        K(L_.single_opt(1, y, g, Val(s.in[2]), Val(s.in[3]), ny, lr, wd, rescale, clip, 0.f, static_cast<float>(a.Float("beta1", 0.9)),
                        static_cast<float>(a.Float("beta2", 0.999)), static_cast<float>(a.Float("epsilon", 1e-8)), 0.f, stream_), "adam_update");
      else
        K(L_.single_opt(0, y, g, op == "sgd_mom_update" ? Val(s.in[2]) : nullptr, nullptr, ny, lr, wd, rescale, clip,
                        op == "sgd_mom_update" ? static_cast<float>(a.Float("momentum", 0)) : 0.f, 0.f, 0.f, 0.f, 0.f, stream_), op.c_str());
    }
  }

  // ---- backward: s.grad holds d loss / d output; adds into the inputs' gradient buffers (only where need_grad)
  void Grad(Slot& s) {
    const Node& n = *s.node;
    const std::string& op = n.op;
    AttrView a(n.attrs);
    const float* dy = s.grad;
    const float* y = s.own;
    const int64_t ny = Numel(s.shape);
    const float* x = Val(s.in[0]);
    const Shape& xs = slots_[s.in[0]].shape;
    float* dx = GradOf(s.in[0]);
    if (op == "FullyConnected") {
      const int64_t h = s.shape.back(), k = slots_[s.in[1]].shape[1], m = Numel(xs) / k;
      if (dx) Gemm(dy, h, 0, Val(s.in[1]), k, 1, m, k, h, dx, k, nullptr, 1);                     // dX += dY . W
      if (float* dw = GradOf(s.in[1])) Gemm(dy, h, 1, x, k, 1, h, k, m, dw, k, nullptr, 1);        // dW += dY^T . X
      if (s.in.size() > 2) if (float* db = GradOf(s.in[2])) K(L_.colsum(dy, db, m, (int)h, h, 1, stream_), "bias gradient");
    } else if (op == "Convolution") {
      const Win w = WinOf(graph::detail::Window(n, false, xs));
      const int64_t N = xs[0], C = xs[1], H = xs[2], W = xs[3], F = s.shape[1], P = s.shape[2] * s.shape[3], G = a.Int("num_group", 1);
      const float* wt = Val(s.in[1]);
      float* dw = GradOf(s.in[1]);
      float* db = s.in.size() > 2 ? GradOf(s.in[2]) : nullptr;
      if (s.depthwise) {
        float* dxt = scratch_;
        if (dw || db) {
          float* dw_to = dw ? dw : scratch_ + N * C * H * W;
          float* db_to = db ? db : (s.in.size() > 2 ? scratch_ + N * C * H * W + F * w.kh * w.kw : nullptr);
          K(L_.depthwise_wgrad(x, dy, dw_to, db_to, (int)N, (int)C, (int)H, (int)W, (int)w.kh, (int)w.kw, (int)w.sh, (int)w.sw, (int)w.ph, (int)w.pw, stream_), "depthwise weight gradient");
        }
        if (dx) {
          K(L_.depthwise_dgrad(dy, wt, dxt, (int)N, (int)C, (int)H, (int)W, (int)w.kh, (int)w.kw, (int)w.sh, (int)w.sw, (int)w.ph, (int)w.pw, stream_), "depthwise data gradient");
          K(L_.axpy(dx, dxt, 1.f, N * C * H * W, stream_), "depthwise data gradient");
        }
        return;
      }
      const int64_t Cg = C / G, Fg = F / G, Kg = Cg * w.kh * w.kw;
      float* dyr = scratch_; float* dcol = scratch_ + N * P * F; float* dxt = dcol + N * P * s.ldc;
      K(L_.nchw_to_rows(dy, dyr, (int)N, (int)F, (int)P, stream_), "NCHW to rows");
      if (dw) for (int64_t g = 0; g < G; ++g) Gemm(dyr + g * Fg, F, 1, s.saved + g * Kg, s.ldc, 1, Fg, Kg, N * P, dw + g * Fg * Kg, Kg, nullptr, 1);
      if (db) K(L_.colsum(dyr, db, N * P, (int)F, F, 1, stream_), "bias gradient");
      if (dx) {
        for (int64_t g = 0; g < G; ++g) Gemm(dyr + g * Fg, F, 0, wt + g * Fg * Kg, Kg, 1, N * P, Kg, Fg, dcol + g * Kg, s.ldc, nullptr, 0);
        K(L_.col2im(dcol, dxt, (int)N, (int)C, (int)H, (int)W, (int)w.kh, (int)w.kw, (int)w.sh, (int)w.sw, (int)w.ph, (int)w.pw, (int)s.ldc, stream_), "col2im");
        K(L_.axpy(dx, dxt, 1.f, N * C * H * W, stream_), "data gradient");
      }
    } else if (op == "BatchNorm") {
      const int64_t N = xs[0], C = xs[1], HW = Numel(xs) / (xs[0] * xs[1]);
      const bool fix_gamma = a.Bool("fix_gamma", true), global = a.Bool("use_global_stats", false) || !is_train_;
      float* dg = fix_gamma ? nullptr : GradOf(s.in[1]);
      float* dbeta = GradOf(s.in[2]);
      if (global) {
        K(L_.bn_global_bwd(x, dy, fix_gamma ? nullptr : Val(s.in[1]), Val(s.in[3]), Val(s.in[4]), static_cast<float>(a.Float("eps", 1e-3)), dx, dg, dbeta,
                           (int)N, (int)C, (int)HW, stream_), "BatchNorm backward");
        return;
      }
      const float* gamma = fix_gamma ? s.saved + 2 * C : Val(s.in[1]);
      float* dxt = scratch_; float* dgt = scratch_ + Numel(xs); float* dbt = dgt + C;
      K(L_.bn_bwd(x, dy, gamma, s.saved, s.saved + C, dxt, dgt, dbt, (int)N, (int)C, (int)HW, stream_), "BatchNorm backward");
      if (dx) K(L_.axpy(dx, dxt, 1.f, Numel(xs), stream_), "BatchNorm backward");
      if (dg) K(L_.axpy(dg, dgt, 1.f, C, stream_), "BatchNorm backward");
      if (dbeta) K(L_.axpy(dbeta, dbt, 1.f, C, stream_), "BatchNorm backward");
    } else if (op == "Pooling") {
      if (!dx) return;
      const Win w = WinOf(graph::detail::Window(n, true, xs));
      const std::string t = a.Str("pool_type", "max");
      K(L_.pool_bwd(t == "max" ? 0 : t == "avg" ? 1 : 2, dy, s.idx, dx, xs[0] * xs[1], (int)xs[2], (int)xs[3], (int)s.shape[2], (int)s.shape[3], (int)w.kh,
                    (int)w.kw, (int)w.sh, (int)w.sw, (int)w.ph, (int)w.pw, a.Bool("count_include_pad", true) ? 1 : 0, stream_), "Pooling backward");
    } else if (op == "Activation" || op == "relu") {
      if (dx) K(L_.act_bwd(op == "relu" ? 0 : ActKind(a.Str("act_type", "relu"), n.name), x, y, dy, dx, ny, 0.f, stream_), "Activation backward");
    } else if (op == "LeakyReLU") {
      if (dx) K(L_.act_bwd(5, x, y, dy, dx, ny, static_cast<float>(a.Float("slope", 0.25)), stream_), "LeakyReLU backward");
    } else if (BinKind(op) >= 0) {
      float* dr = GradOf(s.in[1]);
      if (!dx && !dr) return;
      long long dims[8], ls[8], rs[8];
      for (size_t d = 0; d < s.shape.size(); ++d) dims[d] = s.shape[d];
      BcastStrides(s.shape, xs, ls); BcastStrides(s.shape, slots_[s.in[1]].shape, rs);
      K(L_.binary_bwd(BinKind(op), x, Val(s.in[1]), dy, dx, dr, static_cast<int>(s.shape.size()), dims, ls, rs, stream_), op.c_str());
    } else if (op == "add_n") {
      for (int i : s.in) if (float* d = GradOf(i)) K(L_.axpy(d, dy, 1.f, ny, stream_), "add_n backward");
    } else if (op == "Concat") {
      const int64_t ax = graph::detail::AxisOf(a.Int("dim", 1), s.shape.size(), n.name);
      int64_t outer, C, inner; SplitAxis(s.shape, ax, &outer, &C, &inner);
      int64_t at = 0;
      for (int i : s.in) {
        const int64_t ci = slots_[i].shape[ax];
        if (float* d = GradOf(i)) K(L_.strided_copy(dy + at * inner, d, outer, ci * inner, C * inner, ci * inner, 1, stream_), "Concat backward");
        at += ci;
      }
    } else if (op == "MakeLoss") {
      if (dx) K(L_.add_scalar(dx, static_cast<float>(a.Float("grad_scale", 1.0)), ny, stream_), "MakeLoss backward");
    } else if (op == "BlockGrad" || IsUpdate(op)) {
    } else if (IsCopy(op)) {
      if (dx) K(L_.axpy(dx, dy, 1.f, ny, stream_), "copy backward");
    } else if (op == "Dropout") {
      if (!dx) return;
      if (s.dropped) K(L_.mul_add(dx, dy, s.saved, ny, stream_), "Dropout backward");
      else K(L_.axpy(dx, dy, 1.f, ny, stream_), "Dropout backward");
    } else if (op == "SoftmaxOutput") {
      if (!dx) return;
      const float* label = Val(s.in[1]);
      const float gs = static_cast<float>(a.Float("grad_scale", 1.0));
      if (slots_[s.in[1]].shape == xs) {                         // probability labels
        K(L_.axpy(dx, y, gs, ny, stream_), "SoftmaxOutput backward");
        K(L_.axpy(dx, label, -gs, ny, stream_), "SoftmaxOutput backward");
        return;
      }
      int64_t outer, C, inner; SoftmaxOutputSplit(s, &outer, &C, &inner);
      const std::string norm = a.Str("normalization", "null");
      K(L_.softmax_output_bwd(y, label, dx, outer, (int)C, inner, gs, a.Bool("use_ignore", false) ? 1 : 0, static_cast<float>(a.Float("ignore_label", -1)),
                              norm == "batch" ? 1 : norm == "valid" ? 2 : 0, stream_), "SoftmaxOutput backward");
    } else if (op == "softmax" || op == "log_softmax") {
      if (!dx) return;
      int64_t outer, C, inner; SplitAxis(xs, graph::detail::AxisOf(a.Int("axis", -1), xs.size(), n.name), &outer, &C, &inner);
      K(L_.softmax_bwd(y, dy, dx, outer, (int)C, inner, op == "log_softmax" ? 1 : 0, stream_), op.c_str());
    }
  }
};

}  // namespace exec
}  // namespace gxrt
