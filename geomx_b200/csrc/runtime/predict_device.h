// Device runner of the native predictor: GXPredCreate* with dev_type 2 (c_predict_api.cc).  It executes the GraphPlan of predict.h — the
// same graph loader, shape inference and liveness plan as the host Predictor — with sm_100a kernels of libgeomx_kernels.so (kernel_lib.h).
//
// Memory.  Parameters are uploaded once per create from the native pool (DeviceParams) and shared, by reference count, with the handles of
// GXPredCreateMultiThread and GXPredReshape; BatchNorm's scale and shift are folded on the host at that point, exactly as predict.h does
// at run time.  Every handle owns one arena of the planned size (so GXPredGetPlan reports the host's numbers), its input buffers and one
// workspace shared by all operators: im2col matrix plus GEMM rows for the largest convolution, or the arg-max scratch of max pooling.
// Forward allocates nothing.
//
// Execution.  Every handle has a stream of its own.  The first Forward runs the operators eagerly (kernels do their one-time setup
// then); the second captures the same launches into a CUDA graph, thread-locally, and every later Forward is one graph launch.  The
// graph is valid for the life of the handle because its shapes and buffers never change: Reshape makes a new handle.  PartialForward
// always runs eagerly, one planned operator per step.
//
// Operators: the whole planned set of predict.h.  An attribute the device cannot honour, or a BatchNorm whose statistics are not in the
// parameter file, is refused at create with the node's name; nothing falls back to the host.
#pragma once
#include <algorithm>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "kernel_lib.h"
#include "predict.h"

namespace gxrt {
namespace predict {

// device copies of one create's parameters; freed, on the device's library stream, with the last handle that uses them
struct DeviceParams {
  const kern::Lib* L = nullptr;
  int dev = 0;
  std::map<std::string, float*> ptr;          // parameter name -> device copy
  std::map<int, float*> bn;                   // BatchNorm node -> [scale (C) | shift (C)]
  std::vector<void*> allocs;
  DeviceParams() = default;
  DeviceParams(const DeviceParams&) = delete;
  DeviceParams& operator=(const DeviceParams&) = delete;
  ~DeviceParams() {
    if (!L || allocs.empty()) return;
    L->set_device(dev);
    void* s = L->stream(dev);
    for (void* p : allocs) L->pool_free(dev, p, s);
  }
};

class DevicePredictor : public GraphPlan {
 public:
  DevicePredictor(const std::string& json, const char* params, size_t param_size, const std::vector<std::string>& input_keys,
                  const std::vector<Shape>& input_shapes, const std::vector<std::string>& output_keys, int dev)
      : GraphPlan(json, params, param_size, input_keys, input_shapes, output_keys), L_(&kern::Get()), dev_(dev) {
    kern::DeviceStream(dev, "GXPredCreate");
    SetDevice("GXPredCreate");
    CheckSupported();
    prm_ = Upload();
    Bind();
  }
  // another handle over the same graph and device parameters with its own stream, inputs, arena and workspace
  std::unique_ptr<DevicePredictor> Clone(const std::map<std::string, Shape>* new_shapes) const {
    std::unique_ptr<DevicePredictor> p(new DevicePredictor(*this, 0));
    p->SetDevice("GXPredReshape");
    p->Replan(new_shapes);
    p->CheckSupported();
    p->Bind();
    return p;
  }
  ~DevicePredictor() { Release(); }
  DevicePredictor(const DevicePredictor&) = delete;
  DevicePredictor& operator=(const DevicePredictor&) = delete;

  void SetDevice(const char* what) const { kern::Check(L_->set_device(dev_), what); }
  // host or device memory (cudaMemcpyDefault); returns when `data` has been read
  void SetInput(const std::string& key, const float* data, size_t size) {
    auto it = inputs_.find(key);
    if (it == inputs_.end()) throw std::runtime_error("SetInput: unknown input " + key);
    if (size != it->second.second) throw std::runtime_error("SetInput: " + key + " expects " + std::to_string(it->second.second) + " values, got " + std::to_string(size));
    K(L_->memcpy(it->second.first, data, static_cast<unsigned long long>(size) * 4, 4, stream_), "GXPredSetInput");
    K(L_->stream_sync(stream_), "GXPredSetInput");
  }
  // asynchronous: the work is queued on the handle's stream
  void Forward() {
    if (!eager_done_) { RunAll(); eager_done_ = true; return; }
    if (!graph_) Capture();
    K(L_->graph_launch(graph_, stream_), "GXPredForward: CUDA graph launch");
  }
  void PartialForward(int step, int* step_left) {
    if (step < 0 || step >= static_cast<int>(order_.size())) { *step_left = 0; return; }
    RunOp(order_[step]);
    *step_left = static_cast<int>(order_.size()) - step - 1;
  }
  // waits for the handle's stream; `out` may be host or device memory
  void GetOutput(size_t i, float* out, size_t size) const {
    const Node& n = nodes_[Head(i)];
    if (size != static_cast<size_t>(Numel(n.shape))) throw std::runtime_error("GetOutput: output " + std::to_string(i) + " has " + std::to_string(Numel(n.shape)) + " values, buffer holds " + std::to_string(size));
    K(L_->memcpy(out, ptr_[n.storage], static_cast<unsigned long long>(size) * 4, 4, stream_), "GXPredGetOutput");
    K(L_->stream_sync(stream_), "GXPredGetOutput");
  }

 private:
  const kern::Lib* L_;
  int dev_;
  std::shared_ptr<DeviceParams> prm_;
  kern::Stream stream_ = nullptr;
  void* graph_ = nullptr;
  bool eager_done_ = false;
  std::vector<void*> allocs_;
  std::vector<float*> ptr_;                                            // storage -> device address
  std::map<std::string, std::pair<float*, size_t>> inputs_;           // input key -> buffer, values
  float* ws_ = nullptr;

  DevicePredictor(const DevicePredictor& o, int) : GraphPlan(o), L_(o.L_), dev_(o.dev_), prm_(o.prm_) {}
  static void K(int rc, const char* what) { kern::Check(rc, what); }

  [[noreturn]] static void Refuse(const Node& nd, const std::string& why) { throw std::runtime_error(nd.name + " (" + nd.op + "): " + why + " on the device"); }
  void CheckSupported() const {
    for (int id : order_) {
      const Node& nd = nodes_[id];
      const Attrs& a = nd.attrs;
      if (nd.shape.size() > 8) Refuse(nd, "tensors of more than 8 dimensions are not supported");
      if (nd.op == "Activation") {
        if (UnaryKind(a.Str("act_type", "relu")) < 0) Refuse(nd, "act_type " + a.Str("act_type", "relu") + " is not supported");
      } else if (nd.op == "LeakyReLU") {
        const std::string t = a.Str("act_type", "leaky");
        if (t != "leaky" && t != "elu") Refuse(nd, "LeakyReLU act_type " + t + " is not supported");
      } else if (nd.op == "BatchNorm") {
        for (size_t i = 1; i <= 4; ++i) if (IsInput(In(nd, i))) Refuse(nd, "scale, shift and statistics must come from the parameter file, " + In(nd, i).name + " is an input");
      } else if (nd.op == "Convolution" || nd.op == "FullyConnected") {
        if (Numel(nd.shape) > (int64_t(1) << 31) || Numel(In(nd, 0).shape) > (int64_t(1) << 31)) Refuse(nd, "tensors of 2^31 elements or more are not supported");
      }
    }
  }

  void* Alloc(std::vector<void*>* owner, int64_t floats, kern::Stream s, const char* what) {
    const size_t bytes = static_cast<size_t>(std::max<int64_t>(floats, 1)) * 4;
    void* p = L_->pool_alloc(dev_, bytes, s);
    if (!p) throw std::runtime_error(std::string(what) + ": out of device memory on device " + std::to_string(dev_) + " (" + std::to_string(bytes) + " bytes)");
    owner->push_back(p);
    return p;
  }

  // parameters of the reachable graph, and BatchNorm's folded scale / shift (predict.h Run: scale = gamma / sqrt(var + eps), shift = beta - mean * scale)
  std::shared_ptr<DeviceParams> Upload() {
    auto d = std::make_shared<DeviceParams>();
    d->L = L_; d->dev = dev_;
    kern::Stream s = L_->stream(dev_);
    std::vector<std::vector<float>> staged;                 // host sources stay alive until the copies are done
    for (const Node& nd : nodes_) {
      if (nd.op != "null" || nd.storage < 0 || !nd.known || IsInput(nd) || d->ptr.count(nd.name)) continue;
      const std::vector<float>& v = params_->at(nd.name).second;
      float* p = static_cast<float*>(Alloc(&d->allocs, static_cast<int64_t>(v.size()), s, "GXPredCreate"));
      K(L_->memcpy(p, v.data(), v.size() * 4, 1, s), "GXPredCreate: parameter upload");
      d->ptr[nd.name] = p;
    }
    for (int id : order_) {
      const Node& nd = nodes_[id];
      if (nd.op != "BatchNorm") continue;
      const Attrs& a = nd.attrs;
      const Shape& xs = In(nd, 0).shape;
      const int64_t C = xs[Axis(a.Int("axis", 1), xs.size())];
      const float eps = static_cast<float>(a.Float("eps", 1e-3));
      const bool fix_gamma = a.Bool("fix_gamma", nd.nnvm);
      auto host = [&](size_t i) { return params_->at(In(nd, i).name).second.data(); };
      const float *g = host(1), *b = host(2), *mean = host(3), *var = host(4);
      staged.emplace_back(static_cast<size_t>(2 * C));
      std::vector<float>& ss = staged.back();
      for (int64_t c = 0; c < C; ++c) { ss[c] = (fix_gamma ? 1.f : g[c]) / std::sqrt(var[c] + eps); ss[C + c] = b[c] - mean[c] * ss[c]; }
      float* p = static_cast<float*>(Alloc(&d->allocs, 2 * C, s, "GXPredCreate"));
      K(L_->memcpy(p, ss.data(), ss.size() * 4, 1, s), "GXPredCreate: BatchNorm upload");
      d->bn[id] = p;
    }
    K(L_->stream_sync(s), "GXPredCreate: parameter upload");
    return d;
  }

  static bool Depthwise(const Conv& c, const Shape& xs, const Shape& ys) {
    const int64_t C = xs[1], F = ys[1], HW = xs[2] * xs[3], P = ys[2] * ys[3], KK = c.kh * c.kw;
    return c.groups == C && c.groups == F && c.groups > 1 && c.dh == 1 && c.dw == 1 && (HW + KK) * 4 <= 200 * 1024 && (P + KK) * 4 <= 200 * 1024 &&
           (HW + P) * 4 <= 200 * 1024;
  }
  static int64_t ColStride(const Conv& c, int64_t C) { return (C * c.kh * c.kw + 3) / 4 * 4; }     // a multiple of 4 for the TMA GEMM

  // the handle's stream, arena, input buffers and workspace; on failure everything allocated so far is returned
  void Bind() {
    try {
      K(L_->stream_create(dev_, &stream_), "GXPredCreate: stream");
      ptr_.assign(storages_.size(), nullptr);
      float* arena = static_cast<float*>(Alloc(&allocs_, arena_floats_, stream_, "GXPredCreate"));
      K(L_->memset(arena, 0, static_cast<unsigned long long>(std::max<int64_t>(arena_floats_, 1)) * 4, stream_), "GXPredCreate");
      for (size_t i = 0; i < storages_.size(); ++i) if (!storages_[i].external) ptr_[i] = arena + block_offset_[storages_[i].block];
      inputs_.clear();
      for (const Node& nd : nodes_) {
        if (nd.op != "null" || nd.storage < 0 || !nd.known) continue;
        if (IsInput(nd)) {
          const int64_t n = Numel(nd.shape);
          float* p = static_cast<float*>(Alloc(&allocs_, n, stream_, "GXPredCreate"));
          K(L_->memset(p, 0, static_cast<unsigned long long>(n) * 4, stream_), "GXPredCreate");
          inputs_[nd.name] = {p, static_cast<size_t>(n)};
          ptr_[nd.storage] = p;
        } else {
          ptr_[nd.storage] = prm_->ptr.at(nd.name);
        }
      }
      int64_t ws = 0;
      for (int id : order_) {
        const Node& nd = nodes_[id];
        if (nd.op == "Convolution") {
          const Shape& xs = In(nd, 0).shape;
          const Conv c = ConvAttrs(nd);
          if (Depthwise(c, xs, nd.shape)) continue;
          const int64_t rows = xs[0] * nd.shape[2] * nd.shape[3];
          ws = std::max(ws, rows * (ColStride(c, xs[1]) + nd.shape[1]));
        } else if (nd.op == "Pooling" && PoolAttrs(nd, In(nd, 0).shape).type == 0) {
          ws = std::max(ws, Numel(nd.shape));
        }
      }
      ws_ = ws ? static_cast<float*>(Alloc(&allocs_, ws, stream_, "GXPredCreate")) : nullptr;
      K(L_->stream_sync(stream_), "GXPredCreate");
    } catch (...) {
      Release();
      throw;
    }
  }
  // waits for the stream, then returns memory to the pool on the stream it was allocated with
  void Release() {
    if (!stream_) return;
    L_->set_device(dev_);
    L_->stream_sync(stream_);
    if (graph_) L_->graph_destroy(graph_);
    graph_ = nullptr;
    for (void* p : allocs_) L_->pool_free(dev_, p, stream_);
    allocs_.clear();
    L_->stream_destroy(stream_);
    stream_ = nullptr;
  }

  void Capture() {
    K(L_->graph_begin(stream_), "GXPredForward: begin CUDA graph capture");
    try {
      RunAll();
    } catch (...) {
      void* g = nullptr;
      L_->graph_end(stream_, &g);
      if (g) L_->graph_destroy(g);
      throw;
    }
    void* g = nullptr;
    K(L_->graph_end(stream_, &g), "GXPredForward: CUDA graph capture");
    graph_ = g;
  }
  void RunAll() { for (int id : order_) RunOp(id); }

  float* Ptr(const Node& nd, size_t i) const { return ptr_[In(nd, i).storage]; }
  void Map(int kind, const float* x, float* y, int64_t n, float a = 0.f, float b = 0.f) { K(L_->map_fwd(kind, x, y, n, a, b, stream_), "elementwise map"); }
  static void SplitAxis(const Shape& s, int64_t ax, int64_t* outer, int64_t* c, int64_t* inner) {
    *outer = 1; *inner = 1; *c = s[ax];
    for (int64_t i = 0; i < ax; ++i) *outer *= s[i];
    for (size_t i = ax + 1; i < s.size(); ++i) *inner *= s[i];
  }
  void Softmax(const float* x, float* y, int64_t outer, int64_t C, int64_t inner, bool log) {
    K(L_->softmax_fwd(x, y, outer, static_cast<int>(C), inner, log ? 1 : 0, stream_), "softmax");
  }
  void SoftmaxAxis(const Shape& s, const float* x, float* y, int64_t axis, bool log) {
    int64_t outer, C, inner;
    SplitAxis(s, Axis(axis, s.size()), &outer, &C, &inner);
    Softmax(x, y, outer, C, inner, log);
  }
  // D = A[M, Kd] . B[N, Kd]^T (+ bias), row-major: the tcgen05 GEMM, or the CUDA-core GEMM for operands that miss the TMA alignment
  void Gemm(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int64_t N, int64_t Kd, float* D, int64_t ldd, const float* bias) {
    int rc = L_->gemm_tf32(A, lda, 0, B, ldb, 0, static_cast<int>(M), static_cast<int>(N), static_cast<int>(Kd), D, ldd, bias, nullptr, 0, nullptr, 0, 0, 0, 0,
                           1.f, 1, stream_);
    if (rc < 0) rc = L_->gemm_simt(A, lda, 0, B, ldb, 0, static_cast<int>(M), static_cast<int>(N), static_cast<int>(Kd), D, ldd, bias, nullptr, 0, nullptr, 0, 0,
                                   0, 0, 1.f, stream_);
    K(rc, "GEMM");
  }
  static void BcastStrides(const Shape& out, const Shape& in, long long* st) {
    long long acc = 1;
    for (int i = static_cast<int>(in.size()) - 1, o = static_cast<int>(out.size()) - 1; o >= 0; --i, --o) {
      const int64_t d = i >= 0 ? in[i] : 1;
      st[o] = d == 1 ? 0 : acc;
      acc *= d;
    }
  }

  // one planned operator: the device twin of predict.h Predictor::Run
  void RunOp(int id) {
    const Node& nd = nodes_[id];
    const std::string& op = nd.op;
    const Attrs& a = nd.attrs;
    if (IsView(op)) return;
    float* y = ptr_[nd.storage];
    const int64_t n = Numel(nd.shape);
    const float* x = Ptr(nd, 0);
    const Shape& xs = In(nd, 0).shape;
    int k;
    if (op == "FullyConnected") {
      const Shape& w = In(nd, 1).shape;
      Gemm(x, w[1], Ptr(nd, 1), w[1], n / w[0], w[0], w[1], y, w[0], a.Bool("no_bias", false) ? nullptr : Ptr(nd, 2));
    } else if (op == "Convolution") {
      RunConv(nd, x, xs, y);
    } else if (op == "Pooling") {
      const Pool p = PoolAttrs(nd, xs);
      K(L_->pool_fwd(p.type, x, y, p.type == 0 ? reinterpret_cast<int*>(ws_) : nullptr, xs[0] * xs[1], (int)xs[2], (int)xs[3], (int)nd.shape[2], (int)nd.shape[3],
                     (int)p.kh, (int)p.kw, (int)p.sh, (int)p.sw, (int)p.ph, (int)p.pw, p.count_pad ? 1 : 0, stream_), "Pooling");
    } else if (op == "Activation") {
      Map(UnaryKind(a.Str("act_type", "relu")), x, y, n);
    } else if (op == "LeakyReLU") {
      Map(a.Str("act_type", "leaky") == "leaky" ? 11 : 12, x, y, n, static_cast<float>(a.Float("slope", 0.25)));
    } else if ((k = UnaryKind(op)) >= 0) {
      Map(k, x, y, n);
    } else if (op == "clip") {
      Map(13, x, y, n, static_cast<float>(a.Float("a_min", -std::numeric_limits<float>::infinity())),
          static_cast<float>(a.Float("a_max", std::numeric_limits<float>::infinity())));
    } else if (op == "LogisticRegressionOutput") {
      Map(1, x, y, n);
    } else if (op == "BatchNorm") {
      int64_t outer, C, inner;
      SplitAxis(xs, Axis(a.Int("axis", 1), xs.size()), &outer, &C, &inner);
      const float* ss = prm_->bn.at(id);
      K(L_->channel_affine(x, y, ss, ss + C, outer, static_cast<int>(C), inner, stream_), "BatchNorm");
    } else if (op == "Concat" || op == "concat") {
      int64_t outer, C, inner;
      SplitAxis(nd.shape, Axis(a.Int("dim", 1), nd.shape.size()), &outer, &C, &inner);
      const int64_t ax = Axis(a.Int("dim", 1), nd.shape.size());
      int64_t at = 0;
      for (size_t j = 0; j < nd.inputs.size(); ++j) {
        const int64_t c = In(nd, j).shape[ax];
        K(L_->strided_copy(Ptr(nd, j), y + at * inner, outer, c * inner, c * inner, C * inner, 0, stream_), "Concat");
        at += c;
      }
    } else if (op == "softmax" || op == "log_softmax") {
      SoftmaxAxis(nd.shape, x, y, a.Int("axis", -1), op == "log_softmax");
    } else if (op == "SoftmaxOutput" || op == "Softmax") {
      SoftmaxAxis(nd.shape, x, y, nd.shape.size() < 2 ? 0 : (a.Bool("preserve_shape", false) ? -1 : 1), false);
    } else if (op == "SoftmaxActivation") {
      if (a.Str("mode", "instance") == "channel" || nd.shape.size() <= 2) SoftmaxAxis(nd.shape, x, y, nd.shape.size() < 2 ? 0 : 1, false);
      else Softmax(x, y, nd.shape[0], n / nd.shape[0], 1, false);                     // instance: over everything but the batch axis
    } else if (op == "transpose") {
      auto axes = a.Tuple("axes", {});
      const size_t r = xs.size();
      if (axes.empty()) for (size_t i = 0; i < r; ++i) axes.push_back(static_cast<int64_t>(r - 1 - i));
      long long dims[8]; int ax[8];
      for (size_t i = 0; i < r; ++i) { dims[i] = xs[i]; ax[i] = static_cast<int>(Axis(axes[i], r)); }
      K(L_->transpose(x, y, static_cast<int>(r), dims, ax, stream_), "transpose");
    } else if (op == "Embedding") {
      const Shape& w = In(nd, 1).shape;
      K(L_->embedding_fwd(x, Ptr(nd, 1), y, Numel(xs), w[0], w[1], stream_), "Embedding");
    } else if ((k = BinaryKind(op)) >= 0) {
      long long dims[8], ls[8], rs[8];
      for (size_t d = 0; d < nd.shape.size(); ++d) dims[d] = nd.shape[d];
      BcastStrides(nd.shape, xs, ls); BcastStrides(nd.shape, In(nd, 1).shape, rs);
      K(L_->binary_fwd(k, x, Ptr(nd, 1), y, static_cast<int>(nd.shape.size()), dims, ls, rs, stream_), op.c_str());
    } else if ((k = ScalarKind(op)) >= 0) {
      Map(14 + k, x, y, n, static_cast<float>(a.Float("scalar", 0.0)));
    } else if (op == "add_n" || op == "ElementWiseSum") {
      std::vector<const float*> ins;
      for (size_t j = 0; j < nd.inputs.size(); ++j) ins.push_back(Ptr(nd, j));
      if (ins.size() <= 8) { K(L_->nary_sum(y, ins.data(), static_cast<int>(ins.size()), n, stream_), "add_n"); return; }
      K(L_->memcpy(y, ins[0], static_cast<unsigned long long>(n) * 4, 3, stream_), "add_n");
      for (size_t j = 1; j < ins.size(); ++j) K(L_->axpy(y, ins[j], 1.f, n, stream_), "add_n");
    } else {
      throw std::runtime_error("operator " + op + " has no device kernel");
    }
  }

  // im2col (dilated when asked) into the workspace, one GEMM per group into rows [N * OH * OW][F], rows -> NCHW; depthwise kernels where eligible
  void RunConv(const Node& nd, const float* x, const Shape& xs, float* y) {
    const Conv c = ConvAttrs(nd);
    const float* w = Ptr(nd, 1);
    const float* bias = nd.attrs.Bool("no_bias", false) ? nullptr : Ptr(nd, 2);
    const int64_t B = xs[0], C = xs[1], H = xs[2], W = xs[3], F = nd.shape[1], P = nd.shape[2] * nd.shape[3];
    if (Depthwise(c, xs, nd.shape)) {
      K(L_->depthwise_fwd(x, w, bias, y, (int)B, (int)C, (int)H, (int)W, (int)c.kh, (int)c.kw, (int)c.sh, (int)c.sw, (int)c.ph, (int)c.pw, 0, stream_),
        "depthwise convolution");
      return;
    }
    const int64_t G = c.groups, Cg = C / G, Fg = F / G, Kg = Cg * c.kh * c.kw, ldc = ColStride(c, C);
    float* col = ws_;
    float* rows = ws_ + B * P * ldc;
    if (c.dh == 1 && c.dw == 1)
      K(L_->im2col(x, col, (int)B, (int)C, (int)H, (int)W, (int)c.kh, (int)c.kw, (int)c.sh, (int)c.sw, (int)c.ph, (int)c.pw, (int)ldc, stream_), "im2col");
    else
      K(L_->im2col_dilated(x, col, (int)B, (int)C, (int)H, (int)W, (int)c.kh, (int)c.kw, (int)c.sh, (int)c.sw, (int)c.ph, (int)c.pw, (int)c.dh, (int)c.dw,
                           (int)ldc, stream_), "dilated im2col");
    for (int64_t g = 0; g < G; ++g) Gemm(col + g * Kg, ldc, w + g * Fg * Kg, Kg, B * P, Fg, Kg, rows + g * Fg, F, bias ? bias + g * Fg : nullptr);
    K(L_->rows_to_nchw(rows, y, (int)B, (int)F, (int)P, F, 0, stream_), "rows to NCHW");
  }
};

}  // namespace predict
}  // namespace gxrt
