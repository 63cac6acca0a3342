// Native symbolic graph: the data structure behind the GXSymbol* C API (c_api_graph.cc) and the host training executor (train_exec.h).
//
// Parity: include/mxnet/c_api.h:1040-1530 (MXSymbol*: atomic-symbol creators, Variable / Group / Compose, attributes, List{Arguments,Outputs,
// AuxiliaryStates}, GetInternals / GetOutput / GetChildren, InferShape(+Partial) / InferType, JSON save / load) over what nnvm::Symbol /
// nnvm::Graph provide there (3rdparty/tvm/nnvm/include/nnvm/symbolic.h, src/nnvm/legacy_json_util.cc).  Design differences:
//   * nodes are immutable once composed and shared by reference (a Symbol is a list of (node, output) heads), so Copy is a pointer copy of the
//     heads plus a deep copy only where a later Compose could alias (atomic symbols are deep-copied on Copy);
//   * the operator table is one static array of OpDef records (input names as a function of the attributes, trailing auxiliary states,
//     documented parameters) instead of nnvm's attribute-function registry; shape rules live in ONE function per op that both infers the
//     output and back-fills unknown parameter / label shapes (the reference runs separate forward and backward InferShape passes to a fix point);
//   * both JSON dialects load (the reference's nnvm JSON and this framework's `geomx_b200-symbol-1`); saving writes the nnvm dialect, which the
//     Python front end (symbol.py::load_json), the native predictor (predict.h) and MXNet itself read.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <set>
#include <sstream>
#include <string>
#include <unordered_map>
#include <vector>

#include "predict.h"

namespace gxrt {
namespace graph {

using predict::JParser;
using predict::JValue;
using predict::Numel;
using predict::Shape;
using predict::ShapeStr;
using AttrMap = std::map<std::string, std::string>;

// ------------------------------------------------------------------------------------------------ string-valued attributes (nnvm style)
inline bool IsUserKey(const std::string& k) { return k.size() > 4 && k.compare(0, 2, "__") == 0 && k.compare(k.size() - 2, 2, "__") == 0; }

struct AttrView {
  const AttrMap* m;
  explicit AttrView(const AttrMap& a) : m(&a) {}
  const std::string* Raw(const std::string& k) const {
    auto it = m->find(k);
    return (it == m->end() || it->second.empty() || it->second == "None") ? nullptr : &it->second;
  }
  bool Has(const std::string& k) const { return Raw(k) != nullptr; }
  double Float(const std::string& k, double def) const {
    const std::string* v = Raw(k);
    if (!v) return def;
    if (*v == "True" || *v == "true") return 1;
    if (*v == "False" || *v == "false") return 0;
    try { size_t pos = 0; const double d = std::stod(*v, &pos); return d; } catch (...) {}
    throw std::runtime_error("attribute " + k + "=" + *v + " is not a number");
  }
  int64_t Int(const std::string& k, int64_t def) const { return static_cast<int64_t>(std::llround(Float(k, static_cast<double>(def)))); }
  bool Bool(const std::string& k, bool def) const {
    const std::string* v = Raw(k);
    if (!v) return def;
    return *v == "True" || *v == "true" || *v == "1";
  }
  std::string Str(const std::string& k, const std::string& def) const {
    const std::string* v = Raw(k);
    if (!v) return def;
    if (v->size() >= 2 && (v->front() == '\'' || v->front() == '"') && v->back() == v->front()) return v->substr(1, v->size() - 2);
    return *v;
  }
  std::vector<int64_t> Tuple(const std::string& k, std::vector<int64_t> def) const {
    const std::string* v = Raw(k);
    if (!v) return def;
    std::vector<int64_t> out;
    const std::string& s = *v;
    size_t i = 0;
    while (i < s.size()) {
      if (std::isdigit(static_cast<unsigned char>(s[i])) || (s[i] == '-' && i + 1 < s.size() && std::isdigit(static_cast<unsigned char>(s[i + 1])))) {
        size_t j = i + 1;
        while (j < s.size() && std::isdigit(static_cast<unsigned char>(s[j]))) ++j;
        out.push_back(std::stoll(s.substr(i, j - i)));
        i = j;
      } else { ++i; }
    }
    return out.empty() && s.find('(') == std::string::npos && s.find('[') == std::string::npos ? def : out;
  }
};

inline std::string TupleStr(const Shape& s) {
  std::string o = "(";
  for (size_t i = 0; i < s.size(); ++i) o += (i ? ", " : "") + std::to_string(s[i]);
  if (s.size() == 1) o += ",";
  return o + ")";
}

// ------------------------------------------------------------------------------------------------ nodes
struct Node;
struct Entry { std::shared_ptr<Node> node; int index = 0; };
struct Node {
  std::string op;                    // "null" = variable
  std::string name;
  AttrMap attrs;                     // operator parameters and __user__ attributes, string-valued
  std::vector<Entry> inputs;         // regular inputs followed by auxiliary states
  bool composed = true;              // false: an atomic symbol whose inputs are still to be supplied by Compose
};
struct Symbol { std::vector<Entry> outputs; };

// ------------------------------------------------------------------------------------------------ operator table
struct ParamDoc { const char* name; const char* type; const char* doc; };
struct OpDef {
  const char* name;
  // names of the tensor inputs for these attributes (regular inputs, then auxiliary states)
  std::vector<std::string> (*inputs)(const AttrView&);
  int num_aux;                       // how many TRAILING inputs are auxiliary states
  const char* key_var_num_args;      // the attribute that carries the input count of variadic operators ("" otherwise)
  const char* doc;
  std::vector<ParamDoc> params;
};

namespace detail {
inline std::vector<std::string> InData(const AttrView&) { return {"data"}; }
inline std::vector<std::string> InLR(const AttrView&) { return {"lhs", "rhs"}; }
inline std::vector<std::string> InDataLabel(const AttrView&) { return {"data", "label"}; }
inline std::vector<std::string> InWB(const AttrView& a) { return a.Bool("no_bias", false) ? std::vector<std::string>{"data", "weight"} : std::vector<std::string>{"data", "weight", "bias"}; }
inline std::vector<std::string> InBN(const AttrView&) { return {"data", "gamma", "beta", "moving_mean", "moving_var"}; }
inline std::vector<std::string> InEmb(const AttrView&) { return {"data", "weight"}; }
inline std::vector<std::string> InGB(const AttrView&) { return {"data", "gamma", "beta"}; }
inline std::vector<std::string> InDeconv(const AttrView& a) { return a.Bool("no_bias", true) ? std::vector<std::string>{"data", "weight"} : std::vector<std::string>{"data", "weight", "bias"}; }
inline std::vector<std::string> InTake(const AttrView&) { return {"a", "indices"}; }
inline std::vector<std::string> InPick(const AttrView&) { return {"data", "index"}; }
inline std::vector<std::string> InWhere(const AttrView&) { return {"condition", "x", "y"}; }
inline std::vector<std::string> InIdx(const AttrView&) { return {"indices"}; }
inline std::vector<std::string> InSGD(const AttrView&) { return {"weight", "grad"}; }
inline std::vector<std::string> InSGDMom(const AttrView&) { return {"weight", "grad", "mom"}; }
inline std::vector<std::string> InAdam(const AttrView&) { return {"weight", "grad", "mean", "var"}; }
inline std::vector<std::string> InVar(const AttrView& a) {
  std::vector<std::string> v;
  const int64_t n = a.Int("num_args", 0);
  if (n < 0 || n > 4096) throw std::runtime_error("num_args out of range");
  for (int64_t i = 0; i < n; ++i) v.push_back("arg" + std::to_string(i));
  return v;
}
}  // namespace detail

inline const std::vector<OpDef>& OpTable() {
  using namespace detail;
  static const std::vector<OpDef> t = [] {
    std::vector<OpDef> v;
    const std::vector<ParamDoc> none;
    v.push_back({"FullyConnected", InWB, 0, "", "y = x . W^T + b over the flattened trailing axes (src/operator/nn/fully_connected.cc)",
                 {{"num_hidden", "int, required", "number of output units"}, {"no_bias", "boolean, optional, default=0", "disable the bias"},
                  {"flatten", "boolean, optional, default=1", "collapse all axes but the first"}}});
    v.push_back({"Convolution", InWB, 0, "", "2-D NCHW convolution (src/operator/nn/convolution.cc)",
                 {{"kernel", "Shape(tuple), required", "window (h, w)"}, {"num_filter", "int, required", "output channels"},
                  {"stride", "Shape(tuple), optional, default=(1, 1)", "stride"}, {"pad", "Shape(tuple), optional, default=(0, 0)", "zero padding"},
                  {"dilate", "Shape(tuple), optional, default=(1, 1)", "dilation"}, {"num_group", "int, optional, default=1", "groups"},
                  {"no_bias", "boolean, optional, default=0", "disable the bias"}}});
    v.push_back({"Pooling", InData, 0, "", "2-D max / avg / sum pooling (src/operator/nn/pooling.cc)",
                 {{"kernel", "Shape(tuple), optional", "window"}, {"pool_type", "{'avg', 'max', 'sum'}, optional, default='max'", "reduction"},
                  {"stride", "Shape(tuple), optional, default=(1, 1)", "stride"}, {"pad", "Shape(tuple), optional, default=(0, 0)", "padding"},
                  {"global_pool", "boolean, optional, default=0", "pool over the whole map"},
                  {"pooling_convention", "{'full', 'valid'}, optional, default='valid'", "output size rounding"},
                  {"count_include_pad", "boolean, optional, default=1", "avg divisor counts padding"}}});
    v.push_back({"Activation", InData, 0, "", "elementwise activation (src/operator/nn/activation.cc)",
                 {{"act_type", "{'relu', 'sigmoid', 'softrelu', 'softsign', 'tanh'}, required", "function"}}});
    v.push_back({"LeakyReLU", InData, 0, "", "leaky / elu rectifier (src/operator/leaky_relu.cc)",
                 {{"act_type", "{'elu', 'leaky'}, optional, default='leaky'", "function"}, {"slope", "float, optional, default=0.25", "negative slope"}}});
    v.push_back({"BatchNorm", InBN, 2, "", "batch normalisation with running statistics as auxiliary states (src/operator/nn/batch_norm.cc)",
                 {{"eps", "double, optional, default=0.001", "variance floor"}, {"momentum", "float, optional, default=0.9", "running-average momentum"},
                  {"fix_gamma", "boolean, optional, default=1", "gamma fixed to 1"}, {"use_global_stats", "boolean, optional, default=0", "always use the running statistics"},
                  {"axis", "int, optional, default=1", "channel axis"}}});
    v.push_back({"Dropout", InData, 0, "", "inverted dropout in training mode, identity otherwise (src/operator/nn/dropout.cc)",
                 {{"p", "float, optional, default=0.5", "drop probability"}}});
    v.push_back({"Flatten", InData, 0, "", "collapse all axes but the first", none});
    v.push_back({"Reshape", InData, 0, "", "reshape with the special codes 0, -1, -2, -3 (src/operator/tensor/matrix_op.cc)",
                 {{"shape", "Shape(tuple), required", "target shape"}}});
    v.push_back({"transpose", InData, 0, "", "axis permutation", {{"axes", "Shape(tuple), optional, default=()", "permutation (reverse when empty)"}}});
    v.push_back({"expand_dims", InData, 0, "", "insert an axis of extent 1", {{"axis", "int, required", "position"}}});
    v.push_back({"Concat", InVar, 0, "num_args", "join along one axis (src/operator/nn/concat.cc)",
                 {{"num_args", "int, required", "number of inputs"}, {"dim", "int, optional, default=1", "axis"}}});
    v.push_back({"add_n", InVar, 0, "num_args", "sum of all inputs (src/operator/tensor/elemwise_sum.cc)", {{"num_args", "int, required", "number of inputs"}}});
    v.push_back({"Embedding", InEmb, 0, "", "row lookup (src/operator/tensor/indexing_op.cc)",
                 {{"input_dim", "int, required", "vocabulary"}, {"output_dim", "int, required", "vector width"}}});
    v.push_back({"SoftmaxOutput", InDataLabel, 0, "", "softmax forward, cross-entropy gradient backward (src/operator/softmax_output.cc)",
                 {{"grad_scale", "float, optional, default=1", "gradient scale"}, {"ignore_label", "float, optional, default=-1", "label to skip"},
                  {"use_ignore", "boolean, optional, default=0", "honour ignore_label"}, {"multi_output", "boolean, optional, default=0", "softmax over axis 1 of (n, c, ...)"},
                  {"normalization", "{'batch', 'null', 'valid'}, optional, default='null'", "gradient normalisation"}}});
    v.push_back({"LinearRegressionOutput", InDataLabel, 0, "", "identity forward, (x - y) backward (src/operator/regression_output.cc)", {{"grad_scale", "float, optional, default=1", "gradient scale"}}});
    v.push_back({"LogisticRegressionOutput", InDataLabel, 0, "", "sigmoid forward, (p - y) backward", {{"grad_scale", "float, optional, default=1", "gradient scale"}}});
    v.push_back({"MAERegressionOutput", InDataLabel, 0, "", "identity forward, sign(x - y) backward", {{"grad_scale", "float, optional, default=1", "gradient scale"}}});
    // optimizer steps for imperative use: the output is the updated weight, optimizer states are trailing auxiliary inputs updated in place
    const std::vector<ParamDoc> opt_common = {{"lr", "float, required", "learning rate"}, {"wd", "float, optional, default=0", "weight decay"},
                                              {"rescale_grad", "float, optional, default=1", "gradient scale"},
                                              {"clip_gradient", "float, optional, default=-1", "clip the rescaled gradient to +-value (< 0: off)"}};
    auto with = [&](std::vector<ParamDoc> extra) { std::vector<ParamDoc> p = opt_common; p.insert(p.end(), extra.begin(), extra.end()); return p; };
    v.push_back({"sgd_update", InSGD, 0, "", "w - lr * (clip(rescale_grad * g) + wd * w) (src/operator/optimizer_op.cc)", opt_common});
    v.push_back({"sgd_mom_update", InSGDMom, 1, "", "mom = momentum * mom - lr * (clip(rescale_grad * g) + wd * w); w + mom (src/operator/optimizer_op.cc)",
                 with({{"momentum", "float, optional, default=0", "momentum"}})});
    v.push_back({"adam_update", InAdam, 2, "", "Adam step without bias correction on (weight, grad, mean, var) (src/operator/optimizer_op.cc)",
                 with({{"beta1", "float, optional, default=0.9", "first-moment decay"}, {"beta2", "float, optional, default=0.999", "second-moment decay"},
                       {"epsilon", "float, optional, default=1e-8", "denominator floor"}})});
    v.push_back({"MakeLoss", InData, 0, "", "marks a head as a loss: backward feeds grad_scale (src/operator/make_loss.cc)", {{"grad_scale", "float, optional, default=1", "gradient scale"}}});
    v.push_back({"softmax", InData, 0, "", "softmax along an axis (src/operator/nn/softmax.cc)", {{"axis", "int, optional, default=-1", "axis"}}});
    v.push_back({"log_softmax", InData, 0, "", "log-softmax along an axis", {{"axis", "int, optional, default=-1", "axis"}}});
    v.push_back({"SoftmaxActivation", InData, 0, "", "softmax over axis 1 (legacy name)", none});
    v.push_back({"BlockGrad", InData, 0, "", "identity forward, zero gradient backward", none});
    v.push_back({"identity", InData, 0, "", "copy", none});
    v.push_back({"clip", InData, 0, "", "clamp to [a_min, a_max]", {{"a_min", "float, required", "lower bound"}, {"a_max", "float, required", "upper bound"}}});
    v.push_back({"sum", InData, 0, "", "sum over axes (src/operator/tensor/broadcast_reduce_op_value.cc)",
                 {{"axis", "Shape(tuple), optional, default=()", "axes (all when empty)"}, {"keepdims", "boolean, optional, default=0", "keep reduced axes"}}});
    v.push_back({"mean", InData, 0, "", "mean over axes",
                 {{"axis", "Shape(tuple), optional, default=()", "axes (all when empty)"}, {"keepdims", "boolean, optional, default=0", "keep reduced axes"}}});
    v.push_back({"dot", InLR, 0, "", "matrix product of 2-D operands (src/operator/tensor/dot.cc)",
                 {{"transpose_a", "boolean, optional, default=0", "use lhs^T"}, {"transpose_b", "boolean, optional, default=0", "use rhs^T"}}});
    // ---- second tier: normalisation / transposed convolution / indexing / shape manipulation / more reductions
    v.push_back({"LayerNorm", InGB, 0, "", "normalise over one axis with learned scale and shift (src/operator/nn/layer_norm.cc)",
                 {{"axis", "int, optional, default=-1", "axis"}, {"eps", "float, optional, default=1e-5", "variance floor"}}});
    v.push_back({"InstanceNorm", InGB, 0, "", "normalise every (sample, channel) map (src/operator/instance_norm.cc)", {{"eps", "float, optional, default=0.001", "variance floor"}}});
    v.push_back({"L2Normalization", InData, 0, "", "divide by the L2 norm per instance / channel / spatial position (src/operator/l2_normalization.cc)",
                 {{"mode", "{'channel', 'instance', 'spatial'}, optional, default='instance'", "group"}, {"eps", "float, optional, default=1e-10", "floor"}}});
    v.push_back({"LRN", InData, 0, "", "local response normalisation across channels (src/operator/nn/lrn.cc)",
                 {{"nsize", "int, required", "window"}, {"alpha", "float, optional, default=0.0001", "scale"}, {"beta", "float, optional, default=0.75", "exponent"},
                  {"knorm", "float, optional, default=2", "offset"}}});
    v.push_back({"Deconvolution", InDeconv, 0, "", "2-D transposed convolution (src/operator/nn/deconvolution.cc)",
                 {{"kernel", "Shape(tuple), required", "window"}, {"num_filter", "int, required", "output channels"}, {"stride", "Shape(tuple), optional", "stride"},
                  {"pad", "Shape(tuple), optional", "padding"}, {"adj", "Shape(tuple), optional", "output adjustment"}, {"dilate", "Shape(tuple), optional", "dilation"},
                  {"num_group", "int, optional, default=1", "groups"}, {"no_bias", "boolean, optional, default=1", "disable the bias"}}});
    v.push_back({"UpSampling", InVar, 0, "num_args", "nearest-neighbour upsampling (src/operator/nn/upsampling.cc)",
                 {{"scale", "int, required", "factor"}, {"sample_type", "{'nearest'}, required", "method"}, {"num_args", "int, required", "number of inputs (1)"}}});
    v.push_back({"SliceChannel", InData, 0, "", "split into num_outputs equal parts along an axis — the multi-output operator of the table (src/operator/slice_channel.cc)",
                 {{"num_outputs", "int, required", "number of parts"}, {"axis", "int, optional, default=1", "axis"}, {"squeeze_axis", "boolean, optional, default=0", "drop the axis when the parts have extent 1"}}});
    v.push_back({"softmax_cross_entropy", InDataLabel, 0, "", "summed cross entropy of softmax(data) against integer labels (src/operator/loss_binary_op.cc)", none});
    v.push_back({"smooth_l1", InData, 0, "", "Huber-like loss with transition at 1/sigma^2", {{"scalar", "float, required", "sigma"}}});
    v.push_back({"slice_axis", InData, 0, "", "slice along one axis (src/operator/tensor/matrix_op.cc)",
                 {{"axis", "int, required", "axis"}, {"begin", "int, required", "first index"}, {"end", "int or None, required", "one past the last index"}}});
    v.push_back({"slice", InData, 0, "", "slice by per-axis begin / end (None = full range)", {{"begin", "Shape(tuple), required", "starts"}, {"end", "Shape(tuple), required", "stops"}}});
    v.push_back({"SwapAxis", InData, 0, "", "exchange two axes", {{"dim1", "int, optional, default=0", "axis"}, {"dim2", "int, optional, default=0", "axis"}}});
    v.push_back({"tile", InData, 0, "", "repeat the whole array", {{"reps", "Shape(tuple), required", "repetitions per axis"}}});
    v.push_back({"repeat", InData, 0, "", "repeat elements along an axis", {{"repeats", "int, required", "count"}, {"axis", "int, required", "axis"}}});
    v.push_back({"Pad", InData, 0, "", "pad with a constant, the edge value or a reflection (src/operator/pad.cc)",
                 {{"mode", "{'constant', 'edge', 'reflect'}, required", "fill"}, {"pad_width", "Shape(tuple), required", "(before, after) per axis"},
                  {"constant_value", "double, optional, default=0", "fill value"}}});
    v.push_back({"squeeze", InData, 0, "", "drop axes of extent 1", {{"axis", "Shape(tuple), optional", "axes (all when absent)"}}});
    v.push_back({"broadcast_to", InData, 0, "", "broadcast to a shape (0 keeps the input extent)", {{"shape", "Shape(tuple), required", "target"}}});
    v.push_back({"broadcast_axis", InData, 0, "", "broadcast axes of extent 1", {{"axis", "Shape(tuple), required", "axes"}, {"size", "Shape(tuple), required", "extents"}}});
    v.push_back({"reverse", InData, 0, "", "reverse along axes", {{"axis", "Shape(tuple), required", "axes"}}});
    v.push_back({"take", InTake, 0, "", "gather slices along an axis, indices clipped (src/operator/tensor/indexing_op.cc)", {{"axis", "int, optional, default=0", "axis"}}});
    v.push_back({"pick", InPick, 0, "", "one element per position along an axis", {{"axis", "int, optional, default=-1", "axis"}, {"keepdims", "boolean, optional, default=0", "keep the axis"}}});
    v.push_back({"one_hot", InIdx, 0, "", "one-hot encode indices", {{"depth", "int, required", "classes"}, {"on_value", "double, optional, default=1", "hot"}, {"off_value", "double, optional, default=0", "cold"}}});
    v.push_back({"where", InWhere, 0, "", "x where condition != 0, else y", none});
    v.push_back({"Cast", InData, 0, "", "dtype conversion (the host executor computes in float32)", {{"dtype", "{'float32'}, required", "target dtype"}}});
    for (const char* n : {"max", "min", "prod", "norm"})
      v.push_back({n, InData, 0, "", "reduction over axes (norm: L2)", {{"axis", "Shape(tuple), optional, default=()", "axes (all when empty)"}, {"keepdims", "boolean, optional, default=0", "keep reduced axes"}}});
    for (const char* n : {"argmax", "argmin"})
      v.push_back({n, InData, 0, "", "index of the extreme value along an axis (no gradient)", {{"axis", "int, required", "axis"}, {"keepdims", "boolean, optional, default=0", "keep the axis"}}});
    for (const char* n : {"broadcast_power", "broadcast_equal", "broadcast_not_equal", "broadcast_greater", "broadcast_greater_equal", "broadcast_lesser", "broadcast_lesser_equal"})
      v.push_back({n, InLR, 0, "", "binary power / comparison (1.0 or 0.0) with numpy broadcasting", none});
    for (const char* n : {"_maximum_scalar", "_minimum_scalar", "_rpower_scalar"})
      v.push_back({n, InData, 0, "", "max / min / scalar ** x with a scalar", {{"scalar", "float, required", "the scalar"}}});
    for (const char* n : {"sin", "cos", "tan", "arcsin", "arccos", "arctan", "sinh", "cosh", "log1p", "expm1", "log2", "log10", "rsqrt", "reciprocal", "cbrt", "erf",
                          "floor", "ceil", "round", "sign"})
      v.push_back({n, InData, 0, "", "elementwise function (src/operator/tensor/elemwise_unary_op_{basic,trig}.cc)", none});
    for (const char* n : {"elemwise_add", "elemwise_sub", "elemwise_mul", "elemwise_div", "broadcast_add", "broadcast_sub", "broadcast_mul", "broadcast_div",
                          "broadcast_maximum", "broadcast_minimum"})
      v.push_back({n, InLR, 0, "", "binary arithmetic with numpy broadcasting (src/operator/tensor/elemwise_binary_broadcast_op_basic.cc)", none});
    for (const char* n : {"_plus_scalar", "_minus_scalar", "_rminus_scalar", "_mul_scalar", "_div_scalar", "_rdiv_scalar", "_power_scalar"})
      v.push_back({n, InData, 0, "", "arithmetic with a scalar (src/operator/tensor/elemwise_binary_scalar_op_basic.cc)", {{"scalar", "float, required", "the scalar"}}});
    for (const char* n : {"relu", "sigmoid", "tanh", "exp", "log", "sqrt", "abs", "negative", "square", "softsign"})
      v.push_back({n, InData, 0, "", "elementwise function (src/operator/tensor/elemwise_unary_op_basic.cc)", none});
    return v;
  }();
  return t;
}

// aliases of the reference's registry (capitalised legacy names, underscore forms written by older front ends)
inline std::string CanonicalOp(const std::string& op) {
  static const std::map<std::string, std::string> alias = {
      {"flatten", "Flatten"}, {"reshape", "Reshape"}, {"concat", "Concat"}, {"ElementWiseSum", "add_n"}, {"Softmax", "SoftmaxOutput"}, {"stop_gradient", "BlockGrad"},
      {"_copy", "identity"}, {"make_loss", "MakeLoss"}, {"_plus", "elemwise_add"}, {"_Plus", "elemwise_add"}, {"_add", "elemwise_add"}, {"_minus", "elemwise_sub"},
      {"_Minus", "elemwise_sub"}, {"_sub", "elemwise_sub"}, {"_mul", "elemwise_mul"}, {"_Mul", "elemwise_mul"}, {"_div", "elemwise_div"}, {"_Div", "elemwise_div"},
      {"broadcast_plus", "broadcast_add"}, {"broadcast_minus", "broadcast_sub"}, {"_maximum", "broadcast_maximum"}, {"_minimum", "broadcast_minimum"},
      {"_PlusScalar", "_plus_scalar"}, {"_MinusScalar", "_minus_scalar"}, {"_RMinusScalar", "_rminus_scalar"}, {"_MulScalar", "_mul_scalar"},
      {"_DivScalar", "_div_scalar"}, {"_RDivScalar", "_rdiv_scalar"}, {"_PowerScalar", "_power_scalar"}, {"_MaximumScalar", "_maximum_scalar"},
      {"_MinimumScalar", "_minimum_scalar"}, {"_RPowerScalar", "_rpower_scalar"}, {"_power", "broadcast_power"}, {"_Power", "broadcast_power"}, {"swapaxes", "SwapAxis"},
      {"pad", "Pad"}, {"cast", "Cast"}, {"flip", "reverse"}, {"_equal", "broadcast_equal"}, {"_not_equal", "broadcast_not_equal"}, {"_greater", "broadcast_greater"},
      {"_greater_equal", "broadcast_greater_equal"}, {"_lesser", "broadcast_lesser"}, {"_lesser_equal", "broadcast_lesser_equal"}, {"max_axis", "max"}, {"min_axis", "min"},
      {"sum_axis", "sum"}, {"split", "SliceChannel"}};
  auto it = alias.find(op);
  return it == alias.end() ? op : it->second;
}
inline const OpDef* FindOp(const std::string& op) {
  const std::string c = CanonicalOp(op);
  for (auto& d : OpTable()) if (c == d.name) return &d;
  return nullptr;
}
inline const OpDef& GetOp(const std::string& op) {
  const OpDef* d = FindOp(op);
  if (!d) throw std::runtime_error("operator " + op + " is not registered in the native graph runtime");
  return *d;
}

// visible outputs of a node: 1 for every operator of the table except SliceChannel (all outputs of one node have the same shape)
inline int NumOutputs(const Node& n) {
  if (n.op != "SliceChannel") return 1;
  const int64_t k = AttrView(n.attrs).Int("num_outputs", 0);
  if (k < 1 || k > 4096) throw std::runtime_error(n.name + ": num_outputs must be in 1..4096");
  return static_cast<int>(k);
}

// ------------------------------------------------------------------------------------------------ construction
inline std::string AutoName(const std::string& op) {
  static std::mutex mu;
  static std::map<std::string, int> counter;
  std::string base;
  for (char c : op) base.push_back(static_cast<char>(std::tolower(static_cast<unsigned char>(c))));
  std::lock_guard<std::mutex> lk(mu);
  return base + std::to_string(counter[base]++);
}

inline Symbol Variable(const std::string& name) {
  auto n = std::make_shared<Node>();
  n->op = "null"; n->name = name;
  return Symbol{{Entry{n, 0}}};
}

inline Symbol CreateAtomic(const std::string& op, const AttrMap& attrs) {
  const OpDef& d = GetOp(op);
  auto n = std::make_shared<Node>();
  n->op = d.name; n->attrs = attrs; n->composed = false;
  d.inputs(AttrView(n->attrs));        // validates num_args & co. early
  Symbol out;
  const int k = NumOutputs(*n);
  for (int i = 0; i < k; ++i) out.outputs.push_back(Entry{n, i});
  return out;
}

inline Symbol Group(const std::vector<Symbol>& parts) {
  Symbol g;
  for (auto& p : parts) for (auto& e : p.outputs) g.outputs.push_back(e);
  return g;
}

// Supplies the inputs of an atomic symbol: positional `args` and / or keyword `kwargs`; inputs that are not given become variables named
// `<name>_<input>` (nnvm Symbol::Compose + the front ends' auto-variable rule, python/mxnet/symbol/symbol.py).
inline void Compose(Symbol* s, const std::string& name, const std::vector<Symbol>& args, const std::vector<std::pair<std::string, Symbol>>& kwargs) {
  if (s->outputs.empty() || s->outputs[0].node->composed || s->outputs[0].node->op == "null") throw std::runtime_error("Compose: not an atomic symbol");
  for (auto& e : s->outputs) if (e.node != s->outputs[0].node) throw std::runtime_error("Compose: not an atomic symbol");
  Node& n = *s->outputs[0].node;
  const OpDef& d = GetOp(n.op);
  n.name = name.empty() ? AutoName(n.op) : name;
  if (*d.key_var_num_args && !AttrView(n.attrs).Has(d.key_var_num_args)) n.attrs[d.key_var_num_args] = std::to_string(args.size() + kwargs.size());
  const std::vector<std::string> names = d.inputs(AttrView(n.attrs));
  if (args.size() > names.size()) throw std::runtime_error(n.name + " (" + n.op + "): " + std::to_string(args.size()) + " positional inputs given, the operator takes " + std::to_string(names.size()));
  n.inputs.assign(names.size(), Entry{});
  auto single = [&](const Symbol& a, const std::string& what) {
    if (a.outputs.size() != 1) throw std::runtime_error(n.name + ": input " + what + " must be a single-output symbol");
    if (!a.outputs[0].node->composed) throw std::runtime_error(n.name + ": input " + what + " is an atomic symbol that was never composed");
    return a.outputs[0];
  };
  for (size_t i = 0; i < args.size(); ++i) n.inputs[i] = single(args[i], names[i]);
  for (auto& kv : kwargs) {
    auto it = std::find(names.begin(), names.end(), kv.first);
    if (it == names.end()) throw std::runtime_error(n.name + " (" + n.op + "): no input named " + kv.first);
    Entry& slot = n.inputs[it - names.begin()];
    if (slot.node) throw std::runtime_error(n.name + ": input " + kv.first + " given twice");
    slot = single(kv.second, kv.first);
  }
  for (size_t i = 0; i < names.size(); ++i) if (!n.inputs[i].node) n.inputs[i] = Variable(n.name + "_" + names[i]).outputs[0];
  n.composed = true;
}

inline Symbol Copy(const Symbol& s) {
  Symbol c = s;
  std::map<Node*, std::shared_ptr<Node>> fresh;
  for (auto& e : c.outputs) if (!e.node->composed) {
    auto& f = fresh[e.node.get()];
    if (!f) f = std::make_shared<Node>(*e.node);
    e.node = f;
  }
  return c;
}

// ------------------------------------------------------------------------------------------------ traversal
// nodes reachable from the heads in dependency order (inputs before consumers, first-visit order of a left-to-right DFS = nnvm's DFSVisit)
inline std::vector<Node*> Topo(const Symbol& s) {
  std::vector<Node*> order;
  std::set<Node*> seen;
  struct Frame { Node* n; size_t next; };
  std::vector<Frame> st;
  for (auto& h : s.outputs) {
    if (!h.node) throw std::runtime_error("symbol has an empty head");
    if (seen.insert(h.node.get()).second) st.push_back({h.node.get(), 0});
    while (!st.empty()) {
      Frame& f = st.back();
      if (f.next < f.n->inputs.size()) {
        Node* c = f.n->inputs[f.next++].node.get();
        if (!c) throw std::runtime_error(f.n->name + ": atomic symbol used before Compose");
        if (seen.insert(c).second) st.push_back({c, 0});
      } else { order.push_back(f.n); st.pop_back(); }
    }
  }
  return order;
}

inline std::set<Node*> AuxNodes(const std::vector<Node*>& order) {
  std::set<Node*> aux;
  for (Node* n : order) {
    if (n->op == "null") continue;
    const int na = GetOp(n->op).num_aux;
    for (int i = 0; i < na; ++i) { Node* a = n->inputs[n->inputs.size() - na + i].node.get(); if (a->op == "null") aux.insert(a); }
  }
  return aux;
}
inline std::vector<std::string> ListArguments(const Symbol& s) {
  const auto order = Topo(s); const auto aux = AuxNodes(order);
  std::vector<std::string> out;
  for (Node* n : order) if (n->op == "null" && !aux.count(n)) out.push_back(n->name);
  return out;
}
inline std::vector<std::string> ListAuxiliaryStates(const Symbol& s) {
  const auto order = Topo(s); const auto aux = AuxNodes(order);
  std::vector<std::string> out;
  for (Node* n : order) if (aux.count(n)) out.push_back(n->name);
  return out;
}
inline std::string OutputName(const Entry& e) {
  if (e.node->op == "null") return e.node->name;
  return NumOutputs(*e.node) > 1 ? e.node->name + "_output" + std::to_string(e.index) : e.node->name + "_output";
}
inline std::vector<std::string> ListOutputs(const Symbol& s) {
  std::vector<std::string> out;
  for (auto& e : s.outputs) out.push_back(OutputName(e));
  return out;
}
inline Symbol GetInternals(const Symbol& s) {
  Symbol r;
  std::map<Node*, std::shared_ptr<Node>> owner;
  std::function<void(const Entry&)> own = [&](const Entry& e) { if (owner.emplace(e.node.get(), e.node).second) for (auto& i : e.node->inputs) own(i); };
  for (auto& h : s.outputs) own(h);
  for (Node* n : Topo(s)) for (int i = 0, k = NumOutputs(*n); i < k; ++i) r.outputs.push_back(Entry{owner[n], i});
  return r;
}
inline Symbol GetChildren(const Symbol& s) {
  if (s.outputs.size() != 1) throw std::runtime_error("GetChildren: needs a single-output symbol");
  Symbol r; r.outputs = s.outputs[0].node->inputs;
  return r;
}

// ------------------------------------------------------------------------------------------------ JSON (nnvm dialect out, both dialects in)
inline std::string JEscape(const std::string& s) {
  std::string o;
  for (unsigned char c : s) {
    switch (c) {
      case '"': o += "\\\""; break; case '\\': o += "\\\\"; break; case '\n': o += "\\n"; break; case '\t': o += "\\t"; break; case '\r': o += "\\r"; break;
      default: if (c < 0x20) { char b[8]; snprintf(b, sizeof b, "\\u%04x", c); o += b; } else o.push_back(static_cast<char>(c));
    }
  }
  return o;
}

inline std::string ToJSON(const Symbol& s) {
  const auto order = Topo(s);
  std::unordered_map<Node*, int> id;
  for (size_t i = 0; i < order.size(); ++i) id[order[i]] = static_cast<int>(i);
  std::ostringstream o;
  o << "{\n  \"nodes\": [\n";
  for (size_t i = 0; i < order.size(); ++i) {
    Node* n = order[i];
    o << "    {\n      \"op\": \"" << JEscape(n->op) << "\", \n      \"name\": \"" << JEscape(n->name) << "\", \n";
    if (!n->attrs.empty()) {
      o << "      \"attrs\": {";
      bool first = true;
      for (auto& kv : n->attrs) { o << (first ? "\n" : ", \n") << "        \"" << JEscape(kv.first) << "\": \"" << JEscape(kv.second) << "\""; first = false; }
      o << "\n      }, \n";
    }
    o << "      \"inputs\": [";
    for (size_t k = 0; k < n->inputs.size(); ++k) o << (k ? ", " : "") << "[" << id[n->inputs[k].node.get()] << ", " << n->inputs[k].index << ", 0]";
    o << "]\n    }" << (i + 1 < order.size() ? ", \n" : "\n");
  }
  o << "  ], \n  \"arg_nodes\": [";
  bool first = true;
  for (size_t i = 0; i < order.size(); ++i) if (order[i]->op == "null") { o << (first ? "" : ", ") << i; first = false; }
  o << "], \n  \"node_row_ptr\": [";
  { size_t row = 0; o << 0; for (size_t i = 0; i < order.size(); ++i) { row += static_cast<size_t>(NumOutputs(*order[i])); o << ", " << row; } }
  o << "], \n  \"heads\": [";
  for (size_t i = 0; i < s.outputs.size(); ++i) o << (i ? ", " : "") << "[" << id[s.outputs[i].node.get()] << ", " << s.outputs[i].index << ", 0]";
  o << "], \n  \"attrs\": {\"mxnet_version\": [\"int\", 10400]}\n}";
  return o.str();
}

inline std::string JAttrToString(const JValue& v) {
  switch (v.kind) {
    case JValue::kStr: return v.str;
    case JValue::kBool: return v.b ? "True" : "False";
    case JValue::kNum: {
      if (std::isfinite(v.num) && v.num == std::floor(v.num) && std::fabs(v.num) < 1e15) return std::to_string(static_cast<long long>(v.num));
      char b[40]; snprintf(b, sizeof b, "%.17g", v.num); return b;
    }
    case JValue::kArr: {
      std::string o = "(";
      for (size_t i = 0; i < v.arr.size(); ++i) o += (i ? ", " : "") + JAttrToString(v.arr[i]);
      if (v.arr.size() == 1) o += ",";
      return o + ")";
    }
    default: return "None";
  }
}

inline Symbol FromJSON(const std::string& json) {
  const JValue doc = JParser(json.data(), json.size()).Parse();
  const JValue* jn = doc.Find("nodes");
  if (!jn || jn->kind != JValue::kArr) throw std::runtime_error("symbol JSON: no \"nodes\" array");
  if (jn->arr.size() > (1u << 22)) throw std::runtime_error("symbol JSON: implausible node count");
  std::vector<std::shared_ptr<Node>> nodes(jn->arr.size());
  auto entry = [&](const JValue& e, size_t limit) {
    Entry en; int64_t idx = -1;
    if (e.kind == JValue::kNum) idx = static_cast<int64_t>(e.num);
    else if (e.kind == JValue::kArr && !e.arr.empty() && e.arr[0].kind == JValue::kNum) { idx = static_cast<int64_t>(e.arr[0].num); en.index = e.arr.size() > 1 ? static_cast<int>(e.arr[1].num) : 0; }
    else throw std::runtime_error("symbol JSON: malformed input reference");
    if (idx < 0 || static_cast<size_t>(idx) >= limit) throw std::runtime_error("symbol JSON: node inputs must refer to earlier nodes");
    en.node = nodes[static_cast<size_t>(idx)];
    if (en.index < 0 || en.index >= NumOutputs(*en.node)) throw std::runtime_error("symbol JSON: " + en.node->name + " has no output " + std::to_string(en.index));
    return en;
  };
  for (size_t i = 0; i < nodes.size(); ++i) {
    const JValue& j = jn->arr[i];
    auto n = std::make_shared<Node>();
    const JValue* op = j.Find("op"); const JValue* name = j.Find("name");
    if (!op || op->kind != JValue::kStr) throw std::runtime_error("symbol JSON: node without op");
    n->op = op->str; n->name = name && name->kind == JValue::kStr ? name->str : "node" + std::to_string(i);
    const JValue* at = j.Find("attrs"); if (!at) at = j.Find("param");
    const JValue* usr = j.Find("attr");                     // pre-1.0 files: "param" = operator arguments, "attr" = user annotations
    if (!at) { at = usr; usr = nullptr; }
    if (n->op == "_nd") {                                   // generic imperative-op node of symbol.py: the function name is the operator, kwargs the attributes
      const JValue* fn = at ? at->Find("fn") : nullptr;
      if (!fn || fn->kind != JValue::kStr) throw std::runtime_error(n->name + ": _nd node without fn");
      const size_t dot = fn->str.rfind('.');
      n->op = dot == std::string::npos ? fn->str : fn->str.substr(dot + 1);
      at = at->Find("kwargs");
    }
    for (const JValue* src : {at, usr}) if (src && src->kind == JValue::kObj) for (auto& kv : src->obj) {
      if (kv.first == "__attr__" && kv.second.kind == JValue::kObj) { for (auto& u : kv.second.obj) n->attrs[u.first] = JAttrToString(u.second); continue; }
      if (kv.second.kind != JValue::kNull) n->attrs[kv.first] = JAttrToString(kv.second);
    }
    if (n->op != "null") { n->op = GetOp(n->op).name; }
    if (const JValue* in = j.Find("inputs")) for (auto& e : in->arr) n->inputs.push_back(entry(e, i));
    if (const JValue* aux = j.Find("aux")) for (auto& e : aux->arr) n->inputs.push_back(entry(e, i));
    if (n->op != "null") {
      const OpDef& d = GetOp(n->op);
      if (*d.key_var_num_args && !AttrView(n->attrs).Has(d.key_var_num_args)) n->attrs[d.key_var_num_args] = std::to_string(n->inputs.size());
      if (n->op == "Pooling" && doc.Find("format") && !AttrView(n->attrs).Has("stride") && AttrView(n->attrs).Has("kernel")) n->attrs["stride"] = n->attrs["kernel"];
      const size_t want = d.inputs(AttrView(n->attrs)).size();
      if (n->inputs.size() != want) throw std::runtime_error(n->name + " (" + n->op + "): " + std::to_string(n->inputs.size()) + " inputs in the file, the operator takes " + std::to_string(want));
    } else if (!n->inputs.empty()) throw std::runtime_error(n->name + ": a variable cannot have inputs");
    nodes[i] = n;
  }
  const JValue* heads = doc.Find("heads");
  if (!heads || heads->kind != JValue::kArr || heads->arr.empty()) throw std::runtime_error("symbol JSON: no heads");
  Symbol s;
  for (auto& h : heads->arr) s.outputs.push_back(entry(h, nodes.size()));
  return s;
}

// ------------------------------------------------------------------------------------------------ shape inference
struct ShapeResult {
  std::vector<Node*> order;
  std::unordered_map<Node*, Shape> shape;        // output shape per node (variables: their own shape); absent = unknown
  bool complete = true;
};

namespace detail {
inline int64_t AxisOf(int64_t a, size_t nd, const std::string& who) {
  if (a < 0) a += static_cast<int64_t>(nd);
  if (a < 0 || a >= static_cast<int64_t>(nd)) throw std::runtime_error(who + ": axis out of range");
  return a;
}
inline Shape BroadcastShape(const Shape& a, const Shape& b, const std::string& who) {
  const size_t n = std::max(a.size(), b.size());
  Shape out(n);
  for (size_t i = 0; i < n; ++i) {
    const int64_t x = i + a.size() >= n ? a[i + a.size() - n] : 1, y = i + b.size() >= n ? b[i + b.size() - n] : 1;
    if (x != y && x != 1 && y != 1) throw std::runtime_error(who + ": shapes " + ShapeStr(a) + " and " + ShapeStr(b) + " do not broadcast");
    out[i] = std::max(x, y);
  }
  return out;
}
struct Win { int64_t kh, kw, sh, sw, ph, pw, dh, dw; };
inline Win Window(const Node& n, bool pooling, const Shape& x) {
  AttrView a(n.attrs);
  auto two = [&](const char* key, int64_t def) { auto v = a.Tuple(key, {}); if (v.empty()) v = {def, def}; if (v.size() == 1) v.push_back(v[0]); return v; };
  Win w{};
  if (pooling && a.Bool("global_pool", false)) { w.kh = x[2]; w.kw = x[3]; w.sh = w.sw = w.dh = w.dw = 1; w.ph = w.pw = 0; return w; }
  auto k = a.Tuple("kernel", {});
  if (k.size() == 1 && pooling) k.push_back(k[0]);
  if (k.size() != 2) throw std::runtime_error(n.name + ": only 2-D windows are supported by the native graph runtime");
  const auto s = two("stride", 1), p = two("pad", 0), d = two("dilate", 1);
  w = Win{k[0], k[1], s[0], s[1], p[0], p[1], d[0], d[1]};
  if (w.kh < 1 || w.kw < 1 || w.sh < 1 || w.sw < 1 || w.dh < 1 || w.dw < 1 || w.ph < 0 || w.pw < 0 || w.kh > 4096 || w.kw > 4096 || w.ph > 4096 || w.pw > 4096)
    throw std::runtime_error(n.name + ": kernel / stride / dilate must be positive and pad non-negative");
  if (pooling && (w.ph >= w.kh || w.pw >= w.kw)) throw std::runtime_error(n.name + ": pooling needs pad < kernel");
  return w;
}
inline int64_t PoolOut(int64_t in, int64_t k, int64_t s, int64_t p, bool full) {
  const int64_t span = in + 2 * p - k;
  if (span < 0) throw std::runtime_error("pooling window larger than the padded input");
  return (full ? (span + s - 1) / s : span / s) + 1;
}
inline Shape ReduceShape(const Shape& x, std::vector<int64_t> axes, bool keep, const std::string& who) {
  std::vector<char> red(x.size(), axes.empty());
  for (auto a : axes) red[AxisOf(a, x.size(), who)] = 1;
  Shape out;
  for (size_t i = 0; i < x.size(); ++i) { if (!red[i]) out.push_back(x[i]); else if (keep) out.push_back(1); }
  if (out.empty()) out.push_back(1);
  return out;
}
// "(None, 2, -1)" -> {nullopt, 2, -1}: tuples whose entries may be None (slice begin / end)
inline std::vector<std::pair<bool, int64_t>> TupleOpt(const AttrView& a, const std::string& key) {
  std::vector<std::pair<bool, int64_t>> out;
  const std::string* v = a.Raw(key);
  if (!v) return out;
  std::string tok;
  auto flush = [&] {
    size_t b = 0, e = tok.size();
    while (b < e && (tok[b] == ' ' || tok[b] == '(' || tok[b] == '[')) ++b;
    while (e > b && (tok[e - 1] == ' ' || tok[e - 1] == ')' || tok[e - 1] == ']')) --e;
    const std::string t = tok.substr(b, e - b);
    tok.clear();
    if (t.empty()) return;
    if (t == "None") { out.emplace_back(false, 0); return; }
    try { out.emplace_back(true, std::stoll(t)); } catch (...) { throw std::runtime_error("attribute " + key + ": bad tuple entry " + t); }
  };
  for (char c : *v) { if (c == ',') flush(); else tok.push_back(c); }
  flush();
  return out;
}
// [begin, end) of a slice along an axis of extent n, python style (negative counts from the end, None = open)
inline void SliceRange(bool hb, int64_t b, bool he, int64_t e, int64_t n, const std::string& who, int64_t* lo, int64_t* hi) {
  if (!hb) b = 0;
  if (!he) e = n;
  if (b < 0) b += n;
  if (e < 0) e += n;
  if (b < 0 || e > n || b >= e) throw std::runtime_error(who + ": slice [" + std::to_string(b) + ", " + std::to_string(e) + ") is empty or outside the extent " + std::to_string(n));
  *lo = b; *hi = e;
}
inline Shape ReshapeTo(const Node& n, const Shape& x) {
  const auto spec = AttrView(n.attrs).Tuple("shape", {});
  Shape out; size_t src = 0; int infer = -1;
  for (size_t i = 0; i < spec.size(); ++i) {
    const int64_t d = spec[i];
    if (d > 0) { out.push_back(d); ++src; }
    else if (d == 0) { if (src >= x.size()) throw std::runtime_error(n.name + ": reshape code 0 past the input rank"); out.push_back(x[src++]); }
    else if (d == -1) { if (infer >= 0) throw std::runtime_error(n.name + ": two -1 in reshape"); infer = static_cast<int>(out.size()); out.push_back(1); ++src; }
    else if (d == -2) { while (src < x.size()) out.push_back(x[src++]); }
    else if (d == -3) { if (src + 1 >= x.size()) throw std::runtime_error(n.name + ": reshape code -3 past the input rank"); out.push_back(x[src] * x[src + 1]); src += 2; }
    else throw std::runtime_error(n.name + ": reshape code " + std::to_string(d) + " is not supported");
  }
  if (infer >= 0) { const int64_t rest = Numel(out); if (rest == 0 || Numel(x) % rest) throw std::runtime_error(n.name + ": cannot infer -1"); out[infer] = Numel(x) / rest; }
  if (Numel(out) != Numel(x)) throw std::runtime_error(n.name + ": reshape " + ShapeStr(x) + " -> " + ShapeStr(out) + " changes the size");
  return out;
}
}  // namespace detail

// One rule per operator: `in[i]` are the input shapes (nullptr = unknown).  Returns the output shape (empty optional = cannot tell yet) and may
// assign shapes to unknown inputs through `fill(i, shape)` (parameters from the data shape, labels from the prediction shape).
inline bool InferNode(const Node& n, const std::vector<const Shape*>& in, const std::function<void(size_t, const Shape&)>& fill, Shape* out) {
  using namespace detail;
  AttrView a(n.attrs);
  const std::string& op = n.op;
  auto need = [&](size_t i, const Shape& want) {
    if (!in[i]) { fill(i, want); return; }
    if (*in[i] != want) throw std::runtime_error(n.name + " (" + op + "): input " + n.inputs[i].node->name + " has shape " + ShapeStr(*in[i]) + ", expected " + ShapeStr(want));
  };
  if (in.empty() || !in[0]) {
    // the data input is unknown: binary ops can still take the other side's shape
    if (in.size() == 2 && in[1] && (op.compare(0, 9, "elemwise_") == 0)) { fill(0, *in[1]); *out = *in[1]; return true; }
    return false;
  }
  const Shape& x = *in[0];
  for (auto d : x) if (d < 1) throw std::runtime_error(n.name + ": empty tensors are not supported, shape " + ShapeStr(x));
  if (op == "FullyConnected") {
    const int64_t h = a.Int("num_hidden", 0);
    if (h < 1) throw std::runtime_error(n.name + ": num_hidden must be positive");
    const bool flat = a.Bool("flatten", true);
    if (x.empty()) throw std::runtime_error(n.name + ": scalar input");
    const int64_t k = flat ? Numel(x) / x[0] : x.back();
    need(1, {h, k});
    if (in.size() > 2) need(2, {h});
    if (flat) *out = {x[0], h}; else { *out = x; out->back() = h; }
  } else if (op == "Convolution") {
    if (x.size() != 4) throw std::runtime_error(n.name + ": convolution input must be NCHW, got " + ShapeStr(x));
    const Win w = Window(n, false, x);
    const int64_t f = a.Int("num_filter", 0), g = a.Int("num_group", 1);
    if (f < 1 || g < 1 || x[1] % g || f % g) throw std::runtime_error(n.name + ": num_filter / num_group do not divide the channels");
    need(1, {f, x[1] / g, w.kh, w.kw});
    if (in.size() > 2) need(2, {f});
    const int64_t oh = (x[2] + 2 * w.ph - w.dh * (w.kh - 1) - 1) / w.sh + 1, ow = (x[3] + 2 * w.pw - w.dw * (w.kw - 1) - 1) / w.sw + 1;
    if (oh <= 0 || ow <= 0) throw std::runtime_error(n.name + ": kernel larger than the padded input");
    *out = {x[0], f, oh, ow};
  } else if (op == "Pooling") {
    if (x.size() != 4) throw std::runtime_error(n.name + ": pooling input must be NCHW");
    const Win w = Window(n, true, x);
    const bool full = a.Str("pooling_convention", "valid") == "full", global = a.Bool("global_pool", false);
    *out = {x[0], x[1], global ? 1 : PoolOut(x[2], w.kh, w.sh, w.ph, full), global ? 1 : PoolOut(x[3], w.kw, w.sw, w.pw, full)};
  } else if (op == "Flatten") {
    *out = {x.empty() ? 1 : x[0], x.empty() ? 1 : Numel(x) / std::max<int64_t>(x[0], 1)};
  } else if (op == "Reshape") {
    *out = ReshapeTo(n, x);
  } else if (op == "expand_dims") {
    Shape y = x;
    int64_t ax = a.Int("axis", 0); if (ax < 0) ax += static_cast<int64_t>(x.size()) + 1;
    if (ax < 0 || ax > static_cast<int64_t>(x.size())) throw std::runtime_error(n.name + ": axis out of range");
    y.insert(y.begin() + ax, 1); *out = y;
  } else if (op == "transpose") {
    auto axes = a.Tuple("axes", {});
    if (axes.empty()) for (size_t i = 0; i < x.size(); ++i) axes.push_back(static_cast<int64_t>(x.size() - 1 - i));
    if (axes.size() != x.size()) throw std::runtime_error(n.name + ": axes do not match the input rank");
    std::vector<char> seen(x.size(), 0);
    out->resize(x.size());
    for (size_t i = 0; i < x.size(); ++i) { const int64_t ax = AxisOf(axes[i], x.size(), n.name); if (seen[ax]) throw std::runtime_error(n.name + ": repeated axis"); seen[ax] = 1; (*out)[i] = x[ax]; }
  } else if (op == "BatchNorm") {
    const int64_t ax = AxisOf(a.Int("axis", 1), x.size(), n.name);
    for (size_t i = 1; i <= 4; ++i) need(i, {x[ax]});
    *out = x;
  } else if (op == "Concat") {
    Shape o = x;
    const int64_t ax = AxisOf(a.Int("dim", 1), o.size(), n.name);
    for (size_t i = 1; i < in.size(); ++i) {
      if (!in[i]) return false;
      const Shape& s = *in[i];
      if (s.size() != o.size()) throw std::runtime_error(n.name + ": concat inputs differ in rank");
      for (size_t d = 0; d < s.size(); ++d) if (static_cast<int64_t>(d) != ax && s[d] != o[d]) throw std::runtime_error(n.name + ": concat inputs differ outside the axis");
      o[ax] += s[ax];
    }
    *out = o;
  } else if (op == "add_n" || op == "sgd_update" || op == "sgd_mom_update" || op == "adam_update") {
    for (size_t i = 1; i < in.size(); ++i) need(i, x);
    *out = x;
  } else if (op == "Embedding") {
    const int64_t v = a.Int("input_dim", 0), w = a.Int("output_dim", 0);
    if (v < 1 || w < 1) throw std::runtime_error(n.name + ": input_dim / output_dim must be positive");
    need(1, {v, w});
    *out = x; out->push_back(w);
  } else if (op == "SoftmaxOutput") {
    if (x.size() < 2) throw std::runtime_error(n.name + ": needs at least (batch, classes)");
    if (!in[1]) {
      if (a.Bool("multi_output", false)) { Shape l = {x[0]}; for (size_t i = 2; i < x.size(); ++i) l.push_back(x[i]); fill(1, l); }
      else fill(1, {x[0]});
    }
    *out = x;
  } else if (op == "LinearRegressionOutput" || op == "LogisticRegressionOutput" || op == "MAERegressionOutput") {
    if (!in[1]) fill(1, x);
    *out = x;
  } else if (op == "dot") {
    if (!in[1]) return false;
    const Shape& y = *in[1];
    if (x.size() != 2 || y.size() != 2) throw std::runtime_error(n.name + ": dot takes 2-D operands in the native graph runtime");
    const bool ta = a.Bool("transpose_a", false), tb = a.Bool("transpose_b", false);
    const int64_t m = ta ? x[1] : x[0], k = ta ? x[0] : x[1], k2 = tb ? y[1] : y[0], nn = tb ? y[0] : y[1];
    if (k != k2) throw std::runtime_error(n.name + ": inner dimensions differ, " + ShapeStr(x) + " x " + ShapeStr(y));
    *out = {m, nn};
  } else if (op == "sum" || op == "mean" || op == "max" || op == "min" || op == "prod" || op == "norm") {
    *out = ReduceShape(x, a.Tuple("axis", {}), a.Bool("keepdims", false), n.name);
  } else if (op == "argmax" || op == "argmin") {
    if (!a.Has("axis")) throw std::runtime_error(n.name + ": axis is required");
    *out = ReduceShape(x, {a.Int("axis", 0)}, a.Bool("keepdims", false), n.name);
  } else if (op == "LayerNorm") {
    const int64_t ax = AxisOf(a.Int("axis", -1), x.size(), n.name);
    need(1, {x[ax]}); need(2, {x[ax]});
    *out = x;
  } else if (op == "InstanceNorm") {
    if (x.size() < 3) throw std::runtime_error(n.name + ": InstanceNorm needs (batch, channel, spatial...)");
    need(1, {x[1]}); need(2, {x[1]});
    *out = x;
  } else if (op == "LRN") {
    if (x.size() != 4) throw std::runtime_error(n.name + ": LRN input must be NCHW");
    const int64_t ns = a.Int("nsize", 0);
    if (ns < 1 || ns % 2 == 0) throw std::runtime_error(n.name + ": nsize must be odd and positive");
    *out = x;
  } else if (op == "Deconvolution") {
    if (x.size() != 4) throw std::runtime_error(n.name + ": deconvolution input must be NCHW, got " + ShapeStr(x));
    const Win w = Window(n, false, x);
    auto adj = a.Tuple("adj", {0, 0}); if (adj.empty()) adj = {0, 0}; if (adj.size() == 1) adj.push_back(adj[0]);
    const int64_t f = a.Int("num_filter", 0), g = a.Int("num_group", 1);
    if (f < 1 || g < 1 || x[1] % g || f % g) throw std::runtime_error(n.name + ": num_filter / num_group do not divide the channels");
    if (adj[0] < 0 || adj[1] < 0 || adj[0] >= w.sh || adj[1] >= w.sw) throw std::runtime_error(n.name + ": adj must be in [0, stride)");
    need(1, {x[1], f / g, w.kh, w.kw});
    if (in.size() > 2) need(2, {f});
    const int64_t oh = (x[2] - 1) * w.sh - 2 * w.ph + w.dh * (w.kh - 1) + 1 + adj[0], ow = (x[3] - 1) * w.sw - 2 * w.pw + w.dw * (w.kw - 1) + 1 + adj[1];
    if (oh <= 0 || ow <= 0) throw std::runtime_error(n.name + ": padding larger than the output");
    *out = {x[0], f, oh, ow};
  } else if (op == "UpSampling") {
    if (in.size() != 1 || a.Str("sample_type", "nearest") != "nearest") throw std::runtime_error(n.name + ": the native runtime has single-input nearest-neighbour UpSampling");
    const int64_t sc = a.Int("scale", 0);
    if (x.size() != 4 || sc < 1 || sc > 64) throw std::runtime_error(n.name + ": needs NCHW input and 1 <= scale <= 64");
    *out = {x[0], x[1], x[2] * sc, x[3] * sc};
  } else if (op == "SliceChannel") {
    const int64_t ax = AxisOf(a.Int("axis", 1), x.size(), n.name), k = NumOutputs(n);
    if (x[ax] % k) throw std::runtime_error(n.name + ": extent " + std::to_string(x[ax]) + " of axis " + std::to_string(ax) + " is not divisible into " + std::to_string(k) + " parts");
    *out = x; (*out)[ax] = x[ax] / k;
    if (a.Bool("squeeze_axis", false)) {
      if ((*out)[ax] != 1) throw std::runtime_error(n.name + ": squeeze_axis needs parts of extent 1");
      out->erase(out->begin() + ax);
      if (out->empty()) out->push_back(1);
    }
  } else if (op == "softmax_cross_entropy") {
    if (x.size() != 2) throw std::runtime_error(n.name + ": data must be (batch, classes)");
    need(1, {x[0]});
    *out = {1};
  } else if (op == "slice_axis") {
    const int64_t ax = AxisOf(a.Int("axis", 0), x.size(), n.name);
    int64_t lo, hi; SliceRange(a.Has("begin"), a.Int("begin", 0), a.Has("end"), a.Int("end", 0), x[ax], n.name, &lo, &hi);
    *out = x; (*out)[ax] = hi - lo;
  } else if (op == "slice") {
    const auto b = TupleOpt(a, "begin"), e = TupleOpt(a, "end");
    if (b.size() != e.size() || b.size() > x.size() || b.empty()) throw std::runtime_error(n.name + ": begin / end must have the same length, at most the input rank");
    *out = x;
    for (size_t i = 0; i < b.size(); ++i) { int64_t lo, hi; SliceRange(b[i].first, b[i].second, e[i].first, e[i].second, x[i], n.name, &lo, &hi); (*out)[i] = hi - lo; }
  } else if (op == "SwapAxis") {
    *out = x; std::swap((*out)[AxisOf(a.Int("dim1", 0), x.size(), n.name)], (*out)[AxisOf(a.Int("dim2", 0), x.size(), n.name)]);
  } else if (op == "tile") {
    const auto reps = a.Tuple("reps", {});
    if (reps.empty() || reps.size() > 8) throw std::runtime_error(n.name + ": reps must have 1..8 entries");
    Shape xs = x; while (xs.size() < reps.size()) xs.insert(xs.begin(), 1);
    *out = xs;
    for (size_t i = 0; i < reps.size(); ++i) { const int64_t r = reps[i]; if (r < 1 || r > 4096) throw std::runtime_error(n.name + ": reps out of range"); (*out)[xs.size() - reps.size() + i] *= r; }
  } else if (op == "repeat") {
    if (!a.Has("axis")) throw std::runtime_error(n.name + ": the native runtime needs an explicit axis");
    const int64_t ax = AxisOf(a.Int("axis", 0), x.size(), n.name), r = a.Int("repeats", 0);
    if (r < 1 || r > 4096) throw std::runtime_error(n.name + ": repeats out of range");
    *out = x; (*out)[ax] *= r;
  } else if (op == "Pad") {
    const auto pw = a.Tuple("pad_width", {});
    if (pw.size() != 2 * x.size()) throw std::runtime_error(n.name + ": pad_width needs (before, after) for each of the " + std::to_string(x.size()) + " axes");
    const std::string mode = a.Str("mode", "constant");
    if (mode != "constant" && mode != "edge" && mode != "reflect") throw std::runtime_error(n.name + ": mode " + mode + " is not supported");
    *out = x;
    for (size_t i = 0; i < x.size(); ++i) {
      if (pw[2 * i] < 0 || pw[2 * i + 1] < 0 || pw[2 * i] > 65536 || pw[2 * i + 1] > 65536) throw std::runtime_error(n.name + ": pad_width out of range");
      if (mode == "reflect" && (pw[2 * i] >= x[i] || pw[2 * i + 1] >= x[i])) throw std::runtime_error(n.name + ": reflect padding must be smaller than the extent");
      (*out)[i] += pw[2 * i] + pw[2 * i + 1];
    }
  } else if (op == "squeeze") {
    const auto axes = a.Tuple("axis", {});
    std::vector<char> drop(x.size(), 0);
    if (axes.empty()) { for (size_t i = 0; i < x.size(); ++i) drop[i] = x[i] == 1; }
    else for (auto ax : axes) { const int64_t k = AxisOf(ax, x.size(), n.name); if (x[k] != 1) throw std::runtime_error(n.name + ": cannot squeeze an axis of extent " + std::to_string(x[k])); drop[k] = 1; }
    out->clear();
    for (size_t i = 0; i < x.size(); ++i) if (!drop[i]) out->push_back(x[i]);
    if (out->empty()) out->push_back(1);
  } else if (op == "broadcast_to") {
    const auto t = a.Tuple("shape", {});
    if (t.size() != x.size()) throw std::runtime_error(n.name + ": shape must have the input rank");
    *out = x;
    for (size_t i = 0; i < x.size(); ++i) {
      if (t[i] == 0 || t[i] == x[i]) continue;
      if (x[i] != 1 || t[i] < 1 || t[i] > (int64_t{1} << 24)) throw std::runtime_error(n.name + ": cannot broadcast " + ShapeStr(x) + " to the requested shape");
      (*out)[i] = t[i];
    }
  } else if (op == "broadcast_axis") {
    const auto axes = a.Tuple("axis", {}), sizes = a.Tuple("size", {});
    if (axes.size() != sizes.size() || axes.empty()) throw std::runtime_error(n.name + ": axis and size must have the same length");
    *out = x;
    for (size_t i = 0; i < axes.size(); ++i) {
      const int64_t k = AxisOf(axes[i], x.size(), n.name);
      if (x[k] != 1 || sizes[i] < 1 || sizes[i] > (int64_t{1} << 24)) throw std::runtime_error(n.name + ": only axes of extent 1 can be broadcast");
      (*out)[k] = sizes[i];
    }
  } else if (op == "reverse") {
    for (auto ax : a.Tuple("axis", {})) AxisOf(ax, x.size(), n.name);
    *out = x;
  } else if (op == "take") {
    if (!in[1]) return false;
    const int64_t ax = AxisOf(a.Int("axis", 0), x.size(), n.name);
    out->assign(x.begin(), x.begin() + ax);
    out->insert(out->end(), in[1]->begin(), in[1]->end());
    out->insert(out->end(), x.begin() + ax + 1, x.end());
  } else if (op == "pick") {
    const int64_t ax = AxisOf(a.Int("axis", -1), x.size(), n.name);
    Shape idx = x; idx.erase(idx.begin() + ax); if (idx.empty()) idx.push_back(1);
    if (!in[1]) fill(1, idx);
    else if (Numel(*in[1]) != Numel(idx)) throw std::runtime_error(n.name + ": index has " + std::to_string(Numel(*in[1])) + " elements, expected " + std::to_string(Numel(idx)));
    *out = idx;
    if (a.Bool("keepdims", false)) { *out = x; (*out)[ax] = 1; }
  } else if (op == "one_hot") {
    const int64_t d = a.Int("depth", 0);
    if (d < 1 || d > (int64_t{1} << 24)) throw std::runtime_error(n.name + ": depth out of range");
    *out = x; out->push_back(d);
  } else if (op == "where") {
    if (!in[1]) { fill(1, x); } else if (*in[1] != x) throw std::runtime_error(n.name + ": x must have the condition's shape");
    if (!in[2]) { fill(2, x); } else if (*in[2] != x) throw std::runtime_error(n.name + ": y must have the condition's shape");
    *out = x;
  } else if (op == "Cast") {
    if (a.Str("dtype", "float32") != "float32") throw std::runtime_error(n.name + ": the host executor computes in float32 only");
    *out = x;
  } else if (in.size() == 2) {           // binary arithmetic
    if (!in[1]) { if (op.compare(0, 9, "elemwise_") == 0) { fill(1, x); *out = x; return true; } return false; }
    if (op.compare(0, 9, "elemwise_") == 0 && *in[1] != x) throw std::runtime_error(n.name + ": elementwise operands differ in shape, " + ShapeStr(x) + " vs " + ShapeStr(*in[1]));
    *out = BroadcastShape(x, *in[1], n.name);
  } else {
    *out = x;                            // every remaining registered operator is shape preserving
  }
  return true;
}

// `known`: shapes by argument / auxiliary-state name.  partial = false throws when something stays unknown.
inline ShapeResult InferShapes(const Symbol& s, const std::map<std::string, Shape>& known, bool partial) {
  ShapeResult r;
  r.order = Topo(s);
  std::set<std::string> names;
  for (Node* n : r.order) if (n->op == "null") {
    names.insert(n->name);
    auto it = known.find(n->name);
    if (it != known.end()) r.shape[n] = it->second;
    else if (AttrView(n->attrs).Has("__shape__")) {
      Shape sh = AttrView(n->attrs).Tuple("__shape__", {});
      if (!sh.empty() && std::all_of(sh.begin(), sh.end(), [](int64_t d) { return d > 0; })) r.shape[n] = sh;
    }
  }
  for (auto& kv : known) if (!names.count(kv.first)) throw std::runtime_error("InferShape: " + kv.first + " is not an argument of the symbol");
  for (int sweep = 0; sweep < 3; ++sweep) {
    bool changed = false;
    for (Node* n : r.order) {
      if (n->op == "null" || r.shape.count(n)) continue;
      std::vector<const Shape*> in;
      for (auto& e : n->inputs) { auto it = r.shape.find(e.node.get()); in.push_back(it == r.shape.end() ? nullptr : &it->second); }
      std::vector<std::pair<size_t, Shape>> fills;
      Shape out;
      const bool ok = InferNode(*n, in, [&](size_t i, const Shape& sh) { fills.emplace_back(i, sh); }, &out);
      for (auto& f : fills) {
        Node* src = n->inputs[f.first].node.get();
        if (src->op != "null") continue;                   // only variables are back-filled
        r.shape[src] = f.second; changed = true;
      }
      if (ok) { r.shape[n] = out; changed = true; }
    }
    if (!changed) break;
  }
  for (Node* n : r.order) if (!r.shape.count(n)) {
    r.complete = false;
    if (!partial) throw std::runtime_error("InferShape: the shape of " + n->name + " cannot be determined from the given arguments");
  }
  return r;
}

}  // namespace graph
}  // namespace gxrt
