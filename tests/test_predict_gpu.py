"""The C predict API on a GPU (GXPredCreate* with dev_type 2: csrc/runtime/predict_device.h), driven through ctypes only.  The oracle is
the host predictor (dev_type 1) on the same JSON and parameter blob, itself checked against the Python Executor in test_predict_api.py:
max |device - host| / max |host| <= BOUND, and data-movement operators bitwise."""
import ctypes
import json
import os
import shutil
import subprocess
import threading

import numpy as np
import pytest

import _capi as C
from _capi import ck, lib, u32, vp

BOUND = 1e-4
HINT = "Python Executor"


# ---------------------------------------------------------------------------------------------------------------- JSON + params
class G:
    """a graph in either dialect: the reference's nnvm JSON (string attributes, input triples, arg_nodes) or this framework's"""

    def __init__(self, nnvm=True):
        self.nnvm, self.nodes = nnvm, []

    def var(self, name):
        self.nodes.append({"op": "null", "name": name, "inputs": []})
        return len(self.nodes) - 1

    def op(self, op, name, inputs, **attrs):
        if self.nnvm:
            at = {k: str(v) for k, v in attrs.items()}
            ins = [[i, 0, 0] for i in inputs]
        else:
            at, ins = attrs, list(inputs)
        self.nodes.append({"op": op, "name": name, "attrs": at, "inputs": ins})
        return len(self.nodes) - 1

    def json(self, *heads):
        if self.nnvm:
            return json.dumps({"nodes": self.nodes, "arg_nodes": [i for i, n in enumerate(self.nodes) if n["op"] == "null"], "heads": [[h, 0, 0] for h in heads]})
        return json.dumps({"nodes": self.nodes, "heads": list(heads), "format": "geomx_b200-symbol-1"})


def blob(params, tmp_path):
    import geomx_b200 as mx
    if not params:
        return b""
    f = str(tmp_path / "p.params")
    mx.nd.save(f, {"arg:" + k: mx.nd.array(np.asarray(v, np.float32)) for k, v in params.items()})
    return open(f, "rb").read()


# ---------------------------------------------------------------------------------------------------------------- ctypes predictor
def _shapes(shapes):
    keys = list(shapes)
    ind, data = [0], []
    for k in keys:
        data += list(shapes[k]); ind.append(len(data))
    return len(keys), C.strs(keys), (u32 * len(ind))(*ind), (u32 * max(len(data), 1))(*data)


def create(js, pb, shapes, dev_type, dev_id=0, output_keys=None):
    h = vp()
    n, k, ind, data = _shapes(shapes)
    if output_keys:
        rc = lib().GXPredCreatePartialOut(js.encode(), pb, len(pb), dev_type, dev_id, n, k, ind, data, len(output_keys), C.strs(output_keys), ctypes.byref(h))
    else:
        rc = lib().GXPredCreate(js.encode(), pb, len(pb), dev_type, dev_id, n, k, ind, data, ctypes.byref(h))
    if rc != 0:
        raise RuntimeError(C.err())
    return h


def set_input(h, key, x):
    x = np.ascontiguousarray(x, np.float32)
    ck(lib().GXPredSetInput(h, key.encode(), x.ctypes.data_as(vp), x.size))


def out_shape(h, i=0):
    d, nd = ctypes.POINTER(u32)(), u32()
    ck(lib().GXPredGetOutputShape(h, i, ctypes.byref(d), ctypes.byref(nd)))
    return tuple(d[j] for j in range(nd.value))


def num_outputs(h):
    n = u32(); ck(lib().GXPredGetNumOutputs(h, ctypes.byref(n))); return n.value


def get_output(h, i=0):
    y = np.empty(out_shape(h, i), np.float32)
    ck(lib().GXPredGetOutput(h, i, y.ctypes.data_as(vp), y.size))
    return y


def outputs(h):
    return [get_output(h, i) for i in range(num_outputs(h))]


def plan(h):
    a, n = ctypes.c_uint64(), u32()
    ck(lib().GXPredGetPlan(h, ctypes.byref(a), ctypes.byref(n)))
    return a.value, n.value


def engine(h):
    e = ctypes.c_int(); ck(lib().GXPredGetEngine(h, ctypes.byref(e))); return e.value


def partial_steps(h):
    lefts, step, left = [], 0, 1
    while left:
        lv = ctypes.c_int()
        ck(lib().GXPredPartialForward(h, step, ctypes.byref(lv)))
        left = lv.value; lefts.append(left); step += 1
    return lefts


def free(h):
    ck(lib().GXPredFree(h))


def rel(d, h):
    d, h = np.asarray(d, np.float64), np.asarray(h, np.float64)
    return float(np.abs(d - h).max() / max(np.abs(h).max(), 1e-30))


def serve(js, pb, inputs, dev_type, forwards=1, output_keys=None):
    h = create(js, pb, {k: v.shape for k, v in inputs.items()}, dev_type, output_keys=output_keys)
    runs = []
    for _ in range(forwards):
        for k, v in inputs.items():
            set_input(h, k, v)
        ck(lib().GXPredForward(h))
        runs.append(outputs(h))
    free(h)
    return runs


# ---------------------------------------------------------------------------------------------------------------- CPU: refusals
def test_device_create_errors_point_to_the_python_executor(tmp_path):
    g = G()
    fc = g.op("FullyConnected", "fc", [g.var("data"), g.var("fc_weight"), g.var("fc_bias")], num_hidden=3)
    with pytest.raises(RuntimeError) as e:
        create(g.json(fc), b"", {"data": (2, 4)}, 2)
    assert "fc (FullyConnected): input fc_weight has no value" in str(e.value) and HINT in str(e.value)
    pb = blob({"fc_weight": np.zeros((3, 4)), "fc_bias": np.zeros(3)}, tmp_path)
    with pytest.raises(RuntimeError) as e:                 # no device here, or no device 4096 on a GPU machine
        create(g.json(fc), pb, {"data": (2, 4)}, 2, dev_id=4096)
    assert HINT in str(e.value) and ("device 4096" in str(e.value) or "kernel library" in str(e.value))
    g2 = G()
    c = g2.op("Correlation", "corr_node", [g2.var("data"), g2.var("data2")])
    with pytest.raises(RuntimeError, match="corr_node.*Python Executor"):
        create(g2.json(c), b"", {"data": (1, 2, 4, 4), "data2": (1, 2, 4, 4)}, 2)
    with pytest.raises(RuntimeError, match="dev_type 5"):
        create(g.json(fc), pb, {"data": (2, 4)}, 5)


# ---------------------------------------------------------------------------------------------------------------- GPU: per operator
def _r(rng, *shape, scale=1.0, shift=0.0):
    return (rng.randn(*shape) * scale + shift).astype(np.float32)


def _cases():
    r = np.random.RandomState(3)
    cases = {}

    def add(name, g, head, params, inputs, exact=False):
        cases[name] = (g.json(*head) if isinstance(head, tuple) else g.json(head), params, inputs, exact)

    # FullyConnected
    g = G(); add("fc_flatten", g, g.op("FullyConnected", "fc", [g.var("data"), g.var("w"), g.var("b")], num_hidden=7),
                 {"w": _r(r, 7, 15), "b": _r(r, 7)}, {"data": _r(r, 4, 3, 5)})
    g = G(); add("fc_noflat_nobias", g, g.op("FullyConnected", "fc", [g.var("data"), g.var("w")], num_hidden=6, no_bias=True, flatten=False),
                 {"w": _r(r, 6, 8)}, {"data": _r(r, 3, 2, 8)})
    # Convolution
    convs = {"stride_pad": (dict(kernel=(3, 3), stride=(2, 2), pad=(1, 1), num_filter=8), 3, 1, False),
             "groups": (dict(kernel=(3, 2), pad=(1, 0), num_filter=6, num_group=2), 4, 2, False),
             "depthwise": (dict(kernel=(3, 3), pad=(1, 1), num_filter=4, num_group=4), 4, 4, False),
             "dilate2": (dict(kernel=(3, 3), dilate=(2, 2), pad=(2, 1), num_filter=5), 3, 1, False),
             "dilate2_groups": (dict(kernel=(3, 3), dilate=(2, 2), stride=(2, 1), num_filter=4, num_group=2), 4, 2, False),
             "no_bias": (dict(kernel=(3, 3), num_filter=4, no_bias=True), 3, 1, True),
             "1x1": (dict(kernel=(1, 1), num_filter=16), 8, 1, False)}
    for k, (at, cin, grp, nob) in convs.items():
        g = G()
        ins = [g.var("data"), g.var("w")] + ([] if nob else [g.var("b")])
        p = {"w": _r(r, at["num_filter"], cin // grp, *at["kernel"], scale=0.3)}
        if not nob:
            p["b"] = _r(r, at["num_filter"])
        add("conv_" + k, g, g.op("Convolution", "c", ins, **at), p, {"data": _r(r, 2, cin, 9, 8)})
    # Pooling (max is data movement: bitwise)
    pools = {"max_valid": dict(kernel=(3, 3), stride=(2, 2), pad=(1, 1), pool_type="max"),
             "max_full": dict(kernel=(3, 3), stride=(2, 2), pad=(1, 1), pool_type="max", pooling_convention="full"),
             "avg_pad": dict(kernel=(3, 3), stride=(2, 2), pad=(1, 1), pool_type="avg", count_include_pad=True),
             "avg_nopad": dict(kernel=(3, 3), stride=(2, 2), pad=(1, 1), pool_type="avg", count_include_pad=False),
             "avg_nopad_full": dict(kernel=(3, 3), stride=(2, 2), pad=(1, 1), pool_type="avg", count_include_pad=False, pooling_convention="full"),
             "sum": dict(kernel=(2, 2), stride=(1, 1), pool_type="sum"),
             "global_avg": dict(kernel=(1, 1), global_pool=True, pool_type="avg"), "global_max": dict(kernel=(1, 1), global_pool=True, pool_type="max"),
             "global_sum": dict(kernel=(1, 1), global_pool=True, pool_type="sum"),
             "max_nnvm_default_stride": dict(kernel=(2, 2), pool_type="max"), "avg_nnvm_default_stride": dict(kernel=(3, 2), pool_type="avg")}
    for k, at in pools.items():
        g = G(); add("pool_" + k, g, g.op("Pooling", "p", [g.var("data")], **at), {}, {"data": _r(r, 2, 3, 7, 8)}, exact="max" in k)
    g = G(nnvm=False); add("pool_native_default_stride", g, g.op("Pooling", "p", [g.var("data")], kernel=[2, 2], pool_type="max"), {}, {"data": _r(r, 2, 3, 8, 6)}, exact=True)
    # BatchNorm: axis 1 / -1, fix_gamma, and the dialects' defaults
    for ax, shape in ((1, (4, 3, 5, 5)), (-1, (4, 5, 3)), (1, (6, 3))):
        for fg in (True, False):
            g = G()
            bn = g.op("BatchNorm", "bn", [g.var("data"), g.var("gamma"), g.var("beta"), g.var("mean"), g.var("var")], axis=ax, fix_gamma=fg, eps=1e-4)
            c = shape[ax]
            add("bn_axis%d_%dd_fix%d" % (ax, len(shape), fg), g, bn, {"gamma": _r(r, c, shift=1), "beta": _r(r, c), "mean": _r(r, c), "var": np.abs(_r(r, c)) + 0.5},
                {"data": _r(r, *shape)})
    for nnvm in (True, False):
        g = G(nnvm)
        bn = g.op("BatchNorm", "bn", [g.var("data"), g.var("gamma"), g.var("beta"), g.var("mean"), g.var("var")])     # defaults: fix_gamma, eps
        add("bn_defaults_nnvm%d" % nnvm, g, bn, {"gamma": _r(r, 3, shift=2), "beta": _r(r, 3), "mean": _r(r, 3), "var": np.abs(_r(r, 3)) * 0.01}, {"data": _r(r, 2, 3, 4)})
    # transpose (bitwise)
    for k, (shape, axes) in {"2d_default": ((37, 45), None), "3d_default": ((5, 33, 40), None), "3d_swap_last": ((3, 70, 41), (0, 2, 1)),
                             "3d_keep_last": ((6, 7, 9), (1, 0, 2)), "4d_nhwc": ((2, 5, 33, 34), (0, 2, 3, 1)), "4d_nchw": ((2, 33, 34, 5), (0, 3, 1, 2)),
                             "5d": ((3, 4, 5, 6, 7), (4, 1, 0, 3, 2)), "5d_keep_last": ((3, 4, 5, 6, 7), (2, 0, 3, 1, 4)), "5d_neg": ((2, 3, 4, 5, 6), (-1, 0, -2, 1, 2))}.items():
        g = G()
        t = g.op("transpose", "t", [g.var("data")], **({"axes": axes} if axes else {}))
        add("transpose_" + k, g, t, {}, {"data": _r(r, *shape)}, exact=True)
    # Embedding (bitwise): ids out of range on both sides, fractional ids
    g = G(); e = g.op("Embedding", "emb", [g.var("data"), g.var("w")], input_dim=10, output_dim=6)
    add("embedding", g, e, {"w": _r(r, 10, 6)}, {"data": np.array([[0, 3.7, 9, 12], [-1, -0.5, 5, 100]], np.float32)}, exact=True)
    # binary, with and without broadcast
    for op in ("elemwise_add", "elemwise_sub", "elemwise_mul", "elemwise_div", "_maximum", "_minimum"):
        g = G(); add("binary_" + op, g, g.op(op, "e", [g.var("a"), g.var("b")]), {}, {"a": _r(r, 3, 4), "b": _r(r, 3, 4, shift=0.1)})
    for op in ("broadcast_add", "broadcast_sub", "broadcast_mul", "broadcast_div", "broadcast_maximum", "broadcast_minimum"):
        g = G(); add("binary_" + op, g, g.op(op, "e", [g.var("a"), g.var("b")]), {}, {"a": _r(r, 3, 1, 4), "b": np.abs(_r(r, 2, 1)) + 0.5})
    # scalar, unary, clip, LeakyReLU, Activation, LogisticRegressionOutput: chained, so that most run in place
    for op in ("_plus_scalar", "_minus_scalar", "_mul_scalar", "_div_scalar", "_rminus_scalar", "_rdiv_scalar", "_PlusScalar", "_RDivScalar"):
        g = G(); add("scalar_" + op, g, g.op(op, "s", [g.op("relu", "r", [g.var("data")])], scalar=1.75), {}, {"data": np.abs(_r(r, 5, 9)) + 0.2})
    for op in ("relu", "sigmoid", "tanh", "exp", "log", "sqrt", "abs", "negative", "square", "softsign", "softrelu"):
        g = G(); x = g.var("data")
        add("unary_" + op, g, g.op(op, "u", [g.op("_plus_scalar", "p", [g.op("abs", "a", [x])], scalar=0.25)]), {}, {"data": _r(r, 4, 33, scale=2)})
    g = G(); add("clip", g, g.op("clip", "c", [g.op("identity", "i", [g.var("data")])], a_min=-0.5, a_max=0.7), {}, {"data": _r(r, 6, 7)})
    for t in ("leaky", "elu"):
        g = G(); add("leakyrelu_" + t, g, g.op("LeakyReLU", "l", [g.op("_mul_scalar", "m", [g.var("data")], scalar=2.0)], act_type=t, slope=0.2), {}, {"data": _r(r, 5, 11)})
    for t in ("relu", "sigmoid", "tanh", "softrelu", "softsign"):
        g = G(); add("activation_" + t, g, g.op("Activation", "a", [g.op("_mul_scalar", "m", [g.var("data")], scalar=3.0)], act_type=t), {}, {"data": _r(r, 5, 11)})
    g = G(); add("logistic_regression_output", g, g.op("LogisticRegressionOutput", "lro", [g.op("negative", "n", [g.var("data")]), g.var("label")]), {}, {"data": _r(r, 4, 3)})
    # softmax family
    for k, (op, at, shape) in {"softmax_last": ("softmax", {}, (3, 17)), "softmax_axis1": ("softmax", {"axis": 1}, (2, 5, 3, 4)),
                               "softmax_axis0": ("softmax", {"axis": 0}, (6, 4)), "log_softmax_axis1": ("log_softmax", {"axis": 1}, (2, 40, 3)),
                               "log_softmax_last": ("log_softmax", {}, (4, 1000)), "softmax_output_2d": ("SoftmaxOutput", {}, (4, 10)),
                               "softmax_output_4d": ("SoftmaxOutput", {}, (2, 3, 4, 5)), "softmax_output_preserve": ("SoftmaxOutput", {"preserve_shape": True}, (2, 3, 4)),
                               "softmax_legacy": ("Softmax", {}, (3, 7)), "softmax_activation_instance": ("SoftmaxActivation", {}, (2, 3, 4, 5)),
                               "softmax_activation_channel": ("SoftmaxActivation", {"mode": "channel"}, (2, 3, 4, 5))}.items():
        g = G(); x = g.var("data")
        ins = [x, g.var("label")] if op in ("SoftmaxOutput", "Softmax") else [x]
        add(k, g, g.op(op, "sm", ins, **at), {}, {"data": _r(r, *shape, scale=2)})
    # views (bitwise) and Concat (bitwise)
    g = G(); a = g.var("data")
    v = g.op("Reshape", "r1", [g.op("Flatten", "f", [a])], shape=(0, -1, 4))
    v = g.op("Reshape", "r2", [g.op("expand_dims", "e", [v], axis=1)], shape=(-3, -2))
    v = g.op("BlockGrad", "bg", [g.op("identity", "id", [g.op("Dropout", "do", [v], p=0.5)])])
    v = g.op("MAERegressionOutput", "mae", [g.op("LinearRegressionOutput", "lin", [v, g.var("l1")]), g.var("l2")])
    add("views", g, g.op("_copy", "cp", [v]), {}, {"data": _r(r, 2, 3, 4, 2)}, exact=True)
    for dim, sb in ((1, (2, 5, 4)), (2, (2, 3, 1)), (0, (1, 3, 4))):
        g = G(); add("concat_dim%d" % dim, g, g.op("Concat", "cat", [g.var("a"), g.var("b")], dim=dim, num_args=2), {}, {"a": _r(r, 2, 3, 4), "b": _r(r, *sb)}, exact=True)
    g = G(); add("add_n", g, g.op("add_n", "s", [g.var("a"), g.var("b"), g.var("c")], num_args=3), {}, {k: _r(r, 2, 5) for k in "abc"})
    g = G(); names = ["x%d" % i for i in range(9)]
    add("elementwise_sum_9", g, g.op("ElementWiseSum", "s", [g.var(k) for k in names], num_args=9), {}, {k: _r(r, 3, 7) for k in names})
    # _nd generic nodes of symbol.py's dialect
    g = G(nnvm=False); x = g.var("data")
    n1 = g.op("_nd", "nd_relu", [x], fn="geomx_b200.ndarray.relu", npos=1, kwargs={})
    n2 = g.op("_nd", "nd_clip", [n1], fn="geomx_b200.ndarray.clip", npos=1, kwargs={"a_min": 0.1, "a_max": 0.9})
    n3 = g.op("_nd", "nd_t", [n2], fn="geomx_b200.ndarray.transpose", npos=1, kwargs={"axes": [1, 0]})
    add("nd_generic", g, g.op("_nd", "nd_sm", [n3], fn="geomx_b200.ndarray.softmax", npos=1, kwargs={"axis": 0}), {}, {"data": _r(r, 6, 9)})
    return cases


CASES = _cases()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_operator_device_matches_host(name, tmp_path):
    js, params, inputs, exact = CASES[name]
    pb = blob(params, tmp_path)
    host = serve(js, pb, inputs, 1)[0]
    dev = serve(js, pb, inputs, 2, forwards=3)                # eager, capture + replay, replay
    for i, (d, h) in enumerate(zip(dev[-1], host)):
        assert d.shape == h.shape
        if exact:
            np.testing.assert_array_equal(d, h, err_msg="%s output %d" % (name, i))
        else:
            assert rel(d, h) <= BOUND, (name, i, rel(d, h))
        np.testing.assert_array_equal(dev[0][i], d)             # the graph replays what the eager run computed


# ---------------------------------------------------------------------------------------------------------------- GPU: whole models
def _resnet(tmp_path, nnvm):
    import geomx_b200 as mx
    from geomx_b200.gluon.model_zoo import vision
    rn = vision.get_model("resnet18_v1", classes=1000)
    rn.initialize(mx.init.Xavier())
    x = np.random.RandomState(4).randn(8, 3, 112, 112).astype(np.float32)
    with mx.autograd.predict_mode():
        rn(mx.nd.array(x))
    prefix = str(tmp_path / "rn")
    rn.export(prefix, nnvm=nnvm)
    return open(prefix + "-symbol.json").read(), open(prefix + "-0000.params", "rb").read(), x


@pytest.mark.gpu
@pytest.mark.parametrize("nnvm", [False, True])
def test_resnet18_both_dialects(tmp_path, nnvm):
    js, pb, x = _resnet(tmp_path, nnvm)
    hh, dh = create(js, pb, {"data": x.shape}, 1), create(js, pb, {"data": x.shape}, 2)
    assert engine(hh) == 1 and engine(dh) == 3
    assert plan(dh) == plan(hh), (plan(dh), plan(hh))
    for h in (hh, dh):
        set_input(h, "data", x); ck(lib().GXPredForward(h))
    want, got = get_output(hh), get_output(dh)
    assert got.shape == want.shape == (8, 1000) and rel(got, want) <= BOUND, rel(got, want)
    for _ in range(2):                                            # graph replays
        ck(lib().GXPredForward(dh))
    np.testing.assert_array_equal(get_output(dh), got)
    free(hh); free(dh)


@pytest.mark.gpu
def test_handwritten_reference_file_on_device(tmp_path):
    """MXNet 0.x/1.x style: string attributes, defaults left out, pre-1.0 "param" / "attr" keys (test_predict_api's file)"""
    import geomx_b200 as mx
    nodes = [
        {"op": "null", "name": "data", "inputs": []},
        {"op": "null", "name": "bn_gamma", "attr": {"__lr_mult__": "0.0"}, "inputs": []},
        {"op": "null", "name": "bn_beta", "inputs": []},
        {"op": "null", "name": "bn_moving_mean", "inputs": []},
        {"op": "null", "name": "bn_moving_var", "inputs": []},
        {"op": "BatchNorm", "name": "bn", "param": {}, "attr": {"ctx_group": "dev1"}, "inputs": [[0, 0, 0], [1, 0, 0], [2, 0, 0], [3, 0, 1], [4, 0, 1]]},
        {"op": "Pooling", "name": "pool", "param": {"kernel": "(2, 2)", "pool_type": "max"}, "inputs": [[5, 0, 0]]},
        {"op": "LeakyReLU", "name": "lrelu", "param": {"act_type": "leaky", "slope": "0.1"}, "inputs": [[6, 0, 0]]},
        {"op": "_mul_scalar", "name": "scale", "param": {"scalar": "2.0"}, "inputs": [[7, 0, 0]]},
        {"op": "elemwise_add", "name": "res", "inputs": [[8, 0, 0], [6, 0, 0]]},
        {"op": "transpose", "name": "tr", "param": {"axes": "(0, 2, 3, 1)"}, "inputs": [[9, 0, 0]]},
        {"op": "softmax", "name": "sm", "param": {"axis": "-1"}, "inputs": [[10, 0, 0]]},
    ]
    text = json.dumps({"nodes": nodes, "arg_nodes": [0, 1, 2, 3, 4], "heads": [[11, 0, 0]]})
    rng = np.random.RandomState(2)
    vals = {"bn_gamma": rng.rand(5) + 0.5, "bn_beta": rng.randn(5), "bn_moving_mean": rng.randn(5), "bn_moving_var": rng.rand(5) + 0.5}
    f = str(tmp_path / "hand.params")
    mx.nd.save(f, {("aux:" if "moving" in k else "arg:") + k: mx.nd.array(v.astype(np.float32)) for k, v in vals.items()})
    x = rng.randn(2, 5, 6, 7).astype(np.float32)
    (host,), = serve(text, open(f, "rb").read(), {"data": x}, 1)
    (dev,), = serve(text, open(f, "rb").read(), {"data": x}, 2)[-1:]
    assert dev.shape == (2, 5, 6, 5) and rel(dev, host) <= BOUND


def _small_net(tmp_path, nnvm=True):
    g = G(nnvm)
    r = np.random.RandomState(8)
    c1 = g.op("Convolution", "c1", [g.var("data"), g.var("c1_w"), g.var("c1_b")], kernel=(3, 3), pad=(1, 1), num_filter=8)
    b1 = g.op("BatchNorm", "bn1", [c1, g.var("g1"), g.var("be1"), g.var("m1"), g.var("v1")], fix_gamma=False)
    a1 = g.op("Activation", "relu1", [b1], act_type="relu")
    p1 = g.op("Pooling", "pool1", [a1], kernel=(2, 2), stride=(2, 2), pool_type="max")
    fc = g.op("FullyConnected", "fc", [g.op("Flatten", "fl", [p1]), g.var("fc_w"), g.var("fc_b")], num_hidden=10)
    sm = g.op("SoftmaxOutput", "softmax", [fc, g.var("softmax_label")])
    params = {"c1_w": _r(r, 8, 3, 3, 3, scale=0.3), "c1_b": _r(r, 8), "g1": _r(r, 8, shift=1), "be1": _r(r, 8), "m1": _r(r, 8), "v1": np.abs(_r(r, 8)) + 0.5,
              "fc_w": _r(r, 10, 8 * 5 * 5, scale=0.1), "fc_b": _r(r, 10)}
    return g.json(sm), blob(params, tmp_path)


@pytest.mark.gpu
def test_partial_out_reshape_partial_forward(tmp_path):
    js, pb = _small_net(tmp_path)
    rng = np.random.RandomState(0)
    x = rng.randn(4, 3, 10, 10).astype(np.float32)
    # internal outputs by name
    (hp,), (dp,) = serve(js, pb, {"data": x}, 1, output_keys=["pool1", "fc_output"]), serve(js, pb, {"data": x}, 2, output_keys=["pool1", "fc_output"])
    assert len(dp) == 2 and rel(dp[0], hp[0]) <= BOUND and rel(dp[1], hp[1]) <= BOUND
    # Reshape to another batch: a new handle; the old one stays valid
    h = create(js, pb, {"data": x.shape}, 2)
    set_input(h, "data", x); ck(lib().GXPredForward(h))
    y4 = get_output(h)
    h2, n, k, ind, data = vp(), *_shapes({"data": (2, 3, 10, 10)})
    ck(lib().GXPredReshape(n, k, ind, data, h, ctypes.byref(h2)))
    assert engine(h2) == 3
    set_input(h2, "data", x[:2]); ck(lib().GXPredForward(h2))
    assert out_shape(h2) == (2, 10) and rel(get_output(h2), y4[:2]) <= BOUND
    for _ in range(2):
        ck(lib().GXPredForward(h))
    np.testing.assert_array_equal(get_output(h), y4)
    free(h2)
    ck(lib().GXPredForward(h)); np.testing.assert_array_equal(get_output(h), y4)
    # PartialForward: the host's step_left sequence, and Forward's outputs
    hh = create(js, pb, {"data": x.shape}, 1)
    set_input(hh, "data", x)
    d2 = create(js, pb, {"data": x.shape}, 2)
    set_input(d2, "data", x)
    assert partial_steps(d2) == partial_steps(hh)
    np.testing.assert_array_equal(get_output(d2), y4)
    for p in (h, hh, d2):
        free(p)


@pytest.mark.gpu
def test_graph_replay_equals_eager_and_honours_set_input(tmp_path):
    js, pb = _small_net(tmp_path, nnvm=False)
    rng = np.random.RandomState(1)
    xs = [rng.randn(3, 3, 10, 10).astype(np.float32) for _ in range(3)]
    h = create(js, pb, {"data": xs[0].shape}, 2)
    eager = create(js, pb, {"data": xs[0].shape}, 2)
    seen = []
    for x in xs:                                                  # forward 1 eager, 2 captures and launches, 3 launches
        set_input(h, "data", x); ck(lib().GXPredForward(h))
        got = get_output(h)
        set_input(eager, "data", x); partial_steps(eager)
        np.testing.assert_array_equal(got, get_output(eager))
        seen.append(got)
    assert not np.array_equal(seen[1], seen[2])
    free(h); free(eager)


@pytest.mark.gpu
def test_multi_thread_handles(tmp_path):
    js, pb = _small_net(tmp_path)
    rng = np.random.RandomState(2)
    xs = [rng.randn(2, 3, 10, 10).astype(np.float32) for _ in range(4)]
    single = create(js, pb, {"data": xs[0].shape}, 2)
    want = []
    for x in xs:
        set_input(single, "data", x); ck(lib().GXPredForward(single)); want.append(get_output(single))
    free(single)
    hs = (vp * 4)()
    n, k, ind, data = _shapes({"data": xs[0].shape})
    ck(lib().GXPredCreateMultiThread(js.encode(), pb, len(pb), 2, 0, n, k, ind, data, 4, hs))
    got, errors = [None] * 4, []

    def work(i):
        try:
            for _ in range(6):
                set_input(vp(hs[i]), "data", xs[i]); ck(lib().GXPredForward(vp(hs[i])))
            got[i] = get_output(vp(hs[i]))
        except Exception as e:                                   # noqa: BLE001 - reported below
            errors.append(repr(e))
    th = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    [t.start() for t in th]; [t.join() for t in th]
    assert not errors, errors
    for i in range(4):
        np.testing.assert_array_equal(got[i], want[i])
    free(vp(hs[0]))                                              # the original first: the clones keep the shared parameters
    for i in (3, 1, 2):
        set_input(vp(hs[i]), "data", xs[0]); ck(lib().GXPredForward(vp(hs[i])))
        np.testing.assert_array_equal(get_output(vp(hs[i])), want[0])
        free(vp(hs[i]))


@pytest.mark.gpu
def test_device_pointer_io(tmp_path):
    js, pb = _small_net(tmp_path)
    x = np.random.RandomState(5).randn(4, 3, 10, 10).astype(np.float32)
    h = create(js, pb, {"data": x.shape}, 2)
    set_input(h, "data", x); ck(lib().GXPredForward(h))
    want = get_output(h)
    xd, yd = vp(), vp()
    ck(lib().GXNDArrayCreateEx((u32 * 4)(*x.shape), 4, 2, 0, 0, 0, ctypes.byref(xd)))
    ck(lib().GXNDArrayCreateEx((u32 * 2)(4, 10), 2, 2, 0, 0, 0, ctypes.byref(yd)))
    C.nd_set(xd, x)
    px, py = vp(), vp()
    ck(lib().GXNDArrayGetData(xd, ctypes.byref(px))); ck(lib().GXNDArrayGetData(yd, ctypes.byref(py)))
    set_input(h, "data", np.zeros_like(x)); ck(lib().GXPredForward(h))
    ck(lib().GXPredSetInput(h, b"data", px, x.size))
    ck(lib().GXPredForward(h))
    ck(lib().GXPredGetOutput(h, 0, py, 40))
    np.testing.assert_array_equal(C.nd_get(yd), want)
    # a host handle still refuses device memory
    hh = create(js, pb, {"data": x.shape}, 1)
    assert lib().GXPredSetInput(hh, b"data", px, x.size) == -1 and "GXPredSetInput: device array" in C.err()
    assert lib().GXPredGetOutput(hh, 0, py, 40) == -1 and "GXPredGetOutput: device array" in C.err()
    free(h); free(hh); C.nd_free(xd); C.nd_free(yd)


@pytest.mark.gpu
def test_device_errors(tmp_path):
    js, pb = _small_net(tmp_path)
    g = G()
    c = g.op("Correlation", "corr_node", [g.var("data"), g.var("data2")])
    with pytest.raises(RuntimeError, match="Correlation.*corr_node.*" + HINT):
        create(g.json(c), b"", {"data": (1, 2, 4, 4), "data2": (1, 2, 4, 4)}, 2)
    with pytest.raises(RuntimeError, match="input c1_w has no value.*" + HINT):
        create(js, b"", {"data": (1, 3, 10, 10)}, 2)
    with pytest.raises(RuntimeError, match="no CUDA device 4096.*" + HINT):
        create(js, pb, {"data": (1, 3, 10, 10)}, 2, dev_id=4096)
    g = G()                                                       # an attribute the device cannot honour is refused at create
    a = g.op("Activation", "act_node", [g.var("data")], act_type="gelu_like")
    with pytest.raises(RuntimeError, match="act_node.*act_type.*" + HINT):
        create(g.json(a), b"", {"data": (2, 3)}, 2)
    h = create(js, pb, {"data": (1, 3, 10, 10)}, 2)
    y = np.empty(7, np.float32)
    ck(lib().GXPredForward(h))
    assert lib().GXPredGetOutput(h, 0, y.ctypes.data_as(vp), 7) == -1 and "buffer holds 7" in C.err()
    assert lib().GXPredSetInput(h, b"data", y.ctypes.data_as(vp), 7) == -1 and "expects 300 values" in C.err()
    assert lib().GXPredSetInput(h, b"nope", y.ctypes.data_as(vp), 7) == -1 and "unknown input" in C.err()
    free(h)


# ---------------------------------------------------------------------------------------------------------------- GPU: pure C
@pytest.mark.gpu
def test_pure_c_serve_gpu_example(tmp_path):
    import geomx_b200 as mx
    from geomx_b200.gluon.model_zoo import vision
    so = os.path.join(C.ROOT, "geomx_b200", "lib", "libgeomx_capi.so")
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    exe = str(tmp_path / "serve_gpu")
    subprocess.run([cc, "-O2", "-Wall", "-Werror", "-std=c99", "-I", os.path.join(C.ROOT, "geomx_b200", "include"),
                    os.path.join(C.ROOT, "examples", "c_api", "serve_gpu.c"), "-L", os.path.dirname(so), "-lgeomx_capi",
                    "-Wl,-rpath," + os.path.dirname(so), "-lm", "-o", exe], check=True)
    rn = vision.get_model("resnet18_v1", classes=10)
    rn.initialize(mx.init.Xavier())
    with mx.autograd.predict_mode():
        rn(mx.nd.array(np.zeros((1, 3, 32, 32), np.float32)))
    prefix = str(tmp_path / "rn")
    rn.export(prefix)
    r = subprocess.run([exe, prefix + "-symbol.json", prefix + "-0000.params", "8", "3", "32", "32"], capture_output=True, text=True, timeout=300)
    print(r.stdout)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "max relative difference" in r.stdout and "engine 3" in r.stdout
