"""Device execution through the flat C ABI (GXNDArrayCreateEx, GXExecutorSimpleBindEx, the device executor of csrc/runtime/device_exec.h,
imperative calls on device arrays, the sgd_update / sgd_mom_update / adam_update operators), driven through ctypes only.  The host executor
(train_exec.h, itself checked against torch in test_c_api_graph.py) is the oracle of every device result."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

import _capi as C
from _capi import ck, lib, u32, vp, cp
from test_c_api_graph import _cnn

BOUND = 1e-4          # max |device - host| / max |host|


# ---------------------------------------------------------------------------------------------------------------- helpers
def nd_create_ex(arr, dev_type=2, dev_id=0):
    arr = np.ascontiguousarray(arr, dtype=np.float32)
    h = vp()
    ck(lib().GXNDArrayCreateEx((u32 * max(arr.ndim, 1))(*arr.shape), arr.ndim, dev_type, dev_id, 0, 0, ctypes.byref(h)))
    C.nd_set(h, arr)
    return h


def context(h):
    t, i = ctypes.c_int(), ctypes.c_int()
    ck(lib().GXNDArrayGetContext(h, ctypes.byref(t), ctypes.byref(i)))
    return t.value, i.value


def simple_bind_ex(sym, shapes, dev_type, dev_id=0, grad_req="write", no_grad=()):
    keys = list(shapes.keys())
    ind, data = [0], []
    for k in keys:
        data += list(shapes[k]); ind.append(len(data))
    ex, na, nx = vp(), u32(), u32()
    a, g, x = ctypes.POINTER(vp)(), ctypes.POINTER(vp)(), ctypes.POINTER(vp)()
    rc = lib().GXExecutorSimpleBindEx(sym, dev_type, dev_id, len(keys), C.strs(keys), (u32 * len(ind))(*ind), (u32 * len(data))(*data), grad_req.encode(),
                                      len(no_grad), C.strs(list(no_grad)), ctypes.byref(ex), ctypes.byref(na), ctypes.byref(a), ctypes.byref(g),
                                      ctypes.byref(nx), ctypes.byref(x))
    if rc != 0:
        raise RuntimeError(C.err())
    names, auxn = C.list_arguments(sym), C.list_aux(sym)
    return (ex, {names[i]: vp(a[i]) for i in range(na.value)}, {names[i]: vp(g[i]) for i in range(na.value) if g[i]},
            {auxn[i]: vp(x[i]) for i in range(nx.value)})


def rel(d, h):
    d, h = np.asarray(d, np.float64), np.asarray(h, np.float64)
    return float(np.abs(d - h).max() / max(np.abs(h).max(), 1e-30))


def invoke_into(opname, inputs, out, **attrs):
    keys, vals = list(attrs.keys()), [str(v) for v in attrs.values()]
    n, outs = ctypes.c_int(1), C.handles([out])
    po = ctypes.cast(outs, ctypes.POINTER(vp))
    rc = lib().GXImperativeInvokeByName(opname.encode(), len(inputs), C.handles(list(inputs)), ctypes.byref(n), ctypes.byref(po), len(keys), C.strs(keys),
                                        C.strs(vals))
    if rc != 0:
        raise RuntimeError(C.err())


def run_both(net, shapes, values, is_train=True, grad_req="write", no_grad=(), forwards=1, backward=True):
    """binds `net` on the host and on gpu(0) with the same values and the same random head gradients (loss heads ignore them); returns
    {name: (device, host)} for outputs, gradients and auxiliary states"""
    res = {}
    heads = [np.random.RandomState(17).randn(*s).astype(np.float32) for s in C.infer_shape(net, **shapes)[1]]
    for dev_type in (1, 2):
        ex, args, grads, aux = simple_bind_ex(net, shapes, dev_type, grad_req=grad_req, no_grad=no_grad)
        for k, v in values.items():
            C.nd_set(args[k] if k in args else aux[k], v)
        if grad_req == "add":
            for k, g in grads.items():
                C.nd_set(g, np.full(C.nd_shape(g), 0.25, np.float32))
        for _ in range(forwards):
            outs = C.forward(ex, is_train)
        if backward:
            C.backward(ex, [nd_create_ex(h, dev_type) for h in heads])
        got = {"out%d" % i: o for i, o in enumerate(outs)}
        if backward:
            got.update({"grad:" + k: C.nd_get(g) for k, g in grads.items()})
        got.update({"aux:" + k: C.nd_get(a) for k, a in aux.items()})
        for k, v in got.items():
            res.setdefault(k, [None, None])[dev_type - 1] = v
        ck(lib().GXExecutorFree(ex))
    return {k: (v[1], v[0]) for k, v in res.items()}


def assert_close(res, bound=BOUND):
    for k, (d, h) in res.items():
        assert d.shape == h.shape, (k, d.shape, h.shape)
        assert rel(d, h) <= bound, (k, rel(d, h))


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_create_ex_host_and_refusals():
    a = nd_create_ex(np.arange(6).reshape(2, 3), dev_type=1)
    b = C.nd_create(np.arange(6).reshape(2, 3))
    assert np.array_equal(C.nd_get(a), C.nd_get(b)) and C.nd_shape(a) == (2, 3)
    assert context(a) == (1, 0) and context(b) == (1, 0)
    dt = ctypes.c_int(); ck(lib().GXNDArrayGetDType(a, ctypes.byref(dt))); assert dt.value == 0
    h = vp()
    assert lib().GXNDArrayCreateEx((u32 * 1)(4), 1, 2, 4096, 0, 0, ctypes.byref(h)) == -1
    assert "device 4096" in C.err() or "kernel library" in C.err()
    assert lib().GXNDArrayCreateEx((u32 * 1)(4), 1, 7, 0, 0, 0, ctypes.byref(h)) == -1 and "dev_type 7" in C.err()
    assert lib().GXNDArrayCreateEx((u32 * 1)(4), 1, 2, 0, 0, 1, ctypes.byref(h)) == -1 and "float32" in C.err()
    for x in (a, b):
        C.nd_free(x)


def _update_case(rng, n=37):
    return (rng.randn(n) * 3).astype(np.float32), rng.randn(n).astype(np.float32), rng.randn(n).astype(np.float32) * 0.1, (rng.rand(n) * 0.1).astype(np.float32)


UPDATES = [("sgd_update", dict(lr=0.1, wd=0.01, rescale_grad=0.5, clip_gradient=0.3)), ("sgd_update", dict(lr=0.05)),
           ("sgd_mom_update", dict(lr=0.1, momentum=0.9, wd=0.001, rescale_grad=2.0)), ("sgd_mom_update", dict(lr=0.1, momentum=0.5, clip_gradient=0.4)),
           ("adam_update", dict(lr=0.01, beta1=0.8, beta2=0.99, epsilon=1e-6, wd=0.01, rescale_grad=0.5)), ("adam_update", dict(lr=0.01, clip_gradient=0.5))]


def _mx_update(mx, op, w, g, m, v, attrs, ctx):
    W, G, M, V = (mx.nd.array(a, ctx=ctx) for a in (w, g, m, v))
    if op == "sgd_update":
        r = mx.nd.sgd_update(W, G, out=W, **attrs)
    elif op == "sgd_mom_update":
        r = mx.nd.sgd_mom_update(W, G, M, out=W, **attrs)
    else:
        r = mx.nd.adam_update(W, G, M, V, out=W, **attrs)
    return r.asnumpy(), M.asnumpy(), V.asnumpy()


def _states(op, m, v):
    return {"sgd_update": [], "sgd_mom_update": [m], "adam_update": [m, v]}[op]


@pytest.mark.parametrize("op,attrs", UPDATES)
def test_update_operators_on_host_match_ndarray(op, attrs):
    import geomx_b200 as mx
    w, g, m, v = _update_case(np.random.RandomState(4))
    W, G = C.nd_create(w), C.nd_create(g)
    S = [C.nd_create(s) for s in _states(op, m, v)]
    invoke_into(op, [W, G] + S, W, **attrs)                      # out = weight, states in place
    want_w, want_m, want_v = _mx_update(mx, op, w, g, m, v, attrs, mx.cpu())
    np.testing.assert_allclose(C.nd_get(W), want_w, rtol=1e-6, atol=1e-7)
    if op != "sgd_update":
        np.testing.assert_allclose(C.nd_get(S[0]), want_m, rtol=1e-6, atol=1e-7)
    if op == "adam_update":
        np.testing.assert_allclose(C.nd_get(S[1]), want_v, rtol=1e-6, atol=1e-7)


def test_update_operators_infer_shape():
    w, g, m, v = C.var("w"), C.var("g"), C.var("m"), C.var("v")
    s = C.op("adam_update", "adam", kwinputs={"weight": w, "grad": g, "mean": m, "var": v}, lr=0.1)
    assert C.list_arguments(s) == ["w", "g"] and C.list_aux(s) == ["m", "v"]
    a, o, x, ok = C.infer_shape(s, w=(3, 4))
    assert ok and a == [(3, 4), (3, 4)] and o == [(3, 4)] and x == [(3, 4), (3, 4)]
    s2 = C.op("sgd_mom_update", "mom", kwinputs={"weight": C.var("w2"), "grad": C.var("g2"), "mom": C.var("m2")}, lr=0.1)
    assert C.list_aux(s2) == ["m2"] and C.infer_shape(s2, w2=(5,))[1] == [(5,)]
    s3 = C.op("sgd_update", "sgd", kwinputs={"weight": C.var("w3"), "grad": C.var("g3")}, lr=0.1)
    assert C.list_aux(s3) == [] and C.infer_shape(s3, w3=(2, 2))[1] == [(2, 2)]
    with pytest.raises(RuntimeError, match="expected"):
        C.infer_shape(s3, w3=(2, 2), g3=(3,))


# ---------------------------------------------------------------------------------------------------------------- GPU: arrays
@pytest.mark.gpu
def test_device_arrays_copy_context_save(tmp_path):
    import geomx_b200 as mx
    x = np.random.RandomState(0).randn(3, 5).astype(np.float32)
    d = nd_create_ex(x)
    assert context(d) == (2, 0) and C.nd_shape(d) == (3, 5)
    np.testing.assert_array_equal(C.nd_get(d), x)
    p = vp(); ck(lib().GXNDArrayGetData(d, ctypes.byref(p))); assert p.value
    ck(lib().GXNDArrayWaitToRead(d)); ck(lib().GXNDArrayWaitToWrite(d)); ck(lib().GXNDArrayWaitAll())
    fname = str(tmp_path / "d.params").encode()
    ck(lib().GXNDArraySave(fname, 1, C.handles([d]), C.strs(["arg:x"])))
    np.testing.assert_array_equal(mx.nd.load(fname.decode())["arg:x"].asnumpy(), x)
    size, buf = ctypes.c_size_t(), ctypes.c_char_p()
    ck(lib().GXNDArraySaveRawBytes(d, ctypes.byref(size), ctypes.byref(buf)))
    back = vp(); ck(lib().GXNDArrayLoadFromRawBytes(ctypes.string_at(buf, size.value), size.value, ctypes.byref(back)))
    assert context(back) == (1, 0)
    np.testing.assert_array_equal(C.nd_get(back), x)
    C.nd_free(d); C.nd_free(back)


@pytest.mark.gpu
def test_refusals_name_the_function():
    d = nd_create_ex(np.ones((4, 2)))
    h = C.nd_create(np.ones((4, 2)))
    out = vp()
    for fn, call in (("GXNDArraySlice", lambda: lib().GXNDArraySlice(d, 0, 1, ctypes.byref(out))),
                     ("GXNDArrayAt", lambda: lib().GXNDArrayAt(d, 0, ctypes.byref(out))),
                     ("GXNDArrayReshape", lambda: lib().GXNDArrayReshape(d, 1, (ctypes.c_int * 1)(8), ctypes.byref(out))),
                     ("GXNDArrayDetach", lambda: lib().GXNDArrayDetach(d, ctypes.byref(out))),
                     ("GXAutogradMarkVariables", lambda: lib().GXAutogradMarkVariables(1, C.handles([d]), (u32 * 1)(1), C.handles([d]))),
                     ("GXAutogradBackward", lambda: lib().GXAutogradBackward(1, C.handles([d]), None, 0))):
        assert call() == -1 and fn in C.err() and "device array" in C.err(), (fn, C.err())
    # raw-pointer groups: a device array's buffer is refused
    p = vp(); ck(lib().GXNDArrayGetData(d, ctypes.byref(p)))
    lib().GXGetLastError.restype = cp
    assert lib().GXKVStoreInit(None, 3, p, ctypes.c_size_t(8), 0) == -1 and "GXKVStoreInit: device array" in lib().GXGetLastError().decode()
    assert lib().GXKVStorePush(None, 3, p, ctypes.c_size_t(8), 0, 0, None) == -1 and "GXKVStorePush: device array" in lib().GXGetLastError().decode()
    assert lib().GXPredSetInput(None, b"data", p, 8) == -1 and "GXPredSetInput: device array" in C.err()
    net = C.op("FullyConnected", "fc", [C.var("data")], num_hidden=2)
    # mixed host / device arrays in one Bind
    w, b = nd_create_ex(np.ones((2, 2))), C.nd_create(np.zeros(2))
    ex = vp()
    assert lib().GXExecutorBind(net, 2, 0, 3, C.handles([d, w, b]), None, None, 0, None, ctypes.byref(ex)) == -1 and "GXExecutorBind" in C.err()
    # an operator outside the device set is refused at bind with the node's name
    bad = C.op("MakeLoss", "l", [C.op("LayerNorm", "ln_node", [C.var("data")])])
    with pytest.raises(RuntimeError, match="ln_node"):
        simple_bind_ex(bad, {"data": (2, 4)}, 2)
    dil = C.op("Convolution", "dil_conv", [C.var("data")], kernel="(3, 3)", num_filter=2, dilate="(2, 2)")
    with pytest.raises(RuntimeError, match="dil_conv.*dilated"):
        simple_bind_ex(dil, {"data": (1, 1, 8, 8)}, 2)
    # device inputs while autograd is recording
    with C.record():
        with pytest.raises(RuntimeError, match="GXImperativeInvoke.*recording"):
            C.invoke("relu", [d])
    for x in (d, h, w, b):
        C.nd_free(x)


# ---------------------------------------------------------------------------------------------------------------- GPU: per operator
def _v(rng, *shape, scale=1.0, shift=0.0):
    return (rng.randn(*shape) * scale + shift).astype(np.float32)


def _op_cases():
    x = C.var("data")
    r = np.random.RandomState(7)
    cases = {}

    def loss(sym, name="l"):
        return C.op("MakeLoss", name, [sym], grad_scale=0.5)

    def add(name, sym, shapes, values, **kw):
        cases[name] = (sym, shapes, values, kw)

    add("fc", C.op("FullyConnected", "fc", [x], num_hidden=7), {"data": (4, 3, 5)}, {"data": _v(r, 4, 3, 5), "fc_weight": _v(r, 7, 15), "fc_bias": _v(r, 7)})
    add("fc_nobias_noflat", C.op("FullyConnected", "fc", [x], num_hidden=6, no_bias=True, flatten=False), {"data": (3, 2, 8)},
        {"data": _v(r, 3, 2, 8), "fc_weight": _v(r, 6, 8)})
    add("conv", C.op("Convolution", "c", [x], kernel="(3, 3)", stride="(2, 2)", pad="(1, 1)", num_filter=8), {"data": (2, 3, 9, 9)},
        {"data": _v(r, 2, 3, 9, 9), "c_weight": _v(r, 8, 3, 3, 3, scale=0.3), "c_bias": _v(r, 8)})
    add("conv_groups", C.op("Convolution", "c", [x], kernel="(3, 2)", pad="(1, 0)", num_filter=6, num_group=2, no_bias=True), {"data": (2, 4, 6, 5)},
        {"data": _v(r, 2, 4, 6, 5), "c_weight": _v(r, 6, 2, 3, 2, scale=0.3)})
    add("conv_depthwise", C.op("Convolution", "c", [x], kernel="(3, 3)", pad="(1, 1)", num_filter=4, num_group=4), {"data": (2, 4, 7, 7)},
        {"data": _v(r, 2, 4, 7, 7), "c_weight": _v(r, 4, 1, 3, 3), "c_bias": _v(r, 4)})
    for fg in (True, False):
        add("bn_fix_gamma_%d" % fg, C.op("BatchNorm", "bn", [x], fix_gamma=fg, eps=1e-5, momentum=0.8), {"data": (4, 3, 5, 5)},
            {"data": _v(r, 4, 3, 5, 5, shift=0.5), "bn_gamma": _v(r, 3, shift=1.0), "bn_beta": _v(r, 3), "bn_moving_mean": _v(r, 3), "bn_moving_var": np.ones(3, np.float32)})
    add("bn_global", C.op("BatchNorm", "bn", [x], fix_gamma=False, use_global_stats=True), {"data": (4, 3, 2, 3)},
        {"data": _v(r, 4, 3, 2, 3), "bn_gamma": _v(r, 3, shift=1.0), "bn_beta": _v(r, 3), "bn_moving_mean": _v(r, 3), "bn_moving_var": np.full(3, 2.0, np.float32)})
    add("bn_2d", C.op("BatchNorm", "bn", [x], fix_gamma=False), {"data": (8, 5)},
        {"data": _v(r, 8, 5), "bn_gamma": _v(r, 5, shift=1.0), "bn_beta": _v(r, 5), "bn_moving_mean": np.zeros(5, np.float32), "bn_moving_var": np.ones(5, np.float32)})
    pools = {"max_valid": dict(kernel="(3, 3)", stride="(2, 2)", pad="(1, 1)", pool_type="max"),
             "max_full": dict(kernel="(3, 3)", stride="(2, 2)", pad="(1, 1)", pool_type="max", pooling_convention="full"),
             "avg_pad": dict(kernel="(3, 3)", stride="(2, 2)", pad="(1, 1)", pool_type="avg", count_include_pad=True),
             "avg_nopad": dict(kernel="(3, 3)", stride="(2, 2)", pad="(1, 1)", pool_type="avg", count_include_pad=False, pooling_convention="full"),
             "global_avg": dict(kernel="(1, 1)", global_pool=True, pool_type="avg"), "global_max": dict(kernel="(1, 1)", global_pool=True, pool_type="max"),
             "sum": dict(kernel="(2, 2)", stride="(1, 1)", pool_type="sum")}
    for k, at in pools.items():
        add("pool_" + k, C.op("Pooling", "p", [x], **at), {"data": (2, 3, 7, 7)}, {"data": _v(r, 2, 3, 7, 7)})
    for act in ("relu", "sigmoid", "tanh", "softrelu", "softsign"):
        add("act_" + act, C.op("Activation", "a", [x], act_type=act), {"data": (3, 17)}, {"data": _v(r, 3, 17, scale=2.0)})
    add("leaky", C.op("LeakyReLU", "a", [x], act_type="leaky", slope=0.1), {"data": (3, 17)}, {"data": _v(r, 3, 17)})
    a, b = C.var("a"), C.var("b")
    for op in ("elemwise_add", "elemwise_sub", "elemwise_mul"):
        add(op, C.op(op, "e", [a, b]), {"a": (3, 4), "b": (3, 4)}, {"a": _v(r, 3, 4), "b": _v(r, 3, 4)})
    for op in ("broadcast_add", "broadcast_sub", "broadcast_mul"):
        add(op, C.op(op, "e", [a, b]), {"a": (3, 1, 4), "b": (2, 1)}, {"a": _v(r, 3, 1, 4), "b": _v(r, 2, 1)})
    c = C.var("c")
    add("add_n", C.op("add_n", "s", [a, b, c], num_args=3), {"a": (2, 5), "b": (2, 5), "c": (2, 5)}, {"a": _v(r, 2, 5), "b": _v(r, 2, 5), "c": _v(r, 2, 5)})
    add("concat_axis1", C.op("Concat", "cat", [a, b], dim=1, num_args=2), {"a": (2, 3, 4), "b": (2, 5, 4)}, {"a": _v(r, 2, 3, 4), "b": _v(r, 2, 5, 4)})
    add("concat_axis2", C.op("Concat", "cat", [a, b], dim=2, num_args=2), {"a": (2, 3, 4), "b": (2, 3, 1)}, {"a": _v(r, 2, 3, 4), "b": _v(r, 2, 3, 1)})
    add("copies", loss(C.op("elemwise_add", "e", [C.op("Reshape", "rs", [C.op("Flatten", "fl", [a])], shape="(4, 6)"),
                                                     C.op("BlockGrad", "bg", [C.op("identity", "id", [b])])])),
        {"a": (2, 3, 4), "b": (4, 6)}, {"a": _v(r, 2, 3, 4), "b": _v(r, 4, 6)})
    lab = C.var("label")
    for norm in ("null", "batch", "valid"):
        add("softmax_output_" + norm, C.op("SoftmaxOutput", "sm", kwinputs={"data": x, "label": lab}, normalization=norm, grad_scale=1.5),
            {"data": (6, 10)}, {"data": _v(r, 6, 10), "label": r.randint(0, 10, 6).astype(np.float32)}, no_grad=("label",))
    yn = r.randint(0, 4, (2, 5)).astype(np.float32); yn[0, 1] = -1; yn[1, 3] = -1
    add("softmax_output_ignore", C.op("SoftmaxOutput", "sm", kwinputs={"data": x, "label": lab}, multi_output=True, use_ignore=True, ignore_label=-1,
                                      normalization="valid"), {"data": (2, 4, 5)}, {"data": _v(r, 2, 4, 5), "label": yn}, no_grad=("label",))
    add("softmax_axis1", C.op("softmax", "s", [x], axis=1), {"data": (2, 4, 3)}, {"data": _v(r, 2, 4, 3)})
    add("log_softmax", C.op("log_softmax", "s", [x], axis=-1), {"data": (3, 9)}, {"data": _v(r, 3, 9)})
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(_op_cases().keys()))
def test_operator_device_matches_host(name):
    sym, shapes, values, kw = _op_cases()[name]
    assert_close(run_both(sym, shapes, values, **kw))


# ---------------------------------------------------------------------------------------------------------------- GPU: graphs
def _residual_block():
    x = C.var("data")
    c1 = C.op("Convolution", "c1", [x], kernel="(3, 3)", pad="(1, 1)", num_filter=4, no_bias=True)
    b1 = C.op("BatchNorm", "bn1", [c1], fix_gamma=False)
    r1 = C.op("Activation", "r1", [b1], act_type="relu")
    c2 = C.op("Convolution", "c2", [r1], kernel="(3, 3)", pad="(1, 1)", num_filter=4, no_bias=True)
    b2 = C.op("BatchNorm", "bn2", [c2], fix_gamma=False)
    s = C.op("elemwise_add", "add", [b2, x])                      # fan-out of data: the identity path and c1
    r2 = C.op("Activation", "r2", [s], act_type="relu")
    p = C.op("Pooling", "gp", [r2], kernel="(1, 1)", global_pool=True, pool_type="avg")
    f = C.op("FullyConnected", "fc", [p], num_hidden=3)
    return C.op("SoftmaxOutput", "sm", kwinputs={"data": f, "label": C.var("label")}, normalization="batch")


@pytest.mark.gpu
@pytest.mark.parametrize("grad_req", ["write", "add"])
def test_residual_block_fan_out_and_add(grad_req):
    net = _residual_block()
    r = np.random.RandomState(11)
    shapes = {"data": (4, 4, 6, 6)}
    a, _, x, _ = C.infer_shape(net, **shapes)
    values = {}
    for n, s in zip(C.list_arguments(net), a):
        values[n] = r.randint(0, 3, s).astype(np.float32) if n == "label" else (r.randn(*s) * 0.5).astype(np.float32)
    for n, s in zip(C.list_aux(net), x):
        values[n] = np.ones(s, np.float32) if n.endswith("var") else np.zeros(s, np.float32)
    res = run_both(net, shapes, values, grad_req=grad_req, no_grad=("label",), forwards=3)
    assert "grad:data" in res and "aux:bn1_moving_mean" in res
    assert_close(res)


@pytest.mark.gpu
def test_demo_cnn_training_20_sgd_steps_matches_host():
    net = _cnn()
    B = 16
    r = np.random.RandomState(3)
    names = C.list_arguments(net)
    shapes = dict(zip(names, C.infer_shape(net, data=(B, 1, 28, 28))[0]))
    # Xavier-uniform weights, zero biases and lr 0.01: a regime where 20 steps do not amplify rounding differences (with N(0, 0.1) weights and
    # lr 0.05, a 1e-6 relative perturbation of the initial weights alone moves the host's own loss curve by ~3e-3)
    params = {n: ((r.rand(*s) * 2 - 1) * np.sqrt(3.0 / (np.prod(s) / s[0]))).astype(np.float32) if n.endswith("weight") else np.zeros(s, np.float32)
              for n, s in shapes.items() if n not in ("data", "softmax_label")}
    batches = [(r.rand(B, 1, 28, 28).astype(np.float32), r.randint(0, 10, B).astype(np.float32)) for _ in range(4)]
    curves, finals = [], []
    for dev_type in (1, 2):
        ex, args, grads, _ = simple_bind_ex(net, {"data": (B, 1, 28, 28)}, dev_type, no_grad=("data", "softmax_label"))
        for k, v in params.items():
            C.nd_set(args[k], v)
        losses = []
        for step in range(20):
            X, y = batches[step % len(batches)]
            C.nd_set(args["data"], X); C.nd_set(args["softmax_label"], y)
            p = C.forward(ex, True)[0]
            losses.append(float(-np.log(p[np.arange(B), y.astype(int)] + 1e-12).mean()))
            C.backward(ex)
            for k in params:
                invoke_into("sgd_update", [args[k], grads[k]], args[k], lr=0.01)
        curves.append(np.array(losses)); finals.append({k: C.nd_get(args[k]) for k in params})
        ck(lib().GXExecutorFree(ex))
    host, dev = curves
    assert rel(dev, host) <= 1e-3, (host, dev)
    worst = max(rel(finals[1][k], finals[0][k]) for k in params)
    print("20 SGD steps: loss curve rel err %.3g, worst final-weight rel err %.3g" % (rel(dev, host), worst))
    assert worst <= 1e-3 and host[-1] < host[0]


@pytest.mark.gpu
def test_resnet18_inference_matches_host_predictor(tmp_path):
    import geomx_b200 as mx
    from geomx_b200 import predictor
    from geomx_b200.gluon.model_zoo import vision
    rn = vision.get_model("resnet18_v1", classes=10)
    rn.initialize()
    xi = np.random.RandomState(2).randn(8, 3, 32, 32).astype(np.float32)
    with mx.autograd.predict_mode():
        rn(mx.nd.array(xi))
    rn.export(str(tmp_path / "rn"))
    js = open(str(tmp_path / "rn-symbol.json")).read()
    p = predictor.Predictor(js, open(str(tmp_path / "rn-0000.params"), "rb").read(), {"data": xi.shape})
    p.forward(data=xi)
    want = p.get_output(0)
    sym = C.sym_from_json(js)
    ex, args, _, aux = simple_bind_ex(sym, {"data": xi.shape}, 2, grad_req="null")
    saved = mx.nd.load(str(tmp_path / "rn-0000.params"))
    for k, v in saved.items():
        kind, name = k.split(":", 1)
        C.nd_set((args if kind == "arg" else aux)[name], v.asnumpy())
    C.nd_set(args["data"], xi)
    got = C.forward(ex, False)[0]
    assert got.shape == want.shape and rel(got, want) <= BOUND, rel(got, want)
    ck(lib().GXExecutorFree(ex))


@pytest.mark.gpu
def test_dropout_mask():
    p = 0.3
    net = C.op("Dropout", "do", [C.var("data")], p=p)
    xn = np.random.RandomState(5).rand(64, 256).astype(np.float32) + 0.5

    def run(seed, is_train):
        ck(lib().GXRandomSeed(seed))
        ex, args, grads, _ = simple_bind_ex(net, {"data": xn.shape}, 2)
        C.nd_set(args["data"], xn)
        y = C.forward(ex, is_train)[0]
        g = None
        if is_train:
            C.backward(ex); g = C.nd_get(grads["data"])
        ck(lib().GXExecutorFree(ex))
        return y, g

    y0, _ = run(1, False)
    np.testing.assert_array_equal(y0, xn)
    y, g = run(1, True)
    kept = y != 0
    n = kept.size
    assert abs(kept.mean() - (1 - p)) <= 3 * np.sqrt(p * (1 - p) / n)
    np.testing.assert_allclose(y[kept], xn[kept] / (1 - p), rtol=1e-6)
    np.testing.assert_allclose(g, kept / (1 - p), rtol=1e-6)           # backward with the same mask (head gradient = ones)
    y2, _ = run(1, True)
    np.testing.assert_array_equal(y2 != 0, kept)
    y3, _ = run(2, True)
    assert (y3 != 0).mean() != kept.mean() or not np.array_equal(y3 != 0, kept)


@pytest.mark.gpu
@pytest.mark.parametrize("op,attrs", UPDATES)
def test_update_operators_on_device_match_ndarray_cuda(op, attrs):
    import geomx_b200 as mx
    w, g, m, v = _update_case(np.random.RandomState(9), n=1000)
    W, G = nd_create_ex(w), nd_create_ex(g)
    S = [nd_create_ex(s) for s in _states(op, m, v)]
    invoke_into(op, [W, G] + S, W, **attrs)
    want_w, want_m, want_v = _mx_update(mx, op, w, g, m, v, attrs, mx.gpu(0))
    assert rel(C.nd_get(W), want_w) <= 1e-6
    if op != "sgd_update":
        assert rel(C.nd_get(S[0]), want_m) <= 1e-6
    if op == "adam_update":
        assert rel(C.nd_get(S[1]), want_v) <= 1e-6
    # output created by the call, input untouched when out is not given
    G2 = nd_create_ex(g)
    fresh = C.invoke("sgd_update", [G2, G2], lr=0.5)
    assert context(fresh) == (2, 0)
    np.testing.assert_allclose(C.nd_get(fresh), g * 0.5, rtol=1e-6)
    np.testing.assert_array_equal(C.nd_get(G2), g)


@pytest.mark.gpu
def test_pure_c_gpu_example(tmp_path):
    import geomx_b200 as mx
    so = os.path.join(C.ROOT, "geomx_b200", "lib", "libgeomx_capi.so")
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    exe = str(tmp_path / "train_cnn_gpu")
    subprocess.run([cc, "-O2", "-Wall", "-Werror", "-std=c99", "-I", os.path.join(C.ROOT, "geomx_b200", "include"),
                    os.path.join(C.ROOT, "examples", "c_api", "train_cnn_gpu.c"), "-L", os.path.dirname(so), "-lgeomx_capi",
                    "-Wl,-rpath," + os.path.dirname(so), "-lm", "-o", exe], check=True)
    r = subprocess.run([exe, "40", str(tmp_path / "cnn")], capture_output=True, text=True, timeout=300)
    print(r.stdout)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "predictor agrees with the device executor on 32/32" in r.stdout
    sym, arg, aux = mx.model.load_checkpoint(str(tmp_path / "cnn"), 1)
    assert sym.list_outputs() == ["softmax_output"] and tuple(arg["fc0_weight"].shape) == (256, 512) and aux == {}
