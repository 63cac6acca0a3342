"""GXKVStoreInitND / PushND / PullND / SetUpdater (csrc/runtime/kvstore_nd.h, csrc/kernels/kv_comm.cu): the KVStore on NDArray handles.

CPU: the `local` store against the Python `mx.kv.create('local')`, every refusal, and a 4-process dist_sync job whose workers drive one
parameter through the raw-buffer forms and the same parameter through the NDArray forms.  GPU: the reduction kernels against a numpy port of
Quantize2Bit / Dequantize2Bit, `device` against `local`, device arrays on the dist plane, and the GPU twin of the distributed C example."""
import ctypes
import json
import os
import re
import shutil
import socket
import subprocess
import sys
import time

import numpy as np
import pytest

import _capi as C
from geomx_b200 import runtime

pytestmark = pytest.mark.skipif(not runtime.available(), reason="native runtime not built")
vp = ctypes.c_void_p
HERE = os.path.dirname(os.path.abspath(__file__))
UPDATER = ctypes.CFUNCTYPE(None, ctypes.c_int, vp, vp, vp)


def lib():
    L = C.lib()
    L.GXGetLastError.restype = ctypes.c_char_p
    return L


def kv_err():
    return lib().GXGetLastError().decode(errors="replace")


def kck(rc):
    assert rc == 0, kv_err()


def kv_create(kind):
    h = vp()
    kck(lib().GXKVStoreCreate(kind.encode(), ctypes.byref(h)))
    return h


def keys_of(ks):
    return (ctypes.c_int * max(len(ks), 1))(*ks)


def init(h, ks, vals):
    return lib().GXKVStoreInitND(h, len(ks), keys_of(ks), C.handles(vals))


def push(h, ks, vals):
    return lib().GXKVStorePushND(h, len(ks), keys_of(ks), C.handles(vals), 0)


def pull(h, ks, outs):
    return lib().GXKVStorePullND(h, len(ks), keys_of(ks), C.handles(outs), 0)


def dev_nd(arr, dev):
    arr = np.ascontiguousarray(arr, dtype=np.float32)
    h = vp()
    C.ck(lib().GXNDArrayCreateEx((ctypes.c_uint32 * arr.ndim)(*arr.shape), arr.ndim, 2, dev, 0, 0, ctypes.byref(h)))
    C.nd_set(h, arr)
    return h


def context(h):
    t, d = ctypes.c_int(), ctypes.c_int()
    C.ck(lib().GXNDArrayGetContext(h, ctypes.byref(t), ctypes.byref(d)))
    return t.value, d.value


def host_view(h):
    """numpy view of a host NDArray's bytes (updaters on `local` work in place)"""
    p = vp()
    C.ck(lib().GXNDArrayGetData(h, ctypes.byref(p)))
    shape = C.nd_shape(h)
    return np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctypes.c_float)), shape=shape)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


# ---------------------------------------------------------------------------------------------------------------- numpy oracle of 2-bit
def quantize_2bit(grad, residual, thr):
    """Port of gradient_compression.h Quantize2Bit: returns the words, updates residual in place."""
    n, thr = grad.size, np.float32(thr)
    r = (residual + grad).astype(np.float32)
    code = np.zeros(n, np.uint32)
    pos, neg = r >= thr, r <= -thr
    code[pos] = 3
    code[~pos & neg] = 2
    r[pos] = r[pos] - thr
    r[~pos & neg] = r[~pos & neg] + thr
    residual[:] = r
    words = np.zeros((n + 15) // 16, np.uint32)
    j = np.arange(n) & 15
    shift = ((j >> 2) << 3) + (6 - 2 * (j & 3))
    np.bitwise_or.at(words, np.arange(n) >> 4, code << shift.astype(np.uint32))
    return words


def dequantize_2bit(words, n, thr):
    j = np.arange(n) & 15
    shift = (((j >> 2) << 3) + (6 - 2 * (j & 3))).astype(np.uint32)
    code = (words[np.arange(n) >> 4] >> shift) & 3
    out = np.zeros(n, np.float32)
    out[code == 3] = np.float32(thr)
    out[code == 2] = -np.float32(thr)
    out[out == 0] = 0.0
    return out


# ================================================================================================================ CPU: local store
def test_local_store_matches_python_local():
    """One sequence through GXKVStore*ND on `local` and through mx.kv.create('local'): init, a push with a repeated key, a pull into three
    outputs, assignment without an updater, then a ctypes updater.  Bitwise equal."""
    import geomx_b200 as mx
    rng = np.random.default_rng(0)
    a3, a5 = rng.standard_normal((2, 3)).astype(np.float32), rng.standard_normal(5).astype(np.float32)
    xs = [rng.standard_normal((2, 3)).astype(np.float32) for _ in range(5)]
    y = rng.standard_normal(5).astype(np.float32)

    kv = mx.kv.create("local")
    kv.init(3, mx.nd.array(a3)); kv.init(5, mx.nd.array(a5))
    kv.push(3, [mx.nd.array(xs[0]), mx.nd.array(xs[1]), mx.nd.array(xs[2])]); kv.push(5, mx.nd.array(y))
    po = [mx.nd.zeros((2, 3)) for _ in range(3)]
    kv.pull(3, out=po)
    p5 = mx.nd.zeros(5); kv.pull(5, out=p5)
    py_assign = [o.asnumpy().copy() for o in po] + [p5.asnumpy().copy()]

    def py_upd(key, recv, local):
        local[:] = local + recv * 0.5
    kv._set_updater(py_upd)
    kv.push(3, [mx.nd.array(xs[3]), mx.nd.array(xs[4])])
    kv.pull(3, out=po[0])
    py_updated = po[0].asnumpy().copy()

    h = kv_create("local")
    t = ctypes.c_char_p()
    kck(lib().GXKVStoreGetType(h, ctypes.byref(t))); assert t.value == b"local"
    r, n = ctypes.c_int(-1), ctypes.c_int(-1)
    kck(lib().GXKVStoreGetRank(h, ctypes.byref(r))); kck(lib().GXKVStoreGetGroupSize(h, ctypes.byref(n)))
    assert (r.value, n.value) == (0, 1)
    kck(lib().GXKVStoreBarrier(h))
    kck(init(h, [3, 5], [C.nd_create(a3), C.nd_create(a5)]))
    kck(push(h, [3, 5, 3, 3], [C.nd_create(xs[0]), C.nd_create(y), C.nd_create(xs[1]), C.nd_create(xs[2])]))
    outs = [C.nd_create(np.zeros((2, 3))) for _ in range(3)] + [C.nd_create(np.zeros(5))]
    kck(pull(h, [3, 3, 5, 3], [outs[0], outs[1], outs[3], outs[2]]))
    for got, want in zip(outs, py_assign):
        assert np.array_equal(bits(C.nd_get(got)), bits(want))

    seen = []

    @UPDATER
    def c_upd(key, recv, local, arg):
        seen.append(key)
        loc = host_view(local)
        loc[:] = loc + host_view(recv) * np.float32(0.5)
    kck(lib().GXKVStoreSetUpdater(h, c_upd, None))
    kck(push(h, [3, 3], [C.nd_create(xs[3]), C.nd_create(xs[4])]))
    kck(pull(h, [3], [outs[0]]))
    assert seen == [3]
    assert np.array_equal(bits(C.nd_get(outs[0])), bits(py_updated))
    kck(lib().GXKVStoreFree(h))


def test_local_store_refusals():
    h = kv_create("local")
    a, b = C.nd_create(np.ones((2, 3))), C.nd_create(np.ones(4))

    def fails(rc, *parts):
        assert rc == -1
        for p in parts:
            assert p in kv_err(), kv_err()
    fails(init(h, [1, 1], [a, a]), "GXKVStoreInitND", "key 1", "repeated")
    kck(init(h, [1], [a]))
    fails(init(h, [1], [a]), "GXKVStoreInitND", "key 1", "already initialised")
    fails(push(h, [9], [a]), "GXKVStorePushND", "key 9", "not initialised")
    fails(pull(h, [9], [a]), "GXKVStorePullND", "key 9", "not initialised")
    fails(push(h, [1], [b]), "GXKVStorePushND", "key 1", "shape (4)")
    fails(pull(h, [1], [b]), "GXKVStorePullND", "key 1", "shape")
    buf = (ctypes.c_float * 6)()
    fails(lib().GXKVStoreInit(h, 1, buf, ctypes.c_size_t(6), 0), "GXKVStoreInit", "GXKVStoreInitND")
    fails(lib().GXKVStorePush(h, 1, buf, ctypes.c_size_t(6), 0, 0, None), "GXKVStorePush", "GXKVStorePushND")
    fails(lib().GXKVStorePull(h, 1, buf, ctypes.c_size_t(6), 0, 0, None), "GXKVStorePull", "GXKVStorePullND")
    fails(lib().GXKVStoreRunServer(h), "GXKVStoreRunServer")
    fails(lib().GXKVStoreSetGradientCompression(h, b"2bit", ctypes.c_float(0.5)), "not supported", "'local'")
    kck(lib().GXKVStoreSetGradientCompression(h, b"none", ctypes.c_float(0.0)))
    kck(lib().GXKVStoreFree(h))
    d = kv_create("device")
    kck(lib().GXKVStoreSetGradientCompression(d, b"2bit", ctypes.c_float(0.5)))
    kck(lib().GXKVStoreFree(d))


def test_updater_can_be_cleared_and_null_handles_are_refused():
    """SetUpdater(NULL) returns a local store to assignment; a null handle is an error, not a crash."""
    h = kv_create("local")
    kck(init(h, [4], [C.nd_create(np.ones(3))]))

    @UPDATER
    def double(key, recv, local, arg):
        loc = host_view(local)
        loc[:] = loc + host_view(recv) * np.float32(2.0)
    kck(lib().GXKVStoreSetUpdater(h, double, None))
    kck(push(h, [4], [C.nd_create(np.ones(3))]))
    kck(lib().GXKVStoreSetUpdater(h, None, None))
    kck(push(h, [4, 4], [C.nd_create(np.full(3, 5.0)), C.nd_create(np.full(3, 0.5))]))
    out = C.nd_create(np.zeros(3))
    kck(pull(h, [4], [out]))
    assert np.array_equal(C.nd_get(out), np.full(3, 5.5, np.float32))
    kck(lib().GXKVStoreFree(h))
    assert lib().GXKVStoreSetUpdater(None, None, None) == -1 and "null KVStore handle" in kv_err()
    assert lib().GXKVStorePushND(None, 0, None, None, 0) == -1 and "null KVStore handle" in kv_err()


def free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def run_job(extra, timeout=180):
    """scheduler + server (the Python package's roles) + two _capi_kv_worker.py workers; returns the workers' RESULT dicts"""
    port = free_port()
    base = {"DMLC_PS_ROOT_URI": "127.0.0.1", "DMLC_PS_ROOT_PORT": str(port), "DMLC_NUM_SERVER": "1", "DMLC_NUM_WORKER": "2", "DMLC_NUM_ALL_WORKER": "2"}
    env = {k: v for k, v in os.environ.items() if not k.startswith(("DMLC_", "PS_")) and k not in ("RANK", "WORLD_SIZE")}
    env.update(base); env.update(extra)
    boot = "import sys; sys.path.insert(0, %r); import geomx_b200" % os.path.dirname(HERE)
    cmds = [([sys.executable, "-c", boot], "scheduler"), ([sys.executable, "-c", boot], "server"),
            ([sys.executable, os.path.join(HERE, "_capi_kv_worker.py")], "worker"), ([sys.executable, os.path.join(HERE, "_capi_kv_worker.py")], "worker")]
    procs = [subprocess.Popen(c, env=dict(env, DMLC_ROLE=role), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for c, role in cmds]
    deadline = time.time() + timeout
    try:
        while time.time() < deadline and any(p.poll() is None for p in procs) and all(p.poll() in (None, 0) for p in procs):
            time.sleep(0.1)
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
    outs = [p.communicate()[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n-----\n".join(o[-2000:] for o in outs)
    res = [json.loads(l[7:]) for o in outs for l in o.splitlines() if l.startswith("RESULT {")]
    assert len(res) == 2, outs
    return res


@pytest.mark.parametrize("comp", ["none", "2bit"])
def test_dist_nd_host_arrays_match_raw_buffers(comp):
    res = run_job({"KV_MODE": "host", "KV_COMP": comp})
    assert all(r["equal"] and r["moved"] for r in res), res
    assert res[0]["checksums"] == res[1]["checksums"]


# ================================================================================================================ GPU
def gpu_count():
    n = ctypes.c_int(0)
    C.ck(lib().GXGetGPUCount(ctypes.byref(n)))
    return n.value


def kernels():
    from geomx_b200.ops import _native_sigs
    k = ctypes.CDLL(os.path.join(C.ROOT, "geomx_b200", "lib", "libgeomx_kernels.so"))
    _native_sigs.declare(k)
    return k


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 15, 17, 2 ** 20 + 3])
def test_kernels_bit_exact_against_numpy(n):
    import torch
    k = kernels()
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev).cuda_stream
    thr = 0.37
    rng = np.random.default_rng(n)
    for cnt in range(1, 9):
        res_np = np.zeros(n, np.float32)
        res = torch.zeros(n, device=dev)
        words = torch.zeros((n + 15) // 16, dtype=torch.int32, device=dev)
        out = torch.empty(n, device=dev)
        for _ in range(3):                                          # the residual carries over three calls
            ins_np = [(0.3 * rng.standard_normal(n)).astype(np.float32) for _ in range(cnt)]
            ins = [torch.from_numpy(a).to(dev) for a in ins_np]
            ptrs = (vp * cnt)(*[t.data_ptr() for t in ins])
            assert k.gx_kv_sum_quantize(out.data_ptr(), ptrs, cnt, n, res.data_ptr(), words.data_ptr(), ctypes.c_float(thr), stream) == 0
            s = ins_np[0].copy()
            for a in ins_np[1:]:
                s = (s + a).astype(np.float32)
            want_words = quantize_2bit(s, res_np, thr)
            torch.cuda.synchronize()
            assert np.array_equal(bits(out.cpu().numpy()), bits(s))
            assert np.array_equal(words.cpu().numpy().view(np.uint32), want_words)
            assert np.array_equal(bits(res.cpu().numpy()), bits(res_np))
            # dequantise + sum of cnt word arrays (here: this round's words under cnt different thresholds' worth of inputs)
            wl = [torch.from_numpy(quantize_2bit(a, np.zeros(n, np.float32), thr).view(np.int32)).to(dev) for a in ins_np]
            wp = (vp * cnt)(*[t.data_ptr() for t in wl])
            assert k.gx_kv_dequant_sum(out.data_ptr(), wp, cnt, n, ctypes.c_float(thr), 0, stream) == 0
            want = dequantize_2bit(wl[0].cpu().numpy().view(np.uint32), n, thr)
            for t in wl[1:]:
                want = (want + dequantize_2bit(t.cpu().numpy().view(np.uint32), n, thr)).astype(np.float32)
            torch.cuda.synchronize()
            assert np.array_equal(bits(out.cpu().numpy()), bits(want))


def _device_vs_local(devs, comp=None, updater=False, steps=3):
    """the same device inputs through a `device` store and a `local` store; returns (device pulls, local pulls, home context)"""
    shape = (33, 31)
    rng = np.random.default_rng(len(devs))
    w0 = rng.standard_normal(shape).astype(np.float32)
    pulls, home = {}, None
    upds = {}
    for kind in ("device", "local"):
        h = kv_create(kind)
        if comp and kind == "device":
            kck(lib().GXKVStoreSetGradientCompression(h, b"2bit", ctypes.c_float(comp)))
        if updater:
            @UPDATER
            def upd(key, recv, local, arg):
                out_n, out = ctypes.c_int(1), (vp * 1)(local)
                outs = ctypes.cast(out, ctypes.POINTER(vp))
                C.ck(lib().GXImperativeInvokeByName(b"sgd_update", 2, C.handles([vp(local), vp(recv)]), ctypes.byref(out_n), ctypes.byref(outs), 2,
                                                    C.strs(["lr", "wd"]), C.strs(["0.1", "0.0"])))
            upds[kind] = upd
            kck(lib().GXKVStoreSetUpdater(h, upd, None))
        kck(init(h, [7], [dev_nd(w0, devs[0])]))
        got = []
        grng = np.random.default_rng(11)
        outs = [dev_nd(np.zeros(shape), d) for d in devs]
        for _ in range(steps):
            vals = [dev_nd((0.1 * grng.standard_normal(shape)).astype(np.float32), d) for d in devs]
            kck(push(h, [7] * len(vals), vals))
            kck(pull(h, [7] * len(outs), outs))
            got.append([C.nd_get(o) for o in outs])
            for v in vals:
                C.nd_free(v)
        pulls[kind] = got
        kck(lib().GXKVStoreFree(h))
    return pulls["device"], pulls["local"], w0


@pytest.mark.gpu
@pytest.mark.parametrize("ndev", [1, 2])
def test_device_store_matches_local(ndev):
    if gpu_count() < ndev:
        pytest.skip("needs %d GPUs" % ndev)
    devs = [0, 1, 0] if ndev > 1 else [0, 0]
    d, l, _ = _device_vs_local(devs)
    for a, b in zip(d, l):
        for x, y in zip(a, b):
            assert np.array_equal(bits(x), bits(y))
    # the stored value lives on the device of the init value: an updater sees device arrays there
    h = kv_create("device")
    ctxs = []

    @UPDATER
    def where(key, recv, local, arg):
        ctxs.append((context(vp(recv)), context(vp(local))))
    kck(lib().GXKVStoreSetUpdater(h, where, None))
    kck(init(h, [1], [dev_nd(np.ones(8), devs[-1])]))
    kck(push(h, [1, 1], [dev_nd(np.ones(8), devs[0]), dev_nd(np.ones(8), devs[-1])]))
    kck(lib().GXKVStoreFree(h))
    assert ctxs == [((2, devs[-1]), (2, devs[-1]))]


@pytest.mark.gpu
@pytest.mark.parametrize("ndev", [1, 2])
def test_device_store_updater_sgd_matches_local(ndev):
    if gpu_count() < ndev:
        pytest.skip("needs %d GPUs" % ndev)
    devs = [0, 1] if ndev > 1 else [0, 0]
    d, l, _ = _device_vs_local(devs, updater=True)
    for a, b in zip(d, l):
        for x, y in zip(a, b):
            np.testing.assert_allclose(x, y, rtol=1e-6, atol=1e-7)


@pytest.mark.gpu
@pytest.mark.parametrize("ndev", [1, 2])
def test_device_store_2bit_matches_numpy(ndev):
    if gpu_count() < ndev:
        pytest.skip("needs %d GPUs" % ndev)
    devs = [0, 1, 0] if ndev > 1 else [0, 0, 0]
    thr = 0.05
    d, _, w0 = _device_vs_local(devs, comp=thr)
    shape = w0.shape
    grng = np.random.default_rng(11)
    res = [np.zeros(w0.size, np.float32) for _ in devs]
    for step in range(3):
        vals = [(0.1 * grng.standard_normal(shape)).astype(np.float32).ravel() for _ in devs]
        acc = None
        for i, v in enumerate(vals):
            deq = dequantize_2bit(quantize_2bit(v, res[i], thr), v.size, thr)
            acc = deq if acc is None else (acc + deq).astype(np.float32)
        for out in d[step]:
            assert np.array_equal(bits(out.ravel()), bits(acc))


@pytest.mark.gpu
@pytest.mark.parametrize("comp", ["none", "2bit"])
@pytest.mark.parametrize("mode", ["device", "device2"])
def test_dist_nd_device_arrays_match_raw_buffers(mode, comp):
    if gpu_count() < (2 if mode == "device2" else 1):
        pytest.skip("needs 2 GPUs")
    res = run_job({"KV_MODE": mode, "KV_COMP": comp})
    assert all(r["equal"] and r["moved"] for r in res), res
    assert res[0]["checksums"] == res[1]["checksums"]


@pytest.mark.gpu
def test_gpu_distributed_training_example(tmp_path):
    """examples/c_api/dist_train_cnn_gpu.c: device executors, one PushND of every gradient and one PullND of every weight per step, four
    processes.  Both workers end with the same parameters and the loss falls below 0.3 of its first value."""
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    libdir = os.path.join(C.ROOT, "geomx_b200", "lib")
    exe = str(tmp_path / "dist_train_cnn_gpu")
    subprocess.run([cc, "-O2", "-Wall", "-Werror", "-std=c99", "-I", os.path.join(C.ROOT, "geomx_b200", "include"),
                    os.path.join(C.ROOT, "examples", "c_api", "dist_train_cnn_gpu.c"), "-L", libdir, "-lgeomx_capi", "-Wl,-rpath," + libdir, "-lm",
                    "-o", exe], check=True)
    port = free_port()
    env = {k: v for k, v in os.environ.items() if not k.startswith(("DMLC_", "PS_")) and k not in ("RANK", "WORLD_SIZE")}
    env.update({"DMLC_PS_ROOT_URI": "127.0.0.1", "DMLC_PS_ROOT_PORT": str(port), "DMLC_NUM_SERVER": "1", "DMLC_NUM_WORKER": "2", "DMLC_NUM_ALL_WORKER": "2"})
    procs = [subprocess.Popen([exe, "30"], env=dict(env, DMLC_ROLE=role), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for role in ("scheduler", "server", "worker", "worker")]
    outs = []
    try:
        for p in procs:
            outs.append(p.communicate(timeout=240)[0])
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
    assert all(p.returncode == 0 for p in procs), outs
    finals = [re.search(r"FINAL rank (\d) of 2 loss ([\d.]+) -> ([\d.]+) checksum ([-\d.]+)", o) for o in outs[2:]]
    assert all(finals), outs
    assert sorted(m.group(1) for m in finals) == ["0", "1"]
    assert finals[0].group(4) == finals[1].group(4)
    assert all(float(m.group(3)) < 0.3 * float(m.group(2)) for m in finals)
