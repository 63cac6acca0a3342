"""Serving benchmark of the C predict API: model-zoo ResNet-18 (1000 classes, 3 x 224 x 224) exported to ``-symbol.json`` + ``.params``
and served through the flat C ABI (ctypes on ``geomx_b200/lib/_C*.so``) at several batch sizes by

  * ``host``        the host predictor (GXPredCreate dev_type 1): SetInput + Forward + GetOutput
  * ``gpu``         the device predictor (dev_type 2): Forward + GetOutput into host memory, the input set once before the timed loop
  * ``gpu_devptr``  the device predictor with device-pointer I/O: SetInput from and GetOutput into GXNDArrayCreateEx(dev_type 2) arrays,
                    plus Forward

Each call is timed with a host clock around work that ends in GetOutput's stream synchronise, after warm-up (the device predictor's first
Forward runs eagerly and the second captures the CUDA graph, so warm-up is at least 3 calls).  Reported: p50 / p90 ms per call,
images/s at the p50, the planned arena bytes, the convolution workspace bytes, the GPU's name and power limit (nvidia-smi).  A run
without a GPU fails; nothing falls back to the host.

  python tools/predict_bench.py [--batches 1,8,64] [--iters 50] [--host-iters 3] [--out DIR]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import _capi as C  # noqa: E402
from _capi import ck, lib, u32, vp  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
    except (OSError, subprocess.TimeoutExpired) as e:
        sys.exit("predict_bench: no GPU (nvidia-smi: %s)" % e)
    if out.returncode != 0 or not out.stdout.strip():
        sys.exit("predict_bench: no GPU (nvidia-smi: %s)" % (out.stderr.strip() or "no device"))
    name, power = [s.strip() for s in out.stdout.strip().splitlines()[0].split(",")]
    return name, power


def export_resnet18(d):
    import geomx_b200 as mx
    from geomx_b200.gluon.model_zoo import vision
    net = vision.get_model("resnet18_v1", classes=1000)
    net.initialize(mx.init.Xavier())
    with mx.autograd.predict_mode():
        net(mx.nd.array(np.zeros((1, 3, 224, 224), np.float32)))
    prefix = os.path.join(d, "resnet18")
    net.export(prefix)
    return open(prefix + "-symbol.json").read(), open(prefix + "-0000.params", "rb").read()


def conv_workspace_bytes(js, shape):
    """bytes of the device predictor's shared workspace: im2col matrix (row stride rounded up to 4) + GEMM rows of the largest
    convolution, or the arg-max scratch of the largest max pooling (predict_device.h Bind)"""
    import geomx_b200 as mx
    s = mx.sym.load_json(js).get_internals()
    shapes = dict(zip(s.list_outputs(), s.infer_shape(data=shape)[1]))
    nodes = json.loads(js)["nodes"]
    best = 0
    for n in nodes:
        a = n.get("attrs", {})
        if n["op"] not in ("Convolution", "Pooling"):
            continue
        src = nodes[n["inputs"][0] if isinstance(n["inputs"][0], int) else n["inputs"][0][0]]
        x = shapes[src["name"] if src["op"] == "null" else src["name"] + "_output"]
        y = shapes[n["name"] + "_output"]
        if n["op"] == "Pooling":
            if a.get("pool_type", "max") == "max":
                best = max(best, int(np.prod(y)))
            continue
        k = a["kernel"] if isinstance(a["kernel"], list) else json.loads(str(a["kernel"]).replace("(", "[").replace(")", "]"))
        ldc = (x[1] * k[0] * k[1] + 3) // 4 * 4
        best = max(best, y[0] * y[2] * y[3] * (ldc + y[1]))
    return best * 4


def create(js, pb, shape, dev_type):
    h = vp()
    keys = C.strs(["data"])
    rc = lib().GXPredCreate(js.encode(), pb, len(pb), dev_type, 0, 1, keys, (u32 * 2)(0, 4), (u32 * 4)(*shape), ctypes.byref(h))
    if rc != 0:
        sys.exit("predict_bench: GXPredCreate(dev_type %d) failed: %s" % (dev_type, C.err()))
    return h


def timed(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(iters):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.percentile(ts, 50)), float(np.percentile(ts, 90))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batches", default="1,8,64")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--host-iters", type=int, default=3)
    ap.add_argument("--out", default="predict_bench_out", help="directory for predict_bench.json and the table predict_gpu.txt")
    a = ap.parse_args()
    name, power = gpu_info()
    os.makedirs(a.out, exist_ok=True)
    with tempfile.TemporaryDirectory() as d:
        js, pb = export_resnet18(d)
    rows = []
    rng = np.random.RandomState(0)
    for b in [int(v) for v in a.batches.split(",")]:
        shape = (b, 3, 224, 224)
        x = rng.rand(*shape).astype(np.float32)
        y = np.empty((b, 1000), np.float32)
        px, py = x.ctypes.data_as(vp), y.ctypes.data_as(vp)
        res = {"batch": b, "arena_bytes": None, "conv_workspace_bytes": conv_workspace_bytes(js, shape)}
        hh, dh = create(js, pb, shape, 1), create(js, pb, shape, 2)
        arena, nops = ctypes.c_uint64(), u32()
        ck(lib().GXPredGetPlan(dh, ctypes.byref(arena), ctypes.byref(nops)))
        res["arena_bytes"], res["num_ops"] = arena.value, nops.value

        def host():
            ck(lib().GXPredSetInput(hh, b"data", px, x.size)); ck(lib().GXPredForward(hh)); ck(lib().GXPredGetOutput(hh, 0, py, y.size))
        res["host"] = timed(host, 1, a.host_iters)
        want = y.copy()
        ck(lib().GXPredFree(hh))

        ck(lib().GXPredSetInput(dh, b"data", px, x.size))

        def gpu():
            ck(lib().GXPredForward(dh)); ck(lib().GXPredGetOutput(dh, 0, py, y.size))
        res["gpu"] = timed(gpu, 5, a.iters)
        res["max_rel_diff_vs_host"] = float(np.abs(y.astype(np.float64) - want).max() / np.abs(want).max())

        xd, yd, dx, dy = vp(), vp(), vp(), vp()
        ck(lib().GXNDArrayCreateEx((u32 * 4)(*shape), 4, 2, 0, 0, 0, ctypes.byref(xd)))
        ck(lib().GXNDArrayCreateEx((u32 * 2)(b, 1000), 2, 2, 0, 0, 0, ctypes.byref(yd)))
        C.nd_set(xd, x)
        ck(lib().GXNDArrayGetData(xd, ctypes.byref(dx))); ck(lib().GXNDArrayGetData(yd, ctypes.byref(dy)))

        def gpu_devptr():
            ck(lib().GXPredSetInput(dh, b"data", dx, x.size)); ck(lib().GXPredForward(dh)); ck(lib().GXPredGetOutput(dh, 0, dy, y.size))
        res["gpu_devptr"] = timed(gpu_devptr, 5, a.iters)
        res["devptr_equals_hostptr"] = bool(np.array_equal(C.nd_get(yd), y))
        ck(lib().GXPredFree(dh)); C.nd_free(xd); C.nd_free(yd)
        rows.append(res)
        print(json.dumps(res), flush=True)

    lines = ["ResNet-18 (model zoo, 1000 classes, 3x224x224, fp32) through the C predict API on %s, power limit %s" % (name, power),
             "ms per call: p50 / p90, host clock around work that ends in GetOutput's synchronise; images/s at the p50",
             "%-6s %-22s %-22s %-22s %-14s %-14s %s" % ("batch", "host (dev_type 1)", "gpu (dev_type 2)", "gpu device-pointer I/O", "arena bytes",
                                                      "conv workspace", "max rel diff")]
    for r in rows:
        cell = lambda t: "%.2f / %.2f (%.0f/s)" % (t[0], t[1], r["batch"] * 1e3 / t[0])  # noqa: E731
        lines.append("%-6d %-22s %-22s %-22s %-14d %-14d %.2g" % (r["batch"], cell(r["host"]), cell(r["gpu"]), cell(r["gpu_devptr"]), r["arena_bytes"],
                                                                 r["conv_workspace_bytes"], r["max_rel_diff_vs_host"]))
    table = "\n".join(lines)
    print(table)
    with open(os.path.join(a.out, "predict_bench.json"), "w") as f:
        json.dump({"gpu": name, "power_limit": power, "rows": rows}, f, indent=1)
    with open(os.path.join(a.out, "predict_gpu.txt"), "w") as f:
        f.write(table + "\n")


if __name__ == "__main__":
    main()
