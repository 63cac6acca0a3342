"""Per-step time of the C API KVStore on NDArray handles with a ResNet-18-sized parameter set (62 tensors, 11.7 M float32 values), through

  * ``device``     an in-process ``device`` store, one value per GPU for every key (1, 2, 4, 8 GPUs as far as visible): one PushND of all
                   gradients + one PullND of all weights into every GPU's arrays
  * ``dist host``  ``dist_sync`` over loopback (1 scheduler, 1 server, 1 worker): PushND + PullND of host arrays
  * ``dist dev``   the same job with device arrays on GPU 0 (reduce / quantise on the GPU, page-locked staging)

each without compression and with 2-bit (threshold 0.5).  Times are host-clock p50 / p90 ms per step after warm-up, every step ending in
GXNDArrayWaitAll.  The GPU's name and power limit come from nvidia-smi.  A run without a GPU fails.

  python tools/kv_bench.py [--steps 20] [--out profiles/kv_device.txt]
"""
import argparse
import ctypes
import json
import os
import socket
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import _capi as C  # noqa: E402

vp = ctypes.c_void_p


def resnet18_shapes():
    shapes = [(64, 3, 7, 7), (64,), (64,)]
    cin = 64
    for cout, stride in ((64, 1), (128, 2), (256, 2), (512, 2)):
        for blk in range(2):
            s = stride if blk == 0 else 1
            shapes += [(cout, cin, 3, 3), (cout,), (cout,), (cout, cout, 3, 3), (cout,), (cout,)]
            if s != 1 or cin != cout:
                shapes += [(cout, cin, 1, 1), (cout,), (cout,)]
            cin = cout
    return shapes + [(1000, 512), (1000,)]


def lib():
    L = C.lib()
    L.GXGetLastError.restype = ctypes.c_char_p
    return L


def kck(rc):
    if rc != 0:
        raise RuntimeError(lib().GXGetLastError().decode() + " | " + C.err())


def nd(shape, dev, fill=None):
    h = vp()
    kck(lib().GXNDArrayCreateEx((ctypes.c_uint32 * len(shape))(*shape), len(shape), 2 if dev >= 0 else 1, max(dev, 0), 0, 0, ctypes.byref(h)))
    if fill is not None:
        C.nd_set(h, np.full(shape, fill, np.float32))
    return h


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
    except (OSError, subprocess.TimeoutExpired) as e:
        sys.exit("kv_bench: no GPU (nvidia-smi: %s)" % e)
    if out.returncode != 0 or not out.stdout.strip():
        sys.exit("kv_bench: no GPU (nvidia-smi: %s)" % (out.stderr.strip() or "no device"))
    return out.stdout.strip().splitlines()


def time_steps(h, keys, vals, outs, steps, warm=3):
    k = (ctypes.c_int * len(keys))(*keys)
    v, o = C.handles(vals), C.handles(outs)
    ts = []
    for i in range(warm + steps):
        t0 = time.perf_counter()
        kck(lib().GXKVStorePushND(h, len(keys), k, v, 0))
        kck(lib().GXKVStorePullND(h, len(keys), k, o, 0))
        kck(lib().GXNDArrayWaitAll())
        if i >= warm:
            ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.percentile(ts, 50)), float(np.percentile(ts, 90))


def run_device(ngpu, comp, steps):
    shapes = resnet18_shapes()
    h = vp()
    kck(lib().GXKVStoreCreate(b"device", ctypes.byref(h)))
    if comp:
        kck(lib().GXKVStoreSetGradientCompression(h, b"2bit", ctypes.c_float(0.5)))
    init = [nd(s, 0, 0.0) for s in shapes]
    kck(lib().GXKVStoreInitND(h, len(shapes), (ctypes.c_int * len(shapes))(*range(len(shapes))), C.handles(init)))
    keys, vals, outs = [], [], []
    for d in range(ngpu):
        for i, s in enumerate(shapes):
            keys.append(i); vals.append(nd(s, d, 0.01)); outs.append(nd(s, d))
    r = time_steps(h, keys, vals, outs, steps)
    kck(lib().GXKVStoreFree(h))
    for a in init + vals + outs:
        C.nd_free(a)
    return r


def worker(dev, comp, steps):
    """one dist_sync worker (DMLC_* from the environment); prints the timing as JSON"""
    shapes = resnet18_shapes()
    h = vp()
    kck(lib().GXKVStoreCreate(b"dist_sync", ctypes.byref(h)))
    if comp:
        kck(lib().GXKVStoreSetGradientCompression(h, b"2bit", ctypes.c_float(0.5)))
    kck(lib().GXKVStoreSendCommmandToServers(h, 7, b"name=sgd;lr=0.1;wd=0.0;rescale_grad=1.0;clip_gradient=-1.0;momentum=0.0"))
    keys = list(range(len(shapes)))
    init = [nd(s, dev, 0.0) for s in shapes]
    kck(lib().GXKVStoreInitND(h, len(keys), (ctypes.c_int * len(keys))(*keys), C.handles(init)))
    vals, outs = [nd(s, dev, 0.01) for s in shapes], [nd(s, dev) for s in shapes]
    r = time_steps(h, keys, vals, outs, steps)
    print("TIMING " + json.dumps(r), flush=True)
    kck(lib().GXKVStoreFree(h))


def run_dist(dev, comp, steps):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    env = {k: v for k, v in os.environ.items() if not k.startswith(("DMLC_", "PS_")) and k not in ("RANK", "WORLD_SIZE")}
    env.update({"DMLC_PS_ROOT_URI": "127.0.0.1", "DMLC_PS_ROOT_PORT": str(port), "DMLC_NUM_SERVER": "1", "DMLC_NUM_WORKER": "1", "DMLC_NUM_ALL_WORKER": "1"})
    boot = "import sys; sys.path.insert(0, %r); import geomx_b200" % ROOT
    procs = [subprocess.Popen([sys.executable, "-c", boot], env=dict(env, DMLC_ROLE=r), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in ("scheduler", "server")]
    procs.append(subprocess.Popen([sys.executable, os.path.abspath(__file__), "--worker", str(dev), str(int(comp)), str(steps)], env=dict(env, DMLC_ROLE="worker"),
                                  stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    try:
        outs = [p.communicate(timeout=600)[0] for p in procs]
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
    for line in outs[-1].splitlines():
        if line.startswith("TIMING "):
            return tuple(json.loads(line[7:]))
    raise RuntimeError("dist worker failed:\n" + outs[-1][-3000:])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", nargs=3, default=None)
    a = ap.parse_args()
    if a.worker:
        worker(int(a.worker[0]), bool(int(a.worker[1])), int(a.worker[2]))
        return
    gpus = gpu_info()
    n = ctypes.c_int(0)
    kck(lib().GXGetGPUCount(ctypes.byref(n)))
    if n.value < 1:
        sys.exit("kv_bench: no CUDA device visible to the kernel library")
    total = sum(int(np.prod(s)) for s in resnet18_shapes())
    lines = ["# tools/kv_bench.py --steps %d: C API KVStore on NDArray handles, ResNet-18 parameter set (%d tensors, %.2f M float32)"
             % (a.steps, len(resnet18_shapes()), total / 1e6),
             "# GPU: %s (%d visible); host-clock ms per step (PushND + PullND + WaitAll), p50 / p90" % (gpus[0], n.value),
             "%-24s %-6s %10s %10s" % ("path", "comp", "p50_ms", "p90_ms")]
    for comp in (False, True):
        for g in (1, 2, 4, 8):
            if g <= n.value:
                p50, p90 = run_device(g, comp, a.steps)
                lines.append("%-24s %-6s %10.3f %10.3f" % ("device %d GPU" % g, "2bit" if comp else "none", p50, p90))
        for dev, name in ((-1, "dist_sync host arrays"), (0, "dist_sync device arrays")):
            p50, p90 = run_dist(dev, comp, a.steps)
            lines.append("%-24s %-6s %10.3f %10.3f" % (name, "2bit" if comp else "none", p50, p90))
    text = "\n".join(lines) + "\n"
    print(text, end="")
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
