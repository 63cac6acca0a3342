"""A dist_sync worker over the plain C API (ctypes over lib/_C*.so) that drives one parameter through the raw-buffer forms (key 1) and the same
parameter through the NDArray forms (key 2).  KV_MODE: host (host NDArrays), device (device NDArrays on GPU 0), device2 (one value on GPU 0
and one on GPU 1, summed by the push).  KV_COMP: none | 2bit.  Prints RESULT {"rank", "equal", "checksums"} where `equal` says whether every
pull of key 2 was bitwise equal to the pull of key 1."""
import ctypes
import glob
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
lib = ctypes.CDLL(glob.glob(os.path.join(ROOT, "geomx_b200", "lib", "_C*.so"))[0])
lib.GXGetLastError.restype = ctypes.c_char_p
lib.GXRTGetLastError.restype = ctypes.c_char_p
vp = ctypes.c_void_p


def ck(rc):
    if rc != 0:
        raise RuntimeError(lib.GXGetLastError().decode() + " | " + lib.GXRTGetLastError().decode())


def nd(arr, dev):
    h = vp()
    shape = (ctypes.c_uint32 * arr.ndim)(*arr.shape)
    ck(lib.GXNDArrayCreateEx(shape, arr.ndim, 2 if dev >= 0 else 1, max(dev, 0), 0, 0, ctypes.byref(h)))
    ck(lib.GXNDArraySyncCopyFromCPU(h, arr.ctypes.data_as(vp), ctypes.c_size_t(arr.size)))
    return h


def get(h, shape):
    out = np.empty(shape, np.float32)
    ck(lib.GXNDArraySyncCopyToCPU(h, out.ctypes.data_as(vp), ctypes.c_size_t(out.size)))
    return out


mode, comp = os.environ.get("KV_MODE", "host"), os.environ.get("KV_COMP", "none")
devs = {"host": (-1, -1), "device": (0, 0), "device2": (0, 1)}[mode]
h = vp()
ck(lib.GXKVStoreCreate(b"dist_sync", ctypes.byref(h)))
rank = ctypes.c_int()
ck(lib.GXKVStoreGetRank(h, ctypes.byref(rank)))
if comp != "none":
    ck(lib.GXKVStoreSetGradientCompression(h, comp.encode(), ctypes.c_float(0.05)))
if rank.value == 0:
    ck(lib.GXKVStoreSendCommmandToServers(h, 7, b"name=sgd;lr=0.1;wd=0.0;rescale_grad=1.0;clip_gradient=-1.0;momentum=0.0"))
shape = (37, 29)                                   # 1073 values: not a multiple of 16 or 4
rng = np.random.default_rng(7)
w0 = rng.standard_normal(shape).astype(np.float32)
raw = np.ascontiguousarray(w0.copy())
ck(lib.GXKVStoreInit(h, 1, raw.ctypes.data_as(vp), ctypes.c_size_t(raw.size), 0))
winit = nd(w0, devs[0])
ck(lib.GXKVStoreInitND(h, 1, (ctypes.c_int * 1)(2), (vp * 1)(winit)))
outs = [nd(np.zeros(shape, np.float32), devs[0]), nd(np.zeros(shape, np.float32), devs[1])]
equal, sums = True, []
grng = np.random.default_rng(100 + rank.value)
for step in range(3):
    ga = (0.1 * grng.standard_normal(shape)).astype(np.float32)
    gb = (0.1 * grng.standard_normal(shape)).astype(np.float32)
    gsum = np.ascontiguousarray(ga + gb)
    hp, hl = ctypes.c_int(), ctypes.c_int()
    ck(lib.GXKVStorePush(h, 1, gsum.ctypes.data_as(vp), ctypes.c_size_t(gsum.size), 0, 0, ctypes.byref(hp)))
    ck(lib.GXKVStorePull(h, 1, raw.ctypes.data_as(vp), ctypes.c_size_t(raw.size), 0, 0, ctypes.byref(hl)))
    ck(lib.GXKVStoreWait(h, hl))
    va, vb = nd(ga, devs[0]), nd(gb, devs[1])
    ck(lib.GXKVStorePushND(h, 2, (ctypes.c_int * 2)(2, 2), (vp * 2)(va, vb), 0))
    ck(lib.GXKVStorePullND(h, 2, (ctypes.c_int * 2)(2, 2), (vp * 2)(*outs), 0))
    got = [get(o, shape) for o in outs]
    equal = equal and all(np.array_equal(g.view(np.uint32), raw.view(np.uint32)) for g in got)
    sums.append(float(raw.astype(np.float64).sum()))
    ck(lib.GXNDArrayFree(va)); ck(lib.GXNDArrayFree(vb))
print("RESULT " + json.dumps({"rank": rank.value, "equal": bool(equal), "checksums": sums, "moved": bool(abs(sums[-1] - float(w0.sum())) > 1e-3)}),
      flush=True)
ck(lib.GXKVStoreFree(h))
