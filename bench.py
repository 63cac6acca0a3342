#!/usr/bin/env python
"""Headline benchmark: examples/cnn.py training throughput (samples/sec, whole job) on N B200s of one node.

Contract (driver): ``python bench.py --gpus N --steps K --warmup W`` (N>1: launched by ``torch.distributed.run`` one rank per GPU).
Prints ONE JSON line on rank 0.  Metric / config are BASELINE.json's: the reference demo CNN (178 762 params), per-worker batch 32
(weak scaling), ``dist_sync`` HiPS: workers → local PS (party reduction) → global PS (Adam on the owner shard) → broadcast, synthetic
MNIST-shaped data, random-init (Xavier) weights, fp32 storage with TF32 tensor-core multiplies and fp32 accumulation.

Timed region (device-timed, max over ranks): exactly K full training steps (forward + backward + push + server optimizer + pull), each
bracketed by its own CUDA-event pair; between timed steps a 256 MiB buffer is written to flush the 126 MB L2.  ``e2e`` re-measures the
same K steps through the public API ``HipsCNNTrainStep.step(X_pinned, y_pinned) -> loss`` including the per-step H2D copy of the batch
from pinned host memory and the D2H read of the loss.

``--impl reference`` runs the unmodified reference build under baseline/_ref (baseline/ref_cnn_bench.py; DESIGN.md §Reference arm).
``--impl oracle`` runs the same schedule with library ops only (PyTorch/cuDNN/cuBLAS + NCCL all-reduce + torch Adam, CUDA-graphed) — the
"baseline, not the product" yard-stick of BASELINE.md.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="native", choices=["native", "reference", "oracle"])
    ap.add_argument("--batch-size", type=int, default=32)
    ap.add_argument("--parties", type=int, default=0)
    ap.add_argument("--mode", default="dist_sync", choices=["dist_sync", "dist_async"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-flush", action="store_true")
    ap.add_argument("--no-multicast", action="store_true")
    ap.add_argument("--config", default="fsa", choices=["fsa", "bsc", "mpq_dgt", "hfa", "mixed_sync"],
                    help="BASELINE.json configs: fsa = examples/cnn.py dist_sync (headline); bsc = cnn_bsc.py (Bi-Sparse, threshold 0.01, local Adam); "
                         "mpq_dgt = cnn_mpq.py + DGT (fp16 for keys >= 1000 elements, contribution-ranked tiles, fp8 demotion); hfa = cnn_hfa.py "
                         "(K1=20 local steps, K2=10 party rounds per global round); mixed_sync = cnn.py -ms (dist_async global tier)")
    ap.add_argument("--script", action="store_true", help="time the loop of examples/cnn.py itself (gluon autograd + kv.push/kv.pull per key through "
                                                            "the fabric KVStore) instead of the fused HipsCNNTrainStep engine")
    ap.add_argument("--hybridize", action="store_true", help="--script only: net.hybridize(static_alloc=True) — forward / backward of the gluon net "
                    "replay as CUDA graphs (the CachedOp analogue); the per-key push / pull loop stays eager Python")
    ap.add_argument("--lookahead", action="store_true", help="cut the step after the forward convolutions instead of before them (software "
                    "pipelining across launches, see HipsCNNTrainStep(lookahead=...)); measured: no gain at 1-2 GPUs, so not the default")
    ap.add_argument("--fast", action="store_true", help="plain TF32 tensor-core products instead of the fp32-accurate 3xTF32 default")
    ap.add_argument("--wire-dtype", default="fp32", choices=["fp32", "fp16", "mpq", "fp8"], help="transport format of the fused HiPS step (FP16 / MPQ accelerators)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step computed on rank 0 (per-sample "
                    "loss, logits where the engine keeps them, the updated parameters) as DIR/<name>.npy in float32, so that two builds run with "
                    "the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def step_outputs(eng):
    """The arrays a caller of ``eng.run_device()`` receives from the step just run: per-sample loss, logits (fused engine only) and the
    updated parameters in ``CNN_PARAM_SHAPES`` order."""
    if isinstance(eng, ScriptPathEngine):
        out = {"loss": eng._loss._t}
        params = [p.data()._t for p in eng.params]
    else:
        out = {"loss": eng.loss}
        if getattr(eng, "logits", None) is not None:
            out["logits"] = eng.logits
        params = eng.P
    for i, p in enumerate(params):
        out["param_%02d" % i] = p
    return out


def dump_outputs(arrays, out_dir):
    """Write ``arrays`` as float32 ``.npy`` files.  If they exceed ``DUMP_LIMIT_BYTES`` together, every array larger than an equal share of
    the limit is replaced by a fixed, seeded sample of its flattened elements (same indices on every run)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    host = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    share = DUMP_LIMIT_BYTES // 4 // len(host)
    sample = sum(a.size for a in host.values()) * 4 > DUMP_LIMIT_BYTES
    for name, a in host.items():
        if sample and a.size > share:
            idx = np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True); self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


class ScriptPathEngine:
    """The training loop of examples/cnn.py, verbatim in structure: gluon net, ``autograd.record`` / ``backward``, then for every parameter
    ``kv.push(idx, grad / n, priority=-idx)`` and ``kv.pull(idx, param, priority=-idx)`` through ``mx.kv.create('dist_sync')`` (the fabric
    KVStore under torchrun, the device store on one GPU) with Adam set on the kvstore.  Same interface as HipsCNNTrainStep for the timing code."""

    def __init__(self, mx, B, dev, args):
        import torch
        self.mx, self.torch, self.B = mx, torch, B
        ctx = mx.gpu(dev.index or 0)
        self.ctx = ctx
        net = mx.models.build_cnn()
        net.initialize(force_reinit=True, ctx=ctx, init=mx.init.Xavier())
        net(mx.nd.random.uniform(shape=(B, 1, 28, 28), ctx=ctx))
        if getattr(args, "hybridize", False):
            net.hybridize(static_alloc=True, static_shape=True)
        self.net, self.loss_fn = net, mx.gluon.loss.SoftmaxCrossEntropyLoss()
        self.kv = mx.kv.create("dist_async" if args.config == "mixed_sync" else "dist_sync") if int(os.environ.get("WORLD_SIZE", 1)) > 1 else mx.kv.create("device")
        self.kv.set_optimizer(mx.optimizer.Adam(learning_rate=0.01))
        self.params = list(net.collect_params().values())
        for idx, p in enumerate(self.params):
            self.kv.init(idx, p.data())
            self.kv.pull(idx, p.data())
        mx.nd.waitall()
        self.x = torch.empty(B, 1, 28, 28, device=dev); self.label = torch.empty(B, device=dev)
        self.fabric = getattr(self.kv, "fabric", None)
        self.kernels_per_step = 0
        self._loss = None

    def _iter(self, X, y):
        mx = self.mx
        with mx.autograd.record():
            l = self.loss_fn(self.net(X), y)
        l.backward()
        for idx, p in enumerate(self.params):
            self.kv.push(idx, p.grad() / self.B, priority=-idx)
            self.kv.pull(idx, p.data(), priority=-idx)
        mx.nd.waitall()
        return l

    def run_device(self):
        from geomx_b200.ops import native
        before = native.launch_count
        self._loss = self._iter(self.mx.nd.NDArray(self.x), self.mx.nd.NDArray(self.label))
        self.kernels_per_step = native.launch_count - before

    def step(self, X, y):
        mx = self.mx
        l = self._iter(mx.nd.array(X, ctx=self.ctx), mx.nd.array(y, ctx=self.ctx))
        return float(l.mean().asscalar())

    def h2d_bytes_per_step(self):
        return self.B * 784 * 4 + self.B * 4

    def d2h_bytes_per_step(self):
        return 4


def reference_arm():
    """Run the UNMODIFIED reference (MXNet 1.4.0 / GeoMX, built from /root/reference into baseline/_ref — see baseline/README.md and
    DESIGN.md §3) on the same metric/config through its own public API.  The script imports nothing of geomx_b200."""
    here = os.path.dirname(os.path.abspath(__file__))
    script = os.path.join(here, "baseline", "ref_cnn_bench.py")
    ref_pkg = os.path.join(here, "baseline", "_ref", "mxnet")
    if not (os.path.exists(os.path.join(ref_pkg, "libmxnet.so")) or os.path.exists(os.path.join(ref_pkg, "libmxnet.so.xz"))):
        if int(os.environ.get("RANK", 0)) == 0:
            print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref/mxnet/libmxnet.so(.xz) not present: run baseline/build_reference.sh "
                              "(builds /root/reference with USE_CUDA=1 USE_NCCL=1 USE_DIST_KVSTORE=0 for sm_100, ~45 min on 8 cores)"}))
        return 0
    os.execv(sys.executable, [sys.executable, script] + sys.argv[1:])


def main():
    args = parse()
    if args.impl == "reference":
        return reference_arm()
    import torch
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    if world != args.gpus and world == 1 and args.gpus > 1:
        # convenience: self-launch under torchrun when invoked plainly with --gpus N
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
               "--master-port", str(29500 + os.getpid() % 2000), os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import geomx_b200 as mx
    from geomx_b200.ops import native
    from geomx_b200.parallel import Topology

    B, K, W = args.batch_size, args.steps, max(3, args.warmup)
    parties = args.parties or int(os.environ.get("GEOMX_NUM_PARTIES", 0)) or (2 if (world >= 2 and world % 2 == 0) else 1)
    # DMLC_NUM_GLOBAL_SERVER unset -> 0 = every rank is a global server, ownership sharded tile by tile (the fabric default)
    topo = Topology(world, rank, parties, int(os.environ.get("DMLC_NUM_GLOBAL_SERVER", 0)))
    native.set_gemm_precision("tf32" if args.fast else "3xtf32")
    torch.manual_seed(1234)  # same init on every rank; rank 0's value wins anyway (kv.init semantics)

    # ---- synthetic MNIST-shaped data in pinned host memory (a rotating pool so every step copies a different batch)
    pool = 64
    g = torch.Generator().manual_seed(100 + rank)
    Xs = torch.rand(pool, B, 1, 28, 28, generator=g).pin_memory()
    ys = torch.randint(0, 10, (pool, B), generator=g).float().pin_memory()

    if args.impl == "oracle":
        from geomx_b200.parallel.nccl_oracle import OracleCNNTrainStep
        # multi-rank: eager launches (an NCCL all-reduce captured inside the CUDA graph stalled on the test pod; the single-rank oracle is graphed)
        eng = OracleCNNTrainStep(batch_size=B, optimizer=mx.optimizer.Adam(learning_rate=0.01), topo=topo, device=dev,
                                 use_graph=not args.no_graph and world == 1)
    elif args.script:
        eng = ScriptPathEngine(mx, B, dev, args)
    else:
        kw = {"fsa": {}, "mixed_sync": {"mode": "dist_async"},
              "bsc": {"update": "local", "bsc_threshold": 0.01, "size_lower_bound": 1000},
              "mpq_dgt": {"update": "local", "wire_dtype": "mpq", "size_lower_bound": 1000, "dgt": True},
              "hfa": {"hfa": (int(os.environ.get("MXNET_KVSTORE_HFA_K1", 20)), int(os.environ.get("MXNET_KVSTORE_HFA_K2", 10)))}}[args.config]
        kw.setdefault("mode", args.mode); kw.setdefault("wire_dtype", args.wire_dtype)
        kw["lookahead"] = args.lookahead
        eng = mx.models.HipsCNNTrainStep(net=None, batch_size=B, optimizer=mx.optimizer.Adam(learning_rate=0.01), topo=topo, device=dev,
                                         use_graph=not args.no_graph, use_multicast=not args.no_multicast, **kw)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    flush = None if args.no_flush else torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    # ---------------------------------------------------------------- warm-up (also captures the CUDA graph)
    for i in range(W):
        eng.step(Xs[i % pool], ys[i % pool])
    barrier()

    # ---------------------------------------------------------------- kernel-timed region: K steps, device-resident batch, L2 flushed between steps
    eng.x.copy_(Xs[0], non_blocking=True); eng.label.copy_(ys[0], non_blocking=True)
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    sampler = ClockSampler(local)
    launches0 = native.launch_count
    barrier()
    if rank == 0:
        sampler.start()
    for i in range(K):
        if flush is not None:
            flush.fill_(float(i))
            if world > 1 and getattr(eng, "fabric", None) is not None:
                eng.fabric.barrier()      # untimed: re-align the ranks after the (long) flush so that the timed step does not include peers' flush skew
        starts[i].record()
        eng.run_device()
        ends[i].record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(step_outputs(eng), args.dump_outputs)      # before the e2e region below trains on
    per_step = sorted(s.elapsed_time(e) for s, e in zip(starts, ends))
    dev_ms = sum(per_step)
    pct = lambda q: per_step[min(K - 1, int(q * K))]
    launches_per_step = eng.kernels_per_step
    # ---------------------------------------------------------------- end-to-end region: public API, H2D from pinned + D2H loss every step
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last_loss, pending = 0.0, None
    for i in range(K):
        h = eng.step_async(Xs[(W + i) % pool], ys[(W + i) % pool]) if hasattr(eng, "step_async") else None
        if h is None:
            last_loss = eng.step(Xs[(W + i) % pool], ys[(W + i) % pool])
            continue
        if pending is not None:
            last_loss = pending.item()        # D2H result of step i-1, read while step i runs (every step's loss is read inside the region)
        pending = h
    if pending is not None:
        last_loss = pending.item()
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None

    # ---------------------------------------------------------------- exposed push+pull: duration of the fused HiPS kernel inside the step
    # (%globaltimer stamps of CTA 0, first instruction -> last phase; untimed extra steps; nothing of it overlaps compute, so all of it is exposed)
    comm_us = None
    fab = getattr(eng, "fabric", None)
    if fab is not None and args.mode == "dist_sync" and args.config in ("fsa", "bsc", "mpq_dgt") and not args.script:
        chans = list(fab.channels) or ["fsa"]
        last = "conv" if "conv" in fab.channels else chans[-1]      # the exchange at the end of the step (nothing left to hide it behind)
        look = bool(getattr(eng, "lookahead", False)) and getattr(eng, "direct_conv", False) and "conv" in fab.channels
        fused = bool(getattr(eng, "fused_exchange", False))
        cdbg = None
        if look or fused:
            # the kernels' own %globaltimer stamps are needed (end of the forward convolutions of a look-ahead step; start / end of the
            # exchange tail inside the convolution-backward launch): re-capture the graph with stamping switched on
            cdbg = torch.zeros(1024, dtype=torch.int64, device=dev)
            native.require().gx_cnn_set_debug(ctypes.c_void_p(cdbg.data_ptr()))
            if eng.graph is not None:
                eng.graph = None
                eng.capture()
        for c in chans:
            fab.state[c][3] = 1
        samples = []
        for i in range(9):
            if world > 1:
                fab.barrier()
            eng.run_device()
            torch.cuda.synchronize()
            st = {c: fab.state[c][8:8 + 12].view(torch.int64).tolist() for c in chans}
            cd = cdbg.tolist() if cdbg is not None else None
            if fused:
                # exposed = the tail of the backward launch from "whole grid finished" to "weights written" + whatever of the overlapped
                # channel outlives it (or, look-ahead, outlives the forward convolutions that follow)
                other_end = max([v[5] for k, v in st.items() if k != last] or [0])
                hidden_until = max(cd[24], cd[4]) if look else cd[24]
                if cd[24] > cd[21] > 0:
                    samples.append(((cd[24] - cd[21]) + max(0, other_end - hidden_until)) / 1e3)
            elif st[last][5] > st[last][0] > 0:
                if look:
                    hidden_until = max(cd[4], st[last][5])
                    samples.append(((st[last][5] - st[last][0]) + max(0, max(v[5] for v in st.values()) - hidden_until)) / 1e3)
                else:
                    end = max(v[5] for v in st.values())          # an overlapped channel that outlives the last one is exposed too
                    samples.append((end - st[last][0]) / 1e3)
        if cdbg is not None:
            native.require().gx_cnn_set_debug(ctypes.c_void_p(0))
        for c in chans:
            fab.state[c][3] = 0
        comm_us = statistics.median(samples[1:]) if len(samples) > 1 else None
    proto_err = bool(fab.check_protocol_errors()) if fab is not None else False
    t = torch.tensor([dev_ms, e2e_ms, comm_us or 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, comm_us = float(t[0]), float(t[1]), (float(t[2]) or None)
    if rank == 0:
        value = world * B * K / (dev_ms / 1e3)
        e2e_value = world * B * K / (e2e_ms / 1e3)
        out = {
            "metric": "cnn.py samples/sec (whole box, device-timed, max over ranks)",
            "value": round(value, 1), "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(dev_ms / K, 5), "ms_per_step_p10_p50_p90": [round(pct(0.1), 5), round(pct(0.5), 5), round(pct(0.9), 5)],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "tf32" if args.fast else "fp32 (3xTF32 tensor-core products + fp32 FMA, fp32 accumulate)", "data": "synthetic",
            "impl": args.impl, "baseline_config": args.config, "path": ("examples/cnn.py loop (script%s)" % (", hybridize(static_alloc=True)" if args.hybridize else "")) if args.script else "HipsCNNTrainStep engine",
            "config": {"model": "examples/cnn.py MNIST CNN (Conv16k5-Pool-Conv32k5-Pool-Dense256-Dense128-Dense10, 178762 params)",
                       "global_batch": B * world, "per_gpu_batch": B, "seq_len": None, "kvstore": args.mode,
                       "precision": ("fp32 storage and accumulation, TF32 tcgen05 multiplies (--fast)" if args.fast else
                                     "fp32-accurate: tcgen05 GEMMs run 3xTF32 (hi/lo split, three MMAs per K step, fp32 TMEM accumulate), the M=32 "
                                     "dense chain and conv0 run fp32 FMA; fp32 optimizer state and wire format (reference: fp32 SGEMM)"),
                       "parallelism": "hips-dp%d: %d part%s x %d worker%s, global PS %s" % (
                           world, topo.num_parties, "y" if topo.num_parties == 1 else "ies", topo.party_size, "" if topo.party_size == 1 else "s",
                           "sharded tile-by-tile over all ranks" if topo.tile_sharded else "on rank(s) %s" % topo.gs_ranks),
                       "channels": {k: {"keys": v["keys"], "mode": "replicated 1-hop" if v["replicate"] else "sharded 2-hop", "tiles": v["tiles"]}
                                    for k, v in getattr(getattr(eng, "fabric", None), "channels", {}).items()},
                       "exchange": ("key-group channels: dense keys' two-hop exchange underneath the conv backward, conv keys one-hop after it"
                                    if getattr(eng, "overlap", False) else
                                    ("one fused exchange of all keys after the backward pass (%s protocol)" % (getattr(eng, "single", None) and "direct" or
                                     getattr(getattr(eng, "fabric", None), "protocol", None))) if hasattr(eng, "overlap") else None),
                       "step_cut": ("look-ahead: each launch = head+backward+exchange of batch k, then forward convolutions of batch k+1 (same "
                                    "arithmetic, loss reported one call late)" if getattr(eng, "lookahead", False) else "classic: forward..exchange of one batch per launch"),
                       "optimizer": "Adam(lr=0.01) on the global-PS shard", "cuda_graph": not args.no_graph,
                       "l2": "256 MiB buffer written between timed steps (L2 flush)" if flush is not None else "no flush",
                       "fabric": getattr(getattr(eng, "fabric", None), "heap", None) and eng.fabric.heap.backend,
                       "multicast": bool(getattr(getattr(eng, "fabric", None), "use_multicast", False)),
                       "protocol": getattr(getattr(eng, "fabric", None), "protocol", None), "wire_dtype": args.wire_dtype},
            "e2e": {"value": round(e2e_value, 1), "unit": "samples/s", "ms_per_step": round(e2e_ms / K, 5),
                    "h2d_bytes_per_step": eng.h2d_bytes_per_step(), "d2h_bytes_per_step": eng.d2h_bytes_per_step(), "final_loss": round(last_loss, 5),
                    "api": ("examples/cnn.py loop: mx.nd.array(host batch) -> autograd -> kv.push/pull per key -> loss.asscalar()" if args.script else
                            "HipsCNNTrainStep.step_async(X_pinned, y_pinned) -> LossHandle; loss of step i read (D2H, pinned) after step i+1 was enqueued")},
            "exposed_push_pull_ms_per_step": None if comm_us is None else round(comm_us / 1e3, 5),
            "protocol_errors": proto_err,
            "gpu_launches": int(launches_per_step * K), "gpu_launches_per_step": int(launches_per_step),
            "clocks": clocks,
        }
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
