"""torchrun worker for the gloo collective KVStore test: prints one RESULT line per rank."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import geomx_b200 as mx  # noqa: E402

mode = os.environ.get("TEST_MODE", "sgd")
kv = mx.kv.create("dist_async" if mode == "async" else "dist_sync")
rank = int(os.environ["RANK"])
if getattr(kv, "configures_servers", False) and mode in ("sgd", "async"):
    kv.set_optimizer(mx.optimizer.SGD(learning_rate=0.1))
shapes = [(4, 5), (7,)]
params = [mx.nd.array(np.full(s, 1.0 + i + 10 * rank, dtype=np.float32)) for i, s in enumerate(shapes)]      # only rank 0's values must survive init
for i, p in enumerate(params):
    kv.init(i, p)
    kv.pull(i, p)
mx.nd.waitall()
out = {"rank": rank, "type": type(kv).__name__, "party_rank": kv.rank, "num_workers": kv.num_workers, "num_all_workers": kv.num_all_workers,
       "init": [float(p.asnumpy().reshape(-1)[0]) for p in params], "vals": []}
for step in range(int(os.environ.get("TEST_STEPS", "2"))):
    for i, p in enumerate(params):
        if mode == "hfa":
            kv.push(i, mx.nd.array(np.full(shapes[i], float(step + 1) * (rank + 1), dtype=np.float32)) / kv.num_workers)
        else:
            kv.push(i, mx.nd.array(np.full(shapes[i], 0.5 * (rank + 1), dtype=np.float32)), priority=-i)
        kv.pull(i, p, priority=-i)
    mx.nd.waitall()
    out["vals"].append([float(p.asnumpy().reshape(-1)[0]) for p in params])
kv._barrier()
with open(os.path.join(os.environ["TEST_OUT_DIR"], "rank%d.json" % rank), "w") as f:      # ranks share one stdout: lines may interleave
    json.dump(out, f)
# tear the gloo process group down before interpreter shutdown: left to exit-time destruction it can abort the process
# ("terminate called without an active exception") and fail the launch
import torch.distributed as dist  # noqa: E402
dist.destroy_process_group()
