"""sample_fanout_with_feature against its composition: sample_fanout, then get_dense_feature once per level and feature.

    python benchmarks/fanout_feature.py --out benchmarks/fanout_feature_b200.json [--configs c2,c4] [--iters 50]

Graphs and shapes are bench.py's: c2 (R-MAT 10M nodes / 100M edges, D=128, batch 1024, fanout [25,10]) and the headline c4
(100M / 1B, D=256, batch 8192, [15,10]), same generator seeds.  Both arms run on one Context with the same seeds and are
checked to return the same ids and features before they are timed.  Each arm is warmed up, then timed with CUDA events over
`--iters` calls (per-call mean and the median of 5 such windows); the kernel launches of one call come from eu_launch_count.
R-MAT graphs have no uint64 slots, so the sparse arm (fused vs sample_fanout + get_sparse_feature per level) runs on a
Graph built from arrays with random ragged slots.  The JSON records the GPU name and power limit read in the same run.
The feature tables of c2 (5 GB) and c4 (100 GB) are far larger than the 126 MB L2, so row reads come from HBM.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import euler_b200 as eb  # noqa: E402
from euler_b200 import _lib  # noqa: E402

GRAPH_SEED, FEAT_SEED = 42, 7     # bench.py's
CONFIGS = {
    "c2": dict(nodes=10_000_000, edges=100_000_000, batch=1024, fanout=[25, 10], dim=128),
    "c4": dict(nodes=100_000_000, edges=1_000_000_000, batch=8192, fanout=[15, 10], dim=256),
}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def timed(fn, iters, windows=5):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    n0 = _lib.load().eu_launch_count()
    fn()
    launches = _lib.load().eu_launch_count() - n0
    ms = []
    for _ in range(windows):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1) / iters)
    return {"ms_per_call_median": float(np.median(ms)), "ms_per_call_windows": ms, "launches_per_call": int(launches)}


def compare(seeds, ets, fanout, dense, sparse, iters):
    """dense: (fids, dims); sparse: (fids, defaults).  Returns the timings of both arms after checking they agree."""
    dfids, ddims = dense
    sfids, sdefs = sparse

    def fused():
        return eb.sample_fanout_with_feature(seeds, ets, fanout, -1, dfids, ddims, sfids, sdefs)

    def composed():
        # with default_node -1 the packed ids of default-filled slots are absent ids: the same features as the engine ids
        nb, ws, ts = eb.sample_fanout(seeds, ets, fanout, -1)
        d = [f for lv in nb for f in eb.get_dense_feature(lv, dfids, ddims)]
        s = [f for lv in nb for f in eb.get_sparse_feature(lv, sfids, sdefs)] if sfids else []
        return nb, ws, ts, d, s

    eb.seed(11)
    a = fused()
    eb.seed(11)
    b = composed()
    for x, y in zip(a[0] + a[1] + a[2] + a[3], b[0] + b[1] + b[2] + b[3]):
        assert torch.equal(x, y), "fused and composed arms disagree"
    for (ia, va, sa), (ib, vb, sb) in zip(a[4], b[4]):
        assert torch.equal(ia, ib) and torch.equal(va, vb) and tuple(sa) == tuple(sb), "sparse arms disagree"
    return {"fused": timed(fused, iters), "composed": timed(composed, iters)}


def ragged_graph(n, slots, seed=5):
    """R-MAT-free graph from arrays: n nodes, 10 edges each, `slots` uint64 slots of 0..16 values (30% empty)"""
    rng = np.random.RandomState(seed)
    ids = np.arange(1, n + 1, dtype=np.uint64)
    deg = np.full(n, 10)
    grp_ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int64)
    nbr = rng.randint(1, n + 1, size=int(grp_ptr[-1])).astype(np.uint64)
    lens = rng.randint(0, 17, size=n * slots)
    lens[rng.rand(n * slots) < 0.3] = 0
    u64_ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    u64_val = rng.randint(1, 1 << 40, size=int(u64_ptr[-1])).astype(np.uint64)
    feat = rng.uniform(-1, 1, size=(n, 64)).astype(np.float32)
    return eb.Graph.from_csr(ids, grp_ptr, nbr, w=np.ones(len(nbr), np.float32), feat=feat, u64_ptr=u64_ptr, u64_val=u64_val,
                             n_u64_slots=slots)


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", required=True)
    p.add_argument("--configs", default="c2,c4")
    p.add_argument("--iters", type=int, default=50)
    a = p.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a GPU"
    res = {"gpu": gpu_info(), "iters": a.iters, "rng": "philox",
           "launches_per_call": "kernels of libeuler_b200 in one call (torch's own kernels in the composed sparse arm not counted)",
           "results": []}
    for name in a.configs.split(","):
        cfg = CONFIGS[name]
        g = eb.Graph.rmat(cfg["nodes"], cfg["edges"], seed=GRAPH_SEED, feat_dim=cfg["dim"], feat_seed=FEAT_SEED)
        eb.set_graph(g, rng="philox", seed=1)
        seeds = torch.as_tensor(np.random.RandomState(3).randint(1, cfg["nodes"] + 1, size=cfg["batch"]), device="cuda")
        ets = [[0]] * len(cfg["fanout"])
        for nd in (1, 2):
            # ND = 2: the one stored slot twice, the second at half width
            dense = ([0] * nd, [cfg["dim"], cfg["dim"] // 2][:nd])
            r = compare(seeds, ets, cfg["fanout"], dense, ([], []), a.iters)
            res["results"].append(dict(config=name, batch=cfg["batch"], fanout=cfg["fanout"], dim=cfg["dim"], ND=nd, NS=0, **r))
            print(json.dumps(res["results"][-1]), flush=True)
        eb.set_graph(None)
        del g
        torch.cuda.empty_cache()
    g = ragged_graph(2_000_000, 2)
    eb.set_graph(g, rng="philox", seed=1)
    seeds = torch.as_tensor(np.random.RandomState(4).randint(1, 2_000_001, size=1024), device="cuda")
    for ns in (1, 2):
        r = compare(seeds, [[0], [0]], [25, 10], ([0], [64]), (["u64_%d" % k for k in range(ns)], [0] * ns), a.iters)
        res["results"].append(dict(config="ragged-2M", batch=1024, fanout=[25, 10], dim=64, ND=1, NS=ns, **r))
        print(json.dumps(res["results"][-1]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
