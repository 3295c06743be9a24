#!/usr/bin/env python
"""bench.py -- the minibatch-construction step of alibaba/euler's hot path on N B200s.

    python bench.py --gpus 1 --steps K --warmup W            # our CUDA path (default workload = the north-star config)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path on the host cores
    python bench.py --config c2 ...                          # BASELINE configs[1] instead (RMAT 10M/100M, [25,10], B=1024, D=128)

Default workload = BASELINE.json's north-star headline (configs[3]'s graph and shape): synthetic power-law (R-MAT) graph of
100M nodes / 1B edges resident in HBM -- whole on one GPU at N=1, CSR hash-partitioned by id over the GPUs at N>1 -- batch
8192 seeds per GPU, 2-hop sample_fanout [15,10], dense features (dim 256) of the seeds and of hop 1, GraphSAGE neighbor
mean of hop 1 per seed and of hop 2 per hop-1 node.  A "step" = one pass of that path over one batch.
metric = sampled edges/s (slots delivered: B*15 + B*150 per step per GPU); agg_feat_gbs = algorithmic bytes of the feature
gather + segment mean per second (BASELINE's second number).

Before anything is timed a PARITY GATE runs one seeded launch group through the exact timed code path and compares it with
the CPU oracle (sampling on the exported CSR of this very graph: ids / weights / types bit-exact for every batch of the
group; features and neighbor means of one batch against independently generated feature rows, bit-exact); a mismatch aborts.

One JSON line on stdout (rank 0).  See the task's bench contract for the keys.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

CONFIGS = {
    # north-star headline: BASELINE.json configs[3]'s graph and shape (at N=1 the whole graph lives on one GPU)
    "c4": dict(nodes=100_000_000, edges=1_000_000_000, batch=8192, fanout="15,10", dim=256,
               label="north-star headline (BASELINE configs[3])"),
    "c2": dict(nodes=10_000_000, edges=100_000_000, batch=1024, fanout="25,10", dim=128, label="BASELINE configs[1]"),
    # node2vec biased walk (deepwalk / line example path): metric = walker-steps/s
    "c3": dict(nodes=10_000_000, edges=100_000_000, batch=4096, fanout="80", dim=0, label="BASELINE configs[2]"),
    # heterogeneous graph (3 node types / 5 edge types): per-edge-type SampleNeighbor + RGCN scatter_add aggregation
    "c5": dict(nodes=50_000_000, edges=400_000_000, batch=8192, fanout="10", dim=64, label="BASELINE configs[4]"),
}
C5_ETYPES, C5_NTYPES, C5_SEED = 5, 3, 44
# Launch policy of the library for a throughput run (read once by libeuler_b200.so): the HBM-bound row movers (k_sage_mean,
# k_feature) run on 2 CTAs per SM and the issue-bound sampler on 5, so kernels of different lanes share every SM instead of
# queueing behind each other's full-GPU grids (measured: 7.8 -> 9.2 G edges/s at the headline config).  A latency-sensitive
# single-op caller leaves them unset (uncapped grids).
SM_SHARE = {"EU_SAGE_CTAS": "2", "EU_FEATURE_CTAS": "2", "EU_SAMPLE_CTAS": "5"}
CPU_GRAPH_MAX_NODES = 10_000_000   # the CPU arms build the reference's unordered_map<NodeID,Node*> graph: bounded so the arm fits the driver's time box
GRAPH_SEED, FEAT_SEED = 42, 7


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=40)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--config", default="c4", choices=sorted(CONFIGS))
    p.add_argument("--rng", default="minstd", choices=["minstd", "philox"])
    p.add_argument("--nodes", type=int, default=None)
    p.add_argument("--edges", type=int, default=None)
    p.add_argument("--batch", type=int, default=None)
    p.add_argument("--fanout", default=None)
    p.add_argument("--dim", type=int, default=None)
    p.add_argument("--lanes", type=int, default=4, help="execution contexts (streams) with launch groups in flight")
    p.add_argument("--group", type=int, default=0, help="steps (batches) per launch group, 0 = auto: ceil(steps / lanes) capped by a "
                                                         "row budget.  Each batch keeps its own engine and dedup scope "
                                                         "(eu_sample_fanout_batched), only the kernel launches are shared")
    p.add_argument("--no-fuse", action="store_true", help="get_dense_feature + scatter_mean instead of the fused kernel")
    p.add_argument("--no-graphs", action="store_true", help="launch every kernel from the host instead of replaying a CUDA graph per step")
    p.add_argument("--exchange", default="peer", choices=["peer", "nccl"], help="N>1: in-kernel peer-memory exchange or NCCL")
    p.add_argument("--features", default="replicated", choices=["sharded", "replicated"],
                   help="N>1: every rank holds all feature rows (102 GB at the headline config, fits 180 GB of HBM) and only the CSR "
                        "is sharded -- or Euler's scheme, features live with their rows and are fetched / aggregated by the owners")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-gate", action="store_true", help="skip the pre-timing parity gate (debugging only)")
    p.add_argument("--no-e2e-host", action="store_true", help="skip the e2e leg through the *_host C ABI")
    p.add_argument("--cpu-seconds", type=float, default=12.0)
    p.add_argument("--breakdown-iters", type=int, default=6)
    p.add_argument("--p", type=float, default=0.5, help="config c3: node2vec return parameter")
    p.add_argument("--q", type=float, default=2.0, help="config c3: node2vec in-out parameter")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last timed step returned to DIR/<name>.npy (float32 / float64, "
                        "at most 64 MB in all; arrays too large for that keep a fixed seeded sample of their rows)")
    a = p.parse_args()
    if a.dump_outputs and (a.impl != "ours" or a.config in ("c3", "c5") or int(os.environ.get("WORLD_SIZE", "1")) > 1
                           or os.environ.get("EU_BENCH_FORCE_SHARDED")):
        p.error("--dump-outputs covers the single-GPU minibatch step (--impl ours, config c4 or c2, one rank)")
    cfg = CONFIGS[a.config]
    for k in ("nodes", "edges", "batch", "fanout", "dim"):
        if getattr(a, k) is None:
            setattr(a, k, cfg[k])
    if a.config == "c3" and a.lanes == 4:
        a.lanes = 16      # a walk is a chain of 80 dependent steps whose tail is one hub row: more batches in flight hide it
    if a.config == "c4" and a.lanes == 4:
        a.lanes = 8
    a.label = cfg["label"] if all(getattr(a, k) == cfg[k] for k in ("nodes", "edges", "batch", "fanout", "dim")) else "custom"
    return a


def workload_string(args, counts, n_gpus):
    """identical in both arms (ours / --impl reference)"""
    return ("%s: synthetic power-law (R-MAT 0.57/0.19/0.19/0.05) graph %dM nodes/%dM edges, %d-hop sample_fanout %s "
            "batch=%d per GPU, dense features + GraphSAGE-mean aggregation, feat_dim=%d, %d GPU(s)"
            % (args.label, args.nodes // 10**6, args.edges // 10**6, len(counts), counts, args.batch, args.dim, n_gpus))


def workload_config(args, counts, n_gpus):
    """the `config` object both arms print (arm-specific details live under `arm`)"""
    return {"workload": workload_string(args, counts, n_gpus), "nodes": args.nodes, "edges": args.edges, "batch": args.batch,
            "fanout": counts, "feat_dim": args.dim, "rng": args.rng,
            "l2_policy": "inputs larger than L2 (graph >> 126 MB, fresh random seeds every step)"}


def auto_group(args, counts):
    """steps per launch group: all lanes busy for a short driver run (G = ceil(steps / lanes)), bounded by a row budget
    (the widest hop of a group stays under ~5M rows: 16 at configs[1], 4 at the headline config)"""
    if args.group > 0:
        return max(1, min(args.group, args.steps))
    widest = args.batch
    for c in counts:
        widest *= c
    cap = max(1, min(16, 5_000_000 // max(widest, 1)))
    return max(1, min(cap, -(-args.steps // max(args.lanes, 1))))


# ----------------------------------------------------------------------------- clocks sampler
class Clocks:
    """SM clock + throttle reasons sampled DURING the timed region: NVML from a thread every few ms, nvidia-smi -lms as the
    fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.nv, self.run = index, [], None, None, False
        self.max_mhz = None

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else self.index
            self.h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
            self.nv, self.run = nv, True
            threading.Thread(target=self._poll, daemon=True).start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv = self.nv
        names = [("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"), ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
                 ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"), ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap")]
        get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while self.run:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                bits = get(self.h)
                self.rows.append((time.time(), float(mhz), [n for n, a in names if bits & getattr(nv, a, 0)]))
            except Exception:
                pass
            time.sleep(0.004)

    def _read(self):
        for line in self.proc.stdout:
            r = [x.strip() for x in line.split(",")]
            try:
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                self.max_mhz = float(r[2])
                self.rows.append((time.time(), float(r[1]), [nm for k, nm in enumerate(names) if len(r) > 5 + k and r[5 + k].lower().startswith("active")]))
            except Exception:
                pass

    def stop(self, t0, t1):
        if self.nv is None and self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml / nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.run = False
        if self.proc is not None:
            self.proc.terminate()
        rows = [r for r in self.rows if t0 <= r[0] <= t1 + 0.02] or self.rows[-3:]
        sm = sorted(r[1] for r in rows)
        reasons = set()
        for r in rows:
            reasons.update(r[2])
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(reasons), "samples": len(rows), "source": "nvml" if self.nv is not None else "nvidia-smi"}


# ----------------------------------------------------------------------------- our arm
DUMP_BYTES = 63 * 10**6       # --dump-outputs payload; with the .npy headers the files stay under 64 MB


def last_step_outputs(lane, counts):
    """Host copies of what a caller of the step receives for the last batch of the lane's launch group: per hop the sampled
    ids / weights / types, and per source hop the dense features and the neighbor means."""
    b, G = lane.G - 1, lane.G
    out = {}
    for l in range(len(counts)):
        per = lane.n[l + 1] // G
        for name, xs in (("ids", lane.ids), ("weights", lane.w), ("types", lane.ty)):
            out["%s_hop%d" % (name, l + 1)] = xs[l][b * per:(b + 1) * per].cpu().numpy()
    for l in range(len(counts)):
        per = lane.n[l] // G
        out["features_hop%d" % l] = lane.x[l][b * per:(b + 1) * per].cpu().numpy()
        out["neighbor_mean_hop%d" % l] = lane.agg[l][b * per:(b + 1) * per].cpu().numpy()
    return out


def dump_outputs(dirname, arrays):
    """Writes DIR/<name>.npy per array: 64-bit integers as float64 (ids are exact below 2**53), everything else as float32.
    Arrays are written whole, smallest first, while each fits an equal share of what is left of DUMP_BYTES; from the first that
    does not, every remaining array gets an equal share as a sample of its rows -- the same rows on every run, and the same rows
    for arrays of the same length -- whose indices go to DIR/<name>_rows.npy.  Returns {file: shape}."""
    os.makedirs(dirname, exist_ok=True)
    conv = {k: v.astype(np.float64 if v.dtype.kind in "iu" and v.dtype.itemsize > 4 else np.float32) for k, v in arrays.items()}
    names = sorted(conv, key=lambda k: (conv[k].nbytes, k))
    left, share, written = DUMP_BYTES, None, {}
    for i, name in enumerate(names):
        a = conv[name]
        if share is None and a.nbytes > left // (len(names) - i):
            share = left // (len(names) - i)
        if share is not None:
            k = share // (a[0].nbytes + 8)                      # + the row's float64 index
            rows = np.sort(np.random.RandomState(0).permutation(len(a))[:k]).astype(np.float64)
            np.save(os.path.join(dirname, name + "_rows.npy"), rows)
            written[name + "_rows"] = rows.shape
            a = a[rows.astype(np.int64)]
        np.save(os.path.join(dirname, name + ".npy"), a)
        written[name] = a.shape
        left -= a.nbytes
    return written


def step_bytes(B, counts, D):
    """Algorithmic bytes (SURVEY.md section 8d).  Sampling: 48 B per sampled edge + 40 B per seed (CDF mode,
    mean degree 10).  Aggregation (fused): 8 B id + 4D B row read per edge, 4D B write per output row.
    Self features: 8 B id + 4D read + 4D write per row."""
    rows, edges, seeds = B, 0, 0
    agg = 0
    for c in counts:
        seeds += rows
        edges += rows * c
        agg += rows * c * (8 + 4 * D) + rows * 4 * D
        rows *= c
    self_rows = B + B * counts[0] if len(counts) > 1 else B
    feat = self_rows * (8 + 8 * D)
    return {"sample": edges * 48 + seeds * 40, "agg": agg, "self_feat": feat, "edges": edges}


class Lane:
    """One execution context: own stream, RNG engines, device outputs, pinned host buffers."""

    def __init__(self, eb, graph, args, counts, seed, torch, G):
        self.t = torch
        self.stream = torch.cuda.Stream()
        self.ctx = eb.Context(graph, args.rng, seed, self.stream.cuda_stream)
        B, D = args.batch, args.dim
        dev = "cuda"
        self.B, self.D, self.G, self.counts, self.seed = B, D, G, counts, seed
        self.engine_seeds = [seed * 1000 + b for b in range(G)]
        self.ctx.set_engines(G, self.engine_seeds)
        rows = G * B                      # rows of one launch group = G batches
        self.n = [rows]
        for c in counts:
            rows *= c
            self.n.append(rows)
        self.ctx.reserve(max(self.n))
        self.d_seeds = torch.empty(G * B, dtype=torch.int64, device=dev)
        self.ids = [torch.empty(n, dtype=torch.int64, device=dev) for n in self.n[1:]]
        self.w = [torch.empty(n, dtype=torch.float32, device=dev) for n in self.n[1:]]
        self.ty = [torch.empty(n, dtype=torch.int32, device=dev) for n in self.n[1:]]
        L = len(counts)
        self.x = [torch.empty((self.n[l], D), dtype=torch.float32, device=dev) for l in range(L)]      # self feats
        self.agg = [torch.empty((self.n[l], D), dtype=torch.float32, device=dev) for l in range(L)]    # neighbor means
        self.hop_feat = None
        if args.no_fuse:
            self.hop_feat = [torch.empty((self.n[l + 1], D), dtype=torch.float32, device=dev) for l in range(L)]
            self.src = [torch.arange(self.n[l], dtype=torch.int32, device=dev).repeat_interleave(counts[l]) for l in range(L)]
        # host side of the e2e paths (page-locked: the *_host ABI DMAs pinned caller buffers in place)
        self.h_seeds = torch.empty(G * B, dtype=torch.int64).pin_memory()
        self.h_ids = [torch.empty(n, dtype=torch.int64).pin_memory() for n in self.n[1:]]
        self.h_w = [torch.empty(n, dtype=torch.float32).pin_memory() for n in self.n[1:]]
        self.h_t = [torch.empty(n, dtype=torch.int32).pin_memory() for n in self.n[1:]]
        self.h_x = [torch.empty((self.n[l], D), dtype=torch.float32).pin_memory() for l in range(L)]
        self.h_agg = [torch.empty((self.n[l], D), dtype=torch.float32).pin_memory() for l in range(L)]
        self.h2d = 8 * B                  # per step
        self.d2h = (sum(8 * n for n in self.n[1:]) + 2 * sum(4 * self.n[l] * D for l in range(L))) // G
        # through the *_host ABI: seeds up; ids + weights + types down; per hop the source ids (features) and the neighbor
        # ids (fused mean) go up again, self features and means come down
        self.h2d_host = (8 * self.n[0] + sum(8 * self.n[l] + 8 * self.n[l + 1] for l in range(L))) // G
        self.d2h_host = (sum(16 * n for n in self.n[1:]) + 2 * sum(4 * self.n[l] * D for l in range(L))) // G


def make_step(lib, args, counts, et):
    L = len(counts)
    cs = np.ascontiguousarray(counts, dtype=np.int32)
    P = ctypes.c_void_p * L

    def sample(lane, seeds_dev):
        return lib.eu_sample_fanout_batched(lane.ctx._h, seeds_dev.data_ptr(), lane.G, lane.B, et.ctypes.data, et.shape[1], cs.ctypes.data, L, -1,
                                            P(*[x.data_ptr() for x in lane.ids]), P(*[x.data_ptr() for x in lane.w]),
                                            P(*[x.data_ptr() for x in lane.ty]))

    def aggregate(lane, seeds_dev):
        h = lane.ctx._h
        rc = 0
        for l in range(L):
            src_ids = seeds_dev if l == 0 else lane.ids[l - 1]
            rc |= lib.eu_get_dense_feature(h, src_ids.data_ptr(), lane.n[l], 0, lane.D, lane.x[l].data_ptr())
            if args.no_fuse:
                rc |= lib.eu_get_dense_feature(h, lane.ids[l].data_ptr(), lane.n[l + 1], 0, lane.D, lane.hop_feat[l].data_ptr())
                rc |= lib.eu_scatter_mean(h, lane.hop_feat[l].data_ptr(), lane.D, lane.src[l].data_ptr(), lane.n[l + 1],
                                          lane.n[l], lane.agg[l].data_ptr())
            else:
                rc |= lib.eu_sage_mean_aggregate(h, lane.ids[l].data_ptr(), lane.n[l], counts[l], lane.D, lane.agg[l].data_ptr())
        return rc

    def step(lane, seeds_dev, what="all"):
        rc = 0
        if what in ("all", "sample"):
            rc |= sample(lane, seeds_dev)
        if what in ("all", "aggregate"):
            rc |= aggregate(lane, seeds_dev)
        if rc:
            raise RuntimeError("euler_b200: " + lib.eu_last_error().decode())

    def host_step(lane):
        """the same step through the reference-facing *_host C ABI: HOST buffers in, HOST buffers out (each call returns when
        its results have landed)"""
        h = lane.ctx._h
        rc = lib.eu_sample_fanout_batched_host(h, lane.h_seeds.data_ptr(), lane.G, lane.B, et.ctypes.data, et.shape[1], cs.ctypes.data, L, -1,
                                               P(*[x.data_ptr() for x in lane.h_ids]), P(*[x.data_ptr() for x in lane.h_w]),
                                               P(*[x.data_ptr() for x in lane.h_t]))
        for l in range(L):
            src = lane.h_seeds if l == 0 else lane.h_ids[l - 1]
            rc |= lib.eu_get_dense_feature_host(h, src.data_ptr(), lane.n[l], 0, lane.D, lane.h_x[l].data_ptr())
            rc |= lib.eu_sage_mean_aggregate_host(h, lane.h_ids[l].data_ptr(), lane.n[l], counts[l], lane.D, lane.h_agg[l].data_ptr())
        if rc:
            raise RuntimeError("euler_b200: " + lib.eu_last_error().decode())
    step.host = host_step
    return step


def parity_gate(args, counts, graph, lane, raw_step, host_seeds, torch):
    """One seeded launch group through the timed code path vs the CPU oracle.  Sampling: every batch of the group, ids /
    weights / types bit-exact, on the CSR exported from this very graph.  Features + neighbor means: batch 0 against feature
    rows generated independently on the host (oracle/rmat_gen.c), bit-exact (sorted fixed-fanout segments sum in the
    reference's order).  Raises on any mismatch."""
    from oracle import pyoracle as po
    t0 = time.time()
    G, B, D, L = lane.G, lane.B, lane.D, len(counts)
    ex = graph.export(with_feat=False)
    t_export = time.time() - t0
    og = po.OracleGraph(ex["ids"], ex["node_type"], ex["node_w"], 1, ex["grp_ptr"], ex["nbr"], ex["cum_w"],
                        np.zeros(len(ex["ids"]), np.float32))
    seeds = host_seeds[:G].copy()
    seeds[0, :8] = [0, -1, args.nodes + 12345, seeds[0, 9], seeds[0, 9], 1, args.nodes, seeds[0, 20]]   # placeholders, absent, duplicates, range ends
    lane.ctx.set_engines(G, lane.engine_seeds)
    with torch.cuda.stream(lane.stream):
        lane.d_seeds.copy_(torch.from_numpy(seeds.reshape(-1)))
        raw_step(lane, lane.d_seeds)
    lane.stream.synchronize()
    et = [[0]] * L
    checked = 0
    for b in range(G):
        po.seed(lane.engine_seeds[b])
        o_ids, o_w, o_t = og.op_sample_fanout(seeds[b], et, counts)
        for l in range(L):
            per = lane.n[l + 1] // G
            sl = slice(b * per, (b + 1) * per)
            for name, got, want in (("ids", lane.ids[l], o_ids[l]), ("weights", lane.w[l], o_w[l]), ("types", lane.ty[l], o_t[l])):
                gnp = got[sl].cpu().numpy()
                if not np.array_equal(gnp, want):
                    bad = np.nonzero(gnp != want)[0]
                    raise SystemExit("PARITY GATE FAILED: %s of hop %d, batch %d differ from the oracle at %d of %d slots (first %d: got %r want %r)"
                                     % (name, l + 1, b, len(bad), len(want), bad[0], gnp[bad[0]], want[bad[0]]))
            checked += 3 * per
        if b == 0:
            feats = [po.rmat_feat_rows(seeds[0], args.nodes, D, FEAT_SEED)] + \
                    [po.rmat_feat_rows(o_ids[l], args.nodes, D, FEAT_SEED) for l in range(L)]
            for l in range(L):
                per = lane.n[l] // G
                x = lane.x[l][:per].cpu().numpy()
                if not np.array_equal(x, feats[l]):
                    raise SystemExit("PARITY GATE FAILED: dense features of hop %d differ from the independently generated rows" % l)
                want = po.scatter_mean(feats[l + 1], np.repeat(np.arange(per, dtype=np.int32), counts[l]), per)
                a = lane.agg[l][:per].cpu().numpy()
                if not np.array_equal(a, want):
                    err = float(np.max(np.abs(a - want) / (np.abs(want) + 1e-6)))
                    raise SystemExit("PARITY GATE FAILED: neighbor means of hop %d differ from the oracle (max rel err %.3g)" % (l + 1, err))
                checked += 2 * per * D
    lane.ctx.set_engines(G, lane.engine_seeds)
    del og, ex
    return {"passed": True, "batches": G, "values_compared": int(checked), "seconds": round(time.time() - t0, 2),
            "csr_export_seconds": round(t_export, 2),
            "what": "one launch group of %d batches through the timed code path vs oracle/euler_oracle.c on the exported CSR of the bench "
                    "graph: ids/weights/types of every hop bit-exact; dense features + fused neighbor means of batch 0 bit-exact vs "
                    "oracle/rmat_gen.c feature rows + the oracle's scatter_mean" % G}


def run_ours(args):
    import torch
    import euler_b200 as eb
    from euler_b200 import _lib
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 or os.environ.get("EU_BENCH_FORCE_SHARDED"):   # the env knob runs the sharded pipeline on one rank (no link): its compute-only cost
        return run_sharded(args, world, rank, local)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    for k, v in SM_SHARE.items():
        os.environ.setdefault(k, v)
    lib = _lib.load()
    counts = [int(x) for x in args.fanout.split(",")]
    et = np.zeros((len(counts), 1), np.int32)
    # exactly K steps are timed: K // G full launch groups + one tail group of K % G batches (its own lane + graph)
    G = auto_group(args, counts)
    tail = args.steps % G
    t0 = time.time()
    graph = eb.Graph.rmat(args.nodes, args.edges, seed=GRAPH_SEED, feat_dim=args.dim, feat_seed=FEAT_SEED, device=local)
    torch.cuda.synchronize()
    t_graph = time.time() - t0
    n_lanes = max(1, min(args.lanes, args.steps // G if args.steps >= G else 1))
    lanes = [Lane(eb, graph, args, counts, 12345 + i, torch, G) for i in range(n_lanes)]
    tail_lane = Lane(eb, graph, args, counts, 12345 + n_lanes, torch, tail) if tail else None
    # the *_host calls are synchronous per caller thread: the e2e leg through them runs one thread per lane on HOST_LANES lanes
    # = the reference's client thread pool (euler/client/query_proxy.cc:205-210: 8 threads) so that PCIe stays busy
    HOST_LANES = 8
    raw_step = make_step(lib, args, counts, et)
    nb = args.warmup + args.steps
    n_seed_batches = -(-max(nb, 4 * G) // G) * G
    host_seeds = np.stack([np.random.RandomState(1000 + i).randint(1, args.nodes + 1, size=args.batch)
                           for i in range(n_seed_batches)]).astype(np.int64)
    gate = {"passed": None, "skipped": "--no-gate"}
    if not args.no_gate:
        if args.rng != "minstd":
            gate = {"passed": None, "skipped": "philox mode has no bit-exact oracle stream (statistical tests only)"}
        else:
            gate = parity_gate(args, counts, graph, lanes[0], raw_step, host_seeds, torch)
    per_step_launches = None
    use_graphs = not args.no_graphs
    if use_graphs:
        # the step has static shapes and device-resident RNG state: capture it once per lane and
        # replay (one graph launch per launch group instead of ~14 kernel launches from Python)
        for ln in lanes + ([tail_lane] if tail_lane else []):
            with torch.cuda.stream(ln.stream):
                ln.d_seeds.fill_(1)
                raw_step(ln, ln.d_seeds)          # warm (also sizes every scratch buffer)
            ln.stream.synchronize()
            l_before = lib.eu_launch_count()
            ln.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(ln.graph, stream=ln.stream):
                raw_step(ln, ln.d_seeds)
            ln.launches = lib.eu_launch_count() - l_before
        per_step_launches = ((args.steps // G) * lanes[0].launches + (tail_lane.launches if tail_lane else 0)) / args.steps

    def step(ln, seeds_dev):
        if use_graphs:
            if seeds_dev is not ln.d_seeds:
                ln.d_seeds.copy_(seeds_dev, non_blocking=True)
            ln.graph.replay()
        else:
            raw_step(ln, seeds_dev)
    dev_seeds = torch.from_numpy(host_seeds).cuda()
    n_groups_avail = n_seed_batches // G

    def group_seeds(first, i):
        g0 = ((first // G + i) % n_groups_avail) * G
        return g0, dev_seeds[g0:g0 + G].reshape(-1)
    bts = step_bytes(args.batch, counts, args.dim)
    main = torch.cuda.current_stream()
    all_lanes = lanes + ([tail_lane] if tail_lane else [])

    host_lanes = []
    last = {}                                            # the lane that ran the last step of the latest run()

    def run(n_steps, first, mode):
        """n_steps steps round-robin over the lanes; returns device ms (events on the main stream, lanes fork from / join
        into it).  mode: "dev" = seeds resident in HBM; "e2e" = device entry points + pinned H2D / D2H copies;
        "host" = the *_host C ABI, one host thread per lane (the reference's client pool, query_proxy.cc:205-210)."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        rem = n_steps % G
        use_tail = tail_lane is not None and rem == tail_lane.G
        n_groups = n_steps // G + (1 if rem else 0)     # an untimed (warm-up) remainder is rounded up to a full group
        pool = lanes
        if mode == "host":
            while len(lanes) + len(host_lanes) < min(HOST_LANES, max(n_groups, len(lanes))):
                host_lanes.append(Lane(eb, graph, args, counts, 22345 + len(host_lanes), torch, G))
            pool = lanes + host_lanes
        work = []                                        # (lane, first seed batch, batches)
        for i in range(n_groups):
            ln = pool[i % len(pool)]
            g0, sd = group_seeds(first, i)
            if use_tail and i == n_groups - 1:
                ln, sd = tail_lane, sd[:rem * args.batch]
            work.append((ln, g0, sd))
        if work:
            last["lane"] = work[-1][0]
        torch.cuda.synchronize()
        ev0.record(main)
        for ln in all_lanes + host_lanes:
            ln.stream.wait_event(ev0)
        if mode == "host":
            def worker(ln):
                for (l2, g0, _) in work:
                    if l2 is ln:
                        ln.h_seeds.copy_(torch.from_numpy(host_seeds[g0:g0 + ln.G].reshape(-1)))
                        raw_step.host(ln)
            ths = [threading.Thread(target=worker, args=(ln,)) for ln in all_lanes + host_lanes]
            for t in ths:
                t.start()
            for t in ths:
                t.join()
        else:
            for i, (ln, g0, sd) in enumerate(work):
                with torch.cuda.stream(ln.stream):
                    if mode == "e2e":
                        # the lane's pinned buffers are reused every len(lanes) groups
                        ln.stream.synchronize() if i >= len(lanes) else None
                        ln.h_seeds.copy_(torch.from_numpy(host_seeds[g0:g0 + ln.G].reshape(-1)))
                        ln.d_seeds.copy_(ln.h_seeds, non_blocking=True)
                        step(ln, ln.d_seeds)
                        for l in range(len(counts)):
                            ln.h_ids[l].copy_(ln.ids[l], non_blocking=True)
                            ln.h_x[l].copy_(ln.x[l], non_blocking=True)
                            ln.h_agg[l].copy_(ln.agg[l], non_blocking=True)
                    else:
                        step(ln, sd)
        for ln in all_lanes + host_lanes:
            main.wait_stream(ln.stream)
        ev1.record(main)
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1)

    run(-(-args.warmup // G) * G, 0, "dev")
    if tail_lane:
        run(tail, 0, "dev")
    clocks = Clocks(local)
    clocks.start()
    time.sleep(0.3)
    l0 = lib.eu_launch_count()
    w0 = time.time()
    ms = run(args.steps, args.warmup, "dev")
    w1 = time.time()
    launches = lib.eu_launch_count() - l0
    if use_graphs:
        launches = int(per_step_launches * args.steps)  # kernels of ours inside the replayed graphs
    clk = clocks.stop(w0, w1)
    if args.dump_outputs:
        files = dump_outputs(args.dump_outputs, last_step_outputs(last["lane"], counts))
        print("--dump-outputs: %s" % ", ".join("%s.npy %s" % (k, v) for k, v in files.items()), file=sys.stderr)
    # end-to-end passes: warm EVERY lane the timed pass will use (a lane's first *_host call grows its pinned staging and device
    # scratch -- cudaHostAlloc / cudaMalloc of hundreds of MB, which one box in round 2 took 40 ms per step to do inside the timed
    # region), and the tail lane, before timing
    n_timed_groups = -(-args.steps // G)
    run(G * max(min(n_timed_groups, len(lanes)), 1), 0, "e2e")
    if tail_lane:
        run(tail, 0, "e2e")
    ms_e2e = run(args.steps, args.warmup, "e2e")
    ms_host = None
    if not args.no_e2e_host:
        for _ in range(2):
            run(G * max(min(HOST_LANES, max(n_timed_groups, len(lanes))), 1), 0, "host")
        if tail_lane:
            run(tail, 0, "host")
        ms_host = run(args.steps, args.warmup, "host")
    edges_step = bts["edges"]
    value = edges_step * args.steps / (ms * 1e-3)

    # ---- sub-rates (BASELINE's metric is two numbers): sampling only and feature gather + aggregation only, one lane, serial
    ln = lanes[0]
    sub = {}
    for what in ("sample", "aggregate"):
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        with torch.cuda.stream(ln.stream):
            raw_step(ln, group_seeds(0, 0)[1], "sample")
            raw_step(ln, group_seeds(0, 0)[1], what)
            evs[0].record(ln.stream)
            for it in range(args.breakdown_iters):
                raw_step(ln, group_seeds(0, it)[1] if what == "sample" else ln.d_seeds, what)
            evs[1].record(ln.stream)
        ln.stream.synchronize()
        sub[what] = evs[0].elapsed_time(evs[1]) / (args.breakdown_iters * G)   # ms per step

    # ---- per-kernel breakdown on one lane, serial: the library brackets each of its kernels with CUDA
    # events on the lane's stream (eu_ctx_profile); explains `value` and feeds the roofline
    Lh = len(counts)
    valid_edges = [0] * Lh
    lib.eu_ctx_profile(ln.ctx._h, 1)
    with torch.cuda.stream(ln.stream):
        for it in range(args.breakdown_iters):
            raw_step(ln, group_seeds(0, it)[1])
            for l in range(Lh):
                valid_edges[l] += int((ln.ids[l] != -1).sum().item())
    buf = ctypes.create_string_buffer(1 << 16)
    lib.eu_ctx_profile_read(ln.ctx._h, buf, len(buf))
    lib.eu_ctx_profile(ln.ctx._h, 0)
    kernels = []
    for line in buf.value.decode().strip().splitlines():
        nm, rows, n, ms_tot = line.rsplit(",", 3)
        kernels.append({"kernel": nm, "rows": int(rows), "launches_per_step": int(n) / (args.breakdown_iters * G),
                        "ms_per_launch": float(ms_tot) / int(n), "ms_per_step": float(ms_tot) / (args.breakdown_iters * G)})
    kernels.sort(key=lambda k: -k["ms_per_step"])
    phases = {"%s[rows=%d]" % (k["kernel"], k["rows"]): round(k["ms_per_step"], 5) for k in kernels}
    valid_frac = [valid_edges[l] / (args.breakdown_iters * ln.n[l + 1]) for l in range(Lh)]
    D = args.dim

    def alg_bytes(k):
        """Algorithmic bytes of one launch (SURVEY.md section 8d), counting feature-row reads only for ids that
        exist (default-filled slots read nothing) and sampling reads only for rows that sample."""
        nm, rows = k["kernel"], k["rows"]
        hop = ln.n.index(rows) if rows in ln.n else 0
        if nm.startswith("k_sage_mean"):
            c = counts[hop]
            return rows * c * 8 + valid_frac[hop] * rows * c * 4 * D + rows * 4 * D
        if nm == "k_feature":
            vf = 1.0 if hop == 0 else valid_frac[hop - 1]
            return rows * 8 + vf * rows * 4 * D + rows * 4 * D
        if nm.startswith("k_sample"):
            c = counts[hop]
            # per sampled edge: col_idx 8 + two cumulative weights 8 + CDF probes 4*ceil(log2 deg~10)=16 + output 16;
            # per row: first 4 + mask/offsets 12 + rowof 8 + row_ptr pair 16; default rows only write 16 B / slot
            return rows * 40 + valid_frac[hop] * rows * c * 48 + (1 - valid_frac[hop]) * rows * c * 16
        if nm == "k_prepare":
            return rows * (8 + 16 + 4 + 8 + 16)   # seed id, dedup slot, first, rowof, row_ptr pair
        if nm == "k_dedup_insert":
            return rows * (8 + 16)
        return 0
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    for k in kernels:
        k["algorithmic_bytes_per_launch"] = int(alg_bytes(k))
        k["achieved_gbs"] = round(k["algorithmic_bytes_per_launch"] / (k["ms_per_launch"] * 1e-3) / 1e9, 1)
        k["frac_of_measured_hbm_peak"] = round(k["achieved_gbs"] / peak, 4)
    dom = kernels[0]
    # DRAM traffic of the dominant kernel from the committed ncu capture (same workload and launch shape only)
    traffic, traffic_src, l2_hit = None, None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        ent = tj.get(args.config, {}).get("kernels", {}).get(dom["kernel"].split("<")[0], {}).get(str(dom["rows"]))
        if args.label != "custom" and ent:
            traffic, l2_hit = ent["dram_bytes_per_launch"], ent.get("l2_hit_rate")
            traffic_src = "profiles/r02_traffic.json (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch)"
    except Exception:
        pass
    roof = {"bound": "hbm", "kernel": "%s over %d rows (largest share of the step)" % (dom["kernel"], dom["rows"]),
            "achieved": dom["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": dom["frac_of_measured_hbm_peak"],
            "traffic": traffic, "traffic_source": traffic_src, "l2_hit_rate": l2_hit,
            "note": "achieved = algorithmic bytes / live kernel time; a feature-gathering kernel re-reads hub rows from the 126 MB L2, "
                    "so `traffic` (DRAM bytes) stays below the algorithmic bytes",
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst)" if peaks else "fallback 6650 (B200_PROFILING.md)",
            "algorithmic_bytes_per_launch": dom["algorithmic_bytes_per_launch"], "kernel_ms": round(dom["ms_per_launch"], 5),
            "valid_edge_fraction_per_hop": [round(v, 4) for v in valid_frac],
            "all_kernels": kernels}
    # the step as a whole: the kernels of different lanes overlap (each on its SM share), so the sum of their algorithmic bytes over the
    # timed step is the figure that says how close the PATH is to the HBM roof; the per-kernel lines above are each kernel timed alone
    step_alg = sum(k["algorithmic_bytes_per_launch"] * k["launches_per_step"] for k in kernels)
    step_gbs = step_alg / (ms / args.steps * 1e-3) / 1e9
    roof["step"] = {"algorithmic_bytes_per_step": int(step_alg), "achieved": round(step_gbs, 1), "frac": round(step_gbs / peak, 4),
                    "how": "sum of every kernel's algorithmic bytes per step / timed ms_per_step (all lanes in flight)"}
    if any(os.environ.get(k) not in (None, "0") for k in SM_SHARE):
        roof["note"] += "; per-kernel times are single-lane on the kernel's SM share (%s), not a full-GPU grid" % ", ".join(
            "%s=%s" % (k, os.environ.get(k)) for k in SM_SHARE)
    # aggregated-feature bytes per step with the measured valid fractions (default slots read no row)
    agg_bytes = 0
    for l in range(Lh):
        agg_bytes += ln.n[l] * counts[l] * 8 + valid_frac[l] * ln.n[l] * counts[l] * 4 * D + ln.n[l] * 4 * D
        vf = 1.0 if l == 0 else valid_frac[l - 1]
        agg_bytes += ln.n[l] * 8 + vf * ln.n[l] * 4 * D + ln.n[l] * 4 * D
    agg_bytes /= G   # ln.n counts the rows of a whole launch group
    cfg = workload_config(args, counts, 1)
    e2e_dev = {"value": edges_step * args.steps / (ms_e2e * 1e-3), "ms_per_step": ms_e2e / args.steps,
               "api": "device entry points + pinned-tensor copies issued by the caller"}
    if ms_host is not None:
        e2e = {"value": edges_step * args.steps / (ms_host * 1e-3), "unit": "edges/s", "h2d_bytes_per_step": lanes[0].h2d_host,
               "d2h_bytes_per_step": lanes[0].d2h_host, "ms_per_step": ms_host / args.steps,
               "api": "eu_sample_fanout_batched_host + eu_get_dense_feature_host + eu_sage_mean_aggregate_host (HOST buffers in and out; "
                      "one host thread per lane, %d lanes); PCIe-bound: %.0f MB D2H per step" % (len(lanes) + len(host_lanes), lanes[0].d2h_host / 1e6),
               "pcie_gbs": round((lanes[0].d2h_host + lanes[0].h2d_host) * args.steps / (ms_host * 1e-3) / 1e9, 1),
               "device_api_variant": e2e_dev}
    else:
        e2e = {"value": e2e_dev["value"], "unit": "edges/s", "h2d_bytes_per_step": lanes[0].h2d, "d2h_bytes_per_step": lanes[0].d2h,
               "ms_per_step": e2e_dev["ms_per_step"], "api": e2e_dev["api"]}
    out = {
        "metric": "sampled_edges_per_sec", "value": value, "unit": "edges/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64 ids / f32 weights+features (f64 CDF compare)", "data": "synthetic",
        "config": cfg,
        "arm": {"lanes_in_flight": len(lanes), "steps_per_launch_group": G, "cuda_graphs": use_graphs, "fused_aggregation": not args.no_fuse,
                "graph_hbm_gb": round(graph.hbm_bytes / 1e9, 1),
                "sm_share": {k: os.environ.get(k) for k in SM_SHARE},
                "parallelism": "1 GPU, %d streams x groups of %d independent batches per launch" % (len(lanes), G)},
        "parity_gate": gate,
        "agg_feat_gbs": agg_bytes * args.steps / (ms * 1e-3) / 1e9,
        "sub_rates": {"sampling_only_edges_per_s": edges_step / (sub["sample"] * 1e-3),
                      "aggregation_only_gbs": agg_bytes / (sub["aggregate"] * 1e-3) / 1e9,
                      "ms_per_step": {k: round(v, 5) for k, v in sub.items()}, "how": "one lane, serial launch groups, device-timed"},
        "e2e": e2e,
        "gpu_launches": int(launches),
        "clocks": clk,
        "roofline": roof,
        "phases_ms_single_lane": {k: round(v, 5) for k, v in phases.items()},
        "step_algorithmic_bytes": bts,
        "graph_build_s": round(t_graph, 2), "hbm_graph_bytes": graph.hbm_bytes,
    }
    if not args.no_cpu_baseline and rank == 0:
        for ln_ in all_lanes + host_lanes:
            del ln_.h_x, ln_.h_agg
        out["cpu_baseline"] = cpu_baseline(args, counts)
    emit(out)


def nvlink_counters(index):
    """cumulative NVLink data bytes (tx, rx) of GPU `index` from the driver's own link counters
    (`nvidia-smi nvlink -gt d`: per link "Data Tx: N KiB" / "Data Rx: N KiB"); None when the tool cannot report them"""
    try:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else index
        txt = subprocess.run(["nvidia-smi", "nvlink", "-gt", "d", "-i", str(phys)], capture_output=True, text=True, timeout=20).stdout
        tx = rx = 0
        seen = False
        for line in txt.splitlines():
            line = line.strip()
            if "Data Tx:" in line or "Data Rx:" in line:
                val = line.split(":")[-1].strip().split()
                n = int(val[0]) * {"KiB": 1024, "MiB": 1 << 20, "GiB": 1 << 30, "B": 1}.get(val[1] if len(val) > 1 else "KiB", 1024)
                if "Data Tx:" in line:
                    tx += n
                else:
                    rx += n
                seen = True
        return (tx, rx) if seen else None
    except Exception:
        return None


# ----------------------------------------------------------------------------- sharded arm (N > 1)
def sharded_gate(args, counts, graph, rank, world, torch, dist):
    """N > 1 parity gate: one seeded batch per rank through the peer-memory exchange (csrc/p2p.cu) vs the SAME sharded
    orchestration run with the CPU oracle as every shard's engine over a gloo group (euler_b200/sharded.py::ShardedGraph +
    tests/sharded_common.py::OracleShardOps): ids / weights / types of every hop bit-exact on every rank."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import sharded_common as sc
    from oracle import pyoracle as po
    from euler_b200.sharded import PeerShardedGraph, ShardedGraph, TorchExchange
    t0 = time.time()
    B, L = args.batch, len(counts)
    n = [B]
    for c in counts:
        n.append(n[-1] * c)
    ex = graph.export(with_feat=False)

    class GateOps(sc.OracleShardOps):
        def __init__(self, seed):
            self.torch = torch
            self.og = po.OracleGraph(ex["ids"], ex["node_type"], ex["node_w"], 1, ex["grp_ptr"], ex["nbr"], ex["cum_w"],
                                     np.zeros(len(ex["ids"]), np.float32))
            po.seed(seed)
    seeds = np.random.RandomState(777 + rank).randint(1, args.nodes + 1, size=B).astype(np.int64)
    seeds[:4] = [0, -1, args.nodes + 99, seeds[5]]
    ets = [[0]] * L
    pg = PeerShardedGraph(graph, rank, world, max_rows=max(n[:-1]), max_count=max(counts), max_feat_rows=1, max_dim=4, rng="minstd",
                          seed=9100 + rank)
    p_ids, p_ws, p_ts = pg.sample_fanout(seeds, ets, counts, -1)
    torch.cuda.synchronize()
    err = pg.error()
    gl = dist.new_group(backend="gloo")
    sg = ShardedGraph(GateOps(9100 + rank), TorchExchange(gl))
    o_ids, o_ws, o_ts = sg.sample_fanout(torch.from_numpy(seeds), ets, counts, -1)
    bad = []
    if err:
        bad.append("peer exchange timed out")
    for l in range(L):
        for name, got, want in (("ids", p_ids[l + 1], o_ids[l + 1]), ("weights", p_ws[l], o_ws[l]), ("types", p_ts[l], o_ts[l])):
            if not np.array_equal(got.cpu().numpy().reshape(-1), want.numpy().reshape(-1)):
                bad.append("rank %d: %s of hop %d differ from the oracle-backed sharded run" % (rank, name, l + 1))
    allbad = [None] * world
    dist.all_gather_object(allbad, bad)
    pg.close()
    flat = [b for x in allbad for b in x]
    if flat:
        raise SystemExit("PARITY GATE FAILED: " + "; ".join(flat))
    return {"passed": True, "ranks": world, "values_compared_per_rank": int(3 * sum(n[1:])), "seconds": round(time.time() - t0, 2),
            "what": "one seeded batch per rank through the peer-memory exchange vs ShardedGraph over gloo with the C oracle as every "
                    "shard's engine (same per-shard seeds): ids/weights/types of every hop bit-exact on every rank"}


def run_sharded(args, world, rank, local):
    """Weak scaling: the graph's CSR is hash-partitioned by id over the ranks (owner = id % N, Euler's shard scheme), every
    rank constructs its own batch per step; each hop resolves remote ids through an all-to-all over NVLink -- by default
    done by the kernels themselves on peer memory (csrc/p2p.cu: no NCCL call, no host sync; the whole step is one CUDA graph
    per lane), or with NCCL (--exchange nccl, euler_b200/sharded.py::ShardedGraph).  Dense features: replicated on every
    rank by default (local fetch + aggregation), or sharded with their rows (--features sharded)."""
    import torch
    import torch.distributed as dist
    import euler_b200 as eb
    from euler_b200 import _lib
    from euler_b200.sharded import CudaShardOps, PeerShardedGraph, ShardedGraph, TorchExchange
    torch.cuda.set_device(local)
    if not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    for k, v in SM_SHARE.items():
        os.environ.setdefault(k, v)
    lib = _lib.load()
    counts = [int(x) for x in args.fanout.split(",")]
    L, B, D = len(counts), args.batch, args.dim
    t0 = time.time()
    replicated = args.features == "replicated" and args.exchange == "peer"
    graph = eb.Graph.rmat_shard(args.nodes, args.edges, rank, world, seed=GRAPH_SEED, feat_dim=0 if replicated else D,
                                feat_seed=FEAT_SEED, device=local)
    feat_graph = None
    if replicated:
        # all feature rows on every rank: the generator's features are a hash of (global node index, column), so a full-node
        # graph with a token number of edges carries exactly the rows the shards would hold
        feat_graph = eb.Graph.rmat(args.nodes, 1024, seed=GRAPH_SEED, feat_dim=D, feat_seed=FEAT_SEED, device=local)
    torch.cuda.synchronize()
    t_graph = time.time() - t0
    n = [B]
    for c in counts:
        n.append(n[-1] * c)
    peer = args.exchange == "peer"
    gate = {"passed": None, "skipped": "--no-gate"}
    if not args.no_gate and peer and args.rng == "minstd":
        gate = sharded_gate(args, counts, graph, rank, world, torch, dist)
    # launch group: G batches share every exchange (peer path) -- the kernels and NVLink round trips of an exchange are paid
    # once per G steps; each batch keeps its own engine and dedup scope on every shard (eu_sym_sample_hop_batched)
    G = auto_group(args, counts) if peer else 1
    n_lanes = max(1, min(args.lanes, args.steps // G if args.steps >= G else 1)) if peer else 1
    tail = args.steps % G                 # exactly K steps: K // G full groups + one tail group of K % G batches
    src = [torch.arange(n[l], dtype=torch.int32, device="cuda").repeat_interleave(counts[l]) for l in range(L)] if not peer else None
    n_self = sum(n[:L])                   # rows whose own features are materialised (hop 0 .. L-1)

    class SLane:
        pass
    E2E_LANES = 4
    lanes = []
    for i in range(n_lanes + (1 if tail else 0)):
        ln = SLane()
        ln.G = G if i < n_lanes else tail
        G_main, G = G, ln.G               # the buffers below are sized for this lane's group
        ln.stream = torch.cuda.Stream()
        seed = 12345 + rank * 1000 + i * 64
        if peer:
            feat_rows = 1 if replicated else G * max(max(n), world * max(n[:-1]))
            ln.sg = PeerShardedGraph(graph, rank, world, max_rows=G * max(n[:-1]), max_count=max(counts),
                                     max_feat_rows=feat_rows, max_dim=4 if replicated else D, rng=args.rng, seed=seed, engines=G,
                                     feature_graph=feat_graph)
            ln.ctx = ln.sg.ctx
        else:
            ln.ops = CudaShardOps(graph, args.rng, seed)
            ln.sg = ShardedGraph(ln.ops, TorchExchange())
            ln.ctx = ln.ops.ctx
            ln.ctx.reserve(max(n) * 2 + sum(n))
        # one id buffer: [G*n0 seeds | G*n1 hop-1 ids | ...]; slices of it are the hop outputs and the feature request
        ln.idbuf = torch.empty(G * sum(n), dtype=torch.int64, device="cuda")
        offs = [0]
        for x in n:
            offs.append(offs[-1] + G * x)
        ln.d_seeds = ln.idbuf[:G * B].view(G, B)
        ln.ids = [ln.idbuf[offs[l + 1]:offs[l + 2]] for l in range(L)]
        ln.agg = [torch.empty((G * n[l], D), dtype=torch.float32, device="cuda") for l in range(L)]
        ln.x = torch.empty((G * n_self, D), dtype=torch.float32, device="cuda")
        if i < E2E_LANES or i >= n_lanes:   # pinned host side of the e2e pass: PCIe-bound, 4 lanes (+ the tail) saturate the link
            ln.h_seeds = torch.empty((G, B), dtype=torch.int64).pin_memory()
            ln.h_ids = [torch.empty(G * x, dtype=torch.int64).pin_memory() for x in n[1:]]
            ln.h_x = torch.empty((G * n_self, D), dtype=torch.float32).pin_memory()
            ln.h_agg = [torch.empty((G * n[l], D), dtype=torch.float32).pin_memory() for l in range(L)]
        G = G_main
        lanes.append(ln)
    tail_lane = lanes.pop() if tail else None
    all_lanes = lanes + ([tail_lane] if tail_lane else [])

    def raw_step(ln):
        """one launch group = ln.G steps; seeds are in ln.d_seeds"""
        sg = ln.sg
        G = ln.G
        if peer:
            frontier = ln.d_seeds.view(-1)
            for l in range(L):
                # the frontier of hop l+1 is read straight from the symmetric output of hop l (consumed by the bucket
                # kernels before this rank's push lets any owner overwrite it)
                eng, o_ids, o_w, o_t = sg.hop(frontier, [0], counts[l], -1, nb=G)
                ln.ids[l].copy_(o_ids)
                frontier = eng
            if replicated:
                # every rank holds all feature rows (PeerShardedGraph(feature_graph=...)): fetch + aggregation are the
                # single-GPU kernels, nothing crosses NVLink
                sg.get_dense_feature(ln.idbuf[:G * n_self], 0, D, out=ln.x)
                for l in range(L):
                    sg.sage_mean(ln.ids[l], G * n[l], counts[l], D, out=ln.agg[l])
                ln.x_view = ln.x
                return
            # the hop-(l+1) features are summed by their owners and never cross NVLink row by row
            for l in range(L):
                sg.sage_mean(ln.ids[l], G * n[l], counts[l], D, out=ln.agg[l])
            # own features of the hop-0..L-1 nodes: rows stay in the symmetric region until the next group (a consumer
            # reads them there); the e2e path copies them to the host from there
            ln.x_view = sg.get_dense_feature(ln.idbuf[:G * n_self], 0, D, clone=False)
            return
        seeds_dev = ln.d_seeds.view(-1)
        ids, ws, ts = sg.sample_fanout(seeds_dev, [[0]] * L, counts, -1)
        for l in range(L):
            ln.ids[l].copy_(ids[l + 1])
        feats = sg.get_dense_feature(torch.cat(ids), 0, D)
        ln.ctx.set_stream(torch.cuda.current_stream().cuda_stream)
        ln.x_view = feats[:n_self]
        off = 0
        for l in range(L):
            off += n[l]
            rc = lib.eu_scatter_mean(ln.ctx._h, feats[off:off + n[l + 1]].data_ptr(), D, src[l].data_ptr(), n[l + 1], n[l], ln.agg[l].data_ptr())
            if rc:
                raise RuntimeError(lib.eu_last_error().decode())

    n_seed_groups = max(-(-(args.warmup + args.steps) // G), 8)
    host_seeds = np.stack([np.random.RandomState(1000 + rank * 100003 + i).randint(1, args.nodes + 1, size=(G, B))
                           for i in range(n_seed_groups)]).astype(np.int64)
    dev_seeds = torch.from_numpy(host_seeds).cuda()

    use_graphs = peer and not args.no_graphs
    if use_graphs:
        for ln in all_lanes:
            with torch.cuda.stream(ln.stream):
                ln.d_seeds.copy_(dev_seeds[0][:ln.G])
                raw_step(ln)
            ln.stream.synchronize()
        dist.barrier()
        for ln in all_lanes:
            ln.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(ln.graph, stream=ln.stream):
                raw_step(ln)
        dist.barrier()

    def step(ln):
        if use_graphs:
            ln.graph.replay()
        else:
            raw_step(ln)

    main = torch.cuda.current_stream()

    def run(n_steps, first, e2e):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        ev0.record(main)
        rem = n_steps % G
        use_tail = tail_lane is not None and rem == tail_lane.G
        n_groups = n_steps // G + (1 if rem else 0)     # an untimed (warm-up) remainder is rounded up to a full group
        for ln in all_lanes:
            ln.stream.wait_event(ev0)
        pool = lanes[:E2E_LANES] if e2e else lanes
        for i in range(n_groups):
            ln = pool[i % len(pool)]
            if use_tail and i == n_groups - 1:
                ln = tail_lane
            sd = (first // G + i) % n_seed_groups
            with torch.cuda.stream(ln.stream):
                if e2e:
                    ln.stream.synchronize() if i >= len(pool) else None
                    ln.h_seeds.copy_(torch.from_numpy(host_seeds[sd][:ln.G]))
                    ln.d_seeds.copy_(ln.h_seeds, non_blocking=True)
                    step(ln)
                    ln.h_x.copy_(ln.x_view, non_blocking=True)
                    for l in range(L):
                        ln.h_ids[l].copy_(ln.ids[l], non_blocking=True)
                        ln.h_agg[l].copy_(ln.agg[l], non_blocking=True)
                else:
                    ln.d_seeds.copy_(dev_seeds[sd][:ln.G], non_blocking=True)
                    step(ln)
        for ln in all_lanes:
            main.wait_stream(ln.stream)
        ev1.record(main)
        torch.cuda.synchronize()
        dist.barrier()
        t = torch.tensor([ev0.elapsed_time(ev1)], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    run(-(-max(args.warmup, G * len(lanes)) // G) * G, 0, False)
    if tail_lane:
        run(tail, 0, False)
    clocks = Clocks(local)
    clocks.start()
    time.sleep(0.3)
    nv0 = nvlink_counters(local) if rank == 0 else None
    w0 = time.time()
    ms = run(args.steps, args.warmup, False)
    w1 = time.time()
    nv1 = nvlink_counters(local) if rank == 0 else None
    clk = clocks.stop(w0, w1)
    run(G * min(len(lanes), E2E_LANES), 0, True)
    if tail_lane:
        run(tail, 0, True)
    ms_e2e = run(args.steps, args.warmup, True)
    err = max(ln.sg.error() for ln in all_lanes) if peer else 0
    if err:
        raise SystemExit("bench: the peer exchange was poisoned (a bounded wait timed out): the timed numbers are invalid")
    # per-kernel breakdown + launch count on one lane (library-side CUDA events), serial, no graphs
    prof = {}
    ln = lanes[0]
    reps = 3
    lib.eu_ctx_profile(ln.ctx._h, 1)
    if replicated:
        lib.eu_ctx_profile(ln.sg.fctx._h, 1)
    l0 = lib.eu_launch_count()
    with torch.cuda.stream(ln.stream):
        for it in range(reps):
            ln.d_seeds.copy_(dev_seeds[it % n_seed_groups])
            raw_step(ln)
    ln.stream.synchronize()
    launches_per_group = (lib.eu_launch_count() - l0) / reps
    for hctx in [ln.ctx] + ([ln.sg.fctx] if replicated else []):
        buf = ctypes.create_string_buffer(1 << 16)
        lib.eu_ctx_profile_read(hctx._h, buf, len(buf))
        lib.eu_ctx_profile(hctx._h, 0)
        for line in buf.value.decode().strip().splitlines():
            nm, rows_, cnt_, ms_tot = line.rsplit(",", 3)
            prof["%s[rows=%s]" % (nm, rows_)] = round(float(ms_tot) / reps / G, 4)
    all_prof = [None] * world
    dist.all_gather_object(all_prof, prof)
    if os.environ.get("EU_BENCH_DEBUG") and rank == 0:
        for r_, p_ in enumerate(all_prof):
            print("rank %d profile: %s" % (r_, json.dumps(dict(sorted(p_.items(), key=lambda kv: -kv[1])))), file=sys.stderr)
    prof = {k: max(p_.get(k, 0.0) for p_ in all_prof) for k in prof}
    bts = step_bytes(B, counts, D)
    edges_step = bts["edges"] * world
    remote = (world - 1) / world
    # algorithmic NVLink bytes per rank per step: hop requests (id + src index) and replies (eng id, packed id, w, t);
    # feature requests + rows for the hop-0..L-1 nodes; fused aggregation = neighbor ids out, one partial row per
    # (remote owner, destination) back
    a2a_bytes = 0
    for l in range(L):
        a2a_bytes += remote * n[l] * (12 + 24 * counts[l])
    if peer and replicated:
        pass   # only the hop exchanges cross the link
    elif peer:
        a2a_bytes += remote * n_self * (12 + 4 * D)
        # valid (existing) fraction of the sampled ids of the last profiled group: placeholders are dropped before the
        # aggregation exchange, and an owner sends a partial row only for destinations it owns a neighbor of --
        # expected (world - 1) * (1 - (1 - v / world)^count) rows per destination for uniformly hashed ids
        try:
            vf = [float((lanes[0].ids[l] != -1).float().mean().item()) for l in range(L)]
        except Exception:
            vf = [1.0] * L
        for l in range(L):
            rows_per_dst = (world - 1) * (1.0 - (1.0 - vf[l] / world) ** counts[l])
            a2a_bytes += remote * vf[l] * n[l + 1] * 12 + rows_per_dst * n[l] * 4 * D
    else:
        a2a_bytes += remote * sum(n) * (12 + 4 * D)
    if rank == 0:
        traffic, traffic_src, link = None, None, None
        if nv0 and nv1:
            # measured on the wire: the driver's NVLink data counters of rank 0's GPU around the timed region (KiB granularity;
            # the peer exchange is the only NVLink user in that window)
            tx, rx = nv1[0] - nv0[0], nv1[1] - nv0[1]
            traffic = int((tx + rx) / args.steps)
            traffic_src = "nvidia-smi nvlink -gt d on rank 0's GPU, (tx + rx) delta over the timed region / steps"
            link = {"tx_bytes_per_step": int(tx / args.steps), "rx_bytes_per_step": int(rx / args.steps),
                    "tx_gbs": round(tx / (ms * 1e-3) / 1e9, 2), "rx_gbs": round(rx / (ms * 1e-3) / 1e9, 2),
                    "frac_of_770_gbs_per_direction": round(max(tx, rx) / (ms * 1e-3) / 1e9 / 770.0, 4)}
        out = {
            "metric": "sampled_edges_per_sec", "value": edges_step * args.steps / (ms * 1e-3), "unit": "edges/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64 ids / f32 weights+features (f64 CDF compare)", "data": "synthetic",
            "config": workload_config(args, counts, world),
            "arm": {"global_batch": B * world, "exchange": "peer-memory kernels (NVLink loads/stores, no NCCL)" if peer else "NCCL all_to_all",
                    "lanes_in_flight": n_lanes, "steps_per_launch_group": G, "cuda_graphs": use_graphs, "peer_wait_timeouts": err,
                    "aggregation": ("features replicated on every rank (%.1f GB): local k_feature / k_sage_mean" % (args.nodes * D * 4 / 1e9)) if replicated
                                   else ("fused at the owners (eu_sym_sage_mean: one partial row per owner and destination)" if peer else "materialised rows + scatter_mean"),
                    "features": "replicated" if replicated else "sharded with their rows",
                    "parallelism": "CSR sharded id %% %d, batches data-parallel" % world,
                    "hbm_gb_per_rank": round((graph.hbm_bytes + (feat_graph.hbm_bytes if feat_graph else 0)) / 1e9, 1)},
            "parity_gate": gate,
            "e2e": {"value": edges_step * args.steps / (ms_e2e * 1e-3), "unit": "edges/s", "h2d_bytes_per_step": 8 * B * world,
                    "d2h_bytes_per_step": world * (sum(8 * x for x in n[1:]) + 2 * sum(4 * n[l] * D for l in range(L))),
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(round(launches_per_group * (args.steps // G + (1 if tail else 0)))), "clocks": clk,
            "roofline": {"bound": "nvlink", "kernel": "exchange kernels (k_bucket_place / k_sym_reply_sample%s)" % ("" if replicated else " / k_sym_reply_sage / k_sym_reply_feature") if peer else "NCCL all-to-all",
                         "achieved": round(a2a_bytes / (ms / args.steps * 1e-3) / 1e9, 2), "peak": 770.0, "unit": "GB/s",
                         "frac": round(a2a_bytes / (ms / args.steps * 1e-3) / 1e9 / 770.0, 4), "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": "B200_PROFILING.md measured peer copy 770 GB/s per direction",
                         "algorithmic_bytes_per_step_per_rank": int(a2a_bytes), "nvlink_measured": link,
                         "note": "achieved = algorithmic exchange bytes per rank per step / whole step time (the exchange overlaps the local "
                                 "kernels of the other lanes and is not timed alone)"},
            "graph_build_s": round(t_graph, 2),
            "kernel_ms_per_step_single_lane": dict(sorted(prof.items(), key=lambda kv: -kv[1])),
        }
        if use_graphs:
            out["arm"]["launch"] = "one CUDA graph replay per launch group; gpu_launches counts this library's kernels inside the replays"
        if peer and replicated:
            # With the feature table replicated the exchange is ~2 % of a rank's bytes: a rank's step is bounded by the same local
            # HBM-bound kernels as at N=1.  Headline roofline = that kernel; the link figures move to roofline["nvlink"].
            try:
                vf = [float((lanes[0].ids[l] != -1).float().mean().item()) for l in range(L)]
            except Exception:
                vf = [1.0] * L
            peaks = {}
            try:
                peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            except Exception:
                pass
            peak = float(peaks.get("hbm_gbs", 6650.0))
            hbm_step = 0.0
            for l in range(L):
                c_ = counts[l]
                hbm_step += n[l] * c_ * 8 + vf[l] * n[l] * c_ * 4 * D + n[l] * 4 * D                      # k_sage_mean
                hbm_step += n[l] * 8 + (1.0 if l == 0 else vf[l - 1]) * n[l] * 4 * D + n[l] * 4 * D        # k_feature
                hbm_step += n[l] * 40 + vf[l] * n[l] * c_ * 48 + (1 - vf[l]) * n[l] * c_ * 16 + n[l] * 52  # k_sample + k_prepare (owner side)
            link_roof = out["roofline"]
            rows_dom = G * n[L - 1]
            dom_ms = prof.get("k_sage_mean[rows=%d]" % rows_dom)
            roof = {"bound": "hbm", "peak": peak, "unit": "GB/s", "traffic": None,
                    "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst)" if peaks else "fallback 6650 (B200_PROFILING.md)",
                    "valid_edge_fraction_per_hop": [round(v, 4) for v in vf]}
            if dom_ms:
                dom_bytes = rows_dom * counts[L - 1] * 8 + vf[L - 1] * rows_dom * counts[L - 1] * 4 * D + rows_dom * 4 * D
                ach = dom_bytes / (dom_ms * G * 1e-3) / 1e9
                roof.update({"kernel": "k_sage_mean over %d rows (largest share of a rank's step; timed alone on its SM share, max over ranks)" % rows_dom,
                             "achieved": round(ach, 1), "frac": round(ach / peak, 4), "algorithmic_bytes_per_launch": int(dom_bytes),
                             "kernel_ms": round(dom_ms * G, 5)})
            step_gbs = hbm_step / (ms / args.steps * 1e-3) / 1e9
            roof["step"] = {"algorithmic_bytes_per_step_per_rank": int(hbm_step + a2a_bytes), "achieved": round(step_gbs, 1),
                            "frac": round(step_gbs / peak, 4),
                            "how": "a rank's local algorithmic HBM bytes per step / timed ms_per_step (all lanes in flight, max over ranks)"}
            roof["nvlink"] = link_roof
            roof["traffic_nvlink_bytes_per_step"] = traffic
            out["roofline"] = roof
        emit(out)
    if peer:
        for ln in all_lanes:
            ln.sg.close()
    dist.destroy_process_group()


# ----------------------------------------------------------------------------- CPU arms
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def host_mem_budget():
    """bytes the CPU arms may hold at once: a quarter of what the container may use (cgroup limit when there is one, else
    MemAvailable), never more than 48 GB.  Every reference thread builds the whole minibatch in std::vectors (3 GB per thread
    at the headline config): unbounded, 128 threads would ask for ~400 GB and take the box down with them."""
    limit = None
    for path in ("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory/memory.limit_in_bytes"):
        try:
            v = open(path).read().strip()
            if v.isdigit() and int(v) < (1 << 60):
                limit = int(v)
                break
        except Exception:
            pass
    avail = None
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                avail = int(line.split()[1]) * 1024
    except Exception:
        pass
    cands = [x for x in (limit, avail) if x]
    base = min(cands) if cands else 32 << 30
    return int(min(base // 4, 48 << 30))


def cpu_threads_cap(args, counts, graph_bytes=0):
    """largest thread count whose per-thread minibatch buffers fit the memory budget (see host_mem_budget)"""
    rows = args.batch
    for c in counts:
        rows *= c
    per_thread = int(rows * max(args.dim, 1) * 4 * 2.6) + (64 << 20)   # widest hop: feature matrix + the api's nested vectors + means
    budget = max(host_mem_budget() - graph_bytes, 4 << 30)
    return max(1, min(host_cores(), budget // per_thread))


def cpu_graph(args):
    """The CPU arms' input: the same generator (oracle/rmat_gen.c restates euler_b200/csrc/graph.cu bit-exactly; nothing of
    the product is loaded), at the bench's size when the reference's in-memory graph can be built inside the time box, else
    down-scaled at constant mean degree -- which favours the CPU (its working set shrinks; the GPU arm keeps the full graph)."""
    from oracle import pyoracle as po
    nodes, edges = args.nodes, args.edges
    scale = 1.0
    if nodes > CPU_GRAPH_MAX_NODES:
        scale = CPU_GRAPH_MAX_NODES / nodes
        nodes, edges = CPU_GRAPH_MAX_NODES, int(edges * scale)
    t0 = time.time()
    ex = po.rmat_graph(nodes, edges, seed=GRAPH_SEED, feat_dim=args.dim, feat_seed=FEAT_SEED)
    use_ref = po.have_ref()
    if use_ref:
        # raw weights are needed by Node::Init; de-cumulate exactly as stored differences
        cum, ptr = ex["cum_w"], ex["grp_ptr"]
        w = np.diff(cum, prepend=np.float32(0)).astype(np.float32)
        first = ptr[:-1][np.diff(ptr) > 0]
        w[first] = cum[first]
        rg = po.RefGraph.build(ex["ids"], ex["node_type"], ex["node_w"], 1, ptr, ex["nbr"], w, 1, ex["feat"], sampler=False)
        og = None
    else:
        rg = None
        og = po.OracleGraph(ex["ids"], ex["node_type"], ex["node_w"], 1, ex["grp_ptr"], ex["nbr"], ex["cum_w"],
                            np.zeros(nodes, np.float32), ex["feat"])
    info = {"nodes": nodes, "edges": edges, "scale_vs_gpu_arm": scale, "build_s": round(time.time() - t0, 1),
            "note": "full size" if scale == 1.0 else "down-scaled on the CPU side only (same generator, same mean degree): the reference's "
                    "unordered_map<NodeID,Node*> graph of the full size does not build inside the bench's time box"}
    return rg, og, ex, nodes, info


class CpuStep:
    def __init__(self, args, counts, rg, og, nodes):
        from oracle import pyoracle as po
        self.po, self.rg, self.og, self.args, self.counts = po, rg, og, args, counts
        self.et = [[0]] * len(counts)
        self.seeds = np.stack([np.random.RandomState(1000 + i).randint(1, nodes + 1, size=args.batch) for i in range(64)]).astype(np.int64)

    def step(self, threads, iters):
        """(seconds, edges): every thread runs `iters` full steps (sample_fanout + dense features of every hop + neighbor means)"""
        po = self.po
        if self.rg is not None:
            return po.ref_bench_step(self.seeds, self.et, self.counts, self.args.dim, threads, iters)
        return po.oracle_bench_step(self.og, self.seeds, self.et, self.counts, self.args.dim, threads, iters)

    def fanout(self, threads, iters):
        """(seconds, edges): sampling only"""
        po = self.po
        if self.rg is not None:
            return self.rg.bench_fanout(self.seeds, self.et, self.counts, threads, iters)
        return self.og.bench_fanout(self.seeds, self.et, self.counts, threads, iters)

    def best_threads(self, cores):
        """the reference links jemalloc (CMakeLists.txt:13,41-43), absent here: with glibc malloc its
        vector<vector<vector<float>>> feature path scales badly, so sweep thread counts and keep the best.  The sweep never
        exceeds the memory-derived cap (cpu_threads_cap)."""
        cap = cpu_threads_cap(self.args, self.counts)
        self.thread_cap = cap
        cores = min(cores, cap)
        sweep, best = {}, (0.0, 1)
        for th in sorted({cores, max(1, cores // 2), max(1, cores // 4), min(cores, 16), min(cores, 8), 1}, reverse=True):
            self.step(th, 1)
            sec, edges = self.step(th, 1)
            sweep[str(th)] = edges / sec
            if edges / sec > best[0]:
                best = (edges / sec, th)
        return best[1], sweep


def cpu_sub_rates(cs, args, counts, th, iters):
    """sampling-only edges/s and aggregation-only GB/s (algorithmic bytes) of the CPU path at `th` threads"""
    bts = step_bytes(args.batch, counts, args.dim)
    cs.fanout(th, 1)
    f_sec, f_edges = cs.fanout(th, iters)
    s_sec, s_edges = cs.step(th, iters)
    agg_sec = max(s_sec - f_sec, 1e-9)
    batches = s_edges / bts["edges"]
    out = {"sampling_only_edges_per_s": f_edges / f_sec, "aggregation_only_gbs": (bts["agg"] + bts["self_feat"]) * batches / agg_sec / 1e9,
           "how": "%d threads x %d batches: sampling-only loop timed alone; aggregation = full-step time minus sampling-only time" % (th, iters)}
    cores = host_cores()
    if cores > th:    # the sampler alone needs little memory per thread: also time it on every host core (the north-star's 10x bar)
        cs.fanout(cores, 1)
        a_sec, a_edges = cs.fanout(cores, max(2, iters))
        out["sampling_only_all_cores"] = {"edges_per_s": a_edges / a_sec, "cores": cores}
    return out


def cpu_baseline(args, counts):
    """cpu_baseline leg: the reference's own sources (oracle/_ref, kind "reference") when the prebuilt
    shim travelled with the repo, else the C restatement (kind "port"); best thread count, bounded sample."""
    rg, og, ex, nodes, info = cpu_graph(args)
    cs = CpuStep(args, counts, rg, og, nodes)
    cores = host_cores()
    th, sweep = cs.best_threads(cores)
    sec1, _ = cs.step(th, 1)
    iters = max(1, min(50, int(args.cpu_seconds / max(sec1, 1e-3))))
    sec, edges = cs.step(th, iters)
    one_sec, one_edges = cs.step(1, 1)
    return {"value": edges / sec, "unit": "edges/s", "cores": th, "host_cores": cores, "thread_cap_from_memory_budget": cs.thread_cap,
            "kind": "reference" if rg is not None else "port",
            "sample": "best of a thread sweep: %d threads x %d batches of the same step (sample_fanout + dense features of every hop + "
                      "neighbor means), %.1f s" % (th, iters, sec),
            "one_thread_edges_per_s": one_edges / one_sec,
            "threads_sweep_edges_per_s": sweep, "sub_rates": cpu_sub_rates(cs, args, counts, th, max(1, iters // 2)), "cpu_graph": info}


# ----------------------------------------------------------------------------- config c3: node2vec walk
def walk_workload(args, L, n_gpus):
    return ("%s: synthetic power-law (R-MAT 0.57/0.19/0.19/0.05) graph %dM nodes/%dM edges, node2vec biased walk p=%g q=%g "
            "walk_len=%d batch=%d, %d GPU(s)" % (args.label, args.nodes // 10**6, args.edges // 10**6, args.p, args.q, L, args.batch, n_gpus))


def walk_config(args, L, n_gpus):
    return {"workload": walk_workload(args, L, n_gpus), "nodes": args.nodes, "edges": args.edges, "batch": args.batch, "walk_len": L,
            "p": args.p, "q": args.q, "rng": args.rng,
            "l2_policy": "inputs larger than L2 (graph >> 126 MB, fresh random start nodes every step)"}


def run_walk(args):
    """A step = one random_walk op call: `batch` walkers x walk_len node2vec steps (tf_euler/kernels/random_walk_op.cc:83-289).
    metric = walker-steps/s.  Parity gate: a smaller batch bit-exact against the oracle's restatement of the reference walk."""
    import torch
    import euler_b200 as eb
    from euler_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    lib = _lib.load()
    L, B = int(args.fanout), args.batch
    et = np.zeros((L, 1), np.int32)
    t0 = time.time()
    graph = eb.Graph.rmat(args.nodes, args.edges, seed=GRAPH_SEED, feat_dim=0, device=local)
    torch.cuda.synchronize()
    t_graph = time.time() - t0
    ex = graph.export(with_feat=False)
    deg = torch.from_numpy(np.diff(ex["grp_ptr"]).astype(np.int64)).cuda()
    gate = {"passed": None, "skipped": "--no-gate"}
    if not args.no_gate and args.rng == "minstd":
        from oracle import pyoracle as po
        tg = time.time()
        og = po.OracleGraph(ex["ids"], ex["node_type"], ex["node_w"], 1, ex["grp_ptr"], ex["nbr"], ex["cum_w"], np.zeros(len(ex["ids"]), np.float32))
        Bg, Lg = 1024, 12
        gs = np.random.RandomState(5).randint(1, args.nodes + 1, size=Bg).astype(np.int64)
        gs[:3] = [0, -1, args.nodes + 5]
        ctx = eb.Context(graph, "minstd", 4242)
        d_s = torch.from_numpy(gs).cuda()
        d_o = torch.empty((Bg, Lg + 1), dtype=torch.int64, device="cuda")
        _lib.check(lib.eu_random_walk(ctx._h, d_s.data_ptr(), Bg, et.ctypes.data, 1, Lg, args.p, args.q, -1, d_o.data_ptr()))
        ctx.sync()
        po.seed(4242)
        want = og.op_random_walk(gs, et[:Lg], args.p, args.q, -1)
        got = d_o.cpu().numpy()
        if not np.array_equal(got, want):
            bad = np.argwhere(got != want)
            raise SystemExit("PARITY GATE FAILED: node2vec walk differs from the oracle at %d of %d positions (first: walker %d step %d got %d want %d)"
                             % (len(bad), want.size, bad[0][0], bad[0][1], got[bad[0][0], bad[0][1]], want[bad[0][0], bad[0][1]]))
        gate = {"passed": True, "walkers": Bg, "steps": Lg, "values_compared": int(want.size), "seconds": round(time.time() - tg, 2),
                "what": "eu_random_walk (exact-RNG mode) vs oracle/euler_oracle.c eo_op_random_walk on the exported CSR of the bench graph, bit-exact"}
        ctx.close()
        del og

    class WLane:
        pass
    def make_lanes(rng, count):
        made = []
        for i in range(max(1, count)):
            ln = WLane()
            ln.stream = torch.cuda.Stream()
            ln.ctx = eb.Context(graph, rng, 777 + i, ln.stream.cuda_stream)
            ln.d_seeds = torch.empty(B, dtype=torch.int64, device="cuda")
            ln.out = torch.empty((B, L + 1), dtype=torch.int64, device="cuda")
            ln.h_seeds = torch.empty(B, dtype=torch.int64).pin_memory()
            ln.h_out = torch.empty((B, L + 1), dtype=torch.int64).pin_memory()
            made.append(ln)
        return made
    lanes = make_lanes(args.rng, args.lanes)
    n_sb = max(args.warmup + args.steps, 8)
    host_seeds = np.stack([np.random.RandomState(3000 + i).randint(1, args.nodes + 1, size=B) for i in range(n_sb)]).astype(np.int64)
    dev_seeds = torch.from_numpy(host_seeds).cuda()

    def raw(ln):
        rc = lib.eu_random_walk(ln.ctx._h, ln.d_seeds.data_ptr(), B, et.ctypes.data, 1, L, args.p, args.q, -1, ln.out.data_ptr())
        if rc:
            raise RuntimeError(lib.eu_last_error().decode())
    use_graphs = not args.no_graphs

    def prime(made):
        for ln in made:
            with torch.cuda.stream(ln.stream):
                ln.d_seeds.copy_(dev_seeds[0])
                raw(ln)
            ln.stream.synchronize()
            if use_graphs:
                l_before = lib.eu_launch_count()
                ln.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(ln.graph, stream=ln.stream):
                    raw(ln)
                ln.launches = lib.eu_launch_count() - l_before
    prime(lanes)
    main = torch.cuda.current_stream()

    def run(n_steps, first, mode, lanes=lanes):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record(main)
        for ln in lanes:
            ln.stream.wait_event(ev0)
        if mode == "host":
            def worker(k, ln):
                for i in range(k, n_steps, len(lanes)):
                    ln.h_seeds.copy_(torch.from_numpy(host_seeds[(first + i) % n_sb]))
                    rc = lib.eu_random_walk_host(ln.ctx._h, ln.h_seeds.data_ptr(), B, et.ctypes.data, 1, L, args.p, args.q, -1, ln.h_out.data_ptr())
                    if rc:
                        raise RuntimeError(lib.eu_last_error().decode())
            ths = [threading.Thread(target=worker, args=(k, ln)) for k, ln in enumerate(lanes)]
            for t in ths:
                t.start()
            for t in ths:
                t.join()
        else:
            for i in range(n_steps):
                ln = lanes[i % len(lanes)]
                with torch.cuda.stream(ln.stream):
                    ln.d_seeds.copy_(dev_seeds[(first + i) % n_sb], non_blocking=True)
                    ln.graph.replay() if use_graphs else raw(ln)
        for ln in lanes:
            main.wait_stream(ln.stream)
        ev1.record(main)
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1)
    run(max(args.warmup, 3), 0, "dev")
    clocks = Clocks(local)
    clocks.start()
    time.sleep(0.3)
    w0 = time.time()
    ms = run(args.steps, args.warmup, "dev")
    w1 = time.time()
    clk = clocks.stop(w0, w1)
    run(len(lanes), 0, "host")     # every lane's first *_host call grows its staging buffers: not inside the timed region
    ms_host = run(args.steps, args.warmup, "host")
    # measured sum of degrees: per walker-step 12 * deg(cur) + 8 * deg(prev) + 32 bytes (SURVEY.md section 8d)
    ln = lanes[0]
    with torch.cuda.stream(ln.stream):
        ln.d_seeds.copy_(dev_seeds[1])
        raw(ln)
    ln.stream.synchronize()
    o = ln.out
    row = (o - 1).clamp_(0, args.nodes - 1)
    dcur = torch.where(o > 0, deg[row], torch.zeros_like(o))
    live = (dcur[:, :L] > 0)
    dprev = torch.cat([torch.zeros_like(dcur[:, :1]), dcur[:, :L - 1]], dim=1)
    sum_cur, sum_prev = int(dcur[:, :L].sum().item()), int((dprev * live).sum().item())
    alg_bytes = 12 * sum_cur + 8 * sum_prev + 32 * B * L
    # per-kernel times of one batch (library-side events)
    lib.eu_ctx_profile(ln.ctx._h, 1)
    with torch.cuda.stream(ln.stream):
        raw(ln)
    buf = ctypes.create_string_buffer(1 << 16)
    lib.eu_ctx_profile_read(ln.ctx._h, buf, len(buf))
    lib.eu_ctx_profile(ln.ctx._h, 0)
    prof = {}
    for line in buf.value.decode().strip().splitlines():
        nm, rows_, cnt_, ms_tot = line.rsplit(",", 3)
        prof[nm] = round(float(ms_tot), 4)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    ws = B * L
    value = ws * args.steps / (ms * 1e-3)
    ach = alg_bytes * args.steps / (ms * 1e-3) / 1e9
    out = {"metric": "walker_steps_per_sec", "value": value, "unit": "walker-steps/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "u64 ids / f32 weights (sequential f32 prefix, f64 compare)", "data": "synthetic", "config": walk_config(args, L, 1),
           "arm": {"lanes_in_flight": len(lanes), "cuda_graphs": use_graphs, "graph_hbm_gb": round(graph.hbm_bytes / 1e9, 1),
                   "mode": "exact (bit-exact with the reference's serial engine stream and sequential f32 prefix)" if args.rng == "minstd"
                           else "philox throughput mode (rejection-sampled steps, k_walk_fast)"},
           "parity_gate": gate,
           "e2e": {"value": ws * args.steps / (ms_host * 1e-3), "unit": "walker-steps/s", "h2d_bytes_per_step": 8 * B, "d2h_bytes_per_step": 8 * B * (L + 1),
                   "ms_per_step": ms_host / args.steps, "api": "eu_random_walk_host (HOST buffers in and out), one host thread per lane"},
           "gpu_launches": int(sum(getattr(x, "launches", 0) for x in lanes) / len(lanes) * args.steps) if use_graphs else None,
           "clocks": clk,
           "roofline": {"bound": "hbm", "kernel": "k_walk_weights + k_walk_prefix (whole op: the walk is one chain of dependent steps)",
                        "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4), "traffic": None,
                        "algorithmic_bytes_per_batch": int(alg_bytes), "sum_deg_cur": sum_cur, "sum_deg_prev": sum_prev,
                        "mean_deg_cur_per_live_step": round(sum_cur / max(int(live.sum().item()), 1), 1),
                        "note": "achieved = (12 deg(cur) + 8 deg(prev) + 32) bytes summed over the walker-steps of a batch / batch time; hub "
                                "rows are L2-resident, so this is an algorithmic rate"},
           "kernel_ms_per_batch_single_lane": dict(sorted(prof.items(), key=lambda kv: -kv[1])),
           "graph_build_s": round(t_graph, 2)}
    if args.rng == "minstd":
        # the throughput engine beside the exact one (SURVEY section 7: "fast mode ... report both"): EU_RNG_PHILOX takes a node2vec
        # step by rejection (propose from the stored CDF, accept with bias / max bias): same distribution, O(log deg) per step
        flanes = make_lanes("philox", max(args.lanes, 16))
        prime(flanes)
        fsteps = max(args.steps, 4 * len(flanes))
        run(len(flanes), 0, "dev", flanes)
        ms_f = run(fsteps, 0, "dev", flanes)
        out["fast_mode"] = {"value": ws * fsteps / (ms_f * 1e-3), "unit": "walker-steps/s", "ms_per_step": ms_f / fsteps, "steps": fsteps,
                            "lanes_in_flight": len(flanes), "rng": "philox",
                            "what": "k_walk_fast: rejection-sampled node2vec steps (distribution-exact, not stream-exact), one thread per "
                                    "walker for all %d steps; checked by a chi-square test against the exact transition weights" % L}
    if not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_walk_baseline(args, L, ex)
    emit(out)


def cpu_walk_graph(args, ex):
    from oracle import pyoracle as po
    if ex is None:
        ex = po.rmat_graph(args.nodes, args.edges, seed=GRAPH_SEED, feat_dim=0)
    if po.have_ref():
        cum, ptr = ex["cum_w"], ex["grp_ptr"]
        w = np.diff(cum, prepend=np.float32(0)).astype(np.float32)
        first = ptr[:-1][np.diff(ptr) > 0]
        w[first] = cum[first]
        return po.RefGraph.build(ex["ids"], ex["node_type"], ex["node_w"], 1, ptr, ex["nbr"], w, 1, None, sampler=False), None
    return None, po.OracleGraph(ex["ids"], ex["node_type"], ex["node_w"], 1, ex["grp_ptr"], ex["nbr"], ex["cum_w"], np.zeros(len(ex["ids"]), np.float32))


def cpu_walk_time(args, L, rg, og, threads, walkers):
    """every thread walks `walkers` walkers for L steps (its own engine); returns (seconds, walker-steps)"""
    et = np.zeros((L, 1), np.int32)
    g = rg if rg is not None else og

    def worker(k):
        sd = np.random.RandomState(9000 + k).randint(1, args.nodes + 1, size=walkers).astype(np.int64)
        g.op_random_walk(sd, et, args.p, args.q, -1)
    ths = [threading.Thread(target=worker, args=(k,)) for k in range(threads)]
    t0 = time.time()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    return time.time() - t0, threads * walkers * L


def cpu_walk_baseline(args, L, ex):
    rg, og = cpu_walk_graph(args, ex)
    cores = host_cores()
    th = min(cores, 32) if rg is not None else 1     # the C restatement walks on one global engine: one thread; 32 bounds the
    #                                                   per-thread neighbor-list vectors (hub rows) to a few GB in total
    sec, n = cpu_walk_time(args, L, rg, og, th, 8)
    walkers = max(8, min(256, int(8 * args.cpu_seconds / max(sec, 1e-3))))
    sec, n = cpu_walk_time(args, L, rg, og, th, walkers)
    one_sec, one_n = cpu_walk_time(args, L, rg, og, 1, max(8, walkers // 4))
    return {"value": n / sec, "unit": "walker-steps/s", "cores": th, "host_cores": cores, "kind": "reference" if rg is not None else "port",
            "one_thread_walker_steps_per_s": one_n / one_sec,
            "sample": "%d host threads x %d walkers x %d steps of the reference's node2vec step (ref_shim restatement of random_walk_op.cc:83-168 "
                      "over the reference's own GetFullNeighbor), %.1f s" % (th, walkers, L, sec)}


def run_walk_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    L = int(args.fanout)
    rg, og = cpu_walk_graph(args, None)
    cores = host_cores()
    th = min(cores, 32) if rg is not None else 1
    walkers = 16
    sec1, _ = cpu_walk_time(args, L, rg, og, th, walkers)
    steps = max(1, min(args.steps, int(120.0 / max(sec1, 1e-3)) - args.warmup))
    warm = args.warmup if steps == args.steps else min(args.warmup, 1)
    for _ in range(warm):
        cpu_walk_time(args, L, rg, og, th, walkers)
    tn, ts = 0, 0.0
    for _ in range(steps):
        sec, n = cpu_walk_time(args, L, rg, og, th, walkers)
        tn += n
        ts += sec
    v = tn / ts
    emit({"impl": "reference", "metric": "walker_steps_per_sec", "value": v, "unit": "walker-steps/s", "n_gpus": args.gpus, "steps": steps,
          "warmup": warm, "ms_per_step": 1e3 * ts / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
          "dtype": "u64 ids / f32 weights (sequential f32 prefix, f64 compare)", "data": "synthetic", "config": walk_config(args, L, args.gpus),
          "arm": {"step": "one bounded sample = %d host threads x %d walkers x %d steps" % (th, walkers, L), "host_cores": cores},
          "cpu_baseline": {"value": v, "unit": "walker-steps/s", "cores": th, "kind": "reference" if rg is not None else "port",
                           "sample": "%d steps of %d threads x %d walkers" % (steps, th, walkers)},
          "e2e": {"value": v, "unit": "walker-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0})


# ----------------------------------------------------------------------------- config c5: per-relation sampling + scatter_add
def c5_config(args, count, n_gpus):
    return {"workload": "%s: synthetic heterogeneous R-MAT graph %dM nodes/%dM edges, %d node types / %d edge types, per-edge-type "
                        "sample_neighbor count=%d batch=%d + dense features (dim %d) summed per relation (scatter_add), %d GPU(s)"
                        % (args.label, args.nodes // 10**6, args.edges // 10**6, C5_NTYPES, C5_ETYPES, count, args.batch, args.dim, n_gpus),
            "nodes": args.nodes, "edges": args.edges, "batch": args.batch, "count": count, "feat_dim": args.dim, "edge_types": C5_ETYPES,
            "rng": args.rng, "l2_policy": "inputs larger than L2 (graph >> 126 MB, fresh random seeds every step)"}


def run_c5(args):
    """A step = for every edge type t: sample_neighbor(seeds, [t], count) and the per-relation feature sum of the sampled
    neighbors (get_dense_feature + scatter_add over the fixed-fanout block, fused).  metric = sampled edges/s (T * B * count / step)."""
    import torch
    import euler_b200 as eb
    from euler_b200 import _lib
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    lib = _lib.load()
    T, count, B, D = C5_ETYPES, int(args.fanout), args.batch, args.dim
    t0 = time.time()
    graph = eb.Graph.rmat_hetero(args.nodes, args.edges, T, C5_NTYPES, seed=C5_SEED, feat_dim=D, feat_seed=FEAT_SEED, device=local)
    torch.cuda.synchronize()
    t_graph = time.time() - t0
    G = max(1, min(8, -(-args.steps // max(args.lanes, 1))))
    cs = np.asarray([count], np.int32)
    P1 = ctypes.c_void_p * 1

    class CL:
        pass
    lanes = []
    for i in range(max(1, min(args.lanes, args.steps // G if args.steps >= G else 1))):
        ln = CL()
        ln.stream = torch.cuda.Stream()
        ln.ctx = eb.Context(graph, args.rng, 555 + i, ln.stream.cuda_stream)
        ln.seeds_of = [9000 + 100 * i + b for b in range(G)]
        ln.ctx.set_engines(G, ln.seeds_of)
        ln.ctx.reserve(G * B * count)
        ln.d_seeds = torch.empty(G * B, dtype=torch.int64, device="cuda")
        ln.ids = [torch.empty(G * B * count, dtype=torch.int64, device="cuda") for _ in range(T)]
        ln.w = [torch.empty(G * B * count, dtype=torch.float32, device="cuda") for _ in range(T)]
        ln.ty = [torch.empty(G * B * count, dtype=torch.int32, device="cuda") for _ in range(T)]
        ln.agg = [torch.empty((G * B, D), dtype=torch.float32, device="cuda") for _ in range(T)]
        lanes.append(ln)

    def raw(ln):
        rc = 0
        for t in range(T):
            et = np.asarray([[t]], np.int32)
            rc |= lib.eu_sample_fanout_batched(ln.ctx._h, ln.d_seeds.data_ptr(), G, B, et.ctypes.data, 1, cs.ctypes.data, 1, -1,
                                               P1(ln.ids[t].data_ptr()), P1(ln.w[t].data_ptr()), P1(ln.ty[t].data_ptr()))
            rc |= lib.eu_sage_add_aggregate(ln.ctx._h, ln.ids[t].data_ptr(), G * B, count, D, ln.agg[t].data_ptr())
        if rc:
            raise RuntimeError(lib.eu_last_error().decode())
    n_sb = max(-(-(args.warmup + args.steps) // G), 8)
    host_seeds = np.stack([np.random.RandomState(7000 + i).randint(1, args.nodes + 1, size=G * B) for i in range(n_sb)]).astype(np.int64)
    dev_seeds = torch.from_numpy(host_seeds).cuda()
    gate = {"passed": None, "skipped": "--no-gate"}
    if not args.no_gate and args.rng == "minstd":
        from oracle import pyoracle as po
        tg = time.time()
        ex = graph.export(with_feat=False)
        og = po.OracleGraph(ex["ids"], ex["node_type"], ex["node_w"], T, ex["grp_ptr"], ex["nbr"], ex["cum_w"], ex["grp_cum"])
        ln = lanes[0]
        ln.ctx.set_engines(G, ln.seeds_of)
        with torch.cuda.stream(ln.stream):
            ln.d_seeds.copy_(dev_seeds[0])
            raw(ln)
        ln.stream.synchronize()
        # the engines run relation after relation: batch b's engine serves type 0, then type 1, ... of batch b
        for b in range(G):
            po.seed(ln.seeds_of[b])
            sd = host_seeds[0][b * B:(b + 1) * B]
            for t in range(T):
                o_ids, o_w, o_t = og.op_sample_neighbor(sd, [t], count, -1)
                sl = slice(b * B * count, (b + 1) * B * count)
                for nm, got, want in (("ids", ln.ids[t], o_ids), ("weights", ln.w[t], o_w), ("types", ln.ty[t], o_t)):
                    if not np.array_equal(got[sl].cpu().numpy(), want.reshape(-1)):
                        raise SystemExit("PARITY GATE FAILED: %s of relation %d, batch %d differ from the oracle" % (nm, t, b))
                if b == 0:
                    feat = po.rmat_feat_rows(o_ids.reshape(-1), args.nodes, D, FEAT_SEED)
                    want = po.scatter_add(feat, np.repeat(np.arange(B, dtype=np.int32), count), B)
                    if not np.array_equal(ln.agg[t][:B].cpu().numpy(), want):
                        raise SystemExit("PARITY GATE FAILED: relation %d feature sums differ from the oracle's scatter_add" % t)
        ln.ctx.set_engines(G, ln.seeds_of)
        gate = {"passed": True, "batches": G, "relations": T, "seconds": round(time.time() - tg, 2),
                "what": "per-relation sample_neighbor of %d batches bit-exact vs the oracle on the exported CSR; per-relation feature sums of "
                        "batch 0 bit-exact vs oracle scatter_add over oracle/rmat_gen.c rows" % G}
        del og, ex
    use_graphs = not args.no_graphs
    for ln in lanes:
        with torch.cuda.stream(ln.stream):
            ln.d_seeds.copy_(dev_seeds[0])
            raw(ln)
        ln.stream.synchronize()
        if use_graphs:
            l0 = lib.eu_launch_count()
            ln.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(ln.graph, stream=ln.stream):
                raw(ln)
            ln.launches = lib.eu_launch_count() - l0
    main = torch.cuda.current_stream()

    def run(n_steps, first):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record(main)
        for ln in lanes:
            ln.stream.wait_event(ev0)
        for i in range(-(-n_steps // G)):
            ln = lanes[i % len(lanes)]
            with torch.cuda.stream(ln.stream):
                ln.d_seeds.copy_(dev_seeds[(first // G + i) % n_sb], non_blocking=True)
                ln.graph.replay() if use_graphs else raw(ln)
        for ln in lanes:
            main.wait_stream(ln.stream)
        ev1.record(main)
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1)
    steps = -(-args.steps // G) * G
    run(max(args.warmup, G), 0)
    clocks = Clocks(local)
    clocks.start()
    time.sleep(0.3)
    w0 = time.time()
    ms = run(steps, args.warmup)
    w1 = time.time()
    clk = clocks.stop(w0, w1)
    edges = T * B * count
    valid = float(np.mean([(lanes[0].ids[t] != -1).float().mean().item() for t in range(T)]))
    agg_bytes = T * (B * count * 8 + valid * B * count * 4 * D + B * 4 * D)
    out = {"metric": "sampled_edges_per_sec", "value": edges * steps / (ms * 1e-3), "unit": "edges/s", "n_gpus": 1, "steps": steps,
           "warmup": args.warmup, "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "u64 ids / f32 weights+features (f64 CDF compare)", "data": "synthetic", "config": c5_config(args, count, 1),
           "arm": {"lanes_in_flight": len(lanes), "steps_per_launch_group": G, "cuda_graphs": use_graphs, "graph_hbm_gb": round(graph.hbm_bytes / 1e9, 1)},
           "parity_gate": gate, "agg_feat_gbs": agg_bytes * steps / (ms * 1e-3) / 1e9, "valid_edge_fraction": round(valid, 4),
           "gpu_launches": int(sum(getattr(x, "launches", 0) for x in lanes) / len(lanes) * (steps // G)) if use_graphs else None,
           "clocks": clk, "graph_build_s": round(t_graph, 2)}
    emit(out)


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the same step on the host cores.  Loads nothing of the
    product: the input graph comes from oracle/rmat_gen.c."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    counts = [int(x) for x in args.fanout.split(",")]
    rg, og, ex, nodes, info = cpu_graph(args)
    cs = CpuStep(args, counts, rg, og, nodes)
    cores = host_cores()
    # untimed: pick the thread count the reference runs fastest with on this host -- its best case is the baseline
    th, sweep = cs.best_threads(cores)
    # a "step" of this arm = one bounded sample: every thread runs PER_STEP batches back to back (its first batch after a
    # thread start pays the allocator warm-up; a single batch per step would understate the reference)
    PER_STEP = 2
    sec1, _ = cs.step(th, PER_STEP)
    budget = 150.0                                    # seconds for warm-up + timed steps
    steps = max(1, min(args.steps, int(budget / max(sec1, 1e-3)) - args.warmup))
    warm = args.warmup if steps == args.steps else min(args.warmup, 1)
    for _ in range(warm):
        cs.step(th, PER_STEP)
    t_edges, t_sec = 0, 0.0
    for _ in range(steps):
        sec, edges = cs.step(th, PER_STEP)
        t_edges += edges
        t_sec += sec
    v = t_edges / t_sec
    sub = cpu_sub_rates(cs, args, counts, th, PER_STEP)
    bts = step_bytes(args.batch, counts, args.dim)
    out = {"impl": "reference", "metric": "sampled_edges_per_sec", "value": v, "unit": "edges/s",
           "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": 1e3 * t_sec / steps,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 ids / f32 weights+features (f64 CDF compare)",
           "data": "synthetic", "config": workload_config(args, counts, args.gpus),
           "arm": {"step": "one bounded sample = %d host threads x %d batches each" % (th, PER_STEP), "cpu_graph": info,
                   "threads_sweep_edges_per_s": sweep, "host_cores": cores, "thread_cap_from_memory_budget": cs.thread_cap},
           "agg_feat_gbs": (bts["agg"] + bts["self_feat"]) * (t_edges / bts["edges"]) / t_sec / 1e9,
           "sub_rates": sub,
           "cpu_baseline": {"value": v, "unit": "edges/s", "cores": th, "kind": "reference" if rg is not None else "port",
                            "sample": "%d steps of %d threads x %d batches" % (steps, th, PER_STEP)},
           "e2e": {"value": v, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    emit(out)


_REAL_STDOUT = None


def emit(out):
    """the ONE JSON line goes to the process's real stdout; everything else any library printed went to stderr"""
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(out) + "\n").encode())


if __name__ == "__main__":
    # libraries (NCCL's version banner, torchrun notices) print to fd 1: keep stdout for the JSON line alone
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    a = parse()
    if a.config == "c3":
        run_walk_reference(a) if a.impl == "reference" else run_walk(a)
    elif a.config == "c5" and a.impl == "ours":
        run_c5(a)
    elif a.config == "c5":
        emit({"impl": "reference", "unavailable": "config c5 is a secondary (extras) line: its CPU arm is not wired; the headline, c2 and c3 have one"})
    elif a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
