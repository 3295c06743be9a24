"""Host-side logic of bench.py that the driver depends on (no GPU): defaults, launch-group choice, identical workload strings in
both arms, and the memory cap of the CPU arms (an uncapped thread sweep took the GPU box down twice in round 2)."""
import importlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _parse(argv):
    bench = importlib.import_module("bench")
    old = sys.argv
    sys.argv = ["bench.py"] + argv
    try:
        return bench, bench.parse()
    finally:
        sys.argv = old


def test_defaults_are_the_north_star_headline():
    bench, a = _parse([])
    assert (a.gpus, a.impl, a.config) == (1, "ours", "c4")
    assert (a.nodes, a.edges, a.batch, a.fanout, a.dim) == (100_000_000, 1_000_000_000, 8192, "15,10", 256)
    assert a.warmup >= 3 and a.steps >= 1 and a.label != "custom"


def test_driver_run_keeps_every_lane_busy():
    bench, a = _parse(["--steps", "20", "--warmup", "5"])
    counts = [int(x) for x in a.fanout.split(",")]
    G = bench.auto_group(a, counts)
    assert G == 3                                      # ceil(20 / 8 lanes), under the 5M-row budget of a launch group
    assert G * a.batch * counts[0] * counts[1] <= 5_000_000
    assert -(-a.steps // G) >= a.lanes - 1             # 6 full groups + a tail: 7 of 8 lanes in flight
    bench, c2 = _parse(["--config", "c2", "--steps", "64", "--warmup", "16"])
    assert bench.auto_group(c2, [25, 10]) == 16


def test_both_arms_print_the_same_config():
    bench, ours = _parse(["--steps", "20", "--warmup", "5"])
    _, ref = _parse(["--impl", "reference", "--steps", "20", "--warmup", "5"])
    counts = [15, 10]
    for n in (1, 2, 8):
        assert bench.workload_config(ours, counts, n) == bench.workload_config(ref, counts, n)
    assert (ours.steps, ours.warmup) == (ref.steps, ref.warmup)


def test_cpu_arm_memory_cap():
    bench, a = _parse([])
    assert 0 < bench.host_mem_budget() <= 48 << 30
    cap = bench.cpu_threads_cap(a, [15, 10])
    rows = a.batch * 15 * 10
    assert 1 <= cap <= bench.host_cores()
    assert cap * rows * a.dim * 4 * 2.6 <= 48 << 30    # the threads' minibatch buffers fit the budget


def test_dump_outputs_are_the_last_batch_within_budget_and_repeat(tmp_path, monkeypatch):
    """--dump-outputs: the last batch of the lane's launch group, as float32 / float64 files within the byte budget; arrays
    that do not fit keep the same seeded rows on every run (and equal-length arrays the same rows)"""
    import numpy as np
    import torch
    bench, _ = _parse([])
    budget = 80_000
    monkeypatch.setattr(bench, "DUMP_BYTES", budget)
    B, counts, D, G = 64, [5, 4], 32, 3

    class Lane:
        pass
    ln = Lane()
    ln.G, ln.n = G, [G * B, G * B * 5, G * B * 20]
    torch.manual_seed(0)
    ln.ids = [torch.randint(-1, 10 ** 8, (n,), dtype=torch.int64) for n in ln.n[1:]]
    ln.w = [torch.rand(n) for n in ln.n[1:]]
    ln.ty = [torch.randint(0, 3, (n,), dtype=torch.int32) for n in ln.n[1:]]
    ln.x = [torch.rand(ln.n[l], D) for l in range(2)]
    ln.agg = [torch.rand(ln.n[l], D) for l in range(2)]
    out = bench.last_step_outputs(ln, counts)
    assert np.array_equal(out["ids_hop2"], ln.ids[1][-B * 20:].numpy())
    assert np.array_equal(out["features_hop0"], ln.x[0][-B:].numpy())
    assert np.array_equal(out["neighbor_mean_hop1"], ln.agg[1][-B * 5:].numpy())
    a = bench.dump_outputs(str(tmp_path / "a"), out)
    assert a == bench.dump_outputs(str(tmp_path / "b"), out)
    total = 0
    for name in a:
        x = np.load(tmp_path / "a" / (name + ".npy"))
        assert x.dtype in (np.float32, np.float64) and np.array_equal(x, np.load(tmp_path / "b" / (name + ".npy")))
        total += x.nbytes
    assert total <= budget
    assert np.array_equal(np.load(tmp_path / "a" / "ids_hop2.npy").astype(np.int64), out["ids_hop2"])   # whole and exact
    rows = np.load(tmp_path / "a" / "features_hop1_rows.npy")
    assert 0 < len(rows) < B * 5 and np.array_equal(rows, np.load(tmp_path / "a" / "neighbor_mean_hop1_rows.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "features_hop1.npy"), out["features_hop1"][rows.astype(np.int64)])
