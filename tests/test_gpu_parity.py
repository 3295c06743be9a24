"""GPU parity tests (run on the B200 box): the CUDA path, called through the C ABI / the Python mirror
of tf_euler's op API, against (a) golden vectors produced by the reference itself, (b) the pinned
CPU oracle on fresh seeded inputs, (c) size-independent properties at large sizes.
Integer / id / index outputs and sampled weights: bit-exact.  Float aggregations: bit-exact on the
sorted-index path, 1e-5 relative (north_star tolerance) on the unsorted atomic path."""
import ctypes as C

import numpy as np
import pytest
import torch

import cases
import graphs
from golden import make_golden as mg
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu
RTOL = 1e-5  # BASELINE.json north_star: "within 1e-5 relative for float aggregations"


@pytest.fixture(autouse=True)
def _sync_after():
    yield
    torch.cuda.synchronize()


# ------------------------------------------------------------------ golden replays (reference outputs)
def test_tiny_golden_from_csr():
    g = graphs.load_tiny_csr()
    cases.replay_tiny(cases.CudaBackend(g, g["map_order"]))


def test_tiny_loaded_from_reference_dat_files(tiny_dir):
    import euler_b200
    gr = euler_b200.Graph.load(tiny_dir)
    z = graphs.load_tiny_csr()
    ex = gr.export()
    # rows come in file order (partition 0: ids 2,4,6; partition 1: 1,3,5); compare node by node
    assert sorted(ex["ids"].tolist()) == z["ids"].tolist()
    T = z["T"]
    for r, i in enumerate(ex["ids"]):
        zr = int(np.searchsorted(z["ids"], i))
        assert ex["node_type"][r] == z["node_type"][zr] and ex["node_w"][r] == z["node_w"][zr]
        for t in range(T):
            b, e = ex["grp_ptr"][r * T + t], ex["grp_ptr"][r * T + t + 1]
            zb, ze = z["grp_ptr"][zr * T + t], z["grp_ptr"][zr * T + t + 1]
            assert np.array_equal(ex["nbr"][b:e], z["nbr"][zb:ze]) and np.array_equal(ex["cum_w"][b:e], z["cum_w"][zb:ze])
            assert ex["grp_cum"][r * T + t] == z["grp_cum"][zr * T + t]
        assert np.array_equal(ex["feat"][r], z["feat"][zr])
    # meta: names resolve like type_ops.py (SURVEY Appendix A-11: node "1"->0, "0"->1; edge "0"->0, "1"->1)
    assert gr.node_type_id("1") == 0 and gr.node_type_id("0") == 1
    assert gr.edge_type_id("0") == 0 and gr.edge_type_id("1") == 1
    assert gr.dense_feature_id("f3") == 0 and gr.dense_feature_id("f4") == 1 and gr.dense_feature_dim(1) == 3
    euler_b200.set_graph(gr)
    f3, f4 = euler_b200.get_dense_feature([1, 9, 4], ["f3", "f4"], [2, 3])
    cases.eq(f4.cpu().numpy(), cases.golden()["tiny_feat_f4"], "f4")
    assert np.allclose(f3.cpu().numpy()[0], [1.1, 1.2])
    # config C1: SampleNeighbor fanout=[10] batch=128 on the tools/test_data graph, fixed seed
    og = graphs.oracle_graph(z)
    seeds = np.random.RandomState(0).randint(0, 9, size=128).astype(np.int64)
    euler_b200.seed(2024)
    po.seed(2024)
    got = [x.cpu().numpy() for x in euler_b200.sample_neighbor(seeds, ["0", "1"], 10)]
    for a, b in zip(got, og.op_sample_neighbor(seeds, [0, 1], 10)):
        cases.eq(a, b, "C1 sample_neighbor")


@pytest.mark.parametrize("name", sorted(cases.SYNTH))
@pytest.mark.parametrize("raw", [False, True])
def test_synth_golden(name, raw):
    g = graphs.random_graph(**cases.SYNTH[name])
    cases.replay_synth(name, cases.CudaBackend(g, cases.golden()[name + "_map_order"], raw_weights=raw))


# ------------------------------------------------------------------ fresh inputs vs the oracle
@pytest.mark.parametrize("seed,T,kw", [(21, 1, dict(hub=5000)), (22, 3, dict(zero_w_frac=0.15, id_stride=1009, id_base=77)),
                                       (23, 8, dict(empty_frac=0.4, hub=900, n_node_types=4))])
def test_random_graph_vs_oracle(seed, T, kw):
    n = 20000
    g = graphs.random_graph(seed=seed, n=n, T=T, avg_deg=8, **kw)
    order = np.random.RandomState(seed).permutation(g["ids"])
    be, ob = cases.CudaBackend(g, order), cases.OracleBackend(g, order)
    rs = np.random.RandomState(seed + 1)
    seeds = g["ids"][rs.randint(0, n, size=3000)].astype(np.int64)
    seeds[::13] = 987654321012
    seeds[5::17] = -1
    seeds[3::19] = 0
    for et, cnt in [([0], 25), ([T - 1], 1), (list(range(T)), 70), ([0, T - 1], 33), ([], 10), ([T + 3], 4)]:
        be.seed(seed); ob.seed(seed)
        for a, b in zip(be.op_sample_neighbor(seeds, et, cnt, -5), ob.op_sample_neighbor(seeds, et, cnt, -5)):
            cases.eq(a, b, "sample_neighbor et=%s count=%d" % (et, cnt))
        assert be.draws() == ob.draws()
    ets = [[0, T - 1], [T - 1, 0]]
    be.seed(seed + 2); ob.seed(seed + 2)
    a, b = be.op_sample_fanout(seeds[:600], ets, [25, 10], -1), ob.op_sample_fanout(seeds[:600], ets, [25, 10], -1)
    for x, y in zip(a, b):
        for l in range(2):
            cases.eq(x[l], y[l], "fanout hop %d" % l)
    # engine stream continues across calls exactly like one reference thread
    a2, b2 = be.op_sample_neighbor(seeds, [0], 3, -1), ob.op_sample_neighbor(seeds, [0], 3, -1)
    cases.eq(a2[0], b2[0], "second call on the same stream")
    wet = np.asarray([list(range(T))] * 12, np.int32)
    for p, q in [(0.5, 2.0), (1.0, 1.0), (2.0, 0.5)]:
        be.seed(seed + 3); ob.seed(seed + 3)
        cases.eq(be.op_random_walk(seeds[:500], wet, p, q, -1), ob.op_random_walk(seeds[:500], wet, p, q, -1),
                 "walk p=%s q=%s" % (p, q))
    for types in ([-1], [0], list(range(g["n_node_types"]))):
        be.seed(seed + 4); ob.seed(seed + 4)
        cases.eq(be.sample_node(types, 4097), ob.sample_node(types, 4097), "sample_node %s" % types)


@pytest.mark.parametrize("nb,B,T", [(1, 300, 2), (5, 257, 3), (8, 1024, 1), (16, 33, 4)])
def test_batched_fanout_equals_independent_calls(nb, B, T):
    """eu_sample_fanout_batched: batch b == one sample_fanout call on an engine seeded like engine b."""
    import euler_b200
    g = graphs.random_graph(seed=90 + nb, n=8000, T=T, avg_deg=7, hub=700, id_stride=3, zero_w_frac=0.05)
    gr = graphs.cuda_graph(g)
    og = graphs.oracle_graph(g)
    euler_b200.set_graph(gr)
    ctx = euler_b200.Context(gr, "minstd", 1)
    seeds_e = [1000 + 17 * b for b in range(nb)]
    ctx.set_engines(nb, seeds_e)
    rs = np.random.RandomState(nb)
    nodes = g["ids"][rs.randint(0, 8000, size=(nb, B))].astype(np.int64)
    nodes[:, ::9] = 77777777
    nodes[0, :20] = nodes[0, 0]
    ets = [[0, T - 1], [T - 1, 0]] if T > 1 else [[0], [0]]
    states = {}
    for rep in range(2):  # second call: every engine continues its own stream
        ctx.set_stream(torch.cuda.current_stream().cuda_stream)
        ids, ws, ts = euler_b200.sample_fanout_batched(nodes, ets, [6, 40], -1, ctx=ctx)
        for b in range(nb):
            if rep == 0:
                po.seed(seeds_e[b])
            else:
                po.set_state(states[b])
            o_ids, o_ws, o_ts = _oracle_fanout(og, nodes[b], ets, [6, 40])
            states[b] = po.get_state()
            for l in range(2):
                cases.eq(ids[l + 1][b].cpu().numpy(), o_ids[l], "batch %d rep %d ids hop %d" % (b, rep, l))
                cases.eq(ws[l][b].cpu().numpy(), o_ws[l], "batch %d w hop %d" % (b, l))
                cases.eq(ts[l][b].cpu().numpy(), o_ts[l], "batch %d t hop %d" % (b, l))


def _oracle_fanout(og, nodes, ets, counts):
    """sample_fanout with a different edge-type list length per hop = chained op_sample_neighbor on ENGINE ids."""
    frontier = np.asarray(nodes, np.int64)
    ids, ws, ts = [], [], []
    for et, c in zip(ets, counts):
        e_ids, e_w, e_t = og.op_sample_neighbor(frontier, et, c, 0)      # default_node 0 == engine form
        keep = e_ids[:, :1] != 0
        ids.append(np.where(keep, e_ids, -1).reshape(-1)); ws.append(np.where(keep, e_w, 0).astype(np.float32).reshape(-1))
        ts.append(np.where(keep, e_t, -1).astype(np.int32).reshape(-1))
        frontier = e_ids.reshape(-1)
    return ids, ws, ts


@pytest.mark.parametrize("T,sorted_adj,hub", [(1, True, 3000), (3, True, 500), (2, False, 300), (1, True, 0)])
def test_node2vec_paths_vs_oracle(T, sorted_adj, hub):
    """Both node2vec step kernels: the warp-cooperative one (one edge type per step, sorted adjacency, incl.
    multi-edges and hubs spanning many 32-wide chunks) and the sequential fallback (unsorted / several types)."""
    g = graphs.random_graph(seed=200 + T + hub, n=4000, T=T, avg_deg=9, hub=hub, sorted_adj=sorted_adj, dup_edges=True,
                            empty_frac=0.05)
    be, ob = cases.CudaBackend(g, g["ids"]), cases.OracleBackend(g, g["ids"])
    seeds = g["ids"][np.random.RandomState(7).randint(0, 4000, size=700)].astype(np.int64)
    seeds[::31] = 123456789
    for wet in ([[T - 1]] * 15, [[0], [T - 1]] * 6, [list(range(T))] * 5):
        for p, q in [(0.5, 2.0), (3.0, 0.25)]:
            be.seed(9); ob.seed(9)
            cases.eq(be.op_random_walk(seeds, np.asarray(wet, np.int32), p, q, -1),
                     ob.op_random_walk(seeds, np.asarray(wet, np.int32), p, q, -1), "walk %s p=%s q=%s" % (wet[0], p, q))
            assert be.draws() == ob.draws()


def test_hetero_rmat_graph_vs_oracle():
    """Device-generated heterogeneous graph (configs[4] shape): export -> oracle -> all edge-type modes."""
    import euler_b200
    n, E, T, NT = 30000, 240000, 5, 3
    gr = euler_b200.Graph.rmat_hetero(n, E, T, NT, feat_dim=8)
    ex = gr.export()
    assert (ex["node_type"] == ex["ids"] % NT).all() and ex["grp_ptr"][-1] == E
    og = po.OracleGraph(ex["ids"], ex["node_type"], ex["node_w"], T, ex["grp_ptr"], ex["nbr"], ex["cum_w"], ex["grp_cum"], ex["feat"])
    # the generator's prefix sums equal Node::Init's accumulation of the de-cumulated weights group by group
    euler_b200.set_graph(gr)
    seeds = np.random.RandomState(4).randint(1, n + 1, size=2000).astype(np.int64)
    for et, cnt in [([2], 10), (list(range(T)), 10), ([4, 0, 1], 7), ([], 3)]:
        euler_b200.seed(5); po.seed(5)
        got = [x.cpu().numpy() for x in euler_b200.sample_neighbor(seeds, et, cnt)]
        for a, b in zip(got, og.op_sample_neighbor(seeds, et, cnt)):
            cases.eq(a, b, "hetero sample_neighbor %s" % et)
    og.build_node_sampler(np.arange(n), NT)
    for types in ('-1', [1], [0, 2]):
        euler_b200.seed(6)
        r = po.Rng(6)
        want = og.sample_node([-1] if types == '-1' else types, 3000, r)
        cases.eq(euler_b200.sample_node(3000, types).cpu().numpy().astype(np.uint64), want, "hetero sample_node %s" % (types,))
    x = euler_b200.get_dense_feature(seeds[:50], [0], [8])[0].cpu().numpy()
    cases.eq(x, og.op_get_dense_feature(seeds[:50], 8), "hetero features")


def test_empty_and_degenerate_inputs():
    import euler_b200
    g = graphs.random_graph(seed=31, n=50, T=2)
    be = cases.CudaBackend(g, g["ids"])
    ids, w, t = euler_b200.sample_neighbor(np.zeros(0, np.int64), [0], 5)
    assert ids.shape == (0, 5)
    ids, w, t = euler_b200.sample_neighbor([1, 2], [0], 0)
    assert ids.shape == (2, 0)
    out = euler_b200.random_walk([1, 2, 3], [], 0.5, 2.0)
    assert out.cpu().numpy().tolist() == [[1], [2], [3]]
    # every seed absent -> all defaults, no draws
    be.seed(1)
    ids, w, t = be.op_sample_neighbor(np.asarray([10 ** 12, -1, 0], np.int64), [0, 1], 4, -9)
    assert (ids == -9).all() and (w == 0).all() and (t == -1).all() and be.draws() == 0


def test_host_buffer_entry_points_match_device_ones():
    import euler_b200
    from euler_b200 import _lib
    g = graphs.random_graph(seed=41, n=5000, T=2, feat_dim=16)
    be = cases.CudaBackend(g, g["ids"])
    lib, ctx = _lib.load(), euler_b200.context()
    seeds = g["ids"][np.random.RandomState(3).randint(0, 5000, size=700)].astype(np.int64)
    et = np.asarray([[0, 1], [1, 0]], np.int32)
    cs = np.asarray([6, 5], np.int32)
    be.seed(77)
    d_ids, d_w, d_t = be.op_sample_fanout(seeds, et, [6, 5], -1)
    h_ids = [np.zeros(700 * 6, np.int64), np.zeros(700 * 30, np.int64)]
    h_w = [np.zeros(700 * 6, np.float32), np.zeros(700 * 30, np.float32)]
    h_t = [np.zeros(700 * 6, np.int32), np.zeros(700 * 30, np.int32)]
    P = C.c_void_p * 2
    be.seed(77)
    _lib.check(lib.eu_sample_fanout_host(ctx._h, seeds.ctypes.data, 700, et.ctypes.data, 2, cs.ctypes.data, 2, -1,
                                         P(*[x.ctypes.data for x in h_ids]), P(*[x.ctypes.data for x in h_w]),
                                         P(*[x.ctypes.data for x in h_t])))
    for l in range(2):
        cases.eq(h_ids[l], d_ids[l], "host fanout ids"); cases.eq(h_w[l], d_w[l], "host fanout w"); cases.eq(h_t[l], d_t[l], "host fanout t")
    out = np.zeros((700, 16), np.float32)
    _lib.check(lib.eu_get_dense_feature_host(ctx._h, seeds.ctypes.data, 700, 0, 16, out.ctypes.data))
    cases.eq(out, graphs.oracle_graph(g).op_get_dense_feature(seeds, 16), "host dense feature")
    x = np.random.RandomState(1).randn(300, 8).astype(np.float32)
    idx = np.sort(np.random.RandomState(2).randint(0, 40, size=300)).astype(np.int32)
    o = np.zeros((40, 8), np.float32)
    _lib.check(lib.eu_scatter_add_host(ctx._h, x.ctypes.data, 8, idx.ctypes.data, 300, 40, o.ctypes.data))
    cases.eq(o, po.scatter_add(x, idx, 40), "host scatter_add")
    _lib.check(lib.eu_scatter_max_host(ctx._h, x.ctypes.data, 8, idx.ctypes.data, 300, 40, o.ctypes.data))
    cases.eq(o, po.scatter_max(x, idx, 40), "host scatter_max")
    o2 = np.zeros((300, 8), np.float32)
    _lib.check(lib.eu_gather_host(ctx._h, x.ctypes.data, 300, 8, idx.ctypes.data, 300, o2.ctypes.data))
    cases.eq(o2, po.gather(x, idx), "host gather")
    wk = np.zeros((700, 5), np.int64)
    wet = np.asarray([[0, 1]] * 4, np.int32)
    be.seed(5)
    ref = be.op_random_walk(seeds, wet, 0.25, 4.0, -1)
    be.seed(5)
    _lib.check(lib.eu_random_walk_host(ctx._h, seeds.ctypes.data, 700, wet.ctypes.data, 2, 4, 0.25, 4.0, -1, wk.ctypes.data))
    cases.eq(wk, ref, "host random_walk")
    sn = np.zeros(100, np.int64)
    t0 = np.asarray([0], np.int32)
    be.seed(6)
    ref = be.sample_node([0], 100)
    be.seed(6)
    _lib.check(lib.eu_sample_node_host(ctx._h, 100, t0.ctypes.data, 1, sn.ctypes.data))
    cases.eq(sn.astype(np.uint64), ref, "host sample_node")


# ------------------------------------------------------------------ message passing
@pytest.mark.parametrize("D", [1, 3, 64, 128, 200, 256])
def test_mp_ops_vs_oracle(D):
    import euler_b200
    g = graphs.random_graph(seed=51, n=10, T=1)
    cases.CudaBackend(g, g["ids"])
    rs = np.random.RandomState(D)
    N, E, size = 5000, 40000, 3000
    params = rs.randn(N, D).astype(np.float32)
    idx = rs.randint(0, N, size=E).astype(np.int32)
    cases.eq(euler_b200.gather(params, idx).cpu().numpy(), po.gather(params, idx), "gather")
    upd = rs.randn(E, D).astype(np.float32)
    sidx = np.sort(rs.randint(0, size, size=E)).astype(np.int32)
    sidx[sidx == 7] = 8  # an empty output row
    # sorted indices (what the dataflows emit): the reference's summation order -> bit-exact
    cases.eq(euler_b200.scatter_add(upd, sidx, size).cpu().numpy(), po.scatter_add(upd, sidx, size), "scatter_add sorted")
    cases.eq(euler_b200.scatter_max(upd, sidx, size).cpu().numpy(), po.scatter_max(upd, sidx, size), "scatter_max sorted")
    cases.eq(euler_b200.scatter_mean(upd, sidx, size).cpu().numpy(), po.scatter_mean(upd, sidx, size), "scatter_mean sorted")
    # unsorted indices: order-free atomics, 1e-5 relative (max is exact)
    uidx = rs.permutation(sidx).astype(np.int32)
    for name in ("scatter_add", "scatter_mean"):
        got = getattr(euler_b200, name)(upd, uidx, size).cpu().numpy()
        want = getattr(po, name)(upd, uidx, size)
        scale = np.maximum(np.abs(want), po.scatter_add(np.abs(upd), uidx, size) if name == "scatter_add" else 1.0)
        assert (np.abs(got - want) <= RTOL * np.maximum(scale, 1e-30)).all(), name
    cases.eq(euler_b200.scatter_max(upd, uidx, size).cpu().numpy(), po.scatter_max(upd, uidx, size), "scatter_max unsorted")


def test_mp_ops_reference_test_vectors_and_gradients():
    """tf_euler/python/euler_ops/mp_ops_test.py:30-94 incl. its numeric-gradient checks."""
    import euler_b200 as mp_ops
    g = graphs.random_graph(seed=52, n=10, T=1)
    cases.CudaBackend(g, g["ids"])
    x = torch.tensor([[1., 2.], [3., 4.], [5., 6.]], device="cuda")
    idx = torch.tensor([1, 0, 1], device="cuda")
    assert mp_ops.scatter_add(x, idx, size=2).cpu().tolist() == [[3., 4.], [6., 8.]]
    assert (mp_ops.scatter_mean(x, idx, size=2).cpu() - torch.tensor([[3., 4.], [3., 4.]])).abs().sum() < 1e-6
    x2 = torch.tensor([[1., 6.], [3., 4.], [5., 2.]], device="cuda")
    assert mp_ops.scatter_max(x2, idx, size=2).cpu().tolist() == [[3., 4.], [5., 6.]]
    idx4 = torch.tensor([1, 0, 1, 2], device="cuda")
    assert mp_ops.gather(x, idx4).cpu().tolist() == [[3., 4.], [1., 2.], [3., 4.], [5., 6.]]

    def numeric_grad_err(fn, x0):
        xg = x0.clone().requires_grad_(True)
        y = fn(xg)
        wgt = torch.arange(1, y.numel() + 1, device="cuda", dtype=torch.float32).reshape(y.shape)
        (y * wgt).sum().backward()
        an = xg.grad.clone()
        num = torch.zeros_like(x0)
        eps = 1e-2
        for i in range(x0.numel()):
            d = torch.zeros_like(x0).reshape(-1)
            d[i] = eps
            d = d.reshape(x0.shape)
            num.reshape(-1)[i] = ((fn(x0 + d) * wgt).sum() - (fn(x0 - d) * wgt).sum()) / (2 * eps)
        return (an - num).abs().max().item()

    assert numeric_grad_err(lambda v: mp_ops.scatter_add(v, idx, size=2), x) < 1e-2
    assert numeric_grad_err(lambda v: mp_ops.scatter_mean(v, idx, size=2), x) < 1e-2
    assert numeric_grad_err(lambda v: mp_ops.gather(v, idx4), x) < 1e-2
    x3 = torch.tensor([[1., 2., 7.], [3., 4., 8.], [5., 6., 7.]], device="cuda")
    xg = x3.clone().requires_grad_(True)
    mp_ops.scatter_max(xg, idx, size=2).sum().backward()
    # ties split evenly (mp_ops.py:52-62): column 2 of rows 0 and 2 tie at 7
    assert xg.grad.cpu().tolist() == [[0., 0., .5], [1., 1., 1.], [1., 1., .5]]
    sm = mp_ops.scatter_softmax(x3, idx, size=2).cpu()
    assert torch.allclose(sm[0] + sm[2], torch.ones(3)) and torch.allclose(sm[1], torch.ones(3))


@pytest.mark.parametrize("D,count", [(128, 10), (256, 15), (64, 25), (128, 40)])
def test_dense_feature_and_fused_sage_mean(D, count):
    import euler_b200
    n = 4000
    g = graphs.random_graph(seed=61 + D, n=n, T=1, feat_dim=D, id_stride=3 if D == 64 else 1)
    cases.CudaBackend(g, g["ids"])
    og = graphs.oracle_graph(g)
    rs = np.random.RandomState(D)
    ids = g["ids"][rs.randint(0, n, size=700 * count)].astype(np.int64)
    ids[::29] = -1  # default-filled slots -> zero rows
    (f,) = euler_b200.get_dense_feature(ids, [0], [D])
    want = og.op_get_dense_feature(ids, D)
    cases.eq(f.cpu().numpy(), want, "get_dense_feature")
    (fpad,) = euler_b200.get_dense_feature(ids[:100], [0], [D + 8])
    assert np.array_equal(fpad.cpu().numpy()[:, :D], want[:100]) and not fpad.cpu().numpy()[:, D:].any()
    (fclip,) = euler_b200.get_dense_feature(ids[:100], [0], [D // 2])
    assert np.array_equal(fclip.cpu().numpy(), want[:100, :D // 2])
    (funk,) = euler_b200.get_dense_feature(ids[:10], [3], [4])
    assert not funk.cpu().numpy().any()
    # fused gather + mean == get_dense_feature followed by scatter_mean over repeat(range(rows), count)
    src = np.repeat(np.arange(700, dtype=np.int32), count)
    cases.eq(euler_b200.sage_mean_aggregate(ids, count, D).cpu().numpy(), po.scatter_mean(want, src, 700), "sage_mean")
    cases.eq(euler_b200.scatter_mean(f, src, 700).cpu().numpy(), po.scatter_mean(want, src, 700), "scatter_mean of gathered")


# ------------------------------------------------------------------ throughput engine (philox)
def test_philox_mode_semantics_and_distribution():
    import euler_b200
    g = graphs.random_graph(seed=71, n=3000, T=2, avg_deg=6, hub=400)
    gr = graphs.cuda_graph(g)
    euler_b200.set_graph(gr, rng="philox", seed=9)
    seeds = np.concatenate([g["ids"][:500], g["ids"][:500], [10 ** 12]]).astype(np.int64)
    ids, w, t = [x.cpu().numpy() for x in euler_b200.sample_neighbor(seeds, [0, 1], 16, -1)]
    assert np.array_equal(ids[:500], ids[500:1000])          # duplicate seeds share one sample row
    assert (ids[-1] == -1).all()
    ids2 = euler_b200.sample_neighbor(seeds, [0, 1], 16, -1)[0].cpu().numpy()
    assert not np.array_equal(ids, ids2)                      # next call, new stream position
    # every sampled (neighbor, weight, type) is a real edge of its seed
    og = graphs.oracle_graph(g)
    for i in range(0, 500, 7):
        lens, nb, ww, tt = og.get_full_neighbor([seeds[i]], [0, 1])
        edges = set(zip(nb.tolist(), ww.tolist(), tt.tolist()))
        if not edges:
            assert (ids[i] == -1).all()
        else:
            assert set(zip(ids[i].tolist(), w[i].tolist(), t[i].tolist())) <= edges
    # distribution: hub row, type 0 group, empirical frequencies ~ weights
    hub = int(np.argmax(np.diff(g["grp_ptr"])))
    r, tt = divmod(hub, 2)
    b, e = g["grp_ptr"][hub], g["grp_ptr"][hub + 1]
    wts = g["w"][b:e].astype(np.float64)
    draws = euler_b200.sample_neighbor(np.full(4000, g["ids"][r], np.int64), [tt], 1)[0]
    many = torch.cat([euler_b200.sample_neighbor([g["ids"][r]], [tt], 4096)[0].reshape(-1) for _ in range(40)]).cpu().numpy()
    assert (draws.cpu().numpy() == draws.cpu().numpy()[0]).all()
    exp = {}
    for nid, ww in zip(g["nbr"][b:e].tolist(), wts):
        exp[nid] = exp.get(nid, 0.0) + ww
    tot = sum(exp.values())
    uniq, cnt = np.unique(many, return_counts=True)
    chi2 = sum((c - many.size * exp[int(u)] / tot) ** 2 / (many.size * exp[int(u)] / tot) for u, c in zip(uniq, cnt))
    assert chi2 < 2.0 * len(exp) + 100, chi2


def _node2vec_weights(cids, cw, pids, parent_id, p, q):
    """literal restatement of BuildWeights (tf_euler/kernels/random_walk_op.cc:140-168): two-pointer merge of the child list
    against the parent's list, f64"""
    out = np.array(cw, np.float64)
    j = k = 0
    while j < len(cids) and k < len(pids):
        if cids[j] < pids[k]:
            out[j] /= (q if cids[j] != parent_id else p)
            j += 1
        elif cids[j] == pids[k]:
            j += 1
            k += 1
        else:
            k += 1
    while j < len(cids):
        out[j] /= (q if cids[j] != parent_id else p)
        j += 1
    return out


def test_philox_node2vec_fast_mode_distribution():
    """EU_RNG_PHILOX takes node2vec steps by rejection (k_walk_fast): every step is a real edge, dead walkers go to the
    default node, calls differ, and the transition frequencies match the exact biased weights (chi-square), multi-edges
    and the walker's own parent included."""
    import euler_b200
    g = graphs.random_graph(seed=83, n=60, T=1, avg_deg=14, empty_frac=0.05)
    gr = graphs.cuda_graph(g)
    euler_b200.set_graph(gr, rng="philox", seed=3)
    ids, ptr, nbr, w = g["ids"].astype(np.int64), g["grp_ptr"], g["nbr"].astype(np.int64), g["w"].astype(np.float64)
    row = {int(v): r for r, v in enumerate(ids)}
    p, q = 0.5, 2.0
    deg = np.diff(ptr)
    a = int(ids[int(np.argmax(deg))])
    N = 400_000
    wk = euler_b200.random_walk(np.full(N, a, np.int64), [[0], [0]], p, q, -1).cpu().numpy()
    wk2 = euler_b200.random_walk(np.full(N, a, np.int64), [[0], [0]], p, q, -1).cpu().numpy()
    assert not np.array_equal(wk, wk2)
    assert (wk[:, 0] == a).all()

    def chi2(obs_ids, cand, weights):
        exp = {}
        for v, x in zip(cand.tolist(), weights.tolist()):
            exp[v] = exp.get(v, 0.0) + x
        tot = sum(exp.values())
        uniq, cnt = np.unique(obs_ids, return_counts=True)
        assert set(uniq.tolist()) <= {v for v, x in exp.items() if x > 0}
        got = dict(zip(uniq.tolist(), cnt.tolist()))
        n = obs_ids.size
        stat = sum((got.get(v, 0) - n * x / tot) ** 2 / (n * x / tot) for v, x in exp.items() if x > 0)
        dof = sum(1 for x in exp.values() if x > 0) - 1
        return stat, dof
    ra = row[a]
    ca, wa = nbr[ptr[ra]:ptr[ra + 1]], w[ptr[ra]:ptr[ra + 1]]
    st, dof = chi2(wk[:, 1], ca, _node2vec_weights(ca, wa, [], a, p, q))     # step 0: empty parent list, parent = the start node
    assert st < dof + 6 * np.sqrt(2 * dof) + 10, (st, dof)
    checked = 0
    for b in np.unique(wk[:, 1]):
        sel = wk[wk[:, 1] == b]
        rb = row[int(b)]
        cb, wb = nbr[ptr[rb]:ptr[rb + 1]], w[ptr[rb]:ptr[rb + 1]]
        if len(cb) == 0:
            assert (sel[:, 2] == -1).all()
            continue
        if len(sel) < 20000:
            continue
        st, dof = chi2(sel[:, 2], cb, _node2vec_weights(cb, wb, ca, a, p, q))
        assert st < dof + 6 * np.sqrt(2 * dof) + 10, (int(b), st, dof)
        checked += 1
    assert checked >= 3
    # long walks (two launches of the step loop), unknown / dead seeds
    seeds = np.concatenate([ids[:50], [10 ** 12, 0]]).astype(np.int64)
    L = 130
    lw = euler_b200.random_walk(seeds, [[0]] * L, 0.25, 4.0, -1).cpu().numpy()
    assert (lw[-2:, 1:] == -1).all()
    edges = set()
    for r in range(len(ids)):
        for v in nbr[ptr[r]:ptr[r + 1]]:
            edges.add((int(ids[r]), int(v)))
    for i in range(50):
        for t in range(L):
            u, v = int(lw[i, t]), int(lw[i, t + 1])
            if u == -1:
                assert v == -1
            elif v == -1:
                assert deg[row[u]] == 0
            else:
                assert (u, v) in edges



# ------------------------------------------------------------------ large-size properties
def test_rmat_large_properties():
    """RMAT 2M nodes / 20M edges generated on the device: structure invariants, and at BASELINE's
    fanout [25,10] x batch 1024 every sampled edge is a real edge with its stored weight; minstd
    results equal the oracle run on the exported graph (bit-exact at full fanout)."""
    import euler_b200
    n, E = 2_000_000, 20_000_000
    gr = euler_b200.Graph.rmat(n, E, feat_dim=32)
    ex = gr.export(with_feat=False)
    ptr, nbr, cum = ex["grp_ptr"], ex["nbr"], ex["cum_w"]
    assert ptr[0] == 0 and ptr[-1] == E and (np.diff(ptr) >= 0).all()
    assert nbr.min() >= 1 and nbr.max() <= n
    row_of_edge = np.repeat(np.arange(n), np.diff(ptr))
    key = row_of_edge.astype(np.int64) * (n + 1) + nbr.astype(np.int64)
    assert (np.diff(key) >= 0).all()                      # adjacency sorted by dst within each row
    first = ptr[:-1][np.diff(ptr) > 0]
    w = np.diff(cum, prepend=np.float32(0))
    w[first] = cum[first]
    assert w.min() > 0.5 and w.max() < 11.5               # 1 + (h%100)/10, up to f32 prefix rounding on hub rows
    deg = np.diff(ptr)
    assert deg.max() > 50 * deg.mean()                    # heavy tail
    euler_b200.set_graph(gr, rng="minstd", seed=12345)
    seeds = np.random.RandomState(1000).randint(1, n + 1, size=1024).astype(np.int64)
    ids, ws, ts = euler_b200.sample_fanout(seeds, [[0], [0]], [25, 10])
    og = po.OracleGraph(ex["ids"], ex["node_type"], ex["node_w"], 1, ptr, nbr, cum, np.zeros(n, np.float32))
    po.seed(12345)
    o_ids, o_ws, o_ts = og.op_sample_fanout(seeds, [[0], [0]], [25, 10])
    for l in range(2):
        cases.eq(ids[l + 1].cpu().numpy(), o_ids[l], "rmat fanout ids hop %d" % l)
        cases.eq(ws[l].cpu().numpy(), o_ws[l], "rmat fanout w hop %d" % l)
    # membership: (src row, dst) must exist
    src = np.repeat(ids[1].cpu().numpy(), 10)
    dst = ids[2].cpu().numpy()
    ok = dst != -1
    k2 = (src[ok] - 1) * (n + 1) + dst[ok]
    pos = np.searchsorted(key, k2)
    assert (key[np.minimum(pos, E - 1)] == k2).all()
    # features of the sampled frontier: exact row copies of the generator's U(-1,1) rows
    (f,) = euler_b200.get_dense_feature(ids[1], [0], [32])
    f = f.cpu().numpy()
    valid = ids[1].cpu().numpy() != -1          # RMAT: many seeds have no out-edge -> default rows -> zero features
    assert 0.05 < valid.mean() < 1.0
    assert np.abs(f).max() <= 1.0 and f[valid].std() > 0.5 and not f[~valid].any()
    (f2,) = euler_b200.get_dense_feature(ids[1], [0], [32])
    assert np.array_equal(f, f2.cpu().numpy())


# ---------------------------------------------------------------------------- get_full_neighbor (next-1)
@pytest.mark.gpu
def test_get_full_neighbor_tiny_graph_matches_reference_test_vector():
    """neighbor_ops_test.py:46-57 on the tools/test_data graph + every node / type list against the oracle"""
    import euler_b200
    g = graphs.load_tiny_csr()
    gr = graphs.cuda_graph(g)
    og = graphs.oracle_graph(g)
    euler_b200.set_graph(gr, seed=1)
    for nodes, et in [([1, 2], [0, 1]), ([1, 2, 3, 4, 5, 6], [0]), ([6, 5, 99, 1, 1], [1, 0, 1]), ([3], []), ([], [0, 1]), ([2, 4], [7, 0])]:
        indptr, ids, w, t = euler_b200.get_full_neighbor(np.asarray(nodes, np.int64), et)
        lens, o_ids, o_w, o_t = og.get_full_neighbor(np.asarray(nodes, np.uint64), et)
        cases.eq(np.diff(indptr.cpu().numpy()), np.asarray(lens, np.int64), "lens %s %s" % (nodes, et))
        cases.eq(ids.cpu().numpy(), np.asarray(o_ids).astype(np.int64), "ids")
        cases.eq(w.cpu().numpy(), o_w, "w")
        cases.eq(t.cpu().numpy(), o_t, "t")


@pytest.mark.gpu
@pytest.mark.parametrize("T,stride", [(1, 1), (3, 7)])
def test_get_full_neighbor_random_graph_and_host_entry(T, stride):
    import euler_b200
    g = graphs.random_graph(seed=77 + T, n=5000, T=T, avg_deg=9, id_stride=stride, id_base=3, hub=4000, zero_w_frac=0.1)
    gr = graphs.cuda_graph(g)
    og = graphs.oracle_graph(g)
    euler_b200.set_graph(gr, seed=1)
    rs = np.random.RandomState(5)
    nodes = g["ids"][rs.randint(0, 5000, size=3000)].astype(np.int64)
    nodes[::9] = 10 ** 15
    nodes[0] = g["ids"][int(np.argmax(np.diff(g["grp_ptr"])) // T)]        # the hub
    for et in ([0], list(range(T))[::-1], [T - 1, 0, T - 1]):
        indptr, ids, w, t = euler_b200.get_full_neighbor(nodes, et)
        lens, o_ids, o_w, o_t = og.get_full_neighbor(nodes.astype(np.uint64), et)
        cases.eq(np.diff(indptr.cpu().numpy()), np.asarray(lens, np.int64), "lens")
        cases.eq(ids.cpu().numpy(), np.asarray(o_ids).astype(np.int64), "ids")
        cases.eq(w.cpu().numpy(), o_w, "w")
        cases.eq(t.cpu().numpy(), o_t, "t")
    # host entry point through the C ABI: size with cap = 0, then fetch
    from euler_b200 import _lib
    lib = _lib.load()
    ctx = euler_b200.context()
    et = np.asarray([0], np.int32)
    ptr = np.zeros(len(nodes) + 1, np.int64)
    total = C.c_int64(0)
    _lib.check(lib.eu_get_full_neighbor_host(ctx._h, nodes.ctypes.data, len(nodes), et.ctypes.data, 1, 0, ptr.ctypes.data, None, None, None, C.byref(total)))
    lens, o_ids, o_w, o_t = og.get_full_neighbor(nodes.astype(np.uint64), [0])
    assert total.value == int(np.sum(lens))
    h_ids, h_w, h_t = np.zeros(total.value, np.int64), np.zeros(total.value, np.float32), np.zeros(total.value, np.int32)
    _lib.check(lib.eu_get_full_neighbor_host(ctx._h, nodes.ctypes.data, len(nodes), et.ctypes.data, 1, total.value, ptr.ctypes.data,
                                             h_ids.ctypes.data, h_w.ctypes.data, h_t.ctypes.data, C.byref(total)))
    cases.eq(np.diff(ptr), np.asarray(lens, np.int64), "host lens")
    cases.eq(h_ids, np.asarray(o_ids).astype(np.int64), "host ids")
    cases.eq(h_w, o_w, "host w")
    cases.eq(h_t, o_t, "host t")


# ---------------------------------------------------------------------------- C++ euler::api adapter (seam B3)
@pytest.mark.gpu
def test_cpp_api_adapter(tiny_dir):
    """tests/cpp/api_adapter_main.cc calls include/euler_b200_api.hpp like a C++ user of euler/core/api/api.h; its printed
    results must equal the oracle's on the tools/test_data graph (same seed -> same sampled neighbors)."""
    import os
    import subprocess
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib = os.path.join(root, "euler_b200", "lib")
    exe = os.path.join(tempfile.mkdtemp(), "api_adapter_main")
    subprocess.check_call(["g++", "-std=c++11", "-I" + os.path.join(root, "include"), os.path.join(root, "tests", "cpp", "api_adapter_main.cc"),
                           "-L" + lib, "-leuler_b200", "-Wl,-rpath," + lib, "-o", exe])
    out = subprocess.run([exe, tiny_dir, "5"], capture_output=True, text=True, check=True).stdout
    kv = {}
    for line in out.strip().splitlines():
        k, _, v = line.partition(":")
        kv[k] = v.split()
    g = graphs.load_tiny_csr()
    og = graphs.oracle_graph(g)
    type_of = {int(i): int(t) for i, t in zip(g["ids"], g["node_type"])}
    assert [int(x) for x in kv["node_type"]] == [type_of.get(i, -2 ** 31) for i in [1, 2, 3, 4, 5, 6, 99]]
    # full neighbors
    lens, ids, w, t = og.get_full_neighbor(np.asarray([1, 2, 99, 6], np.uint64), [0, 1])
    off = 0
    for i, n in enumerate(lens):
        got = kv["full[%d]" % i]
        want = []
        for k in range(off, off + n):
            want += [str(int(ids[k])), "%.9g" % float(w[k]), str(int(t[k]))]
        assert got == want, (i, got, want)
        off += n
    # sampled neighbors: engine stream seeded 4242; euler::SampleNeighbor = api.cc:223-236 (every occurrence of an id draws
    # independently, in order), empty vector for absent rows
    rng = po.Rng(4242)

    def fmt_rows(o_ids, o_w, o_t, n_rows, cnt, lens=None):
        out = []
        for i in range(n_rows):
            want = []
            if (lens[i] if lens is not None else o_ids[i, 0] != 0):
                for j in range(cnt):
                    want += [str(int(o_ids[i, j])), "%.9g" % float(o_w[i, j]), str(int(o_t[i, j]))]
            out.append(want)
        return out
    for key, nodes, et in [("sample", [1, 2, 3, 99, 1, 6], [0, 1]), ("sample2", [4, 5], [1])]:
        o_ids, o_w, o_t, o_len = og.sample_neighbor_api(np.asarray(nodes, np.uint64), et, 5, rng)
        for i, want in enumerate(fmt_rows(o_ids, o_w, o_t, len(nodes), 5, o_len)):
            assert kv["%s[%d]" % (key, i)] == want, (key, i, kv["%s[%d]" % (key, i)], want)
    # dense features: node 1 and 3 per slot, absent node -> empty vectors, unknown slot -> empty
    feat = g["feat"].reshape(len(g["ids"]), -1)
    rows = {int(i): r for r, i in enumerate(g["ids"])}
    dims = [int(d) for d in g["feat_slot_dims"]] if "feat_slot_dims" in g else None
    for i, node in enumerate([1, 99, 3]):
        for k in range(3):
            vals = kv["feat[%d][%d]" % (i, k)]
            if node not in rows or k == 2:
                assert vals == []
            elif dims is not None:
                lo = sum(dims[:k])
                assert vals == ["%.9g" % float(x) for x in feat[rows[node], lo:lo + dims[k]]]
            else:
                assert len(vals) > 0
    assert len(kv["sample_node"]) == 8 and all(int(x) in rows for x in kv["sample_node"])
    assert kv["names"] == ["1", "-1", "0", "-1"]
    # the op-level variant continues the same engine: sample_node drew 8 x 3 uniforms (a list of 2 types) in between
    for _ in range(24):
        rng.uniform()
    po.set_state((rng.x, rng.draws))
    nodes = [1, 2, 3, 99, 1, 6]
    o_ids, o_w, o_t = og.op_sample_neighbor(np.asarray(nodes, np.int64), [0, 1], 5, 0)
    for i, want in enumerate(fmt_rows(o_ids.reshape(6, 5), o_w.reshape(6, 5), o_t.reshape(6, 5), 6, 5)):
        assert kv["unique[%d]" % i] == want, ("unique", i)
    assert kv["unique[0]"] == kv["unique[4]"]          # duplicates share one row under the op semantics
    st = po.get_state()
    rng.x, rng.draws = st[0], st[1]
    # euler::Graph / euler::Node
    r1 = rows[1]
    assert kv["graph_node"] == ["1", "1", str(int(g["node_type"][r1])), "%.9g" % float(g["node_w"][r1]), "1"]
    o_ids, o_w, o_t, o_len = og.sample_neighbor_api(np.asarray([1], np.uint64), [0, 1], 5, rng)
    assert kv["node_sample[0]"] == fmt_rows(o_ids, o_w, o_t, 1, 5, o_len)[0]
    lens, f_ids, f_w, f_t = og.get_full_neighbor(np.asarray([1], np.uint64), [0, 1])
    full = [(int(f_ids[k]), float(f_w[k]), int(f_t[k])) for k in range(int(lens[0]))]
    flat = lambda v: [x for (a, b, c) in v for x in (str(a), "%.9g" % b, str(c))]  # noqa: E731
    assert kv["node_full[0]"] == flat(full)
    assert kv["node_sorted[0]"] == flat(sorted(full, key=lambda z: z[0]))
    assert kv["node_topk[0]"] == flat(sorted(full, key=lambda z: -z[1])[:2])
    assert len(kv["graph_sample_node"]) == 6 and all(type_of[int(x)] == 0 for x in kv["graph_sample_node"])
    assert kv["graph_init_bad"] == ["0"]
    assert kv["out_of_scope"] == ["throws"]


# ---------------------------------------------------------------------------- device-side unique + dataflow (next-1)
@pytest.mark.gpu
def test_unique_first_occurrence_and_sage_dataflow():
    import euler_b200
    from euler_b200.dataflow import SageDataFlow
    from test_dataflow_cpu import CpuSampler, np_unique_first
    g = graphs.random_graph(seed=11, n=800, T=2, avg_deg=4, id_stride=3, id_base=2, hub=90)
    euler_b200.set_graph(graphs.cuda_graph(g), seed=77)
    rs = np.random.RandomState(2)
    for n in (1, 31, 1000, 70001):
        x = rs.randint(-3, 400, size=n).astype(np.int64)
        x[::17] = -1
        x[5::29] = 0
        v, inv = euler_b200.unique(x)
        wv, winv = np_unique_first(x)
        cases.eq(v.cpu().numpy(), wv, "unique values n=%d" % n)
        cases.eq(inv.cpu().numpy().astype(np.int64), winv.astype(np.int64), "unique inverse n=%d" % n)
    v, inv = euler_b200.unique(np.zeros(0, np.int64))
    assert v.numel() == 0 and inv.numel() == 0
    roots = g["ids"][rs.randint(0, 800, size=64)].astype(np.int64)
    roots[::9] = 10 ** 9
    for self_loops in (True, False):
        euler_b200.seed(77)
        flow = SageDataFlow([5, 3], [[0, 1], [1]], add_self_loops=self_loops, max_id=10 ** 7)(torch.as_tensor(roots, device="cuda"))
        want = SageDataFlow([5, 3], [[0, 1], [1]], add_self_loops=self_loops, max_id=10 ** 7, sampler=CpuSampler(g, 77))(torch.from_numpy(roots))
        for a, b in zip(flow, want):
            cases.eq(a.n_id.cpu().numpy(), b.n_id.numpy(), "flow n_id")
            cases.eq(a.res_n_id.cpu().numpy(), b.res_n_id.numpy(), "flow res_n_id")
            cases.eq(a.edge_index.cpu().numpy(), b.edge_index.numpy(), "flow edge_index")
            assert a.size == b.size


# ------------------------------------------------------------------ round 2: generator restatement, pinned host buffers
@pytest.mark.parametrize("n,E,T,NT", [(50_000, 600_000, 1, 1), (30_011, 250_000, 5, 3)])
def test_device_rmat_generator_equals_host_restatement(n, E, T, NT):
    """euler_b200/csrc/graph.cu (k_rmat_edges, k_rmat_fill, k_build_cum, k_fill_feat) vs oracle/rmat_gen.c: bit-identical
    CSR, cumulative weights and features -- bench.py's CPU arms and its parity gate rely on this equality."""
    import euler_b200
    if T == 1:
        gr = euler_b200.Graph.rmat(n, E, seed=42, feat_dim=24, feat_seed=7)
    else:
        gr = euler_b200.Graph.rmat_hetero(n, E, T, NT, seed=42, feat_dim=24, feat_seed=7)
    ex = gr.export()
    host = po.rmat_graph(n, E, seed=42, feat_dim=24, feat_seed=7, T=T, NT=NT, threads=3)
    for k in ("ids", "node_type", "node_w", "grp_ptr", "nbr", "cum_w", "feat") + (("grp_cum",) if T > 1 else ()):
        cases.eq(ex[k], host[k], "rmat " + k)
    ids = np.array([1, n, n + 1, 0, -1, 17], np.int64)
    want = np.where(((ids >= 1) & (ids <= n))[:, None], host["feat"][np.clip(ids - 1, 0, n - 1)], 0).astype(np.float32)
    cases.eq(po.rmat_feat_rows(ids, n, 24, 7), want, "rmat_feat_rows")


def test_host_entry_points_dma_pinned_buffers_in_place():
    """*_host with page-locked caller buffers (no staging copy) == the same calls with pageable buffers == device entry points"""
    import euler_b200
    from euler_b200 import _lib
    lib = _lib.load()
    g = graphs.random_graph(seed=77, n=20000, T=2, avg_deg=8, feat_dim=128, hub=400)
    gr = graphs.cuda_graph(g)
    B, counts, nb = 300, [6, 5], 3
    cs = np.asarray(counts, np.int32)
    et = np.asarray([[0, 1], [1, 0]], np.int32)
    seeds = g["ids"][np.random.RandomState(5).randint(0, 20000, size=nb * B)].astype(np.int64)
    seeds[::7] = 0
    n1, n2 = nb * B * 6, nb * B * 30
    P = C.c_void_p * 2
    outs = {}
    for mode in ("pinned", "pageable"):
        ctx = euler_b200.Context(gr, "minstd", 99)
        ctx.set_engines(nb, [500 + b for b in range(nb)])
        mk = (lambda n_, dt: torch.empty(n_, dtype=dt).pin_memory()) if mode == "pinned" else (lambda n_, dt: torch.empty(n_, dtype=dt))
        h_seeds = mk(nb * B, torch.int64); h_seeds.copy_(torch.from_numpy(seeds))
        ids = [mk(n1, torch.int64), mk(n2, torch.int64)]
        ws = [mk(n1, torch.float32), mk(n2, torch.float32)]
        ts = [mk(n1, torch.int32), mk(n2, torch.int32)]
        _lib.check(lib.eu_sample_fanout_batched_host(ctx._h, h_seeds.data_ptr(), nb, B, et.ctypes.data, 2, cs.ctypes.data, 2, -1,
                                                     P(*[x.data_ptr() for x in ids]), P(*[x.data_ptr() for x in ws]), P(*[x.data_ptr() for x in ts])))
        x = mk(n1 * 128, torch.float32)
        _lib.check(lib.eu_get_dense_feature_host(ctx._h, ids[0].data_ptr(), n1, 0, 128, x.data_ptr()))
        agg = mk(n1 * 128, torch.float32)
        _lib.check(lib.eu_sage_mean_aggregate_host(ctx._h, ids[1].data_ptr(), n1, 5, 128, agg.data_ptr()))
        outs[mode] = [t.clone().numpy() for t in ids + ws + ts + [x, agg]]
    for a, b in zip(outs["pinned"], outs["pageable"]):
        cases.eq(a, b, "pinned vs pageable host buffers")
    # device entry points, same engines
    ctx = euler_b200.Context(gr, "minstd", 99)
    ctx.set_engines(nb, [500 + b for b in range(nb)])
    d_seeds = torch.from_numpy(seeds).cuda()
    d_ids = [torch.empty(n1, dtype=torch.int64, device="cuda"), torch.empty(n2, dtype=torch.int64, device="cuda")]
    d_ws = [torch.empty(n1, dtype=torch.float32, device="cuda"), torch.empty(n2, dtype=torch.float32, device="cuda")]
    d_ts = [torch.empty(n1, dtype=torch.int32, device="cuda"), torch.empty(n2, dtype=torch.int32, device="cuda")]
    _lib.check(lib.eu_sample_fanout_batched(ctx._h, d_seeds.data_ptr(), nb, B, et.ctypes.data, 2, cs.ctypes.data, 2, -1,
                                            P(*[x.data_ptr() for x in d_ids]), P(*[x.data_ptr() for x in d_ws]), P(*[x.data_ptr() for x in d_ts])))
    d_agg = torch.empty(n1 * 128, dtype=torch.float32, device="cuda")
    _lib.check(lib.eu_sage_mean_aggregate(ctx._h, d_ids[1].data_ptr(), n1, 5, 128, d_agg.data_ptr()))
    ctx.sync()
    cases.eq(outs["pinned"][0], d_ids[0].cpu().numpy(), "host vs device ids hop 1")
    cases.eq(outs["pinned"][1], d_ids[1].cpu().numpy(), "host vs device ids hop 2")
    cases.eq(outs["pinned"][7], d_agg.cpu().numpy(), "host vs device sage mean")


def test_fanout_with_zero_count_leaves_the_dedup_tables_clean():
    """counts = [5, 0]: the chain stops before the empty hop; the next op on the same ctx still matches the oracle"""
    import euler_b200
    g = graphs.random_graph(seed=78, n=3000, T=1, avg_deg=5)
    euler_b200.set_graph(graphs.cuda_graph(g), rng="minstd", seed=31)
    og = graphs.oracle_graph(g)
    seeds = g["ids"][np.random.RandomState(1).randint(0, 3000, size=200)].astype(np.int64)
    po.seed(31)
    ids, ws, ts = euler_b200.sample_fanout(seeds, [[0], [0]], [5, 0])
    o_ids, _, _ = og.op_sample_fanout(seeds, [[0]], [5])
    cases.eq(ids[1].cpu().numpy(), o_ids[0], "hop 1 of [5, 0]")
    assert ids[2].numel() == 0
    ids2, _, _ = euler_b200.sample_fanout(seeds, [[0], [0]], [4, 3])
    o2, _, _ = og.op_sample_fanout(seeds, [[0], [0]], [4, 3])
    cases.eq(ids2[2].cpu().numpy(), o2[1], "fanout after a zero-count call")


def test_sample_node_on_a_loaded_graph_follows_the_reference_map_order(tiny_dir):
    """eu_graph_load replays the reference's node_map_ insert sequence into the same std::unordered_map, so the global node
    sampler enumerates nodes in the reference's order: sample_node on Graph.load(dir) == the reference's own SampleNode on the
    same directory under the same seed (tests/golden/ref_checks.npz), all three type modes (graph.cc:221-275,333-370)."""
    import euler_b200
    gr = euler_b200.Graph.load(tiny_dir)
    euler_b200.set_graph(gr, rng="minstd", seed=1)
    for i, (types, nt) in enumerate(mg.TINY_SAMPLE_NODE):
        for s in mg.TINY_SAMPLE_NODE_SEEDS:
            euler_b200.seed(s)
            got = euler_b200.sample_node(200, nt).cpu().numpy()
            cases.eq_ref(got, "tiny_sn%d_s%d" % (i, s), "sample_node types=%s seed=%d on the loaded graph" % (types, s))


# ------------------------------------------------------------------ next-1: sorted / top-k listings, gen_pair, raw api sampling
def test_sorted_and_topk_neighbors_reference_vectors_and_random_graph():
    """tiny graph: the reference's own expectations (tf_euler/python/euler_ops/neighbor_ops_test.py:73-110); random graph:
    stable sort by id / by weight descending of the oracle's full listing."""
    import euler_b200
    z = graphs.load_tiny_csr()
    euler_b200.set_graph(graphs.cuda_graph(z))
    ptr, ids, w, t = euler_b200.get_sorted_full_neighbor([1, 2], [0, 1])
    cases.eq(ptr.cpu().numpy(), np.array([0, 3, 5]), "sorted indptr")
    cases.eq(ids.cpu().numpy(), np.array([2, 3, 4, 3, 5]), "sorted ids (neighbor_ops_test.py:73-84)")
    assert np.allclose(w.cpu().numpy(), [2.0, 3.0, 4.0, 3.0, 5.0])
    cases.eq(t.cpu().numpy(), np.array([0, 1, 0, 1, 1], np.int32), "sorted types")
    k_ids, k_w, k_t = euler_b200.get_top_k_neighbor([1, 2], [0, 1], 2)
    cases.eq(k_ids.cpu().numpy(), np.array([[4, 3], [5, 3]]), "top-k ids (neighbor_ops_test.py:102-110)")
    assert np.allclose(k_w.cpu().numpy(), [[4.0, 3.0], [5.0, 3.0]])
    cases.eq(k_t.cpu().numpy(), np.array([[0, 1], [1, 1]], np.int32), "top-k types")
    g = graphs.random_graph(seed=301, n=3000, T=3, avg_deg=9, hub=700, dup_edges=True, empty_frac=0.1)
    euler_b200.set_graph(graphs.cuda_graph(g))
    og = graphs.oracle_graph(g)
    nodes = g["ids"][np.random.RandomState(2).randint(0, 3000, size=500)].astype(np.int64)
    nodes[::17] = 987654321
    for et in ([0, 2], [1], [2, 0, 1]):
        lens, f_ids, f_w, f_t = og.get_full_neighbor(nodes.astype(np.uint64), et)
        ptr, ids, w, t = euler_b200.get_sorted_full_neighbor(nodes, et)
        k_ids, k_w, k_t = euler_b200.get_top_k_neighbor(nodes, et, 7, default_node=-5)
        off = 0
        s_ids, s_w, s_t = [], [], []
        want_k = np.full((len(nodes), 7), -5, np.int64); want_kw = np.zeros((len(nodes), 7), np.float32); want_kt = np.full((len(nodes), 7), -1, np.int32)
        for i, n in enumerate(lens):
            sl = slice(off, off + n)
            o = np.argsort(f_ids[sl], kind="stable")
            s_ids.append(f_ids[sl][o]); s_w.append(f_w[sl][o]); s_t.append(f_t[sl][o])
            o2 = np.argsort(-f_w[sl], kind="stable")[:7]
            want_k[i, :len(o2)] = f_ids[sl][o2]; want_kw[i, :len(o2)] = f_w[sl][o2]; want_kt[i, :len(o2)] = f_t[sl][o2]
            off += n
        cases.eq(ptr.cpu().numpy(), np.concatenate([[0], np.cumsum(lens)]), "sorted indptr %s" % et)
        cases.eq(ids.cpu().numpy(), np.concatenate(s_ids).astype(np.int64), "sorted ids %s" % et)
        cases.eq(w.cpu().numpy(), np.concatenate(s_w), "sorted weights %s" % et)
        cases.eq(t.cpu().numpy(), np.concatenate(s_t), "sorted types %s" % et)
        cases.eq(k_ids.cpu().numpy(), want_k, "top-k ids %s" % et)
        cases.eq(k_w.cpu().numpy(), want_kw, "top-k weights %s" % et)
        cases.eq(k_t.cpu().numpy(), want_kt, "top-k types %s" % et)


@pytest.mark.parametrize("plen,lw,rw", [(6, 1, 1), (11, 2, 3), (5, 7, 0), (1, 2, 2), (81, 5, 5)])
def test_gen_pair_matches_the_reference_loop(plen, lw, rw):
    """literal restatement of tf_euler/kernels/gen_pair_op.cc:61-80 on the host vs the closed-form kernel"""
    import euler_b200
    g = graphs.random_graph(seed=5, n=50, T=1)
    euler_b200.set_graph(graphs.cuda_graph(g))
    paths = np.random.RandomState(plen).randint(1, 1000, size=(37, plen)).astype(np.int64)
    want = []
    for path in paths:
        row = []
        for j in range(plen):
            k = 0
            while j - k - 1 >= 0 and k < lw:
                row += [path[j], path[j - k - 1]]; k += 1
            k = 0
            while j + k + 1 < plen and k < rw:
                row += [path[j], path[j + k + 1]]; k += 1
        want.append(row)
    want = np.asarray(want, np.int64).reshape(37, -1, 2)
    got = euler_b200.gen_pair(paths, lw, rw).cpu().numpy()
    assert got.shape == want.shape, (got.shape, want.shape)
    cases.eq(got, want, "gen_pair")


def test_raw_api_sample_neighbor_draws_duplicates_independently():
    """eu_sample_neighbor_raw == euler::SampleNeighbor (api.cc:223-236) on the oracle: no unique, serial draw order"""
    import euler_b200
    for T, et in ((1, [0]), (3, [0, 2]), (3, [0, 1, 2])):
        g = graphs.random_graph(seed=410 + T, n=5000, T=T, avg_deg=8, hub=600, empty_frac=0.1, zero_w_frac=0.05)
        euler_b200.set_graph(graphs.cuda_graph(g), rng="minstd", seed=55)
        og = graphs.oracle_graph(g)
        nodes = g["ids"][np.random.RandomState(3).randint(0, 5000, size=2000)].astype(np.int64)
        nodes[::7] = nodes[0]
        nodes[5::31] = 424242424242
        rng = po.Rng(55)
        for rep in range(2):
            o_ids, o_w, o_t, o_len = og.sample_neighbor_api(nodes.astype(np.uint64), et, 6, rng)
            ids, w, t = euler_b200.sample_neighbor_api(nodes, et, 6)
            keep = (o_len > 0)[:, None]
            cases.eq(ids.cpu().numpy(), np.where(keep, o_ids.astype(np.int64), 0), "raw ids T=%d rep=%d" % (T, rep))
            cases.eq(w.cpu().numpy(), np.where(keep, o_w, 0).astype(np.float32), "raw weights")
            cases.eq(t.cpu().numpy(), np.where(keep, o_t, -1).astype(np.int32), "raw types")
        assert euler_b200.context().draws() == rng.draws


def test_sparse_and_binary_features_reference_test_vectors(tiny_dir):
    """the reference's own expectations on the tools/test_data graph (tf_euler/python/euler_ops/feature_ops_test.py:46-85):
    sparse f1 / f2 of nodes [1, -1, 2, 3, 4] and binary f5 / f6 of nodes [1, 2], through Graph.load of the converter's files"""
    import euler_b200
    gr = euler_b200.Graph.load(tiny_dir)
    euler_b200.set_graph(gr)
    sp = euler_b200.get_sparse_feature([1, -1, 2, 3, 4], ['f1', 'f2'], None, 2)
    want = [[[11, 12], [0, 0], [21, 22], [31, 32], [41, 42]], [[13, 14], [0, 0], [23, 24], [33, 34], [43, 44]]]
    for (idx, vals, shape), w in zip(sp, want):
        dense = np.zeros(shape, np.int64)
        i = idx.cpu().numpy()
        dense[i[:, 0], i[:, 1]] = vals.cpu().numpy()
        cases.eq(dense, np.asarray(w, np.int64), "sparse feature (dense view)")
        assert shape == (5, 2)
    # the absent node (-1) owns exactly one entry (1, 0) = default value
    idx, vals, _ = euler_b200.get_sparse_feature([1, -1], ['f1'], [77])[0]
    cases.eq(idx.cpu().numpy(), np.array([[0, 0], [0, 1], [1, 0]]), "sparse indices")
    cases.eq(vals.cpu().numpy(), np.array([11, 12, 77]), "sparse values with default")
    assert euler_b200.get_binary_feature([1, 2], ['f5', 'f6'], 3) == [[b'1a', b'2a'], [b'1b', b'2b']]
    assert euler_b200.get_binary_feature([99, 1], ['graph_label', 'nope']) == [[b'', b'1'], [b'', b'']]
    # unknown sparse feature: every node gets the default entry
    idx, vals, shape = euler_b200.get_sparse_feature([1, 2], ['nope'], [5])[0]
    cases.eq(vals.cpu().numpy(), np.array([5, 5]), "unknown sparse feature")


# ------------------------------------------------------------------ next-4: edge sampling and edge features
def test_edge_features_reference_test_vectors_and_sample_edge(tiny_dir):
    """edge features: the reference's own expectations (tf_euler/python/euler_ops/feature_ops_test.py:62-140);
    sample_edge: the reference's Graph::SampleEdge on the same directory under the same seed (tests/golden/ref_checks.npz;
    one type; several types return nothing upstream and are refused here)."""
    import euler_b200
    gr = euler_b200.Graph.load(tiny_dir)
    assert gr.num_edge_records == 12
    euler_b200.set_graph(gr, rng="minstd", seed=1)
    edges = [[1, 2, 0], [2, 3, 1]]
    sp = euler_b200.get_edge_sparse_feature(edges, ['f1', 'f2'], None)
    for (idx, vals, shape), want in zip(sp, ([[121, 122], [231, 232]], [[123, 124], [233, 234]])):
        dense = np.zeros(shape, np.int64)
        i = idx.cpu().numpy()
        dense[i[:, 0], i[:, 1]] = vals.cpu().numpy()
        cases.eq(dense, np.asarray(want, np.int64), "edge sparse feature")
    assert euler_b200.get_edge_binary_feature(edges, ['f5']) == [[b'12a', b'23a']]
    f3, f4 = euler_b200.get_edge_dense_feature(edges + [[9, 9, 0]], ["f3", "f4"], [2, 3], 2)
    assert np.allclose(f3.cpu().numpy(), [[12.1, 12.2], [23.1, 23.2], [0, 0]])
    assert np.allclose(f4.cpu().numpy(), [[12.3, 12.4, 12.5], [23.3, 23.4, 23.5], [0, 0, 0]])
    for t in (0, 1):
        for s in mg.TINY_SAMPLE_EDGE_SEEDS:
            euler_b200.seed(s)
            got = euler_b200.sample_edge(64, t).cpu().numpy()
            cases.eq_ref(got, "tiny_se%d_s%d" % (t, s), "sample_edge type %d seed %d" % (t, s))
            cases.eq_ref(euler_b200.context().draws(), "tiny_se%d_s%d_draws" % (t, s), "draws of sample_edge type %d seed %d" % (t, s))
    with pytest.raises(euler_b200.EulerError):
        euler_b200.sample_edge(4, [0, 1])


# ------------------------------------------------------------------ next-3: layerwise sampling and batch adjacency
@pytest.mark.parametrize("weight_func", ['', 'sqrt'])
def test_layerwise_sampling_candidates_distribution_and_adj(weight_func):
    """sample_neighbor_layerwise: the candidate set and every candidate's summed weight are the reference's
    (local_sample_layer_op.cc:66-101, restated here from the oracle's full-neighbor listing); the draws must stay inside the
    set, follow those weights (5-sigma band over 6000 draws per row), adj must equal membership exactly; rows without
    candidates are default-filled.  The reference's own tests check the same properties (neighbor_ops_test.py:142-181)."""
    import euler_b200
    g = graphs.random_graph(seed=640, n=300, T=2, avg_deg=5, dup_edges=True, empty_frac=0.2)
    euler_b200.set_graph(graphs.cuda_graph(g), rng="minstd", seed=3)
    og = graphs.oracle_graph(g)
    rs = np.random.RandomState(4)
    batch, n, count = 6, 4, 6000
    nodes = g["ids"][rs.randint(0, 300, size=(batch, n))].astype(np.int64)
    nodes[2, :] = 10 ** 12            # a row of absent nodes: no candidates
    nodes[3, 1] = nodes[3, 0]         # a repeated node: its edges count twice
    et = [0, 1]
    out, adj = euler_b200.sample_neighbor_layerwise(nodes, et, count, -7, weight_func)
    out, adj = out.cpu().numpy(), adj.cpu().numpy()
    lens, f_ids, f_w, f_t = og.get_full_neighbor(nodes.reshape(-1).astype(np.uint64), et)
    ptr = np.concatenate([[0], np.cumsum(lens)])
    for b in range(batch):
        lo, hi = ptr[b * n], ptr[(b + 1) * n]
        cand = {}
        for k in range(lo, hi):
            key = (int(f_ids[k]), int(f_t[k]))
            cand[key] = np.float32(cand.get(key, np.float32(0)) + f_w[k]) if key in cand else np.float32(f_w[k])
        if weight_func == 'sqrt':
            cand = {k: np.float32(np.sqrt(v)) for k, v in cand.items()}
        if not cand:
            assert (out[b] == -7).all() and (adj[b] == 0).all()
            continue
        by_dst = {}
        for (d, _), v in cand.items():
            by_dst[d] = by_dst.get(d, 0.0) + float(v)
        tot = sum(by_dst.values())
        vals, cnts = np.unique(out[b], return_counts=True)
        assert set(vals.tolist()) <= set(by_dst), "draws outside the candidate set"
        for d, c in zip(vals, cnts):
            p = by_dst[int(d)] / tot
            assert abs(c - count * p) <= 5 * np.sqrt(count * p * (1 - p)) + 3, (b, d, c, count * p)
        for j in range(n):
            nbrs = set(int(x) for x in f_ids[ptr[b * n + j]:ptr[b * n + j + 1]])
            want = np.array([1.0 if int(x) in nbrs else 0.0 for x in out[b]], np.float32)
            cases.eq(adj[b, j], want, "adj row")
    # sparse_get_adj: membership of given neighbor candidates
    nb = g["ids"][rs.randint(0, 300, size=(batch, 7))].astype(np.int64)
    nb[:, 0] = out[:, 0]
    a2 = euler_b200.sparse_get_adj(nodes.reshape(-1), nb.reshape(-1), et, n, 7).cpu().numpy()
    for b in range(batch):
        for j in range(n):
            nbrs = set(int(x) for x in f_ids[ptr[b * n + j]:ptr[b * n + j + 1]])
            cases.eq(a2[b, j], np.array([1.0 if int(x) in nbrs else 0.0 for x in nb[b]], np.float32), "sparse_get_adj row")


# ------------------------------------------------------------------ a-13: GCN / RGCN / SAGE aggregation blocks
@pytest.mark.parametrize("D", [64, 128])
def test_gcn_relation_and_sage_blocks_vs_literal_restatement(D):
    """euler_b200/convolution.py (GCNConv / RelationConv / SAGEConv message passing over the mp ops) against numpy
    restatements of gcn_conv.py:32-55, relation_conv.py:53-70, sage_conv.py:33-38 on a SageDataFlow-shaped block (sorted,
    fixed-fanout edge_src + appended self loops) and on an unsorted edge list; 1e-5 relative (north_star float tolerance)."""
    import euler_b200  # noqa: F401
    from euler_b200 import convolution as conv
    g = graphs.random_graph(seed=5, n=50, T=1)
    euler_b200.set_graph(graphs.cuda_graph(g))
    rs = np.random.RandomState(D)
    n0, n1, fan = 200, 700, 6
    src = np.repeat(np.arange(n0), fan)
    dst = rs.randint(0, n1, size=n0 * fan)
    loops = np.arange(n0)                                  # add_self_loops (neighbor_dataflow.py:98-100)
    blocks = {"sorted+self-loops": (np.concatenate([src, loops]), np.concatenate([dst, loops])),
              "unsorted": (rs.randint(0, n0, size=900), rs.randint(0, n1, size=900))}
    x1 = rs.randn(n1, D).astype(np.float32)
    R, dim = 5, 32
    mat = rs.randn(R, dim, D).astype(np.float32) * 0.1
    for name, (e0, e1) in blocks.items():
        ei = torch.from_numpy(np.stack([e0, e1])).cuda()
        X = torch.from_numpy(x1).cuda()
        # GCN
        deg0 = np.bincount(e0, minlength=n0).astype(np.float64)
        deg1 = np.bincount(e1, minlength=n1).astype(np.float64)
        with np.errstate(divide="ignore"):
            w = (deg0[e0] ** -0.5) * (deg1[e1] ** -0.5)
        want = np.zeros((n0, D), np.float64)
        np.add.at(want, e0, w[:, None] * x1[e1].astype(np.float64))
        got = conv.gcn_aggregate((None, X), ei, (n0, n1)).cpu().numpy()
        has = deg0 > 0
        assert np.allclose(got[has], want[has], rtol=RTOL, atol=1e-5), "gcn block " + name
        # SAGE mean
        s = np.zeros((n0, D), np.float64)
        np.add.at(s, e0, x1[e1].astype(np.float64))
        want = s / (deg0[:, None] + 1e-7)
        got = conv.sage_aggregate((None, X), ei, (n0, n1)).cpu().numpy()
        assert np.allclose(got, want, rtol=RTOL, atol=1e-5), "sage block " + name
        # Relation (RGCN): per-edge relation matrix, then mean
        attr = rs.randint(0, R, size=len(e0))
        msg = np.einsum("eij,ej->ei", mat[attr].astype(np.float64), x1[e1].astype(np.float64))
        s = np.zeros((n0, dim), np.float64)
        np.add.at(s, e0, msg)
        want = s / (deg0[:, None] + 1e-7)
        got = conv.relation_aggregate((None, X), ei, (n0, n1), torch.from_numpy(attr).cuda(), torch.from_numpy(mat).cuda()).cpu().numpy()
        assert np.allclose(got, want, rtol=1e-4, atol=1e-4), "relation block " + name


def test_fused_add_aggregate_equals_scatter_add_composition():
    """eu_sage_add_aggregate (aggr='add' over a fixed-fanout block, D = 64 of configs[4]) == get_dense_feature + scatter_add"""
    import euler_b200
    from euler_b200 import _lib
    g = graphs.random_graph(seed=77, n=3000, T=2, avg_deg=5, feat_dim=64)
    euler_b200.set_graph(graphs.cuda_graph(g))
    ids = g["ids"][np.random.RandomState(3).randint(0, 3000, size=512 * 10)].astype(np.int64)
    ids[::9] = -1
    d_ids = torch.from_numpy(ids).cuda()
    out = torch.empty((512, 64), dtype=torch.float32, device="cuda")
    ctx = euler_b200.context()
    _lib.check(_lib.load().eu_sage_add_aggregate(ctx._h, d_ids.data_ptr(), 512, 10, 64, out.data_ptr()))
    feat = euler_b200.get_dense_feature(d_ids, [0], [64])[0]
    want = euler_b200.scatter_add(feat, torch.arange(512, dtype=torch.int32, device="cuda").repeat_interleave(10), 512)
    cases.eq(out.cpu().numpy(), want.cpu().numpy(), "fused add aggregate")
