"""sample_fanout_with_feature: the sample_fanout chain plus the dense and uint64 features of every level in one device op.

The oracle is the C restatement's fanout (oracle/) followed by a numpy lookup of every level's ENGINE ids (0 where a slot was
default-filled) in the graph's slot arrays.  tests/golden/fanout_feature.npz holds what the reference itself returns for the
tiny graph (tests/golden/make_fanout_feature_golden.py); the CPU test pins the oracle to it, the GPU tests hold the
product to both."""
import ctypes as C
import os

import numpy as np
import pytest

import graphs
from oracle import pyoracle as po

GOLDEN = os.path.join(graphs.GOLDEN, "fanout_feature.npz")
# (name, nodes, edge types, counts, default_node, dense names, dense dims, sparse names, sparse defaults): the cases of
# tests/golden/make_fanout_feature_golden.py::FANOUT_FEATURE_CASES, over FANOUT_FEATURE_SEEDS
CASES = [
    ("reftest", [1, 2, 0, 3], [[0, 1], [0, 1]], [3, 3], -1, ["f3", "f4"], [2, 3], ["f1", "f2"], [0, 0]),
    ("defnode", [1, 2, 3, 4, 5, 6, 0, 99, 6], [[0, 1], [1, 0]], [4, 2], 5, ["f3", "f4"], [2, 3], ["f2", "f1"], [7, -3]),
    ("wide", [6, 5, 4, 3, 2, 1, 1], [[1], [0]], [2, 5], -1, ["f4", "f3"], [8, 5], ["f1"], [11]),
]
SEEDS = (3, 1234, 987654)


def golden():
    return np.load(GOLDEN)


# ----------------------------------------------------------------------------------------------- the oracle
class Slots:
    """A graph's feature slots as numpy arrays: dense[k] f32[n, stored width], uint64 slot k of row r =
    u64_val[u64_ptr[r*S+k] : u64_ptr[r*S+k+1]]"""

    def __init__(self, ids, dense, u64_ptr, u64_val, n_u64):
        self.row = {int(i): r for r, i in enumerate(ids)}
        self.dense, self.u64_ptr, self.u64_val, self.S = dense, u64_ptr, u64_val, n_u64

    def rows(self, ids):
        return np.asarray([self.row.get(int(i), -1) for i in np.asarray(ids, np.uint64)], np.int64)

    def get_dense(self, ids, fid, dim):
        out = np.zeros((len(ids), dim), np.float32)
        if 0 <= fid < len(self.dense):
            w = min(dim, self.dense[fid].shape[1])
            r = self.rows(ids)
            out[r >= 0, :w] = self.dense[fid][r[r >= 0], :w]
        return out

    def get_sparse(self, ids, fid, default):
        """CSR (ptr, values), a row without values owns one default entry"""
        vals = []
        for r in self.rows(ids):
            v = np.zeros(0, np.int64)
            if r >= 0 and 0 <= fid < self.S:
                v = self.u64_val[self.u64_ptr[r * self.S + fid]:self.u64_ptr[r * self.S + fid + 1]].astype(np.int64)
            vals.append(v if len(v) else np.asarray([default], np.int64))
        ptr = np.concatenate([[0], np.cumsum([len(v) for v in vals])]).astype(np.int64)
        return ptr, (np.concatenate(vals) if vals else np.zeros(0, np.int64))


def oracle_fanout_feature(og, slots, seed, nodes, ets, counts, dflt, dfids, ddims, sfids, sdefs):
    po.seed(seed)
    ids, ws, ts = og.op_sample_fanout(np.asarray(nodes, np.int64), np.asarray(ets, np.int32), counts, dflt)
    draws = po.draws()
    levels = [np.asarray(nodes, np.int64).astype(np.uint64)] + [np.where(t == -1, 0, i).astype(np.uint64) for i, t in zip(ids, ts)]
    dense = [slots.get_dense(lv, f, d) for lv in levels for f, d in zip(dfids, ddims)]
    sparse = [slots.get_sparse(lv, f, v) for lv in levels for f, v in zip(sfids, sdefs)]
    return ids, ws, ts, draws, dense, sparse


def tiny_slots():
    g, z = graphs.load_tiny_csr(), golden()
    dims = list(g["feat_slot_dims"])
    offs = np.concatenate([[0], np.cumsum(dims)])
    dense = [g["feat"][:, offs[k]:offs[k + 1]] for k in range(len(dims))]
    return g, Slots(g["ids"], dense, z["u64_ptr"], z["u64_val"], len(z["u64_names"]))


TINY_DENSE, TINY_SPARSE = {"f3": 0, "f4": 1}, {"f1": 0, "f2": 1}   # slot order of tiny_csr.npz / u64_names


def eq(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a, b), "%s: %s vs %s" % (what, a, b)


def check_against_golden(z, key, ids, ws, ts, draws, dense, sparse, L, ND, NS):
    assert draws == int(z[key + "draws"]), key + "draws"
    for l in range(L):
        eq(ids[l], z[key + "ids%d" % l], key + "ids%d" % l)
        eq(ws[l], z[key + "w%d" % l], key + "w%d" % l)
        eq(ts[l], z[key + "t%d" % l], key + "t%d" % l)
    for i in range(L + 1):
        for j in range(ND):
            eq(dense[i * ND + j], z[key + "dense%d_%d" % (i, j)], key + "dense%d_%d" % (i, j))
        for j in range(NS):
            eq(sparse[i * NS + j][0], z[key + "sp%d_%d_ptr" % (i, j)], key + "sp%d_%d_ptr" % (i, j))
            eq(sparse[i * NS + j][1], z[key + "sp%d_%d_val" % (i, j)], key + "sp%d_%d_val" % (i, j))


def test_oracle_reproduces_the_reference_golden():
    g, slots = tiny_slots()
    og = graphs.oracle_graph(g)
    z = golden()
    for name, nodes, ets, counts, dflt, dn, dd, sn, sd in CASES:
        for seed in SEEDS:
            out = oracle_fanout_feature(og, slots, seed, nodes, ets, counts, dflt, [TINY_DENSE[n] for n in dn], dd,
                                        [TINY_SPARSE[n] for n in sn], sd)
            check_against_golden(z, "%s_s%d_" % (name, seed), *out, len(counts), len(dn), len(sn))


# ----------------------------------------------------------------------------------------------- GPU
def to_csr(sp):
    """(indices, values, dense_shape) -> (ptr, values) as numpy"""
    idx, vals, shape = sp
    n = shape[0]
    lens = np.bincount(idx[:, 0].cpu().numpy(), minlength=n) if n else np.zeros(0, np.int64)
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    cols = idx[:, 1].cpu().numpy()
    assert np.array_equal(cols, np.arange(len(cols)) - ptr[:-1][idx[:, 0].cpu().numpy()]), "column indices"
    assert shape[1] == (int(lens.max()) if n else 0), "dense_shape"
    return ptr, vals.cpu().numpy()


def run_op(nodes, ets, counts, dflt, dn, dd, sn, sd):
    import euler_b200
    nb, ws, ts, dense, sparse = euler_b200.sample_fanout_with_feature(nodes, ets, counts, dflt, dn, dd, sn, sd)
    draws = euler_b200.context().draws()
    return ([x.cpu().numpy() for x in nb[1:]], [x.cpu().numpy() for x in ws], [x.cpu().numpy() for x in ts], draws,
            [x.cpu().numpy() for x in dense], [to_csr(s) for s in sparse])


@pytest.mark.gpu
def test_reference_golden_on_the_tiny_graph(tiny_dir):
    import euler_b200
    z = golden()
    euler_b200.set_graph(euler_b200.Graph.load(tiny_dir), rng="minstd", seed=1)
    for name, nodes, ets, counts, dflt, dn, dd, sn, sd in CASES:
        for seed in SEEDS:
            euler_b200.seed(seed)
            out = run_op(nodes, [[str(t) for t in e] for e in ets], counts, dflt, dn, dd, sn, sd)
            check_against_golden(z, "%s_s%d_" % (name, seed), *out, len(counts), len(dn), len(sn))


@pytest.mark.gpu
def test_sparse_feature_max_len_on_the_tiny_graph(tiny_dir):
    import euler_b200
    from euler_b200 import _lib
    z = golden()
    gr = euler_b200.Graph.load(tiny_dir)
    S = len(z["u64_names"])
    lens = np.diff(z["u64_ptr"]).reshape(-1, S)
    for k, nm in enumerate(z["u64_names"]):
        assert _lib.load().eu_graph_sparse_feature_max_len(gr._h, gr.sparse_feature_id(nm.decode())) == lens[:, k].max()
    assert _lib.load().eu_graph_sparse_feature_max_len(gr._h, -1) == 0
    assert _lib.load().eu_graph_sparse_feature_max_len(gr._h, 1000) == 0


DENSE_WIDTHS = [3, 8, 5, 2, 4]      # stored widths of the random graphs' dense slots


def random_setup(seed, T, n=600):
    """a random graph with dense slots DENSE_WIDTHS and 3 ragged uint64 slots (many empty rows), on the device and as Slots"""
    import euler_b200
    g = graphs.random_graph(seed=seed, n=n, T=T, avg_deg=5, hub=300, id_stride=3, id_base=2)
    rng = np.random.RandomState(seed + 7)
    feat = rng.uniform(-1, 1, size=(n, sum(DENSE_WIDTHS))).astype(np.float32)
    S = 3
    lens = rng.randint(0, 6, size=n * S)
    lens[rng.rand(n * S) < 0.3] = 0
    u64_ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    u64_val = rng.randint(1, 1 << 40, size=int(u64_ptr[-1])).astype(np.uint64)
    gr = euler_b200.Graph.from_csr(g["ids"], g["grp_ptr"], g["nbr"], n_edge_types=T, cum_w=g["cum_w"],
                                   grp_cum=g["grp_cum"] if T > 1 else None, node_type=g["node_type"], node_w=g["node_w"],
                                   n_node_types=g["n_node_types"], feat=feat, feat_slot_dims=DENSE_WIDTHS, u64_ptr=u64_ptr,
                                   u64_val=u64_val, n_u64_slots=S)
    offs = np.concatenate([[0], np.cumsum(DENSE_WIDTHS)])
    slots = Slots(g["ids"], [feat[:, offs[k]:offs[k + 1]] for k in range(len(DENSE_WIDTHS))], u64_ptr, u64_val, S)
    seeds = g["ids"][rng.randint(0, n, size=200)].astype(np.int64)
    seeds[::9] = 10 ** 9 + 7   # absent
    seeds[3::13] = 0
    return g, gr, slots, seeds


# slot 1 (width 8) fetched narrower (clipped), slot 2 (width 5) wider (zero padded), slot 0 at 3 (not a multiple of 4), an
# unknown slot (-1) gives zeros; sparse slot -1 gives only defaults
RANDOM_DENSE = ([0, 1, 2, 3, -1], [3, 4, 7, 2, 6])
RANDOM_SPARSE = ([0, 2, 1, -1], [0, -5, 99, 3])


@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 3])
def test_random_graphs_against_the_oracle(T):
    import euler_b200
    g, gr, slots, seeds = random_setup(40 + T, T)
    euler_b200.set_graph(gr, rng="minstd", seed=1)
    og = graphs.oracle_graph(g)
    for ci, counts in enumerate([[6], [4, 3], [3, 2, 2], [5, 0, 3], [25, 10]]):
        L = len(counts)
        ets = [[0] if T == 1 else [0, T - 1]] * L
        dfids, ddims = RANDOM_DENSE if ci != 4 else (RANDOM_DENSE[0][:2], RANDOM_DENSE[1][:2])
        sfids, sdefs = RANDOM_SPARSE
        s = 100 + ci
        euler_b200.seed(s)
        got = run_op(seeds, ets, counts, -1 if ci % 2 else int(g["ids"][5]), dfids, ddims, sfids, sdefs)
        want = oracle_fanout_feature(og, slots, s, seeds, ets, counts, -1 if ci % 2 else int(g["ids"][5]), dfids, ddims,
                                     sfids, sdefs)
        assert got[3] == want[3], "draws"
        for what, a, b in zip(("ids", "w", "t"), got[:3], want[:3]):
            for l in range(L):
                eq(a[l], b[l], "case %d %s%d" % (ci, what, l))
        for k, (a, b) in enumerate(zip(got[4], want[4])):
            eq(a, b, "case %d dense %d" % (ci, k))
        for k, (a, b) in enumerate(zip(got[5], want[5])):
            eq(a[0], b[0], "case %d sparse ptr %d" % (ci, k))
            eq(a[1], b[1], "case %d sparse values %d" % (ci, k))
        if 0 in counts:   # a count-0 hop ends the chain: every later level is empty
            z = counts.index(0)
            for l in range(z + 1, L + 1):
                assert all(x.shape[0] == 0 for x in got[4][l * len(dfids):(l + 1) * len(dfids)])


@pytest.mark.gpu
def test_same_draws_as_sample_fanout():
    import euler_b200
    g, gr, slots, seeds = random_setup(51, 3)
    euler_b200.set_graph(gr, rng="minstd", seed=1)
    ets, counts = [[0, 2], [2, 1]], [5, 4]
    euler_b200.seed(77)
    a_ids, a_w, a_t = euler_b200.sample_fanout(seeds, ets, counts, default_node=-3)
    a_draws = euler_b200.context().draws()
    euler_b200.seed(77)
    b_ids, b_w, b_t, _, _ = euler_b200.sample_fanout_with_feature(seeds, ets, counts, -3, [0], [4], [1], [0])
    assert euler_b200.context().draws() == a_draws
    for l in range(len(counts)):
        assert np.array_equal(a_ids[l + 1].cpu().numpy(), b_ids[l + 1].cpu().numpy())
        assert np.array_equal(a_w[l].cpu().numpy().view(np.uint32), b_w[l].cpu().numpy().view(np.uint32))
        assert np.array_equal(a_t[l].cpu().numpy(), b_t[l].cpu().numpy())


@pytest.mark.gpu
def test_default_filled_slots_get_no_features_even_when_default_node_exists():
    """The op fetches features of the ENGINE ids (v_select(nb_i)); the composition sample_fanout + get_dense_feature on the
    TF-packed ids fetches default_node's own features instead.  Both are asserted: the difference is deliberate."""
    import euler_b200
    g, gr, slots, seeds = random_setup(52, 1)
    euler_b200.set_graph(gr, rng="minstd", seed=1)
    dn = int(g["ids"][5])
    euler_b200.seed(5)
    nb, ws, ts, dense, sparse = euler_b200.sample_fanout_with_feature(seeds, [[0]], [4], dn, [1], [8], [0], [-9])
    t = ts[0].cpu().numpy()
    filled = t == -1
    assert filled.any() and (nb[1].cpu().numpy()[filled] == dn).all()
    d = dense[1].cpu().numpy()
    assert (d[filled] == 0).all()
    ptr, vals = to_csr(sparse[1])
    assert all(ptr[k + 1] - ptr[k] == 1 and vals[ptr[k]] == -9 for k in np.nonzero(filled)[0])
    own = euler_b200.get_dense_feature(nb[1], [1], [8])[0].cpu().numpy()
    assert np.array_equal(own[filled], np.repeat(slots.get_dense([dn], 1, 8), filled.sum(), axis=0))
    assert (own[filled] != 0).any()
    assert np.array_equal(own[~filled], d[~filled])


def _alloc(rows, ddims, maxlens, dev):
    import torch
    ids = [torch.empty(r, dtype=torch.int64, device=dev) for r in rows[1:]]
    ws = [torch.empty(r, dtype=torch.float32, device=dev) for r in rows[1:]]
    ts = [torch.empty(r, dtype=torch.int32, device=dev) for r in rows[1:]]
    dense = [torch.empty((r, d), dtype=torch.float32, device=dev) for r in rows for d in ddims]
    ptr = [torch.empty(r + 1, dtype=torch.int64, device=dev) for r in rows for _ in maxlens]
    val = [torch.empty(r * m, dtype=torch.int64, device=dev) for r in rows for m in maxlens]
    return ids, ws, ts, dense, ptr, val


def _ptrs(xs):
    return (C.c_void_p * max(len(xs), 1))(*[x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data for x in xs])


class Call:
    """the C entry points with explicit output buffers on one Context"""

    def __init__(self, gr, seeds, ets, counts, dfids, ddims, sfids, sdefs, dflt=-1):
        from euler_b200 import _lib
        self.lib = _lib.load()
        self.gr, self.seeds, self.counts = gr, np.ascontiguousarray(seeds, np.int64), np.asarray(counts, np.int32)
        self.et = np.ascontiguousarray(ets, np.int32)
        self.dfids, self.ddims = np.asarray(dfids, np.int32), np.asarray(ddims, np.int32)
        self.sfids, self.sdefs = np.asarray(sfids, np.int32), np.asarray(sdefs, np.int64)
        self.dflt = dflt
        self.rows = [len(self.seeds)]
        for c in counts:
            self.rows.append(self.rows[-1] * c)
        self.maxlens = [max(1, self.lib.eu_graph_sparse_feature_max_len(gr._h, int(f))) for f in self.sfids]

    def args(self, ctx_h, nodes_ptr, bufs):
        ids, ws, ts, dense, ptr, val = bufs
        return (ctx_h, nodes_ptr, len(self.seeds), self.et.ctypes.data, self.et.shape[1], self.counts.ctypes.data, len(self.counts),
                self.dflt, _ptrs(ids), _ptrs(ws), _ptrs(ts), len(self.dfids), self.dfids.ctypes.data, self.ddims.ctypes.data,
                _ptrs(dense), len(self.sfids), self.sfids.ctypes.data, self.sdefs.ctypes.data, _ptrs(ptr), _ptrs(val))

    def device(self, ctx, bufs, nodes_t):
        from euler_b200._lib import check
        check(self.lib.eu_sample_fanout_with_feature(*self.args(ctx._h, nodes_t.data_ptr(), bufs)))

    def host(self, ctx):
        from euler_b200._lib import check
        ids = [np.zeros(r, np.int64) for r in self.rows[1:]]
        ws = [np.zeros(r, np.float32) for r in self.rows[1:]]
        ts = [np.zeros(r, np.int32) for r in self.rows[1:]]
        dense = [np.zeros((r, d), np.float32) for r in self.rows for d in self.ddims]
        ptr = [np.zeros(r + 1, np.int64) for r in self.rows for _ in self.maxlens]
        val = [np.zeros(r * m, np.int64) for r in self.rows for m in self.maxlens]
        check(self.lib.eu_sample_fanout_with_feature_host(*self.args(ctx._h, self.seeds.ctypes.data, (ids, ws, ts, dense, ptr, val))))
        return ids, ws, ts, dense, ptr, val


def _np(bufs, sparse_cut=True):
    ids, ws, ts, dense, ptr, val = [[x.cpu().numpy() if hasattr(x, "cpu") else x for x in b] for b in bufs]
    if sparse_cut:
        val = [v[:p[-1]] for p, v in zip(ptr, val)]
    return ids, ws, ts, dense, ptr, val


def _same(a, b):
    for xa, xb in zip(a, b):
        for u, v in zip(xa, xb):
            assert u.shape == v.shape and np.array_equal(u.view(np.uint8) if u.dtype == np.float32 else u,
                                                         v.view(np.uint8) if v.dtype == np.float32 else v)


@pytest.mark.gpu
def test_host_and_device_entry_points_agree():
    import euler_b200
    import torch
    g, gr, slots, seeds = random_setup(53, 3)
    call = Call(gr, seeds, [[0, 2], [1, 2], [2, 0]], [3, 2, 3], *RANDOM_DENSE, *RANDOM_SPARSE, dflt=int(g["ids"][0]))
    ctx = euler_b200.Context(gr, "minstd", 9)
    dev = torch.device("cuda", 0)
    bufs = _alloc(call.rows, list(call.ddims), call.maxlens, dev)
    call.device(ctx, bufs, torch.as_tensor(call.seeds, device=dev))
    ctx.sync()
    d = _np(bufs)
    ctx.seed(9)
    h = _np(call.host(ctx))
    _same(d, h)


@pytest.mark.gpu
def test_launch_count_is_the_fanout_plus_one_dense_and_three_sparse():
    import euler_b200
    import torch
    from euler_b200 import _lib
    lib = _lib.load()
    g, gr, slots, seeds = random_setup(54, 3)
    euler_b200.set_graph(gr, rng="minstd", seed=1)
    ets, counts = [[0, 2], [2, 1]], [4, 3]
    for _ in range(2):   # the second round counts: scratch is sized
        n0 = lib.eu_launch_count()
        euler_b200.sample_fanout(seeds, ets, counts)
        n1 = lib.eu_launch_count()
        euler_b200.sample_fanout_with_feature(seeds, ets, counts, -1, [0, 2], [3, 7], [0, 1], [0, 0])
        n2 = lib.eu_launch_count()
    torch.cuda.synchronize()
    assert n2 - n1 == (n1 - n0) + 1 + 3, (n1 - n0, n2 - n1)


@pytest.mark.gpu
def test_cuda_graph_capture_replays_the_eager_call():
    import euler_b200
    import torch
    g, gr, slots, seeds = random_setup(55, 3)
    call = Call(gr, seeds, [[0, 2], [1, 2]], [5, 3], *RANDOM_DENSE, *RANDOM_SPARSE)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    ctx = euler_b200.Context(gr, "minstd", 1, stream=stream.cuda_stream)
    ctx.reserve(max(call.rows))
    nodes = torch.as_tensor(call.seeds, device=dev)
    bufs = _alloc(call.rows, list(call.ddims), call.maxlens, dev)
    with torch.cuda.stream(stream):
        call.device(ctx, bufs, nodes)   # warm call: sizes the remaining scratch
    ctx.sync()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=stream):
        call.device(ctx, bufs, nodes)
    ctx.seed(321)
    graph.replay()
    ctx.sync()
    replayed = _np(bufs)
    eager_bufs = _alloc(call.rows, list(call.ddims), call.maxlens, dev)
    ctx.seed(321)
    call.device(ctx, eager_bufs, nodes)
    ctx.sync()
    _same(replayed, _np(eager_bufs))
