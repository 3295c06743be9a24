"""Backend-agnostic replay of the golden cases (tests/golden/golden_ops.npz, written from the
reference itself by tests/golden/make_golden.py).  A backend provides seed(), op_sample_neighbor(),
op_sample_fanout(), op_random_walk(), sample_node(), draws() with the oracle's signatures."""
import os

import numpy as np

import graphs
from golden.make_golden import NB_CASES, SYNTH, digest  # noqa: F401

_G = None
_REF = None


def golden():
    global _G
    if _G is None:
        _G = np.load(os.path.join(graphs.GOLDEN, "golden_ops.npz"))
    return _G


def ref_checks():
    """tests/golden/ref_checks.npz: the reference's outputs (as digests) and the map orders of the random graphs"""
    global _REF
    if _REF is None:
        z = np.load(os.path.join(graphs.GOLDEN, "ref_checks.npz"))
        _REF = {k: z[k] for k in z.files}
        _REF["digests"] = {k.decode(): v.tobytes() for k, v in zip(z["keys"], z["sha256"])}
    return _REF


def eq_ref(got, key, what):
    """`got` is bit for bit what the reference returned for `key` (same shape, dtype and values; integers of any width)"""
    assert digest(got) == ref_checks()["digests"][key], "%s: differs from the reference's output" % what


def eq(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, "%s: shape %s vs %s" % (what, a.shape, b.shape)
    if a.dtype.kind == "f":
        same = a.view(np.uint32) == b.view(np.uint32)  # bit-exact, also for -0.0
    else:
        same = a == b
    assert same.all(), "%s: %d / %d mismatches, first at %s: %s vs %s" % (
        what, (~same).sum(), same.size, np.argwhere(~same)[0], a[~same][:4], b[~same][:4])


def replay_tiny(be):
    G = golden()
    seeds = G["tiny_seeds"]
    for ci, (et, cnt) in enumerate(NB_CASES):
        be.seed(100 + ci)
        ids, w, t = be.op_sample_neighbor(seeds, et, cnt, -1)
        eq(ids, G["tiny_nb%d_ids" % ci], "tiny nb%d ids" % ci)
        eq(w, G["tiny_nb%d_w" % ci], "tiny nb%d w" % ci)
        eq(t, G["tiny_nb%d_t" % ci], "tiny nb%d t" % ci)
        assert be.draws() == int(G["tiny_nb%d_draws" % ci]), "tiny nb%d draws" % ci
    be.seed(200)
    ids, ws, ts = be.op_sample_fanout(seeds, [[0, 1], [0, 1]], [3, 4], -1)
    for l in range(2):
        eq(ids[l], G["tiny_fan%d_ids" % l], "tiny fanout ids hop %d" % l)
        eq(ws[l], G["tiny_fan%d_w" % l], "tiny fanout w hop %d" % l)
        eq(ts[l], G["tiny_fan%d_t" % l], "tiny fanout t hop %d" % l)
    be.seed(300)
    eq(be.op_random_walk(seeds, np.asarray([[0, 1]] * 6, np.int32), 0.5, 2.0, -1), G["tiny_walk_n2v"], "tiny node2vec")
    be.seed(301)
    eq(be.op_random_walk(seeds, np.asarray([[0, 1]] * 6, np.int32), 1.0, 1.0, -1), G["tiny_walk_uni"], "tiny walk p=q=1")
    be.seed(400)
    eq(be.sample_node([0], 64), G["tiny_sn_t0"], "tiny sample_node type 0")
    be.seed(401)
    eq(be.sample_node([-1], 64), G["tiny_sn_all"], "tiny sample_node all")
    be.seed(402)
    eq(be.sample_node([0, 1], 64), G["tiny_sn_01"], "tiny sample_node [0,1]")


def replay_synth(name, be):
    G = golden()
    seeds = G[name + "_seeds"]
    for ci in range(int(G[name + "_ncases"])):
        et, cnt = G["%s_nb%d_et" % (name, ci)], int(G["%s_nb%d_cnt" % (name, ci)])
        be.seed(500 + ci)
        ids, w, t = be.op_sample_neighbor(seeds, et, cnt, -1)
        eq(ids, G["%s_nb%d_ids" % (name, ci)], "%s nb%d ids" % (name, ci))
        eq(w, G["%s_nb%d_w" % (name, ci)], "%s nb%d w" % (name, ci))
        eq(t, G["%s_nb%d_t" % (name, ci)], "%s nb%d t" % (name, ci))
        assert be.draws() == int(G["%s_nb%d_draws" % (name, ci)]), "%s nb%d draws" % (name, ci)
    be.seed(600)
    ids, ws, ts = be.op_sample_fanout(seeds, G[name + "_fan_et"], [5, 3], -1)
    for l in range(2):
        eq(ids[l], G["%s_fan%d_ids" % (name, l)], "%s fanout ids hop %d" % (name, l))
        eq(ws[l], G["%s_fan%d_w" % (name, l)], "%s fanout w hop %d" % (name, l))
        eq(ts[l], G["%s_fan%d_t" % (name, l)], "%s fanout t hop %d" % (name, l))
    T = SYNTH[name].get("T", 1)
    wet = np.asarray([list(range(T))] * 8, np.int32)
    be.seed(700)
    eq(be.op_random_walk(seeds[:64], wet, 0.5, 2.0, -1), G[name + "_walk_n2v"], name + " node2vec")
    be.seed(701)
    eq(be.op_random_walk(seeds[:64], wet, 1.0, 1.0, -1), G[name + "_walk_uni"], name + " walk p=q=1")
    be.seed(800)
    eq(be.sample_node([-1], 500), G[name + "_sn_all"], name + " sample_node all")
    be.seed(801)
    eq(be.sample_node([0], 500), G[name + "_sn_t0"], name + " sample_node type 0")


def rows_in_order(g, id_order):
    """rows of g["ids"] in the given id order (the reference's unordered_map iteration order)."""
    pos = {int(i): r for r, i in enumerate(g["ids"])}
    return np.asarray([pos[int(i)] for i in id_order], np.int64)


class OracleBackend:
    """The C restatement (oracle/euler_oracle.c) behind the op-level signatures."""

    def __init__(self, g, map_order):
        from oracle import pyoracle as po
        self.po = po
        self.og = graphs.oracle_graph(g)
        self.og.build_node_sampler(rows_in_order(g, map_order), g["n_node_types"])
        self._rng = None

    def seed(self, s):
        self.po.seed(s)
        self._rng = self.po.Rng(s)
        self._sn = 0

    def draws(self):
        return self.po.draws()

    def op_sample_neighbor(self, *a):
        return self.og.op_sample_neighbor(*a)

    def op_sample_fanout(self, *a):
        return self.og.op_sample_fanout(*a)

    def op_random_walk(self, *a):
        return self.og.op_random_walk(*a)

    def sample_node(self, types, count):
        return self.og.sample_node(types, count, self._rng)

    def sampler_tables(self, t):
        return self.og.node_sampler_tables(t)


class CudaBackend:
    """The product, through the Python mirror of tf_euler's op API (euler_b200.ops -> C ABI)."""

    def __init__(self, g, map_order, raw_weights=False):
        import euler_b200
        self.eb = euler_b200
        self.graph = graphs.cuda_graph(g, raw_weights=raw_weights, sampler_order=rows_in_order(g, map_order))
        euler_b200.set_graph(self.graph, rng="minstd", seed=1)

    def seed(self, s):
        self.eb.seed(s)

    def draws(self):
        return self.eb.context().draws()

    def op_sample_neighbor(self, seeds, et, cnt, dn):
        return tuple(x.cpu().numpy() for x in self.eb.sample_neighbor(seeds, et, cnt, dn))

    def op_sample_fanout(self, seeds, ets, counts, dn):
        ids, ws, ts = self.eb.sample_fanout(seeds, list(ets), counts, dn)
        f = lambda xs: [x.cpu().numpy() for x in xs]  # noqa: E731
        return f(ids[1:]), f(ws), f(ts)

    def op_random_walk(self, seeds, wet, p, q, dn):
        return self.eb.random_walk(seeds, list(wet), p, q, dn).cpu().numpy()

    def sample_node(self, types, count):
        t = '-1' if list(types) == [-1] else list(types)
        return self.eb.sample_node(count, t).cpu().numpy().astype(np.uint64)
