"""Generates the golden vectors under tests/golden/ from the REFERENCE ITSELF (oracle/_ref: the
unmodified reference sources + a seedable random.cc).  Runs only where oracle/_ref has been built,
i.e. where the reference sources were present at build time:

    oracle/tools/make_tiny_fixture.sh /tmp/euler      # reference converter -> .dat files
    python tests/golden/make_golden.py

Outputs (committed):
  tiny_euler/            the .dat/.meta files written by the reference converter
  tiny_csr.npz           that graph as loaded by the reference's Graph::Init, exported via the shim
  golden_ops.npz         outputs of the reference for seeded op calls on the tiny graph and on
                         seeded synthetic graphs (tests/graphs.py::random_graph)
  ref_checks.npz         the reference's side of the tests that compare the oracle or the product
                         with it (write_ref_checks), so that they run without the reference: one
                         sha256 digest per output (shape, dtype and every value), under its key
The reference's own deterministic test vectors for this path (mp_ops_test.py:30-94,
neighbor_ops_test.py:46-57, compact_weighted_collection_test.cc:43-55) are written out in
tests/test_oracle_golden.py directly.
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import pyoracle as po  # noqa: E402
import graphs  # noqa: E402

# (name, random_graph kwargs) -- regenerated identically by the tests
SYNTH = {
    "s1": dict(seed=11, n=300, T=1, avg_deg=5, feat_dim=8),
    "s3": dict(seed=12, n=200, T=3, avg_deg=4, n_node_types=2, zero_w_frac=0.1, id_stride=7, id_base=5),
    "s5": dict(seed=13, n=150, T=5, avg_deg=3, n_node_types=3, empty_frac=0.3, hub=200),
}
NB_CASES = [([0], 10), ([1], 4), ([0, 1], 5), ([], 3), ([1, 0], 40), ([7], 2)]


def seeds_for(g, rs, n):
    ids = g["ids"]
    s = ids[rs.randint(0, len(ids), size=n)].astype(np.int64)
    s[::7] = 10 ** 9 + 7  # absent id
    s[1::11] = 0
    return s


# ---- ref_checks.npz: the reference's side of the tests that compare with it.  The cases below are shared with those tests
UNIFORM_SEEDS = (1, 12345, 0, 2147483647, 1758564000)
UNIFORM_DRAWS = 50000
RANDOM_OPS = [(1, 1, {}), (2, 2, dict(zero_w_frac=0.2)), (3, 4, dict(hub=300, id_stride=13)),
              (4, 6, dict(empty_frac=0.5, n_node_types=3))]
FEAT_GRAPH = dict(seed=9, n=200, T=3, avg_deg=4, feat_dim=12)
FULL_NEIGHBOR_ETS = ([0], [2, 0], [1, 1], [5])
TINY_SAMPLE_NODE = (([0], 0), ([1], 1), ([-1], '-1'), ([0, 1], [0, 1]))   # (reference's types, euler_b200's node_type argument)
TINY_SAMPLE_NODE_SEEDS, TINY_SAMPLE_EDGE_SEEDS = (77, 12345), (5, 777)


def digest(a):
    """sha256 of an array's shape, dtype and bytes (integers as int64): pins an output with 32 bytes of golden data"""
    a = np.asarray(a)
    if a.dtype.kind in "iu":
        a = a.astype(np.int64)
    h = hashlib.sha256(repr((a.shape, a.dtype.str)).encode())
    h.update(np.ascontiguousarray(a).tobytes())
    return h.digest()


def uniform_stream(uniform):
    return np.fromiter((uniform() for _ in range(UNIFORM_DRAWS)), np.float64, UNIFORM_DRAWS)


def random_ops_graph(seed, T, kw):
    return graphs.random_graph(seed=seed, n=400, T=T, avg_deg=5, **kw)


def random_ops(be, g, seed):
    """The seeded op calls of test_oracle_vs_ref.py::test_random_graph_ops on backend `be` (the reference's RefGraph or
    tests/cases.py::OracleBackend) -> {name: output}"""
    T = g["T"]
    out = {}
    rs = np.random.RandomState(seed)
    seeds = g["ids"][rs.randint(0, len(g["ids"]), size=300)].astype(np.int64)
    seeds[::9] = 12345678901
    for ci, (et, cnt) in enumerate([([0], 7), (list(range(T)), 20), ([T - 1, 0], 5), ([], 2), ([0, 0], 3)]):
        be.seed(seed)
        for k, x in zip(("ids", "w", "t"), be.op_sample_neighbor(seeds, et, cnt, -7)):
            out["nb%d_%s" % (ci, k)] = x
        out["nb%d_draws" % ci] = be.draws()
    be.seed(seed + 1)
    for k, xs in zip(("ids", "w", "t"), be.op_sample_fanout(seeds, [[0, T - 1], [0, T - 1], [T - 1, 0]], [4, 3, 2], -1)):
        for l in range(3):
            out["fan%d_%s" % (l, k)] = xs[l]
    wet = np.asarray([list(range(T))] * 10, np.int32)
    for i, (p, q) in enumerate([(0.5, 2.0), (1.0, 1.0), (4.0, 0.25), (1.0, 2.0)]):
        be.seed(seed + 2)
        out["walk%d" % i] = be.op_random_walk(seeds[:100], wet, p, q, -1)
    for i, types in enumerate(([-1], [0], list(range(g["n_node_types"])))):
        be.seed(seed + 3)
        out["sn%d" % i] = be.sample_node(types, 300)
    for t in range(g["n_node_types"]):
        for k, x in zip(("ids", "w", "prob", "alias"), be.sampler_tables(t)):
            out["tables%d_%s" % (t, k)] = x
    return out


def full_neighbor_ids(g):
    return np.concatenate([g["ids"][:50], [999999]]).astype(np.uint64)


def alias_weights():
    """the weight vectors of test_abi.py::test_alias_tables_match_the_reference_on_the_host"""
    rng = np.random.RandomState(11)
    for _ in range(300):
        n = int(rng.randint(1, 400))
        w = (rng.randint(0, 1000, size=n) / np.float32(7)).astype(np.float32)
        w[rng.rand(n) < 0.2] = 0
        if w.sum() == 0:
            w[0] = 1
        yield w


def write_ref_checks():
    import ctypes as C
    out, sums = {}, {}

    def put(key, x):
        sums[key] = digest(x)
    R = po.ref()
    for s in UNIFORM_SEEDS:
        R.ref_seed(s)
        put("uniform%d" % s, uniform_stream(R.ref_uniform))
    # the committed fixture through the reference's own loader: global node sampler, then global edge sampler
    tiny = os.path.join(HERE, "tiny_euler")
    g = po.RefGraph.load(tiny)
    for i, (types, _) in enumerate(TINY_SAMPLE_NODE):
        for s in TINY_SAMPLE_NODE_SEEDS:
            g.seed(s)
            put("tiny_sn%d_s%d" % (i, s), g.sample_node(types, 200))
    g = po.RefGraph.load(tiny, "all", "all")
    for t in (0, 1):
        for s in TINY_SAMPLE_EDGE_SEEDS:
            g.seed(s)
            put("tiny_se%d_s%d" % (t, s), g.sample_edge([t], 64))
            put("tiny_se%d_s%d_draws" % (t, s), g.draws())
    for seed, T, kw in RANDOM_OPS:
        g = random_ops_graph(seed, T, kw)
        rg = graphs.ref_graph(g)
        out["rops%d_map_order" % seed] = rg.node_ids_in_map_order()     # an input of the replay: always in full
        for k, x in random_ops(rg, g, seed).items():
            put("rops%d_%s" % (seed, k), x)
    g = graphs.random_graph(**FEAT_GRAPH)
    rg = graphs.ref_graph(g)
    ids = full_neighbor_ids(g)
    put("feat", rg.get_dense_feature(ids, 0, FEAT_GRAPH["feat_dim"])[0])
    for i, et in enumerate(FULL_NEIGHBOR_ETS):
        for k, x in zip(("lens", "ids", "w", "t"), rg.get_full_neighbor(ids, et)):
            put("full%d_%s" % (i, k), x)
    # AliasMethod::Init on the weights FastWeightedCollection normalised with the f32 sum (the oracle's, equal to the product's)
    for rep, w in enumerate(alias_weights()):
        n = len(w)
        p2, a2, s2 = np.empty(n, np.float32), np.empty(n, np.int64), C.c_float(0)
        po.lib().eo_fwc_build(w, n, p2, a2, C.byref(s2))
        p3, a3 = np.empty(n, np.float32), np.empty(n, np.int64)
        R.ref_alias_build((w / np.float32(s2.value)).astype(np.float32), n, p3, a3)
        put("alias%d_prob" % rep, p3)
        put("alias%d_alias" % rep, a3)
    out["keys"] = np.asarray(list(sums), "S")
    out["sha256"] = np.frombuffer(b"".join(sums.values()), np.uint8).reshape(len(sums), 32)
    np.savez_compressed(os.path.join(HERE, "ref_checks.npz"), **out)
    print("wrote", len(sums), "digests to ref_checks.npz")


def main():
    out = {}
    # ---- tiny graph through the reference loader
    tiny = os.path.join(HERE, "tiny_euler")
    g = po.RefGraph.load(tiny, "node", "node")
    csr = g.export_csr()
    n = len(csr["ids"])
    dims = [2, 3]  # dense_f3, dense_f4 (euler.meta)
    feat = np.zeros((n, sum(dims)), np.float32)
    for r in range(n):
        ends, vals = csr["f32_ends"][r], csr["f32_vals"][r]
        off = 0
        for s, d in enumerate(dims):
            b = 0 if s == 0 else ends[s - 1]
            feat[r, off:off + min(d, ends[s] - b)] = vals[b:b + min(d, ends[s] - b)]
            off += d
    map_order = g.node_ids_in_map_order()
    np.savez(os.path.join(HERE, "tiny_csr.npz"), ids=csr["ids"], node_type=csr["node_type"],
             node_w=csr["node_w"], T=csr["T"], grp_ptr=csr["grp_ptr"], nbr=csr["nbr"],
             cum_w=csr["cum_w"], grp_cum=csr["grp_cum"], feat=feat, feat_slot_dims=np.asarray(dims, np.int32),
             n_node_types=2, map_order=map_order)
    tiny_seeds = np.asarray([1, 2, 3, 4, 5, 6, 7, 3, 1, 0, 6, 6], np.int64)
    out["tiny_seeds"] = tiny_seeds
    for ci, (et, cnt) in enumerate(NB_CASES):
        g.seed(100 + ci)
        ids, w, t = g.op_sample_neighbor(tiny_seeds, et, cnt, -1)
        out["tiny_nb%d_ids" % ci], out["tiny_nb%d_w" % ci], out["tiny_nb%d_t" % ci] = ids, w, t
        out["tiny_nb%d_draws" % ci] = g.draws()
    g.seed(200)
    ids, ws, ts = g.op_sample_fanout(tiny_seeds, [[0, 1], [0, 1]], [3, 4], -1)
    for l in range(2):
        out["tiny_fan%d_ids" % l], out["tiny_fan%d_w" % l], out["tiny_fan%d_t" % l] = ids[l], ws[l], ts[l]
    g.seed(300)
    out["tiny_walk_n2v"] = g.op_random_walk(tiny_seeds, np.asarray([[0, 1]] * 6, np.int32), 0.5, 2.0, -1)
    g.seed(301)
    out["tiny_walk_uni"] = g.op_random_walk(tiny_seeds, np.asarray([[0, 1]] * 6, np.int32), 1.0, 1.0, -1)
    for t in (0, 1):
        sid, sw, prob, alias = g.sampler_tables(t)
        out["tiny_sampler%d_ids" % t], out["tiny_sampler%d_prob" % t], out["tiny_sampler%d_alias" % t] = sid, prob, alias
    g.seed(400)
    out["tiny_sn_t0"] = g.sample_node([0], 64)
    g.seed(401)
    out["tiny_sn_all"] = g.sample_node([-1], 64)
    g.seed(402)
    out["tiny_sn_01"] = g.sample_node([0, 1], 64)
    f, lens = g.get_dense_feature(np.asarray([1, 9, 4], np.uint64), 1, 3)
    out["tiny_feat_f4"] = f

    # ---- seeded synthetic graphs through Node::Init
    for name, kw in SYNTH.items():
        sg = graphs.random_graph(**kw)
        rg = graphs.ref_graph(sg)
        rs = np.random.RandomState(kw["seed"] + 1000)
        seeds = seeds_for(sg, rs, 257)
        out[name + "_seeds"] = seeds
        T = sg["T"]
        cases = [([0], 10), (list(range(T)), 25), ([T - 1], 3)] + ([([0, T - 1], 7), ([1, 0], 33)] if T > 2 else [])
        out[name + "_ncases"] = len(cases)
        for ci, (et, cnt) in enumerate(cases):
            rg.seed(500 + ci)
            ids, w, t = rg.op_sample_neighbor(seeds, et, cnt, -1)
            out["%s_nb%d_et" % (name, ci)] = np.asarray(et, np.int32)
            out["%s_nb%d_cnt" % (name, ci)] = cnt
            out["%s_nb%d_ids" % (name, ci)], out["%s_nb%d_w" % (name, ci)], out["%s_nb%d_t" % (name, ci)] = ids, w, t
            out["%s_nb%d_draws" % (name, ci)] = rg.draws()
        rg.seed(600)
        ets = [[0]] * 2 if T == 1 else [[0, T - 1], [T - 1, 0]]
        ids, ws, ts = rg.op_sample_fanout(seeds, ets, [5, 3], -1)
        out[name + "_fan_et"] = np.asarray(ets, np.int32)
        for l in range(2):
            out["%s_fan%d_ids" % (name, l)], out["%s_fan%d_w" % (name, l)], out["%s_fan%d_t" % (name, l)] = ids[l], ws[l], ts[l]
        rg.seed(700)
        wet = np.asarray([list(range(T))] * 8, np.int32)
        out[name + "_walk_n2v"] = rg.op_random_walk(seeds[:64], wet, 0.5, 2.0, -1)
        rg.seed(701)
        out[name + "_walk_uni"] = rg.op_random_walk(seeds[:64], wet, 1.0, 1.0, -1)
        out[name + "_map_order"] = rg.node_ids_in_map_order()
        rg.seed(800)
        out[name + "_sn_all"] = rg.sample_node([-1], 500)
        rg.seed(801)
        out[name + "_sn_t0"] = rg.sample_node([0], 500)
    np.savez_compressed(os.path.join(HERE, "golden_ops.npz"), **out)
    print("wrote", len(out), "arrays")
    write_ref_checks()


if __name__ == "__main__":
    main()
