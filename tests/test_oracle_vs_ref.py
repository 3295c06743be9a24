"""CPU: the C restatement against what the UNMODIFIED reference sources returned on fresh random graphs (not only the
committed golden cases), stored by tests/golden/make_golden.py::write_ref_checks in tests/golden/ref_checks.npz."""
import numpy as np
import pytest

import cases
import graphs
from golden import make_golden as mg
from oracle import pyoracle as po


def test_uniform_stream_bit_exact():
    for s in mg.UNIFORM_SEEDS:
        cases.eq_ref(mg.uniform_stream(po.Rng(s).uniform), "uniform%d" % s, "uniform stream of seed %d" % s)


@pytest.mark.skipif(not po.have_ref(), reason="checks the reference's own loader: needs oracle/_ref (the reference sources at build time)")
def test_reference_loader_reads_committed_fixture(tiny_dir):
    g = po.RefGraph.load(tiny_dir, "node", "node")
    csr = g.export_csr()
    z = graphs.load_tiny_csr()
    for k in ("ids", "node_type", "node_w", "grp_ptr", "nbr", "cum_w", "grp_cum"):
        assert np.array_equal(csr[k], z[k]), k
    assert np.array_equal(g.node_ids_in_map_order(), z["map_order"])


@pytest.mark.parametrize("seed,T,kw", mg.RANDOM_OPS)
def test_random_graph_ops(seed, T, kw):
    g = mg.random_ops_graph(seed, T, kw)
    be = cases.OracleBackend(g, cases.ref_checks()["rops%d_map_order" % seed])
    for k, x in mg.random_ops(be, g, seed).items():
        cases.eq_ref(x, "rops%d_%s" % (seed, k), "graph %d: %s" % (seed, k))


def test_dense_feature_and_full_neighbor():
    g = graphs.random_graph(**mg.FEAT_GRAPH)
    og = graphs.oracle_graph(g)
    ids = mg.full_neighbor_ids(g)
    cases.eq_ref(og.op_get_dense_feature(ids.astype(np.int64), mg.FEAT_GRAPH["feat_dim"]), "feat", "dense feature")
    for i, et in enumerate(mg.FULL_NEIGHBOR_ETS):
        for k, x in zip(("lens", "ids", "w", "t"), og.get_full_neighbor(ids, et)):
            cases.eq_ref(x, "full%d_%s" % (i, k), "full neighbor %s: %s" % (et, k))
