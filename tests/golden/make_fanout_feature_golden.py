"""Generates tests/golden/fanout_feature.npz from the REFERENCE ITSELF (oracle/_ref, as tests/golden/make_golden.py does):
sample_fanout_with_feature on the tiny graph -- the reference's fanout, then its Node feature getters on every level's
engine ids -- plus the tiny graph's uint64 slots as the reference's loader holds them.  Runs only where oracle/_ref has been
built and the reference sources are present (the uint64 accessor below is compiled against their headers):

    python tests/golden/make_fanout_feature_golden.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import pyoracle as po  # noqa: E402


# ---- fanout_feature.npz: sample_fanout_with_feature on the tiny graph.  (name, nodes, edge types, counts, default_node,
# dense names, dense dims, sparse names, sparse defaults); shared with tests/test_fanout_with_feature.py
FANOUT_FEATURE_CASES = [
    # neighbor_ops_test.py:203-217
    ("reftest", [1, 2, 0, 3], [[0, 1], [0, 1]], [3, 3], -1, ["f3", "f4"], [2, 3], ["f1", "f2"], [0, 0]),
    # default_node is a node with features: filled slots still get zeros / the sparse default
    ("defnode", [1, 2, 3, 4, 5, 6, 0, 99, 6], [[0, 1], [1, 0]], [4, 2], 5, ["f3", "f4"], [2, 3], ["f2", "f1"], [7, -3]),
    # requested widths above the stored ones: zero padding
    ("wide", [6, 5, 4, 3, 2, 1, 1], [[1], [0]], [2, 5], -1, ["f4", "f3"], [8, 5], ["f1"], [11]),
]
FANOUT_FEATURE_SEEDS = (3, 1234, 987654)

_SPARSE_HELPER = r"""
#include <stdint.h>
#include <string>
#include <vector>
#include "euler/core/api/api.h"
#include "euler/core/graph/graph.h"
extern "C" int32_t ref_feature_id(const char* name) { return euler::Graph::Instance().graph_meta().GetFeatureId(name); }
// euler::GetNodeUint64Feature (api.cc) for one slot: out_len[i] values of node i, back to back in out_vals (first cap)
extern "C" int64_t ref_get_sparse_feature(const uint64_t* ids, int64_t n, int32_t fid, int64_t cap, int64_t* out_len,
                                          uint64_t* out_vals) {
  euler::NodeIdVec v(ids, ids + n);
  auto res = euler::GetNodeUint64Feature(v, std::vector<int>(1, fid));
  int64_t tot = 0;
  for (int64_t i = 0; i < n; ++i) {
    out_len[i] = res[i].empty() ? 0 : (int64_t)res[i][0].size();
    for (int64_t k = 0; k < out_len[i]; ++k, ++tot) if (tot < cap) out_vals[tot] = res[i][0][k];
  }
  return tot;
}
"""


def sparse_helper():
    """ref_feature_id / ref_get_sparse_feature over the reference's GraphMeta and Node::GetUint64Feature, compiled against
    oracle/_ref/libeuler_ref.so (the graph singleton pyoracle.RefGraph loads)"""
    import ctypes as C
    import subprocess
    import tempfile
    po.ref()
    d = tempfile.mkdtemp()
    src, so = os.path.join(d, "sparse_helper.cc"), os.path.join(d, "libsparse_helper.so")
    with open(src, "w") as f:
        f.write(_SPARSE_HELPER)
    refdir = os.environ.get("REF", "/root/reference")
    subprocess.check_call(["g++", "-std=c++11", "-O2", "-fPIC", "-shared", "-include", "cstdint", "-include", "stdexcept",
                           "-D_GLIBCXX_USE_CXX11_ABI=0", "-I" + refdir, "-I" + os.path.join(refdir, "third_party"), "-w",
                           src, "-o", so, po.REF_SO])
    H = C.CDLL(so)
    H.ref_feature_id.restype = C.c_int32
    H.ref_feature_id.argtypes = [C.c_char_p]
    H.ref_get_sparse_feature.restype = C.c_int64
    H.ref_get_sparse_feature.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p]
    return H


def ref_sparse(H, ids, fid):
    """(lens, values) of slot fid for ids, as the reference's Node getter returns them"""
    ids = np.ascontiguousarray(ids, np.uint64)
    n = len(ids)
    lens = np.zeros(n, np.int64)
    tot = H.ref_get_sparse_feature(ids.ctypes.data, n, fid, 0, lens.ctypes.data, None)
    vals = np.zeros(max(tot, 1), np.uint64)
    H.ref_get_sparse_feature(ids.ctypes.data, n, fid, tot, lens.ctypes.data, vals.ctypes.data)
    return lens, vals[:tot]


def write_fanout_feature():
    out = {}
    tiny = os.path.join(HERE, "tiny_euler")
    g = po.RefGraph.load(tiny, "node", "node")
    H = sparse_helper()
    ids = np.sort(g.node_ids_in_map_order())
    # the graph's uint64 slots, rows in tiny_csr.npz order: slot k of row r = u64_val[u64_ptr[r*S+k] : u64_ptr[r*S+k+1]]
    names = ["f1", "f2"]
    S = len(names)
    per = [ref_sparse(H, ids, H.ref_feature_id(("sparse_" + nm).encode())) for nm in names]
    lens = np.stack([p[0] for p in per], axis=1).reshape(-1)
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    vals = []
    offs = [np.concatenate([[0], np.cumsum(p[0])]) for p in per]
    for r in range(len(ids)):
        for k in range(S):
            vals.append(per[k][1][offs[k][r]:offs[k][r + 1]])
    out["u64_names"] = np.asarray(names, "S")
    out["u64_ptr"], out["u64_val"] = ptr, np.concatenate(vals).astype(np.uint64)
    for name, nodes, ets, counts, dflt, dn, dd, sn, sd in FANOUT_FEATURE_CASES:
        for seed in FANOUT_FEATURE_SEEDS:
            key = "%s_s%d_" % (name, seed)
            g.seed(seed)
            f_ids, f_w, f_t = g.op_sample_fanout(np.asarray(nodes, np.int64), ets, counts, dflt)
            out[key + "draws"] = g.draws()
            levels = [np.asarray(nodes, np.int64).astype(np.uint64)]
            for l in range(len(counts)):
                out[key + "ids%d" % l], out[key + "w%d" % l], out[key + "t%d" % l] = f_ids[l], f_w[l], f_t[l]
                levels.append(np.where(f_t[l] == -1, 0, f_ids[l]).astype(np.uint64))   # engine ids: 0 where default-filled
            for i, lv in enumerate(levels):
                for j, (nm, dim) in enumerate(zip(dn, dd)):
                    out[key + "dense%d_%d" % (i, j)] = g.get_dense_feature(lv, H.ref_feature_id(("dense_" + nm).encode()), dim)[0]
                for j, (nm, dv) in enumerate(zip(sn, sd)):
                    ln, vl = ref_sparse(H, lv, H.ref_feature_id(("sparse_" + nm).encode()))
                    # the op's SparseTensor (sample_fanout_with_feature_op.cc:238-257): a row without values gets (k, 0) = default
                    rows = [vl[o:o + n].astype(np.int64) if n else np.asarray([dv], np.int64)
                            for o, n in zip(np.concatenate([[0], np.cumsum(ln)])[:-1], ln)]
                    out[key + "sp%d_%d_ptr" % (i, j)] = np.concatenate([[0], np.cumsum([len(x) for x in rows])]).astype(np.int64)
                    out[key + "sp%d_%d_val" % (i, j)] = np.concatenate(rows) if rows else np.zeros(0, np.int64)
    np.savez_compressed(os.path.join(HERE, "fanout_feature.npz"), **out)
    print("wrote", len(out), "arrays to fanout_feature.npz")


if __name__ == "__main__":
    write_fanout_feature()
