"""CPU: the C-ABI library builds, loads, and exports every symbol include/euler_b200.h declares;
without a GPU it refuses to work instead of falling back."""
import ctypes as C
import os
import re

import pytest
import torch

import graphs  # noqa: F401  (sys.path)
from euler_b200 import _lib, build

HEADER = os.path.join(graphs.ROOT, "include", "euler_b200.h")


def _declared():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"\b((?:eu_[a-z0-9_]+|InitQueryProxy))\s*\(", src)
    return sorted(set(names) - {"eu_status", "eu_rng_kind"})


def test_library_builds_and_exports_header_symbols():
    build.build()
    lib = _lib.load()
    names = _declared()
    assert len(names) >= 45
    for n in names:
        assert hasattr(lib, n), "missing export " + n
        assert n in _lib.SIGNATURES, "python binding lacks " + n
    assert set(_lib.SIGNATURES) <= set(names), set(_lib.SIGNATURES) - set(names)
    assert b"sm_100a" in lib.eu_version()


def test_sass_is_sm100a():
    out = os.popen("cuobjdump -lelf %s 2>/dev/null" % _lib.SO_PATH).read()
    assert "sm_100a" in out


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_gpu_means_loud_failure_not_fallback():
    lib = _lib.load()
    h = C.c_void_p()
    rc = lib.eu_graph_create_rmat(100, 1000, 0.57, 0.19, 0.19, 42, 0, 7, 0, C.byref(h))
    assert rc == 3  # EU_ERR_NO_GPU
    assert b"no CPU fallback" in lib.eu_last_error()
    import euler_b200
    with pytest.raises(euler_b200.EulerError):
        euler_b200.Graph.rmat(100, 1000)
    with pytest.raises(euler_b200.EulerError):
        euler_b200.sample_neighbor([1], [0], 3)  # no graph initialised


def test_init_query_proxy_contract():
    # tf_euler/utils/init_query_proxy.cc:19-36: false only for an empty / malformed k=v list
    lib = _lib.load()
    assert lib.InitQueryProxy(b"") is False
    assert lib.InitQueryProxy(b"mode") is False
    assert lib.InitQueryProxy(b"a=b=c") is False
    assert lib.InitQueryProxy(b"mode=remote;zk_server=x") is True   # logged, not propagated (:34)
    import euler_b200
    with pytest.raises(TypeError):
        euler_b200.initialize_graph(42)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(graphs.ROOT, "euler_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "pyoracle" not in txt and "euler_oracle" not in txt and "libeuler_ref" not in txt, f


def test_cpp_api_adapter_compiles_and_links():
    """include/euler_b200_api.hpp (the reference's euler/core/api/api.h surface over the C ABI) compiles as C++11 and links
    against the shared library; with no GPU the program refuses to start (no CPU fallback)."""
    import shutil
    import subprocess
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib = os.path.join(root, "euler_b200", "lib")
    if shutil.which("g++") is None or not os.path.exists(os.path.join(lib, "libeuler_b200.so")):
        pytest.skip("g++ or the built library is missing")
    exe = os.path.join(tempfile.mkdtemp(), "api_adapter_main")
    subprocess.check_call(["g++", "-std=c++11", "-Wall", "-Werror", "-I" + os.path.join(root, "include"),
                           os.path.join(root, "tests", "cpp", "api_adapter_main.cc"), "-L" + lib, "-leuler_b200",
                           "-Wl,-rpath," + lib, "-o", exe])
    import torch
    if not torch.cuda.is_available():
        r = subprocess.run([exe, os.path.join(root, "tests", "golden", "tiny_euler")], capture_output=True, text=True)
        assert r.returncode != 0 and "no CPU fallback" in r.stderr


def test_alias_tables_match_the_reference_on_the_host():
    """eu_build_alias_table (host-only): the tables the global node / edge samplers are built from are bit-identical to the
    oracle's restatement of AliasMethod::Init / FastWeightedCollection::Init and to the reference's own AliasMethod
    (euler/common/alias_method.cc:23-63), as stored in tests/golden/ref_checks.npz."""
    import ctypes as C
    import numpy as np
    import cases
    from euler_b200 import _lib
    from golden import make_golden as mg
    from oracle import pyoracle as po
    lib = _lib.load()
    ol = po.lib()
    for rep, w in enumerate(mg.alias_weights()):
        n = len(w)
        prob, alias = np.empty(n, np.float32), np.empty(n, np.int32)
        s = C.c_float(0)
        assert lib.eu_build_alias_table(w.ctypes.data, n, prob.ctypes.data, alias.ctypes.data, C.addressof(s)) == 0
        p2, a2 = np.empty(n, np.float32), np.empty(n, np.int64)
        s2 = C.c_float(0)
        ol.eo_fwc_build(w, n, p2, a2, C.byref(s2))
        assert prob.tobytes() == p2.tobytes() and np.array_equal(alias, a2) and s.value == s2.value, rep
        # FastWeightedCollection normalises in f32 before AliasMethod: the reference's tables of w / sum
        cases.eq_ref(prob, "alias%d_prob" % rep, "prob of weight vector %d" % rep)
        cases.eq_ref(alias, "alias%d_alias" % rep, "alias of weight vector %d" % rep)


def test_loader_replays_the_reference_sampler_order_on_the_host():
    """eu_graph_load_inspect (host-only parse of an Euler 2.0 directory): node / edge counts of the converter's files and the
    global-sampler enumeration order == the reference's own loader on the same directory (its unordered_map<NodeID, Node*>
    iteration order, euler/core/graph/graph.cc:349-354), per node type, as stored in tests/golden/golden_ops.npz."""
    import ctypes as C
    import os
    import numpy as np
    import cases
    from euler_b200 import _lib
    lib = _lib.load()
    tiny = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "tiny_euler")
    nn, ne = C.c_int64(0), C.c_int64(0)
    T, NT = C.c_int32(0), C.c_int32(0)
    assert lib.eu_graph_load_inspect(tiny.encode(), 0, 1, C.addressof(nn), C.addressof(ne), C.addressof(T), C.addressof(NT), 0, None, None) == 0
    assert (nn.value, T.value, NT.value) == (6, 2, 2) and ne.value > 0       # the reference's 6-node test graph (tf_euler/python/euler_ops/testdata)
    ids, types = np.zeros(nn.value, np.int64), np.zeros(nn.value, np.int32)
    assert lib.eu_graph_load_inspect(tiny.encode(), 0, 1, None, None, None, None, nn.value, ids.ctypes.data, types.ctypes.data) == 0
    assert sorted(ids.tolist()) == [1, 2, 3, 4, 5, 6]
    # sharded load: shard s of 2 sees the partitions p with p % 2 == s (graph_builder.cc:230-246); together they see every node
    seen = []
    for s in range(2):
        n_s = C.c_int64(0)
        assert lib.eu_graph_load_inspect(tiny.encode(), s, 2, C.addressof(n_s), None, None, None, 0, None, None) == 0
        part = np.zeros(n_s.value, np.int64)
        lib.eu_graph_load_inspect(tiny.encode(), s, 2, None, None, None, None, n_s.value, part.ctypes.data, None)
        seen += part.tolist()
    assert sorted(seen) == [1, 2, 3, 4, 5, 6]
    assert lib.eu_graph_load_inspect(b"/nonexistent/dir", 0, 1, None, None, None, None, 0, None, None) != 0
    for t in range(NT.value):
        ref_ids = cases.golden()["tiny_sampler%d_ids" % t]       # the reference's sampler table of type t on this directory
        assert np.array_equal(ids[types == t].astype(np.uint64), ref_ids), (t, ids, types, ref_ids)


def test_gen_pair_count_is_the_reference_formula():
    """eu_gen_pair_count (host): pairs per path of tf_euler gen_pair (tf_euler/kernels/gen_pair_op.cc:41-60) == the number of
    (j, k) with k in [j - left, j + right] inside the path, k != j -- counted literally."""
    from euler_b200 import _lib
    lib = _lib.load()
    for plen in range(0, 12):
        for lw in range(0, 6):
            for rw in range(0, 6):
                want = sum(1 for j in range(plen) for k in range(j - lw, j + rw + 1) if k != j and 0 <= k < plen)
                assert lib.eu_gen_pair_count(plen, lw, rw) == want, (plen, lw, rw)
