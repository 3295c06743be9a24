"""tf_euler's Python op API for the minibatch-construction path, over torch CUDA tensors.

Same names, argument meaning and error behaviour as the reference wrappers
(tf_euler/python/euler_ops/{base,neighbor_ops,walk_ops,sample_ops,feature_ops,mp_ops,type_ops}.py);
each function cites the wrapper it mirrors.  Tensors are torch tensors on the graph's device; every
op enqueues kernels from libeuler_b200.so on the current torch stream.  Nothing here computes on the
CPU and nothing falls back to PyTorch ops: if the library or the GPU is missing, calls raise.
"""
import ctypes as C
import threading

import numpy as np
import torch

from . import _lib
from ._lib import EulerError, check
from .graph import Context, Graph

_state = threading.local()
_default = {"graph": None, "rng": "minstd", "seed": 1}


# ------------------------------------------------------------------------------------ init
def initialize_graph(config):
    """base.initialize_graph (tf_euler/python/euler_ops/base.py:37-60): str or dict of k=v;
    TypeError otherwise.  Returns what InitQueryProxy returns."""
    if isinstance(config, dict):
        config = ';'.join('{}={}'.format(key, value) for key, value in config.items())
    if not isinstance(config, str):
        raise TypeError('Expect str or dict for graph config, got {}.'.format(type(config).__name__))
    lib = _lib.load()
    ok = bool(lib.InitQueryProxy(config.encode()))
    h = lib.eu_default_graph()
    if h:
        kv = dict(item.split('=') for item in config.split(';') if item)
        g = Graph(C.c_void_p(h), int(kv.get('device', 0)))
        g.close = lambda: None  # owned by the library's default slot
        set_graph(g, rng=kv.get('rng', 'minstd'), seed=int(kv.get('seed', 1)))
    return ok


def initialize_embedded_graph(data_dir, sampler_type='all', data_type='all'):
    """base.initialize_embedded_graph (base.py:63-67)."""
    return initialize_graph({'mode': 'local', 'data_path': data_dir, 'data_type': data_type,
                             'sampler_type': sampler_type})


def set_graph(graph, rng="minstd", seed=1):
    """Install an already-built Graph (synthetic / from arrays) as the process default."""
    _default.update(graph=graph, rng=rng, seed=seed)
    _state.__dict__.pop("ctx", None)


def get_graph():
    if _default["graph"] is None:
        raise EulerError("graph is not initialized: call initialize_graph / set_graph first")
    return _default["graph"]


def context():
    """Per-thread Context of the default graph (one engine per client thread, like
    euler/common/random.cc:22's thread_local engine)."""
    ctx = getattr(_state, "ctx", None)
    if ctx is None or ctx.graph is not _default["graph"]:
        ctx = Context(get_graph(), _default["rng"], _default["seed"])
        _state.ctx = ctx
        _state.stream = None    # a fresh Context is not bound to any torch stream yet
    return ctx


def seed(s):
    """Re-seed this thread's engine (the reference has no seed API; parity tests need one)."""
    context().seed(s)


def _dev():
    return torch.device("cuda", get_graph().device)


def _ctx_on_stream():
    """This thread's Context, bound to torch's current stream.  All ops of a Context share its scratch (dedup tables, engine
    state, staging), so when the current stream CHANGES the new stream is first ordered after everything the Context issued on
    the old one (an event, no host sync)."""
    ctx = context()
    cur = torch.cuda.current_stream(_dev())
    prev = getattr(_state, "stream", None)
    if prev is not None and prev.cuda_stream != cur.cuda_stream:
        ev = torch.cuda.Event()
        ev.record(prev)
        cur.wait_event(ev)
    if prev is None or prev.cuda_stream != cur.cuda_stream:
        ctx.set_stream(cur.cuda_stream)
        _state.stream = cur
    return ctx


def _t(x, dtype):
    if isinstance(x, torch.Tensor):
        return x.to(device=_dev(), dtype=dtype).contiguous()
    return torch.as_tensor(np.asarray(x), dtype=dtype, device=_dev()).contiguous()


def _i32_host(x):
    if isinstance(x, torch.Tensor):
        x = x.detach().cpu().numpy()
    return np.ascontiguousarray(np.asarray(x).reshape(-1), dtype=np.int32)


# ------------------------------------------------------------------------------------ type ops
def get_edge_type_id(type_id_or_names):
    """type_ops.get_edge_type_id (type_ops.py:57-68): names resolved through graph meta."""
    return _type_ids(type_id_or_names, get_graph().edge_type_id)


def get_node_type_id(type_id_or_names):
    """type_ops.get_node_type_id (type_ops.py:42-54)."""
    return _type_ids(type_id_or_names, get_graph().node_type_id)


def _type_ids(v, lookup):
    if isinstance(v, torch.Tensor):
        return _i32_host(v)
    arr = np.asarray(v).reshape(-1)
    if arr.dtype.kind in "US":
        return np.asarray([lookup(str(s)) for s in arr], np.int32)
    return arr.astype(np.int32)


# ------------------------------------------------------------------------------------ sampling
def sample_neighbor(nodes, edge_types, count, default_node=-1, condition=''):
    """neighbor_ops.sample_neighbor (neighbor_ops.py:39-41).  Returns (neighbors i64[B,count],
    weights f32[B,count], types i32[B,count])."""
    if condition:
        raise EulerError("sample_neighbor: `condition` (index queries) is outside this path")
    nodes = _t(nodes, torch.int64).reshape(-1)
    et = get_edge_type_id(edge_types)
    B = nodes.numel()
    ids = torch.empty((B, count), dtype=torch.int64, device=nodes.device)
    w = torch.empty((B, count), dtype=torch.float32, device=nodes.device)
    t = torch.empty((B, count), dtype=torch.int32, device=nodes.device)
    ctx = _ctx_on_stream()
    check(_lib.load().eu_sample_neighbor(ctx._h, nodes.data_ptr(), B, et.ctypes.data, len(et), count,
                                         default_node, ids.data_ptr(), w.data_ptr(), t.data_ptr()))
    return ids, w, t


def sample_fanout(nodes, edge_types, counts, default_node=-1):
    """neighbor_ops.sample_fanout (neighbor_ops.py:122-158).  edge_types: list (per hop) of 1-D
    type lists of equal length.  Returns (neighbors_list[L+1], weights_list[L], types_list[L]),
    all flattened like the reference."""
    nodes = _t(nodes, torch.int64).reshape(-1)
    L = len(counts)
    ets = [get_edge_type_id(e) for e in edge_types]
    if len(ets) != L or any(len(e) != len(ets[0]) for e in ets):
        raise EulerError("sample_fanout: edge_types must hold one equal-length type list per hop")
    et = np.ascontiguousarray(np.stack(ets) if L else np.zeros((0, 0)), dtype=np.int32)
    cs = np.ascontiguousarray(counts, dtype=np.int32)
    B = nodes.numel()
    ids, ws, ts, rows = [], [], [], B
    for c in counts:
        rows *= int(c)
        ids.append(torch.empty(rows, dtype=torch.int64, device=nodes.device))
        ws.append(torch.empty(rows, dtype=torch.float32, device=nodes.device))
        ts.append(torch.empty(rows, dtype=torch.int32, device=nodes.device))
    P = C.c_void_p * max(L, 1)
    ctx = _ctx_on_stream()
    check(_lib.load().eu_sample_fanout(ctx._h, nodes.data_ptr(), B, et.ctypes.data,
                                       et.shape[1] if L else 0, cs.ctypes.data, L, default_node,
                                       P(*[x.data_ptr() for x in ids]), P(*[x.data_ptr() for x in ws]),
                                       P(*[x.data_ptr() for x in ts])))
    return [nodes] + ids, ws, ts


def sample_fanout_with_feature(nodes, edge_types, count, default_node, dense_feature_names, dense_dimensions,
                               sparse_feature_names, sparse_default_values):
    """neighbor_ops.sample_fanout_with_feature (neighbor_ops.py:49-69; kernel sample_fanout_with_feature_op.cc).  sample_fanout
    (same draws) plus the features of every level: level 0 is `nodes`, level l the ids hop l drew, where a default-filled slot
    has no node and gets zeros / the sparse default whatever default_node is.  Returns (neighbors[L+1], weights[L], types[L],
    dense[(L+1)*ND], sparse[(L+1)*NS]), features level-major (level i, feature j at i*ND + j); each sparse entry is
    (indices i64[nnz, 2], values i64[nnz], dense_shape) as get_sparse_feature returns.  Names are looked up as "dense_"+name /
    "sparse_"+name; ints are slot ids."""
    nodes = _t(nodes, torch.int64).reshape(-1)
    L = len(count)
    ets = [get_edge_type_id(e) for e in edge_types]
    if len(ets) != L or any(len(e) != len(ets[0]) for e in ets):
        raise EulerError("sample_fanout_with_feature: edge_types must hold one equal-length type list per hop")
    if len(dense_feature_names) != len(dense_dimensions) or len(sparse_feature_names) != len(sparse_default_values):
        raise EulerError("sample_fanout_with_feature: one dimension per dense feature and one default per sparse feature")
    g, lib = get_graph(), _lib.load()
    et = np.ascontiguousarray(np.stack(ets) if L else np.zeros((0, 0)), dtype=np.int32)
    cs = np.ascontiguousarray(count, dtype=np.int32)
    dfid = np.asarray([n if isinstance(n, (int, np.integer)) else g.dense_feature_id(n) for n in dense_feature_names], np.int32)
    ddim = np.asarray([int(d) for d in dense_dimensions], np.int32)
    sfid = np.asarray([n if isinstance(n, (int, np.integer)) else g.sparse_feature_id(n) for n in sparse_feature_names], np.int32)
    sdef = np.asarray([int(v) for v in sparse_default_values], np.int64)
    dev = nodes.device
    rows = [nodes.numel()]
    for c in count:
        rows.append(rows[-1] * int(c))
    ids = [torch.empty(r, dtype=torch.int64, device=dev) for r in rows[1:]]
    ws = [torch.empty(r, dtype=torch.float32, device=dev) for r in rows[1:]]
    ts = [torch.empty(r, dtype=torch.int32, device=dev) for r in rows[1:]]
    dense = [torch.empty((r, int(d)), dtype=torch.float32, device=dev) for r in rows for d in ddim]
    maxlen = [max(1, lib.eu_graph_sparse_feature_max_len(g._h, int(f))) for f in sfid]
    sp_ptr = [torch.empty(r + 1, dtype=torch.int64, device=dev) for r in rows for _ in sfid]
    sp_val = [torch.empty(r * m, dtype=torch.int64, device=dev) for r in rows for m in maxlen]

    def P(ts_):
        return (C.c_void_p * max(len(ts_), 1))(*[x.data_ptr() for x in ts_])
    ctx = _ctx_on_stream()
    check(lib.eu_sample_fanout_with_feature(ctx._h, nodes.data_ptr(), rows[0], et.ctypes.data, et.shape[1] if L else 0,
                                            cs.ctypes.data, L, int(default_node), P(ids), P(ws), P(ts), len(dfid),
                                            dfid.ctypes.data, ddim.ctypes.data, P(dense), len(sfid), sfid.ctypes.data,
                                            sdef.ctypes.data, P(sp_ptr), P(sp_val)))
    sparse = []
    if sp_ptr:
        lens = [p[1:] - p[:-1] for p in sp_ptr]
        zero = torch.zeros(1, dtype=torch.int64, device=dev)
        # the one host sync: value counts (to cut the value arrays) and row maxima (dense_shape) of every feature
        sizes = torch.stack([torch.cat([p[-1:], n.max().reshape(1) if n.numel() else zero]) for p, n in zip(sp_ptr, lens)]).cpu().tolist()
        for indptr, vals, ln, (total, width) in zip(sp_ptr, sp_val, lens, sizes):
            n = ln.numel()
            r = torch.repeat_interleave(torch.arange(n, device=dev), ln, output_size=total)
            cols = torch.arange(total, device=dev) - indptr[:-1][r]
            sparse.append((torch.stack([r, cols], dim=1), vals[:total], (n, width)))
    return [nodes] + ids, ws, ts, dense, sparse


def sample_fanout_batched(nodes, edge_types, counts, default_node=-1, ctx=None):
    """nb independent sample_fanout calls in one set of kernel launches.  nodes: [nb, B]; batch b runs on engine b
    of `ctx` (Context.set_engines), i.e. it returns exactly what sample_fanout(nodes[b]) returns on a context
    seeded like engine b.  Returns (neighbors_list[L+1], weights_list[L], types_list[L]) with a leading nb dim."""
    nodes = _t(nodes, torch.int64)
    nb, B = nodes.shape
    L = len(counts)
    ets = [get_edge_type_id(e) for e in edge_types]
    et = np.ascontiguousarray(np.stack(ets) if L else np.zeros((0, 0)), dtype=np.int32)
    cs = np.ascontiguousarray(counts, dtype=np.int32)
    ids, ws, ts, rows = [], [], [], B
    for c in counts:
        rows *= int(c)
        ids.append(torch.empty((nb, rows), dtype=torch.int64, device=nodes.device))
        ws.append(torch.empty((nb, rows), dtype=torch.float32, device=nodes.device))
        ts.append(torch.empty((nb, rows), dtype=torch.int32, device=nodes.device))
    P = C.c_void_p * max(L, 1)
    ctx = ctx or _ctx_on_stream()
    check(_lib.load().eu_sample_fanout_batched(ctx._h, nodes.data_ptr(), nb, B, et.ctypes.data,
                                               et.shape[1] if L else 0, cs.ctypes.data, L, default_node,
                                               P(*[x.data_ptr() for x in ids]), P(*[x.data_ptr() for x in ws]),
                                               P(*[x.data_ptr() for x in ts])))
    return [nodes] + ids, ws, ts


def sample_node(count, node_type, condition=''):
    """sample_ops.sample_node (sample_ops.py:38-54); node_type '-1' (or -1) = all types."""
    if condition:
        raise EulerError("sample_node: `condition` (index queries) is outside this path")
    if isinstance(node_type, str) and node_type == '-1':
        types = np.asarray([-1], np.int32)
    else:
        types = get_node_type_id(node_type)
    count = int(count)
    out = torch.empty(count, dtype=torch.int64, device=_dev())
    ctx = _ctx_on_stream()
    check(_lib.load().eu_sample_node(ctx._h, count, types.ctypes.data, len(types), out.data_ptr()))
    return out


def random_walk(nodes, edge_types, p=1.0, q=1.0, default_node=-1):
    """walk_ops.random_walk (walk_ops.py:29-43).  edge_types: list of L 1-D type lists.
    Returns i64[B, L+1]."""
    nodes = _t(nodes, torch.int64).reshape(-1)
    ets = [get_edge_type_id(e) for e in edge_types]
    L = len(ets)
    if any(len(e) != len(ets[0]) for e in ets):
        raise EulerError("random_walk: every step needs the same number of edge types here")
    et = np.ascontiguousarray(np.stack(ets) if L else np.zeros((0, 0)), dtype=np.int32)
    B = nodes.numel()
    out = torch.empty((B, L + 1), dtype=torch.int64, device=nodes.device)
    ctx = _ctx_on_stream()
    check(_lib.load().eu_random_walk(ctx._h, nodes.data_ptr(), B, et.ctypes.data,
                                     et.shape[1] if L else 0, L, float(p), float(q), default_node,
                                     out.data_ptr()))
    return out


def get_dense_feature(nodes, feature_names, dimensions, thread_num=1):
    """feature_ops.get_dense_feature (feature_ops.py:111-125): list of f32[M, dim_i]; names are
    looked up as "dense_"+name in the graph meta (get_dense_feature_op.cc:83); ints are slot ids."""
    del thread_num  # the reference splits the batch over TF threads; one launch here
    nodes = _t(nodes, torch.int64).reshape(-1)
    g = get_graph()
    outs = []
    ctx = _ctx_on_stream()
    for name, dim in zip(feature_names, dimensions):
        fid = name if isinstance(name, (int, np.integer)) else g.dense_feature_id(name)
        out = torch.empty((nodes.numel(), int(dim)), dtype=torch.float32, device=nodes.device)
        check(_lib.load().eu_get_dense_feature(ctx._h, nodes.data_ptr(), nodes.numel(), int(fid),
                                               int(dim), out.data_ptr()))
        outs.append(out)
    return outs


def _ragged(fn, nodes, fid, *mid):
    """two-phase ragged fetch: lengths, then values"""
    nodes = _t(nodes, torch.int64).reshape(-1)
    n = nodes.numel()
    ctx = _ctx_on_stream()
    indptr = torch.empty(n + 1, dtype=torch.int64, device=nodes.device)
    check(fn(ctx._h, nodes.data_ptr(), n, int(fid), *mid, 0, indptr.data_ptr(), None))
    total = int(indptr[-1].item())
    return nodes, n, ctx, indptr, total


def get_sparse_feature(nodes, feature_names, default_values=None, thread_num=1):
    """feature_ops.get_sparse_feature (feature_ops.py:57-73; kernel get_sparse_feature_op.cc:52-130).  Per feature the
    reference returns a SparseTensor; here the same content as (indices i64[nnz, 2], values i64[nnz], dense_shape (N, max_len)):
    row i lists the uint64 values of the node, a node without values gets the single entry (i, 0) = default value."""
    g, lib = get_graph(), _lib.load()
    names = [str(x) for x in feature_names]
    defaults = [0] * len(names) if default_values is None else [int(x) for x in default_values]
    outs = []
    for name, dv in zip(names, defaults):
        fid = g.sparse_feature_id(name)
        nd, n, ctx, indptr, total = _ragged(lib.eu_get_sparse_feature, nodes, fid, dv)
        vals = torch.empty(total, dtype=torch.int64, device=nd.device)
        if total:
            check(lib.eu_get_sparse_feature(ctx._h, nd.data_ptr(), n, int(fid), dv, total, indptr.data_ptr(), vals.data_ptr()))
        lens = indptr[1:] - indptr[:-1]
        rows = torch.repeat_interleave(torch.arange(n, device=nd.device), lens)
        cols = torch.arange(total, device=nd.device) - indptr[:-1][rows]
        outs.append((torch.stack([rows, cols], dim=1), vals, (n, int(lens.max().item()) if n else 0)))
    return outs


def get_binary_feature(nodes, feature_names, thread_num=1):
    """feature_ops.get_binary_feature (feature_ops.py:158-171): per feature a list of N byte strings (b'' for absent nodes)."""
    g, lib = get_graph(), _lib.load()
    outs = []
    for name in [str(x) for x in feature_names]:
        fid = g.binary_feature_id(name)
        nd, n, ctx, indptr, total = _ragged(lib.eu_get_binary_feature, nodes, fid)
        buf = torch.empty(max(total, 1), dtype=torch.uint8, device=nd.device)
        if total:
            check(lib.eu_get_binary_feature(ctx._h, nd.data_ptr(), n, int(fid), total, indptr.data_ptr(), buf.data_ptr()))
        raw, ptr = bytes(buf[:total].cpu().numpy().tobytes()), indptr.cpu().tolist()
        outs.append([raw[ptr[i]:ptr[i + 1]] for i in range(n)])
    return outs


def sample_edge(count, edge_type):
    """sample_ops.sample_edge (tf_euler/python/euler_ops/sample_ops.py; kernel sample_edge_op.cc): i64[count, 3] rows of
    (src, dst, type), drawn by edge weight among the edges of ONE type (several types return nothing in the reference)."""
    types = get_edge_type_id(edge_type)
    count = int(count)
    out = torch.empty((count, 3), dtype=torch.int64, device=_dev())
    ctx = _ctx_on_stream()
    check(_lib.load().eu_sample_edge(ctx._h, count, types.ctypes.data, len(types), out.data_ptr()))
    return out


def _edges(edges):
    e = _t(edges, torch.int64)
    if e.dim() != 2 or e.shape[1] != 3:
        raise EulerError("edges must be a matrix with shape [n, 3]")
    return e.contiguous()


def get_edge_dense_feature(edges, feature_names, dimensions, thread_num=1):
    """feature_ops.get_edge_dense_feature: list of f32[E, dim] (zeros for unknown edges / features)"""
    e = _edges(edges)
    g, lib, outs = get_graph(), _lib.load(), []
    ctx = _ctx_on_stream()
    for name, dim in zip(feature_names, dimensions):
        out = torch.empty((e.shape[0], int(dim)), dtype=torch.float32, device=e.device)
        check(lib.eu_get_edge_dense_feature(ctx._h, e.data_ptr(), e.shape[0], g.edge_feature_id("dense", name), int(dim), out.data_ptr()))
        outs.append(out)
    return outs


def get_edge_sparse_feature(edges, feature_names, default_values=None, thread_num=1):
    """feature_ops.get_edge_sparse_feature: per feature (indices i64[nnz, 2], values i64[nnz], dense_shape)"""
    e = _edges(edges)
    g, lib, outs = get_graph(), _lib.load(), []
    names = [str(x) for x in feature_names]
    defaults = [0] * len(names) if default_values is None else [int(x) for x in default_values]
    ctx = _ctx_on_stream()
    n = e.shape[0]
    for name, dv in zip(names, defaults):
        fid = g.edge_feature_id("sparse", name)
        indptr = torch.empty(n + 1, dtype=torch.int64, device=e.device)
        check(lib.eu_get_edge_sparse_feature(ctx._h, e.data_ptr(), n, fid, dv, 0, indptr.data_ptr(), None))
        total = int(indptr[-1].item())
        vals = torch.empty(total, dtype=torch.int64, device=e.device)
        if total:
            check(lib.eu_get_edge_sparse_feature(ctx._h, e.data_ptr(), n, fid, dv, total, indptr.data_ptr(), vals.data_ptr()))
        lens = indptr[1:] - indptr[:-1]
        rows = torch.repeat_interleave(torch.arange(n, device=e.device), lens)
        cols = torch.arange(total, device=e.device) - indptr[:-1][rows]
        outs.append((torch.stack([rows, cols], dim=1), vals, (n, int(lens.max().item()) if n else 0)))
    return outs


def get_edge_binary_feature(edges, feature_names, thread_num=1):
    """feature_ops.get_edge_binary_feature: per feature a list of E byte strings"""
    e = _edges(edges)
    g, lib, outs = get_graph(), _lib.load(), []
    ctx = _ctx_on_stream()
    n = e.shape[0]
    for name in [str(x) for x in feature_names]:
        fid = g.edge_feature_id("binary", name)
        indptr = torch.empty(n + 1, dtype=torch.int64, device=e.device)
        check(lib.eu_get_edge_binary_feature(ctx._h, e.data_ptr(), n, fid, 0, indptr.data_ptr(), None))
        total = int(indptr[-1].item())
        buf = torch.empty(max(total, 1), dtype=torch.uint8, device=e.device)
        if total:
            check(lib.eu_get_edge_binary_feature(ctx._h, e.data_ptr(), n, fid, total, indptr.data_ptr(), buf.data_ptr()))
        raw, ptr = bytes(buf[:total].cpu().numpy().tobytes()), indptr.cpu().tolist()
        outs.append([raw[ptr[i]:ptr[i + 1]] for i in range(n)])
    return outs


def get_full_neighbor(nodes, edge_types):
    """neighbor_ops.get_full_neighbor (tf_euler/python/euler_ops/neighbor_ops.py; kernel get_full_neighbor_op.cc over
    euler::GetFullNeighbor api.cc:208-221).  The reference returns three SparseTensors [N, max_degree] (ids, weights,
    types) whose values are listed node by node; here the same values come back ragged: (indptr i64[N+1], ids i64[nnz],
    weights f32[nnz], types i32[nnz]) -- SparseTensor indices are (i, k - indptr[i]) for k in [indptr[i], indptr[i+1])."""
    nodes = _t(nodes, torch.int64).reshape(-1)
    et = np.ascontiguousarray(edge_types, dtype=np.int32).reshape(-1)
    ctx = _ctx_on_stream()
    lib = _lib.load()
    n = nodes.numel()
    indptr = torch.empty(n + 1, dtype=torch.int64, device=nodes.device)
    check(lib.eu_get_full_neighbor(ctx._h, nodes.data_ptr(), n, et.ctypes.data, len(et), 0, indptr.data_ptr(), None, None, None))
    total = int(indptr[-1].item())
    ids = torch.empty(total, dtype=torch.int64, device=nodes.device)
    w = torch.empty(total, dtype=torch.float32, device=nodes.device)
    t = torch.empty(total, dtype=torch.int32, device=nodes.device)
    if total:
        check(lib.eu_get_full_neighbor(ctx._h, nodes.data_ptr(), n, et.ctypes.data, len(et), total, indptr.data_ptr(),
                                       ids.data_ptr(), w.data_ptr(), t.data_ptr()))
    return indptr, ids, w, t


def get_sorted_full_neighbor(nodes, edge_types, condition=''):
    """neighbor_ops.get_sorted_full_neighbor (neighbor_ops.py:100-119): get_full_neighbor with every node's entries ordered by
    neighbor id; same ragged return."""
    if condition:
        raise EulerError("get_sorted_full_neighbor: `condition` (index queries) is outside this path")
    nodes = _t(nodes, torch.int64).reshape(-1)
    et = get_edge_type_id(edge_types)
    ctx = _ctx_on_stream()
    lib = _lib.load()
    n = nodes.numel()
    indptr = torch.empty(n + 1, dtype=torch.int64, device=nodes.device)
    check(lib.eu_get_sorted_full_neighbor(ctx._h, nodes.data_ptr(), n, et.ctypes.data, len(et), 0, indptr.data_ptr(), None, None, None))
    total = int(indptr[-1].item())
    ids = torch.empty(total, dtype=torch.int64, device=nodes.device)
    w = torch.empty(total, dtype=torch.float32, device=nodes.device)
    t = torch.empty(total, dtype=torch.int32, device=nodes.device)
    if total:
        check(lib.eu_get_sorted_full_neighbor(ctx._h, nodes.data_ptr(), n, et.ctypes.data, len(et), total, indptr.data_ptr(),
                                              ids.data_ptr(), w.data_ptr(), t.data_ptr()))
    return indptr, ids, w, t


def get_top_k_neighbor(nodes, edge_types, k, default_node=-1, condition=''):
    """neighbor_ops.get_top_k_neighbor (neighbor_ops.py:44-46): (ids i64[N,k], weights f32[N,k], types i32[N,k]), the k
    heaviest edges of each node, heaviest first, filled with default_node / 0 / -1."""
    if condition:
        raise EulerError("get_top_k_neighbor: `condition` (index queries) is outside this path")
    nodes = _t(nodes, torch.int64).reshape(-1)
    et = get_edge_type_id(edge_types)
    n, k = nodes.numel(), int(k)
    ids = torch.empty((n, k), dtype=torch.int64, device=nodes.device)
    w = torch.empty((n, k), dtype=torch.float32, device=nodes.device)
    t = torch.empty((n, k), dtype=torch.int32, device=nodes.device)
    ctx = _ctx_on_stream()
    check(_lib.load().eu_get_top_k_neighbor(ctx._h, nodes.data_ptr(), n, et.ctypes.data, len(et), k, default_node,
                                            ids.data_ptr(), w.data_ptr(), t.data_ptr()))
    return ids, w, t


def sample_neighbor_layerwise(nodes, edge_types, count, default_node=-1, weight_func=''):
    """neighbor_ops.sample_neighbor_layerwise (neighbor_ops.py:72-77): nodes [batch, n] -> (neighbors i64[batch, count],
    adj f32[batch, n, count]); adj is the dense view of the reference's SparseTensor (1.0 where neighbors[b, k] is a neighbor of
    nodes[b, j]).  weight_func: '' or 'sqrt'."""
    nd = _t(nodes, torch.int64)
    if nd.dim() != 2:
        raise EulerError("sample_neighbor_layerwise: nodes must be [batch, n]")
    if weight_func not in ('', 'sqrt'):
        raise EulerError("sample_neighbor_layerwise: weight_func must be '' or 'sqrt' (local_sample_layer_op.cc:93-101)")
    nd = nd.contiguous()
    batch, n = nd.shape
    et = get_edge_type_id(edge_types)
    out = torch.empty((batch, int(count)), dtype=torch.int64, device=nd.device)
    adj = torch.empty((batch, n, int(count)), dtype=torch.float32, device=nd.device)
    ctx = _ctx_on_stream()
    check(_lib.load().eu_sample_neighbor_layerwise(ctx._h, nd.data_ptr(), batch, n, et.ctypes.data, len(et), int(count), default_node,
                                                   1 if weight_func == 'sqrt' else 0, out.data_ptr(), adj.data_ptr()))
    return out, adj


def sparse_get_adj(nodes, nb_nodes, edge_types, n=-1, m=-1):
    """neighbor_ops.sparse_get_adj (neighbor_ops.py:33-36): nodes [batch * n], nb_nodes [batch * m] (n / m = -1: one batch row)
    -> f32[batch, n, m], the dense view of the reference's SparseTensor."""
    nd = _t(nodes, torch.int64).reshape(-1).contiguous()
    nb = _t(nb_nodes, torch.int64).reshape(-1).contiguous()
    N = nd.numel() if n == -1 else int(n)
    M = nb.numel() if m == -1 else int(m)
    batch = nd.numel() // max(N, 1)
    et = get_edge_type_id(edge_types)
    adj = torch.empty((batch, N, M), dtype=torch.float32, device=nd.device)
    ctx = _ctx_on_stream()
    check(_lib.load().eu_sparse_get_adj(ctx._h, nd.data_ptr(), nb.data_ptr(), batch, N, M, et.ctypes.data, len(et), adj.data_ptr()))
    return adj


def gen_pair(paths, left_win_size, right_win_size):
    """walk_ops.gen_pair (tf_euler/kernels/gen_pair_op.cc): skip-gram pairs i64[B, n_pairs, 2] of walks i64[B, path_len]."""
    paths = _t(paths, torch.int64)
    if paths.dim() != 2:
        raise EulerError("gen_pair: paths must be [batch, path_len]")
    paths = paths.contiguous()
    B, plen = paths.shape
    lib = _lib.load()
    pc = lib.eu_gen_pair_count(plen, int(left_win_size), int(right_win_size))
    out = torch.empty((B, pc, 2), dtype=torch.int64, device=paths.device)
    ctx = _ctx_on_stream()
    check(lib.eu_gen_pair(ctx._h, paths.data_ptr(), B, plen, int(left_win_size), int(right_win_size), out.data_ptr()))
    return out


def sample_neighbor_api(nodes, edge_types, count):
    """euler::SampleNeighbor of the C++ api (api.cc:223-236): NO unique / gather -- a repeated id draws again.  Returns
    engine-form (ids i64[N,count], w, t); rows without a result are (0, 0.0, -1)."""
    nodes = _t(nodes, torch.int64).reshape(-1)
    et = get_edge_type_id(edge_types)
    n, count = nodes.numel(), int(count)
    ids = torch.empty((n, count), dtype=torch.int64, device=nodes.device)
    w = torch.empty((n, count), dtype=torch.float32, device=nodes.device)
    t = torch.empty((n, count), dtype=torch.int32, device=nodes.device)
    ctx = _ctx_on_stream()
    check(_lib.load().eu_sample_neighbor_raw(ctx._h, nodes.data_ptr(), n, et.ctypes.data, len(et), count,
                                             ids.data_ptr(), w.data_ptr(), t.data_ptr()))
    return ids, w, t


def unique(ids):
    """tf.unique on the device (eu_unique): (values in first-occurrence order, inverse i32 with ids == values[inverse])."""
    ids = _t(ids, torch.int64).reshape(-1)
    n = ids.numel()
    vals = torch.empty(n, dtype=torch.int64, device=ids.device)
    inv = torch.empty(n, dtype=torch.int32, device=ids.device)
    cnt = torch.zeros(1, dtype=torch.int64, device=ids.device)
    ctx = _ctx_on_stream()
    check(_lib.load().eu_unique(ctx._h, ids.data_ptr(), n, vals.data_ptr(), inv.data_ptr(), cnt.data_ptr()))
    return vals[:int(cnt.item())], inv


def sage_mean_aggregate(neighbor_ids, count, dim):
    """Fused get_dense_feature + scatter_mean for fixed-fanout blocks (SAGEConv's neighbor mean,
    tf_euler/python/convolution/sage_conv.py:33-38 over sage_dataflow.py:43-46 blocks)."""
    ids = _t(neighbor_ids, torch.int64).reshape(-1)
    rows = ids.numel() // int(count)
    out = torch.empty((rows, int(dim)), dtype=torch.float32, device=ids.device)
    ctx = _ctx_on_stream()
    check(_lib.load().eu_sage_mean_aggregate(ctx._h, ids.data_ptr(), rows, int(count), int(dim),
                                             out.data_ptr()))
    return out


# ------------------------------------------------------------------------------------ mp ops
def _raw_gather(params, indices):
    params = params.contiguous()
    out = torch.empty((indices.numel(), params.shape[1]), dtype=torch.float32, device=params.device)
    ctx = _ctx_on_stream()
    check(_lib.load().eu_gather(ctx._h, params.data_ptr(), params.shape[0], params.shape[1],
                                indices.data_ptr(), indices.numel(), out.data_ptr()))
    return out


def _raw_scatter(name, updates, indices, size):
    updates = updates.contiguous()
    out = torch.empty((int(size), updates.shape[1]), dtype=torch.float32, device=updates.device)
    ctx = _ctx_on_stream()
    check(getattr(_lib.load(), name)(ctx._h, updates.data_ptr(), updates.shape[1], indices.data_ptr(),
                                     indices.numel(), int(size), out.data_ptr()))
    return out


class _Gather(torch.autograd.Function):
    """MPGather with gradient scatter_add(grad, indices, N) (mp_ops.py:39-43)."""

    @staticmethod
    def forward(ctx, params, indices):
        ctx.save_for_backward(indices)
        ctx.n = params.shape[0]
        return _raw_gather(params, indices)

    @staticmethod
    def backward(ctx, grad):
        (indices,) = ctx.saved_tensors
        return _raw_scatter("eu_scatter_add", grad, indices, ctx.n), None


class _ScatterAdd(torch.autograd.Function):
    """MPScatterAdd with gradient gather(grad, indices) (mp_ops.py:46-49)."""

    @staticmethod
    def forward(ctx, updates, indices, size):
        ctx.save_for_backward(indices)
        return _raw_scatter("eu_scatter_add", updates, indices, size)

    @staticmethod
    def backward(ctx, grad):
        (indices,) = ctx.saved_tensors
        return _raw_gather(grad, indices), None, None


class _ScatterMax(torch.autograd.Function):
    """MPScatterMax; gradient splits evenly among ties (mp_ops.py:52-62)."""

    @staticmethod
    def forward(ctx, updates, indices, size):
        out = _raw_scatter("eu_scatter_max", updates, indices, size)
        ctx.save_for_backward(updates, indices, out)
        ctx.size = size
        return out

    @staticmethod
    def backward(ctx, grad):
        updates, indices, out = ctx.saved_tensors
        indicators = (updates == _raw_gather(out, indices)).to(updates.dtype)
        num_selected = _raw_scatter("eu_scatter_add", indicators, indices, ctx.size)
        indicators = indicators / _raw_gather(num_selected, indices)
        return indicators * _raw_gather(grad, indices), None, None


def _f32(x):
    x = _t(x, torch.float32)
    return x if x.dim() == 2 else x.reshape(x.shape[0], -1)


def gather(params, indices):
    """mp_ops.gather = MPGather (mp_ops.py:27): out[i,:] = params[indices[i],:]."""
    return _Gather.apply(_f32(params), _t(indices, torch.int32).reshape(-1))


def scatter_add(updates, indices, size=None):
    """mp_ops.scatter_add = MPScatterAdd (mp_ops.py:28)."""
    return _ScatterAdd.apply(_f32(updates), _t(indices, torch.int32).reshape(-1), int(size))


def scatter_max(updates, indices, size=None):
    """mp_ops.scatter_max = MPScatterMax (mp_ops.py:29); output initialised to -1e9."""
    return _ScatterMax.apply(_f32(updates), _t(indices, torch.int32).reshape(-1), int(size))


def scatter_mean(updates, indices, size=None):
    """mp_ops.scatter_mean (mp_ops.py:65-69): scatter_add / (scatter_add(ones) + 1e-7).
    Without autograd the fused kernel is used (same arithmetic)."""
    updates = _f32(updates)
    indices = _t(indices, torch.int32).reshape(-1)
    if not (torch.is_grad_enabled() and updates.requires_grad):
        return _raw_scatter("eu_scatter_mean", updates, indices, int(size))
    out = scatter_add(updates, indices, size)
    ep = 1e-7
    ones = torch.ones((updates.shape[0], 1), dtype=torch.float32, device=updates.device)
    count = scatter_add(ones, indices, size) + ep
    return out / count


def scatter_(op, updates, indices, size):
    """mp_ops.scatter_ (mp_ops.py:72-73)."""
    return globals()['scatter_' + op](updates, indices, size)


def scatter_softmax(updates, indices, size=None):
    """mp_ops.scatter_softmax (mp_ops.py:76-79)."""
    updates = _f32(updates)
    updates = updates - gather(scatter_max(updates, indices, size), indices)
    updates = torch.exp(updates)
    return updates / gather(scatter_add(updates, indices, size), indices)
