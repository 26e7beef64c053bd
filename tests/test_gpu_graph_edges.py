"""Keyphrase graphs assembled on the device from their co-occurrence counts (east_graph_edges_host / _dev,
applications.graph_on_device): supports and edges come back, the K x K counts stay where they are.  Every graph is compared
dict for dict with applications.graph_from_cooccurrence on the host, confidences by float.hex."""
import ctypes

import numpy as np
import pytest

P_VALUES = [0, 1, 2.5, float("nan"), float("inf"), -float("inf")]
C_VALUES = [-0.5, 0, 5e-324, 0.6, 1, 1.5, float("nan"), float("inf")]


def _key(graph):
    """a graph dict with its confidences as float.hex (NaN parameters as their repr, so that they compare equal)"""
    return ({k: repr(v) for k, v in graph.items() if k not in ("nodes", "edges")}, graph["nodes"],
            [(e["source"], e["target"], float(e["confidence"]).hex()) for e in graph["edges"]])


def _host(kps, kept, cooc, c, r, p):
    from east import applications
    return applications.graph_from_cooccurrence(kps, kept, cooc, c, r, p)


def _device(kps, kept, cooc, c, r, p):
    from east import applications
    return applications.graph_on_device(kps, kept, cooc, c, r, p)


def _counts(K, D, seed, zero_rows=()):
    """symmetric int32 counts C = B B^T of random relevance bits with some all-zero rows (zero supports)"""
    rng = np.random.default_rng(seed)
    dens = np.clip(0.6 / np.sqrt(np.arange(1, K + 1)), 0.02, 1)
    B = (rng.random((K, D)) < dens[rng.permutation(K)][:, None]).astype(np.int64)
    B[list(zero_rows)] = 0
    return (B @ B.T).astype(np.int32)


def _labels(K, seed):
    """(keyphrases, kept): kept has K columns, two of which repeat a label (the last one wins); the keyphrases repeat
    some labels and skip others"""
    rng = np.random.default_rng(seed)
    kept = ["kp%d" % k for k in range(K)]
    if K > 6:
        kept[5], kept[K - 1] = kept[2], kept[3]
    labels = sorted(set(kept))
    kps = [labels[i] for i in rng.integers(0, len(labels), size=K + K // 3)]
    return kps, kept


def _call(entry, C, node_col, c, p, cap, stream=None):
    """one raw call of east_graph_edges_host (entry "host", C numpy) or _dev ("dev", C a CUDA tensor)"""
    from east import _capi
    L = _capi.load()
    T, cols, N = (1 if C.ndim == 2 else C.shape[0]), C.shape[-1], len(node_col)
    support, n_edges = np.full((T, max(N, 1)), -7, dtype=np.int32), np.full(T, -7, dtype=np.int64)
    src, dst, conf = np.zeros(max(cap, 1), np.int32), np.zeros(max(cap, 1), np.int32), np.zeros(max(cap, 1))
    i32, i64, f64 = ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_double)
    outs = (support.ctypes.data_as(i32), n_edges.ctypes.data_as(i64), cap, src.ctypes.data_as(i32), dst.ctypes.data_as(i32),
            conf.ctypes.data_as(f64))
    nodes = (np.ascontiguousarray(node_col, dtype=np.int32).ctypes.data_as(i32), N, c, p)
    if entry == "host":
        rc = L.east_graph_edges_host(C.ctypes.data_as(i32), cols, T, *nodes, 0, *outs)
    else:
        rc = L.east_graph_edges_dev(ctypes.c_void_p(C.data_ptr()), cols, T, *nodes, C.device.index, ctypes.c_void_p(stream or 0),
                                    *outs)
    return rc, support[:, :N], n_edges, src, dst, conf


def test_argument_order_needs_no_gpu():
    # every check runs before the first CUDA call, in one order: the outputs, the counts, the nodes
    from east import _capi
    L = _capi.load()
    i32, i64, f64 = ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_double)
    C = np.zeros((2, 2), dtype=np.int32)
    fake = ctypes.c_void_p(1 << 20)   # a device address the calls must never reach
    sup, ne = np.zeros(4, np.int32).ctypes.data_as(i32), np.zeros(2, np.int64).ctypes.data_as(i64)
    s, d, cf = np.zeros(4, np.int32).ctypes.data_as(i32), np.zeros(4, np.int32).ctypes.data_as(i32), np.zeros(4).ctypes.data_as(f64)
    good_nodes, bad_nodes = np.array([0, 1], np.int32), np.array([0, 2], np.int32)

    def both(counts, cols, T, nodes, n, outs):
        """the rc and message of each entry with these arguments"""
        got = []
        nd = nodes.ctypes.data_as(i32) if nodes is not None else None
        got.append((L.east_graph_edges_host(counts, cols, T, nd, n, 0.5, 1.0, 0, *outs), L.east_last_error()))
        got.append((L.east_graph_edges_dev(fake if counts is not None else None, cols, T, nd, n, 0.5, 1.0, 0, None, *outs),
                    L.east_last_error()))
        return got

    Cp = C.ctypes.data_as(i32)
    cases = [   # (arguments, the message of the first failing check)
        ((Cp, 0, 9, bad_nodes, 2, (None, ne, 4, s, d, cf)), b"bad output"),
        ((Cp, 0, 9, bad_nodes, 2, (sup, None, 4, s, d, cf)), b"bad output"),
        ((Cp, 0, 9, bad_nodes, 2, (sup, ne, -1, s, d, cf)), b"bad output"),
        ((Cp, 0, 9, bad_nodes, 2, (sup, ne, 4, s, None, cf)), b"bad output"),
        ((Cp, 0, 1, bad_nodes, 2, (sup, ne, 4, s, d, cf)), b"bad counts"),
        ((Cp, 2, 0, bad_nodes, 2, (sup, ne, 4, s, d, cf)), b"bad counts"),
        ((Cp, 2, 9, bad_nodes, 2, (sup, ne, 4, s, d, cf)), b"bad counts"),
        ((None, 2, 1, bad_nodes, 2, (sup, ne, 0, None, None, None)), b"bad counts"),
        ((Cp, 2, 1, bad_nodes, 2, (sup, ne, 0, None, None, None)), b"node column out of range"),
        ((Cp, 2, 1, np.array([-1, 0], np.int32), 2, (sup, ne, 4, s, d, cf)), b"node column out of range"),
        ((Cp, 2, 1, None, 2, (sup, ne, 4, s, d, cf)), b"bad nodes"),
        ((Cp, 2, 1, good_nodes, -1, (sup, ne, 4, s, d, cf)), b"bad nodes"),
    ]
    for args, msg in cases:
        for rc, err in both(*args):
            assert rc == -1 and msg in err, (msg, err)
    # the Python binding reports them as ValueError
    with pytest.raises(ValueError):
        _capi.graph_edges(C, bad_nodes, 0.5, 1.0)


@pytest.mark.gpu
@pytest.mark.parametrize("on", ["numpy", "tensor"])
def test_golden_graphs(golden, on):
    import torch
    hse = golden["hse"]
    kps = hse["keyphrases"]
    names = [d["name"] for d in hse["docs"]]
    table = np.array([[float.fromhex(hse["table_norm"][kp][n]) for kp in kps] for n in names])
    for g in hse["graphs"]:
        B = (table >= g["r"]).astype(np.int64)
        cooc = (B.T @ B).astype(np.int32)
        counts = cooc if on == "numpy" else torch.from_numpy(cooc).cuda()
        graph = _device(kps, kps, counts, g["c"], g["r"], g["p"])
        assert _key(graph) == _key(_host(kps, kps, cooc, g["c"], g["r"], g["p"]))
        assert graph["nodes"] == g["nodes"]
        assert [(e["source"], e["target"], e["confidence"].hex()) for e in graph["edges"]] == \
               [(e["source"], e["target"], e["confidence"]) for e in g["edges"]]


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 7, 40, 200])
@pytest.mark.parametrize("on", ["numpy", "tensor"])
def test_random_counts_every_threshold(K, on):
    import torch
    cooc = _counts(K, 64, seed=K, zero_rows=range(0, K, 5))
    kps, kept = _labels(K, seed=K + 1)
    counts = cooc if on == "numpy" else torch.from_numpy(cooc).cuda()
    for p in P_VALUES:
        for c in C_VALUES:
            assert _key(_device(kps, kept, counts, c, 0.25, p)) == _key(_host(kps, kept, cooc, c, 0.25, p)), (p, c)


@pytest.mark.gpu
def test_large_random_counts():
    import torch
    K = 2500
    cooc = _counts(K, 400, seed=3, zero_rows=range(7, K, 11))
    kps, kept = _labels(K, seed=4)
    dev = torch.from_numpy(cooc).cuda()
    for p, c in ((1, 0.6), (2.5, 0.3), (0, 1), (1, 1.5), (3, 0.2)):
        exp = _key(_host(kps, kept, cooc, c, 0.25, p))
        assert _key(_device(kps, kept, cooc, c, 0.25, p)) == exp, (p, c)
        assert _key(_device(kps, kept, dev, c, 0.25, p)) == exp, (p, c)


@pytest.mark.gpu
@pytest.mark.parametrize("on", ["numpy", "tensor"])
def test_eight_planes_in_one_call(on):
    import torch
    K = 200
    planes = np.stack([_counts(K, 50 + 10 * t, seed=100 + t, zero_rows=range(t, K, 9)) for t in range(8)])
    kps, kept = _labels(K, seed=5)
    thresholds = [0.1 * t for t in range(8)]
    counts = planes if on == "numpy" else torch.from_numpy(planes).cuda()
    for p, c in ((1, 0.6), (0, 0), (2.5, 0.3), (float("nan"), 0.5), (1, float("nan"))):
        got = _device(kps, kept, counts, c, thresholds, p)
        assert isinstance(got, list) and len(got) == 8
        for t, r in enumerate(thresholds):
            assert _key(got[t]) == _key(_host(kps, kept, planes[t], c, r, p)), (p, c, t)


@pytest.mark.gpu
def test_tensor_on_a_non_default_stream():
    import torch
    K = 600
    B = (torch.rand((K, 300), generator=torch.Generator().manual_seed(8)) < 0.1).float()
    kps, kept = _labels(K, seed=9)
    exp = (B @ B.T).to(torch.int32).numpy()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        Bd = B.cuda(non_blocking=False)
        counts = torch.zeros((1, K, K), dtype=torch.int32, device="cuda")
        counts[0] = (Bd @ Bd.T).to(torch.int32)   # queued on `side`: the graph call must be ordered after it
        got = _device(kps, kept, counts, 0.4, [0.25], 2)
    assert _key(got[0]) == _key(_host(kps, kept, exp, 0.4, 0.25, 2))


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["host", "dev"])
def test_edge_cap_sizing(entry):
    import torch
    K = 150
    planes = np.stack([_counts(K, 60, seed=20 + t) for t in range(3)])
    kps, kept = _labels(K, seed=21)
    from east import applications
    node_col = applications._node_columns(kps, kept)
    C = planes if entry == "host" else torch.from_numpy(planes).cuda()
    exp = [_host(kps, kept, planes[t], 0.3, 0.0, 1) for t in range(3)]
    want = [len(g["edges"]) for g in exp]
    exact = sum(want)
    assert exact > 1
    for cap in (0, exact - 1):
        rc, support, n_edges, *_ = _call(entry, C, node_col, 0.3, 1.0, cap)
        assert rc == -5 and n_edges.tolist() == want, cap
        assert np.array_equal(support, planes[:, node_col, node_col])
    rc, support, n_edges, src, dst, conf = _call(entry, C, node_col, 0.3, 1.0, exact)
    assert rc == 0 and n_edges.dtype == np.int64 and n_edges.tolist() == want
    flat = [e for g in exp for e in g["edges"]]
    assert [(int(s), int(d), float(c).hex()) for s, d, c in zip(src, dst, conf)] == \
           [(e["source"], e["target"], e["confidence"].hex()) for e in flat]


@pytest.mark.gpu
def test_dense_planes_count_in_int64():
    # c <= 0 and p = -inf: every ordered pair of distinct nodes is an edge, N (N - 1) per plane.  The row counts are
    # int32 (a row has < 2^31 edges) and the scan over the rows of all planes is int64 (csrc/graph_edges.cu); 2^31 edges
    # (> 34 GB of host output) are not allocated here.
    import torch
    from east import _capi
    N, T = 2000, 8
    C = torch.zeros((T, N, N), dtype=torch.int32, device="cuda")
    node_col = np.arange(N, dtype=np.int32)[::-1].copy()
    support, n_edges, src, dst, conf = _capi.graph_edges(C, node_col, 0.0, -float("inf"))
    assert n_edges.dtype == np.int64 and n_edges.tolist() == [N * (N - 1)] * T
    assert not support.any() and len(src) == T * N * (N - 1) and not conf.any()
    assert (src[:N - 1] == 0).all() and np.array_equal(dst[:N - 1], np.arange(1, N))
    last = T * N * (N - 1)
    assert (src[last - (N - 1):] == N - 1).all() and np.array_equal(dst[last - (N - 1):], np.arange(N - 1))


@pytest.mark.gpu
def test_self_loops_are_never_emitted():
    # graph_from_cooccurrence pairs a node with itself at referral_confidence <= -1 (fill_diagonal(-1.0), then >= c);
    # the reference's permutations never does, nor does the device assembly
    K = 30
    cooc = _counts(K, 40, seed=31)
    kps, kept = _labels(K, seed=32)
    for c in (-1, -2.5, -float("inf")):
        host = _host(kps, kept, cooc, c, 0.25, 0)
        got = _device(kps, kept, cooc, c, 0.25, 0)
        assert any(e["source"] == e["target"] for e in host["edges"])
        host["edges"] = [e for e in host["edges"] if e["source"] != e["target"]]
        assert _key(got) == _key(host)


@pytest.mark.gpu
def test_missing_and_empty_keyphrases():
    from east import applications
    cooc = _counts(4, 10, seed=1)
    with pytest.raises(KeyError):
        applications.graph_on_device(["kp0", "nope"], ["kp0", "kp1", "kp2", "kp3"], cooc, 0.5, 0.25, 1)
    assert applications.graph_on_device([], [], np.zeros((0, 0), np.int32), 0.5, 0.25, 1) == \
        _host([], [], np.zeros((0, 0), np.int32), 0.5, 0.25, 1)


@pytest.mark.gpu
def test_public_routes_assemble_on_the_device(golden, monkeypatch, tmp_path):
    from east import applications, relevance
    from test_gpu_synonym_tables import _hse
    texts, kps = _hse()
    settings = [(g["c"], g["r"], g["p"]) for g in golden["hse"]["graphs"]]
    measure = relevance.ASTRelevanceMeasure()
    measure.set_text_collection(list(texts.values()))
    measure.save_index(str(tmp_path / "idx"))
    kept = [k for k in kps if k]
    from east import utils
    prepared = [utils.prepare_text(k) for k in kept]
    planes = relevance.ASTRelevanceMeasure.load_index(str(tmp_path / "idx")).cooccurrence(prepared, [r for _, r, _ in settings])
    expect = [_host(kps, kept, planes[t], c, r, p) for t, (c, r, p) in enumerate(settings)]
    host = {(c, r, p): _host(kps, kept, planes[t], c, r, p) for c, _, p in settings for t, (_, r, _) in enumerate(settings)}

    def refuse(*a, **k):
        raise AssertionError("the graph was assembled on the host")
    with monkeypatch.context() as m:
        m.setattr(applications, "graph_from_cooccurrence", refuse)
        for (c, r, p), exp in zip(settings, expect):
            graph = applications.keyphrases_graph(kps, texts, c, r, p, similarity_measure=relevance.ASTRelevanceMeasure())
            assert _key(graph) == _key(exp), (c, r, p)
        loaded = relevance.ASTRelevanceMeasure.load_index(str(tmp_path / "idx"))
        for c, _, p in settings:
            got = loaded.graphs(kps, c, [r for _, r, _ in settings], p)
            for t, (_, r, _) in enumerate(settings):
                assert _key(got[t]) == _key(host[c, r, p]), (c, r, p)
        assert [_key(g) for g in [loaded.graphs(kps, c, [r], p)[0] for c, r, p in settings]] == [_key(e) for e in expect]
