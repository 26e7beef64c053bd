"""Keyphrase graphs on an existing index (east_graph_index_host / _dev, DeviceIndex.graph, ASTRelevanceMeasure.cooccurrence):
the counts of a built, table-returned, loaded or globally sorted index at one or several relevance thresholds, without a
score table.  Every plane is compared element for element with east_cooc_host of the index's own score_table /
score_groups table."""
import ctypes
import struct

import numpy as np
import pytest

from test_gpu_graphs import _collection, _public_collection, _queries, _thresholds
from test_gpu_synonym_tables import _concat, _word_synonyms
from test_gpu_synonyms import _rich_synonyms, _Synonimizer


def _capi():
    from east import _capi
    return _capi


def test_index_graph_entries_check_their_arguments_in_order_without_a_gpu():
    # output (C, the number of thresholds, the thresholds), then the index and the range, then the groups, then the
    # keyphrases -- all before the first CUDA call
    capi = _capi()
    L = capi.load()
    # stands in for an index of 4 documents: the checks read only n_docs, which follows `device` at the head of
    # struct east_index (csrc/capi.cu); device -1 makes any call that got past the checks fail before a launch
    fake_index = ctypes.create_string_buffer(4096)
    struct.pack_into("<ii", fake_index, 0, -1, 4)
    idx = ctypes.cast(fake_index, ctypes.c_void_p)
    fake = 1 << 20   # device addresses the calls must never reach
    codes = np.array([65], dtype=np.uint32)
    empty = np.array([0, 1, 1], dtype=np.int64)   # the second keyphrase is empty
    groups, bad_groups = np.array([0, 2], dtype=np.int64), np.array([0, 3], dtype=np.int64)
    thr = np.array([0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9])
    C = np.zeros(9 * 4, dtype=np.int32)
    p = capi._ptr

    def host(index=idx, off=empty, g=None, thresholds=thr, T=1, begin=0, count=4, out=C):
        return L.east_graph_index_host(index, p(codes, capi._u32p), p(off, capi._i64p), len(off) - 1,
                                       None if g is None else p(g, capi._i64p), 0 if g is None else len(g) - 1, 1,
                                       None if thresholds is None else p(thresholds, capi._f64p), T, begin, count,
                                       None if out is None else p(out, capi._i32p))

    def dev(index=idx, off=empty, g=None, thresholds=thr, T=1, begin=0, count=4, out=fake):
        return L.east_graph_index_dev(index, fake, None, p(off, capi._i64p), len(off) - 1,
                                      None if g is None else p(g, capi._i64p), 0 if g is None else len(g) - 1, 0,
                                      None if thresholds is None else p(thresholds, capi._f64p), T, begin, count, out, None)

    def error(rc):
        with pytest.raises((ValueError, ZeroDivisionError)) as e:
            capi._check(rc)
        return e.type, L.east_last_error().decode()

    capi.launch_count(reset=True)
    for call in (host, dev):
        for g in (None, groups):
            assert error(call(g=g))[0] is ZeroDivisionError, call.__name__   # everything else is well-formed
            for bad in ({"index": None}, {"T": 0}, {"T": 9}, {"thresholds": None}, {"out": None}, {"begin": -1},
                        {"count": 0}, {"begin": 3, "count": 2}, {"begin": 4, "count": 1}):
                assert error(call(g=g, **bad))[0] is ValueError, (call.__name__, g, bad)
        assert error(call(g=bad_groups))[0] is ValueError, call.__name__
        # the first failure in the stated order is the one reported
        assert "threshold" in error(call(T=9, begin=-1, g=bad_groups))[1]
        assert "threshold" in error(call(thresholds=None, index=None, g=bad_groups))[1]
        assert "document range" in error(call(begin=-1, g=bad_groups))[1]
        assert "group" in error(call(g=bad_groups))[1]
    assert capi.launch_count() == 0


def _index(kind, packed, ms, q, tmp_path):
    """an index of `packed` made the way `kind` says"""
    capi = _capi()
    codes, off, group_off, normalized = q
    text, doc_off = _concat(packed)
    if kind == "table":
        out = np.empty((len(ms), len(off) - 1 if group_off is None else len(group_off) - 1))
        return capi.DeviceIndex.build_host_and_score(text, doc_off, ms, codes, off, out, normalized, group_off=group_off)
    idx = capi.DeviceIndex.build_host(text, doc_off, ms)
    if kind == "loaded":
        path = str(tmp_path / "index.eastidx")
        idx.save(path)
        idx.close()
        idx = capi.DeviceIndex.load(path)
    return idx


def _own_table(idx, q):
    codes, off, group_off, normalized = q
    if group_off is None:
        return idx.score_table(codes, off, normalized)
    return idx.score_groups(codes, off, group_off)


def _graph(idx, q, thr, **kw):
    codes, off, group_off, normalized = q
    return idx.graph(codes, off, thr, normalized=normalized, group_off=group_off, **kw)


def _with_big_document(packed, ms):
    """the first five documents and one of more than 64 Ki code points: the index comes from the global sort"""
    import synth
    from east import utils
    from east.asts import utils as au
    big = utils.text_to_strings_collection(synth.document(90000, 78))
    return list(packed[:5]) + [au.pack_strings_collection(big)], list(ms[:5]) + [len(big)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["norm", "denorm", "groups"])
def test_every_index_kind_and_threshold_equals_cooc_of_its_table(mode, tmp_path):
    capi = _capi()
    texts, cols, packed, ms, prepared = _collection(first_seed=9300)
    q = _queries(prepared, mode)
    for kind in ("built", "table", "loaded", "global"):
        parts, m = _with_big_document(packed, ms) if kind == "global" else (packed, ms)
        idx = _index(kind, parts, m, q, tmp_path)
        assert bool(idx.info()["doc_sorted"]) == (kind != "global"), kind
        table = _own_table(idx, q)
        thrs = _thresholds(table)
        capi.launch_count(reset=True)
        planes = _graph(idx, q, thrs)
        assert planes.shape == (len(thrs), table.shape[1], table.shape[1]) and planes.dtype == np.int32
        for t, thr in enumerate(thrs):
            exp = capi.cooc_host(table, thr)
            assert np.array_equal(planes[t], exp), (kind, thr)
            one = _graph(idx, q, thr)
            assert one.shape == exp.shape and np.array_equal(one, exp), (kind, thr)
        # thresholds in any order, one of them twice
        mixed = [thrs[4], thrs[0], thrs[4], thrs[2]]
        got = _graph(idx, q, mixed)
        assert all(np.array_equal(got[t], capi.cooc_host(table, r)) for t, r in enumerate(mixed)), kind
        idx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["denorm", "groups"])
def test_document_ranges_count_their_documents_and_add_up(mode):
    capi = _capi()
    texts, cols, packed, ms, prepared = _collection(first_seed=9400)
    q = _queries(prepared, mode)
    idx = _index("built", packed, ms, q, None)
    table = _own_table(idx, q)
    thrs = _thresholds(table)
    n = len(ms)
    for begin in (0, 1, 17, 133):
        for count in (1, 37, n - begin):
            got = _graph(idx, q, thrs, doc_begin=begin, doc_count=count)
            for t, thr in enumerate(thrs):
                assert np.array_equal(got[t], capi.cooc_host(table[begin:begin + count], thr)), (begin, count, thr)
    bounds = [0, 1, 17, 133, n]
    parts = [_graph(idx, q, thrs, doc_begin=a, doc_count=b - a) for a, b in zip(bounds, bounds[1:])]
    assert np.array_equal(sum(parts), _graph(idx, q, thrs))
    idx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["norm", "groups"])
def test_tiles_are_thresholded_once_per_tile_whatever_the_number_of_thresholds(mode):
    capi = _capi()
    texts, cols, packed, ms, prepared = _collection(first_seed=9450)
    q = _queries(prepared, mode)
    idx = _index("built", packed, ms, q, None)
    table = _own_table(idx, q)
    thrs = _thresholds(table)
    exp = np.stack([capi.cooc_host(table, r) for r in thrs])
    try:
        # the fp64 scratch holds 20 documents: 15 tiles per call, most of them at column offsets that are not multiples of 16
        capi.set_option("score_tmp_doubles", table.shape[1] * 20)
        for T in (1, len(thrs)):
            capi.set_option("time_kernels", 0)
            capi.set_option("time_kernels", 1)
            got = _graph(idx, q, thrs[:T])
            names = capi.kernel_stats()
            capi.set_option("time_kernels", 0)
            assert np.array_equal(got, exp[:T]), T
            assert names["k_threshold_bytes"]["launches"] >= len(ms) // 20, (T, names["k_threshold_bytes"])
            assert not any(k.startswith("k_doc_suffix_sort") for k in names), (T, sorted(names))
        for variant in (0, 2, 3):
            capi.set_option("cooc_variant", variant)
            assert np.array_equal(_graph(idx, q, thrs), exp), variant
    finally:
        capi.set_option("time_kernels", 0)
        capi.set_option("score_tmp_doubles", 0)
        capi.set_option("cooc_variant", 0)
    idx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["norm", "groups"])
def test_device_entry_writes_every_count_on_the_callers_stream(mode):
    import torch
    capi = _capi()
    texts, cols, packed, ms, prepared = _collection(first_seed=9550)
    q = _queries(prepared, mode)
    codes, off, group_off, normalized = q
    idx = _index("built", packed, ms, q, None)
    table = _own_table(idx, q)
    thrs = _thresholds(table)
    k = table.shape[1]
    kp_t = torch.from_numpy(codes.view(np.int32).copy()).cuda()
    stream = torch.cuda.Stream()
    for host_copy, begin, count in ((codes, 0, len(ms)), (None, 17, 100)):
        C_t = torch.full((len(thrs), k, k), -1, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        idx.graph_dev(kp_t.data_ptr(), host_copy, off, thrs, C_t.data_ptr(), normalized=normalized, group_off=group_off,
                      doc_begin=begin, doc_count=count, stream=stream.cuda_stream)
        stream.synchronize()
        got = C_t.cpu().numpy()
        for t, thr in enumerate(thrs):
            assert np.array_equal(got[t], capi.cooc_host(table[begin:begin + count], thr)), (begin, thr)
    idx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("collection", ["ascii", "several_batches", "hse"])
@pytest.mark.parametrize("synonyms", [False, True])
def test_loaded_collection_gives_graphs_without_a_table(golden, monkeypatch, tmp_path, collection, synonyms):
    from east import applications, relevance, utils
    capi = _capi()
    texts, kps = _public_collection(collection)
    kept = [kp for kp in kps if kp]
    prepared = [utils.prepare_text(k) for k in kept]
    syn = None
    if synonyms:
        syn = _Synonimizer(_rich_synonyms(prepared) if collection != "hse" else _word_synonyms(prepared))
    settings = [(g["c"], g["r"], g["p"]) for g in golden["hse"]["graphs"]] + [(0.5, 0.0, 1), (0.5, 2.0, 1)]
    rs = [r for _, r, _ in settings]
    fresh = relevance.ASTRelevanceMeasure()
    fresh.set_text_collection(list(texts.values()))
    table = fresh.relevance_table(prepared, syn)
    expect = [capi.cooc_host(table, r) for r in rs]
    graphs = [applications.keyphrases_graph(kps, texts, c, r, p, similarity_measure=relevance.ASTRelevanceMeasure(),
                                            synonimizer=syn) for c, r, p in settings]
    fresh.save_index(str(tmp_path / "saved"))

    def refuse(*a, **k):
        raise AssertionError("a score table was formed")
    with monkeypatch.context() as m:
        m.setattr(capi, "cooc_host", refuse)
        m.setattr(capi.DeviceIndex, "score_table", refuse)
        m.setattr(capi.DeviceIndex, "score_groups", refuse)
        loaded = relevance.ASTRelevanceMeasure.load_index(str(tmp_path / "saved"))
        assert len(loaded._batches) == (2 if collection == "several_batches" else 1)
        planes = loaded.cooccurrence(prepared, rs, syn)
        assert planes.shape == (len(rs), len(kept), len(kept))
        for t, r in enumerate(rs):
            assert np.array_equal(planes[t], expect[t]), r
            one = loaded.cooccurrence(prepared, r, syn)
            assert np.array_equal(one, expect[t]), r
            assert loaded._cooc is None
        for (c, r, p), t, graph in zip(settings, range(len(rs)), graphs):
            assert applications.graph_from_cooccurrence(kps, kept, planes[t], c, r, p) == graph, (c, r, p)
    if collection == "hse" and not synonyms:
        for g, t in zip(golden["hse"]["graphs"], range(3)):
            graph = applications.graph_from_cooccurrence(kps, kept, planes[t], g["c"], g["r"], g["p"])
            assert graph["nodes"] == g["nodes"]
            assert [(e["source"], e["target"], float(e["confidence"]).hex()) for e in graph["edges"]] == \
                   [(e["source"], e["target"], e["confidence"]) for e in g["edges"]]


@pytest.mark.gpu
def test_measure_routes_counts_by_what_it_holds(monkeypatch):
    import synth
    from east import relevance, utils
    capi = _capi()
    texts = synth.documents(6, 3000, first_seed=8950)
    prepared = [utils.prepare_text(k) for k in synth.keyphrases(30, seed=9)]
    syn = _Synonimizer(_rich_synonyms(prepared))
    fresh = relevance.ASTRelevanceMeasure()
    fresh.set_text_collection(texts)
    plain, grouped = fresh.relevance_table(prepared), fresh.relevance_table(prepared, syn)
    # a table scored while indexing answers, per threshold, through cooc_host; other variants go to the index
    measure = relevance.ASTRelevanceMeasure()
    measure.set_text_collection(texts, prepared_keyphrases=prepared)
    calls = []
    real_cooc, real_graph = capi.cooc_host, capi.DeviceIndex.graph
    with monkeypatch.context() as m:
        m.setattr(capi, "cooc_host", lambda *a, **k: calls.append("cooc_host") or real_cooc(*a, **k))
        m.setattr(capi.DeviceIndex, "graph", lambda self, *a, **k: calls.append("graph") or real_graph(self, *a, **k))
        got = measure.cooccurrence(prepared, [0.2, 0.3])
        assert calls == ["cooc_host", "cooc_host"]
        assert all(np.array_equal(got[t], real_cooc(plain, r)) for t, r in enumerate((0.2, 0.3)))
        del calls[:]
        got = measure.cooccurrence(prepared, 0.3, syn)
        assert calls == ["graph"] and np.array_equal(got, real_cooc(grouped, 0.3))
        # stored counts of a graph call answer only their own scalar threshold
        measure.set_text_collection(texts, prepared_keyphrases=prepared, relevance_threshold=0.3)
        del calls[:]
        assert measure.cooccurrence(prepared, 0.3) is measure._cooc and calls == []
        got = measure.cooccurrence(prepared, [0.3])
        assert calls == ["graph"] and got.shape == (1, 30, 30) and np.array_equal(got[0], measure._cooc)
    for bad in ([0.1] * 9, []):   # 1 to 8 thresholds
        with pytest.raises(ValueError):
            measure.cooccurrence(prepared, bad)
