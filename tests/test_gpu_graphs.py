"""Keyphrase graphs without the score table (east_graph_host / _dev / _texts_host): the per-document kernel writes the
relevance bytes the tensor-core co-occurrence count reads (k_doc_suffix_sort_graph, k_doc_suffix_sort_groups_graph), and
every fallback thresholds bounded tiles of documents into the same bytes.  Every count matrix is compared element for
element with east_cooc_host of the matching table entry's table; graph dicts with the table route and the reference."""
import json
import os

import numpy as np
import pytest

from test_gpu_synonym_tables import _concat, _hse, _word_synonyms
from test_gpu_synonyms import _defaultdict, _rich_synonyms, _Synonimizer


def _capi():
    from east import _capi
    return _capi


def _collection(n_docs=300, n_bytes=1200, first_seed=9100, n_kps=40):
    import synth
    from east import utils
    from east.asts import utils as au
    texts = synth.documents(n_docs, n_bytes, first_seed)
    cols = [utils.text_to_strings_collection(t) for t in texts]
    packed = [au.pack_strings_collection(c) for c in cols]
    prepared = [utils.prepare_text(k) for k in synth.keyphrases(n_kps, seed=17)]
    return texts, cols, packed, [len(c) for c in cols], prepared


def _queries(prepared, mode):
    """(codes, off, group_off, normalized) of a plain ("norm" / "denorm") or grouped ("groups") call"""
    capi = _capi()
    if mode == "groups":
        codes, off, group_off = capi.pack_variant_groups(prepared, _rich_synonyms(prepared))
        return codes, off, group_off, True
    codes, off = capi.pack_keyphrases(prepared)
    return codes, off, None, mode == "norm"


def _table(parts, ms, q):
    """the matching table entry's table (east_table_host / east_table_groups_host)"""
    codes, off, group_off, normalized = q
    text, doc_off = _concat(parts)
    out = np.empty((len(ms), len(off) - 1 if group_off is None else len(group_off) - 1))
    _capi().DeviceIndex.build_host_and_score(text, doc_off, ms, codes, off, out, normalized, group_off=group_off).close()
    return out


def _graph_host(parts, ms, q, thr):
    codes, off, group_off, normalized = q
    text, doc_off = _concat(parts)
    C, idx = _capi().DeviceIndex.build_host_and_graph(text, doc_off, ms, codes, off, thr, normalized=normalized,
                                                      group_off=group_off)
    return idx, C


def _graph_dev(parts, ms, q, thr):
    import torch
    codes, off, group_off, normalized = q
    text, doc_off = _concat(parts)
    cols = len(off) - 1 if group_off is None else len(group_off) - 1
    text_t = torch.from_numpy(text.view(np.int32)).cuda()
    kp_t = torch.from_numpy(codes.view(np.int32).copy()).cuda()
    C_t = torch.full((cols, cols), -1, dtype=torch.int32, device="cuda")
    idx = _capi().DeviceIndex.build_dev_and_graph(text_t.data_ptr(), doc_off, ms, kp_t.data_ptr(), codes, off, thr, C_t.data_ptr(),
                                                  normalized=normalized, group_off=group_off)
    torch.cuda.synchronize()
    return idx, C_t.cpu().numpy()


def _graph_texts(texts, q, thr):
    codes, off, group_off, normalized = q
    C, idx = _capi().DeviceIndex.graph_from_texts(texts, codes, off, thr, normalized=normalized, group_off=group_off)
    return idx, C


def _kernels(fn, *args):
    """(counts of fn, {kernel name: stats} of the kernels it launched)"""
    capi = _capi()
    capi.set_option("time_kernels", 0)
    capi.set_option("time_kernels", 1)
    try:
        idx, C = fn(*args)
        idx.close()
        names = capi.kernel_stats()
    finally:
        capi.set_option("time_kernels", 0)
    return C, names


def _in_kernel(names, grouped):
    graph_kernel = "k_doc_suffix_sort_groups_graph" if grouped else "k_doc_suffix_sort_graph"
    return (graph_kernel in names and "k_threshold_bytes" not in names
            and not {"k_doc_suffix_sort", "k_doc_suffix_sort_groups"} & set(names)
            and not any(n.startswith("k_score_combine") or n.startswith("k_score_suffixes") for n in names))


def _thresholds(table):
    """every cell counts (0 and below), none counts, and values of the table itself (ties of >=)"""
    values = np.unique(table)
    picks = [float(values[int(q * (len(values) - 1))]) for q in (0.2, 0.5, 0.8)]
    return [0.0, -0.5, float(table.max()) + 1.0] + picks


def _expect(table, thr):
    return _capi().cooc_host(table, thr)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["norm", "denorm", "groups"])
def test_every_graph_entry_equals_cooc_of_the_table(mode):
    from east.asts import utils as au
    capi = _capi()
    texts, cols, packed, ms, prepared = _collection()
    q = _queries(prepared, mode)
    table = _table(packed, ms, q)
    narrow = [au.pack_strings_collection_u8(c) for c in cols]
    grouped = mode == "groups"
    for thr in _thresholds(table):
        exp = _expect(table, thr)
        B = table >= thr
        assert np.array_equal(exp, (B.T.astype(np.int64) @ B.astype(np.int64)).astype(np.int32))
        try:
            capi.set_option("pipeline_chunk", 40000)   # several runs: the bytes are written while later runs are on their way
            for name, parts in (("host width 4", packed), ("host width 1", narrow)):
                idx, C = _graph_host(parts, ms, q, thr)
                assert idx.stat("pipelined") == 1 and idx.info()["doc_sorted"], name
                idx.close()
                assert np.array_equal(C, exp), (name, thr)
        finally:
            capi.set_option("pipeline_chunk", 0)
        idx, C = _graph_dev(packed, ms, q, thr)
        idx.close()
        assert np.array_equal(C, exp), ("dev", thr)
        idx, C = _graph_texts(texts, q, thr)
        idx.close()
        assert np.array_equal(C, exp), ("texts", thr)
    thr = _thresholds(table)[4]
    exp = _expect(table, thr)
    for name, fn, args in (("host", _graph_host, (packed, ms)), ("host width 1", _graph_host, (narrow, ms)),
                           ("dev", _graph_dev, (packed, ms)), ("texts", _graph_texts, (texts,))):
        C, names = _kernels(fn, *args, q, thr)
        assert _in_kernel(names, grouped), (name, sorted(names))
        assert "k_cooc_umma_tma" in names or "k_cooc_umma_pipe" in names, (name, sorted(names))
        assert np.array_equal(C, exp), name


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["norm", "groups"])
def test_every_fallback_fills_the_same_bytes(mode):
    import synth
    from east import utils
    from east.asts import utils as au
    capi = _capi()
    texts, cols, packed, ms, prepared = _collection(first_seed=9500)
    q = _queries(prepared, mode)
    table = _table(packed, ms, q)
    thr = _thresholds(table)[3]
    exp = _expect(table, thr)
    try:
        capi.set_option("no_fused_score", 1)   # the per-run batched scorer, its rows thresholded tile by tile
        for fn in (_graph_host, _graph_dev):
            C, names = _kernels(fn, packed, ms, q, thr)
            assert "k_threshold_bytes" in names and not any(n.endswith("_graph") for n in names), (fn.__name__, sorted(names))
            assert np.array_equal(C, exp), fn.__name__
        capi.set_option("no_fused_score", 0)
        # the fp64 scratch holds budget / cols documents: 20 here, so 15 tiles per call, each thresholded into its columns
        # (offsets that are not multiples of 16: the byte-by-byte edges of k_threshold_bytes); the per-suffix scratch,
        # budget / distinct suffixes documents, is tiled as well
        capi.set_option("score_tmp_doubles", len(prepared) * 20)
        for fn in (_graph_host, _graph_dev):
            C, names = _kernels(fn, packed, ms, q, thr)
            assert np.array_equal(C, exp), fn.__name__
            assert not any(n.endswith("_graph") for n in names), (fn.__name__, sorted(names))
            assert names["k_threshold_bytes"]["launches"] >= len(ms) // 20, (fn.__name__, names["k_threshold_bytes"])
    finally:
        capi.set_option("no_fused_score", 0)
        capi.set_option("score_tmp_doubles", 0)
    # an alphabet miss in the middle of a batch: the speculative pass's bytes are overwritten by the pass that stands
    digits = au.pack_strings_collection(["0123456789 QUIZ7", "ZEBRA9 J"])
    with_digits = (list(packed[:200]) + [digits] + list(packed[200:]), list(ms[:200]) + [2] + list(ms[200:]))
    exp_digits = _expect(_table(with_digits[0], with_digits[1], q), thr)
    try:
        capi.set_option("alphabet_sample", 100000)
        capi.set_option("pipeline_chunk", 40000)
        for fn in (_graph_host, _graph_dev):
            capi.set_option("forget_alphabet_guess", 1)
            idx, _ = fn(packed, ms, q, thr)   # leaves this batch's alphabet as the guess
            idx.close()
            idx, C = fn(with_digits[0], with_digits[1], q, thr)
            assert idx.stat("pipeline_miss") == 1 or idx.stat("alphabet_miss") == 1, fn.__name__
            idx.close()
            assert np.array_equal(C, exp_digits), fn.__name__
    finally:
        capi.set_option("alphabet_sample", 0)
        capi.set_option("pipeline_chunk", 0)
    # a document of more than 64 Ki code points: the global sort, then the scorer after the build
    big_col = utils.text_to_strings_collection(synth.document(90000, 78))
    batch = (packed[:5] + [au.pack_strings_collection(big_col)], ms[:5] + [len(big_col)])
    exp_big = _expect(_table(batch[0], batch[1], q), thr)
    for fn in (_graph_host, _graph_dev):
        idx, C = fn(batch[0], batch[1], q, thr)
        assert not idx.info()["doc_sorted"], fn.__name__
        idx.close()
        assert np.array_equal(C, exp_big), fn.__name__


@pytest.mark.gpu
def test_more_groups_than_the_kernel_keeps_in_shared_memory():
    import collections
    import synth
    from east import utils
    capi = _capi()
    texts, cols, packed, ms, _ = _collection(n_docs=40, n_bytes=2000, first_seed=9600)
    prepared = [utils.prepare_text(k) for k in synth.keyphrases(12300, seed=23)]
    codes, off, group_off = capi.pack_variant_groups(prepared, collections.defaultdict(list))
    q = (codes, off, group_off, True)
    table = _table(packed, ms, q)
    thr = _thresholds(table)[4]
    exp = _expect(table, thr)
    for fn in (_graph_host, _graph_dev):
        C, names = _kernels(fn, packed, ms, q, thr)
        assert "k_score_combine_max" in names and "k_threshold_bytes" in names, (fn.__name__, sorted(names))
        assert not any(n.endswith("_graph") for n in names), fn.__name__
        assert np.array_equal(C, exp), fn.__name__


@pytest.mark.gpu
def test_errors_are_raised_before_anything_is_built():
    capi = _capi()
    texts, cols, packed, ms, _ = _collection(n_docs=20, first_seed=9800)
    empty = capi.pack_variant_groups(["FOX", "DOG"], _defaultdict({"FOX": [""]}))   # the variant "" of FOX
    codes, off = capi.pack_keyphrases(["FOX", "DOG", "CAT"])
    bad = [(codes, off, np.array(g, dtype=np.int64), True) for g in ([0], [1, 3], [0, 2], [0, 2, 2, 3], [0, 4])]
    no_keyphrases = (np.zeros(1, dtype=np.uint32), np.zeros(1, dtype=np.int64), None, True)
    empty_plain = capi.pack_keyphrases(["FOX", ""])
    for fn, args in ((_graph_host, (packed, ms)), (_graph_dev, (packed, ms)), (_graph_texts, (texts,))):
        capi.launch_count(reset=True)
        with pytest.raises(ZeroDivisionError):
            fn(*args, (*empty, True), 0.1)
        with pytest.raises(ZeroDivisionError):
            fn(*args, (*empty_plain, None, True), 0.1)
        for g in bad:
            with pytest.raises(ValueError):
                fn(*args, g, 0.1)
        with pytest.raises(ValueError):
            fn(*args, no_keyphrases, 0.1)
        assert capi.launch_count() == 0, fn.__name__


def _public_collection(collection):
    import synth
    if collection == "hse":
        return _hse()
    docs = synth.documents(8, 3000, first_seed=8800)
    if collection == "several_batches":
        docs.insert(3, synth.documents(1, 90000, first_seed=600)[0])
    return {"t%d" % i: d for i, d in enumerate(docs)}, synth.keyphrases(30, seed=9)


def _table_route(kps, texts, r, c, p, measure, synonimizer=None):
    """keyphrases_graph as it was built before: the score table, then east_cooc_host"""
    from east import applications
    kept, _, scores = applications._score_matrix(kps, texts, measure, synonimizer, "english")
    cooc = _capi().cooc_host(scores, r) if scores.size else np.zeros((len(kept), len(kept)), dtype=np.int32)
    return applications.graph_from_cooccurrence(kps, kept, cooc, c, r, p)


def _no_table(monkeypatch):
    """make every way of forming a score table fail"""
    from east import _capi as capi

    def refuse(*a, **k):
        raise AssertionError("a score table was formed")
    monkeypatch.setattr(capi, "cooc_host", refuse)
    monkeypatch.setattr(capi.DeviceIndex, "build_host_and_score", classmethod(refuse))
    monkeypatch.setattr(capi.DeviceIndex, "table_from_texts", classmethod(refuse))
    monkeypatch.setattr(capi.DeviceIndex, "score_table", refuse)
    monkeypatch.setattr(capi.DeviceIndex, "score_groups", refuse)


@pytest.mark.gpu
@pytest.mark.parametrize("collection", ["ascii", "hse", "several_batches"])
@pytest.mark.parametrize("synonyms", [False, True])
def test_keyphrases_graph_without_a_table(golden, monkeypatch, collection, synonyms):
    from east import applications, relevance, utils
    texts, kps = _public_collection(collection)
    prepared = [utils.prepare_text(k) for k in kps if k]
    syn = None
    if synonyms:
        syn = _Synonimizer(_rich_synonyms(prepared) if collection != "hse" else _word_synonyms(prepared))
    settings = [(g["c"], g["r"], g["p"]) for g in golden["hse"]["graphs"]] + [(0.5, 0.0, 1), (0.5, 2.0, 1)]
    expect = [_table_route(kps, texts, r, c, p, relevance.ASTRelevanceMeasure(), syn) for c, r, p in settings]
    with monkeypatch.context() as m:
        _no_table(m)
        for (c, r, p), exp in zip(settings, expect):
            measure = relevance.ASTRelevanceMeasure()
            graph = applications.keyphrases_graph(kps, texts, c, r, p, similarity_measure=measure, synonimizer=syn)
            assert graph == exp, (c, r, p)
            assert measure._table is None and measure._cooc is not None
            assert len(measure._batches) == (2 if collection == "several_batches" else 1)
            assert (measure.asts[0]._strings_collection is None) == (collection != "several_batches")
    if collection == "hse" and not synonyms:
        for g in golden["hse"]["graphs"]:
            graph = applications.keyphrases_graph(kps, texts, g["c"], g["r"], g["p"],
                                                  similarity_measure=relevance.ASTRelevanceMeasure("easa", True))
            assert graph["nodes"] == g["nodes"]
            assert [(e["source"], e["target"], float(e["confidence"]).hex()) for e in graph["edges"]] == \
                   [(e["source"], e["target"], e["confidence"]) for e in g["edges"]]


@pytest.mark.gpu
def test_empty_keyphrases_and_collections_behave_as_before():
    import synth
    from east import applications, relevance
    texts = {"t%d" % i: d for i, d in enumerate(synth.documents(3, 2000, first_seed=50))}
    for kps, coll in (([], texts), (synth.keyphrases(5), {}), ([], {})):
        assert applications.keyphrases_graph(kps, coll, similarity_measure=relevance.ASTRelevanceMeasure()) == \
            _table_route(kps, coll, 0.25, 0.6, 1, relevance.ASTRelevanceMeasure())
    with pytest.raises(KeyError):
        applications.keyphrases_graph(["FOX", ""], texts, similarity_measure=relevance.ASTRelevanceMeasure())


@pytest.mark.gpu
@pytest.mark.parametrize("host", [False, True])
def test_counts_and_tables_never_stand_in_for_each_other(host):
    import synth
    from east import relevance, utils
    texts = synth.documents(6, 3000, first_seed=8900)
    prepared = [utils.prepare_text(k) for k in synth.keyphrases(30, seed=9)]
    syn = _Synonimizer(_rich_synonyms(prepared))
    fresh = relevance.ASTRelevanceMeasure("easa", False)
    fresh.set_text_collection(texts)
    plain, grouped = fresh.relevance_table(prepared), fresh.relevance_table(prepared, syn)
    capi = _capi()
    measure = relevance.ASTRelevanceMeasure("easa", False, device_preprocessing=not host)
    measure.set_text_collection(texts, prepared_keyphrases=prepared, relevance_threshold=0.3)
    stored = measure.cooccurrence(prepared, 0.3)
    assert stored is measure._cooc and np.array_equal(stored, capi.cooc_host(plain, 0.3))
    # a table after a graph is a table
    assert np.array_equal(measure.relevance_table(prepared).view(np.uint64), plain.view(np.uint64))
    # other thresholds, variants or normalization: the counts of the table
    for args, table in (((prepared, 0.2), plain), ((prepared, 0.3, syn), grouped)):
        got = measure.cooccurrence(*args)
        assert got is not measure._cooc and np.array_equal(got, capi.cooc_host(table, args[1])), args[1:]
    measure.normalized = True
    assert measure.cooccurrence(prepared, 0.3) is not measure._cooc
    measure.normalized = False
    # a graph after a table: counts, computed from the table that was scored while indexing
    measure.set_text_collection(texts, prepared_keyphrases=prepared, synonimizer=syn)
    assert measure._cooc is None
    assert np.array_equal(measure.cooccurrence(prepared, 0.3, syn), capi.cooc_host(grouped, 0.3))
    assert np.array_equal(measure.relevance_table(prepared, syn).view(np.uint64), grouped.view(np.uint64))
    measure.set_text_collection(texts, prepared_keyphrases=prepared, synonimizer=syn, relevance_threshold=0.3)
    assert measure._table is None
    assert np.array_equal(measure.cooccurrence(prepared, 0.3, syn), capi.cooc_host(grouped, 0.3))
    assert measure.cooccurrence(prepared, 0.3, syn) is measure._cooc
    assert np.array_equal(measure.relevance_table(prepared, syn).view(np.uint64), grouped.view(np.uint64))
    assert measure.cooccurrence(prepared, 0.3) is not measure._cooc


def _sharded_worker(rank, world, port, out_dir):
    import sys
    from conftest import PKG, ROOT
    for p in (PKG, ROOT):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from east import distributed

        def refuse(*a, **k):
            raise AssertionError("SymmetricTable constructed")
        distributed.SymmetricTable = refuse
        distributed.relevance_table_sharded = refuse
        docs, ragged, names, syn = _sharded_inputs()
        graphs = {}
        for key, collection in (("even", docs), ("ragged", ragged)):
            texts = {"t%d" % j: d for j, d in enumerate(collection)}
            graphs[key] = distributed.keyphrases_graph_sharded(names, texts, 0.5, 0.1, 1, device=rank)
            graphs[key + "_syn"] = distributed.keyphrases_graph_sharded(names, texts, 0.5, 0.1, 1, device=rank, synonimizer=syn)
        with open(os.path.join(out_dir, "graphs%d.json" % rank), "w") as f:
            json.dump(graphs, f)
    finally:
        dist.destroy_process_group()


def _sharded_inputs():
    import synth
    from east import utils
    docs = [synth.document(3000 + 1000 * (j % 4), 300 + j) for j in range(7)]
    names = synth.keyphrases(9)
    prepared = [utils.prepare_text(k) for k in names]
    ragged = docs[:3] + [synth.document(90000, 999)] + docs[3:]
    return docs, ragged, names, _Synonimizer(_rich_synonyms(prepared))


@pytest.mark.gpu
def test_two_gpu_sharded_graph_equals_one_gpu(tmp_path):
    import socket
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from east import applications, relevance
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_sharded_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    docs, ragged, names, syn = _sharded_inputs()
    for r in range(2):
        with open(str(tmp_path / ("graphs%d.json" % r))) as f:
            graphs = json.load(f)
        for key, collection in (("even", docs), ("ragged", ragged)):
            texts = {"t%d" % j: d for j, d in enumerate(collection)}
            for suffix, s_ in (("", None), ("_syn", syn)):
                one = applications.keyphrases_graph(names, texts, 0.5, 0.1, 1, similarity_measure=relevance.ASTRelevanceMeasure(),
                                                    synonimizer=s_)
                assert graphs[key + suffix] == json.loads(json.dumps(one)), (key + suffix, r)
