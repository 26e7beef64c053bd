"""Synonym-expanded keyphrase tables in ONE engine call (east_table_groups_host / _dev, east_table_texts_groups_host): the
per-document kernel keeps the best variant of every group itself (k_doc_suffix_sort_groups).  Every table is compared bit
for bit with the two-call path -- build, then DeviceIndex.score_groups, which is pinned to the oracle's group maximum by
test_gpu_synonyms.py -- and sampled rows with the oracle itself."""
import collections
import json
import os

import numpy as np
import pytest

from test_gpu_synonyms import _PerPair, _Synonimizer, _defaultdict, _hex, _oracle_groups, _reference_table, _rich_synonyms


def _capi():
    from east import _capi
    return _capi


def _concat(parts):
    doc_off = np.zeros(len(parts) + 1, dtype=np.int64)
    np.cumsum([len(p) for p in parts], out=doc_off[1:])
    return np.ascontiguousarray(np.concatenate(parts)), doc_off


def _groups(prepared, synonyms):
    return _capi().pack_variant_groups(prepared, synonyms)


def _two_call(packed, ms, codes, off, group_off):
    idx = _capi().DeviceIndex(packed, ms)
    try:
        return idx.score_groups(codes, off, group_off)
    finally:
        idx.close()


def _host(parts, ms, codes, off, group_off):
    text, doc_off = _concat(parts)
    out = np.full((len(ms), len(group_off) - 1), -1.0)
    idx = _capi().DeviceIndex.build_host_and_score(text, doc_off, ms, codes, off, out, group_off=group_off)
    return idx, out


def _dev(packed, ms, codes, off, group_off):
    import torch
    text, doc_off = _concat(packed)
    text_t = torch.from_numpy(text.view(np.int32)).cuda()
    kp_t = torch.from_numpy(codes.view(np.int32).copy()).cuda()
    out_t = torch.full((len(ms), len(group_off) - 1), -1.0, dtype=torch.float64, device="cuda")
    idx = _capi().DeviceIndex.build_dev_and_score(text_t.data_ptr(), doc_off, ms, kp_t.data_ptr(), codes, off, out_t.data_ptr(),
                                                  group_off=group_off)
    torch.cuda.synchronize()
    return idx, out_t.cpu().numpy()


def _texts(texts, codes, off, group_off):
    out = np.full((len(texts), len(group_off) - 1), -1.0)
    idx = _capi().DeviceIndex.table_from_texts(texts, codes, off, out, group_off=group_off)
    return idx, out


def _kernels(fn, *args):
    """(result of fn, names of the kernels it launched)"""
    capi = _capi()
    capi.set_option("time_kernels", 0)
    capi.set_option("time_kernels", 1)
    try:
        idx, out = fn(*args)
        idx.close()
        names = set(capi.kernel_stats())
    finally:
        capi.set_option("time_kernels", 0)
    return out, names


def _in_kernel(names):
    return ("k_doc_suffix_sort_groups" in names and "k_score_combine_max" not in names
            and not any(n.startswith("k_score_suffixes") for n in names))


def _collection(n_docs=300, n_bytes=1200, first_seed=9100, n_kps=40):
    import synth
    from east import utils
    from east.asts import utils as au
    texts = synth.documents(n_docs, n_bytes, first_seed)
    cols = [utils.text_to_strings_collection(t) for t in texts]
    packed = [au.pack_strings_collection(c) for c in cols]
    prepared = [utils.prepare_text(k) for k in synth.keyphrases(n_kps, seed=17)]
    codes, off, group_off = _groups(prepared, _rich_synonyms(prepared))
    sizes = np.diff(group_off)
    assert sizes.min() == 1 and sizes.max() > 1
    return texts, cols, packed, [len(c) for c in cols], codes, off, group_off


@pytest.mark.gpu
def test_every_one_call_entry_equals_the_two_call_path(oracle_mod):
    from east.asts import utils as au
    capi = _capi()
    texts, cols, packed, ms, codes, off, group_off = _collection()
    ref = _two_call(packed, ms, codes, off, group_off)
    for d in (0, 150, 299):
        assert _hex(ref[d]) == _hex(_oracle_groups(oracle_mod, packed[d], ms[d], codes, off, group_off)), d
    narrow = [au.pack_strings_collection_u8(c) for c in cols]
    try:
        capi.set_option("pipeline_chunk", 40000)   # several runs: the rows are scored while later runs are on their way
        for name, fn, parts in (("host width 4", _host, packed), ("host width 1", _host, narrow)):
            idx, out = fn(parts, ms, codes, off, group_off)
            assert idx.stat("pipelined") == 1 and idx.info()["doc_sorted"], name
            idx.close()
            assert _hex(out) == _hex(ref), name
            out, names = _kernels(fn, parts, ms, codes, off, group_off)
            assert _in_kernel(names) and _hex(out) == _hex(ref), (name, sorted(names))
    finally:
        capi.set_option("pipeline_chunk", 0)
    for name, fn, arg in (("dev", _dev, packed), ("texts", _texts, texts)):
        out, names = _kernels(fn, *((arg, ms) if name == "dev" else (arg,)), codes, off, group_off)
        assert _in_kernel(names), (name, sorted(names))
        assert _hex(out) == _hex(ref), name


@pytest.mark.gpu
def test_batched_tiled_alphabet_miss_and_large_document_paths(oracle_mod):
    import synth
    from east import utils
    from east.asts import utils as au
    capi = _capi()
    texts, cols, packed, ms, codes, off, group_off = _collection(first_seed=9500)
    ref = _two_call(packed, ms, codes, off, group_off)
    try:
        capi.set_option("no_fused_score", 1)   # the per-run batched scorer with groups
        for fn in (_host, _dev):
            out, names = _kernels(fn, packed, ms, codes, off, group_off)
            assert "k_score_combine_max" in names and "k_doc_suffix_sort_groups" not in names, fn.__name__
            assert _hex(out) == _hex(ref), fn.__name__
        capi.set_option("no_fused_score", 0)
        capi.set_option("score_tmp_doubles", int(off[-1]) * 4)   # a few documents per tile: tiled, overlapped
        for fn in (_host, _dev):
            out, names = _kernels(fn, packed, ms, codes, off, group_off)
            assert "k_score_combine_max" in names and "k_doc_suffix_sort_groups" not in names, fn.__name__
            assert _hex(out) == _hex(ref), fn.__name__
    finally:
        capi.set_option("no_fused_score", 0)
        capi.set_option("score_tmp_doubles", 0)
    # the alphabet of the previous batch is only a guess: new symbols in the middle redo the batch
    digits = au.pack_strings_collection(["0123456789 QUIZ7", "ZEBRA9 J"])
    with_digits = (list(packed[:200]) + [digits] + list(packed[200:]), list(ms[:200]) + [2] + list(ms[200:]))
    ref_digits = _two_call(with_digits[0], with_digits[1], codes, off, group_off)
    try:
        capi.set_option("alphabet_sample", 100000)   # device-resident batches above this size sample / guess
        capi.set_option("pipeline_chunk", 40000)     # host batches: pipelined, from the guess
        for fn in (_host, _dev):
            capi.set_option("forget_alphabet_guess", 1)        # (the reference build above left the digits in the guess)
            idx, out = fn(packed, ms, codes, off, group_off)   # leaves this batch's alphabet as the guess
            idx.close()
            idx, out = fn(with_digits[0], with_digits[1], codes, off, group_off)
            assert idx.stat("pipeline_miss") == 1 or idx.stat("alphabet_miss") == 1, fn.__name__
            idx.close()
            assert _hex(out) == _hex(ref_digits), fn.__name__
    finally:
        capi.set_option("alphabet_sample", 0)
        capi.set_option("pipeline_chunk", 0)
    assert _hex(ref_digits[200]) == _hex(_oracle_groups(oracle_mod, digits, 2, codes, off, group_off))
    # a document of more than 64 Ki code points: the global sort, then the grouped scorer after the build
    big_col = utils.text_to_strings_collection(synth.document(90000, 78))
    big = au.pack_strings_collection(big_col)
    batch = (packed[:5] + [big], ms[:5] + [len(big_col)])
    ref_big = _two_call(batch[0], batch[1], codes, off, group_off)
    for fn in (_host, _dev):
        idx, out = fn(batch[0], batch[1], codes, off, group_off)
        assert not idx.info()["doc_sorted"], fn.__name__
        idx.close()
        assert _hex(out) == _hex(ref_big), fn.__name__
    assert _hex(ref_big[5]) == _hex(_oracle_groups(oracle_mod, big, len(big_col), codes, off, group_off))


@pytest.mark.gpu
def test_single_variant_groups_equal_the_plain_normalized_table():
    capi = _capi()
    texts, cols, packed, ms, _, _, _ = _collection(n_docs=200, first_seed=9700)
    from east import utils
    import synth
    prepared = [utils.prepare_text(k) for k in synth.keyphrases(40, seed=17)]
    codes, off, group_off = _groups(prepared, collections.defaultdict(list))
    assert np.array_equal(group_off, np.arange(len(prepared) + 1))
    pcodes, poff = capi.pack_keyphrases(prepared)
    text, doc_off = _concat(packed)
    plain = np.empty((len(ms), len(prepared)))
    capi.DeviceIndex.build_host_and_score(text, doc_off, ms, pcodes, poff, plain, True).close()
    for fn in (_host, _dev):
        idx, out = fn(packed, ms, codes, off, group_off)
        idx.close()
        assert _hex(out) == _hex(plain), fn.__name__
    idx, out = _texts(texts, codes, off, group_off)
    idx.close()
    assert _hex(out) == _hex(plain)


@pytest.mark.gpu
def test_errors_are_raised_before_anything_is_built():
    capi = _capi()
    texts, cols, packed, ms, _, _, _ = _collection(n_docs=20, first_seed=9800)
    empty = _groups(["FOX", "DOG"], _defaultdict({"FOX": [""]}))   # the variant "" of FOX
    codes, off = capi.pack_keyphrases(["FOX", "DOG", "CAT"])
    bad = [(codes, off, np.array(g, dtype=np.int64)) for g in ([0], [1, 3], [0, 2], [0, 2, 2, 3], [0, 4])]
    for fn, args in ((_host, (packed, ms)), (_dev, (packed, ms)), (_texts, (texts,))):
        capi.launch_count(reset=True)
        with pytest.raises(ZeroDivisionError):
            fn(*args, *empty)
        for g in bad:
            with pytest.raises(ValueError):
                fn(*args, *g)
        assert capi.launch_count() == 0, fn.__name__


def _hse():
    from conftest import GOLDEN_DIR
    with open(os.path.join(GOLDEN_DIR, "golden.json"), encoding="utf-8") as f:
        hse = json.load(f)["hse"]
    with open(os.path.join(GOLDEN_DIR, "hse_texts.json"), encoding="utf-8") as f:
        raw = json.load(f)
    return {d["name"]: raw[d["name"]] for d in hse["docs"]}, hse["keyphrases"]


def _word_synonyms(prepared):
    """every third keyphrase word gets the next word as a synonym, one word also a synonym with a space"""
    from east import utils
    words = sorted({t for kp in prepared for t in utils.tokenize(kp)})
    syn = collections.defaultdict(list)
    for i in range(0, len(words) - 1, 3):
        syn[words[i]] = [words[i + 1]]
    syn[words[1]] = syn[words[1]] + [words[2] + " " + words[0]]
    return syn


@pytest.mark.gpu
@pytest.mark.parametrize("collection", ["ascii", "hse", "host_preprocessing", "several_batches"])
def test_keyphrases_table_and_graph_in_one_engine_call(oracle_mod, monkeypatch, collection):
    import synth
    from east import _capi as capi
    from east import applications, relevance, utils
    if collection == "hse":
        texts, kps = _hse()
    else:
        docs = synth.documents(8, 3000, first_seed=8800)
        if collection == "host_preprocessing":
            docs[2] = docs[2] + " ΑΛΦΑ ΒΗΤΑ"   # Greek: Python's Unicode tables, the host-packed path
        elif collection == "several_batches":
            docs.insert(3, synth.documents(1, 90000, first_seed=600)[0])
        texts = {"t%d" % i: d for i, d in enumerate(docs)}
        kps = synth.keyphrases(30, seed=9)
    prepared = [utils.prepare_text(k) for k in kps]
    syn = _Synonimizer(_rich_synonyms(prepared) if collection != "hse" else _word_synonyms(prepared))
    exp = _reference_table(oracle_mod, texts, prepared, syn.get_synonyms())
    pairs = applications.keyphrases_table(kps, texts, _PerPair(), synonimizer=syn)
    old = relevance.ASTRelevanceMeasure()     # the previous route: build, then the grouped call
    old.set_text_collection(list(texts.values()))
    old_table = old.relevance_table(prepared, syn)
    assert _hex(old_table) == _hex(exp)

    calls = []
    real = capi.DeviceIndex.score_groups
    monkeypatch.setattr(capi.DeviceIndex, "score_groups", lambda self, *a, **k: calls.append(1) or real(self, *a, **k))
    measure = relevance.ASTRelevanceMeasure()
    table = applications.keyphrases_table(kps, texts, measure, synonimizer=syn)
    assert not calls, "the table was scored while the collection was indexed"
    assert len(measure._batches) == (2 if collection == "several_batches" else 1)
    on_device = collection in ("ascii", "hse")
    assert (measure.asts[0]._strings_collection is None) == on_device   # raw texts: device preprocessing
    for k, kp in enumerate(kps):
        for j, name in enumerate(texts):
            assert float(table[kp][name]).hex() == float(exp[j, k]).hex(), (kp, name)
            assert type(table[kp][name]) is type(pairs[kp][name])
            assert float(pairs[kp][name]).hex() == float(exp[j, k]).hex(), (kp, name)
    graph = applications.keyphrases_graph(kps, texts, relevance_threshold=0.2, similarity_measure=relevance.ASTRelevanceMeasure(),
                                          synonimizer=syn)
    assert not calls
    assert graph == applications.keyphrases_graph(kps, texts, relevance_threshold=0.2, similarity_measure=_PerPair(),
                                                  synonimizer=syn)


@pytest.mark.gpu
def test_a_synonym_table_and_a_plain_table_never_stand_in_for_each_other():
    import synth
    from east import relevance, utils
    texts = synth.documents(6, 3000, first_seed=8900)
    prepared = [utils.prepare_text(k) for k in synth.keyphrases(30, seed=9)]
    syn = _Synonimizer(_rich_synonyms(prepared))
    other = _Synonimizer(_defaultdict({}))
    fresh = relevance.ASTRelevanceMeasure("easa", False)   # unnormalized: plain and synonym tables differ everywhere
    fresh.set_text_collection(texts)
    plain, grouped, grouped_other = (fresh.relevance_table(prepared), fresh.relevance_table(prepared, syn),
                                     fresh.relevance_table(prepared, other))
    assert _hex(plain) != _hex(grouped) and _hex(grouped) != _hex(grouped_other)
    for host in (False, True):
        measure = relevance.ASTRelevanceMeasure("easa", False, device_preprocessing=not host)
        measure.set_text_collection(texts, prepared_keyphrases=prepared, synonimizer=syn)
        assert _hex(measure.relevance_table(prepared, syn)) == _hex(grouped)
        assert measure.relevance_table(prepared, syn) is measure._table
        assert _hex(measure.relevance_table(prepared)) == _hex(plain)
        assert _hex(measure.relevance_table(prepared, other)) == _hex(grouped_other)   # re-packing differs
        measure.set_text_collection(texts, prepared_keyphrases=prepared)
        assert _hex(measure.relevance_table(prepared, syn)) == _hex(grouped)
        assert _hex(measure.relevance_table(prepared)) == _hex(plain)


@pytest.mark.gpu
def test_benchmark_sized_collection(oracle_mod):
    # the headline collection of bench.py (10^3 documents of 50 KB) with the seeded dictionary of its 10^3 keyphrases
    import torch
    import synth
    from east import utils
    capi = _capi()
    prepared = [utils.prepare_text(k) for k in synth.keyphrases(1000)]
    codes, off, group_off = _groups(prepared, synth.synonyms(prepared))
    text, doc_off, doc_m = synth.packed_collection_fast(1000, 50000)
    text_t = torch.from_numpy(text.view(np.int32)).cuda()
    kp_t = torch.from_numpy(codes.view(np.int32).copy()).cuda()
    out_t = torch.full((1000, len(prepared)), -1.0, dtype=torch.float64, device="cuda")
    capi.set_option("time_kernels", 0)
    capi.set_option("time_kernels", 1)
    try:
        capi.DeviceIndex.build_dev_and_score(text_t.data_ptr(), doc_off, doc_m, kp_t.data_ptr(), codes, off, out_t.data_ptr(),
                                             group_off=group_off).close()
        names = set(capi.kernel_stats())   # (the event pairs are read once the call's work is done)
    finally:
        capi.set_option("time_kernels", 0)
    assert _in_kernel(names), sorted(names)
    table = out_t.cpu().numpy()
    idx = capi.DeviceIndex.build_dev(text_t.data_ptr(), doc_off, doc_m)
    ref = idx.score_groups(codes, off, group_off)
    idx.close()
    assert _hex(table) == _hex(ref)
    for d in (0, 500, 999):
        seg = text[doc_off[d]:doc_off[d + 1]]
        assert _hex(table[d]) == _hex(_oracle_groups(oracle_mod, seg, int(doc_m[d]), codes, off, group_off)), d


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
        from east import _capi, distributed
        docs, prepared, syn, ragged, names = _sharded_inputs()

        def save(name, t):
            np.save(os.path.join(out_dir, "%s%d.npy" % (name, rank)), t.cpu().numpy())
        save("fused", distributed.relevance_table_sharded(docs, prepared, device=rank, synonimizer=syn))
        save("gather", distributed.relevance_table_sharded(docs, prepared, device=rank, fused_gather=False, synonimizer=syn))
        try:
            _capi.set_option("score_tmp_doubles", 150)   # the batched scorer stores the rows to the peers
            save("tiled", distributed.relevance_table_sharded(docs, prepared, device=rank, synonimizer=syn))
        finally:
            _capi.set_option("score_tmp_doubles", 0)
        save("ragged", distributed.relevance_table_sharded(ragged, prepared, device=rank, synonimizer=syn))
        graph = distributed.keyphrases_graph_sharded(names, {"t%d" % j: d for j, d in enumerate(docs)}, 0.5, 0.1, 1, device=rank,
                                                     synonimizer=syn)
        with open(os.path.join(out_dir, "graph%d.json" % rank), "w") as f:
            json.dump(graph, f)
    finally:
        dist.destroy_process_group()


def _sharded_inputs():
    import synth
    from east import utils
    docs = [synth.document(3000 + 1000 * (j % 4), 300 + j) for j in range(7)]
    names = synth.keyphrases(9)
    prepared = [utils.prepare_text(k) for k in names]
    ragged = docs[:3] + [synth.document(90000, 999)] + docs[3:]
    return docs, prepared, _Synonimizer(_rich_synonyms(prepared)), ragged, names


@pytest.mark.gpu
def test_two_gpu_sharded_synonym_tables_equal_one_gpu(tmp_path):
    import socket
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from east import applications, relevance
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_sharded_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    docs, prepared, syn, ragged, names = _sharded_inputs()
    expect = {}
    for key, collection in (("plain", docs), ("ragged", ragged)):
        measure = relevance.ASTRelevanceMeasure()
        measure.set_text_collection(collection)
        expect[key] = measure.relevance_table(prepared, syn)
    graph = applications.keyphrases_graph(names, {"t%d" % j: d for j, d in enumerate(docs)}, 0.5, 0.1, 1,
                                          similarity_measure=relevance.ASTRelevanceMeasure(), synonimizer=syn)
    for r in range(2):
        for name in ("fused", "gather", "tiled"):
            assert _hex(np.load(str(tmp_path / ("%s%d.npy" % (name, r))))) == _hex(expect["plain"]), (name, r)
        assert _hex(np.load(str(tmp_path / ("ragged%d.npy" % r)))) == _hex(expect["ragged"]), r
        with open(str(tmp_path / ("graph%d.json" % r))) as f:
            assert json.load(f) == json.loads(json.dumps(graph))
