"""Synonym-expanded scoring (easa.py:27-34): the score of a keyphrase with a synonimizer is the best normalized score
over every substitution of its words by their synonyms.  CPU tests of the variant expansion and its packing; GPU tests
of the grouped scoring call (east_score_groups_host, k_score_combine_max) bit for bit against the CPU oracle's maximum
over each group."""
import collections

import numpy as np
import pytest


def _capi():
    from east import _capi
    return _capi


class _Synonimizer(object):
    def __init__(self, synonyms):
        self.synonyms = synonyms

    def get_synonyms(self):
        return self.synonyms


def _defaultdict(d):
    out = collections.defaultdict(list)
    out.update(d)
    return out


# ---- variant expansion (host) ----------------------------------------------------------------------------------------

def test_variants_of_unknown_words_with_a_defaultdict_and_keyerror_with_a_dict():
    from east import utils
    syn = _defaultdict({"QUICK": ["FAST", "SPEEDY"]})
    assert utils.synonym_variants("QUICK FOX", syn) == ["FASTFOX", "SPEEDYFOX", "QUICKFOX"]
    assert utils.synonym_variants("LAZY DOG", syn) == ["LAZYDOG"]
    with pytest.raises(KeyError):
        utils.synonym_variants("QUICK FOX", {"QUICK": ["FAST"]})


def test_variant_keeps_the_space_of_a_synonym():
    from east import utils
    assert utils.synonym_variants("CAR PARK", _defaultdict({"CAR": ["RED CAR"]})) == ["RED CARPARK", "CARPARK"]


def test_empty_synonym_duplicate_variants_and_a_tokenless_keyphrase():
    from east import utils
    syn = _defaultdict({"AB": ["ABCD", ""], "CD": [""]})
    assert utils.synonym_variants("AB CD", syn) == ["ABCD", "ABCDCD", "", "CD", "AB", "ABCD"]   # "ABCD" twice
    assert utils.synonym_variants("AB", syn) == ["ABCD", "", "AB"]
    assert utils.synonym_variants("!!! ...", syn) == [""]
    assert utils.synonym_variants("", syn) == [""]


def test_group_offsets_of_the_packed_variants():
    capi = _capi()
    syn = _defaultdict({"QUICK": ["FAST", "A B"], "FOX": ["ਅX"]})
    codes, off, group_off = capi.pack_variant_groups(["QUICK FOX", "DOG", "!!"], syn)
    assert group_off.tolist() == [0, 6, 7, 8]
    variants = ["FASTਅX", "FASTFOX", "A BਅX", "A BFOX", "QUICKਅX", "QUICKFOX", "DOG", ""]
    assert off.tolist() == [0] + np.cumsum([len(v) for v in variants]).tolist()
    assert codes.dtype == np.uint32 and codes.tolist() == [ord(c) for c in "".join(variants)]
    codes, off, group_off = capi.pack_variant_groups([], syn)
    assert codes.size == 0 and off.tolist() == [0] and group_off.tolist() == [0]


def test_seeded_dictionary_of_the_benchmark():
    import synth
    from east import utils
    kps = [utils.prepare_text(k) for k in synth.keyphrases(1000)]
    codes, off, group_off = _capi().pack_variant_groups(kps, synth.synonyms(kps))
    assert len(off) - 1 == 9277 and int(np.diff(group_off).max()) == 64 and int(off[-1]) == 159333


# ---- grouped scoring on the device ----------------------------------------------------------------------------------

def _group_max(scores, group_off):
    """max(...) of easa.py:34 over each group, starting from the group's first variant"""
    out = np.empty(len(group_off) - 1, dtype=np.float64)
    for g in range(len(group_off) - 1):
        best = scores[group_off[g]]
        for v in range(group_off[g] + 1, group_off[g + 1]):
            if scores[v] > best:
                best = scores[v]
        out[g] = best
    return out


def _oracle_groups(oracle_mod, text, m, codes, off, group_off):
    return _group_max(oracle_mod.OracleEASA(text=text, m=m).score_many(codes, off, True), group_off)


def _hex(a):
    return [float(x).hex() for x in np.ravel(a)]


def _rich_synonyms(prepared):
    """synth.synonyms plus, for one word, a synonym with a space, one with code points >= 0x0A00 and the word itself
    (duplicate variants)"""
    import synth
    from east import utils
    syn = _defaultdict(synth.synonyms(prepared))
    words = sorted({t for kp in prepared for t in utils.tokenize(kp)})
    syn[words[0]] = syn[words[0]] + [words[1] + " " + words[2], "中文" + words[0], words[0]]
    return syn


@pytest.mark.gpu
def test_grouped_table_on_both_build_paths(oracle_mod):
    import synth
    from east import utils
    from east.asts import utils as au
    capi = _capi()
    kps = [utils.prepare_text(k) for k in synth.keyphrases(60)]
    codes, off, group_off = capi.pack_variant_groups(kps, _rich_synonyms(kps))
    packed, ms, _ = synth.packed_collection(4, 4000, first_seed=31)
    small = capi.DeviceIndex(packed, ms)
    assert small.info()["doc_sorted"]
    big_col = utils.text_to_strings_collection(synth.document(90000, 77))
    big = au.pack_strings_collection(big_col)
    large = capi.DeviceIndex([big], [len(big_col)])
    assert big.size > 65535 and not large.info()["doc_sorted"]
    for idx, texts, tms in ((small, packed, ms), (large, [big], [len(big_col)])):
        table = idx.score_groups(codes, off, group_off)
        assert table.shape == (len(texts), len(kps))
        for d in range(len(texts)):
            assert _hex(table[d]) == _hex(_oracle_groups(oracle_mod, texts[d], tms[d], codes, off, group_off)), d
        # a document range: the rows of those documents
        if len(texts) > 1:
            part = idx.score_groups(codes, off, group_off, doc_begin=1, doc_count=2)
            assert _hex(part) == _hex(table[1:3])


@pytest.mark.gpu
def test_fast_and_generic_walks_with_code_points_beyond_the_terminators(oracle_mod):
    from east.asts import utils as au
    capi = _capi()
    strings = ["FOXDOG", "QUICKFOX", "THEXLAZY", "FOXFOX"]
    packed = au.pack_strings_collection(strings)
    syn = _defaultdict({"QUICK": ["中文", "FAST"], "FOX": ["ਅX", "DOG"]})
    codes, off, group_off = capi.pack_variant_groups(["QUICK FOX", "FOX", "LAZY DOG"], syn)
    exp = _oracle_groups(oracle_mod, packed, len(strings), codes, off, group_off)
    idx = capi.DeviceIndex([packed], [len(strings)])
    assert idx.info()["fast_path"]
    fast = idx.score_groups(codes, off, group_off)
    try:
        capi.set_option("score_generic", 1)
        generic = idx.score_groups(codes, off, group_off)
    finally:
        capi.set_option("score_generic", 0)
    assert _hex(fast[0]) == _hex(exp) and _hex(generic[0]) == _hex(exp)


@pytest.mark.gpu
def test_a_spaced_synonym_is_scored_with_its_space(oracle_mod):
    from east.asts import base
    from east.asts import utils as au
    capi = _capi()
    strings = ["A RED CAR", "BLUE"]
    syn = _Synonimizer(_defaultdict({"CAR": ["RED CAR"]}))
    codes, off, group_off = capi.pack_variant_groups(["CAR"], syn.get_synonyms())
    packed = au.pack_strings_collection(strings)
    exp = _oracle_groups(oracle_mod, packed, 2, codes, off, group_off)
    stripped, soff = capi.pack_keyphrases(["RED CAR", "CAR"])
    exp_stripped = _group_max(oracle_mod.OracleEASA(text=packed, m=2).score_many(stripped, soff, True), [0, 2])
    assert float(exp[0]) != float(exp_stripped[0])
    ast = base.AST.get_ast(strings)
    got = ast.score("CAR", synonimizer=syn)
    assert isinstance(got, np.float64) and float(got).hex() == float(exp[0]).hex()
    assert ast.score("NOTHING", synonimizer=syn) == 0 and type(ast.score("NOTHING", synonimizer=syn)) is int


def _collection_texts():
    import synth
    docs = synth.documents(6, 3000, first_seed=500)
    docs.insert(3, synth.documents(1, 90000, first_seed=600)[0])   # ~82 k code points: a second device batch
    return {"t%d" % i: d for i, d in enumerate(docs)}


def _reference_table(oracle_mod, texts, prepared, synonyms):
    from east import utils
    codes, off, group_off = _capi().pack_variant_groups(prepared, synonyms)
    rows = []
    for t in texts.values():
        o = oracle_mod.OracleEASA(utils.text_to_strings_collection(t))
        rows.append(_group_max(o.score_many(codes, off, True), group_off))
    return np.array(rows)


@pytest.mark.gpu
def test_several_device_batches_and_a_loaded_index(oracle_mod, tmp_path):
    import synth
    from east import relevance, utils
    texts = _collection_texts()
    prepared = [utils.prepare_text(k) for k in synth.keyphrases(40, seed=21)]
    syn = _Synonimizer(_rich_synonyms(prepared))
    measure = relevance.ASTRelevanceMeasure("easa", True)
    measure.set_text_collection(list(texts.values()))
    assert len(measure._batches) == 2
    table = measure.relevance_table(prepared, syn)
    exp = _reference_table(oracle_mod, texts, prepared, syn.get_synonyms())
    assert _hex(table) == _hex(exp)
    measure.save_index(str(tmp_path / "collection"))
    loaded = relevance.ASTRelevanceMeasure.load_index(str(tmp_path / "collection"))
    assert _hex(loaded.relevance_table(prepared, syn)) == _hex(exp)
    assert float(loaded.relevance(prepared[0], text=3, synonimizer=syn)).hex() == float(exp[3, 0]).hex()


@pytest.mark.gpu
def test_overlapped_tiles_equal_one_tile():
    import synth
    from east import utils
    capi = _capi()
    prepared = [utils.prepare_text(k) for k in synth.keyphrases(50, seed=5)]
    codes, off, group_off = capi.pack_variant_groups(prepared, _rich_synonyms(prepared))
    packed, ms, _ = synth.packed_collection(40, 2000, first_seed=700)
    idx = capi.DeviceIndex(packed, ms)
    one = idx.score_groups(codes, off, group_off)
    try:
        # n_uniq <= total suffixes: at most a few documents per tile, many tiles -> the two-halves branch
        capi.set_option("score_tmp_doubles", int(off[-1]) * 4)
        tiled = idx.score_groups(codes, off, group_off)
        capi.set_option("score_no_overlap", 1)
        plain = idx.score_groups(codes, off, group_off)
    finally:
        capi.set_option("score_tmp_doubles", 0)
        capi.set_option("score_no_overlap", 0)
    assert _hex(tiled) == _hex(one) and _hex(plain) == _hex(one)


@pytest.mark.gpu
def test_benchmark_sized_documents_past_the_one_kernel_preparation(oracle_mod):
    # 50 KB documents, the keyphrases of the benchmark and the seeded dictionary: 159 k query suffixes, more than the
    # 64 Ki the one-cluster preparation takes (sampled rows checked)
    import synth
    from east import utils
    capi = _capi()
    prepared = [utils.prepare_text(k) for k in synth.keyphrases(1000)]
    codes, off, group_off = capi.pack_variant_groups(prepared, synth.synonyms(prepared))
    assert off[-1] > 65536
    packed, ms, _ = synth.packed_collection(6, 50000, first_seed=40)
    idx = capi.DeviceIndex(packed, ms)
    table = idx.score_groups(codes, off, group_off)
    for d in (0, 5):
        assert _hex(table[d]) == _hex(_oracle_groups(oracle_mod, packed[d], ms[d], codes, off, group_off)), d


class _PerPair(object):
    """A measure that is not an ASTRelevanceMeasure: keyphrases_table scores it pair by pair, as the reference does"""

    def __init__(self):
        from east import relevance
        self.inner = relevance.ASTRelevanceMeasure("easa", True)

    def set_text_collection(self, texts, language=None):
        self.inner.set_text_collection(texts)

    def relevance(self, keyphrase, text, synonimizer=None):
        return self.inner.relevance(keyphrase, text, synonimizer)


@pytest.mark.gpu
def test_keyphrases_table_and_graph_with_a_synonimizer(oracle_mod):
    import synth
    from east import applications, relevance, utils
    texts = {"t%d" % i: d for i, d in enumerate(synth.documents(8, 3000, first_seed=800))}
    kps = synth.keyphrases(30, seed=9)
    prepared = [utils.prepare_text(k) for k in kps]
    syn = _Synonimizer(_rich_synonyms(prepared))
    exp = _reference_table(oracle_mod, texts, prepared, syn.get_synonyms())
    table = applications.keyphrases_table(kps, texts, relevance.ASTRelevanceMeasure(), synonimizer=syn)
    pairs = applications.keyphrases_table(kps, texts, _PerPair(), synonimizer=syn)
    for k, kp in enumerate(kps):
        for j, name in enumerate(texts):
            assert float(table[kp][name]).hex() == float(exp[j, k]).hex(), (kp, name)
            assert type(table[kp][name]) is type(pairs[kp][name])
            assert float(pairs[kp][name]).hex() == float(exp[j, k]).hex(), (kp, name)
    graph = applications.keyphrases_graph(kps, texts, relevance_threshold=0.2, similarity_measure=relevance.ASTRelevanceMeasure(),
                                          synonimizer=syn)
    assert graph == applications.keyphrases_graph(kps, texts, relevance_threshold=0.2, similarity_measure=_PerPair(),
                                                  synonimizer=syn)


@pytest.mark.gpu
def test_synonym_scores_are_normalized_whatever_the_measure_says():
    import synth
    from east import relevance, utils
    texts = [synth.document(3000, 900 + i) for i in range(4)]
    prepared = [utils.prepare_text(k) for k in synth.keyphrases(20, seed=3)]
    syn = _Synonimizer(_rich_synonyms(prepared))
    tables = []
    for normalized in (True, False):
        measure = relevance.ASTRelevanceMeasure("easa", normalized)
        measure.set_text_collection(texts)
        tables.append(measure.relevance_table(prepared, syn))
    assert _hex(tables[0]) == _hex(tables[1])
    assert not np.array_equal(measure.relevance_table(prepared), tables[0])   # without synonyms it is unnormalized


@pytest.mark.gpu
def test_tokenless_keyphrase_raises_zero_division():
    from east import relevance
    from east.asts import base
    syn = _Synonimizer(_defaultdict({"FOX": ["DOG"]}))
    ast = base.AST.get_ast(["QUICKFOX", "DOG"])
    with pytest.raises(ZeroDivisionError):
        ast.score("!!!", synonimizer=syn)
    with pytest.raises(ZeroDivisionError):
        ast.score("FOX", synonimizer=_Synonimizer(_defaultdict({"FOX": [""]})))   # the empty variant
    measure = relevance.ASTRelevanceMeasure()
    measure.set_text_collection(["the quick fox and the lazy dog"])
    with pytest.raises(ZeroDivisionError):
        measure.relevance_table(["FOX", "..."], syn)


@pytest.mark.gpu
def test_malformed_group_offsets_are_rejected():
    from east.asts import utils as au
    capi = _capi()
    strings = ["QUICKFOX", "DOG"]
    idx = capi.DeviceIndex([au.pack_strings_collection(strings)], [2])
    codes, off = capi.pack_keyphrases(["FOX", "DOG", "CAT"])
    assert idx.score_groups(codes, off, [0, 2, 3]).shape == (1, 2)
    for bad in ([0], [], [1, 3], [0, 2], [0, 2, 2, 3], [0, 3, 2, 3], [0, 4]):
        with pytest.raises(ValueError):
            idx.score_groups(codes, off, bad)
    for begin, count in ((1, 1), (-1, 1), (0, 0)):
        with pytest.raises(ValueError):
            idx.score_groups(codes, off, [0, 3], doc_begin=begin, doc_count=count)
