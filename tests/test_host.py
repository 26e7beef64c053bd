"""CPU: host-side mirror of the EAST API and the C-ABI surface (no compute without a GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT, have_gpu


def test_tokenize_reference_known_answer(golden):
    from east import utils
    # tests/test_utils.py:10-13
    assert utils.tokenize("Well, what a sunny day!") == ["Well", "what", "a", "sunny", "day"]
    assert utils.tokenize(golden["prep"]["tokenize"]["in"]) == golden["prep"]["tokenize"]["out"]


def test_text_to_strings_collection_matches_reference(golden):
    from east import utils
    for item in golden["prep"]["collections"]:
        assert utils.text_to_strings_collection(item["in"]) == item["out"]
    assert utils.text_to_strings_collection("") == [" "]
    assert utils.prepare_text(b"caf\xc3\xa9 \xff") == "CAFÉ �"  # upper-case, errors=replace


def test_asts_utils_known_answers():
    from east.asts import utils
    # tests/asts/test_utils.py:10-30
    assert utils.match_strings("", "") == 0 and utils.match_strings("a", "") == 0
    assert utils.match_strings("a", "ab") == 1 and utils.match_strings("abc", "abd") == 2
    assert utils.match_strings("abc", "abc") == 3 and utils.match_strings("abcd", "abc") == 3
    assert utils.index([1, 2, 3, 2], 2) == 1 and utils.index([1, 2, 3, 2], 2, 2) == 3
    assert utils.index("abcabc", "c", 3) == 5
    assert utils.make_unique_endings(["ab", "c"]) == ["ab਀", "cਁ"]


def test_pack_strings_collection(oracle_mod):
    from east.asts import utils
    for strings in (["XABXAC", "HI"], [" "], ["", "A", ""], ["Жук", "x" * 50, "\U0001F600!"]):
        packed = utils.pack_strings_collection(strings)
        assert packed.dtype == np.uint32
        expect = [ord(ch) for s in utils.make_unique_endings(strings) for ch in s]
        assert packed.tolist() == expect
        assert np.array_equal(packed, oracle_mod.pack(strings))
    # no 0x110000 cap on the number of strings
    many = utils.pack_strings_collection(["A"] * 1200000)
    assert many[-1] == 0x0A00 + 1199999


def test_registry_and_exceptions(golden):
    import east  # noqa: F401  (registers engines)
    from east import consts, exceptions
    from east.asts import base, easa
    assert golden["errors"] == {"empty_collection": "EmptyStringsCollectionException",
                                "unknown_algorithm": "NoSuchASTAlgorithm"}
    with pytest.raises(exceptions.EmptyStringsCollectionException):
        base.AST.get_ast([])
    with pytest.raises(exceptions.NoSuchASTAlgorithm) as ei:
        base.AST.get_ast(["A"], "nope")
    assert "nope" in str(ei.value)
    assert easa.EnhancedAnnotatedSuffixArray.__algorithm__ == consts.ASTAlgorithm.EASA == "easa"
    assert consts.String.UNICODE_SPECIAL_SYMBOLS_START == 0x0A00
    with pytest.raises(TypeError):
        consts.String.UNICODE_SPECIAL_SYMBOLS_START = 1
    assert sorted(consts.ASTAlgorithm) == ["ast_linear", "ast_naive", "easa"]


def test_capi_library_exports_every_declared_symbol():
    from east import _capi
    header = open(os.path.join(ROOT, "include", "east_b200.h")).read()
    declared = set(re.findall(r"\b(east_[a-z_0-9]+)\s*\(", header))
    declared.discard("east_index")
    assert declared == set(_capi.EXPORTED_SYMBOLS)
    assert os.path.exists(_capi.LIB_PATH), "build the engine first: python -c 'import __graft_entry__ as g; g.build()'"
    lib = ctypes.CDLL(_capi.LIB_PATH)
    for sym in sorted(declared):
        assert hasattr(lib, sym), sym
    assert b"sm_100a" in ctypes.c_char_p(ctypes.cast(lib.east_version, ctypes.CFUNCTYPE(ctypes.c_char_p))()).value


@pytest.mark.skipif(have_gpu(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback_without_gpu():
    from east import exceptions
    from east.asts import base
    with pytest.raises(exceptions.DeviceError):
        base.AST.get_ast(["XABXAC", "HI"])
    from east import applications
    with pytest.raises(exceptions.DeviceError):
        applications.keyphrases_table(["abc"], {"t": "some text here"})


def test_argument_validation_needs_no_gpu():
    from east import _capi
    L = _capi.load()
    h = ctypes.c_void_p()
    text = np.array([65, 0x0A00], dtype=np.uint32)
    off = np.array([0, 0], dtype=np.int64)  # empty document
    m = np.array([1], dtype=np.int32)
    rc = L.east_build_host(text.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)),
                           off.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
                           m.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), 1, 0, ctypes.byref(h))
    assert rc == -1 and b"empty document" in L.east_last_error()
    # the one-call entry validates the documents AND the keyphrases before it touches the device: an empty
    # query is the reference's ZeroDivisionError (easa.py:134), whatever else would happen later
    out = np.zeros((1, 2))
    with pytest.raises(ValueError):
        _capi.DeviceIndex.build_host_and_score(text, off, m, np.array([65], dtype=np.uint32), np.array([0, 1, 1]), out)
    good_off = np.array([0, 2], dtype=np.int64)
    with pytest.raises(ZeroDivisionError):
        _capi.DeviceIndex.build_host_and_score(text, good_off, m, np.array([65], dtype=np.uint32), np.array([0, 1, 1]), out)


def test_every_build_and_score_entry_checks_its_arguments_in_one_order_without_a_gpu():
    # every check runs before the first CUDA call (no DeviceError without a GPU, no fake pointer is ever dereferenced),
    # in one order: output, documents (raw texts: their offsets), groups, keyphrases
    from east import _capi
    Dx = _capi.DeviceIndex
    fake = 1 << 20   # device addresses the calls must never reach
    text32, text8 = np.array([65, 0x0A00], dtype=np.uint32), np.array([65, 0xFF], dtype=np.uint8)
    m = np.array([1], dtype=np.int32)
    docs = {"bad": np.array([0, 0], dtype=np.int64), "good": np.array([0, 2], dtype=np.int64)}
    texts = {"bad": (np.frombuffer(b"ABC DEF", dtype=np.uint8), np.array([0, 7, 3], dtype=np.int64)),
             "good": (np.frombuffer(b"ABC DEF", dtype=np.uint8), np.array([0, 3, 7], dtype=np.int64))}
    codes, empty_kp = np.array([65], dtype=np.uint32), np.array([0, 1, 1], dtype=np.int64)   # the second keyphrase is empty
    groups, bad_groups = np.array([0, 2], dtype=np.int64), np.array([0, 3], dtype=np.int64)

    def table(n, g):
        return np.zeros((n, 2 if g is None else len(g) - 1))

    def host(t):
        return lambda d, g: Dx.build_host_and_score(t, docs[d], m, codes, empty_kp, table(1, g), group_off=g)

    entries = {   # C entry: call(documents, group_off)
        "east_table_host": host(text32),
        "east_table_host_u8": host(text8),
        "east_table_host_gather": lambda d, g: Dx.build_host_and_score(text32, docs[d], m, codes, empty_kp, table(1, g),
                                                                       own_rows=fake),
        "east_table_dev": lambda d, g: Dx.build_dev_and_score(fake, docs[d], m, fake, None, empty_kp, fake),   # no host copy
        "east_table_dev_gather": lambda d, g: Dx.build_dev_and_score(fake, docs[d], m, fake, codes, empty_kp, fake,
                                                                     peer_rows=[fake]),
        "east_table_texts_host": lambda d, g: Dx.table_from_texts(texts[d], codes, empty_kp, table(2, g)),
        "east_table_groups_host": host(text32),
        "east_table_groups_dev": lambda d, g: Dx.build_dev_and_score(fake, docs[d], m, fake, codes, empty_kp, fake, group_off=g),
        "east_table_texts_groups_host": lambda d, g: Dx.table_from_texts(texts[d], codes, empty_kp, table(2, g),
                                                                         group_off=g),
        "east_graph_host": lambda d, g: Dx.build_host_and_graph(text32, docs[d], m, codes, empty_kp, 0.5, group_off=g),
        "east_graph_dev": lambda d, g: Dx.build_dev_and_graph(fake, docs[d], m, fake, None, empty_kp, 0.5, fake, group_off=g),
        "east_graph_texts_host": lambda d, g: Dx.graph_from_texts(texts[d], codes, empty_kp, 0.5, group_off=g),
    }
    for name, call in entries.items():
        # the groups entries always take groups; the graph entries with and without them
        for g in ([groups] if "_groups_" in name else [None, groups] if "_graph_" in name else [None]):
            with pytest.raises(ValueError):   # malformed documents before the empty keyphrase
                call("bad", g)
            with pytest.raises(ZeroDivisionError):
                call("good", g)
        if "_groups_" in name or "_graph_" in name:
            with pytest.raises(ValueError):   # malformed groups before the empty keyphrase
                call("good", bad_groups)
    # the score calls on an index: a NULL index before the (empty) keyphrases
    L = _capi.load()
    kp, off = codes.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)), empty_kp.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
    gp = groups.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
    out = np.zeros(4).ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    probes, score = ctypes.c_int64(), ctypes.c_double()
    for rc in (L.east_score_table_host(None, kp, off, 2, 1, out),
               L.east_score_table_dev(None, fake, off, 2, 1, fake, None),
               L.east_score_range_dev(None, fake, off, 2, 1, 0, 1, fake, None),
               L.east_score_probes_dev(None, fake, off, 2, fake, None, ctypes.byref(probes)),
               L.east_score_groups_host(None, kp, off, 2, gp, 1, 0, 1, out),
               L.east_score_groups_dev(None, fake, off, 2, gp, 1, 0, 1, fake, None),
               L.east_score_one(None, 0, kp, 0, 1, ctypes.byref(score), None)):
        assert rc == -1, L.east_last_error()


def test_synthetic_generator_is_deterministic():
    import synth
    d1, d2 = synth.document(10000, 1), synth.document(10000, 1)
    assert d1 == d2 and len(d1) == 10000 and d1 != synth.document(10000, 2)
    kps = synth.keyphrases(50)
    assert kps == synth.keyphrases(50) and all(1 <= len(k.split(" ")) <= 3 for k in kps)
    from east import utils
    col = utils.text_to_strings_collection(d1)
    n = sum(len(s) for s in col) + len(col)
    assert 0.85 < n / 10000.0 < 0.97  # SURVEY 8: n ~ 0.911 x bytes


def test_plan_batches_separates_large_documents_and_bounds_the_batch():
    from east.relevance import plan_batches
    sizes = [100, 70000, 200, 300, 65535, 65536, 50]
    assert plan_batches(sizes) == [[0, 2, 3, 4, 6], [1, 5]]
    assert plan_batches([10, 20, 30, 40], small_limit=100, max_batch=50) == [[0, 1], [2], [3]]
    assert plan_batches([500, 10, 500], small_limit=100, max_batch=600) == [[1], [0], [2]]
    assert plan_batches([]) == []
    flat = sorted(j for b in plan_batches(list(range(1, 200)), small_limit=50, max_batch=300) for j in b)
    assert flat == list(range(199))


def test_host_preprocessing_reproduces_the_reference_on_its_sample_corpus(golden):
    # raw texts of doc/samples (tests/golden/hse_texts.json) -> the strings collections the REFERENCE produced (golden.json)
    import json
    from east import utils
    with open(os.path.join(ROOT, "tests", "golden", "hse_texts.json"), encoding="utf-8") as f:
        texts = json.load(f)
    assert len(texts) == len(golden["hse"]["docs"]) == 30
    for d in golden["hse"]["docs"]:
        assert utils.text_to_strings_collection(texts[d["name"]]) == d["strings"], d["name"]


def test_narrow_packing_and_batch_planning():
    from east import relevance
    from east.asts import utils as au
    col = ["AB", "C D", "XYZ"]
    p8, p32 = au.pack_strings_collection_u8(col), au.pack_strings_collection(col)
    assert p8.dtype == np.uint8 and p8.size == p32.size
    assert p8.tolist() == [65, 66, 255, 67, 32, 68, 255, 88, 89, 90, 255]
    assert [int(x) for x in p32[p32 >= 0x0A00]] == [0x0A00, 0x0A01, 0x0A02]
    assert np.array_equal(np.where(p8 == 255, 0, p8), np.where(p32 >= 0x0A00, 0, p32))
    assert au.pack_strings_collection_u8(["ÿ"]) is None and au.pack_strings_collection_u8(["Ж"]) is None
    assert au.pack_strings_collection_u8(["été"]) is not None      # Latin-1 fits one byte per code point
    # small and large documents go to separate device batches; no batch exceeds the limit
    assert relevance.plan_batches([10, 70000, 20, 30]) == [[0, 2, 3], [1]]
    assert relevance.plan_batches([5, 5, 5], small_limit=10, max_batch=10) == [[0, 1], [2]]
    assert relevance.plan_batches([]) == []
    # what the device preprocessing accepts (mirror of csrc/tokenize.cu)
    ok = relevance._DEVICE_TEXT_RE.match
    assert ok("plain ASCII, it's 100% fine_") and ok("«Привет» – №5…") and ok("﻿BOM first")
    assert not ok("café") and not ok("x²") and not ok("中文") and not ok("Ѡ")


def test_bench_dump_outputs_writes_the_table_or_a_fixed_sample(tmp_path, monkeypatch):
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_for_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    table = np.random.default_rng(3).random((50, 7))
    bench.dump_table(str(tmp_path / "full"), "scores", table)
    assert os.listdir(str(tmp_path / "full")) == ["scores.npy"]
    got = np.load(str(tmp_path / "full" / "scores.npy"))
    assert got.dtype == np.float64 and np.array_equal(got, table)
    monkeypatch.setattr(bench, "DUMP_BYTES", 20 * (7 * 8 + 8))   # room for 20 rows and their row numbers
    samples = []
    for run in ("a", "b"):
        bench.dump_table(str(tmp_path / run), "scores", table)
        rows = np.load(str(tmp_path / run / "scores_rows.npy"))
        got = np.load(str(tmp_path / run / "scores.npy"))
        assert rows.dtype == got.dtype == np.float64 and got.shape == (20, 7)
        assert np.all(np.diff(rows) > 0) and np.array_equal(got, table[rows.astype(np.int64)])
        samples.append(rows)
    assert np.array_equal(samples[0], samples[1])


def test_graph_from_cooccurrence_matches_the_reference_graphs(golden):
    # the graph assembly (applications.py:115-149) from exact co-occurrence counts computed on the host from the golden table
    from east import applications
    hse = golden["hse"]
    kps = hse["keyphrases"]
    names = [d["name"] for d in hse["docs"]]
    table = np.array([[float.fromhex(hse["table_norm"][kp][n]) for kp in kps] for n in names])
    for g in hse["graphs"]:
        B = (table >= g["r"]).astype(np.int64)
        graph = applications.graph_from_cooccurrence(kps, kps, (B.T @ B).astype(np.int32), g["c"], g["r"], g["p"])
        assert graph["nodes"] == g["nodes"]
        assert [(e["source"], e["target"], float(e["confidence"]).hex()) for e in graph["edges"]] == \
               [(e["source"], e["target"], e["confidence"]) for e in g["edges"]]
    with pytest.raises(KeyError):
        applications.graph_from_cooccurrence(["a", ""], ["a"], np.zeros((1, 1), dtype=np.int32), 0.5, 0.5, 1)
