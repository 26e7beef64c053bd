"""GPU: the child table and annotation of the per-document kernel (phase 8 of doc_sort.cu) on inputs built to hit the
edges of its tiles of 32 ranks and of its pyramid searches, by both implementations: tiles of 32 ranks, one lane per
rank (the default), and the per-thread stack walk (EAST_DOC_SORT_STACK_WALK=1).  The switch is read once per process,
so each implementation runs in a child process of its own that writes its arrays to a file; both are compared with each other and with the
CPU oracle, array for array."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "ast-text-analysis_b200")
NAMES = ["suftab", "lcptab", "childtab_up", "childtab_down", "childtab_next_l_index", "anntab"]


def _document_of(rng, target):
    """Zipf-distributed words in strings of three; the packed document has exactly `target` code points."""
    words = ["".join(rng.choice(list("ABCDEFGHIJKLMNOPQRSTUVWXYZ"), size=int(rng.integers(3, 9)))) for _ in range(2000)]
    p = 1.0 / np.arange(1, len(words) + 1)
    p /= p.sum()
    strings, total = [], 0
    while total < target:
        s_ = "".join(rng.choice(words, size=3, p=p))
        if total + len(s_) + 1 > target:
            s_ = s_[: max(1, target - total - 1)]
        strings.append(s_)
        total += len(s_) + 1
    if total != target:
        strings[0] = strings[0][: len(strings[0]) - (total - target)] or "A"
    return strings


def _batches():
    """Batches of documents (lists of strings); every document stays below the kernel's bucket limit."""
    rng = np.random.default_rng(11)
    twice = "".join(rng.choice(list("ABCD"), size=2000))
    return [
        # n not a multiple of 32, and n = 65 535 (2 048 tiles, four pyramid levels)
        [_document_of(rng, 1001), _document_of(rng, 4133), _document_of(rng, 65535)],
        # one symbol: LCP falls from 2 999 to 1 across tiles and 1 024-rank blocks (16 bit planes)
        [["A" * 3000]],
        # runs of A of every length 1..79: LCP rises and falls across tile boundaries
        [["A" * i for i in range(1, 80)]],
        # all-equal LCP (next chains thousands of ranks long), a string twice (LCP ~2 000), single strings
        [["XY"] * 2000, [twice, twice], ["AB" * 1500], ["".join(_document_of(rng, 8000))], ["A"]],
    ]


def _dump(out):
    """Child process: index every batch, write its arrays to `out` (.npz)."""
    for p in (PKG, ROOT):
        sys.path.insert(0, p)
    from east import _capi
    from east.asts import utils as au
    arrays = {}
    for b, batch in enumerate(_batches()):
        idx = _capi.DeviceIndex([au.pack_strings_collection(c) for c in batch], [len(c) for c in batch])
        assert idx.info()["doc_sorted"] and idx.stat("tables_fused") == 1, b
        for d in range(len(batch)):
            for which, name in enumerate(NAMES):
                arrays["%d/%d/%s" % (b, d, name)] = idx.array(d, which)
        idx.close()
    np.savez(out, **arrays)


def _run(tmp_path, stack_walk):
    out = str(tmp_path / ("stack_walk.npz" if stack_walk else "tiles.npz"))
    env = dict(os.environ)
    env.pop("EAST_DOC_SORT_STACK_WALK", None)
    if stack_walk:
        env["EAST_DOC_SORT_STACK_WALK"] = "1"
    flags = ["-s"] if sys.flags.no_user_site else []
    subprocess.run([sys.executable] + flags + [os.path.abspath(__file__), out], env=env, cwd=ROOT, check=True)
    return dict(np.load(out))


@pytest.fixture(scope="module")
def both(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("child_table")
    return {"tiles": _run(tmp, False), "stack_walk": _run(tmp, True)}


@pytest.fixture(scope="module")
def expected(oracle_mod):
    from east.asts import utils as au
    exp = {}
    for b, batch in enumerate(_batches()):
        for d, c in enumerate(batch):
            o = oracle_mod.OracleEASA(text=au.pack_strings_collection(c), m=len(c))
            for name in NAMES:
                exp["%d/%d/%s" % (b, d, name)] = getattr(o, name)
    return exp


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["tiles", "stack_walk"])
def test_child_table_and_annotation_match_the_oracle(both, expected, path):
    got = both[path]
    assert sorted(got) == sorted(expected)
    for key, exp in expected.items():
        assert np.array_equal(got[key], exp), (path, key, np.nonzero(got[key] != exp)[0][:5])


@pytest.mark.gpu
def test_tiles_and_stack_walk_agree(both):
    assert sorted(both["tiles"]) == sorted(both["stack_walk"])
    for key, a in both["tiles"].items():
        assert np.array_equal(a, both["stack_walk"][key]), key


if __name__ == "__main__":
    _dump(sys.argv[1])
