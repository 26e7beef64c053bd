"""Synthetic Zipf word text of SURVEY.md section 8(d): the workload of bench.py and of the
size-independent parity tests.

  vocabulary : V = 50 000 words, word i = lowercase a-z string, length uniform in [3, 10],
               numpy.random.default_rng(0)
  documents  : words drawn with p(rank) ~ 1/rank, default_rng(doc seed), joined by single
               spaces, truncated at the target byte size; doc j of a collection has seed j + 1
  keyphrases : 1-3 words (uniform) from the same Zipf, default_rng(7), joined by spaces
"""
import numpy as np

V = 50000
_vocab_cache = {}


def vocabulary(v=V):
    if v not in _vocab_cache:
        rng = np.random.default_rng(0)
        lengths = rng.integers(3, 11, size=v)
        letters = rng.integers(0, 26, size=int(lengths.sum()))
        chars = (letters + ord("a")).astype(np.uint8).tobytes().decode("ascii")
        offs = np.concatenate([[0], np.cumsum(lengths)])
        words = [chars[offs[i]:offs[i + 1]] for i in range(v)]
        ranks = np.arange(1, v + 1, dtype=np.float64)
        cdf = np.cumsum(1.0 / ranks)
        cdf /= cdf[-1]
        _vocab_cache[v] = (words, cdf, lengths)
    return _vocab_cache[v]


def document(n_bytes, seed, v=V):
    """One synthetic .txt document of exactly n_bytes ASCII bytes (last word may be cut)."""
    words, cdf, lengths = vocabulary(v)
    rng = np.random.default_rng(seed)
    # mean word length 6.5 + 1 space; oversample, then truncate
    count = int(n_bytes / 5.0) + 16
    ids = np.searchsorted(cdf, rng.random(count), side="right")
    text = " ".join(words[i] for i in ids)
    while len(text) < n_bytes:
        ids = np.searchsorted(cdf, rng.random(count), side="right")
        text += " " + " ".join(words[i] for i in ids)
    return text[:n_bytes]


def documents(n_docs, n_bytes, first_seed=1, v=V):
    return [document(n_bytes, first_seed + j, v) for j in range(n_docs)]


def keyphrases(k, seed=7, v=V):
    words, cdf, _ = vocabulary(v)
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(k):
        nw = int(rng.integers(1, 4))
        ids = np.searchsorted(cdf, rng.random(nw), side="right")
        out.append(" ".join(words[i] for i in ids))
    return out


def synonyms(prepared_keyphrases, seed=11, v=V):
    """Seeded synonym dictionary of profiles/bench_synonyms.py: every distinct word of the (upper-cased) keyphrases,
    in sorted order, gets rng.integers(0, 4) synonyms drawn from the same Zipf, upper-cased.  For keyphrases(1000):
    9 277 variants, at most 64 per keyphrase."""
    from east import utils
    words, cdf, _ = vocabulary(v)
    rng = np.random.default_rng(seed)
    out = {}
    for w in sorted({t for kp in prepared_keyphrases for t in utils.tokenize(kp)}):
        ids = np.searchsorted(cdf, rng.random(int(rng.integers(0, 4))), side="right")
        out[w] = [words[i].upper() for i in ids]
    return out


def packed_collection(n_docs, n_bytes, first_seed=1):
    """Documents run through the host preprocessing of the product package and packed:
    returns (list of uint32 arrays, list of m, list of strings collections)."""
    from east import utils
    from east.asts import utils as asts_utils
    cols = [utils.text_to_strings_collection(d) for d in documents(n_docs, n_bytes, first_seed)]
    packed = [asts_utils.pack_strings_collection(c) for c in cols]
    return packed, [len(c) for c in cols], cols


def packed_big_document(n_bytes, seed=1, v=V):
    """Packed form (uint32 code points + terminators, string count m) of a synthetic document of
    ~n_bytes, built with numpy only -- the same result as
    pack_strings_collection(text_to_strings_collection(text)) for a text made of whole vocabulary
    words (every word has 3..10 letters, so the token filter of utils.py:63 drops nothing), but
    without materialising tens of millions of Python strings.  Returns (packed, m, text_bytes)."""
    words, cdf, lengths = vocabulary(v)
    rng = np.random.default_rng(seed)
    mean_len = float((lengths * np.diff(np.concatenate([[0.0], cdf]))).sum()) + 1.0
    count = max(1, int(n_bytes / mean_len))
    ids = np.searchsorted(cdf, rng.random(count), side="right")
    wl = lengths[ids].astype(np.int64)
    # flat upper-case code points of the chosen words
    vocab_codes = np.frombuffer("".join(words).upper().encode("ascii"), dtype=np.uint8)
    vocab_off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    total_chars = int(wl.sum())
    word_start_out = np.concatenate([[0], np.cumsum(wl)[:-1]])
    idx = np.arange(total_chars, dtype=np.int64)
    word_of = np.repeat(np.arange(count, dtype=np.int64), wl)
    src = vocab_off[ids][word_of] + (idx - word_start_out[word_of])
    chars = vocab_codes[src].astype(np.uint32)
    # strings = groups of 3 consecutive words (utils.py:66-73)
    m = (count + 2) // 3
    str_len = np.add.reduceat(wl, np.arange(0, count, 3))
    n = total_chars + m
    term_pos = np.cumsum(str_len + 1) - 1
    out = np.empty(n, dtype=np.uint32)
    is_char = np.ones(n, dtype=bool)
    is_char[term_pos] = False
    out[is_char] = chars
    out[term_pos] = 0x0A00 + np.arange(m, dtype=np.uint32)
    text_bytes = total_chars + count - 1  # words joined by single spaces
    return out, int(m), int(text_bytes), ids


def packed_collection_fast(n_docs, n_bytes, first_seed=1, v=V, chunk_docs=4096):
    """n_docs synthetic documents of ~n_bytes each, already packed (uint32 code points + terminators), built with numpy
    only: the same result as pack_strings_collection(text_to_strings_collection(" ".join(words))) for documents made
    of whole vocabulary words (3..10 letters each: the token filter of utils.py:63 drops nothing).  Every document has
    the same number of words (n_bytes / mean word length), drawn from the Zipf distribution with default_rng(first_seed
    + chunk number).  Returns (text uint32 [N], doc_off int64 [n_docs + 1], doc_m int32 [n_docs])."""
    words, cdf, lengths = vocabulary(v)
    mean_len = float((lengths * np.diff(np.concatenate([[0.0], cdf]))).sum()) + 1.0
    wpd = max(1, int(n_bytes / mean_len))
    m_doc = (wpd + 2) // 3
    vocab_codes = np.frombuffer("".join(words).upper().encode("ascii"), dtype=np.uint8)
    vocab_off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    texts, sizes = [], []
    for c0 in range(0, n_docs, chunk_docs):
        nd = min(chunk_docs, n_docs - c0)
        rng = np.random.default_rng(first_seed + c0 // chunk_docs)
        count = nd * wpd
        ids = np.searchsorted(cdf, rng.random(count), side="right")
        wl = lengths[ids].astype(np.int64)
        j = np.arange(count, dtype=np.int64) % wpd
        ends_string = (j % 3 == 2) | (j == wpd - 1)
        out_len = wl + ends_string
        start = np.concatenate([[0], np.cumsum(out_len)[:-1]])
        n = int(out_len.sum())
        out = np.empty(n, dtype=np.uint32)
        term_pos = (start + wl)[ends_string]
        is_char = np.ones(n, dtype=bool)
        is_char[term_pos] = False
        total_chars = int(wl.sum())
        word_of = np.repeat(np.arange(count, dtype=np.int64), wl)
        char_start = np.concatenate([[0], np.cumsum(wl)[:-1]])
        src = vocab_off[ids][word_of] + (np.arange(total_chars, dtype=np.int64) - char_start[word_of])
        out[is_char] = vocab_codes[src]
        out[term_pos] = 0x0A00 + (j[ends_string] // 3).astype(np.uint32)
        texts.append(out)
        sizes.append(np.add.reduceat(out_len, np.arange(0, count, wpd)))
    sizes = np.concatenate(sizes)
    doc_off = np.zeros(n_docs + 1, dtype=np.int64)
    np.cumsum(sizes, out=doc_off[1:])
    return np.concatenate(texts), doc_off, np.full(n_docs, m_doc, dtype=np.int32)
