# -*- coding: utf-8 -*-
"""ctypes binding of libeast_b200.so (C ABI in include/east_b200.h).

There is no CPU fallback: if the shared library is missing, or no CUDA device is visible,
every entry point raises east.exceptions.DeviceError.
"""
import ctypes
import os

import numpy as np

from east import exceptions

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("EAST_B200_LIB",
                          os.path.join(os.path.dirname(_HERE), "lib", "libeast_b200.so"))

# east_array ids (include/east_b200.h)
SUFTAB, LCPTAB, CHILDTAB_UP, CHILDTAB_DOWN, CHILDTAB_NEXT_L_INDEX, ANNTAB, PACKED_TEXT = range(7)
TEXT_DEVPTR = 100

EAST_ERR_ZERODIV = -4
EAST_ERR_UNSUPPORTED = -6


class UnsupportedText(ValueError):
    """The device preprocessing met a character outside ASCII / U+0400-045F: use the host preprocessing."""


EXPORTED_SYMBOLS = [
    "east_last_error", "east_device_count", "east_version", "east_build_host", "east_build_dev",
    "east_free", "east_index_info", "east_index_doc", "east_index_copy", "east_index_devptr",
    "east_score_table_host", "east_score_table_dev", "east_score_one", "east_cooc_dev",
    "east_cooc_host", "east_last_timings", "east_launch_count", "east_set_option", "east_kernel_stats",
    "east_score_probes_dev", "east_index_stat", "east_score_range_dev", "east_table_host", "east_table_dev",
    "east_build_host_u8", "east_table_host_u8", "east_table_dev_gather", "east_trim", "east_table_host_gather", "east_index_save", "east_index_load", "east_texts_to_packed_host", "east_table_texts_host",
    "east_score_groups_host", "east_score_groups_dev",
    "east_table_groups_host", "east_table_groups_dev", "east_table_texts_groups_host",
    "east_graph_host", "east_graph_dev", "east_graph_texts_host",
]

_lib = None

_u32p = ctypes.POINTER(ctypes.c_uint32)
_u8p = ctypes.POINTER(ctypes.c_uint8)
_i32p = ctypes.POINTER(ctypes.c_int32)
_i64p = ctypes.POINTER(ctypes.c_int64)
_f64p = ctypes.POINTER(ctypes.c_double)
_f32p = ctypes.POINTER(ctypes.c_float)
_vp = ctypes.c_void_p


def load():
    """dlopen the engine and declare prototypes; raises DeviceError if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise exceptions.DeviceError(
            reason="%s not found -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                   "or `make -C ast-text-analysis_b200`" % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    L.east_last_error.restype = ctypes.c_char_p
    L.east_version.restype = ctypes.c_char_p
    L.east_device_count.restype = ctypes.c_int
    L.east_build_host.argtypes = [_u32p, _i64p, _i32p, ctypes.c_int32, ctypes.c_int, ctypes.POINTER(_vp)]
    L.east_build_dev.argtypes = [_vp, _i64p, _i32p, ctypes.c_int32, ctypes.c_int, _vp, ctypes.POINTER(_vp)]
    L.east_free.argtypes = [_vp]
    L.east_free.restype = None
    L.east_index_info.argtypes = [_vp, _i32p, _i64p, _i32p, _i32p, _i32p]
    L.east_index_doc.argtypes = [_vp, ctypes.c_int32, _i64p, _i64p, _i32p]
    L.east_index_stat.argtypes = [_vp, ctypes.c_char_p, _i64p]
    L.east_index_copy.argtypes = [_vp, ctypes.c_int32, ctypes.c_int, _i32p]
    L.east_index_devptr.argtypes = [_vp, ctypes.c_int, ctypes.POINTER(_vp)]
    L.east_score_table_host.argtypes = [_vp, _u32p, _i64p, ctypes.c_int32, ctypes.c_int, _f64p]
    L.east_score_table_dev.argtypes = [_vp, _vp, _i64p, ctypes.c_int32, ctypes.c_int, _vp, _vp]
    L.east_table_host.argtypes = [_u32p, _i64p, _i32p, ctypes.c_int32, ctypes.c_int, _u32p, _i64p, ctypes.c_int32,
                                  ctypes.c_int, _f64p, ctypes.POINTER(_vp)]
    L.east_build_host_u8.argtypes = [_u8p, _i64p, _i32p, ctypes.c_int32, ctypes.c_int, ctypes.POINTER(_vp)]
    L.east_table_host_u8.argtypes = [_u8p, _i64p, _i32p, ctypes.c_int32, ctypes.c_int, _u32p, _i64p, ctypes.c_int32,
                                     ctypes.c_int, _f64p, ctypes.POINTER(_vp)]
    L.east_table_dev.argtypes = [_vp, _i64p, _i32p, ctypes.c_int32, ctypes.c_int, _vp, _u32p, _i64p, ctypes.c_int32,
                                 ctypes.c_int, _vp, _vp, ctypes.POINTER(_vp)]
    L.east_table_dev_gather.argtypes = [_vp, _i64p, _i32p, ctypes.c_int32, ctypes.c_int, _vp, _u32p, _i64p, ctypes.c_int32,
                                        ctypes.c_int, _vp, ctypes.POINTER(_vp), ctypes.c_int32, _vp, ctypes.POINTER(_vp)]
    L.east_table_host_gather.argtypes = [_vp, ctypes.c_int32, _i64p, _i32p, ctypes.c_int32, ctypes.c_int, _u32p, _i64p, ctypes.c_int32,
                                         ctypes.c_int, _f64p, _vp, ctypes.POINTER(_vp), ctypes.c_int32, ctypes.POINTER(_vp)]
    L.east_index_save.argtypes = [_vp, ctypes.c_char_p]
    L.east_index_load.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.POINTER(_vp)]
    L.east_texts_to_packed_host.argtypes = [_u8p, _i64p, ctypes.c_int32, ctypes.c_int, _u32p, ctypes.c_int64, _i64p, _i32p]
    L.east_table_texts_host.argtypes = [_u8p, _i64p, ctypes.c_int32, ctypes.c_int, _u32p, _i64p, ctypes.c_int32, ctypes.c_int, _f64p,
                                        _i64p, _i32p, ctypes.POINTER(_vp)]
    L.east_score_range_dev.argtypes = [_vp, _vp, _i64p, ctypes.c_int32, ctypes.c_int, ctypes.c_int32, ctypes.c_int32, _vp, _vp]
    L.east_score_groups_host.argtypes = [_vp, _u32p, _i64p, ctypes.c_int32, _i64p, ctypes.c_int32, ctypes.c_int32,
                                         ctypes.c_int32, _f64p]
    L.east_score_groups_dev.argtypes = [_vp, _vp, _i64p, ctypes.c_int32, _i64p, ctypes.c_int32, ctypes.c_int32,
                                        ctypes.c_int32, _vp, _vp]
    L.east_table_groups_host.argtypes = [_vp, ctypes.c_int32, _i64p, _i32p, ctypes.c_int32, ctypes.c_int, _u32p, _i64p,
                                         ctypes.c_int32, _i64p, ctypes.c_int32, _f64p, ctypes.POINTER(_vp)]
    L.east_table_groups_dev.argtypes = [_vp, _i64p, _i32p, ctypes.c_int32, ctypes.c_int, _vp, _u32p, _i64p, ctypes.c_int32,
                                        _i64p, ctypes.c_int32, _vp, ctypes.POINTER(_vp), ctypes.c_int32, _vp, ctypes.POINTER(_vp)]
    L.east_table_texts_groups_host.argtypes = [_u8p, _i64p, ctypes.c_int32, ctypes.c_int, _u32p, _i64p, ctypes.c_int32, _i64p,
                                               ctypes.c_int32, _f64p, _i64p, _i32p, ctypes.POINTER(_vp)]
    L.east_graph_host.argtypes = [_vp, ctypes.c_int32, _i64p, _i32p, ctypes.c_int32, ctypes.c_int, _u32p, _i64p, ctypes.c_int32,
                                  _i64p, ctypes.c_int32, ctypes.c_int, ctypes.c_double, _i32p, ctypes.POINTER(_vp)]
    L.east_graph_dev.argtypes = [_vp, _i64p, _i32p, ctypes.c_int32, ctypes.c_int, _vp, _u32p, _i64p, ctypes.c_int32, _i64p,
                                 ctypes.c_int32, ctypes.c_int, ctypes.c_double, _vp, _vp, ctypes.POINTER(_vp)]
    L.east_graph_texts_host.argtypes = [_u8p, _i64p, ctypes.c_int32, ctypes.c_int, _u32p, _i64p, ctypes.c_int32, _i64p,
                                        ctypes.c_int32, ctypes.c_int, ctypes.c_double, _i32p, _i64p, _i32p, ctypes.POINTER(_vp)]
    L.east_score_probes_dev.argtypes = [_vp, _vp, _i64p, ctypes.c_int32, _vp, _vp, _i64p]
    L.east_score_one.argtypes = [_vp, ctypes.c_int32, _u32p, ctypes.c_int32, ctypes.c_int, _f64p, _f64p]
    L.east_cooc_dev.argtypes = [_vp, ctypes.c_int64, ctypes.c_int32, ctypes.c_double, _vp, ctypes.c_int, _vp]
    L.east_cooc_host.argtypes = [_f64p, ctypes.c_int64, ctypes.c_int32, ctypes.c_double, _i32p, ctypes.c_int]
    L.east_last_timings.argtypes = [_f32p, ctypes.c_char_p, ctypes.c_int32, ctypes.c_int32]
    L.east_launch_count.argtypes = [ctypes.c_int]
    L.east_launch_count.restype = ctypes.c_int64
    L.east_set_option.argtypes = [ctypes.c_char_p, ctypes.c_int64]
    L.east_kernel_stats.argtypes = [ctypes.c_char_p, ctypes.c_int32, _f64p, _i64p, _f64p, ctypes.c_int32]
    _lib = L
    return L


def _check(rc):
    if rc == 0:
        return
    msg = load().east_last_error().decode("utf-8", "replace")
    if rc == EAST_ERR_ZERODIV:
        raise ZeroDivisionError(msg or "float division by zero")  # easa.py:134 on an empty query
    if rc == -3:
        raise MemoryError(msg)
    if rc == EAST_ERR_UNSUPPORTED:
        raise UnsupportedText(msg)
    if rc == -1 or rc == -5:
        raise ValueError(msg)
    raise exceptions.DeviceError(reason=msg)


def _ptr(a, t):
    return a.ctypes.data_as(t)


def device_count():
    return load().east_device_count()


def trim(device=0):
    """Return the memory the library keeps for reuse (its private pools) to the driver."""
    _check(load().east_trim(int(device)))


def set_option(name, value):
    _check(load().east_set_option(name.encode(), int(value)))


def launch_count(reset=False):
    return int(load().east_launch_count(1 if reset else 0))


def last_timings():
    """[(stage name, device ms)] of the last build/score/cooc call of this thread."""
    L = load()
    ms = (ctypes.c_float * 64)()
    names = ctypes.create_string_buffer(4096)
    n = L.east_last_timings(ms, names, 64, 4096)
    parts = names.raw.split(b"\0")
    return [(parts[i].decode(), float(ms[i])) for i in range(min(n, 64))]


def kernel_stats():
    """{kernel name: {"launches", "ms", "bytes"}} accumulated while option time_kernels == 1."""
    L = load()
    cap = 64
    names = ctypes.create_string_buffer(8192)
    ms = (ctypes.c_double * cap)()
    launches = (ctypes.c_int64 * cap)()
    nbytes = (ctypes.c_double * cap)()
    n = L.east_kernel_stats(names, 8192, ms, launches, nbytes, cap)
    parts = names.raw.split(b"\0")
    return {parts[i].decode(): {"launches": int(launches[i]), "ms": float(ms[i]), "bytes": float(nbytes[i])}
            for i in range(min(n, cap))}


def pack_keyphrases(queries):
    """Space-stripped queries (easa.py:36 query.replace(" ", "")) -> (uint32 codes, int64 offsets)."""
    from east.asts.utils import codepoints
    stripped = [q.replace(" ", "") for q in queries]
    off = np.zeros(len(stripped) + 1, dtype=np.int64)
    np.cumsum([len(q) for q in stripped], out=off[1:])
    codes = np.ascontiguousarray(codepoints("".join(stripped)), dtype=np.uint32)
    if codes.size != off[-1]:
        raise ValueError("keyphrases contain lone surrogates")
    return codes, off


def pack_variant_groups(queries, synonyms):
    """Synonym-expanded queries -> (uint32 codes, int64 variant offsets [V + 1], int64 group offsets [len(queries) + 1]):
    the variants of query k (utils.synonym_variants) are variants group_off[k] .. group_off[k + 1] - 1, packed as they
    are -- the reference scores them with _score, which does not strip spaces (easa.py:34)."""
    from east import utils
    from east.asts.utils import codepoints
    variants = []
    group_off = np.zeros(len(queries) + 1, dtype=np.int64)
    for k, q in enumerate(queries):
        variants.extend(utils.synonym_variants(q, synonyms))
        group_off[k + 1] = len(variants)
    off = np.zeros(len(variants) + 1, dtype=np.int64)
    np.cumsum([len(v) for v in variants], out=off[1:])
    codes = np.ascontiguousarray(codepoints("".join(variants)), dtype=np.uint32)
    if codes.size != off[-1]:
        raise ValueError("synonym variants contain lone surrogates")
    return codes, off, group_off


def _columns(K, group_off):
    """Columns of a table: one per keyphrase, or one per group of synonym variants."""
    return K if group_off is None else len(group_off) - 1


def _keyphrases_args(kp_codes, kp_off):
    """(uint32 code points, int64 offsets, K) of packed keyphrases or variants; kp_codes may be None (the optional host
    copy of device-resident code points)"""
    kp_off = np.ascontiguousarray(kp_off, dtype=np.int64)
    codes = None if kp_codes is None else np.ascontiguousarray(kp_codes, dtype=np.uint32)
    return codes, kp_off, len(kp_off) - 1


def _kp_host_arg(kp_codes):
    """pointer to the optional host copy of device-resident code points (None: no copy)"""
    return None if kp_codes is None else _ptr(kp_codes, _u32p)


def _documents_args(doc_off, doc_m):
    """(int64 offsets [n + 1], int32 string counts [n]) of packed documents"""
    return np.ascontiguousarray(doc_off, dtype=np.int64), np.ascontiguousarray(doc_m, dtype=np.int32)


def _texts_args(texts):
    """raw texts (list of str / UTF-8 bytes, or (uint8 buffer, int64 offsets) already laid out back to back, e.g. in
    pinned memory) -> (buffer, offsets, n, doc_off and doc_m for the packed documents the call returns)"""
    buf, off = texts if isinstance(texts, tuple) else concat_utf8(texts)
    n = len(off) - 1
    return buf, off, n, np.zeros(n + 1, dtype=np.int64), np.zeros(n, dtype=np.int32)


def _peers_arg(peer_rows):
    """(ctypes array of the peer row addresses, their number)"""
    peer_rows = list(peer_rows or [])
    return (_vp * max(len(peer_rows), 1))(*[int(a) for a in peer_rows]), len(peer_rows)


def _groups_arg(group_off):
    """(int64 array or None, pointer or None, G) of optional group offsets"""
    if group_off is None:
        return None, None, 0
    group_off = np.ascontiguousarray(group_off, dtype=np.int64)
    return group_off, _ptr(group_off, _i64p), len(group_off) - 1


def _counts_out(C, K, group_off):
    cols = _columns(K, group_off)
    if C is None:
        return np.empty((cols, cols), dtype=np.int32)
    assert C.dtype == np.int32 and C.flags["C_CONTIGUOUS"] and C.size == cols * cols
    return C


def concat_utf8(texts):
    """list of str / bytes -> (uint8 buffer of the UTF-8 texts back to back, int64 offsets [n + 1])"""
    raws = [t if isinstance(t, (bytes, bytearray)) else t.encode("utf-8", errors="surrogatepass") for t in texts]
    off = np.zeros(len(raws) + 1, dtype=np.int64)
    np.cumsum([len(r) for r in raws], out=off[1:])
    buf = np.frombuffer(b"".join(raws), dtype=np.uint8) if off[-1] else np.zeros(1, dtype=np.uint8)
    return buf, off


def texts_to_packed(texts, device=0):
    """utils.text_to_strings_collection + pack_strings_collection of every text ON THE DEVICE (east_texts_to_packed_host).
    texts: list of str or UTF-8 bytes.  Returns (uint32 packed text, int64 doc_off [n + 1], int32 doc_m [n]); raises
    UnsupportedText when a text has characters outside ASCII / U+0400-045F."""
    L = load()
    buf, off = concat_utf8(texts)
    n = len(texts)
    doc_off = np.zeros(n + 1, dtype=np.int64)
    doc_m = np.zeros(n, dtype=np.int32)
    cap = int(off[-1]) + 2 * n + 2     # a packed document never has more entries than its text has bytes, + 2
    packed = np.empty(cap, dtype=np.uint32)
    _check(L.east_texts_to_packed_host(_ptr(buf, _u8p), _ptr(off, _i64p), n, int(device), _ptr(packed, _u32p), cap,
                                       _ptr(doc_off, _i64p), _ptr(doc_m, _i32p)))
    return packed[: int(doc_off[-1])], doc_off, doc_m


class DeviceIndex(object):
    """A batch of documents indexed on one GPU (opaque east_index handle)."""

    def __init__(self, packed_docs, doc_m, device=0):
        """packed_docs: list of uint32 arrays (east.asts.utils.pack_strings_collection),
        doc_m: number of strings of each document."""
        L = load()
        if len(packed_docs) == 0:
            raise exceptions.EmptyStringsCollectionException()
        self.n_docs = len(packed_docs)
        self.doc_off = np.zeros(self.n_docs + 1, dtype=np.int64)
        np.cumsum([len(p) for p in packed_docs], out=self.doc_off[1:])
        self.doc_m = np.ascontiguousarray(doc_m, dtype=np.int32)
        text = np.ascontiguousarray(np.concatenate(packed_docs) if self.n_docs > 1 else packed_docs[0],
                                    dtype=np.uint32)
        self.device = int(device)
        self._h = _vp()
        _check(L.east_build_host(_ptr(text, _u32p), _ptr(self.doc_off, _i64p), _ptr(self.doc_m, _i32p),
                                 self.n_docs, self.device, ctypes.byref(self._h)))
        self.build_timings = []  # filled by close(): the table kernels may still be running

    @classmethod
    def from_handle(cls, handle, doc_off, doc_m, device):
        self = cls.__new__(cls)
        self._h = handle
        self.doc_off = np.ascontiguousarray(doc_off, dtype=np.int64)
        self.doc_m = np.ascontiguousarray(doc_m, dtype=np.int32)
        self.n_docs = len(self.doc_m)
        self.device = device
        self.build_timings = []
        return self

    @classmethod
    def build_host(cls, text, doc_off, doc_m, device=0):
        """Build from an already concatenated host buffer (uint32, may be pinned)."""
        L = load()
        doc_off = np.ascontiguousarray(doc_off, dtype=np.int64)
        doc_m = np.ascontiguousarray(doc_m, dtype=np.int32)
        assert text.dtype == np.uint32 and text.flags["C_CONTIGUOUS"]
        h = _vp()
        _check(L.east_build_host(_ptr(text, _u32p), _ptr(doc_off, _i64p), _ptr(doc_m, _i32p), len(doc_m),
                                 int(device), ctypes.byref(h)))
        return cls.from_handle(h, doc_off, doc_m, int(device))

    @classmethod
    def _adopt(cls, entry, doc_off, doc_m, device, *args):
        """Call a build entry with its arguments and the out_idx pointer; the index it returns (doc_off / doc_m may be
        filled by the call)."""
        h = _vp()
        _check(entry(*args, ctypes.byref(h)))
        return cls.from_handle(h, doc_off, doc_m, int(device))

    @classmethod
    def table_from_texts(cls, texts, kp_codes, kp_off, out, normalized=True, device=0, group_off=None):
        """Raw texts in, score table out, in ONE engine call (east_table_texts_host): the texts are upper-cased,
        tokenised, grouped and packed on the device (tokenize.cu), indexed and scored.  texts: list of str / UTF-8
        bytes (ASCII and Cyrillic; anything else raises UnsupportedText).  Returns the index.
        group_off (pack_variant_groups): the keyphrases are synonym variants in G groups and `out` has G columns, the
        best normalized variant of each group (east_table_texts_groups_host)."""
        L = load()
        buf, off, n, doc_off, doc_m = _texts_args(texts)
        kp_codes, kp_off, K = _keyphrases_args(kp_codes, kp_off)
        group_off, gp, G = _groups_arg(group_off)
        assert out.dtype == np.float64 and out.flags["C_CONTIGUOUS"] and out.size == n * _columns(K, group_off)
        texts_args = (_ptr(buf, _u8p), _ptr(off, _i64p), n, int(device), _ptr(kp_codes, _u32p), _ptr(kp_off, _i64p), K)
        outs = (_ptr(out, _f64p), _ptr(doc_off, _i64p), _ptr(doc_m, _i32p))
        if group_off is not None:
            return cls._adopt(L.east_table_texts_groups_host, doc_off, doc_m, device, *texts_args, gp, G, *outs)
        return cls._adopt(L.east_table_texts_host, doc_off, doc_m, device, *texts_args, 1 if normalized else 0, *outs)

    @classmethod
    def graph_from_texts(cls, texts, kp_codes, kp_off, threshold, C=None, normalized=True, device=0, group_off=None):
        """table_from_texts() for a keyphrase graph (east_graph_texts_host): raw texts in, the int32 co-occurrence counts
        C[i][j] = number of texts in which columns i and j both score >= threshold out, without a score table.
        Returns (C, index); C: [cols, cols], cols = K, or G with group_off (always normalized)."""
        buf, off, n, doc_off, doc_m = _texts_args(texts)
        kp_codes, kp_off, K = _keyphrases_args(kp_codes, kp_off)
        group_off, gp, G = _groups_arg(group_off)
        C = _counts_out(C, K, group_off)
        return C, cls._adopt(load().east_graph_texts_host, doc_off, doc_m, device, _ptr(buf, _u8p), _ptr(off, _i64p), n,
                             int(device), _ptr(kp_codes, _u32p), _ptr(kp_off, _i64p), K, gp, G, 1 if normalized else 0,
                             float(threshold), _ptr(C, _i32p), _ptr(doc_off, _i64p), _ptr(doc_m, _i32p))

    @classmethod
    def build_host_and_graph(cls, text, doc_off, doc_m, kp_codes, kp_off, threshold, C=None, normalized=True, device=0,
                             group_off=None):
        """build_host_and_score() for a keyphrase graph (east_graph_host): text uint32 code points or one byte per code
        point (pack_strings_collection_u8).  Returns (int32 counts [cols, cols], index); no score table is formed."""
        doc_off, doc_m = _documents_args(doc_off, doc_m)
        kp_codes, kp_off, K = _keyphrases_args(kp_codes, kp_off)
        assert text.dtype in (np.uint32, np.uint8) and text.flags["C_CONTIGUOUS"]
        group_off, gp, G = _groups_arg(group_off)
        C = _counts_out(C, K, group_off)
        return C, cls._adopt(load().east_graph_host, doc_off, doc_m, device, _vp(text.ctypes.data), int(text.itemsize),
                             _ptr(doc_off, _i64p), _ptr(doc_m, _i32p), len(doc_m), int(device), _ptr(kp_codes, _u32p),
                             _ptr(kp_off, _i64p), K, gp, G, 1 if normalized else 0, float(threshold), _ptr(C, _i32p))

    @classmethod
    def build_dev_and_graph(cls, text_devptr, doc_off, doc_m, kp_devptr, kp_codes, kp_off, threshold, C_devptr, normalized=True,
                            device=0, stream=0, group_off=None):
        """build_dev_and_score() for a keyphrase graph (east_graph_dev): the int32 [cols, cols] counts go to C_devptr.
        Returns the index."""
        doc_off, doc_m = _documents_args(doc_off, doc_m)
        kp_codes, kp_off, K = _keyphrases_args(kp_codes, kp_off)
        group_off, gp, G = _groups_arg(group_off)
        return cls._adopt(load().east_graph_dev, doc_off, doc_m, device, _vp(text_devptr), _ptr(doc_off, _i64p),
                          _ptr(doc_m, _i32p), len(doc_m), int(device), _vp(kp_devptr), _kp_host_arg(kp_codes),
                          _ptr(kp_off, _i64p), K, gp, G, 1 if normalized else 0, float(threshold), _vp(C_devptr), _vp(stream))

    @classmethod
    def build_host_u8(cls, text8, doc_off, doc_m, device=0):
        """build_host() for a text shipped as one byte per code point (pack_strings_collection_u8)."""
        L = load()
        doc_off = np.ascontiguousarray(doc_off, dtype=np.int64)
        doc_m = np.ascontiguousarray(doc_m, dtype=np.int32)
        assert text8.dtype == np.uint8 and text8.flags["C_CONTIGUOUS"]
        h = _vp()
        _check(L.east_build_host_u8(_ptr(text8, _u8p), _ptr(doc_off, _i64p), _ptr(doc_m, _i32p), len(doc_m),
                                    int(device), ctypes.byref(h)))
        return cls.from_handle(h, doc_off, doc_m, int(device))

    @classmethod
    def build_host_and_score(cls, text, doc_off, doc_m, kp_codes, kp_off, out, normalized=True, device=0, own_rows=None,
                             peer_rows=None, group_off=None):
        """build_host() + score_table_into() as ONE engine call (east_table_host): on a large batch of small
        documents the runs of documents already sorted are scored, and their rows of `out` copied back, while
        the rest of the text is still on its way to the device.  Returns the index; `out` ([n_docs, K] float64,
        may be pinned) holds the table.
        group_off (pack_variant_groups): the keyphrases are synonym variants in G groups and `out` ([n_docs, G]) holds
        the best normalized variant of each group (east_table_groups_host; not with own_rows / peer_rows)."""
        L = load()
        doc_off, doc_m = _documents_args(doc_off, doc_m)
        kp_codes, kp_off, K = _keyphrases_args(kp_codes, kp_off)
        assert text.dtype in (np.uint32, np.uint8) and text.flags["C_CONTIGUOUS"]
        assert out.dtype == np.float64 and out.flags["C_CONTIGUOUS"] and out.size == len(doc_m) * _columns(K, group_off)
        group_off, gp, G = _groups_arg(group_off)
        norm = 1 if normalized else 0
        docs = (_ptr(doc_off, _i64p), _ptr(doc_m, _i32p), len(doc_m), int(device))
        kps = (_ptr(kp_codes, _u32p), _ptr(kp_off, _i64p), K)
        if group_off is not None:
            if own_rows or peer_rows:
                raise ValueError("a sharded synonym table is built from device-resident text (build_dev_and_score)")
            return cls._adopt(L.east_table_groups_host, doc_off, doc_m, device, _vp(text.ctypes.data), int(text.itemsize),
                              *docs, *kps, gp, G, _ptr(out, _f64p))
        if own_rows or peer_rows:   # sharded table: rows also to the gathered tables on the devices (east_table_host_gather)
            peers, n_peers = _peers_arg(peer_rows)
            return cls._adopt(L.east_table_host_gather, doc_off, doc_m, device, _vp(text.ctypes.data), int(text.itemsize),
                              *docs, *kps, norm, _ptr(out, _f64p), _vp(own_rows or 0), peers, n_peers)
        if text.dtype == np.uint8:   # one byte per code point, 0xFF ends a string (pack_strings_collection_u8)
            return cls._adopt(L.east_table_host_u8, doc_off, doc_m, device, _ptr(text, _u8p), *docs, *kps, norm, _ptr(out, _f64p))
        return cls._adopt(L.east_table_host, doc_off, doc_m, device, _ptr(text, _u32p), *docs, *kps, norm, _ptr(out, _f64p))

    @classmethod
    def build_dev_and_score(cls, text_devptr, doc_off, doc_m, kp_devptr, kp_codes, kp_off, out_devptr, normalized=True,
                            device=0, stream=0, peer_rows=None, group_off=None):
        """build_dev() + score_table_dev() as ONE engine call (east_table_dev): the per-document kernel scores every
        document right after indexing it.  kp_codes: host copy of the keyphrase code points (or None).
        peer_rows: device addresses in the OTHER ranks' gathered tables where this rank's rows start (mapped peer
        memory): the kernel stores every row there too (east_table_dev_gather, the fused all-gather).
        group_off (pack_variant_groups): the keyphrases are synonym variants in G groups and the table has G columns,
        the best normalized variant of each group (east_table_groups_dev, with or without peer_rows)."""
        L = load()
        doc_off, doc_m = _documents_args(doc_off, doc_m)
        kp_codes, kp_off, K = _keyphrases_args(kp_codes, kp_off)
        group_off, gp, G = _groups_arg(group_off)
        args = (_vp(text_devptr), _ptr(doc_off, _i64p), _ptr(doc_m, _i32p), len(doc_m), int(device), _vp(kp_devptr),
                _kp_host_arg(kp_codes), _ptr(kp_off, _i64p), K)
        if group_off is not None:
            return cls._adopt(L.east_table_groups_dev, doc_off, doc_m, device, *args, gp, G, _vp(out_devptr),
                              *_peers_arg(peer_rows), _vp(stream))
        if peer_rows:
            return cls._adopt(L.east_table_dev_gather, doc_off, doc_m, device, *args, 1 if normalized else 0, _vp(out_devptr),
                              *_peers_arg(peer_rows), _vp(stream))
        return cls._adopt(L.east_table_dev, doc_off, doc_m, device, *args, 1 if normalized else 0, _vp(out_devptr), _vp(stream))

    def score_table_into(self, kp_codes, kp_off, out, normalized=True):
        """score_table() into a caller-provided float64 [n_docs, K] host array (may be pinned)."""
        K = len(kp_off) - 1
        assert out.dtype == np.float64 and out.flags["C_CONTIGUOUS"] and out.size == self.n_docs * K
        kp_codes = np.ascontiguousarray(kp_codes, dtype=np.uint32)
        kp_off = np.ascontiguousarray(kp_off, dtype=np.int64)
        _check(load().east_score_table_host(self._h, _ptr(kp_codes, _u32p), _ptr(kp_off, _i64p), K,
                                            1 if normalized else 0, _ptr(out, _f64p)))
        self.score_timings = last_timings()
        return out

    @classmethod
    def build_dev(cls, text_devptr, doc_off, doc_m, device=0, stream=0):
        """Build from a device-resident packed text (bench: inputs already in HBM)."""
        L = load()
        doc_off = np.ascontiguousarray(doc_off, dtype=np.int64)
        doc_m = np.ascontiguousarray(doc_m, dtype=np.int32)
        h = _vp()
        _check(L.east_build_dev(_vp(text_devptr), _ptr(doc_off, _i64p), _ptr(doc_m, _i32p), len(doc_m),
                                int(device), _vp(stream), ctypes.byref(h)))
        return cls.from_handle(h, doc_off, doc_m, int(device))

    def save(self, path):
        """Write the index (text, suffix array, tables, scorer side tables) to `path` (east_index_save)."""
        _check(load().east_index_save(self._h, os.fsencode(path)))

    @classmethod
    def load(cls, path, device=0):
        """Load an index written by save() onto `device`; scores and arrays equal the saved index's."""
        L = load()
        h = _vp()
        _check(L.east_index_load(os.fsencode(path), int(device), ctypes.byref(h)))
        n_docs = ctypes.c_int32()
        _check(L.east_index_info(h, ctypes.byref(n_docs), None, None, None, None))
        doc_off, doc_m = [0], []
        off, n, m = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int32()
        for d in range(n_docs.value):
            _check(L.east_index_doc(h, d, ctypes.byref(off), ctypes.byref(n), ctypes.byref(m)))
            doc_off.append(off.value + n.value)
            doc_m.append(m.value)
        return cls.from_handle(h, doc_off, doc_m, int(device))

    def strings_collection(self, doc):
        """The strings of a document, decoded from the packed text of the index (for indexes loaded from a file)."""
        text = self.array(doc, PACKED_TEXT).view(np.uint32)
        ends = np.nonzero(text >= 0x0A00)[0]
        out, start = [], 0
        for e in ends.tolist():
            out.append(text[start:e].astype("<u4").tobytes().decode("utf-32-le", errors="surrogatepass"))
            start = e + 1
        return out

    def close(self):
        """Free the index (waits for its table kernels); afterwards build_timings holds the per-stage
        device times of its build."""
        if getattr(self, "_h", None):
            load().east_free(self._h)
            self._h = None
            self.build_timings = last_timings()

    def wait(self):
        """Block until every table of the index is complete (build calls return once the suffix array
        is final; LCP / child / annotation tables finish on an auxiliary stream)."""
        p = _vp()
        _check(load().east_index_devptr(self._h, LCPTAB, ctypes.byref(p)))
        self.build_timings = last_timings()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self):
        n_docs, n_total, dev, rounds, fast = (ctypes.c_int32(), ctypes.c_int64(), ctypes.c_int32(),
                                              ctypes.c_int32(), ctypes.c_int32())
        _check(load().east_index_info(self._h, ctypes.byref(n_docs), ctypes.byref(n_total), ctypes.byref(dev),
                                      ctypes.byref(rounds), ctypes.byref(fast)))
        return {"n_docs": n_docs.value, "n_total": n_total.value, "device": dev.value,
                "rounds": rounds.value, "fast_path": bool(fast.value),
                "doc_sorted": bool(self.stat("doc_sorted")), "doc_sort_overflow": bool(self.stat("doc_sort_overflow"))}

    def stat(self, name):
        v = ctypes.c_int64(0)
        _check(load().east_index_stat(self._h, name.encode(), ctypes.byref(v)))
        return int(v.value)

    def array(self, doc, which):
        if not 0 <= doc < self.n_docs:
            raise ValueError("document %r out of range" % (doc,))
        n = int(self.doc_off[doc + 1] - self.doc_off[doc])
        out = np.empty(n, dtype=np.int32)
        _check(load().east_index_copy(self._h, int(doc), int(which), _ptr(out, _i32p)))
        return out

    def devptr(self, which):
        p = _vp()
        _check(load().east_index_devptr(self._h, int(which), ctypes.byref(p)))
        return p.value

    def score_table(self, kp_codes, kp_off, normalized=True):
        """-> float64 array [n_docs, K] (doc-major, SURVEY 5.8)."""
        K = len(kp_off) - 1
        kp_codes = np.ascontiguousarray(kp_codes, dtype=np.uint32)
        kp_off = np.ascontiguousarray(kp_off, dtype=np.int64)
        out = np.empty((self.n_docs, K), dtype=np.float64)
        if kp_codes.size == 0:
            kp_codes = np.zeros(1, dtype=np.uint32)
        _check(load().east_score_table_host(self._h, _ptr(kp_codes, _u32p), _ptr(kp_off, _i64p), K,
                                            1 if normalized else 0, _ptr(out, _f64p)))
        self.score_timings = last_timings()
        return out

    def score_table_dev(self, kp_devptr, kp_off, out_devptr, normalized=True, stream=0):
        kp_off = np.ascontiguousarray(kp_off, dtype=np.int64)
        _check(load().east_score_table_dev(self._h, _vp(kp_devptr), _ptr(kp_off, _i64p), len(kp_off) - 1,
                                           1 if normalized else 0, _vp(out_devptr), _vp(stream)))
        self.score_timings = last_timings()

    def score_range_dev(self, kp_devptr, kp_off, doc_begin, doc_count, out_devptr, normalized=True, stream=0):
        """Rows of documents [doc_begin, doc_begin + doc_count) into out[doc_count, K] (device)."""
        kp_off = np.ascontiguousarray(kp_off, dtype=np.int64)
        _check(load().east_score_range_dev(self._h, _vp(kp_devptr), _ptr(kp_off, _i64p), len(kp_off) - 1,
                                           1 if normalized else 0, int(doc_begin), int(doc_count), _vp(out_devptr), _vp(stream)))
        self.score_timings = last_timings()

    def score_groups(self, kp_codes, kp_off, group_off, doc_begin=0, doc_count=None):
        """Synonym-expanded scores (pack_variant_groups) of documents [doc_begin, doc_begin + doc_count): float64
        [doc_count, G], the best normalized score over the variants of each group (east_score_groups_host)."""
        kp_codes = np.ascontiguousarray(kp_codes, dtype=np.uint32)
        kp_off = np.ascontiguousarray(kp_off, dtype=np.int64)
        group_off = np.ascontiguousarray(group_off, dtype=np.int64)
        if len(kp_off) and kp_codes.size < kp_off[-1]:
            raise ValueError("variant offsets run past the code points")
        if doc_count is None:
            doc_count = self.n_docs - doc_begin
        G = len(group_off) - 1
        out = np.empty((max(int(doc_count), 0), max(G, 0)), dtype=np.float64)
        if kp_codes.size == 0:
            kp_codes = np.zeros(1, dtype=np.uint32)
        _check(load().east_score_groups_host(self._h, _ptr(kp_codes, _u32p), _ptr(kp_off, _i64p), len(kp_off) - 1,
                                             _ptr(group_off, _i64p), G, int(doc_begin), int(doc_count), _ptr(out, _f64p)))
        self.score_timings = last_timings()
        return out

    def score_groups_dev(self, kp_devptr, kp_off, group_off, out_devptr, doc_begin=0, doc_count=None, stream=0):
        """score_groups() with the code points and the [doc_count, G] table on the device (east_score_groups_dev)."""
        kp_off = np.ascontiguousarray(kp_off, dtype=np.int64)
        group_off = np.ascontiguousarray(group_off, dtype=np.int64)
        if doc_count is None:
            doc_count = self.n_docs - doc_begin
        _check(load().east_score_groups_dev(self._h, _vp(kp_devptr), _ptr(kp_off, _i64p), len(kp_off) - 1,
                                            _ptr(group_off, _i64p), len(group_off) - 1, int(doc_begin), int(doc_count),
                                            _vp(out_devptr), _vp(stream)))
        self.score_timings = last_timings()

    def score_probes_dev(self, kp_devptr, kp_off, out_devptr, stream=0):
        """Normalized table via the probe-counting scorer; returns the number of probes."""
        kp_off = np.ascontiguousarray(kp_off, dtype=np.int64)
        probes = ctypes.c_int64(0)
        _check(load().east_score_probes_dev(self._h, _vp(kp_devptr), _ptr(kp_off, _i64p), len(kp_off) - 1,
                                            _vp(out_devptr), _vp(stream), ctypes.byref(probes)))
        return probes.value

    def score_one(self, doc, q_codes, normalized=True, want_suffix_scores=False):
        q_codes = np.ascontiguousarray(q_codes, dtype=np.uint32)
        L = int(q_codes.size)
        score = ctypes.c_double(0.0)
        ss = np.zeros(max(L, 1), dtype=np.float64)
        qp = _ptr(q_codes, _u32p) if L else None
        _check(load().east_score_one(self._h, int(doc), qp, L, 1 if normalized else 0, ctypes.byref(score),
                                     _ptr(ss, _f64p) if want_suffix_scores else None))
        return (score.value, ss[:L]) if want_suffix_scores else score.value


def cooc_host(S, threshold, device=0):
    """C = B B^T with B[k][d] = S[d][k] >= threshold; S float64 [D, K] -> int32 [K, K]."""
    S = np.ascontiguousarray(S, dtype=np.float64)
    D, K = S.shape
    C = np.empty((K, K), dtype=np.int32)
    _check(load().east_cooc_host(_ptr(S, _f64p), D, K, float(threshold), _ptr(C, _i32p), int(device)))
    return C


def cooc_dev(S_devptr, D, K, threshold, C_devptr, device=0, stream=0):
    _check(load().east_cooc_dev(_vp(S_devptr), int(D), int(K), float(threshold), _vp(C_devptr), int(device),
                                _vp(stream)))
