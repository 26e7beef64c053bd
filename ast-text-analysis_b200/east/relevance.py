# -*- coding: utf-8 -*-
"""Relevance measures (mirror of east/relevance.py:16-53; the cosine measure is out of scope).

ASTRelevanceMeasure keeps the reference's interface -- set_text_collection(texts, language)
and relevance(keyphrase, text=j) -- but indexes the whole collection as ONE device batch and
adds relevance_table(), which scores every (keyphrase, text) pair in one call; that is what
east.applications.keyphrases_table uses instead of K x D single-pair calls.
"""
import numpy as np

from east import _capi
from east import consts
from east import logging
from east import utils
from east.asts import base
from east.asts import easa
from east.asts import utils as asts_utils


import re

# what csrc/tokenize.cu handles: ASCII, the Cyrillic block up to U+045F and -- as separators -- the non-alphanumeric signs of
# U+0080-00BF (mask TK_LATIN1_SEPARATORS), General Punctuation, the numero sign and the byte order mark
_LATIN1_SEPARATORS = 0x89d3fbffffffffff
_DEVICE_TEXT_RE = re.compile("[\\x00-\\x7f\\u0400-\\u045f\\u2000-\\u206f\\u2116\\ufeff%s]*\\Z" % "".join(
    "\\x%02x" % (0x80 + i) for i in range(64) if (_LATIN1_SEPARATORS >> i) & 1))
SMALL_DOCUMENT_LIMIT = 65535   # code points: the per-document shared-memory kernel (csrc/doc_sort.cu) takes these
MAX_BATCH_CODE_POINTS = 1 << 29   # one device index addresses < 2^30 code points (int32 ranks)


def plan_batches(sizes, small_limit=SMALL_DOCUMENT_LIMIT, max_batch=MAX_BATCH_CODE_POINTS):
    """Split a collection into device batches: documents the per-document kernel can take are kept apart from
    larger ones (one large text would otherwise send the whole batch to the global sort), and no batch exceeds
    what one index addresses.  Returns lists of document numbers, original order kept inside a batch."""
    batches = []
    for wanted_small in (True, False):
        cur, cur_size = [], 0
        for j, size in enumerate(sizes):
            if (size <= small_limit) != wanted_small:
                continue
            if cur and cur_size + size > max_batch:
                batches.append(cur)
                cur, cur_size = [], 0
            cur.append(j)
            cur_size += size
        if cur:
            batches.append(cur)
    return batches


class RelevanceMeasure(object):

    def set_text_collection(self, texts, language=consts.Language.ENGLISH):
        raise NotImplementedError()

    def relevance(self, keyphrase, text, synonimizer=None):
        raise NotImplementedError()


class ASTRelevanceMeasure(RelevanceMeasure):

    def __init__(self, ast_algorithm=consts.ASTAlgorithm.EASA, normalized=True, device=0, device_preprocessing=True):
        super(ASTRelevanceMeasure, self).__init__()
        self.device_preprocessing = device_preprocessing
        self.ast_algorithm = ast_algorithm
        self.normalized = normalized
        self.device = device
        self.asts = []
        self._index = None
        self._batches = []
        self._table = None
        self._table_keyphrases = None
        self._table_groups = None
        self._cooc = None
        self._cooc_key = None

    def set_text_collection(self, texts, language=consts.Language.ENGLISH, prepared_keyphrases=None, synonimizer=None,
                            relevance_threshold=None):
        """relevance.py:34-49: one AST per text; here all of them in one batched build.

        prepared_keyphrases (optional, what keyphrases_table passes): the keyphrases relevance_table() is
        going to be asked for.  Each batch is then built AND scored by one engine call, which overlaps the
        scoring of the documents already indexed with the transfer of the rest (east_table_host).
        synonimizer (optional, with prepared_keyphrases): the table scored while indexing is the synonym table of
        relevance_table(prepared_keyphrases, synonimizer) -- the best variant of each keyphrase, always normalized
        (east_table_groups_host / east_table_texts_groups_host).
        relevance_threshold (optional, with prepared_keyphrases): what keyphrases_graph passes.  Each batch is then built
        and counted by one graph call instead (east_graph_host / east_graph_texts_host): the co-occurrence counts of
        cooccurrence(prepared_keyphrases, relevance_threshold, synonimizer) are summed over the batches and no score
        table is formed."""
        self.texts = texts
        self.language = language
        self.asts = []
        self._index = None
        self._batches = []
        self._table = None
        self._table_keyphrases = None
        self._table_groups = None
        self._cooc = None
        self._cooc_key = None
        total_texts = len(texts)
        if self.ast_algorithm not in tuple(consts.ASTAlgorithm):
            # other registered engines (none ship in this package) go through the registry
            for i in range(total_texts):
                self.asts.append(base.AST.get_ast(utils.text_to_strings_collection(texts[i]),
                                                  self.ast_algorithm))
                logging.progress("Indexing texts with ASTs", i + 1, total_texts)
            logging.clear()
            return
        if not texts:
            return
        # the synonym variants are expanded and packed once: the same arrays go to every device batch
        groups = (_capi.pack_variant_groups(prepared_keyphrases, synonimizer.get_synonyms())
                  if prepared_keyphrases and synonimizer else None)
        graph = bool(prepared_keyphrases) and relevance_threshold is not None
        threshold = relevance_threshold if graph else None
        if prepared_keyphrases and self.device_preprocessing and self._set_text_collection_on_device(texts, prepared_keyphrases,
                                                                                                    groups, threshold):
            return
        collections = [utils.text_to_strings_collection(text) for text in texts]
        # one byte per code point where the text allows it (ASCII / Latin-1: a quarter of the bytes over the host link),
        # uint32 code points otherwise; both have one entry per code point + one per string
        packed = [asts_utils.pack_strings_collection_u8(c) for c in collections]
        packed = [p if p is not None else asts_utils.pack_strings_collection(c) for p, c in zip(packed, collections)]
        fused = (groups[:2] if groups else _capi.pack_keyphrases(prepared_keyphrases)) if prepared_keyphrases else None
        # everything is built into locals: a batch that raises leaves the measure empty, not half-initialised
        asts = [None] * len(collections)
        batches = []
        table = np.empty((len(collections), len(prepared_keyphrases)), dtype=np.float64) if fused and not graph else None
        cooc = None
        for docs in plan_batches([len(p) for p in packed]):
            narrow = all(packed[j].dtype == np.uint8 for j in docs)
            parts = [packed[j] if narrow or packed[j].dtype == np.uint32 else asts_utils.pack_strings_collection(collections[j])
                     for j in docs]
            doc_off = np.zeros(len(docs) + 1, dtype=np.int64)
            np.cumsum([len(p) for p in parts], out=doc_off[1:])
            text = np.ascontiguousarray(np.concatenate(parts) if len(parts) > 1 else parts[0])
            doc_m = [len(collections[j]) for j in docs]
            if fused is None:
                build = _capi.DeviceIndex.build_host_u8 if narrow else _capi.DeviceIndex.build_host
                index = build(text, doc_off, doc_m, device=self.device)
            elif graph:
                counts, index = _capi.DeviceIndex.build_host_and_graph(text, doc_off, doc_m, fused[0], fused[1], threshold,
                                                                       normalized=self.normalized, device=self.device,
                                                                       group_off=groups[2] if groups else None)
                cooc = counts if cooc is None else cooc + counts   # int32: exact (counts <= number of texts)
            else:
                rows = np.empty((len(docs), len(prepared_keyphrases)), dtype=np.float64)
                index = _capi.DeviceIndex.build_host_and_score(text, doc_off, doc_m, fused[0], fused[1], rows,
                                                               normalized=self.normalized, device=self.device,
                                                               group_off=groups[2] if groups else None)
                table[docs] = rows
            batches.append((index, docs))
            for local, j in enumerate(docs):
                asts[j] = easa.EnhancedAnnotatedSuffixArray(collections[j], _index=index, _doc=local)
        self.asts, self._batches, self._index = asts, batches, batches[0][0]
        if graph:
            self._cooc, self._cooc_key = cooc, self._counts_key(prepared_keyphrases, groups, threshold)
        elif fused:
            self._table, self._table_keyphrases, self._table_groups = table, list(prepared_keyphrases), groups

    def _counts_key(self, prepared_keyphrases, groups, threshold):
        return list(prepared_keyphrases), groups, float(threshold), bool(self.normalized)

    def _set_text_collection_on_device(self, texts, prepared_keyphrases, groups=None, threshold=None):
        """keyphrases_table for a collection of small ASCII / Cyrillic texts: ONE engine call takes the raw texts,
        does the preprocessing of utils.text_to_strings_collection on the device (csrc/tokenize.cu), indexes and scores
        (east_table_texts_host; with groups -- pack_variant_groups -- the synonym table, east_table_texts_groups_host).
        Returns False when the collection needs the host preprocessing (other scripts -- Python's Unicode tables --, a
        text too large for the per-document kernel, several device batches).  threshold: the co-occurrence counts of a
        keyphrase graph instead of the table (east_graph_texts_host)."""
        total = 0
        for t in texts:
            if isinstance(t, (bytes, bytearray)):
                size = len(t)
            elif t.isascii():
                size = len(t)
            elif _DEVICE_TEXT_RE.match(t):
                size = 3 * len(t)   # bound on the UTF-8 size
            else:
                return False
            if size > SMALL_DOCUMENT_LIMIT - 2:
                return False
            total += size
        if total >= MAX_BATCH_CODE_POINTS:
            return False
        fused = groups[:2] if groups else _capi.pack_keyphrases(prepared_keyphrases)
        group_off = groups[2] if groups else None
        table = None
        try:
            if threshold is None:
                table = np.empty((len(texts), len(prepared_keyphrases)), dtype=np.float64)
                index = _capi.DeviceIndex.table_from_texts(texts, fused[0], fused[1], table, normalized=self.normalized,
                                                           device=self.device, group_off=group_off)
            else:
                cooc, index = _capi.DeviceIndex.graph_from_texts(texts, fused[0], fused[1], threshold, normalized=self.normalized,
                                                                 device=self.device, group_off=group_off)
        except _capi.UnsupportedText:
            return False
        docs = list(range(len(texts)))
        self.asts = [easa.EnhancedAnnotatedSuffixArray(None, _index=index, _doc=j) for j in docs]
        self._batches, self._index = [(index, docs)], index
        if table is None:
            self._cooc, self._cooc_key = cooc, self._counts_key(prepared_keyphrases, groups, threshold)
        else:
            self._table, self._table_keyphrases, self._table_groups = table, list(prepared_keyphrases), groups
        return True

    def save_index(self, directory):
        """Write the indexed collection to `directory` (one file per device batch + the batch layout), so that a later
        run loads it instead of rebuilding every structure (the reference rebuilds them on every run, relevance.py:38-47)."""
        import json
        import os
        if not self._batches:
            raise ValueError("no text collection has been indexed")
        os.makedirs(directory, exist_ok=True)
        layout = {"normalized": bool(self.normalized), "ast_algorithm": self.ast_algorithm, "n_texts": len(self.asts), "batches": []}
        for b, (index, docs) in enumerate(self._batches):
            name = "batch%04d.eastidx" % b
            index.save(os.path.join(directory, name))
            layout["batches"].append({"file": name, "docs": [int(j) for j in docs]})
        with open(os.path.join(directory, "layout.json"), "w") as f:
            json.dump(layout, f)

    @classmethod
    def load_index(cls, directory, device=0):
        """A measure over the collection saved by save_index(): relevance(), relevance_table() and the asts' attributes
        work as after set_text_collection()."""
        import json
        import os
        with open(os.path.join(directory, "layout.json")) as f:
            layout = json.load(f)
        self = cls(layout["ast_algorithm"], layout["normalized"], device=device)
        asts = [None] * layout["n_texts"]
        batches = []
        for entry in layout["batches"]:
            index = _capi.DeviceIndex.load(os.path.join(directory, entry["file"]), device=device)
            batches.append((index, entry["docs"]))
            for local, j in enumerate(entry["docs"]):
                asts[j] = easa.EnhancedAnnotatedSuffixArray(index.strings_collection(local), _index=index, _doc=local)
        self.asts, self._batches, self._index = asts, batches, batches[0][0]
        return self

    def relevance(self, keyphrase, text, synonimizer=None):
        return self.asts[text].score(keyphrase, normalized=self.normalized, synonimizer=synonimizer)

    def relevance_table(self, prepared_keyphrases, synonimizer=None):
        """Scores of every prepared keyphrase against every text: float64 [n_texts, K].  With a synonimizer, the best
        score over the synonym substitutions of each keyphrase, always normalized (easa.py:27-34)."""
        if synonimizer:
            if self._index is None:
                return np.array([[ast.score(kp, normalized=self.normalized, synonimizer=synonimizer)
                                  for kp in prepared_keyphrases] for ast in self.asts], dtype=np.float64)
            # expanded once; every device batch is one grouped call (the batches after the first reuse the preparation)
            codes, off, group_off = _capi.pack_variant_groups(prepared_keyphrases, synonimizer.get_synonyms())
            if (self._table_groups is not None and list(prepared_keyphrases) == self._table_keyphrases
                    and all(np.array_equal(a, b) for a, b in zip((codes, off, group_off), self._table_groups))):
                return self._table   # the same variants were scored while the collection was being indexed
            table = np.empty((len(self.asts), len(prepared_keyphrases)), dtype=np.float64)
            for index, docs in self._batches:
                table[docs] = index.score_groups(codes, off, group_off)
            return table
        if self._index is None:
            return np.array([[ast.score(kp, normalized=self.normalized) for kp in prepared_keyphrases]
                             for ast in self.asts], dtype=np.float64)
        if self._table is not None and self._table_groups is None and list(prepared_keyphrases) == self._table_keyphrases:
            return self._table   # scored while the collection was being indexed
        codes, off = _capi.pack_keyphrases(prepared_keyphrases)
        if len(self._batches) == 1:
            return self._index.score_table(codes, off, normalized=self.normalized)
        table = np.empty((len(self.asts), len(prepared_keyphrases)), dtype=np.float64)
        for index, docs in self._batches:
            table[docs] = index.score_table(codes, off, normalized=self.normalized)
        return table

    def cooccurrence(self, prepared_keyphrases, relevance_threshold, synonimizer=None):
        """int32 [K, K] co-occurrence counts: C[i][j] = number of texts in which prepared keyphrases i and j both score
        >= relevance_threshold (with a synonimizer: their best synonym variants), C[k][k] the support of k.  The counts
        of the graph calls made while indexing (set_text_collection with relevance_threshold) when they were made for
        these keyphrases, variants, threshold and normalization; otherwise those of relevance_table()."""
        K = len(prepared_keyphrases)
        if self._cooc is not None:
            groups = _capi.pack_variant_groups(prepared_keyphrases, synonimizer.get_synonyms()) if synonimizer else None
            kps, kgroups, kthr, knorm = self._cooc_key
            same_groups = (groups is None) == (kgroups is None) and (
                groups is None or all(np.array_equal(a, b) for a, b in zip(groups, kgroups)))
            if (list(prepared_keyphrases) == kps and same_groups and float(relevance_threshold) == kthr
                    and bool(self.normalized) == knorm):
                return self._cooc
        if not K or not self.asts:
            return np.zeros((K, K), dtype=np.int32)
        return _capi.cooc_host(self.relevance_table(prepared_keyphrases, synonimizer), relevance_threshold)
