# -*- coding: utf-8 -*-
"""The "easa" engine: Enhanced Annotated Suffix Array, built and queried on a B200.

Drop-in for east/asts/easa.py:12-400.  Same class name, constructor, attributes
(string, suftab, lcptab, childtab_up, childtab_down, childtab_next_l_index, anntab;
easa.py:18-24) and score()/traverse_*() behaviour; the arrays live in HBM and are copied
to numpy (int64, like the reference's np.int) on first access.

Construction and scoring run in libeast_b200.so (hand-written sm_100a CUDA); there is no
CPU implementation in this package.
"""
import numpy as np

from east import _capi
from east import consts
from east.asts import base
from east.asts import utils


class EnhancedAnnotatedSuffixArray(base.AST):

    __algorithm__ = consts.ASTAlgorithm.EASA

    def __init__(self, strings_collection, _index=None, _doc=0, device=0):
        if strings_collection is None and _index is not None:
            # indexed from raw text on the device (or loaded from a file): the strings are decoded on first use
            self._strings_collection = None
        else:
            super(EnhancedAnnotatedSuffixArray, self).__init__(strings_collection)
            self._strings_collection = strings_collection
        if _index is None:
            packed = utils.pack_strings_collection(strings_collection)
            _index = _capi.DeviceIndex([packed], [len(strings_collection)], device=device)
            _doc = 0
        self._index = _index
        self._doc = _doc
        self._cache = {}

    @property
    def strings_collection(self):
        if self._strings_collection is None:
            self._strings_collection = self._index.strings_collection(self._doc)
        return self._strings_collection

    # ---- the reference's attributes, materialised lazily from device memory ----
    def _array(self, which):
        if which not in self._cache:
            self._cache[which] = self._index.array(self._doc, which).astype(np.int64)
        return self._cache[which]

    @property
    def string(self):
        if "string" not in self._cache:
            self._cache["string"] = "".join(utils.make_unique_endings(self.strings_collection))
        return self._cache["string"]

    suftab = property(lambda self: self._array(_capi.SUFTAB))
    lcptab = property(lambda self: self._array(_capi.LCPTAB))
    childtab_up = property(lambda self: self._array(_capi.CHILDTAB_UP))
    childtab_down = property(lambda self: self._array(_capi.CHILDTAB_DOWN))
    childtab_next_l_index = property(lambda self: self._array(_capi.CHILDTAB_NEXT_L_INDEX))
    anntab = property(lambda self: self._array(_capi.ANNTAB))

    # ---- scoring (easa.py:26-36) ----
    def score(self, query, normalized=True, synonimizer=None, return_suffix_scores=False):
        if synonimizer:
            # easa.py:27-34: best score over all synonym substitutions, always normalized -- one grouped engine call
            codes, off, group_off = _capi.pack_variant_groups([query], synonimizer.get_synonyms())
            result = self._index.score_groups(codes, off, group_off, doc_begin=self._doc, doc_count=1)[0, 0]
            return np.float64(result) if result != 0 else 0  # the reference's max keeps _score's int 0
        return self._score(query.replace(" ", ""), normalized, return_suffix_scores)

    def _score(self, query, normalized=True, return_suffix_scores=False):
        codes = utils.codepoints(query)
        if return_suffix_scores:
            result, per_suffix = self._index.score_one(self._doc, codes, normalized, True)
            suffix_scores = {}
            for s in range(len(query)):
                v = per_suffix[s]
                suffix_scores[query[s:]] = np.float64(v) if v != 0 else 0
            return (np.float64(result) if result != 0 else 0), suffix_scores
        result = self._index.score_one(self._doc, codes, normalized, False)
        return np.float64(result) if result != 0 else 0  # the reference returns int 0 on no match

    # ---- traversals (easa.py:38-89), host side over the downloaded tables ----
    def _lcp_value(self, i, j):
        """lcp value of the interval [i..j] read off the child table (easa.py:349-356), including
        the reference's treatment of the root and of singleton intervals."""
        n = len(self.suftab)
        if (i == 0 or i == n - 1) and j == n - 1:
            return 0
        up_next = self.childtab_up[j + 1]  # IndexError for j == n - 1, exactly as the reference
        if i < up_next <= j:
            return self.lcptab[up_next]
        return self.lcptab[self.childtab_down[i]]

    def _get_child_intervals(self, i, j):
        """Child intervals (l, i', j', first character of the edge) of [i..j] in rank order:
        first l-index from up[j+1] / down[i], then the next-l-index chain (easa.py:358-377)."""
        if i == j:
            return []
        n = len(self.suftab)
        depth = self._lcp_value(i, j)
        sa, text, nxt = self.suftab, self.string, self.childtab_next_l_index
        out = []
        if i == 0 and j == n - 1:
            cut = 0
        else:
            cut = self.childtab_up[j + 1] if i < self.childtab_up[j + 1] else self.childtab_down[i]
            out.append((self._lcp_value(i, cut - 1), i, cut - 1, text[sa[i] + depth]))
        while nxt[cut] != 0:
            following = nxt[cut]
            out.append((self._lcp_value(cut, following - 1), cut, following - 1, text[sa[cut] + depth]))
            cut = following
        out.append((self._lcp_value(cut, j), cut, j, text[sa[cut] + depth]))
        return out

    def traverse_depth_first_pre_order(self, callback):
        n = len(self.suftab)

        def visit(node):
            callback(node)
            if node[1] != node[2]:
                for child in sorted(self._get_child_intervals(node[1], node[2]), key=lambda c: c[3]):
                    visit(child)

        visit([0, 0, n - 1, ""])

    def traverse_depth_first_post_order(self, callback):
        """Bottom-up over lcp-intervals; callback receives [l, i, j, children]."""
        lcp = self.lcptab
        n = len(lcp)
        stack = [[0, 0, None, []]]
        for k in range(1, n):
            left = k - 1
            pending = None
            while lcp[k] < stack[-1][0]:
                done = stack.pop()
                done[2] = k - 1
                callback(done)
                left = done[1]
                if lcp[k] <= stack[-1][0]:
                    stack[-1][3].append(done)
                    pending = None
                else:
                    pending = done
            if lcp[k] > stack[-1][0]:
                stack.append([int(lcp[k]), left, None, [pending] if pending else []])
        stack[-1][2] = n - 1
        callback(stack[-1])

    def traverse_breadth_first(self, callback):
        raise NotImplementedError


class _TreeAlias(EnhancedAnnotatedSuffixArray):
    """The reference's pointer-tree engines give exactly the scores of EASA (its own test,
    tests/asts/test_base.py:16-24, asserts equality); their names resolve to the B200 engine."""

    __algorithm__ = None


class LinearAnnotatedSuffixTreeAlias(_TreeAlias):
    __algorithm__ = consts.ASTAlgorithm.AST_LINEAR


class NaiveAnnotatedSuffixTreeAlias(_TreeAlias):
    __algorithm__ = consts.ASTAlgorithm.AST_NAIVE
