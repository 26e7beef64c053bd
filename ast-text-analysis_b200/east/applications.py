# -*- coding: utf-8 -*-
"""Keyphrase table and keyphrase graph (mirror of east/applications.py:11-149).

Same signatures and return structures as the reference.  With an ASTRelevanceMeasure the
K x D scoring loop (applications.py:43-52) is one batched device call, and the K^2 set
intersections of the graph (applications.py:136-147) are one boolean matrix product
C = B B^T on the device.
"""
import itertools

import numpy as np

from east import _capi
from east import consts
from east import logging
from east import relevance
from east import utils


def _score_matrix(keyphrases, texts, similarity_measure, synonimizer, language):
    """(kept keyphrases, text titles, float64 [D, K] scores) -- the table before dict-ification."""
    similarity_measure = similarity_measure or relevance.ASTRelevanceMeasure()
    text_titles = list(texts.keys())
    text_collection = list(texts.values())
    kept = [kp for kp in keyphrases if kp]  # empty keyphrases are skipped (applications.py:44-45)
    prepared = [utils.prepare_text(kp) for kp in kept]
    if isinstance(similarity_measure, relevance.ASTRelevanceMeasure) and prepared:
        # the measure scores the keyphrases -- with a synonimizer, their best synonym variants -- while it indexes the
        # collection (one overlapped engine call)
        similarity_measure.set_text_collection(text_collection, language, prepared_keyphrases=prepared,
                                               synonimizer=synonimizer)
    else:
        similarity_measure.set_text_collection(text_collection, language)
    if not kept or not text_titles:
        return kept, text_titles, np.zeros((len(text_titles), len(kept)))
    if synonimizer is not None and isinstance(similarity_measure, relevance.ASTRelevanceMeasure):
        # the table scored while indexing (a grouped call per device batch for other indexes)
        scores = similarity_measure.relevance_table(prepared, synonimizer)
    elif synonimizer is None and hasattr(similarity_measure, "relevance_table"):
        scores = similarity_measure.relevance_table(prepared)
    else:
        scores = np.empty((len(text_titles), len(kept)), dtype=np.float64)
        total = scores.size
        step = 0
        for k, kp in enumerate(prepared):
            for j in range(len(text_titles)):
                step += 1
                logging.progress("Calculating matching scores", step, total)
                scores[j, k] = similarity_measure.relevance(kp, text=j, synonimizer=synonimizer)
        logging.clear()
    return kept, text_titles, scores


def keyphrases_table(keyphrases, texts, similarity_measure=None, synonimizer=None,
                     language=consts.Language.ENGLISH):
    """{keyphrase: {text name: matching score}} -- east/applications.py:11-56."""
    kept, titles, scores = _score_matrix(keyphrases, texts, similarity_measure, synonimizer, language)
    res = {}
    for k, kp in enumerate(kept):
        column = scores[:, k]
        res[kp] = {titles[j]: (column[j] if column[j] != 0 else 0) for j in range(len(titles))}
    return res


def keyphrases_graph(keyphrases, texts, referral_confidence=0.6, relevance_threshold=0.25,
                     support_threshold=1, similarity_measure=None, synonimizer=None,
                     language=consts.Language.ENGLISH):
    """Keyphrase relation graph -- east/applications.py:59-149.

    Node ids are positions in `keyphrases`; nodes below the support threshold are dropped
    without renumbering; edges are ordered pairs (permutations order) whose confidence
    |T1 & T2| / max(|T1|, 1) reaches referral_confidence.
    """
    similarity_measure = similarity_measure or relevance.ASTRelevanceMeasure()
    if isinstance(similarity_measure, relevance.ASTRelevanceMeasure):
        # the measure counts the co-occurrences while it indexes the collection (one graph call per device batch): the
        # relevance bytes come out of the scoring kernel and no score table is formed
        kept = [kp for kp in keyphrases if kp]
        prepared = [utils.prepare_text(kp) for kp in kept]
        text_collection = list(texts.values())
        if prepared:
            similarity_measure.set_text_collection(text_collection, language, prepared_keyphrases=prepared,
                                                   synonimizer=synonimizer, relevance_threshold=relevance_threshold)
        else:
            similarity_measure.set_text_collection(text_collection, language)
        if kept and texts:
            cooc = similarity_measure.cooccurrence(prepared, relevance_threshold, synonimizer)
        else:
            cooc = np.zeros((len(kept), len(kept)), dtype=np.int32)
        return graph_on_device(keyphrases, kept, cooc, referral_confidence, relevance_threshold, support_threshold)
    kept, titles, scores = _score_matrix(keyphrases, texts, similarity_measure, synonimizer, language)
    if scores.size:
        cooc = _capi.cooc_host(scores, relevance_threshold)
    else:
        cooc = np.zeros((len(kept), len(kept)), dtype=np.int32)
    return graph_on_device(keyphrases, kept, cooc, referral_confidence, relevance_threshold, support_threshold)


def graph_on_device(keyphrases, kept, cooc, referral_confidence, relevance_threshold, support_threshold):
    """graph_from_cooccurrence assembled where the counts are (east_graph_edges_*): the same graph dict, and only the
    supports and the edges come back from the device.  cooc: int32 [K, K], or [T, K, K] with T relevance thresholds
    (relevance_threshold then a sequence of T: a list of T graphs comes back); a numpy array or a CUDA torch tensor.
    The one difference from graph_from_cooccurrence: no node is paired with itself, whatever referral_confidence (the
    host function pairs every node with itself at referral_confidence <= -1; the reference never does)."""
    planes = np.ndim(relevance_threshold) != 0
    thresholds = list(relevance_threshold) if planes else [relevance_threshold]
    node_col = _node_columns(keyphrases, kept)
    if len(keyphrases):
        support, n_edges, src, dst, conf = _capi.graph_edges(cooc, node_col, referral_confidence, support_threshold)
        bounds = np.concatenate([[0], np.cumsum(n_edges)]).tolist()
    else:   # no node, nothing to count
        support, bounds = np.zeros((len(thresholds), 0), dtype=np.int32), [0] * (len(thresholds) + 1)
        src = dst = conf = np.zeros(0)
    graphs = [graph_from_edges(keyphrases, support[t], src[bounds[t]:bounds[t + 1]], dst[bounds[t]:bounds[t + 1]],
                               conf[bounds[t]:bounds[t + 1]], referral_confidence, r, support_threshold)
              for t, r in enumerate(thresholds)]
    return graphs if planes else graphs[0]


def _node_columns(keyphrases, kept):
    """the column of every keyphrase, as graph_from_cooccurrence picks it"""
    column_of = {}
    for k, kp in enumerate(kept):
        column_of[kp] = k  # duplicate keyphrases share one table row (last wins, like a dict)
    for kp in keyphrases:
        if kp not in column_of:
            raise KeyError(kp)  # the reference indexes table[keyphrase] for skipped empty keyphrases
    return np.array([column_of[kp] for kp in keyphrases], dtype=np.int32)


def graph_from_edges(keyphrases, support, src, dst, conf, referral_confidence, relevance_threshold, support_threshold):
    """The graph dict of graph_from_cooccurrence from one plane of _capi.graph_edges: support[n] of every keyphrase,
    the edges (node positions src -> dst, their confidences) in permutations order."""
    support = support.tolist()
    return {
        "nodes": [{"id": i, "label": kp, "support": support[i]} for i, kp in enumerate(keyphrases)
                  if support[i] >= support_threshold],
        "edges": [{"source": s, "target": d, "confidence": c} for s, d, c in zip(src.tolist(), dst.tolist(), conf.tolist())],
        "referral_confidence": referral_confidence,
        "relevance_threshold": relevance_threshold,
        "support_threshold": support_threshold,
    }


def graph_from_cooccurrence(keyphrases, kept, cooc, referral_confidence, relevance_threshold, support_threshold):
    """The graph dict of east/applications.py:115-149 from the co-occurrence counts cooc[k1][k2] = number of texts
    in which both kept keyphrases k1 and k2 reach the relevance threshold (diagonal: the support)."""
    column_of = {}
    for k, kp in enumerate(kept):
        column_of[kp] = k  # duplicate keyphrases share one table row (last wins, like a dict)
    for kp in keyphrases:
        if kp not in column_of:
            raise KeyError(kp)  # the reference indexes table[keyphrase] for skipped empty keyphrases
    support = {kp: int(cooc[column_of[kp], column_of[kp]]) for kp in keyphrases}

    graph = {
        "nodes": [{"id": i, "label": kp, "support": support[kp]} for i, kp in enumerate(keyphrases)],
        "edges": [],
        "referral_confidence": referral_confidence,
        "relevance_threshold": relevance_threshold,
        "support_threshold": support_threshold,
    }
    graph["nodes"] = [n for n in graph["nodes"] if support[n["label"]] >= support_threshold]
    nodes = graph["nodes"]
    if len(nodes) > 1:
        cols = np.array([column_of[n["label"]] for n in nodes])
        counts = cooc[np.ix_(cols, cols)].astype(np.float64)
        sup = np.array([max(support[n["label"]], 1) for n in nodes], dtype=np.float64)
        confidence = counts / sup[:, None]  # IEEE double divide, as float(len(..)) / max(len(..), 1)
        np.fill_diagonal(confidence, -1.0)
        src, dst = np.nonzero(confidence >= referral_confidence)  # row-major == permutations order
        for i1, i2 in zip(src.tolist(), dst.tolist()):
            graph["edges"].append({"source": nodes[i1]["id"], "target": nodes[i2]["id"],
                                   "confidence": float(confidence[i1, i2])})
    return graph
