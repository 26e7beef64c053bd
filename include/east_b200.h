/*
 * east_b200.h -- C ABI of libeast_b200.so, the B200 (sm_100a) engine behind EAST's
 * `east.asts` "easa" algorithm.
 *
 * The reference (mikhaildubov/AST-text-analysis, pure Python) has no FFI; its boundary for
 * this path is the Python class east.asts.easa.EnhancedAnnotatedSuffixArray
 * (east/asts/easa.py:12-400) reached through east.asts.base.AST.get_ast
 * (east/asts/base.py:13-18).  Each entry point below names the reference code it replaces.
 * INTEGRATION.md shows the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes, no C++/torch types;
 *   - every function returns 0 on success, a negative east_status on failure, and leaves a
 *     message retrievable with east_last_error() (thread-local);
 *   - "text" is the packed document: the code points of string 0, then 0x0A00+0, the code
 *     points of string 1, then 0x0A00+1, ... (east/asts/utils.py:25-40 + east/asts/easa.py:19);
 *     several documents are concatenated and delimited by doc_off[n_docs+1];
 *   - *_host entry points take host buffers and do their own H<->D copies;
 *     *_dev entry points take device pointers that live on the index's device;
 *   - there is no CPU fallback: without a usable CUDA device every entry point fails;
 *   - the build-and-score entries (east_table_*, east_graph_*) and the score entries (east_score_*) check their
 *     arguments before they touch the device, in one order, and report the first failure: the output (and the peer
 *     list, text_width); the documents (raw texts: their offsets; a score entry: the index and the document range);
 *     the groups; the keyphrases (EAST_ERR_ZERODIV for an empty one).
 */
#ifndef EAST_B200_H
#define EAST_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct east_index east_index; /* opaque, immutable after build */

typedef enum east_status {
    EAST_OK = 0,
    EAST_ERR_INVALID = -1, /* bad argument (NULL, negative size, empty document, ...) */
    EAST_ERR_CUDA = -2,    /* CUDA runtime error or no device */
    EAST_ERR_NOMEM = -3,
    EAST_ERR_ZERODIV = -4, /* empty query: the reference raises ZeroDivisionError (easa.py:134) */
    EAST_ERR_RANGE = -5,   /* size exceeds the int32/2^30 limits of one index */
    EAST_ERR_UNSUPPORTED = -6 /* device preprocessing: a text has characters outside ASCII / U+0400-045F */
} east_status;

/* which array east_index_copy() exports; names follow east/asts/easa.py:18-24 */
typedef enum east_array {
    EAST_SUFTAB = 0,             /* easa.py:141-245  _compute_suftab (values local to the doc) */
    EAST_LCPTAB = 1,             /* easa.py:247-266  _compute_lcptab */
    EAST_CHILDTAB_UP = 2,        /* easa.py:268-287  _compute_childtab */
    EAST_CHILDTAB_DOWN = 3,      /* easa.py:268-287 */
    EAST_CHILDTAB_NEXT_L_INDEX = 4, /* easa.py:289-304 _compute_childtab_next_l_index */
    EAST_ANNTAB = 5,             /* easa.py:306-331  _compute_anntab */
    EAST_PACKED_TEXT = 6         /* easa.py:19  self.string as code points (terminators 0x0A00 + i) */
} east_array;

const char *east_last_error(void);
int east_device_count(void);
const char *east_version(void);

/* ---- build: replaces EnhancedAnnotatedSuffixArray.__init__ (easa.py:16-24) for a batch of
 * documents, i.e. the loop of ASTRelevanceMeasure.set_text_collection (relevance.py:41-47).
 *   text      : concatenated packed documents, doc_off[n_docs] code points
 *   doc_off   : n_docs+1 offsets into text (doc_off[0] == 0)
 *   doc_m     : number of strings (= terminators) of each document
 * Limits: doc_off[n_docs] < 2^30 per index.
 * The call returns once the suffix array (all a scorer needs) is final; the LCP, child and annotation
 * tables are completed on an auxiliary stream so that a following east_score_table_* overlaps them.
 * east_index_copy / east_index_devptr / east_free wait for them (option "sync_build" = 1 makes the
 * build itself wait). */
int east_build_host(const uint32_t *text, const int64_t *doc_off, const int32_t *doc_m,
                    int32_t n_docs, int device, east_index **out);
int east_build_dev(const uint32_t *text_dev, const int64_t *doc_off_host, const int32_t *doc_m_host,
                   int32_t n_docs, int device, void *stream, east_index **out);
void east_free(east_index *idx);

/* ---- introspection (parity checks; the reference exposes these as numpy attributes) */
int east_index_info(const east_index *idx, int32_t *n_docs, int64_t *n_total, int32_t *device,
                    int32_t *rounds, int32_t *fast_path);
int east_index_doc(const east_index *idx, int32_t doc, int64_t *offset, int64_t *n, int32_t *m);
/* how the suffix array was built (tests assert which kernel path ran): name is one of
 * "doc_sorted" (1 = the per-document shared-memory sort, doc_sort.cu), "doc_sort_overflow",
 * "key_chars", "key_bits", "rounds", "active_after_round0", "fast_path" */
int east_index_stat(const east_index *idx, const char *name, int64_t *value);
/* copy one array of one document to a host int32 buffer of n entries */
int east_index_copy(const east_index *idx, int32_t doc, int which, int32_t *dst_host);
/* device pointer to the whole-batch array (global ranks/positions); for tests and benches */
int east_index_devptr(const east_index *idx, int which, const void **ptr);

/* ---- scoring: replaces EnhancedAnnotatedSuffixArray.score/_score (easa.py:26-36, 91-139)
 * for every (document, keyphrase) pair, i.e. the K x D loop of
 * applications.keyphrases_table (applications.py:43-52).
 *   kp      : concatenated code points of the K queries AFTER query.replace(" ", "")
 *   kp_off  : K+1 offsets
 *   out     : doc-major table out[d * K + k], IEEE double
 * A zero-length query makes the call fail with EAST_ERR_ZERODIV. */
int east_score_table_host(const east_index *idx, const uint32_t *kp, const int64_t *kp_off,
                          int32_t K, int normalized, double *out_DxK);
int east_score_table_dev(const east_index *idx, const uint32_t *kp_dev, const int64_t *kp_off_host,
                         int32_t K, int normalized, double *out_DxK_dev, void *stream);
/* Build and score in ONE call: what applications.keyphrases_table does per text (build the structure,
 * applications.py:25 -> relevance.py:34-49, then score every keyphrase, applications.py:43-52), for the
 * whole collection.  Arguments as in east_build_host + east_score_table_host.  On a large batch of small
 * documents the text is copied in runs of whole documents; each run is sorted and scored, and its rows of
 * out_DxK copied back, while the later runs are still arriving.  Results are identical to the two calls.
 * out_idx may be NULL; otherwise it receives the index (east_free it). */
int east_table_host(const uint32_t *text, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs,
                    int device, const uint32_t *kp, const int64_t *kp_off, int32_t K, int normalized,
                    double *out_DxK, east_index **out_idx);
/* The same two host entries for a text shipped as ONE BYTE per code point -- four times fewer bytes over the host link.
 * text8: the code points of string 0 (each < 0xFF, as themselves), then 0xFF, the code points of string 1, then 0xFF, ...:
 * the k-th 0xFF of a document stands for the terminator 0x0A00 + k of east/asts/utils.py:35-39; doc_off / doc_m as above
 * (offsets in code points = bytes).  Texts with a code point >= 0xFF (Cyrillic, CJK) use the uint32 entries.  On a large
 * batch of small documents the per-document kernel byte-codes straight from these bytes and writes the uint32 code
 * points of the index itself; otherwise they are expanded on the device first.  Results are identical to the uint32
 * entries on the equivalent packed text.  EAST_ERR_INVALID when a document does not hold exactly doc_m bytes 0xFF or does
 * not end with one. */
int east_build_host_u8(const uint8_t *text8, const int64_t *doc_off, const int32_t *doc_m,
                       int32_t n_docs, int device, east_index **out);
int east_table_host_u8(const uint8_t *text8, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs,
                       int device, const uint32_t *kp, const int64_t *kp_off, int32_t K, int normalized,
                       double *out_DxK, east_index **out_idx);
/* the same with text, keyphrases and table resident on the device (kp_host: optional host copy of the
 * keyphrase code points, saves a device-to-host round trip; may be NULL) */
int east_table_dev(const uint32_t *text_dev, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs,
                   int device, const uint32_t *kp_dev, const uint32_t *kp_host, const int64_t *kp_off, int32_t K,
                   int normalized, double *out_DxK_dev, void *stream, east_index **out_idx);
/* east_table_dev for a table whose documents are sharded over several GPUs (one process per GPU; the documents are
 * independent: east/relevance.py:41-47), with the all-gather of the per-rank slices fused into the scoring kernel:
 * every row this rank produces is also stored, by the CTA that computed it, at peer_rows[i] + the same row offset --
 * peer_rows[i] = where this rank's slice starts in the gathered table of the i-th other rank, a pointer into that rank's
 * memory mapped into this process (CUDA peer access / torch symmetric memory: the stores travel over NVLink).  The call
 * returns when this rank's kernels are done and its stores are fenced system-wide; the caller then runs a barrier
 * across ranks, after which every rank holds the whole table.  n_peers <= 15.  Without peers it is east_table_dev. */
int east_table_dev_gather(const uint32_t *text_dev, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs,
                          int device, const uint32_t *kp_dev, const uint32_t *kp_host, const int64_t *kp_off, int32_t K,
                          int normalized, double *out_DxK_dev, double *const *peer_rows, int32_t n_peers, void *stream,
                          east_index **out_idx);
/* The host-buffer entries (text_width 4: east_table_host, 1: east_table_host_u8) with the same fused all-gather: the
 * rows go to out_DxK on the host AND to own_rows_dev (this rank's rows of its own gathered table on the device; may be
 * NULL) AND to the other ranks' tables at peer_rows[i]. */
int east_table_host_gather(const void *text, int32_t text_width, const int64_t *doc_off, const int32_t *doc_m,
                           int32_t n_docs, int device, const uint32_t *kp, const int64_t *kp_off, int32_t K,
                           int normalized, double *out_DxK, double *own_rows_dev, double *const *peer_rows,
                           int32_t n_peers, east_index **out_idx);
/* the rows of documents [doc_begin, doc_begin + doc_count) only: out[(d - doc_begin) * K + k].  Lets a caller
 * that shards documents over GPUs overlap the collective of one document tile with the scoring of the next. */
int east_score_range_dev(const east_index *idx, const uint32_t *kp_dev, const int64_t *kp_off_host,
                         int32_t K, int normalized, int32_t doc_begin, int32_t doc_count,
                         double *out_dev, void *stream);
/* synonym-expanded scoring (easa.py:27-34): V variants in kp/kp_off (NOT space-stripped), grouped by
 * group_off[G+1] (host, int64, group_off[0] = 0, strictly increasing, group_off[G] = V); for documents
 * [doc_begin, doc_begin + doc_count): out[(d - doc_begin) * G + g] = max over the group's variants of the
 * normalized score.  Always normalized, as the reference's synonym branch.
 * A group is every substitution of one keyphrase's words by their synonyms: the call walks each distinct query
 * suffix of all variants once per document and keeps only the best variant of each group, so the document x
 * variant table is never formed.  Malformed groups fail with EAST_ERR_INVALID, an empty variant with
 * EAST_ERR_ZERODIV.  The _host entry takes host buffers; the _dev entry takes kp_dev and out_dev on the index's
 * device (kp_off and group_off stay on the host). */
int east_score_groups_host(const east_index *idx, const uint32_t *kp, const int64_t *kp_off, int32_t V,
                           const int64_t *group_off, int32_t G, int32_t doc_begin, int32_t doc_count,
                           double *out_host);
int east_score_groups_dev(const east_index *idx, const uint32_t *kp_dev, const int64_t *kp_off, int32_t V,
                          const int64_t *group_off, int32_t G, int32_t doc_begin, int32_t doc_count,
                          double *out_dev, void *stream);
/* same table through an instrumented scorer that also counts the algorithmic bytes it reads:
 * 8 per (SA word, text word) probe (SURVEY 8(d)); on the fast path 5 per (SA word, text byte)
 * probe and 8 per 2-gram bucket lookup.  *probes receives that byte count. */
int east_score_probes_dev(const east_index *idx, const uint32_t *kp_dev, const int64_t *kp_off_host,
                          int32_t K, double *out_DxK_dev, void *stream, int64_t *probes);
/* single query against one document, with the per-suffix results of
 * return_suffix_scores=True (easa.py:132-137); suffix_scores may be NULL, else len doubles */
int east_score_one(const east_index *idx, int32_t doc, const uint32_t *q, int32_t len,
                   int normalized, double *score, double *suffix_scores);

/* ---- keyphrase graph support: replaces the pair loop of applications.keyphrases_graph
 * (applications.py:111-113, 136-147).  B[k][d] = S[d][k] >= threshold; C = B * B^T (int32);
 * support[k] = C[k][k]. */
int east_cooc_dev(const double *S_DxK_dev, int64_t D, int32_t K, double threshold,
                  int32_t *C_KxK_dev, int device, void *stream);
int east_cooc_host(const double *S_DxK, int64_t D, int32_t K, double threshold,
                   int32_t *C_KxK, int device);

/* ---- measurement hooks (bench.py): per-stage device time of the last build/score call on
 * this thread, measured with CUDA events on the launching stream.
 * names: NUL-separated list written to buf; returns the number of stages. */
int east_last_timings(float *ms, char *names, int32_t cap, int32_t names_cap);
/* per-kernel device time, measured with a CUDA event pair around every launch while the
 * per-thread option "time_kernels" is 1 (set it to 0 to stop and clear).  names: NUL-separated.
 * bytes: algorithmic bytes moved by those launches (roofline numerator).  Returns #kernels. */
int east_kernel_stats(char *names, int32_t names_cap, double *ms, int64_t *launches, double *bytes,
                      int32_t cap);
/* number of kernel launches issued by the library on this thread since the last reset */
int64_t east_launch_count(int reset);
/* ---- preprocessing on the device: replaces utils.text_to_strings_collection (east/utils.py:31-79: utf-8 decode, upper(),
 * [\w']+ tokens, tokens of <= 2 characters and all-digit tokens dropped, every 3 consecutive tokens joined, [" "] for a text
 * without tokens) + make_unique_endings (east/asts/utils.py:25-40) for raw UTF-8 texts of ASCII and Cyrillic (U+0400-045F)
 * characters.  utf8: the texts concatenated, text_off: n_texts + 1 byte offsets.  A text with any other character (or
 * invalid UTF-8) makes the call fail with EAST_ERR_UNSUPPORTED: the caller then uses the host preprocessing (Python's
 * full Unicode tables), which stays the reference behaviour.
 * east_texts_to_packed_host returns the packed documents (uint32 code points, what east_build_host takes), their
 * offsets (n_texts + 1) and string counts; EAST_ERR_RANGE when packed_cap is too small (doc_off_out is valid then).
 * east_table_texts_host = that + east_table_dev + the table back on the host: raw text in, scores out, one call. */
int east_texts_to_packed_host(const uint8_t *utf8, const int64_t *text_off, int32_t n_texts, int device,
                              uint32_t *packed_out, int64_t packed_cap, int64_t *doc_off_out, int32_t *doc_m_out);
int east_table_texts_host(const uint8_t *utf8, const int64_t *text_off, int32_t n_texts, int device,
                          const uint32_t *kp, const int64_t *kp_off, int32_t K, int normalized, double *out_DxK,
                          int64_t *doc_off_out /* optional */, int32_t *doc_m_out /* optional */, east_index **out_idx);

/* ---- synonym-expanded tables in one call: build and score as the table entries above, with the queries of
 * east_score_groups_* -- V variants in kp/kp_off (NOT space-stripped), grouped by group_off[G+1] (host, int64,
 * group_off[0] = 0, strictly increasing, group_off[G] = V) -- and a table G wide: out[d * G + g] = max over the
 * variants of group g of the normalized score of document d (always normalized, as the reference's synonym branch).
 * The tables are bit-identical to the entry's build followed by east_score_groups_host on the index.  On a batch of
 * small documents the per-document kernel keeps the best variant of every group itself (up to 12 288 groups), so the
 * synonym table inherits the pipelined host build, the one-byte text and the fused all-gather of the plain entries;
 * otherwise the batched scorer combines the groups after the build.  Groups and variants are checked before anything
 * is built: malformed groups fail with EAST_ERR_INVALID, an empty variant with EAST_ERR_ZERODIV; a text outside
 * ASCII / Cyrillic fails the _texts_ entry with EAST_ERR_UNSUPPORTED, as in east_table_texts_host.
 *   east_table_groups_host: host text (text_width 4: uint32 code points as east_table_host, 1: one byte per code point
 *     as east_table_host_u8), out_DxG on the host.
 *   east_table_groups_dev: as east_table_dev_gather (n_peers = 0: no gather; peer_rows then may be NULL).
 *   east_table_texts_groups_host: raw UTF-8 texts, as east_table_texts_host. */
int east_table_groups_host(const void *text, int32_t text_width, const int64_t *doc_off, const int32_t *doc_m,
                           int32_t n_docs, int device, const uint32_t *kp, const int64_t *kp_off, int32_t V,
                           const int64_t *group_off, int32_t G, double *out_DxG, east_index **out_idx);
int east_table_groups_dev(const uint32_t *text_dev, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs,
                          int device, const uint32_t *kp_dev, const uint32_t *kp_host, const int64_t *kp_off, int32_t V,
                          const int64_t *group_off, int32_t G, double *out_DxG_dev, double *const *peer_rows,
                          int32_t n_peers, void *stream, east_index **out_idx);
int east_table_texts_groups_host(const uint8_t *utf8, const int64_t *text_off, int32_t n_texts, int device,
                                 const uint32_t *kp, const int64_t *kp_off, int32_t V, const int64_t *group_off,
                                 int32_t G, double *out_DxG, int64_t *doc_off_out /* optional */,
                                 int32_t *doc_m_out /* optional */, east_index **out_idx);

/* ---- keyphrase graphs in one call: build and score as the table entries above, but return the co-occurrence counts
 * C[i][j] = number of documents in which both column i and column j score >= threshold (applications.py:111-147:
 * C[k][k] is the support of k), int32, cols x cols row-major, where cols = G with group_off and V without it (group_off
 * may be NULL: then kp holds V plain keyphrases, space-stripped as for east_table_host, scored with `normalized`; with
 * group_off the variants of east_table_groups_* are scored, always normalized).  The documents x columns score table is
 * never formed: the per-document kernel stores one relevance byte per (column, document) -- score >= threshold, the fp64
 * compare of east_cooc_* -- into the keyphrase-major byte matrix the tensor-core product C = B B^T reads; the paths that
 * score after the build (batched or tiled scorer, failed speculation, global sort) score bounded tiles of documents and
 * threshold each tile.  C equals east_cooc_host(table, threshold) of the matching table entry's table element for element.
 * Arguments, keyphrases and groups are checked before anything is built (EAST_ERR_INVALID, EAST_ERR_ZERODIV for an empty
 * keyphrase or variant); the _texts_ entry fails with EAST_ERR_UNSUPPORTED as east_table_texts_host does.  Every entry
 * optionally returns the index (out_idx may be NULL).
 *   east_graph_host: host text (text_width 4: uint32 code points, 1: one byte per code point), C_host on the host.
 *   east_graph_dev: device-resident text and keyphrases (kp_host: optional host copy), C_dev on the device, queued on
 *     `stream` (the call returns once C_dev is written).
 *   east_graph_texts_host: raw UTF-8 texts, as east_table_texts_host. */
int east_graph_host(const void *text, int32_t text_width, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs,
                    int device, const uint32_t *kp, const int64_t *kp_off, int32_t V, const int64_t *group_off, int32_t G,
                    int normalized, double threshold, int32_t *C_host, east_index **out_idx);
int east_graph_dev(const uint32_t *text_dev, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs, int device,
                   const uint32_t *kp_dev, const uint32_t *kp_host, const int64_t *kp_off, int32_t V, const int64_t *group_off,
                   int32_t G, int normalized, double threshold, int32_t *C_dev, void *stream, east_index **out_idx);
int east_graph_texts_host(const uint8_t *utf8, const int64_t *text_off, int32_t n_texts, int device, const uint32_t *kp,
                          const int64_t *kp_off, int32_t V, const int64_t *group_off, int32_t G, int normalized,
                          double threshold, int32_t *C_host, int64_t *doc_off_out /* optional */,
                          int32_t *doc_m_out /* optional */, east_index **out_idx);

/* ---- persistence: the reference rebuilds every structure on every run (relevance.py:38-47); an index -- packed text,
 * suffix array, LCP, child table, annotation and the scorer's side tables of one batch of documents -- can be written
 * to a file and loaded back onto any device.  Scores and arrays of a loaded index are identical to the saved one's. */
int east_index_save(const east_index *idx, const char *path);
int east_index_load(const char *path, int device, east_index **out);

/* The library allocates from two private stream-ordered memory pools per device (the device's default pool is not
 * touched) and keeps freed blocks for the next call, up to a quarter of the device memory.  east_trim waits for the
 * device and returns everything that is not in use to the driver (also drops the calling thread's cached keyphrase
 * preparation and alphabet guess). */
int east_trim(int device);
/* Process-wide switches and tuning knobs (0 = default), mostly for A/B measurements and tests.  The ones that change what a
 * call does rather than how fast:
 *   "no_alphabet_guess" = 1   batches of small documents always scan for their alphabet.  Default: a batch starts from the
 *                             alphabet of the calling thread's previous batch on the device -- a guess the per-document
 *                             kernel checks against every code point; a miss redoes the batch from a scan (index stats
 *                             "alphabet_guessed", "alphabet_miss", "pipeline_miss").  Results never depend on it.
 *   "forget_alphabet_guess" = 1  (an action, per thread) the calling thread's next batch scans.
 *   "alphabet_sample"   = n   device-resident batches take their alphabet from the first n code points (default 2 M;
 *                             -1: the whole text); checked and redone the same way.
 *   "kp_prep_host"      = 1   keyphrase preparation on the host (round 1; cross-check of the device variants);
 *   "kp_small_max"      = n   largest number of query suffixes the one-kernel preparation takes (default and limit 65 536).
 *   "drop_kp_cache"     = 1   forget the keyphrase preparation kept for score calls on an existing index.
 * Others ("key_chars", "rs_variant", "cooc_variant", "time_kernels", ...) are described where they are read (csrc/capi.cu). */
int east_set_option(const char *name, int64_t value);

#ifdef __cplusplus
}
#endif
#endif /* EAST_B200_H */
