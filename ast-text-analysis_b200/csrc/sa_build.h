// sa_build.h -- internal interfaces between the build stages of libeast_b200.
#pragma once
#include "common.cuh"

namespace east {

struct SufRec;
// Keyphrases to score INSIDE the per-document kernel: once a CTA has indexed its document it walks every distinct
// query suffix (score_walk.cuh) while suffix array, key words and bucket rows are still hot in L2, and stores the
// per-suffix results to tmp[(document - doc_begin) * n_uniq + position], then adds them up per keyphrase.
struct DocScore {
    const SufRec *recs = nullptr;     // distinct query suffixes in visiting order
    int32_t n_uniq = 0;
    const uint8_t *q8 = nullptr;      // dense byte codes of the concatenated keyphrases
    const uint32_t *kp = nullptr;     // their code points (walks of suffixes with code points >= 0x0A00)
    double *tmp = nullptr;
    int normalized = 0;
    // the keyphrase sums (k_score_combine's arithmetic) are taken by the same CTA: out[(document - doc_begin) * K + k]
    const int32_t *kp_off = nullptr;  // K + 1
    const int32_t *uniq_of = nullptr; // per suffix of the concatenated keyphrases: position of its distinct twin
    int32_t K = 0;
    double *out = nullptr;
    // synonym-expanded table (k_doc_suffix_sort_groups): the K queries are variants grouped by group_off[G + 1] (device);
    // the row is G wide, out[(document - doc_begin) * G + g] = the best variant of group g (k_score_combine_max's
    // arithmetic).  The groups' running maxima live in the CTA's shared memory: at most MAX_GROUPS groups.
    const int32_t *group_off = nullptr;
    int32_t G = 0;
    static constexpr int32_t MAX_GROUPS = 12288;
    // the all-gather of a documents-sharded table, fused: every row is also stored into the gathered tables of the other
    // ranks (their memory mapped into this process: NVLink peer stores), at the same row offset as `out`
    static constexpr int MAX_PEERS = 15;
    double *peer_out[MAX_PEERS] = {};
    int32_t n_peers = 0;
    double algorithmic_bytes = 0.0;   // of the walks of this launch (measurement only: added to the kernel's byte count)
    // the per-rank key words (sk) only serve LATER score calls on the index (the in-kernel walks read the staged text): a
    // launch that scores its documents itself may leave them to the first such call (ensure_suffix_keys in capi.cu)
    int skip_suffix_keys = 0;
    // keyphrase graph (k_doc_suffix_sort_graph, k_doc_suffix_sort_groups_graph): instead of its row the CTA stores the
    // relevance bytes graph[k * graph_pitch + graph_col0 + (document - doc_begin)] = (score >= threshold), k < K (G with
    // groups): the keyphrase-major matrix C = B B^T reads (cooc_tc.cu).  No peers in this mode.
    uint8_t *graph = nullptr;
    int64_t graph_pitch = 0, graph_col0 = 0;
    double threshold = 0.0;
};

// What a caller-supplied hook sees once the per-document kernel of one run of
// documents has been queued on `stream` -- everything the scorer needs for these documents is ordered
// before whatever the hook queues on the same stream (east_table_host scores the run there).
struct RunReady {
    int32_t doc_begin, doc_count;
    cudaStream_t stream;
    const uint8_t *t8;
    const uint32_t *bkt, *bkt3;   // whole-batch tables (row of document 0 first); bkt3 may be NULL
    int sym_bits;
    const std::vector<uint8_t> *code_table;
    int speculative;              // 1 = pipelined host build: the run stands only if the build ends with pipelined = 1
};

struct SaInput {
    const uint32_t *text;     // device, n code points (packed documents, concatenated)
    // pipelined host build of east_*_host_u8: the text arrives as one byte per code point (0xFF = end of a string);
    // `text` is then an OUTPUT of the per-document kernel (the code points with their terminators 0x0A00 + k)
    const uint8_t *text8 = nullptr;
    const int32_t *doc_off;   // device, n_docs + 1
    const int32_t *doc_m;     // device, n_docs
    int32_t n;
    int32_t n_docs;
    int64_t m_total;
    int key_chars;            // 0 = as many symbols as fit the 64-bit key
    int force_general;        // testing: never take the terminator-class fast path
    int rs_variant = 0;       // tuning: radix-sort kernel shape (see radix_sort_pairs)
    const int32_t *doc_off_host = nullptr;  // host copy of doc_off
    int segmented_sort = 1;                 // round 0: per-document tiles / histograms when documents are large
    int local_group_sort = 1;               // doubling rounds: rank inside small groups instead of radix passes
    int64_t sort_batch_elems = 0;           // round-0 sort batch in suffixes (0 = whole batch at once)
    int doc_sort = 1;                       // small documents: one CTA sorts a whole document in shared memory
    // destination of the LCP / child / annotation tables: the per-document kernel fills them itself
    int32_t *lcp = nullptr, *up = nullptr, *down = nullptr, *next = nullptr, *ann = nullptr;
    uint32_t *sk = nullptr;                 // destination of the scorer's per-rank key bytes (fast path only)
    int light_scan = 1;                     // small documents: alphabet-only scan first (the per-document kernel validates)
    int64_t alphabet_sample = 0;            // ... over this many leading code points only (speculation, checked by the kernel); 0 = all
    int alphabet_guess = 0;                 // batches of small documents may start from the alphabet of this thread's previous batch
                                            // (the same speculation without the scan and its host round trip; checked by the kernel)
    int want_bkt3 = 1;                      // per-document kernel: also keep its 3-gram bucket starts for the scorer
    int fused_encode = 1;                   // per-document kernel: byte-code the text itself (no separate k_encode_text pass)
    // pipelined host build: the text arrives in n_chunks runs of whole documents; chunk c = documents
    // [chunk_doc[c], chunk_doc[c+1]) is resident once chunk_ready[c] has fired (recorded on the copy stream)
    int n_chunks = 0;
    const int32_t *chunk_doc = nullptr;
    const cudaEvent_t *chunk_ready = nullptr;
    cudaStream_t helper_stream = nullptr;   // odd runs are sorted here, so that consecutive one-wave kernels overlap their tails
    cudaStream_t prep_stream = nullptr;     // pipelined build: the runs are byte-coded here (high priority) as soon as they arrive
    // Hooks around every launch of the per-document kernel (each run of the pipelined build; the whole batch
    // otherwise), only when the 2-gram table and the key words exist.  run_begin may fill `score` to have the
    // kernel score the documents; run_hook is called after the launch (in the ordinary build: after the launch
    // is known to have succeeded) with in_kernel = whether that happened.
    void (*run_begin)(void *ctx, const RunReady &run, DocScore &score) = nullptr;
    void (*run_hook)(void *ctx, const RunReady &run, int in_kernel) = nullptr;
    void *run_ctx = nullptr;
    // called once the text scan has been queued, before the host waits for its result: host work (launches on other
    // streams) that does not depend on the alphabet hides under the scan's round trip
    void (*scan_queued)(void *ctx) = nullptr;
    Arena *arena = nullptr;   // where the arrays that stay with the index (byte text, bucket tables) are taken from
};

struct SaOutput {
    int32_t *sa;              // device, n  (global text positions, doc-major rank order)
    DevBuf<uint8_t> t8;       // fast path: dense byte codes of the text (kept for later stages)
    DevBuf<uint32_t> bkt;     // fast path: 2-gram bucket table [n_docs << 2*sym_bits] + sentinel
    DevBuf<uint32_t> bkt3;    // per-document kernel with 5-bit symbols: 3-gram table [n_docs << 3*sym_bits] + sentinel
    std::vector<uint8_t> code_table;  // code point (< 0x0A00) -> dense code (0 = absent)
    int sym_bits = 0;
    int term_code = 0;
    int fast_path = 0;
    int sigma = 0;
    int key_chars = 0;
    int key_bits = 0;
    int rounds = 0;
    uint32_t active_after_round0 = 0;
    int segmented = 0;               // round 0 used the per-document sort
    int radix_fallback_rounds = 0;   // doubling rounds that met a group > GS_MAX and used the radix sort
    int doc_sorted = 0;              // the per-document shared-memory sort produced the suffix array
    int doc_sort_overflow = 0;       // it met a bucket it cannot sort and the global sort took over
    int tables_done = 0;             // LCP / child / annotation tables were produced by the per-document kernel
    int sk_done = 0;                 // the scorer's per-rank key bytes were produced
    int sk_skipped = 0;              // ... except by launches that scored their documents themselves (made on first use)
    int pipelined = 0;               // the build overlapped the host-to-device copy (speculative alphabet held)
    int pipeline_miss = 0;           // it did not hold (later chunks brought new symbols / bad layout): redone
    int alphabet_guessed = 0;        // the build started from the alphabet of the thread's previous batch (and it held, or see the misses)
    int alphabet_miss = 0;           // the alphabet sampled from a prefix of a device-resident text did not hold: redone
};

void build_suffix_array(const SaInput &in, SaOutput &out, StageTimer &tm, cudaStream_t s);
// one byte per code point (0xFF = end of a string) -> packed code points with terminators 0x0A00 + k; *bad |= 1 when a
// document does not hold exactly doc_m terminators or does not end with one
void expand_text8(const uint8_t *text8, const int32_t *doc_off, const int32_t *doc_m, int n_docs, uint32_t *text, uint32_t *bad,
                  cudaStream_t s);

// per-document shared-memory suffix sort (doc_sort.cu)
struct DocSortPlan {
    int b = 0, G = 0, S2 = 0;   // bits per symbol, symbols per bucket id, symbols per refinement level
    int text_cap = 0, bits_words = 0;
    size_t smem = 0;
    int tables_fit = 0;         // the fused LCP / child / annotation phases fit the shared memory too
};
struct DocSortTables { int32_t *lcp, *up, *down, *next, *ann; };   // every entry of the launched documents is written
bool doc_sort_plan(int sigma, int32_t max_doc_n, DocSortPlan &plan);
void doc_sort_launch(const DocSortPlan &plan, const uint8_t *t8, const uint32_t *text, const int32_t *doc_off,
                     const int32_t *doc_m, int doc_begin, int n_docs,
                     int64_t n_total /* code points of these documents */, uint32_t term, int32_t *sa, uint32_t *bkt, uint32_t *bkt3, uint32_t *overflow, cudaStream_t s,
                     unsigned long long *phase_clk = nullptr /* profiling: 8 cycle counters */,
                     const DocSortTables *tables = nullptr /* also produce LCP, child table, annotation */,
                     uint32_t *sk = nullptr /* also produce the scorer's per-rank key bytes */,
                     const DocScore *score = nullptr /* also score keyphrases (needs bkt and sk) */,
                     const uint8_t *code_table = nullptr /* byte-code the text in the kernel (writes t8, sets *miss) */,
                     uint32_t *miss = nullptr, int64_t text_len = 0 /* code points of the whole batch */,
                     const uint8_t *text8 = nullptr /* with code_table: one byte per code point in, code points out to `text` */);

// device preprocessing of raw UTF-8 texts (tokenize.cu): sizes[3 d] = code points of the packed document d, [3 d + 1] = its
// strings, [3 d + 2] != 0 = the text has characters the device does not handle; then the packed documents themselves
void tokenize_texts(const uint8_t *raw_dev, const int64_t *raw_off_dev, int32_t n_texts, int32_t *sizes_dev, cudaStream_t s);
void tokenize_emit(const uint8_t *raw_dev, const int64_t *raw_off_dev, int32_t n_texts, const int64_t *doc_off_dev, uint32_t *text_dev,
                   cudaStream_t s);

// Kasai-equivalent LCP (easa.py:247-266), child table (easa.py:268-304) and annotation
// (easa.py:306-331) of the whole batch
void build_lcp_tables(const uint32_t *text, const uint8_t *t8 /*or null*/, int term_code, const int32_t *sa, const int32_t *doc_off, const int32_t *doc_m,
                      int n_docs, int32_t n, int32_t *lcp, int32_t *up, int32_t *down, int32_t *next,
                      int32_t *ann, StageTimer &tm, cudaStream_t s, int child_variant = 0);

// batched scorer (easa.py:91-139)
// one record per DISTINCT query suffix, in visiting order (thread order): everything a walk needs to start
bool alphabet_guess_code_table(uint8_t *table /* EAST_TERM_BASE entries */);   // sa_build.cu: see AlphabetGuess
void alphabet_guess_forget();                                                  // the calling thread's guess

struct SufRec {
    uint64_t q8_first;   // dense codes of the first 8 symbols (fast path; symbol d in byte d)
    int32_t sidx;        // index of (one of) the suffix(es) in the concatenated keyphrases
    uint16_t len;        // symbols to the end of its keyphrase
    uint8_t generic;     // 1 = contains a code point >= 0x0A00 (or no fast path): generic walk on code points
    uint8_t pad;
};
struct ScoreInput {
    const uint32_t *text;
    const int32_t *sa;
    const int32_t *doc_off;
    const int32_t *doc_m;
    int n_docs;
    const uint32_t *kp;        // device, concatenated queries
    const int32_t *kp_off;     // device, K + 1
    int32_t K;
    int32_t total_suffixes;
    int normalized;
    // fast path (terminator-class alphabet): dense byte text, byte-coded queries, 2-gram buckets
    const uint8_t *t8 = nullptr;
    const uint32_t *bkt = nullptr;      // [n_docs << 2*sym_bits] + 1, rows of the docs being scored
    const uint32_t *bkt3 = nullptr;     // optional [n_docs << 3*sym_bits] + 1: depth 2 is a table lookup too
    const uint32_t *sk = nullptr;       // per rank: text bytes at offsets 2..5 of the suffix (saves the SA -> text hop)
    const uint8_t *q8 = nullptr;        // dense codes of kp (0 = symbol absent from the batch)
    // identical query suffixes (same code points to the end of their keyphrase) are walked once:
    const int32_t *uniq_of = nullptr;   // device, total_suffixes: position (in visiting order) of the suffix's distinct twin
    const SufRec *recs = nullptr;       // device, n_uniq: the distinct suffixes in visiting order
    int32_t n_uniq = 0;
    int sym_bits = 0;
    unsigned long long *probe_count = nullptr;  // device counter: run the probe-counting variant
    double algorithmic_bytes = 0.0;             // 8 B x probes of this workload, if known (roofline numerator)
    // sharded table: k_score_combine also stores every cell into the gathered tables of the other ranks (mapped peer
    // memory, same offset as out_DxK): the all-gather of the batched scorer path (k_score_combine, k_score_combine_max)
    double *peer_out[DocScore::MAX_PEERS] = {};
    int32_t n_peers = 0;
    // synonym-expanded scoring: the K queries are variants, grouped by group_off[G + 1] (device); the combine step then
    // stores out[doc][g] = the best variant of group g (k_score_combine_max).  nullptr: one column per query.
    const int32_t *group_off = nullptr;
    int32_t G = 0;
};
// the second half of score_table alone: tmp[doc][distinct suffix] (here: written by the per-document kernel) -> out[doc][k]
// (out[doc][g] with groups)
void score_combine(const ScoreInput &in, const double *suffix_tmp, double *out_DxK, cudaStream_t s);
void score_table(const ScoreInput &in, double *suffix_tmp /*n_docs x n_uniq*/, double *out_DxK,
                 cudaStream_t s);
// the first half alone: the walks of every (document, distinct suffix) -> suffix_tmp
void score_suffixes(const ScoreInput &in, double *suffix_tmp, cudaStream_t s);

// sk[r] = the 4 byte codes at offsets 2..5 of suffix sa[r] (for indexes built by the global sort)
void fill_suffix_keys(const uint8_t *t8, const int32_t *sa, int32_t n, uint32_t *sk, cudaStream_t s);

void cooc_counts(const double *S_DxK, int64_t D, int32_t K, double threshold, int32_t *C, cudaStream_t s);     // AND + POPC
// tcgen05 co-occurrence counts = threshold_bytes into a zeroed Kp x Dp byte matrix (cooc_padding) + cooc_counts_bytes
void cooc_counts_tc(const double *S_DxK, int64_t D, int32_t K, double threshold, int32_t *C, cudaStream_t s,
                    int simple = 0 /* 0: TMA-fed cluster kernel, 1: the non-pipelined 128 x 128 kernel, 2: the cp.async pipeline */);
// the relevance bytes of D documents x K keyphrases: Bm[Kp][Dp], Dp = D rounded up to 128, Kp = K rounded up to 256
void cooc_padding(int64_t D, int32_t K, int64_t *Dp, int32_t *Kp);
// Bm[k][col0 + d] = (S[d][k] >= threshold) for d < D, k < K (S: D x K doc-major); nothing else of Bm is written
void threshold_bytes(const double *S_DxK, int64_t D, int32_t K, double threshold, uint8_t *Bm, int64_t Dp, int64_t col0,
                     cudaStream_t s);
// C = Bm Bm^T (K x K int32) from a prepared, zero-padded Kp x Dp matrix
void cooc_counts_bytes(const uint8_t *Bm, int64_t Dp, int32_t Kp, int32_t K, int32_t *C, cudaStream_t s, int simple = 0);

}  // namespace east
