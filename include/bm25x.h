/*
 * bm25x.h — C ABI of the B200-native BM25 top-k engine (libbm25x.so).
 *
 * This is the drop-in boundary for ONE path of tensorchord/VectorChord-bm25: the
 * ranked top-k query `bm25::search` (and, next, `bm25::evaluate`).  Each entry
 * point cites the reference interface it replaces (paths relative to the
 * reference tree).  Plain pointers and sizes only: no C++/torch types, no
 * exceptions or unwinding across the boundary (the reference denies
 * ffi_unwind_calls, src/lib.rs:16): every call returns an int status and
 * bm25x_last_error() holds a thread-local message.
 *
 * There is NO CPU fallback: every search entry point fails with
 * BM25X_ERR_CUDA when no sm_100 device / kernel image is available.
 */
#ifndef BM25X_H
#define BM25X_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BM25X_OK 0
#define BM25X_ERR_INVALID 1     /* bad argument / corrupt corpus ("data corruption" panics in the reference) */
#define BM25X_ERR_CUDA 2        /* CUDA runtime / launch failure, or no usable device */
#define BM25X_ERR_OOM 3
#define BM25X_ERR_UNSUPPORTED 4 /* k > BM25X_MAX_K, > BM25X_MAX_QUERY_TERMS live terms, tf >= 2^24 */
#define BM25X_ERR_LIMIT_ZERO 5  /* k == 0: "number of needed rows is set to 0" (scanners/default.rs:114-116) */

#define BM25X_MAX_K 65535 /* the reference's bm25.limit maximum (src/index/gucs.rs:37-46) */
#define BM25X_MAX_QUERY_TERMS 64 /* live (known, distinct) tokens per query; more than 32 run as two passes over term groups */
#define BM25X_TERM_MISSING 0xFFFFFFFFu
#define BM25X_KEY_WIDTH 16 /* crates/bm25/src/lib.rs:37 WIDTH */

typedef struct bm25x_index bm25x_index;
typedef struct bm25x_batch bm25x_batch;

/* The sealed segment as the reference hands it to flush():
 * `Segment{records: Record(len, payload), mappings: Mapping(key, doc, tf)}` sorted by (key, doc)
 * (crates/bm25/src/segment.rs:19-45, flush.rs:40-67).  Term-major CSR on the host. */
typedef struct {
    uint32_t n_docs;          /* number_of_documents; doc id = record order (io.rs:52-60) */
    const uint32_t *doc_len;  /* [n_docs] exact document length = Σ tf (vector.rs:77-83) */
    const uint16_t *payload;  /* [n_docs*3] heap ctid of each record, or NULL (payload = doc id split) */
    uint32_t n_terms;         /* distinct tokens */
    const uint8_t *term_key;  /* [n_terms*16] interned keys, strictly ascending (vector.rs:19-35), or NULL when
                                 callers address terms by dense ordinal (the bm25vector u32-token-id surface) */
    const uint64_t *post_off; /* [n_terms+1] */
    const uint32_t *post_doc; /* [P] doc ids, strictly ascending inside a term */
    const uint32_t *post_tf;  /* [P] term frequencies, != 0 */
    double k1, b;             /* Bm25IndexOptions (crates/bm25/src/types.rs:18-45): defaults 1.2 / 0.75 */
} bm25x_corpus;

typedef struct {
    uint32_t n_docs, n_terms;
    uint64_t n_postings;
    uint64_t sum_doc_len;  /* JumpTuple.sum_of_document_lengths (tuples.rs:141-160) */
    double avgdl, k1, b;
    uint64_t device_bytes; /* HBM held by the index */
    uint64_t n_blocks;     /* 128-posting blocks (flush.rs:78-125) */
    int device;
} bm25x_index_info;

typedef struct {
    double kernel_ms;        /* device time of the search kernels, CUDA events on the launch stream */
    double h2d_ms, d2h_ms;   /* bm25x_search_batch only (host clock): canonicalise + upload, download of the results */
    uint64_t postings;       /* Σ df over live query terms (algorithmic postings touched, exhaustive) */
    uint64_t bytes_algo;     /* 8 B/posting + 8 B/result slot + 16 B/query term (SURVEY §8d) */
    uint32_t launches;       /* kernels launched */
    uint32_t queries;        /* live queries (>= 1 known term) */
    uint64_t postings_fetched; /* postings actually streamed into shared memory (< postings when pruning bites) */
} bm25x_search_stats;

/* ---- index lifetime: replaces bm25::build → flush (crates/bm25/src/build.rs:22-71, flush.rs:40-158) for the
 * read path: lays the postings out in HBM and precomputes per-term s0 and per-fieldnorm s1 (bm25.rs:334-354). */
int bm25x_index_create(const bm25x_corpus *corpus, int device, bm25x_index **out);
void bm25x_index_destroy(bm25x_index *idx);
int bm25x_index_get_info(const bm25x_index *idx, bm25x_index_info *out);

/* ---- the sealed segment AS STORED by the reference (SURVEY §8 f1: ingest of the on-page format).  While walking the
 * index pages the caller flattens, per token, the chain of SummaryTuples (crates/bm25/src/tuples.rs:900-910) and the
 * BlockTuples they point to (tuples.rs:973-983) that flush() wrote (flush.rs:78-120); the block payloads are taken
 * exactly as compression.rs:36-136 left them (4-lane vertical bit packing with delta-coded doc ids for full blocks,
 * byte packing for a token's last block) and are decoded on the GPU — replacing fill_block (search.rs:498-518) +
 * crates/simd/src/bitpacking*.rs / bytepacking*.rs on the CPU.  Searches on the resulting index are identical to those
 * on an index created from the same postings with bm25x_index_create. */
typedef struct {
    uint32_t n_docs;
    const uint32_t *doc_len;       /* [n_docs] exact lengths, or NULL: then the two fields below (what the pages hold) */
    const uint8_t *doc_fieldnorm;  /* [n_docs] DocumentTuple.fieldnorm (tuples.rs:756-762); used when doc_len == NULL */
    uint64_t sum_doc_len;          /* JumpTuple.sum_of_document_lengths (tuples.rs:141-160); used when doc_len == NULL */
    const uint16_t *payload;       /* [n_docs*3] DocumentTuple.payload (ctid), or NULL */
    uint32_t n_terms;
    const uint8_t *term_key;       /* [n_terms*16] TokenTuple.id, strictly ascending, or NULL */
    const uint64_t *term_blk_off;  /* [n_terms+1] first block of each token; term_blk_off[n_terms] == n_blocks */
    uint64_t n_blocks;
    const uint32_t *blk_min_doc;   /* [n_blocks] SummaryTuple.min_document_id: the delta seed of the block */
    const uint32_t *blk_n;         /* [n_blocks] SummaryTuple.number_of_documents: 128 except a token's last block */
    const uint8_t *blk_meta_doc;   /* [n_blocks] BlockTuple.metadata_document_ids: flag << 7 | width */
    const uint8_t *blk_meta_tf;    /* [n_blocks] BlockTuple.metadata_term_frequencies */
    const uint64_t *blk_doc_off;   /* [n_blocks] byte offset of compressed_document_ids inside `bytes` */
    const uint64_t *blk_tf_off;    /* [n_blocks] byte offset of compressed_term_frequencies inside `bytes` */
    const uint8_t *bytes;          /* concatenated block payloads */
    uint64_t n_bytes;
    double k1, b;
    /* SummaryTuple.wand_fieldnorm / wand_term_frequency (tuples.rs:900-910; written by flush.rs:101-120): the arg-max
     * posting of each block, whose score is the block's upper bound (search.rs:381,426-429).  Optional (both or
     * neither): when given they are checked against the decoded postings ("corrupt blocks" on mismatch); the bounds
     * the kernels use are always computed from the decoded postings themselves. */
    const uint8_t *blk_wand_fieldnorm; /* [n_blocks] or NULL */
    const uint32_t *blk_wand_tf;       /* [n_blocks] or NULL */
} bm25x_blocks;
int bm25x_index_create_from_blocks(const bm25x_blocks *blocks, int device, bm25x_index **out);

/* ---- replication across the GPUs of one box (queries shard, the index is replicated; NCCL broadcast at load
 * only).  The library stays NCCL-free: it exposes the device arrays, the caller moves the bytes (bench.py uses
 * torch.distributed.broadcast over NVLink).  Sender: bm25x_index_get_layout.  Receiver: bm25x_index_alloc_replica
 * with the sender's layout (scalars only are read), fill the arrays named by its own layout, then
 * bm25x_index_finalize_replica. */
#define BM25X_N_ARRAYS 13
typedef struct {
    uint32_t n_docs, n_terms;
    uint64_t n_postings, n_postings_padded, n_blocks, sum_doc_len;
    double k1, b, avgdl;
    void *dev_ptr[BM25X_N_ARRAYS];     /* device addresses of the index arrays (valid on `device` only) */
    uint64_t bytes[BM25X_N_ARRAYS];
    int device;
} bm25x_index_layout;
int bm25x_index_get_layout(const bm25x_index *idx, bm25x_index_layout *out);
int bm25x_index_alloc_replica(const bm25x_index_layout *like, int device, bm25x_index **out);
int bm25x_index_finalize_replica(bm25x_index *idx);
/* Options.  "prune" (default 1): MaxScore-style pruning in the warp-per-query kernel — terms whose summed score upper
 * bounds (the token-level WAND bound of the reference: TokenTuple.wand_fieldnorm/wand_term_frequency,
 * flush.rs:101-120, search.rs:363) stay below 5 % of the current k-th score are no longer streamed; their postings
 * are looked up in HBM only for the candidates.  Results are identical with it on or off.
 * "seed" (default 1): queries of 2..8 terms with limit <= 128 and no prefilter bitmap run through the SEEDED kernel —
 * the documents that hold a single query term come from per-term champion lists (the term's best 128 postings in
 * result order, built with the index), so the stream reads doc ids only (half the bytes) and never tests a posting on
 * its own; "seed_max_terms" (4 | 8), "seed_dense_div" (default 64: queries with a list of >= n_docs / 64 postings go
 * back to the plain kernel; 0: never), "seed_prune_min" (default 32768: so do queries with a list this long and 8x
 * their shortest one — pruning pays).  "twophase" (default 0): queries of 2..4 terms with limit <= 224 that the seeded
 * kernel does not take run as two launches — 8-byte postings while single postings can still enter the top-k, then
 * doc ids only.  "slice_min" (default 32768): bm25x_search_batch pipelines batches of >= 2 x this many queries as slices
 * (upload / kernels / download overlap; 0: one piece).  None of these changes a result bit. */
int bm25x_index_set_option(bm25x_index *idx, const char *name, int64_t value);
/* df of every term (TokenTuple.number_of_documents), host copy. */
int bm25x_index_get_df(const bm25x_index *idx, uint32_t *df_out);

/* address_tokens::read (crates/bm25/src/address_tokens.rs:61-98): key → dense term ordinal,
 * BM25X_TERM_MISSING when absent (search.rs:60-62 then skips it).  Needs term_key at create time. */
int bm25x_lookup_terms(const bm25x_index *idx, const uint8_t *keys, uint32_t n, uint32_t *ordinals_out);

/* vector::intern (crates/bm25/src/vector.rs:19-35): the 16-byte key of a token under the index's 32-byte seed.  Tokens
 * shorter than 16 bytes without a NUL byte are their own zero-padded key; all others are the first 16 bytes of
 * blake3::keyed_hash(seed, token) with a zero last byte replaced by 1.  Host-only (no device involved). */
int bm25x_intern(const uint8_t seed[32], const uint8_t *token, size_t len, uint8_t key_out[BM25X_KEY_WIDTH]);
/* Test hook: first 16 bytes of BLAKE3 keyed_hash(key, data) without the interning rules (known-answer tests). */
int bm25x_blake3_keyed16(const uint8_t key[32], const uint8_t *data, size_t len, uint8_t out[16]);

/* ---- bm25::search (crates/bm25/src/search.rs:28-282) for a whole batch of queries, called where
 * DefaultBuilder::build calls it (src/index/bm25/scanners/default.rs:117-129).
 *   q_off[nq+1], q_terms[]: query i = term ordinals q_terms[q_off[i]..q_off[i+1]) — any order, duplicates and
 *     BM25X_TERM_MISSING / df==0 terms allowed (they are dropped exactly as search.rs:55-62 drops them).
 *   k: `limit` (NonZero<usize>, 1..=BM25X_MAX_K).
 *   allow: optional prefilter bitmap [ceil(n_docs/8)], bit d set ⇒ filter(payload(d)) is true
 *     (search.rs:230; the per-candidate callback of the reference cannot cross a batch ABI); NULL ⇒ all pass.
 *   outputs, row i at offset i*k, best first (score desc, then doc id asc — the canonical tie rule):
 *     out_doc u32, out_score f32 (positive; the SQL binding negates, operators.rs:54),
 *     out_score64 f64 or NULL (bit-identical to Cache::evaluate summed in ascending term order),
 *     out_payload u16[3] or NULL, out_n[i] = rows returned (<= k).
 * Host pointers; the call copies H2D, runs the sm_100a kernels, copies D2H. */
int bm25x_search_batch(bm25x_index *idx, uint32_t nq, const uint32_t *q_off, const uint32_t *q_terms, uint32_t k,
                       const uint8_t *allow, uint32_t *out_doc, float *out_score, double *out_score64,
                       uint16_t *out_payload, uint32_t *out_n, bm25x_search_stats *stats);

/* Split form of the same call, for pipelining and for timing the device part alone:
 * prepare = canonicalise + upload queries; run = kernels only, everything resident in HBM
 * (stream = cudaStream_t as void*, NULL = the library's stream; asynchronous unless stats != NULL);
 * fetch = D2H of the results. */
int bm25x_batch_prepare(bm25x_index *idx, uint32_t nq, const uint32_t *q_off, const uint32_t *q_terms, uint32_t k,
                        const uint8_t *allow, bm25x_batch **out);
int bm25x_batch_run(bm25x_batch *batch, void *stream, bm25x_search_stats *stats);
int bm25x_batch_fetch(bm25x_batch *batch, uint32_t *out_doc, float *out_score, double *out_score64,
                      uint16_t *out_payload, uint32_t *out_n);
/* Device addresses of the batch's result rows ([nq*k] u32 / f32 / f64 / u16[3], [nq] u32; any pointer may be NULL),
 * written by bm25x_batch_run on its stream and valid until bm25x_batch_destroy — for callers that move results
 * GPU → GPU (the NCCL gather of sharded results to one rank, vectorchord-bm25_b200/shard.py) instead of fetching. */
int bm25x_batch_device_results(bm25x_batch *batch, void **doc, void **score, void **score64, void **payload, void **n);
void bm25x_batch_destroy(bm25x_batch *batch);

/* ---- the growing segment (SURVEY §8 f3): documents inserted since the last seal.  bm25::search scans them one by one
 * before it walks the sealed postings (crates/bm25/src/search.rs:83-135): every non-deleted growing document is scored
 * over the query tokens that exist in the SEALED segment with the sealed statistics — Cache::new(sealed N, sealed df,
 * k1, b, sealed avgdl) (search.rs:49-51,66-77; `insert` does not update them) — and shares the Results heap with the
 * sealed documents.  Here the growing documents are inverted once into a second, small index handle that carries
 * the sealed statistics, so the same kernels unite their postings; a query then is two top-k searches + a merge.
 * Doc ids of the growing handle are growing ordinals (insertion order).  Re-create the handle after inserts/deletes
 * (it is as cheap as the segment is small); bm25x_index_maintain (below) folds the growing documents and the delete
 * marks into a new sealed index, after which the growing segment starts empty again. */
typedef struct {
    uint32_t n_docs;               /* growing documents, in VectorTuple-chain order */
    const uint32_t *doc_len;       /* [n_docs] exact lengths, or NULL: then doc_fieldnorm */
    const uint8_t *doc_fieldnorm;  /* [n_docs] VectorTuple fieldnorm (search.rs:96-98); used when doc_len == NULL */
    const uint16_t *payload;       /* [n_docs*3] VectorTuple.payload (ctid), or NULL */
    const uint8_t *deleted;        /* [n_docs] VectorTuple.deleted (search.rs:110): non-zero = skipped; or NULL */
    const uint64_t *elem_off;      /* [n_docs+1] */
    const uint32_t *elem_term;     /* Element.key as term ordinal of the SEALED index (bm25x_lookup_terms), strictly
                                      ascending inside a document; BM25X_TERM_MISSING = token unknown to the sealed
                                      segment: it can never match a query token (search.rs:60-62) */
    const uint32_t *elem_tf;       /* Element.value, != 0 */
} bm25x_growing_docs;
int bm25x_growing_create(const bm25x_index *sealed, const bm25x_growing_docs *docs, bm25x_index **out);
/* bm25::search over sealed + growing: bm25x_search_batch on both handles and the merge below.  `growing` may be NULL
 * (sealed only).  Doc ids >= n_docs(sealed) denote growing ordinal (id - n_docs(sealed)); on equal scores sealed
 * documents come first, then ascending id (the reference's order of equal scores is not pinned, see bm25x_search_batch).
 * allow_growing: optional prefilter bitmap over growing ordinals. */
int bm25x_search_batch_growing(bm25x_index *sealed, bm25x_index *growing, uint32_t nq, const uint32_t *q_off,
                               const uint32_t *q_terms, uint32_t k, const uint8_t *allow_sealed,
                               const uint8_t *allow_growing, uint32_t *out_doc, float *out_score, double *out_score64,
                               uint16_t *out_payload, uint32_t *out_n, bm25x_search_stats *stats);
/* Host-only: row-wise merge of two top-k result sets (score desc; equal scores: list a first, then ascending id);
 * ids of list b are shifted by doc_base_b.  f64 scores of both lists are required; f32 scores / payloads optional. */
int bm25x_merge_topk(uint32_t nq, uint32_t k, const uint32_t *doc_a, const float *score_a, const double *score64_a,
                     const uint16_t *payload_a, const uint32_t *n_a, const uint32_t *doc_b, const float *score_b,
                     const double *score64_b, const uint16_t *payload_b, const uint32_t *n_b, uint32_t doc_base_b,
                     uint32_t *out_doc, float *out_score, double *out_score64, uint16_t *out_payload, uint32_t *out_n);

/* ---- the write side: bm25::maintain (crates/bm25/src/maintain.rs:27-311) and bm25::bulkdelete (bulkdelete.rs:20-112),
 * called where amvacuumcleanup / ambulkdelete call them.  maintain rewrites every posting on the device: the sealed
 * postings never cross PCIe (only per-document and per-term arrays and the growing elements do). */
#define BM25X_DOC_NONE 0xFFFFFFFFu /* relabel entry of a document that did not survive */

/* The VectorTuple chain as stored (Element.key + value), for maintain.  Exactly one of elem_key / elem_term:
 * elem_key  [n_elem*16]  when the sealed index has term keys (keys strictly ascending inside a document);
 * elem_term [n_elem]     when it has none (dense-ordinal surface; strictly ascending; ordinals >= n_terms(sealed)
 *                        are new tokens and extend the vocabulary to max+1 over the surviving documents, the ones in
 *                        between having df 0). */
typedef struct {
    uint32_t n_docs;
    const uint16_t *payload;   /* [n_docs*3], or NULL = the synthetic ctid of the growing ordinal (what bm25x_growing_create
                                  gives the same documents) */
    const uint8_t *deleted;    /* [n_docs] VectorTuple.deleted, or NULL */
    const uint64_t *elem_off;  /* [n_docs+1] */
    const uint8_t *elem_key;
    const uint32_t *elem_term;
    const uint32_t *elem_tf;   /* != 0, < 2^24 */
} bm25x_vectors;

typedef struct {
    double total_ms, device_ms;      /* host clock around the call; CUDA events from the first upload to the last kernel */
    uint64_t h2d_bytes, d2h_bytes;   /* everything the call copied across PCIe */
    uint64_t postings_in, postings_out; /* sealed postings + growing elements read; postings of the new index */
} bm25x_maintain_stats;

/* bm25::maintain: a NEW sealed index on the same device.  `sealed` is read, never modified, and stays valid; the caller
 * swaps handles and destroys the old one.  sealed_deleted [n_docs(sealed)] or NULL; docs NULL = compaction only.
 * relabel_out [n_docs(sealed) + docs->n_docs] or NULL: new doc id or BM25X_DOC_NONE.  Options set on `sealed`
 * (prune, seed, seed_*, twophase, slice_min) carry over.
 * New documents: the surviving sealed ones in doc-id order, then the surviving growing ones in chain order; payloads
 * (ctids) carry over, doc ids do not.  Tokens: those with at least one surviving posting, ascending (keyed indexes drop
 * the others; keyless ones keep every ordinal, with df 0).  Lengths follow the reference exactly, quirk included: a
 * surviving SEALED document gets its number of distinct tokens (maintain.rs:337,356-360), not Σ tf; a growing one gets
 * Σ tf (vector.rs:77-83).  So maintaining an index with some tf > 1 changes its fieldnorms and avgdl even with no
 * deletes and no inserts.  The peak device memory is the old plus the new index.
 * BM25X_ERR_INVALID: growing handle as `sealed`, keys for a keyless index or ordinals for a keyed one, documents that
 * break vector.rs:39-75, BM25X_TERM_MISSING as an ordinal, no surviving document.  BM25X_ERR_UNSUPPORTED: tf >= 2^24.
 * A failed call returns no handle and leaves `sealed` untouched. */
int bm25x_index_maintain(const bm25x_index *sealed, const uint8_t *sealed_deleted, const bm25x_vectors *docs,
                         bm25x_index **out, uint32_t *relabel_out, bm25x_maintain_stats *stats);

/* bm25::bulkdelete for one handle (sealed or growing): deleted[d] |= payload(d) is in `dead` ([n_dead*3] ctids,
 * ascending by (hi, lo, offset), duplicates allowed; else BM25X_ERR_INVALID).  Marks are only set, never cleared.
 * n_marked (or NULL) = marks newly set by this call.  Searches do not consult the marks (search.rs:227-237): a deleted
 * sealed row is returned until the next maintain, as in the reference. */
int bm25x_bulkdelete(const bm25x_index *idx, const uint16_t *dead, uint64_t n_dead, uint8_t *deleted,
                     uint32_t *n_marked);

/* Invariants of the reference's vector types (crates/bm25/src/vector.rs:46-134): n vectors in CSR form, keys strictly
 * ascending inside a vector, term frequencies (tfs, NULL for Query-like vectors) non-zero — what Document::new / Query::new
 * enforce with expect("invalid data").  BM25X_ERR_INVALID names the first offending vector.  Host only. */
int bm25x_check_vectors(uint32_t n, const uint32_t *off, const uint32_t *terms, const uint32_t *tfs);

/* ---- bm25::evaluate (crates/bm25/src/evaluate.rs:22-74) behind `<&>` without an index scan
 * (src/index/operators.rs:22-55): pair p scores document [d_off[p], d_off[p+1]) (sorted distinct term ordinals
 * with tfs) against query [q_off[p], q_off[p+1]) (sorted distinct ordinals).  out[p] = positive f64 score. */
int bm25x_evaluate_batch(bm25x_index *idx, uint32_t n_pairs, const uint32_t *d_off, const uint32_t *d_terms,
                         const uint32_t *d_tfs, const uint32_t *q_off, const uint32_t *q_terms, double *out);

/* ---- synthetic corpus generator (bench/test utility; spec in DESIGN.md, mirrors tests/fuzz:168-205).
 * Fills a host CSR the caller frees with bm25x_synth_free. zipf_s == 0 ⇒ uniform vocabulary. */
typedef struct {
    uint32_t n_docs, n_terms;
    uint64_t n_postings;
    uint32_t *doc_len;
    uint64_t *post_off;
    uint32_t *post_doc;
    uint32_t *post_tf;
} bm25x_synth_corpus;
int bm25x_synth_generate(uint64_t seed, uint32_t n_docs, uint32_t vocab, uint32_t len_min, uint32_t len_max,
                         double zipf_s, int nthreads, bm25x_synth_corpus *out);
void bm25x_synth_free(bm25x_synth_corpus *c);
/* Queries: n_min..n_max distinct terms with df > 0 drawn from the same distribution. q_off[nq+1], q_terms[nq*n_max]. */
int bm25x_synth_queries(uint64_t seed, uint32_t nq, uint32_t vocab, uint32_t n_min, uint32_t n_max, double zipf_s,
                        const uint64_t *post_off, uint32_t *q_off, uint32_t *q_terms);

const char *bm25x_last_error(void);
int bm25x_device_count(void);

#ifdef __cplusplus
}
#endif
#endif
