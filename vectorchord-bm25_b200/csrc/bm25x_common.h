// bm25x_common.h — internal types shared by the host library and the sm_100a kernels.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>
#include <string>
#include <vector>

#include "../../include/bm25x.h"

#define BM25X_BLOCK 128u            // postings per block, as the reference (crates/bm25/src/flush.rs:84)
#define BM25X_DOC_INF 0xFFFFFFFFu   // exhausted-cursor sentinel, as search.rs:484-496
#define BM25X_POST_ALIGN 4u         // every term's posting list starts on a multiple of 4 postings: 16-byte TMA granularity of
                                    // the doc-id-only copy (pdoc, 4 B per posting) as well as of the 8-byte postings
#define BM25X_CHAMP_L 128u          // champion list: the best min(df, 128) postings of every term by single-term score
#define BM25X_POST_SLACK 4u         // slack slots behind the last list, reading as exhausted cursors

#ifndef BM25X_SEED_MAX_TERMS
#define BM25X_SEED_MAX_TERMS 8
#endif
#ifndef BM25X_TWOPHASE_DEFAULT
#define BM25X_TWOPHASE_DEFAULT 0
#endif

void bm25x_set_error(const char *fmt, ...);
// Host threads this process may really use: the affinity mask capped by the cgroup CPU quota (omp_get_max_threads()
// ignores the quota: 128 threads spinning on a dozen granted cores cost the batch canonicalisation tens of ms).
int bm25x_host_threads(int cap);

#define BM25X_CUDA_TRY(expr)                                                                   \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            bm25x_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__,  \
                            __LINE__);                                                         \
            return _e == cudaErrorMemoryAllocation ? BM25X_ERR_OOM : BM25X_ERR_CUDA;           \
        }                                                                                      \
    } while (0)

// A posting as it lives in HBM: 8 bytes, the reference's logical Mapping(doc u32, tf u32)
// (segment.rs:23-25) with the document's fieldnorm byte folded into the low 8 bits of the
// second word: w = tf << 8 | fieldnorm(doc).  tf < 2^24 is enforced at index build.
struct Posting {
    uint32_t doc;
    uint32_t w;
};

// Device-resident index (flat arrays; replaces the reference's 8 KiB pages, tapes and address trees).
struct DeviceIndex {
    uint32_t n_docs = 0, n_terms = 0;
    uint64_t n_post = 0;      // real postings
    uint64_t n_post_pad = 0;  // incl. the pad slots that round every term up to BM25X_POST_ALIGN postings
    uint64_t n_blocks = 0;
    Posting *post = nullptr;        // [n_post_pad] term-major, doc-ascending inside a term
    uint32_t *pdoc = nullptr;       // [n_post_pad] the doc ids of `post` alone (derived on the device, not replicated): what the
                                    // 2..4-term classes of k_search_ring stream — their hot loop never reads tf / fieldnorm
    // Champion lists (derived on the device, not replicated): per term its best min(df, BM25X_CHAMP_L) postings in the
    // result order (exact single-term score desc, doc id asc).  A document that holds ONE query term can only be in the
    // top-k if it is among the first k champions of that term (every posting ranked before it belongs to a document that
    // beats it), so a query seeds its pool from these and its stream never tests single postings (RCfg::SEEDED).
    Posting *champ = nullptr;       // [champ_off[n_terms]]
    uint64_t *champ_off = nullptr;  // [n_terms+1]
    uint64_t n_champ = 0;
    uint64_t *post_off = nullptr;   // [n_terms+1] padded offsets (multiples of BM25X_POST_ALIGN)
    uint32_t *df = nullptr;         // [n_terms] TokenTuple.number_of_documents
    uint64_t *blk_off = nullptr;    // [n_terms+1] first block index of each term
    uint2 *blk = nullptr;           // [n_blocks] (first doc, last doc) — SummaryTuple.{min,max}_document_id
    float *blk_ub = nullptr;        // [n_blocks] upper bound of one posting's score inside the block (SummaryTuple.wand_*)
    float *s0f = nullptr;           // [n_terms] float(s0)
    double *s0d = nullptr;          // [n_terms] idf*(k1+1), bm25.rs:348
    double *s1d = nullptr;          // [256] k1*(1-b+b*len(fn)/avgdl), bm25.rs:349-352
    float *s1f = nullptr;           // [256]
    double *ubd = nullptr;          // [n_terms] upper bound of one posting's exact score (token-level WAND bound)
    uint8_t *fieldnorm = nullptr;   // [n_docs]
    uint16_t *payload = nullptr;    // [n_docs*3]
};

struct bm25x_index {
    int device = 0;
    int sm_count = 0;
    DeviceIndex d;
    double k1 = 1.2, b = 0.75, avgdl = 0;
    float s1f_min = 0.f;               // min over the documents of s1f[fieldnorm]: one-compare single-term test (k_search_ring)
    uint64_t sum_len = 0;
    uint64_t device_bytes = 0;
    std::vector<uint32_t> h_df;        // host copy for query canonicalisation
    std::vector<uint8_t> h_keys;       // [n_terms*16] sorted keys (optional)
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;  // bm25x_search_batch: result downloads of one slice while the next one runs (lazy)
    uint32_t slice_min = 32768;          // bm25x_search_batch cuts batches of >= 2 x this many queries into slices (0: never)
    std::vector<void *> allocs;
    int prune = 1;                     // MaxScore-style pruning in the search kernels
    uint32_t seed_dense_div = 64;      // seeded launches hand queries with a list of n_docs / 64 postings or more to the plain kernel
    uint32_t seed_prune_min = 32768;   // seeded launches hand queries with a list this long (and 8x their shortest) to the pruning kernel
    int seed_max_terms = BM25X_SEED_MAX_TERMS;  // widest term-count class that runs seeded (4 or 8)
    int seed = 1;                      // 2..4-term classes, k <= BM25X_CHAMP_L, no prefilter: pools seeded from the champion lists
    int twophase = BM25X_TWOPHASE_DEFAULT;  // 2..4-term classes, k <= 224: two launches (8-byte postings, then doc ids only)
    bool growing = false;              // made by bm25x_growing_create: scores with another index's statistics
    // page-locked staging buffer of bm25x_batch_prepare (grow-only, shared by the batches of this index)
    uint32_t *h_stage = nullptr;
    size_t h_stage_words = 0;
    cudaEvent_t h_stage_free = nullptr;  // recorded after the upload that last read h_stage
    bool h_stage_busy = false;
    std::mutex stage_mutex;
    // bm25x_evaluate_batch: tables that depend on the index alone, built on first use (idf per term with the host libm,
    // fieldnorm -> length), kept on the device
    double *eval_idf = nullptr;
    uint32_t *eval_fn_len = nullptr;
    std::mutex eval_mutex;
};

// ---- index construction, shared by every way an index comes to life (bm25x_index.cu) ----

// What the index sources (CSR columns, reference-format blocks, growing documents, maintain) share: statistics, tables,
// allocations.
struct BuildMeta {
    uint32_t n_docs, n_terms;
    const uint32_t *doc_len;
    const uint16_t *payload;
    const uint8_t *term_key;
    double k1, b;
    const uint32_t *df;  // [n_terms]
    uint64_t n_post;
    const uint8_t *fieldnorm = nullptr;  // when doc_len == NULL: DocumentTuple.fieldnorm per doc + JumpTuple.sum_of_document_lengths
    uint64_t sum_len = 0;
    // growing segment (search.rs:66-77): score with the SEALED segment's statistics instead of the index's own
    const uint32_t *stat_df = nullptr;  // [n_terms] sealed TokenTuple.number_of_documents
    uint32_t stat_n_docs = 0;           // sealed JumpTuple.number_of_documents
    double stat_avgdl = 0.0;            // sealed sum_of_document_lengths / number_of_documents
};

// Allocates the index and fills everything except the postings (statistics, s0/s1 tables, fieldnorms, payload, keys,
// padded offsets).  On failure the index is destroyed and *ixp is NULL.
int bm25x_index_begin(const BuildMeta &m, int device, bm25x_index **ixp);
// Bytes bm25x_index_begin + bm25x_index_finish_device copy host → device for an index of this shape.
uint64_t bm25x_index_build_h2d_bytes(uint32_t n_docs, uint32_t n_terms);
// After the postings are in place: pad slots, pdoc, block descriptors, per-term score bounds, champion lists.
cudaError_t bm25x_index_finish_device(bm25x_index *ix);
// Chunked H2D of a term-major CSR (T terms, P postings) and its scatter into ix->d.post: posting p of term t lands at
// d_dst[t] + (p - off[t]) as {doc, tf << 8 | fieldnorm[doc]}.  d_dst: device array [T].
cudaError_t bm25x_scatter_csr(bm25x_index *ix, uint32_t T, uint64_t P, const uint64_t *off, const uint32_t *doc,
                              const uint32_t *tf, const uint64_t *d_dst);
// The ctid given to document i of an index created without payloads: (block hi, block lo, offset) of a 291-tuple page.
void bm25x_synthetic_ctid(uint32_t i, uint16_t out[3]);

// Inversion of doc-major vectors (a VectorTuple chain, vector.rs:46-98) into a term-major CSR over T terms.  Documents
// are visited in order, so every term's list comes out ascending.  Deleted documents are skipped; term_of(e) is the
// term of element e, or BM25X_TERM_MISSING to drop it; doc_id(d) is the id document d gets in the lists.
template <class TermOf, class DocId>
void bm25x_invert_docs(uint32_t G, const uint64_t *elem_off, const uint8_t *deleted, const uint32_t *elem_tf, uint32_t T,
                       TermOf term_of, DocId doc_id, std::vector<uint64_t> &off, std::vector<uint32_t> &doc,
                       std::vector<uint32_t> &tf) {
    off.assign((size_t)T + 1, 0);
    for (uint32_t d = 0; d < G; d++) {
        if (deleted && deleted[d]) continue;
        for (uint64_t e = elem_off[d]; e < elem_off[d + 1]; e++) {
            const uint32_t t = term_of(e);
            if (t != BM25X_TERM_MISSING) off[(size_t)t + 1]++;
        }
    }
    for (uint32_t t = 0; t < T; t++) off[(size_t)t + 1] += off[t];
    const uint64_t P = off[T];
    doc.assign(P ? P : 1, 0);
    tf.assign(P ? P : 1, 0);
    std::vector<uint64_t> cur(off.begin(), off.end() - 1);
    for (uint32_t d = 0; d < G; d++) {
        if (deleted && deleted[d]) continue;
        const uint32_t id = doc_id(d);
        for (uint64_t e = elem_off[d]; e < elem_off[d + 1]; e++) {
            const uint32_t t = term_of(e);
            if (t == BM25X_TERM_MISSING) continue;
            doc[cur[t]] = id;
            tf[cur[t]] = elem_tf[e];
            cur[t]++;
        }
    }
}
