// bm25x_index.cu — index lifetime: host CSR (the reference's sealed Segment) → flat HBM layout.
//
// Replaces, for the read path, bm25::build → flush (crates/bm25/src/build.rs:22-71,
// crates/bm25/src/flush.rs:40-158): same semantics (N, Σlen → avgdl from exact lengths, per-document
// quantised fieldnorm, 128-posting blocks in (term, doc) order with min/max doc per block, df per
// token) but none of its page / tape / address-tree machinery.  Layout in DESIGN.md §3.
#include <math.h>
#include <omp.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "bm25x_common.h"
#include "bm25x_blocks.cuh"

static thread_local char g_err[512] = "";

void bm25x_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char *bm25x_last_error(void) { return g_err; }

int bm25x_host_threads(int cap) {
    static const int granted = [] {
        if (const char *e = getenv("BM25X_HOST_THREADS")) {  // explicit share, e.g. cores / ranks when several ranks share a box
            const int v = atoi(e);
            if (v >= 1) return v;
        }
        int n = omp_get_num_procs();  // honours the affinity mask
        FILE *f = fopen("/sys/fs/cgroup/cpu.max", "r");
        if (f) {
            char q[64];
            long long per = 0;
            if (fscanf(f, "%63s %lld", q, &per) == 2 && strcmp(q, "max") != 0 && per > 0) {
                const long long quota = (atoll(q) + per / 2) / per;
                if (quota >= 1 && quota < n) n = (int)quota;
            }
            fclose(f);
        } else if ((f = fopen("/sys/fs/cgroup/cpu/cpu.cfs_quota_us", "r"))) {
            long long quota = -1, per = 100000;
            if (fscanf(f, "%lld", &quota) != 1) quota = -1;
            fclose(f);
            FILE *g = fopen("/sys/fs/cgroup/cpu/cpu.cfs_period_us", "r");
            if (g) {
                if (fscanf(g, "%lld", &per) != 1) per = 100000;
                fclose(g);
            }
            if (quota > 0 && per > 0 && (quota + per / 2) / per < n) n = (int)std::max<long long>(1, (quota + per / 2) / per);
        }
        return n < 1 ? 1 : n;
    }();
    return cap > 0 && granted > cap ? cap : granted;
}

extern "C" int bm25x_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// ---- fieldnorm codec (crates/bm25/src/bm25.rs:15-283): 0..=40 step 1, then groups of 8 whose step
// doubles per group.  Generated, and pinned against the reference's literal table by the tests. ----
static uint32_t g_fn_len[256];
static bool g_fn_ready = false;
static void fn_init() {
    if (g_fn_ready) return;
    int n = 0;
    for (; n <= 40; n++) g_fn_len[n] = (uint32_t)n;
    uint32_t v = 40, step = 2;
    while (n < 256) {
        for (int i = 0; i < 8 && n < 256; i++) {
            v += step;
            g_fn_len[n++] = v;
        }
        step *= 2;
    }
    g_fn_ready = true;
}
uint32_t bm25x_fieldnorm_to_length(uint8_t fn) {
    fn_init();
    return g_fn_len[fn];
}
uint8_t bm25x_length_to_fieldnorm(uint32_t len) {  // bm25.rs:278-283
    fn_init();
    int lo = 0, hi = 256;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (g_fn_len[mid] <= len) lo = mid + 1;
        else hi = mid;
    }
    return (uint8_t)(lo - 1);
}

// ---- device transforms ----

// CSR chunk → AoS postings at their padded positions, with the fieldnorm byte folded in.
__global__ void k_build_postings(const uint32_t *__restrict__ c_doc, const uint32_t *__restrict__ c_tf,
                                 uint64_t chunk_base, uint64_t chunk_n, const uint64_t *__restrict__ off,
                                 const uint64_t *__restrict__ off_pad, uint32_t n_terms,
                                 const uint8_t *__restrict__ fieldnorm, Posting *__restrict__ post) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= chunk_n) return;
    uint64_t gi = chunk_base + i;
    // term = last t with off[t] <= gi
    uint32_t lo = 0, hi = n_terms;
    while (lo < hi) {
        uint32_t mid = (lo + hi + 1) >> 1;
        if (off[mid] <= gi) lo = mid;
        else hi = mid - 1;
    }
    uint32_t d = c_doc[i];
    Posting p;
    p.doc = d;
    p.w = (c_tf[i] << 8) | fieldnorm[d];
    post[off_pad[lo] + (gi - off[lo])] = p;
}

__global__ void k_pad_slots(const uint64_t *__restrict__ off_pad, const uint32_t *__restrict__ df, uint32_t n_terms,
                            Posting *__restrict__ post) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_terms) return;
    Posting p;
    p.doc = BM25X_DOC_INF;
    p.w = 0;
    const uint32_t end = (df[t] + BM25X_POST_ALIGN - 1u) & ~(BM25X_POST_ALIGN - 1u);
    for (uint32_t i = df[t]; i < end; i++) post[off_pad[t] + i] = p;
}

// pdoc[i] = post[i].doc: the doc-id-only copy streamed by the 2..4-term classes of k_search_ring (bm25x_search_ring.cuh,
// RCfg::DOCRING).  Derived data: built here for every way an index comes to life (postings, stored blocks, replica).
__global__ void k_extract_docs(const Posting *__restrict__ post, uint64_t n, uint32_t *__restrict__ pdoc) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) pdoc[i] = post[i].doc;
}

// Per 128-posting block: (first doc, last doc) = SummaryTuple.{min,max}_document_id, and the block's score bound =
// Cache::evaluate of the block's arg-max posting, what the reference keeps as SummaryTuple.(wand_fieldnorm,
// wand_term_frequency) (flush.rs:101-120) and evaluates per block at query time (search.rs:381,426-429).  Stored as f32
// rounded UP after the same 2^-40 inflation as the token-level bound.
__global__ void k_block_desc(const uint64_t *__restrict__ off_pad, const uint32_t *__restrict__ df,
                             const uint64_t *__restrict__ blk_off, uint32_t n_terms, uint64_t n_blocks,
                             const Posting *__restrict__ post, const double *__restrict__ s0d,
                             const double *__restrict__ s1d, uint2 *__restrict__ blk, float *__restrict__ blk_ub) {
    uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_blocks) return;
    uint32_t lo = 0, hi = n_terms;
    while (lo < hi) {
        uint32_t mid = (lo + hi + 1) >> 1;
        if (blk_off[mid] <= g) lo = mid;
        else hi = mid - 1;
    }
    uint64_t b = g - blk_off[lo];
    uint64_t first = b * BM25X_BLOCK;
    uint64_t last = first + BM25X_BLOCK;
    if (last > df[lo]) last = df[lo];
    blk[g] = make_uint2(post[off_pad[lo] + first].doc, post[off_pad[lo] + last - 1].doc);
    const double s0 = s0d[lo];
    double best = 0.0;
    for (uint64_t i = first; i < last; i++) {
        const uint32_t w = post[off_pad[lo] + i].w;
        const double tfd = (double)(w >> 8);
        const double v = __ddiv_rn(__dmul_rn(tfd, s0), __dadd_rn(tfd, s1d[w & 0xFFu]));
        best = v > best ? v : best;
    }
    blk_ub[g] = __double2float_ru(best * (1.0 + 9.094947017729282e-13));
}

// Ingest check: the stored SummaryTuple.(wand_fieldnorm, wand_term_frequency) of a block must evaluate to the block's
// real maximum (it is the arg-max of the block's own postings, flush.rs:101-110); anything else is a corrupt index.
__global__ void k_check_block_wand(uint64_t n_blocks, const uint64_t *__restrict__ blk_off, uint32_t n_terms,
                                   const uint8_t *__restrict__ wand_fn, const uint32_t *__restrict__ wand_tf,
                                   const double *__restrict__ s0d, const double *__restrict__ s1d,
                                   const float *__restrict__ blk_ub, uint32_t *__restrict__ err) {
    uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_blocks) return;
    uint32_t lo = 0, hi = n_terms;
    while (lo < hi) {
        uint32_t mid = (lo + hi + 1) >> 1;
        if (blk_off[mid] <= g) lo = mid;
        else hi = mid - 1;
    }
    const double tfd = (double)wand_tf[g];
    const double v = __ddiv_rn(__dmul_rn(tfd, s0d[lo]), __dadd_rn(tfd, s1d[wand_fn[g]]));
    const float ub = __double2float_ru(v * (1.0 + 9.094947017729282e-13));
    // tf() and Cache::evaluate round differently: allow the last f32 ulp either way
    if (!(ub <= blk_ub[g] * 1.0000003f && ub >= blk_ub[g] * 0.9999997f)) atomicOr(err, 8u);
}

// Per-term upper bound of a single posting's exact score: max over the term's postings of Cache::evaluate
// (bm25.rs:355-358) — what the reference stores as the token-level (wand_fieldnorm, wand_term_frequency) arg-max
// (flush.rs:101-120) and evaluates at query time (search.rs:363).  One block per term; inflated by 2^-40 so that the
// bound also dominates any later re-association of the f64 sum.
__global__ void k_term_ub(const uint64_t *__restrict__ off_pad, const uint32_t *__restrict__ df,
                          const Posting *__restrict__ post, const double *__restrict__ s0d,
                          const double *__restrict__ s1d, uint32_t n_terms, double *__restrict__ ubd) {
    __shared__ double red[256];
    for (uint32_t t = blockIdx.x; t < n_terms; t += gridDim.x) {
        const Posting *pp = post + off_pad[t];
        const double s0 = s0d[t];
        double best = 0.0;
        for (uint32_t i = threadIdx.x; i < df[t]; i += blockDim.x) {
            uint32_t w = pp[i].w;
            double tfd = (double)(w >> 8);
            double v = __ddiv_rn(__dmul_rn(tfd, s0), __dadd_rn(tfd, s1d[w & 0xFFu]));
            best = v > best ? v : best;
        }
        red[threadIdx.x] = best;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if ((int)threadIdx.x < o && red[threadIdx.x + o] > red[threadIdx.x]) red[threadIdx.x] = red[threadIdx.x + o];
            __syncthreads();
        }
        if (threadIdx.x == 0) ubd[t] = red[0] * (1.0 + 9.094947017729282e-13);
        __syncthreads();
    }
}

// Champion lists: one warp per term keeps the best L postings by (exact single-term score desc, doc id asc) — the order in
// which single-term documents enter a result (Cache::evaluate, bm25.rs:355-358, is the whole score of such a document).
// The list is scanned once in doc order; a posting is buffered only if it beats the current L-th best (later documents
// lose ties), and the 2L-entry buffer is sorted and cut back to L when it fills.
#define CHAMP_WARPS 4
__global__ void __launch_bounds__(CHAMP_WARPS * 32) k_champions(const uint64_t *__restrict__ off_pad, const uint32_t *__restrict__ df,
                                                                const Posting *__restrict__ post, const double *__restrict__ s0d,
                                                                const double *__restrict__ s1d, uint32_t n_terms,
                                                                const uint64_t *__restrict__ champ_off, Posting *__restrict__ champ) {
    constexpr int L = (int)BM25X_CHAMP_L, CAP = 2 * L;
    __shared__ double bs[CHAMP_WARPS][CAP];
    __shared__ uint32_t bd[CHAMP_WARPS][CAP], bw[CHAMP_WARPS][CAP];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    double *ss = bs[wid];
    uint32_t *sd = bd[wid], *sw = bw[wid];
    const uint32_t lt = (1u << lane) - 1u;
    auto sort_buf = [&](int n) {  // bitonic over CAP entries, best first; entries >= n are padding (score -1)
        for (int i = n + lane; i < CAP; i += 32) {
            ss[i] = -1.0;
            sd[i] = BM25X_DOC_INF;
            sw[i] = 0;
        }
        __syncwarp();
        for (int size = 2; size <= CAP; size <<= 1)
            for (int stride = size >> 1; stride > 0; stride >>= 1) {
                for (int i = lane; i < CAP / 2; i += 32) {
                    const int a = 2 * i - (i & (stride - 1)), b = a + stride;
                    const double sa = ss[a], sb = ss[b];
                    const uint32_t da = sd[a], db = sd[b];
                    const bool a_first = sa > sb || (sa == sb && da < db);
                    const bool desc = (a & size) == 0;
                    if (desc ? !a_first : a_first) {
                        ss[a] = sb;
                        ss[b] = sa;
                        sd[a] = db;
                        sd[b] = da;
                        const uint32_t t = sw[a];
                        sw[a] = sw[b];
                        sw[b] = t;
                    }
                }
                __syncwarp();
            }
    };
    for (uint32_t t = blockIdx.x * CHAMP_WARPS + wid; t < n_terms; t += gridDim.x * CHAMP_WARPS) {
        const Posting *pp = post + off_pad[t];
        const uint32_t n = df[t];
        const double s0 = s0d[t];
        int cnt = 0;
        bool have = false;
        double thr = 0.0;
        for (uint32_t base = 0; base < n; base += 32) {
            const uint32_t i = base + lane;
            Posting v;
            v.doc = 0;
            v.w = 0;
            double sc = -1.0;
            if (i < n) {
                v = pp[i];
                const double tfd = (double)(v.w >> 8);
                sc = __ddiv_rn(__dmul_rn(tfd, s0), __dadd_rn(tfd, s1d[v.w & 0xFFu]));
            }
            const bool acc = i < n && (!have || sc > thr);
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, acc);
            if (acc) {
                const int at = cnt + __popc(m & lt);
                ss[at] = sc;
                sd[at] = v.doc;
                sw[at] = v.w;
            }
            cnt += __popc(m);
            if (cnt > CAP - 32) {
                __syncwarp();
                sort_buf(cnt);
                cnt = L;
                thr = ss[L - 1];
                have = true;
                __syncwarp();
            }
        }
        __syncwarp();
        sort_buf(cnt);
        const int keep = cnt < L ? cnt : L;
        Posting *out = champ + champ_off[t];
        for (int i = lane; i < keep; i += 32) {
            Posting v;
            v.doc = sd[i];
            v.w = sw[i];
            out[i] = v;
        }
        __syncwarp();
    }
}

// champ_off from the host copy of df, then the lists (bm25x_index_finish_device / finalize_replica; needs post, s0d, s1d)
static cudaError_t build_champions(bm25x_index *ix);

template <typename T>
static int dev_alloc(bm25x_index *ix, T **p, size_t n) {
    size_t bytes = sizeof(T) * (n ? n : 1);
    BM25X_CUDA_TRY(cudaMalloc((void **)p, bytes));
    ix->allocs.push_back((void *)*p);
    ix->device_bytes += bytes;
    return BM25X_OK;
}

static cudaError_t build_champions(bm25x_index *ix) {
    DeviceIndex &d = ix->d;
    const uint32_t T = d.n_terms;
    std::vector<uint64_t> h_off((size_t)T + 1);
    uint64_t run = 0;
    for (uint32_t t = 0; t < T; t++) {
        h_off[t] = run;
        run += std::min<uint32_t>(ix->h_df[t], BM25X_CHAMP_L);
    }
    h_off[T] = run;
    d.n_champ = run;
    cudaError_t e = cudaMalloc((void **)&d.champ, sizeof(Posting) * (size_t)(run ? run : 1));
    if (e != cudaSuccess) return e;
    ix->allocs.push_back((void *)d.champ);
    ix->device_bytes += sizeof(Posting) * (size_t)(run ? run : 1);
    e = cudaMalloc((void **)&d.champ_off, sizeof(uint64_t) * ((size_t)T + 1));
    if (e != cudaSuccess) return e;
    ix->allocs.push_back((void *)d.champ_off);
    ix->device_bytes += sizeof(uint64_t) * ((size_t)T + 1);
    e = cudaMemcpy(d.champ_off, h_off.data(), sizeof(uint64_t) * ((size_t)T + 1), cudaMemcpyHostToDevice);
    if (e != cudaSuccess || !T) return e;
    const unsigned blocks = (unsigned)std::min<uint64_t>(((uint64_t)T + CHAMP_WARPS - 1) / CHAMP_WARPS, 148ull * 16ull);
    k_champions<<<blocks, CHAMP_WARPS * 32>>>(d.post_off, d.df, d.post, d.s0d, d.s1d, T, d.champ_off, d.champ);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    return e;
}

#define TRY(x)                      \
    do {                            \
        int _rc = (x);              \
        if (_rc != BM25X_OK) {      \
            bm25x_index_destroy(ix); \
            return _rc;             \
        }                           \
    } while (0)
#define CU(x)                                                                                       \
    do {                                                                                            \
        cudaError_t _e = (x);                                                                       \
        if (_e != cudaSuccess) {                                                                    \
            bm25x_set_error("%s failed: %s (%s:%d)", #x, cudaGetErrorString(_e), __FILE__, __LINE__); \
            bm25x_index_destroy(ix);                                                                \
            return _e == cudaErrorMemoryAllocation ? BM25X_ERR_OOM : BM25X_ERR_CUDA;                \
        }                                                                                           \
    } while (0)

static int check_common(const char *who, uint32_t n_docs, const void *doc_len, double k1, double b, int device) {
    if (n_docs == 0 || n_docs == BM25X_DOC_INF || !doc_len) {
        bm25x_set_error("%s: empty or malformed corpus", who);
        return BM25X_ERR_INVALID;
    }
    if (!(k1 >= 0.0) || !(b >= 0.0 && b <= 1.0)) {
        bm25x_set_error("%s: k1/b out of range", who);
        return BM25X_ERR_INVALID;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
        cudaGetLastError();
        bm25x_set_error("%s: CUDA device %d not available (%d devices); there is no CPU fallback", who, device, ndev);
        return BM25X_ERR_CUDA;
    }
    return BM25X_OK;
}

static int check_keys(const char *who, const uint8_t *term_key, uint32_t T) {
    if (term_key)
        for (uint32_t t = 1; t < T; t++)
            if (memcmp(term_key + (size_t)(t - 1) * 16, term_key + (size_t)t * 16, 16) >= 0) {
                bm25x_set_error("%s: term_key must be strictly ascending", who);
                return BM25X_ERR_INVALID;
            }
    return BM25X_OK;
}

// Allocates the index and fills everything except the postings.  On failure the index is destroyed.
// Environment overrides of the option defaults (test matrix: BM25X_SEED=0 / BM25X_TWOPHASE=1 run the same tests through
// the other kernel paths); bm25x_index_set_option still wins.
static void apply_env_options(bm25x_index *ix) {
    if (const char *e = getenv("BM25X_SEED")) ix->seed = atoi(e) != 0;
    if (const char *e = getenv("BM25X_TWOPHASE")) ix->twophase = atoi(e) != 0;
    if (const char *e = getenv("BM25X_SEED_FORCE")) {  // every eligible query through the seeded kernel, dense or skewed
        if (atoi(e) != 0) {
            ix->seed_prune_min = 0xFFFFFFFFu;
            ix->seed_dense_div = 0u;
        }
    }
}

void bm25x_synthetic_ctid(uint32_t i, uint16_t out[3]) {
    const uint32_t blkno = i / 291;
    out[0] = (uint16_t)(blkno >> 16);
    out[1] = (uint16_t)(blkno & 0xFFFF);
    out[2] = (uint16_t)(i % 291 + 1);
}

uint64_t bm25x_index_build_h2d_bytes(uint32_t n_docs, uint32_t n_terms) {
    const uint64_t N = n_docs, T = n_terms;
    // post_off, blk_off, champ_off; df, s0d, s0f; s1d, s1f; fieldnorm, payload
    return 3 * 8 * (T + 1) + (T ? (4 + 8 + 4) * T : 0) + 256 * (8 + 4) + N + 6 * N;
}

int bm25x_index_begin(const BuildMeta &m, int device, bm25x_index **ixp) {
    *ixp = nullptr;
    fn_init();
    const uint32_t N = m.n_docs, T = m.n_terms;
    const uint64_t P = m.n_post;
    bm25x_index *ix = new bm25x_index();
    apply_env_options(ix);
    ix->device = device;
    ix->k1 = m.k1;
    ix->b = m.b;
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        bm25x_set_error("bm25x_index_create: device %d is sm_%d%d; this library only carries sm_100a kernels", device,
                        prop.major, prop.minor);
        bm25x_index_destroy(ix);
        return BM25X_ERR_CUDA;
    }
    ix->sm_count = prop.multiProcessorCount;
    CU(cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking));
    {   // keep freed batch buffers cached in the default pool (bm25x_batch_* allocate stream-ordered)
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            uint64_t thr = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        }
    }

    // ---- flush.rs:52-66: N, Σlen (exact), per-doc fieldnorm (quantised), avgdl ----
    std::vector<uint8_t> h_fn(N);
    uint64_t sum_len = 0;
    if (m.doc_len) {
#pragma omp parallel for reduction(+ : sum_len) num_threads(bm25x_host_threads(0))
        for (uint32_t d = 0; d < N; d++) {
            sum_len += m.doc_len[d];
            h_fn[d] = bm25x_length_to_fieldnorm(m.doc_len[d]);
        }
    } else {  // the stored index keeps only the quantised norm per document and the exact total (tuples.rs:141-160,756-762)
        memcpy(h_fn.data(), m.fieldnorm, N);
        sum_len = m.sum_len;
    }
    ix->sum_len = sum_len;
    ix->avgdl = m.stat_df ? m.stat_avgdl : (double)sum_len / (double)N;

    // ---- per-term df, padded offsets, block offsets, s0 (bm25.rs:285-289,348) ----
    ix->h_df.resize(T);
    std::vector<uint64_t> h_off_pad(T + 1), h_blk_off(T + 1);
    std::vector<double> h_s0d(T);
    std::vector<float> h_s0f(T);
    uint64_t pp = 0, nb = 0;
    for (uint32_t t = 0; t < T; t++) {
        uint64_t n = m.df[t];
        ix->h_df[t] = (uint32_t)n;
        h_off_pad[t] = pp;
        h_blk_off[t] = nb;
        pp += (n + BM25X_POST_ALIGN - 1) & ~(uint64_t)(BM25X_POST_ALIGN - 1);
        nb += (n + BM25X_BLOCK - 1) / BM25X_BLOCK;
        const double n_stat = m.stat_df ? (double)m.stat_df[t] : (double)n, N_stat = m.stat_df ? (double)m.stat_n_docs : (double)N;
        double idf = log((N_stat + 1.0) / (n_stat + 0.5));
        h_s0d[t] = idf * (m.k1 + 1.0);
        h_s0f[t] = (float)h_s0d[t];
    }
    h_off_pad[T] = pp;
    h_blk_off[T] = nb;
    // bm25.rs:349-352 — identical for every term: depends only on (k1, b, avgdl)
    double h_s1d[256];
    float h_s1f[256];
    for (int f = 0; f < 256; f++) {
        double dl = (double)g_fn_len[f];
        h_s1d[f] = m.k1 * (1.0 - m.b + m.b * dl / ix->avgdl);
        h_s1f[f] = (float)h_s1d[f];
    }
    {   // smallest s1 over the documents present: the one-compare single-term test of k_search_ring needs a lower bound
        bool seen[256] = {false};
        for (uint32_t d = 0; d < N; d++) seen[h_fn[d]] = true;
        float mn = 3.0e38f;
        for (int f = 0; f < 256; f++)
            if (seen[f] && h_s1f[f] < mn) mn = h_s1f[f];
        ix->s1f_min = mn;
    }
    if (m.term_key) ix->h_keys.assign(m.term_key, m.term_key + (size_t)T * 16);

    DeviceIndex &d = ix->d;
    d.n_docs = N;
    d.n_terms = T;
    d.n_post = P;
    d.n_post_pad = pp;
    d.n_blocks = nb;
    TRY(dev_alloc(ix, &d.post, pp + BM25X_POST_SLACK));
    TRY(dev_alloc(ix, &d.pdoc, pp + BM25X_POST_SLACK));
    TRY(dev_alloc(ix, &d.post_off, (size_t)T + 1));
    TRY(dev_alloc(ix, &d.df, T));
    TRY(dev_alloc(ix, &d.blk_off, (size_t)T + 1));
    TRY(dev_alloc(ix, &d.blk, nb));
    TRY(dev_alloc(ix, &d.blk_ub, nb));
    TRY(dev_alloc(ix, &d.s0f, T));
    TRY(dev_alloc(ix, &d.s0d, T));
    TRY(dev_alloc(ix, &d.s1d, 256));
    TRY(dev_alloc(ix, &d.s1f, 256));
    TRY(dev_alloc(ix, &d.ubd, T));
    TRY(dev_alloc(ix, &d.fieldnorm, N));
    TRY(dev_alloc(ix, &d.payload, (size_t)N * 3));
    CU(cudaMemset((void *)(d.post + pp), 0xFF, BM25X_POST_SLACK * sizeof(Posting)));  // the slack slots read as exhausted cursors
    CU(cudaMemcpy(d.post_off, h_off_pad.data(), sizeof(uint64_t) * (T + 1), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d.blk_off, h_blk_off.data(), sizeof(uint64_t) * (T + 1), cudaMemcpyHostToDevice));
    if (T) {
        CU(cudaMemcpy(d.df, ix->h_df.data(), sizeof(uint32_t) * T, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(d.s0d, h_s0d.data(), sizeof(double) * T, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(d.s0f, h_s0f.data(), sizeof(float) * T, cudaMemcpyHostToDevice));
    }
    CU(cudaMemcpy(d.s1d, h_s1d, sizeof(h_s1d), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d.s1f, h_s1f, sizeof(h_s1f), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d.fieldnorm, h_fn.data(), N, cudaMemcpyHostToDevice));
    if (m.payload) {
        CU(cudaMemcpy(d.payload, m.payload, sizeof(uint16_t) * 3 * (size_t)N, cudaMemcpyHostToDevice));
    } else {
        std::vector<uint16_t> pl((size_t)N * 3);
        for (uint32_t i = 0; i < N; i++) bm25x_synthetic_ctid(i, &pl[(size_t)i * 3]);
        CU(cudaMemcpy(d.payload, pl.data(), sizeof(uint16_t) * pl.size(), cudaMemcpyHostToDevice));
    }

    *ixp = ix;
    return BM25X_OK;
}

cudaError_t bm25x_index_finish_device(bm25x_index *ix) {
    DeviceIndex &d = ix->d;
    const uint32_t T = d.n_terms;
    const uint64_t nb = d.n_blocks;
    cudaError_t e = cudaSuccess;
    if (T) {
        k_pad_slots<<<(T + 255) / 256, 256>>>(d.post_off, d.df, T, d.post);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) {
        k_extract_docs<<<148 * 8, 256>>>(d.post, d.n_post_pad + BM25X_POST_SLACK, d.pdoc);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess && nb) {
        k_block_desc<<<(unsigned)((nb + 255) / 256), 256>>>(d.post_off, d.df, d.blk_off, T, nb, d.post, d.s0d, d.s1d, d.blk,
                                                            d.blk_ub);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess && T) {
        k_term_ub<<<(unsigned)std::min<uint32_t>(T, 148u * 16u), 256>>>(d.post_off, d.df, d.post, d.s0d, d.s1d, T, d.ubd);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = build_champions(ix);
    return e;
}

cudaError_t bm25x_scatter_csr(bm25x_index *ix, uint32_t T, uint64_t P, const uint64_t *post_off, const uint32_t *post_doc,
                              const uint32_t *post_tf, const uint64_t *d_dst) {
    DeviceIndex &d = ix->d;
    uint64_t *d_off = nullptr;
    uint32_t *d_cdoc = nullptr, *d_ctf = nullptr;
    const uint64_t CH = 64ull << 20;  // postings per chunk
    uint64_t chn = std::min<uint64_t>(CH, P ? P : 1);
    cudaError_t e1 = cudaMalloc((void **)&d_off, sizeof(uint64_t) * ((size_t)T + 1));
    cudaError_t e2 = cudaMalloc((void **)&d_cdoc, sizeof(uint32_t) * chn);
    cudaError_t e3 = cudaMalloc((void **)&d_ctf, sizeof(uint32_t) * chn);
    cudaError_t e = e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3);
    if (e == cudaSuccess) e = cudaMemcpy(d_off, post_off, sizeof(uint64_t) * ((size_t)T + 1), cudaMemcpyHostToDevice);
    for (uint64_t base = 0; base < P && e == cudaSuccess; base += CH) {
        uint64_t n = std::min<uint64_t>(CH, P - base);
        e = cudaMemcpy(d_cdoc, post_doc + base, sizeof(uint32_t) * n, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(d_ctf, post_tf + base, sizeof(uint32_t) * n, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) {
            k_build_postings<<<(unsigned)((n + 255) / 256), 256>>>(d_cdoc, d_ctf, base, n, d_off, d_dst, T, d.fieldnorm,
                                                                   d.post);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
    }
    cudaFree(d_off);
    cudaFree(d_cdoc);
    cudaFree(d_ctf);
    return e;
}

// Postings of a term-major CSR: chunked H2D of the columns + device transform to the padded AoS, then the derived arrays.
// Destroys the index on failure.
static int upload_csr(bm25x_index *ix, const char *who, uint32_t T, uint64_t P, const uint64_t *post_off,
                      const uint32_t *post_doc, const uint32_t *post_tf) {
    cudaError_t e = bm25x_scatter_csr(ix, T, P, post_off, post_doc, post_tf, ix->d.post_off);
    if (e == cudaSuccess) e = bm25x_index_finish_device(ix);
    if (e != cudaSuccess) {
        bm25x_set_error("%s: posting upload failed: %s", who, cudaGetErrorString(e));
        bm25x_index_destroy(ix);
        return e == cudaErrorMemoryAllocation ? BM25X_ERR_OOM : BM25X_ERR_CUDA;
    }
    return BM25X_OK;
}

extern "C" int bm25x_index_create(const bm25x_corpus *c, int device, bm25x_index **out) {
    if (!c || !out) {
        bm25x_set_error("bm25x_index_create: null argument");
        return BM25X_ERR_INVALID;
    }
    *out = nullptr;
    if (!c->post_off || (c->post_off[c->n_terms] && (!c->post_doc || !c->post_tf))) {
        bm25x_set_error("bm25x_index_create: empty or malformed corpus");
        return BM25X_ERR_INVALID;
    }
    int rc = check_common("bm25x_index_create", c->n_docs, c->doc_len, c->k1, c->b, device);
    if (rc != BM25X_OK) return rc;
    const uint32_t N = c->n_docs, T = c->n_terms;
    const uint64_t P = c->post_off[T];

    // ---- host-side validation of the CSR (the reference panics with "data corruption") ----
    int bad = 0;  // 1 = ordering/ranges, 2 = tf too large
#pragma omp parallel for schedule(dynamic, 256) reduction(| : bad) num_threads(bm25x_host_threads(0))
    for (uint32_t t = 0; t < T; t++) {
        uint64_t p0 = c->post_off[t], p1 = c->post_off[t + 1];
        if (p1 < p0 || p1 > P) {
            bad |= 1;
            continue;
        }
        if (p1 - p0 > N) bad |= 1;
        uint32_t prev = 0;
        for (uint64_t p = p0; p < p1; p++) {
            uint32_t d = c->post_doc[p], f = c->post_tf[p];
            if (d >= N || f == 0 || (p > p0 && d <= prev)) bad |= 1;
            if (f >= (1u << 24)) bad |= 2;
            prev = d;
        }
    }
    if (bad & 1) {
        bm25x_set_error("bm25x_index_create: corrupt corpus (doc ids must be < n_docs and strictly ascending per term, tf != 0)");
        return BM25X_ERR_INVALID;
    }
    if (bad & 2) {
        bm25x_set_error("bm25x_index_create: term frequency >= 2^24 is not supported by the packed posting layout");
        return BM25X_ERR_UNSUPPORTED;
    }
    rc = check_keys("bm25x_index_create", c->term_key, T);
    if (rc != BM25X_OK) return rc;

    std::vector<uint32_t> df(T);
    for (uint32_t t = 0; t < T; t++) df[t] = (uint32_t)(c->post_off[t + 1] - c->post_off[t]);
    BuildMeta m{N, T, c->doc_len, c->payload, c->term_key, c->k1, c->b, df.data(), P};
    bm25x_index *ix = nullptr;
    rc = bm25x_index_begin(m, device, &ix);
    if (rc != BM25X_OK) return rc;

    rc = upload_csr(ix, "bm25x_index_create", T, P, c->post_off, c->post_doc, c->post_tf);
    if (rc != BM25X_OK) return rc;
    *out = ix;
    return BM25X_OK;
}

// ---- f1: the sealed segment as the reference stores it (blocks in the codec of compression.rs), decoded on the GPU ----
extern "C" int bm25x_index_create_from_blocks(const bm25x_blocks *c, int device, bm25x_index **out) {
    const char *who = "bm25x_index_create_from_blocks";
    if (!c || !out) {
        bm25x_set_error("%s: null argument", who);
        return BM25X_ERR_INVALID;
    }
    *out = nullptr;
    const uint32_t N = c->n_docs, T = c->n_terms;
    const uint64_t NB = c->n_blocks;
    if (!c->term_blk_off || (NB && (!c->blk_min_doc || !c->blk_n || !c->blk_meta_doc || !c->blk_meta_tf ||
                                    !c->blk_doc_off || !c->blk_tf_off || (c->n_bytes && !c->bytes)))) {
        bm25x_set_error("%s: empty or malformed corpus", who);
        return BM25X_ERR_INVALID;
    }
    int rc = check_common(who, N, c->doc_len ? (const void *)c->doc_len : (const void *)c->doc_fieldnorm, c->k1, c->b, device);
    if (rc != BM25X_OK) return rc;
    if (c->term_blk_off[0] != 0 || c->term_blk_off[T] != NB) {
        bm25x_set_error("%s: term_blk_off must run from 0 to n_blocks", who);
        return BM25X_ERR_INVALID;
    }
    // ---- host-side validation of the block directory (payloads are validated by the decoder on the device) ----
    std::vector<uint32_t> df(T);
    uint64_t P = 0;
    int bad = 0;
#pragma omp parallel for schedule(dynamic, 256) reduction(| : bad) reduction(+ : P) num_threads(bm25x_host_threads(0))
    for (uint32_t t = 0; t < T; t++) {
        const uint64_t b0 = c->term_blk_off[t], b1 = c->term_blk_off[t + 1];
        if (b1 < b0 || b1 > NB) {
            bad |= 1;
            df[t] = 0;
            continue;
        }
        uint64_t n_t = 0;
        for (uint64_t g = b0; g < b1; g++) {
            const uint32_t n = c->blk_n[g];
            // flush.rs:80-90: every block of a token holds 128 postings except the last one
            if (n == 0 || n > BM25X_BLOCK || (n < BM25X_BLOCK && g + 1 != b1)) bad |= 1;
            const uint8_t metas[2] = {c->blk_meta_doc[g], c->blk_meta_tf[g]};
            const uint64_t offs[2] = {c->blk_doc_off[g], c->blk_tf_off[g]};
            for (int s = 0; s < 2; s++) {
                const uint32_t w = metas[s] & 0x7Fu;
                uint64_t nbytes;
                if ((metas[s] >> 7) == 0) {  // compression.rs:43-52: bit packing only for full blocks, width <= 32
                    if (w > 32 || n != BM25X_BLOCK) bad |= 2;
                    nbytes = (uint64_t)w * 16;
                } else {                      // compression.rs:53-62: 1..4 bytes per value
                    if (w < 1 || w > 4) bad |= 2;
                    nbytes = (uint64_t)w * n;
                }
                if (offs[s] > c->n_bytes || nbytes > c->n_bytes - offs[s]) bad |= 1;
            }
            n_t += n;
        }
        if (n_t > N) bad |= 1;
        df[t] = (uint32_t)std::min<uint64_t>(n_t, N);
        P += n_t;
    }
    if (bad & 1) {
        bm25x_set_error("%s: corrupt block directory (block sizes, token ranges or payload offsets)", who);
        return BM25X_ERR_INVALID;
    }
    if (bad & 2) {
        bm25x_set_error("%s: corrupt block metadata (bitwidth out of bound / unexpected input len)", who);
        return BM25X_ERR_INVALID;
    }
    rc = check_keys(who, c->term_key, T);
    if (rc != BM25X_OK) return rc;

    BuildMeta m{N, T, c->doc_len, c->payload, c->term_key, c->k1, c->b, df.data(), P};
    m.fieldnorm = c->doc_fieldnorm;
    m.sum_len = c->sum_doc_len;
    bm25x_index *ix = nullptr;
    rc = bm25x_index_begin(m, device, &ix);
    if (rc != BM25X_OK) return rc;
    DeviceIndex &d = ix->d;

    // ---- upload the directory + payloads, decode on the device ----
    uint64_t *d_tbo = nullptr, *d_doff = nullptr, *d_toff = nullptr;
    uint32_t *d_min = nullptr, *d_n = nullptr, *d_err = nullptr;
    uint8_t *d_md = nullptr, *d_mt = nullptr, *d_bytes = nullptr;
    uint32_t h_err = 0;
    cudaError_t e = cudaSuccess;
    auto up = [&](auto **dp, const auto *hp, size_t n) {
        using E = std::remove_pointer_t<std::remove_pointer_t<decltype(dp)>>;
        if (e != cudaSuccess) return;
        e = cudaMalloc((void **)dp, sizeof(E) * (n ? n : 1));
        if (e == cudaSuccess && n) e = cudaMemcpy(*dp, hp, sizeof(E) * n, cudaMemcpyHostToDevice);
    };
    up(&d_tbo, c->term_blk_off, (size_t)T + 1);
    up(&d_min, c->blk_min_doc, NB);
    up(&d_n, c->blk_n, NB);
    up(&d_md, c->blk_meta_doc, NB);
    up(&d_mt, c->blk_meta_tf, NB);
    up(&d_doff, c->blk_doc_off, NB);
    up(&d_toff, c->blk_tf_off, NB);
    up(&d_bytes, c->bytes, c->n_bytes);
    up(&d_err, &h_err, 1);
    if (e == cudaSuccess && NB) {
        k_decode_blocks<<<(unsigned)((NB + DEC_WARPS - 1) / DEC_WARPS), DEC_WARPS * 32>>>(
            NB, d_tbo, T, d_min, d_n, d_md, d_mt, d_doff, d_toff, d_bytes, d.post_off, d.fieldnorm, N, d.post, d_err);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = bm25x_index_finish_device(ix);
    uint8_t *d_wfn = nullptr;
    uint32_t *d_wtf = nullptr;
    if (c->blk_wand_fieldnorm && c->blk_wand_tf) {  // the stored per-block bounds must be those of the decoded postings
        up(&d_wfn, c->blk_wand_fieldnorm, NB);
        up(&d_wtf, c->blk_wand_tf, NB);
        if (e == cudaSuccess && NB) {
            k_check_block_wand<<<(unsigned)((NB + 255) / 256), 256>>>(NB, d.blk_off, T, d_wfn, d_wtf, d.s0d, d.s1d, d.blk_ub,
                                                                     d_err);
            e = cudaGetLastError();
        }
    }
    if (e == cudaSuccess && NB > 1) {
        k_check_block_order<<<(unsigned)((NB + 255) / 256), 256>>>(d.blk_off, T, NB, d.blk, d_err);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(&h_err, d_err, sizeof(h_err), cudaMemcpyDeviceToHost);
    cudaFree(d_wfn);
    cudaFree(d_wtf);
    cudaFree(d_tbo);
    cudaFree(d_min);
    cudaFree(d_n);
    cudaFree(d_md);
    cudaFree(d_mt);
    cudaFree(d_doff);
    cudaFree(d_toff);
    cudaFree(d_bytes);
    cudaFree(d_err);
    if (e != cudaSuccess) {
        bm25x_set_error("%s: block upload/decode failed: %s", who, cudaGetErrorString(e));
        bm25x_index_destroy(ix);
        return e == cudaErrorMemoryAllocation ? BM25X_ERR_OOM : BM25X_ERR_CUDA;
    }
    if (h_err & BM25X_BLKERR_RANGE) {
        bm25x_set_error("%s: corrupt blocks (doc ids must be < n_docs and strictly ascending per token, tf != 0)", who);
        bm25x_index_destroy(ix);
        return BM25X_ERR_INVALID;
    }
    if (h_err & BM25X_BLKERR_TF) {
        bm25x_set_error("%s: term frequency >= 2^24 is not supported by the packed posting layout", who);
        bm25x_index_destroy(ix);
        return BM25X_ERR_UNSUPPORTED;
    }
    if (h_err & 8u) {
        bm25x_set_error("%s: corrupt blocks (SummaryTuple wand_fieldnorm/wand_term_frequency is not the block's maximum)", who);
        bm25x_index_destroy(ix);
        return BM25X_ERR_INVALID;
    }
    *out = ix;
    return BM25X_OK;
}

// ---- f3: the growing segment (documents inserted since the last seal, search.rs:83-135) as a second, small index that
// scores with the sealed segment's statistics.  The reference scans these documents one by one per query; here they
// are inverted once (term-major postings over growing ordinals) so that the same kernels unite them. ----
extern "C" int bm25x_growing_create(const bm25x_index *sealed, const bm25x_growing_docs *g, bm25x_index **out) {
    const char *who = "bm25x_growing_create";
    if (!sealed || !g || !out) {
        bm25x_set_error("%s: null argument", who);
        return BM25X_ERR_INVALID;
    }
    *out = nullptr;
    const uint32_t G = g->n_docs, T = sealed->d.n_terms;
    if (!g->elem_off || (g->elem_off[G] && (!g->elem_term || !g->elem_tf))) {
        bm25x_set_error("%s: empty or malformed corpus", who);
        return BM25X_ERR_INVALID;
    }
    int rc = check_common(who, G, g->doc_len ? (const void *)g->doc_len : (const void *)g->doc_fieldnorm, sealed->k1,
                          sealed->b, sealed->device);
    if (rc != BM25X_OK) return rc;
    // validate the documents (vector.rs:39-75: keys strictly ascending, tf != 0)
    int bad = 0;
    for (uint32_t d = 0; d < G; d++) {
        const uint64_t e0 = g->elem_off[d], e1 = g->elem_off[d + 1];
        if (e1 < e0 || e1 > g->elem_off[G]) {
            bad |= 1;
            break;
        }
        if (g->deleted && g->deleted[d]) continue;  // VectorTuple.deleted (search.rs:110)
        bool have_prev = false;
        uint32_t prev = 0;
        for (uint64_t e = e0; e < e1; e++) {
            const uint32_t t = g->elem_term[e], f = g->elem_tf[e];
            if (f == 0) bad |= 1;
            if (t == BM25X_TERM_MISSING) continue;  // token unknown to the sealed segment: never matches (search.rs:60-62)
            if (have_prev && t <= prev) bad |= 1;
            have_prev = true;
            prev = t;
            if (t >= T || sealed->h_df[t] == 0) continue;
            if (f >= (1u << 24)) bad |= 2;
        }
    }
    if (bad & 1) {
        bm25x_set_error("%s: corrupt documents (term ordinals must be strictly ascending per document, tf != 0)", who);
        return BM25X_ERR_INVALID;
    }
    if (bad & 2) {
        bm25x_set_error("%s: term frequency >= 2^24 is not supported by the packed posting layout", who);
        return BM25X_ERR_UNSUPPORTED;
    }
    // invert; doc ids are growing ordinals, deleted documents keep theirs
    std::vector<uint64_t> off;
    std::vector<uint32_t> post_doc, post_tf;
    bm25x_invert_docs(
        G, g->elem_off, g->deleted, g->elem_tf, T,
        [&](uint64_t e) {
            const uint32_t t = g->elem_term[e];
            return t == BM25X_TERM_MISSING || t >= T || sealed->h_df[t] == 0 ? BM25X_TERM_MISSING : t;
        },
        [](uint32_t d) { return d; }, off, post_doc, post_tf);
    std::vector<uint32_t> df(T);
    for (uint32_t t = 0; t < T; t++) df[t] = (uint32_t)(off[(size_t)t + 1] - off[t]);
    const uint64_t P = off[T];
    BuildMeta m{G, T, g->doc_len, g->payload, sealed->h_keys.empty() ? nullptr : sealed->h_keys.data(), sealed->k1,
                sealed->b, df.data(), P};
    m.fieldnorm = g->doc_fieldnorm;
    m.stat_df = sealed->h_df.data();
    m.stat_n_docs = sealed->d.n_docs;
    m.stat_avgdl = sealed->avgdl;
    bm25x_index *ix = nullptr;
    rc = bm25x_index_begin(m, sealed->device, &ix);
    if (rc != BM25X_OK) return rc;
    rc = upload_csr(ix, who, T, P, off.data(), post_doc.data(), post_tf.data());
    if (rc != BM25X_OK) return rc;
    ix->prune = sealed->prune;
    ix->growing = true;
    *out = ix;
    return BM25X_OK;
}

extern "C" void bm25x_index_destroy(bm25x_index *ix) {
    if (!ix) return;
    cudaSetDevice(ix->device);
    if (ix->stream) cudaStreamSynchronize(ix->stream);
    for (void *p : ix->allocs) cudaFree(p);
    if (ix->h_stage) cudaFreeHost(ix->h_stage);
    if (ix->h_stage_free) cudaEventDestroy(ix->h_stage_free);
    if (ix->copy_stream) cudaStreamDestroy(ix->copy_stream);
    if (ix->stream) cudaStreamDestroy(ix->stream);
    delete ix;
}

extern "C" int bm25x_index_get_info(const bm25x_index *ix, bm25x_index_info *out) {
    if (!ix || !out) {
        bm25x_set_error("bm25x_index_get_info: null argument");
        return BM25X_ERR_INVALID;
    }
    out->n_docs = ix->d.n_docs;
    out->n_terms = ix->d.n_terms;
    out->n_postings = ix->d.n_post;
    out->sum_doc_len = ix->sum_len;
    out->avgdl = ix->avgdl;
    out->k1 = ix->k1;
    out->b = ix->b;
    out->device_bytes = ix->device_bytes;
    out->n_blocks = ix->d.n_blocks;
    out->device = ix->device;
    return BM25X_OK;
}

// ---- replication: expose / adopt the device arrays (the bytes travel by NCCL in the caller) ----
static void layout_arrays(const bm25x_index *ix, void **ptr, uint64_t *bytes) {
    const DeviceIndex &d = ix->d;
    const uint64_t T = d.n_terms, N = d.n_docs;
    void *p[BM25X_N_ARRAYS] = {d.post, d.post_off, d.df, d.blk_off, d.blk, d.s0f, d.s0d, d.s1d, d.s1f, d.fieldnorm, d.payload,
                               d.ubd, d.blk_ub};
    uint64_t b[BM25X_N_ARRAYS] = {sizeof(Posting) * (d.n_post_pad + BM25X_POST_SLACK), 8 * (T + 1), 4 * (T ? T : 1), 8 * (T + 1),
                                  8 * (d.n_blocks ? d.n_blocks : 1), 4 * (T ? T : 1), 8 * (T ? T : 1), 8 * 256, 4 * 256,
                                  N, 6 * N, 8 * (T ? T : 1), 4 * (d.n_blocks ? d.n_blocks : 1)};
    for (int i = 0; i < BM25X_N_ARRAYS; i++) {
        ptr[i] = p[i];
        bytes[i] = b[i];
    }
}

extern "C" int bm25x_index_get_layout(const bm25x_index *ix, bm25x_index_layout *out) {
    if (!ix || !out) {
        bm25x_set_error("bm25x_index_get_layout: null argument");
        return BM25X_ERR_INVALID;
    }
    out->n_docs = ix->d.n_docs;
    out->n_terms = ix->d.n_terms;
    out->n_postings = ix->d.n_post;
    out->n_postings_padded = ix->d.n_post_pad;
    out->n_blocks = ix->d.n_blocks;
    out->sum_doc_len = ix->sum_len;
    out->k1 = ix->k1;
    out->b = ix->b;
    out->avgdl = ix->avgdl;
    out->device = ix->device;
    layout_arrays(ix, out->dev_ptr, out->bytes);
    return BM25X_OK;
}

extern "C" int bm25x_index_alloc_replica(const bm25x_index_layout *like, int device, bm25x_index **out) {
    if (!like || !out) {
        bm25x_set_error("bm25x_index_alloc_replica: null argument");
        return BM25X_ERR_INVALID;
    }
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
        cudaGetLastError();
        bm25x_set_error("bm25x_index_alloc_replica: CUDA device %d not available; there is no CPU fallback", device);
        return BM25X_ERR_CUDA;
    }
    bm25x_index *ix = new bm25x_index();
    apply_env_options(ix);
    ix->device = device;
    ix->k1 = like->k1;
    ix->b = like->b;
    ix->avgdl = like->avgdl;
    ix->sum_len = like->sum_doc_len;
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        bm25x_set_error("bm25x_index_alloc_replica: device %d is sm_%d%d; this library only carries sm_100a kernels", device,
                        prop.major, prop.minor);
        bm25x_index_destroy(ix);
        return BM25X_ERR_CUDA;
    }
    ix->sm_count = prop.multiProcessorCount;
    CU(cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking));
    {
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            uint64_t thr = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        }
    }
    DeviceIndex &d = ix->d;
    d.n_docs = like->n_docs;
    d.n_terms = like->n_terms;
    d.n_post = like->n_postings;
    d.n_post_pad = like->n_postings_padded;
    d.n_blocks = like->n_blocks;
    const size_t T = d.n_terms, N = d.n_docs;
    TRY(dev_alloc(ix, &d.post, d.n_post_pad + BM25X_POST_SLACK));
    TRY(dev_alloc(ix, &d.pdoc, d.n_post_pad + BM25X_POST_SLACK));
    TRY(dev_alloc(ix, &d.post_off, T + 1));
    TRY(dev_alloc(ix, &d.df, T));
    TRY(dev_alloc(ix, &d.blk_off, T + 1));
    TRY(dev_alloc(ix, &d.blk, d.n_blocks));
    TRY(dev_alloc(ix, &d.blk_ub, d.n_blocks));
    TRY(dev_alloc(ix, &d.s0f, T));
    TRY(dev_alloc(ix, &d.s0d, T));
    TRY(dev_alloc(ix, &d.s1d, 256));
    TRY(dev_alloc(ix, &d.s1f, 256));
    TRY(dev_alloc(ix, &d.fieldnorm, N));
    TRY(dev_alloc(ix, &d.payload, N * 3));
    TRY(dev_alloc(ix, &d.ubd, T));
    *out = ix;
    return BM25X_OK;
}

extern "C" int bm25x_index_finalize_replica(bm25x_index *ix) {
    if (!ix) {
        bm25x_set_error("bm25x_index_finalize_replica: null argument");
        return BM25X_ERR_INVALID;
    }
    BM25X_CUDA_TRY(cudaSetDevice(ix->device));
    // derived data that does not travel: the doc-id-only copy of the postings
    k_extract_docs<<<148 * 8, 256>>>(ix->d.post, ix->d.n_post_pad + BM25X_POST_SLACK, ix->d.pdoc);
    BM25X_CUDA_TRY(cudaGetLastError());
    BM25X_CUDA_TRY(cudaDeviceSynchronize());
    ix->h_df.resize(ix->d.n_terms);
    if (ix->d.n_terms)
        BM25X_CUDA_TRY(cudaMemcpy(ix->h_df.data(), ix->d.df, sizeof(uint32_t) * ix->d.n_terms, cudaMemcpyDeviceToHost));
    if (!ix->d.champ) BM25X_CUDA_TRY(build_champions(ix));  // derived data: built here from the replicated arrays
    {   // s1f_min from the replicated arrays (see bm25x_index_begin)
        std::vector<uint8_t> h_fn(ix->d.n_docs);
        float h_s1f[256];
        BM25X_CUDA_TRY(cudaMemcpy(h_fn.data(), ix->d.fieldnorm, ix->d.n_docs, cudaMemcpyDeviceToHost));
        BM25X_CUDA_TRY(cudaMemcpy(h_s1f, ix->d.s1f, sizeof(h_s1f), cudaMemcpyDeviceToHost));
        bool seen[256] = {false};
        for (uint32_t d = 0; d < ix->d.n_docs; d++) seen[h_fn[d]] = true;
        float mn = 3.0e38f;
        for (int f = 0; f < 256; f++)
            if (seen[f] && h_s1f[f] < mn) mn = h_s1f[f];
        ix->s1f_min = mn;
    }
    return BM25X_OK;
}

extern "C" int bm25x_index_set_option(bm25x_index *ix, const char *name, int64_t value) {
    if (!ix || !name) {
        bm25x_set_error("bm25x_index_set_option: null argument");
        return BM25X_ERR_INVALID;
    }
    if (strcmp(name, "prune") == 0) {
        ix->prune = value != 0;
        return BM25X_OK;
    }
    if (strcmp(name, "seed") == 0) {  // 2..4-term classes: pools seeded from the champion lists, doc-id-only stream
        ix->seed = value != 0;
        return BM25X_OK;
    }
    if (strcmp(name, "seed_prune_min") == 0) {  // seeded launches: list length from which a skewed query goes to the pruning kernel
        ix->seed_prune_min = value < 0 ? 0u : (value > 0xFFFFFFFFll ? 0xFFFFFFFFu : (uint32_t)value);
        return BM25X_OK;
    }
    if (strcmp(name, "slice_min") == 0) {  // bm25x_search_batch: queries per slice of a pipelined call (0: one piece)
        ix->slice_min = value < 0 ? 0u : (value > 0xFFFFFFFFll ? 0xFFFFFFFFu : (uint32_t)value);
        return BM25X_OK;
    }
    if (strcmp(name, "seed_dense_div") == 0) {  // seeded launches: lists of n_docs / this or more go to the plain kernel (0: never)
        ix->seed_dense_div = value < 0 ? 0u : (value > 0xFFFFFFFFll ? 0xFFFFFFFFu : (uint32_t)value);
        return BM25X_OK;
    }
    if (strcmp(name, "seed_max_terms") == 0) {  // widest term-count class that runs seeded: 4 or 8
        ix->seed_max_terms = value >= 8 ? 8 : 4;
        return BM25X_OK;
    }
    if (strcmp(name, "twophase") == 0) {  // 2..4-term classes: 8-byte postings first, doc ids only once no posting passes alone
        ix->twophase = value != 0;
        return BM25X_OK;
    }
    bm25x_set_error("bm25x_index_set_option: unknown option '%s'", name);
    return BM25X_ERR_INVALID;
}

extern "C" int bm25x_index_get_df(const bm25x_index *ix, uint32_t *df_out) {
    if (!ix || (!df_out && ix->d.n_terms)) {
        bm25x_set_error("bm25x_index_get_df: null argument");
        return BM25X_ERR_INVALID;
    }
    if (ix->h_df.size() != ix->d.n_terms) {
        bm25x_set_error("bm25x_index_get_df: replica not finalized");
        return BM25X_ERR_INVALID;
    }
    memcpy(df_out, ix->h_df.data(), sizeof(uint32_t) * ix->d.n_terms);
    return BM25X_OK;
}

// address_tokens::read (crates/bm25/src/address_tokens.rs:61-98) over the sorted key array.
extern "C" int bm25x_lookup_terms(const bm25x_index *ix, const uint8_t *keys, uint32_t n, uint32_t *out) {
    if (!ix || (!keys && n) || (!out && n)) {
        bm25x_set_error("bm25x_lookup_terms: null argument");
        return BM25X_ERR_INVALID;
    }
    if (ix->h_keys.empty() && ix->d.n_terms) {
        bm25x_set_error("bm25x_lookup_terms: index was created without term keys");
        return BM25X_ERR_INVALID;
    }
    const uint8_t *base = ix->h_keys.data();
    for (uint32_t i = 0; i < n; i++) {
        const uint8_t *key = keys + (size_t)i * 16;
        uint32_t lo = 0, hi = ix->d.n_terms;
        while (lo < hi) {
            uint32_t mid = (lo + hi) >> 1;
            if (memcmp(base + (size_t)mid * 16, key, 16) < 0) lo = mid + 1;
            else hi = mid;
        }
        out[i] = (lo < ix->d.n_terms && memcmp(base + (size_t)lo * 16, key, 16) == 0) ? lo : BM25X_TERM_MISSING;
    }
    return BM25X_OK;
}
