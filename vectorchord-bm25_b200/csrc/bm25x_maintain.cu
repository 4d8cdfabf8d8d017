// bm25x_maintain.cu — the write side of the freshness model: bm25::maintain (crates/bm25/src/maintain.rs:27-311) folds
// the growing documents and the delete marks into a NEW sealed index, bm25::bulkdelete (bulkdelete.rs:20-112) sets the
// delete marks from a list of dead heap tuples.  DESIGN.md §4.7.
//
// Rule of the device path: arrays with one entry per posting never cross PCIe.  Per-document (N), per-term (T) arrays
// and the growing elements do; the sealed postings are relabelled and compacted in HBM, straight into the new handle.
#include <string.h>

#include <algorithm>
#include <chrono>

#include "bm25x_common.h"

#define MT_THREADS 256
#define MT_ITEMS 16                          // documents / postings per thread (4 aligned groups of 4 postings)
#define MT_TILE (MT_THREADS * MT_ITEMS)      // documents / postings per block

// Exclusive scan of one value per thread across the block (MT_THREADS threads); *total = the block's sum.
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t *total) {
    __shared__ uint32_t ws[MT_THREADS / 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t x = v;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) ws[wid] = x;
    __syncthreads();
    if (wid == 0) {
        uint32_t s = lane < MT_THREADS / 32 ? ws[lane] : 0u;
        for (int o = 1; o < MT_THREADS / 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, s, o);
            if (lane >= o) s += y;
        }
        if (lane < MT_THREADS / 32) ws[lane] = s;
    }
    __syncthreads();
    const uint32_t before = wid ? ws[wid - 1] : 0u;
    *total = ws[MT_THREADS / 32 - 1];
    __syncthreads();
    return before + x - v;
}

// In-place exclusive scan of the per-tile counts v[0..n), v[n] = the total.  One block; the tiles are few (n_post / 4096).
__global__ void __launch_bounds__(1024) k_mt_scan_tiles(uint64_t *__restrict__ v, uint64_t n) {
    __shared__ uint64_t ws[32];
    __shared__ uint64_t carry;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint64_t base = 0; base < n; base += 1024) {
        const uint64_t i = base + threadIdx.x;
        const uint64_t x0 = i < n ? v[i] : 0;
        uint64_t x = x0;
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) ws[wid] = x;
        __syncthreads();
        if (wid == 0) {
            uint64_t s = ws[lane];
            for (int o = 1; o < 32; o <<= 1) {
                const uint64_t y = __shfl_up_sync(0xFFFFFFFFu, s, o);
                if (lane >= o) s += y;
            }
            ws[lane] = s;
        }
        __syncthreads();
        const uint64_t incl = carry + (wid ? ws[wid - 1] : 0) + x;
        if (i < n) v[i] = incl - x0;
        __syncthreads();
        if (threadIdx.x == 1023) carry = incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) v[n] = carry;
}

// ---- 1. survivor relabel: relabel[d] = number of surviving documents before d, BM25X_DOC_NONE for a deleted one ----
__device__ __forceinline__ uint32_t mt_alive_docs(const uint8_t *__restrict__ del, uint32_t N, uint64_t d0) {
    uint32_t c = 0;
    for (int i = 0; i < MT_ITEMS; i++) c += (d0 + i < N && !del[d0 + i]) ? 1u : 0u;
    return c;
}

__global__ void __launch_bounds__(MT_THREADS) k_mt_alive_count(const uint8_t *__restrict__ del, uint32_t N,
                                                               uint64_t *__restrict__ tile_cnt) {
    const uint64_t d0 = (uint64_t)blockIdx.x * MT_TILE + threadIdx.x * MT_ITEMS;
    uint32_t total;
    block_excl_scan(mt_alive_docs(del, N, d0), &total);
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = total;
}

__global__ void __launch_bounds__(MT_THREADS) k_mt_relabel(const uint8_t *__restrict__ del, uint32_t N,
                                                           const uint64_t *__restrict__ tile_pref,
                                                           uint32_t *__restrict__ relabel) {
    const uint64_t d0 = (uint64_t)blockIdx.x * MT_TILE + threadIdx.x * MT_ITEMS;
    uint32_t total;
    uint32_t r = (uint32_t)tile_pref[blockIdx.x] + block_excl_scan(mt_alive_docs(del, N, d0), &total);
    for (int i = 0; i < MT_ITEMS && d0 + i < N; i++) relabel[d0 + i] = del[d0 + i] ? BM25X_DOC_NONE : r++;
}

// Terms of the postings [p0, p0 + MT_ITEMS) of every thread: the block finds the terms of its tile's first and last
// posting, each thread narrows that range to its own first posting.  Last t with off_pad[t] <= p (empty terms share
// their start with the next one, so this is the term that holds p).
__device__ __forceinline__ uint32_t mt_term_of(const uint64_t *__restrict__ off_pad, uint32_t T, uint64_t n_pad,
                                               uint64_t p0) {
    __shared__ uint32_t range[2];
    auto search = [&](uint64_t p, uint32_t lo, uint32_t hi) {
        while (lo < hi) {
            const uint32_t mid = (lo + hi + 1) >> 1;
            if (off_pad[mid] <= p) lo = mid;
            else hi = mid - 1;
        }
        return lo;
    };
    const uint64_t tile0 = (uint64_t)blockIdx.x * MT_TILE;
    if (threadIdx.x == 0) range[0] = search(tile0, 0, T - 1);
    if (threadIdx.x == 1) range[1] = search((tile0 + MT_TILE < n_pad ? tile0 + MT_TILE : n_pad) - 1, 0, T - 1);
    __syncthreads();
    return p0 < n_pad ? search(p0, range[0], range[1]) : 0u;
}

// ---- 2 + 3. per-document posting counts of the survivors (their new length, maintain.rs:356-360), per-term survivor
// counts, per-tile survivor counts.  pdoc is read in 16-byte groups: a group never straddles two terms
// (BM25X_POST_ALIGN), pad slots read BM25X_DOC_INF and count as dead. ----
__global__ void __launch_bounds__(MT_THREADS) k_mt_post_count(const uint32_t *__restrict__ pdoc, uint64_t n_pad,
                                                              const uint8_t *__restrict__ del,
                                                              const uint64_t *__restrict__ off_pad, uint32_t T,
                                                              uint32_t *__restrict__ doc_cnt,
                                                              uint32_t *__restrict__ term_cnt,
                                                              uint64_t *__restrict__ tile_cnt) {
    const uint64_t p0 = (uint64_t)blockIdx.x * MT_TILE + threadIdx.x * MT_ITEMS;
    uint32_t t = mt_term_of(off_pad, T, n_pad, p0);
    const uint32_t t_first = t;
    uint32_t c_all = 0, c_first = 0;
    for (int gq = 0; gq < MT_ITEMS / 4; gq++) {
        const uint64_t p = p0 + 4 * gq;
        if (p >= n_pad) break;
        while (t + 1 < T && off_pad[t + 1] <= p) t++;
        const uint4 q = *reinterpret_cast<const uint4 *>(pdoc + p);
        const uint32_t ds[4] = {q.x, q.y, q.z, q.w};
        uint32_t c = 0;
        for (int j = 0; j < 4; j++)
            if (ds[j] != BM25X_DOC_INF && !del[ds[j]]) {
                atomicAdd(&doc_cnt[ds[j]], 1u);
                c++;
            }
        c_all += c;
        if (t == t_first) c_first += c;
        else if (c) atomicAdd(&term_cnt[t], c);
    }
    // most threads of a warp hold postings of one term: one atomic per term and warp for the first run
    const uint32_t key = p0 < n_pad ? t_first : 0xFFFFFFFFu;
    const uint32_t peers = __match_any_sync(0xFFFFFFFFu, key);
    const uint32_t sum = __reduce_add_sync(peers, c_first);
    if (key != 0xFFFFFFFFu && sum && (threadIdx.x & 31) == (uint32_t)(__ffs(peers) - 1)) atomicAdd(&term_cnt[key], sum);
    uint32_t total;
    block_excl_scan(c_all, &total);
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = total;
}

// ---- 4. order-preserving compaction of the sealed postings into the new handle.  S = the survivor's rank among all
// surviving postings (tile prefix + block scan); its slot is S + base[t] with base[t] = new_off[t'] - (survivors of the
// terms before t), i.e. new_off[t'] + rank within the term.  New doc id, same tf, the NEW document's fieldnorm. ----
__global__ void __launch_bounds__(MT_THREADS) k_mt_compact(const Posting *__restrict__ post, uint64_t n_pad,
                                                           const uint8_t *__restrict__ del,
                                                           const uint32_t *__restrict__ relabel,
                                                           const uint8_t *__restrict__ fn_new,
                                                           const uint64_t *__restrict__ off_pad, uint32_t T,
                                                           const uint64_t *__restrict__ tile_pref,
                                                           const uint64_t *__restrict__ base, Posting *__restrict__ out) {
    const uint64_t p0 = (uint64_t)blockIdx.x * MT_TILE + threadIdx.x * MT_ITEMS;
    uint32_t t = mt_term_of(off_pad, T, n_pad, p0);
    Posting v[MT_ITEMS];
    uint32_t alive = 0;
    for (int gq = 0; gq < MT_ITEMS / 4; gq++) {
        const uint64_t p = p0 + 4 * gq;
        if (p >= n_pad) break;
        const uint4 *src = reinterpret_cast<const uint4 *>(post + p);
        for (int h = 0; h < 2; h++) {
            const uint4 q = src[h];
            v[4 * gq + 2 * h] = Posting{q.x, q.y};
            v[4 * gq + 2 * h + 1] = Posting{q.z, q.w};
        }
        for (int j = 0; j < 4; j++) {
            const uint32_t d = v[4 * gq + j].doc;
            if (d != BM25X_DOC_INF && !del[d]) alive |= 1u << (4 * gq + j);
        }
    }
    uint32_t total;
    uint64_t s = tile_pref[blockIdx.x] + block_excl_scan(__popc(alive), &total);
    for (int gq = 0; gq < MT_ITEMS / 4; gq++) {
        const uint64_t p = p0 + 4 * gq;
        if (p >= n_pad) break;
        while (t + 1 < T && off_pad[t + 1] <= p) t++;
        const uint64_t b = base[t];
        for (int j = 0; j < 4; j++) {
            const int i = 4 * gq + j;
            if (!((alive >> i) & 1u)) continue;
            const uint32_t nd = relabel[v[i].doc];
            out[s + b] = Posting{nd, (v[i].w & 0xFFFFFF00u) | fn_new[nd]};
            s++;
        }
    }
}

// ---- 6. bulkdelete: hit[d] = payload(d) is in the sorted dead list ----
__device__ __forceinline__ uint64_t mt_ctid(const uint16_t *__restrict__ p) {
    return (uint64_t)p[0] << 32 | (uint64_t)p[1] << 16 | (uint64_t)p[2];
}

__global__ void k_mt_bulkdelete(const uint16_t *__restrict__ payload, uint32_t N, const uint16_t *__restrict__ dead,
                                uint64_t n_dead, uint8_t *__restrict__ hit) {
    const uint64_t d = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= N) return;
    const uint64_t key = mt_ctid(payload + 3 * d);
    uint64_t lo = 0, hi = n_dead;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (mt_ctid(dead + 3 * mid) < key) lo = mid + 1;
        else hi = mid;
    }
    hit[d] = lo < n_dead && mt_ctid(dead + 3 * lo) == key;
}

// ---- host side ----

namespace {

// Device scratch of one call, freed on every return path.
struct Scratch {
    std::vector<void *> p;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    ~Scratch() {
        for (void *x : p) cudaFree(x);
        for (cudaEvent_t e : ev)
            if (e) cudaEventDestroy(e);
    }
    template <typename T>
    cudaError_t alloc(T **q, size_t n) {
        cudaError_t e = cudaMalloc((void **)q, sizeof(T) * (n ? n : 1));
        if (e == cudaSuccess) p.push_back((void *)*q);
        return e;
    }
};

int cuda_fail(const char *who, cudaError_t e) {
    bm25x_set_error("%s: %s", who, cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? BM25X_ERR_OOM : BM25X_ERR_CUDA;
}

// Lower bound of a 16-byte key in a sorted key table of n keys.
uint32_t key_lower_bound(const uint8_t *table, uint32_t n, const uint8_t *key) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (memcmp(table + (size_t)mid * 16, key, 16) < 0) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

uint32_t key_find(const uint8_t *table, uint32_t n, const uint8_t *key) {
    const uint32_t i = key_lower_bound(table, n, key);
    return i < n && memcmp(table + (size_t)i * 16, key, 16) == 0 ? i : BM25X_TERM_MISSING;
}

}  // namespace

#define MT_CU(x)                                 \
    do {                                         \
        cudaError_t _e = (x);                    \
        if (_e != cudaSuccess) {                 \
            if (nix) bm25x_index_destroy(nix);   \
            return cuda_fail(who, _e);           \
        }                                        \
    } while (0)

extern "C" int bm25x_index_maintain(const bm25x_index *sealed, const uint8_t *sealed_deleted, const bm25x_vectors *docs,
                                    bm25x_index **out, uint32_t *relabel_out, bm25x_maintain_stats *stats) {
    const char *who = "bm25x_index_maintain";
    const auto t_start = std::chrono::steady_clock::now();
    if (!sealed || !out) {
        bm25x_set_error("%s: null argument", who);
        return BM25X_ERR_INVALID;
    }
    *out = nullptr;
    if (sealed->growing) {
        bm25x_set_error("%s: a growing handle is not a sealed index (maintain the sealed index, pass the growing "
                        "documents as docs)", who);
        return BM25X_ERR_INVALID;
    }
    if (sealed->h_df.size() != sealed->d.n_terms) {
        bm25x_set_error("%s: replica not finalized", who);
        return BM25X_ERR_INVALID;
    }
    const uint32_t N = sealed->d.n_docs, T = sealed->d.n_terms;
    const bool keyed = !sealed->h_keys.empty();
    const uint8_t *old_keys = sealed->h_keys.data();

    // ---- the growing documents must be what Document::new accepts (vector.rs:39-75) ----
    const uint32_t G = docs ? docs->n_docs : 0;
    const uint64_t n_elem = docs && docs->elem_off ? docs->elem_off[G] : 0;
    if (docs) {
        if (!docs->elem_off || (n_elem && !docs->elem_tf)) {
            bm25x_set_error("%s: malformed documents (elem_off / elem_tf missing)", who);
            return BM25X_ERR_INVALID;
        }
        if (docs->elem_key && docs->elem_term) {
            bm25x_set_error("%s: give exactly one of elem_key / elem_term", who);
            return BM25X_ERR_INVALID;
        }
        if (docs->elem_key && !keyed) {
            bm25x_set_error("%s: term keys given, but the sealed index has none (give elem_term)", who);
            return BM25X_ERR_INVALID;
        }
        if (docs->elem_term && keyed) {
            bm25x_set_error("%s: term ordinals given, but the sealed index has term keys (give elem_key)", who);
            return BM25X_ERR_INVALID;
        }
        if (n_elem && !docs->elem_key && !docs->elem_term) {
            bm25x_set_error("%s: documents without elem_key / elem_term", who);
            return BM25X_ERR_INVALID;
        }
        int bad = 0;  // 1 = order / ranges / tf == 0, 2 = tf too large, 4 = BM25X_TERM_MISSING used as an ordinal
        for (uint32_t d = 0; d < G && !(bad & 1); d++) {
            const uint64_t e0 = docs->elem_off[d], e1 = docs->elem_off[d + 1];
            if (e1 < e0 || e1 > n_elem) {
                bad |= 1;
                break;
            }
            for (uint64_t e = e0; e < e1; e++) {
                const uint32_t f = docs->elem_tf[e];
                if (f == 0) bad |= 1;
                if (f >= (1u << 24)) bad |= 2;
                if (keyed) {
                    if (e > e0 && memcmp(docs->elem_key + (e - 1) * 16, docs->elem_key + e * 16, 16) >= 0) bad |= 1;
                } else {
                    if (docs->elem_term[e] == BM25X_TERM_MISSING) bad |= 4;
                    if (e > e0 && docs->elem_term[e - 1] >= docs->elem_term[e]) bad |= 1;
                }
            }
        }
        if (bad & 4) {
            bm25x_set_error("%s: BM25X_TERM_MISSING is not a term ordinal (every element of a document is a token)", who);
            return BM25X_ERR_INVALID;
        }
        if (bad & 1) {
            bm25x_set_error("%s: corrupt documents (term keys / ordinals must be strictly ascending per document, "
                            "tf != 0)", who);
            return BM25X_ERR_INVALID;
        }
        if (bad & 2) {
            bm25x_set_error("%s: term frequency >= 2^24 is not supported by the packed posting layout", who);
            return BM25X_ERR_UNSUPPORTED;
        }
    }
    const uint8_t *g_del = docs ? docs->deleted : nullptr;

    // ---- new document order (maintain.rs:55-73, io.rs:52-60): sealed survivors by doc id, then growing survivors ----
    uint32_t n_sealed_alive = 0, n_new = 0;
    for (uint32_t d = 0; d < N; d++) n_sealed_alive += !(sealed_deleted && sealed_deleted[d]);
    std::vector<uint32_t> grow_new(G, BM25X_DOC_NONE);
    n_new = n_sealed_alive;
    for (uint32_t g = 0; g < G; g++)
        if (!(g_del && g_del[g])) {
            if (n_new == BM25X_DOC_INF - 1) {
                bm25x_set_error("%s: more than 2^32 - 2 documents", who);
                return BM25X_ERR_INVALID;
            }
            grow_new[g] = n_new++;
        }
    if (n_new == 0) {
        bm25x_set_error("%s: no document survives (an index cannot be empty)", who);
        return BM25X_ERR_INVALID;
    }

    bm25x_index *nix = nullptr;
    Scratch s;
    uint64_t h2d = 0, d2h = 0;
    MT_CU(cudaSetDevice(sealed->device));
    MT_CU(cudaEventCreate(&s.ev[0]));
    MT_CU(cudaEventCreate(&s.ev[1]));
    MT_CU(cudaEventRecord(s.ev[0], 0));

    // ---- device pass over the sealed segment: relabel, per-doc / per-term / per-tile survivor counts ----
    const DeviceIndex &od = sealed->d;
    const uint64_t n_pad = od.n_post_pad;
    const uint64_t n_rt = ((uint64_t)N + MT_TILE - 1) / MT_TILE, n_pt = std::max<uint64_t>(1, (n_pad + MT_TILE - 1) / MT_TILE);
    uint8_t *d_del = nullptr;
    uint32_t *d_relabel = nullptr, *d_doc_cnt = nullptr, *d_term_cnt = nullptr;
    uint64_t *d_rtile = nullptr, *d_ptile = nullptr;
    MT_CU(s.alloc(&d_del, N));
    MT_CU(s.alloc(&d_relabel, N));
    MT_CU(s.alloc(&d_doc_cnt, N));
    MT_CU(s.alloc(&d_term_cnt, T));
    MT_CU(s.alloc(&d_rtile, n_rt + 1));
    MT_CU(s.alloc(&d_ptile, n_pt + 1));
    if (sealed_deleted) {
        MT_CU(cudaMemcpy(d_del, sealed_deleted, N, cudaMemcpyHostToDevice));
        h2d += N;
    } else {
        MT_CU(cudaMemset(d_del, 0, N));
    }
    MT_CU(cudaMemset(d_doc_cnt, 0, sizeof(uint32_t) * N));
    MT_CU(cudaMemset(d_term_cnt, 0, sizeof(uint32_t) * (T ? T : 1)));
    k_mt_alive_count<<<(unsigned)n_rt, MT_THREADS>>>(d_del, N, d_rtile);
    k_mt_scan_tiles<<<1, 1024>>>(d_rtile, n_rt);
    k_mt_relabel<<<(unsigned)n_rt, MT_THREADS>>>(d_del, N, d_rtile, d_relabel);
    if (T) k_mt_post_count<<<(unsigned)n_pt, MT_THREADS>>>(od.pdoc, n_pad, d_del, od.post_off, T, d_doc_cnt, d_term_cnt, d_ptile);
    else MT_CU(cudaMemset(d_ptile, 0, sizeof(uint64_t) * (n_pt + 1)));
    k_mt_scan_tiles<<<1, 1024>>>(d_ptile, n_pt);
    MT_CU(cudaGetLastError());
    std::vector<uint32_t> term_cnt(T), doc_cnt(N);
    std::vector<uint16_t> old_pl((size_t)N * 3);
    if (T) MT_CU(cudaMemcpy(term_cnt.data(), d_term_cnt, sizeof(uint32_t) * T, cudaMemcpyDeviceToHost));
    MT_CU(cudaMemcpy(doc_cnt.data(), d_doc_cnt, sizeof(uint32_t) * N, cudaMemcpyDeviceToHost));
    MT_CU(cudaMemcpy(old_pl.data(), od.payload, sizeof(uint16_t) * 3 * (size_t)N, cudaMemcpyDeviceToHost));
    d2h += 4ull * T + 4ull * N + 6ull * N;
    if (relabel_out) {
        MT_CU(cudaMemcpy(relabel_out, d_relabel, sizeof(uint32_t) * N, cudaMemcpyDeviceToHost));
        d2h += 4ull * N;
        for (uint32_t g = 0; g < G; g++) relabel_out[(size_t)N + g] = grow_new[g];
    }

    // ---- new documents: length (maintain.rs:337,356-360 for sealed survivors = their number of postings; vector.rs:77-83
    // saturating Σ tf for growing ones) and payload ----
    std::vector<uint32_t> new_len(n_new);
    std::vector<uint16_t> new_pl((size_t)n_new * 3);
    {
        uint32_t r = 0;
        for (uint32_t d = 0; d < N; d++) {
            if (sealed_deleted && sealed_deleted[d]) continue;
            new_len[r] = doc_cnt[d];
            memcpy(&new_pl[(size_t)r * 3], &old_pl[(size_t)d * 3], 6);
            r++;
        }
        for (uint32_t g = 0; g < G; g++) {
            if (grow_new[g] == BM25X_DOC_NONE) continue;
            uint64_t len = 0;
            for (uint64_t e = docs->elem_off[g]; e < docs->elem_off[g + 1]; e++) len += docs->elem_tf[e];
            new_len[r] = (uint32_t)std::min<uint64_t>(len, 0xFFFFFFFFull);
            if (docs->payload) memcpy(&new_pl[(size_t)r * 3], docs->payload + (size_t)g * 3, 6);
            else bm25x_synthetic_ctid(g, &new_pl[(size_t)r * 3]);
            r++;
        }
    }

    // ---- new token set (io.rs locally_merge, flush.rs): tokens with at least one posting, ascending; growing-only
    // tokens are new terms.  Keyless: ordinals stay, the vocabulary grows to the largest ordinal + 1. ----
    std::vector<uint32_t> old_to_new(T);
    std::vector<uint8_t> new_keys;
    uint32_t T_new = T;
    if (keyed) {
        std::vector<uint32_t> g_cnt(T, 0);
        std::vector<const uint8_t *> unknown;
        for (uint32_t g = 0; g < G; g++) {
            if (grow_new[g] == BM25X_DOC_NONE) continue;
            for (uint64_t e = docs->elem_off[g]; e < docs->elem_off[g + 1]; e++) {
                const uint8_t *k = docs->elem_key + e * 16;
                const uint32_t t = key_find(old_keys, T, k);
                if (t != BM25X_TERM_MISSING) g_cnt[t]++;
                else unknown.push_back(k);
            }
        }
        auto less = [](const uint8_t *a, const uint8_t *b) { return memcmp(a, b, 16) < 0; };
        std::sort(unknown.begin(), unknown.end(), less);
        unknown.erase(std::unique(unknown.begin(), unknown.end(),
                                  [](const uint8_t *a, const uint8_t *b) { return memcmp(a, b, 16) == 0; }),
                      unknown.end());
        new_keys.reserve(((size_t)T + unknown.size()) * 16);
        size_t j = 0;
        for (uint32_t t = 0; t <= T; t++) {
            while (j < unknown.size() && (t == T || less(unknown[j], old_keys + (size_t)t * 16)))
                new_keys.insert(new_keys.end(), unknown[j], unknown[j] + 16), j++;
            if (t == T) break;
            old_to_new[t] = BM25X_TERM_MISSING;
            if (term_cnt[t] + g_cnt[t] == 0) continue;  // every posting of the token died
            old_to_new[t] = (uint32_t)(new_keys.size() / 16);
            new_keys.insert(new_keys.end(), old_keys + (size_t)t * 16, old_keys + (size_t)t * 16 + 16);
        }
        T_new = (uint32_t)(new_keys.size() / 16);
    } else {
        for (uint32_t t = 0; t < T; t++) old_to_new[t] = t;
        for (uint32_t g = 0; g < G; g++)
            if (grow_new[g] != BM25X_DOC_NONE && docs->elem_off[g + 1] > docs->elem_off[g])
                T_new = std::max(T_new, docs->elem_term[docs->elem_off[g + 1] - 1] + 1);  // ascending: the last is the largest
    }

    // growing postings, term-major over the new ordinals (the inversion bm25x_growing_create uses)
    std::vector<uint64_t> g_off;
    std::vector<uint32_t> g_doc, g_tf;
    const uint8_t *nk = new_keys.data();
    bm25x_invert_docs(
        G, docs ? docs->elem_off : nullptr, g_del, docs ? docs->elem_tf : nullptr, T_new,
        [&](uint64_t e) { return keyed ? key_find(nk, T_new, docs->elem_key + e * 16) : docs->elem_term[e]; },
        [&](uint32_t g) { return grow_new[g]; }, g_off, g_doc, g_tf);
    const uint64_t P_g = g_off[T_new];

    // df, padded offsets (as bm25x_index_begin lays them out), destinations of both parts
    std::vector<uint32_t> df(T_new), s_cnt(T_new, 0);
    for (uint32_t t = 0; t < T; t++)
        if (old_to_new[t] != BM25X_TERM_MISSING) s_cnt[old_to_new[t]] = term_cnt[t];
    uint64_t P_new = 0;
    std::vector<uint64_t> off_pad(T_new), g_dst(T_new ? T_new : 1), base(T ? T : 1, 0);
    {
        uint64_t pp = 0;
        for (uint32_t t = 0; t < T_new; t++) {
            df[t] = s_cnt[t] + (uint32_t)(g_off[(size_t)t + 1] - g_off[t]);
            P_new += df[t];
            off_pad[t] = pp;
            g_dst[t] = pp + s_cnt[t];
            pp += ((uint64_t)df[t] + BM25X_POST_ALIGN - 1) & ~(uint64_t)(BM25X_POST_ALIGN - 1);
        }
        uint64_t before = 0;  // surviving sealed postings of the terms before t
        for (uint32_t t = 0; t < T; t++) {
            if (old_to_new[t] != BM25X_TERM_MISSING) base[t] = off_pad[old_to_new[t]] - before;
            before += term_cnt[t];
        }
    }

    // ---- the new handle: statistics and tables from the new lengths (flush.rs:50-66), then its postings ----
    BuildMeta m{n_new, T_new, new_len.data(), new_pl.data(), keyed ? nk : nullptr, sealed->k1, sealed->b, df.data(), P_new};
    int rc = bm25x_index_begin(m, sealed->device, &nix);
    if (rc != BM25X_OK) return rc;
    h2d += bm25x_index_build_h2d_bytes(n_new, T_new);
    uint64_t *d_base = nullptr, *d_gdst = nullptr;
    MT_CU(s.alloc(&d_base, T));
    MT_CU(s.alloc(&d_gdst, T_new));
    if (T) {
        MT_CU(cudaMemcpy(d_base, base.data(), sizeof(uint64_t) * T, cudaMemcpyHostToDevice));
        k_mt_compact<<<(unsigned)n_pt, MT_THREADS>>>(od.post, n_pad, d_del, d_relabel, nix->d.fieldnorm, od.post_off, T,
                                                     d_ptile, d_base, nix->d.post);
        MT_CU(cudaGetLastError());
    }
    h2d += 8ull * T;
    if (P_g) {
        MT_CU(cudaMemcpy(d_gdst, g_dst.data(), sizeof(uint64_t) * T_new, cudaMemcpyHostToDevice));
        MT_CU(bm25x_scatter_csr(nix, T_new, P_g, g_off.data(), g_doc.data(), g_tf.data(), d_gdst));
        h2d += 8ull * T_new + 8ull * ((uint64_t)T_new + 1) + 8ull * P_g;
    }
    MT_CU(bm25x_index_finish_device(nix));
    MT_CU(cudaEventRecord(s.ev[1], 0));
    MT_CU(cudaEventSynchronize(s.ev[1]));

    // options set on the sealed handle carry over
    nix->prune = sealed->prune;
    nix->seed = sealed->seed;
    nix->seed_dense_div = sealed->seed_dense_div;
    nix->seed_prune_min = sealed->seed_prune_min;
    nix->seed_max_terms = sealed->seed_max_terms;
    nix->twophase = sealed->twophase;
    nix->slice_min = sealed->slice_min;
    if (stats) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, s.ev[0], s.ev[1]);
        stats->device_ms = ms;
        stats->h2d_bytes = h2d;
        stats->d2h_bytes = d2h;
        stats->postings_in = od.n_post + n_elem;
        stats->postings_out = P_new;
        stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count();
    }
    *out = nix;
    return BM25X_OK;
}

extern "C" int bm25x_bulkdelete(const bm25x_index *idx, const uint16_t *dead, uint64_t n_dead, uint8_t *deleted,
                                uint32_t *n_marked) {
    const char *who = "bm25x_bulkdelete";
    if (!idx || !deleted || (n_dead && !dead)) {
        bm25x_set_error("%s: null argument", who);
        return BM25X_ERR_INVALID;
    }
    for (uint64_t i = 1; i < n_dead; i++) {
        const uint16_t *a = dead + 3 * (i - 1), *b = dead + 3 * i;
        if (a[0] > b[0] || (a[0] == b[0] && (a[1] > b[1] || (a[1] == b[1] && a[2] > b[2])))) {
            bm25x_set_error("%s: dead tids must be sorted ascending by (hi, lo, offset)", who);
            return BM25X_ERR_INVALID;
        }
    }
    if (n_marked) *n_marked = 0;
    const uint32_t N = idx->d.n_docs;
    if (!n_dead || !N) return BM25X_OK;
    bm25x_index *nix = nullptr;  // MT_CU cleans up a new index; there is none here
    Scratch s;
    uint16_t *d_dead = nullptr;
    uint8_t *d_hit = nullptr;
    MT_CU(cudaSetDevice(idx->device));
    MT_CU(s.alloc(&d_dead, 3 * n_dead));
    MT_CU(s.alloc(&d_hit, N));
    MT_CU(cudaMemcpy(d_dead, dead, sizeof(uint16_t) * 3 * n_dead, cudaMemcpyHostToDevice));
    k_mt_bulkdelete<<<(N + 255) / 256, 256>>>(idx->d.payload, N, d_dead, n_dead, d_hit);
    MT_CU(cudaGetLastError());
    std::vector<uint8_t> hit(N);
    MT_CU(cudaMemcpy(hit.data(), d_hit, N, cudaMemcpyDeviceToHost));
    uint32_t n = 0;
    for (uint32_t d = 0; d < N; d++)
        if (hit[d] && !deleted[d]) {
            deleted[d] = 1;
            n++;
        }
    if (n_marked) *n_marked = n;
    return BM25X_OK;
}
