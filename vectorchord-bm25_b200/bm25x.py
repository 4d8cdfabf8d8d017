"""ctypes binding of include/bm25x.h (the drop-in C ABI).  No torch types cross this boundary."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# BM25X_LIBRARY: load another build of the same library (tools/time_variants.py times tuning variants side by side)
_SO = os.environ.get("BM25X_LIBRARY") or os.path.join(_HERE, "libbm25x.so")

MAX_K = 65535
MAX_QUERY_TERMS = 64
TERM_MISSING = 0xFFFFFFFF
DOC_NONE = 0xFFFFFFFF


class Bm25xError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"bm25x error {code}: {msg}")
        self.code = code


class _Corpus(C.Structure):
    _fields_ = [("n_docs", C.c_uint32), ("doc_len", C.POINTER(C.c_uint32)), ("payload", C.POINTER(C.c_uint16)),
                ("n_terms", C.c_uint32), ("term_key", C.POINTER(C.c_uint8)), ("post_off", C.POINTER(C.c_uint64)),
                ("post_doc", C.POINTER(C.c_uint32)), ("post_tf", C.POINTER(C.c_uint32)), ("k1", C.c_double),
                ("b", C.c_double)]


class _Blocks(C.Structure):
    _fields_ = [("n_docs", C.c_uint32), ("doc_len", C.POINTER(C.c_uint32)), ("doc_fieldnorm", C.POINTER(C.c_uint8)),
                ("sum_doc_len", C.c_uint64), ("payload", C.POINTER(C.c_uint16)), ("n_terms", C.c_uint32),
                ("term_key", C.POINTER(C.c_uint8)), ("term_blk_off", C.POINTER(C.c_uint64)), ("n_blocks", C.c_uint64),
                ("blk_min_doc", C.POINTER(C.c_uint32)), ("blk_n", C.POINTER(C.c_uint32)),
                ("blk_meta_doc", C.POINTER(C.c_uint8)), ("blk_meta_tf", C.POINTER(C.c_uint8)),
                ("blk_doc_off", C.POINTER(C.c_uint64)), ("blk_tf_off", C.POINTER(C.c_uint64)),
                ("bytes", C.POINTER(C.c_uint8)), ("n_bytes", C.c_uint64), ("k1", C.c_double), ("b", C.c_double),
                ("blk_wand_fieldnorm", C.POINTER(C.c_uint8)), ("blk_wand_tf", C.POINTER(C.c_uint32))]


class _GrowingDocs(C.Structure):
    _fields_ = [("n_docs", C.c_uint32), ("doc_len", C.POINTER(C.c_uint32)), ("doc_fieldnorm", C.POINTER(C.c_uint8)),
                ("payload", C.POINTER(C.c_uint16)), ("deleted", C.POINTER(C.c_uint8)),
                ("elem_off", C.POINTER(C.c_uint64)), ("elem_term", C.POINTER(C.c_uint32)),
                ("elem_tf", C.POINTER(C.c_uint32))]


class _Vectors(C.Structure):  # bm25x_vectors
    _fields_ = [("n_docs", C.c_uint32), ("payload", C.POINTER(C.c_uint16)), ("deleted", C.POINTER(C.c_uint8)),
                ("elem_off", C.POINTER(C.c_uint64)), ("elem_key", C.POINTER(C.c_uint8)),
                ("elem_term", C.POINTER(C.c_uint32)), ("elem_tf", C.POINTER(C.c_uint32))]


class MaintainStats(C.Structure):  # bm25x_maintain_stats
    _fields_ = [("total_ms", C.c_double), ("device_ms", C.c_double), ("h2d_bytes", C.c_uint64),
                ("d2h_bytes", C.c_uint64), ("postings_in", C.c_uint64), ("postings_out", C.c_uint64)]


class IndexInfo(C.Structure):
    _fields_ = [("n_docs", C.c_uint32), ("n_terms", C.c_uint32), ("n_postings", C.c_uint64),
                ("sum_doc_len", C.c_uint64), ("avgdl", C.c_double), ("k1", C.c_double), ("b", C.c_double),
                ("device_bytes", C.c_uint64), ("n_blocks", C.c_uint64), ("device", C.c_int)]


N_ARRAYS = 13


class IndexLayout(C.Structure):
    _fields_ = [("n_docs", C.c_uint32), ("n_terms", C.c_uint32), ("n_postings", C.c_uint64),
                ("n_postings_padded", C.c_uint64), ("n_blocks", C.c_uint64), ("sum_doc_len", C.c_uint64),
                ("k1", C.c_double), ("b", C.c_double), ("avgdl", C.c_double), ("dev_ptr", C.c_void_p * N_ARRAYS),
                ("bytes", C.c_uint64 * N_ARRAYS), ("device", C.c_int)]


class BrokerOptions(C.Structure):  # bm25x_broker_options (include/bm25x_broker.h)
    _fields_ = [("max_batch", C.c_uint32), ("max_wait_us", C.c_uint32), ("ring_slots", C.c_uint32), ("reserved", C.c_uint32)]


class BrokerStats(C.Structure):  # bm25x_broker_stats
    _fields_ = [("requests", C.c_uint64), ("batches", C.c_uint64), ("max_batch_seen", C.c_uint64),
                ("ring_full_waits", C.c_uint64), ("rejected", C.c_uint64)]


# bm25x_broker_backend: (ctx, nq, q_off, q_terms, k, out_doc, out_score, out_score64, out_payload, out_n) -> status
BROKER_BACKEND = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.c_uint32,
                             C.POINTER(C.c_uint32), C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_uint16),
                             C.POINTER(C.c_uint32))


class SearchStats(C.Structure):
    _fields_ = [("kernel_ms", C.c_double), ("h2d_ms", C.c_double), ("d2h_ms", C.c_double), ("postings", C.c_uint64),
                ("bytes_algo", C.c_uint64), ("launches", C.c_uint32), ("queries", C.c_uint32),
                ("postings_fetched", C.c_uint64)]


class _Synth(C.Structure):
    _fields_ = [("n_docs", C.c_uint32), ("n_terms", C.c_uint32), ("n_postings", C.c_uint64),
                ("doc_len", C.POINTER(C.c_uint32)), ("post_off", C.POINTER(C.c_uint64)),
                ("post_doc", C.POINTER(C.c_uint32)), ("post_tf", C.POINTER(C.c_uint32))]


def build_library(force: bool = False) -> str:
    """nvcc -gencode arch=compute_100a,code=sm_100a build of csrc/ → libbm25x.so (in-tree)."""
    srcdir = os.path.join(_HERE, "csrc")
    srcs = [os.path.join(srcdir, f) for f in os.listdir(srcdir)] + [os.path.join(_HERE, "..", "include", "bm25x.h")]
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call(["make", "-C", srcdir, "-s"], stdout=subprocess.DEVNULL)
    return _SO


_lib = None


def load_library():
    """Loads libbm25x.so; raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise Bm25xError(-1, f"{_SO} not built: run `python -c 'import __graft_entry__ as g; g.build()'`")
    L = C.CDLL(_SO)
    vp, u8p, u16p, u32p, u64p, f32p, f64p = (C.c_void_p, C.POINTER(C.c_uint8), C.POINTER(C.c_uint16),
                                             C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_float),
                                             C.POINTER(C.c_double))
    L.bm25x_index_create.argtypes = [C.POINTER(_Corpus), C.c_int, C.POINTER(vp)]
    L.bm25x_index_create_from_blocks.argtypes = [C.POINTER(_Blocks), C.c_int, C.POINTER(vp)]
    L.bm25x_growing_create.argtypes = [vp, C.POINTER(_GrowingDocs), C.POINTER(vp)]
    L.bm25x_search_batch_growing.argtypes = [vp, vp, C.c_uint32, u32p, u32p, C.c_uint32, u8p, u8p, u32p, f32p, f64p,
                                             u16p, u32p, C.POINTER(SearchStats)]
    L.bm25x_index_maintain.argtypes = [vp, u8p, C.POINTER(_Vectors), C.POINTER(vp), u32p, C.POINTER(MaintainStats)]
    L.bm25x_bulkdelete.argtypes = [vp, u16p, C.c_uint64, u8p, u32p]
    L.bm25x_merge_topk.argtypes = [C.c_uint32, C.c_uint32, u32p, f32p, f64p, u16p, u32p, u32p, f32p, f64p, u16p, u32p,
                                   C.c_uint32, u32p, f32p, f64p, u16p, u32p]
    L.bm25x_index_destroy.argtypes = [vp]
    L.bm25x_index_destroy.restype = None
    L.bm25x_index_get_info.argtypes = [vp, C.POINTER(IndexInfo)]
    L.bm25x_lookup_terms.argtypes = [vp, u8p, C.c_uint32, u32p]
    L.bm25x_index_get_layout.argtypes = [vp, C.POINTER(IndexLayout)]
    L.bm25x_index_alloc_replica.argtypes = [C.POINTER(IndexLayout), C.c_int, C.POINTER(vp)]
    L.bm25x_index_finalize_replica.argtypes = [vp]
    L.bm25x_index_get_df.argtypes = [vp, u32p]
    L.bm25x_index_set_option.argtypes = [vp, C.c_char_p, C.c_int64]
    L.bm25x_search_batch.argtypes = [vp, C.c_uint32, u32p, u32p, C.c_uint32, u8p, u32p, f32p, f64p, u16p, u32p,
                                     C.POINTER(SearchStats)]
    L.bm25x_batch_prepare.argtypes = [vp, C.c_uint32, u32p, u32p, C.c_uint32, u8p, C.POINTER(vp)]
    L.bm25x_batch_run.argtypes = [vp, vp, C.POINTER(SearchStats)]
    L.bm25x_batch_fetch.argtypes = [vp, u32p, f32p, f64p, u16p, u32p]
    L.bm25x_batch_device_results.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    L.bm25x_batch_destroy.argtypes = [vp]
    L.bm25x_batch_destroy.restype = None
    L.bm25x_evaluate_batch.argtypes = [vp, C.c_uint32, u32p, u32p, u32p, u32p, u32p, f64p]
    L.bm25x_check_vectors.argtypes = [C.c_uint32, u32p, u32p, u32p]
    L.bm25x_synth_generate.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_double,
                                       C.c_int, C.POINTER(_Synth)]
    L.bm25x_synth_free.argtypes = [C.POINTER(_Synth)]
    L.bm25x_synth_free.restype = None
    L.bm25x_synth_queries.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_double, u64p,
                                      u32p, u32p]
    L.bm25x_intern.argtypes = [u8p, u8p, C.c_size_t, u8p]
    L.bm25x_blake3_keyed16.argtypes = [u8p, u8p, C.c_size_t, u8p]
    L.bm25x_broker_create.argtypes = [vp, C.POINTER(BrokerOptions), C.POINTER(vp)]
    L.bm25x_broker_create_with_backend.argtypes = [BROKER_BACKEND, vp, C.POINTER(BrokerOptions), C.POINTER(vp)]
    L.bm25x_broker_search.argtypes = [vp, u32p, C.c_uint32, C.c_uint32, u32p, f64p, u16p, u32p]
    L.bm25x_broker_get_stats.argtypes = [vp, C.POINTER(BrokerStats)]
    L.bm25x_broker_destroy.argtypes = [vp]
    L.bm25x_broker_destroy.restype = None
    L.bm25x_last_error.restype = C.c_char_p
    L.bm25x_device_count.restype = C.c_int
    _lib = L
    return L


def intern(seed: bytes, token: bytes) -> bytes:
    """vector::intern (crates/bm25/src/vector.rs:19-35): 16-byte key of a token under the index seed."""
    assert len(seed) == 32
    out = (C.c_uint8 * 16)()
    sd = (C.c_uint8 * 32).from_buffer_copy(seed)
    tk = (C.c_uint8 * max(len(token), 1)).from_buffer_copy(token if token else b"\0")
    _check(load_library().bm25x_intern(sd, tk, len(token), out))
    return bytes(out)


def blake3_keyed16(key: bytes, data: bytes) -> bytes:
    out = (C.c_uint8 * 16)()
    kk = (C.c_uint8 * 32).from_buffer_copy(key)
    dd = (C.c_uint8 * max(len(data), 1)).from_buffer_copy(data if data else b"\0")
    _check(load_library().bm25x_blake3_keyed16(kk, dd, len(data), out))
    return bytes(out)


def _check(rc):
    if rc != 0:
        raise Bm25xError(rc, load_library().bm25x_last_error().decode())


def _p(a, ty):
    return a.ctypes.data_as(C.POINTER(ty)) if a is not None else None


def check_vectors(off, terms, tfs=None):
    """bm25x_check_vectors: the Document / Query invariants of crates/bm25/src/vector.rs:46-134 for n vectors in CSR form
    (keys strictly ascending, tfs non-zero); raises Bm25xError(1, "invalid data: ...")."""
    off = np.ascontiguousarray(off, dtype=np.uint32)
    terms = np.ascontiguousarray(terms, dtype=np.uint32)
    tfs = np.ascontiguousarray(tfs, dtype=np.uint32) if tfs is not None else None
    _check(load_library().bm25x_check_vectors(len(off) - 1, _p(off, C.c_uint32), _p(terms, C.c_uint32), _p(tfs, C.c_uint32)))


def device_count() -> int:
    return load_library().bm25x_device_count()


class Document:
    """crates/bm25/src/vector.rs:46-98 `Document`: strictly ascending term ordinals with tf != 0."""

    def __init__(self, terms, tfs):
        self.terms = np.ascontiguousarray(terms, dtype=np.uint32)
        self.tfs = np.ascontiguousarray(tfs, dtype=np.uint32)
        if len(self.terms) != len(self.tfs) or np.any(np.diff(self.terms.astype(np.int64)) <= 0) or np.any(self.tfs == 0):
            raise ValueError("invalid data")  # Document::new → expect("invalid data")

    def length(self) -> int:
        return int(min(int(self.tfs.astype(np.uint64).sum()), 0xFFFFFFFF))


class Query:
    """crates/bm25/src/vector.rs:100-134 `Query`: strictly ascending term ordinals."""

    def __init__(self, terms):
        self.terms = np.ascontiguousarray(terms, dtype=np.uint32)
        if np.any(np.diff(self.terms.astype(np.int64)) <= 0):
            raise ValueError("invalid data")


class SyntheticCorpus:
    """Host CSR owned by libbm25x (malloc); numpy views without copying (10 GB at the 10M-doc config)."""

    def __init__(self, raw: _Synth):
        self._raw = raw
        self.n_docs, self.n_terms, self.n_postings = raw.n_docs, raw.n_terms, raw.n_postings
        self.doc_len = np.ctypeslib.as_array(raw.doc_len, shape=(raw.n_docs,))
        self.post_off = np.ctypeslib.as_array(raw.post_off, shape=(raw.n_terms + 1,))
        n = max(int(raw.n_postings), 1)
        self.post_doc = np.ctypeslib.as_array(raw.post_doc, shape=(n,))[:raw.n_postings]
        self.post_tf = np.ctypeslib.as_array(raw.post_tf, shape=(n,))[:raw.n_postings]
        self.k1, self.b = 1.2, 0.75

    def free(self):
        if self._raw is not None:
            self.doc_len = self.post_off = self.post_doc = self.post_tf = None
            load_library().bm25x_synth_free(C.byref(self._raw))
            self._raw = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def synth_corpus(seed, n_docs, vocab, len_min, len_max=None, zipf_s=0.0, nthreads=0) -> SyntheticCorpus:
    raw = _Synth()
    _check(load_library().bm25x_synth_generate(seed, n_docs, vocab, len_min, len_min if len_max is None else len_max,
                                               float(zipf_s), nthreads, C.byref(raw)))
    return SyntheticCorpus(raw)


def synth_queries(seed, nq, vocab, n_min, n_max, post_off, zipf_s=0.0):
    post_off = np.ascontiguousarray(post_off, dtype=np.uint64)
    q_off = np.zeros(nq + 1, dtype=np.uint32)
    q_terms = np.zeros(nq * n_max, dtype=np.uint32)
    _check(load_library().bm25x_synth_queries(seed, nq, vocab, n_min, n_max, float(zipf_s), _p(post_off, C.c_uint64),
                                              _p(q_off, C.c_uint32), _p(q_terms, C.c_uint32)))
    return q_off, q_terms[:q_off[-1]].copy()


class Index:
    """Sealed-segment index resident in one GPU's HBM (bm25x_index_*)."""

    def __init__(self, n_docs, doc_len, n_terms, post_off, post_doc, post_tf, k1=1.2, b=0.75, payload=None,
                 term_keys=None, device=0):
        L = load_library()
        self._keep = [np.ascontiguousarray(doc_len, dtype=np.uint32), np.ascontiguousarray(post_off, dtype=np.uint64),
                      np.ascontiguousarray(post_doc, dtype=np.uint32), np.ascontiguousarray(post_tf, dtype=np.uint32)]
        c = _Corpus()
        c.n_docs, c.n_terms, c.k1, c.b = int(n_docs), int(n_terms), float(k1), float(b)
        c.doc_len = _p(self._keep[0], C.c_uint32)
        c.post_off = _p(self._keep[1], C.c_uint64)
        c.post_doc = _p(self._keep[2], C.c_uint32)
        c.post_tf = _p(self._keep[3], C.c_uint32)
        if payload is not None:
            pl = np.ascontiguousarray(payload, dtype=np.uint16)
            self._keep.append(pl)
            c.payload = _p(pl, C.c_uint16)
        if term_keys is not None:
            tk = np.ascontiguousarray(term_keys, dtype=np.uint8)
            self._keep.append(tk)
            c.term_key = _p(tk, C.c_uint8)
        h = C.c_void_p()
        _check(L.bm25x_index_create(C.byref(c), device, C.byref(h)))
        self.h = h
        self._keep = None  # the library copied everything to the device
        self.n_docs, self.n_terms = int(n_docs), int(n_terms)

    @classmethod
    def from_blocks(cls, n_docs, n_terms, term_blk_off, blk_min_doc, blk_n, blk_meta_doc, blk_meta_tf, blk_doc_off,
                    blk_tf_off, data, doc_len=None, doc_fieldnorm=None, sum_doc_len=0, k1=1.2, b=0.75, payload=None,
                    term_keys=None, device=0, blk_wand_fieldnorm=None, blk_wand_tf=None) -> "Index":
        """Index from the sealed segment as the reference stores it: per-token chains of 128-posting blocks in the
        codec of compression.rs, decoded on the GPU (bm25x_index_create_from_blocks).  Document norms come either from
        exact lengths (`doc_len`) or, as on the pages, from `doc_fieldnorm` + `sum_doc_len`."""
        L = load_library()
        c = _Blocks()
        keep = []

        def arr(a, dt, ct):
            a = np.ascontiguousarray(a, dtype=dt)
            keep.append(a)
            return _p(a, ct)

        c.n_docs, c.n_terms, c.k1, c.b = int(n_docs), int(n_terms), float(k1), float(b)
        if doc_len is not None:
            c.doc_len = arr(doc_len, np.uint32, C.c_uint32)
        if doc_fieldnorm is not None:
            c.doc_fieldnorm = arr(doc_fieldnorm, np.uint8, C.c_uint8)
        c.sum_doc_len = int(sum_doc_len)
        if payload is not None:
            c.payload = arr(payload, np.uint16, C.c_uint16)
        if term_keys is not None:
            c.term_key = arr(term_keys, np.uint8, C.c_uint8)
        c.term_blk_off = arr(term_blk_off, np.uint64, C.c_uint64)
        c.n_blocks = int(keep[-1][int(n_terms)]) if len(keep[-1]) > int(n_terms) else 0
        c.blk_min_doc = arr(blk_min_doc, np.uint32, C.c_uint32)
        c.blk_n = arr(blk_n, np.uint32, C.c_uint32)
        c.blk_meta_doc = arr(blk_meta_doc, np.uint8, C.c_uint8)
        c.blk_meta_tf = arr(blk_meta_tf, np.uint8, C.c_uint8)
        c.blk_doc_off = arr(blk_doc_off, np.uint64, C.c_uint64)
        c.blk_tf_off = arr(blk_tf_off, np.uint64, C.c_uint64)
        c.bytes = arr(data, np.uint8, C.c_uint8)
        c.n_bytes = len(keep[-1])
        if blk_wand_fieldnorm is not None and blk_wand_tf is not None:   # SummaryTuple.wand_* (checked against the blocks)
            c.blk_wand_fieldnorm = arr(blk_wand_fieldnorm, np.uint8, C.c_uint8)
            c.blk_wand_tf = arr(blk_wand_tf, np.uint32, C.c_uint32)
        h = C.c_void_p()
        _check(L.bm25x_index_create_from_blocks(C.byref(c), device, C.byref(h)))
        return cls._adopt(h, n_docs, n_terms)

    @classmethod
    def _adopt(cls, handle, n_docs, n_terms):
        self = cls.__new__(cls)
        self.h, self._keep, self.n_docs, self.n_terms = handle, None, int(n_docs), int(n_terms)
        return self

    def layout(self) -> IndexLayout:
        out = IndexLayout()
        _check(load_library().bm25x_index_get_layout(self.h, C.byref(out)))
        return out

    @classmethod
    def alloc_replica(cls, like: IndexLayout, device: int) -> "Index":
        """Empty index of the same shape on `device`; fill the arrays of .layout() (e.g. by NCCL broadcast), then
        call finalize_replica()."""
        h = C.c_void_p()
        _check(load_library().bm25x_index_alloc_replica(C.byref(like), device, C.byref(h)))
        return cls._adopt(h, like.n_docs, like.n_terms)

    def finalize_replica(self):
        _check(load_library().bm25x_index_finalize_replica(self.h))

    def set_option(self, name: str, value: int):
        _check(load_library().bm25x_index_set_option(self.h, name.encode(), int(value)))

    def df(self):
        out = np.zeros(self.n_terms, np.uint32)
        _check(load_library().bm25x_index_get_df(self.h, _p(out, C.c_uint32)))
        return out

    @staticmethod
    def from_corpus(c, device=0, **kw):
        return Index(c.n_docs, c.doc_len, c.n_terms, c.post_off, c.post_doc, c.post_tf, getattr(c, "k1", 1.2),
                     getattr(c, "b", 0.75), device=device, **kw)

    def close(self):
        if getattr(self, "h", None):
            load_library().bm25x_index_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self) -> IndexInfo:
        out = IndexInfo()
        _check(load_library().bm25x_index_get_info(self.h, C.byref(out)))
        return out

    def lookup_terms(self, keys):
        keys = np.ascontiguousarray(keys, dtype=np.uint8).reshape(-1, 16)
        out = np.zeros(len(keys), dtype=np.uint32)
        _check(load_library().bm25x_lookup_terms(self.h, _p(keys, C.c_uint8), len(keys), _p(out, C.c_uint32)))
        return out

    # ---- bm25::search for a batch (host buffers in, host buffers out) ----
    def search_batch(self, q_off, q_terms, k, allow=None, want_f64=True, want_payload=False, out=None):
        q_off = np.ascontiguousarray(q_off, dtype=np.uint32)
        q_terms = np.ascontiguousarray(q_terms, dtype=np.uint32)
        nq = len(q_off) - 1
        kk = max(int(k), 1)
        if out is None:
            out = {"doc": np.empty((nq, kk), np.uint32), "score": np.empty((nq, kk), np.float32),
                   "score64": np.empty((nq, kk), np.float64) if want_f64 else None,
                   "payload": np.empty((nq, kk, 3), np.uint16) if want_payload else None,
                   "n": np.empty(nq, np.uint32)}
        al = np.ascontiguousarray(allow, dtype=np.uint8) if allow is not None else None
        st = SearchStats()
        _check(load_library().bm25x_search_batch(self.h, nq, _p(q_off, C.c_uint32), _p(q_terms, C.c_uint32), int(k),
                                                 _p(al, C.c_uint8), _p(out["doc"], C.c_uint32),
                                                 _p(out["score"], C.c_float), _p(out["score64"], C.c_double),
                                                 _p(out["payload"], C.c_uint16), _p(out["n"], C.c_uint32),
                                                 C.byref(st)))
        out["stats"] = st
        return out

    def search(self, query, k, allow=None):
        """One query, the shape of bm25::search(&index, k, &query, filter): [(score f64, doc id)] best first."""
        terms = query.terms if isinstance(query, Query) else np.asarray(query, dtype=np.uint32)
        r = self.search_batch(np.array([0, len(terms)], np.uint32), terms, k, allow=allow)
        n = int(r["n"][0])
        return r["doc"][0, :n].copy(), r["score64"][0, :n].copy()

    # ---- growing segment (documents inserted since the last seal; search.rs:83-135) ----
    def growing(self, elem_off, elem_term, elem_tf, doc_len=None, doc_fieldnorm=None, payload=None,
                deleted=None) -> "Index":
        """Handle over the growing documents (doc-major: document g holds elements elem_off[g]..elem_off[g+1], term
        ordinals of THIS sealed index ascending, TERM_MISSING for tokens it does not know) that scores with this
        index's statistics (bm25x_growing_create).  Search it like any index; ids are growing ordinals."""
        g = _GrowingDocs()
        keep = []

        def arr(a, dt, ct):
            a = np.ascontiguousarray(a, dtype=dt)
            keep.append(a)
            return _p(a, ct)

        g.elem_off = arr(elem_off, np.uint64, C.c_uint64)
        g.n_docs = len(keep[-1]) - 1
        g.elem_term = arr(elem_term, np.uint32, C.c_uint32)
        g.elem_tf = arr(elem_tf, np.uint32, C.c_uint32)
        if doc_len is not None:
            g.doc_len = arr(doc_len, np.uint32, C.c_uint32)
        if doc_fieldnorm is not None:
            g.doc_fieldnorm = arr(doc_fieldnorm, np.uint8, C.c_uint8)
        if payload is not None:
            g.payload = arr(payload, np.uint16, C.c_uint16)
        if deleted is not None:
            g.deleted = arr(deleted, np.uint8, C.c_uint8)
        h = C.c_void_p()
        _check(load_library().bm25x_growing_create(self.h, C.byref(g), C.byref(h)))
        return Index._adopt(h, g.n_docs, self.n_terms)

    # ---- the write side: bm25::maintain / bm25::bulkdelete ----
    def maintain(self, deleted=None, elem_off=None, elem_key=None, elem_term=None, elem_tf=None, payload=None,
                 growing_deleted=None):
        """bm25x_index_maintain: a NEW sealed index from this one's surviving documents (`deleted` marks, or None) and
        the growing documents (doc-major elem_off / elem_tf with elem_key [n_elem, 16] on a keyed index or elem_term on
        a keyless one; None = compaction only).  Returns (Index, relabel, stats): relabel[d] = new doc id of sealed
        document d, then of growing document g at n_docs + g, DOC_NONE for the dead.  This index is left unchanged."""
        keep = []

        def arr(a, dt, ct):
            a = np.ascontiguousarray(a, dtype=dt)
            keep.append(a)
            return _p(a, ct)

        v, vp = None, None
        n_grow = 0
        if elem_off is not None:
            v = _Vectors()
            v.elem_off = arr(elem_off, np.uint64, C.c_uint64)
            v.n_docs = n_grow = len(keep[-1]) - 1
            v.elem_tf = arr(elem_tf, np.uint32, C.c_uint32)
            if elem_key is not None:
                v.elem_key = arr(elem_key, np.uint8, C.c_uint8)
            if elem_term is not None:
                v.elem_term = arr(elem_term, np.uint32, C.c_uint32)
            if payload is not None:
                v.payload = arr(payload, np.uint16, C.c_uint16)
            if growing_deleted is not None:
                v.deleted = arr(growing_deleted, np.uint8, C.c_uint8)
            vp = C.byref(v)
        dl = arr(deleted, np.uint8, C.c_uint8) if deleted is not None else None
        relabel = np.empty(self.n_docs + n_grow, np.uint32)
        st = MaintainStats()
        h = C.c_void_p()
        _check(load_library().bm25x_index_maintain(self.h, dl, vp, C.byref(h), _p(relabel, C.c_uint32), C.byref(st)))
        info = IndexInfo()
        _check(load_library().bm25x_index_get_info(h, C.byref(info)))
        return Index._adopt(h, info.n_docs, info.n_terms), relabel, st

    def bulkdelete(self, dead, deleted=None):
        """bm25x_bulkdelete: marks every document whose payload (ctid) is in `dead` ([n, 3] u16, sorted by (hi, lo,
        offset)).  Returns (deleted, n_marked): the updated marks (a copy of `deleted`, or fresh zeros) and how many
        this call set."""
        dead = np.ascontiguousarray(dead, dtype=np.uint16).reshape(-1, 3)
        out = np.zeros(self.n_docs, np.uint8) if deleted is None else np.array(deleted, dtype=np.uint8, copy=True)
        n = C.c_uint32(0)
        _check(load_library().bm25x_bulkdelete(self.h, _p(dead, C.c_uint16), len(dead), _p(out, C.c_uint8), C.byref(n)))
        return out, n.value

    def search_batch_growing(self, growing, q_off, q_terms, k, allow=None, allow_growing=None, want_payload=False):
        """bm25::search over this sealed index + a growing handle (None = sealed only): ids >= n_docs are growing
        ordinal + n_docs."""
        q_off = np.ascontiguousarray(q_off, dtype=np.uint32)
        q_terms = np.ascontiguousarray(q_terms, dtype=np.uint32)
        nq, kk = len(q_off) - 1, int(k)
        out = {"doc": np.empty((nq, kk), np.uint32), "score": np.empty((nq, kk), np.float32),
               "score64": np.empty((nq, kk), np.float64),
               "payload": np.empty((nq, kk, 3), np.uint16) if want_payload else None, "n": np.empty(nq, np.uint32)}
        al = np.ascontiguousarray(allow, dtype=np.uint8) if allow is not None else None
        alg = np.ascontiguousarray(allow_growing, dtype=np.uint8) if allow_growing is not None else None
        st = SearchStats()
        _check(load_library().bm25x_search_batch_growing(
            self.h, growing.h if growing is not None else None, nq, _p(q_off, C.c_uint32), _p(q_terms, C.c_uint32), kk,
            _p(al, C.c_uint8), _p(alg, C.c_uint8), _p(out["doc"], C.c_uint32), _p(out["score"], C.c_float),
            _p(out["score64"], C.c_double), _p(out["payload"], C.c_uint16), _p(out["n"], C.c_uint32), C.byref(st)))
        out["stats"] = st
        return out

    def prepare(self, q_off, q_terms, k, allow=None) -> "Batch":
        return Batch(self, q_off, q_terms, k, allow)

    # ---- bm25::evaluate for a batch of (document, query) pairs ----
    def evaluate_batch(self, docs, queries):
        d_off = np.zeros(len(docs) + 1, np.uint32)
        q_off = np.zeros(len(docs) + 1, np.uint32)
        for i, (d, q) in enumerate(zip(docs, queries)):
            d_off[i + 1] = d_off[i] + len(d.terms)
            q_off[i + 1] = q_off[i] + len(q.terms)
        cat = lambda xs: np.ascontiguousarray(np.concatenate(xs) if xs else np.zeros(0), dtype=np.uint32)
        d_terms, d_tfs, q_terms = cat([d.terms for d in docs]), cat([d.tfs for d in docs]), cat([q.terms for q in queries])
        out = np.zeros(len(docs), np.float64)
        _check(load_library().bm25x_evaluate_batch(self.h, len(docs), _p(d_off, C.c_uint32), _p(d_terms, C.c_uint32),
                                                   _p(d_tfs, C.c_uint32), _p(q_off, C.c_uint32),
                                                   _p(q_terms, C.c_uint32), _p(out, C.c_double)))
        return out

    def evaluate(self, document: Document, query: Query) -> float:
        return float(self.evaluate_batch([document], [query])[0])


def merge_topk(a, b, doc_base_b, k):
    """Host-only bm25x_merge_topk of two result dicts (as returned by search_batch with f64 scores)."""
    nq = len(a["n"])
    assert a["doc"].shape == (nq, k) and b["doc"].shape == (nq, k)
    pay = a.get("payload") is not None and b.get("payload") is not None
    out = {"doc": np.empty((nq, k), np.uint32), "score": np.empty((nq, k), np.float32),
           "score64": np.empty((nq, k), np.float64), "payload": np.empty((nq, k, 3), np.uint16) if pay else None,
           "n": np.empty(nq, np.uint32)}
    c = lambda x, dt: np.ascontiguousarray(x, dtype=dt)
    keep = [c(a["doc"], np.uint32), c(a["score"], np.float32), c(a["score64"], np.float64),
            c(a["payload"], np.uint16) if pay else None, c(a["n"], np.uint32),
            c(b["doc"], np.uint32), c(b["score"], np.float32), c(b["score64"], np.float64),
            c(b["payload"], np.uint16) if pay else None, c(b["n"], np.uint32)]
    ty = [C.c_uint32, C.c_float, C.c_double, C.c_uint16, C.c_uint32] * 2
    _check(load_library().bm25x_merge_topk(nq, int(k), *[_p(x, t) for x, t in zip(keep[:5], ty[:5])],
                                           *[_p(x, t) for x, t in zip(keep[5:], ty[5:])], int(doc_base_b),
                                           _p(out["doc"], C.c_uint32), _p(out["score"], C.c_float),
                                           _p(out["score64"], C.c_double), _p(out["payload"], C.c_uint16),
                                           _p(out["n"], C.c_uint32)))
    return out


class Batch:
    """Split form: prepare (canonicalise + upload) / run (kernels only, inputs resident in HBM) / fetch (D2H)."""

    def __init__(self, index: Index, q_off, q_terms, k, allow=None):
        self.index = index
        q_off = np.ascontiguousarray(q_off, dtype=np.uint32)
        q_terms = np.ascontiguousarray(q_terms, dtype=np.uint32)
        self.nq, self.k = len(q_off) - 1, int(k)
        al = np.ascontiguousarray(allow, dtype=np.uint8) if allow is not None else None
        h = C.c_void_p()
        _check(load_library().bm25x_batch_prepare(index.h, self.nq, _p(q_off, C.c_uint32), _p(q_terms, C.c_uint32),
                                                  self.k, _p(al, C.c_uint8), C.byref(h)))
        self.h = h

    def run(self, stream=None, timed=True):
        st = SearchStats()
        _check(load_library().bm25x_batch_run(self.h, C.c_void_p(stream) if stream else None,
                                              C.byref(st) if timed else None))
        return st

    def fetch(self, want_f64=True, want_payload=False):
        out = {"doc": np.empty((self.nq, self.k), np.uint32), "score": np.empty((self.nq, self.k), np.float32),
               "score64": np.empty((self.nq, self.k), np.float64) if want_f64 else None,
               "payload": np.empty((self.nq, self.k, 3), np.uint16) if want_payload else None,
               "n": np.empty(self.nq, np.uint32)}
        _check(load_library().bm25x_batch_fetch(self.h, _p(out["doc"], C.c_uint32), _p(out["score"], C.c_float),
                                                _p(out["score64"], C.c_double), _p(out["payload"], C.c_uint16),
                                                _p(out["n"], C.c_uint32)))
        return out

    def device_results(self):
        """Raw device addresses of the result rows: {"doc": (ptr, nbytes), "score": ..., "score64": ..., "n": ...}
        (bm25x_batch_device_results) — for GPU → GPU transport of sharded results (shard.py)."""
        p = [C.c_void_p() for _ in range(5)]
        _check(load_library().bm25x_batch_device_results(self.h, *[C.byref(x) for x in p]))
        slots = self.nq * self.k
        return {"doc": (p[0].value, 4 * slots), "score": (p[1].value, 4 * slots), "score64": (p[2].value, 8 * slots),
                "payload": (p[3].value, 6 * slots), "n": (p[4].value, 4 * self.nq)}

    def close(self):
        if getattr(self, "h", None):
            load_library().bm25x_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Broker:
    """Batching broker (include/bm25x_broker.h): concurrent single-query callers, one backend call per batch.
    Broker(index) batches into bm25x_search_batch; Broker(backend=callable) into any function of the backend signature
    (the callable receives raw ctypes pointers)."""

    def __init__(self, index=None, backend=None, max_batch=0, max_wait_us=0, ring_slots=0):
        L = load_library()
        opt = BrokerOptions(max_batch, max_wait_us, ring_slots, 0)
        self.h = C.c_void_p()
        self._keep = None
        if backend is not None:
            self._keep = BROKER_BACKEND(backend)
            _check(L.bm25x_broker_create_with_backend(self._keep, None, C.byref(opt), C.byref(self.h)))
        else:
            self._keep = index
            _check(L.bm25x_broker_create(index.h, C.byref(opt), C.byref(self.h)))

    def search(self, terms, k, want_payload=False):
        terms = np.ascontiguousarray(terms, dtype=np.uint32)
        kk = max(int(k), 1)
        doc, s64, n = np.empty(kk, np.uint32), np.empty(kk, np.float64), C.c_uint32(0)
        pay = np.empty((kk, 3), np.uint16) if want_payload else None
        _check(load_library().bm25x_broker_search(self.h, _p(terms, C.c_uint32), len(terms), int(k), _p(doc, C.c_uint32),
                                                  _p(s64, C.c_double), _p(pay, C.c_uint16), C.byref(n)))
        return (doc[:n.value], s64[:n.value]) + ((pay[:n.value],) if want_payload else ())

    def stats(self) -> BrokerStats:
        st = BrokerStats()
        _check(load_library().bm25x_broker_get_stats(self.h, C.byref(st)))
        return st

    def close(self):
        if self.h:
            load_library().bm25x_broker_destroy(self.h)
            self.h = C.c_void_p()
