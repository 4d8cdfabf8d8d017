"""Plain numpy restatement of bm25::maintain (crates/bm25/src/maintain.rs:27-311) and of the bulkdelete predicate
(bulkdelete.rs:20-112): the expected value of every maintain test, and the input of an independent
bm25x_index_create of the same index for byte comparisons.  Test infrastructure, like oracle/."""
from __future__ import annotations

import numpy as np

from oracle import oracle

DOC_NONE = 0xFFFFFFFF
TERM_MISSING = 0xFFFFFFFF


def synthetic_ctid(ids):
    """The ctid the library gives document i of an index made without payloads: (block hi, block lo, offset) of a
    291-tuple page."""
    i = np.asarray(ids, dtype=np.int64)
    blk = i // 291
    return np.stack([blk >> 16, blk & 0xFFFF, i % 291 + 1], axis=-1).astype(np.uint16).reshape(-1, 3)


class Vectors:
    """The VectorTuple chain (bm25x_vectors): document g holds elements elem_off[g]..elem_off[g+1], each a token
    (elem_key [n, 16] on a keyed index, elem_term on a keyless one) with its tf."""

    def __init__(self, elem_off, elem_tf, elem_term=None, elem_key=None, payload=None, deleted=None):
        self.elem_off = np.ascontiguousarray(elem_off, dtype=np.uint64)
        self.elem_tf = np.ascontiguousarray(elem_tf, dtype=np.uint32)
        self.elem_term = None if elem_term is None else np.ascontiguousarray(elem_term, dtype=np.uint32)
        self.elem_key = None if elem_key is None else np.ascontiguousarray(elem_key, dtype=np.uint8).reshape(-1, 16)
        self.payload = None if payload is None else np.ascontiguousarray(payload, dtype=np.uint16).reshape(-1, 3)
        self.n_docs = len(self.elem_off) - 1
        self.deleted = (np.zeros(self.n_docs, bool) if deleted is None else np.asarray(deleted).astype(bool))

    @staticmethod
    def from_docs(docs, keys=None, payload=None, deleted=None):
        """docs: list of dict{token: tf}; tokens are ordinals, or indices into `keys` ([n, 16]) for a keyed index."""
        off = np.cumsum([0] + [len(d) for d in docs]).astype(np.uint64)
        if keys is None:
            terms = [t for d in docs for t in sorted(d)]
            tfs = [d[t] for d in docs for t in sorted(d)]
            return Vectors(off, tfs, elem_term=terms, payload=payload, deleted=deleted)
        keys = np.asarray(keys, dtype=np.uint8).reshape(-1, 16)
        rows, tfs = [], []
        for d in docs:
            for t in sorted(d, key=lambda t: bytes(keys[t])):
                rows.append(keys[t])
                tfs.append(d[t])
        return Vectors(off, tfs, elem_key=np.array(rows, np.uint8).reshape(-1, 16), payload=payload, deleted=deleted)


def _key_u64(keys):
    """16-byte keys as (hi, lo) big-endian u64 pairs: lexicographic row order = byte order (memcmp)."""
    k = np.ascontiguousarray(keys, dtype=np.uint8).reshape(-1, 16)
    return k.view(">u8").astype(np.uint64).reshape(-1, 2)


def maintain(corpus, payload, term_keys, sealed_deleted, growing):
    """-> (Corpus, payload [N', 3] u16, term_keys [T', 16] u8 or None, relabel [N + G] u32)

    corpus: the sealed segment (oracle.Corpus); payload [N, 3] or None (= synthetic_ctid of the doc id); term_keys
    [T, 16] or None (keyless); sealed_deleted [N] or None; growing: Vectors or None."""
    N, T = corpus.n_docs, corpus.n_terms
    sdel = np.zeros(N, bool) if sealed_deleted is None else np.asarray(sealed_deleted).astype(bool)
    G = growing.n_docs if growing is not None else 0
    gdel = growing.deleted if growing is not None else np.zeros(0, bool)

    # 1. new document order (maintain.rs:55-73,167-255; io.rs:52-60,187-197): sealed survivors by doc id, then growing
    #    survivors in chain order; dense ids from 0
    alive_s, alive_g = np.nonzero(~sdel)[0], np.nonzero(~gdel)[0]
    ns = len(alive_s)
    relabel = np.full(N + G, DOC_NONE, dtype=np.uint32)
    relabel[alive_s] = np.arange(ns)
    relabel[N + alive_g] = ns + np.arange(len(alive_g))

    # deleted documents and their postings vanish (add_element returns early on u32::MAX, maintain.rs:353-355)
    df = (corpus.post_off[1:] - corpus.post_off[:-1]).astype(np.int64)
    s_term = np.repeat(np.arange(T, dtype=np.int64), df)
    keep = ~sdel[corpus.post_doc] if len(corpus.post_doc) else np.zeros(0, bool)
    s_term, s_old, s_tf = s_term[keep], corpus.post_doc[keep], corpus.post_tf[keep]
    s_doc = relabel[s_old].astype(np.int64)

    # 2. lengths: a sealed survivor is re-recorded as Record(0, payload) (maintain.rs:337) and each of its postings adds 1
    #    (maintain.rs:356-360): its number of distinct tokens.  A growing one: saturating Σ tf over all its elements
    #    (vector.rs:77-83, io.rs:193)
    s_len = np.bincount(s_old, minlength=N)[alive_s] if N else np.zeros(0, np.int64)
    if growing is not None:
        cnt = (growing.elem_off[1:] - growing.elem_off[:-1]).astype(np.int64)
        g_doc_of_elem = np.repeat(np.arange(G), cnt)
        tf_sum = np.bincount(g_doc_of_elem, weights=growing.elem_tf.astype(np.float64), minlength=G)
        g_len = np.minimum(tf_sum[alive_g], 0xFFFFFFFF)
        e_keep = ~gdel[g_doc_of_elem]
        g_doc = relabel[N + g_doc_of_elem[e_keep]].astype(np.int64)
        g_tf = growing.elem_tf[e_keep]
    else:
        g_len, g_doc, g_tf = np.zeros(0), np.zeros(0, np.int64), np.zeros(0, np.uint32)
    doc_len = np.concatenate([s_len, g_len]).astype(np.uint32)

    # 3. tokens: those that still have a posting, ascending by byte order (io::locally_merge sorts Mapping(key, doc, tf);
    #    flush.rs writes the tokens of the mappings).  Keyless surface: ordinals stay, the vocabulary grows to
    #    max ordinal + 1
    if term_keys is not None:
        sk = _key_u64(term_keys)[s_term] if len(s_term) else np.zeros((0, 2), np.uint64)
        gk = _key_u64(growing.elem_key[e_keep]) if growing is not None and len(g_tf) else np.zeros((0, 2), np.uint64)
        allk = np.concatenate([sk, gk])
        uniq, inv = np.unique(allk, axis=0, return_inverse=True) if len(allk) else (np.zeros((0, 2), np.uint64),
                                                                                    np.zeros(0, np.int64))
        inv = np.asarray(inv).reshape(-1)
        new_term = inv.astype(np.int64)
        T_new = len(uniq)
        new_keys = uniq.astype(">u8").view(np.uint8).reshape(-1, 16).copy()
    else:
        g_term = growing.elem_term[e_keep].astype(np.int64) if growing is not None else np.zeros(0, np.int64)
        new_term = np.concatenate([s_term, g_term])
        T_new = max(T, int(g_term.max()) + 1 if len(g_term) else 0)
        new_keys = None

    # inside a token: sealed survivors (relabelled, order kept) then growing postings — sorting by (token, new doc id)
    doc = np.concatenate([s_doc, g_doc])
    tf = np.concatenate([s_tf, g_tf]).astype(np.uint32)
    order = np.lexsort((doc, new_term))
    off = np.zeros(T_new + 1, dtype=np.uint64)
    np.cumsum(np.bincount(new_term, minlength=T_new), out=off[1:])
    new_corpus = oracle.Corpus(ns + len(alive_g), doc_len, T_new, off, doc[order].astype(np.uint32), tf[order],
                               corpus.k1, corpus.b)

    # 4. payload (ctid) carried over unchanged
    spl = synthetic_ctid(np.arange(N)) if payload is None else np.asarray(payload, np.uint16).reshape(-1, 3)
    if growing is not None:
        gpl = synthetic_ctid(np.arange(G)) if growing.payload is None else growing.payload
    else:
        gpl = np.zeros((0, 3), np.uint16)
    new_payload = np.concatenate([spl[alive_s], gpl[alive_g]]).astype(np.uint16)
    return new_corpus, new_payload, new_keys, relabel


def bulkdelete(payload, dead, deleted=None):
    """bulkdelete.rs:20-112 with the callback "is this ctid in the dead list": -> (marks, newly set)."""
    pl = np.asarray(payload, np.uint64).reshape(-1, 3)
    dd = np.asarray(dead, np.uint64).reshape(-1, 3)
    key = lambda a: (a[:, 0] << np.uint64(32)) | (a[:, 1] << np.uint64(16)) | a[:, 2]
    hit = np.isin(key(pl), key(dd))
    old = np.zeros(len(pl), bool) if deleted is None else np.asarray(deleted).astype(bool)
    return (old | hit).astype(np.uint8), int(np.count_nonzero(hit & ~old))
