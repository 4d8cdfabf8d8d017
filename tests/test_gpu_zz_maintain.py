"""GPU: bm25x_index_maintain / bm25x_bulkdelete (bm25::maintain, maintain.rs:27-311; bm25::bulkdelete,
bulkdelete.rs:20-112).

Expected values come from the numpy restatement (tests/maintain_oracle.py) only.  Bar: the maintained handle is
byte-identical (all 13 device arrays) to bm25x_index_create of the restated corpus with its payload and keys, and its
searches are bit-exact against the oracle's exhaustive scorer on that corpus.  (File name: runs after the other GPU
tests.)"""
import struct

import numpy as np
import pytest

import _pkg
import maintain_oracle as mo
from test_gpu_blocks import _device_arrays, _from_blocks
from test_gpu_parity import _compare

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def m():
    mod = _pkg.load()
    mod.load_library()
    assert mod.device_count() >= 1, "no CUDA device: the engine has no CPU fallback"
    return mod


def _oc(orc, c):
    return orc.Corpus(c.n_docs, c.doc_len, c.n_terms, c.post_off, c.post_doc, c.post_tf)


def _create(m, c, payload=None, keys=None):
    return m.Index(c.n_docs, c.doc_len, c.n_terms, c.post_off, c.post_doc, c.post_tf, c.k1, c.b, payload=payload,
                   term_keys=keys)


def _bits(x):
    return struct.pack("<d", x)


def _vectors(m, orc, seed, n, vocab, zipf, keys=None, deleted_every=5):
    """Growing documents over ordinals [0, vocab); with `keys` ([vocab, 16], sorted) their tokens are those keys."""
    fresh = orc.Corpus.synth(seed, n, vocab, 1, 60, zipf_s=zipf)
    g = orc.GrowingDocs.from_corpus(fresh)
    deleted = (np.arange(n) % deleted_every == 2).astype(np.uint8)
    if keys is None:
        return mo.Vectors(g.elem_off, g.elem_tf, elem_term=g.elem_term, deleted=deleted)
    return mo.Vectors(g.elem_off, g.elem_tf, elem_key=keys[g.elem_term], deleted=deleted)


def _maintain(ix, sdel, vec):
    if vec is None:
        return ix.maintain(deleted=sdel)
    return ix.maintain(deleted=sdel, elem_off=vec.elem_off, elem_key=vec.elem_key, elem_term=vec.elem_term,
                       elem_tf=vec.elem_tf, payload=vec.payload, growing_deleted=vec.deleted)


def _check(m, orc, new, relabel, sealed_corpus, payload, keys, sdel, vec, what, search=True):
    """The maintained handle against the restatement; returns the expected (corpus, payload, keys)."""
    ec, epl, ek, erel = mo.maintain(sealed_corpus, payload, keys, sdel, vec)
    assert np.array_equal(relabel, erel), f"{what}: relabel"
    ref = _create(m, ec, payload=epl, keys=ek)
    for i, (a, b) in enumerate(zip(_device_arrays(ref), _device_arrays(new))):
        assert np.array_equal(a, b), f"{what}: device array {i} differs from create() of the maintained corpus"
    gi, ri = new.info(), ref.info()
    for f in ("n_docs", "n_terms", "n_postings", "n_blocks", "sum_doc_len"):
        assert getattr(gi, f) == getattr(ri, f), f"{what}: info.{f}"
    assert _bits(gi.avgdl) == _bits(ri.avgdl) and gi.n_docs == ec.n_docs and gi.n_terms == ec.n_terms
    if ek is not None and len(ek):
        assert new.lookup_terms(ek).tolist() == list(range(len(ek)))
    if search:
        oix = orc.OracleIndex(ec)
        q_off, q_terms = m.synth_queries(len(what) * 7919 + 5, 40, ec.n_terms, 1, 8, ec.post_off)
        for seed in (1, 0):
            new.set_option("seed", seed)
            for k in (1, 10, 100, 1000):
                _compare(new.search_batch(q_off, q_terms, k), oix, q_off, q_terms, k, what=f"{what} seed={seed}")
        new.set_option("seed", 1)
    ref.close()
    return ec, epl, ek


def _random_keys(rng, n):
    k = rng.integers(1, 256, size=(n * 2, 16), dtype=np.uint8)
    k = np.unique(k, axis=0)[:n]                  # rows sorted = byte order
    assert len(k) == n
    return np.ascontiguousarray(k)


CONFIGS = [
    dict(name="uniform", seed=301, n=20000, vocab=3000, lmin=8, lmax=80, zipf=0.0, ng=1500, extra=0),
    dict(name="zipf_new_ordinals", seed=302, n=30000, vocab=5000, lmin=16, lmax=96, zipf=1.0, ng=2000, extra=300),
    dict(name="keyed", seed=303, n=20000, vocab=3000, lmin=8, lmax=80, zipf=0.8, ng=1500, extra=400, keyed=True),
    dict(name="from_blocks", seed=304, n=12000, vocab=800, lmin=4, lmax=200, zipf=0.7, ng=1000, extra=50, blocks=True),
    dict(name="dense", seed=305, n=6000, vocab=60, lmin=5, lmax=300, zipf=1.1, ng=800, extra=5),
]


@pytest.mark.parametrize("cfg", CONFIGS, ids=[c["name"] for c in CONFIGS])
def test_maintain_byte_identical_and_search_exact(m, orc, cfg):
    c = m.synth_corpus(cfg["seed"], cfg["n"], cfg["vocab"], cfg["lmin"], cfg["lmax"], cfg["zipf"])
    oc = _oc(orc, c)
    rng = np.random.default_rng(cfg["seed"])
    sdel = (rng.integers(0, 7, c.n_docs) == 0).astype(np.uint8)
    keys = gkeys = None
    if cfg.get("keyed"):
        universe = _random_keys(rng, cfg["vocab"] + cfg["extra"])
        sel = np.sort(rng.choice(len(universe), cfg["vocab"], replace=False))
        keys, gkeys = universe[sel], universe
    vec = _vectors(m, orc, cfg["seed"] + 1, cfg["ng"], cfg["vocab"] + cfg["extra"], cfg["zipf"], keys=gkeys)
    if cfg.get("blocks"):
        fn = np.array([orc.lib().orc_length_to_fieldnorm(int(x)) for x in c.doc_len], dtype=np.uint8)
        _, ix = _from_blocks(m, orc, c, doc_len=None, doc_fieldnorm=fn, sum_doc_len=int(c.doc_len.astype(np.uint64).sum()))
    else:
        ix = m.Index.from_corpus(c, term_keys=keys)
    new, relabel, st = _maintain(ix, sdel, vec)
    _check(m, orc, new, relabel, oc, None, keys, sdel, vec, cfg["name"])
    assert st.postings_in == c.n_postings + len(vec.elem_tf) and st.postings_out == new.info().n_postings
    assert st.device_ms > 0 and st.total_ms >= st.device_ms
    new.close()
    ix.close()


def test_length_quirk_on_the_device(m, orc):
    rng = np.random.default_rng(7)
    docs = [{int(t): 1 for t in rng.choice(50, rng.integers(1, 12), replace=False)} for _ in range(3000)]
    ones = orc.Corpus.from_docs(docs, n_terms=50)
    ix = _create(m, ones)
    new, relabel, _ = ix.maintain()
    assert relabel.tolist() == list(range(3000))
    for a, b in zip(_device_arrays(ix), _device_arrays(new)):     # all tf = 1: nothing changes
        assert np.array_equal(a, b)
    new.close()
    ix.close()
    for d in docs[::3]:
        for t in d:
            d[t] = int(rng.integers(1, 9))
    heavy = orc.Corpus.from_docs(docs, n_terms=50)
    ix = _create(m, heavy)
    new, _, _ = ix.maintain()
    distinct = orc.Corpus(heavy.n_docs, [len(d) for d in docs], heavy.n_terms, heavy.post_off, heavy.post_doc,
                          heavy.post_tf)
    ref = _create(m, distinct)
    got, want, old = _device_arrays(new), _device_arrays(ref), _device_arrays(ix)
    assert all(np.array_equal(a, b) for a, b in zip(got, want))   # lengths = distinct tokens (maintain.rs:337,356-360)
    assert not all(np.array_equal(a, b) for a, b in zip(got, old))
    assert _bits(new.info().avgdl) == _bits(ref.info().avgdl) != _bits(ix.info().avgdl)
    for x in (new, ref, ix):
        x.close()


def test_edges(m, orc):
    c = m.synth_corpus(311, 5000, 400, 4, 60, 0.6)
    oc = _oc(orc, c)
    ix = m.Index.from_corpus(c)
    vec = _vectors(m, orc, 312, 600, 450, 0.6)
    # every growing document deleted
    gone = mo.Vectors(vec.elem_off, vec.elem_tf, elem_term=vec.elem_term, deleted=np.ones(vec.n_docs, np.uint8))
    sdel = (np.arange(c.n_docs) % 9 == 4).astype(np.uint8)
    new, relabel, _ = _maintain(ix, sdel, gone)
    _check(m, orc, new, relabel, oc, None, None, sdel, gone, "growing_all_deleted", search=False)
    new.close()
    # every sealed document deleted, growing ones survive
    alld = np.ones(c.n_docs, np.uint8)
    new, relabel, _ = _maintain(ix, alld, vec)
    _check(m, orc, new, relabel, oc, None, None, alld, vec, "sealed_all_deleted")
    # maintain of a maintained handle = the restatement applied twice
    ec, epl, _, _ = mo.maintain(oc, None, None, alld, vec)
    sdel2 = (np.arange(ec.n_docs) % 4 == 1).astype(np.uint8)
    vec2 = _vectors(m, orc, 313, 300, 470, 0.6)
    pl2 = np.arange(vec2.n_docs * 3, dtype=np.uint16).reshape(-1, 3) + 7
    vec2.payload = pl2
    new2, relabel2, _ = _maintain(new, sdel2, vec2)
    ec2, epl2, _ = _check(m, orc, new2, relabel2, ec, epl, None, sdel2, vec2, "twice")
    head = int(np.argmax(np.diff(ec2.post_off.astype(np.int64))))
    res = new2.search_batch(np.array([0, 1], np.uint32), np.array([head], np.uint32), 50, want_payload=True)
    assert res["n"][0] == 50
    for r in range(50):                                              # payloads travel with their documents
        assert res["payload"][0, r].tolist() == epl2[res["doc"][0, r]].tolist()
    # growing() on a maintained handle
    fresh = orc.Corpus.synth(314, 400, new2.n_terms, 1, 40)
    g = orc.GrowingDocs.from_corpus(fresh)
    gix = new2.growing(g.elem_off, g.elem_term, g.elem_tf, doc_len=g.doc_len)
    oix2 = orc.OracleIndex(ec2)
    q_off, q_terms = m.synth_queries(315, 30, ec2.n_terms, 1, 6, ec2.post_off)
    r = gix.search_batch(q_off, q_terms, 20)
    for i in range(len(q_off) - 1):
        gd, gs = oix2.search_growing(g, q_terms[q_off[i]:q_off[i + 1]], 20)
        n = int(r["n"][i])
        assert n == len(gd) and np.array_equal(r["doc"][i, :n], gd) and np.array_equal(r["score64"][i, :n], gs)
    for x in (gix, new2, new, ix):
        x.close()


def test_dead_token(m, orc):
    kA, kB, kC = (np.array([v] + [0] * 15, np.uint8) for v in (0x11, 0x22, 0x33))
    docs = [{0: 1, 2: 1}, {1: 3}, {0: 2}, {2: 1}]
    c = orc.Corpus.from_docs(docs)
    keys = np.stack([kA, kB, kC])
    sdel = np.array([0, 1, 0, 0], np.uint8)                         # kB lives in document 1 only
    ix = _create(m, c, keys=keys)
    new, relabel, _ = ix.maintain(deleted=sdel)
    _check(m, orc, new, relabel, c, None, keys, sdel, None, "dead_key", search=False)
    assert new.lookup_terms(keys).tolist() == [0, m.TERM_MISSING, 1]
    new.close()
    ix.close()
    ix = _create(m, c)                                               # keyless: the ordinal stays with df 0
    new, relabel, _ = ix.maintain(deleted=sdel)
    _check(m, orc, new, relabel, c, None, None, sdel, None, "dead_ordinal", search=False)
    assert new.df().tolist() == [2, 0, 2]
    assert new.search([1], 10)[0].size == 0
    assert new.search([0, 1], 10)[0].tolist() == [1, 0]             # doc 2 (tf 2, length 1 now) ranks first
    new.close()
    ix.close()


def test_errors_leave_the_sealed_handle_alone(m, orc):
    c = m.synth_corpus(321, 3000, 200, 4, 40, 0.5)
    ix = m.Index.from_corpus(c)
    q_off, q_terms = m.synth_queries(322, 30, 200, 1, 5, c.post_off)
    before = ix.search_batch(q_off, q_terms, 50)
    off = np.array([0, 2], np.uint64)
    E = m.Bm25xError

    def raises(code, match, **kw):
        with pytest.raises(E, match=match) as ei:
            ix.maintain(**kw)
        assert ei.value.code == code
    raises(1, "strictly ascending", elem_off=off, elem_term=[5, 4], elem_tf=[1, 1])
    raises(1, "tf != 0", elem_off=off, elem_term=[4, 5], elem_tf=[1, 0])
    raises(1, "TERM_MISSING", elem_off=off, elem_term=[4, m.TERM_MISSING], elem_tf=[1, 1])
    raises(1, "term keys given", elem_off=off, elem_key=np.zeros((2, 16), np.uint8), elem_tf=[1, 1])
    raises(4, "2\\^24", elem_off=off, elem_term=[4, 5], elem_tf=[1, 1 << 24])
    raises(1, "no document survives", deleted=np.ones(c.n_docs, np.uint8))
    raises(1, "no document survives", deleted=np.ones(c.n_docs, np.uint8), elem_off=off, elem_term=[4, 5],
           elem_tf=[1, 1], growing_deleted=[1])
    keys = _random_keys(np.random.default_rng(3), c.n_terms)
    kix = m.Index.from_corpus(c, term_keys=keys)
    with pytest.raises(E, match="term ordinals given") as ei:
        kix.maintain(elem_off=off, elem_term=[4, 5], elem_tf=[1, 1])
    assert ei.value.code == 1
    with pytest.raises(E, match="strictly ascending"):
        kix.maintain(elem_off=off, elem_key=keys[[5, 4]], elem_tf=[1, 1])
    kix.close()
    g = ix.growing(off, [1, 2], [1, 1], doc_len=[2])
    with pytest.raises(E, match="growing handle") as ei:
        g.maintain()
    assert ei.value.code == 1
    g.close()
    h = m.Index._adopt(None, 0, 0)
    with pytest.raises(E, match="null argument"):
        h.maintain()
    after = ix.search_batch(q_off, q_terms, 50)                     # after failed calls
    assert np.array_equal(before["doc"], after["doc"]) and np.array_equal(before["score64"], after["score64"])
    new, _, _ = ix.maintain(deleted=(np.arange(c.n_docs) % 2).astype(np.uint8))
    after = ix.search_batch(q_off, q_terms, 50)                     # after a successful one
    assert np.array_equal(before["doc"], after["doc"]) and np.array_equal(before["score64"], after["score64"])
    new.close()
    ix.close()


def test_pcie_rule(m, orc):
    c = m.synth_corpus(331, 20000, 5000, 64, 128)                    # >= 64 postings per document
    ix = m.Index.from_corpus(c)
    sdel = (np.arange(c.n_docs) % 7 == 3).astype(np.uint8)
    vec = _vectors(m, orc, 332, 300, 5100, 0.0)
    new, relabel, st = _maintain(ix, sdel, vec)
    assert st.h2d_bytes + st.d2h_bytes < st.postings_in, (st.h2d_bytes, st.d2h_bytes, st.postings_in)
    _check(m, orc, new, relabel, _oc(orc, c), None, None, sdel, vec, "pcie", search=False)
    new.close()
    ix.close()


def test_bulkdelete(m, orc):
    c = m.synth_corpus(341, 4000, 300, 4, 40, 0.5)
    rng = np.random.default_rng(341)
    default_pl = mo.synthetic_ctid(np.arange(c.n_docs))
    explicit_pl = np.sort(rng.integers(0, 1 << 16, size=(c.n_docs, 3)).astype(np.uint16), axis=0)
    for pl, kw in ((default_pl, {}), (explicit_pl, {"payload": explicit_pl})):
        ix = m.Index.from_corpus(c, **kw)
        dead = pl[rng.choice(c.n_docs, 500)]
        dead = np.concatenate([dead, rng.integers(0, 1 << 16, size=(50, 3)).astype(np.uint16)])   # unknown tids too
        dead = dead[np.lexsort((dead[:, 2], dead[:, 1], dead[:, 0]))]
        want, want_n = mo.bulkdelete(pl, dead)
        got, n = ix.bulkdelete(dead)
        assert np.array_equal(got, want) and n == want_n
        earlier = (np.arange(c.n_docs) % 11 == 0).astype(np.uint8)  # marks are kept, only new ones are counted
        want, want_n = mo.bulkdelete(pl, dead, earlier)
        got, n = ix.bulkdelete(dead, earlier)
        assert np.array_equal(got, want) and n == want_n
        assert ix.bulkdelete(dead, got)[1] == 0
        with pytest.raises(m.Bm25xError, match="sorted") as ei:
            ix.bulkdelete(dead[::-1])
        assert ei.value.code == 1
        # bulkdelete -> maintain end to end
        new, relabel, _ = ix.maintain(deleted=got)
        _check(m, orc, new, relabel, _oc(orc, c), kw.get("payload"), None, got, None, "bulkdelete", search=False)
        new.close()
        ix.close()
    # a growing handle: its own payloads (default = synthetic ctid of the growing ordinal, or explicit)
    ix = m.Index.from_corpus(c)
    g = orc.GrowingDocs.from_corpus(orc.Corpus.synth(342, 700, 300, 1, 30))
    for gpl in (None, np.sort(rng.integers(0, 1 << 16, size=(700, 3)).astype(np.uint16), axis=0)):
        gix = ix.growing(g.elem_off, g.elem_term, g.elem_tf, doc_len=g.doc_len, payload=gpl)
        pl = mo.synthetic_ctid(np.arange(700)) if gpl is None else gpl
        dead = pl[np.sort(rng.choice(700, 90, replace=False))]
        got, n = gix.bulkdelete(dead)
        want, want_n = mo.bulkdelete(pl, dead)
        assert np.array_equal(got, want) and n == want_n >= 90
        gix.close()
    ix.close()
