"""CPU: the numpy restatement of bm25::maintain (tests/maintain_oracle.py) on hand-worked cases.  Every expected corpus
is written out literally; the GPU tests take their expected values from this restatement."""
import numpy as np

from oracle import oracle
import maintain_oracle as mo

NONE = mo.DOC_NONE


def _key(b):
    return np.array([b] + [0] * 15, dtype=np.uint8)


def _same(c, n_docs, doc_len, off, doc, tf):
    assert c.n_docs == n_docs and c.n_terms == len(off) - 1
    assert c.doc_len.tolist() == doc_len
    assert c.post_off.tolist() == off
    assert c.post_doc.tolist() == doc and c.post_tf.tolist() == tf


def test_keyless_deletes_lengths_and_vocabulary():
    sealed = oracle.Corpus.from_docs([{0: 3, 1: 1}, {1: 2, 2: 1}, {2: 1}, {0: 1, 3: 1}])
    growing = mo.Vectors.from_docs([{1: 3, 5: 1}, {0: 1}, {2: 2}], deleted=[0, 1, 0])
    c, pl, keys, relabel = mo.maintain(sealed, None, None, [0, 1, 0, 0], growing)
    # sealed 0, 2, 3 then growing 0, 2; sealed doc 0 has tfs (3, 1): length 2; growing doc 0 has tfs (3, 1): length 4
    assert relabel.tolist() == [0, NONE, 1, 2, 3, NONE, 4]
    _same(c, 5, [2, 1, 2, 4, 2],
          off=[0, 2, 4, 6, 7, 7, 8],          # ordinal 4 is nobody's (df 0); ordinal 5 is new: vocabulary = 6
          doc=[0, 2, 0, 3, 1, 4, 2, 3],
          tf=[3, 1, 1, 3, 1, 2, 1, 1])
    assert keys is None
    # payloads: the synthetic ctids of sealed doc ids 0, 2, 3 and of growing ordinals 0, 2
    assert pl.tolist() == [[0, 0, 1], [0, 0, 3], [0, 0, 4], [0, 0, 1], [0, 0, 3]]


def test_keyed_dead_key_vanishes_new_key_sorted_in():
    kA, kB, kC, kD, kE = (_key(v) for v in (0x10, 0x20, 0x30, 0x40, 0x50))
    sealed_keys = np.stack([kA, kC, kD])
    sealed = oracle.Corpus.from_docs([{0: 1, 1: 2}, {2: 5}, {0: 2}])
    gkeys = np.stack([kA, kB, kC, kD, kE])
    growing = mo.Vectors.from_docs([{1: 1, 2: 1}, {4: 2}], keys=gkeys, payload=[[0, 2, 1], [0, 2, 2]],
                                   deleted=[0, 1])
    c, pl, keys, relabel = mo.maintain(sealed, [[0, 1, 1], [0, 1, 2], [0, 1, 3]], sealed_keys, [0, 1, 0], growing)
    assert relabel.tolist() == [0, NONE, 1, 2, NONE]
    # kD held only the deleted document: gone; kE only a deleted growing one: never there; kB is inserted before kC.
    # sealed doc 2 has one token with tf 2: length 1
    assert keys.tolist() == [kA.tolist(), kB.tolist(), kC.tolist()]
    _same(c, 3, [2, 1, 2], off=[0, 2, 3, 5], doc=[0, 1, 2, 0, 2], tf=[1, 2, 1, 2, 1])
    assert pl.tolist() == [[0, 1, 1], [0, 1, 3], [0, 2, 1]]


def test_compaction_only_changes_lengths_only_when_some_tf_exceeds_one():
    ones = oracle.Corpus.from_docs([{0: 1, 2: 1}, {1: 1}, {0: 1, 1: 1, 2: 1}])
    c, _, _, relabel = mo.maintain(ones, None, None, None, None)
    assert relabel.tolist() == [0, 1, 2]
    _same(c, 3, [2, 1, 3], ones.post_off.tolist(), ones.post_doc.tolist(), ones.post_tf.tolist())
    heavy = oracle.Corpus.from_docs([{0: 4, 2: 1}, {1: 7}])
    assert heavy.doc_len.tolist() == [5, 7]
    c, _, _, _ = mo.maintain(heavy, None, None, None, None)
    _same(c, 2, [2, 1], heavy.post_off.tolist(), heavy.post_doc.tolist(), heavy.post_tf.tolist())


def test_everything_sealed_deleted_growing_survives():
    sealed = oracle.Corpus.from_docs([{0: 1}, {1: 1}])
    growing = mo.Vectors.from_docs([{1: 2}, {3: 1}])
    c, pl, _, relabel = mo.maintain(sealed, None, None, [1, 1], growing)
    assert relabel.tolist() == [NONE, NONE, 0, 1]
    _same(c, 2, [2, 1], off=[0, 0, 1, 1, 2], doc=[0, 1], tf=[2, 1])
    assert pl.tolist() == [[0, 0, 1], [0, 0, 2]]


def test_bulkdelete_predicate():
    payload = [[0, 0, 1], [0, 0, 2], [0, 1, 1], [1, 0, 1]]
    marks, n = mo.bulkdelete(payload, [[0, 0, 2], [0, 0, 2], [1, 0, 1]], deleted=[1, 0, 0, 1])
    assert marks.tolist() == [1, 1, 0, 1] and n == 1   # doc 3 was marked already; doc 1 is new
