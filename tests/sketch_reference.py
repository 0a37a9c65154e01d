"""numpy references of the per-sequence MinHash sketches and of the all-pairs sketch comparison.

The sketches come from the oracle's k-mer streams (`oracle.batch_iterate`); the comparison is written from the set
definitions alone and is itself pinned against brute force over Python sets
(tests/test_oracle_minhash_compare.py).
"""
import numpy as np

from oracle import oracle as ko


def minhash_sketches(words, n_seqs, k, s, canonical=True, *, word_off=None, seq_len=None, uniform_len=0, uniform_stride=0):
    """The bottom-s sketch of every sequence on its own, from the oracle's k-mer streams: row i = np.unique(h_i)[:s],
    padded with ~0, and the row lengths.  Arguments as for oracle.batch_iterate."""
    _, _, h, off = ko.batch_iterate(words, n_seqs, k, ko.CANON if canonical else ko.FW, word_off=word_off, seq_len=seq_len,
                                    uniform_len=uniform_len, uniform_stride=uniform_stride, want_hash=True)
    if off is None:
        w = max(0, uniform_len - k + 1)
        off = np.arange(n_seqs + 1, dtype=np.uint64) * np.uint64(w)
    rows = np.full((n_seqs, s), ~np.uint64(0), dtype=np.uint64)
    lens = np.zeros(n_seqs, dtype=np.uint32)
    for i in range(n_seqs):
        u = np.unique(h[int(off[i]):int(off[i + 1])])[:s]
        rows[i, :len(u)] = u
        lens[i] = len(u)
    return rows, lens


def minhash_compare(a, a_n, b, b_n, s):
    """All pairs of two lists of bottom-s sketches, from the set definitions: for rows A_i = a[i, :min(a_n[i], s)] and
    B_j = b[j, :min(b_n[j], s)], shared[i, j] = |A_i ∩ B_j| and shared_bottom[i, j] = |S_s(A_i ∪ B_j) ∩ A_i ∩ B_j|,
    S_s = the s smallest values (the numerator of Mash's Jaccard estimate)."""
    a, b = np.asarray(a, dtype=np.uint64), np.asarray(b, dtype=np.uint64)
    rows_a = [np.unique(a[i, :min(int(a_n[i]), s)]) for i in range(len(a_n))]
    rows_b = [np.unique(b[j, :min(int(b_n[j]), s)]) for j in range(len(b_n))]
    shared = np.zeros((len(rows_a), len(rows_b)), dtype=np.uint32)
    bottom = np.zeros_like(shared)
    for i, x in enumerate(rows_a):
        for j, y in enumerate(rows_b):
            both = np.intersect1d(x, y, assume_unique=True)
            shared[i, j] = len(both)
            bottom[i, j] = len(np.intersect1d(np.union1d(x, y)[:s], both, assume_unique=True))
    return shared, bottom
