"""Consumers of the k-mer stream that never write it: the bottom-s MinHash sketch under fx_hash
(`sketch(fx_hash, CanonicalDNAMers{16}(seq), 1000)`, /root/reference/docs/src/minhash.md:31-36) and
the composition vector (`counts[as_integer(kmer) + 1] += 1` over FwDNAMers{4},
/root/reference/docs/src/composition.md:28-39), against the oracle's k-mer streams."""
import numpy as np
import pytest

import kmertools as kt
from oracle import oracle as ko

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def kc():
    import kmerscuda
    return kmerscuda


def oracle_hashes(words, n, k, canonical):
    a, _, h = ko.iterate(words, n, k, ko.CANON if canonical else ko.FW, want_hash=True)
    return a, h


@pytest.mark.parametrize("k", [1, 4, 16, 31, 32, 33, 63])
def test_minhash_sketch_single_sequence(kc, k):
    rng = np.random.default_rng(k)
    for n in (0, k - 1, k, 5000, 200_003):
        words = rng.integers(0, 2**64, size=max((n + 31) // 32, 1), dtype=np.uint64)
        rs = kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, words, n))
        for canonical in (True, False):
            for s in (1, 10, 1000, 100_000):
                got = kc.minhash_sketch(rs, k, s, canonical=canonical)
                assert np.array_equal(got, ko.minhash_sketch(words, n, k, s, canonical)), (k, n, canonical, s)


def test_minhash_sketch_duplicates_force_a_higher_threshold(kc):
    """A set whose small hashes are heavily duplicated: the first threshold bucket holds >= s k-mers
    but fewer than s distinct ones, so the second pass has to be repeated."""
    rng = np.random.default_rng(5)
    unit = kt.random_dna(rng, 40)
    s_txt = unit * 2000 + kt.random_dna(rng, 3000)
    words = kt.pack2(s_txt)
    n = len(s_txt)
    rs = kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, words, n))
    _, h = oracle_hashes(words, n, 16, True)
    distinct = np.unique(h)
    for s in (5, 64, 1000, 5000):
        assert np.array_equal(kc.minhash_sketch(rs, 16, s), distinct[:s])
    # homopolymer: one distinct k-mer
    words = kt.pack2("A" * 10_000)
    rs = kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, words, 10_000))
    _, h = oracle_hashes(words, 10_000, 21, True)
    assert np.array_equal(kc.minhash_sketch(rs, 21, 100), np.unique(h))


def test_minhash_sketch_read_sets(kc):
    rng = np.random.default_rng(6)
    n_reads, length, stride, k = 5000, 150, 5, 21
    words = rng.integers(0, 2**64, size=n_reads * stride, dtype=np.uint64)
    rs = kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride)
    _, _, h, _ = ko.batch_iterate(words, n_reads, k, ko.CANON, uniform_len=length, uniform_stride=stride, want_hash=True)
    assert np.array_equal(kc.minhash_sketch(rs, k, 1000), np.unique(h)[:1000])
    lens = rng.integers(0, 400, size=700).astype(np.uint64)
    off = np.zeros(len(lens) + 1, dtype=np.uint64)
    off[1:] = np.cumsum((lens + 31) // 32)
    words = rng.integers(0, 2**64, size=int(off[-1]) + 1, dtype=np.uint64)
    rs = kc.ReadSet(2, words, len(lens), seq_word_offset=off[:-1].copy(), seq_len=lens)
    _, _, h, _ = ko.batch_iterate(words, len(lens), k, ko.CANON, word_off=off[:-1].copy(), seq_len=lens, want_hash=True)
    assert np.array_equal(kc.minhash_sketch(rs, k, 333), np.unique(h)[:333])


@pytest.mark.parametrize("k", [1, 2, 4, 6, 7, 8, 11])
def test_composition(kc, k):
    rng = np.random.default_rng(100 + k)
    n = 300_007
    words = rng.integers(0, 2**64, size=(n + 31) // 32, dtype=np.uint64)
    rs = kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, words, n))
    for canonical in (False, True):
        want = ko.composition(words, n, k, canonical)
        got, total, _ = kc.composition(rs, k, canonical=canonical)
        assert total == n - k + 1 and np.array_equal(got, want)
    # the reference's own example shape: FwDNAMers{4} over a 10 000 bp record
    n_reads, length, stride = 999, 150, 5
    words = rng.integers(0, 2**64, size=n_reads * stride, dtype=np.uint64)
    rs = kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride)
    a, _, _, _ = ko.batch_iterate(words, n_reads, k, ko.FW, uniform_len=length, uniform_stride=stride)
    got, total, _ = kc.composition(rs, k)
    assert np.array_equal(got, np.bincount(a[:, 0].astype(np.int64), minlength=4**k).astype(np.uint32))


def test_argument_checks(kc):
    rs = kc.ReadSet.single(kc.LongDNA2("ACGT" * 50))
    with pytest.raises(kc.KmersCUDAError):
        kc.composition(rs, 15)
    with pytest.raises(kc.KmersCUDAError):
        kc.minhash_sketch(rs, 65, 10)
    with pytest.raises(kc.KmersCUDAError):
        kc.minhash_sketch(rs, 16, 0)


# ------------------------------------------------------------------------------ exact k-mer counts
@pytest.mark.parametrize("k,canonical", [(1, True), (5, False), (16, True), (21, True), (31, False), (32, True)])
def test_kmer_table_matches_unique_counts(kc, k, canonical):
    rng = np.random.default_rng(500 + k)
    # a genome sampled by overlapping reads: most k-mers occur many times
    genome = rng.integers(0, 4, size=20_000).astype(np.uint64)
    n_reads, length, stride = 4000, 150, 5
    starts = rng.integers(0, len(genome) - length, size=n_reads)
    codes = np.zeros((n_reads, stride * 32), dtype=np.uint64)
    for r, s0 in enumerate(starts):
        codes[r, :length] = genome[s0:s0 + length]
    words = np.concatenate([kt.pack_codes(row, 2) for row in codes])
    rs = kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride)
    a, _, _, _ = ko.batch_iterate(words, n_reads, k, ko.CANON if canonical else ko.FW, uniform_len=length, uniform_stride=stride)
    want_k, want_c = np.unique(a[:, 0], return_counts=True)
    t = kc.KmerTable(17)
    n, _ = t.count(rs, k, canonical=canonical)
    assert n == a.shape[0] and t.n_keys == len(want_k)
    got_k, got_c = t.items()
    assert np.array_equal(got_k, want_k) and np.array_equal(got_c, want_c.astype(np.uint32))
    # counting the set again doubles every count; merging a second table adds it
    t.count(rs, k, canonical=canonical)
    t2 = kc.KmerTable(16)
    t2.count(rs, k, canonical=canonical)
    t.merge(t2)
    got_k, got_c = t.items()
    assert np.array_equal(got_k, want_k) and np.array_equal(got_c, 3 * want_c.astype(np.uint32))
    for x in (t, t2):
        x.free()


@pytest.mark.parametrize("k,canonical,log2cap,ragged", [(21, True, 24, False), (31, False, 24, True), (32, True, 28, True)])
def test_kmer_table_beyond_l2_takes_the_binned_path(kc, k, canonical, log2cap, ragged):
    """Tables larger than L2 (more than 96 MiB: 12 bytes per slot) are filled slice by slice from binned k-mers (64 bins
    for 2^24 slots, 256 for 2^28), from a uniform and from ragged sets; the result is the same table content."""
    count_twice(kc, k, canonical, log2cap, ragged)


def test_kmer_table_at_exactly_the_l2_budget_streams(kc):
    """2^23 one-limb slots are 96 MiB, exactly the L2 budget: the largest table that is still updated directly (the
    binned path starts above it)."""
    count_twice(kc, 21, True, 23, False)


def count_twice(kc, k, canonical, log2cap, ragged):
    """A 3000-read set from a 60 kbp genome counted into a fresh table of 2^log2cap slots, then once more."""
    rng = np.random.default_rng(900 + k)
    genome = rng.integers(0, 4, size=60_000).astype(np.uint64)
    n_reads = 3000
    lens = rng.integers(0, 260, size=n_reads) if ragged else np.full(n_reads, 150)
    seq_codes = []
    for ln in lens:
        s0 = int(rng.integers(0, len(genome) - 260))
        seq_codes.append(genome[s0:s0 + int(ln)])
    if ragged:
        words_l, off = [], [0]
        for c in seq_codes:
            w = kt.pack_codes(c, 2) if len(c) else np.zeros(0, dtype=np.uint64)
            words_l.append(w)
            off.append(off[-1] + len(w))
        words = np.concatenate(words_l) if words_l else np.zeros(0, dtype=np.uint64)
        off = np.asarray(off, dtype=np.uint64)
        ln = np.asarray(lens, dtype=np.uint64)
        rs = kc.ReadSet(2, words, n_reads, seq_word_offset=off, seq_len=ln)
        a, _, _, _ = ko.batch_iterate(words, n_reads, k, ko.CANON if canonical else ko.FW, word_off=off, seq_len=ln)
    else:
        codes = np.zeros((n_reads, 5 * 32), dtype=np.uint64)
        for r, c in enumerate(seq_codes):
            codes[r, :150] = c
        words = np.concatenate([kt.pack_codes(row, 2) for row in codes])
        rs = kc.ReadSet(2, words, n_reads, uniform_len=150, uniform_stride_words=5)
        a, _, _, _ = ko.batch_iterate(words, n_reads, k, ko.CANON if canonical else ko.FW, uniform_len=150, uniform_stride=5)
    want_k, want_c = np.unique(a[:, 0], return_counts=True)
    t = kc.KmerTable(log2cap)
    n, _ = t.count(rs, k, canonical=canonical)
    assert n == a.shape[0] and t.n_keys == len(want_k)
    got_k, got_c = t.items()
    assert np.array_equal(got_k, want_k) and np.array_equal(got_c, want_c.astype(np.uint32))
    n, _ = t.count(rs, k, canonical=canonical)  # every key is already there
    assert t.n_keys == len(want_k)
    got_k, got_c = t.items()
    assert np.array_equal(got_k, want_k) and np.array_equal(got_c, 2 * want_c.astype(np.uint32))
    t.free()


def test_kmer_table_full_and_argument_checks(kc):
    rng = np.random.default_rng(1)
    n = 10_000
    words = rng.integers(0, 2**64, size=(n + 31) // 32, dtype=np.uint64)
    rs = kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, words, n))
    t = kc.KmerTable(8)  # 256 slots for ~10 000 distinct 21-mers
    with pytest.raises(kc.KmersCUDAError, match="full"):
        t.count(rs, 21)
    t.free()
    t = kc.KmerTable(10)
    with pytest.raises(kc.KmersCUDAError):
        t.count(rs, 33)
    with pytest.raises(kc.KmersCUDAError):
        t.count(rs, 32, canonical=False)
    t.free()
