"""A bottom-s MinHash sketch per sequence (kmc_minhash_sketch_each) and all-pairs sketch comparison
(kmc_minhash_compare), exactly against the references: every row equals np.unique(h_i)[:s] of the oracle's stream of
sequence i and the single-set sketch of that sequence alone; every pair count equals the set definitions."""
import numpy as np
import pytest

import kmertools as kt
import sketch_reference as ref
from oracle import oracle as ko

pytestmark = pytest.mark.gpu

ALL = ~np.uint64(0)


@pytest.fixture(scope="module")
def kc():
    import kmerscuda
    return kmerscuda


def ragged(rng, lens, gap_words=0):
    """A ragged set of random sequences with the given lengths, each starting on its own word."""
    lens = np.asarray(lens, dtype=np.uint64)
    need = (lens + 31) // 32 + gap_words
    off = np.zeros(len(lens) + 1, dtype=np.uint64)
    off[1:] = np.cumsum(need)
    words = rng.integers(0, 2**64, size=max(int(off[-1]), 1), dtype=np.uint64)
    return words, off[:-1].copy(), lens


def check_rows(kc, rows, lens, want_rows, want_lens, s):
    assert rows.shape == want_rows.shape and np.array_equal(lens, want_lens)
    assert np.array_equal(rows, want_rows)
    for i in np.flatnonzero(lens < s)[:50]:
        assert np.all(rows[i, lens[i]:] == ALL)


def single_sketch(kc, words, off, n, k, s, canonical):
    """kmc_minhash_sketch of one sequence of a set on its own"""
    nw = max((n + 31) // 32, 1)
    w = np.zeros(nw, dtype=np.uint64)
    part = words[int(off): int(off) + nw]
    w[: len(part)] = part
    return kc.minhash_sketch(kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, w, n)), k, s, canonical=canonical)


@pytest.mark.parametrize("k", [1, 16, 21, 31, 32, 33, 63, 64])
@pytest.mark.parametrize("canonical", [False, True])
def test_rows_equal_the_single_set_sketch(kc, k, canonical):
    rng = np.random.default_rng(1000 + 2 * k + canonical)
    g = 8 if k <= 32 else 4
    for s in (1, 10, 1000):
        # uniform sets: windows per read a multiple of G (aligned work items) and not
        for wpr in (8 * g, 8 * g - 3, 1500):
            n_reads, length = 37, k - 1 + wpr
            stride = (length + 31) // 32 + 1
            words = rng.integers(0, 2**64, size=n_reads * stride, dtype=np.uint64)
            rs = kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride)
            rows, lens = kc.minhash_sketches(rs, k, s, canonical=canonical)
            want = ref.minhash_sketches(words, n_reads, k, s, canonical, uniform_len=length, uniform_stride=stride)
            check_rows(kc, rows, lens, *want, s)
            for i in (0, 17, n_reads - 1):
                one = single_sketch(kc, words, i * stride, length, k, s, canonical)
                assert np.array_equal(rows[i, : lens[i]], one), (k, s, wpr, i)
        # ragged: lengths 0..K-1 give empty rows, mixed with longer sequences
        lens_in = np.concatenate([np.arange(0, k), rng.integers(k, 3 * k + 2500, size=40)])
        rng.shuffle(lens_in)
        words, off, sl = ragged(rng, lens_in, gap_words=1)
        rs = kc.ReadSet(2, words, len(sl), seq_word_offset=off, seq_len=sl)
        rows, lens = kc.minhash_sketches(rs, k, s, canonical=canonical)
        want = ref.minhash_sketches(words, len(sl), k, s, canonical, word_off=off, seq_len=sl)
        check_rows(kc, rows, lens, *want, s)
        assert np.all(lens[sl < k] == 0)
        for i in range(0, len(sl), 9):
            one = single_sketch(kc, words, off[i], int(sl[i]), k, s, canonical)
            assert np.array_equal(rows[i, : lens[i]], one), (k, s, i)


@pytest.mark.parametrize("k", [21, 33])
def test_single_sequence_set_equals_the_set_sketch(kc, k):
    rng = np.random.default_rng(7 + k)
    for n in (0, k - 1, k, 5000, 200_003):
        words = rng.integers(0, 2**64, size=max((n + 31) // 32, 1), dtype=np.uint64)
        rs = kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, words, n))
        for canonical in (True, False):
            for s in (1, 1000):
                rows, lens = kc.minhash_sketches(rs, k, s, canonical=canonical)
                one = kc.minhash_sketch(rs, k, s, canonical=canonical)
                assert rows.shape == (1, s) and lens[0] == len(one) and np.array_equal(rows[0, : lens[0]], one)
                assert np.array_equal(one, ko.minhash_sketch(words, n, k, s, canonical))


def test_first_symbol_offset_views(kc):
    rng = np.random.default_rng(11)
    k, s, first = 21, 100, 13
    # a view of one sequence
    n_total = 50_000
    words = rng.integers(0, 2**64, size=(n_total + 31) // 32, dtype=np.uint64)
    n = n_total - first - 7
    rs = kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, words, n_total), first_symbol_offset=first, length=n)
    rows, lens = kc.minhash_sketches(rs, k, s)
    _, _, h = ko.iterate(words, n, k, ko.CANON, first=first, want_hash=True)
    assert np.array_equal(rows[0, : lens[0]], np.unique(h)[:s])
    # a uniform set of views: every read skips its first symbols
    n_reads, length, stride = 300, 150, 6
    words = rng.integers(0, 2**64, size=n_reads * stride, dtype=np.uint64)
    rs = kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride, first_symbol_offset=first)
    rows, lens = kc.minhash_sketches(rs, k, s, canonical=False)
    for i in range(n_reads):
        _, _, h = ko.iterate(words[i * stride:(i + 1) * stride], length, k, ko.FW, first=first, want_hash=True)
        u = np.unique(h)[:s]
        assert lens[i] == len(u) and np.array_equal(rows[i, : lens[i]], u), i


def test_a_tile_of_more_than_512_sequences(kc):
    """Short ragged reads: one tile of work items spans more than 512 sequences, so their descriptors are read from
    global memory (the unstaged locator path)."""
    rng = np.random.default_rng(12)
    k = 16
    lens_in = rng.integers(k, k + 3, size=6000)
    words, off, sl = ragged(rng, lens_in)
    rs = kc.ReadSet(2, words, len(sl), seq_word_offset=off, seq_len=sl)
    for s in (1, 10):
        rows, lens = kc.minhash_sketches(rs, k, s)
        check_rows(kc, rows, lens, *ref.minhash_sketches(words, len(sl), k, s, True, word_off=off, seq_len=sl), s)


def test_one_long_sequence_among_short_ones(kc):
    rng = np.random.default_rng(13)
    k, s = 21, 1000
    lens_in = np.concatenate([rng.integers(0, 3000, size=300), [10_000_000], rng.integers(0, 3000, size=300)])
    words, off, sl = ragged(rng, lens_in)
    rs = kc.ReadSet(2, words, len(sl), seq_word_offset=off, seq_len=sl)
    rows, lens, st = kc.minhash_sketches(rs, k, s, stats=True)
    check_rows(kc, rows, lens, *ref.minhash_sketches(words, len(sl), k, s, True, word_off=off, seq_len=sl), s)
    assert st["n_written"] == int(lens.sum())


def test_repeats_go_through_the_retry(kc):
    """A sequence of repeats has far fewer distinct k-mers than windows, so its first limit yields fewer than s distinct
    candidates and it is sketched again with a higher one; a homopolymer (one k-mer) goes up to the limit ~0."""
    rng = np.random.default_rng(5)
    unit = kt.random_dna(rng, 40)
    texts = [unit * 2000 + kt.random_dna(rng, 3000), "A" * 10_000, kt.random_dna(rng, 200_000)]
    seqs = [kc.LongSequence(kc.DNAAlphabet2, kt.pack2(t), len(t)) for t in texts]
    rs = kc.ReadSet.from_sequences(seqs)
    for s in (5, 64, 1000, 5000):
        rows, lens, st = kc.minhash_sketches(rs, 16, s, stats=True)
        for i, q in enumerate(seqs):
            want = ko.minhash_sketch(q.data, len(q), 16, s, True)
            assert lens[i] == len(want) and np.array_equal(rows[i, : lens[i]], want), (s, i)
        assert st["extra_rounds"] >= 1 and st["resketched"] >= 1, st
    rows, lens, st = kc.minhash_sketches(kc.ReadSet.from_sequences(seqs[1:2]), 21, 100, stats=True)
    assert lens[0] == 1 and st["extra_rounds"] == 2 and st["resketched"] == 2


def test_scale_2000_sequences(kc):
    rng = np.random.default_rng(14)
    k, s = 21, 1000
    lens_in = rng.integers(1000, 300_001, size=2000)
    words, off, sl = ragged(rng, lens_in)
    rs = kc.ReadSet(2, words, len(sl), seq_word_offset=off, seq_len=sl)
    rows, lens = kc.minhash_sketches(rs, k, s)
    for c0 in range(0, len(sl), 250):
        c1 = min(c0 + 250, len(sl))
        want = ref.minhash_sketches(words, c1 - c0, k, s, True, word_off=off[c0:c1], seq_len=sl[c0:c1])
        check_rows(kc, rows[c0:c1], lens[c0:c1], *want, s)


# ------------------------------------------------------------------------------------------------ all pairs
def random_sketches(rng, n, s, lens, universe):
    """n rows of distinct values drawn from `universe` (unique), ascending, ~0 past each row's length"""
    rows = np.full((n, s), ALL, dtype=np.uint64)
    lens = np.minimum(np.asarray(lens, dtype=np.int64), s).astype(np.uint32)
    for i in range(n):
        rows[i, : lens[i]] = np.sort(rng.choice(universe, size=int(lens[i]), replace=False))
    return rows, lens


def compare_both(kc, a, a_n, b, b_n, s):
    got = kc.minhash_compare(a, a_n, b, b_n)
    want = ref.minhash_compare(a, a_n, b, b_n, s)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    return got


@pytest.mark.parametrize("s", [1, 31, 32, 33, 1000, 4096, 16384])
def test_compare_random_shapes(kc, s):
    rng = np.random.default_rng(s)
    # a shared universe so that rows overlap; values near ~0 included
    universe = np.unique(np.concatenate([rng.integers(0, 2**64, size=3 * s + 64, dtype=np.uint64),
                                         np.array([0, 1, ALL - np.uint64(1), ALL], dtype=np.uint64)]))
    shapes = [(1, 1), (3, 70)] + ([(257, 129)] if s <= 1000 else [])
    for n_a, n_b in shapes:
        la = rng.integers(0, s + 1, size=n_a)
        lb = rng.integers(0, s + 1, size=n_b)
        la[: min(3, n_a)] = [0, 1, s][: min(3, n_a)]
        lb[: min(3, n_b)] = [s, 0, 1][: min(3, n_b)]
        if n_b > 5:
            lb[4] = s
        a, a_n = random_sketches(rng, n_a, s, la, universe)
        b, b_n = random_sketches(rng, n_b, s, lb, universe)
        if n_b > 5:
            b_n[4] = s + 5            # a length above s is read as s
            b[5] = a[min(2, n_a - 1)]  # identical rows
            b_n[5] = a_n[min(2, n_a - 1)]
        compare_both(kc, a, a_n, b, b_n, s)


@pytest.mark.parametrize("s", [1, 32, 1000])
def test_compare_identical_disjoint_nested_and_all_ones(kc, s):
    rng = np.random.default_rng(77 + s)
    base = np.unique(rng.integers(0, 2**63, size=2 * s + 10, dtype=np.uint64))
    even, odd = base[0::2][:s], base[1::2][:s]
    rows = [base[:s], base[:s], even, odd, base[: max(s // 2, 1)], np.append(base[: s - 1], ALL), np.array([ALL]), np.array([], np.uint64)]
    a = np.full((len(rows), s), ALL, dtype=np.uint64)
    a_n = np.zeros(len(rows), dtype=np.uint32)
    for i, r in enumerate(rows):
        r = np.sort(r)[:s]
        a[i, : len(r)] = r
        a_n[i] = len(r)
    shared, bottom = kc.minhash_compare(a, a_n)
    want = ref.minhash_compare(a, a_n, a, a_n, s)
    assert np.array_equal(shared, want[0]) and np.array_equal(bottom, want[1])
    assert np.array_equal(shared, shared.T) and np.array_equal(bottom, bottom.T)
    assert np.array_equal(np.diag(shared), a_n) and np.array_equal(np.diag(bottom), a_n)
    j = kc.mash_jaccard(shared, bottom, a_n, a_n, s)
    assert j[0, 1] == 1.0 and (s == 1 or j[2, 3] == 0.0)
    d = kc.mash_distance(j, 21)
    assert d[0, 1] == 0.0 and (s == 1 or d[2, 3] == 1.0)


def test_compare_self_is_symmetric(kc):
    rng = np.random.default_rng(3)
    s = 200
    universe = np.unique(rng.integers(0, 2**64, size=600, dtype=np.uint64))
    a, a_n = random_sketches(rng, 150, s, rng.integers(0, s + 1, size=150), universe)
    shared, bottom = kc.minhash_compare(a, a_n)
    assert np.array_equal(shared, shared.T) and np.array_equal(bottom, bottom.T)
    assert np.array_equal(np.diag(shared), np.minimum(a_n, s))
    want = ref.minhash_compare(a, a_n, a, a_n, s)
    assert np.array_equal(shared, want[0]) and np.array_equal(bottom, want[1])


def mutate(rng, seq, rate):
    out = seq.copy()
    m = rng.random(len(seq)) < rate
    out[m] = (out[m] + rng.integers(1, 4, size=int(m.sum()))) % 4
    return out


def test_compare_sketches_of_related_genomes(kc):
    rng = np.random.default_rng(21)
    k, s, n = 21, 1000, 200_000
    root = rng.integers(0, 4, size=n)
    genomes = [mutate(rng, root, r) for r in (0.0, 0.001, 0.01, 0.05, 0.1, 0.2)]
    seqs = [kc.LongSequence(kc.DNAAlphabet2, kt.pack_codes(g, 2), n) for g in genomes]
    rows, lens = kc.minhash_sketches(kc.ReadSet.from_sequences(seqs), k, s)
    shared, bottom = kc.minhash_compare(rows, lens)
    want = ref.minhash_compare(rows, lens, rows, lens, s)
    assert np.array_equal(shared, want[0]) and np.array_equal(bottom, want[1])
    j = kc.mash_jaccard(shared, bottom, lens, lens, s)
    assert np.all(np.diff(j[0]) <= 0)  # further from the root, fewer shared k-mers
    assert j[0, 0] == 1.0 and j[0, -1] < 0.05


def test_argument_checks(kc):
    import ctypes as C
    from kmerscuda import _abi
    ctx = kc.default_context()
    lib = ctx.lib
    rs = kc.ReadSet.single(kc.LongDNA2("ACGT" * 50))
    with pytest.raises(kc.KmersCUDAError):
        kc.minhash_sketches(rs, 65, 10)  # K > 64
    with pytest.raises(kc.KmersCUDAError):
        kc.minhash_sketches(rs, 16, 0)   # s < 1
    drs = kc.DeviceReadSet(ctx, rs)
    buf = ctx.alloc(1 << 12)
    res = _abi.kmc_result()
    f = lib.kmc_minhash_sketch_each
    assert f(ctx.handle, C.byref(drs.desc), 16, _abi.KMC_CANON, 0, buf.ptr, buf.ptr, C.byref(res)) == _abi.KMC_E_BAD_ARG
    assert f(ctx.handle, C.byref(drs.desc), 16, _abi.KMC_CANON, 2**62, buf.ptr, buf.ptr, C.byref(res)) == _abi.KMC_E_BAD_ARG
    assert f(ctx.handle, C.byref(drs.desc), 16, _abi.KMC_FWRV, 10, buf.ptr, buf.ptr, C.byref(res)) == _abi.KMC_E_BAD_ARG
    assert f(ctx.handle, C.byref(drs.desc), 16, _abi.KMC_CANON, 10, None, buf.ptr, C.byref(res)) == _abi.KMC_E_BAD_ARG
    assert f(ctx.handle, C.byref(drs.desc), 16, _abi.KMC_CANON, 10, buf.ptr, None, C.byref(res)) == _abi.KMC_E_BAD_ARG
    assert f(ctx.handle, C.byref(drs.desc), 16, _abi.KMC_CANON, 10, buf.ptr, buf.ptr, None) == _abi.KMC_E_BAD_ARG
    assert f(ctx.handle, C.byref(drs.desc), 65, _abi.KMC_CANON, 10, buf.ptr, buf.ptr, C.byref(res)) == _abi.KMC_E_UNSUPPORTED
    assert f(None, C.byref(drs.desc), 16, _abi.KMC_CANON, 10, buf.ptr, buf.ptr, C.byref(res)) == _abi.KMC_E_BAD_ARG
    four = _abi.kmc_seqs(drs.desc.words, drs.desc.n_words, 1, None, None, 50, drs.desc.n_words, 4, 0)
    assert f(ctx.handle, C.byref(four), 16, _abi.KMC_CANON, 10, buf.ptr, buf.ptr, C.byref(res)) == _abi.KMC_E_UNSUPPORTED
    # n_seqs = 0 writes nothing
    ctx._check(lib.kmc_memset(ctx.handle, buf.ptr, 0x5a, 1 << 12))
    empty = _abi.kmc_seqs(drs.desc.words, drs.desc.n_words, 0, None, None, 0, 0, 2, 0)
    assert f(ctx.handle, C.byref(empty), 16, _abi.KMC_CANON, 10, buf.ptr, buf.ptr, C.byref(res)) == _abi.KMC_OK
    assert res.n_written == 0 and np.all(buf.download(np.uint8, 1 << 12) == 0x5a)

    g = lib.kmc_minhash_compare
    assert g(ctx.handle, buf.ptr, buf.ptr, 1, buf.ptr, buf.ptr, 1, 0, buf.ptr, buf.ptr) == _abi.KMC_E_BAD_ARG
    assert g(ctx.handle, buf.ptr, buf.ptr, 1, buf.ptr, buf.ptr, 1, 16385, buf.ptr, buf.ptr) == _abi.KMC_E_UNSUPPORTED
    assert g(ctx.handle, None, buf.ptr, 1, buf.ptr, buf.ptr, 1, 4, buf.ptr, buf.ptr) == _abi.KMC_E_BAD_ARG
    assert g(ctx.handle, buf.ptr, buf.ptr, 1, buf.ptr, None, 1, 4, buf.ptr, buf.ptr) == _abi.KMC_E_BAD_ARG
    assert g(None, buf.ptr, buf.ptr, 1, buf.ptr, buf.ptr, 1, 4, buf.ptr, buf.ptr) == _abi.KMC_E_BAD_ARG
    ctx._check(lib.kmc_memset(ctx.handle, buf.ptr, 0x5a, 1 << 12))
    assert g(ctx.handle, None, None, 0, None, None, 5, 4, buf.ptr, buf.ptr) == _abi.KMC_OK  # n_a = 0 does nothing
    assert g(ctx.handle, buf.ptr, buf.ptr, 3, None, None, 0, 4, buf.ptr, buf.ptr) == _abi.KMC_OK
    assert np.all(buf.download(np.uint8, 1 << 12) == 0x5a)
    # one output may be NULL
    a = np.array([[1, 2, 3, 4]], dtype=np.uint64)
    da, dn, out = ctx.to_device(a), ctx.to_device(np.array([4], np.uint32)), ctx.alloc(8)
    assert g(ctx.handle, da.ptr, dn.ptr, 1, da.ptr, dn.ptr, 1, 4, None, out.ptr) == _abi.KMC_OK
    assert out.download(np.uint32, 1)[0] == 4
    for d in (buf, da, dn, out):
        d.free()
