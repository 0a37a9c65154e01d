"""Read-only queries of the exact k-mer tables (one and two limbs): the count of every window of a read set
(KmerTable.lookup / kmc_kmer_lookup(2)), of given keys (get), the count spectrum (histogram) and the count-filtered
export (items(min_count, max_count)).  Every expectation comes from np.unique(..., return_counts=True) of the oracle's
k-mer stream.  The tables are counted from one read set and looked up with another, half of whose reads come from a
second genome, so that hits and misses both occur."""
import ctypes as C

import numpy as np
import pytest

import kmertools as kt
from oracle import oracle as ko

ALL_ONES = np.uint64(2**64 - 1)


@pytest.fixture(scope="module")
def kc():
    import kmerscuda
    return kmerscuda


def n_limbs_of(k):
    return 1 if k <= 32 else 2


# ------------------------------------------------------------------------------------------------------ read sets
def uniform_reads(kc, rng, genome, n_reads, length):
    stride = (length + 31) // 32
    starts = rng.integers(0, len(genome) - length + 1, size=n_reads)
    codes = np.zeros((n_reads, stride * 32), dtype=np.uint64)
    codes[:, :length] = genome[starts[:, None] + np.arange(length)[None, :]]
    words = kt.pack_codes(codes.reshape(-1), 2)
    return kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride), words, n_reads, dict(
        uniform_len=length, uniform_stride=stride)


def ragged_reads(kc, rng, genome, n_reads, max_len):
    """Reads of 0 .. max_len symbols, empty reads and reads shorter than K among them."""
    lens = rng.integers(0, max_len + 1, size=n_reads)
    lens[:6] = [0, 1, 14, 31, 32, 63]
    words_l, off = [], [0]
    for ln in lens:
        s0 = int(rng.integers(0, len(genome) - max_len))
        w = kt.pack_codes(genome[s0:s0 + int(ln)], 2) if ln else np.zeros(0, dtype=np.uint64)
        words_l.append(w)
        off.append(off[-1] + len(w))
    words = np.concatenate(words_l)
    off = np.asarray(off[:-1], dtype=np.uint64)
    ln = np.asarray(lens, dtype=np.uint64)
    return kc.ReadSet(2, words, n_reads, seq_word_offset=off, seq_len=ln), words, n_reads, dict(word_off=off, seq_len=ln)


def single_sequence(kc, codes):
    words = kt.pack_codes(codes, 2)
    return kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, words, len(codes))), words, len(codes)


def stream(words, n_reads, k, canonical, layout):
    """The oracle's k-mer stream (rows of limbs, kmc_extract's order)."""
    a, _, _, _ = ko.batch_iterate(words, n_reads, k, ko.CANON if canonical else ko.FW, **layout)
    return a


def counts_of(table_stream, query_stream):
    """For every row of query_stream, how often it occurs in table_stream (np.unique with counts over both)."""
    both = np.concatenate([table_stream, query_stream])
    _, inv, _ = np.unique(both, axis=0, return_inverse=True, return_counts=True)
    inv = inv.reshape(-1)
    in_table = np.bincount(inv[:len(table_stream)], minlength=int(inv.max()) + 1 if len(inv) else 0)
    return in_table[inv[len(table_stream):]].astype(np.uint32)


def unique_counts(a):
    uk, uc = np.unique(a, axis=0, return_counts=True)
    return (uk[:, 0] if a.shape[1] == 1 else uk), uc.astype(np.uint32)


def table_from(kc, rs, k, canonical, log2cap):
    t = kc.KmerTable(log2cap, n_limbs=n_limbs_of(k))
    t.count(rs, k, canonical=canonical)
    return t


def genomes(seed, n=30_000):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 4, size=n).astype(np.uint64)
    b = rng.integers(0, 4, size=n).astype(np.uint64)
    return rng, a, np.concatenate([a, b])  # the query genome: the table's genome and a second one


# ------------------------------------------------------------------------------------------------------ lookup parity
LOOKUP_CASES = [(1, False), (1, True), (15, False), (15, True), (31, False), (31, True), (32, True),
                (33, False), (33, True), (47, False), (47, True), (63, False), (63, True), (64, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("k,canonical", LOOKUP_CASES)
def test_lookup_matches_oracle_counts(kc, k, canonical):
    from kmerscuda import _abi
    rng, ga, gb = genomes(1000 + 2 * k + canonical)
    rs_a, wa, na, la = uniform_reads(kc, rng, ga, 3000, 150)
    sa = stream(wa, na, k, canonical, la)
    t = table_from(kc, rs_a, k, canonical, 17)
    for make, arg in ((uniform_reads, 150), (ragged_reads, 200)):
        rs_b, wb, nb, lb = make(kc, rng, gb, 3000, arg)
        sb = stream(wb, nb, k, canonical, lb)
        want = counts_of(sa, sb)
        assert (want > 0).any() and (k < 8 or (want == 0).any())  # (every 1-mer occurs in both sets)
        got = t.lookup(rs_b, k, canonical=canonical)
        assert got.dtype == np.uint32 and np.array_equal(got, want)
    # one sequence whose last group of windows is partial (for G = 8 and G = 4)
    length = 40_000 + k - 1 + 3
    rs_s, ws, ns = single_sequence(kc, gb[:length])
    a, _, _ = ko.iterate(ws, ns, k, ko.CANON if canonical else ko.FW)
    assert np.array_equal(t.lookup(rs_s, k, canonical=canonical), counts_of(sa, a))
    # out_counts 4 bytes past an aligned base: every group takes the scalar stores
    rs_b, wb, nb, lb = uniform_reads(kc, rng, gb, 2000, 150)
    want = counts_of(sa, stream(wb, nb, k, canonical, lb))
    n = len(want)
    buf = t.ctx.alloc(4 * (n + 2))
    t.ctx._check(t.ctx.lib.kmc_memset(t.ctx.handle, buf.ptr, 0xAB, 4 * (n + 2)))
    drs = kc.DeviceReadSet(t.ctx, rs_b)
    res = _abi.kmc_result()
    fn = t._fn("kmc_kmer_lookup")
    t.ctx._check(fn(t.ctx.handle, C.byref(drs.desc), k, kc.KMC_CANON if canonical else kc.KMC_FW, t.keys.ptr, t.vals.ptr,
                    t.log2_capacity, buf.ptr + 4, n, C.byref(res)))
    assert res.n_written == n
    out = buf.download(np.uint32, n + 2)
    assert np.array_equal(out[1:n + 1], want)
    assert out[0] == 0xABABABAB and out[n + 1] == 0xABABABAB
    buf.free()
    # the counts can stay on the device
    d = t.lookup(rs_b, k, canonical=canonical, device_out=True)
    assert np.array_equal(d.download(np.uint32, n), want)
    d.free()
    t.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k,log2cap", [(31, 24), (63, 23)])
def test_lookup_beyond_l2(kc, k, log2cap):
    """2^24 one-limb slots (192 MB) and 2^23 two-limb slots (160 MB): filled by the binned count, probed directly."""
    rng, ga, gb = genomes(77 + k, 60_000)
    rs_a, wa, na, la = uniform_reads(kc, rng, ga, 4000, 150)
    sa = stream(wa, na, k, True, la)
    t = table_from(kc, rs_a, k, True, log2cap)
    for make, arg in ((uniform_reads, 150), (ragged_reads, 260)):
        rs_b, wb, nb, lb = make(kc, rng, gb, 4000, arg)
        assert np.array_equal(t.lookup(rs_b, k), counts_of(sa, stream(wb, nb, k, True, lb)))
    t.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [21, 40])
def test_lookup_and_get_in_a_full_table(kc, k):
    """A completely full table (the count overflowed): the probe of an absent key ends after 2^cap slots."""
    rng = np.random.default_rng(5 + k)
    codes = rng.integers(0, 4, size=5000).astype(np.uint64)
    rs, w, n = single_sequence(kc, codes)
    t = kc.KmerTable(8, n_limbs=n_limbs_of(k))
    with pytest.raises(kc.KmersCUDAError, match="full"):
        t.count(rs, k)
    L = t.n_limbs
    dk, dv = t.ctx.alloc(8 * L * 256), t.ctx.alloc(4 * 256)
    n_out = C.c_uint64(0)
    t.ctx._check(t._fn("kmc_kmer_table_export")(t.ctx.handle, t.keys.ptr, t.vals.ptr, 8, dk.ptr, dv.ptr, 256, C.byref(n_out)))
    assert n_out.value == 256  # every slot holds a key
    keys, vals = dk.download(np.uint64, 256 * L).reshape(256, L), dv.download(np.uint32, 256)
    a, _, _ = ko.iterate(w, n, k, ko.CANON)
    # a key in the table holds its exact count; every other k-mer of the sequence is absent
    uk, uc = np.unique(a, axis=0, return_counts=True)
    present = counts_of(keys, uk) > 0
    assert present.sum() == 256
    assert np.array_equal(counts_of(a, keys), vals)
    q = uk if L == 2 else uk[:, 0]
    assert np.array_equal(t.get(q), np.where(present, uc, 0).astype(np.uint32))
    free = np.full((1, 2), ALL_ONES) if L == 2 else np.full(1, ALL_ONES)
    assert t.get(free)[0] == 0
    per_window = counts_of(uk[present], a)  # 0 for the k-mers that found no slot
    want = np.where(per_window > 0, counts_of(a, a), 0).astype(np.uint32)
    assert np.array_equal(t.lookup(rs, k), want)
    dk.free()
    dv.free()
    t.free()


# ------------------------------------------------------------------------------------------------------ get
@pytest.mark.gpu
def test_get_edge_keys(kc):
    from kmerscuda import _abi
    rng, ga, gb = genomes(31)
    for k in (31, 63):
        rs, w, n, lay = uniform_reads(kc, rng, ga, 2000, 150)
        a = stream(w, n, k, True, lay)
        uk, uc = unique_counts(a)
        t = table_from(kc, rs, k, True, 16)
        assert np.array_equal(t.get(uk), uc)
        # absent keys, the free marker(s), n = 0
        if k == 31:
            q = np.concatenate([uk[:10] ^ np.uint64(1 << 61), np.array([ALL_ONES], dtype=np.uint64)])
        else:
            q = np.concatenate([uk[:10] ^ np.uint64(1 << 61), np.array([[ALL_ONES, ALL_ONES], [ALL_ONES, 7]], dtype=np.uint64)])
        q = q[counts_of(a, q if k == 63 else q[:, None]) == 0]
        assert len(q) >= 10 and not t.get(q).any()
        assert t.get(np.zeros((0,) if k == 31 else (0, 2), dtype=np.uint64)).shape == (0,)
        assert t._fn("kmc_kmer_table_get")(t.ctx.handle, t.keys.ptr, t.vals.ptr, t.log2_capacity, None, 0, None) == 0
        with pytest.raises(ValueError):
            t.get(np.zeros((3, 2) if k == 31 else (3,), dtype=np.uint64))
        t.free()
    # K = 64: T^32 A^32 is canonical and has limb 0 = ~0; {~0, x} for another x is absent
    special = np.array([3] * 32 + [0] * 32, dtype=np.uint64)
    codes = rng.integers(0, 4, size=(500, 150)).astype(np.uint64)
    codes[:, 40:104] = special
    stride = 5
    padded = np.zeros((500, stride * 32), dtype=np.uint64)
    padded[:, :150] = codes
    words = kt.pack_codes(padded.reshape(-1), 2)
    rs = kc.ReadSet(2, words, 500, uniform_len=150, uniform_stride_words=stride)
    a = stream(words, 500, 64, True, dict(uniform_len=150, uniform_stride=stride))
    uk, uc = unique_counts(a)
    t = table_from(kc, rs, 64, True, 16)
    got = t.get(np.array([[ALL_ONES, 0], [ALL_ONES, 1], [ALL_ONES, ALL_ONES]], dtype=np.uint64))
    row = np.flatnonzero((uk[:, 0] == ALL_ONES) & (uk[:, 1] == 0))
    assert len(row) == 1 and got[0] == uc[row[0]] >= 500
    assert got[1] == 0 and got[2] == 0
    assert np.array_equal(t.get(uk), uc)
    # misaligned two-limb queries are a status, not a device fault
    q = t.ctx.to_device(uk[:4].copy())
    out = t.ctx.alloc(16)
    lib = t.ctx.lib
    assert lib.kmc_kmer_table2_get(t.ctx.handle, t.keys.ptr, t.vals.ptr, 16, q.ptr + 8, 2, out.ptr) == _abi.KMC_E_BAD_ARG
    assert lib.kmc_kmer_table2_get(t.ctx.handle, t.keys.ptr + 8, t.vals.ptr, 16, q.ptr, 2, out.ptr) == _abi.KMC_E_BAD_ARG
    assert lib.kmc_kmer_table2_get(t.ctx.handle, t.keys.ptr, t.vals.ptr, 0, q.ptr, 2, out.ptr) == _abi.KMC_E_BAD_ARG
    assert lib.kmc_kmer_table2_get(t.ctx.handle, t.keys.ptr, t.vals.ptr, 16, None, 2, out.ptr) == _abi.KMC_E_BAD_ARG
    q.free()
    out.free()
    t.free()


# ------------------------------------------------------------------------------------------------------ histogram
@pytest.mark.gpu
@pytest.mark.parametrize("k", [31, 63])
def test_histogram(kc, k):
    from kmerscuda import _abi
    rng, ga, _ = genomes(50 + k, 20_000)
    rs, w, n, lay = uniform_reads(kc, rng, ga, 4000, 150)
    _, uc = unique_counts(stream(w, n, k, True, lay))
    t = table_from(kc, rs, k, True, 17)
    for n_bins in (1, 2, 256, 16384):
        want = np.bincount(np.minimum(uc, n_bins - 1), minlength=n_bins).astype(np.uint64)
        assert np.array_equal(t.histogram(n_bins), want), n_bins
    # it accumulates: twice into one buffer doubles it
    lib, ctx = t.ctx.lib, t.ctx
    h = ctx.alloc(8 * 256)
    ctx._check(lib.kmc_memset(ctx.handle, h.ptr, 0, 8 * 256))
    for _ in range(2):
        ctx._check(t._fn("kmc_kmer_table_histogram")(ctx.handle, t.keys.ptr, t.vals.ptr, t.log2_capacity, h.ptr, 256))
    assert np.array_equal(h.download(np.uint64, 256), 2 * np.bincount(np.minimum(uc, 255), minlength=256).astype(np.uint64))
    fn = t._fn("kmc_kmer_table_histogram")
    assert fn(ctx.handle, t.keys.ptr, t.vals.ptr, t.log2_capacity, h.ptr, 0) == _abi.KMC_E_BAD_ARG
    assert fn(ctx.handle, t.keys.ptr, t.vals.ptr, t.log2_capacity, h.ptr, 16385) == _abi.KMC_E_BAD_ARG
    assert fn(ctx.handle, t.keys.ptr, t.vals.ptr, 41, h.ptr, 16) == _abi.KMC_E_BAD_ARG
    assert fn(ctx.handle, t.keys.ptr, t.vals.ptr, t.log2_capacity, None, 16) == _abi.KMC_E_BAD_ARG
    if k == 63:
        assert fn(ctx.handle, t.keys.ptr + 8, t.vals.ptr, t.log2_capacity, h.ptr, 16) == _abi.KMC_E_BAD_ARG
    # a merged entry with count 0 is a key in bin 0
    key = np.array([[5, 9]] if k == 63 else [5], dtype=np.uint64)
    dkey, dval = ctx.to_device(key), ctx.to_device(np.zeros(1, dtype=np.uint32))
    ctx._check(t._fn("kmc_kmer_table_merge")(ctx.handle, t.keys.ptr, t.vals.ptr, t.log2_capacity, dkey.ptr, dval.ptr, 1, None))
    hist = t.histogram(256)
    assert hist[0] == 1 and hist[1:].sum() == len(uc)
    h.free()
    t.free()
    # poly-A: one key, counted once per window, lands in the last bin
    codes = np.zeros((300, 150), dtype=np.uint64)
    padded = np.zeros((300, 160), dtype=np.uint64)
    padded[:, :150] = codes
    rs = kc.ReadSet(2, kt.pack_codes(padded.reshape(-1), 2), 300, uniform_len=150, uniform_stride_words=5)
    t = table_from(kc, rs, k, True, 10)
    hist = t.histogram(256)
    assert hist[255] == 1 and hist.sum() == 1
    t.free()


# ------------------------------------------------------------------------------------------------------ filtered export
@pytest.mark.gpu
@pytest.mark.parametrize("k", [31, 63])
def test_export_range(kc, k):
    from kmerscuda import _abi
    rng, ga, _ = genomes(60 + k, 20_000)
    rs, w, n, lay = uniform_reads(kc, rng, ga, 4000, 150)
    uk, uc = unique_counts(stream(w, n, k, True, lay))
    t = table_from(kc, rs, k, True, 17)
    all_k, all_v = t.items()
    for lo, hi in ((1, 2**32 - 1), (0, 2**32 - 1), (5, 10), (20, 20), (0, 0), (10**6, 10**6), (int(uc.max()), 2**32 - 1)):
        keep = (uc >= lo) & (uc <= hi)
        gk, gv = t.items(min_count=lo, max_count=hi)
        assert np.array_equal(gk, uk[keep]) and np.array_equal(gv, uc[keep]), (lo, hi)
    gk, gv = t.items(min_count=1, max_count=2**32 - 1)
    assert np.array_equal(gk, all_k) and np.array_equal(gv, all_v)
    gk, _ = t.items(min_count=3)
    assert np.array_equal(gk, uk[uc >= 3])
    # a too-small capacity: KMC_E_OUT_TOO_SMALL, *n_out = how many there are, nothing past the buffer
    ctx, L = t.ctx, t.n_limbs
    m = int(((uc >= 2) & (uc <= 30)).sum())
    cap, guard = m - 7, 64
    dk, dv = ctx.alloc(8 * L * (cap + guard)), ctx.alloc(4 * (cap + guard))
    ctx._check(ctx.lib.kmc_memset(ctx.handle, dk.ptr, 0x5A, 8 * L * (cap + guard)))
    ctx._check(ctx.lib.kmc_memset(ctx.handle, dv.ptr, 0x5A, 4 * (cap + guard)))
    n_out = C.c_uint64(0)
    fn = t._fn("kmc_kmer_table_export_range")
    assert fn(ctx.handle, t.keys.ptr, t.vals.ptr, t.log2_capacity, 2, 30, dk.ptr, dv.ptr, cap, C.byref(n_out)) == _abi.KMC_E_OUT_TOO_SMALL
    assert n_out.value == m
    assert (dk.download(np.uint64, L * (cap + guard))[L * cap:] == np.uint64(0x5A5A5A5A5A5A5A5A)).all()
    assert (dv.download(np.uint32, cap + guard)[cap:] == np.uint32(0x5A5A5A5A)).all()
    assert fn(ctx.handle, t.keys.ptr, t.vals.ptr, t.log2_capacity, 31, 30, dk.ptr, dv.ptr, cap, C.byref(n_out)) == _abi.KMC_E_BAD_ARG
    assert fn(ctx.handle, t.keys.ptr, t.vals.ptr, 0, 2, 30, dk.ptr, dv.ptr, cap, C.byref(n_out)) == _abi.KMC_E_BAD_ARG
    assert fn(ctx.handle, t.keys.ptr, t.vals.ptr, t.log2_capacity, 2, 30, dk.ptr, dv.ptr, cap, None) == _abi.KMC_E_BAD_ARG
    if k == 63:
        assert fn(ctx.handle, t.keys.ptr, t.vals.ptr, t.log2_capacity, 2, 30, dk.ptr + 8, dv.ptr, cap, C.byref(n_out)) == _abi.KMC_E_BAD_ARG
    dk.free()
    dv.free()
    t.free()


# ------------------------------------------------------------------------------------------------------ lookup checks
@pytest.mark.gpu
def test_lookup_argument_checks(kc):
    from kmerscuda import _abi
    rng, ga, _ = genomes(9, 5000)
    rs, w, n, lay = uniform_reads(kc, rng, ga, 500, 150)
    one, two = table_from(kc, rs, 31, True, 14), table_from(kc, rs, 63, True, 14)
    for t, bad in ((one, [(33, True), (32, False)]), (two, [(32, True), (64, False), (65, True)])):
        for k, canonical in bad:
            with pytest.raises(kc.KmersCUDAError):
                t.lookup(rs, k, canonical=canonical)
    rs4 = kc.ReadSet.single(kc.LongDNA4("ACGT" * 50))
    with pytest.raises(kc.KmersCUDAError, match="2-bit"):
        one.lookup(rs4, 21)
    with pytest.raises(kc.KmersCUDAError, match="2-bit"):
        two.lookup(rs4, 41)
    # capacity < windows: KMC_E_OUT_TOO_SMALL and nothing written
    ctx, lib = one.ctx, one.ctx.lib
    drs = kc.DeviceReadSet(ctx, rs)
    windows = 500 * (150 - 31 + 1)
    buf = ctx.alloc(4 * windows)
    ctx._check(lib.kmc_memset(ctx.handle, buf.ptr, 0x77, 4 * windows))
    res = _abi.kmc_result()
    st = lib.kmc_kmer_lookup(ctx.handle, C.byref(drs.desc), 31, kc.KMC_CANON, one.keys.ptr, one.vals.ptr, 14, buf.ptr, windows - 1,
                             C.byref(res))
    assert st == _abi.KMC_E_OUT_TOO_SMALL and res.n_written == windows
    assert (buf.download(np.uint32, windows) == np.uint32(0x77777777)).all()
    # NULL pointers, log2_capacity, misaligned two-limb keys
    assert lib.kmc_kmer_lookup(ctx.handle, C.byref(drs.desc), 31, kc.KMC_CANON, None, one.vals.ptr, 14, buf.ptr, windows,
                               C.byref(res)) == _abi.KMC_E_BAD_ARG
    assert lib.kmc_kmer_lookup(ctx.handle, C.byref(drs.desc), 31, kc.KMC_CANON, one.keys.ptr, one.vals.ptr, 14, None, windows,
                               C.byref(res)) == _abi.KMC_E_BAD_ARG
    assert lib.kmc_kmer_lookup(ctx.handle, C.byref(drs.desc), 31, kc.KMC_CANON, one.keys.ptr, one.vals.ptr, 41, buf.ptr, windows,
                               C.byref(res)) == _abi.KMC_E_BAD_ARG
    assert lib.kmc_kmer_lookup2(ctx.handle, C.byref(drs.desc), 63, kc.KMC_CANON, two.keys.ptr + 8, two.vals.ptr, 14, buf.ptr, windows,
                                C.byref(res)) == _abi.KMC_E_BAD_ARG
    assert "aligned" in lib.kmc_last_error(ctx.handle).decode()
    buf.free()
    one.free()
    two.free()
