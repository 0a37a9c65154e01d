"""GPU parity: libkmerscuda (through the C ABI) against the CPU oracle, bit-exact.

Every test here calls the CUDA library; the oracle (oracle/) is only the checker.  The bar is
bit-exact equality of every limb, hash and index.
"""
import ctypes as C
import json
import os

import numpy as np
import pytest

import kmertools as kt
from oracle import oracle as ko

pytestmark = pytest.mark.gpu

KATS = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_kats.json")))
DIFF = KATS["differential_sequences"]
MODES = {"fw": 0, "fwrv": 1, "canon": 2, "unambig": 3}


@pytest.fixture(scope="module")
def kc():
    import kmerscuda
    return kmerscuda


@pytest.fixture(scope="module")
def ctx(kc):
    return kc.default_context()


def dna(s):
    return s.upper().replace("U", "T")


def rows(a):
    return [tuple(int(v) for v in r) for r in a]


# ----------------------------------------------------------------------------- golden vectors
def test_kat_fx_hash(kc):
    for e in KATS["fx_hash"]:
        limbs = [int(x, 16) for x in e["limbs"]] if "limbs" in e else list(kt.kmer_limbs(dna(e["kmer"])))
        got = kc.fx_hash(np.array([limbs], dtype=np.uint64).reshape(1, len(limbs)))
        assert int(got[0]) == int(e["hash"], 16), e


def test_kat_canonical(kc):
    for e in KATS["canonical"]:
        got = kc.CanonicalDNAMers(e["k"], kc.LongDNA2(dna(e["seq"]))).collect()
        assert rows(got) == [kt.kmer_limbs(dna(x)) for x in e["expect"]]


def test_kat_fwrv(kc):
    for e in KATS["fwrv"]:
        got = kc.FwRvDNAIterator(e["k"], kc.LongDNA2(dna(e["seq"]))).collect()  # [n, 2, N]
        assert rows(got[:, 0, :]) == [kt.kmer_limbs(p[0]) for p in e["expect"]]
        assert rows(got[:, 1, :]) == [kt.kmer_limbs(p[1]) for p in e["expect"]]


def test_kat_encoding(kc):
    for e in KATS["as_integer"]:
        got = kc.FwDNAMers(len(e["kmer"]), kc.LongDNA2(e["kmer"])).collect()
        assert rows(got) == [(int(e["value"], 16),)]


def test_kat_iscanonical(kc):
    for e in KATS["iscanonical"]:
        k = len(e["kmer"])
        fwrv = kc.FwRvDNAIterator(k, kc.LongDNA2(e["kmer"])).collect()
        fw, rv = tuple(map(int, fwrv[0, 0])), tuple(map(int, fwrv[0, 1]))
        assert (fw <= rv) == e["value"]
        assert rv == kt.kmer_limbs(kt.revcomp(e["kmer"]))


@pytest.mark.parametrize("key", ["fw_2bit", "smaller_than_k", "fwrv", "fwrv_k9", "canonical", "unambiguous_2bit"])
def test_reference_differential_sequences_2bit(kc, key):
    e = DIFF[key]
    k = e["k"]
    for s in map(dna, e["seqs"]):
        seq = kc.LongDNA2(s)
        assert rows(kc.FwDNAMers(k, seq).collect()) == kt.naive_fw(s, k)
        fr = kc.FwRvDNAIterator(k, seq).collect()
        want = kt.naive_fwrv(s, k)
        assert rows(fr[:, 0, :]) == [w[0] for w in want] and rows(fr[:, 1, :]) == [w[1] for w in want]
        assert rows(kc.CanonicalDNAMers(k, seq).collect()) == kt.naive_canonical(s, k)
        km, pos = kc.UnambiguousDNAMers(k, seq).collect()
        assert rows(km) == kt.naive_fw(s, k) and pos.tolist() == list(range(1, len(s) - k + 2))


# ------------------------------------------------------------------- randomised, vs the oracle
KS = [1, 2, 5, 13, 14, 16, 29, 30, 31, 32, 33, 47, 48, 49, 63, 64, 65, 80, 81, 96, 97, 112, 113, 127, 128]


@pytest.mark.parametrize("k", KS)
def test_single_sequence_all_modes(kc, k):
    rng = np.random.default_rng(0xCCFB + k)
    for length in sorted({0, k - 1, k, k + 1, k + 2, k + 3, k + 4, k + 5, k + 31, k + 32, k + 33, 3 * k + 257, 1000}):
        s = kt.random_dna(rng, max(length, 0))
        w = kt.pack2(s)
        seq = kc.LongSequence(kc.DNAAlphabet2, w, len(s))
        rs = kc.ReadSet.single(seq)
        a, b, h = ko.iterate(w, len(s), k, ko.FWRV, want_hash=True)
        e = kc.extract(MODES["fwrv"], rs, k, hash=True)
        assert np.array_equal(e.kmers, a) and np.array_equal(e.rv, b) and np.array_equal(e.hash, h)
        e = kc.extract(MODES["fwrv"], rs, k, aos=True)
        assert np.array_equal(e.kmers[:, 0, :], a) and np.array_equal(e.kmers[:, 1, :], b)
        c, _, hc = ko.iterate(w, len(s), k, ko.CANON, want_hash=True)
        e = kc.extract(MODES["canon"], rs, k, hash=True)
        assert np.array_equal(e.kmers, c) and np.array_equal(e.hash, hc)
        e = kc.extract(MODES["fw"], rs, k)
        assert np.array_equal(e.kmers, a)
        km, pos = ko.unambiguous(w, len(s), k, src_bits=2)
        e = kc.extract(MODES["unambig"], rs, k)
        assert np.array_equal(e.kmers, km) and np.array_equal(e.index, pos)
        e = kc.extract(MODES["unambig"], rs, k, aos=True)
        N = kc.n_limbs(k)
        assert np.array_equal(e.kmers[:, :N], km) and np.array_equal(e.kmers[:, N].astype(np.int64), pos)


def make_ragged(rng, lens):
    seqs = [kt.random_dna(rng, n) for n in lens]
    packed = [kt.pack2(s) for s in seqs]
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(p) for p in packed])
    words = np.concatenate([p for p in packed if len(p)] + [np.zeros(1, np.uint64)])
    return seqs, words, off[:-1].copy(), np.array(lens, dtype=np.uint64)


@pytest.mark.parametrize("k", [1, 7, 31, 32, 33, 63, 64, 96, 127])
def test_ragged_read_set(kc, k):
    rng = np.random.default_rng(100 + k)
    lens = [0, 1, k - 1, k, k + 1, k + 2, k + 3, 150, 151, 152, 153, 0, 0, k, 40, 999, k + 5] + \
        rng.integers(0, 400, size=300).tolist()
    lens = [max(0, int(x)) for x in lens]
    seqs, words, off, ln = make_ragged(rng, lens)
    rs = kc.ReadSet(2, words, len(lens), seq_word_offset=off, seq_len=ln)
    for mode, omode in (("fw", ko.FW), ("fwrv", ko.FWRV), ("canon", ko.CANON)):
        a, b, h, out_off = ko.batch_iterate(words, len(lens), k, omode, word_off=off, seq_len=ln, want_hash=True)
        e = kc.extract(MODES[mode], rs, k, hash=True, want_seq_offsets=True)
        assert e.n == a.shape[0]
        assert np.array_equal(e.kmers, a) and np.array_equal(e.hash, h)
        assert np.array_equal(e.seq_out_offset, out_off)
        if b is not None:
            assert np.array_equal(e.rv, b)
    # UnambiguousKmers over 2-bit reads: every window, 1-based index within its read
    e = kc.extract(MODES["unambig"], rs, k)
    want_idx = np.concatenate([np.arange(1, max(0, n - k + 1) + 1) for n in lens] + [np.zeros(0, np.int64)])
    assert np.array_equal(e.index, want_idx)


@pytest.mark.parametrize("k", [4, 31, 63])
def test_ragged_many_short_reads(kc, k):
    """Thousands of reads of 0-2 work items each: a tile spans more sequences than the kernel
    stages in shared memory, so the global-array fallback of the item search runs."""
    rng = np.random.default_rng(900 + k)
    lens = rng.integers(max(0, k - 2), k + 6, size=20_000).tolist()
    seqs, words, off, ln = make_ragged(rng, lens)
    rs = kc.ReadSet(2, words, len(lens), seq_word_offset=off, seq_len=ln)
    a, _, h, out_off = ko.batch_iterate(words, len(lens), k, ko.CANON, word_off=off, seq_len=ln, want_hash=True)
    e = kc.extract(MODES["canon"], rs, k, hash=True, want_seq_offsets=True)
    assert e.n == a.shape[0] and np.array_equal(e.kmers, a) and np.array_equal(e.hash, h)
    assert np.array_equal(e.seq_out_offset, out_off)


@pytest.mark.parametrize("k,length", [(31, 150), (31, 151), (31, 149), (21, 100), (63, 150), (63, 151), (5, 36),
                                      (31, 31), (31, 30), (32, 250), (97, 300)])
def test_uniform_read_set(kc, k, length):
    rng = np.random.default_rng(k * 1000 + length)
    n_reads = 3000
    stride = (length + 31) // 32 + (1 if length % 7 == 0 else 0)  # sometimes padded strides
    words = rng.integers(0, 2**64, size=n_reads * stride, dtype=np.uint64)
    rs = kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride)
    for mode, omode in (("canon", ko.CANON), ("fwrv", ko.FWRV)):
        a, b, h, _ = ko.batch_iterate(words, n_reads, k, omode, uniform_len=length, uniform_stride=stride,
                                      want_hash=True)
        e = kc.extract(MODES[mode], rs, k, hash=True)
        assert e.n == a.shape[0]
        assert np.array_equal(e.kmers, a) and np.array_equal(e.hash, h)
        if b is not None:
            assert np.array_equal(e.rv, b)


# windows per read a multiple of the group size G (8 / 4 / 4 / 2 for 1..4 limbs): extract_aligned_kernel, every
# (limbs, block width) class of its launcher tables; the read count leaves a partial last tile
@pytest.mark.parametrize("k,length", [(3, 10), (9, 24), (10, 25), (16, 31), (25, 64), (26, 65), (31, 150), (32, 63),
                                      (33, 36), (40, 47), (47, 54), (48, 59), (57, 64), (64, 151),
                                      (65, 72), (72, 75), (81, 88), (96, 211),
                                      (97, 98), (104, 113), (113, 126), (128, 255)])
def test_aligned_uniform_sets(kc, k, length):
    rng = np.random.default_rng(k * 977 + length)
    g = {1: 8, 2: 4, 3: 4, 4: 2}[(2 * k + 63) // 64]
    assert (length - k + 1) % g == 0
    stride = (length + 31) // 32 + (k % 2)
    n_reads = 2048 * 3 * g // (length - k + 1) + 37
    words = rng.integers(0, 2**64, size=n_reads * stride, dtype=np.uint64)
    rs = kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride)
    for mode, omode, hash_ in (("canon", ko.CANON, True), ("fwrv", ko.FWRV, False), ("fw", ko.FW, True), ("canon", ko.CANON, False)):
        a, b, h, _ = ko.batch_iterate(words, n_reads, k, omode, uniform_len=length, uniform_stride=stride, want_hash=True)
        e = kc.extract(MODES[mode], rs, k, hash=hash_)
        assert e.n == a.shape[0] and np.array_equal(e.kmers, a)
        if hash_:
            assert np.array_equal(e.hash, h)
        if b is not None:
            assert np.array_equal(e.rv, b)
    # the Julia tuple layouts (one-limb k-mers with an even window count: the lean kernel with groups of two windows)
    a, b, h, _ = ko.batch_iterate(words, n_reads, k, ko.FWRV, uniform_len=length, uniform_stride=stride, want_hash=True)
    N = a.shape[1]
    for hash_ in (False, True):
        e = kc.extract(MODES["fwrv"], rs, k, aos=True, hash=hash_)
        assert e.n == a.shape[0] and np.array_equal(e.kmers[:, 0, :], a) and np.array_equal(e.kmers[:, 1, :], b)
        if hash_:
            assert np.array_equal(e.hash, h)
        e = kc.extract(MODES["unambig"], rs, k, aos=True, hash=hash_)
        wpr = length - k + 1
        assert e.n == a.shape[0] and np.array_equal(e.kmers[:, :N], a)
        assert np.array_equal(e.kmers[:, N].astype(np.int64), np.tile(np.arange(1, wpr + 1, dtype=np.int64), n_reads))
        if hash_:
            assert np.array_equal(e.hash, h)


def test_aligned_single_sequence_and_views(kc):
    """One long sequence (one read of the uniform locator: the quotient of every item is 0): its window count need not be a
    multiple of G -- the last group is then partial (al_tail) -- and views may start inside a word; the last tile
    reaches the end of the buffer (clamped loads)."""
    rng = np.random.default_rng(4242)
    for k in (31, 63, 21, 97):
        g = {1: 8, 2: 4, 3: 4, 4: 2}[(2 * k + 63) // 64]
        for first, tail in ((0, 0), (5, 1), (17, g - 1), (0, g // 2)):
            n = 40_000 * g + k - 1 + tail
            w = rng.integers(0, 2**64, size=(n + first + 31) // 32, dtype=np.uint64)
            rs = kc.ReadSet(2, w, 1, uniform_len=n, uniform_stride_words=w.size, first_symbol_offset=first)
            a, _, h = ko.iterate(w, n, k, ko.CANON, first=first, want_hash=True)
            e = kc.extract(MODES["canon"], rs, k, hash=True)
            assert e.n == a.shape[0] and np.array_equal(e.kmers, a) and np.array_equal(e.hash, h)
            f, r, _ = ko.iterate(w, n, k, ko.FWRV, first=first, want_hash=False)
            e = kc.extract(MODES["fwrv"], rs, k)
            assert e.n == f.shape[0] and np.array_equal(e.kmers, f) and np.array_equal(e.rv, r)
            e = kc.extract(MODES["fwrv"], rs, k, aos=True)
            assert e.n == f.shape[0] and np.array_equal(e.kmers[:, 0, :], f) and np.array_equal(e.kmers[:, 1, :], r)
            e = kc.extract(MODES["unambig"], rs, k, aos=True)
            N = f.shape[1]
            assert np.array_equal(e.kmers[:, :N], f) and np.array_equal(e.kmers[:, N].astype(np.int64), np.arange(1, f.shape[0] + 1))


def test_subsequence_views(kc):
    """first_symbol_offset: a LongSubSeq-style view starting inside a word."""
    rng = np.random.default_rng(77)
    s = kt.random_dna(rng, 700)
    w = kt.pack2(s)
    for first in (1, 15, 16, 31, 32, 33, 77):
        for k in (5, 31, 33, 64):
            n = 400
            rs = kc.ReadSet(2, w, 1, uniform_len=n, uniform_stride_words=w.size, first_symbol_offset=first)
            a, _, h = ko.iterate(w, n, k, ko.CANON, first=first, want_hash=True)
            e = kc.extract(MODES["canon"], rs, k, hash=True)
            assert np.array_equal(e.kmers, a) and np.array_equal(e.hash, h)


def test_unaligned_output_buffers(kc, ctx):
    """Output pointers that are only 8-byte aligned take the scalar-store path."""
    from kmerscuda import _abi
    rng = np.random.default_rng(5)
    k, n = 31, 5000
    s = kt.random_dna(rng, n)
    w = kt.pack2(s)
    drs = kc.DeviceReadSet(ctx, kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, w, n)))
    nw = n - k + 1
    da, dh = ctx.alloc((nw + 4) * 8), ctx.alloc((nw + 4) * 8)
    out = _abi.kmc_out(da.ptr + 8, None, dh.ptr + 24, None, None, nw, 0)
    res = _abi.kmc_result()
    st = ctx.lib.kmc_extract(ctx.handle, C.byref(drs.desc), k, MODES["canon"], _abi.KMC_HASH_FX, C.byref(out),
                             C.byref(res))
    assert st == 0 and res.n_written == nw
    a, _, h = ko.iterate(w, n, k, ko.CANON, want_hash=True)
    assert np.array_equal(da.download(np.uint64, nw, 8), a[:, 0])
    assert np.array_equal(dh.download(np.uint64, nw, 24), h)


def test_errors(kc, ctx):
    from kmerscuda import _abi
    rs = kc.ReadSet.single(kc.LongDNA2("ACGTACGTAC"))
    drs = kc.DeviceReadSet(ctx, rs)
    da = ctx.alloc(64)
    res = _abi.kmc_result()
    out = _abi.kmc_out(da.ptr, None, None, None, None, 2, 0)  # too small: 8 windows for K=3
    assert ctx.lib.kmc_extract(ctx.handle, C.byref(drs.desc), 3, 0, 0, C.byref(out), C.byref(res)) == _abi.KMC_E_OUT_TOO_SMALL
    assert ctx.lib.kmc_extract(ctx.handle, C.byref(drs.desc), 0, 0, 0, C.byref(out), C.byref(res)) == _abi.KMC_E_BAD_K
    assert b"at least 1" in ctx.lib.kmc_last_error(ctx.handle)
    assert ctx.lib.kmc_extract(ctx.handle, C.byref(drs.desc), 129, 0, 0, C.byref(out), C.byref(res)) == _abi.KMC_E_BAD_K
    assert ctx.lib.kmc_extract(ctx.handle, C.byref(drs.desc), 3, 9, 0, C.byref(out), C.byref(res)) == _abi.KMC_E_BAD_ARG
    n = C.c_uint64()
    assert ctx.lib.kmc_count(ctx.handle, C.byref(drs.desc), 3, 0, C.byref(n)) == 0 and n.value == 8


def test_standalone_fx_hash(kc):
    rng = np.random.default_rng(9)
    for N in (1, 2, 3, 4):
        km = rng.integers(0, 2**64, size=(10_000, N), dtype=np.uint64)
        for h0 in (0, 1, 0xDEADBEEF12345678):
            assert np.array_equal(kc.fx_hash(km, h0), ko.fx_hash(km, h0))


def test_base_hash(kc):
    """Base.hash.(v) (src/kmer.jl:206, Julia 1.10 / 1.11 hashing): the documented value and the oracle."""
    for e in KATS["base_hash"]:
        s = dna(e["kmer"])
        got = kc.base_hash(np.array([kt.kmer_limbs(s)], dtype=np.uint64), len(s))
        assert int(got[0]) == int(e["hash"], 16)
    rng = np.random.default_rng(10)
    for N, K in ((1, 1), (1, 31), (2, 63), (3, 96), (4, 128)):
        km = rng.integers(0, 2**64, size=(10_000, N), dtype=np.uint64)
        for h0 in (0, 7, 0xDEADBEEF12345678):
            assert np.array_equal(kc.base_hash(km, K, h0), ko.base_hash(km, K, h0))


# --------------------------------------------------------------------- pipelined host path
@pytest.mark.parametrize("k", [31, 63])
def test_host_path_single_sequence_chunked(kc, k):
    """> 4 Mi windows so that kmc_extract_host splits the sequence into several chunks."""
    n = 9_000_011
    words = kt.splitmix64(np.arange((n + 31) // 32, dtype=np.uint64) + np.uint64(0xCCFB2D5055D8C990))
    rs = kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, words, n))
    a, _, h = ko.iterate(words, n, k, ko.CANON, want_hash=True)
    e = kc.extract(MODES["canon"], rs, k, hash=True, host_path=True)
    assert e.n == n - k + 1 and np.array_equal(e.kmers, a) and np.array_equal(e.hash, h)
    km, pos = ko.unambiguous(words, n, k, src_bits=2)
    e = kc.extract(MODES["unambig"], rs, k, host_path=True)
    assert np.array_equal(e.kmers, km) and np.array_equal(e.index, pos)


def test_host_path_uniform_reads_chunked(kc):
    k, length, stride, n_reads = 31, 150, 5, 90_000  # 10.8 M windows -> 3 chunks
    words = kt.splitmix64(np.arange(n_reads * stride, dtype=np.uint64) + np.uint64(439824))
    rs = kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride)
    a, b, h, _ = ko.batch_iterate(words, n_reads, k, ko.FWRV, uniform_len=length, uniform_stride=stride, want_hash=True)
    e = kc.extract(MODES["fwrv"], rs, k, hash=True, host_path=True, want_seq_offsets=True)
    assert np.array_equal(e.kmers, a) and np.array_equal(e.rv, b) and np.array_equal(e.hash, h)
    assert np.array_equal(e.seq_out_offset, np.arange(n_reads + 1, dtype=np.uint64) * np.uint64(120))
    e = kc.extract(MODES["fwrv"], rs, k, aos=True, host_path=True)
    assert np.array_equal(e.kmers[:, 0, :], a) and np.array_equal(e.kmers[:, 1, :], b)


def test_host_path_ragged_reads_chunked(kc):
    rng = np.random.default_rng(21)
    k = 31
    lens = rng.integers(0, 400, size=60_000).tolist()  # ~ 10 M windows -> several chunks
    ln = np.array(lens, dtype=np.uint64)
    nw = (ln + np.uint64(31)) // np.uint64(32)
    off = np.zeros(len(lens) + 1, dtype=np.uint64)
    off[1:] = np.cumsum(nw)
    words = kt.splitmix64(np.arange(int(off[-1]) + 1, dtype=np.uint64) + np.uint64(7))
    rs = kc.ReadSet(2, words, len(lens), seq_word_offset=off[:-1].copy(), seq_len=ln)
    a, _, h, out_off = ko.batch_iterate(words, len(lens), k, ko.CANON, word_off=off[:-1].copy(), seq_len=ln,
                                        want_hash=True)
    e = kc.extract(MODES["canon"], rs, k, hash=True, host_path=True, want_seq_offsets=True)
    assert e.n == a.shape[0] and np.array_equal(e.kmers, a) and np.array_equal(e.hash, h)
    assert np.array_equal(e.seq_out_offset, out_off)
    e2 = kc.extract(MODES["canon"], rs, k, hash=True)
    assert np.array_equal(e2.kmers, a) and np.array_equal(e2.hash, h)


def test_host_sequences_device_outputs_and_digest(kc, ctx):
    """KMC_OUT_DEVICE: sequences from the host, streams left in device memory; kmc_digest is the
    fingerprint a caller reads back instead of the streams."""
    k, length, stride, n_reads = 31, 150, 5, 90_000
    words = kt.splitmix64(np.arange(n_reads * stride, dtype=np.uint64) + np.uint64(99))
    rs = kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride)
    a, _, h, _ = ko.batch_iterate(words, n_reads, k, ko.CANON, uniform_len=length, uniform_stride=stride, want_hash=True)
    e = kc.extract(MODES["canon"], rs, k, hash=True, host_path=True, device_out=True)
    assert np.array_equal(e.kmers, a) and np.array_equal(e.hash, h)
    # ragged + single long sequence + 4-bit unambiguous through the same flag
    rng = np.random.default_rng(4)
    lens = rng.integers(0, 400, size=60_000).tolist()
    seqs, w2, off, ln = make_ragged(rng, [int(x) for x in lens])
    rs2 = kc.ReadSet(2, w2, len(lens), seq_word_offset=off, seq_len=ln)
    a2, b2, h2, _ = ko.batch_iterate(w2, len(lens), k, ko.FWRV, word_off=off, seq_len=ln, want_hash=True)
    e = kc.extract(MODES["fwrv"], rs2, k, hash=True, host_path=True, device_out=True)
    assert np.array_equal(e.kmers, a2) and np.array_equal(e.rv, b2) and np.array_equal(e.hash, h2)
    n = 9_000_011
    codes = np.where(kt.splitmix64(np.arange(n, dtype=np.uint64)) % np.uint64(100) == 0, np.uint64(15),
                     np.uint64(1) << (kt.splitmix64(np.arange(n, dtype=np.uint64) + np.uint64(5)) & np.uint64(3)))
    w4 = kt.pack_codes(codes, 4)
    km, pos = ko.unambiguous(w4, n, k, src_bits=4)
    e = kc.extract(MODES["unambig"], kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet4, w4, n)), k, hash=True,
                   host_path=True, device_out=True)
    assert np.array_equal(e.kmers, km) and np.array_equal(e.index, pos) and np.array_equal(e.hash, ko.fx_hash(km))
    # KMC_DIGEST fused into the pipeline == fingerprint of what the call wrote
    from kmerscuda import _abi
    cap = a.shape[0]
    da, dh = ctx.alloc(cap * 8), ctx.alloc(cap * 8)
    desc = _abi.kmc_seqs(words.ctypes.data, words.size, n_reads, None, None, length, stride, 2, 0)
    out = _abi.kmc_out(da.ptr, None, dh.ptr, None, None, cap, 0)
    res = _abi.kmc_result()
    ctx._check(ctx.lib.kmc_extract_host(ctx.handle, C.byref(desc), k, MODES["canon"],
                                        _abi.KMC_HASH_FX | _abi.KMC_OUT_DEVICE | _abi.KMC_DIGEST, C.byref(out), C.byref(res)))
    assert list(res.digest) == [int(np.bitwise_xor.reduce(a.reshape(-1))), int(a.sum(dtype=np.uint64)),
                                int(np.bitwise_xor.reduce(h)), int(h.sum(dtype=np.uint64))]
    assert np.array_equal(da.download(np.uint64, cap), a[:, 0])
    # digest == numpy xor / wrapping sum, at odd offsets and lengths
    d = ctx.to_device(a)
    for o, m in ((0, a.size), (1, a.size - 1), (3, 1001), (0, 0), (2, 1)):
        x, s = ctx.digest(d.ptr + 8 * o, m)
        sl = a.reshape(-1)[o:o + m]
        assert x == int(np.bitwise_xor.reduce(sl)) if m else x == 0
        assert s == int(sl.sum(dtype=np.uint64)) if m else s == 0


@pytest.mark.parametrize("mode,k,hash_,ragged", [("fw", 31, False, False), ("canon", 63, True, True), ("fw", 5, True, True),
                                                 ("canon", 32, False, False), ("canon", 31, True, False),
                                                 ("canon", 63, True, False)])
def test_digest_fused_into_the_extraction_kernel(kc, ctx, mode, k, hash_, ragged):
    """KMC_DIGEST for the SoA forms of FwKmers / CanonicalKmers over 2-bit sources comes out of the extraction kernel
    itself (no second pass over the streams): one- and two-limb k-mers, with and without the hash stream, uniform and
    ragged sets with partial groups at every read boundary."""
    from kmerscuda import _abi
    rng = np.random.default_rng(k + 7)
    omode = ko.CANON if mode == "canon" else ko.FW
    if ragged:
        lens = rng.integers(0, 300, size=20_000).tolist()
        seqs, words, off, ln = make_ragged(rng, [int(x) for x in lens])
        n_seqs = len(lens)
        a, _, h, _ = ko.batch_iterate(words, n_seqs, k, omode, word_off=off, seq_len=ln, want_hash=True)
        desc = _abi.kmc_seqs(words.ctypes.data, words.size, n_seqs, off.ctypes.data, ln.ctypes.data, 0, 0, 2, 0)
    else:
        n_seqs, length, stride = 30_000, 150, 5
        words = rng.integers(0, 2**64, size=n_seqs * stride, dtype=np.uint64)
        a, _, h, _ = ko.batch_iterate(words, n_seqs, k, omode, uniform_len=length, uniform_stride=stride, want_hash=True)
        desc = _abi.kmc_seqs(words.ctypes.data, words.size, n_seqs, None, None, length, stride, 2, 0)
    n, limbs = a.shape
    da, dh = ctx.alloc(max(n, 1) * limbs * 8), ctx.alloc(max(n, 1) * 8)
    out = _abi.kmc_out(da.ptr, None, dh.ptr if hash_ else None, None, None, n, 0)
    res = _abi.kmc_result()
    flags = (_abi.KMC_HASH_FX if hash_ else 0) | _abi.KMC_OUT_DEVICE | _abi.KMC_DIGEST
    ctx._check(ctx.lib.kmc_extract_host(ctx.handle, C.byref(desc), k, MODES[mode], flags, C.byref(out), C.byref(res)))
    want = [int(np.bitwise_xor.reduce(a.reshape(-1))), int(a.sum(dtype=np.uint64)),
            int(np.bitwise_xor.reduce(h)) if hash_ else 0, int(h.sum(dtype=np.uint64)) if hash_ else 0]
    assert int(res.n_written) == n and list(res.digest) == want
    assert np.array_equal(da.download(np.uint64, n * limbs).reshape(n, limbs), a)
    if hash_:
        assert np.array_equal(dh.download(np.uint64, n), h)
    da.free()
    dh.free()


# ---------------------------------------------------------------------- bucket count table
def test_bucket_count_binned_ragged(kc):
    """Tables beyond L2 take the binned path (ids -> bins -> apply); ragged set, one- and two-limb k-mers."""
    rng = np.random.default_rng(5)
    lens = rng.integers(0, 300, size=30_000).tolist()
    seqs, words, off, ln = make_ragged(rng, [int(x) for x in lens])
    rs = kc.ReadSet(2, words, len(lens), seq_word_offset=off, seq_len=ln)
    for k, bits in ((31, 26), (63, 27), (5, 30), (100, 25)):
        _, _, h, _ = ko.batch_iterate(words, len(lens), k, ko.CANON, word_off=off, seq_len=ln, want_hash=True)
        table, n, _ = kc.bucket_count(rs, k, bits)
        assert n == h.size
        idx, cnt = np.unique((h >> np.uint64(64 - bits)).astype(np.int64), return_counts=True)
        assert int(table.sum(dtype=np.int64)) == h.size
        assert np.array_equal(np.nonzero(table)[0], idx) and np.array_equal(table[idx], cnt.astype(np.uint32))


def test_bucket_count_fused_bins_and_spill_list(kc):
    """Tables beyond L2, one-limb k-mers, aligned uniform set: ids and bins come from one kernel with bins of a fixed
    capacity.  Random reads fit; a set dominated by one repeated k-mer fills a bin, whose later runs go to the spill list
    (the run that straddles the capacity included: the bin ends where it would have begun) -- the table is the exact
    histogram either way."""
    rng = np.random.default_rng(99)
    n_reads, length, stride, k = 40_000, 150, 5, 31
    words = rng.integers(0, 2**64, size=n_reads * stride, dtype=np.uint64)
    cases = {"random": words.copy()}
    w = words.copy()
    w.reshape(n_reads, stride)[n_reads // 3:] = 0  # two thirds of the reads are poly-A: one bucket gets 67 % of the k-mers
    cases["crowded"] = w
    cases["single k-mer"] = np.zeros_like(words)
    for name, ww in cases.items():
        rs = kc.ReadSet(2, ww, n_reads, uniform_len=length, uniform_stride_words=stride)
        _, _, h, _ = ko.batch_iterate(ww, n_reads, k, ko.CANON, uniform_len=length, uniform_stride=stride, want_hash=True)
        for bits in (26, 28):
            table, n, _ = kc.bucket_count(rs, k, bits)
            idx, cnt = np.unique((h >> np.uint64(64 - bits)).astype(np.int64), return_counts=True)
            assert n == h.size and int(table.sum(dtype=np.int64)) == h.size, name
            assert np.array_equal(np.nonzero(table)[0], idx) and np.array_equal(table[idx], cnt.astype(np.uint32)), name
    # a partial last tile and a partial last iteration of the binning step
    for n_small in (1, 7, 300, 2048 // 15 + 1, 4500):
        ww = words[: n_small * stride]
        rs = kc.ReadSet(2, ww, n_small, uniform_len=length, uniform_stride_words=stride)
        _, _, h, _ = ko.batch_iterate(ww, n_small, k, ko.CANON, uniform_len=length, uniform_stride=stride, want_hash=True)
        table, n, _ = kc.bucket_count(rs, k, 27)
        idx, cnt = np.unique((h >> np.uint64(64 - 27)).astype(np.int64), return_counts=True)
        assert n == h.size and np.array_equal(np.nonzero(table)[0], idx) and np.array_equal(table[idx], cnt.astype(np.uint32))


# (63, 27) and (21, 26): tables beyond L2 that the fused bins do not take, so the exact path bins the ids of
# extract_aligned_kernel (88 windows per read, a multiple of G = 4) and of extract_kernel (130 windows, not a multiple of 8)
@pytest.mark.parametrize("k,bits", [(31, 20), (63, 12), (15, 28), (63, 27), (21, 26)])
def test_bucket_count(kc, k, bits):
    rng = np.random.default_rng(k)
    n_reads, length, stride = 20_000, 150, 5
    words = rng.integers(0, 2**64, size=n_reads * stride, dtype=np.uint64)
    rs = kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride)
    table, n, _ = kc.bucket_count(rs, k, bits)
    _, _, h, _ = ko.batch_iterate(words, n_reads, k, ko.CANON, uniform_len=length, uniform_stride=stride, want_hash=True)
    want = np.bincount((h >> np.uint64(64 - bits)).astype(np.int64), minlength=1 << bits).astype(np.uint32)
    assert n == h.size and int(table.sum()) == h.size
    assert np.array_equal(table, want)


@pytest.mark.parametrize("bits,n_parts", [(20, 4), (26, 8), (27, 32), (26, 1)])
def test_bucket_count_async_progress_events(kc, ctx, bits, n_parts):
    """kmc_bucket_count_async: same table as the synchronous call; every progress event completes; a range whose
    event has fired is final (checked by copying it out on a second stream that only waits for that event).  At bits = 26
    also over a ragged set, which the exact binned path counts (the uniform set takes the fused bins)."""
    import ctypes as C
    import torch
    from kmerscuda import _abi, sharding
    rng = np.random.default_rng(bits)
    n_reads, length, stride, k = 30_000, 150, 5, 31
    words = rng.integers(0, 2**64, size=n_reads * stride, dtype=np.uint64)
    sets = [kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride)]
    if bits == 26:
        lens = [int(x) for x in rng.integers(0, 300, size=30_000)]
        _, rwords, off, ln = make_ragged(rng, lens)
        sets.append(kc.ReadSet(2, rwords, len(lens), seq_word_offset=off, seq_len=ln))
    for rs in sets:
        want, n, _ = kc.bucket_count(rs, k, bits, ctx=ctx)
        drs = kc.DeviceReadSet(ctx, rs)
        main, side = torch.cuda.Stream(), torch.cuda.Stream()
        with torch.cuda.stream(main):
            ctx.set_stream(main.cuda_stream)
            try:
                table = torch.zeros(1 << bits, dtype=torch.int32, device="cuda")
                events = [torch.cuda.Event() for _ in range(n_parts)]
                for e in events:
                    e.record(main)
                handles = (C.c_void_p * n_parts)(*[C.c_void_p(e.cuda_event) for e in events])
                res = _abi.kmc_result()
                ctx._check(ctx.lib.kmc_bucket_count_async(ctx.handle, C.byref(drs.desc), k, bits, table.data_ptr(), n_parts, handles,
                                                          C.byref(res)))
                part = table.numel() // n_parts
                copies = []
                with torch.cuda.stream(side):
                    for i, e in enumerate(events):
                        side.wait_event(e)
                        copies.append(table[i * part:(i + 1) * part].clone())
                side.synchronize()
                main.synchronize()
                assert all(e.query() for e in events)
                assert int(res.n_written) == n
                assert np.array_equal(table.cpu().numpy().view(np.uint32), want)
                assert np.array_equal(torch.cat(copies).cpu().numpy().view(np.uint32), want)
                # one rank: the overlapped count + merge helper is the same count
                table.zero_()
                assert sharding.count_and_merge_table(ctx, drs.desc, k, bits, table, n_parts=n_parts) == n
                main.synchronize()
                assert np.array_equal(table.cpu().numpy().view(np.uint32), want)
                # argument checks
                bad = (C.c_void_p * 3)(*[C.c_void_p(e.cuda_event) for e in events[:1] * 3])
                assert ctx.lib.kmc_bucket_count_async(ctx.handle, C.byref(drs.desc), k, bits, table.data_ptr(), 3, bad, C.byref(res)) != 0
            finally:
                ctx.set_stream(None)


# ----------------------------------------------- full-size properties (BASELINE config C2 shape)
def test_full_size_properties(kc, ctx):
    """10 M x 150 bp reads, K=31, canonical + fx_hash, outputs resident on the device (19.2 GB).
    Size-independent checks: (1) the fused hash stream equals kmc_fx_hash over the canonical
    stream, (2) canonical(read) == canonical(reverse-complemented read) reversed -- checked on
    the device with torch, (3) a random sample of reads equals the oracle bit for bit."""
    import torch
    from kmerscuda import _abi
    free, _ = torch.cuda.mem_get_info()
    n_reads = 10_000_000 if free > 60e9 else 1_000_000
    k, length, stride = 31, 150, 5
    wpr = length - k + 1
    g = torch.Generator(device="cuda").manual_seed(439824)
    words = torch.randint(-2**63, 2**63 - 1, (n_reads * stride,), dtype=torch.int64, device="cuda", generator=g)
    # trailing bits of each read's last word are zero in a LongSequence (150 = 4*32 + 22 symbols)
    words.view(n_reads, stride)[:, stride - 1] &= (1 << (2 * (length - 32 * (stride - 1)))) - 1
    canon = torch.empty(n_reads * wpr, dtype=torch.int64, device="cuda")
    hsh = torch.empty(n_reads * wpr, dtype=torch.int64, device="cuda")
    desc = _abi.kmc_seqs(words.data_ptr(), words.numel(), n_reads, None, None, length, stride, 2, 0)
    out = _abi.kmc_out(canon.data_ptr(), None, hsh.data_ptr(), None, None, n_reads * wpr, 0)
    res = _abi.kmc_result()
    torch.cuda.synchronize()
    ctx._check(ctx.lib.kmc_extract(ctx.handle, C.byref(desc), k, MODES["canon"], _abi.KMC_HASH_FX, C.byref(out), C.byref(res)))
    assert res.n_written == n_reads * wpr
    # (1) fused hash == standalone hash of the canonical stream
    h2 = torch.empty_like(hsh)
    ctx._check(ctx.lib.kmc_fx_hash(ctx.handle, canon.data_ptr(), canon.numel(), 1, 0, h2.data_ptr()))
    ctx.sync()
    assert torch.equal(hsh, h2)
    del h2
    # (2) strand symmetry: the canonical k-mers of the reverse-complemented reads are the same
    #     multiset per read, in reverse order.  Build the RC reads with the library itself:
    #     rv k-mer of window 0 of a K=L "read" is the RC read; cheaper: check on a 200k-read slice.
    m = min(n_reads, 200_000)
    sl = words[: m * stride].cpu().numpy().view(np.uint64)
    codes = ((sl.reshape(m, stride, 1) >> (np.arange(32, dtype=np.uint64) * np.uint64(2))) & np.uint64(3)).reshape(m, -1)[:, :length]
    rc_codes = (3 - codes[:, ::-1]).astype(np.uint64)
    pad = np.zeros((m, stride * 32), dtype=np.uint64)
    pad[:, :length] = rc_codes
    rc_words = np.bitwise_or.reduce(pad.reshape(m, stride, 32) << (np.arange(32, dtype=np.uint64) * np.uint64(2)), axis=2).reshape(-1)
    rs_rc = kc.ReadSet(2, rc_words, m, uniform_len=length, uniform_stride_words=stride)
    e = kc.extract(MODES["canon"], rs_rc, k, hash=True)
    fwd = canon[: m * wpr].cpu().numpy().view(np.uint64).reshape(m, wpr)
    assert np.array_equal(e.kmers.reshape(m, wpr)[:, ::-1], fwd)
    # (3) sampled reads against the oracle
    rng = np.random.default_rng(1)
    idx = np.sort(rng.choice(n_reads, size=2000, replace=False))
    for r in idx[:: 1 if n_reads <= 1_000_000 else 1]:
        w = words[r * stride:(r + 1) * stride].cpu().numpy().view(np.uint64)
        a, _, h = ko.iterate(w, length, k, ko.CANON, want_hash=True)
        assert np.array_equal(canon[r * wpr:(r + 1) * wpr].cpu().numpy().view(np.uint64), a[:, 0])
        assert np.array_equal(hsh[r * wpr:(r + 1) * wpr].cpu().numpy().view(np.uint64), h)


# ----------------------------------------------- full-size properties (BASELINE config C4 shape)
def test_full_size_properties_c4(kc, ctx):
    """CanonicalDNAMers{63} (two limbs) + fx_hash over one 1 Gbp 2-bit sequence, streams resident (24 GB).
    Size-independent checks: (1) the fused hash equals kmc_fx_hash over the canonical stream, (2) the
    8 shards of the 1/2/4/8-GPU plan (window ranges with a K-1 halo, kmerscuda.sharding), run one after
    the other into their slices, reproduce the unsharded streams exactly, (3) strand symmetry on a slice,
    (4) sampled windows against the oracle."""
    import torch
    from kmerscuda import _abi, sharding
    free, _ = torch.cuda.mem_get_info()
    n = 1_000_000_000 if free > 80e9 else 50_000_000
    k, N = 63, 2
    nwin = n - k + 1
    g = torch.Generator(device="cuda").manual_seed(63)
    words = torch.randint(-2**63, 2**63 - 1, ((n + 31) // 32,), dtype=torch.int64, device="cuda", generator=g)
    canon = torch.empty(nwin * N, dtype=torch.int64, device="cuda")
    hsh = torch.empty(nwin, dtype=torch.int64, device="cuda")
    desc = _abi.kmc_seqs(words.data_ptr(), words.numel(), 1, None, None, n, words.numel(), 2, 0)
    out = _abi.kmc_out(canon.data_ptr(), None, hsh.data_ptr(), None, None, nwin, 0)
    res = _abi.kmc_result()
    torch.cuda.synchronize()
    ctx._check(ctx.lib.kmc_extract(ctx.handle, C.byref(desc), k, MODES["canon"], _abi.KMC_HASH_FX, C.byref(out), C.byref(res)))
    assert res.n_written == nwin
    # (1)
    h2 = torch.empty_like(hsh)
    ctx._check(ctx.lib.kmc_fx_hash(ctx.handle, canon.data_ptr(), nwin, N, 0, h2.data_ptr()))
    ctx.sync()
    assert torch.equal(hsh, h2)
    # (2) the sharded plan, into h2 / a second canonical buffer slice by slice
    ref_digest = ctx.digest(canon.data_ptr(), nwin * N), ctx.digest(hsh.data_ptr(), nwin)
    h2.zero_()
    c2 = torch.zeros_like(canon)
    for sh in sharding.plan_sequence_shards(n, k, 2, 8):
        if sh.n_windows == 0:
            continue
        d = _abi.kmc_seqs(words.data_ptr() + 8 * sh.word0, sh.n_words, 1, None, None, sh.length, sh.n_words, 2, sh.first_symbol_offset)
        o = _abi.kmc_out(c2.data_ptr() + 8 * N * sh.window0, None, h2.data_ptr() + 8 * sh.window0, None, None, sh.n_windows, 0)
        ctx._check(ctx.lib.kmc_extract(ctx.handle, C.byref(d), k, MODES["canon"], _abi.KMC_HASH_FX, C.byref(o), C.byref(res)))
        assert res.n_written == sh.n_windows
    assert (ctx.digest(c2.data_ptr(), nwin * N), ctx.digest(h2.data_ptr(), nwin)) == ref_digest
    assert torch.equal(c2, canon) and torch.equal(h2, hsh)
    del c2, h2
    # (3) strand symmetry on the first 1 M symbols
    m = 1_000_000
    sl = words[: m // 32].cpu().numpy().view(np.uint64)
    codes = ((sl.reshape(-1, 1) >> (np.arange(32, dtype=np.uint64) * np.uint64(2))) & np.uint64(3)).reshape(-1)
    rc = kt.pack_codes((3 - codes[::-1]).astype(np.uint64), 2)
    e = kc.extract(MODES["canon"], kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, rc, m)), k)
    fwd = canon[: (m - k + 1) * N].cpu().numpy().view(np.uint64).reshape(-1, N)
    assert np.array_equal(e.kmers[::-1], fwd)
    # (4) sampled windows (slices of 200 windows at random places, limb / word boundaries included)
    rng = np.random.default_rng(4)
    for s in np.concatenate([[0, nwin - 200], rng.integers(0, nwin - 200, size=300)]):
        s = int(s)
        w0 = s // 32
        w = words[w0: w0 + (200 + k + 62) // 32 + 1].cpu().numpy().view(np.uint64)
        a, _, h = ko.iterate(w, 200 + k - 1, k, ko.CANON, first=s - 32 * w0, want_hash=True)
        assert np.array_equal(canon[s * N:(s + 200) * N].cpu().numpy().view(np.uint64).reshape(-1, N), a)
        assert np.array_equal(hsh[s:s + 200].cpu().numpy().view(np.uint64), h)
