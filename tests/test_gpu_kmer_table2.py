"""Exact counts of two-limb k-mers (K = 33..64): KmerTable(..., n_limbs=2) over kmc_kmer_count2 and the other `*2`
entry points, against np.unique of the oracle's k-mer stream (u64[n, 2], limb 0 = head first, rows in Kmer order).
The owner function of the multi-GPU exchange is checked on the CPU; everything else needs a GPU.  The two-GPU forms
are skipped on boxes with fewer than two GPUs."""
import os
import socket

import numpy as np
import pytest

import kmertools as kt
from oracle import oracle as ko

FX = np.uint64(0x517CC1B727220A95)


@pytest.fixture(scope="module")
def kc():
    import kmerscuda
    return kmerscuda


def owner2_numpy(keys, n_ranks):
    """kmc_kmer_owner2 restated: fx_hash of the two limbs, the second mix of owner_of, a multiply-shift."""
    h = ko.fx_hash(keys)
    with np.errstate(over="ignore"):
        h = h ^ (h >> np.uint64(32))
        h = h * np.uint64(0x9E3779B97F4A7C15)
        return ((h >> np.uint64(32)) * np.uint64(n_ranks)) >> np.uint64(32)


def test_owner2_matches_numpy_restatement():
    from kmerscuda import _abi
    lib = _abi.load()
    rng = np.random.default_rng(2)
    keys = rng.integers(0, 2**64, size=(500, 2), dtype=np.uint64)
    keys[0] = [np.uint64(2**64 - 1), 0]  # the canonical 64-mer T^32 A^32
    keys[1] = [0, 0]
    keys[2] = [1, np.uint64(2**64 - 1)]
    # the hash the owner is taken over is fx_hash<2>: limb 0 first
    with np.errstate(over="ignore"):
        h0 = keys[:, 0] * FX
        h = (((h0 << np.uint64(5)) | (h0 >> np.uint64(59))) ^ keys[:, 1]) * FX
    assert np.array_equal(ko.fx_hash(keys), h)
    for n in range(1, 65):
        want = owner2_numpy(keys, n)
        got = np.array([lib.kmc_kmer_owner2(int(a), int(b), n) for a, b in keys], dtype=np.uint64)
        assert np.array_equal(got, want), n
        assert int(got.max()) < n
    assert lib.kmc_kmer_owner2(5, 7, 0) == 0


# ------------------------------------------------------------------------------------------------------ read sets
def uniform_reads(kc, rng, genome, n_reads, length):
    """n_reads reads of `length` symbols drawn from `genome` (2-bit codes): most k-mers occur many times."""
    stride = (length + 31) // 32
    starts = rng.integers(0, len(genome) - length + 1, size=n_reads)
    codes = np.zeros((n_reads, stride * 32), dtype=np.uint64)
    codes[:, :length] = genome[starts[:, None] + np.arange(length)[None, :]]
    words = kt.pack_codes(codes.reshape(-1), 2)
    rs = kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride)
    return rs, dict(uniform_len=length, uniform_stride=stride), words, n_reads


def ragged_reads(kc, rng, genome, n_reads, max_len):
    """Reads of 0 .. max_len symbols (empty reads and reads shorter than K among them)."""
    lens = rng.integers(0, max_len + 1, size=n_reads)
    lens[:5] = [0, 1, 32, 33, 63]
    words_l, off = [], [0]
    for ln in lens:
        s0 = int(rng.integers(0, len(genome) - max_len))
        w = kt.pack_codes(genome[s0:s0 + int(ln)], 2) if ln else np.zeros(0, dtype=np.uint64)
        words_l.append(w)
        off.append(off[-1] + len(w))
    words = np.concatenate(words_l)
    off = np.asarray(off[:-1], dtype=np.uint64)
    ln = np.asarray(lens, dtype=np.uint64)
    rs = kc.ReadSet(2, words, n_reads, seq_word_offset=off, seq_len=ln)
    return rs, dict(word_off=off, seq_len=ln), words, n_reads


def oracle_counts(words, n_reads, k, canonical, layout):
    a, _, _, _ = ko.batch_iterate(words, n_reads, k, ko.CANON if canonical else ko.FW, **layout)
    assert a.shape[1] == 2
    uk, uc = np.unique(a, axis=0, return_counts=True)
    return a.shape[0], uk, uc.astype(np.uint32)


def check_table(t, uk, uc, times=1):
    assert t.n_keys == len(uk)
    gk, gc = t.items()
    assert gk.shape == uk.shape and gc.shape == uc.shape
    assert np.array_equal(gk, uk) and np.array_equal(gc, times * uc)


# ------------------------------------------------------------------------------------------------------ parity
@pytest.mark.gpu
@pytest.mark.parametrize("k,canonical", [(33, False), (33, True), (40, False), (40, True), (47, False), (47, True),
                                         (63, False), (63, True), (64, True)])
def test_kmer_table2_matches_unique_counts(kc, k, canonical):
    rng = np.random.default_rng(700 + k + canonical)
    genome = rng.integers(0, 4, size=20_000).astype(np.uint64)
    for make in (uniform_reads, ragged_reads):
        rs, layout, words, n_reads = make(kc, rng, genome, 4000, 150)
        n_k, uk, uc = oracle_counts(words, n_reads, k, canonical, layout)
        t = kc.KmerTable(17, n_limbs=2)
        n, ms = t.count(rs, k, canonical=canonical)
        assert n == n_k and ms > 0
        check_table(t, uk, uc)
        # counting the set again doubles every count; merging a second table adds it
        t.count(rs, k, canonical=canonical)
        check_table(t, uk, uc, 2)
        t2 = kc.KmerTable(16, n_limbs=2)
        t2.count(rs, k, canonical=canonical)
        t.merge(t2)
        check_table(t, uk, uc, 3)
        t.free()
        t2.free()
    # one sequence whose last group of windows is partial
    n = 200_003
    w = rng.integers(0, 2**64, size=(n + 31) // 32, dtype=np.uint64)
    a, _, _ = ko.iterate(w, n, k, ko.CANON if canonical else ko.FW)
    uk, uc = np.unique(a, axis=0, return_counts=True)
    t = kc.KmerTable(19, n_limbs=2)
    n_c, _ = t.count(kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, w, n)), k, canonical=canonical)
    assert n_c == n - k + 1
    check_table(t, uk, uc.astype(np.uint32))
    t.free()


def fixed_reads(kc, codes):
    """Reads given as rows of 2-bit codes, all of the same length."""
    n_reads, length = codes.shape
    stride = (length + 31) // 32
    padded = np.zeros((n_reads, stride * 32), dtype=np.uint64)
    padded[:, :length] = codes
    words = kt.pack_codes(padded.reshape(-1), 2)
    return kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride), words, dict(uniform_len=length,
                                                                                                     uniform_stride=stride)


@pytest.mark.gpu
def test_both_limbs_decide_equality(kc):
    rng = np.random.default_rng(11)
    # K = 63 forward, reads of exactly 63 symbols: limb 0 holds the first 31 symbols, limb 1 the last 32.  All reads share
    # limb 1 and differ (among 400 variants) in limb 0 -- and then the other way round.
    tail = rng.integers(0, 4, size=32).astype(np.uint64)
    heads = rng.integers(0, 4, size=(400, 31)).astype(np.uint64)
    pick = rng.integers(0, 400, size=5000)
    for codes in (np.concatenate([heads[pick], np.tile(tail, (5000, 1))], axis=1),
                  np.concatenate([np.tile(heads[0], (5000, 1)), rng.integers(0, 4, size=(400, 32)).astype(np.uint64)[pick]],
                                 axis=1)):
        rs, words, layout = fixed_reads(kc, codes)
        n_k, uk, uc = oracle_counts(words, 5000, 63, False, layout)
        assert n_k == 5000 and len(uk) == len(np.unique(pick))
        t = kc.KmerTable(12, n_limbs=2)
        t.count(rs, 63, canonical=False)
        check_table(t, uk, uc)
        t.free()
    # K = 64 canonical over reads containing T^32 A^32 (its own reverse complement: limb 0 = ~0, limb 1 = 0) -- a key, not
    # a free slot
    special = np.array([3] * 32 + [0] * 32, dtype=np.uint64)
    codes = rng.integers(0, 4, size=(3000, 150)).astype(np.uint64)
    at = rng.integers(0, 150 - 64 + 1, size=3000)
    for r in range(3000):
        codes[r, at[r]:at[r] + 64] = special
    rs, words, layout = fixed_reads(kc, codes)
    n_k, uk, uc = oracle_counts(words, 3000, 64, True, layout)
    row = np.flatnonzero((uk[:, 0] == np.uint64(2**64 - 1)) & (uk[:, 1] == 0))
    assert len(row) == 1 and uc[row[0]] >= 3000
    for log2cap in (18, 23):  # streaming and binned insert
        t = kc.KmerTable(log2cap, n_limbs=2)
        t.count(rs, 64, canonical=True)
        check_table(t, uk, uc)
        t.free()


# ------------------------------------------------------------------------------------------------------ binned path
@pytest.mark.gpu
@pytest.mark.parametrize("k,canonical,log2cap", [(63, True, 23), (41, False, 23), (55, True, 26)])
def test_kmer_table2_beyond_l2_takes_the_binned_path(kc, k, canonical, log2cap):
    """Tables beyond 96 MB (2^23 slots = 160 MB, 2^26 = 1.25 GB) are filled slice by slice from binned k-mers."""
    rng = np.random.default_rng(900 + k)
    genome = rng.integers(0, 4, size=60_000).astype(np.uint64)
    for make in (uniform_reads, ragged_reads):
        rs, layout, words, n_reads = make(kc, rng, genome, 3000, 150 if make is uniform_reads else 260)
        n_k, uk, uc = oracle_counts(words, n_reads, k, canonical, layout)
        t = kc.KmerTable(log2cap, n_limbs=2)
        n, _ = t.count(rs, k, canonical=canonical)
        assert n == n_k
        check_table(t, uk, uc)
        t.count(rs, k, canonical=canonical)  # every key is already there
        check_table(t, uk, uc, 2)
        t.free()


# ------------------------------------------------------------------------------------------------------ probing, checks
@pytest.mark.gpu
def test_kmer_table2_probing_full_and_argument_checks(kc):
    rng = np.random.default_rng(3)
    # ~3000 distinct keys in 4096 slots: long probe runs that wrap around the end of the table
    n = 3000 + 40 - 1
    w = rng.integers(0, 2**64, size=(n + 31) // 32, dtype=np.uint64)
    rs = kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, w, n))
    a, _, _ = ko.iterate(w, n, 40, ko.CANON)
    uk, uc = np.unique(a, axis=0, return_counts=True)
    t = kc.KmerTable(12, n_limbs=2)
    t.count(rs, 40)
    check_table(t, uk, uc.astype(np.uint32))
    t.free()
    # too many keys
    n = 10_000
    w = rng.integers(0, 2**64, size=(n + 31) // 32, dtype=np.uint64)
    rs = kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, w, n))
    t = kc.KmerTable(8, n_limbs=2)
    with pytest.raises(kc.KmersCUDAError, match="full"):
        t.count(rs, 40)
    t.free()
    t = kc.KmerTable(10, n_limbs=2)
    for k, canonical in ((32, True), (65, True), (64, False)):
        with pytest.raises(kc.KmersCUDAError):
            t.count(rs, k, canonical=canonical)
    with pytest.raises(kc.KmersCUDAError):
        t.count(kc.ReadSet.single(kc.LongDNA4("ACGT" * 50)), 40)
    one = kc.KmerTable(10)
    with pytest.raises(kc.KmersCUDAError):
        one.count(rs, 33)
    with pytest.raises(ValueError):
        t.merge(one)
    with pytest.raises(ValueError):
        kc.KmerTable(10, n_limbs=3)
    # the C entry points reject two-limb keys that are not 16-byte aligned (a status, not a device fault)
    import ctypes as C
    from kmerscuda import _abi
    ctx, lib = t.ctx, t.ctx.lib
    bad = t.keys.ptr + 8
    n_out = C.c_uint64(0)
    res = _abi.kmc_result()
    drs = kc.DeviceReadSet(ctx, rs)
    assert lib.kmc_kmer_count2(ctx.handle, C.byref(drs.desc), 40, kc.KMC_CANON, bad, t.vals.ptr, 8, C.byref(res)) == _abi.KMC_E_BAD_ARG
    assert lib.kmc_kmer_table2_merge(ctx.handle, bad, t.vals.ptr, 8, t.keys.ptr, t.vals.ptr, 4, C.byref(n_out)) == _abi.KMC_E_BAD_ARG
    assert lib.kmc_kmer_table2_export(ctx.handle, bad, t.vals.ptr, 8, t.keys.ptr, t.vals.ptr, 4, C.byref(n_out)) == _abi.KMC_E_BAD_ARG
    assert lib.kmc_kmer_table2_exchange(ctx.handle, bad, t.vals.ptr, 8, t.keys.ptr, t.vals.ptr, 8, C.byref(n_out)) == _abi.KMC_E_BAD_ARG
    assert "aligned" in lib.kmc_last_error(ctx.handle).decode()
    one.free()
    t.free()


# ------------------------------------------------------------------------------------------------------ multi-GPU
def _small_set(kc, seed=17):
    rng = np.random.default_rng(seed)
    genome = rng.integers(0, 4, size=20_000).astype(np.uint64)
    return uniform_reads(kc, rng, genome, 4000, 150)


@pytest.mark.gpu
def test_kmer_table2_one_rank_exchange_and_one_device_group(kc):
    rs, layout, words, n_reads = _small_set(kc)
    ctx = kc.Context(0)
    ctx.comm_init(1, 0, kc.Context.comm_unique_id())
    t = kc.KmerTable(16, ctx=ctx, n_limbs=2)
    t.count(rs, 63)
    owned = t.exchange(16)
    assert owned.n_limbs == 2
    k0, v0 = t.items()
    k1, v1 = owned.items()
    assert k0.shape[1] == 2 and np.array_equal(k0, k1) and np.array_equal(v0, v1)
    _, uk, uc = oracle_counts(words, n_reads, 63, True, layout)
    assert np.array_equal(k0, uk) and np.array_equal(v0, uc)
    ctx.comm_destroy()
    ctx.close()

    g = kc.Group([0])
    t = kc.KmerTable(16, ctx=g.ctx[0], n_limbs=2)
    t.count(rs, 63)
    owned = g.kmer_table_exchange([t], 16)
    k1, v1 = owned[0].items()
    assert np.array_equal(k1, uk) and np.array_equal(v1, uc)
    with pytest.raises(ValueError):
        g.kmer_table_exchange([t, kc.KmerTable(10, ctx=g.ctx[0])], 16)
    g.close()


@pytest.mark.gpu
def test_kmer_table2_group_two_gpus_single_process(kc):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from kmerscuda import sharding
    rs, layout, words, n_reads = _small_set(kc)
    g = kc.Group([0, 1])
    tabs = []
    for r, c in enumerate(g.ctx):
        t = kc.KmerTable(16, ctx=c, n_limbs=2)
        t.count(sharding.read_shard(rs, 2, r), 63)
        tabs.append(t)
    owned = g.kmer_table_exchange(tabs, 16)
    _, uk, uc = oracle_counts(words, n_reads, 63, True, layout)
    own = np.array([g.lib.kmc_kmer_owner2(int(a), int(b), 2) for a, b in uk])
    for r in range(2):
        gk, gv = owned[r].items()
        assert np.array_equal(gk, uk[own == r]) and np.array_equal(gv, uc[own == r])
    g.close()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, ret):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, "kmers.jl_b200"), os.path.join(root, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import kmerscuda as kc
    from kmerscuda import sharding
    ctx = kc.Context(rank)
    ctx.comm_init_torch()
    rs, layout, words, n_reads = _small_set(kc)
    t = kc.KmerTable(16, ctx=ctx, n_limbs=2)
    t.count(sharding.read_shard(rs, world, rank), 63)
    owned = t.exchange(16)
    _, uk, uc = oracle_counts(words, n_reads, 63, True, layout)
    mine = np.array([ctx.lib.kmc_kmer_owner2(int(a), int(b), world) == rank for a, b in uk])
    gk, gv = owned.items()
    ret[rank] = bool(np.array_equal(gk, uk[mine]) and np.array_equal(gv, uc[mine]))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_kmer_table2_two_process_exchange():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    with ctx.Manager() as mgr:
        ret = mgr.dict()
        port = _free_port()
        procs = [ctx.Process(target=_worker, args=(r, 2, port, ret)) for r in range(2)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(300)
            assert p.exitcode == 0
        assert ret.get(0) is True and ret.get(1) is True
