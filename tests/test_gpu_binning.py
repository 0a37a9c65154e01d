"""The beyond-L2 binned path, checked directly and end to end.

binning.cuh partitions the keys of a table too large for L2 by table slice (`partition`: hist64_kernel / scatter64_kernel
for 64 bins, hist_kernel<P> / scatter_kernel<P> for 2^7 .. 2^10) and walks the slices in groups (`apply_groups`).  The
final tables hide a key in the wrong bin or run -- every key is inserted by its own hash -- so the partition is checked
on its own here, through tests/device_harness/binning_harness.cu (built at test time with nvcc, like the host harness of
test_core_host.py), against an exact numpy reference: for every (bin, block) the count matrix, its bin-major exclusive
prefix and the multiset of keys in the run, for 4-byte ids, one-limb and two-limb k-mers at every bin count.  Then the
table entry points at the bin counts and inputs the other suites do not reach: P > 6, one key everywhere, a binned table
at more than 90 % load and one that overflows while binned."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import oracle as ko

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "kmers.jl_b200", "csrc")
FX = 0x517CC1B727220A95
FX_INV = pow(FX, -1, 1 << 64)
WIDTHS = (4, 8, 16)
PS = (6, 7, 8, 9, 10)
CUDA_SUCCESS, CUDA_INVALID_VALUE = 0, 1


# ------------------------------------------------------------------------------------------------------ the harness
@pytest.fixture(scope="module")
def bh(tmp_path_factory):
    nvcc = shutil.which("nvcc") or ("/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else None)
    if nvcc is None:
        pytest.skip("no nvcc")
    so = str(tmp_path_factory.mktemp("binning_harness") / "libbinning_harness.so")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
                    "-Xcompiler", "-fPIC", "-shared", "-I", CSRC, os.path.join(ROOT, "tests", "device_harness", "binning_harness.cu"),
                    os.path.join(CSRC, "scan.cu"), "-o", so], check=True)
    lib = C.CDLL(so)
    P = C.POINTER
    lib.bh_shape.restype = C.c_int
    lib.bh_shape.argtypes = [C.c_int, P(C.c_int), P(C.c_int), P(C.c_int)]
    lib.bh_blocks_for.restype = C.c_uint64
    lib.bh_blocks_for.argtypes = [C.c_int, C.c_uint64]
    lib.bh_bin_range.restype = C.c_int
    lib.bh_bin_range.argtypes = [P(C.c_int), P(C.c_int)]
    lib.bh_partition.restype = C.c_int
    lib.bh_partition.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p,
                                 P(C.c_int), P(C.c_int)]
    lib.bh_partition_check_large.restype = C.c_int
    lib.bh_partition_check_large.argtypes = [C.c_int, C.c_int, C.c_uint64, C.c_uint64, C.c_void_p]
    lib.bh_apply_groups_schedule.restype = C.c_int
    lib.bh_apply_groups_schedule.argtypes = [C.c_int, C.c_int, C.c_uint, C.c_void_p, C.c_void_p]
    lib.bh_mem_get_info.restype = C.c_int
    lib.bh_mem_get_info.argtypes = [P(C.c_uint64), P(C.c_uint64)]
    return lib


def shape(bh, key_bytes):
    """(kPerVec, kPerIter, kChunk) of binning::Shape for the key width, as the harness compiled it."""
    v, it, ch = C.c_int(), C.c_int(), C.c_int()
    assert bh.bh_shape(key_bytes, C.byref(v), C.byref(it), C.byref(ch)) == 0
    return v.value, it.value, ch.value


def partition(bh, key_bytes, p, shift, keys):
    """One binning::partition on the device: (status, out, offs, matrix, guard intact, input unchanged)."""
    n = len(keys)
    cells = (1 << p) * bh.bh_blocks_for(key_bytes, n)
    keys = np.ascontiguousarray(keys)
    out = np.zeros_like(keys) if n else np.zeros(1, dtype=keys.dtype)
    offs = np.zeros(cells + 1, dtype=np.uint64)
    matrix = np.zeros(max(cells, 1), dtype=np.uint64)
    g, i = C.c_int(), C.c_int()
    st = bh.bh_partition(key_bytes, p, shift, keys.ctypes.data if n else None, n, out.ctypes.data, offs.ctypes.data,
                         matrix.ctypes.data, C.byref(g), C.byref(i))
    return st, out[:n], offs, matrix[:cells], bool(g.value), bool(i.value)


# ------------------------------------------------------------------------------------------------------ exact reference
def rotl5(x):
    return (x << np.uint64(5)) | (x >> np.uint64(59))


def hash_of(keys, key_bytes):
    """The 64-bit hash whose top bits are the bin: fx_hash of a one-limb k-mer, key_hash of a two-limb one (table_keys.cuh)."""
    with np.errstate(over="ignore"):
        if key_bytes == 8:
            return keys * np.uint64(FX)
        return (rotl5(keys[:, 0] * np.uint64(FX)) ^ keys[:, 1]) * np.uint64(FX)


def bin_of(keys, key_bytes, p, shift):
    if key_bytes == 4:
        return (keys >> np.uint32(shift)).astype(np.int64)
    return (hash_of(keys, key_bytes) >> np.uint64(64 - p)).astype(np.int64)


def keys_in_bins(rng, key_bytes, p, shift, bins, low=None):
    """Keys whose bin is bins[i], by inverting the bin function: ids (b << shift) | low; one limb h * FX^-1 with
    h = (b << (64 - P)) | low; two limbs a random head x and y = (h * FX^-1) ^ rotl(x * FX, 5)."""
    bins = np.asarray(bins, dtype=np.uint64)
    n = len(bins)
    low_bits = shift if key_bytes == 4 else 64 - p
    if low is None:
        low = rng.integers(0, 2**64, size=n, dtype=np.uint64) & np.uint64((1 << low_bits) - 1)
    if key_bytes == 4:
        return ((bins << np.uint64(shift)) | low).astype(np.uint32)
    h = (bins << np.uint64(64 - p)) | low
    with np.errstate(over="ignore"):
        k = h * np.uint64(FX_INV)
        if key_bytes == 8:
            return k
        x = rng.integers(0, 2**64, size=n, dtype=np.uint64)
        return np.stack([x, k ^ rotl5(x * np.uint64(FX))], axis=1)


def sorted_by_run(keys, run):
    """keys ordered by (run, key): two arrays equal <=> every run holds the same multiset of keys."""
    if keys.dtype == np.uint32:  # (run, id) packed in one word sorts faster than a lexsort
        return np.sort((run.astype(np.uint64) << np.uint64(32)) | keys)
    cols = (keys,) if keys.ndim == 1 else (keys[:, 1], keys[:, 0])
    return keys[np.lexsort(cols + (run,))]


def check_partition(keys, bins, p, chunk, out, offs, matrix):
    """What binning::partition promises, exactly: matrix[b * nb + blk] = keys of chunk blk (kChunk keys per block) in
    bin b; offs = its bin-major exclusive prefix, offs[cells] = n; out[offs[c] .. offs[c + 1]) = the keys of cell c."""
    n = len(bins)
    nb = -(-n // chunk)
    cells = (1 << p) * nb
    cell = bins * nb + np.arange(n, dtype=np.int64) // chunk
    want_m = np.bincount(cell, minlength=cells).astype(np.uint64)
    assert matrix.shape == (cells,) and np.array_equal(matrix, want_m), "count matrix"
    want_o = np.zeros(cells + 1, dtype=np.uint64)
    want_o[1:] = np.cumsum(want_m)
    assert np.array_equal(offs, want_o), "offsets"
    assert out.shape == keys.shape, "output size"
    run = np.searchsorted(offs, np.arange(n, dtype=np.uint64), side="right").astype(np.int64) - 1  # cell of each position
    assert np.array_equal(sorted_by_run(out, run), sorted_by_run(keys, cell)), "keys of a (bin, block) run"


# ------------------------------------------------------------------------------------------------------ inputs
def thread_of(n, key_bytes):
    """The thread of the block that load_iter hands key i to (warp w: 32 * kPerThread keys as four rows of one 128-bit
    vector per lane)."""
    v = 16 // key_bytes
    pt = 4 * v
    j = np.arange(n, dtype=np.int64) % (256 * pt)
    return (j // (32 * pt)) * 32 + (j % (32 * v)) // v


BIG_N = 2_000_003
BIG_N_DISTRIBUTIONS = ("uniform", "one bin per thread")  # (the small sizes take every distribution)


def distributions(rng, key_bytes, p, shift, n, only=None):
    """(name, keys) for the inputs where a partition goes wrong: uniform, everything in the first / last / a middle bin,
    two alternating bins, round robin, ascending bins, and every thread's keys in one bin."""
    nb = 1 << p
    top = shift + p if key_bytes == 4 else 64
    if only is None or "uniform" in only:
        if key_bytes == 4:
            u = (rng.integers(0, 2**top, size=n, dtype=np.uint64)).astype(np.uint32)
            u[-1:] = (1 << top) - 1  # (shift 22, P 10: id 0xFFFFFFFF)
        else:
            u = keys_in_bins(rng, key_bytes, p, shift, rng.integers(0, nb, size=n))
        yield "uniform", u
    i = np.arange(n, dtype=np.int64)
    for name, bins in (("first bin", lambda: np.zeros(n, np.int64)), ("last bin", lambda: np.full(n, nb - 1)),
                       ("middle bin", lambda: np.full(n, nb // 2 + 1)),
                       ("two alternating", lambda: np.where(i % 2 == 0, 3, nb - 2)), ("round robin", lambda: i % nb),
                       ("ascending", lambda: np.sort(rng.integers(0, nb, size=n))),
                       ("one bin per thread", lambda: thread_of(n, key_bytes) % nb)):
        if only is not None and name not in only:
            continue
        bins = bins()
        low = None
        if name == "last bin":  # the largest key of the last bin as well
            low_bits = shift if key_bytes == 4 else 64 - p
            low = rng.integers(0, 2**64, size=n, dtype=np.uint64) & np.uint64((1 << low_bits) - 1)
            low[::7] = np.uint64((1 << low_bits) - 1)
        yield name, keys_in_bins(rng, key_bytes, p, shift, bins, low)


def sizes(bh, key_bytes):
    v, it, ch = shape(bh, key_bytes)
    return sorted({1, v - 1, v + 1, it - 1, it, it + 1, ch - 1, ch, ch + 1, 3 * ch + 5, BIG_N} - {0})


# ------------------------------------------------------------------------------------------------------ CPU tests
def test_shape_constants_and_blocks(bh):
    """The harness's view of binning::Shape: four 128-bit loads per thread and iteration, four iterations per block."""
    lo, hi = C.c_int(), C.c_int()
    bh.bh_bin_range(C.byref(lo), C.byref(hi))
    assert (lo.value, hi.value) == (min(PS), max(PS))
    for kb in WIDTHS:
        v, it, ch = shape(bh, kb)
        assert v == 16 // kb and it == 256 * 4 * v and ch == 4 * it
        for n in (0, 1, ch - 1, ch, ch + 1, 2**32 + 12_345):
            assert bh.bh_blocks_for(kb, n) == -(-n // ch)
    assert bh.bh_shape(12, C.byref(lo), C.byref(hi), C.byref(lo)) == -1


@pytest.mark.parametrize("key_bytes", WIDTHS)
def test_the_partition_checker_rejects_corrupted_partitions(bh, key_bytes):
    """check_partition accepts a correct partition (built in numpy, any order inside a run) and rejects four corrupted
    ones: two keys swapped across bins, a run boundary moved by one, a key dropped, a key duplicated."""
    rng = np.random.default_rng(40 + key_bytes)
    _, _, chunk = shape(bh, key_bytes)
    p, shift = 6, 26
    n = 2 * chunk + 77
    keys = keys_in_bins(rng, key_bytes, p, shift, rng.integers(0, 1 << p, size=n))
    bins = bin_of(keys, key_bytes, p, shift)
    nb = -(-n // chunk)
    cell = bins * nb + np.arange(n) // chunk
    order = np.lexsort((rng.random(n), cell))
    out = keys[order]
    matrix = np.bincount(cell, minlength=(1 << p) * nb).astype(np.uint64)
    offs = np.concatenate([[0], np.cumsum(matrix)]).astype(np.uint64)
    check_partition(keys, bins, p, chunk, out, offs, matrix)
    out_bins = bin_of(out, key_bytes, p, shift)

    swapped = out.copy()
    i = 0
    j = int(np.flatnonzero(out_bins != out_bins[i])[0])
    swapped[[i, j]] = swapped[[j, i]]
    moved = offs.copy()
    c = int(np.flatnonzero(matrix)[3]) + 1  # a boundary between two non-empty runs
    moved[c] += np.uint64(1)
    dropped = out.copy()
    dropped[5] = keys_in_bins(rng, key_bytes, p, shift, [out_bins[5]])[0]  # a key of the same bin that is not in the input
    run = np.searchsorted(offs, np.arange(n, dtype=np.uint64), side="right") - 1
    k = int(np.flatnonzero(run[1:] == run[:-1])[0])
    duplicated = out.copy()
    duplicated[k + 1] = duplicated[k]  # (its own run: the bins and the matrix still add up)
    for o, f, why in ((swapped, offs, "keys of a"), (out, moved, "offsets"), (dropped, offs, "keys of a"),
                      (duplicated, offs, "keys of a")):
        with pytest.raises(AssertionError, match=why):
            check_partition(keys, bins, p, chunk, o, f, matrix)


# ------------------------------------------------------------------------------------------------------ partition on the GPU
@pytest.mark.gpu
@pytest.mark.parametrize("p", PS)
@pytest.mark.parametrize("key_bytes", WIDTHS)
def test_partition_matches_the_exact_reference(bh, key_bytes, p):
    """Every (key width, P) instance of partition -- 64 bins: hist64 / scatter64; more: hist_kernel<P> / scatter_kernel<P>
    -- at sizes around the vector, iteration and block boundaries for every distribution, and at two million keys uniform
    and one bin per thread; ids at shifts 0, 16 and 22 (two million: 0 and 22).  Each run is checked against the reference, leaves the input and the 4 KB behind the output
    alone, and a second run gives the same bytes."""
    rng = np.random.default_rng(1000 * key_bytes + p)
    _, _, chunk = shape(bh, key_bytes)
    for shift in ((0, 16, 22) if key_bytes == 4 else (0,)):
        for n in sizes(bh, key_bytes):
            if n == BIG_N and shift not in (0, 22):
                continue
            for name, keys in distributions(rng, key_bytes, p, shift, n, BIG_N_DISTRIBUTIONS if n == BIG_N else None):
                what = (key_bytes, p, shift, n, name)
                st, out, offs, matrix, guard, same_in = partition(bh, key_bytes, p, shift, keys)
                assert st == CUDA_SUCCESS, what
                assert guard and same_in, what
                check_partition(keys, bin_of(keys, key_bytes, p, shift), p, chunk, out, offs, matrix)
                st2, out2, offs2, matrix2, _, _ = partition(bh, key_bytes, p, shift, keys)
                assert st2 == CUDA_SUCCESS and out2.tobytes() == out.tobytes(), what
                assert np.array_equal(offs2, offs) and np.array_equal(matrix2, matrix), what


@pytest.mark.gpu
@pytest.mark.parametrize("key_bytes", WIDTHS)
def test_partition_rejects_bin_counts_out_of_range(bh, key_bytes):
    rng = np.random.default_rng(key_bytes)
    keys = keys_in_bins(rng, key_bytes, 6, 0, np.zeros(100, np.int64))
    for p in (5, 11):
        assert partition(bh, key_bytes, p, 0, keys)[0] == CUDA_INVALID_VALUE, p
    st, out, offs, _, guard, _ = partition(bh, key_bytes, 6, 0, keys[:0])
    assert st == CUDA_SUCCESS and out.size == 0 and guard


def free_device_bytes(bh):
    f, t = C.c_uint64(), C.c_uint64()
    assert bh.bh_mem_get_info(C.byref(f), C.byref(t)) == CUDA_SUCCESS
    return f.value


@pytest.mark.gpu
@pytest.mark.parametrize("key_bytes,p,n", [(4, 7, 2**29 + 3), (8, 6, 2**29 + 1), (8, 9, 2**29 - 7), (16, 6, 2**29 - 1),
                                           (16, 10, 2**29 + 5), (4, 10, 2**32 + 12_345)])
def test_partition_of_large_inputs_verified_on_the_device(bh, key_bytes, p, n):
    """Half a billion keys of every width, and 2^32 + 12 345 ids (34 GB of input and output: flat indices past 32 bits),
    generated, partitioned and checked on the device: every key lies in the range of its own bin, the per-bin count,
    xor and sum of the keys agree between input and output, offs is the scan of the matrix and ends at n, the guard
    behind the output is intact."""
    need = 2 * n * key_bytes + 16 * (1 << p) * bh.bh_blocks_for(key_bytes, n) + (2 << 30)
    free = free_device_bytes(bh)
    if free < need:
        pytest.skip(f"needs about {need / 2**30:.0f} GiB of free device memory, {free / 2**30:.0f} GiB free")
    report = np.zeros(6, dtype=np.uint64)
    assert bh.bh_partition_check_large(key_bytes, p, n, 0x5EED + p, report.ctypes.data) == CUDA_SUCCESS
    misplaced, bins_differ, bad_cells, total, guard_bytes, bad_input = (int(x) for x in report)
    assert (misplaced, bins_differ, bad_cells, guard_bytes, bad_input) == (0, 0, 0, 0, 0)
    assert total == n


# ------------------------------------------------------------------------------------------------------ progress events
@pytest.mark.gpu
def test_apply_groups_records_each_event_once_its_range_is_final(bh):
    """apply_groups records event i once the bins [0, (i + 1) * n_bins / n_parts) are applied: a second stream that waits
    for event i and reads the last applied bin end must see at least that (the apply holds its stream ~10 us before it
    writes, so an event recorded ahead of its group would be read too early).  Every event is recorded."""
    for n_bins in (64, 128, 256, 512, 1024):
        for group in (1, 2, 3, 6):
            for n_parts in (1, 2, 4, 8, 16, 32):
                seen = np.zeros(n_parts, dtype=np.uint32)
                rec = np.zeros(n_parts, dtype=np.int32)
                assert bh.bh_apply_groups_schedule(n_bins, group, n_parts, seen.ctypes.data, rec.ctypes.data) == CUDA_SUCCESS
                what = (n_bins, group, n_parts)
                assert rec.all(), what
                i = np.arange(n_parts, dtype=np.int64)
                assert np.all((i + 1) * n_bins <= seen.astype(np.int64) * n_parts), (what, seen)
                assert np.all(seen <= n_bins), (what, seen)


# ------------------------------------------------------------------------------------------------------ end to end
@pytest.fixture(scope="module")
def kc():
    import kmerscuda
    return kmerscuda


def pack_codes(codes):
    """2-bit codes -> u64 words, symbol i at bits 2i of word i // 32."""
    codes = np.asarray(codes, dtype=np.uint64)
    pad = (-len(codes)) % 32
    c = np.concatenate([codes, np.zeros(pad, np.uint64)]).reshape(-1, 32)
    return np.bitwise_or.reduce(c << (np.uint64(2) * np.arange(32, dtype=np.uint64)), axis=1)


def uniform_set(kc, rng, genome, n_reads=3000, length=150):
    stride = (length + 31) // 32
    starts = rng.integers(0, len(genome) - length + 1, size=n_reads)
    codes = np.zeros((n_reads, stride * 32), dtype=np.uint64)
    codes[:, :length] = genome[starts[:, None] + np.arange(length)[None, :]]
    words = pack_codes(codes.reshape(-1))
    layout = dict(uniform_len=length, uniform_stride=stride)
    return kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride), words, n_reads, layout


def ragged_set(kc, rng, genome, n_reads=3000, max_len=260):
    lens = rng.integers(0, max_len + 1, size=n_reads)
    lens[:4] = [0, 1, 63, 64]
    parts, off = [], [0]
    for ln in lens:
        s0 = int(rng.integers(0, len(genome) - max_len))
        w = pack_codes(genome[s0:s0 + int(ln)]) if ln else np.zeros(0, np.uint64)
        parts.append(w)
        off.append(off[-1] + len(w))
    words = np.concatenate(parts + [np.zeros(1, np.uint64)])
    off, ln = np.asarray(off[:-1], np.uint64), np.asarray(lens, np.uint64)
    return kc.ReadSet(2, words, n_reads, seq_word_offset=off, seq_len=ln), words, n_reads, dict(word_off=off, seq_len=ln)


def unique_counts(a):
    """np.unique(..., return_counts=True) of a k-mer stream u64[n, limbs], rows in the order KmerTable.items() returns."""
    if a.shape[1] == 1:
        k, c = np.unique(a[:, 0], return_counts=True)
        return k, c.astype(np.uint32)
    s = a[np.lexsort((a[:, 1], a[:, 0]))]
    first = np.ones(len(s), dtype=bool)
    first[1:] = (s[1:] != s[:-1]).any(axis=1)
    idx = np.flatnonzero(first)
    return s[idx], np.diff(np.append(idx, len(s))).astype(np.uint32)


def check_table(t, uk, uc, times=1):
    assert t.n_keys == len(uk)
    gk, gc = t.items()
    assert np.array_equal(gk, uk) and np.array_equal(gc, times * uc)


def mode(canonical):
    return ko.CANON if canonical else ko.FW


@pytest.mark.gpu
@pytest.mark.parametrize("n_limbs,k,log2cap", [(1, 31, 27), (1, 21, 29), (2, 63, 27), (2, 41, 28)])
def test_kmer_tables_with_more_than_64_bins(kc, n_limbs, k, log2cap):
    """kmc_kmer_count at 2^27 and 2^29 slots (128 and 512 bins: 1.5 and 6 GB), kmc_kmer_count2 at 2^27 and 2^28 (128 and
    256 bins of 16-byte keys: 2.5 and 5 GB), over a uniform and a ragged set, counted twice."""
    rng = np.random.default_rng(50 + log2cap + k)
    genome = rng.integers(0, 4, size=60_000).astype(np.uint64)
    for make in (uniform_set, ragged_set):
        rs, words, n_reads, layout = make(kc, rng, genome)
        a, _, _, _ = ko.batch_iterate(words, n_reads, k, ko.CANON, **layout)
        uk, uc = unique_counts(a)
        t = kc.KmerTable(log2cap, n_limbs=n_limbs)
        n, _ = t.count(rs, k)
        assert n == a.shape[0]
        check_table(t, uk, uc)
        t.count(rs, k)
        check_table(t, uk, uc, 2)
        t.free()


@pytest.mark.gpu
def test_bucket_count_with_128_bins(kc):
    """kmc_bucket_count at B = 29 (128 bins of 2^22 counters, 2 GB) over a ragged set: the exact path; counted twice."""
    rng = np.random.default_rng(29)
    genome = rng.integers(0, 4, size=2_000_000).astype(np.uint64)
    rs, words, n_reads, layout = ragged_set(kc, rng, genome, n_reads=40_000, max_len=300)
    bits, k = 29, 31
    _, _, h, _ = ko.batch_iterate(words, n_reads, k, ko.CANON, want_hash=True, **layout)
    idx, cnt = np.unique((h >> np.uint64(64 - bits)).astype(np.int64), return_counts=True)
    ctx = kc.default_context()
    table = ctx.alloc(4 << bits)
    try:
        ctx._check(ctx.lib.kmc_memset(ctx.handle, table.ptr, 0, 4 << bits))
        for times in (1, 2):
            got, n, _ = kc.bucket_count(rs, k, bits, ctx=ctx, table=table)
            assert n == h.size
            assert int(got.sum(dtype=np.int64)) == times * h.size
            assert np.array_equal(np.flatnonzero(got), idx) and np.array_equal(got[idx], times * cnt.astype(np.uint32))
            del got
    finally:
        table.free()


@pytest.mark.gpu
@pytest.mark.parametrize("n_limbs,k,canonical,base", [(1, 31, False, 0), (1, 31, True, 0), (1, 31, False, 3), (1, 31, True, 3),
                                                      (2, 63, False, 3), (2, 64, True, 3)])
def test_one_key_everywhere(kc, n_limbs, k, canonical, base):
    """Poly-A (base 0) and poly-T (base 3) reads: every window is one k-mer (K = 63 forward over poly-T is {2^62 - 1, ~0},
    so every two-limb insert re-reads its slot through the compare-and-swap, all at once).  In a streaming table and in a
    binned one, where every key falls into one bin: one key, counted once per window."""
    n_reads, length = 2000, 150
    rng = np.random.default_rng(k)
    rs, words, _, layout = uniform_set(kc, rng, np.full(length, base, np.uint64), n_reads, length)
    a, _, _, _ = ko.batch_iterate(words, n_reads, k, mode(canonical), **layout)
    uk, uc = unique_counts(a)
    assert len(uk) == 1 and uc[0] == n_reads * (length - k + 1)
    for log2cap in (16, 24 if n_limbs == 1 else 23):  # streaming; binned (192 / 160 MB)
        t = kc.KmerTable(log2cap, n_limbs=n_limbs)
        n, _ = t.count(rs, k, canonical=canonical)
        assert n == a.shape[0]
        check_table(t, uk, uc)
        t.free()


def random_sequence(kc, rng, n):
    w = rng.integers(0, 2**64, size=(n + 31) // 32, dtype=np.uint64)
    return kc.ReadSet.single(kc.LongSequence(kc.DNAAlphabet2, w, n)), w


@pytest.mark.gpu
@pytest.mark.parametrize("n_limbs,k,log2cap,n_bases", [(1, 31, 24, 15_200_000), (2, 41, 23, 7_600_000)])
def test_binned_table_at_high_load_and_overflow(kc, n_limbs, k, log2cap, n_bases):
    """A binned table (64 bins) filled past 90 % with distinct k-mers of one random sequence: probe chains cross the slice
    boundaries between apply launches and the last slice wraps to slot 0.  Exact, then doubled by a second count.  Then
    a second sequence brings the distinct keys to 512 more than the slots, which must report the table full."""
    rng = np.random.default_rng(log2cap)
    rs, w = random_sequence(kc, rng, n_bases)
    a, _, _ = ko.iterate(w, n_bases, k, ko.CANON)
    uk, uc = unique_counts(a)
    slots = 1 << log2cap
    assert len(uk) >= 0.9 * slots
    t = kc.KmerTable(log2cap, n_limbs=n_limbs)
    try:
        n, _ = t.count(rs, k)
        assert n == n_bases - k + 1
        check_table(t, uk, uc)
        t.count(rs, k)
        check_table(t, uk, uc, 2)
        extra = slots - len(uk) + 512  # new distinct keys: 512 of them find no slot
        rs2, w2 = random_sequence(kc, rng, extra + k - 1)
        a2, _, _ = ko.iterate(w2, extra + k - 1, k, ko.CANON)
        both = unique_counts(np.concatenate([a, a2]))[0]
        assert len(both) == slots + 512
        with pytest.raises(kc.KmersCUDAError, match="full"):
            t.count(rs2, k)
    finally:
        t.free()
