"""Every k-mer consumer on every read-set layout of the launch planner, against the oracle's k-mer stream.

The consumers -- minhash_sketch, minhash_sketches, composition, the exact k-mer tables (count, lookup, one and two
limbs), bucket_count and minimizers -- reduce the k-mer stream on the device instead of writing it out.  All of them
but the minimizers are laid out by plan_layout (api.cu), which sends a set down a different kernel path by its shape:
the aligned consume kernel or the general tile cursor, a partial last group (al_tail), views (first_symbol_offset),
clamped loads at the end of the buffer, one block width (nx) per K class, and the binned paths of tables beyond L2.
Each layout below is built to reach one of those cases, and asserts that it does by restating the planner's predicate
(set_iteration_strides) before it is used.

The reference stream of a set is oracle.iterate over each of its sequences (`(words, length, first)`), concatenated;
every reference below is an exact integer reduction of that stream in numpy, and every comparison is exact: values,
n_written, and the number of keys or the row lengths.

test_general_path_on_aligned_sets runs the file once more with KMC_ALIGNED_KERNEL=0, which sends the aligned sets
through the general kernel.
"""
import ctypes as C
import functools
import os
import subprocess
import sys
import zlib
from dataclasses import dataclass

import numpy as np
import pytest

from oracle import oracle as ko

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

FW, CANON = ko.FW, ko.CANON
MODES = (FW, CANON)
# K at both ends of every (limbs, nx) class: one limb (G = 8) nx = 1: 1..9, 2: 10..25, 3: 26..32; two limbs (G = 4)
# nx = 3: 33..45, 4: 46..61, 5: 62..64
K_ONE = (5, 9, 10, 25, 26, 31, 32)
K_TWO = (33, 45, 46, 61, 62, 63, 64)
K_ALL = K_ONE + K_TWO
K_PER_LIMB = (25, 61)  # one K per limb count on the layouts that do not run the full list
COMP_K = (1, 6, 7, 9, 10, 12)  # composition: shared-memory counters up to K = 9 or so, direct atomics above
FULL_LAYOUTS = ("S1", "U0", "U1")
OTHER_LAYOUTS = ("S0", "U2", "U3", "U4", "R0")
TILE_ITEMS = 256 * 8  # kTileItems: work items per tile (extract_kernels.cuh)


def group_of(k):
    return 8 if k <= 32 else 4


def nx_of(k):
    if k <= 32:
        return 1 if k <= 9 else 2 if k <= 25 else 3
    return 3 if k <= 45 else 4 if k <= 61 else 5


def planner_class(rs, k):
    """("aligned", al_tail), ("general", 0) or ("ragged", 0): plan_layout's group slots per read and the predicate of
    set_iteration_strides (extract_kernels.cuh), restated."""
    if rs.seq_len is not None:
        return ("ragged", 0)
    g = group_of(k)
    wpr = max(0, rs.uniform_len - k + 1)
    if rs.n_seqs == 1:
        gprm = -(-wpr // g)
    else:
        gprm = wpr // g if wpr % g == 0 else -(-wpr // g) + 1
    whole = wpr > 0 and wpr % g == 0 and gprm == wpr // g
    single = wpr > 0 and rs.n_seqs == 1 and gprm == -(-wpr // g)
    if (whole or single) and rs.seq_word_offset is None:
        return ("aligned", 0 if whole else wpr % g)
    return ("general", 0)


@pytest.fixture(scope="module")
def kc():
    import kmerscuda
    return kmerscuda


@pytest.fixture(scope="module")
def ctx(kc):
    return kc.default_context()


# ----------------------------------------------------------------------------------------------------- layouts
@dataclass
class Case:
    name: str
    rs: object
    per: list     # (words, length, first) of every sequence
    expect: tuple  # planner_class


def _rand_words(rng, n):
    return rng.integers(0, 2**64, size=max(int(n), 0), dtype=np.uint64)


def _uniform(kc, rng, name, k, n_seqs, length, first, stride_extra, expect):
    stride = -(-(first + length) // 32) + stride_extra
    words = _rand_words(rng, max(n_seqs * stride, 1))  # random bits in the padding too
    rs = kc.ReadSet(2, words, n_seqs, uniform_len=length, uniform_stride_words=stride, first_symbol_offset=first)
    per = [(words[i * stride:(i + 1) * stride], length, first) for i in range(n_seqs)]
    return Case(name, rs, per, expect)


def _single(kc, rng, name, k, n_words, length, first, expect):
    words = _rand_words(rng, n_words)
    rs = kc.ReadSet(2, words, 1, uniform_len=length, uniform_stride_words=n_words, first_symbol_offset=first)
    return Case(name, rs, [(words, length, first)], expect)


def build_S0(kc, rng, k):
    # one sequence whose last window ends on the last symbol of the buffer (n_words tight) with whole groups only:
    # K = 1 mod G
    g = group_of(k)
    assert (k - 1) % g == 0, "S0 needs K = 1 mod G"
    nw = 1536
    return [_single(kc, rng, "S0", k, nw, 32 * nw, 0, ("aligned", 0))]


def build_S1(kc, rng, k):
    # one sequence with a partial last group, and views starting inside a word, ending inside the buffer or at its end
    g = group_of(k)
    m = 2600
    out = []
    for first, tail in ((0, 1), (0, g - 1), (1, 1), (33, g - 1)):
        length = g * m + tail + k - 1
        nw = -(-(first + length) // 32) + 2
        out.append(_single(kc, rng, f"S1-f{first}-t{tail}", k, nw, length, first, ("aligned", tail)))
    for first in (31, 70):  # the view ends on the buffer's last symbol
        nw = -(-(g * m + k + first) // 32)
        length = 32 * nw - first
        out.append(_single(kc, rng, f"S1-f{first}-end", k, nw, length, first, ("aligned", (length - k + 1) % g)))
    return out


def _u_reads(g):
    # 12 groups per read; enough reads for more than two tiles, the last one partial
    n = 2 * TILE_ITEMS // 12 + 5
    assert (n * 12) % TILE_ITEMS != 0
    return n


def build_U0(kc, rng, k):
    g = group_of(k)
    return [_uniform(kc, rng, "U0", k, _u_reads(g), 12 * g + k - 1, 0, 1, ("aligned", 0))]


def build_U1(kc, rng, k):
    g = group_of(k)
    return [_uniform(kc, rng, "U1", k, _u_reads(g), 12 * g + 3 + k - 1, 0, 0, ("general", 0))]


def build_U2(kc, rng, k):
    g = group_of(k)
    out = []
    for first in (7, 40):
        out.append(_uniform(kc, rng, f"U2-aligned-f{first}", k, _u_reads(g), 12 * g + k - 1, first, 1, ("aligned", 0)))
        out.append(_uniform(kc, rng, f"U2-general-f{first}", k, _u_reads(g), 12 * g + 3 + k - 1, first, 0, ("general", 0)))
    return out


def build_U3(kc, rng, k):
    short = _uniform(kc, rng, "U3-short", k, 5, k - 1, 0, 1, ("general", 0))
    empty = Case("U3-empty", kc.ReadSet(2, _rand_words(rng, 4), 0, uniform_len=3 * k, uniform_stride_words=4), [], None)
    return [short, empty]


def build_U4(kc, rng, k):
    # uniform length, explicit word offsets in permuted order (with gaps): the aligned form is off however the windows fall
    g = group_of(k)
    n, length = 300, 12 * g + k - 1
    nw = -(-length // 32)
    order = rng.permutation(n)
    off = np.zeros(n, dtype=np.uint64)
    at = 0
    for i in order:
        at += int(rng.integers(0, 2))
        off[i] = at
        at += nw
    words = _rand_words(rng, at + 1)
    rs = kc.ReadSet(2, words, n, seq_word_offset=off, uniform_len=length)
    per = [(words[int(o):int(o) + nw + 1], length, 0) for o in off]
    return [Case("U4", rs, per, ("general", 0))]


def build_R0(kc, rng, k):
    g = group_of(k)
    out = []
    for first in (0, 9):
        lens = np.concatenate([[0, k - 1, k, k + g - 1], rng.integers(0, 400, size=300)]).astype(np.uint64)
        rng.shuffle(lens)
        nws = [-(-(first + int(n)) // 32) + int(rng.integers(0, 2)) for n in lens]
        off = np.zeros(len(lens), dtype=np.uint64)
        off[1:] = np.cumsum(nws)[:-1]
        words = _rand_words(rng, sum(nws) + 1)
        rs = kc.ReadSet(2, words, len(lens), seq_word_offset=off, seq_len=lens, first_symbol_offset=first)
        per = [(words[int(o):int(o) + w + 1], int(n), first) for o, w, n in zip(off, nws, lens)]
        out.append(Case(f"R0-f{first}", rs, per, ("ragged", 0)))
    return out


BUILDERS = {"S0": build_S0, "S1": build_S1, "U0": build_U0, "U1": build_U1, "U2": build_U2, "U3": build_U3, "U4": build_U4,
            "R0": build_R0}


@functools.lru_cache(maxsize=None)
def cases(layout, k):
    import kmerscuda as kc
    rng = np.random.default_rng(zlib.crc32(f"{layout}-{k}".encode()))
    cs = BUILDERS[layout](kc, rng, k)
    for c in cs:
        if c.expect is not None:
            assert planner_class(c.rs, k) == c.expect, (c.name, k)
    return cs


@functools.lru_cache(maxsize=None)
def device_set(layout, k, i):
    import kmerscuda as kc
    return kc.DeviceReadSet(kc.default_context(), cases(layout, k)[i].rs)


class Stream:
    """The oracle's k-mer stream of one set: a [n, N], hashes h [n], per-sequence offsets."""

    def __init__(self, per, k, mode):
        parts = [ko.iterate(w, n, k, mode, first=f, want_hash=True) for w, n, f in per]
        N = ko.n_limbs(k)
        self.k, self.N = k, N
        self.a = np.concatenate([p[0] for p in parts]) if parts else np.zeros((0, N), np.uint64)
        self.h = np.concatenate([p[2] for p in parts]) if parts else np.zeros(0, np.uint64)
        self.off = np.zeros(len(per) + 1, dtype=np.int64)
        self.off[1:] = np.cumsum([p[0].shape[0] for p in parts])
        self.total = int(self.off[-1])

    def seq(self, i):
        return self.a[self.off[i]:self.off[i + 1]], self.h[self.off[i]:self.off[i + 1]]

    @functools.cached_property
    def table(self):
        """(distinct keys sorted as KmerTable.items returns them, inverse of every window, counts)"""
        if self.N == 1:
            u, inv, c = np.unique(self.a[:, 0], return_inverse=True, return_counts=True)
        else:
            u, inv, c = np.unique(self.a, axis=0, return_inverse=True, return_counts=True)
        return u, inv.reshape(-1), c.astype(np.uint32)


@functools.lru_cache(maxsize=None)
def stream(layout, k, i, mode):
    return Stream(cases(layout, k)[i].per, k, mode)


def plan(layouts_full, layouts_other, k_full, k_other):
    return [(lay, k) for lay in layouts_full for k in k_full] + [(lay, k) for lay in layouts_other for k in k_other]


def each(layout, k):
    return range(len(cases(layout, k)))


def table_modes(k):
    """the modes the exact tables take at this K: forward up to 31 / 63, canonical up to 32 / 64"""
    return [m for m in MODES if not (m == FW and k in (32, 64))]


LAYOUT_K = plan(FULL_LAYOUTS, OTHER_LAYOUTS, K_ALL, K_PER_LIMB)


def test_layouts_cover_every_block_width_aligned_and_not():
    """Every (limbs, nx) class at both of its ends, on an aligned and on an unaligned set."""
    classes = {(1 if k <= 32 else 2, nx_of(k)) for k in K_ALL}
    assert classes == {(1, 1), (1, 2), (1, 3), (2, 3), (2, 4), (2, 5)}
    for k in K_ALL:
        kinds = {c.expect[0] for lay in FULL_LAYOUTS for c in cases(lay, k)}
        assert {"aligned", "general"} <= kinds, k
        assert any(c.expect[1] for c in cases("S1", k)), k  # a partial last group


# ------------------------------------------------------------------------------------------------ MinHash sketches
@pytest.mark.parametrize("layout,k", LAYOUT_K)
def test_minhash_sketch(kc, ctx, layout, k):
    for i in each(layout, k):
        drs = device_set(layout, k, i)
        for mode in MODES:
            u = np.unique(stream(layout, k, i, mode).h)
            for s in (1, 100, 5000, len(u) + 7):
                got = kc.minhash_sketch(drs, k, s, canonical=mode == CANON, ctx=ctx)
                assert np.array_equal(got, u[:s]), (cases(layout, k)[i].name, mode, s)


@pytest.mark.parametrize("layout,k", LAYOUT_K)
def test_minhash_sketches(kc, ctx, layout, k):
    for i in each(layout, k):
        drs = device_set(layout, k, i)
        n = drs.host.n_seqs
        for mode in MODES:
            st = stream(layout, k, i, mode)
            for s in (1, 100):
                rows, lens, info = kc.minhash_sketches(drs, k, s, canonical=mode == CANON, ctx=ctx, stats=True)
                exp = np.full((n, s), ~np.uint64(0), dtype=np.uint64)
                exp_n = np.zeros(n, dtype=np.uint32)
                for r in range(n):
                    u = np.unique(st.seq(r)[1])[:s]
                    exp[r, :len(u)] = u
                    exp_n[r] = len(u)
                assert np.array_equal(lens, exp_n) and np.array_equal(rows, exp), (cases(layout, k)[i].name, mode, s)
                assert info["n_written"] == int(exp_n.sum())


# ------------------------------------------------------------------------------------------------------- composition
def composition_twice(kc, ctx, drs, k, mode, st):
    """kmc_composition twice into one table: the counts of the stream, then every count doubled (the call accumulates)."""
    from kmerscuda import _abi
    n = 1 << (2 * k)
    table = ctx.alloc(4 * n)
    try:
        ctx._check(ctx.lib.kmc_memset(ctx.handle, table.ptr, 0, 4 * n))
        u, c = np.unique(st.a[:, 0], return_counts=True)
        for rep in (1, 2):
            res = _abi.kmc_result()
            ctx._check(ctx.lib.kmc_composition(ctx.handle, C.byref(drs.desc), k, mode, table.ptr, C.byref(res)))
            assert res.n_written == st.total
            if rep == 2 or k <= 12:
                host = table.download(np.uint32, n)
                nz = np.flatnonzero(host)
                assert np.array_equal(nz, u) and np.array_equal(host[nz], rep * c), (k, mode, rep)
    finally:
        table.free()


COMP_PLAN = (plan(FULL_LAYOUTS, (), COMP_K, ()) + [("S0", 1), ("S0", 9)] +
             plan((), ("U2", "U3", "U4", "R0"), (), (9, 12)) + [("U1", 14), ("R0", 14)])


@pytest.mark.parametrize("layout,k", COMP_PLAN)
def test_composition(kc, ctx, layout, k):
    for i in each(layout, k):
        for mode in MODES:
            composition_twice(kc, ctx, device_set(layout, k, i), k, mode, stream(layout, k, i, mode))


# ------------------------------------------------------------------------------------------------ exact k-mer tables
def check_table(kc, ctx, drs, k, mode, st, log2_capacity, what):
    t = kc.KmerTable(log2_capacity, ctx=ctx, n_limbs=1 if k <= 32 else 2)
    try:
        n, _ = t.count(drs, k, canonical=mode == CANON)
        u, inv, c = st.table
        assert n == st.total and t.n_keys == len(c), what
        keys, vals = t.items()
        assert np.array_equal(keys, u) and np.array_equal(vals, c), what
        assert np.array_equal(t.lookup(drs, k, canonical=mode == CANON), c[inv]), what
    finally:
        t.free()


def direct_capacity(st):
    return max(10, int(2 * len(st.table[2]) + 1).bit_length())


@pytest.mark.parametrize("layout,k", LAYOUT_K)
def test_kmer_table_count_and_lookup(kc, ctx, layout, k):
    for i in each(layout, k):
        for mode in table_modes(k):
            st = stream(layout, k, i, mode)
            check_table(kc, ctx, device_set(layout, k, i), k, mode, st, direct_capacity(st), (cases(layout, k)[i].name, mode))


@pytest.mark.parametrize("layout,k", plan(("S1", "U2", "R0", "U0", "S0"), (), K_PER_LIMB, ()))
def test_kmer_table_beyond_l2(kc, ctx, layout, k):
    """2^24 one-limb / 2^23 two-limb slots: the k-mers are written out, binned by table slice and inserted slice by slice."""
    for i in each(layout, k):
        for mode in table_modes(k):
            check_table(kc, ctx, device_set(layout, k, i), k, mode, stream(layout, k, i, mode), 24 if k <= 32 else 23,
                        (cases(layout, k)[i].name, mode, "beyond L2"))


@pytest.mark.parametrize("layout,k", [("U0", 25), ("U0", 61), ("S1", 25), ("R0", 61)])
def test_kmer_lookup_abi_edges(kc, ctx, layout, k):
    """out_counts 4 bytes past an aligned base (scalar stores), and capacity = windows - 1: KMC_E_OUT_TOO_SMALL, nothing
    written."""
    from kmerscuda import _abi
    drs = device_set(layout, k, 0)
    st = stream(layout, k, 0, CANON)
    t = kc.KmerTable(direct_capacity(st), ctx=ctx, n_limbs=1 if k <= 32 else 2)
    n = st.total
    out = ctx.alloc(4 * (n + 8))
    try:
        t.count(drs, k, canonical=True)
        u, inv, c = st.table
        fn = t._fn("kmc_kmer_lookup")
        res = _abi.kmc_result()
        ctx._check(fn(ctx.handle, C.byref(drs.desc), k, CANON, t.keys.ptr, t.vals.ptr, t.log2_capacity, out.ptr + 4, n, C.byref(res)))
        assert res.n_written == n
        assert np.array_equal(out.download(np.uint32, n, 4), c[inv])
        ctx._check(ctx.lib.kmc_memset(ctx.handle, out.ptr, 0xA5, 4 * (n + 8)))
        res = _abi.kmc_result()
        st_ = fn(ctx.handle, C.byref(drs.desc), k, CANON, t.keys.ptr, t.vals.ptr, t.log2_capacity, out.ptr, n - 1, C.byref(res))
        assert st_ == _abi.KMC_E_OUT_TOO_SMALL
        assert np.all(out.download(np.uint32, n + 8) == 0xA5A5A5A5)
    finally:
        out.free()
        t.free()


# ------------------------------------------------------------------------------------------------------ bucket count
def check_buckets(kc, ctx, drs, k, st, bits, what):
    table, n, _ = kc.bucket_count(drs, k, bits, ctx=ctx)
    u, c = np.unique(st.h >> np.uint64(64 - bits), return_counts=True)
    nz = np.flatnonzero(table)
    assert n == st.total and np.array_equal(nz, u) and np.array_equal(table[nz], c), what


@pytest.mark.parametrize("layout,k", LAYOUT_K)
def test_bucket_count_l2(kc, ctx, layout, k):
    for i in each(layout, k):
        check_buckets(kc, ctx, device_set(layout, k, i), k, stream(layout, k, i, CANON), 12, (cases(layout, k)[i].name, 12))


@pytest.mark.parametrize("layout,k", plan(FULL_LAYOUTS + OTHER_LAYOUTS, (), K_PER_LIMB, ()))
def test_bucket_count_beyond_l2(kc, ctx, layout, k):
    """2^26 buckets: one-limb k-mers of S0, U0 and their aligned views take the fused bins, the rest the exact binned path."""
    for i in each(layout, k):
        check_buckets(kc, ctx, device_set(layout, k, i), k, stream(layout, k, i, CANON), 26, (cases(layout, k)[i].name, 26))


# -------------------------------------------------------------------------------------------------------- minimizers
def minimizer_reference(st, W, step):
    """per sequence: for the window starts 0, step, ... the first k-mer of least hash among W consecutive ones"""
    km, ix, hh, off = [], [], [], [0]
    for r in range(len(st.off) - 1):
        a, h = st.seq(r)
        if len(h) >= W:
            win = np.lib.stride_tricks.sliding_window_view(h, W)[::step]
            pos = np.arange(0, len(h) - W + 1, step) + win.argmin(axis=1)
            km.append(a[pos, 0])
            ix.append(pos + 1)
            hh.append(h[pos])
        off.append(off[-1] + (len(h) - W) // step + 1 if len(h) >= W else off[-1])
    cat = lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt)  # noqa: E731
    return cat(km, np.uint64), cat(ix, np.int64), cat(hh, np.uint64), np.array(off, dtype=np.uint64)


MIN_PLAN = plan(FULL_LAYOUTS, OTHER_LAYOUTS, (5, 25, 32), (25,))


@pytest.mark.parametrize("layout,k", MIN_PLAN)
def test_minimizers(kc, ctx, layout, k):
    for i in each(layout, k):
        drs = device_set(layout, k, i)
        for mode in MODES:
            st = stream(layout, k, i, mode)
            for W in sorted({1, 10, 31, 32, 65 - k}):
                for step in (1, 3):
                    km, ix, hh, so = kc.minimizers(drs, k, W, step, canonical=mode == CANON, hash=True, ctx=ctx)
                    ekm, eix, ehh, eoff = minimizer_reference(st, W, step)
                    what = (cases(layout, k)[i].name, mode, W, step)
                    assert np.array_equal(km, ekm) and np.array_equal(ix, eix) and np.array_equal(hh, ehh), what
                    assert np.array_equal(so, eoff), what


@pytest.mark.parametrize("layout", ["U0", "U4", "R0", "S1"])
def test_minimizers_abi_index_base_and_offsets(kc, ctx, layout):
    """index_base is added to every index; outputs 8 bytes past an aligned base (scalar stores) and 16 bytes past it (the
    dense kernel's two-word stores)."""
    from kmerscuda import _abi
    k, W = 25, 10
    drs = device_set(layout, k, 0)
    st = stream(layout, k, 0, FW)
    ekm, eix, ehh, eoff = minimizer_reference(st, W, 1)
    n = len(ekm)
    bufs = [ctx.alloc(8 * (n + 4)) for _ in range(3)]
    try:
        for shift in (8, 16):
            out = _abi.kmc_out(bufs[0].ptr + shift, None, bufs[1].ptr + shift, bufs[2].ptr + shift, None, n, 1000)
            res = _abi.kmc_result()
            ctx._check(ctx.lib.kmc_minimizers(ctx.handle, C.byref(drs.desc), k, W, 1, FW, _abi.KMC_HASH_FX, C.byref(out), C.byref(res)))
            assert res.n_written == n
            assert np.array_equal(bufs[0].download(np.uint64, n, shift), ekm)
            assert np.array_equal(bufs[1].download(np.uint64, n, shift), ehh)
            assert np.array_equal(bufs[2].download(np.int64, n, shift), eix + 1000)
    finally:
        for b in bufs:
            b.free()


# ------------------------------------------------------------------------- R1: overlapping views of one long sequence
R1_SEQS, R1_LEN = 1000, 100_000


@pytest.fixture(scope="module")
def r1(kc):
    rng = np.random.default_rng(1001)
    words = _rand_words(rng, R1_LEN // 32)
    # the tiles of one-limb windows against the planner's bound for sets that do not overlap (tiles_upper_bound, plan.h)
    assert R1_SEQS * (R1_LEN // 8) // TILE_ITEMS > 100 * ((32 * words.size + 2 * R1_SEQS) // TILE_ITEMS + 2)
    rs = kc.ReadSet(2, words, R1_SEQS, seq_word_offset=np.zeros(R1_SEQS, np.uint64), seq_len=np.full(R1_SEQS, R1_LEN, np.uint64))
    return rs, {(k, m): Stream([(words, R1_LEN, 0)], k, m) for k in (12, 25, 61) for m in MODES}


@pytest.fixture
def fresh(kc):
    """A context of its own: its scratch window has not grown in earlier calls."""
    c = kc.Context(0)
    yield c
    c.close()


def test_overlapping_views_count_and_sketches(kc, fresh, r1):
    """1000 ragged views, all at word 0 of one 100 kbp buffer: about 6100 tiles of windows over a buffer of 3125 words."""
    rs, ref = r1
    drs = kc.DeviceReadSet(fresh, rs)
    for k in (25, 61):
        for mode in MODES:
            st = ref[(k, mode)]
            n = C.c_uint64(0)
            fresh._check(fresh.lib.kmc_count(fresh.handle, C.byref(drs.desc), k, mode, C.byref(n)))
            assert n.value == R1_SEQS * st.total
            u = np.unique(st.h)
            assert np.array_equal(kc.minhash_sketch(drs, k, 1000, canonical=mode == CANON, ctx=fresh), u[:1000])
            rows, lens = kc.minhash_sketches(drs, k, 64, canonical=mode == CANON, ctx=fresh)
            assert np.all(lens == 64) and np.array_equal(rows, np.tile(u[:64], (R1_SEQS, 1)))


@pytest.mark.parametrize("k", [25, 61])
def test_overlapping_views_tables(kc, fresh, r1, k):
    rs, ref = r1
    drs = kc.DeviceReadSet(fresh, rs)
    for mode in table_modes(k):
        st = ref[(k, mode)]
        u, inv, c = st.table
        t = kc.KmerTable(direct_capacity(st), ctx=fresh, n_limbs=1 if k <= 32 else 2)
        try:
            n, _ = t.count(drs, k, canonical=mode == CANON)
            assert n == R1_SEQS * st.total and t.n_keys == len(c)
            keys, vals = t.items()
            assert np.array_equal(keys, u) and np.array_equal(vals, R1_SEQS * c)
            got = t.lookup(drs, k, canonical=mode == CANON).reshape(R1_SEQS, st.total)
            assert np.all(got == (R1_SEQS * c)[inv][None, :])
        finally:
            t.free()


def test_overlapping_views_composition_and_buckets(kc, fresh, r1):
    rs, ref = r1
    drs = kc.DeviceReadSet(fresh, rs)
    for mode in MODES:
        st = ref[(12, mode)]
        table, n, _ = kc.composition(drs, 12, canonical=mode == CANON, ctx=fresh)
        u, c = np.unique(st.a[:, 0], return_counts=True)
        nz = np.flatnonzero(table)
        assert n == R1_SEQS * st.total and np.array_equal(nz, u) and np.array_equal(table[nz], R1_SEQS * c)
    for k in (25, 61):
        st = ref[(k, CANON)]
        for bits in (12, 26):
            table, n, _ = kc.bucket_count(drs, k, bits, ctx=fresh)
            u, c = np.unique(st.h >> np.uint64(64 - bits), return_counts=True)
            nz = np.flatnonzero(table)
            assert n == R1_SEQS * st.total and np.array_equal(nz, u) and np.array_equal(table[nz], R1_SEQS * c)


def test_overlapping_views_minimizers(kc, fresh, r1):
    rs, ref = r1
    drs = kc.DeviceReadSet(fresh, rs)
    for mode in MODES:
        st = ref[(25, mode)]
        ekm, eix, ehh, eoff = minimizer_reference(st, 31, 101)
        km, ix, hh, so = kc.minimizers(drs, 25, 31, 101, canonical=mode == CANON, hash=True, ctx=fresh)
        m = len(ekm)
        assert np.array_equal(so, np.arange(R1_SEQS + 1, dtype=np.uint64) * np.uint64(m))
        assert np.array_equal(km, np.tile(ekm, R1_SEQS)) and np.array_equal(ix, np.tile(eix, R1_SEQS))
        assert np.array_equal(hh, np.tile(ehh, R1_SEQS))


def test_overlapping_views_fourbit_unambiguous(kc, fresh):
    """UnambiguousKmers over a 4-bit source whose views overlap: compact_kernel's look-back descriptors (tile_state), one
    per tile of windows, outnumber the tiles of the buffer."""
    from kmerscuda import _abi
    rng = np.random.default_rng(4004)
    n_seqs, length, k = 400, 20_000, 21
    codes = rng.choice(np.array([1, 2, 4, 8], dtype=np.uint64), size=length)
    codes[rng.random(length) < 0.002] = 15  # N
    import kmertools as kt
    words = kt.pack_codes(codes, 4)
    rs = kc.ReadSet(4, words, n_seqs, seq_word_offset=np.zeros(n_seqs, np.uint64), seq_len=np.full(n_seqs, length, np.uint64))
    km1, pos1 = ko.unambiguous(words, length, k, src_bits=4)
    drs = kc.DeviceReadSet(fresh, rs)
    n = C.c_uint64(0)
    fresh._check(fresh.lib.kmc_count(fresh.handle, C.byref(drs.desc), k, _abi.KMC_UNAMBIG, C.byref(n)))
    assert n.value == n_seqs * len(pos1)
    e = kc.extract(_abi.KMC_UNAMBIG, drs, k, ctx=fresh)
    assert e.n == n_seqs * len(pos1)
    assert np.array_equal(e.kmers.reshape(n_seqs, -1), np.tile(km1[:, 0], (n_seqs, 1)))
    assert np.array_equal(e.index.reshape(n_seqs, -1), np.tile(pos1, (n_seqs, 1)))
    # the count pass lays windows out in groups of 32: 6000 views of 1 Mbp need about 92,000 tiles of it, against a
    # bound of about 250 for a buffer of 1 Mbp
    n_seqs, length = 6000, 1_000_000
    codes = rng.choice(np.array([1, 2, 4, 8], dtype=np.uint64), size=length)
    codes[rng.random(length) < 0.002] = 15
    words = kt.pack_codes(codes, 4)
    rs = kc.ReadSet(4, words, n_seqs, seq_word_offset=np.zeros(n_seqs, np.uint64), seq_len=np.full(n_seqs, length, np.uint64))
    _, pos1 = ko.unambiguous(words, length, k, src_bits=4)
    drs = kc.DeviceReadSet(fresh, rs)
    fresh._check(fresh.lib.kmc_count(fresh.handle, C.byref(drs.desc), k, _abi.KMC_UNAMBIG, C.byref(n)))
    assert n.value == n_seqs * len(pos1)


# ------------------------------------------------------------------------------------------- sources they refuse
def test_consumers_refuse_fourbit_and_ascii_sources(kc, ctx):
    four = kc.ReadSet.single(kc.LongDNA4("ACGTNACGTA" * 20))
    ascii_ = kc.ReadSet.from_strings(["ACGTACGTAC" * 20, "ACGT" * 30])
    for rs in (four, ascii_):
        drs = kc.DeviceReadSet(ctx, rs)
        calls = [
            lambda: kc.minhash_sketch(drs, 21, 10, ctx=ctx),
            lambda: kc.minhash_sketches(drs, 21, 10, ctx=ctx),
            lambda: kc.composition(drs, 5, ctx=ctx),
            lambda: kc.KmerTable(10, ctx=ctx).count(drs, 21),
            lambda: kc.KmerTable(10, ctx=ctx, n_limbs=2).count(drs, 41),
            lambda: kc.KmerTable(10, ctx=ctx).lookup(drs, 21),
            lambda: kc.KmerTable(10, ctx=ctx, n_limbs=2).lookup(drs, 41),
            lambda: kc.bucket_count(drs, 21, 12, ctx=ctx),
            lambda: kc.minimizers(drs, 21, 10, ctx=ctx),
        ]
        for call in calls:
            with pytest.raises(kc.KmersCUDAError, match=r"status 6:"):
                call()


# ------------------------------------------------------------------------------- the general path on aligned sets
def test_general_path_on_aligned_sets():
    """KMC_ALIGNED_KERNEL=0 (read once per process) sends the aligned sets through the general tile cursor: this file
    once more in a process of its own."""
    if os.environ.get("KMC_ALIGNED_KERNEL") == "0":
        pytest.skip("already running with KMC_ALIGNED_KERNEL=0")
    env = dict(os.environ, KMC_ALIGNED_KERNEL="0")
    r = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", "-p", "no:cacheprovider", os.path.abspath(__file__),
                        "-k", "not overlapping and not general_path and not refuse"],
                       env=env, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
