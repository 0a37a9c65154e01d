#!/usr/bin/env python
"""Device-resident timings of the BASELINE.json configs other than the headline one (C2 is
bench.py): C3 UnambiguousDNAMers{31} over 4-bit reads / one long sequence with 1 % N,
C4 CanonicalDNAMers{63} over 1 Gbp, C5 canonical 31-mer bucket-count table (per-GPU part), plus
the other iterator modes on the C2 shape.  One JSON line per case: k-mers/s, algorithmic GB/s
(SURVEY.md 8d) and the fraction of the measured HBM peak.  Inputs are generated on the device with
torch (plumbing); every timed call goes through the C ABI.

  python tools/bench_configs.py [--cases c3,c4,c5,modes] [--steps 10] [--scale 1.0]
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "kmers.jl_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import kmerscuda as kc  # noqa: E402
from kmerscuda import _abi  # noqa: E402

FW, FWRV, CANON, UNAMBIG = 0, 1, 2, 3


def peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        return 6650.0


WARMUP = 3


def timed(ctx, fn, steps, warmup=None):
    for _ in range(WARMUP if warmup is None else warmup):
        fn()
    ctx.sync()
    ms = []
    for _ in range(steps):
        ctx.timer_begin()
        fn()
        ms.append(ctx.timer_end())
    return float(np.median(ms)), float(np.min(ms))


def rand_words_2bit(n_words, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randint(-2**63, 2**63 - 1, (n_words,), dtype=torch.int64, device="cuda", generator=g)


def rand_words_4bit(n_rows, syms_per_row, valid_len, seed, p_n=0.01, chunk_rows=1_000_000):
    """n_rows x (syms_per_row/16) words; symbols beyond valid_len are gap (0)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    wpr = syms_per_row // 16
    out = torch.empty(n_rows * wpr, dtype=torch.int64, device="cuda")
    shifts = torch.arange(16, device="cuda", dtype=torch.int64) * 4
    for r0 in range(0, n_rows, chunk_rows):
        r1 = min(n_rows, r0 + chunk_rows)
        base = torch.randint(0, 4, (r1 - r0, syms_per_row), dtype=torch.int64, device="cuda", generator=g)
        nib = torch.ones_like(base) << base
        nib[torch.rand(nib.shape, device="cuda", generator=g) < p_n] = 15
        nib[:, valid_len:] = 0
        out[r0 * wpr:r1 * wpr] = (nib.view(r1 - r0, wpr, 16) << shifts).sum(dim=2).reshape(-1)
    return out


def emit(name, n_kmers, bytes_total, ms_med, ms_min, extra=None):
    pk = peak()
    gbs = bytes_total / (ms_med / 1e3) / 1e9
    line = {"case": name, "kmers": n_kmers, "kmers_per_s": n_kmers / (ms_med / 1e3), "ms_median": ms_med, "ms_min": ms_min,
            "algorithmic_bytes": bytes_total, "achieved_GBps": gbs, "peak_GBps": pk, "frac_of_measured_peak": gbs / pk}
    if extra:
        line.update(extra)
    print(json.dumps(line), flush=True)


def run_extract(ctx, desc, k, mode, flags, out, res):
    st = ctx.lib.kmc_extract(ctx.handle, C.byref(desc), k, mode, flags, C.byref(out), C.byref(res))
    if st != 0:
        raise RuntimeError(ctx.lib.kmc_last_error(ctx.handle).decode())


def case_c3_reads(ctx, steps, scale):
    n_reads, length, stride, k = int(10_000_000 * scale), 150, 10, 31
    wpr = length - k + 1
    words = rand_words_4bit(n_reads, stride * 16, length, 439824)
    cap = n_reads * wpr
    km = torch.empty(cap, dtype=torch.int64, device="cuda")
    idx = torch.empty(cap, dtype=torch.int64, device="cuda")
    desc = _abi.kmc_seqs(words.data_ptr(), words.numel(), n_reads, None, None, length, stride, 4, 0)
    out = _abi.kmc_out(km.data_ptr(), None, None, idx.data_ptr(), None, cap, 0)
    res = _abi.kmc_result()
    torch.cuda.synchronize()
    med, mn = timed(ctx, lambda: run_extract(ctx, desc, k, UNAMBIG, 0, out, res), steps)
    n = int(res.n_written)
    emit("C3i UnambiguousDNAMers{31}, 4-bit, 1%% N, %d x 150 bp reads (SoA kmer+index)" % n_reads, n,
         0.5 * n_reads * length + 16 * n, med, mn, {"windows": cap, "survivors_frac": n / cap})
    km2 = torch.empty(2 * cap, dtype=torch.int64, device="cuda")
    out = _abi.kmc_out(km2.data_ptr(), None, None, None, None, cap, 0)
    med, mn = timed(ctx, lambda: run_extract(ctx, desc, k, UNAMBIG, _abi.KMC_AOS, out, res), steps)
    emit("C3i same, AoS Vector{Tuple{Kmer,Int}}", n, 0.5 * n_reads * length + 16 * n, med, mn)


def case_c3_long(ctx, steps, scale):
    length, k = int(1_000_000_000 * scale), 31
    nw = (length + 15) // 16
    rows = 1024
    per = (nw + rows - 1) // rows
    words = rand_words_4bit(rows, per * 16, per * 16, 7, chunk_rows=32)[:nw].contiguous()
    cap = length - k + 1
    km = torch.empty(cap, dtype=torch.int64, device="cuda")
    idx = torch.empty(cap, dtype=torch.int64, device="cuda")
    desc = _abi.kmc_seqs(words.data_ptr(), words.numel(), 1, None, None, length, words.numel(), 4, 0)
    out = _abi.kmc_out(km.data_ptr(), None, None, idx.data_ptr(), None, cap, 0)
    res = _abi.kmc_result()
    torch.cuda.synchronize()
    med, mn = timed(ctx, lambda: run_extract(ctx, desc, k, UNAMBIG, 0, out, res), steps)
    n = int(res.n_written)
    emit("C3ii UnambiguousDNAMers{31}, 4-bit, 1%% N, one %d bp sequence" % length, n, 0.5 * length + 16 * n, med, mn,
         {"windows": cap, "survivors_frac": n / cap})


def case_c4(ctx, steps, scale):
    length, k = int(1_000_000_000 * scale), 63
    words = rand_words_2bit((length + 31) // 32, 11)
    cap = length - k + 1
    km = torch.empty(2 * cap, dtype=torch.int64, device="cuda")
    desc = _abi.kmc_seqs(words.data_ptr(), words.numel(), 1, None, None, length, words.numel(), 2, 0)
    out = _abi.kmc_out(km.data_ptr(), None, None, None, None, cap, 0)
    res = _abi.kmc_result()
    torch.cuda.synchronize()
    med, mn = timed(ctx, lambda: run_extract(ctx, desc, k, CANON, _abi.KMC_NO_SYNC, out, res), steps)
    emit("C4 CanonicalDNAMers{63} (2 limbs), one %d bp 2-bit sequence" % length, cap, (0.25 + 16) * cap, med, mn)
    hs = torch.empty(cap, dtype=torch.int64, device="cuda")
    out = _abi.kmc_out(km.data_ptr(), None, hs.data_ptr(), None, None, cap, 0)
    med, mn = timed(ctx, lambda: run_extract(ctx, desc, k, CANON, _abi.KMC_NO_SYNC | _abi.KMC_HASH_FX, out, res), steps)
    emit("C4 same + fx_hash", cap, (0.25 + 24) * cap, med, mn)


def case_c5(ctx, steps, scale):
    """K = 31 at B = 20 and 24 (direct increments) and 28 (fused bins); K = 63 at B = 28 (two limbs: the exact binned path)."""
    n_reads, length, stride = int(25_000_000 * scale), 150, 5
    words = rand_words_2bit(n_reads * stride, 13)
    words.view(n_reads, stride)[:, stride - 1] &= (1 << (2 * (length - 32 * (stride - 1)))) - 1
    desc = _abi.kmc_seqs(words.data_ptr(), words.numel(), n_reads, None, None, length, stride, 2, 0)
    res = _abi.kmc_result()
    for k, bits in ((31, 20), (31, 24), (31, 28), (63, 28)):
        wpr = length - k + 1
        table = torch.zeros(1 << bits, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()

        def step():
            st = ctx.lib.kmc_bucket_count(ctx.handle, C.byref(desc), k, bits, table.data_ptr(), C.byref(res))
            if st != 0:
                raise RuntimeError(ctx.lib.kmc_last_error(ctx.handle).decode())
        med, mn = timed(ctx, step, steps)
        n = n_reads * wpr
        emit("C5 (per-GPU part) canonical %d-mer bucket table, B=%d, %d x 150 bp reads" % (k, bits, n_reads), n,
             (0.25 * length / wpr + 8) * n, med, mn, {"table_bytes": 4 << bits})
        del table


def case_modes(ctx, steps, scale):
    n_reads, length, stride, k = int(10_000_000 * scale), 150, 5, 31
    wpr = length - k + 1
    n = n_reads * wpr
    words = rand_words_2bit(n_reads * stride, 439824)
    desc = _abi.kmc_seqs(words.data_ptr(), words.numel(), n_reads, None, None, length, stride, 2, 0)
    a = torch.empty(2 * n, dtype=torch.int64, device="cuda")
    b = torch.empty(n, dtype=torch.int64, device="cuda")
    res = _abi.kmc_result()
    inb = 0.25 * length / wpr
    cases = [("FwDNAMers{31}", FW, 0, _abi.kmc_out(a.data_ptr(), None, None, None, None, n, 0), inb + 8),
             ("FwRvIterator{31} SoA", FWRV, 0, _abi.kmc_out(a.data_ptr(), b.data_ptr(), None, None, None, n, 0), inb + 16),
             ("FwRvIterator{31} AoS Tuple{Kmer,Kmer}", FWRV, _abi.KMC_AOS, _abi.kmc_out(a.data_ptr(), None, None, None, None, n, 0), inb + 16),
             ("CanonicalDNAMers{31} (no hash)", CANON, 0, _abi.kmc_out(a.data_ptr(), None, None, None, None, n, 0), inb + 8),
             ("UnambiguousDNAMers{31} over 2-bit (kmer + index)", UNAMBIG, 0, _abi.kmc_out(a.data_ptr(), None, None, b.data_ptr(), None, n, 0), inb + 16)]
    for name, mode, fl, out, bpk in cases:
        med, mn = timed(ctx, lambda: run_extract(ctx, desc, k, mode, fl | _abi.KMC_NO_SYNC, out, res), steps)
        emit("C2-shape %s, %d x 150 bp" % (name, n_reads), n, bpk * n, med, mn)


def case_ragged(ctx, steps, scale):
    """C2 workload through the ragged (CSR) descriptors: (a) all reads 150 bp, (b) lengths uniform in [100, 250]."""
    n_reads, k = int(10_000_000 * scale), 31
    g = torch.Generator(device="cuda").manual_seed(5)
    for name, lens in (("all 150 bp", torch.full((n_reads,), 150, dtype=torch.int64, device="cuda")),
                       ("lengths U[100,250]", torch.randint(100, 251, (n_reads,), dtype=torch.int64, device="cuda", generator=g))):
        nw = (lens + 31) // 32
        off = torch.zeros(n_reads + 1, dtype=torch.int64, device="cuda")
        off[1:] = torch.cumsum(nw, 0)
        words = rand_words_2bit(int(off[-1]) + 1, 439824)
        n = int((lens - k + 1).clamp(min=0).sum())
        a = torch.empty(n, dtype=torch.int64, device="cuda")
        h = torch.empty(n, dtype=torch.int64, device="cuda")
        desc = _abi.kmc_seqs(words.data_ptr(), words.numel(), n_reads, off.data_ptr(), lens.data_ptr(), 0, 0, 2, 0)
        out = _abi.kmc_out(a.data_ptr(), None, h.data_ptr(), None, None, n, 0)
        res = _abi.kmc_result()
        torch.cuda.synchronize()
        med, mn = timed(ctx, lambda: run_extract(ctx, desc, k, CANON, _abi.KMC_HASH_FX, out, res), steps)
        sym = int(lens.sum())
        emit("ragged CSR CanonicalDNAMers{31}+fx_hash, %d reads, %s (incl. layout scans)" % (n_reads, name), n,
             0.25 * sym + 16 * n, med, mn)
        del words, a, h


def case_ascii(ctx, steps, scale):
    """C2 workload from ASCII bytes (what a FASTQ parser hands over): 150 bytes per read, recoded on the device."""
    n_reads, length, k = int(10_000_000 * scale), 150, 31
    wpr = length - k + 1
    n = n_reads * wpr
    g = torch.Generator(device="cuda").manual_seed(3)
    lut = torch.tensor([65, 67, 71, 84], dtype=torch.uint8, device="cuda")
    data = lut[torch.randint(0, 4, (n_reads * length,), device="cuda", generator=g)]
    a = torch.empty(n, dtype=torch.int64, device="cuda")
    h = torch.empty(n, dtype=torch.int64, device="cuda")
    desc = _abi.kmc_seqs(data.data_ptr(), data.numel(), n_reads, None, None, length, length, 8, 0)
    out = _abi.kmc_out(a.data_ptr(), None, h.data_ptr(), None, None, n, 0)
    res = _abi.kmc_result()
    torch.cuda.synchronize()
    med, mn = timed(ctx, lambda: run_extract(ctx, desc, k, CANON, _abi.KMC_HASH_FX, out, res), steps)
    emit("ASCII source: CanonicalDNAMers{31}+fx_hash, %d x 150-byte reads (strict, recoded on device)" % n_reads, n,
         1.0 * n_reads * length + 16 * n, med, mn)
    data[torch.rand(data.numel(), device="cuda", generator=g) < 0.01] = 78  # 'N'
    idx = torch.empty(n, dtype=torch.int64, device="cuda")
    out = _abi.kmc_out(a.data_ptr(), None, None, idx.data_ptr(), None, n, 0)
    med, mn = timed(ctx, lambda: run_extract(ctx, desc, k, UNAMBIG, 0, out, res), steps)
    nw = int(res.n_written)
    emit("ASCII source: UnambiguousDNAMers{31}, 1%% N, %d x 150-byte reads" % n_reads, nw, 1.0 * n_reads * length + 16 * nw, med, mn)


def case_minimizers(ctx, steps, scale):
    """Minimizers over one 1 Gbp 2-bit sequence: benchmark.jl's (K=8, W=20, step 20) and dense canonical (K=31, W=10, step 1)."""
    length = int(1_000_000_000 * scale)
    words = rand_words_2bit((length + 31) // 32, 19)
    desc = _abi.kmc_seqs(words.data_ptr(), words.numel(), 1, None, None, length, words.numel(), 2, 0)
    res = _abi.kmc_result()
    for k, w, step, mode, name in ((8, 20, 20, FW, "forward, non-overlapping windows (test/benchmark.jl:96-119)"),
                                   (31, 10, 1, CANON, "canonical, every window start")):
        n = (length - (k + w - 1)) // step + 1
        a = torch.empty(n, dtype=torch.int64, device="cuda")
        idx = torch.empty(n, dtype=torch.int64, device="cuda")
        out = _abi.kmc_out(a.data_ptr(), None, None, idx.data_ptr(), None, n, 0)
        torch.cuda.synchronize()

        def stepf():
            st = ctx.lib.kmc_minimizers(ctx.handle, C.byref(desc), k, w, step, mode, 0, C.byref(out), C.byref(res))
            if st != 0:
                raise RuntimeError(ctx.lib.kmc_last_error(ctx.handle).decode())
        med, mn = timed(ctx, stepf, steps)
        emit("minimizers K=%d W=%d step=%d, %s, one %d bp sequence" % (k, w, step, name, length), n,
             0.25 * length + 16 * n, med, mn, {"kmers_ordered_per_s": n * w / (med / 1e3)})
        del a, idx


def case_kmer4(ctx, steps, scale):
    """k-mers over the 4-bit alphabet on the C2 shape: CanonicalKmers{DNAAlphabet{4},31} (2 limbs) + fx_hash from a
    4-bit source (Copyable; any IUPAC symbol) and from a 2-bit source (TwoToFour), FwKmers{DNAAlphabet{4},16} (1 limb)."""
    n_reads, length, k = int(10_000_000 * scale), 150, 31
    wpr = length - k + 1
    n = n_reads * wpr
    a = torch.empty(2 * n, dtype=torch.int64, device="cuda")
    h = torch.empty(n, dtype=torch.int64, device="cuda")
    res = _abi.kmc_result()
    w4 = rand_words_2bit(n_reads * 10, 7)   # random nibbles: every IUPAC symbol
    w2 = rand_words_2bit(n_reads * 5, 8)
    fl = _abi.KMC_KMER4 | _abi.KMC_NO_SYNC
    out = _abi.kmc_out(a.data_ptr(), None, h.data_ptr(), None, None, n, 0)
    d4 = _abi.kmc_seqs(w4.data_ptr(), w4.numel(), n_reads, None, None, length, 10, 4, 0)
    d2 = _abi.kmc_seqs(w2.data_ptr(), w2.numel(), n_reads, None, None, length, 5, 2, 0)
    med, mn = timed(ctx, lambda: run_extract(ctx, d4, k, CANON, fl | _abi.KMC_HASH_FX, out, res), steps)
    emit("C2-shape CanonicalKmers{DNAAlphabet{4},31}+fx_hash (2 limbs), 4-bit source (Copyable), %d x 150 bp" % n_reads, n,
         (0.5 * length / wpr + 24) * n, med, mn)
    med, mn = timed(ctx, lambda: run_extract(ctx, d2, k, CANON, fl | _abi.KMC_HASH_FX, out, res), steps)
    emit("C2-shape CanonicalKmers{DNAAlphabet{4},31}+fx_hash (2 limbs), 2-bit source (TwoToFour), %d x 150 bp" % n_reads, n,
         (0.25 * length / wpr + 24) * n, med, mn)
    k16 = 16
    n16 = n_reads * (length - k16 + 1)
    a16 = torch.empty(n16, dtype=torch.int64, device="cuda")
    out16 = _abi.kmc_out(a16.data_ptr(), None, None, None, None, n16, 0)
    med, mn = timed(ctx, lambda: run_extract(ctx, d4, k16, FW, fl, out16, res), steps)
    emit("C2-shape FwKmers{DNAAlphabet{4},16} (1 limb), 4-bit source, %d x 150 bp" % n_reads, n16,
         (0.5 * length / (length - k16 + 1) + 8) * n16, med, mn)


def case_sketch(ctx, steps, scale):
    """Consumers that never write the stream: the bottom-1000 MinHash sketch of the reference's example
    (docs/src/minhash.md:31-36, CanonicalDNAMers{16}) and K = 31, and the composition vector
    (docs/src/composition.md:28-39, FwDNAMers{4}) and K = 11, over one 1 Gbp 2-bit sequence.
    Algorithmic bytes: the sequence is read (twice for the sketch); the outputs are O(s) / O(4^K)."""
    length = int(1_000_000_000 * scale)
    words = rand_words_2bit((length + 31) // 32, 23)
    desc = _abi.kmc_seqs(words.data_ptr(), words.numel(), 1, None, None, length, words.numel(), 2, 0)
    res = _abi.kmc_result()
    for k in (16, 31):
        s = 1000
        out = torch.empty(s, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()

        def stepf():
            st = ctx.lib.kmc_minhash_sketch(ctx.handle, C.byref(desc), k, CANON, s, out.data_ptr(), C.byref(res))
            if st != 0:
                raise RuntimeError(ctx.lib.kmc_last_error(ctx.handle).decode())
        med, mn = timed(ctx, stepf, steps)
        emit("MinHash sketch s=1000 of CanonicalDNAMers{%d} under fx_hash, one %d bp sequence (no stream written)" % (k, length),
             length - k + 1, 2 * 0.25 * length + 8 * s, med, mn)
    for k, mode, name in ((4, FW, "FwDNAMers{4}"), (11, CANON, "CanonicalDNAMers{11}")):
        table = torch.zeros(4 ** k, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()

        def stepc():
            st = ctx.lib.kmc_composition(ctx.handle, C.byref(desc), k, mode, table.data_ptr(), C.byref(res))
            if st != 0:
                raise RuntimeError(ctx.lib.kmc_last_error(ctx.handle).decode())
        med, mn = timed(ctx, stepc, steps)
        emit("composition vector of %s, one %d bp sequence" % (name, length), length - k + 1, 0.25 * length + 4.0 * 4 ** k, med, mn)


def case_count(ctx, steps, scale):
    """Exact canonical 31-mer counts (kmc_kmer_count) over reads sampled from a genome at 30x coverage:
    4 M x 150 bp reads of a 20 Mbp genome (about 20 M distinct canonical 31-mers, each seen ~24 times), table of 2^26
    slots (768 MB: beyond L2); and over a 1 Mbp genome (table of 2^22 slots = 48 MB: L2-resident)."""
    n_reads, length, stride, k = int(4_000_000 * scale), 150, 5, 31
    wpr = length - k + 1
    res = _abi.kmc_result()
    g = torch.Generator(device="cuda").manual_seed(77)
    shifts = (torch.arange(32, device="cuda", dtype=torch.int64) * 2)
    for genome_len, log2cap in ((int(20_000_000 * scale), 26), (1_000_000, 22)):
        genome = torch.randint(0, 4, (genome_len,), dtype=torch.int64, device="cuda", generator=g)
        words = torch.empty(n_reads * stride, dtype=torch.int64, device="cuda")
        pos = torch.arange(stride * 32, device="cuda")
        for c0 in range(0, n_reads, 250_000):
            c1 = min(n_reads, c0 + 250_000)
            starts = torch.randint(0, genome_len - length, (c1 - c0, 1), device="cuda", generator=g)
            codes = genome[(starts + pos).clamp(max=genome_len - 1)] * (pos < length)
            words[c0 * stride:c1 * stride] = (codes.view(c1 - c0, stride, 32) << shifts).sum(-1).view(-1)
        desc = _abi.kmc_seqs(words.data_ptr(), words.numel(), n_reads, None, None, length, stride, 2, 0)
        keys = torch.empty(1 << log2cap, dtype=torch.int64, device="cuda")
        vals = torch.empty(1 << log2cap, dtype=torch.int32, device="cuda")
        distinct = [0]

        def stepf():
            keys.fill_(-1)
            vals.zero_()
            st = ctx.lib.kmc_kmer_count(ctx.handle, C.byref(desc), k, CANON, keys.data_ptr(), vals.data_ptr(), log2cap, C.byref(res))
            if st != 0:
                raise RuntimeError(ctx.lib.kmc_last_error(ctx.handle).decode())
            distinct[0] = int(res.digest[0])
        torch.cuda.synchronize()
        ms = []
        for i in range(WARMUP + steps):
            stepf()
            if i >= WARMUP:
                ms.append(float(res.kernel_ms))
        med, mn = float(np.median(ms)), float(np.min(ms))
        n = n_reads * wpr
        emit("exact canonical 31-mer count table, %d x 150 bp reads at 30x of a %d bp genome, 2^%d slots" % (n_reads, genome_len, log2cap),
             n, 0.25 * length / wpr * n + 12.0 * distinct[0], med, mn, {"distinct_keys": distinct[0], "table_bytes": 12 << log2cap})
        del words, keys, vals, genome


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="c3,c3long,c4,c5,modes")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    global WARMUP
    WARMUP = args.warmup
    torch.cuda.set_device(0)
    ctx = kc.Context(0)
    table = {"c3": case_c3_reads, "c3long": case_c3_long, "c4": case_c4, "c5": case_c5, "modes": case_modes, "ragged": case_ragged, "ascii": case_ascii, "minimizers": case_minimizers, "sketch": case_sketch, "kmer4": case_kmer4, "count": case_count}
    for c in args.cases.split(","):
        table[c](ctx, args.steps, args.scale)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
