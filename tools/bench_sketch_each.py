#!/usr/bin/env python
"""Device time of the per-sequence MinHash sketches (kmc_minhash_sketch_each) and of the all-pairs comparison
(kmc_minhash_compare), in one command:

  * collection: 1000 ragged random sequences of 0.5-2 Mbp (about 1.25 Gbp, beyond L2), canonical 21-mers, s = 1000.
    Three ways alternate step by step after warm-up: kmc_minhash_sketch_each; a loop of kmc_minhash_sketch over the
    same device buffer, one sequence per call; kmc_minhash_sketch of the whole set.  Rates are windows over the span
    of the call(s), cudaEvents on the context's stream.  The rows of the batched call are checked against the loop's.
  * read set: 4 M x 150 bp, s = 1000 (every window is a candidate: this measures the segmented sort); the temporary
    memory is the growth of the context's memory pool over the call.
  * all pairs: 4096 sketches of s = 1000, A against itself.  Pairs/s and element probes/s, probes = sum over pairs of
    n_B * ceil(log2(n_A + 1)), and the kernel's share of the shared-memory probe bound: one 8-byte load per probe,
    128 bytes per clock per SM at the card's maximum SM clock.  A seeded sample of pairs is checked against numpy.

One JSON line per case, then the GPU's name, power limit and maximum SM clock (read in the same command).

  python tools/bench_sketch_each.py [--steps 5] [--warmup 2] [--out profiles/r09_sketch_each.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "kmers.jl_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import kmerscuda as kc  # noqa: E402
from kmerscuda import _abi  # noqa: E402
from oracle import oracle as ko  # noqa: E402
import sketch_reference as ref  # noqa: E402

K, S = 21, 1000


def check(ctx, st):
    if st != 0:
        raise RuntimeError(ctx.lib.kmc_last_error(ctx.handle).decode())


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": power, "clocks_max_sm": clock}


def span_ms(ctx, fn):
    ctx.timer_begin()
    fn()
    return ctx.timer_end()


def collection(ctx, steps, warmup, rows_out):
    rng = np.random.default_rng(9)
    lens = rng.integers(500_000, 2_000_001, size=1000).astype(np.uint64)
    nw = (lens + 31) // 32
    off = np.zeros(len(lens) + 1, dtype=np.uint64)
    off[1:] = np.cumsum(nw)
    words = rng.integers(0, 2**64, size=int(off[-1]), dtype=np.uint64)
    rs = kc.ReadSet(2, words, len(lens), seq_word_offset=off[:-1].copy(), seq_len=lens)
    drs = kc.DeviceReadSet(ctx, rs)
    n = len(lens)
    windows = int((lens - K + 1).sum())
    d_each, d_n = ctx.alloc(n * S * 8), ctx.alloc(n * 4)
    d_loop, d_one = ctx.alloc(n * S * 8), ctx.alloc(S * 8)
    loop_n = np.zeros(n, dtype=np.uint32)
    singles = [_abi.kmc_seqs(drs.words.ptr + int(off[i]) * 8, int(nw[i]), 1, None, None, int(lens[i]), int(nw[i]), 2, 0)
               for i in range(n)]
    res = _abi.kmc_result()
    lib, h = ctx.lib, ctx.handle

    def each():
        check(ctx, lib.kmc_minhash_sketch_each(h, C.byref(drs.desc), K, _abi.KMC_CANON, S, d_each.ptr, d_n.ptr, C.byref(res)))

    def loop():
        for i in range(n):
            check(ctx, lib.kmc_minhash_sketch(h, C.byref(singles[i]), K, _abi.KMC_CANON, S, d_loop.ptr + i * S * 8, C.byref(res)))
            loop_n[i] = res.n_written

    def whole():
        check(ctx, lib.kmc_minhash_sketch(h, C.byref(drs.desc), K, _abi.KMC_CANON, S, d_one.ptr, C.byref(res)))

    cases = {"sketch_each": each, "sketch_loop": loop, "sketch_whole_set": whole}
    for _ in range(warmup):
        for fn in cases.values():
            fn()
    ms = {name: [] for name in cases}
    for _ in range(steps):
        for name, fn in cases.items():
            ms[name].append(span_ms(ctx, fn))
    each()
    got = d_each.download(np.uint64, n * S).reshape(n, S)
    got_n = d_n.download(np.uint32, n)
    want = d_loop.download(np.uint64, n * S).reshape(n, S)
    ok = bool(np.array_equal(got_n, loop_n) and all(np.array_equal(got[i, : got_n[i]], want[i, : loop_n[i]]) for i in range(n))
              and np.all(got_n == S))
    for name in cases:
        med = float(np.median(ms[name]))
        rows_out.append({"case": "collection", "call": name, "n_seqs": n, "bp": int(lens.sum()), "windows": windows, "s": S, "k": K,
                         "ms_median": med, "ms_min": float(np.min(ms[name])), "gkmers_per_s": windows / (med / 1e3) / 1e9,
                         "rows_equal_loop": ok})
    for d in (d_each, d_n, d_loop, d_one):
        d.free()
    del drs


def read_set(ctx, steps, warmup, rows_out):
    rng = np.random.default_rng(10)
    n_reads, length, stride = 4_000_000, 150, 5
    words = rng.integers(0, 2**64, size=n_reads * stride, dtype=np.uint64)
    rs = kc.ReadSet(2, words, n_reads, uniform_len=length, uniform_stride_words=stride)
    drs = kc.DeviceReadSet(ctx, rs)
    windows = n_reads * (length - K + 1)
    d_rows, d_n = ctx.alloc(n_reads * S * 8), ctx.alloc(n_reads * 4)
    res = _abi.kmc_result()

    def each():
        check(ctx, ctx.lib.kmc_minhash_sketch_each(ctx.handle, C.byref(drs.desc), K, _abi.KMC_CANON, S, d_rows.ptr, d_n.ptr,
                                                   C.byref(res)))

    ctx.trim()
    free0 = torch.cuda.mem_get_info(0)[0]
    each()
    temp = free0 - torch.cuda.mem_get_info(0)[0]
    for _ in range(warmup):
        each()
    ms = [span_ms(ctx, each) for _ in range(steps)]
    lens = d_n.download(np.uint32, n_reads)
    sample = rng.choice(n_reads, size=200, replace=False)
    ok = True
    for i in sample:
        row = d_rows.download(np.uint64, S, offset_bytes=int(i) * S * 8)
        want = ko.minhash_sketch(words[i * stride:(i + 1) * stride], length, K, S, True)
        ok &= bool(lens[i] == len(want) and np.array_equal(row[: lens[i]], want) and np.all(row[lens[i]:] == ~np.uint64(0)))
    med = float(np.median(ms))
    rows_out.append({"case": "read_set", "call": "sketch_each", "n_seqs": n_reads, "windows": windows, "s": S, "k": K,
                     "ms_median": med, "ms_min": float(np.min(ms)), "gkmers_per_s": windows / (med / 1e3) / 1e9,
                     "temp_bytes": int(temp), "temp_bytes_per_window": temp / windows, "out_bytes": n_reads * S * 8,
                     "sampled_rows_equal_oracle": ok})
    for d in (d_rows, d_n):
        d.free()
    ctx.trim()
    del drs


def all_pairs(ctx, steps, warmup, rows_out, info):
    rng = np.random.default_rng(11)
    n = 4096
    pool = rng.integers(0, 2**64, size=4096, dtype=np.uint64)
    rows = np.empty((n, S), dtype=np.uint64)
    for i in range(n):  # 300 values from a shared pool (overlaps between rows), 700 of the row's own
        v = np.concatenate([rng.choice(pool, size=300, replace=False), rng.integers(0, 2**64, size=S - 300, dtype=np.uint64)])
        v = np.unique(v)
        assert len(v) == S
        rows[i] = v
    lens = np.full(n, S, dtype=np.uint32)
    da, dn = ctx.to_device(rows), ctx.to_device(lens)
    d_sh, d_bt = ctx.alloc(n * n * 4), ctx.alloc(n * n * 4)

    def cmp():
        check(ctx, ctx.lib.kmc_minhash_compare(ctx.handle, da.ptr, dn.ptr, n, da.ptr, dn.ptr, n, S, d_sh.ptr, d_bt.ptr))

    for _ in range(warmup):
        cmp()
    launches = 10
    ms = []
    for _ in range(steps):
        ctx.timer_begin()
        for _ in range(launches):
            cmp()
        ms.append(ctx.timer_end() / launches)
    shared = d_sh.download(np.uint32, n * n).reshape(n, n)
    bottom = d_bt.download(np.uint32, n * n).reshape(n, n)
    ok = bool(np.array_equal(np.diag(shared), lens) and np.array_equal(shared, shared.T))
    for _ in range(300):
        i, j = rng.integers(0, n, size=2)
        w = ref.minhash_compare(rows[i:i + 1], lens[i:i + 1], rows[j:j + 1], lens[j:j + 1], S)
        ok &= bool(shared[i, j] == w[0][0, 0] and bottom[i, j] == w[1][0, 0])
    med = float(np.median(ms))
    probes = float(lens.astype(np.float64).sum()) * float(np.ceil(np.log2(lens.astype(np.float64) + 1)).sum())
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    clock_hz = float(info["clocks_max_sm"].split()[0]) * 1e6
    bound_s = probes * 8 / (128.0 * sm * clock_hz)
    rows_out.append({"case": "all_pairs", "call": "minhash_compare", "n_a": n, "n_b": n, "s": S, "ms_median": med,
                     "ms_min": float(np.min(ms)), "pairs_per_s": n * n / (med / 1e3), "probes": probes,
                     "probes_per_s": probes / (med / 1e3), "smem_probe_bound_ms": bound_s * 1e3,
                     "share_of_smem_probe_bound": bound_s / (med / 1e3), "sm_count": sm, "sampled_pairs_equal_numpy": ok})
    for d in (da, dn, d_sh, d_bt):
        d.free()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_sketch_each.jsonl"))
    ap.add_argument("--cases", default="collection,read_set,all_pairs")
    a = ap.parse_args()
    info = gpu_info()
    ctx = kc.default_context(0)
    rows = []
    cases = a.cases.split(",")
    if "collection" in cases:
        collection(ctx, a.steps, a.warmup, rows)
    if "read_set" in cases:
        read_set(ctx, a.steps, a.warmup, rows)
    if "all_pairs" in cases:
        all_pairs(ctx, a.steps, a.warmup, rows, info)
    rows.append(info)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for r in rows:
            line = json.dumps(r)
            print(line)
            f.write(line + "\n")


if __name__ == "__main__":
    main()
