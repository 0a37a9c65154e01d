#!/usr/bin/env python
"""Device time of the read-only queries of the exact k-mer tables, next to the count that fills them, in one command:

  * the per-window lookup (kmc_kmer_lookup / kmc_kmer_lookup2) of the reads the table was counted from, against the
    count of the same reads into the same table (alternating, step by step).  The reads are those of
    `tools/bench_configs.py --cases count` and `tools/bench_count2.py`: 4 M x 150 bp at 30x of a 20 Mbp genome (2^26
    slots: beyond L2, counted by the binned path, looked up by direct probes) and of a 1 Mbp genome (2^22 slots,
    L2-resident); canonical 31-mers (one limb) and 63-mers (two limbs);
  * the count spectrum (kmc_kmer_table_histogram) and the count-filtered export (kmc_kmer_table_export_range) of the
    2^26-slot tables: 12 (one limb) or 20 (two limbs) bytes read per slot, over kernel time, against the copy rate of
    a 4 GB device-to-device copy measured in the same command.

One JSON line per case, then the GPU's name and power limit.

  python tools/bench_lookup.py [--steps 5] [--warmup 2] [--scale 1.0]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "kmers.jl_b200"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import kmerscuda as kc  # noqa: E402
from kmerscuda import _abi  # noqa: E402
from bench_configs import CANON  # noqa: E402
from bench_count2 import sampled_reads  # noqa: E402


def check(ctx, st):
    if st != 0:
        raise RuntimeError(ctx.lib.kmc_last_error(ctx.handle).decode())


def copy_peak_gbs():
    """Device-to-device copy of 4 GB: (read + written bytes) / time, the best of 5."""
    n = 1 << 29
    a = torch.empty(n, dtype=torch.int64, device="cuda").fill_(1)
    b = torch.empty_like(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 0.0
    for _ in range(7):
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, 2 * 8 * n / (e0.elapsed_time(e1) / 1e3) / 1e9)
    del a, b
    return best


def timed_call(ctx, fn, steps, warmup):
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(steps):
        ctx.timer_begin()
        fn()
        ms.append(ctx.timer_end())
    return float(np.median(ms)), float(np.min(ms))


def run(ctx, steps, warmup, scale, peak):
    n_reads, length, stride = int(4_000_000 * scale), 150, 5
    g = torch.Generator(device="cuda").manual_seed(77)
    for genome_len, log2cap in ((int(20_000_000 * scale), 26), (1_000_000, 22)):
        words = sampled_reads(n_reads, length, stride, genome_len, g)
        desc = _abi.kmc_seqs(words.data_ptr(), words.numel(), n_reads, None, None, length, stride, 2, 0)
        for nl, k in ((1, 31), (2, 63)):
            wpr = length - k + 1
            n = n_reads * wpr
            slot_bytes = 8 * nl + 4
            keys = torch.empty(nl << log2cap, dtype=torch.int64, device="cuda")
            vals = torch.empty(1 << log2cap, dtype=torch.int32, device="cuda")
            out = torch.empty(n, dtype=torch.int32, device="cuda")
            count_fn = ctx.lib.kmc_kmer_count if nl == 1 else ctx.lib.kmc_kmer_count2
            lookup_fn = ctx.lib.kmc_kmer_lookup if nl == 1 else ctx.lib.kmc_kmer_lookup2
            res = _abi.kmc_result()
            count_ms, lookup_ms, distinct = [], [], 0
            for i in range(warmup + steps):
                keys.fill_(-1)
                vals.zero_()
                check(ctx, count_fn(ctx.handle, C.byref(desc), k, CANON, keys.data_ptr(), vals.data_ptr(), log2cap, C.byref(res)))
                distinct = int(res.digest[0])
                c_ms = float(res.kernel_ms)
                check(ctx, lookup_fn(ctx.handle, C.byref(desc), k, CANON, keys.data_ptr(), vals.data_ptr(), log2cap, out.data_ptr(), n,
                                     C.byref(res)))
                if i >= warmup:
                    count_ms.append(c_ms)
                    lookup_ms.append(float(res.kernel_ms))
            # every window's k-mer is in the table, and the counts of the windows sum to sum(count^2) over the keys
            v = vals.to(torch.int64)
            if int(out.min().item()) < 1 or int(out.to(torch.int64).sum().item()) != int((v * v).sum().item()):
                raise RuntimeError("the looked-up counts disagree with the table")
            path = "binned count, direct lookup" if (slot_bytes << log2cap) > (96 << 20) else "streaming"
            c_med, l_med = float(np.median(count_ms)), float(np.median(lookup_ms))
            print(json.dumps({
                "case": "per-window lookup vs count, canonical %d-mers (%d limb%s), %d x 150 bp reads at 30x of a %d bp genome, 2^%d slots"
                        % (k, nl, "s" if nl == 2 else "", n_reads, genome_len, log2cap),
                "kmers": n, "distinct_keys": distinct, "table_bytes": slot_bytes << log2cap, "path": path,
                "count_ms_median": c_med, "count_ms_min": float(np.min(count_ms)), "count_G_kmers_per_s": n / (c_med / 1e3) / 1e9,
                "lookup_ms_median": l_med, "lookup_ms_min": float(np.min(lookup_ms)), "lookup_G_kmers_per_s": n / (l_med / 1e3) / 1e9,
                "lookup_over_count_time": l_med / c_med}), flush=True)
            del out
            if log2cap == 26:
                scan_bytes = slot_bytes << log2cap
                hist = torch.zeros(256, dtype=torch.int64, device="cuda")
                hist_fn = ctx.lib.kmc_kmer_table_histogram if nl == 1 else ctx.lib.kmc_kmer_table2_histogram
                med, mn = timed_call(ctx, lambda: check(ctx, hist_fn(ctx.handle, keys.data_ptr(), vals.data_ptr(), log2cap, hist.data_ptr(),
                                                                      256)), steps, warmup)
                if int(hist.sum().item()) != (warmup + steps) * distinct:
                    raise RuntimeError("the histogram does not hold every key")
                print(json.dumps({"case": "count spectrum (256 bins) of the 2^26-slot %d-limb table" % nl, "ms_median": med, "ms_min": mn,
                                  "bytes_read": scan_bytes, "achieved_GBps": scan_bytes / (med / 1e3) / 1e9, "copy_peak_GBps": peak,
                                  "frac_of_copy_peak": scan_bytes / (med / 1e3) / 1e9 / peak}), flush=True)
                solid = int(((vals >= 2)).sum().item())
                ok = torch.empty(nl * solid + 2, dtype=torch.int64, device="cuda")
                ov = torch.empty(solid + 1, dtype=torch.int32, device="cuda")
                n_out = C.c_uint64(0)
                exp_fn = ctx.lib.kmc_kmer_table_export_range if nl == 1 else ctx.lib.kmc_kmer_table2_export_range
                med, mn = timed_call(ctx, lambda: check(ctx, exp_fn(ctx.handle, keys.data_ptr(), vals.data_ptr(), log2cap, 2, 0xFFFFFFFF,
                                                                     ok.data_ptr(), ov.data_ptr(), solid, C.byref(n_out))), steps, warmup)
                if n_out.value != solid:
                    raise RuntimeError("the filtered export did not return every solid key")
                moved = scan_bytes + solid * slot_bytes
                print(json.dumps({"case": "solid keys (count >= 2) of the 2^26-slot %d-limb table" % nl, "ms_median": med, "ms_min": mn,
                                  "keys_out": solid, "bytes_read": scan_bytes, "bytes_read_and_written": moved,
                                  "achieved_GBps": moved / (med / 1e3) / 1e9, "copy_peak_GBps": peak,
                                  "frac_of_copy_peak": moved / (med / 1e3) / 1e9 / peak}), flush=True)
                del hist, ok, ov
            del keys, vals
            torch.cuda.empty_cache()
        del words


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--scale", type=float, default=1.0)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    ctx = kc.Context(0)
    peak = copy_peak_gbs()
    print(json.dumps({"case": "device-to-device copy, 4 GB", "copy_peak_GBps": peak}), flush=True)
    run(ctx, args.steps, args.warmup, args.scale, peak)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        smi = "unknown"
    print(json.dumps({"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi}), flush=True)


if __name__ == "__main__":
    main()
