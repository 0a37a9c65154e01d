#!/usr/bin/env python
"""Device time of the exact count table of two-limb k-mers (kmc_kmer_count2), the counterpart of
`tools/bench_configs.py --cases count` (one-limb canonical 31-mers) with canonical 63-mers: 4 M x 150 bp reads sampled
at 30x coverage from a 20 Mbp genome (2^26 slots = 1.25 GB: the k-mers are written out, binned by table slice and
inserted slice after slice) and from a 1 Mbp genome (table of 2^22 slots = 80 MB, L2-resident: the k-mers are inserted
as they are produced).  The same generator, seed and order of draws as the one-limb case, so the reads are the same.
One JSON line per case, then the GPU's name and power limit.

  python tools/bench_count2.py [--steps 10] [--warmup 3] [--scale 1.0]
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
from bench_configs import CANON, emit  # noqa: E402


def sampled_reads(n_reads, length, stride, genome_len, g):
    """n_reads reads of `length` symbols at random positions of a random genome, 2-bit packed, `stride` words per read."""
    shifts = torch.arange(32, device="cuda", dtype=torch.int64) * 2
    genome = torch.randint(0, 4, (genome_len,), dtype=torch.int64, device="cuda", generator=g)
    words = torch.empty(n_reads * stride, dtype=torch.int64, device="cuda")
    pos = torch.arange(stride * 32, device="cuda")
    for c0 in range(0, n_reads, 250_000):
        c1 = min(n_reads, c0 + 250_000)
        starts = torch.randint(0, genome_len - length, (c1 - c0, 1), device="cuda", generator=g)
        codes = genome[(starts + pos).clamp(max=genome_len - 1)] * (pos < length)
        words[c0 * stride:c1 * stride] = (codes.view(c1 - c0, stride, 32) << shifts).sum(-1).view(-1)
    return words


def case_count2(ctx, steps, warmup, scale):
    n_reads, length, stride, k = int(4_000_000 * scale), 150, 5, 63
    wpr = length - k + 1
    res = _abi.kmc_result()
    g = torch.Generator(device="cuda").manual_seed(77)
    for genome_len, log2cap in ((int(20_000_000 * scale), 26), (1_000_000, 22)):
        words = sampled_reads(n_reads, length, stride, genome_len, g)
        desc = _abi.kmc_seqs(words.data_ptr(), words.numel(), n_reads, None, None, length, stride, 2, 0)
        keys = torch.empty(2 << log2cap, dtype=torch.int64, device="cuda")  # u64[2^cap][2]
        vals = torch.empty(1 << log2cap, dtype=torch.int32, device="cuda")
        distinct = [0]

        def stepf():
            keys.fill_(-1)
            vals.zero_()
            st = ctx.lib.kmc_kmer_count2(ctx.handle, C.byref(desc), k, CANON, keys.data_ptr(), vals.data_ptr(), log2cap, C.byref(res))
            if st != 0:
                raise RuntimeError(ctx.lib.kmc_last_error(ctx.handle).decode())
            distinct[0] = int(res.digest[0])
        torch.cuda.synchronize()
        ms = []
        for i in range(warmup + steps):
            stepf()
            if i >= warmup:
                ms.append(float(res.kernel_ms))
        n = n_reads * wpr
        total = int(vals.sum(dtype=torch.int64).item())
        if total != n:
            raise RuntimeError(f"the table holds {total} counts for {n} k-mers")
        emit("exact canonical 63-mer count table (two limbs), %d x 150 bp reads at 30x of a %d bp genome, 2^%d slots"
             % (n_reads, genome_len, log2cap), n, 0.25 * length / wpr * n + 20.0 * distinct[0], float(np.median(ms)), float(np.min(ms)),
             {"distinct_keys": distinct[0], "table_bytes": 20 << log2cap, "path": "binned" if (20 << log2cap) > (96 << 20) else "streaming",
              "G_kmers_per_s": n / (float(np.median(ms)) / 1e3) / 1e9})
        del words, keys, vals


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    ctx = kc.Context(0)
    case_count2(ctx, args.steps, args.warmup, args.scale)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        smi = "unknown"
    print(json.dumps({"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi}), flush=True)


if __name__ == "__main__":
    main()
