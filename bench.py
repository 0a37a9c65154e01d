#!/usr/bin/env python
"""bench.py -- canonical 31-mers + fx_hash per second (BASELINE.json metric, config C2).

One "step" is one pass of the hot path over one batch of synthetic reads:
CanonicalDNAMers{31} + fx_hash over 10 M x 150 bp 2-bit reads per GPU (1.2 G k-mers, 400 MB in,
19.2 GB out), weak scaling (every rank owns its own 10 M reads; no data-path collective).

  value     device-resident throughput (inputs in HBM, outputs stay in HBM), CUDA events, max over ranks
  e2e       the same metric through kmc_extract_host with pinned HOST sequence buffers: H2D of the
            step's reads inside, streams left in HBM (KMC_OUT_DEVICE), 32-byte result fingerprint read
            back; e2e_host_streams = the same with both full streams copied to pinned host memory
  roofline  algorithmic bytes (16.3125 B / k-mer) / measured kernel time vs MEASURED_PEAKS.json
  cpu_baseline / --impl reference   the CPU restatement of the reference's per-symbol recurrence
            (oracle/, OpenMP over reads, all host cores) -- Julia is not installed, so the reference
            itself cannot run; see DESIGN.md.
  c4, c5    the two multi-GPU configs BASELINE.json names, timed in the same run (extra keys of the line):
            c4 = CanonicalDNAMers{63} over ONE 1 Gbp sequence, strong-scaled over the ranks by window range with a
            K-1 halo; c5 = the canonical 31-mer bucket-count table (B = 28) over 25 M reads per GPU, count +
            NCCL merge inside libkmerscuda (kmc_bucket_count_merge)
Every rank checks its own output against the oracle (full-stream fingerprints + sampled reads); a failure on any
rank aborts the run without a number.
"""
import argparse
import datetime
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "kmers.jl_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

K = 31
READ_LEN = 150
STRIDE = 5  # words per read (word-aligned CSR)
WPR = READ_LEN - K + 1
BYTES_PER_KMER = 0.25 * READ_LEN / WPR + 8 + 8  # SURVEY.md 8(d): 16.3125
SEED = 439824  # test/benchmark.jl:19
METRIC = "canonical 31-mers+hash/sec"
UNIT = "kmers/s"


def splitmix64(x):
    with np.errstate(over="ignore"):
        z = x + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def synth_reads(n_reads, rank=0, out=None):
    """word[j] = splitmix64(seed + j); trailing bits of each read's last word zeroed."""
    n = n_reads * STRIDE
    base = np.uint64(SEED) + np.uint64(rank) * np.uint64(1 << 40)
    words = out if out is not None else np.empty(n, dtype=np.uint64)
    step = 1 << 24
    for s in range(0, n, step):
        e = min(n, s + step)
        words[s:e] = splitmix64(np.arange(s, e, dtype=np.uint64) + base)
    tail = READ_LEN - 32 * (STRIDE - 1)
    words.reshape(n_reads, STRIDE)[:, STRIDE - 1] &= np.uint64((1 << (2 * tail)) - 1)
    return words


def host_cores():
    """Cores this process may run on.  (OMP_NUM_THREADS is NOT consulted: torchrun exports OMP_NUM_THREADS=1 to its
    workers, which made the round-1 reference arm report 1 core at N >= 2.)"""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def config_dict(n_reads, world):
    """The `config` of the JSON line -- the same dict in both arms."""
    return {"workload": workload_name(n_reads), "k": K, "read_len": READ_LEN, "reads_per_gpu": n_reads,
            "parallelism": f"reads sharded over {world} GPU(s), no data-path collective",
            "l2": "no explicit flush: each step streams 0.4 GB in + 19.2 GB out, far larger than the 126 MB L2"}


def workload_name(n_reads):
    return (f"C2: CanonicalDNAMers{{{K}}} + fx_hash over {n_reads:,} x {READ_LEN} bp 2-bit reads per GPU "
            f"({n_reads * WPR:,} k-mers, SoA canon u64 + hash u64)")


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    # (timestamp last: it contains no comma-separated sub-fields, but keeps the indices below stable)
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,timestamp")

    def __init__(self, device):
        self.device, self.proc, self.path = device, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self, t0=None, t1=None):
        """Median SM clock, maximum power and the throttle reasons over the samples taken between the wall-clock
        times t0 and t1 (the timed region), all samples if none fall inside."""
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = []
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    row = {"sm": float(f[1]), "mx": float(f[2]), "w": float(f[3]), "t": None,
                           "reasons": {name for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                                                "sw_power_cap"), f[5:9]) if v.lower().startswith("active")}}
                except ValueError:
                    continue
                if len(f) > 9:
                    try:
                        row["t"] = datetime.datetime.strptime(f[9], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    except ValueError:
                        pass
                rows.append(row)
            os.unlink(self.path)
        except Exception:
            pass
        inside = [r for r in rows if t0 is not None and r["t"] is not None and t0 <= r["t"] <= t1]
        use = inside or rows
        if use:
            reasons = set().union(*[r["reasons"] for r in use])
            out.update(sm_mhz=float(np.median([r["sm"] for r in use])), sm_max_mhz=float(max(r["mx"] for r in use)),
                       reasons=sorted(reasons), samples=len(use), power_w_max=float(max(r["w"] for r in use)),
                       window="timed region" if inside else "whole run (no sample carried a timestamp inside the timed region)")
        return out


# --------------------------------------------------------------------------------------------
# CPU arm: the oracle's literal per-symbol recurrence, OpenMP over reads (test infrastructure
# used here only as the measured CPU baseline, never on the product path)
# --------------------------------------------------------------------------------------------
def cpu_throughput(sample_reads, min_seconds, threads=0):
    from oracle import oracle as ko
    cores = host_cores() if threads <= 0 else threads
    words = synth_reads(sample_reads)
    n = sample_reads * WPR
    a = np.empty((n, 1), dtype=np.uint64)
    h = np.empty(n, dtype=np.uint64)
    ko.batch_iterate(words, sample_reads, K, ko.CANON, uniform_len=READ_LEN, uniform_stride=STRIDE,
                     want_hash=True, threads=cores, out=(a, None, h))  # warm-up (page faults, threads)
    passes, t0 = 0, time.perf_counter()
    while True:
        ko.batch_iterate(words, sample_reads, K, ko.CANON, uniform_len=READ_LEN, uniform_stride=STRIDE,
                         want_hash=True, threads=cores, out=(a, None, h))
        passes += 1
        dt = time.perf_counter() - t0
        if dt >= min_seconds:
            break
    return n * passes / dt, cores, passes, dt


def run_reference(args, rank, world):
    """The reference arm: the oracle port on all host cores, one step = one GPU's share of the workload (all
    args.reads reads, processed in slabs that reuse one output buffer so that host memory stays bounded).  Under
    torchrun rank 0 alone runs; throughput does not depend on N (there is one host)."""
    if rank != 0:
        return 0
    cores = host_cores()
    julia = shutil.which("julia")
    if julia:
        # the real reference, if a Julia toolchain with Kmers.jl ever is on this machine (baseline/julia_ref.jl)
        try:
            env = dict(os.environ, JULIA_NUM_THREADS=str(cores))
            r = subprocess.run([julia, os.path.join(ROOT, "baseline", "julia_ref.jl"), str(args.reads), str(args.steps)],
                               capture_output=True, text=True, timeout=3600, env=env)
            jl = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
            line = {
                "impl": "reference", "metric": METRIC, "value": jl["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": 1, "ms_per_step": jl["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u64", "data": "synthetic", "config": config_dict(args.reads, world),
                "cpu_baseline": {"value": jl["value"], "unit": UNIT, "cores": jl["cores"], "kind": "reference",
                                 "sample": f"Kmers.jl's own CanonicalDNAMers{{31}} + fx_hash under Threads.@threads, Julia {jl['julia']}, "
                                           f"all {args.reads:,} reads per step"},
                "e2e": {"value": jl["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
            print(json.dumps(line), flush=True)
            return 0
        except Exception as e:  # noqa: BLE001  (no Kmers.jl in that Julia, ...): fall through to the restatement
            print(f"bench.py: julia is on PATH but baseline/julia_ref.jl failed ({e}); timing the C restatement", file=sys.stderr)
    from oracle import oracle as ko
    slab = min(args.reads, args.cpu_sample_reads)
    words = synth_reads(args.reads)
    a = np.empty((slab * WPR, 1), dtype=np.uint64)
    h = np.empty(slab * WPR, dtype=np.uint64)

    def step():
        for r0 in range(0, args.reads, slab):
            r1 = min(args.reads, r0 + slab)
            m = (r1 - r0) * WPR
            ko.batch_iterate(words[r0 * STRIDE:r1 * STRIDE], r1 - r0, K, ko.CANON, uniform_len=READ_LEN, uniform_stride=STRIDE,
                             want_hash=True, threads=cores, out=(a[:m], None, h[:m]))
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    n = args.reads * WPR
    value = n * args.steps / dt
    sample_desc = (f"all {args.reads:,} reads of one GPU's share per step ({n:,} k-mers/step, in slabs of {slab:,} reads), "
                   f"literal per-symbol recurrence, OpenMP parallel-for over reads, {cores} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": config_dict(args.reads, world),
        "note": "Julia is not installed: this arm times the C restatement of the reference algorithm (oracle/) on the host "
                "cores; one host serves all N GPUs, so the value does not scale with N",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample_desc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def _digest(arr):
    """(xor, wrapping sum) of a uint64 array -- what kmc_digest computes on the device."""
    a = arr.reshape(-1)
    return int(np.bitwise_xor.reduce(a)) if a.size else 0, int(a.sum(dtype=np.uint64)) if a.size else 0


def oracle_stream_digests(words, n_reads, threads, slab=1_000_000):
    """Fingerprints of the canonical stream and of the hash stream of a uniform read set, computed by the oracle
    over ALL reads (in slabs): ((xor, sum) of canon, (xor, sum) of hash)."""
    from oracle import oracle as ko
    xa = sa = xh = sh = 0
    a = np.empty((slab * WPR, 1), dtype=np.uint64)
    h = np.empty(slab * WPR, dtype=np.uint64)
    for r0 in range(0, n_reads, slab):
        r1 = min(n_reads, r0 + slab)
        m = (r1 - r0) * WPR
        ko.batch_iterate(words[r0 * STRIDE:r1 * STRIDE], r1 - r0, K, ko.CANON, uniform_len=READ_LEN, uniform_stride=STRIDE,
                         want_hash=True, threads=threads, out=(a[:m], None, h[:m]))
        x, y = _digest(a[:m])
        xa ^= x
        sa = (sa + y) & 0xFFFFFFFFFFFFFFFF
        x, y = _digest(h[:m])
        xh ^= x
        sh = (sh + y) & 0xFFFFFFFFFFFFFFFF
    return (xa, sa), (xh, sh)


DUMP_SAMPLE = 1 << 20  # k-mers per stream written by --dump-outputs: 5 float64 arrays of 8 MiB
DUMP_SEED = 20240611


def dump_outputs(path, ctx, d_canon, d_hash, n_kmers):
    """Writes what the timed call returned, for comparing two builds output for output: a fixed seeded sample of
    DUMP_SAMPLE k-mer positions (all of them for a smaller run) of the canonical and the hash stream, and the
    fingerprints of both full streams.  A u64 is split into its upper and lower 32 bits, each exact as a float64."""
    import torch
    os.makedirs(path, exist_ok=True)
    if n_kmers <= DUMP_SAMPLE:
        idx = np.arange(n_kmers, dtype=np.int64)
    else:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n_kmers, DUMP_SAMPLE, replace=False)).astype(np.int64)
    d_idx = torch.from_numpy(idx).cuda()

    def halves(x):
        x = np.asarray(x, dtype=np.uint64)
        return (x >> np.uint64(32)).astype(np.float64), (x & np.uint64(0xFFFFFFFF)).astype(np.float64)
    arrays = {"kmer_index": idx.astype(np.float64)}
    for name, d in (("canon", d_canon), ("hash", d_hash)):
        arrays[f"{name}_hi"], arrays[f"{name}_lo"] = halves(d[d_idx].cpu().numpy().view(np.uint64))
    # rows: canonical xor, canonical wrapping sum, hash xor, hash wrapping sum; columns: upper, lower 32 bits
    dg = [*ctx.digest(d_canon.data_ptr(), n_kmers), *ctx.digest(d_hash.data_ptr(), n_kmers)]
    arrays["stream_digest"] = np.stack(halves(dg), axis=1)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def splitmix_words(first, count, seed):
    """words[first : first + count) of the counter-based stream word[j] = splitmix64(seed + j)."""
    out = np.empty(count, dtype=np.uint64)
    step = 1 << 24
    for s0 in range(0, count, step):
        e = min(count, s0 + step)
        out[s0:e] = splitmix64(np.arange(first + s0, first + e, dtype=np.uint64) + np.uint64(seed))
    return out


# --------------------------------------------------------------------------------------------
# the multi-GPU configs BASELINE.json names, as extra legs of the same run
# --------------------------------------------------------------------------------------------
C4_LEN = 1_000_000_000
C4_K = 63


def leg_c4(env, steps):
    """C4: CanonicalDNAMers{63} (two limbs) over ONE 1 Gbp 2-bit sequence, STRONG-scaled: rank g extracts the window
    starts [g * ceil(n / N), (g + 1) * ceil(n / N)) from its slice of the words plus a K-1-symbol halo; the concatenation
    in rank order is the unsharded stream.  No collective.  Every rank checks three stretches of its range against the
    oracle, and the fingerprint of all shards together against rank 0's unsharded run (which also gives the N = 1
    time of the same box for the efficiency)."""
    import ctypes as C

    import torch
    import torch.distributed as dist
    from kmerscuda import _abi, sharding
    from oracle import oracle as ko
    ctx, lib, stream, rank, world = env["ctx"], env["lib"], env["stream"], env["rank"], env["world"]
    seed = SEED + (1 << 50)
    n_total = C4_LEN - C4_K + 1

    def run(sh, n_steps):
        words = splitmix_words(sh.word0, sh.n_words, seed)
        d_words = torch.from_numpy(words.view(np.int64)).cuda()
        d_out = torch.empty(sh.n_windows * 2, dtype=torch.int64, device="cuda")
        desc = _abi.kmc_seqs(d_words.data_ptr(), sh.n_words, 1, None, None, sh.length, sh.n_words, 2, sh.first_symbol_offset)
        out = _abi.kmc_out(d_out.data_ptr(), None, None, None, None, sh.n_windows, sh.index_base)
        res = _abi.kmc_result()

        def one():
            st = lib.kmc_extract(ctx.handle, C.byref(desc), C4_K, _abi.KMC_CANON, _abi.KMC_NO_SYNC, C.byref(out), C.byref(res))
            if st != 0:
                raise RuntimeError(f"c4: kmc_extract failed: {lib.kmc_last_error(ctx.handle).decode()}")
        for _ in range(3):
            one()
        return words, d_out, one, res

    sh = sharding.plan_sequence_shards(C4_LEN, C4_K, 2, world)[rank]
    words, d_out, one, res = run(sh, steps)
    env["barrier"]()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for _ in range(steps):
        one()
    t1.record(stream)
    env["barrier"]()
    ms = env["max_over_ranks"](t0.elapsed_time(t1) / steps)
    assert res.n_written == sh.n_windows
    # parity: three stretches of this rank's range against the oracle
    ok = True
    span = 20_000
    for w0 in (0, max(0, sh.n_windows // 2 - span // 2), max(0, sh.n_windows - span)):
        nwin = min(span, sh.n_windows - w0)
        if nwin <= 0:
            continue
        sym0 = sh.first_symbol_offset + w0
        ww = words[sym0 // 32: (sym0 + nwin + C4_K - 1 + 31) // 32 + 1]
        a, _, _ = ko.iterate(ww, nwin + C4_K - 1, C4_K, ko.CANON, first=sym0 % 32)
        got = d_out[2 * w0: 2 * (w0 + nwin)].cpu().numpy().view(np.uint64).reshape(-1, 2)
        ok &= bool(np.array_equal(got, a))
    dg = ctx.digest(d_out.data_ptr(), sh.n_windows * 2)
    # fingerprints of all shards: xor of the xors, wrapping sum of the sums
    t = torch.tensor([dg[0] - (1 << 64) if dg[0] >= (1 << 63) else dg[0], dg[1] - (1 << 64) if dg[1] >= (1 << 63) else dg[1]],
                     dtype=torch.int64, device="cuda")
    parts = [torch.zeros_like(t) for _ in range(world)]
    if world > 1:
        dist.all_gather(parts, t)
    else:
        parts = [t]
    x = s_ = 0
    for q in parts:
        x ^= int(q[0].item()) & 0xFFFFFFFFFFFFFFFF
        s_ = (s_ + int(q[1].item())) & 0xFFFFFFFFFFFFFFFF
    del d_out
    torch.cuda.empty_cache()
    ms1 = ms
    if world > 1:
        # the unsharded run on rank 0 (the other ranks wait): the N = 1 time, and the fingerprint the shards must add up to
        full = [0, 0, 0.0]
        if rank == 0:
            sh1 = sharding.plan_sequence_shards(C4_LEN, C4_K, 2, 1)[0]
            _, d1, one1, _ = run(sh1, steps)
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(stream)
            for _ in range(steps):
                one1()
            a1.record(stream)
            torch.cuda.synchronize()
            d = ctx.digest(d1.data_ptr(), n_total * 2)
            full = [d[0], d[1], a0.elapsed_time(a1) / steps]
            del d1
            torch.cuda.empty_cache()
        box = [full]
        dist.broadcast_object_list(box, src=0)
        ok &= (x, s_) == (box[0][0], box[0][1])
        ms1 = box[0][2]
    env["all_ranks_ok"](ok, "c4: sharded CanonicalDNAMers{63} differs from the oracle / the unsharded run")
    bytes_per = 0.25 + 16
    return {"workload": f"C4: CanonicalDNAMers{{{C4_K}}} (2 limbs) over one {C4_LEN:,} bp 2-bit sequence, window ranges + K-1 halo "
                        f"over {world} GPU(s)", "scaling": "strong", "steps": steps, "ms_per_step": ms,
            "value": n_total / (ms / 1e3), "unit": UNIT, "ms_per_step_1gpu_same_box": ms1,
            "strong_scaling_efficiency": ms1 / (world * ms), "achieved_GBps_per_gpu": bytes_per * n_total / world / (ms / 1e3) / 1e9,
            "bytes_per_kmer": bytes_per, "collective": None,
            "parity": "every rank: 3 x 20,000 windows of its range == oracle; fingerprint of all shards == the unsharded run"}


def leg_c5(env, reads_per_gpu, bits, steps):
    """C5: the canonical 31-mer bucket-count table, table[fx_hash(canon) >> (64 - B)] += 1, over reads_per_gpu x 150 bp
    reads per GPU (25 M x 8 GPUs = the 200 M reads of BASELINE.json), merged with the path's only collective inside
    libkmerscuda: kmc_bucket_count_merge all-reduces every eighth of the table (ncclAllReduce on a communication
    stream) as soon as the count has finished it.  Times: the count alone, the all-reduce alone, the overlapped call."""
    import ctypes as C

    import torch
    from kmerscuda import _abi
    from oracle import oracle as ko
    ctx, lib, stream, rank, world = env["ctx"], env["lib"], env["stream"], env["rank"], env["world"]
    n_kmers = reads_per_gpu * WPR
    g = torch.Generator(device="cuda").manual_seed(SEED + 1000 + rank)
    words = torch.randint(-2**63, 2**63 - 1, (reads_per_gpu * STRIDE,), dtype=torch.int64, device="cuda", generator=g)
    words.view(reads_per_gpu, STRIDE)[:, STRIDE - 1] &= (1 << (2 * (READ_LEN - 32 * (STRIDE - 1)))) - 1
    desc = _abi.kmc_seqs(words.data_ptr(), words.numel(), reads_per_gpu, None, None, READ_LEN, STRIDE, 2, 0)
    table = torch.zeros(1 << bits, dtype=torch.int32, device="cuda")
    res = _abi.kmc_result()
    ctx.comm_init_torch() if world > 1 else ctx.comm_init(1, 0, type(ctx).comm_unique_id())

    def timed(fn, n):
        out = []
        for i in range(n + 1):
            table.zero_()
            env["barrier"]()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            env["barrier"]()
            if i:
                out.append(a.elapsed_time(b))
        return env["max_over_ranks"](float(np.mean(out)))

    def count_only():
        ctx._check(lib.kmc_bucket_count(ctx.handle, C.byref(desc), K, bits, table.data_ptr(), C.byref(res)))

    def merge_only():
        ctx.allreduce(table.data_ptr(), 1 << bits)

    def count_merge():
        ctx._check(lib.kmc_bucket_count_merge(ctx.handle, C.byref(desc), K, bits, table.data_ptr(), C.byref(res)))

    count_ms = timed(count_only, steps)
    merge_ms = timed(merge_only, steps)
    total_ms = timed(count_merge, steps)
    # parity (the table of the last count_merge call): the merged total, the same table on every rank, and this rank's
    # first 100,000 reads counted alone against bincount of the oracle's hashes
    ok = int(res.n_written) == n_kmers
    ok &= int(table.sum(dtype=torch.int64).item()) == n_kmers * world
    dg = ctx.digest(table.data_ptr(), (1 << bits) // 2)
    if world > 1:
        import torch.distributed as dist
        box = [None] * world
        dist.all_gather_object(box, dg)
        ok &= all(b == box[0] for b in box)
    n_s = min(100_000, reads_per_gpu)
    table.zero_()
    sdesc = _abi.kmc_seqs(words.data_ptr(), n_s * STRIDE, n_s, None, None, READ_LEN, STRIDE, 2, 0)
    ctx._check(lib.kmc_bucket_count(ctx.handle, C.byref(sdesc), K, bits, table.data_ptr(), C.byref(res)))
    hw = words[: n_s * STRIDE].cpu().numpy().view(np.uint64)
    _, _, h, _ = ko.batch_iterate(hw, n_s, K, ko.CANON, uniform_len=READ_LEN, uniform_stride=STRIDE, want_hash=True,
                                  threads=max(1, host_cores() // world))
    ub, uc = np.unique((h >> np.uint64(64 - bits)).astype(np.int64), return_counts=True)
    got = table[torch.from_numpy(ub).cuda()].cpu().numpy()
    ok &= bool(np.array_equal(got.astype(np.int64), uc)) and int(table.sum(dtype=torch.int64).item()) == n_s * WPR
    env["all_ranks_ok"](ok, "c5: bucket-count table differs from the oracle / between ranks")
    ctx.comm_destroy()
    del table, words
    torch.cuda.empty_cache()
    ctx.trim()
    tb = 4 << bits
    return {"workload": f"C5: canonical {K}-mer hash-bucket count table, B = {bits} ({tb >> 20} MiB of u32 counters per GPU), "
                        f"{reads_per_gpu:,} x {READ_LEN} bp reads per GPU x {world} GPU(s), count + NCCL merge",
            "scaling": "weak", "steps": steps, "count_ms": count_ms, "merge_ms": merge_ms, "total_ms_overlapped": total_ms,
            "total_ms_sequential": count_ms + merge_ms, "value": n_kmers * world / (total_ms / 1e3), "unit": UNIT,
            "kmers_per_s_count_only_per_gpu": n_kmers / (count_ms / 1e3),
            "allreduce_busbw_GBps": (2 * (world - 1) / world * tb / (merge_ms / 1e3) / 1e9) if world > 1 else None,
            "collective": "ncclAllReduce(u32, sum) of 8 table ranges on a communication stream, inside kmc_bucket_count_merge "
                          "(libkmerscuda binds libnccl at run time; the communicator id is broadcast by torch.distributed)",
            "parity": "every rank: merged total == k-mers of all ranks; identical table on every rank; 100,000 reads counted "
                      "alone == bincount of the oracle's hashes"}


# --------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------
def run_ours(args, rank, local_rank, world):
    import ctypes as C

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    # NCCL_DEBUG=VERSION makes NCCL print a banner on stdout, which must carry exactly one JSON line (at N = 1 too:
    # the c5 leg attaches a one-rank communicator inside libkmerscuda)
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import kmerscuda as kc
    from kmerscuda import _abi

    ctx = kc.Context(local_rank)
    lib = ctx.lib
    n_reads = args.reads
    n_kmers = n_reads * WPR

    # ---- inputs: generated on the host once, resident in HBM before the timed region ----------
    pinned_in = ctx.pinned(n_reads * STRIDE * 8, np.uint64)
    synth_reads(n_reads, rank, out=pinned_in)
    d_words = torch.empty(n_reads * STRIDE, dtype=torch.int64, device="cuda")
    d_canon = torch.empty(n_kmers, dtype=torch.int64, device="cuda")
    d_hash = torch.empty(n_kmers, dtype=torch.int64, device="cuda")
    # a dedicated (non-default) torch stream: the library launches on it and torch.cuda.Event
    # records on it, so the events bracket exactly the kernels they are meant to time
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    ctx.set_stream(stream.cuda_stream)
    ctx._check(lib.kmc_upload(ctx.handle, d_words.data_ptr(), pinned_in.ctypes.data, pinned_in.nbytes))
    ctx.sync()
    desc = _abi.kmc_seqs(d_words.data_ptr(), d_words.numel(), n_reads, None, None, READ_LEN, STRIDE, 2, 0)
    out = _abi.kmc_out(d_canon.data_ptr(), None, d_hash.data_ptr(), None, None, n_kmers, 0)
    res = _abi.kmc_result()
    flags = _abi.KMC_HASH_FX | _abi.KMC_NO_SYNC

    def step():
        st = lib.kmc_extract(ctx.handle, C.byref(desc), K, _abi.KMC_CANON, flags, C.byref(out), C.byref(res))
        if st != 0:
            raise RuntimeError(f"kmc_extract failed: {lib.kmc_last_error(ctx.handle).decode()}")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.15)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    wall0 = time.time()
    t_begin.record(stream)
    for i in range(args.steps):
        ev[i][0].record(stream)
        step()
        ev[i][1].record(stream)
    t_end.record(stream)
    barrier()
    wall1 = time.time()
    total_ms = t_begin.elapsed_time(t_end)
    kernel_ms = [a.elapsed_time(b) for a, b in ev]
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    assert res.n_written == n_kmers
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx, d_canon, d_hash, n_kmers)

    # The same launch with idle gaps (outside the timed region, reported beside the roofline): back to back the
    # kernel runs into the board's power cap and the SM clock drops (tools/diag_power.py: 1000 W, ~1650 of 1965 MHz);
    # with 25 ms of idle between launches it runs at full clock.  The gap between the two is power, not the kernel.
    gap_ms = []
    if rank == 0:
        for _ in range(12):
            time.sleep(0.025)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            step()
            b.record(stream)
            torch.cuda.synchronize()
            gap_ms.append(a.elapsed_time(b))
    barrier()

    t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    max_ms = float(t.item())
    value = n_kmers * world * args.steps / (max_ms / 1e3)

    # ---- the same launch in a sustained loop of about one second (outside the timed region): the board's power
    #      cap only bites after a few hundred milliseconds, so a short timed region reads as a burst
    sus_ms = None
    if not args.no_sustained:
        n_sus = max(50, int(1000.0 / max(np.mean(kernel_ms), 0.1)))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sus_sampler = ClockSampler(local_rank)
        if rank == 0:
            sus_sampler.start()
        w0 = time.time()
        a.record(stream)
        for _ in range(n_sus):
            step()
        b.record(stream)
        torch.cuda.synchronize()
        w1 = time.time()
        sus_ms = a.elapsed_time(b) / n_sus
        sus_clocks = sus_sampler.stop(w0, w1) if rank == 0 else None
    barrier()

    # ---- parity, on EVERY rank (outside the timed region): the fingerprints of both full streams against the
    #      oracle's over all of the rank's reads, and sampled reads element by element.  One failing rank aborts
    #      the whole run without a number.
    def all_ranks_ok(ok, what):
        f = torch.tensor([1 if ok else 0], dtype=torch.int32, device="cuda")
        if world > 1:
            dist.all_reduce(f, op=dist.ReduceOp.MIN)
        if int(f.item()) != 1:
            raise SystemExit(f"bench.py: {what} (rank {rank}: {'ok' if ok else 'MISMATCH'}); refusing to report a number")

    checked = {"ranks": world, "what": "skipped (--no-check)"}
    if not args.no_check:
        from oracle import oracle as ko
        ok = True
        want = oracle_stream_digests(pinned_in, n_reads, max(1, host_cores() // world))
        got = (ctx.digest(d_canon.data_ptr(), n_kmers), ctx.digest(d_hash.data_ptr(), n_kmers))
        ok &= got == want
        rng = np.random.default_rng(7 + rank)
        for r in rng.choice(n_reads, size=64, replace=False):
            w = pinned_in[r * STRIDE:(r + 1) * STRIDE]
            a, _, h = ko.iterate(w, READ_LEN, K, ko.CANON, want_hash=True)
            got_a = d_canon[r * WPR:(r + 1) * WPR].cpu().numpy().view(np.uint64)
            got_h = d_hash[r * WPR:(r + 1) * WPR].cpu().numpy().view(np.uint64)
            ok &= bool(np.array_equal(got_a, a[:, 0]) and np.array_equal(got_h, h))
        all_ranks_ok(ok, "GPU output differs from the oracle")
        checked = {"ranks": world, "what": "every rank: xor + wrapping-sum fingerprints of the full canonical and hash streams "
                                           f"({n_kmers:,} k-mers) == the oracle's over all its reads; 64 sampled reads element-wise"}

    # ---- end to end through the C ABI with HOST sequence buffers ---------------------------------
    # e2e (headline): every step uploads that step's reads from pinned host memory (chunked H2D
    # overlapped with the kernels inside kmc_extract_host), leaves the canonical + hash streams in
    # HBM for a device consumer (KMC_OUT_DEVICE -- the deployment north_star describes: each GPU
    # emits its streams, only tables / sketches / fingerprints leave the GPU), and reads back the
    # step's result fingerprint (KMC_DIGEST: xor + wrapping sum of both streams, 32 bytes).
    # e2e_host_streams: the same call materialising both full streams in pinned HOST memory
    # (19.2 GB over PCIe per step) -- reported beside it; it is PCIe-bound by construction.
    e2e = e2e_host = None
    if not args.no_e2e:
        hdesc = _abi.kmc_seqs(pinned_in.ctypes.data, n_reads * STRIDE, n_reads, None, None, READ_LEN, STRIDE, 2, 0)
        dout = _abi.kmc_out(d_canon.data_ptr(), None, d_hash.data_ptr(), None, None, n_kmers, 0)
        hres = _abi.kmc_result()
        want_dig = (ctx.digest(d_canon.data_ptr(), n_kmers), ctx.digest(d_hash.data_ptr(), n_kmers))  # from the resident run
        d_canon.zero_()
        d_hash.zero_()
        torch.cuda.synchronize()

        def e2e_step():
            st = lib.kmc_extract_host(ctx.handle, C.byref(hdesc), K, _abi.KMC_CANON,
                                      _abi.KMC_HASH_FX | _abi.KMC_OUT_DEVICE | _abi.KMC_DIGEST, C.byref(dout), C.byref(hres))
            if st != 0:
                raise RuntimeError(f"e2e step failed: {lib.kmc_last_error(ctx.handle).decode()}")
        for _ in range(2):
            e2e_step()  # warm-up (allocates the pipeline slots)
        dig = hres.digest
        got_dig = ((int(dig[0]), int(dig[1])), (int(dig[2]), int(dig[3])))
        all_ranks_ok(got_dig == want_dig, "e2e result fingerprint differs from the device-resident run")
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            e2e_step()
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {"value": n_kmers * world * args.e2e_steps / float(dt.item()), "unit": UNIT,
               "h2d_bytes_per_step": n_reads * STRIDE * 8, "d2h_bytes_per_step": 32, "steps": args.e2e_steps,
               "ms_per_step": float(dt.item()) / args.e2e_steps * 1e3,
               "h2d_GBps_per_gpu": n_reads * STRIDE * 8 * args.e2e_steps / float(dt.item()) / 1e9,
               "timer": "host wall clock around the calls (each synchronises), max over ranks",
               "path": "one kmc_extract_host call: pinned host words -> chunked H2D overlapped with the kernels -> canonical "
                       "+ hash streams resident in HBM (KMC_OUT_DEVICE), fingerprinted chunk by chunk (KMC_DIGEST) -> "
                       "32-byte result to host",
               "result_check": "digest equals the device-resident run's; sampled reads equal the oracle"}

        # -- the same call with both streams written to pinned host memory
        del d_canon, d_hash
        torch.cuda.empty_cache()
        # 16 bytes of pinned host memory per k-mer: the full 19.2 GB on one GPU, a 1/world share per rank
        # otherwise (all ranks share one host's memory and one root complex; the number is PCIe-bound anyway)
        e2e_reads = max(1, n_reads // world)
        try:
            h_canon = ctx.pinned(e2e_reads * WPR * 8, np.uint64)
            h_hash = ctx.pinned(e2e_reads * WPR * 8, np.uint64)
        except kc.KmersCUDAError:
            e2e_reads = max(1, e2e_reads // 10)
            h_canon = ctx.pinned(e2e_reads * WPR * 8, np.uint64)
            h_hash = ctx.pinned(e2e_reads * WPR * 8, np.uint64)
        hdesc2 = _abi.kmc_seqs(pinned_in.ctypes.data, e2e_reads * STRIDE, e2e_reads, None, None, READ_LEN, STRIDE, 2, 0)
        hout = _abi.kmc_out(h_canon.ctypes.data, None, h_hash.ctypes.data, None, None, e2e_reads * WPR, 0)

        def host_step():
            st = lib.kmc_extract_host(ctx.handle, C.byref(hdesc2), K, _abi.KMC_CANON, _abi.KMC_HASH_FX, C.byref(hout), C.byref(hres))
            if st != 0:
                raise RuntimeError(f"kmc_extract_host failed: {lib.kmc_last_error(ctx.handle).decode()}")
        host_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.host_steps):
            host_step()
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        if not args.no_check:
            from oracle import oracle as ko
            ok = True
            for r in (0, e2e_reads // 2, e2e_reads - 1):
                a, _, h = ko.iterate(pinned_in[r * STRIDE:(r + 1) * STRIDE], READ_LEN, K, ko.CANON, want_hash=True)
                ok &= bool(np.array_equal(h_canon[r * WPR:(r + 1) * WPR], a[:, 0]) and np.array_equal(h_hash[r * WPR:(r + 1) * WPR], h))
            all_ranks_ok(ok, "host-path output differs from the oracle")
        e2e_host = {"value": e2e_reads * WPR * world * args.host_steps / float(dt.item()), "unit": UNIT,
                    "h2d_bytes_per_step": e2e_reads * STRIDE * 8, "d2h_bytes_per_step": e2e_reads * WPR * 16,
                    "steps": args.host_steps, "reads_per_gpu": e2e_reads,
                    "path": "kmc_extract_host: pinned host words -> 3-slot H2D/kernel/D2H pipeline -> BOTH full streams in "
                            "pinned host memory (PCIe-bound: 16 B per k-mer over the link)"}

    # ---- the multi-GPU configs (C4 strong-scaled, C5 count + NCCL merge), every rank verified -----------------
    try:
        del d_canon, d_hash
    except NameError:
        pass
    torch.cuda.empty_cache()

    def max_over_ranks(v):
        tt = torch.tensor([v], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    env = {"ctx": ctx, "lib": lib, "stream": stream, "rank": rank, "world": world, "barrier": barrier,
           "max_over_ranks": max_over_ranks, "all_ranks_ok": all_ranks_ok}
    c4 = c5 = None
    if not args.no_legs:
        c4 = leg_c4(env, args.leg_steps)
        c5 = leg_c5(env, args.c5_reads, args.c5_bits, max(3, args.leg_steps // 2))

    if rank == 0:
        peak, peak_src = measured_peak()
        k_ms = float(np.mean(kernel_ms))
        achieved = BYTES_PER_KMER * n_kmers / (k_ms / 1e3) / 1e9
        traffic = traffic_src = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                traffic = tj.get("extract_kernel_c2_dram_bytes_per_launch")
                traffic_src = "NOT measured in this run: one ncu --set full capture of the same kernel, " + tj.get("source", tp)
            except Exception:
                traffic = traffic_src = None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": max_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": config_dict(n_reads, world),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "frac_timed_region_is": "sustained" if max_ms > 250.0 else "burst (timed region shorter than 0.25 s: the "
                                                 "board's power cap has not bitten yet; see frac_sustained)",
                         "frac_sustained": (BYTES_PER_KMER * n_kmers / (sus_ms / 1e3) / 1e9 / peak) if sus_ms else None,
                         "sustained": {"kernel_ms": sus_ms, "clocks": sus_clocks,
                                       "how": "the same launch back to back for about one second, outside the timed region"}
                         if sus_ms else None,
                         "frac_burst": (BYTES_PER_KMER * n_kmers / (float(np.median(gap_ms)) / 1e3) / 1e9 / peak) if gap_ms else None,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "extract_aligned_kernel<N=1,NX=3,CANON,HASH,SINK_STREAMS,BPS=2> (G=8; aligned uniform set: extract_kernels.cuh)",
                         "kernel_ms": k_ms, "bytes_per_kmer": BYTES_PER_KMER, "peak_source": peak_src,
                         "idle_gaps": {"kernel_ms": float(np.median(gap_ms)),
                                       "achieved": BYTES_PER_KMER * n_kmers / (float(np.median(gap_ms)) / 1e3) / 1e9,
                                       "how": "the same launch, 12 times with 25 ms of idle before each (full SM clock, no "
                                              "power cap); not the timed region"} if gap_ms else None,
                         "write_ceiling_note": "the peak is a copy (half reads); this kernel is 98 % writes, whose ceiling "
                                               "measures 7480 GB/s (profiles/r01_bw_probe_v2.json, tools/bw_probe.py)"},
            "gpu_launches": args.steps,
            "clocks": clocks,
            "parity": checked,
        }
        if c4:
            line["c4"] = c4
        if c5:
            line["c5"] = c5
        if e2e:
            line["e2e"] = e2e
            line["e2e_host_streams"] = e2e_host
        if world == 1 and not args.no_cpu:
            v, cores, passes, dt = cpu_throughput(min(n_reads, args.cpu_sample_reads), args.cpu_seconds)
            line["cpu_baseline"] = {
                "value": v, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": (f"{min(n_reads, args.cpu_sample_reads):,} of the {n_reads:,} reads x {passes} passes in {dt:.1f} s; "
                           "C restatement of the reference's per-symbol recurrence, OpenMP over reads")}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=10_000_000, help="reads per GPU")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--host-steps", type=int, default=2)
    ap.add_argument("--cpu-sample-reads", type=int, default=2_000_000)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--no-sustained", action="store_true")
    ap.add_argument("--no-legs", action="store_true", help="skip the c4 / c5 legs")
    ap.add_argument("--leg-steps", type=int, default=10)
    ap.add_argument("--c5-reads", type=int, default=25_000_000, help="reads per GPU of the c5 leg")
    ap.add_argument("--c5-bits", type=int, default=28)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write rank 0's outputs of the last step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and "RANK" not in os.environ:
        # launched directly: re-exec under torchrun, one rank per GPU
        port = 29500 + os.getpid() % 2000
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                                   f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
                                   "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:])
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    return run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    sys.exit(main())
