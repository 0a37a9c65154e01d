// buckets.cu -- the canonical k-mer bucket-count table (north_star extension; not in the reference):
// table[fx_hash(canonical k-mer) >> (64 - B)] += 1 over a read set.
//
// Two regimes, both bound by how fast an SM can issue scattered 4-byte increments (1.29 cycles per lane:
// 2.2e11 / s measured; shared-memory atomics are no faster, so there is nothing to privatise):
//   * the table fits L2 (<= 96 MB): extract_kernel<SINK_BUCKETS> increments it directly;
//   * larger tables (B = 28 is 1 GiB): random increments miss L2 and serialise at DRAM latency (measured
//     24 G k-mers/s).  So the bucket ids are first written out (SINK_IDS), partitioned by their high bits into
//     bins whose table slice is <= 16 MB (binning.cuh: no atomics, exact placement from a count matrix), and
//     then applied bin after bin, so that all SMs work on an L2-resident part of the table at a time.  The
//     table is final range by range, which kmc_bucket_count_async reports through events so that the merge of
//     several GPUs' tables can overlap the count.
// This file holds the whole count, from kmc_bucket_count / kmc_bucket_count_async to the last event; enqueue_count
// chooses the path.
#include <type_traits>

#include "binning.cuh"
#include "plan.h"

namespace kmc {

namespace {

// An increment that MISSES L2 is far more expensive than its 64 bytes of DRAM traffic: the L2 slice's
// atomic unit waits for the fill, so misses serialise at DRAM latency (tools/micro/atomics_probe.cu:
// 2.2e11 increments/s on a warm 16 MB table, 2.3e10/s when every increment misses -- and still only
// 2.7e10/s on binned ids, because each slice is cold when its bin starts).  So every bin first pulls
// its table slice into L2 with plain coalesced loads (bandwidth-bound, 16 MB), then applies its ids.
__global__ void __launch_bounds__(256) warm_slice_kernel(const uint32_t *__restrict__ slice, uint64_t n_counters,
                                                         uint32_t *__restrict__ sink)
{
    const uint4 *p = reinterpret_cast<const uint4 *>(slice);
    const uint64_t n4 = n_counters / 4;
    uint32_t acc = 0;
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4;
         i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        uint4 v;
        // evict_last: the slice is to stay in L2 while its bins are applied, whatever streams through beside it
        asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                     : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                     : "l"(p + i), "l"(0x14F0000000000000ull));
        acc |= v.x & v.y & v.z & v.w;
    }
    if (acc == 0xffffffffu) *sink = acc; // keeps the loads alive; a count of 2^32-1 in four neighbours does not happen
}

// the ids of bins [bin, bin_end) are binned[offs[bin * n_blocks] .. offs[bin_end * n_blocks])
__global__ void __launch_bounds__(256) bin_apply_kernel(const uint32_t *__restrict__ binned, const uint64_t *__restrict__ offs,
                                                        uint64_t n_blocks, int bin, int bin_end, uint32_t *__restrict__ table)
{
    const uint64_t begin = __ldg(offs + static_cast<uint64_t>(bin) * n_blocks);
    const uint64_t end = __ldg(offs + static_cast<uint64_t>(bin_end) * n_blocks);
    const uint64_t a4 = (begin + 3) & ~3ull; // 16-byte aligned middle part
    const uint64_t tid = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const uint64_t threads = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    if (tid < a4 - begin && begin + tid < end) atomicAdd(table + binned[begin + tid], 1u);
    for (uint64_t i = a4 + tid * 4; i < end; i += threads * 4) {
        if (i + 4 <= end) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(binned + i));
            atomicAdd(table + v.x, 1u);
            atomicAdd(table + v.y, 1u);
            atomicAdd(table + v.z, 1u);
            atomicAdd(table + v.w, 1u);
        } else {
            for (uint64_t j = i; j < end; ++j) atomicAdd(table + binned[j], 1u);
        }
    }
}


// ---------------------------------------------------------------------------------------------
// The fused first half of the binned count for the common case -- one-limb k-mers (K <= 32) over an aligned uniform
// read set (extract_kernels.cuh: AlignedItems; C5 is 150 bp reads, K = 31).  The three passes of the exact path
// (bucket ids written out, per-chunk bin histogram, scatter) read and write 12 bytes per k-mer three times over and
// need the histogram only to know where every chunk's run of every bin goes.  Counting does not care about the order
// inside a bin, so here ONE kernel produces the ids and bins them: a block computes the canonical k-mers and hashes
// of 4096 windows per iteration (16 per thread, in registers), runs the same shared-memory binning step
// (binning.cuh: scatter64_iter) and reserves the place of each of its 64 runs with one atomicAdd on the bin's
// cursor.  The bins have a fixed capacity, mean + 12.5 % + 8192 ids: fx_hash spreads distinct k-mers evenly.  A set in which
// one bucket range attracts much more than its share (reads of one repeated k-mer, say) fills a bin; a run that no longer
// fits goes to the SPILL list instead (one more atomicAdd; the list can hold every id of the call, so nothing is ever
// dropped and there is nothing to fall back to), and the bin ends where that run would have begun.  The spilled ids are
// applied to the table directly, before the bins -- they are few, or they are many and hit the same few counters.
// 4.2 + 1.9 + 7.9 ms of the 30.6 ms per 3 G k-mers become one kernel of 9.7 ms, and the call stays asynchronous.
// ---------------------------------------------------------------------------------------------
constexpr int kStateBinEnd = binning::kTpBins;      // state[64 .. 128): where a full bin ends (~0: it never filled up)
constexpr int kStateSpill = 2 * binning::kTpBins;   // state[128]: ids in the spill list
constexpr int kStateWords = 2 * binning::kTpBins + 2;

struct FusedBins {
    uint32_t *binned;             // 64 bins of `cap` ids each, then the spill list
    uint64_t cap;                 // a multiple of 4 (the apply kernel loads 16 bytes at a time)
    unsigned long long *state;    // [64] ids reserved per bin, [64] bin ends, [1] spill cursor
    int bin_shift;                // bin = id >> bin_shift
};

template <int NX>
__global__ void __launch_bounds__(binning::kBlock, 3) bucket_bin_kernel(const ExtractParams p, const FusedBins f)
{
    using S = binning::Shape<uint32_t>;
    constexpr int G = 8, PT = S::kPerThread;
    static_assert(PT == 2 * G && S::kChunk == kTileItems * G, "a thread bins the ids of two work items per iteration");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    binning::Scatter64Smem<uint32_t> &sm = *reinterpret_cast<binning::Scatter64Smem<uint32_t> *>(smem_raw);
    const uint32_t n_items = static_cast<uint32_t>(p.items);
    const uint32_t tile_base = blockIdx.x * static_cast<uint32_t>(kTileItems);
    if (p.pf_tiles) burst_prefetch<false, G, 2>(p, n_items);
    const AlignedItems<G, 2> items(p);
    const uint32_t tile_end = n_items - tile_base > static_cast<uint32_t>(kTileItems) ? tile_base + kTileItems : n_items;
    const bool inside = items.template loads_inside<NX>(p, tile_end - 1u);
    const binning::IdBin bin_of{f.bin_shift};
    constexpr int kItemsPerIter = 2 * binning::kBlock;
    // where the run of `count` ids of bin b goes
    auto reserve = [&](int b, uint32_t count) -> uint64_t {
        if (count == 0) return 0;
        const uint64_t at = atomicAdd(f.state + b, static_cast<unsigned long long>(count));
        if (at + count > f.cap) {
            // the bin is full: it ends where this run would have begun (every run reserved before it fits, every later
            // one starts beyond the capacity too), and the run goes to the spill list
            atomicMin(f.state + kStateBinEnd + b, static_cast<unsigned long long>(at));
            return binning::kTpBins * f.cap + atomicAdd(f.state + kStateSpill, static_cast<unsigned long long>(count));
        }
        return static_cast<uint64_t>(b) * f.cap + at;
    };
    // the bucket ids of one work item (its G windows)
    auto ids_of = [&](uint32_t item, uint32_t *key) {
        uint32_t x[NX];
        load_block_at<NX>(p, items.bit_of(item), inside, x);
        uint64_t fw[G][1], rv[G][1];
        block_kmers<1, NX, G, true, true, 2>(x, p.s0, p.head_mask, fw, rv);
#pragma unroll
        for (int j = 0; j < G; ++j) {
            const uint64_t c[1] = {fw[j][0] < rv[j][0] ? fw[j][0] : rv[j][0]};
            key[j] = static_cast<uint32_t>(fx_hash<1>(c, 0) >> p.bucket_shift);
        }
    };
#pragma unroll 1
    for (uint32_t it_base = tile_base; it_base < tile_end; it_base += kItemsPerIter) {
        uint32_t key[PT];
        if (tile_end - it_base >= static_cast<uint32_t>(kItemsPerIter)) { // block-uniform: every iteration but the set's last
            ids_of(it_base + threadIdx.x, key);
            ids_of(it_base + binning::kBlock + threadIdx.x, key + G);
            binning::scatter64_iter<uint32_t, true>(sm, key, 0xffffu, bin_of, reserve, f.binned);
        } else {
            uint32_t ok_mask = 0;
#pragma unroll
            for (int j = 0; j < PT; ++j) key[j] = 0;
            if (it_base + threadIdx.x < tile_end) {
                ids_of(it_base + threadIdx.x, key);
                ok_mask = 0xffu;
            }
            if (it_base + binning::kBlock + threadIdx.x < tile_end) {
                ids_of(it_base + binning::kBlock + threadIdx.x, key + G);
                ok_mask |= 0xff00u;
            }
            binning::scatter64_iter<uint32_t, false>(sm, key, ok_mask, bin_of, reserve, f.binned);
        }
    }
}

// The ids of bin b are binned[b * cap .. b * cap + min(reserved, bin end)).  The next 16 bytes of ids are loaded before the
// current four are applied.
__device__ __forceinline__ uint4 ld_ids(const uint32_t *p)
{
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "l"(p), "l"(0x12F0000000000000ull));
    return v;
}
__device__ __forceinline__ void inc_counter(uint32_t *p)
{
    asm volatile("red.global.add.L2::cache_hint.u32 [%0], 1, %1;" ::"l"(p), "l"(0x14F0000000000000ull) : "memory");
}

__global__ void __launch_bounds__(256) bin_apply_fused_kernel(const uint32_t *__restrict__ binned, uint64_t cap,
                                                              const unsigned long long *__restrict__ state, int bin, int bin_end,
                                                              uint32_t *__restrict__ table)
{
    const uint64_t tid = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const uint64_t step = static_cast<uint64_t>(gridDim.x) * blockDim.x * 4;
    for (int b = bin; b < bin_end; ++b) {
        const uint32_t *ids = binned + static_cast<uint64_t>(b) * cap; // 16-byte aligned: cap is a multiple of 4
        const uint64_t reserved = state[b], full_at = state[kStateBinEnd + b];
        const uint64_t n = reserved < full_at ? reserved : full_at, n4 = n & ~3ull;
        uint64_t i = tid * 4;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (i < n4) v = ld_ids(ids + i);
        while (i < n4) {
            const uint64_t nxt = i + step;
            uint4 w = make_uint4(0, 0, 0, 0);
            if (nxt < n4) w = ld_ids(ids + nxt);
            inc_counter(table + v.x);
            inc_counter(table + v.y);
            inc_counter(table + v.z);
            inc_counter(table + v.w);
            v = w;
            i = nxt;
        }
        if (tid < n - n4) inc_counter(table + ids[n4 + tid]);
    }
}

// the spill list: ids whose bin was full, applied to the table as they come (no slice of it is resident for them)
__global__ void __launch_bounds__(256) spill_apply_kernel(const uint32_t *__restrict__ spill, const unsigned long long *__restrict__ state,
                                                          uint32_t *__restrict__ table)
{
    const uint64_t n = state[kStateSpill];
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<uint64_t>(gridDim.x) * blockDim.x)
        atomicAdd(table + spill[i], 1u);
}

uint64_t fused_bin_capacity(uint64_t n_ids)
{
    const uint64_t cap = n_ids / binning::kTpBins + n_ids / (8 * binning::kTpBins) + 8192;
    return (cap + 3) & ~3ull;
}
// ids the binned buffer holds: the 64 bins and a spill list long enough for every id of the call
uint64_t fused_bin_buffer_ids(uint64_t n_ids) { return binning::kTpBins * fused_bin_capacity(n_ids) + n_ids + 4096; }

// First half: one kernel bins the bucket ids of every window into the 64 bins.  p: the parameter block of an aligned uniform
// set of one-limb k-mers with whole groups and fewer than 2^32 - kTileItems work items, strides and bucket_shift set (the
// caller has checked that).  bin = id >> shift.
cudaError_t fused_bin_ids(ExtractParams p, int nx, int shift, uint32_t *binned, uint64_t cap, unsigned long long *state,
                          cudaStream_t stream)
{
    const uint64_t tiles = (p.items + kTileItems - 1) / kTileItems;
    p.al_magic = aligned_magic(p.gprm);
    p.pf_tiles = 0;
    if (prefetch_enabled()) {
        const uint64_t per_tile = static_cast<uint64_t>(p.nw32) * 4 / tiles + 1, t = kPfChunkBytes / per_tile;
        p.pf_tiles = static_cast<uint32_t>(t < 2 * kPfLead ? 2 * kPfLead : (t > (1u << 20) ? (1u << 20) : t));
    }
    cudaError_t e = cudaMemsetAsync(state, 0, kStateWords * sizeof(unsigned long long), stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(state + kStateBinEnd, 0xff, binning::kTpBins * sizeof(unsigned long long), stream);
    if (e != cudaSuccess) return e;
    const FusedBins f{binned, cap, state, shift};
    constexpr int smem = static_cast<int>(sizeof(binning::Scatter64Smem<uint32_t>));
    auto launch = [&](auto tag) -> cudaError_t {
        constexpr int NX = decltype(tag)::value;
        cudaError_t e2 = cudaFuncSetAttribute(bucket_bin_kernel<NX>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e2 != cudaSuccess) return e2;
        bucket_bin_kernel<NX><<<static_cast<unsigned>(tiles), binning::kBlock, smem, stream>>>(p, f);
        return cudaGetLastError();
    };
    switch (nx) {
    case 1: return launch(std::integral_constant<int, 1>());
    case 2: return launch(std::integral_constant<int, 2>());
    case 3: return launch(std::integral_constant<int, 3>());
    }
    return cudaErrorInvalidValue;
}

// Second half: the spill list, then the bins in table order.
cudaError_t fused_bin_apply(const uint32_t *binned, uint64_t cap, const unsigned long long *state, int shift, uint32_t *table,
                            uint32_t *sink, int sm_count, cudaStream_t stream, uint32_t n_parts, void *const *events)
{
    const uint64_t slice = 1ull << shift;
    spill_apply_kernel<<<static_cast<unsigned>(sm_count * 8), 256, 0, stream>>>(binned + binning::kTpBins * cap, state, table);
    auto apply = [&](int b, int b_end) {
        const cudaError_t e = warm_table(table + static_cast<uint64_t>(b) * slice, slice * (b_end - b), sm_count, sink, stream);
        if (e != cudaSuccess) return e;
        bin_apply_fused_kernel<<<static_cast<unsigned>(sm_count * 16), 256, 0, stream>>>(binned, cap, state, b, b_end, table);
        return cudaGetLastError();
    };
    return binning::apply_groups(binning::kTpBins, binning::kBucketGroup, n_parts, events, stream, apply);
}

// Enqueues the count on the first path that applies:
//   * no windows: nothing to count;
//   * the table fits L2: the extraction kernel increments it directly (SINK_BUCKETS);
//   * one-limb k-mers over an aligned uniform set in 64 bins (C5), and the fused bins fit in memory: ids and bins from one
//     kernel, bins of a fixed capacity and a spill list for the runs of a bin that filled up;
//   * the temporaries of the exact path fit in memory: ids written out (SINK_IDS), partitioned, applied bin after bin;
//   * otherwise direct increments.
// Every path records the n_parts progress events (events may be NULL) once their ranges of the table are final.
int32_t enqueue_count(kmc_ctx *ctx, const Geometry &ge, const Layout &L, ExtractParams p, int bucket_bits, uint32_t *table,
                      uint32_t n_parts, void *const *events, cudaStream_t stream)
{
    auto record_all = [&]() -> int32_t {
        for (uint32_t i = 0; i < n_parts; ++i) CU(cudaEventRecord(static_cast<cudaEvent_t>(events[i]), stream));
        return KMC_OK;
    };
    if (L.total == 0) return record_all();
    int32_t st = ensure_host_small(ctx); // allocates dev_small, where the warm-up kernel's sink lives
    if (st) return st;
    const bool fits_l2 = (4ull << bucket_bits) <= binning::kL2Budget;
    if (!fits_l2) {
        const int pbits = binning::bin_bits(bucket_bits, binning::kBucketSliceBits), shift = bucket_bits - pbits;
        ExtractParams pa = p;
        set_iteration_strides(pa, ge.g);
        if (ge.n_limbs == 1 && L.uniform_len && pbits == 6 && pa.aligned && pa.al_tail == 0 && pa.items < 0xffffffffull - kTileItems) {
            AsyncBuf bins_buf, state_buf;
            const uint64_t cap = fused_bin_capacity(L.total);
            cudaError_t e = bins_buf.alloc(ctx, fused_bin_buffer_ids(L.total) * 4, stream);
            if (e == cudaSuccess) e = state_buf.alloc(ctx, kStateWords * sizeof(unsigned long long), stream);
            if (e == cudaSuccess) {
                CU(fused_bin_ids(pa, ge.nx, shift, bins_buf.as<uint32_t>(), cap, state_buf.as<unsigned long long>(), stream));
                CU(fused_bin_apply(bins_buf.as<uint32_t>(), cap, state_buf.as<unsigned long long>(), shift, table, warm_sink(ctx),
                                   ctx->sm_count, stream, n_parts, events));
                return KMC_OK;
            }
            (void)cudaGetLastError();
        }
        // the flat id array is exactly the flat window array: every flat index < windows is written once (slots of partial
        // groups that are not windows are not written and not binned)
        binning::BinnedKeys<uint32_t> bk;
        if (bk.alloc(ctx, (L.items + 1) * static_cast<uint64_t>(ge.g), pbits, stream)) {
            p.out_a = bk.written.as<uint64_t>();
            p.vec_ok = 1;
            ExtractLaunchFn fn = get_launcher(ge, MODE_BUCKET_IDS, true, !L.uniform_len);
            if (!fn) return fail(ctx, KMC_E_UNSUPPORTED, "no kernel for this K");
            CU(fn(p, ctx->sm_count, stream));
            CU(bk.partition(L.total, binning::IdBin{shift}, stream));
            const uint64_t slice = 1ull << shift;
            auto apply = [&](int b, int b_end) {
                const cudaError_t e = warm_table(table + static_cast<uint64_t>(b) * slice, slice * (b_end - b), ctx->sm_count,
                                                 warm_sink(ctx), stream);
                if (e != cudaSuccess) return e;
                bin_apply_kernel<<<static_cast<unsigned>(ctx->sm_count * 16), 256, 0, stream>>>(bk.binned.as<uint32_t>(), bk.offs.as<uint64_t>(),
                                                                                                bk.n_blocks, b, b_end, table);
                return cudaGetLastError();
            };
            CU(binning::apply_groups(1 << pbits, binning::kBucketGroup, n_parts, events, stream, apply));
            return KMC_OK;
        }
    }
    // a table that fits L2 is pulled into it first: increments that miss L2 serialise at DRAM latency
    if (fits_l2) CU(warm_table(table, 1ull << bucket_bits, ctx->sm_count, warm_sink(ctx), stream));
    p.bucket_table = table;
    ExtractLaunchFn fn = get_launcher(ge, MODE_BUCKETS, true, !L.uniform_len);
    if (!fn) return fail(ctx, KMC_E_UNSUPPORTED, "no kernel for this K");
    CU(fn(p, ctx->sm_count, stream));
    return record_all();
}

// n_parts == 0: the synchronous call (kernel_ms measured); otherwise progress events and no synchronisation
int32_t bucket_count(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t bucket_bits, uint32_t *table, uint32_t n_parts,
                     void *const *events, kmc_result *result)
{
    int32_t st = check_common(ctx, seqs, k);
    if (st) return st;
    if (!table || !result) return fail(ctx, KMC_E_BAD_ARG, "table / result is NULL");
    if (bucket_bits < 1 || bucket_bits > 32) return fail(ctx, KMC_E_BAD_ARG, "bucket_bits must be in 1..32");
    if (seqs->src_bits != 2) return fail(ctx, KMC_E_UNSUPPORTED, "bucket count needs a 2-bit source");
    CU(cudaSetDevice(ctx->device));
    result->n_written = 0;
    result->err_seq = result->err_pos = 0;
    result->err_sym = 0;
    result->kernel_ms = 0.f;
    const Geometry ge = geometry(k);
    cudaStream_t stream = ctx->stream;
    CU(cudaEventRecord(ctx->ev_k0, stream));
    st = ensure_scratch(ctx, layout_scratch_bytes(seqs) + 256);
    if (st) return st;
    Scratch scratch{static_cast<char *>(ctx->scratch), ctx->scratch_bytes, 0};
    Layout L;
    st = plan_layout(ctx, seqs, k, ge, stream, KnownTotals(), scratch, &L);
    if (st) return st;
    result->n_written = L.total;
    ExtractParams p = base_params(seqs, k, ge, L, 0);
    p.bucket_shift = static_cast<uint32_t>(64 - bucket_bits);
    st = enqueue_count(ctx, ge, L, p, bucket_bits, table, n_parts, events, stream);
    if (st || n_parts || L.total == 0) return st; // the asynchronous form: the caller waits for its events
    CU(cudaEventRecord(ctx->ev_k1, stream));
    CU(cudaStreamSynchronize(stream));
    CU(cudaEventElapsedTime(&result->kernel_ms, ctx->ev_k0, ctx->ev_k1));
    return KMC_OK;
}

} // namespace

cudaError_t warm_table(const uint32_t *table, uint64_t n_counters, int sm_count, uint32_t *sink, cudaStream_t stream)
{
    warm_slice_kernel<<<static_cast<unsigned>(sm_count * 8), 256, 0, stream>>>(table, n_counters, sink);
    return cudaGetLastError();
}

} // namespace kmc

using namespace kmc;

extern "C" int32_t kmc_bucket_count(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t bucket_bits, uint32_t *table,
                                    kmc_result *result)
{
    return bucket_count(ctx, seqs, k, bucket_bits, table, 0, nullptr, result);
}

extern "C" int32_t kmc_bucket_count_async(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t bucket_bits, uint32_t *table,
                                          uint32_t n_parts, void *const *events, kmc_result *result)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (!events || n_parts < 1 || n_parts > 32 || (n_parts & (n_parts - 1)))
        return fail(ctx, KMC_E_BAD_ARG, "n_parts must be a power of two <= 32 and events non-NULL");
    for (uint32_t i = 0; i < n_parts; ++i)
        if (!events[i]) return fail(ctx, KMC_E_BAD_ARG, "NULL event");
    return bucket_count(ctx, seqs, k, bucket_bits, table, n_parts, events, result);
}
