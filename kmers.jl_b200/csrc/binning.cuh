// binning.cuh -- partition an array of keys into 2^P bins on the device (P = 6 .. 10).
//
// Used where a table is too large for L2 and random updates to it would run at DRAM latency: the
// updates are first sorted by the table slice they touch, then applied slice after slice
// (buckets.cu: 32-bit bucket ids; sketch.cu: 64-bit one-limb and 128-bit two-limb (ulonglong2) k-mers of the
// exact count tables).
//
// One block owns a chunk of the input.  Pass 1 counts the chunk's keys per bin (count matrix
// [bin][block]), an exclusive scan of the matrix gives every (bin, block) its place in the output, pass
// 2 moves the keys: staged in shared memory in bin order, written out as runs.  No global cursors, no
// atomics on global memory, deterministic sizes.
//
// Shared-memory atomics cost about two cycles per lane on this machine -- as much as the L2 updates
// the binning is there to save -- so neither pass uses them:
//   * 64 bins (the common case): no warp cooperation at all.  A thread counts the bins of its own keys
//     in byte counters that only it touches -- the four bins 4g..4g+3 share the word [g][thread], so a
//     warp's accesses fall into 32 different banks -- and the value a counter had before a key was
//     counted is that key's rank among the thread's keys of the bin.  Threads are ordered by
//     (lane, warp) for the prefix sums, which lets a lane sum the words of "its" eight threads without
//     bank conflicts, four 8-bit (then two 16-bit) fields at a time.
//   * more bins: the lanes of a warp that hold the same bin find each other with one ballot per bin
//     bit (the way a radix sort ranks its digits); the lowest of them adds their number to a counter
//     that only this warp touches, and a lane's rank is the counter before that plus the number of
//     peers below it.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <type_traits>

#include "kmc_internal.h"
#include "table_keys.cuh"

namespace kmc {
namespace binning {

constexpr int kBlock = 256;
constexpr int kWarps = kBlock / 32;
constexpr int kIters = 4;
constexpr int kMinBits = 6, kMaxBits = 10;

template <typename Key> struct Shape {
    static constexpr int kPerVec = 16 / sizeof(Key);           // keys per 128-bit load
    static constexpr int kPerThread = 4 * kPerVec;             // keys per thread per iteration (four 128-bit loads)
    static constexpr int kPerIter = kBlock * kPerThread;       // keys staged per iteration
    static constexpr int kChunk = kPerIter * kIters;           // keys per block
    static_assert(kIters * kPerThread < 256, "a byte counts a thread's keys of one bin");
};

template <typename Key> inline uint64_t blocks_for(uint64_t n) { return (n + Shape<Key>::kChunk - 1) / Shape<Key>::kChunk; }

// bin of a 32-bit bucket id: its high bits
struct IdBin {
    int shift;
    __device__ __forceinline__ uint32_t operator()(uint32_t id) const { return id >> shift; }
};
// bin of a one-limb k-mer: the high bits of its fx_hash (src/kmer.jl:255-261 with h = 0: one multiplication)
struct KmerHashBin {
    int shift; // 64 - P
    __device__ __forceinline__ uint32_t operator()(uint64_t kmer) const
    {
        return static_cast<uint32_t>((kmer * 0x517cc1b727220a95ull) >> shift);
    }
};

// bin of a two-limb k-mer: the high bits of the hash that picks its table slot (table_keys.cuh)
struct KmerHashBin2 {
    int shift; // 64 - P
    __device__ __forceinline__ uint32_t operator()(ulonglong2 kmer) const { return static_cast<uint32_t>(key_hash(kmer) >> shift); }
};

// Loads this thread's keys of the iteration starting at it_base: warp w owns the keys [w * 32 * kPerThread,
// + 32 * kPerThread) of the iteration as four rows of one 128-bit vector per lane.  `in` must be 16-byte
// aligned; the tail of the array is loaded key by key (16-byte keys: a row is one key).
template <typename Key>
__device__ __forceinline__ void load_iter(const Key *__restrict__ in, uint64_t n, uint64_t it_base,
                                          Key (&key)[Shape<Key>::kPerThread], uint32_t &ok_mask)
{
    constexpr int V = Shape<Key>::kPerVec, PT = Shape<Key>::kPerThread;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    ok_mask = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const uint64_t e = it_base + static_cast<uint64_t>(warp) * (32 * PT) + r * (32 * V) + lane * V;
        if (e + V <= n) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(in + e));
            if constexpr (sizeof(Key) == 4) {
                key[V * r + 0] = v.x;
                key[V * r + 1] = v.y;
                key[V * r + 2] = v.z;
                key[V * r + 3] = v.w;
            } else if constexpr (sizeof(Key) == 8) {
                key[V * r + 0] = (static_cast<uint64_t>(v.y) << 32) | v.x;
                key[V * r + 1] = (static_cast<uint64_t>(v.w) << 32) | v.z;
            } else {
                key[r] = make_ulonglong2((static_cast<uint64_t>(v.y) << 32) | v.x, (static_cast<uint64_t>(v.w) << 32) | v.z);
            }
            ok_mask |= ((1u << V) - 1u) << (V * r);
        } else if constexpr (V == 1) {
            key[r] = Key{};
        } else {
#pragma unroll
            for (int q = 0; q < V; ++q) {
                const bool ok = e + q < n;
                key[V * r + q] = ok ? __ldg(in + e + q) : Key(0);
                ok_mask |= (ok ? 1u : 0u) << (V * r + q);
            }
        }
    }
}

// ------------------------------------------------------------------------------------ 64 bins
constexpr int kTpBins = 64, kTpGroups = kTpBins / 4;

__device__ __forceinline__ uint32_t tp_count(uint8_t *cnt, uint32_t bin)
{
    uint8_t *c = cnt + (bin >> 2) * (kBlock * 4) + threadIdx.x * 4 + (bin & 3u);
    const uint32_t before = *c;
    *c = static_cast<uint8_t>(before + 1);
    return before;
}

// matrix[bin * n_blocks + block] = number of keys of bin `bin` in the block's chunk
template <typename Key, typename BinOf>
__global__ void __launch_bounds__(kBlock) hist64_kernel(const Key *__restrict__ in, uint64_t n, BinOf bin_of, uint64_t n_blocks,
                                                       uint64_t *__restrict__ matrix)
{
    using S = Shape<Key>;
    __shared__ uint32_t s_cnt[kTpGroups][kBlock];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int g = 0; g < kTpGroups; ++g) s_cnt[g][threadIdx.x] = 0;
    uint8_t *cnt = reinterpret_cast<uint8_t *>(&s_cnt[0][0]);
    const uint64_t base = static_cast<uint64_t>(blockIdx.x) * S::kChunk;
    for (int it = 0; it < kIters; ++it) {
        const uint64_t it_base = base + static_cast<uint64_t>(it) * S::kPerIter;
        if (it_base >= n) break; // block-uniform
        Key key[S::kPerThread];
        uint32_t ok_mask;
        load_iter(in, n, it_base, key, ok_mask);
        if (it_base + S::kPerIter <= n) {
#pragma unroll
            for (int j = 0; j < S::kPerThread; ++j) tp_count(cnt, bin_of(key[j]));
        } else {
#pragma unroll
            for (int j = 0; j < S::kPerThread; ++j)
                if ((ok_mask >> j) & 1u) tp_count(cnt, bin_of(key[j]));
        }
    }
    __syncthreads();
    // warp w sums groups 2w, 2w+1 over the 256 threads (two 16-bit fields per word: a bin total is <= kChunk)
    static_assert(S::kChunk <= 65535, "bin totals are summed in 16-bit fields");
#pragma unroll
    for (int q = 0; q < kTpGroups / kWarps; ++q) {
        const int g = warp * (kTpGroups / kWarps) + q;
        uint32_t lo = 0, hi = 0;
#pragma unroll
        for (int i = 0; i < kBlock / 32; ++i) {
            const uint32_t x = s_cnt[g][lane + 32 * i];
            lo += x & 0x00ff00ffu;
            hi += (x >> 8) & 0x00ff00ffu;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            lo += __shfl_xor_sync(0xffffffffu, lo, d);
            hi += __shfl_xor_sync(0xffffffffu, hi, d);
        }
        if (lane < 4) { // bins 4g + {0: lo.low, 1: hi.low, 2: lo.high, 3: hi.high}
            const uint32_t v = (lane & 1) ? hi : lo;
            matrix[static_cast<uint64_t>(4 * g + lane) * n_blocks + blockIdx.x] = (lane & 2) ? (v >> 16) : (v & 0xffffu);
        }
    }
}

template <typename Key> struct Scatter64Smem {
    uint32_t cnt[kTpGroups][kBlock];      // byte counters, four bins per word
    uint32_t off[kTpGroups * 2][kBlock];  // keys of the bin held by the threads before this one: two 16-bit fields per
                                          // word, bin b in word [(b >> 2) * 2 + (b & 1)], field (b >> 1) & 1
    Key keys[Shape<Key>::kPerIter];
    uint8_t bins[sizeof(Key) >= 8 ? Shape<Key>::kPerIter : 16]; // 64- and 128-bit keys: the bin of every staged key
    uint64_t dst[kTpBins];                // output index of staging slot 0 of each bin (wraps; only sums are used)
    uint64_t glob[kTpBins];               // where the block's next key of each bin goes
    uint32_t start[kTpBins + 1];
    uint32_t tot[kTpBins];
};

// The binned keys are written once and read back much later (or by another kernel): no L1 allocation, first in line for
// eviction from L2 -- so that they do not push out what a kernel running beside this one keeps there (buckets.cu: the table
// slice the increments of the previous piece are working on).
template <typename Key> __device__ __forceinline__ void st_binned(Key *p, Key v)
{
    if constexpr (sizeof(Key) == 4)
        asm volatile("st.global.L1::no_allocate.L2::cache_hint.u32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(0x12F0000000000000ull) : "memory");
    else if constexpr (sizeof(Key) == 8)
        asm volatile("st.global.L1::no_allocate.L2::cache_hint.u64 [%0], %1, %2;" ::"l"(p), "l"(v), "l"(0x12F0000000000000ull) : "memory");
    else
        asm volatile("st.global.L1::no_allocate.L2::cache_hint.v2.u64 [%0], {%1, %2}, %3;" ::"l"(p), "l"(v.x), "l"(v.y),
                     "l"(0x12F0000000000000ull)
                     : "memory");
}

// One iteration of the 64-bin scatter: the block's kPerIter keys (PT per thread, in registers) are counted per bin,
// ranked, staged in shared memory in bin order and written out as one run per bin.  reserve(bin, count), called by the
// lanes of warp 0 for the bins 2 * lane and 2 * lane + 1, returns the index in `out` of the run of `count` keys of `bin`.
// FULL (block-uniform, a template parameter so that the common case carries no per-key tests or branches): all
// kPerIter keys exist; otherwise bit j of ok_mask says whether key[j] does.  Ends without a barrier: the next
// iteration's writes to cnt / off / start / dst are ordered behind this one's reads by its own barriers.
template <typename Key, bool FULL, typename BinOf, typename Reserve>
__device__ __forceinline__ void scatter64_iter(Scatter64Smem<Key> &sm, const Key (&key)[Shape<Key>::kPerThread], uint32_t ok_mask,
                                               BinOf bin_of, Reserve reserve, Key *__restrict__ out)
{
    using S = Shape<Key>;
    constexpr int PT = S::kPerThread;
    static_assert(PT * kBlock == S::kPerIter, "the write-out of a full iteration takes PT keys per thread");
    constexpr bool kStageBins = sizeof(Key) >= 8; // recomputing a hash bin at write-out costs more than a byte of staging
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int g = 0; g < kTpGroups; ++g) sm.cnt[g][threadIdx.x] = 0;
    uint32_t rank[PT / 4], bins[kStageBins ? PT / 4 : 1]; // four byte fields per word (a rank is < PT, a bin < 64)
    uint8_t *cnt = reinterpret_cast<uint8_t *>(&sm.cnt[0][0]);
#pragma unroll
    for (int j = 0; j < PT; ++j) {
        const uint32_t b = bin_of(key[j]);
        uint32_t r = 0;
        if (FULL || ((ok_mask >> j) & 1u)) r = tp_count(cnt, b);
        rank[j / 4] = (j % 4 == 0) ? r : (rank[j / 4] | (r << (8 * (j % 4))));
        if (kStageBins) bins[j / 4] = (j % 4 == 0) ? b : (bins[j / 4] | (b << (8 * (j % 4))));
    }
    __syncthreads();
    // exclusive prefix of every bin's counters over the threads in (lane, warp) order
#pragma unroll
    for (int q = 0; q < kTpGroups / kWarps; ++q) {
        const int g = warp * (kTpGroups / kWarps) + q;
        uint32_t lo[kBlock / 32], hi[kBlock / 32], slo = 0, shi = 0;
#pragma unroll
        for (int i = 0; i < kBlock / 32; ++i) {
            const uint32_t x = sm.cnt[g][lane + 32 * i];
            lo[i] = slo;
            hi[i] = shi;
            slo += x & 0x00ff00ffu;
            shi += (x >> 8) & 0x00ff00ffu;
        }
        uint32_t ilo = slo, ihi = shi;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t a = __shfl_up_sync(0xffffffffu, ilo, d), b = __shfl_up_sync(0xffffffffu, ihi, d);
            if (lane >= d) {
                ilo += a;
                ihi += b;
            }
        }
        const uint32_t blo = ilo - slo, bhi = ihi - shi;
#pragma unroll
        for (int i = 0; i < kBlock / 32; ++i) {
            sm.off[2 * g + 0][lane + 32 * i] = blo + lo[i]; // bins 4g (low field) and 4g + 2 (high field)
            sm.off[2 * g + 1][lane + 32 * i] = bhi + hi[i]; // bins 4g + 1 and 4g + 3
        }
        if (lane == 31) {
            sm.tot[4 * g + 0] = ilo & 0xffffu;
            sm.tot[4 * g + 1] = ihi & 0xffffu;
            sm.tot[4 * g + 2] = ilo >> 16;
            sm.tot[4 * g + 3] = ihi >> 16;
        }
    }
    __syncthreads();
    if (warp == 0) { // exclusive scan of the 64 totals
        const uint32_t t0 = sm.tot[2 * lane], t1 = sm.tot[2 * lane + 1];
        uint32_t incl = t0 + t1;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t a = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += a;
        }
        const uint32_t s0 = incl - t0 - t1, s1 = incl - t1;
        sm.start[2 * lane] = s0;
        sm.start[2 * lane + 1] = s1;
        sm.dst[2 * lane] = reserve(2 * lane, t0) - s0;
        sm.dst[2 * lane + 1] = reserve(2 * lane + 1, t1) - s1;
        if (lane == 31) sm.start[kTpBins] = incl;
    }
    __syncthreads();
    const uint32_t *off_col = &sm.off[0][threadIdx.x];
#pragma unroll
    for (int j = 0; j < PT; ++j) {
        if (FULL || ((ok_mask >> j) & 1u)) {
            const uint32_t b = kStageBins ? ((bins[j / 4] >> (8 * (j % 4))) & 0xffu) : bin_of(key[j]);
            const uint32_t w = off_col[(((b >> 1) & ~1u) | (b & 1u)) * kBlock];
            const uint32_t slot = sm.start[b] + ((w >> ((b & 2u) << 3)) & 0xffffu) + ((rank[j / 4] >> (8 * (j % 4))) & 0xffu);
            sm.keys[slot] = key[j];
            if (kStageBins) sm.bins[slot] = static_cast<uint8_t>(b);
        }
    }
    __syncthreads();
    if (FULL) {
#pragma unroll
        for (int i = 0; i < PT; ++i) {
            const uint32_t t = threadIdx.x + i * kBlock;
            const Key v = sm.keys[t];
            const uint32_t b = kStageBins ? static_cast<uint32_t>(sm.bins[t]) : bin_of(v);
            st_binned(out + (sm.dst[b] + t), v); // (dst wraps; only the sum is used)
        }
    } else {
        const uint32_t total = sm.start[kTpBins];
        for (uint32_t t = threadIdx.x; t < total; t += kBlock) {
            const Key v = sm.keys[t];
            const uint32_t b = kStageBins ? static_cast<uint32_t>(sm.bins[t]) : bin_of(v);
            st_binned(out + (sm.dst[b] + t), v);
        }
    }
}

// out[offs[bin * n_blocks + block] ...) receives the block's keys of bin `bin` (any order within the bin)
template <typename Key, typename BinOf>
__global__ void __launch_bounds__(kBlock, 3) scatter64_kernel(const Key *__restrict__ in, uint64_t n, BinOf bin_of, uint64_t n_blocks,
                                                             const uint64_t *__restrict__ offs, Key *__restrict__ out)
{
    using S = Shape<Key>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Scatter64Smem<Key> &sm = *reinterpret_cast<Scatter64Smem<Key> *>(smem_raw);
    if (threadIdx.x < kTpBins) sm.glob[threadIdx.x] = offs[static_cast<uint64_t>(threadIdx.x) * n_blocks + blockIdx.x];
    const uint64_t base = static_cast<uint64_t>(blockIdx.x) * S::kChunk;
    for (int it = 0; it < kIters; ++it) {
        const uint64_t it_base = base + static_cast<uint64_t>(it) * S::kPerIter;
        if (it_base >= n) break; // block-uniform
        const bool full = it_base + S::kPerIter <= n; // block-uniform: all but the last iteration of the last block
        Key key[S::kPerThread];
        uint32_t ok_mask;
        load_iter(in, n, it_base, key, ok_mask);
        // (sm.glob was filled before the first iteration's barriers; only warp 0 touches it afterwards)
        auto reserve = [&](int b, uint32_t count) {
            const uint64_t g = sm.glob[b];
            sm.glob[b] = g + count;
            return g;
        };
        if (full)
            scatter64_iter<Key, true>(sm, key, ok_mask, bin_of, reserve, out);
        else
            scatter64_iter<Key, false>(sm, key, ok_mask, bin_of, reserve, out);
    }
}

// ------------------------------------------------------------------------------------ 2^P bins, P > 6
template <int P> __device__ __forceinline__ uint32_t bin_peers(uint32_t bin, bool ok)
{
    uint32_t peers = __ballot_sync(0xffffffffu, ok);
#pragma unroll
    for (int b = 0; b < P; ++b) {
        const bool bit = (bin >> b) & 1u;
        const uint32_t set = __ballot_sync(0xffffffffu, bit);
        peers &= bit ? set : ~set;
    }
    return peers;
}

template <int P, typename Key, typename BinOf>
__global__ void __launch_bounds__(kBlock) hist_kernel(const Key *__restrict__ in, uint64_t n, BinOf bin_of, uint64_t n_blocks,
                                                     uint64_t *__restrict__ matrix)
{
    using S = Shape<Key>;
    constexpr int NB = 1 << P;
    __shared__ uint32_t s_cnt[kWarps][NB];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int b = lane; b < NB; b += 32) s_cnt[warp][b] = 0;
    __syncwarp();
    const uint64_t base = static_cast<uint64_t>(blockIdx.x) * S::kChunk;
    for (int it = 0; it < kIters; ++it) {
        const uint64_t it_base = base + static_cast<uint64_t>(it) * S::kPerIter;
        if (it_base >= n) break; // block-uniform
        Key key[S::kPerThread];
        uint32_t ok_mask;
        load_iter(in, n, it_base, key, ok_mask);
#pragma unroll
        for (int j = 0; j < S::kPerThread; ++j) {
            const bool ok = (ok_mask >> j) & 1u;
            const uint32_t bin = bin_of(key[j]);
            const uint32_t peers = bin_peers<P>(bin, ok);
            if (ok && lane == __ffs(peers) - 1) s_cnt[warp][bin] += __popc(peers);
            __syncwarp();
        }
    }
    __syncthreads();
    for (int b = threadIdx.x; b < NB; b += kBlock) {
        uint32_t c = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) c += s_cnt[w][b];
        matrix[static_cast<uint64_t>(b) * n_blocks + blockIdx.x] = c;
    }
}

template <int P, typename Key> struct ScatterSmem {
    uint16_t wcnt[kWarps][1 << P]; // per warp: count, then the warp's offset within the bin
    uint32_t start[(1 << P) + 1];  // first staging slot of each bin in this iteration
    uint64_t glob[1 << P];         // where the block's next key of each bin goes
    Key keys[Shape<Key>::kPerIter];
    uint16_t bins[Shape<Key>::kPerIter];
    uint32_t wsum[kWarps];
};

template <int P, typename Key, typename BinOf>
__global__ void __launch_bounds__(kBlock, 2) scatter_kernel(const Key *__restrict__ in, uint64_t n, BinOf bin_of, uint64_t n_blocks,
                                                           const uint64_t *__restrict__ offs, Key *__restrict__ out)
{
    using S = Shape<Key>;
    constexpr int NB = 1 << P, PT = S::kPerThread;
    constexpr int BPT = (NB + kBlock - 1) / kBlock; // bins per thread in the block scan
    extern __shared__ __align__(16) unsigned char smem_raw[];
    ScatterSmem<P, Key> &sm = *reinterpret_cast<ScatterSmem<P, Key> *>(smem_raw);
    for (int b = threadIdx.x; b < NB; b += kBlock) sm.glob[b] = offs[static_cast<uint64_t>(b) * n_blocks + blockIdx.x];
    const uint64_t base = static_cast<uint64_t>(blockIdx.x) * S::kChunk;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t lt_mask = (1u << lane) - 1u;
    for (int it = 0; it < kIters; ++it) {
        const uint64_t it_base = base + static_cast<uint64_t>(it) * S::kPerIter;
        if (it_base >= n) break; // block-uniform
        for (int b = lane; b < NB; b += 32) sm.wcnt[warp][b] = 0;
        __syncwarp();
        Key key[PT];
        uint32_t ok_mask;
        uint16_t bin[PT], rank[PT];
        load_iter(in, n, it_base, key, ok_mask);
#pragma unroll
        for (int j = 0; j < PT; ++j) {
            const bool ok = (ok_mask >> j) & 1u;
            bin[j] = static_cast<uint16_t>(bin_of(key[j]));
            const uint32_t peers = bin_peers<P>(bin[j], ok);
            const uint32_t before = ok ? sm.wcnt[warp][bin[j]] : 0u;
            rank[j] = static_cast<uint16_t>(before + __popc(peers & lt_mask));
            __syncwarp();
            if (ok && lane == __ffs(peers) - 1) sm.wcnt[warp][bin[j]] = static_cast<uint16_t>(before + __popc(peers));
            __syncwarp();
        }
        __syncthreads();
        // per bin: exclusive prefix over the warps (in place) and the total; exclusive scan of the totals -> start
        {
            uint32_t tot[BPT], sum = 0;
#pragma unroll
            for (int q = 0; q < BPT; ++q) {
                const int b = BPT * threadIdx.x + q;
                uint32_t run = 0;
                if (b < NB) {
#pragma unroll
                    for (int w = 0; w < kWarps; ++w) {
                        const uint32_t c = sm.wcnt[w][b];
                        sm.wcnt[w][b] = static_cast<uint16_t>(run);
                        run += c;
                    }
                }
                tot[q] = run;
                sum += run;
            }
            uint32_t incl = sum;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += t;
            }
            if (lane == 31) sm.wsum[warp] = incl;
            __syncthreads();
            uint32_t run = incl - sum;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) run += (w < warp) ? sm.wsum[w] : 0u;
#pragma unroll
            for (int q = 0; q < BPT; ++q) {
                const int b = BPT * threadIdx.x + q;
                if (b < NB) sm.start[b] = run;
                run += tot[q];
            }
            if (threadIdx.x == kBlock - 1) sm.start[NB] = run;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < PT; ++j) {
            if ((ok_mask >> j) & 1u) {
                const uint32_t slot = sm.start[bin[j]] + sm.wcnt[warp][bin[j]] + rank[j];
                sm.keys[slot] = key[j];
                sm.bins[slot] = bin[j];
            }
        }
        __syncthreads();
        const uint32_t total = sm.start[NB];
        for (uint32_t t = threadIdx.x; t < total; t += kBlock) {
            const uint32_t b = sm.bins[t];
            out[sm.glob[b] + (t - sm.start[b])] = sm.keys[t];
        }
        __syncthreads();
        for (int b = threadIdx.x; b < NB; b += kBlock) sm.glob[b] += sm.start[b + 1] - sm.start[b];
        // the next iteration's writes to wcnt / start / keys are ordered behind this by its barriers
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------ host side
// cells of the count matrix (and of its scan) for n keys in 2^p bins
template <typename Key> inline uint64_t matrix_cells(uint64_t n, int p) { return (static_cast<uint64_t>(1) << p) * blocks_for<Key>(n); }

// Partitions in[0..n) into 2^p bins by bin_of.  Afterwards the keys of bin b are
// out[offs[b * n_blocks] .. offs[(b + 1) * n_blocks]) with n_blocks = blocks_for<Key>(n).
// matrix / offs: matrix_cells + 1 (+ 2) u64; scan_tmp: scan_tmp_elems(matrix_cells) u64.  in / out 16-byte aligned.
template <typename Key, typename BinOf>
cudaError_t partition(const Key *in, uint64_t n, int p, BinOf bin_of, Key *out, uint64_t *matrix, uint64_t *offs, uint64_t *scan_tmp,
                      cudaStream_t stream)
{
    if (n == 0) return cudaSuccess;
    if (p < kMinBits || p > kMaxBits) return cudaErrorInvalidValue;
    const uint64_t n_blocks = blocks_for<Key>(n);
    if (n_blocks > 0x7fffffffull) return cudaErrorInvalidConfiguration;
    const unsigned grid = static_cast<unsigned>(n_blocks);
    const uint64_t cells = matrix_cells<Key>(n, p);
    if (p == 6) {
        constexpr int smem = static_cast<int>(sizeof(Scatter64Smem<Key>));
        cudaError_t e = cudaFuncSetAttribute(scatter64_kernel<Key, BinOf>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        hist64_kernel<Key, BinOf><<<grid, kBlock, 0, stream>>>(in, n, bin_of, n_blocks, matrix);
        e = inclusive_offsets_u64(matrix, offs, cells, scan_tmp, stream);
        if (e != cudaSuccess) return e;
        scatter64_kernel<Key, BinOf><<<grid, kBlock, smem, stream>>>(in, n, bin_of, n_blocks, offs, out);
        return cudaGetLastError();
    }
    auto run = [&](auto tag) -> cudaError_t {
        constexpr int P = decltype(tag)::value;
        constexpr int smem = static_cast<int>(sizeof(ScatterSmem<P, Key>));
        cudaError_t e = cudaFuncSetAttribute(scatter_kernel<P, Key, BinOf>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        hist_kernel<P, Key, BinOf><<<grid, kBlock, 0, stream>>>(in, n, bin_of, n_blocks, matrix);
        e = inclusive_offsets_u64(matrix, offs, cells, scan_tmp, stream);
        if (e != cudaSuccess) return e;
        scatter_kernel<P, Key, BinOf><<<grid, kBlock, smem, stream>>>(in, n, bin_of, n_blocks, offs, out);
        return cudaGetLastError();
    };
    switch (p) {
    case 7: return run(std::integral_constant<int, 7>());
    case 8: return run(std::integral_constant<int, 8>());
    case 9: return run(std::integral_constant<int, 9>());
    default: return run(std::integral_constant<int, 10>());
    }
}

// The binned path of a table too large for L2: one key per update is written out, the keys are partitioned by table slice,
// and the slices are walked in groups, each group pulled into L2 and then given its keys.
//
// A table of up to kL2Budget bytes is updated directly: it stays in L2 (126 MB) beside the stream that updates it.
constexpr uint64_t kL2Budget = 96ull << 20;

// Table slice per bin: 2^22 counters = 16 MB of bucket table; 2^20 slots = 12 MB of one-limb, 20 MB of two-limb k-mer table.
constexpr int kBucketSliceBits = 22, kKmerSliceBits = 20;

// log2 of the bins of a table of 2^table_bits entries in slices of at most 2^slice_bits entries
inline int bin_bits(int table_bits, int slice_bits)
{
    const int p = table_bits - slice_bits;
    return p < kMinBits ? kMinBits : (p > kMaxBits ? kMaxBits : p);
}

// Bins applied per launch.  Measured on a B200: the bucket table (16 MB slices, increments) is fastest with 2 bins = 32 MB
// per launch (1: +1 %, 4: +6 %, 8 = 128 MB: 2x slower -- the slices no longer fit L2); the one-limb k-mer table (12 MB
// slices, a load and an increment per k-mer) keeps improving up to 8 bins = 96 MB (1: 10.7 ms, 2: 9.8, 4: 9.6, 8: 9.3 ms
// per 480 M k-mers); 6 leaves room for the k-mer stream itself.  The two-limb table takes 3 bins = 60 MB.
constexpr int kBucketGroup = 2;
constexpr int kmer_group(int n_limbs) { return n_limbs == 1 ? 6 : 3; }

// The temporaries of the binned path for up to n keys in 2^p bins: the keys as they are written (one per flat window),
// the binned keys, the count matrix, its offsets and the scan scratch.  Stream-ordered, freed when this goes out of scope.
template <typename Key> struct BinnedKeys {
    AsyncBuf written, binned, matrix, offs, scan;
    int p = 0;
    uint64_t n_blocks = 0; // of the last partition: the keys of bin b are binned[offs[b * n_blocks] .. offs[(b + 1) * n_blocks])

    // false when the memory is not there (the CUDA error is cleared): the caller then updates the table directly
    bool alloc(kmc_ctx *ctx, uint64_t n, int bits, cudaStream_t stream)
    {
        p = bits;
        const uint64_t key_bytes = (n * sizeof(Key) + 255) / 256 * 256, cells = matrix_cells<Key>(n, p);
        cudaError_t e = written.alloc(ctx, key_bytes, stream);
        if (e == cudaSuccess) e = binned.alloc(ctx, key_bytes, stream);
        if (e == cudaSuccess) e = matrix.alloc(ctx, (cells + 1) * 8, stream);
        if (e == cudaSuccess) e = offs.alloc(ctx, (cells + 2) * 8, stream);
        if (e == cudaSuccess) e = scan.alloc(ctx, (scan_tmp_elems(cells) + 1) * 8, stream);
        if (e != cudaSuccess) (void)cudaGetLastError();
        return e == cudaSuccess;
    }

    // bins the first n written keys by bin_of
    template <typename BinOf> cudaError_t partition(uint64_t n, BinOf bin_of, cudaStream_t stream)
    {
        n_blocks = blocks_for<Key>(n);
        return binning::partition<Key>(written.as<Key>(), n, p, bin_of, binned.as<Key>(), matrix.as<uint64_t>(), offs.as<uint64_t>(),
                                       scan.as<uint64_t>(), stream);
    }
};

// Walks the bins [0, n_bins) in groups of `group`: apply(bin, bin_end) enqueues the warm-ups of the group's table slices and
// the kernel that applies its keys.  events (may be NULL): events[i] is recorded once the i-th of n_parts equal ranges of
// the table is final, i.e. once the bins [i * n_bins / n_parts, (i + 1) * n_bins / n_parts) are applied.
template <typename Apply>
cudaError_t apply_groups(int n_bins, int group, uint32_t n_parts, void *const *events, cudaStream_t stream, Apply apply)
{
    if (!events) n_parts = 0;
    uint32_t parts_done = 0;
    for (int b = 0; b < n_bins; b += group) {
        const int b_end = b + group < n_bins ? b + group : n_bins;
        cudaError_t e = apply(b, b_end);
        if (e != cudaSuccess) return e;
        while (parts_done < n_parts && static_cast<uint64_t>(parts_done + 1) * n_bins <= static_cast<uint64_t>(b_end) * n_parts) {
            e = cudaEventRecord(static_cast<cudaEvent_t>(events[parts_done++]), stream);
            if (e != cudaSuccess) return e;
        }
    }
    return cudaGetLastError();
}

} // namespace binning
} // namespace kmc
