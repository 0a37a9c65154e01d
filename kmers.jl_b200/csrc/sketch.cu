// sketch.cu -- consumers of the k-mer stream that never write it (SURVEY.md 8f ranks 2 and 4):
//
//   kmc_minhash_sketch  bottom-s MinHash sketch under fx_hash -- the reference's example
//                       `sketch(fx_hash, CanonicalDNAMers{16}(seq), 1000)` (docs/src/minhash.md:31-36;
//                       MinHash.jl is not vendored: the published bottom-s definition is restated --
//                       the s smallest DISTINCT hash values over all k-mers, ascending)
//   kmc_minhash_sketch_each  the same sketch of every sequence of the set on its own, in one call (per-sequence hash
//                       limits, candidates in per-sequence segments, cub's segmented sort; kmc_minhash_compare
//                       compares the rows, compare.cu)
//   kmc_composition     k-mer composition vector -- `counts[as_integer(kmer) + 1] += 1` over
//                       FwDNAMers{K} (docs/src/composition.md:28-39), K <= 14
//   kmc_kmer_count      exact k-mer counts keyed by the k-mer itself (the `Dict{Kmer,Int}` a user of the
//                       iterators builds; CanonicalKmers.jl:183-185 on counting), K <= 32: an
//                       open-addressing table in device memory (fx_hash of the k-mer picks the slot,
//                       linear probing, 64-bit compare-and-swap on the key, 32-bit add on the count);
//                       kmc_kmer_table_merge / _export move entries between tables (multi-GPU merge)
//   kmc_kmer_count2     the same table for two-limb k-mers, K = 33..64 (table_keys.cuh): 16-byte keys, claimed by
//                       one 128-bit compare-and-swap; kmc_kmer_table2_merge / _export
//   kmc_kmer_lookup(2)  read-only queries of a counted table: the count of every window of a read set (in
//                       kmc_extract's order), of a list of keys (_get), the count spectrum (_histogram) and the
//                       keys whose count lies in a range (_export_range)
//
// Both run consume_kernel: the same (read, group slot) work items, block load and static funnel
// shifts as extract_kernel (kmer_core.cuh), with the stores replaced by a small functor.
//
// Sketch: (1) histogram of the top 12 hash bits (4096 counters: every block counts in shared memory
// and adds its non-zero counters to the global table once), (2) the host picks the smallest
// threshold bucket t whose cumulative count reaches s (control logic over 4096 integers), (3) a second pass appends every hash whose top bits are <= t to a candidate array
// sized exactly by the histogram, (4) the candidates -- s plus at most one bucket's worth -- are
// sorted and deduplicated on the device (cub radix sort + unique: library plumbing on a tiny
// array), and if duplicates left fewer than s distinct values the threshold moves up and (3)-(4)
// repeat.  The k-mers are read twice (2 x 0.25 B/symbol) and nothing proportional to them is written.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_segmented_sort.cuh>
#include <cub/device/device_select.cuh>

#include <algorithm>
#include <vector>

#include "binning.cuh"
#include "plan.h"
#include "table_keys.cuh"

namespace kmc {

namespace {

enum : int {
    OP_HASH_HIST = 0,
    OP_HASH_BELOW = 1,
    OP_COMPOSITION = 2,
    OP_COMPOSITION_SHARED = 3,
    OP_TABLE = 4,
    OP_TABLE2 = 5,
    OP_LOOKUP = 6,
    OP_LOOKUP2 = 7,
    OP_SKETCH_COUNT = 8,
    OP_SKETCH_APPEND = 9
};

// kEmptyKey (table_keys.cuh) is never a k-mer: one limb, K <= 31, or K = 32 canonical (the all-T 32-mer is not
// canonical); two limbs {~0, ~0}, K <= 63, or K = 64 canonical.

// table[key] += inc.  Returns kTableFull when no slot is left, kTableNew when the key was not in the table
// before.  Most k-mers of a read set are already in the table, so the slot is read before the
// compare-and-swap is attempted.
enum : int { kTableFull = 0, kTableCounted = 1, kTableNew = 2 };

__device__ __forceinline__ int table_add(unsigned long long *keys, uint32_t *vals, uint32_t log2cap, uint64_t key, uint64_t hash,
                                         uint32_t inc)
{
    const uint64_t mask = (1ull << log2cap) - 1;
    uint64_t slot = hash >> (64 - log2cap);
    for (uint64_t probes = 0; probes <= mask; ++probes) {
        unsigned long long cur = keys[slot];
        int st = kTableCounted;
        if (cur == kEmptyKey) {
            cur = atomicCAS(keys + slot, kEmptyKey, static_cast<unsigned long long>(key));
            if (cur == kEmptyKey) {
                st = kTableNew;
                cur = key;
            }
        }
        if (cur == key) {
            atomicAdd(vals + slot, inc);
            return st;
        }
        slot = (slot + 1) & mask;
    }
    return kTableFull;
}

// The same for a two-limb key.  The slot is read with one 16-byte load, but a vector load is not promised to be
// single-copy atomic: a slot being claimed could be seen half written, and a half-written slot has a limb that is
// still ~0.  So a slot with any ~0 limb is read again through the compare-and-swap itself, which claims it if it is
// free and returns its true content otherwise (keys whose limbs are ~0 -- the all-T tail of a k-mer -- are rare).
__device__ __forceinline__ int table_add(ulonglong2 *keys, uint32_t *vals, uint32_t log2cap, ulonglong2 key, uint64_t hash,
                                         uint32_t inc)
{
    const uint64_t mask = (1ull << log2cap) - 1;
    const ulonglong2 empty = make_ulonglong2(kEmptyKey, kEmptyKey);
    uint64_t slot = hash >> (64 - log2cap);
    for (uint64_t probes = 0; probes <= mask; ++probes) {
        ulonglong2 cur = keys[slot];
        int st = kTableCounted;
        if (cur.x == kEmptyKey || cur.y == kEmptyKey) {
            cur = atomicCAS(keys + slot, empty, key);
            if (key_free(cur)) {
                st = kTableNew;
                cur = key;
            }
        }
        if (cur.x == key.x && cur.y == key.y) {
            atomicAdd(vals + slot, inc);
            return st;
        }
        slot = (slot + 1) & mask;
    }
    return kTableFull;
}

// table[key], 0 for a key that is not in the table: the probe of table_add without its atomics.  Precondition: no
// count or merge into the same table is in flight (calls on one context are stream ordered), so a two-limb slot read
// by one 16-byte load is never half written.  A full table that lacks the key ends after 2^log2cap probes.
template <typename Key>
__device__ __forceinline__ uint32_t table_find(const Key *__restrict__ keys, const uint32_t *__restrict__ vals, uint32_t log2cap,
                                               Key key, uint64_t hash)
{
    const uint64_t mask = (1ull << log2cap) - 1;
    uint64_t slot = hash >> (64 - log2cap);
    for (uint64_t probes = 0; probes <= mask; ++probes) {
        const Key cur = keys[slot];
        if (key_free(cur)) return 0;
        if (key_equal(cur, key)) return vals[slot];
        slot = (slot + 1) & mask;
    }
    return 0;
}

// adds the new keys a thread has seen to *distinct: one atomic per warp (all 32 lanes must call)
__device__ __forceinline__ void add_distinct(unsigned long long *distinct, uint32_t n_new)
{
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) n_new += __shfl_xor_sync(0xffffffffu, n_new, d);
    if ((threadIdx.x & 31) == 0 && n_new) atomicAdd(distinct, static_cast<unsigned long long>(n_new));
}

struct ConsumeParams {
    uint32_t *table;               // OP_HASH_HIST: u32[2^12]; OP_COMPOSITION*: u32[4^K]
    uint32_t shift;                // OP_HASH_HIST / OP_HASH_BELOW: 64 - bits
    uint64_t limit;                // OP_HASH_BELOW: keep h <= limit
    uint64_t *cand;                // OP_HASH_BELOW: candidate array
    unsigned long long *cursor;    // OP_HASH_BELOW: elements appended so far
    uint64_t cand_cap;
    uint32_t table_entries;        // OP_HASH_HIST, OP_COMPOSITION_SHARED: counters kept in shared memory
    unsigned long long *keys;      // OP_TABLE: u64[2^log2cap] keys (kEmptyKey = free), vals = table
    uint32_t log2cap;
    unsigned long long *distinct;  // OP_TABLE: keys in the table
    uint32_t *overflow;            // OP_TABLE*: set when a k-mer found no slot
    ulonglong2 *keys2;             // OP_TABLE2: two-limb keys, ulonglong2[2^log2cap] ({~0, ~0} = free), vals = table
    uint32_t *out_counts;          // OP_LOOKUP*: u32 per window, at its flat window index (kmc_extract's order)
    const uint64_t *seq_lim;       // OP_SKETCH_*: per sequence, keep h < lim (~0: every k-mer; 0: skip the sequence)
    unsigned long long *seq_cnt;   // OP_SKETCH_COUNT: candidates per sequence
    unsigned long long *seq_cursor; // OP_SKETCH_APPEND: next free candidate slot of each sequence (starts at its offset)
};

constexpr int kSharedCompositionMax = 4096; // 4^6 counters = 16 KB of shared memory
constexpr int kSketchBits = 12;             // top hash bits of the sketch histogram (also kept in shared memory)
static_assert((1 << kSketchBits) <= kSharedCompositionMax, "the sketch histogram lives in the same shared array");

// ALIGNED: the work items of an aligned uniform set or of a single sequence (extract_kernels.cuh: AlignedItems) -- no
// cursor, one bounds test per tile, every slot a window except in the last group of a single sequence.
template <int N, int NX, bool RAGGED, bool CANON, int OP, bool ALIGNED = false>
__global__ void __launch_bounds__(kBlockThreads) consume_kernel(const ExtractParams p, const ConsumeParams c)
{
    static_assert(!(ALIGNED && RAGGED), "aligned sets are uniform");
    constexpr int G = GroupOf<N>::G;
    __shared__ TileShared<RAGGED> sh;
    constexpr bool SHARED_HIST = (OP == OP_COMPOSITION_SHARED || OP == OP_HASH_HIST);
    constexpr bool LOOKUP = (OP == OP_LOOKUP || OP == OP_LOOKUP2);
    constexpr bool SKETCH = (OP == OP_SKETCH_COUNT || OP == OP_SKETCH_APPEND);
    __shared__ uint32_t s_hist[SHARED_HIST ? kSharedCompositionMax : 1];
    const uint64_t tile_base = static_cast<uint64_t>(blockIdx.x) * kTileItems;
    if (SHARED_HIST) {
        for (uint32_t i = threadIdx.x; i < c.table_entries; i += kBlockThreads) s_hist[i] = 0;
    }
    TileCursor<RAGGED, G> cur;
    if (!ALIGNED) cur.init(p, tile_base, sh, threadIdx.x); // (block-wide barriers inside: also orders the zeroing above)
    if (SHARED_HIST) __syncthreads();
    uint32_t n_new = 0; // OP_TABLE*: keys this thread put into the table
    const AlignedItems<G, 2> items(p);
    const uint32_t n_items32 = static_cast<uint32_t>(p.items);
    bool inside = false;
    if (ALIGNED) {
        const uint32_t tb = static_cast<uint32_t>(tile_base);
        const uint32_t tile_last = (n_items32 - tb > static_cast<uint32_t>(kTileItems) ? tb + kTileItems : n_items32) - 1u;
        inside = items.template loads_inside<NX>(p, tile_last);
    }

#pragma unroll 1
    for (int it = 0; it < kTileIters; ++it) {
        const uint32_t li = static_cast<uint32_t>(it) * kBlockThreads + threadIdx.x;
        const uint64_t item = tile_base + li;
        if (item >= p.items) break;
        int jlo, jhi;
        uint32_t x[NX];
        uint64_t seq = 0, lim = 0; // OP_SKETCH_*: the item's sequence and its limit (0: skipped this round)
        if (ALIGNED) {
            jlo = 0;
            jhi = (p.al_tail != 0 && static_cast<uint32_t>(item) == n_items32 - 1u) ? static_cast<int>(p.al_tail) : G;
            if constexpr (SKETCH) {
                seq = items.read_of(static_cast<uint32_t>(item));
                lim = __ldg(c.seq_lim + seq);
                if (lim == 0) jhi = 0;
            }
            load_block_at<NX>(p, items.bit_of(static_cast<uint32_t>(item)), inside, x);
        } else {
            cur.locate(p, item, li, sh);
            jlo = cur.jlo;
            jhi = cur.jhi;
            if constexpr (SKETCH) {
                seq = cur.r;
                lim = __ldg(c.seq_lim + seq);
                if (lim == 0) jhi = jlo;
            }
            if (jhi > jlo) load_block<NX>(p.w32, p.nw32, cur.bit(p), x);
        }
        if (jhi > jlo) {
            uint64_t fw[G][N], rv[G][N];
            block_kmers<N, NX, G, true, CANON>(x, p.s0, p.head_mask, fw, rv);
            uint32_t found[LOOKUP ? G : 1]; // OP_LOOKUP*: the counts of the item's windows [jlo, jhi)
            uint64_t hs[OP == OP_SKETCH_APPEND ? G : 1]; // OP_SKETCH_APPEND: the hashes of the windows
            uint32_t take = 0;                            // OP_SKETCH_*: bit j = window j is a candidate
#pragma unroll
            for (int j = 0; j < G; ++j) {
                if (j < jlo || j >= jhi) continue;
                bool take_fw = true;
                if (CANON) take_fw = limbs_less<N>(fw[j], rv[j]);
                uint64_t a[N];
#pragma unroll
                for (int i = 0; i < N; ++i) a[i] = take_fw ? fw[j][i] : rv[j][i];
                if constexpr (OP == OP_LOOKUP) {
                    found[j] = table_find<unsigned long long>(c.keys, c.table, c.log2cap, a[N - 1], fx_hash<N>(a, 0));
                    continue;
                } else if constexpr (OP == OP_LOOKUP2) {
                    const ulonglong2 key = make_ulonglong2(a[0], a[N - 1]);
                    found[j] = table_find(c.keys2, c.table, c.log2cap, key, key_hash(key));
                    continue;
                } else if constexpr (SKETCH) {
                    const uint64_t h = fx_hash<N>(a, 0);
                    if (h < lim || lim == ~0ull) take |= 1u << j;
                    if constexpr (OP == OP_SKETCH_APPEND) hs[j] = h;
                    continue;
                }
                if (OP == OP_HASH_HIST) {
                    atomicAdd(s_hist + (fx_hash<N>(a, 0) >> c.shift), 1u);
                } else if (OP == OP_HASH_BELOW) {
                    const uint64_t h = fx_hash<N>(a, 0);
                    if (h <= c.limit) {
                        const unsigned long long at = atomicAdd(c.cursor, 1ull);
                        if (at < c.cand_cap) c.cand[at] = h;
                    }
                } else if (OP == OP_TABLE) {
                    const int st = table_add(c.keys, c.table, c.log2cap, a[N - 1], fx_hash<N>(a, 0), 1u);
                    if (st == kTableFull) *c.overflow = 1u;
                    n_new += st == kTableNew;
                } else if (OP == OP_TABLE2) {
                    const ulonglong2 key = make_ulonglong2(a[0], a[N - 1]);
                    const int st = table_add(c.keys2, c.table, c.log2cap, key, key_hash(key), 1u);
                    if (st == kTableFull) *c.overflow = 1u;
                    n_new += st == kTableNew;
                } else if (OP == OP_COMPOSITION) {
                    atomicAdd(c.table + a[N - 1], 1u); // as_integer(kmer): K <= 14, one limb
                } else {
                    atomicAdd(s_hist + a[N - 1], 1u);
                }
            }
            if constexpr (SKETCH) {
                // The lanes of a warp that hold candidates of one sequence add them with one atomic: the counts (<= G)
                // are summed bit by bit over the lanes of the same sequence (__match_any_sync), and the appending
                // lanes write at their prefix from the base the first of them reserved.
                const uint32_t active = __activemask();
                if (__any_sync(active, take != 0)) {
                    constexpr int kCountBits = G >= 8 ? 4 : G >= 4 ? 3 : G >= 2 ? 2 : 1;
                    static_assert(G < 16, "a lane's candidate count fits kCountBits bits");
                    const uint32_t lane = threadIdx.x & 31;
                    const uint32_t peers = __match_any_sync(active, static_cast<unsigned long long>(seq));
                    const int leader = __ffs(peers) - 1;
                    const uint32_t n_take = __popc(take), lower = peers & ((1u << lane) - 1u);
                    uint32_t total = 0, before = 0;
#pragma unroll
                    for (int b = 0; b < kCountBits; ++b) {
                        const uint32_t m = __ballot_sync(active, (n_take >> b) & 1u) & peers;
                        total += static_cast<uint32_t>(__popc(m)) << b;
                        before += static_cast<uint32_t>(__popc(m & lower)) << b;
                    }
                    if constexpr (OP == OP_SKETCH_COUNT) {
                        if (static_cast<int>(lane) == leader && total) atomicAdd(c.seq_cnt + seq, static_cast<unsigned long long>(total));
                    } else {
                        unsigned long long base = 0;
                        if (static_cast<int>(lane) == leader && total) base = atomicAdd(c.seq_cursor + seq, static_cast<unsigned long long>(total));
                        uint64_t at = __shfl_sync(active, base, leader) + before;
#pragma unroll
                        for (int j = 0; j < G; ++j)
                            if ((take >> j) & 1u) c.cand[at++] = hs[j];
                    }
                }
            }
            if constexpr (LOOKUP) {
                // a whole group is 4 G bytes at a multiple of 4 G: one vector store when the base allows it (p.vec_ok)
                uint32_t *dst = c.out_counts + (ALIGNED ? item : cur.q) * G;
                if (jlo == 0 && jhi == G && p.vec_ok && (G == 8 || G == 4)) {
                    uint64_t w[G / 2];
#pragma unroll
                    for (int t = 0; t < G / 2; ++t) w[t] = found[2 * t] | (static_cast<uint64_t>(found[2 * t + 1]) << 32);
                    if (G == 8) st_v4(reinterpret_cast<uint64_t *>(dst), w[0], w[1 % (G / 2)], w[2 % (G / 2)], w[3 % (G / 2)]);
                    else st_v2(reinterpret_cast<uint64_t *>(dst), w[0], w[1 % (G / 2)]);
                } else {
#pragma unroll
                    for (int j = 0; j < G; ++j)
                        if (j >= jlo && j < jhi) dst[j] = found[j];
                }
            }
        }
        if (!ALIGNED) cur.advance(p);
    }
    if (OP == OP_TABLE || OP == OP_TABLE2) add_distinct(c.distinct, n_new);
    if (SHARED_HIST) {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < c.table_entries; i += kBlockThreads) {
            const uint32_t v = s_hist[i];
            if (v) atomicAdd(c.table + i, v);
        }
    }
}

using ConsumeLaunchFn = cudaError_t (*)(ExtractParams, ConsumeParams, cudaStream_t);

template <int N, int NX, bool RAGGED, bool CANON, int OP>
cudaError_t launch_consume(ExtractParams p, ConsumeParams c, cudaStream_t stream)
{
    const uint64_t tiles = (p.items + kTileItems - 1) / kTileItems;
    if (tiles == 0) return cudaSuccess;
    if (tiles > 0x7fffffffull) return cudaErrorInvalidConfiguration;
    set_iteration_strides(p, RAGGED ? 0 : GroupOf<N>::G);
    if constexpr (!RAGGED) {
        if (p.aligned && !p.items_dev && p.gprm < 0x80000000ull && p.items < 0xffffffffull - kTileItems && aligned_kernel_enabled()) {
            p.al_magic = aligned_magic(p.gprm);
            consume_kernel<N, NX, false, CANON, OP, true><<<static_cast<unsigned>(tiles), kBlockThreads, 0, stream>>>(p, c);
            return cudaGetLastError();
        }
        p.aligned = 0; // the general locator below must not take its aligned fast path for a partial tail it cannot see
        p.al_tail = 0;
    }
    consume_kernel<N, NX, RAGGED, CANON, OP><<<static_cast<unsigned>(tiles), kBlockThreads, 0, stream>>>(p, c);
    return cudaGetLastError();
}

template <int N, int NX, int OP>
ConsumeLaunchFn pick_consume(bool ragged, bool canon)
{
    if (ragged) return canon ? &launch_consume<N, NX, true, true, OP> : &launch_consume<N, NX, true, false, OP>;
    return canon ? &launch_consume<N, NX, false, true, OP> : &launch_consume<N, NX, false, false, OP>;
}

template <int N, int OP>
ConsumeLaunchFn pick_consume_nx(int nx, bool ragged, bool canon)
{
    constexpr int NXMAX = (64 * N + 2 * GroupOf<N>::G - 2 + 31) / 32;
    if (nx == NXMAX) return pick_consume<N, NXMAX, OP>(ragged, canon);
    if (nx == NXMAX - 1) return pick_consume<N, (NXMAX - 1 > 0 ? NXMAX - 1 : 1), OP>(ragged, canon);
    if (nx == NXMAX - 2) return pick_consume<N, (NXMAX - 2 > 0 ? NXMAX - 2 : 1), OP>(ragged, canon);
    return nullptr;
}

template <int OP>
ConsumeLaunchFn consume_launcher(const Geometry &ge, bool ragged, bool canon)
{
    switch (ge.n_limbs) {
    case 1: return pick_consume_nx<1, OP>(ge.nx, ragged, canon);
    case 2: return pick_consume_nx<2, OP>(ge.nx, ragged, canon);
    }
    return nullptr;
}

// every non-empty (key, count) of a source table / entry list into the destination table
// (Key: unsigned long long for one-limb tables, ulonglong2 for two-limb ones)
template <typename Key>
__global__ void __launch_bounds__(256) table_merge_kernel(Key *keys, uint32_t *vals, uint32_t log2cap, const Key *__restrict__ src_keys,
                                                          const uint32_t *__restrict__ src_vals, uint64_t n,
                                                          unsigned long long *distinct, uint32_t *overflow)
{
    uint32_t n_new = 0;
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const Key key = src_keys[i];
        if (key_free(key)) continue;
        const int st = table_add(keys, vals, log2cap, key, key_hash(key), src_vals[i]);
        if (st == kTableFull) *overflow = 1u;
        n_new += st == kTableNew;
    }
    add_distinct(distinct, n_new);
}

// Tables beyond L2: an insertion that misses L2 waits for DRAM (13.9 G k-mers/s measured against 123 G/s on an
// L2-resident table).  So the k-mers are written out, partitioned by the high bits of their slot (binning.cuh)
// and inserted slice after slice, each slice pulled into L2 first.  The k-mers of bin `bin` are
// binned[offs[bin * n_blocks] .. offs[(bin + 1) * n_blocks]); one launch inserts the bins [bin, bin_end).
template <typename Key>
__global__ void __launch_bounds__(256) bin_insert_kernel(const Key *__restrict__ binned, const uint64_t *__restrict__ offs,
                                                         uint64_t n_blocks, int bin, int bin_end, Key *keys, uint32_t *vals,
                                                         uint32_t log2cap, unsigned long long *distinct, uint32_t *overflow)
{
    const uint64_t begin = __ldg(offs + static_cast<uint64_t>(bin) * n_blocks);
    const uint64_t end = __ldg(offs + static_cast<uint64_t>(bin_end) * n_blocks);
    uint32_t n_new = 0;
    for (uint64_t i = begin + static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < end;
         i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const Key key = __ldg(binned + i);
        const int st = table_add(keys, vals, log2cap, key, key_hash(key), 1u);
        if (st == kTableFull) *overflow = 1u;
        n_new += st == kTableNew;
    }
    add_distinct(distinct, n_new);
}

// RANGE: only the entries with min_count <= count <= max_count
template <typename Key, bool RANGE = false>
__global__ void __launch_bounds__(256) table_export_kernel(const Key *__restrict__ keys, const uint32_t *__restrict__ vals,
                                                           uint64_t n_slots, Key *__restrict__ out_keys,
                                                           uint32_t *__restrict__ out_vals, uint64_t capacity,
                                                           unsigned long long *cursor, uint32_t min_count = 0,
                                                           uint32_t max_count = ~0u)
{
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_slots;
         i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const Key key = keys[i];
        if (key_free(key)) continue;
        if (RANGE && (vals[i] < min_count || vals[i] > max_count)) continue;
        const uint32_t active = __activemask(); // warp-aggregated append: one atomic per converged group
        const int leader = __ffs(active) - 1;
        unsigned long long base = 0;
        if ((threadIdx.x & 31) == leader) base = atomicAdd(cursor, static_cast<unsigned long long>(__popc(active)));
        base = __shfl_sync(active, base, leader);
        const uint64_t at = base + __popc(active & ((1u << (threadIdx.x & 31)) - 1u));
        if (at < capacity) {
            out_keys[at] = key;
            out_vals[at] = vals[i];
        }
    }
}

// out[i] = table[query[i]], 0 for a key that is not in the table
template <typename Key>
__global__ void __launch_bounds__(256) table_get_kernel(const Key *__restrict__ keys, const uint32_t *__restrict__ vals, uint32_t log2cap,
                                                        const Key *__restrict__ query, uint64_t n, uint32_t *__restrict__ out)
{
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const Key key = query[i];
        out[i] = table_find(keys, vals, log2cap, key, key_hash(key));
    }
}

// The count spectrum: hist[min(count, n_bins - 1)] += 1 for every key of the table.  Each block counts into n_bins
// shared counters (dynamic shared memory) and adds its non-zero bins once.  Most keys of a read set share a few small
// counts, so the lanes of a warp that fall into one bin add together (one shared atomic per distinct bin).  A thread
// loads kHistUnroll slots before it counts any, to keep enough loads in flight for a pass bound by HBM.
constexpr int kHistUnroll = 4;

template <typename Key>
__global__ void __launch_bounds__(256) table_histogram_kernel(const Key *__restrict__ keys, const uint32_t *__restrict__ vals,
                                                              uint64_t n_slots, unsigned long long *hist, uint32_t n_bins)
{
    extern __shared__ uint32_t s_bins[];
    for (uint32_t b = threadIdx.x; b < n_bins; b += blockDim.x) s_bins[b] = 0;
    __syncthreads();
    const uint64_t step = static_cast<uint64_t>(gridDim.x) * blockDim.x * kHistUnroll;
    for (uint64_t base = static_cast<uint64_t>(blockIdx.x) * blockDim.x * kHistUnroll + threadIdx.x; base < n_slots; base += step) {
        uint32_t bin[kHistUnroll];
#pragma unroll
        for (int u = 0; u < kHistUnroll; ++u) {
            const uint64_t i = base + static_cast<uint64_t>(u) * blockDim.x;
            const bool inside = i < n_slots;
            const Key key = inside ? keys[i] : Key{};
            const uint32_t val = inside ? vals[i] : 0u;
            bin[u] = inside && !key_free(key) ? min(val, n_bins - 1) : ~0u; // ~0: no key
        }
        const uint32_t active = __activemask();
#pragma unroll
        for (int u = 0; u < kHistUnroll; ++u) {
            const uint32_t peers = __match_any_sync(active, bin[u]);
            if (bin[u] != ~0u && (threadIdx.x & 31) == static_cast<unsigned>(__ffs(peers) - 1)) atomicAdd(s_bins + bin[u], __popc(peers));
        }
    }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < n_bins; b += blockDim.x)
        if (s_bins[b]) atomicAdd(hist + b, static_cast<unsigned long long>(s_bins[b]));
}

// ---- a bottom-s sketch per sequence (kmc_minhash_sketch_each) ----------------------------------------------------
// The first limit of each sequence: every k-mer when its windows are few against s, otherwise the hash below which
// s + 4 sqrt(s) + 16 of its windows are expected (windows hash uniformly), so that distinct k-mers below it fall short of
// s only when repeats remove that margin -- and the retry catches those.  No windows: an empty row, no candidates.
__global__ void sketch_limits_kernel(const uint64_t *__restrict__ win_off, uint64_t wpr, uint64_t n, uint64_t s,
                                     uint64_t *__restrict__ lim)
{
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const uint64_t w = win_off ? win_off[i + 1] - win_off[i] : wpr;
        const double want = static_cast<double>(s) + 4.0 * sqrt(static_cast<double>(s)) + 16.0;
        const double frac = w ? want / static_cast<double>(w) : 1.0;
        lim[i] = frac >= 0.5 ? ~0ull : static_cast<uint64_t>(frac * 18446744073709551616.0);
    }
}

// the segment offsets of sequences [seg0, seg0 + nseg] relative to the first one, as the int offsets cub takes
__global__ void segment_offsets_kernel(const uint64_t *__restrict__ off, uint64_t seg0, uint64_t nseg, int *__restrict__ out)
{
    const uint64_t base = off[seg0];
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i <= nseg;
         i += static_cast<uint64_t>(gridDim.x) * blockDim.x)
        out[i] = static_cast<int>(off[seg0 + i] - base);
}

// One warp per sequence of the round (lim != 0): its sorted candidates [off[i], off[i+1]) give the first min(s, distinct)
// distinct values to row i, the rest of the row is ~0 and out_n[i] its length.  A row that is final adds its length to
// *n_total.  A row with fewer than s distinct candidates under a limit below ~0 may be missing values above the limit: its
// limit becomes 4x (then ~0) and it is counted in *n_retry; every other sequence gets limit 0, which the next round skips.
__global__ void __launch_bounds__(256) sketch_finish_kernel(const uint64_t *__restrict__ sorted, const uint64_t *__restrict__ off,
                                                            uint64_t *__restrict__ lim, uint64_t n, uint64_t s, int round,
                                                            uint64_t *__restrict__ out_hashes, uint32_t *__restrict__ out_n,
                                                            unsigned long long *n_retry, unsigned long long *n_total)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t warps = static_cast<uint64_t>(gridDim.x) * (blockDim.x / 32);
    for (uint64_t i = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) / 32; i < n; i += warps) {
        const uint64_t l = lim[i];
        if (l == 0) continue;
        const uint64_t beg = off[i], end = off[i + 1];
        uint64_t *row = out_hashes + i * s;
        uint64_t distinct = 0;
        for (uint64_t p0 = beg; p0 < end && distinct < s; p0 += 32) {
            const uint64_t q = p0 + lane;
            const bool in = q < end;
            const uint64_t v = in ? sorted[q] : 0;
            const bool keep = in && (q == beg || sorted[q - 1] != v);
            const uint32_t m = __ballot_sync(0xffffffffu, keep);
            const uint64_t rank = distinct + __popc(m & ((1u << lane) - 1u));
            if (keep && rank < s) row[rank] = v;
            distinct += __popc(m);
        }
        const uint64_t nd = distinct < s ? distinct : s;
        for (uint64_t t = nd + lane; t < s; t += 32) row[t] = ~0ull;
        if (lane == 0) {
            out_n[i] = static_cast<uint32_t>(nd);
            const bool retry = distinct < s && l != ~0ull;
            lim[i] = retry ? (round == 0 && l < (1ull << 62) ? 4 * l : ~0ull) : 0;
            if (retry) atomicAdd(n_retry, 1ull);
            else atomicAdd(n_total, static_cast<unsigned long long>(nd));
        }
    }
}

} // namespace

} // namespace kmc

using namespace kmc;

extern "C" int32_t kmc_minhash_sketch(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint64_t s,
                                      uint64_t *out_hashes, kmc_result *result)
{
    int32_t st = check_common(ctx, seqs, k);
    if (st) return st;
    if (!out_hashes || !result) return fail(ctx, KMC_E_BAD_ARG, "out_hashes / result is NULL");
    if (mode != KMC_FW && mode != KMC_CANON) return fail(ctx, KMC_E_BAD_ARG, "mode must be KMC_FW or KMC_CANON");
    if (seqs->src_bits != 2) return fail(ctx, KMC_E_UNSUPPORTED, "the sketch needs a 2-bit source");
    if (k > 64) return fail(ctx, KMC_E_UNSUPPORTED, "the sketch supports K <= 64");
    if (s < 1) return fail(ctx, KMC_E_BAD_ARG, "the sketch size must be at least 1");
    CU(cudaSetDevice(ctx->device));
    memset(result, 0, sizeof *result);
    const Geometry ge = geometry(k);
    const bool canon = mode == KMC_CANON;
    cudaStream_t stream = ctx->stream;
    CU(cudaEventRecord(ctx->ev_k0, stream));
    constexpr int kBits = kSketchBits;
    constexpr uint64_t kBuckets = 1ull << kBits;
    st = ensure_scratch(ctx, layout_scratch_bytes(seqs) + kBuckets * 4 + 1024);
    if (st) return st;
    st = ensure_host_small(ctx);
    if (st) return st;
    Scratch scratch{static_cast<char *>(ctx->scratch), ctx->scratch_bytes, 0};
    uint32_t *table = static_cast<uint32_t *>(scratch.take(kBuckets * 4));
    unsigned long long *cursor = static_cast<unsigned long long *>(scratch.take(16));
    Layout L;
    st = plan_layout(ctx, seqs, k, ge, stream, KnownTotals(), scratch, &L);
    if (st) return st;
    if (L.total == 0) return KMC_OK;
    ExtractParams p = base_params(seqs, k, ge, L, 0);
    const bool ragged = !L.uniform_len;

    // (1) histogram of the top hash bits
    ConsumeParams c{};
    c.table = table;
    c.shift = 64 - kBits;
    c.table_entries = static_cast<uint32_t>(kBuckets);
    CU(cudaMemsetAsync(table, 0, kBuckets * 4, stream));
    ConsumeLaunchFn hist = consume_launcher<OP_HASH_HIST>(ge, ragged, canon);
    ConsumeLaunchFn below = consume_launcher<OP_HASH_BELOW>(ge, ragged, canon);
    if (!hist || !below) return fail(ctx, KMC_E_UNSUPPORTED, "no kernel for this K");
    CU(hist(p, c, stream));
    std::vector<uint32_t> counts(kBuckets);
    CU(cudaMemcpyAsync(counts.data(), table, kBuckets * 4, cudaMemcpyDeviceToHost, stream));
    CU(cudaStreamSynchronize(stream));

    // (2)-(4) threshold bucket, candidates, sort + unique; repeat with a higher threshold while
    // duplicates leave fewer than s distinct values
    uint64_t want = s; // candidates to collect (counting duplicates)
    for (;;) {
        uint64_t cum = 0;
        uint64_t t = 0;
        for (; t < kBuckets; ++t) {
            cum += counts[t];
            if (cum >= want) break;
        }
        const bool all = t >= kBuckets - 1;
        if (t >= kBuckets) t = kBuckets - 1;
        AsyncBuf cand, sorted, uniq, tmp, nsel;
        CU(cand.alloc(ctx, cum * 8, stream));
        CU(sorted.alloc(ctx, cum * 8, stream));
        CU(uniq.alloc(ctx, cum * 8, stream));
        CU(nsel.alloc(ctx, 8, stream));
        c.limit = all ? ~0ull : (((t + 1) << (64 - kBits)) - 1);
        c.cand = static_cast<uint64_t *>(cand.p);
        c.cursor = cursor;
        c.cand_cap = cum;
        CU(cudaMemsetAsync(cursor, 0, 8, stream));
        CU(below(p, c, stream));
        size_t b1 = 0, b2 = 0;
        CU(cub::DeviceRadixSort::SortKeys(nullptr, b1, static_cast<uint64_t *>(cand.p), static_cast<uint64_t *>(sorted.p), cum, 0,
                                          64, stream));
        CU(cub::DeviceSelect::Unique(nullptr, b2, static_cast<uint64_t *>(sorted.p), static_cast<uint64_t *>(uniq.p),
                                     static_cast<uint64_t *>(nsel.p), cum, stream));
        CU(tmp.alloc(ctx, b1 > b2 ? b1 : b2, stream));
        CU(cub::DeviceRadixSort::SortKeys(tmp.p, b1, static_cast<uint64_t *>(cand.p), static_cast<uint64_t *>(sorted.p), cum, 0, 64,
                                          stream));
        CU(cub::DeviceSelect::Unique(tmp.p, b2, static_cast<uint64_t *>(sorted.p), static_cast<uint64_t *>(uniq.p),
                                     static_cast<uint64_t *>(nsel.p), cum, stream));
        CU(cudaMemcpyAsync(&ctx->host_small[100], nsel.p, 8, cudaMemcpyDeviceToHost, stream));
        CU(cudaMemcpyAsync(&ctx->host_small[101], cursor, 8, cudaMemcpyDeviceToHost, stream));
        CU(cudaStreamSynchronize(stream));
        const uint64_t distinct = ctx->host_small[100];
        if (ctx->host_small[101] != cum) return fail(ctx, KMC_E_BAD_ARG, "internal: the two sketch passes disagree");
        if (distinct >= s || all) {
            const uint64_t n = distinct < s ? distinct : s;
            CU(cudaMemcpyAsync(out_hashes, uniq.p, n * 8, cudaMemcpyDeviceToDevice, stream));
            result->n_written = n;
            break;
        }
        want = cum + 2 * (s - distinct) + 1; // at least one more bucket
    }
    CU(cudaEventRecord(ctx->ev_k1, stream));
    CU(cudaStreamSynchronize(stream));
    CU(cudaEventElapsedTime(&result->kernel_ms, ctx->ev_k0, ctx->ev_k1));
    return KMC_OK;
}

// Every sequence's own sketch in one pass per round over the set (DESIGN.md 3.2d): per-sequence limits, a count pass
// (OP_SKETCH_COUNT) and a scan give each sequence a segment of the candidate array, an append pass (OP_SKETCH_APPEND)
// fills the segments, cub's segmented sort orders them and sketch_finish_kernel takes each row's distinct prefix.  Rows
// whose repeats left fewer than s distinct candidates go round again with a higher limit; the others are skipped.
extern "C" int32_t kmc_minhash_sketch_each(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint64_t s,
                                           uint64_t *out_hashes, uint32_t *out_n, kmc_result *result)
{
    int32_t st = check_common(ctx, seqs, k);
    if (st) return st;
    if (!out_hashes || !out_n || !result) return fail(ctx, KMC_E_BAD_ARG, "out_hashes / out_n / result is NULL");
    if (mode != KMC_FW && mode != KMC_CANON) return fail(ctx, KMC_E_BAD_ARG, "mode must be KMC_FW or KMC_CANON");
    if (seqs->src_bits != 2) return fail(ctx, KMC_E_UNSUPPORTED, "the sketch needs a 2-bit source");
    if (k > 64) return fail(ctx, KMC_E_UNSUPPORTED, "the sketch supports K <= 64");
    if (s < 1) return fail(ctx, KMC_E_BAD_ARG, "the sketch size must be at least 1");
    const uint64_t n = seqs->n_seqs;
    if (n && s > ~0ull / 8 / n) return fail(ctx, KMC_E_BAD_ARG, "n_seqs * s * 8 bytes overflows");
    memset(result, 0, sizeof *result);
    if (n == 0) return KMC_OK;
    CU(cudaSetDevice(ctx->device));
    const Geometry ge = geometry(k);
    const bool canon = mode == KMC_CANON;
    cudaStream_t stream = ctx->stream;
    CU(cudaEventRecord(ctx->ev_k0, stream));
    st = ensure_scratch(ctx, layout_scratch_bytes(seqs) + 1024);
    if (st) return st;
    st = ensure_host_small(ctx);
    if (st) return st;
    Scratch scratch{static_cast<char *>(ctx->scratch), ctx->scratch_bytes, 0};
    unsigned long long *counters = static_cast<unsigned long long *>(scratch.take(32)); // n_retry, n_total
    Layout L;
    st = plan_layout(ctx, seqs, k, ge, stream, KnownTotals(), scratch, &L);
    if (st) return st;
    ExtractParams p = base_params(seqs, k, ge, L, 0);
    const bool ragged = !L.uniform_len;
    ConsumeLaunchFn count = consume_launcher<OP_SKETCH_COUNT>(ge, ragged, canon);
    ConsumeLaunchFn append = consume_launcher<OP_SKETCH_APPEND>(ge, ragged, canon);
    if (!count || !append) return fail(ctx, KMC_E_UNSUPPORTED, "no kernel for this K");

    AsyncBuf lim, cnt, off, cursor, scan_tmp;
    CU(lim.alloc(ctx, n * 8, stream));
    CU(cnt.alloc(ctx, n * 8, stream));
    CU(off.alloc(ctx, (n + 1) * 8, stream));
    CU(cursor.alloc(ctx, n * 8, stream));
    CU(scan_tmp.alloc(ctx, scan_tmp_elems(n) * 8, stream));
    const unsigned blocks = static_cast<unsigned>(std::min<uint64_t>((n + 255) / 256, static_cast<uint64_t>(ctx->sm_count) * 16));
    sketch_limits_kernel<<<blocks, 256, 0, stream>>>(L.win_off, L.wpr, n, s, lim.as<uint64_t>());
    CU(cudaGetLastError());
    CU(cudaMemsetAsync(counters, 0, 16, stream));
    ConsumeParams c{};
    c.seq_lim = lim.as<uint64_t>();
    c.seq_cnt = cnt.as<unsigned long long>();
    c.seq_cursor = cursor.as<unsigned long long>();
    constexpr int kMaxRounds = 3; // the first limit, 4x, ~0: the last round flags nothing
    for (int round = 0; round < kMaxRounds; ++round) {
        // (1) candidates per sequence, their offsets and total
        CU(cudaMemsetAsync(cnt.p, 0, n * 8, stream));
        CU(count(p, c, stream));
        CU(inclusive_offsets_u64(cnt.as<uint64_t>(), off.as<uint64_t>(), n, scan_tmp.as<uint64_t>(), stream));
        CU(cudaMemcpyAsync(&ctx->host_small[100], off.as<uint64_t>() + n, 8, cudaMemcpyDeviceToHost, stream));
        CU(cudaStreamSynchronize(stream));
        const uint64_t total = ctx->host_small[100];
        // (2) the candidates into their segments
        AsyncBuf cand, sorted;
        CU(cand.alloc(ctx, total * 8, stream));
        CU(sorted.alloc(ctx, total * 8, stream));
        c.cand = cand.as<uint64_t>();
        CU(cudaMemcpyAsync(cursor.p, off.p, n * 8, cudaMemcpyDeviceToDevice, stream));
        CU(append(p, c, stream));
        // (3) sort every segment: cub counts items and segments in int, so runs of whole segments of at most 2^31 - 1
        // candidates each (one download of the offsets when the total is larger)
        if (total) {
            std::vector<uint64_t> h_off;
            if (total > 0x7fffffffull || n > 0x7fffffffull) {
                h_off.resize(n + 1);
                CU(cudaMemcpyAsync(h_off.data(), off.p, (n + 1) * 8, cudaMemcpyDeviceToHost, stream));
                CU(cudaStreamSynchronize(stream));
            }
            AsyncBuf seg_off, sort_tmp;
            const uint64_t max_run = std::min<uint64_t>(n, 0x7ffffffeull);
            CU(seg_off.alloc(ctx, (max_run + 1) * 4, stream));
            size_t tmp_bytes = 0;
            CU(cub::DeviceSegmentedSort::SortKeys(nullptr, tmp_bytes, cand.as<const uint64_t>(), sorted.as<uint64_t>(),
                                                  static_cast<int>(std::min<uint64_t>(total, 0x7fffffffull)), static_cast<int>(max_run),
                                                  seg_off.as<int>(), seg_off.as<int>() + 1, stream));
            CU(sort_tmp.alloc(ctx, tmp_bytes, stream));
            for (uint64_t seg0 = 0; seg0 < n;) {
                uint64_t seg1 = n;
                if (!h_off.empty()) {
                    seg1 = seg0 + 1;
                    if (h_off[seg1] - h_off[seg0] > 0x7fffffffull)
                        return fail(ctx, KMC_E_UNSUPPORTED, "a sequence has more than 2^31 - 1 sketch candidates");
                    while (seg1 < n && seg1 - seg0 < max_run && h_off[seg1 + 1] - h_off[seg0] <= 0x7fffffffull) ++seg1;
                }
                const uint64_t items = h_off.empty() ? total : h_off[seg1] - h_off[seg0];
                const uint64_t base = h_off.empty() ? 0 : h_off[seg0];
                const unsigned ob = static_cast<unsigned>(std::min<uint64_t>((seg1 - seg0 + 256) / 256, static_cast<uint64_t>(ctx->sm_count) * 16));
                segment_offsets_kernel<<<ob, 256, 0, stream>>>(off.as<uint64_t>(), seg0, seg1 - seg0, seg_off.as<int>());
                CU(cudaGetLastError());
                if (items)
                    CU(cub::DeviceSegmentedSort::SortKeys(sort_tmp.p, tmp_bytes, cand.as<const uint64_t>() + base, sorted.as<uint64_t>() + base,
                                                          static_cast<int>(items), static_cast<int>(seg1 - seg0), seg_off.as<int>(),
                                                          seg_off.as<int>() + 1, stream));
                seg0 = seg1;
            }
        }
        // (4) the rows; sequences left short go round again
        CU(cudaMemsetAsync(counters, 0, 8, stream));
        const unsigned fb = static_cast<unsigned>(std::min<uint64_t>((n + 7) / 8, static_cast<uint64_t>(ctx->sm_count) * 32));
        sketch_finish_kernel<<<fb, 256, 0, stream>>>(sorted.as<uint64_t>(), off.as<uint64_t>(), lim.as<uint64_t>(), n, s, round,
                                                     out_hashes, out_n, counters, counters + 1);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(&ctx->host_small[100], counters, 16, cudaMemcpyDeviceToHost, stream));
        CU(cudaStreamSynchronize(stream));
        const uint64_t n_retry = ctx->host_small[100];
        if (n_retry == 0) break;
        result->digest[0] += 1;       // rounds past the first
        result->digest[1] += n_retry; // sequences sketched again
    }
    result->n_written = ctx->host_small[101];
    CU(cudaEventRecord(ctx->ev_k1, stream));
    CU(cudaStreamSynchronize(stream));
    CU(cudaEventElapsedTime(&result->kernel_ms, ctx->ev_k0, ctx->ev_k1));
    return KMC_OK;
}

extern "C" int32_t kmc_composition(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint32_t *table,
                                   kmc_result *result)
{
    int32_t st = check_common(ctx, seqs, k);
    if (st) return st;
    if (!table || !result) return fail(ctx, KMC_E_BAD_ARG, "table / result is NULL");
    if (mode != KMC_FW && mode != KMC_CANON) return fail(ctx, KMC_E_BAD_ARG, "mode must be KMC_FW or KMC_CANON");
    if (seqs->src_bits != 2) return fail(ctx, KMC_E_UNSUPPORTED, "the composition needs a 2-bit source");
    if (k > 14) return fail(ctx, KMC_E_UNSUPPORTED, "the dense composition table supports K <= 14 (4^K counters)");
    CU(cudaSetDevice(ctx->device));
    memset(result, 0, sizeof *result);
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
    if (L.total == 0) return KMC_OK;
    ExtractParams p = base_params(seqs, k, ge, L, 0);
    ConsumeParams c{};
    c.table = table;
    c.table_entries = 1u << (2 * k);
    // few counters: every block counts in shared memory and adds its non-zero counters once (global
    // atomics on a handful of addresses serialise); many counters: direct increments, L2-resident up to K = 12
    const bool shared = c.table_entries <= static_cast<uint32_t>(kSharedCompositionMax);
    ConsumeLaunchFn fn = shared ? consume_launcher<OP_COMPOSITION_SHARED>(ge, !L.uniform_len, mode == KMC_CANON)
                                : consume_launcher<OP_COMPOSITION>(ge, !L.uniform_len, mode == KMC_CANON);
    if (!fn) return fail(ctx, KMC_E_UNSUPPORTED, "no kernel for this K");
    CU(fn(p, c, stream));
    CU(cudaEventRecord(ctx->ev_k1, stream));
    CU(cudaStreamSynchronize(stream));
    CU(cudaEventElapsedTime(&result->kernel_ms, ctx->ev_k0, ctx->ev_k1));
    return KMC_OK;
}

// ---- exact k-mer counts ------------------------------------------------------------------------
static int32_t table_status(kmc_ctx *ctx, cudaStream_t stream, unsigned long long *distinct, uint32_t *overflow, kmc_result *result)
{
    CU(cudaMemcpyAsync(&ctx->host_small[100], distinct, 8, cudaMemcpyDeviceToHost, stream));
    CU(cudaMemcpyAsync(&ctx->host_small[101], overflow, 4, cudaMemcpyDeviceToHost, stream));
    CU(cudaStreamSynchronize(stream));
    if (result) result->digest[0] = ctx->host_small[100]; // keys added by this call
    if (static_cast<uint32_t>(ctx->host_small[101]) != 0)
        return fail(ctx, KMC_E_OUT_TOO_SMALL, "the k-mer table is full");
    return KMC_OK;
}

// The key of a table of NL limbs (table_keys.cuh), and the same k-mer as binning.cuh partitions it
template <int NL> using TableKey = typename std::conditional<NL == 1, unsigned long long, ulonglong2>::type;
template <int NL> using BinKey = typename std::conditional<NL == 1, uint64_t, ulonglong2>::type;

// kmc_kmer_count (NL = 1) and kmc_kmer_count2 (NL = 2) past their K checks
template <int NL>
static int32_t kmer_count(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint64_t *keys, uint32_t *vals,
                          uint32_t log2_capacity, kmc_result *result)
{
    using Key = TableKey<NL>;
    if (log2_capacity < 1 || log2_capacity > 40) return fail(ctx, KMC_E_BAD_ARG, "log2_capacity must be in 1..40");
    CU(cudaSetDevice(ctx->device));
    memset(result, 0, sizeof *result);
    const Geometry ge = geometry(k);
    if (ge.n_limbs != NL) return fail(ctx, KMC_E_UNSUPPORTED, "no kernel for this K");
    cudaStream_t stream = ctx->stream;
    CU(cudaEventRecord(ctx->ev_k0, stream));
    int32_t st = ensure_scratch(ctx, layout_scratch_bytes(seqs) + 1024);
    if (st) return st;
    st = ensure_host_small(ctx);
    if (st) return st;
    Scratch scratch{static_cast<char *>(ctx->scratch), ctx->scratch_bytes, 0};
    unsigned long long *distinct = static_cast<unsigned long long *>(scratch.take(16));
    uint32_t *overflow = reinterpret_cast<uint32_t *>(distinct + 1);
    Layout L;
    st = plan_layout(ctx, seqs, k, ge, stream, KnownTotals(), scratch, &L);
    if (st) return st;
    result->n_written = L.total;
    if (L.total == 0) return KMC_OK;
    ExtractParams p = base_params(seqs, k, ge, L, 0);
    Key *table_keys = reinterpret_cast<Key *>(keys);
    ConsumeParams c{};
    c.table = vals;
    if constexpr (NL == 1)
        c.keys = table_keys;
    else
        c.keys2 = table_keys;
    c.log2cap = log2_capacity;
    c.distinct = distinct;
    c.overflow = overflow;
    CU(cudaMemsetAsync(distinct, 0, 16, stream));
    // A table beyond L2 (12 bytes per slot for one limb, 20 for two): write the k-mers out, bin them by the table slice
    // they fall into and insert slice after slice (bin_insert_kernel), a group of slices per launch (binning.cuh).  Needs
    // 16 (32) bytes per k-mer of temporary memory; without it the k-mers are inserted as they are produced.
    const uint64_t table_bytes = (8 * NL + 4ull) << log2_capacity;
    const int bin_bits = binning::bin_bits(static_cast<int>(log2_capacity), binning::kKmerSliceBits);
    binning::BinnedKeys<BinKey<NL>> bk;
    if (table_bytes > binning::kL2Budget && bk.alloc(ctx, (L.items + 1) * static_cast<uint64_t>(ge.g), bin_bits, stream)) {
        p.out_a = bk.written.template as<uint64_t>();
        p.vec_ok = 1;
        ExtractLaunchFn xfn = get_launcher(ge, mode == KMC_CANON ? MODE_CANON : MODE_FW, false, !L.uniform_len);
        if (!xfn) return fail(ctx, KMC_E_UNSUPPORTED, "no kernel for this K");
        CU(xfn(p, ctx->sm_count, stream));
        if constexpr (NL == 1)
            CU(bk.partition(L.total, binning::KmerHashBin{64 - bin_bits}, stream));
        else
            CU(bk.partition(L.total, binning::KmerHashBin2{64 - bin_bits}, stream));
        const Key *sorted = bk.binned.template as<const Key>();
        const uint64_t slice = 1ull << (log2_capacity - bin_bits); // slots per bin
        auto apply = [&](int b, int b_end) {
            const uint64_t slots = slice * static_cast<uint64_t>(b_end - b);
            cudaError_t e = warm_table(reinterpret_cast<const uint32_t *>(table_keys + static_cast<uint64_t>(b) * slice), 2 * NL * slots,
                                       ctx->sm_count, warm_sink(ctx), stream);
            if (e == cudaSuccess) e = warm_table(vals + static_cast<uint64_t>(b) * slice, slots, ctx->sm_count, warm_sink(ctx), stream);
            if (e != cudaSuccess) return e;
            bin_insert_kernel<Key><<<static_cast<unsigned>(ctx->sm_count * 16), 256, 0, stream>>>(
                sorted, bk.offs.template as<uint64_t>(), bk.n_blocks, b, b_end, table_keys, vals, log2_capacity, distinct, overflow);
            return cudaGetLastError();
        };
        CU(binning::apply_groups(1 << bin_bits, binning::kmer_group(NL), 0, nullptr, stream, apply));
    } else {
        const bool ragged = !L.uniform_len, canon = mode == KMC_CANON;
        ConsumeLaunchFn fn = NL == 1 ? consume_launcher<OP_TABLE>(ge, ragged, canon) : pick_consume_nx<2, OP_TABLE2>(ge.nx, ragged, canon);
        if (!fn) return fail(ctx, KMC_E_UNSUPPORTED, "no kernel for this K");
        CU(fn(p, c, stream));
    }
    CU(cudaEventRecord(ctx->ev_k1, stream));
    st = table_status(ctx, stream, distinct, overflow, result);
    CU(cudaEventElapsedTime(&result->kernel_ms, ctx->ev_k0, ctx->ev_k1));
    return st;
}

template <int NL>
static int32_t kmer_table_merge(kmc_ctx *ctx, uint64_t *keys, uint32_t *vals, uint32_t log2_capacity, const uint64_t *src_keys,
                                const uint32_t *src_vals, uint64_t n_src, uint64_t *n_new)
{
    using Key = TableKey<NL>;
    if (!ctx) return KMC_E_BAD_ARG;
    if (!keys || !vals || (n_src && (!src_keys || !src_vals))) return fail(ctx, KMC_E_BAD_ARG, "NULL table");
    if (log2_capacity < 1 || log2_capacity > 40) return fail(ctx, KMC_E_BAD_ARG, "log2_capacity must be in 1..40");
    CU(cudaSetDevice(ctx->device));
    int32_t st = ensure_scratch(ctx, 1024);
    if (st) return st;
    st = ensure_host_small(ctx);
    if (st) return st;
    cudaStream_t stream = ctx->stream;
    unsigned long long *distinct = static_cast<unsigned long long *>(ctx->scratch);
    uint32_t *overflow = reinterpret_cast<uint32_t *>(distinct + 1);
    CU(cudaMemsetAsync(distinct, 0, 16, stream));
    if (n_src) {
        const uint64_t blocks = std::min<uint64_t>((n_src + 255) / 256, static_cast<uint64_t>(ctx->sm_count) * 16);
        table_merge_kernel<Key><<<static_cast<unsigned>(blocks), 256, 0, stream>>>(reinterpret_cast<Key *>(keys), vals, log2_capacity,
                                                                                   reinterpret_cast<const Key *>(src_keys), src_vals,
                                                                                   n_src, distinct, overflow);
        CU(cudaGetLastError());
    }
    kmc_result r{};
    st = table_status(ctx, stream, distinct, overflow, &r);
    if (n_new) *n_new = r.digest[0];
    return st;
}

// RANGE: kmc_kmer_table(2)_export_range, the entries whose count lies in [min_count, max_count]
template <int NL, bool RANGE = false>
static int32_t kmer_table_export(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity, uint64_t *out_keys,
                                 uint32_t *out_vals, uint64_t capacity, uint64_t *n_out, uint32_t min_count = 0, uint32_t max_count = ~0u)
{
    using Key = TableKey<NL>;
    if (!ctx) return KMC_E_BAD_ARG;
    if (!keys || !vals || !n_out || (capacity && (!out_keys || !out_vals))) return fail(ctx, KMC_E_BAD_ARG, "NULL buffer");
    if (log2_capacity < 1 || log2_capacity > 40) return fail(ctx, KMC_E_BAD_ARG, "log2_capacity must be in 1..40");
    if (min_count > max_count) return fail(ctx, KMC_E_BAD_ARG, "min_count is larger than max_count");
    CU(cudaSetDevice(ctx->device));
    int32_t st = ensure_scratch(ctx, 1024);
    if (st) return st;
    st = ensure_host_small(ctx);
    if (st) return st;
    cudaStream_t stream = ctx->stream;
    unsigned long long *cursor = static_cast<unsigned long long *>(ctx->scratch);
    CU(cudaMemsetAsync(cursor, 0, 8, stream));
    const uint64_t n_slots = 1ull << log2_capacity;
    const uint64_t blocks = std::min<uint64_t>((n_slots + 255) / 256, static_cast<uint64_t>(ctx->sm_count) * 16);
    table_export_kernel<Key, RANGE><<<static_cast<unsigned>(blocks), 256, 0, stream>>>(
        reinterpret_cast<const Key *>(keys), vals, n_slots, reinterpret_cast<Key *>(out_keys), out_vals, capacity, cursor, min_count,
        max_count);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(&ctx->host_small[100], cursor, 8, cudaMemcpyDeviceToHost, stream));
    CU(cudaStreamSynchronize(stream));
    *n_out = ctx->host_small[100];
    if (*n_out > capacity) return fail(ctx, KMC_E_OUT_TOO_SMALL, "export capacity smaller than the number of keys in the table");
    return KMC_OK;
}

// The checks a count into a table of NL limbs and a lookup in it share, past their NULL checks: 16-byte aligned
// two-limb keys, the mode, a 2-bit source and a K of the table's width
template <int NL>
static int32_t check_table_kmers(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, const uint64_t *keys)
{
    if (NL == 2 && reinterpret_cast<uintptr_t>(keys) % 16) return fail(ctx, KMC_E_BAD_ARG, "the two-limb keys must be 16-byte aligned");
    if (mode != KMC_FW && mode != KMC_CANON) return fail(ctx, KMC_E_BAD_ARG, "mode must be KMC_FW or KMC_CANON");
    if (seqs->src_bits != 2) return fail(ctx, KMC_E_UNSUPPORTED, "the k-mer table needs a 2-bit source");
    if (NL == 1 && (k > 32 || (k == 32 && mode == KMC_FW)))
        return fail(ctx, KMC_E_UNSUPPORTED, "the k-mer table supports K <= 31, and K = 32 for canonical k-mers");
    if (NL == 2 && (k < 33 || k > 64 || (k == 64 && mode == KMC_FW)))
        return fail(ctx, KMC_E_UNSUPPORTED, "the two-limb k-mer table supports K = 33..63, and K = 64 for canonical k-mers");
    return KMC_OK;
}

template <int NL>
static int32_t kmer_count_checked(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint64_t *keys, uint32_t *vals,
                                  uint32_t log2_capacity, kmc_result *result)
{
    int32_t st = check_common(ctx, seqs, k);
    if (st) return st;
    if (!keys || !vals || !result) return fail(ctx, KMC_E_BAD_ARG, "keys / vals / result is NULL");
    st = check_table_kmers<NL>(ctx, seqs, k, mode, keys);
    if (st) return st;
    return kmer_count<NL>(ctx, seqs, k, mode, keys, vals, log2_capacity, result);
}

extern "C" int32_t kmc_kmer_count(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint64_t *keys, uint32_t *vals,
                                  uint32_t log2_capacity, kmc_result *result)
{
    return kmer_count_checked<1>(ctx, seqs, k, mode, keys, vals, log2_capacity, result);
}

extern "C" int32_t kmc_kmer_count2(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint64_t *keys, uint32_t *vals,
                                   uint32_t log2_capacity, kmc_result *result)
{
    return kmer_count_checked<2>(ctx, seqs, k, mode, keys, vals, log2_capacity, result);
}

// kmc_kmer_lookup (NL = 1) and kmc_kmer_lookup2 (NL = 2): the count of every window, direct probes at any table size
template <int NL>
static int32_t kmer_lookup(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, const uint64_t *keys, const uint32_t *vals,
                           uint32_t log2_capacity, uint32_t *out_counts, uint64_t capacity, kmc_result *result)
{
    int32_t st = check_common(ctx, seqs, k);
    if (st) return st;
    if (!keys || !vals || !out_counts || !result) return fail(ctx, KMC_E_BAD_ARG, "keys / vals / out_counts / result is NULL");
    st = check_table_kmers<NL>(ctx, seqs, k, mode, keys);
    if (st) return st;
    if (log2_capacity < 1 || log2_capacity > 40) return fail(ctx, KMC_E_BAD_ARG, "log2_capacity must be in 1..40");
    CU(cudaSetDevice(ctx->device));
    memset(result, 0, sizeof *result);
    const Geometry ge = geometry(k);
    if (ge.n_limbs != NL) return fail(ctx, KMC_E_UNSUPPORTED, "no kernel for this K");
    cudaStream_t stream = ctx->stream;
    CU(cudaEventRecord(ctx->ev_k0, stream));
    st = ensure_scratch(ctx, layout_scratch_bytes(seqs) + 256);
    if (st) return st;
    Scratch scratch{static_cast<char *>(ctx->scratch), ctx->scratch_bytes, 0};
    Layout L;
    st = plan_layout(ctx, seqs, k, ge, stream, KnownTotals(), scratch, &L);
    if (st) return st;
    result->n_written = L.total;
    if (capacity < L.total) return fail(ctx, KMC_E_OUT_TOO_SMALL, "out_counts capacity smaller than the number of windows");
    if (L.total == 0) return KMC_OK;
    ExtractParams p = base_params(seqs, k, ge, L, 0);
    p.vec_ok = reinterpret_cast<uintptr_t>(out_counts) % (4u * ge.g) == 0;
    ConsumeParams c{};
    c.table = const_cast<uint32_t *>(vals); // read only: OP_LOOKUP* never writes the table
    if constexpr (NL == 1)
        c.keys = reinterpret_cast<unsigned long long *>(const_cast<uint64_t *>(keys));
    else
        c.keys2 = reinterpret_cast<ulonglong2 *>(const_cast<uint64_t *>(keys));
    c.log2cap = log2_capacity;
    c.out_counts = out_counts;
    ConsumeLaunchFn fn = pick_consume_nx<NL, NL == 1 ? OP_LOOKUP : OP_LOOKUP2>(ge.nx, !L.uniform_len, mode == KMC_CANON);
    if (!fn) return fail(ctx, KMC_E_UNSUPPORTED, "no kernel for this K");
    CU(fn(p, c, stream));
    CU(cudaEventRecord(ctx->ev_k1, stream));
    CU(cudaStreamSynchronize(stream));
    CU(cudaEventElapsedTime(&result->kernel_ms, ctx->ev_k0, ctx->ev_k1));
    return KMC_OK;
}

// the argument checks every read-only query of a table shares
template <int NL>
static int32_t check_table_query(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (!keys || !vals) return fail(ctx, KMC_E_BAD_ARG, "NULL table");
    if (log2_capacity < 1 || log2_capacity > 40) return fail(ctx, KMC_E_BAD_ARG, "log2_capacity must be in 1..40");
    if (NL == 2 && reinterpret_cast<uintptr_t>(keys) % 16) return fail(ctx, KMC_E_BAD_ARG, "the two-limb keys must be 16-byte aligned");
    return KMC_OK;
}

template <int NL>
static int32_t kmer_table_get(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity, const uint64_t *query,
                              uint64_t n, uint32_t *out_counts)
{
    using Key = TableKey<NL>;
    int32_t st = check_table_query<NL>(ctx, keys, vals, log2_capacity);
    if (st) return st;
    if (n && (!query || !out_counts)) return fail(ctx, KMC_E_BAD_ARG, "query / out_counts is NULL");
    if (NL == 2 && reinterpret_cast<uintptr_t>(query) % 16) return fail(ctx, KMC_E_BAD_ARG, "the two-limb keys must be 16-byte aligned");
    if (n == 0) return KMC_OK;
    CU(cudaSetDevice(ctx->device));
    cudaStream_t stream = ctx->stream;
    const uint64_t blocks = std::min<uint64_t>((n + 255) / 256, static_cast<uint64_t>(ctx->sm_count) * 16);
    table_get_kernel<Key><<<static_cast<unsigned>(blocks), 256, 0, stream>>>(reinterpret_cast<const Key *>(keys), vals, log2_capacity,
                                                                              reinterpret_cast<const Key *>(query), n, out_counts);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(stream));
    return KMC_OK;
}

constexpr uint32_t kMaxHistBins = 16384; // 64 KB of shared counters per block

template <int NL>
static int32_t kmer_table_histogram(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity, uint64_t *hist,
                                    uint32_t n_bins)
{
    using Key = TableKey<NL>;
    int32_t st = check_table_query<NL>(ctx, keys, vals, log2_capacity);
    if (st) return st;
    if (!hist) return fail(ctx, KMC_E_BAD_ARG, "hist is NULL");
    if (n_bins < 1 || n_bins > kMaxHistBins) return fail(ctx, KMC_E_BAD_ARG, "n_bins must be in 1..16384");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t stream = ctx->stream;
    const size_t smem = 4ull * n_bins;
    CU(cudaFuncSetAttribute(table_histogram_kernel<Key>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * kMaxHistBins));
    const uint64_t n_slots = 1ull << log2_capacity;
    const uint64_t blocks = std::min<uint64_t>((n_slots + 256 * kHistUnroll - 1) / (256 * kHistUnroll), static_cast<uint64_t>(ctx->sm_count) * 8);
    table_histogram_kernel<Key><<<static_cast<unsigned>(blocks), 256, smem, stream>>>(
        reinterpret_cast<const Key *>(keys), vals, n_slots, reinterpret_cast<unsigned long long *>(hist), n_bins);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(stream));
    return KMC_OK;
}

template <int NL>
static int32_t kmer_table_export_range(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                                       uint32_t min_count, uint32_t max_count, uint64_t *out_keys, uint32_t *out_vals, uint64_t capacity,
                                       uint64_t *n_out)
{
    if (ctx && NL == 2 && (reinterpret_cast<uintptr_t>(keys) % 16 || reinterpret_cast<uintptr_t>(out_keys) % 16))
        return fail(ctx, KMC_E_BAD_ARG, "the two-limb keys must be 16-byte aligned");
    return kmer_table_export<NL, true>(ctx, keys, vals, log2_capacity, out_keys, out_vals, capacity, n_out, min_count, max_count);
}

extern "C" int32_t kmc_kmer_lookup(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, const uint64_t *keys, const uint32_t *vals,
                                   uint32_t log2_capacity, uint32_t *out_counts, uint64_t capacity, kmc_result *result)
{
    return kmer_lookup<1>(ctx, seqs, k, mode, keys, vals, log2_capacity, out_counts, capacity, result);
}

extern "C" int32_t kmc_kmer_lookup2(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, const uint64_t *keys,
                                    const uint32_t *vals, uint32_t log2_capacity, uint32_t *out_counts, uint64_t capacity,
                                    kmc_result *result)
{
    return kmer_lookup<2>(ctx, seqs, k, mode, keys, vals, log2_capacity, out_counts, capacity, result);
}

extern "C" int32_t kmc_kmer_table_get(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                                      const uint64_t *query, uint64_t n, uint32_t *out_counts)
{
    return kmer_table_get<1>(ctx, keys, vals, log2_capacity, query, n, out_counts);
}

extern "C" int32_t kmc_kmer_table2_get(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                                       const uint64_t *query, uint64_t n, uint32_t *out_counts)
{
    return kmer_table_get<2>(ctx, keys, vals, log2_capacity, query, n, out_counts);
}

extern "C" int32_t kmc_kmer_table_histogram(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                                            uint64_t *hist, uint32_t n_bins)
{
    return kmer_table_histogram<1>(ctx, keys, vals, log2_capacity, hist, n_bins);
}

extern "C" int32_t kmc_kmer_table2_histogram(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                                             uint64_t *hist, uint32_t n_bins)
{
    return kmer_table_histogram<2>(ctx, keys, vals, log2_capacity, hist, n_bins);
}

extern "C" int32_t kmc_kmer_table_export_range(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                                               uint32_t min_count, uint32_t max_count, uint64_t *out_keys, uint32_t *out_vals,
                                               uint64_t capacity, uint64_t *n_out)
{
    return kmer_table_export_range<1>(ctx, keys, vals, log2_capacity, min_count, max_count, out_keys, out_vals, capacity, n_out);
}

extern "C" int32_t kmc_kmer_table2_export_range(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                                                uint32_t min_count, uint32_t max_count, uint64_t *out_keys, uint32_t *out_vals,
                                                uint64_t capacity, uint64_t *n_out)
{
    return kmer_table_export_range<2>(ctx, keys, vals, log2_capacity, min_count, max_count, out_keys, out_vals, capacity, n_out);
}

extern "C" int32_t kmc_kmer_table_merge(kmc_ctx *ctx, uint64_t *keys, uint32_t *vals, uint32_t log2_capacity,
                                        const uint64_t *src_keys, const uint32_t *src_vals, uint64_t n_src, uint64_t *n_new)
{
    return kmer_table_merge<1>(ctx, keys, vals, log2_capacity, src_keys, src_vals, n_src, n_new);
}

extern "C" int32_t kmc_kmer_table2_merge(kmc_ctx *ctx, uint64_t *keys, uint32_t *vals, uint32_t log2_capacity,
                                         const uint64_t *src_keys, const uint32_t *src_vals, uint64_t n_src, uint64_t *n_new)
{
    if (ctx && (reinterpret_cast<uintptr_t>(keys) % 16 || reinterpret_cast<uintptr_t>(src_keys) % 16))
        return fail(ctx, KMC_E_BAD_ARG, "the two-limb keys must be 16-byte aligned");
    return kmer_table_merge<2>(ctx, keys, vals, log2_capacity, src_keys, src_vals, n_src, n_new);
}

extern "C" int32_t kmc_kmer_table_export(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                                         uint64_t *out_keys, uint32_t *out_vals, uint64_t capacity, uint64_t *n_out)
{
    return kmer_table_export<1>(ctx, keys, vals, log2_capacity, out_keys, out_vals, capacity, n_out);
}

extern "C" int32_t kmc_kmer_table2_export(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                                          uint64_t *out_keys, uint32_t *out_vals, uint64_t capacity, uint64_t *n_out)
{
    if (ctx && (reinterpret_cast<uintptr_t>(keys) % 16 || reinterpret_cast<uintptr_t>(out_keys) % 16))
        return fail(ctx, KMC_E_BAD_ARG, "the two-limb keys must be 16-byte aligned");
    return kmer_table_export<2>(ctx, keys, vals, log2_capacity, out_keys, out_vals, capacity, n_out);
}
