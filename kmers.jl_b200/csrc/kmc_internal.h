// kmc_internal.h -- shared host-side declarations of libkmerscuda (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <string>

#include "../../include/kmerscuda.h"

struct kmc_comm;

struct kmc_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr; // the stream launches go to (own_stream or the caller's)
    cudaStream_t pipe_streams[3] = {nullptr, nullptr, nullptr}; // kmc_extract_host pipeline slots
    cudaEvent_t pipe_events[3] = {nullptr, nullptr, nullptr};   // phase-A completion per slot
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;  // kmc_timer_*
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;      // per-call kernel timing
    // grow-only scratch (scans, recoded 4-bit streams, compaction counters)
    void *scratch = nullptr;
    uint64_t scratch_bytes = 0;
    // host-pipeline device buffers, one per slot (grow-only)
    void *pipe_buf[3] = {nullptr, nullptr, nullptr};
    uint64_t pipe_bytes[3] = {0, 0, 0};
    // small pinned host block for device->host read-backs of counts and error records:
    // 16 u64 per pipeline slot, slot 3 = the context's own stream
    uint64_t *host_small = nullptr;
    uint64_t *dev_small = nullptr; // 128 bytes of device memory: KMC_DIGEST accumulators (first 64), warm_table's sink (byte 96)
    // stream-ordered temporaries (binned counts, sketch candidates) come from a pool the context owns, so the
    // process's default pool is left alone and kmc_trim / kmc_ctx_destroy give the memory back
    cudaMemPool_t pool = nullptr;
    kmc_comm *comm = nullptr; // comm.cu: the NCCL communicator attached to this context, if any
    std::string last_error;
};

namespace kmc {

// stream-ordered temporary from the context's pool; freed (stream-ordered) when it goes out of scope
struct AsyncBuf {
    void *p = nullptr;
    cudaStream_t s = nullptr;
    cudaError_t alloc(kmc_ctx *ctx, uint64_t bytes, cudaStream_t stream)
    {
        s = stream;
        return ctx->pool ? cudaMallocFromPoolAsync(&p, bytes ? bytes : 1, ctx->pool, stream)
                         : cudaMallocAsync(&p, bytes ? bytes : 1, stream);
    }
    template <typename T> T *as() const { return static_cast<T *>(p); }
    AsyncBuf() = default;
    AsyncBuf(const AsyncBuf &) = delete;
    AsyncBuf &operator=(const AsyncBuf &) = delete;
    ~AsyncBuf()
    {
        if (p) cudaFreeAsync(p, s);
    }
};

inline uint32_t *warm_sink(kmc_ctx *ctx) { return reinterpret_cast<uint32_t *>(ctx->dev_small) + 24; }

// comm.cu: destroys the context's communicator (rank) and its stream / events
void comm_detach(kmc_ctx *ctx);

// scratch carving -------------------------------------------------------------------------
int32_t ensure_scratch(kmc_ctx *ctx, uint64_t bytes);
int32_t ensure_host_small(kmc_ctx *ctx);

// scan.cu -----------------------------------------------------------------------------------
// out[0] = 0, out[i+1] = sum_{j<=i} in[j]  (n+1 outputs), all on `stream`.
// tmp must hold scan_tmp_elems(n) u64.
uint64_t scan_tmp_elems(uint64_t n);
cudaError_t inclusive_offsets_u64(const uint64_t *in, uint64_t *out, uint64_t n, uint64_t *tmp, cudaStream_t stream);
// per-sequence window counts (FwKmers.jl:40-43: max(0, len - K + 1)) -> cnt[n]
cudaError_t window_counts(const uint64_t *seq_len, uint64_t n, int k, uint64_t *cnt, cudaStream_t stream);
// group slots per sequence from the window offsets: slots[r] = #aligned groups of G that intersect
// [win_off[r], win_off[r+1])
cudaError_t group_slots(const uint64_t *win_off, uint64_t n, int g, uint64_t *slots, cudaStream_t stream);

cudaError_t tile_first_reads(const uint64_t *item_off, uint64_t n_seqs, uint64_t tile_items, uint64_t n_tiles,
                             uint64_t *tile_first, cudaStream_t stream);

// buckets.cu: pulls table[0..n_counters) into L2; sink: 4 bytes of device memory on the table's device (never written in
// practice)
cudaError_t warm_table(const uint32_t *table, uint64_t n_counters, int sm_count, uint32_t *sink, cudaStream_t stream);

// misc_kernels.cu -----------------------------------------------------------------------------
cudaError_t launch_fx_hash(const uint64_t *kmers, uint64_t n, int n_limbs, uint64_t h0, uint64_t *out, int sm_count,
                           cudaStream_t stream);
// acc[0] ^= xor of the words, acc[1] += their sum (zero = clear acc first)
cudaError_t launch_digest(const uint64_t *p, uint64_t n, uint64_t *acc, int sm_count, cudaStream_t stream, bool zero = true);
cudaError_t launch_base_hash(const uint64_t *kmers, uint64_t n, int n_limbs, uint64_t h, uint64_t *out, int sm_count,
                             cudaStream_t stream);
cudaError_t launch_store_probe(void *dptr, uint64_t bytes, int sm_count, cudaStream_t stream);

} // namespace kmc
