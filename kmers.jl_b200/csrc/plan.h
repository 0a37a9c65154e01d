// plan.h -- host-side launch planning shared by the 2-bit (api.cu) and 4-bit (fourbit.cu) paths:
// k-mer geometry, the window / group-slot layout of a read set, scratch carving and the source
// side of the kernel parameter block.  Nothing here computes k-mers on the host.
#pragma once
#include <cstring>
#include <memory>

#include "extract_kernels.cuh"
#include "kmc_internal.h"

namespace kmc {

int32_t fail_cuda(kmc_ctx *ctx, cudaError_t e, const char *what);
int32_t fail(kmc_ctx *ctx, int32_t code, const char *msg);

#define CU(call)                                                   \
    do {                                                           \
        cudaError_t e__ = (call);                                  \
        if (e__ != cudaSuccess) return fail_cuda(ctx, e__, #call); \
    } while (0)

// (Geometry / geometry(): kmer_core.cuh)

inline uint64_t round_up(uint64_t x, uint64_t m) { return (x + m - 1) / m * m; }

// A window of device scratch memory handed to one call (or one pipeline slot); carved by bumping.
struct Scratch {
    char *base = nullptr;
    uint64_t bytes = 0, used = 0;
    void *take(uint64_t n)
    {
        n = round_up(n ? n : 1, 256);
        if (used + n > bytes) return nullptr;
        void *p = base + used;
        used += n;
        return p;
    }
};

// Totals a caller may already know (the host pipeline computes them from host-side lengths), so
// the device path does not have to synchronise to read them back.
struct KnownTotals {
    bool valid = false;
    uint64_t windows = 0;
    uint64_t items = 0;
    // KMC_DIGEST of the host pipeline: if not NULL and digest_fusable(), the extraction kernel adds the xor / wrapping
    // sum of what it writes to digest[0..1] (stream a) and digest[2..3] (hash stream) itself, instead of a second
    // pass that re-reads both streams
    unsigned long long *digest = nullptr;
    // UnambiguousKmers over a recoded source: whether the sequences are ascending and disjoint in the buffer
    // (1 / 0), or -1 when the caller does not know (device-resident offsets are then checked on the device)
    int linear = -1;
};

// the fused fingerprint exists for the SoA forms of FwKmers / CanonicalKmers over 2-bit sources, K <= 64
inline bool digest_fusable(const kmc_seqs *s, int n_limbs, int mode, uint32_t flags)
{
    return s->src_bits == 2 && !(flags & (KMC_AOS | KMC_KMER4)) && (mode == KMC_FW || mode == KMC_CANON) && n_limbs <= 2;
}

struct Layout {
    bool uniform_len, uniform_off;
    uint64_t wpr;   // uniform_len only
    uint64_t total; // windows
    uint64_t items;
    uint64_t gprm;
    const uint64_t *win_off = nullptr;  // device, ragged
    const uint64_t *item_off = nullptr; // device, ragged
    const uint64_t *tile_first = nullptr; // device, ragged
    // tile_first when the scratch window cannot hold it (sequences that overlap in the buffer can have more windows
    // than the buffer has symbols): a temporary from the context's pool, freed (stream-ordered) with the last copy of
    // the Layout, so after the launches that read it have been enqueued
    std::shared_ptr<AsyncBuf> tile_buf;
};

// upper bound of the tiles a layout of sequences that do not overlap in the buffer can need (windows <= symbols, at
// most two partial group slots per sequence), for scratch sizing before the exact totals are known.  Overlapping
// sequences can need more: plan_layout() then takes the tile array from the context's pool.
inline uint64_t tiles_upper_bound(const kmc_seqs *s)
{
    const uint64_t spu = s->src_bits == 8 ? 1 : s->src_bits == 4 ? 16 : 32; // symbols per unit of n_words
    return (s->n_words * spu + 2 * s->n_seqs) / kTileItems + 2;
}

int32_t check_common(kmc_ctx *ctx, const kmc_seqs *s, int32_t k);

// bytes plan_layout() takes from the scratch window
uint64_t layout_scratch_bytes(const kmc_seqs *s);

// Window / group-slot layout of a set whose descriptor arrays live on the DEVICE.
int32_t plan_layout(kmc_ctx *ctx, const kmc_seqs *s, int k, const Geometry &ge, cudaStream_t stream,
                    const KnownTotals &known, Scratch &scratch, Layout *L);

// Source-side fields of the kernel parameter block (2-bit stream).
ExtractParams base_params(const kmc_seqs *s, int k, const Geometry &ge, const Layout &L, uint64_t unit_bias);

// Output-side fields + argument checks shared by both paths.  Returns KMC_OK or an error.
int32_t bind_outputs(kmc_ctx *ctx, const kmc_out *out, int mode, uint32_t flags, ExtractParams *p);

cudaError_t fill_uniform_offsets(uint64_t *out, uint64_t n_plus_1, uint64_t step, cudaStream_t stream);

ExtractLaunchFn get_launcher(const Geometry &ge, int mode, bool hash, bool ragged);
ExtractLaunchFn get_digest_launcher(const Geometry &ge, int mode, bool hash, bool ragged); // MODE_FW / MODE_CANON, N <= 2

// The device-resident extraction for 2-bit sources; everything is enqueued on `stream`.
int32_t extract_device(kmc_ctx *ctx, const kmc_seqs *s, int32_t k, int32_t mode, uint32_t flags, const kmc_out *out,
                       kmc_result *res, cudaStream_t stream, const KnownTotals &known, uint64_t unit_bias, bool sync,
                       Scratch &scratch);
uint64_t extract_scratch_bytes(const kmc_seqs *s, int k, int mode);

// kmer4.cu: k-mers over a 4-bit alphabet (KMC_KMER4) from 4-bit (Copyable) or 2-bit (TwoToFour) sources
int32_t check_kmer4(kmc_ctx *ctx, const kmc_seqs *s, int32_t k, int32_t mode);
uint64_t kmer4_scratch_bytes(const kmc_seqs *s);
int32_t extract_device_kmer4(kmc_ctx *ctx, const kmc_seqs *s, int32_t k, int32_t mode, uint32_t flags, const kmc_out *out,
                             kmc_result *res, cudaStream_t stream, const KnownTotals &known, uint64_t unit_bias, bool sync,
                             Scratch &scratch);

} // namespace kmc
