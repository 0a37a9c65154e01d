// api.cu -- the C ABI of libkmerscuda.so (include/kmerscuda.h): contexts, memory, and the host-side
// planning of every launch.  No compute happens on the host: a missing device is an error, never a
// fallback.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <new>
#include <vector>

#include "fourbit.h"
#include "plan.h"

// ---------------------------------------------------------------------------------------------
// helpers
// ---------------------------------------------------------------------------------------------
namespace kmc {

int32_t fail_cuda(kmc_ctx *ctx, cudaError_t e, const char *what)
{
    if (ctx) {
        char buf[512];
        snprintf(buf, sizeof buf, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
        ctx->last_error = buf;
    }
    return -static_cast<int32_t>(e);
}

int32_t fail(kmc_ctx *ctx, int32_t code, const char *msg)
{
    if (ctx) ctx->last_error = msg;
    return code;
}

ExtractLaunchFn get_launcher(const Geometry &ge, int mode, bool hash, bool ragged)
{
    switch (ge.n_limbs) {
    case 1: return get_extract_launcher_n1(ge.nx, mode, hash, ragged);
    case 2: return get_extract_launcher_n2(ge.nx, mode, hash, ragged);
    case 3: return get_extract_launcher_n3(ge.nx, mode, hash, ragged);
    case 4: return get_extract_launcher_n4(ge.nx, mode, hash, ragged);
    }
    return nullptr;
}

ExtractLaunchFn get_digest_launcher(const Geometry &ge, int mode, bool hash, bool ragged)
{
    switch (ge.n_limbs) {
    case 1: return get_digest_launcher_n1(ge.nx, mode, hash, ragged);
    case 2: return get_digest_launcher_n2(ge.nx, mode, hash, ragged);
    }
    return nullptr;
}

namespace {

bool aligned32(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 31) == 0; }

__global__ void fill_uniform_offsets_kernel(uint64_t *out, uint64_t n_plus_1, uint64_t step)
{
    uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n_plus_1) out[i] = i * step;
}

} // namespace

cudaError_t fill_uniform_offsets(uint64_t *out, uint64_t n_plus_1, uint64_t step, cudaStream_t stream)
{
    fill_uniform_offsets_kernel<<<static_cast<unsigned>((n_plus_1 + 255) / 256), 256, 0, stream>>>(out, n_plus_1, step);
    return cudaGetLastError();
}

int32_t check_common(kmc_ctx *ctx, const kmc_seqs *s, int32_t k)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (!s) return fail(ctx, KMC_E_BAD_ARG, "kmc_seqs is NULL");
    if (k < 1) return fail(ctx, KMC_E_BAD_K, "K must be at least 1");
    if (k > KMC_MAX_K) return fail(ctx, KMC_E_BAD_K, "K exceeds KMC_MAX_K (128)");
    if (s->src_bits != 2 && s->src_bits != 4 && s->src_bits != 8)
        return fail(ctx, KMC_E_BAD_ARG, "src_bits must be 2, 4 (LongSequence words) or 8 (ASCII bytes)");
    if (s->n_seqs > 0 && s->words == nullptr && s->n_words > 0) return fail(ctx, KMC_E_BAD_ARG, "words is NULL");
    return KMC_OK;
}

uint64_t layout_scratch_bytes(const kmc_seqs *s)
{
    if (s->seq_len == nullptr) return 0;
    const uint64_t n = s->n_seqs;
    return 4 * round_up((n + 1) * 8, 256) + round_up(scan_tmp_elems(n) * 8, 256) +
           round_up((tiles_upper_bound(s) + 1) * 8, 256);
}

int32_t plan_layout(kmc_ctx *ctx, const kmc_seqs *s, int k, const Geometry &ge, cudaStream_t stream,
                    const KnownTotals &known, Scratch &scratch, Layout *L)
{
    L->uniform_len = (s->seq_len == nullptr);
    L->uniform_off = (s->seq_word_offset == nullptr);
    L->tile_first = nullptr;
    L->tile_buf.reset(); // (a pipeline slot's layout of its previous chunk, whose launches are enqueued)
    const uint64_t G = static_cast<uint64_t>(ge.g);
    if (L->uniform_len) {
        L->wpr = s->uniform_len >= static_cast<uint64_t>(k) ? s->uniform_len - k + 1 : 0;
        L->total = L->wpr * s->n_seqs;
        L->gprm = (L->wpr % G == 0) ? L->wpr / G : (L->wpr + G - 1) / G + 1;
        if (s->n_seqs == 1) L->gprm = (L->wpr + G - 1) / G;
        L->items = L->gprm * s->n_seqs;
        return KMC_OK;
    }
    // ragged: cnt -> win_off ; slots -> item_off   (all in scratch)
    const uint64_t n = s->n_seqs;
    uint64_t *cnt = static_cast<uint64_t *>(scratch.take((n + 1) * 8));
    uint64_t *win_off = static_cast<uint64_t *>(scratch.take((n + 1) * 8));
    uint64_t *slots = static_cast<uint64_t *>(scratch.take((n + 1) * 8));
    uint64_t *item_off = static_cast<uint64_t *>(scratch.take((n + 1) * 8));
    uint64_t *tmp = static_cast<uint64_t *>(scratch.take(scan_tmp_elems(n) * 8));
    if (!cnt || !win_off || !slots || !item_off || !tmp) return fail(ctx, KMC_E_BAD_ARG, "internal: scratch window too small");
    CU(window_counts(s->seq_len, n, k, cnt, stream));
    CU(inclusive_offsets_u64(cnt, win_off, n, tmp, stream));
    CU(group_slots(win_off, n, ge.g, slots, stream));
    CU(inclusive_offsets_u64(slots, item_off, n, tmp, stream));
    L->win_off = win_off;
    L->item_off = item_off;
    L->wpr = 0;
    L->gprm = 1;
    if (known.valid) {
        L->total = known.windows;
        L->items = known.items;
    } else {
        uint64_t h[2] = {0, 0};
        CU(cudaMemcpyAsync(&h[0], win_off + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
        CU(cudaMemcpyAsync(&h[1], item_off + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
        CU(cudaStreamSynchronize(stream));
        L->total = h[0];
        L->items = h[1];
    }
    const uint64_t tiles = (L->items + kTileItems - 1) / kTileItems;
    if (tiles) {
        uint64_t *tile_first = static_cast<uint64_t *>(scratch.take((tiles + 1) * 8));
        if (!tile_first) { // more tiles than tiles_upper_bound(): sequences that overlap in the buffer
            L->tile_buf = std::make_shared<AsyncBuf>();
            CU(L->tile_buf->alloc(ctx, (tiles + 1) * 8, stream));
            tile_first = L->tile_buf->as<uint64_t>();
        }
        CU(tile_first_reads(item_off, n, kTileItems, tiles, tile_first, stream));
        L->tile_first = tile_first;
    }
    return KMC_OK;
}

ExtractParams base_params(const kmc_seqs *s, int k, const Geometry &ge, const Layout &L, uint64_t unit_bias)
{
    ExtractParams p;
    memset(&p, 0, sizeof p);
    p.w32 = reinterpret_cast<const uint32_t *>(s->words);
    p.nw32 = static_cast<int64_t>(s->n_words) * 2;
    p.unit_bits = 64;
    p.unit_bias = unit_bias;
    p.first = s->first_symbol_offset;
    p.k = k;
    p.s0 = ge.s0;
    p.head_mask = ge.head_mask;
    p.n_seqs = s->n_seqs;
    p.items = L.items;
    p.stride_units = s->uniform_stride_words;
    p.wpr = L.wpr;
    p.gprm = L.gprm;
    p.seq_unit_off = s->seq_word_offset;
    p.win_off = L.win_off;
    p.item_off = L.item_off;
    p.tile_first = L.tile_first;
    return p;
}

int32_t bind_outputs(kmc_ctx *ctx, const kmc_out *out, int mode, uint32_t flags, ExtractParams *p)
{
    const bool hash = (flags & KMC_HASH_FX) != 0;
    const bool aos = (flags & KMC_AOS) != 0;
    const bool want_index = (mode == KMC_UNAMBIG);
    if (!out->a) return fail(ctx, KMC_E_BAD_ARG, "out.a is NULL");
    if (mode == KMC_FWRV && !aos && !out->b) return fail(ctx, KMC_E_BAD_ARG, "out.b is NULL (FWRV, SoA)");
    if (hash && !out->hash) return fail(ctx, KMC_E_BAD_ARG, "out.hash is NULL (KMC_HASH_FX)");
    if (want_index && !aos && !out->index) return fail(ctx, KMC_E_BAD_ARG, "out.index is NULL (UNAMBIG, SoA)");
    p->out_a = out->a;
    p->out_b = out->b;
    p->out_hash = hash ? out->hash : nullptr;
    // AoS index lives inside out.a; the kernels key "emit an index" on out_index != NULL
    p->out_index = want_index ? (aos ? reinterpret_cast<int64_t *>(out->a) : out->index) : nullptr;
    p->index_base = out->index_base;
    p->aos = aos ? 1u : 0u;
    p->vec_ok = aligned32(out->a) && (!p->out_b || aligned32(p->out_b)) && (!p->out_hash || aligned32(p->out_hash)) &&
                (!p->out_index || aligned32(p->out_index));
    return KMC_OK;
}

uint64_t extract_scratch_bytes(const kmc_seqs *s, int k, int mode)
{
    if (s->src_bits != 2) return fourbit_scratch_bytes(s, k, mode);
    return layout_scratch_bytes(s) + 256;
}

// The device-resident extraction (2-bit sources); everything is enqueued on `stream`.
int32_t extract_device(kmc_ctx *ctx, const kmc_seqs *s, int32_t k, int32_t mode, uint32_t flags, const kmc_out *out,
                       kmc_result *res, cudaStream_t stream, const KnownTotals &known, uint64_t unit_bias, bool sync,
                       Scratch &scratch)
{
    const Geometry ge = geometry(k);
    const bool hash = (flags & KMC_HASH_FX) != 0;
    const int kmode = (mode == KMC_UNAMBIG) ? MODE_FW : mode; // 2-bit source: every window + its index (UnambiguousKmers.jl:64-77)

    if (sync) CU(cudaEventRecord(ctx->ev_k0, stream));
    // The Julia tuple layouts of one-limb k-mers over a uniform set: Vector{Tuple{Kmer,Kmer}} (FwRvIterator) and
    // Vector{Tuple{Kmer,Int}} (UnambiguousKmers over a 2-bit source) through the lean kernel with groups of two windows, so
    // that one work item is one 32-byte sector of the output (extract_kernels.cuh: launch_extract_aos).
    if ((flags & KMC_AOS) && (mode == KMC_FWRV || mode == KMC_UNAMBIG) && ge.n_limbs == 1 && !s->seq_len && !s->seq_word_offset) {
        const Geometry g2 = geometry(k, 2, kAosGroup);
        Layout L2;
        int32_t st2 = plan_layout(ctx, s, k, g2, stream, known, scratch, &L2); // (uniform: arithmetic only)
        if (st2) return st2;
        AosLaunchFn afn = get_aos_launcher_n1(g2.nx, mode == KMC_FWRV, hash);
        if (afn && L2.total > 0 && L2.total <= out->capacity) {
            ExtractParams p2 = base_params(s, k, g2, L2, unit_bias);
            st2 = bind_outputs(ctx, out, mode, flags, &p2);
            if (st2) return st2;
            const cudaError_t e = afn(p2, stream);
            if (e == cudaSuccess) {
                res->n_written = L2.total;
                if (out->seq_out_offset) CU(fill_uniform_offsets(out->seq_out_offset, s->n_seqs + 1, L2.wpr, stream));
                if (sync) {
                    CU(cudaEventRecord(ctx->ev_k1, stream));
                    CU(cudaStreamSynchronize(stream));
                    CU(cudaEventElapsedTime(&res->kernel_ms, ctx->ev_k0, ctx->ev_k1));
                }
                return KMC_OK;
            }
            if (e != cudaErrorNotSupported) return fail_cuda(ctx, e, "launch_extract_aos");
            (void)cudaGetLastError();
        }
    }
    Layout L;
    int32_t st = plan_layout(ctx, s, k, ge, stream, known, scratch, &L);
    if (st) return st;
    res->n_written = L.total;
    if (out->seq_out_offset) {
        if (L.uniform_len)
            CU(fill_uniform_offsets(out->seq_out_offset, s->n_seqs + 1, L.wpr, stream));
        else
            CU(cudaMemcpyAsync(out->seq_out_offset, L.win_off, (s->n_seqs + 1) * sizeof(uint64_t), cudaMemcpyDeviceToDevice, stream));
    }
    if (L.total == 0) return KMC_OK;
    if (L.total > out->capacity) return fail(ctx, KMC_E_OUT_TOO_SMALL, "output capacity smaller than the number of k-mers");
    ExtractParams p = base_params(s, k, ge, L, unit_bias);
    st = bind_outputs(ctx, out, mode, flags, &p);
    if (st) return st;

    const bool fused_digest = known.digest && digest_fusable(s, ge.n_limbs, mode, flags);
    if (fused_digest) p.digest = known.digest;
    ExtractLaunchFn fn = fused_digest ? get_digest_launcher(ge, kmode, hash, !L.uniform_len) : get_launcher(ge, kmode, hash, !L.uniform_len);
    if (!fn) return fail(ctx, KMC_E_UNSUPPORTED, "no kernel for this K");
    CU(fn(p, ctx->sm_count, stream));
    if (sync) {
        CU(cudaEventRecord(ctx->ev_k1, stream));
        CU(cudaStreamSynchronize(stream));
        CU(cudaEventElapsedTime(&res->kernel_ms, ctx->ev_k0, ctx->ev_k1));
    }
    return KMC_OK;
}

int32_t ensure_scratch(kmc_ctx *ctx, uint64_t bytes)
{
    if (bytes <= ctx->scratch_bytes) return KMC_OK;
    if (ctx->scratch) {
        CU(cudaStreamSynchronize(ctx->stream));
        for (int i = 0; i < 3; ++i) CU(cudaStreamSynchronize(ctx->pipe_streams[i]));
        CU(cudaFree(ctx->scratch));
        ctx->scratch = nullptr;
        ctx->scratch_bytes = 0;
    }
    uint64_t want = bytes + bytes / 4 + 4096;
    CU(cudaMalloc(&ctx->scratch, want));
    ctx->scratch_bytes = want;
    return KMC_OK;
}

int32_t ensure_host_small(kmc_ctx *ctx)
{
    if (ctx->host_small) return KMC_OK;
    CU(cudaHostAlloc(reinterpret_cast<void **>(&ctx->host_small), 4096, cudaHostAllocDefault));
    memset(ctx->host_small, 0, 4096);
    CU(cudaMalloc(reinterpret_cast<void **>(&ctx->dev_small), 128));
    return KMC_OK;
}

} // namespace kmc

using namespace kmc;

// ---------------------------------------------------------------------------------------------
// lifecycle
// ---------------------------------------------------------------------------------------------
extern "C" {

int32_t kmc_version(void) { return KMC_VERSION; }

int32_t kmc_device_count(int32_t *n)
{
    if (!n) return KMC_E_BAD_ARG;
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) {
        *n = 0;
        return (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? KMC_E_NO_DEVICE : -static_cast<int32_t>(e);
    }
    *n = c;
    return KMC_OK;
}

int32_t kmc_ctx_create(int32_t device, kmc_ctx **out)
{
    if (!out) return KMC_E_BAD_ARG;
    *out = nullptr;
    int32_t n = 0;
    int32_t st = kmc_device_count(&n);
    if (st) return st;
    if (n == 0 || device < 0 || device >= n) return KMC_E_NO_DEVICE;
    kmc_ctx *ctx = new (std::nothrow) kmc_ctx();
    if (!ctx) return KMC_E_BAD_ARG;
    ctx->device = device;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) {
        // Stream-ordered temporaries (binned counts, sketch candidates) come from a pool this context owns.  It keeps
        // what it has allocated (a binned count of 3 G k-mers takes 24 GB: re-allocating it per call costs
        // milliseconds) until kmc_trim or kmc_ctx_destroy; the process's default pool is not touched.
        cudaMemPoolProps props;
        memset(&props, 0, sizeof props);
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        if (cudaMemPoolCreate(&ctx->pool, &props) == cudaSuccess) {
            uint64_t keep = ~0ull;
            cudaMemPoolSetAttribute(ctx->pool, cudaMemPoolAttrReleaseThreshold, &keep);
        } else {
            ctx->pool = nullptr; // AsyncBuf falls back to the device's default pool
        }
        (void)cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking);
    for (int i = 0; i < 3 && e == cudaSuccess; ++i) e = cudaStreamCreateWithFlags(&ctx->pipe_streams[i], cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev_begin);
    if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev_end);
    if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev_k0);
    if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev_k1);
    if (e != cudaSuccess) {
        delete ctx;
        return -static_cast<int32_t>(e);
    }
    ctx->stream = ctx->own_stream;
    *out = ctx;
    return KMC_OK;
}

int32_t kmc_ctx_destroy(kmc_ctx *ctx)
{
    if (!ctx) return KMC_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->scratch) cudaFree(ctx->scratch);
    if (ctx->host_small) cudaFreeHost(ctx->host_small);
    if (ctx->dev_small) cudaFree(ctx->dev_small);
    for (int i = 0; i < 3; ++i) {
        if (ctx->pipe_buf[i]) cudaFree(ctx->pipe_buf[i]);
        if (ctx->pipe_streams[i]) cudaStreamDestroy(ctx->pipe_streams[i]);
        if (ctx->pipe_events[i]) cudaEventDestroy(ctx->pipe_events[i]);
    }
    if (ctx->ev_begin) cudaEventDestroy(ctx->ev_begin);
    if (ctx->ev_end) cudaEventDestroy(ctx->ev_end);
    if (ctx->ev_k0) cudaEventDestroy(ctx->ev_k0);
    if (ctx->ev_k1) cudaEventDestroy(ctx->ev_k1);
    if (ctx->comm) comm_detach(ctx);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->pool) cudaMemPoolDestroy(ctx->pool);
    delete ctx;
    return KMC_OK;
}

int32_t kmc_ctx_set_stream(kmc_ctx *ctx, void *cuda_stream)
{
    if (!ctx) return KMC_E_BAD_ARG;
    ctx->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
    return KMC_OK;
}

int32_t kmc_sync(kmc_ctx *ctx)
{
    if (!ctx) return KMC_E_BAD_ARG;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    return KMC_OK;
}

int32_t kmc_trim(kmc_ctx *ctx)
{
    if (!ctx) return KMC_E_BAD_ARG;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < 3; ++i) CU(cudaStreamSynchronize(ctx->pipe_streams[i]));
    if (ctx->pool) CU(cudaMemPoolTrimTo(ctx->pool, 0));
    return KMC_OK;
}

const char *kmc_last_error(kmc_ctx *ctx) { return ctx ? ctx->last_error.c_str() : "kmc_ctx is NULL"; }

const char *kmc_status_string(int32_t status)
{
    switch (status) {
    case KMC_OK: return "ok";
    case KMC_E_BAD_K: return "K must be at least 1 (and at most KMC_MAX_K)";
    case KMC_E_BAD_ARG: return "bad argument";
    case KMC_E_AMBIGUOUS: return "cannot encode an uncertain symbol in a 2-bit alphabet";
    case KMC_E_OUT_TOO_SMALL: return "output buffer too small";
    case KMC_E_NO_DEVICE: return "no CUDA device";
    case KMC_E_UNSUPPORTED: return "unsupported configuration";
    case KMC_E_NCCL: return "NCCL error (or NCCL could not be loaded)";
    }
    if (status < 0) return cudaGetErrorString(static_cast<cudaError_t>(-status));
    return "unknown status";
}

int32_t kmc_device_info(kmc_ctx *ctx, int32_t *sm_count, uint64_t *total_mem, char *name, int32_t name_len)
{
    if (!ctx) return KMC_E_BAD_ARG;
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, ctx->device));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (total_mem) *total_mem = prop.totalGlobalMem;
    if (name && name_len > 0) {
        strncpy(name, prop.name, static_cast<size_t>(name_len) - 1);
        name[name_len - 1] = 0;
    }
    return KMC_OK;
}

// ---------------------------------------------------------------------------------------------
// memory
// ---------------------------------------------------------------------------------------------
int32_t kmc_malloc(kmc_ctx *ctx, uint64_t bytes, void **dptr)
{
    if (!ctx || !dptr) return KMC_E_BAD_ARG;
    CU(cudaSetDevice(ctx->device));
    CU(cudaMalloc(dptr, bytes ? bytes : 1));
    return KMC_OK;
}

int32_t kmc_free(kmc_ctx *ctx, void *dptr)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (!dptr) return KMC_OK;
    CU(cudaSetDevice(ctx->device));
    CU(cudaFree(dptr));
    return KMC_OK;
}

int32_t kmc_memset(kmc_ctx *ctx, void *dptr, int32_t value, uint64_t bytes)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (bytes == 0) return KMC_OK;
    CU(cudaSetDevice(ctx->device));
    CU(cudaMemsetAsync(dptr, value, bytes, ctx->stream));
    return KMC_OK;
}

int32_t kmc_upload(kmc_ctx *ctx, void *dptr, const void *host, uint64_t bytes)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (bytes == 0) return KMC_OK;
    CU(cudaSetDevice(ctx->device));
    CU(cudaMemcpyAsync(dptr, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return KMC_OK;
}

int32_t kmc_download(kmc_ctx *ctx, void *host, const void *dptr, uint64_t bytes)
{
    if (!ctx) return KMC_E_BAD_ARG;
    CU(cudaSetDevice(ctx->device));
    if (bytes) CU(cudaMemcpyAsync(host, dptr, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return KMC_OK;
}

int32_t kmc_host_alloc(kmc_ctx *ctx, uint64_t bytes, void **hptr)
{
    if (!ctx || !hptr) return KMC_E_BAD_ARG;
    CU(cudaSetDevice(ctx->device));
    CU(cudaHostAlloc(hptr, bytes ? bytes : 1, cudaHostAllocDefault));
    return KMC_OK;
}

int32_t kmc_host_free(kmc_ctx *ctx, void *hptr)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (!hptr) return KMC_OK;
    CU(cudaFreeHost(hptr));
    return KMC_OK;
}

int32_t kmc_host_register(kmc_ctx *ctx, void *hptr, uint64_t bytes)
{
    if (!ctx || !hptr) return KMC_E_BAD_ARG;
    CU(cudaSetDevice(ctx->device));
    CU(cudaHostRegister(hptr, bytes, cudaHostRegisterDefault));
    return KMC_OK;
}

int32_t kmc_host_unregister(kmc_ctx *ctx, void *hptr)
{
    if (!ctx || !hptr) return KMC_E_BAD_ARG;
    CU(cudaHostUnregister(hptr));
    return KMC_OK;
}

// ---------------------------------------------------------------------------------------------
// hot path
// ---------------------------------------------------------------------------------------------
int32_t kmc_count(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint64_t *n_out)
{
    int32_t st = check_common(ctx, seqs, k);
    if (st) return st;
    if (!n_out) return fail(ctx, KMC_E_BAD_ARG, "n_out is NULL");
    if (mode < KMC_FW || mode > KMC_UNAMBIG) return fail(ctx, KMC_E_BAD_ARG, "unknown mode");
    CU(cudaSetDevice(ctx->device));
    if (mode == KMC_UNAMBIG && seqs->src_bits != 2) return count_unambiguous_4bit(ctx, seqs, k, n_out, ctx->stream);
    const Geometry ge = geometry(k);
    st = ensure_scratch(ctx, layout_scratch_bytes(seqs) + 256);
    if (st) return st;
    Scratch scratch{static_cast<char *>(ctx->scratch), ctx->scratch_bytes, 0};
    Layout L;
    st = plan_layout(ctx, seqs, k, ge, ctx->stream, KnownTotals(), scratch, &L);
    if (st) return st;
    *n_out = L.total;
    return KMC_OK;
}

int32_t kmc_extract(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint32_t flags, const kmc_out *out,
                    kmc_result *result)
{
    int32_t st = check_common(ctx, seqs, k);
    if (st) return st;
    if (!out || !result) return fail(ctx, KMC_E_BAD_ARG, "kmc_out / kmc_result is NULL");
    if (mode < KMC_FW || mode > KMC_UNAMBIG) return fail(ctx, KMC_E_BAD_ARG, "unknown mode");
    CU(cudaSetDevice(ctx->device));
    result->n_written = 0;
    result->err_seq = result->err_pos = 0;
    result->err_sym = 0;
    result->kernel_ms = 0.f;
    if (flags & KMC_KMER4) {
        st = check_kmer4(ctx, seqs, k, mode);
        if (st) return st;
        st = ensure_scratch(ctx, kmer4_scratch_bytes(seqs));
        if (st) return st;
        Scratch scratch{static_cast<char *>(ctx->scratch), ctx->scratch_bytes, 0};
        return extract_device_kmer4(ctx, seqs, k, mode, flags, out, result, ctx->stream, KnownTotals(), 0,
                                    (flags & KMC_NO_SYNC) == 0, scratch);
    }
    if (seqs->src_bits != 2) return extract_device_4bit(ctx, seqs, k, mode, flags, out, result, ctx->stream);
    st = ensure_scratch(ctx, extract_scratch_bytes(seqs, k, mode));
    if (st) return st;
    Scratch scratch{static_cast<char *>(ctx->scratch), ctx->scratch_bytes, 0};
    return extract_device(ctx, seqs, k, mode, flags, out, result, ctx->stream, KnownTotals(), 0,
                          (flags & KMC_NO_SYNC) == 0, scratch);
}

int32_t kmc_fx_hash(kmc_ctx *ctx, const uint64_t *kmers, uint64_t n, int32_t n_limbs, uint64_t h0, uint64_t *out)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (n_limbs < 0 || n_limbs > 4) return fail(ctx, KMC_E_BAD_ARG, "n_limbs must be in 0..4");
    if (n && (!out || (n_limbs && !kmers))) return fail(ctx, KMC_E_BAD_ARG, "NULL buffer");
    CU(cudaSetDevice(ctx->device));
    CU(launch_fx_hash(kmers, n, n_limbs, h0, out, ctx->sm_count, ctx->stream));
    return KMC_OK;
}

int32_t kmc_base_hash(kmc_ctx *ctx, const uint64_t *kmers, uint64_t n, int32_t n_limbs, int32_t k, uint64_t h0, uint64_t *out)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (n_limbs < 0 || n_limbs > 4) return fail(ctx, KMC_E_BAD_ARG, "n_limbs must be in 0..4");
    if (k < 0) return fail(ctx, KMC_E_BAD_K, "K must not be negative");
    if (n && (!out || (n_limbs && !kmers))) return fail(ctx, KMC_E_BAD_ARG, "NULL buffer");
    CU(cudaSetDevice(ctx->device));
    CU(launch_base_hash(kmers, n, n_limbs, h0 ^ static_cast<uint64_t>(k), out, ctx->sm_count, ctx->stream));
    return KMC_OK;
}

int32_t kmc_digest(kmc_ctx *ctx, const uint64_t *dptr, uint64_t n, uint64_t *out)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (!out || (n && !dptr)) return fail(ctx, KMC_E_BAD_ARG, "NULL buffer");
    CU(cudaSetDevice(ctx->device));
    int32_t st = ensure_scratch(ctx, 256);
    if (st) return st;
    uint64_t *acc = static_cast<uint64_t *>(ctx->scratch);
    CU(launch_digest(dptr, n, acc, ctx->sm_count, ctx->stream));
    CU(cudaMemcpyAsync(out, acc, 16, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return KMC_OK;
}

int32_t kmc_timer_begin(kmc_ctx *ctx)
{
    if (!ctx) return KMC_E_BAD_ARG;
    CU(cudaSetDevice(ctx->device));
    CU(cudaEventRecord(ctx->ev_begin, ctx->stream));
    return KMC_OK;
}

int32_t kmc_timer_end(kmc_ctx *ctx, float *ms)
{
    if (!ctx || !ms) return KMC_E_BAD_ARG;
    CU(cudaSetDevice(ctx->device));
    CU(cudaEventRecord(ctx->ev_end, ctx->stream));
    CU(cudaEventSynchronize(ctx->ev_end));
    CU(cudaEventElapsedTime(ms, ctx->ev_begin, ctx->ev_end));
    return KMC_OK;
}

int32_t kmc_store_probe(kmc_ctx *ctx, void *dptr, uint64_t bytes)
{
    if (!ctx || !dptr) return KMC_E_BAD_ARG;
    CU(cudaSetDevice(ctx->device));
    CU(launch_store_probe(dptr, bytes, ctx->sm_count, ctx->stream));
    return KMC_OK;
}

} // extern "C"
