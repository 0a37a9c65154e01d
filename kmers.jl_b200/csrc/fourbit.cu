// fourbit.cu -- 4-bit sources (FourToTwo, src/construction.jl:85-86): device recoding, the
// valid-start bit stream, the strict-mode error resolution and the two-phase orchestration of
// UnambiguousKmers' ordered compaction.  See fourbit.h for the scheme.
#include "compact_kernels.cuh"
#include "fourbit.h"

namespace kmc {

namespace {

constexpr uint64_t kNone = ~0ull;
constexpr int kCountLayoutG = 32; // windows per work item when the survivors are only counted (valid_count.cu)

// (recode_word: fourbit_core.cuh)

// One thread per PAIR of source words (= one group of 32 symbols): 2 x u32 of 2-bit codes, 1 x u32 of
// uncertainty flags -- and, fused, the group's valid-start word: the block keeps its 256 flag words
// (+ a 5-word halo recomputed from the neighbouring block's source words) in shared memory, so the
// flags are never re-read from global memory and no second pass is launched.
// rev (optional): the same codes as one stream in REVERSED symbol order -- group g goes, its 32 symbols reversed, to
// 64-bit word n_groups - 1 - g -- in which the forward k-mer of every window is a plain run of 2K bits (lincompact.cuh).
// FULL: every group of the block and of its halo exists, both source words of each lie inside the array, and the
// array is 16-byte aligned -- all blocks but the last one or two.  The bounds tests and 64-bit index arithmetic of the
// general form were 40 % of the pass's instructions, and the pass is bound by its integer instructions.
template <bool FULL>
__device__ __forceinline__ void recode_vstart_block(const uint64_t *__restrict__ words, uint64_t n_words, int k,
                                                    uint32_t *__restrict__ rec, uint32_t *__restrict__ bad,
                                                    uint32_t *__restrict__ vstart, uint64_t n_groups, uint64_t n_vstart,
                                                    uint32_t *__restrict__ rev, uint32_t *s_bad)
{
    // kRecodeGroups groups per thread, all their source words requested before the first is used: with one 16-byte
    // load per short-lived thread the pass was latency-bound, and the halo below was recomputed once per 256 groups
    const uint64_t g0 = static_cast<uint64_t>(blockIdx.x) * (256 * kRecodeGroups);
    const uint32_t t = threadIdx.x;
    const uint4 *src = reinterpret_cast<const uint4 *>(words) + g0; // (FULL: 16-byte aligned)
    const bool aligned = (reinterpret_cast<uintptr_t>(words) & 15) == 0;
    // words past the end read as 'A' (one-hot): never part of a window, never flagged
    auto load_pair = [&](uint32_t i) -> uint4 { // group g0 + i
        if (FULL) return __ldg(src + i);
        const uint64_t g = g0 + i;
        if (2 * g + 1 < n_words && aligned) return __ldg(src + i);
        const uint64_t a = 2 * g < n_words ? __ldg(words + 2 * g) : 0x1111111111111111ull;
        const uint64_t b = 2 * g + 1 < n_words ? __ldg(words + 2 * g + 1) : 0x1111111111111111ull;
        return make_uint4(static_cast<uint32_t>(a), static_cast<uint32_t>(a >> 32), static_cast<uint32_t>(b), static_cast<uint32_t>(b >> 32));
    };
    uint4 w[kRecodeGroups];
#pragma unroll
    for (int j = 0; j < kRecodeGroups; ++j) w[j] = load_pair(256 * j + t);
    uint4 h = make_uint4(0x11111111u, 0x11111111u, 0x11111111u, 0x11111111u);
    if (t < kRecodeHalo) h = load_pair(256 * kRecodeGroups + t);
    auto recode = [](const uint4 &v, uint32_t &c0, uint32_t &c1) -> uint32_t { // 32 symbols: codes of the two words, 32 flags
        uint32_t a, b, fa, fb;
        recode_half(v.x, a, fa);
        recode_half(v.y, b, fb);
        c0 = a | (b << 16);
        uint32_t f = fa | (fb << 8);
        recode_half(v.z, a, fa);
        recode_half(v.w, b, fb);
        c1 = a | (b << 16);
        return f | (fa << 16) | (fb << 24);
    };
    uint2 *rec2 = reinterpret_cast<uint2 *>(rec) + g0;
    uint2 *rev2 = reinterpret_cast<uint2 *>(rev) + (n_groups - 1 - g0); // group g0 + i goes to rev2[-i]
    uint32_t *bad0 = bad + g0;
#pragma unroll
    for (int j = 0; j < kRecodeGroups; ++j) {
        const uint32_t i = 256 * j + t;
        uint32_t c0, c1;
        const uint32_t f = recode(w[j], c0, c1); // (a group past the end: all 'A', no flag)
        if (FULL || g0 + i < n_groups) {
            if (rec) rec2[i] = make_uint2(c0, c1);
            if (rev) *(rev2 - i) = make_uint2(rev2_32(c1), rev2_32(c0));
            if (bad) bad0[i] = f;
        }
        s_bad[i] = f;
    }
    if (t < kRecodeHalo) {
        uint32_t c0, c1;
        s_bad[256 * kRecodeGroups + t] = recode(h, c0, c1);
    }
    __syncthreads();
    uint32_t *vs0 = vstart + g0;
#pragma unroll
    for (int j = 0; j < kRecodeGroups; ++j) {
        const uint32_t i = 256 * j + t;
        if (FULL || g0 + i < n_vstart) {
            uint32_t a[6];
#pragma unroll
            for (int d = 0; d < 5; ++d) a[d] = s_bad[i + d];
            a[5] = 0;
            vs0[i] = valid_start_word(a, k);
        }
    }
}

__global__ void __launch_bounds__(256) recode_vstart_kernel(const uint64_t *__restrict__ words, uint64_t n_words, int k,
                                                            uint32_t *__restrict__ rec, uint32_t *__restrict__ bad,
                                                            uint32_t *__restrict__ vstart, uint64_t n_groups,
                                                            uint64_t n_vstart, uint32_t *__restrict__ rev)
{
    __shared__ uint32_t s_bad[256 * kRecodeGroups + 8];
    const uint64_t g_end = (static_cast<uint64_t>(blockIdx.x) + 1) * (256 * kRecodeGroups) + kRecodeHalo; // one past the halo
    const bool full = g_end <= n_groups && 2 * g_end <= n_words && (reinterpret_cast<uintptr_t>(words) & 15) == 0; // block-uniform
    if (full)
        recode_vstart_block<true>(words, n_words, k, rec, bad, vstart, n_groups, n_vstart, rev, s_bad);
    else
        recode_vstart_block<false>(words, n_words, k, rec, bad, vstart, n_groups, n_vstart, rev, s_bad);
}

// Turns the first offending flat window of a strict mode into what the reference throws on:
// the first symbol with count_ones != 1 of that sequence (its 0-based sequence, 1-based position
// and 4-bit encoding).  One thread.
__global__ void resolve_error_kernel(ExtractParams p, int src_bits, const uint64_t *__restrict__ words4,
                                     const uint32_t *__restrict__ bad, uint64_t flat, uint64_t *__restrict__ err_out)
{
    uint64_t r, f0;
    if (p.win_off) {
        uint64_t lo = 0, hi = p.n_seqs;
        while (hi - lo > 1) {
            uint64_t mid = (lo + hi) >> 1;
            if (p.win_off[mid] <= flat) lo = mid; else hi = mid;
        }
        // skip sequences without windows that share the same offset
        r = lo;
        f0 = p.win_off[r];
    } else {
        r = flat / p.wpr;
        f0 = r * p.wpr;
    }
    const uint64_t w = flat - f0;
    const uint64_t unit_off = p.seq_unit_off ? p.seq_unit_off[r] - p.unit_bias : r * p.stride_units;
    const uint64_t s0 = unit_off * (p.unit_bits >> 1) + p.first; // absolute symbol index of the sequence's first symbol
    uint64_t pos0 = w + static_cast<uint64_t>(p.k) - 1; // windows before w were clean => only the last symbol can be new
    if (w == 0) {
        for (uint64_t j = 0; j < static_cast<uint64_t>(p.k); ++j) {
            const uint64_t a = s0 + j;
            if ((bad[a >> 5] >> (a & 31)) & 1u) {
                pos0 = j;
                break;
            }
        }
    }
    const uint64_t a = s0 + pos0;
    err_out[0] = r;
    err_out[1] = pos0 + 1;
    err_out[2] = src_bits == 8 ? reinterpret_cast<const uint8_t *>(words4)[a] : (words4[a >> 4] >> (4 * (a & 15))) & 15u;
}

// Emitted k-mers per sequence (UnambiguousKmers): popcount of the valid-start bits over the
// sequence's windows.  One warp per sequence.
__global__ void __launch_bounds__(256) seq_valid_counts_kernel(ExtractParams p, uint64_t *__restrict__ cnt)
{
    const uint64_t r = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= p.n_seqs) return;
    uint64_t wcount;
    if (p.win_off) wcount = p.win_off[r + 1] - p.win_off[r]; else wcount = p.wpr;
    const uint64_t unit_off = p.seq_unit_off ? p.seq_unit_off[r] - p.unit_bias : r * p.stride_units;
    const uint64_t a = unit_off * (p.unit_bits >> 1) + p.first, b = a + wcount; // valid-start bits [a, b)
    uint64_t c = 0;
    if (wcount) {
        for (uint64_t w = (a >> 5) + lane; w <= ((b - 1) >> 5); w += 32) {
            uint32_t v = __ldg(p.vstart + w);
            if (w == (a >> 5)) v &= 0xffffffffu << (a & 31);
            if (w == ((b - 1) >> 5)) v &= 0xffffffffu >> (31 - ((b - 1) & 31));
            c += __popc(v);
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
    if (lane == 0) cnt[r] = c;
}

ExtractLaunchFn strict_launcher(const Geometry &ge, int mode, bool hash, bool ragged)
{
    switch (ge.n_limbs) {
    case 1: return get_strict4_launcher_n1(ge.nx, mode, hash, ragged);
    case 2: return get_strict4_launcher_n2(ge.nx, mode, hash, ragged);
    case 3: return get_strict4_launcher_n3(ge.nx, mode, hash, ragged);
    case 4: return get_strict4_launcher_n4(ge.nx, mode, hash, ragged);
    }
    return nullptr;
}

LinLaunchFn lin_launcher(const Geometry &ge, bool hash, bool offsets)
{
    switch (ge.n_limbs) {
    case 1: return get_lin_launcher_n1(hash, offsets);
    case 2: return get_lin_launcher_n2(hash, offsets);
    case 3: return get_lin_launcher_n3(hash, offsets);
    case 4: return get_lin_launcher_n4(hash, offsets);
    }
    return nullptr;
}

CompactLaunchFn compact_launcher(const Geometry &ge, bool hash, bool ragged)
{
    switch (ge.n_limbs) {
    case 1: return get_compact_launcher_n1(ge.nx, hash, ragged);
    case 2: return get_compact_launcher_n2(ge.nx, hash, ragged);
    case 3: return get_compact_launcher_n3(ge.nx, hash, ragged);
    case 4: return get_compact_launcher_n4(ge.nx, hash, ragged);
    }
    return nullptr;
}

} // namespace

cudaError_t fourbit_recode(const uint64_t *words, uint64_t n_words, int k, uint32_t *rec, uint32_t *bad, uint32_t *vstart,
                           uint64_t n_groups, uint64_t n_vstart, cudaStream_t stream, uint32_t *rev)
{
    recode_vstart_kernel<<<static_cast<unsigned>((n_vstart + 256 * kRecodeGroups - 1) / (256 * kRecodeGroups)), 256, 0, stream>>>(words, n_words, k, rec, bad, vstart, n_groups,
                                                                                           n_vstart, rev);
    return cudaGetLastError();
}

uint64_t fourbit_scratch_bytes(const kmc_seqs *s, int k, int mode)
{
    (void)k;
    const uint64_t nb = s->src_bits == 8 ? (s->n_words + 31) / 32 : (s->n_words + 1) / 2; // groups of 32 symbols
    const uint64_t tb = tiles_upper_bound(s);
    uint64_t need = 0;
    need += round_up(8 * (nb + 2), 256);     // rec32
    need += 3 * round_up(4 * (nb + 8), 256); // bad, vstart, err
    need += 4 * kLinChunkWords + 256;        // vstart rounded up to whole chunks of the source-order compaction
    if (mode == KMC_UNAMBIG) need += lin_scratch_bytes(32 * (nb + 2), s->n_seqs) + round_up(8 * (nb + 2), 256) + 256; // + the reversed stream
    need += 3 * 256;                         // err_flat, err_out, total
    need += layout_scratch_bytes(s);
    if (mode == KMC_UNAMBIG) {
        need += round_up(8 * (tb + 1), 256);                                                        // tile_state
        need += round_up(8 * (s->n_seqs + 1), 256) + round_up(8 * scan_tmp_elems(s->n_seqs), 256); // seq_out_offset
    }
    return need + 1024;
}

int32_t fourbit_phase_a(kmc_ctx *ctx, const kmc_seqs *s, int32_t k, int32_t mode, uint32_t flags, const kmc_out *out,
                        cudaStream_t stream, const KnownTotals &known, uint64_t unit_bias, Scratch &scratch,
                        uint64_t *host_small, bool count_first, FourBitState *st)
{
    st->seqs = s;
    st->words4 = s->words;
    st->k = k;
    st->mode = mode;
    st->flags = flags;
    st->ge = geometry(k);
    st->host_small = host_small;
    st->unit_bias = unit_bias;
    st->unambig = (mode == KMC_UNAMBIG);
    st->counted = false;
    host_small[0] = 0;
    host_small[1] = kNone;
    const Geometry &ge = st->ge;
    const bool hash = (flags & KMC_HASH_FX) != 0;

    const bool ascii = s->src_bits == 8;
    // groups of 32 symbols = u32 words of flag bits (4-bit: pairs of source words; ASCII: 32 bytes)
    const uint64_t nb = ascii ? (s->n_words + 31) / 32 : (s->n_words + 1) / 2;
    // UnambiguousKmers over a uniform set that the source-order compaction will take for certain (lin_uniform_ok: no
    // device-side check is needed) reads neither the forward stream nor the flags: the recoding pass then writes only
    // the reversed stream and the valid-start bits -- a third of its traffic less
    const bool rev_only = st->unambig && out && lin_enabled() && known.linear != 0 && lin_uniform_ok(s, k);
    uint32_t *rec = rev_only ? nullptr : static_cast<uint32_t *>(scratch.take(8 * (nb + 2)));
    uint32_t *bad = rev_only ? nullptr : static_cast<uint32_t *>(scratch.take(4 * (nb + 8)));
    uint32_t *vstart = static_cast<uint32_t *>(scratch.take(4 * (lin_chunks(32 * (nb + 2)) * kLinChunkWords + 8)));
    uint32_t *err = (ascii && st->unambig) ? static_cast<uint32_t *>(scratch.take(4 * (nb + 8))) : nullptr;
    if (ascii && st->unambig && !err) return fail(ctx, KMC_E_BAD_ARG, "internal: scratch window too small");
    // UnambiguousKmers: the source-order compaction reads its k-mers from the stream in reversed symbol order
    uint32_t *rev = (st->unambig && out && lin_enabled()) ? static_cast<uint32_t *>(scratch.take(8 * (nb + 2) + 256)) : nullptr;
    if (rev) rev += 64; // (lin_compact2_kernel may read the word before the stream)
    st->err = err;
    unsigned long long *err_flat = static_cast<unsigned long long *>(scratch.take(16)); // [1]: "the recoding pass flagged an error byte"
    uint64_t *err_out = static_cast<uint64_t *>(scratch.take(24));
    if ((!rev_only && (!rec || !bad)) || !vstart || !err_flat || !err_out) return fail(ctx, KMC_E_BAD_ARG, "internal: scratch window too small");
    st->bad = bad;
    st->err_out = err_out;

    if (ascii) {
        const int lut = st->unambig ? 2 : ((flags & KMC_RNA) ? 1 : 0);
        CU(ascii_recode(reinterpret_cast<const uint8_t *>(s->words), s->n_words, lut, k, rec, bad, err, vstart, nb, nb + 2, stream, rev,
                        err ? err_flat + 1 : nullptr));
    } else {
        CU(fourbit_recode(s->words, s->n_words, k, rec, bad, vstart, nb, nb + 2, stream, rev));
    }

    // the set is laid out for the extraction / compaction kernel's G; a count-only call (out == NULL)
    // lays it out in groups of 32 windows
    Geometry lay = ge;
    if (st->unambig && !out) lay.g = kCountLayoutG;
    int32_t rc = plan_layout(ctx, s, k, lay, stream, known, scratch, &st->L);
    if (rc) return rc;
    const Layout &L = st->L;

    ExtractParams p = base_params(s, k, ge, L, unit_bias);
    p.w32 = rec;
    p.nw32 = static_cast<int64_t>(2 * nb);
    p.unit_bits = ascii ? 2 : 32; // offsets are in bytes = symbols (ASCII) or in source words = 16 symbols
    p.vstart = vstart;
    p.err_flat = err_flat;
    st->p = p;
    if (ascii && st->unambig) {
        // every byte of every sequence is read (UnambiguousKmers.jl:109-132), whatever its length
        CU(cudaMemsetAsync(err_flat, 0xff, 8, stream));
        CU(ascii_first_error_seq(st->p, err, s->seq_len, s->uniform_len, err_flat, ctx->sm_count, stream, 0, err_flat + 1));
        CU(cudaMemcpyAsync(&host_small[1], err_flat, 8, cudaMemcpyDeviceToHost, stream));
    }
    if (L.total == 0) {
        if (st->unambig && out && out->seq_out_offset)
            CU(cudaMemsetAsync(out->seq_out_offset, 0, (s->n_seqs + 1) * sizeof(uint64_t), stream));
        return KMC_OK;
    }

    if (!st->unambig) {
        if (L.total > out->capacity) return fail(ctx, KMC_E_OUT_TOO_SMALL, "output capacity smaller than the number of k-mers");
        rc = bind_outputs(ctx, out, mode, flags, &st->p);
        if (rc) return rc;
        CU(cudaMemsetAsync(err_flat, 0xff, 8, stream));
        ExtractLaunchFn fn = strict_launcher(ge, mode, hash, !L.uniform_len);
        if (!fn) return fail(ctx, KMC_E_UNSUPPORTED, "no kernel for this K");
        CU(fn(st->p, ctx->sm_count, stream));
        CU(cudaMemcpyAsync(&host_small[1], err_flat, 8, cudaMemcpyDeviceToHost, stream));
        return KMC_OK;
    }

    // UnambiguousKmers.  Sets whose sequences are ascending and disjoint in the buffer are compacted in source
    // order (lincompact.cuh): the preparation masks the valid-start bits down to window starts and scans the
    // survivors per chunk, so the total is known before the k-mers exist.  Any other layout goes through
    // compact_kernel, which places its tiles itself (the survivors are then counted up front only for callers that
    // need the number before the k-mers exist).
    rc = lin_prepare(ctx, st->p, s, k, nb + 2, rev ? known.linear : 0, &host_small[8], stream, scratch, &st->lin);
    if (rc) return rc;
    st->lin.lp.rev32 = rev;
    st->lin.lp.t_syms = 32 * nb;
    if (rev_only && !st->lin.linear) return fail(ctx, KMC_E_BAD_ARG, "internal: the source-order compaction declined a set it had accepted");
    if (st->lin.linear) {
        st->total_dev = const_cast<unsigned long long *>(reinterpret_cast<const unsigned long long *>(st->lin.total_dev));
        if (count_first || !out) {
            CU(cudaMemcpyAsync(&host_small[0], st->total_dev, 8, cudaMemcpyDeviceToHost, stream));
            st->counted = true;
        }
    } else {
        const uint64_t tiles = (L.items + kTileItems - 1) / kTileItems;
        st->total_dev = static_cast<unsigned long long *>(scratch.take(8));
        st->tile_state = static_cast<unsigned long long *>(scratch.take(8 * (tiles + 2)));
        st->tile_state_buf.reset();
        if (st->total_dev && !st->tile_state) { // more tiles than tiles_upper_bound(): sequences that overlap in the buffer
            st->tile_state_buf = std::make_shared<AsyncBuf>();
            CU(st->tile_state_buf->alloc(ctx, 8 * (tiles + 2), stream));
            st->tile_state = st->tile_state_buf->as<unsigned long long>();
        }
        if (!st->total_dev || !st->tile_state) return fail(ctx, KMC_E_BAD_ARG, "internal: scratch window too small");
        if (count_first || !out) {
            CU(cudaMemsetAsync(st->total_dev, 0, 8, stream));
            CU(count_valid(st->p, !L.uniform_len, lay.g, st->total_dev, stream));
            CU(cudaMemcpyAsync(&host_small[0], st->total_dev, 8, cudaMemcpyDeviceToHost, stream));
            st->counted = true;
        }
    }
    if (out && out->seq_out_offset) {
        uint64_t *cnt = static_cast<uint64_t *>(scratch.take(8 * (s->n_seqs + 1)));
        uint64_t *tmp2 = static_cast<uint64_t *>(scratch.take(8 * scan_tmp_elems(s->n_seqs)));
        if (!cnt || !tmp2) return fail(ctx, KMC_E_BAD_ARG, "internal: scratch window too small");
        const uint64_t threads = s->n_seqs * 32;
        seq_valid_counts_kernel<<<static_cast<unsigned>((threads + 255) / 256), 256, 0, stream>>>(st->p, cnt);
        CU(cudaGetLastError());
        CU(inclusive_offsets_u64(cnt, out->seq_out_offset, s->n_seqs, tmp2, stream));
    }
    return KMC_OK;
}

int32_t fourbit_phase_b(kmc_ctx *ctx, FourBitState *st, const kmc_out *out, cudaStream_t stream, kmc_result *res)
{
    const Layout &L = st->L;
    if (!st->unambig) {
        if (st->host_small[1] != kNone) {
            resolve_error_kernel<<<1, 1, 0, stream>>>(st->p, static_cast<int>(st->seqs->src_bits), st->words4, st->bad,
                                                      st->host_small[1], st->err_out);
            CU(cudaGetLastError());
            CU(cudaMemcpyAsync(&st->host_small[2], st->err_out, 24, cudaMemcpyDeviceToHost, stream));
            CU(cudaStreamSynchronize(stream));
            res->n_written = 0;
            res->err_seq = st->host_small[2];
            res->err_pos = st->host_small[3];
            res->err_sym = static_cast<uint32_t>(st->host_small[4]);
            return fail(ctx, KMC_E_AMBIGUOUS, "cannot encode an uncertain symbol in a 2-bit alphabet");
        }
        res->n_written = L.total;
        return KMC_OK;
    }
    if (st->err && st->host_small[1] != kNone) { // ASCII: a byte outside the skipping table
        CU(ascii_resolve_error(st->p, reinterpret_cast<const uint8_t *>(st->words4), st->err, st->seqs->seq_len,
                               st->seqs->uniform_len, st->host_small[1], st->err_out, stream));
        CU(cudaMemcpyAsync(&st->host_small[4], st->err_out, 24, cudaMemcpyDeviceToHost, stream));
        CU(cudaStreamSynchronize(stream));
        res->n_written = 0;
        res->err_seq = st->host_small[4];
        res->err_pos = st->host_small[5];
        res->err_sym = static_cast<uint32_t>(st->host_small[6]);
        return fail(ctx, KMC_E_AMBIGUOUS, "cannot encode this byte in a 2-bit alphabet");
    }
    res->n_written = 0;
    if (L.total == 0) {
        st->counted = true; // nothing to emit: host_small[0] is already 0
        return KMC_OK;
    }
    if (st->counted) {
        const uint64_t total = st->host_small[0];
        res->n_written = total;
        if (total == 0) return KMC_OK;
        if (total > out->capacity) return fail(ctx, KMC_E_OUT_TOO_SMALL, "output capacity smaller than the number of k-mers");
    }

    // ---- ordered compaction of the surviving windows (forward k-mer + 1-based start) ------------
    ExtractParams p = st->p;
    int32_t rc = bind_outputs(ctx, out, KMC_UNAMBIG, st->flags, &p);
    if (rc) return rc;
    const bool hash = (st->flags & KMC_HASH_FX) != 0;
    if (st->lin.linear) {
        LinParams lp = st->lin.lp;
        lp.capacity = out->capacity;
        LinLaunchFn fn = lin_launcher(st->ge, hash, st->lin.offsets);
        if (!fn) return fail(ctx, KMC_E_UNSUPPORTED, "no kernel for this K");
        CU(fn(p, lp, stream));
    } else {
        const uint64_t tiles = (L.items + kTileItems - 1) / kTileItems;
        CompactParams cp{st->tile_state, reinterpret_cast<uint64_t *>(st->total_dev), out->capacity};
        CU(cudaMemsetAsync(st->tile_state, 0, 8 * (tiles + 1), stream)); // the look-back descriptors and the ticket counter
        CompactLaunchFn fn = compact_launcher(st->ge, hash, !L.uniform_len);
        if (!fn) return fail(ctx, KMC_E_UNSUPPORTED, "no kernel for this K");
        CU(fn(p, cp, stream));
    }
    if (!st->counted) CU(cudaMemcpyAsync(&st->host_small[0], st->total_dev, 8, cudaMemcpyDeviceToHost, stream));
    return KMC_OK;
}

// After the stream has been synchronised: what the compaction emitted (when it was not counted first).
int32_t fourbit_unambig_result(kmc_ctx *ctx, const FourBitState *st, const kmc_out *out, kmc_result *res)
{
    if (!st->unambig || st->counted) return KMC_OK;
    const uint64_t total = st->host_small[0];
    if (total > out->capacity) {
        res->n_written = 0;
        return fail(ctx, KMC_E_OUT_TOO_SMALL, "output capacity smaller than the number of k-mers");
    }
    res->n_written = total;
    return KMC_OK;
}

int32_t extract_device_4bit(kmc_ctx *ctx, const kmc_seqs *s, int32_t k, int32_t mode, uint32_t flags,
                            const kmc_out *out, kmc_result *res, cudaStream_t stream)
{
    int32_t rc = ensure_scratch(ctx, fourbit_scratch_bytes(s, k, mode));
    if (rc) return rc;
    rc = ensure_host_small(ctx);
    if (rc) return rc;
    Scratch scratch{static_cast<char *>(ctx->scratch), ctx->scratch_bytes, 0};
    FourBitState st;
    CU(cudaEventRecord(ctx->ev_k0, stream));
    rc = fourbit_phase_a(ctx, s, k, mode, flags, out, stream, KnownTotals(), 0, scratch, ctx->host_small, false, &st);
    if (rc) return rc;
    // strict modes and ASCII sources can fail: phase B needs the error word.  UnambiguousKmers over a
    // 4-bit source cannot, and its compaction is enqueued right behind the recoding.
    if (!st.unambig || st.err) CU(cudaStreamSynchronize(stream));
    rc = fourbit_phase_b(ctx, &st, out, stream, res);
    if (rc) return rc;
    if (mode != KMC_UNAMBIG && out->seq_out_offset) {
        if (st.L.uniform_len)
            CU(fill_uniform_offsets(out->seq_out_offset, s->n_seqs + 1, st.L.wpr, stream));
        else
            CU(cudaMemcpyAsync(out->seq_out_offset, st.L.win_off, (s->n_seqs + 1) * sizeof(uint64_t), cudaMemcpyDeviceToDevice, stream));
    }
    CU(cudaEventRecord(ctx->ev_k1, stream));
    CU(cudaStreamSynchronize(stream));
    CU(cudaEventElapsedTime(&res->kernel_ms, ctx->ev_k0, ctx->ev_k1));
    return fourbit_unambig_result(ctx, &st, out, res);
}

int32_t count_unambiguous_4bit(kmc_ctx *ctx, const kmc_seqs *s, int32_t k, uint64_t *n_out, cudaStream_t stream)
{
    int32_t rc = ensure_scratch(ctx, fourbit_scratch_bytes(s, k, KMC_UNAMBIG));
    if (rc) return rc;
    rc = ensure_host_small(ctx);
    if (rc) return rc;
    Scratch scratch{static_cast<char *>(ctx->scratch), ctx->scratch_bytes, 0};
    FourBitState st;
    rc = fourbit_phase_a(ctx, s, k, KMC_UNAMBIG, 0, nullptr, stream, KnownTotals(), 0, scratch, ctx->host_small, true, &st);
    if (rc) return rc;
    CU(cudaStreamSynchronize(stream));
    if (st.err && ctx->host_small[1] != kNone) { // ASCII: the iteration would throw before finishing
        kmc_result r{};
        return fourbit_phase_b(ctx, &st, nullptr, stream, &r);
    }
    *n_out = st.L.total ? ctx->host_small[0] : 0;
    return KMC_OK;
}

} // namespace kmc
