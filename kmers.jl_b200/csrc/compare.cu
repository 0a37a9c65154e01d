// compare.cu -- kmc_minhash_compare: every bottom-s sketch of list A against every sketch of list B (DESIGN.md 3.2d).
//
// For a pair (A_i, B_j) of ascending, distinct rows the kernel counts
//   shared        = |A_i ∩ B_j|
//   shared_bottom = |S_s(A_i ∪ B_j) ∩ A_i ∩ B_j|      (S_s = the s smallest values: Mash's estimator numerator)
// A block holds TA rows of A in shared memory and its warps stream rows of B.  A lane takes one element x = B_j[t] and
// finds a = |{y in A_i : y < x}| by a binary search in each of the TA rows, the TA searches interleaved step by step so
// that one lane has TA independent shared-memory loads in flight.  x is in A_i when A_i[a] == x; a warp prefix over
// those ballots gives c = |{y in A_i ∩ B_j : y < x}|, so a + t - c is x's rank in A_i ∪ B_j and x counts towards
// shared_bottom exactly when x is in A_i and a + t - c < s.  Each element of B is loaded once for TA pairs.
#include <algorithm>

#include "plan.h"

namespace kmc {

namespace {

constexpr int kCompareThreads = 256;
constexpr uint32_t kCompareMaxS = 16384;          // one row of A is at most 128 KB of shared memory
constexpr uint64_t kCompareTileBytes = 96 << 10;  // A rows per block: as many as fit here, up to 8 (at least one)
constexpr uint64_t kCompareBRows = 64;            // rows of B per block

template <int TA>
__global__ void __launch_bounds__(kCompareThreads) minhash_compare_kernel(const uint64_t *__restrict__ a, const uint32_t *__restrict__ a_n,
                                                                          uint64_t n_a, const uint64_t *__restrict__ b,
                                                                          const uint32_t *__restrict__ b_n, uint64_t n_b, uint32_t s,
                                                                          uint64_t b_rows, uint32_t *__restrict__ shared,
                                                                          uint32_t *__restrict__ shared_bottom)
{
    extern __shared__ uint64_t s_a[]; // [TA][s]
    const uint64_t i0 = static_cast<uint64_t>(blockIdx.x) * TA;
    uint32_t len[TA];
    uint32_t longest = 0;
#pragma unroll
    for (int i = 0; i < TA; ++i) {
        len[i] = i0 + i < n_a ? min(__ldg(a_n + i0 + i), s) : 0u;
        longest = max(longest, len[i]);
    }
    // a row is read up to its length only
#pragma unroll
    for (int i = 0; i < TA; ++i)
        for (uint32_t t = threadIdx.x; t < len[i]; t += kCompareThreads) s_a[static_cast<uint64_t>(i) * s + t] = __ldg(a + (i0 + i) * s + t);
    __syncthreads();
    // the largest power of two not above the longest row: the first step of the lower-bound search (the steps sum to at
    // least any row's length)
    const uint32_t top = longest ? 1u << (31 - __clz(longest)) : 0u;

    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x / 32;
    const uint32_t lower = (1u << lane) - 1u;
    const uint64_t j_end = min(n_b, (static_cast<uint64_t>(blockIdx.y) + 1) * b_rows);
    for (uint64_t j = static_cast<uint64_t>(blockIdx.y) * b_rows + warp; j < j_end; j += kCompareThreads / 32) {
        const uint32_t nb = min(__ldg(b_n + j), s);
        const uint64_t *brow = b + j * s;
        uint32_t n_shared[TA], n_bottom[TA]; // warp-uniform
#pragma unroll
        for (int i = 0; i < TA; ++i) n_shared[i] = n_bottom[i] = 0;
        for (uint32_t t0 = 0; t0 < nb; t0 += 32) {
            const uint32_t t = t0 + lane;
            const bool in = t < nb;
            const uint64_t x = in ? __ldg(brow + t) : 0;
            uint32_t lo[TA];
#pragma unroll
            for (int i = 0; i < TA; ++i) lo[i] = 0;
            for (uint32_t step = top; step; step >>= 1) {
#pragma unroll
                for (int i = 0; i < TA; ++i) {
                    const uint32_t q = lo[i] + step;
                    if (q <= len[i] && s_a[static_cast<uint64_t>(i) * s + q - 1] < x) lo[i] = q;
                }
            }
#pragma unroll
            for (int i = 0; i < TA; ++i) {
                const bool found = in && lo[i] < len[i] && s_a[static_cast<uint64_t>(i) * s + lo[i]] == x;
                const uint32_t m = __ballot_sync(0xffffffffu, found);
                const uint32_t c = n_shared[i] + __popc(m & lower); // |A ∩ B| below x
                const bool bottom = found && lo[i] + t - c < s;
                n_shared[i] += __popc(m);
                n_bottom[i] += __popc(__ballot_sync(0xffffffffu, bottom));
            }
        }
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < TA; ++i) {
                if (i0 + i >= n_a) break;
                const uint64_t at = (i0 + i) * n_b + j;
                if (shared) shared[at] = n_shared[i];
                if (shared_bottom) shared_bottom[at] = n_bottom[i];
            }
        }
    }
}

template <int TA>
cudaError_t launch_compare(const uint64_t *a, const uint32_t *a_n, uint64_t n_a, const uint64_t *b, const uint32_t *b_n, uint64_t n_b,
                           uint32_t s, uint32_t *shared, uint32_t *shared_bottom, cudaStream_t stream)
{
    const size_t smem = static_cast<size_t>(TA) * s * 8;
    cudaError_t e = cudaFuncSetAttribute(minhash_compare_kernel<TA>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    // grid.y is at most 65535: more rows of B per block for very long lists
    const uint64_t b_rows = std::max<uint64_t>(kCompareBRows, (n_b + 65534) / 65535);
    const dim3 grid(static_cast<unsigned>((n_a + TA - 1) / TA), static_cast<unsigned>((n_b + b_rows - 1) / b_rows));
    minhash_compare_kernel<TA><<<grid, kCompareThreads, smem, stream>>>(a, a_n, n_a, b, b_n, n_b, s, b_rows, shared, shared_bottom);
    return cudaGetLastError();
}

} // namespace

} // namespace kmc

using namespace kmc;

extern "C" int32_t kmc_minhash_compare(kmc_ctx *ctx, const uint64_t *a, const uint32_t *a_n, uint64_t n_a, const uint64_t *b,
                                       const uint32_t *b_n, uint64_t n_b, uint64_t s, uint32_t *shared, uint32_t *shared_bottom)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (s < 1) return fail(ctx, KMC_E_BAD_ARG, "the sketch size must be at least 1");
    if (s > kCompareMaxS) return fail(ctx, KMC_E_UNSUPPORTED, "kmc_minhash_compare supports s <= 16384");
    if (n_a == 0 || n_b == 0) return KMC_OK;
    if (!a || !a_n || !b || !b_n) return fail(ctx, KMC_E_BAD_ARG, "a / a_n / b / b_n is NULL");
    if (n_a > ~0ull / n_b || n_a > 0x7fffffffull) return fail(ctx, KMC_E_BAD_ARG, "n_a * n_b is too large");
    if (!shared && !shared_bottom) return KMC_OK;
    CU(cudaSetDevice(ctx->device));
    cudaStream_t stream = ctx->stream;
    const uint64_t fit = kCompareTileBytes / (8 * s);
    const uint32_t s32 = static_cast<uint32_t>(s);
    if (fit >= 8) CU(launch_compare<8>(a, a_n, n_a, b, b_n, n_b, s32, shared, shared_bottom, stream));
    else if (fit >= 4) CU(launch_compare<4>(a, a_n, n_a, b, b_n, n_b, s32, shared, shared_bottom, stream));
    else if (fit >= 2) CU(launch_compare<2>(a, a_n, n_a, b, b_n, n_b, s32, shared, shared_bottom, stream));
    else CU(launch_compare<1>(a, a_n, n_a, b, b_n, n_b, s32, shared, shared_bottom, stream));
    CU(cudaStreamSynchronize(stream));
    return KMC_OK;
}
