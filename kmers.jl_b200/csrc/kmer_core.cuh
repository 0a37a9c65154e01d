// kmer_core.cuh -- register-level k-mer primitives for sm_100a.
//
// The reference derives k-mer i from k-mer i-1 (shift_encoding,
// src/construction_utils.jl:129-134; shift_first_encoding, src/kmer.jl:511-518).  Here every
// window is computed independently from the packed sequence words:
//
//   Let S be the little-endian 2-bit stream of a LongSequence (symbol i at bits [2i, 2i+2)) and
//   W_p = S[2p, 2p+2K) the raw bits of the window starting at symbol p.  Because LongSequence
//   stores the first symbol in the LOWEST bits while Kmer stores it in the HIGHEST,
//     reverse-complement k-mer  rv = ~W_p  (masked to 2K bits)          -- no bit reversal at all
//     forward k-mer             fw = rev2(W_p)  (order of 2-bit groups reversed)
//   (the closed form the reference itself uses in build_kmer(::Copyable), src/construction.jl:213-219:
//   reversebits of the raw words, right-aligned).
//
// A thread owns G consecutive windows.  It loads a block of NX 32-bit words that covers the
// 2K + 2(G-1) bits of its windows, aligns it once with funnel shifts, bit-reverses the block once,
// and then every window is two static funnel shifts per 32-bit half:
//   x-stream (aligned to the first window) -> rv_j  = ~(x >> 2j)
//   t-stream (rev2 of the block, aligned to the LAST window) -> fw_j = t >> 2(G-1-j)
// NX is a template parameter chosen as ceil((2K + 2G - 2) / 32) so that every word index is a
// compile-time constant (registers, never local memory) and the run-time alignment shifts are < 32.
#pragma once
#include <cstdint>

namespace kmc {

#define KMC_DEV __device__ __forceinline__

constexpr uint64_t FX_CONSTANT = 0x517cc1b727220a95ull; // src/kmer.jl:218

// Windows per work item (= per thread) for k-mers of n limbs.  G*n*8 bytes is a multiple of 32, so
// a full group goes out as whole 256-bit stores; 64-96 bytes per thread and stream amortise the
// per-item address arithmetic over more windows (profiles/: G = 4 -> 8 for one limb).
#ifndef KMC_GROUP_1
#define KMC_GROUP_1 8
#define KMC_GROUP_2 4
#define KMC_GROUP_3 4
#define KMC_GROUP_4 2
#endif
constexpr int group_of(int n) { return n == 1 ? KMC_GROUP_1 : n == 2 ? KMC_GROUP_2 : n == 3 ? KMC_GROUP_3 : KMC_GROUP_4; }

// The shape of a work item for K symbols of bps bits: limbs, windows per item, 32-bit words per block, and the
// two constants block_kmers needs.  Plain host code (the launch planner, plan.h) -- here so that the CPU test of
// these primitives (tests/host_core) takes the geometry from the same place as the kernels' launchers.
struct Geometry {
    int n_limbs, g, nx;
    uint32_t s0;
    uint64_t head_mask;
};

// src/kmer.jl:117-137 (N = cld(K * bps, 64)) and :603-605 (get_mask); bps = bits per symbol of the k-mer alphabet
// g = 0: the group size of the limb count (group_of); otherwise the given one (the AoS kernels use smaller groups)
inline Geometry geometry(int k, int bps = 2, int g = 0)
{
    Geometry ge;
    ge.n_limbs = (bps * k + 63) / 64;
    ge.g = g > 0 ? g : group_of(ge.n_limbs);
    ge.nx = (bps * k + bps * ge.g - bps + 31) / 32;
    ge.s0 = static_cast<uint32_t>(32 * ge.nx - bps * k - bps * (ge.g - 1));
    int used = bps * k - 64 * (ge.n_limbs - 1); // bits used in the head limb, bps..64
    ge.head_mask = used >= 64 ? ~0ull : ((1ull << used) - 1);
    return ge;
}

// Work item -> (read, group within the read) -> stream bit for an aligned uniform set: every read owns gprm groups of G
// windows, none of which straddles two reads.  The quotient item / gprm comes from a multiply-high by
// magic = floor(2^32 / gprm) (2^32 - 1 for gprm = 1) and one correction step: the estimate is the quotient or one below
// it for every item < 2^32 and gprm < 2^31.
inline uint32_t aligned_magic(uint64_t gprm) { return gprm == 1 ? 0xffffffffu : static_cast<uint32_t>(0x100000000ull / gprm); }

template <int G, int BPS> struct AlignedLocator {
    uint32_t gprm, magic, read_bits;
    uint64_t first_bits;
    KMC_DEV AlignedLocator(uint32_t gprm_, uint32_t magic_, uint32_t read_bits_, uint32_t first_symbol)
        : gprm(gprm_), magic(magic_), read_bits(read_bits_), first_bits(static_cast<uint64_t>(BPS) * first_symbol)
    {
    }
    // bit offset in the stream of the item's first symbol; gi = the item's group within its read
    KMC_DEV uint64_t bit_of(uint32_t item, uint32_t &gi) const
    {
        uint32_t r = __umulhi(item, magic); // the quotient or one below it
        gi = item - r * gprm;
        if (gi >= gprm) {
            gi -= gprm;
            ++r;
        }
        return static_cast<uint64_t>(r) * read_bits + (first_bits + gi * static_cast<uint32_t>(G * BPS));
    }
    KMC_DEV uint64_t bit_of(uint32_t item) const
    {
        uint32_t gi;
        return bit_of(item, gi);
    }
    // the read that owns the item: the quotient bit_of computes
    KMC_DEV uint32_t read_of(uint32_t item) const
    {
        const uint32_t r = __umulhi(item, magic);
        return item - r * gprm >= gprm ? r + 1 : r;
    }
};

// reversebits(x, BitsPerSymbol{2}) on a 32-bit word: reverse the order of the 16 two-bit groups.
KMC_DEV uint32_t rev2_32(uint32_t x)
{
    x = __brev(x);
    return ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
}

// 4-bit alphabets (Kmer{DNAAlphabet{4}} / Kmer{RNAAlphabet{4}}, SURVEY.md 8f rank 3).  The closed form is
// the same with nibbles for bit pairs: LongSequence stores the first symbol lowest, Kmer highest, so
//   forward k-mer             fw = rev4(W)   reversebits(x, BitsPerSymbol{4}): nibble order reversed
//   reverse-complement k-mer  rv = comp4(W)  complement_bitpar for 4-bit alphabets reverses the four
//                                            bits of every nibble (A=1<->T=8, C=2<->G=4, IUPAC sets
//                                            likewise; src/transformations.jl:14-18) -- in place
KMC_DEV uint32_t rev4_32(uint32_t x)
{
    x = __byte_perm(x, 0u, 0x0123);
    return ((x >> 4) & 0x0f0f0f0fu) | ((x & 0x0f0f0f0fu) << 4);
}
KMC_DEV uint32_t comp4_32(uint32_t x) { return __brev(rev4_32(x)); }

KMC_DEV uint64_t pack64(uint32_t lo, uint32_t hi) { return (static_cast<uint64_t>(hi) << 32) | lo; }

// 64 bits of a 32-bit-word stream starting at bit offset `off`.  `off` is a compile-time
// constant at every call site once the caller's loops are unrolled, so all indices are static
// (words past the end of the block read as zero; they only ever feed masked-out bits).
template <int NW>
KMC_DEV uint64_t stream64(const uint32_t (&s)[NW], int off)
{
    const int c = off >> 5, sh = off & 31;
    auto W = [&](int i) -> uint32_t { return i < NW ? s[i < NW ? i : 0] : 0u; };
    uint32_t lo, hi;
    if (sh == 0) {
        lo = W(c);
        hi = W(c + 1);
    } else {
        lo = __funnelshift_r(W(c), W(c + 1), sh);
        hi = __funnelshift_r(W(c + 1), W(c + 2), sh);
    }
    return pack64(lo, hi);
}

// cmp(x.data, y.data) == -1 (src/kmer.jl:176-201): limb-lexicographic, head first.
template <int N>
KMC_DEV bool limbs_less(const uint64_t (&a)[N], const uint64_t (&b)[N])
{
    bool lt = false, decided = false;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        lt = lt || (!decided && a[i] < b[i]);
        decided = decided || (a[i] != b[i]);
    }
    return lt;
}

// x * C mod 2^64 for a compile-time C.  On the device: one 32 x 32 -> 64-bit product and two multiply-adds into its high
// half (the compiler's own expansion takes a fourth instruction; fx_hash runs this once per k-mer and limb).
template <uint64_t C> KMC_DEV uint64_t mul_c64(uint64_t x)
{
#ifdef __CUDA_ARCH__
    uint64_t r;
    asm("{\n\t"
        ".reg .u32 xl, xh, pl, ph;\n\t"
        "mov.b64 {xl, xh}, %1;\n\t"
        "mul.lo.u32 pl, xl, %2;\n\t"
        "mul.hi.u32 ph, xl, %2;\n\t"
        "mad.lo.u32 ph, xh, %2, ph;\n\t"
        "mad.lo.u32 ph, xl, %3, ph;\n\t"
        "mov.b64 %0, {pl, ph};\n\t"
        "}"
        : "=l"(r)
        : "l"(x), "n"(static_cast<uint32_t>(C)), "n"(static_cast<uint32_t>(C >> 32)));
    return r;
#else
    return x * C;
#endif
}
KMC_DEV uint64_t mul_fx(uint64_t x) { return mul_c64<FX_CONSTANT>(x); }

// fx_hash (src/kmer.jl:255-261)
template <int N>
KMC_DEV uint64_t fx_hash(const uint64_t (&d)[N], uint64_t h)
{
#pragma unroll
    for (int i = 0; i < N; ++i) h = mul_fx(((h << 5) | (h >> 59)) ^ d[i]);
    return h;
}

// ---- streaming stores --------------------------------------------------------------------
// The output streams are written once and never read by the kernel that writes them: no L1 allocation, and
// first in line for eviction from L2 (so that they do not displace the prefetched source, extract_kernels.cuh).
// kEvictFirst is what `createpolicy.fractional.L2::evict_first.b64 p, 1.0` returns (a constant encoding).
#ifndef KMC_STORE_EVICT_FIRST
#define KMC_STORE_EVICT_FIRST 1
#endif
constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;

KMC_DEV void st_u64(uint64_t *p, uint64_t v)
{
#if KMC_STORE_EVICT_FIRST
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.u64 [%0], %1, %2;" ::"l"(p), "l"(v), "l"(kEvictFirst) : "memory");
#else
    asm volatile("st.global.L1::no_allocate.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
#endif
}
KMC_DEV void st_v2(uint64_t *p, uint64_t a, uint64_t b)
{
#if KMC_STORE_EVICT_FIRST
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v2.u64 [%0], {%1,%2}, %3;" ::"l"(p), "l"(a), "l"(b), "l"(kEvictFirst)
                 : "memory");
#else
    asm volatile("st.global.L1::no_allocate.v2.u64 [%0], {%1,%2};" ::"l"(p), "l"(a), "l"(b) : "memory");
#endif
}
// 256-bit store: one STG.E.256 on sm_100a
KMC_DEV void st_v4(uint64_t *p, uint64_t a, uint64_t b, uint64_t c, uint64_t d)
{
#if KMC_STORE_EVICT_FIRST
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v4.u64 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "l"(a), "l"(b), "l"(c), "l"(d),
                 "l"(kEvictFirst)
                 : "memory");
#else
    asm volatile("st.global.L1::no_allocate.v4.u64 [%0], {%1,%2,%3,%4};" ::"l"(p), "l"(a), "l"(b), "l"(c), "l"(d)
                 : "memory");
#endif
}

// CNT contiguous u64 values; `aligned32` says p is 32-byte aligned.
template <int CNT>
KMC_DEV void store_run(uint64_t *p, const uint64_t (&v)[CNT], bool aligned32)
{
    if (CNT % 4 == 0 && aligned32) {
#pragma unroll
        for (int i = 0; i + 3 < CNT; i += 4) st_v4(p + i, v[i], v[i + 1], v[i + 2], v[i + 3]);
    } else if (CNT % 2 == 0 && (reinterpret_cast<uintptr_t>(p) & 15) == 0) {
#pragma unroll
        for (int i = 0; i + 1 < CNT; i += 2) st_v2(p + i, v[i], v[i + 1]);
    } else {
#pragma unroll
        for (int i = 0; i < CNT; ++i) st_u64(p + i, v[i]);
    }
}

// CNT words staged for the address p; only the words [lo, hi) are to be written.
//   fast     all of them, and p is 32-byte aligned (whole 256-bit stores when CNT % 4 == 0)
//   base_ok  the stream's base pointer is 32-byte aligned, so p is aligned to CNT*8 bytes (mod 32):
//            aligned quads / pairs that lie inside [lo, hi) still go out as 256- / 128-bit stores
template <int CNT>
KMC_DEV void store_words(uint64_t *p, const uint64_t (&v)[CNT], int lo, int hi, bool fast, bool base_ok)
{
    if (fast) {
        store_run<CNT>(p, v, CNT % 4 == 0);
        return;
    }
    const bool quad_ok = base_ok && (CNT % 4 == 0), pair_ok = base_ok && (CNT % 2 == 0);
#pragma unroll
    for (int i = 0; i < CNT; i += 4) {
        if (i + 4 <= CNT && quad_ok && lo <= i && hi >= i + 4) {
            st_v4(p + i, v[i], v[i + 1], v[i + 2], v[i + 3]);
            continue;
        }
#pragma unroll
        for (int j = i; j < i + 4 && j < CNT; j += 2) {
            if (j + 2 <= CNT && pair_ok && lo <= j && hi >= j + 2) {
                st_v2(p + j, v[j], v[j + 1]);
            } else {
                if (j >= lo && j < hi) st_u64(p + j, v[j]);
                if (j + 1 < CNT && j + 1 >= lo && j + 1 < hi) st_u64(p + j + 1, v[j + 1]);
            }
        }
    }
}

// Base.hash(x::Kmer, h) = hash(x.data, h ⊻ K) (src/kmer.jl:206) with the tuple / UInt64 hashing of Julia 1.10 and
// 1.11 (misc_kernels.cu: base_hash_kernel folds the limbs from the last to the first):
//   hash(::Tuple{}, h) = h + 0x77cfa1eef01bca90 ; hash(t::Tuple, h) = hash(t[1], hash(tail(t), h))   (tuple.jl)
//   hash(x::UInt64, h) = hash_64_64(x) - 3h                                                          (hashing.jl)
KMC_DEV uint64_t hash_64_64(uint64_t a)
{
    a = ~a + (a << 21);
    a = a ^ (a >> 24);
    a = a + (a << 3) + (a << 8);
    a = a ^ (a >> 14);
    a = a + (a << 2) + (a << 4);
    a = a ^ (a >> 28);
    a = a + (a << 31);
    return a;
}
KMC_DEV uint64_t base_hash_seed(uint64_t h) { return h + 0x77cfa1eef01bca90ull; }
KMC_DEV uint64_t base_hash_fold(uint64_t limb, uint64_t acc) { return hash_64_64(limb) - 3 * acc; }

// ---- the window block ----------------------------------------------------------------------
// Loads NX+1 words at 32-bit word index floor(bit/32) (clamped into [0, nw32) so that slots
// outside the sequence buffer never fault; such bits only ever feed windows that are not
// emitted) and produces the aligned x-stream.
template <int NX>
KMC_DEV void load_raw(const uint32_t *__restrict__ w32, int64_t nw32, int64_t bit, uint32_t (&a)[NX + 1])
{
    const int64_t idx = bit >> 5;
    if (idx >= 0 && idx + NX < nw32) {
#pragma unroll
        for (int i = 0; i <= NX; ++i) a[i] = __ldg(w32 + idx + i);
    } else {
#pragma unroll
        for (int i = 0; i <= NX; ++i) {
            int64_t k = idx + i;
            k = k < 0 ? 0 : (k >= nw32 ? nw32 - 1 : k);
            a[i] = __ldg(w32 + k);
        }
    }
}

template <int NX>
KMC_DEV void load_block(const uint32_t *__restrict__ w32, int64_t nw32, int64_t bit, uint32_t (&x)[NX])
{
    uint32_t a[NX + 1];
    load_raw<NX>(w32, nw32, bit, a);
    const uint32_t s = static_cast<uint32_t>(bit) & 31u;
#pragma unroll
    for (int i = 0; i < NX; ++i) x[i] = __funnelshift_r(a[i], a[i + 1], s);
}

// fw[j] / rv[j] for the G windows of a block, limbs head first.  BPS = bits per symbol of the k-mer
// alphabet (and of the stream): 2 or 4.
//   s0        = 32*NX - BPS*K - BPS*(G-1), in [0, 32)
//   head_mask = get_mask (src/kmer.jl:603-605)
// The head limb holds BPS*K - 64(N-1) bits, and a block of NX words only serves K with BPS*K + BPS*(G-1) > 32(NX-1): where
// that leaves at least 32 bits in the head limb, the low half of head_mask is all ones and only the high half is applied.
template <int N, int NX, int G, int BPS> KMC_DEV uint64_t mask_head(uint64_t v, uint64_t head_mask)
{
    constexpr bool kLoFull = 32 * (NX - 1) - BPS * (G - 1) + 1 - 64 * (N - 1) >= 32;
    if (kLoFull) return pack64(static_cast<uint32_t>(v), static_cast<uint32_t>(v >> 32) & static_cast<uint32_t>(head_mask >> 32));
    return v & head_mask;
}

template <int N, int NX, int G, bool WANT_FW, bool WANT_RV, int BPS = 2>
KMC_DEV void block_kmers(const uint32_t (&x)[NX], uint32_t s0, uint64_t head_mask, uint64_t (&fw)[G][N],
                         uint64_t (&rv)[G][N])
{
    if (WANT_RV) {
        // complement once per block (complement_bitpar for 2-bit alphabets is ~x,
        // src/transformations.jl:21-25), then each window is a static funnel shift.
        uint32_t nx[NX];
#pragma unroll
        for (int i = 0; i < NX; ++i) nx[i] = BPS == 2 ? ~x[i] : comp4_32(x[i]);
#pragma unroll
        for (int j = 0; j < G; ++j) {
#pragma unroll
            for (int m = 0; m < N; ++m) { // m = 0 is the least significant limb
                uint64_t v = stream64<NX>(nx, BPS * j + 64 * m);
                if (m == N - 1) v = mask_head<N, NX, G, BPS>(v, head_mask);
                rv[j][N - 1 - m] = v;
            }
        }
    }
    if (WANT_FW) {
        // rev2 of the whole block: symbol i of the x-stream lands at symbol 16*NX-1-i.
        uint32_t y[NX];
#pragma unroll
        for (int i = 0; i < NX; ++i) y[i] = BPS == 2 ? rev2_32(x[NX - 1 - i]) : rev4_32(x[NX - 1 - i]);
        // drop the s0 bits that lie beyond the last window
        uint32_t t[NX];
#pragma unroll
        for (int i = 0; i < NX; ++i) t[i] = __funnelshift_r(y[i], i + 1 < NX ? y[i + 1 < NX ? i + 1 : 0] : 0u, s0);
#pragma unroll
        for (int j = 0; j < G; ++j) {
#pragma unroll
            for (int m = 0; m < N; ++m) {
                uint64_t v = stream64<NX>(t, BPS * (G - 1 - j) + 64 * m);
                if (m == N - 1) v = mask_head<N, NX, G, BPS>(v, head_mask);
                fw[j][N - 1 - m] = v;
            }
        }
    }
}

} // namespace kmc
