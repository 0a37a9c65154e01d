// table_keys.cuh -- the keys of the exact k-mer count tables (sketch.cu) and of their exchange across GPUs (comm.cu).
//
// A one-limb k-mer (K <= 32) is one 64-bit word.  A two-limb k-mer (K = 33..64) is a ulonglong2 {x = limb 0 (the head
// limb, Kmer{A,K,2}.data[1]), y = limb 1}: 16-byte aligned, so that a slot is read by one 128-bit load and claimed by one
// 128-bit compare-and-swap.  A free slot is all ones in every limb; whether a key is free is decided on all its limbs
// (the canonical 64-mer T^32 A^32 has limb 0 = ~0).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "kmer_core.cuh"

namespace kmc {

constexpr uint64_t kEmptyKey = ~0ull;

__host__ __device__ __forceinline__ bool key_free(uint64_t k) { return k == kEmptyKey; }
__host__ __device__ __forceinline__ bool key_free(ulonglong2 k) { return k.x == kEmptyKey && k.y == kEmptyKey; }
__host__ __device__ __forceinline__ bool key_equal(uint64_t a, uint64_t b) { return a == b; }
__host__ __device__ __forceinline__ bool key_equal(ulonglong2 a, ulonglong2 b) { return a.x == b.x && a.y == b.y; }

// fx_hash(k-mer, 0) (src/kmer.jl:255-261): its top bits pick the table slot (and the bin of the binned insert), a
// second mix of it the owner rank of the multi-GPU exchange (comm.cu)
KMC_DEV uint64_t key_hash(uint64_t k)
{
    const uint64_t d[1] = {k};
    return fx_hash<1>(d, 0);
}
// The one definition of a two-limb key's hash that the slot, the bin and the owner are all taken from; host code
// (kmc_kmer_owner2) computes it too, so it is plain arithmetic rather than kmer_core.cuh's device-only fx_hash<2>.
__host__ __device__ __forceinline__ uint64_t key_hash(ulonglong2 k)
{
    uint64_t h = k.x * FX_CONSTANT; // limb 0 first: (rotl(0, 5) ^ limb0) * FX
    h = (((h << 5) | (h >> 59)) ^ k.y) * FX_CONSTANT;
    return h;
}

} // namespace kmc
