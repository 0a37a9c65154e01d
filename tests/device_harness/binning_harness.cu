// binning_harness.cu -- the device half of tests/test_gpu_binning.py: binning.cuh's partition and apply_groups, called
// through a plain C interface with the bin functors the library uses (IdBin for 32-bit bucket ids, KmerHashBin for
// one-limb and KmerHashBin2 for two-limb k-mers).  Every entry point allocates, copies and frees its own device memory
// and returns a cudaError_t, so the caller hands over host arrays only.  Test infrastructure: the library does not link
// it, and nothing in binning.cuh is changed for it.
//
// nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 --expt-relaxed-constexpr -Xcompiler -fPIC -shared
//      -I kmers.jl_b200/csrc tests/device_harness/binning_harness.cu kmers.jl_b200/csrc/scan.cu -o libbinning_harness.so
#include <cuda_runtime.h>

#include <cstdint>
#include <cstring>
#include <vector>

#include "binning.cuh"

using namespace kmc;

namespace {

constexpr uint64_t kGuardBytes = 4096;
constexpr unsigned char kSentinel = 0xA5;

// device memory freed on every return path
struct DevMem {
    void *p = nullptr;
    cudaError_t alloc(uint64_t bytes) { return cudaMalloc(&p, bytes ? bytes : 16); }
    template <typename T> T *as() const { return static_cast<T *>(p); }
    DevMem() = default;
    DevMem(const DevMem &) = delete;
    DevMem &operator=(const DevMem &) = delete;
    ~DevMem()
    {
        if (p) cudaFree(p);
    }
};

struct Stream {
    cudaStream_t s = nullptr;
    cudaError_t create() { return cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking); }
    ~Stream()
    {
        if (s) cudaStreamDestroy(s);
    }
};

#define TRY(x)                                                                                                                   \
    do {                                                                                                                         \
        const cudaError_t e_ = (x);                                                                                              \
        if (e_ != cudaSuccess) return e_;                                                                                        \
    } while (0)

template <typename Key> struct BinOfWidth;
template <> struct BinOfWidth<uint32_t> {
    static binning::IdBin make(int p, int shift) { return binning::IdBin{shift}; }
};
template <> struct BinOfWidth<uint64_t> {
    static binning::KmerHashBin make(int p, int) { return binning::KmerHashBin{64 - p}; }
};
template <> struct BinOfWidth<ulonglong2> {
    static binning::KmerHashBin2 make(int p, int) { return binning::KmerHashBin2{64 - p}; }
};

template <typename Key> cudaError_t partition_once(int p, int shift, const void *in, uint64_t n, void *out, uint64_t *offs,
                                                    uint64_t *matrix, int *guard_ok, int *input_ok)
{
    *guard_ok = 0;
    *input_ok = 0;
    const uint64_t bytes = n * sizeof(Key), cells = binning::matrix_cells<Key>(n, p);
    DevMem d_in, d_out, d_matrix, d_offs, d_scan;
    TRY(d_in.alloc(bytes));
    TRY(d_out.alloc(bytes + kGuardBytes));
    TRY(d_matrix.alloc((cells + 1) * 8));
    TRY(d_offs.alloc((cells + 2) * 8));
    TRY(d_scan.alloc((scan_tmp_elems(cells) + 1) * 8));
    Stream st;
    TRY(st.create());
    if (bytes) TRY(cudaMemcpyAsync(d_in.p, in, bytes, cudaMemcpyHostToDevice, st.s));
    TRY(cudaMemsetAsync(d_out.p, kSentinel, bytes + kGuardBytes, st.s));
    TRY(cudaMemsetAsync(d_matrix.p, 0xff, (cells + 1) * 8, st.s));
    TRY(cudaMemsetAsync(d_offs.p, 0xff, (cells + 2) * 8, st.s));
    TRY(binning::partition<Key>(d_in.as<const Key>(), n, p, BinOfWidth<Key>::make(p, shift), d_out.as<Key>(), d_matrix.as<uint64_t>(),
                                d_offs.as<uint64_t>(), d_scan.as<uint64_t>(), st.s));
    std::vector<unsigned char> back(bytes > kGuardBytes ? bytes : kGuardBytes);
    if (bytes) TRY(cudaMemcpyAsync(out, d_out.p, bytes, cudaMemcpyDeviceToHost, st.s));
    if (cells) TRY(cudaMemcpyAsync(matrix, d_matrix.p, cells * 8, cudaMemcpyDeviceToHost, st.s));
    TRY(cudaMemcpyAsync(offs, d_offs.p, (cells + 1) * 8, cudaMemcpyDeviceToHost, st.s));
    TRY(cudaMemcpyAsync(back.data(), d_out.as<unsigned char>() + bytes, kGuardBytes, cudaMemcpyDeviceToHost, st.s));
    TRY(cudaStreamSynchronize(st.s));
    bool guard = true;
    for (uint64_t i = 0; i < kGuardBytes; ++i) guard = guard && back[i] == kSentinel;
    if (bytes) TRY(cudaMemcpyAsync(back.data(), d_in.p, bytes, cudaMemcpyDeviceToHost, st.s));
    TRY(cudaStreamSynchronize(st.s));
    *guard_ok = guard ? 1 : 0;
    *input_ok = (bytes == 0 || std::memcmp(back.data(), in, bytes) == 0) ? 1 : 0;
    return cudaSuccess;
}

// ------------------------------------------------------------------------------------------- the large, device-verified case
__device__ __forceinline__ uint64_t mix64(uint64_t z)
{
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

__device__ __forceinline__ void make_key(uint64_t seed, uint64_t i, uint32_t &k) { k = static_cast<uint32_t>(mix64(seed + i) >> 17); }
__device__ __forceinline__ void make_key(uint64_t seed, uint64_t i, uint64_t &k) { k = mix64(seed + i); }
__device__ __forceinline__ void make_key(uint64_t seed, uint64_t i, ulonglong2 &k)
{
    k = make_ulonglong2(mix64(seed + 2 * i), mix64(seed + 2 * i + 1));
}

// what a key adds to the fingerprints of its bin: itself, spread over 64 bits
__device__ __forceinline__ uint64_t key_print(uint32_t k) { return mix64(k + 0x9e3779b97f4a7c15ull); }
__device__ __forceinline__ uint64_t key_print(uint64_t k) { return mix64(k + 0x9e3779b97f4a7c15ull); }
__device__ __forceinline__ uint64_t key_print(ulonglong2 k) { return mix64(mix64(k.x + 0x9e3779b97f4a7c15ull) ^ k.y); }

template <typename Key> __global__ void generate_kernel(Key *keys, uint64_t n, uint64_t seed)
{
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<uint64_t>(gridDim.x) * blockDim.x)
        make_key(seed, i, keys[i]);
}

// per bin: count, xor and wrapping sum of key_print.  by_position: the bin of keys[i] is the bin whose range of the
// partitioned output holds i (starts[b] .. starts[b + 1]), and a key whose own bin differs is counted in *misplaced;
// otherwise the bin is the key's own.
constexpr int kMaxBins = 1 << binning::kMaxBits;
template <typename Key, typename BinOf>
__global__ void __launch_bounds__(256) bin_stats_kernel(const Key *__restrict__ keys, uint64_t n, BinOf bin_of, int n_bins,
                                                       const uint64_t *__restrict__ starts, bool by_position, unsigned long long *stats,
                                                       unsigned long long *misplaced)
{
    __shared__ unsigned long long s_cnt[kMaxBins], s_xor[kMaxBins], s_sum[kMaxBins];
    __shared__ uint64_t s_start[kMaxBins + 1];
    for (int b = threadIdx.x; b < n_bins; b += blockDim.x) s_cnt[b] = s_xor[b] = s_sum[b] = 0;
    if (by_position)
        for (int b = threadIdx.x; b <= n_bins; b += blockDim.x) s_start[b] = starts[b];
    __syncthreads();
    unsigned long long bad = 0;
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const Key k = keys[i];
        const uint32_t own = bin_of(k);
        uint32_t b = own;
        if (by_position) { // largest b with s_start[b] <= i
            int lo = 0, hi = n_bins;
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if (s_start[mid] <= i) lo = mid; else hi = mid;
            }
            b = static_cast<uint32_t>(lo);
            bad += b != own;
        }
        if (b >= static_cast<uint32_t>(n_bins)) { // (a key of a bin that does not exist: count it, keep the stats in range)
            bad += 1;
            continue;
        }
        const uint64_t f = key_print(k);
        atomicAdd(&s_cnt[b], 1ull);
        atomicXor(&s_xor[b], static_cast<unsigned long long>(f));
        atomicAdd(&s_sum[b], static_cast<unsigned long long>(f));
    }
    if (bad) atomicAdd(misplaced, bad);
    __syncthreads();
    for (int b = threadIdx.x; b < n_bins; b += blockDim.x) {
        if (s_cnt[b]) {
            atomicAdd(&stats[3 * b + 0], s_cnt[b]);
            atomicXor(&stats[3 * b + 1], s_xor[b]);
            atomicAdd(&stats[3 * b + 2], s_sum[b]);
        }
    }
}

// starts[b] = offs[b * n_blocks]: the first output index of bin b (b = n_bins: offs[cells], which must be n)
__global__ void bin_starts_kernel(const uint64_t *offs, uint64_t n_blocks, int n_bins, uint64_t *starts)
{
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b <= n_bins; b += gridDim.x * blockDim.x) starts[b] = offs[static_cast<uint64_t>(b) * n_blocks];
}

// cells whose offsets are not the exclusive prefix of the matrix: offs[c + 1] - offs[c] != matrix[c] (or offs[0] != 0)
__global__ void scan_check_kernel(const uint64_t *matrix, const uint64_t *offs, uint64_t cells, unsigned long long *bad)
{
    unsigned long long b = 0;
    for (uint64_t c = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; c < cells; c += static_cast<uint64_t>(gridDim.x) * blockDim.x)
        b += (offs[c + 1] - offs[c] != matrix[c]) || (c == 0 && offs[0] != 0);
    if (b) atomicAdd(bad, b);
}

__global__ void guard_check_kernel(const unsigned char *guard, uint64_t bytes, unsigned long long *bad)
{
    unsigned long long b = 0;
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < bytes; i += static_cast<uint64_t>(gridDim.x) * blockDim.x)
        b += guard[i] != kSentinel;
    if (b) atomicAdd(bad, b);
}

// report: [0] keys out of their bin's range, [1] bins whose count / xor / sum differ between input and output,
// [2] cells of offs that are not the scan of the matrix, [3] offs[cells] (must be n), [4] changed guard bytes,
// [5] input keys whose bin is out of range (must be 0)
template <typename Key> cudaError_t partition_check_large(int p, uint64_t n, uint64_t seed, uint64_t *report)
{
    for (int i = 0; i < 6; ++i) report[i] = ~0ull;
    if (p < binning::kMinBits || p > binning::kMaxBits || n == 0) return cudaErrorInvalidValue;
    const int n_bins = 1 << p;
    const auto bin_of = BinOfWidth<Key>::make(p, 32 - p);
    const uint64_t bytes = n * sizeof(Key), cells = binning::matrix_cells<Key>(n, p), n_blocks = binning::blocks_for<Key>(n);
    int dev = 0, sms = 0;
    TRY(cudaGetDevice(&dev));
    TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const unsigned grid = static_cast<unsigned>(sms * 8);
    DevMem d_in, d_out, d_matrix, d_offs, d_scan, d_small;
    TRY(d_in.alloc(bytes));
    TRY(d_out.alloc(bytes + kGuardBytes));
    TRY(d_matrix.alloc((cells + 1) * 8));
    TRY(d_offs.alloc((cells + 2) * 8));
    TRY(d_scan.alloc((scan_tmp_elems(cells) + 1) * 8));
    // two stats tables (input, output), the bin starts, and the counters
    const uint64_t small_words = 6 * kMaxBins + (kMaxBins + 1) + 8;
    TRY(d_small.alloc(small_words * 8));
    unsigned long long *st_in = d_small.as<unsigned long long>(), *st_out = st_in + 3 * kMaxBins;
    uint64_t *starts = reinterpret_cast<uint64_t *>(st_out + 3 * kMaxBins);
    unsigned long long *ctr = reinterpret_cast<unsigned long long *>(starts + kMaxBins + 1);
    Stream st;
    TRY(st.create());
    TRY(cudaMemsetAsync(d_small.p, 0, small_words * 8, st.s));
    TRY(cudaMemsetAsync(d_out.p, kSentinel, bytes + kGuardBytes, st.s));
    generate_kernel<Key><<<grid, 256, 0, st.s>>>(d_in.as<Key>(), n, seed);
    TRY(cudaGetLastError());
    TRY(binning::partition<Key>(d_in.as<const Key>(), n, p, bin_of, d_out.as<Key>(), d_matrix.as<uint64_t>(), d_offs.as<uint64_t>(),
                                d_scan.as<uint64_t>(), st.s));
    bin_starts_kernel<<<(n_bins + 256) / 256, 256, 0, st.s>>>(d_offs.as<uint64_t>(), n_blocks, n_bins, starts);
    bin_stats_kernel<<<grid, 256, 0, st.s>>>(d_in.as<const Key>(), n, bin_of, n_bins, starts, false, st_in, ctr + 5);
    bin_stats_kernel<<<grid, 256, 0, st.s>>>(d_out.as<const Key>(), n, bin_of, n_bins, starts, true, st_out, ctr + 0);
    scan_check_kernel<<<grid, 256, 0, st.s>>>(d_matrix.as<uint64_t>(), d_offs.as<uint64_t>(), cells, ctr + 2);
    guard_check_kernel<<<16, 256, 0, st.s>>>(d_out.as<unsigned char>() + bytes, kGuardBytes, ctr + 4);
    TRY(cudaGetLastError());
    std::vector<unsigned long long> host(small_words);
    TRY(cudaMemcpyAsync(host.data(), d_small.p, small_words * 8, cudaMemcpyDeviceToHost, st.s));
    TRY(cudaStreamSynchronize(st.s));
    const unsigned long long *h_in = host.data(), *h_out = h_in + 3 * kMaxBins, *h_ctr = h_out + 3 * kMaxBins + kMaxBins + 1;
    uint64_t bins_differ = 0;
    for (int b = 0; b < n_bins; ++b) bins_differ += std::memcmp(h_in + 3 * b, h_out + 3 * b, 24) != 0;
    report[0] = h_ctr[0];
    report[1] = bins_differ;
    report[2] = h_ctr[2];
    report[3] = h_out[3 * kMaxBins + n_bins]; // starts[n_bins] = offs[cells]
    report[4] = h_ctr[4];
    report[5] = h_ctr[5];
    return cudaSuccess;
}

// ------------------------------------------------------------------------------------------- apply_groups
__global__ void mark_applied_kernel(unsigned *done, unsigned b_end)
{
    // hold the stream a little, so that an event recorded before this group's apply would be seen ahead of the write
    const uint64_t t0 = clock64();
    while (clock64() - t0 < 20000) {
    }
    *done = b_end;
}

template <typename Key> void shape(int *per_vec, int *per_iter, int *chunk)
{
    *per_vec = binning::Shape<Key>::kPerVec;
    *per_iter = binning::Shape<Key>::kPerIter;
    *chunk = binning::Shape<Key>::kChunk;
}

} // namespace

extern "C" {

// kPerVec, kPerIter, kChunk of a key width (4, 8 or 16 bytes); -1 for another width.  No device needed.
int bh_shape(int key_bytes, int *per_vec, int *per_iter, int *chunk)
{
    switch (key_bytes) {
    case 4: shape<uint32_t>(per_vec, per_iter, chunk); return 0;
    case 8: shape<uint64_t>(per_vec, per_iter, chunk); return 0;
    case 16: shape<ulonglong2>(per_vec, per_iter, chunk); return 0;
    default: return -1;
    }
}

uint64_t bh_blocks_for(int key_bytes, uint64_t n)
{
    switch (key_bytes) {
    case 4: return binning::blocks_for<uint32_t>(n);
    case 8: return binning::blocks_for<uint64_t>(n);
    case 16: return binning::blocks_for<ulonglong2>(n);
    default: return 0;
    }
}

int bh_bin_range(int *min_bits, int *max_bits)
{
    *min_bits = binning::kMinBits;
    *max_bits = binning::kMaxBits;
    return 0;
}

// One binning::partition of in[0..n) into 2^p bins (ids: IdBin{shift}; 8 / 16-byte keys: the k-mer hash bins).  out: n
// keys; matrix: 2^p * blocks_for(n) counts; offs: that + 1.  guard_ok: the 4 KB behind the output kept their sentinel;
// input_ok: the input is unchanged.
int bh_partition(int key_bytes, int p, int shift, const void *in, uint64_t n, void *out, uint64_t *offs, uint64_t *matrix,
                 int *guard_ok, int *input_ok)
{
    switch (key_bytes) {
    case 4: return partition_once<uint32_t>(p, shift, in, n, out, offs, matrix, guard_ok, input_ok);
    case 8: return partition_once<uint64_t>(p, shift, in, n, out, offs, matrix, guard_ok, input_ok);
    case 16: return partition_once<ulonglong2>(p, shift, in, n, out, offs, matrix, guard_ok, input_ok);
    default: return cudaErrorInvalidValue;
    }
}

// n keys generated on the device from `seed` (ids: 32 bits, binned by their top p bits), partitioned and checked there;
// report: see partition_check_large
int bh_partition_check_large(int key_bytes, int p, uint64_t n, uint64_t seed, uint64_t *report)
{
    switch (key_bytes) {
    case 4: return partition_check_large<uint32_t>(p, n, seed, report);
    case 8: return partition_check_large<uint64_t>(p, n, seed, report);
    case 16: return partition_check_large<ulonglong2>(p, n, seed, report);
    default: return cudaErrorInvalidValue;
    }
}

// binning::apply_groups(n_bins, group, n_parts) with an apply that writes b_end into a device cell.  seen[i]: that cell
// as a second stream read it once it had waited for event i.  recorded[i]: whether event i was recorded at all.
int bh_apply_groups_schedule(int n_bins, int group, unsigned n_parts, unsigned *seen, int *recorded)
{
    for (unsigned i = 0; i < n_parts; ++i) {
        seen[i] = ~0u;
        recorded[i] = 0;
    }
    Stream main, side;
    TRY(main.create());
    TRY(side.create());
    DevMem d_done, d_seen;
    TRY(d_done.alloc(4));
    TRY(d_seen.alloc(4ull * (n_parts ? n_parts : 1)));
    struct Events {
        std::vector<cudaEvent_t> ev;
        ~Events()
        {
            for (cudaEvent_t e : ev) cudaEventDestroy(e);
        }
    } events;
    for (unsigned i = 0; i <= n_parts; ++i) { // the last one marks the start
        cudaEvent_t e;
        TRY(cudaEventCreate(&e));
        events.ev.push_back(e);
    }
    cudaEvent_t t0 = events.ev[n_parts];
    TRY(cudaMemsetAsync(d_done.p, 0, 4, main.s));
    TRY(cudaMemsetAsync(d_seen.p, 0xff, 4ull * n_parts, main.s));
    TRY(cudaEventRecord(t0, main.s));
    TRY(cudaStreamWaitEvent(side.s, t0, 0));
    unsigned *done = d_done.as<unsigned>();
    auto apply = [&](int, int b_end) {
        mark_applied_kernel<<<1, 1, 0, main.s>>>(done, static_cast<unsigned>(b_end));
        return cudaGetLastError();
    };
    std::vector<void *> handles(events.ev.begin(), events.ev.begin() + n_parts);
    TRY(binning::apply_groups(n_bins, group, n_parts, handles.data(), main.s, apply));
    // the side stream reads the cell behind each event, in event order (an event never recorded is no wait at all)
    for (unsigned i = 0; i < n_parts; ++i) {
        TRY(cudaStreamWaitEvent(side.s, events.ev[i], 0));
        TRY(cudaMemcpyAsync(d_seen.as<unsigned>() + i, done, 4, cudaMemcpyDeviceToDevice, side.s));
    }
    TRY(cudaStreamSynchronize(main.s));
    TRY(cudaStreamSynchronize(side.s));
    TRY(cudaMemcpy(seen, d_seen.p, 4ull * n_parts, cudaMemcpyDeviceToHost));
    for (unsigned i = 0; i < n_parts; ++i) {
        float ms = 0;
        const cudaError_t e = cudaEventElapsedTime(&ms, t0, events.ev[i]); // an event never recorded: an error
        recorded[i] = e == cudaSuccess;
        if (e != cudaSuccess) (void)cudaGetLastError();
    }
    return cudaSuccess;
}

// free and total device memory, for the test that needs tens of GB
int bh_mem_get_info(uint64_t *free_bytes, uint64_t *total_bytes)
{
    size_t f = 0, t = 0;
    const cudaError_t e = cudaMemGetInfo(&f, &t);
    *free_bytes = f;
    *total_bytes = t;
    return e;
}

} // extern "C"
