// comm.cu -- the multi-GPU surface of the C ABI (include/kmerscuda.h, "multi-GPU"): NCCL communicators
// attached to contexts, the single-process device group, and the two places where the path exchanges data
// between GPUs:
//   * the sum of the per-GPU bucket-count tables (north_star's only collective): kmc_bucket_count_merge /
//     kmc_group_bucket_count all-reduce every range of the table on a communication stream as soon as the
//     count has finished it, while the later ranges are still being counted;
//   * the exact k-mer table across GPUs (SURVEY.md 8f rank 4): every key has one owner rank (a second mix of
//     its fx_hash), entries travel to their owner by grouped ncclSend / ncclRecv over NVLink, the owner merges.
// The k-mer / hash / index streams themselves never cross GPUs (reads shard by sequence, one long sequence by
// window range with a K-1 halo): kmc_group_extract* only runs the per-device calls side by side.
//
// NCCL is bound at run time (dlopen of libnccl.so.2: inside a torch process that is the copy torch already
// loaded, otherwise the system one), so that libkmerscuda.so loads -- and the single-GPU path works -- on a
// machine without NCCL; the multi-GPU entry points then fail with KMC_E_NCCL and say why.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "plan.h"
#include "table_keys.cuh"

namespace kmc {

namespace {

constexpr uint32_t kMergeParts = 8; // ranges of a bucket table that are all-reduced separately

struct NcclApi {
    void *handle = nullptr;
    std::string error;
    decltype(&ncclGetVersion) GetVersion = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommInitAll) CommInitAll = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    decltype(&ncclAllReduce) AllReduce = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclSend) Send = nullptr;
    decltype(&ncclRecv) Recv = nullptr;
    decltype(&ncclGroupStart) GroupStart = nullptr;
    decltype(&ncclGroupEnd) GroupEnd = nullptr;
};

NcclApi &nccl()
{
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        std::vector<std::string> names;
        if (const char *e = getenv("KMERSCUDA_NCCL")) names.push_back(e);
        names.push_back("libnccl.so.2");
        names.push_back("libnccl.so");
        for (const std::string &n : names) {
            api.handle = dlopen(n.c_str(), RTLD_NOW | RTLD_GLOBAL);
            if (api.handle) break;
        }
        if (!api.handle) {
            api.error = std::string("NCCL is not available: ") + (dlerror() ? dlerror() : "dlopen(libnccl.so.2) failed");
            return;
        }
        bool ok = true;
        auto sym = [&](const char *name) -> void * {
            void *p = dlsym(api.handle, name);
            if (!p) {
                ok = false;
                api.error = std::string("NCCL symbol missing: ") + name;
            }
            return p;
        };
#define KMC_NCCL_SYM(F) api.F = reinterpret_cast<decltype(api.F)>(sym("nccl" #F))
        KMC_NCCL_SYM(GetVersion);
        KMC_NCCL_SYM(GetUniqueId);
        KMC_NCCL_SYM(CommInitRank);
        KMC_NCCL_SYM(CommInitAll);
        KMC_NCCL_SYM(CommDestroy);
        KMC_NCCL_SYM(GetErrorString);
        KMC_NCCL_SYM(AllReduce);
        KMC_NCCL_SYM(AllGather);
        KMC_NCCL_SYM(Send);
        KMC_NCCL_SYM(Recv);
        KMC_NCCL_SYM(GroupStart);
        KMC_NCCL_SYM(GroupEnd);
#undef KMC_NCCL_SYM
        if (!ok) {
            dlclose(api.handle);
            api.handle = nullptr;
        }
    });
    return api;
}

int32_t fail_nccl(kmc_ctx *ctx, ncclResult_t r, const char *what)
{
    if (ctx) {
        char buf[512];
        snprintf(buf, sizeof buf, "%s: NCCL error %d (%s)", what, static_cast<int>(r),
                 nccl().GetErrorString ? nccl().GetErrorString(r) : "?");
        ctx->last_error = buf;
    }
    return KMC_E_NCCL;
}

#define NC(ctx, call)                                              \
    do {                                                           \
        ncclResult_t r__ = (call);                                 \
        if (r__ != ncclSuccess) return fail_nccl(ctx, r__, #call); \
    } while (0)

int32_t need_nccl(kmc_ctx *ctx)
{
    if (nccl().handle) return KMC_OK;
    return fail(ctx, KMC_E_NCCL, nccl().error.c_str());
}

} // namespace

} // namespace kmc

// One communicator rank, attached to a context.  Collectives run on `stream` (the communication stream) so that
// they overlap the kernels of the context's own stream; `done` orders the context's stream behind them.
struct kmc_comm {
    ncclComm_t comm = nullptr;
    int rank = 0, n_ranks = 1;
    cudaStream_t stream = nullptr;
    cudaEvent_t part[kmc::kMergeParts] = {};
    cudaEvent_t done = nullptr;
};

struct kmc_group {
    std::vector<kmc_ctx *> ctx; // one per device, each with a comm of the group's communicator (rank = index)
};

namespace kmc {

namespace {

int32_t comm_finish_init(kmc_ctx *ctx, ncclComm_t comm, int rank, int n_ranks)
{
    kmc_comm *c = new (std::nothrow) kmc_comm();
    if (!c) return fail(ctx, KMC_E_BAD_ARG, "out of host memory");
    c->comm = comm;
    c->rank = rank;
    c->n_ranks = n_ranks;
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    for (uint32_t i = 0; i < kMergeParts && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&c->part[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->done, cudaEventDisableTiming);
    ctx->comm = c;
    if (e != cudaSuccess) {
        comm_detach(ctx);
        return fail_cuda(ctx, e, "communicator streams / events");
    }
    return KMC_OK;
}

// ---- the exact k-mer table across GPUs: entries -> owner ranks ---------------------------------------------------
// (keys: uint64_t for one-limb tables, ulonglong2 for two-limb ones; table_keys.cuh)
constexpr int kMaxRanks = 64;

// The owner of a key: a second mix of its fx_hash (the table's slot is the TOP bits of fx_hash; an owner taken from
// the same bits would leave every owner's table with a 1/n_ranks sliver of its slots in use), range-reduced by a
// multiply-shift.  Host and device agree (kmc_kmer_owner, kmc_kmer_owner2).
__host__ __device__ inline uint32_t owner_of_hash(uint64_t h, uint32_t n_ranks)
{
    h ^= h >> 32;
    h *= 0x9E3779B97F4A7C15ull;
    return static_cast<uint32_t>(((h >> 32) * n_ranks) >> 32);
}
__host__ __device__ inline uint32_t owner_of(uint64_t key, uint32_t n_ranks)
{
    return owner_of_hash(key * FX_CONSTANT, n_ranks); // fx_hash of a one-limb k-mer with h0 = 0: (rotl(0,5) ^ key) * FX
}
__host__ __device__ inline uint32_t owner_of(ulonglong2 key, uint32_t n_ranks) { return owner_of_hash(key_hash(key), n_ranks); }

// pass 1: entries per owner
template <typename Key>
__global__ void __launch_bounds__(256) owner_count_kernel(const Key *__restrict__ keys, uint64_t n_slots, uint32_t n_ranks,
                                                          unsigned long long *__restrict__ counts)
{
    __shared__ uint32_t s_cnt[kMaxRanks];
    if (threadIdx.x < kMaxRanks) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_slots;
         i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const Key key = keys[i];
        if (!key_free(key)) atomicAdd(s_cnt + owner_of(key, n_ranks), 1u);
    }
    __syncthreads();
    if (threadIdx.x < n_ranks && s_cnt[threadIdx.x]) atomicAdd(counts + threadIdx.x, static_cast<unsigned long long>(s_cnt[threadIdx.x]));
}

// pass 2: the entries, grouped by owner (segment o starts at base[o]); one block reserves a run per owner for the
// chunk of slots it handles, so the global cursors see one atomic per (block, chunk, owner)
template <typename Key>
__global__ void __launch_bounds__(256) owner_scatter_kernel(const Key *__restrict__ keys, const uint32_t *__restrict__ vals,
                                                            uint64_t n_slots, uint32_t n_ranks, const uint64_t *__restrict__ base,
                                                            unsigned long long *__restrict__ cursor, Key *__restrict__ out_keys,
                                                            uint32_t *__restrict__ out_vals)
{
    __shared__ uint32_t s_cnt[kMaxRanks];
    __shared__ unsigned long long s_base[kMaxRanks];
    constexpr int kPer = 8;
    const uint64_t chunk = 256ull * kPer;
    for (uint64_t c0 = static_cast<uint64_t>(blockIdx.x) * chunk; c0 < n_slots; c0 += static_cast<uint64_t>(gridDim.x) * chunk) {
        if (threadIdx.x < kMaxRanks) s_cnt[threadIdx.x] = 0;
        __syncthreads();
        Key key[kPer];
        uint32_t val[kPer], own[kPer], rank[kPer];
#pragma unroll
        for (int j = 0; j < kPer; ++j) {
            const uint64_t i = c0 + static_cast<uint64_t>(j) * 256 + threadIdx.x;
            if constexpr (sizeof(Key) == 8)
                key[j] = i < n_slots ? keys[i] : kEmptyKey;
            else
                key[j] = i < n_slots ? keys[i] : make_ulonglong2(kEmptyKey, kEmptyKey);
            if (!key_free(key[j])) {
                val[j] = vals[i];
                own[j] = owner_of(key[j], n_ranks);
                rank[j] = atomicAdd(s_cnt + own[j], 1u);
            }
        }
        __syncthreads();
        if (threadIdx.x < n_ranks)
            s_base[threadIdx.x] = base[threadIdx.x] + atomicAdd(cursor + threadIdx.x, static_cast<unsigned long long>(s_cnt[threadIdx.x]));
        __syncthreads();
#pragma unroll
        for (int j = 0; j < kPer; ++j)
            if (!key_free(key[j])) {
                const uint64_t at = s_base[own[j]] + rank[j];
                out_keys[at] = key[j];
                out_vals[at] = val[j];
            }
        __syncthreads();
    }
}

// what one local rank holds during an exchange (keys: n_limbs u64 per entry)
struct ExchangeRank {
    kmc_ctx *ctx;
    const uint64_t *keys;
    const uint32_t *vals;
    uint64_t *owned_keys;
    uint32_t *owned_vals;
    AsyncBuf counts_dev, cursor_dev, base_dev, matrix_dev, send_keys, send_vals, recv_keys, recv_vals;
    std::vector<uint64_t> counts, matrix; // host copies: entries per owner; the n x n matrix [sender][owner]
    uint64_t n_entries = 0, n_recv = 0, n_new = 0;
};

// The exchange for the local ranks `rs` (one per context of this process: all of the communicator's ranks in the
// single-process group, exactly one under one-process-per-GPU launchers).  Every rank of the communicator must make
// the call (it is a collective).  Key: uint64_t (one-limb tables) or ulonglong2 (two-limb tables, sent as 2n u64).
template <typename Key>
int32_t table_exchange(std::vector<ExchangeRank> &rs, uint32_t log2_capacity, uint32_t owned_log2_capacity, uint64_t *n_owned)
{
    constexpr uint64_t NL = sizeof(Key) / 8;
    kmc_ctx *c0 = rs[0].ctx;
    int32_t st = need_nccl(c0);
    if (st) return st;
    NcclApi &N = nccl();
    const uint32_t n_ranks = static_cast<uint32_t>(c0->comm->n_ranks);
    if (n_ranks > kMaxRanks) return fail(c0, KMC_E_UNSUPPORTED, "the k-mer table exchange supports up to 64 ranks");
    const uint64_t n_slots = 1ull << log2_capacity;
    const bool grouped = rs.size() > 1;

    // (1) entries per owner, on every local rank; all-gather into the [sender][owner] matrix
    for (ExchangeRank &r : rs) {
        kmc_ctx *ctx = r.ctx;
        CU(cudaSetDevice(ctx->device));
        cudaStream_t s = ctx->stream;
        CU(r.counts_dev.alloc(ctx, 8 * n_ranks, s));
        CU(r.matrix_dev.alloc(ctx, 8ull * n_ranks * n_ranks, s));
        CU(cudaMemsetAsync(r.counts_dev.p, 0, 8 * n_ranks, s));
        const uint64_t blocks = std::min<uint64_t>((n_slots + 255) / 256, static_cast<uint64_t>(ctx->sm_count) * 16);
        owner_count_kernel<Key><<<static_cast<unsigned>(blocks), 256, 0, s>>>(reinterpret_cast<const Key *>(r.keys), n_slots, n_ranks,
                                                                             r.counts_dev.as<unsigned long long>());
        CU(cudaGetLastError());
    }
    if (grouped) NC(c0, N.GroupStart());
    for (ExchangeRank &r : rs) {
        kmc_ctx *ctx = r.ctx;
        CU(cudaSetDevice(ctx->device));
        NC(ctx, N.AllGather(r.counts_dev.p, r.matrix_dev.p, n_ranks, ncclUint64, ctx->comm->comm, ctx->stream));
    }
    if (grouped) NC(c0, N.GroupEnd());
    for (ExchangeRank &r : rs) {
        kmc_ctx *ctx = r.ctx;
        CU(cudaSetDevice(ctx->device));
        r.matrix.resize(static_cast<size_t>(n_ranks) * n_ranks);
        CU(cudaMemcpyAsync(r.matrix.data(), r.matrix_dev.p, 8ull * n_ranks * n_ranks, cudaMemcpyDeviceToHost, ctx->stream));
    }
    for (ExchangeRank &r : rs) {
        kmc_ctx *ctx = r.ctx;
        CU(cudaSetDevice(ctx->device));
        CU(cudaStreamSynchronize(ctx->stream));
    }

    // (2) group the entries by owner; size the receive buffers from the matrix
    for (ExchangeRank &r : rs) {
        kmc_ctx *ctx = r.ctx;
        const uint32_t me = static_cast<uint32_t>(ctx->comm->rank);
        CU(cudaSetDevice(ctx->device));
        cudaStream_t s = ctx->stream;
        r.counts.assign(r.matrix.begin() + static_cast<size_t>(me) * n_ranks, r.matrix.begin() + static_cast<size_t>(me + 1) * n_ranks);
        std::vector<uint64_t> base(n_ranks + 1, 0);
        for (uint32_t o = 0; o < n_ranks; ++o) base[o + 1] = base[o] + r.counts[o];
        r.n_entries = base[n_ranks];
        r.n_recv = 0;
        for (uint32_t q = 0; q < n_ranks; ++q)
            if (q != me) r.n_recv += r.matrix[static_cast<size_t>(q) * n_ranks + me];
        CU(r.base_dev.alloc(ctx, 8 * (n_ranks + 1), s));
        CU(r.cursor_dev.alloc(ctx, 8 * n_ranks, s));
        CU(r.send_keys.alloc(ctx, 8 * NL * r.n_entries, s));
        CU(r.send_vals.alloc(ctx, 4 * r.n_entries, s));
        CU(r.recv_keys.alloc(ctx, 8 * NL * r.n_recv, s));
        CU(r.recv_vals.alloc(ctx, 4 * r.n_recv, s));
        // (base is a host vector that dies with this iteration: a synchronous copy)
        CU(cudaMemcpyAsync(r.base_dev.p, base.data(), 8 * (n_ranks + 1), cudaMemcpyHostToDevice, s));
        CU(cudaStreamSynchronize(s));
        CU(cudaMemsetAsync(r.cursor_dev.p, 0, 8 * n_ranks, s));
        const uint64_t blocks = std::min<uint64_t>((n_slots + 2047) / 2048, static_cast<uint64_t>(ctx->sm_count) * 8);
        owner_scatter_kernel<Key><<<static_cast<unsigned>(blocks), 256, 0, s>>>(
            reinterpret_cast<const Key *>(r.keys), r.vals, n_slots, n_ranks, r.base_dev.as<uint64_t>(), r.cursor_dev.as<unsigned long long>(),
            r.send_keys.as<Key>(), r.send_vals.as<uint32_t>());
        CU(cudaGetLastError());
    }

    // (3) every entry to its owner: one grouped batch of sends and receives per rank (NVLink peer copies under NCCL)
    NC(c0, N.GroupStart());
    for (ExchangeRank &r : rs) {
        kmc_ctx *ctx = r.ctx;
        const uint32_t me = static_cast<uint32_t>(ctx->comm->rank);
        CU(cudaSetDevice(ctx->device));
        uint64_t send_at = 0, recv_at = 0;
        for (uint32_t q = 0; q < n_ranks; ++q) {
            const uint64_t ns = r.counts[q];
            if (q != me && ns) {
                NC(ctx, N.Send(r.send_keys.as<uint64_t>() + NL * send_at, NL * ns, ncclUint64, static_cast<int>(q), ctx->comm->comm, ctx->stream));
                NC(ctx, N.Send(r.send_vals.as<uint32_t>() + send_at, ns, ncclUint32, static_cast<int>(q), ctx->comm->comm, ctx->stream));
            }
            send_at += ns;
            const uint64_t nr = q != me ? r.matrix[static_cast<size_t>(q) * n_ranks + me] : 0;
            if (nr) {
                NC(ctx, N.Recv(r.recv_keys.as<uint64_t>() + NL * recv_at, NL * nr, ncclUint64, static_cast<int>(q), ctx->comm->comm, ctx->stream));
                NC(ctx, N.Recv(r.recv_vals.as<uint32_t>() + recv_at, nr, ncclUint32, static_cast<int>(q), ctx->comm->comm, ctx->stream));
                recv_at += nr;
            }
        }
    }
    NC(c0, N.GroupEnd());

    // (4) the owner merges its own share and what it received
    for (size_t i = 0; i < rs.size(); ++i) {
        ExchangeRank &r = rs[i];
        kmc_ctx *ctx = r.ctx;
        const uint32_t me = static_cast<uint32_t>(ctx->comm->rank);
        uint64_t own0 = 0;
        for (uint32_t o = 0; o < me; ++o) own0 += r.counts[o];
        uint64_t added = 0, a2 = 0;
        auto merge = NL == 1 ? kmc_kmer_table_merge : kmc_kmer_table2_merge;
        st = merge(ctx, r.owned_keys, r.owned_vals, owned_log2_capacity, r.send_keys.as<uint64_t>() + NL * own0,
                   r.send_vals.as<uint32_t>() + own0, r.counts[me], &added);
        if (st) return st;
        st = merge(ctx, r.owned_keys, r.owned_vals, owned_log2_capacity, r.recv_keys.as<uint64_t>(), r.recv_vals.as<uint32_t>(),
                   r.n_recv, &a2);
        if (st) return st;
        if (n_owned) n_owned[i] = added + a2;
    }
    return KMC_OK;
}

// count on every local rank, all-reduce range by range behind the count
int32_t bucket_count_merge(const std::vector<kmc_ctx *> &cs, const kmc_seqs *seqs, size_t seqs_stride, int32_t k, int32_t bucket_bits,
                           uint32_t *const *tables, kmc_result *results)
{
    kmc_ctx *c0 = cs[0];
    int32_t st = need_nccl(c0);
    if (st) return st;
    NcclApi &N = nccl();
    if (bucket_bits < 1 || bucket_bits > 32) return fail(c0, KMC_E_BAD_ARG, "bucket_bits must be in 1..32");
    const uint32_t n_parts = bucket_bits >= 8 ? kMergeParts : 1;
    const uint64_t part = (1ull << bucket_bits) / n_parts;
    for (kmc_ctx *ctx : cs)
        if (!ctx->comm) return fail(ctx, KMC_E_BAD_ARG, "the context has no communicator (kmc_comm_init_rank / kmc_group_create)");
    // The counts of the devices are enqueued side by side, each from its own host thread.  kmc_bucket_count_async only
    // enqueues, but that is about seventy launches per device: one thread walking eight devices starts the last one 2 ms
    // after the first (27.7 ms per step on eight GPUs from plain C; 26.1 ms with one thread per device).  (With the first
    // version of the fused count, which waited for its binning kernel on the host, the plain loop serialised the GPUs
    // outright: 95.7 ms.)
    auto start = [&](size_t i) -> int32_t {
        kmc_ctx *ctx = cs[i];
        CU(cudaSetDevice(ctx->device));
        CU(cudaEventRecord(ctx->ev_begin, ctx->stream));
        const kmc_seqs *s = reinterpret_cast<const kmc_seqs *>(reinterpret_cast<const char *>(seqs) + i * seqs_stride);
        return kmc_bucket_count_async(ctx, s, k, bucket_bits, tables[i], n_parts, reinterpret_cast<void *const *>(ctx->comm->part), &results[i]);
    };
    if (cs.size() == 1) {
        st = start(0);
        if (st) return st;
    } else {
        std::vector<int32_t> sts(cs.size(), KMC_OK);
        std::vector<std::thread> th;
        th.reserve(cs.size());
        for (size_t i = 0; i < cs.size(); ++i) th.emplace_back([&, i] { sts[i] = start(i); });
        for (std::thread &t : th) t.join();
        for (int32_t v : sts)
            if (v) return v;
    }
    const bool grouped = cs.size() > 1;
    for (uint32_t p = 0; p < n_parts; ++p) {
        if (grouped) NC(c0, N.GroupStart());
        for (size_t i = 0; i < cs.size(); ++i) {
            kmc_ctx *ctx = cs[i];
            CU(cudaSetDevice(ctx->device));
            CU(cudaStreamWaitEvent(ctx->comm->stream, ctx->comm->part[p], 0));
            uint32_t *range = tables[i] + p * part;
            NC(ctx, N.AllReduce(range, range, part, ncclUint32, ncclSum, ctx->comm->comm, ctx->comm->stream));
        }
        if (grouped) NC(c0, N.GroupEnd());
    }
    for (size_t i = 0; i < cs.size(); ++i) {
        kmc_ctx *ctx = cs[i];
        CU(cudaSetDevice(ctx->device));
        CU(cudaEventRecord(ctx->comm->done, ctx->comm->stream));
        CU(cudaStreamWaitEvent(ctx->stream, ctx->comm->done, 0));
        CU(cudaEventRecord(ctx->ev_end, ctx->stream));
    }
    for (size_t i = 0; i < cs.size(); ++i) {
        kmc_ctx *ctx = cs[i];
        CU(cudaSetDevice(ctx->device));
        CU(cudaEventSynchronize(ctx->ev_end));
        CU(cudaEventElapsedTime(&results[i].kernel_ms, ctx->ev_begin, ctx->ev_end));
    }
    return KMC_OK;
}

int32_t allreduce(const std::vector<kmc_ctx *> &cs, void *const *bufs, uint64_t n, ncclDataType_t type)
{
    kmc_ctx *c0 = cs[0];
    int32_t st = need_nccl(c0);
    if (st) return st;
    NcclApi &N = nccl();
    const bool grouped = cs.size() > 1;
    if (grouped) NC(c0, N.GroupStart());
    for (size_t i = 0; i < cs.size(); ++i) {
        kmc_ctx *ctx = cs[i];
        if (!ctx->comm) return fail(ctx, KMC_E_BAD_ARG, "the context has no communicator (kmc_comm_init_rank / kmc_group_create)");
        CU(cudaSetDevice(ctx->device));
        NC(ctx, N.AllReduce(bufs[i], bufs[i], n, type, ncclSum, ctx->comm->comm, ctx->stream));
    }
    if (grouped) NC(c0, N.GroupEnd());
    return KMC_OK;
}

// runs fn(i) for every device of the group on its own host thread (calls that synchronise internally -- 4-bit
// sources, the host pipeline -- would otherwise serialise the devices); returns the first non-zero status
template <typename F> int32_t for_each_device(kmc_group *g, F fn)
{
    const size_t n = g->ctx.size();
    std::vector<int32_t> st(n, KMC_OK);
    if (n == 1) return fn(0);
    std::vector<std::thread> th;
    th.reserve(n);
    for (size_t i = 0; i < n; ++i) th.emplace_back([&, i] { st[i] = fn(i); });
    for (std::thread &t : th) t.join();
    for (size_t i = 0; i < n; ++i)
        if (st[i]) return st[i];
    return KMC_OK;
}

} // namespace

void comm_detach(kmc_ctx *ctx)
{
    kmc_comm *c = ctx->comm;
    if (!c) return;
    cudaSetDevice(ctx->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->comm && nccl().CommDestroy) nccl().CommDestroy(c->comm);
    for (uint32_t i = 0; i < kMergeParts; ++i)
        if (c->part[i]) cudaEventDestroy(c->part[i]);
    if (c->done) cudaEventDestroy(c->done);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    ctx->comm = nullptr;
}

} // namespace kmc

using namespace kmc;

extern "C" {

int32_t kmc_nccl_version(int32_t *version)
{
    if (!version) return KMC_E_BAD_ARG;
    *version = 0;
    if (!nccl().handle) return KMC_E_NCCL;
    int v = 0;
    if (nccl().GetVersion(&v) != ncclSuccess) return KMC_E_NCCL;
    *version = v;
    return KMC_OK;
}

// ---- one process per GPU (torchrun / MPI launchers) ------------------------------------------------------------------
int32_t kmc_comm_unique_id(void *id128)
{
    if (!id128) return KMC_E_BAD_ARG;
    if (!nccl().handle) return KMC_E_NCCL;
    static_assert(sizeof(ncclUniqueId) == KMC_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    if (nccl().GetUniqueId(&id) != ncclSuccess) return KMC_E_NCCL;
    memcpy(id128, &id, sizeof id);
    return KMC_OK;
}

int32_t kmc_comm_init_rank(kmc_ctx *ctx, int32_t n_ranks, int32_t rank, const void *id128)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (!id128 || n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(ctx, KMC_E_BAD_ARG, "bad communicator arguments");
    if (ctx->comm) return fail(ctx, KMC_E_BAD_ARG, "the context already has a communicator");
    int32_t st = need_nccl(ctx);
    if (st) return st;
    CU(cudaSetDevice(ctx->device));
    ncclUniqueId id;
    memcpy(&id, id128, sizeof id);
    ncclComm_t comm = nullptr;
    NC(ctx, nccl().CommInitRank(&comm, n_ranks, id, rank));
    return comm_finish_init(ctx, comm, rank, n_ranks);
}

int32_t kmc_comm_destroy(kmc_ctx *ctx)
{
    if (!ctx) return KMC_E_BAD_ARG;
    comm_detach(ctx);
    return KMC_OK;
}

int32_t kmc_comm_info(kmc_ctx *ctx, int32_t *rank, int32_t *n_ranks)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (rank) *rank = ctx->comm ? ctx->comm->rank : 0;
    if (n_ranks) *n_ranks = ctx->comm ? ctx->comm->n_ranks : 1;
    return KMC_OK;
}

int32_t kmc_allreduce_u32(kmc_ctx *ctx, uint32_t *buf, uint64_t n)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (n && !buf) return fail(ctx, KMC_E_BAD_ARG, "NULL buffer");
    void *b = buf;
    return allreduce({ctx}, &b, n, ncclUint32);
}

int32_t kmc_allreduce_u64(kmc_ctx *ctx, uint64_t *buf, uint64_t n)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (n && !buf) return fail(ctx, KMC_E_BAD_ARG, "NULL buffer");
    void *b = buf;
    return allreduce({ctx}, &b, n, ncclUint64);
}

int32_t kmc_bucket_count_merge(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t bucket_bits, uint32_t *table,
                               kmc_result *result)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (!seqs || !table || !result) return fail(ctx, KMC_E_BAD_ARG, "NULL argument");
    uint32_t *t = table;
    return bucket_count_merge({ctx}, seqs, 0, k, bucket_bits, &t, result);
}

uint32_t kmc_kmer_owner(uint64_t key, uint32_t n_ranks) { return n_ranks ? owner_of(key, n_ranks) : 0; }

uint32_t kmc_kmer_owner2(uint64_t limb0, uint64_t limb1, uint32_t n_ranks)
{
    return n_ranks ? owner_of(make_ulonglong2(limb0, limb1), n_ranks) : 0;
}

} // extern "C"

template <typename Key>
static int32_t kmer_table_exchange(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity, uint64_t *owned_keys,
                                   uint32_t *owned_vals, uint32_t owned_log2_capacity, uint64_t *n_owned)
{
    if (!ctx) return KMC_E_BAD_ARG;
    if (!keys || !vals || !owned_keys || !owned_vals) return fail(ctx, KMC_E_BAD_ARG, "NULL table");
    if (log2_capacity < 1 || log2_capacity > 40 || owned_log2_capacity < 1 || owned_log2_capacity > 40)
        return fail(ctx, KMC_E_BAD_ARG, "log2_capacity must be in 1..40");
    if (sizeof(Key) == 16 && (reinterpret_cast<uintptr_t>(keys) % 16 || reinterpret_cast<uintptr_t>(owned_keys) % 16))
        return fail(ctx, KMC_E_BAD_ARG, "the two-limb keys must be 16-byte aligned");
    if (!ctx->comm) return fail(ctx, KMC_E_BAD_ARG, "the context has no communicator (kmc_comm_init_rank / kmc_group_create)");
    std::vector<ExchangeRank> rs(1);
    rs[0].ctx = ctx;
    rs[0].keys = keys;
    rs[0].vals = vals;
    rs[0].owned_keys = owned_keys;
    rs[0].owned_vals = owned_vals;
    return table_exchange<Key>(rs, log2_capacity, owned_log2_capacity, n_owned);
}

template <typename Key>
static int32_t group_kmer_table_exchange(kmc_group *g, const uint64_t *const *keys, const uint32_t *const *vals, uint32_t log2_capacity,
                                         uint64_t *const *owned_keys, uint32_t *const *owned_vals, uint32_t owned_log2_capacity,
                                         uint64_t *n_owned)
{
    if (!g || !keys || !vals || !owned_keys || !owned_vals) return KMC_E_BAD_ARG;
    const size_t n = g->ctx.size();
    if (sizeof(Key) == 16)
        for (size_t i = 0; i < n; ++i)
            if (reinterpret_cast<uintptr_t>(keys[i]) % 16 || reinterpret_cast<uintptr_t>(owned_keys[i]) % 16)
                return fail(g->ctx[i], KMC_E_BAD_ARG, "the two-limb keys must be 16-byte aligned");
    if (n == 1) { // one owner: the exchange is a merge into the owned table
        auto merge = sizeof(Key) == 8 ? kmc_kmer_table_merge : kmc_kmer_table2_merge;
        return merge(g->ctx[0], owned_keys[0], owned_vals[0], owned_log2_capacity, keys[0], vals[0], 1ull << log2_capacity, n_owned);
    }
    std::vector<ExchangeRank> rs(n);
    for (size_t i = 0; i < n; ++i) {
        rs[i].ctx = g->ctx[i];
        rs[i].keys = keys[i];
        rs[i].vals = vals[i];
        rs[i].owned_keys = owned_keys[i];
        rs[i].owned_vals = owned_vals[i];
    }
    return table_exchange<Key>(rs, log2_capacity, owned_log2_capacity, n_owned);
}

extern "C" {

int32_t kmc_kmer_table_exchange(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                                uint64_t *owned_keys, uint32_t *owned_vals, uint32_t owned_log2_capacity, uint64_t *n_owned)
{
    return kmer_table_exchange<uint64_t>(ctx, keys, vals, log2_capacity, owned_keys, owned_vals, owned_log2_capacity, n_owned);
}

int32_t kmc_kmer_table2_exchange(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                                 uint64_t *owned_keys, uint32_t *owned_vals, uint32_t owned_log2_capacity, uint64_t *n_owned)
{
    return kmer_table_exchange<ulonglong2>(ctx, keys, vals, log2_capacity, owned_keys, owned_vals, owned_log2_capacity, n_owned);
}

// ---- one process, several GPUs (what a Julia session is) -------------------------------------------------------------
int32_t kmc_group_create(int32_t n, const int32_t *devices, kmc_group **out)
{
    if (!out) return KMC_E_BAD_ARG;
    *out = nullptr;
    if (n < 1 || n > kMaxRanks) return KMC_E_BAD_ARG;
    int32_t have = 0;
    int32_t st = kmc_device_count(&have);
    if (st) return st;
    std::vector<int> devs(static_cast<size_t>(n));
    for (int32_t i = 0; i < n; ++i) {
        devs[i] = devices ? devices[i] : i;
        if (devs[i] < 0 || devs[i] >= have) return KMC_E_NO_DEVICE;
    }
    kmc_group *g = new (std::nothrow) kmc_group();
    if (!g) return KMC_E_BAD_ARG;
    for (int32_t i = 0; i < n; ++i) {
        kmc_ctx *ctx = nullptr;
        st = kmc_ctx_create(devs[i], &ctx);
        if (st) {
            kmc_group_destroy(g);
            return st;
        }
        g->ctx.push_back(ctx);
    }
    // a group of one device needs no communicator (and no NCCL): its collectives are the identity
    if (n > 1) {
        if (!nccl().handle) {
            kmc_group_destroy(g);
            return KMC_E_NCCL;
        }
        std::vector<ncclComm_t> comms(static_cast<size_t>(n), nullptr);
        if (nccl().CommInitAll(comms.data(), n, devs.data()) != ncclSuccess) {
            kmc_group_destroy(g);
            return KMC_E_NCCL;
        }
        for (int32_t i = 0; i < n; ++i) {
            cudaSetDevice(devs[i]);
            st = comm_finish_init(g->ctx[i], comms[i], i, n);
            if (st) {
                for (int32_t j = i + 1; j < n; ++j) nccl().CommDestroy(comms[j]);
                kmc_group_destroy(g);
                return st;
            }
        }
    }
    *out = g;
    return KMC_OK;
}

int32_t kmc_group_destroy(kmc_group *g)
{
    if (!g) return KMC_OK;
    for (kmc_ctx *ctx : g->ctx) kmc_ctx_destroy(ctx); // detaches and destroys the rank's communicator
    delete g;
    return KMC_OK;
}

int32_t kmc_group_size(kmc_group *g, int32_t *n)
{
    if (!g || !n) return KMC_E_BAD_ARG;
    *n = static_cast<int32_t>(g->ctx.size());
    return KMC_OK;
}

int32_t kmc_group_ctx(kmc_group *g, int32_t i, kmc_ctx **ctx)
{
    if (!g || !ctx || i < 0 || i >= static_cast<int32_t>(g->ctx.size())) return KMC_E_BAD_ARG;
    *ctx = g->ctx[i];
    return KMC_OK;
}

int32_t kmc_group_sync(kmc_group *g)
{
    if (!g) return KMC_E_BAD_ARG;
    for (kmc_ctx *ctx : g->ctx) {
        int32_t st = kmc_sync(ctx);
        if (st) return st;
    }
    return KMC_OK;
}

int32_t kmc_group_allreduce_u32(kmc_group *g, uint32_t *const *bufs, uint64_t n)
{
    if (!g || !bufs) return KMC_E_BAD_ARG;
    if (g->ctx.size() == 1) return KMC_OK;
    return allreduce(g->ctx, reinterpret_cast<void *const *>(bufs), n, ncclUint32);
}

int32_t kmc_group_allreduce_u64(kmc_group *g, uint64_t *const *bufs, uint64_t n)
{
    if (!g || !bufs) return KMC_E_BAD_ARG;
    if (g->ctx.size() == 1) return KMC_OK;
    return allreduce(g->ctx, reinterpret_cast<void *const *>(bufs), n, ncclUint64);
}

int32_t kmc_group_bucket_count(kmc_group *g, const kmc_seqs *seqs, int32_t k, int32_t bucket_bits, uint32_t *const *tables,
                               kmc_result *results)
{
    if (!g || !seqs || !tables || !results) return KMC_E_BAD_ARG;
    if (g->ctx.size() == 1) return kmc_bucket_count(g->ctx[0], seqs, k, bucket_bits, tables[0], results);
    return bucket_count_merge(g->ctx, seqs, sizeof(kmc_seqs), k, bucket_bits, tables, results);
}

int32_t kmc_group_extract(kmc_group *g, const kmc_seqs *seqs, int32_t k, int32_t mode, uint32_t flags, const kmc_out *outs,
                          kmc_result *results)
{
    if (!g || !seqs || !outs || !results) return KMC_E_BAD_ARG;
    return for_each_device(g, [&](size_t i) { return kmc_extract(g->ctx[i], &seqs[i], k, mode, flags & ~KMC_NO_SYNC, &outs[i], &results[i]); });
}

int32_t kmc_group_extract_host(kmc_group *g, const kmc_seqs *host_seqs, int32_t k, int32_t mode, uint32_t flags,
                               const kmc_out *outs, kmc_result *results)
{
    if (!g || !host_seqs || !outs || !results) return KMC_E_BAD_ARG;
    return for_each_device(g, [&](size_t i) { return kmc_extract_host(g->ctx[i], &host_seqs[i], k, mode, flags, &outs[i], &results[i]); });
}

int32_t kmc_group_kmer_table_exchange(kmc_group *g, const uint64_t *const *keys, const uint32_t *const *vals, uint32_t log2_capacity,
                                      uint64_t *const *owned_keys, uint32_t *const *owned_vals, uint32_t owned_log2_capacity,
                                      uint64_t *n_owned)
{
    return group_kmer_table_exchange<uint64_t>(g, keys, vals, log2_capacity, owned_keys, owned_vals, owned_log2_capacity, n_owned);
}

int32_t kmc_group_kmer_table2_exchange(kmc_group *g, const uint64_t *const *keys, const uint32_t *const *vals, uint32_t log2_capacity,
                                       uint64_t *const *owned_keys, uint32_t *const *owned_vals, uint32_t owned_log2_capacity,
                                       uint64_t *n_owned)
{
    return group_kmer_table_exchange<ulonglong2>(g, keys, vals, log2_capacity, owned_keys, owned_vals, owned_log2_capacity, n_owned);
}

} // extern "C"
