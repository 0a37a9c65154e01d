/*
 * kmerscuda.h -- C ABI of libkmerscuda.so: B200 (sm_100a) k-mer extraction behind
 * the Kmers.jl iterator API.
 *
 * The reference (BioJulia/Kmers.jl v1.2.0, pure Julia) has no FFI; its boundary for
 * this path is Julia's iteration protocol on four iterator types plus fx_hash.  Each
 * entry point below names the reference interface it replaces (paths relative to the
 * reference tree).  A Julia module (KmersCUDA, see INTEGRATION.md) binds these with
 * `ccall`; in this repository the same symbols are bound with Python ctypes
 * (kmers.jl_b200/kmerscuda/_abi.py).
 *
 * Conventions
 *  - every function returns an int32 status: 0 = KMC_OK, > 0 = domain error below,
 *    < 0 = -(cudaError_t).  No C++ exception crosses the ABI.
 *  - plain pointers and sizes only.  "device" pointers are CUDA device addresses on
 *    the context's device (from kmc_malloc or from any other allocator, e.g. a torch
 *    tensor's data_ptr); "host" pointers are ordinary host addresses.
 *  - k-mers are Kmer{A,K,N}.data: N = cld(2K, 64) UInt64 limbs, head (most
 *    significant) limb first, first symbol in the highest used bits, unused bits
 *    (top of limb 0) zero (src/kmer.jl:32-51).  Output alphabets are the 2-bit ones
 *    (DNAAlphabet{2} / RNAAlphabet{2} are bit-identical: A,C,G,T/U = 0,1,2,3).
 *  - sequences are LongSequence{<:NucleicAcidAlphabet{2|4}}.data words: symbol i
 *    (0-based) at bits [i*bps mod 64, +bps) of word i*bps div 64.
 *  - one stream per context; calls on one context must be serialised by the caller;
 *    distinct contexts are independent.
 */
#ifndef KMERSCUDA_H
#define KMERSCUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KMC_VERSION 100 /* 0.1.0 */
#define KMC_MAX_K 128   /* N <= 4 limbs */
#define KMC_MAX_K4 64   /* k-mers over a 4-bit alphabet (KMC_KMER4): N <= 4 limbs */

/* status codes */
#define KMC_OK 0
#define KMC_E_BAD_K 1         /* K < 1 ("K must be at least 1", FwKmers.jl:32-33) or K > KMC_MAX_K */
#define KMC_E_BAD_ARG 2       /* null / inconsistent descriptor */
#define KMC_E_AMBIGUOUS 3     /* a symbol cannot be encoded in the 2-bit alphabet: strict 4->2 recoding hit an
                                 uncertain symbol (construction.jl:108-110), or an ASCII source holds a byte
                                 that is not a valid letter (FwKmers.jl:124-126, UnambiguousKmers.jl:123-124).
                                 The caller throws BioSequences.EncodeError; result->err_* say where / what */
#define KMC_E_OUT_TOO_SMALL 4 /* kmc_out.capacity < number of elements to write */
#define KMC_E_NO_DEVICE 5
#define KMC_E_UNSUPPORTED 6
#define KMC_E_NCCL 7          /* a multi-GPU entry point failed inside NCCL, or NCCL could not be loaded
                                 (libnccl.so.2 is bound at run time); kmc_last_error says which */

/* iterator selected (kmc_extract `mode`) */
#define KMC_FW 0      /* FwKmers{A,K}            src/iterators/FwKmers.jl:28-59,88-115      */
#define KMC_FWRV 1    /* FwRvIterator{A,K}       src/iterators/CanonicalKmers.jl:25-56,94-144 */
#define KMC_CANON 2   /* CanonicalKmers{A,K}     src/iterators/CanonicalKmers.jl:199-225    */
#define KMC_UNAMBIG 3 /* UnambiguousKmers{A,K}   src/iterators/UnambiguousKmers.jl:29-148   */

/* flags */
#define KMC_HASH_FX 0x1u /* also emit fx_hash(x, 0) (src/kmer.jl:255-261) of the k-mer written to
                            out.a (fw for FW/FWRV/UNAMBIG, canonical for CANON) */
#define KMC_AOS 0x2u     /* Julia element layout for tuple eltypes: FWRV -> out.a holds
                            Tuple{Kmer,Kmer} = u64[n][2][N]; UNAMBIG -> out.a holds
                            Tuple{Kmer,Int} = {u64[N]; i64}[n].  Default is SoA
                            (out.a / out.b / out.index separate). */
#define KMC_NO_SYNC 0x4u /* do not synchronise the stream before returning (2-bit sources,
                            fixed-count modes only; result->n_written is still exact) */
#define KMC_OUT_DEVICE 0x8u /* kmc_extract_host only: the kmc_out buffers are DEVICE memory (the
                            sequences still come from the host).  The streams stay in HBM for a
                            device consumer; out.seq_out_offset must be NULL. */
#define KMC_RNA 0x20u    /* the k-mer alphabet is RNAAlphabet{2} (default DNAAlphabet{2}).  The limbs are
                            bit-identical; it only matters for strict iteration over ASCII sources,
                            where U (not T) is the fourth valid letter. */
#define KMC_KMER4 0x40u  /* the k-mers are over a 4-bit alphabet, Kmer{DNAAlphabet{4},K,N} / Kmer{RNAAlphabet{4},K,N}
                            with N = cld(4K, 64) limbs, K <= KMC_MAX_K4: FW / FWRV / CANON from a 4-bit source
                            (Copyable, FwKmers.jl:88-94, CanonicalKmers.jl:107-120; every symbol is allowed),
                            from a 2-bit source (TwoToFour, FwKmers.jl:96-102, CanonicalKmers.jl:122-129) or from
                            ASCII bytes (AsciiEncode, FwKmers.jl:117-129, CanonicalKmers.jl:146-174: every IUPAC
                            letter and the gap '-' in either case, T for DNA / U with KMC_RNA; any other byte in
                            a sequence of at least K symbols is KMC_E_AMBIGUOUS). */
#define KMC_DIGEST 0x10u /* kmc_extract_host only: also fingerprint what was written -- xor and wrapping
                            sum of the out.a words and of the out.hash words -> result->digest[4].
                            For FwKmers / CanonicalKmers over 2-bit sources (SoA, K <= 64) the extraction
                            kernel accumulates it from its own registers; other forms are fingerprinted
                            chunk by chunk by a second kernel right behind the one that wrote the chunk. */

typedef struct kmc_ctx kmc_ctx;
typedef struct kmc_group kmc_group; /* one process driving several GPUs: a context per device + one NCCL communicator */
#define KMC_COMM_ID_BYTES 128       /* size of the communicator id of kmc_comm_unique_id (an ncclUniqueId) */

/* A set of sequences resident in device memory.  n_seqs == 1 is a single LongSequence.
 * Ragged sets give word-aligned CSR offsets; uniform sets (every read the same length,
 * fixed word stride) leave seq_word_offset / seq_len NULL.
 * src_bits == 8 describes ASCII sources (String / codeunits / Vector{UInt8}: the AsciiEncode scheme,
 * construction.jl:95-96): `words` then points at BYTES (no alignment required) and every "word"
 * quantity below -- n_words, seq_word_offset, uniform_stride_words -- counts bytes. */
typedef struct kmc_seqs {
    const uint64_t *words;           /* device: concatenated LongSequence.data */
    uint64_t n_words;                /* number of u64 words addressable at `words` */
    uint64_t n_seqs;
    const uint64_t *seq_word_offset; /* device u64[n_seqs] first word of each sequence, or NULL */
    const uint64_t *seq_len;         /* device u64[n_seqs] symbols per sequence, or NULL */
    uint64_t uniform_len;            /* used when seq_len == NULL */
    uint64_t uniform_stride_words;   /* used when seq_word_offset == NULL */
    uint32_t src_bits;               /* 2 (Copyable, construction.jl:75-80), 4 (FourToTwo, :85-86) or
                                        8 (ASCII bytes, AsciiEncode, :95-96) */
    uint32_t first_symbol_offset;    /* symbols skipped at the start of every sequence (LongSubSeq view) */
} kmc_seqs;

/* Output buffers (device for kmc_extract, host for kmc_extract_host).  Unused ones NULL. */
typedef struct kmc_out {
    uint64_t *a;              /* FW/FWRV: fw k-mers; CANON: canonical; UNAMBIG: k-mers. (AoS: tuples) */
    uint64_t *b;              /* FWRV SoA: reverse-complement k-mers */
    uint64_t *hash;           /* KMC_HASH_FX: u64[n] */
    int64_t *index;           /* UNAMBIG SoA: 1-based start of each k-mer in its sequence */
    uint64_t *seq_out_offset; /* optional u64[n_seqs+1]: element offset of each sequence's output */
    uint64_t capacity;        /* elements (k-mers) each buffer can hold */
    int64_t index_base;       /* added to every emitted index (shards of one long sequence) */
} kmc_out;

typedef struct kmc_result {
    uint64_t n_written; /* elements produced (== length(iterator) summed over sequences) */
    uint64_t err_seq;   /* KMC_E_AMBIGUOUS: 0-based sequence, */
    uint64_t err_pos;   /*   1-based symbol position within it, */
    uint32_t err_sym;   /*   and the offending 4-bit encoding (reinterpret(DNA, x)) or ASCII byte */
    float kernel_ms;    /* device time of the launches of this call (cudaEvents), 0 with KMC_NO_SYNC */
    uint64_t digest[4]; /* KMC_DIGEST: xor(a), sum(a), xor(hash), sum(hash) */
} kmc_result;

/* ---- lifecycle ------------------------------------------------------------------ */
int32_t kmc_version(void);
int32_t kmc_device_count(int32_t *n);
int32_t kmc_ctx_create(int32_t device, kmc_ctx **ctx);
int32_t kmc_ctx_destroy(kmc_ctx *ctx);
/* Launch on an existing CUDA stream (cudaStream_t / CUstream handle, e.g. torch's current
 * stream) instead of the context's own.  NULL restores the context's own stream. */
int32_t kmc_ctx_set_stream(kmc_ctx *ctx, void *cuda_stream);
int32_t kmc_sync(kmc_ctx *ctx);
/* Stream-ordered temporaries (the binned counts take 8-16 bytes per k-mer) are cached in a memory pool the
 * context owns; this gives the cached memory back to the device.  Synchronises. */
int32_t kmc_trim(kmc_ctx *ctx);
const char *kmc_last_error(kmc_ctx *ctx);
const char *kmc_status_string(int32_t status);
int32_t kmc_device_info(kmc_ctx *ctx, int32_t *sm_count, uint64_t *total_mem, char *name, int32_t name_len);

/* ---- memory ----------------------------------------------------------------------- */
int32_t kmc_malloc(kmc_ctx *ctx, uint64_t bytes, void **dptr);
int32_t kmc_free(kmc_ctx *ctx, void *dptr);
int32_t kmc_memset(kmc_ctx *ctx, void *dptr, int32_t value, uint64_t bytes);
int32_t kmc_upload(kmc_ctx *ctx, void *dptr, const void *host, uint64_t bytes);   /* async on the stream */
int32_t kmc_download(kmc_ctx *ctx, void *host, const void *dptr, uint64_t bytes); /* synchronises */
int32_t kmc_host_alloc(kmc_ctx *ctx, uint64_t bytes, void **hptr); /* pinned */
int32_t kmc_host_free(kmc_ctx *ctx, void *hptr);
int32_t kmc_host_register(kmc_ctx *ctx, void *hptr, uint64_t bytes); /* pin caller memory (a Julia Vector) */
int32_t kmc_host_unregister(kmc_ctx *ctx, void *hptr);

/* ---- the hot path ------------------------------------------------------------------- */
/* Base.length(it) summed over the set (FwKmers.jl:40-43); for KMC_UNAMBIG over a 4-bit
 * source (IteratorSize = SizeUnknown, UnambiguousKmers.jl:33-37) runs the count pass. */
int32_t kmc_count(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint64_t *n_out);

/* collect(Iterator{A,K}(seq)) for every sequence of the set, concatenated in order.
 * Replaces the per-symbol loops of FwKmers.jl:88-115, CanonicalKmers.jl:94-144,220-225
 * and UnambiguousKmers.jl:64-77,134-148 with batched device launches. */
int32_t kmc_extract(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint32_t flags,
                    const kmc_out *out, kmc_result *result);

/* Same call with HOST buffers (seqs->words/offsets/lens and every kmc_out pointer are host
 * addresses, ideally pinned): uploads, extracts and downloads in pipelined chunks on
 * internal streams.  This is the call a Julia `collect(it)` replacement makes. */
int32_t kmc_extract_host(kmc_ctx *ctx, const kmc_seqs *host_seqs, int32_t k, int32_t mode, uint32_t flags,
                         const kmc_out *host_out, kmc_result *result);

/* collect(SpacedKmers{A,K,J}(seq)) for every sequence of the set (src/iterators/SpacedKmers.jl:22-139; each_codon =
 * SpacedKmers{A,3,3}, :78-82): the k-mers at the 1-based starts 1, 1+J, 1+2J, ... -- div(L - K, J) + 1 per sequence
 * of L >= K symbols (:36-40) -- concatenated in order into out.a (N limbs each), out.hash (KMC_HASH_FX) and
 * optionally out.seq_out_offset.  Device buffers.  Every recoding scheme of the nucleotide alphabets
 * (construction.jl:75-100): 2-bit / 4-bit / ASCII sources into 2-bit k-mers (K <= KMC_MAX_K) or, with KMC_KMER4,
 * 4-bit k-mers (K <= KMC_MAX_K4); KMC_RNA as for kmc_extract.  A symbol that cannot be encoded INSIDE a sampled
 * window is KMC_E_AMBIGUOUS (result->err_*); symbols between the windows of a step J > K are not read, as in the
 * reference.  step < 1 is KMC_E_BAD_K ("J must be at least 1", SpacedKmers.jl:30). */
int32_t kmc_extract_spaced(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t step, uint32_t flags,
                           const kmc_out *out, kmc_result *result);

/* fx_hash.(v, h0) over n k-mers of n_limbs limbs each already in device memory
 * (src/kmer.jl:255-261). */
int32_t kmc_fx_hash(kmc_ctx *ctx, const uint64_t *kmers, uint64_t n, int32_t n_limbs, uint64_t h0,
                    uint64_t *out);

/* Base.hash.(v, h0) (src/kmer.jl:206: hash(x.data, h ⊻ K)) over n k-mers of K symbols and n_limbs limbs
 * in device memory, with the tuple / UInt64 hashing of Julia 1.10 and 1.11 (hash_64_64).  Pinned by
 * the reference's documented hash(mer"UGCUGUAC"r) == 0xe5057d38c8907b22 (docs/src/hashing.md:18-20);
 * the reference warns that values change between Julia minors (hashing.md:10-13), so a binding must
 * check that value against its own Julia before using this entry point. */
int32_t kmc_base_hash(kmc_ctx *ctx, const uint64_t *kmers, uint64_t n, int32_t n_limbs, int32_t k, uint64_t h0,
                      uint64_t *out);

/* north_star extension (not in the reference): histogram of
 * fx_hash(canonical k-mer) >> (64 - bucket_bits) over the set, accumulated into
 * table[2^bucket_bits] (u32, device, caller-zeroed).  Tables of several GPUs are summed by
 * kmc_bucket_count_merge / kmc_group_bucket_count below (NCCL all-reduce over NVLink). */
int32_t kmc_bucket_count(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t bucket_bits,
                         uint32_t *table, kmc_result *result);

/* kmc_bucket_count without the final synchronisation and with progress events, so that the merge of
 * the tables of several GPUs -- the path's only collective -- overlaps the counting: the table is cut
 * into n_parts equal contiguous ranges (n_parts = 1, 2, 4, ... 32) and events[i] (a cudaEvent_t created
 * by the caller) is recorded on the context's stream as soon as range i holds its final counts.  A
 * caller all-reduces range i on a second stream that waits for events[i] while later ranges are still
 * being counted (tables beyond L2 are filled slice after slice; an L2-sized table is final only at the
 * end, and all events are recorded there).  result->n_written is set; result->kernel_ms is not.  The
 * call is complete when events[n_parts - 1] has completed (or after kmc_sync). */
int32_t kmc_bucket_count_async(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t bucket_bits,
                               uint32_t *table, uint32_t n_parts, void *const *events, kmc_result *result);

/* Minimizers: "the minimum of W consecutive kmers, as ordered by some ordering O"
 * (docs/src/replacements.md:28-30) with fx_hash as the ordering (replacements.md:32-58,
 * test/benchmark.jl:96-119).  For every window start i = 1, 1+step, 1+2*step, ... that has W
 * k-mers available, out.a gets the k-mer with the smallest fx_hash among the k-mers starting at
 * i .. i+W-1 (ties: the first), out.hash (KMC_HASH_FX) its hash and out.index (optional) its
 * 1-based start.  mode KMC_FW orders forward k-mers as the reference example does, KMC_CANON
 * canonical k-mers.  Device buffers; 2-bit sources; K <= 32 and K + W - 1 <= 64.  The full
 * k-mer stream is never written. */
int32_t kmc_minimizers(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t w, int32_t step, int32_t mode,
                       uint32_t flags, const kmc_out *out, kmc_result *result);

/* Bottom-s MinHash sketch under fx_hash: the reference's example
 * `sketch(fx_hash, CanonicalDNAMers{16}(seq), 1000)` (docs/src/minhash.md:31-36; MinHash.jl is an
 * external package: the published bottom-s definition is used) -- the s smallest DISTINCT fx_hash
 * values over all (forward: KMC_FW, canonical: KMC_CANON) k-mers of the set, ascending, into
 * out_hashes (device u64[s]); result->n_written = how many there are (< s if the set has fewer
 * distinct k-mers).  2-bit sources, K <= 64.  The k-mer stream is never written: two passes over
 * the sequence (a 4096-bucket histogram of the top hash bits, then the candidates below the
 * threshold bucket), a sort of s + one bucket's worth of candidates. */
int32_t kmc_minhash_sketch(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint64_t s,
                           uint64_t *out_hashes, kmc_result *result);

/* The bottom-s sketch of every sequence of the set on its own: row i of out_hashes (device u64[n_seqs][s]) holds,
 * ascending, exactly what kmc_minhash_sketch returns for a set made of sequence i alone; out_n[i] (device u32[n_seqs])
 * is its length: min(s, distinct k-mers of sequence i), 0 for a sequence shorter than K.  Slots past out_n[i] are ~0.
 * KMC_FW / KMC_CANON, 2-bit sources, K <= 64, single sequences, uniform and ragged sets, first_symbol_offset views.
 * result->n_written = sum of out_n; result->kernel_ms as for the other consumers; result->digest[0] = rounds run past
 * the first, result->digest[1] = sequences those rounds sketched again (sequences whose repeats left fewer than s
 * distinct k-mers below their first hash limit).  s < 1, n_seqs * s * 8 overflowing u64, a mode other than KMC_FW /
 * KMC_CANON and NULL pointers are KMC_E_BAD_ARG; K > 64 and other sources are KMC_E_UNSUPPORTED; n_seqs = 0 writes
 * nothing.  Temporary memory: 32 bytes per sequence and 16 bytes per candidate (about s + 4 sqrt(s) + 16 per long
 * sequence, every window of a sequence of fewer than about 2s + 8 sqrt(s) + 32 windows) plus the sort's scratch. */
int32_t kmc_minhash_sketch_each(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint64_t s,
                                uint64_t *out_hashes, uint32_t *out_n, kmc_result *result);

/* Every sketch of list A against every sketch of list B (device rows of s u64, ascending and distinct, lengths a_n /
 * b_n; a length above s is read as s; A and B may be the same arrays).  For pair (i, j), at i * n_b + j (device u32):
 *   shared[]        = |A_i ∩ B_j|
 *   shared_bottom[] = |S_s(A_i ∪ B_j) ∩ A_i ∩ B_j|, S_s = the s smallest values   (Mash's estimator numerator)
 * so the Mash Jaccard estimate is shared_bottom / min(s, n_A + n_B - shared).  Either output may be NULL.  s in
 * 1..16384 (KMC_E_UNSUPPORTED above, KMC_E_BAD_ARG for 0); n_a = 0 or n_b = 0 does nothing.  No row is read past its
 * length, whatever the rows contain.  Synchronises. */
int32_t kmc_minhash_compare(kmc_ctx *ctx, const uint64_t *a, const uint32_t *a_n, uint64_t n_a,
                            const uint64_t *b, const uint32_t *b_n, uint64_t n_b, uint64_t s,
                            uint32_t *shared, uint32_t *shared_bottom);

/* k-mer composition vector: table[as_integer(kmer)] += 1 for every k-mer of the set
 * (docs/src/composition.md:28-39 counts FwDNAMers{4}; as_integer: src/kmer.jl:305-326), forward
 * (KMC_FW) or canonical (KMC_CANON) k-mers, K <= 14.  table: device u32[4^K], caller-zeroed
 * (accumulates, so several sets / GPUs can be summed).  2-bit sources. */
int32_t kmc_composition(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint32_t *table,
                        kmc_result *result);

/* Exact k-mer counts, keyed by the k-mer: the `Dict{Kmer,Int}` a user of the iterators builds (the reference
 * discusses counting in src/iterators/CanonicalKmers.jl:183-185 and docs/src/composition.md).  The table is
 * open addressing in caller-owned device memory: keys u64[2^log2_capacity] (free slot = ~0: initialise with
 * kmc_memset(keys, 0xff, ...)), vals u32[2^log2_capacity] (zeroed); fx_hash of the k-mer picks the slot, linear
 * probing.  Accumulates, so several sets can be counted into one table.  Forward (KMC_FW, K <= 31) or canonical
 * (KMC_CANON, K <= 32) k-mers of a 2-bit source.  result->n_written = k-mers counted, result->digest[0] = keys
 * this call added; KMC_E_OUT_TOO_SMALL when the table is full (its contents are then incomplete). */
int32_t kmc_kmer_count(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint64_t *keys, uint32_t *vals,
                       uint32_t log2_capacity, kmc_result *result);
/* Adds every (key, count) with key != ~0 of src (another table, or an entry list from kmc_kmer_table_export:
 * n_src slots) into the table -- the merge step of a multi-GPU count: each rank exports, the entries travel
 * (all-gather / all-to-all by key owner), the owner merges.  *n_new (optional) = keys added. */
int32_t kmc_kmer_table_merge(kmc_ctx *ctx, uint64_t *keys, uint32_t *vals, uint32_t log2_capacity,
                             const uint64_t *src_keys, const uint32_t *src_vals, uint64_t n_src, uint64_t *n_new);
/* The table's entries as two dense device arrays (unordered); *n_out = how many. */
int32_t kmc_kmer_table_export(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                              uint64_t *out_keys, uint32_t *out_vals, uint64_t capacity, uint64_t *n_out);
/* The same table for two-limb k-mers: forward (KMC_FW, K = 33..63) or canonical (KMC_CANON, K = 33..64) k-mers of a
 * 2-bit source.  keys: device u64[2^log2_capacity][2], 16-byte aligned, each entry Kmer{A,K,2}.data (head limb
 * first, unused top bits of limb 0 zero); free slot = both limbs ~0 (initialise with kmc_memset(keys, 0xff, 16 << cap));
 * vals u32[2^log2_capacity] (zeroed).  fx_hash of the k-mer picks the slot, linear probing; a free slot is claimed
 * with one 128-bit compare-and-swap.  Results and status as for kmc_kmer_count. */
int32_t kmc_kmer_count2(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, uint64_t *keys /* [2^cap][2] */,
                        uint32_t *vals, uint32_t log2_capacity, kmc_result *result);
/* kmc_kmer_table_merge / kmc_kmer_table_export of two-limb tables: src_keys u64[n_src][2], out_keys u64[capacity][2] */
int32_t kmc_kmer_table2_merge(kmc_ctx *ctx, uint64_t *keys, uint32_t *vals, uint32_t log2_capacity,
                              const uint64_t *src_keys /* [n_src][2] */, const uint32_t *src_vals, uint64_t n_src, uint64_t *n_new);
int32_t kmc_kmer_table2_export(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                               uint64_t *out_keys /* [capacity][2] */, uint32_t *out_vals, uint64_t capacity, uint64_t *n_out);
/* Read-only queries of a table filled by kmc_kmer_count / kmc_kmer_count2 (or merged into).  Precondition: no count or
 * merge into the same table is in flight -- calls on one context are stream ordered, so this holds unless another
 * context writes the table.  A key that is not in the table has count 0.  Every entry point below returns
 * KMC_E_BAD_ARG for a NULL pointer, log2_capacity outside 1..40, and two-limb keys / query / out_keys that are not
 * 16-byte aligned.
 *
 * The count of every window of a read set: out_counts[i] (device u32[capacity]) = table[k-mer i], in the order
 * kmc_extract writes the same k-mers (so out_counts[i] belongs to out.a[i]) -- the second pass of a k-mer-spectrum
 * error corrector or read filter.  The k-mers must be looked up with the mode the table was counted with (KMC_FW or
 * KMC_CANON); K, mode and source are checked as by kmc_kmer_count.  result->n_written = windows; capacity < windows is
 * KMC_E_OUT_TOO_SMALL and nothing is written.  Tables of any size are probed directly. */
int32_t kmc_kmer_lookup(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, const uint64_t *keys, const uint32_t *vals,
                        uint32_t log2_capacity, uint32_t *out_counts, uint64_t capacity, kmc_result *result);
/* The same for a two-limb table (kmc_kmer_count2): K and mode as there, keys u64[2^cap][2] */
int32_t kmc_kmer_lookup2(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t mode, const uint64_t *keys /* [2^cap][2] */,
                         const uint32_t *vals, uint32_t log2_capacity, uint32_t *out_counts, uint64_t capacity, kmc_result *result);
/* out_counts[i] = table[query[i]] for n keys in device memory (query u64[n] / u64[n][2]); n = 0 does nothing */
int32_t kmc_kmer_table_get(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                           const uint64_t *query, uint64_t n, uint32_t *out_counts);
int32_t kmc_kmer_table2_get(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                            const uint64_t *query /* [n][2] */, uint64_t n, uint32_t *out_counts);
/* The count spectrum: hist[min(count, n_bins - 1)] += 1 for every key of the table, so the last bin holds every count
 * of n_bins - 1 and more (bin 0 holds keys merged in with a zero count).  hist: device u64[n_bins], caller-zeroed; it
 * accumulates, so after kmc_kmer_table_exchange the histograms of the owned tables summed over the ranks with
 * kmc_allreduce_u64 are the spectrum of the whole input.  n_bins in 1..16384. */
int32_t kmc_kmer_table_histogram(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity, uint64_t *hist,
                                 uint32_t n_bins);
int32_t kmc_kmer_table2_histogram(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity, uint64_t *hist,
                                  uint32_t n_bins);
/* kmc_kmer_table_export of the entries with min_count <= count <= max_count only (the solid k-mers); *n_out and
 * KMC_E_OUT_TOO_SMALL as there, nothing is written past capacity.  min_count > max_count is KMC_E_BAD_ARG. */
int32_t kmc_kmer_table_export_range(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                                    uint32_t min_count, uint32_t max_count, uint64_t *out_keys, uint32_t *out_vals,
                                    uint64_t capacity, uint64_t *n_out);
int32_t kmc_kmer_table2_export_range(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                                     uint32_t min_count, uint32_t max_count, uint64_t *out_keys /* [capacity][2] */,
                                     uint32_t *out_vals, uint64_t capacity, uint64_t *n_out);

/* ---- multi-GPU (SURVEY.md 8b / 8e) ---------------------------------------------------------------
 * The reference has no collective (it is single-threaded Julia); north_star shards reads over the GPUs of a box
 * by sequence and merges ONE thing: the optional canonical k-mer count table (the consumer discussed at
 * src/iterators/CanonicalKmers.jl:183-185, docs/src/composition.md:28-39).  The k-mer / hash / index streams never
 * cross GPUs.  Two ways to drive several GPUs, over the same code:
 *   - one process, a kmc_group (what a Julia session is): kmc_group_create makes a context per device and an NCCL
 *     communicator over them (ncclCommInitAll); per-device descriptors are passed as arrays indexed by device;
 *   - one process per GPU (torchrun, MPI): rank 0 makes an id (kmc_comm_unique_id), the launcher broadcasts its
 *     128 bytes, every rank attaches a communicator to its context (kmc_comm_init_rank).
 * NCCL is loaded at run time; without it these entry points return KMC_E_NCCL (a group of ONE device needs none). */
int32_t kmc_nccl_version(int32_t *version);
int32_t kmc_comm_unique_id(void *id128);
int32_t kmc_comm_init_rank(kmc_ctx *ctx, int32_t n_ranks, int32_t rank, const void *id128);
int32_t kmc_comm_destroy(kmc_ctx *ctx);
int32_t kmc_comm_info(kmc_ctx *ctx, int32_t *rank, int32_t *n_ranks);
/* in-place sum over the ranks of n counters in device memory, enqueued on the context's stream */
int32_t kmc_allreduce_u32(kmc_ctx *ctx, uint32_t *buf, uint64_t n);
int32_t kmc_allreduce_u64(kmc_ctx *ctx, uint64_t *buf, uint64_t n);
/* kmc_bucket_count of this rank's reads + the sum over all ranks, the merge overlapping the count: every eighth of
 * the table is all-reduced on a communication stream as soon as the count has finished it.  On return (it
 * synchronises) every rank's table holds the merged counts; result->n_written = k-mers THIS rank counted,
 * result->kernel_ms = device time from the first count kernel to the end of the last all-reduce.  Collective. */
int32_t kmc_bucket_count_merge(kmc_ctx *ctx, const kmc_seqs *seqs, int32_t k, int32_t bucket_bits, uint32_t *table,
                               kmc_result *result);
/* The exact k-mer table across GPUs.  Every key has one owner rank, kmc_kmer_owner(key, n_ranks) (a second mix of
 * the key's fx_hash, independent of the bits that pick its slot).  The call sends every (key, count) of this
 * rank's table (kmc_kmer_count) to its owner -- grouped ncclSend / ncclRecv, NVLink peer traffic -- and the owner
 * adds what it receives, and its own share, into owned_keys / owned_vals (a table like kmc_kmer_count's,
 * initialised by the caller).  *n_owned = keys added to the owned table.  Afterwards the union of the owned tables
 * is the count of the whole input, each key on exactly one rank.  Collective. */
uint32_t kmc_kmer_owner(uint64_t key, uint32_t n_ranks);
int32_t kmc_kmer_table_exchange(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                                uint64_t *owned_keys, uint32_t *owned_vals, uint32_t owned_log2_capacity, uint64_t *n_owned);
/* The same for two-limb tables (kmc_kmer_count2): the owner of {limb0, limb1} is the same second mix taken over
 * fx_hash of both limbs; entries travel as 2n u64, the owner merges with kmc_kmer_table2_merge. */
uint32_t kmc_kmer_owner2(uint64_t limb0, uint64_t limb1, uint32_t n_ranks);
int32_t kmc_kmer_table2_exchange(kmc_ctx *ctx, const uint64_t *keys, const uint32_t *vals, uint32_t log2_capacity,
                                 uint64_t *owned_keys, uint32_t *owned_vals, uint32_t owned_log2_capacity, uint64_t *n_owned);

/* devices == NULL selects devices 0 .. n-1 */
int32_t kmc_group_create(int32_t n, const int32_t *devices, kmc_group **group);
int32_t kmc_group_destroy(kmc_group *group);
int32_t kmc_group_size(kmc_group *group, int32_t *n);
int32_t kmc_group_ctx(kmc_group *group, int32_t i, kmc_ctx **ctx); /* device i's context (memory, uploads, single-GPU calls) */
int32_t kmc_group_sync(kmc_group *group);
/* bufs[i]: n counters on device i; in-place sum, enqueued on every context's stream */
int32_t kmc_group_allreduce_u32(kmc_group *group, uint32_t *const *bufs, uint64_t n);
int32_t kmc_group_allreduce_u64(kmc_group *group, uint64_t *const *bufs, uint64_t n);
/* seqs[i] / tables[i] / results[i] belong to device i: kmc_bucket_count_merge on every device of the group (C5) */
int32_t kmc_group_bucket_count(kmc_group *group, const kmc_seqs *seqs, int32_t k, int32_t bucket_bits,
                               uint32_t *const *tables, kmc_result *results);
/* kmc_extract / kmc_extract_host on every device side by side (one host thread per device); shard i of a read
 * set (or the i-th window range of one long sequence, out.index_base = its first window) goes to device i, and
 * the concatenation of the outputs in device order is the single-GPU (= reference) order */
int32_t kmc_group_extract(kmc_group *group, const kmc_seqs *seqs, int32_t k, int32_t mode, uint32_t flags,
                          const kmc_out *outs, kmc_result *results);
int32_t kmc_group_extract_host(kmc_group *group, const kmc_seqs *host_seqs, int32_t k, int32_t mode, uint32_t flags,
                               const kmc_out *host_outs, kmc_result *results);
int32_t kmc_group_kmer_table_exchange(kmc_group *group, const uint64_t *const *keys, const uint32_t *const *vals,
                                      uint32_t log2_capacity, uint64_t *const *owned_keys, uint32_t *const *owned_vals,
                                      uint32_t owned_log2_capacity, uint64_t *n_owned);
int32_t kmc_group_kmer_table2_exchange(kmc_group *group, const uint64_t *const *keys, const uint32_t *const *vals,
                                       uint32_t log2_capacity, uint64_t *const *owned_keys, uint32_t *const *owned_vals,
                                       uint32_t owned_log2_capacity, uint64_t *n_owned);

/* XOR and wrapping sum of n u64 words in device memory -> out[0], out[1] (host).  A cheap
 * fingerprint of a device-resident stream: parity checks and result read-back at sizes where
 * downloading the stream itself would only measure PCIe.  Synchronises. */
int32_t kmc_digest(kmc_ctx *ctx, const uint64_t *dptr, uint64_t n, uint64_t *out);

/* ---- timing (cudaEvents on the context's stream) ------------------------------------ */
int32_t kmc_timer_begin(kmc_ctx *ctx);
int32_t kmc_timer_end(kmc_ctx *ctx, float *ms); /* synchronises */

/* ---- measurement aid: pure 256-bit streaming store of `bytes` (write roofline probe) --
 * The environment variable KMC_STORE_PROBE_PATTERN selects variants of the probe that reproduce the
 * extraction kernels' store pattern with and without their source reads (tools/bw_probe.py; the
 * experiments behind DESIGN.md 3.1).  Not part of the drop-in boundary. */
int32_t kmc_store_probe(kmc_ctx *ctx, void *dptr, uint64_t bytes);

#ifdef __cplusplus
}
#endif
#endif /* KMERSCUDA_H */
