// fourbit.h -- sources that are recoded on the device before extraction: 4-bit (DNAAlphabet{4} /
// RNAAlphabet{4}) LongSequences, the FourToTwo scheme (src/construction.jl:85-86), and ASCII byte
// strings, the AsciiEncode scheme (construction.jl:95-96, ascii.cu).
//
// A 4-bit source is first recoded on the device into (i) a 2-bit stream (trailing_zeros of each
// one-hot nibble, construction_utils.jl:41-54) and (ii) a bit stream that flags every uncertain
// symbol (count_ones != 1: IUPAC ambiguity codes, N and gap).  From (ii) a "valid start" bit
// stream is derived: bit P = no uncertain symbol in [P, P+K).  The 2-bit extraction kernels then
// run unchanged on (i) and consult the valid-start bits:
//   strict FwKmers / FwRvIterator / CanonicalKmers (FwKmers.jl:104-115, CanonicalKmers.jl:131-144):
//     the first window with an uncertain symbol is reported; the call fails with KMC_E_AMBIGUOUS
//     and the position / encoding the reference's throw_uncertain (construction.jl:108-110) names;
//   UnambiguousKmers (UnambiguousKmers.jl:134-148): windows with an uncertain symbol are skipped.
//     compact_kernel (compact_kernels.cuh) computes the windows like the 2-bit kernels do and
//     compacts the survivors in order, each k-mer with its 1-based start inside its read, in a
//     single pass (decoupled look-back over the tiles; aligned 256-bit stores from a staging buffer).
#pragma once
#include "fourbit_core.cuh"
#include "lincompact.cuh"
#include "plan.h"

namespace kmc {

// The source-order compaction's layout (lincompact.cuh, lin_prepare in valid_count.cu)
struct LinPlan {
    bool linear = false;  // the set's sequences are ascending and disjoint in the buffer: lin_compact_kernel runs
    bool offsets = false; // the set gives per-sequence offsets
    LinParams lp{};
    const uint64_t *total_dev = nullptr; // device: the number of k-mers the set emits (last entry of the chunk scan)
};
bool lin_enabled();
bool lin_uniform_ok(const kmc_seqs *s, int k);
uint64_t lin_chunks(uint64_t n_positions);
uint64_t lin_scratch_bytes(uint64_t n_symbols, uint64_t n_seqs);
int32_t lin_prepare(kmc_ctx *ctx, const ExtractParams &p, const kmc_seqs *s, int k, uint64_t n_vstart_words,
                    int known_linear, uint64_t *host_flag, cudaStream_t stream, Scratch &scratch, LinPlan *plan);

// What one 4-bit extraction needs between its two phases.  Phase A enqueues the recoding (and, for
// strict modes, the extraction) and leaves two words in `host_small` (pinned): [0] = number of k-mers
// UnambiguousKmers will emit (only when asked to count first), [1] = first offending flat window of a
// strict mode / first sequence with an invalid byte (~0 = none).
// Phase B runs after the caller has synchronised the stream.
struct FourBitState {
    const kmc_seqs *seqs = nullptr; // device descriptor (must outlive phase B)
    const uint64_t *words4 = nullptr;
    int k = 0, mode = 0;
    uint32_t flags = 0;
    Geometry ge{};
    Layout L{};      // layout for the kernel's G (count only: G = 32)
    ExtractParams p{};
    uint32_t *bad = nullptr;
    uint32_t *err = nullptr; // ASCII UnambiguousKmers: hard-error flags (bytes outside the skipping table)
    unsigned long long *tile_state = nullptr; // UnambiguousKmers: look-back descriptors of compact_kernel
    std::shared_ptr<AsyncBuf> tile_state_buf; // tile_state when the scratch window cannot hold it (overlapping sequences)
    unsigned long long *total_dev = nullptr;  // UnambiguousKmers: emitted k-mers (device)
    LinPlan lin;                              // UnambiguousKmers: the source-order compaction, when the layout allows it
    bool counted = false;                     // host_small[0] holds the count when phase A has completed
    uint64_t *err_out = nullptr; // device u64[3]: seq, 1-based pos, encoding
    uint64_t *host_small = nullptr;
    uint64_t unit_bias = 0;
    bool unambig = false;
};

// valid_count.cu: *total += survivors of the set laid out in groups of g windows (g = 2, 4, 8 or 32)
cudaError_t count_valid(const ExtractParams &p, bool ragged, int g, unsigned long long *total, cudaStream_t stream);

// (valid_start_word: fourbit_core.cuh)
constexpr int kRecodeGroups = 4; // groups of 32 symbols per thread of the 4-bit recoding pass
constexpr int kRecodeHalo = 5; // flag words beyond a group that its windows can reach (31 + K - 1 <= 158 bits)

// ascii.cu: byte sources (AsciiEncode).  lut: 0 = strict DNAAlphabet{2}, 1 = strict RNAAlphabet{2},
// 2 = the UnambiguousKmers skipping table.  n_groups = groups of 32 bytes.
// Writes rec / bad / err for the groups [0, n_groups) and the valid-start words [0, n_vstart).
// rev (optional, both recoding passes): the codes once more as a stream in REVERSED symbol order (2 u32 per group)
cudaError_t ascii_recode(const uint8_t *bytes, uint64_t n_bytes, int lut, int k, uint32_t *rec, uint32_t *bad, uint32_t *err,
                         uint32_t *vstart, uint64_t n_groups, uint64_t n_vstart, cudaStream_t stream, uint32_t *rev = nullptr,
                         unsigned long long *any_err = nullptr);
// (any_err, optional: a device word the pass clears and then sets if it flags any byte as an error)
// the first sequence (of at least min_len symbols) that holds a flagged byte -> atomicMin into *err_seq
cudaError_t ascii_first_error_seq(const ExtractParams &p, const uint32_t *err, const uint64_t *seq_len, uint64_t uniform_len,
                                  unsigned long long *err_seq, int sm_count, cudaStream_t stream, uint64_t min_len = 0,
                                  const unsigned long long *any_err = nullptr);
// ASCII bytes -> nibbles of a 4-bit alphabet (2 u64 per group of 32 bytes) + error flags + the valid-start words
cudaError_t ascii4_recode(const uint8_t *bytes, uint64_t n_bytes, bool rna, int k, uint64_t *nib, uint32_t *bad, uint32_t *vstart,
                          uint64_t n_groups, uint64_t n_vstart, cudaStream_t stream, unsigned long long *any_err = nullptr);
// fourbit.cu: the FourToTwo recoding pass (2-bit codes, uncertainty flags, valid-start words); n_groups = groups of 32 symbols
cudaError_t fourbit_recode(const uint64_t *words, uint64_t n_words, int k, uint32_t *rec, uint32_t *bad, uint32_t *vstart,
                           uint64_t n_groups, uint64_t n_vstart, cudaStream_t stream, uint32_t *rev = nullptr);
// kmer4.cu: TwoToFour, every 2-bit source word -> 128 bits of one-hot nibbles
cudaError_t expand_two_to_four(const uint64_t *words, uint64_t n_words, void *wide, cudaStream_t stream);
cudaError_t ascii_resolve_error(const ExtractParams &p, const uint8_t *bytes, const uint32_t *err, const uint64_t *seq_len,
                                uint64_t uniform_len, uint64_t r, uint64_t *err_out, cudaStream_t stream);

uint64_t fourbit_scratch_bytes(const kmc_seqs *s, int k, int mode);

// count_first (UnambiguousKmers): also count the survivors, so that phase B knows n_written before it
// enqueues the compaction (the host pipeline needs it to place the next chunk).  out == NULL: count only.
int32_t fourbit_phase_a(kmc_ctx *ctx, const kmc_seqs *s, int32_t k, int32_t mode, uint32_t flags, const kmc_out *out,
                        cudaStream_t stream, const KnownTotals &known, uint64_t unit_bias, Scratch &scratch,
                        uint64_t *host_small, bool count_first, FourBitState *st);
// Fills res->n_written (and err_* with KMC_E_AMBIGUOUS).  For UnambiguousKmers: enqueues the compaction;
// without count_first, n_written is host_small[0] once the stream has been synchronised
// (fourbit_unambig_result).
int32_t fourbit_phase_b(kmc_ctx *ctx, FourBitState *st, const kmc_out *out, cudaStream_t stream, kmc_result *res);
int32_t fourbit_unambig_result(kmc_ctx *ctx, const FourBitState *st, const kmc_out *out, kmc_result *res);

// kmc_extract on device buffers: phase A, sync, phase B, sync.
int32_t extract_device_4bit(kmc_ctx *ctx, const kmc_seqs *s, int32_t k, int32_t mode, uint32_t flags,
                            const kmc_out *out, kmc_result *res, cudaStream_t stream);
int32_t count_unambiguous_4bit(kmc_ctx *ctx, const kmc_seqs *s, int32_t k, uint64_t *n_out, cudaStream_t stream);

} // namespace kmc
