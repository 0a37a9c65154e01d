"""
    KmersCUDA

Drop-in GPU (NVIDIA B200, sm_100a) replacement for the k-mer *extraction* path of Kmers.jl:
`collect` of `FwKmers`, `FwRvIterator`, `CanonicalKmers` and `UnambiguousKmers` over
`LongSequence` / `LongSubSeq{<:NucleicAcidAlphabet{2|4}}` and ASCII sources (`String`, `SubString`,
`codeunits`, byte vectors, `StringView`), plus `fx_hash`.  Every number is computed by
`libkmerscuda.so` (hand-written CUDA) through `ccall`; there is no CUDA.jl codegen and no CPU
fallback.  Results are bit-identical to the reference's own iterators.

Three ways to get results, from the drop-in to the fast one:

  * `KmersCUDA.collect(it)`                 what `Base.collect(it)` returns, in host memory (PCIe-bound for large inputs:
                                            16 bytes per k-mer cross the link);
  * `KmersCUDA.extract(Iter, reads; device = true)`   the streams stay in HBM as `DeviceVector`s (`Array(dv)` copies one to
                                            the host) for device consumers: `fx_hash_device`, `bucket_count`, `count_kmers`,
                                            `minhash_sketch`, ...; only the reads cross PCIe;
  * `Group(devices)`                        one process driving several GPUs: `extract(...; group)` shards the reads by
                                            sequence, `bucket_count(reads...; group)` counts on every GPU and merges the
                                            tables with NCCL inside the library (`kmc_group_bucket_count`).

NOTE: this module is written against include/kmerscuda.h but could not be executed in the build
environment (no Julia toolchain there); the Python mirror `kmers.jl_b200/kmerscuda` binds the
same symbols and is what the test-suite exercises.  test/runtests.jl is the parity suite to run
where Julia, Kmers.jl, BioSequences.jl and a B200 are present.
"""
module KmersCUDA

using BioSequences
using Kmers
using Kmers: FwKmers, FwRvIterator, CanonicalKmers, UnambiguousKmers, SpacedKmers, Kmer, derive_type
using Libdl

export fx_hash_device, hash_device, extract, set_library!, minhash_sketch, minhash_sketches, minhash_compare, composition, minimizers, count_kmers,
    bucket_count, DeviceVector, Group, free!, KmerCountTable, counts, spectrum

# ---------------------------------------------------------------------------------------------
# library handle
# ---------------------------------------------------------------------------------------------
const LIB = Ref{String}(get(ENV, "KMERSCUDA_LIB", "libkmerscuda.so"))
set_library!(path::AbstractString) = (LIB[] = String(path))

const KMC_OK = Int32(0)
const KMC_E_BAD_K = Int32(1)
const KMC_E_AMBIGUOUS = Int32(3)
const KMC_FW, KMC_FWRV, KMC_CANON, KMC_UNAMBIG = Int32(0), Int32(1), Int32(2), Int32(3)
const KMC_HASH_FX, KMC_AOS, KMC_OUT_DEVICE = UInt32(1), UInt32(2), UInt32(8)
const KMC_RNA = UInt32(0x20)     # strict iteration over ASCII: U, not T, is the fourth letter
const KMC_KMER4 = UInt32(0x40)   # k-mers over a 4-bit alphabet (Copyable 4 -> 4, TwoToFour)

# struct kmc_seqs / kmc_out / kmc_result of include/kmerscuda.h (same field order and sizes).  KmcResult is
# mutable and passed as Ref{KmcResult}: ccall hands the library the address of the object itself.
struct KmcSeqs
    words::Ptr{UInt64}
    n_words::UInt64
    n_seqs::UInt64
    seq_word_offset::Ptr{UInt64}
    seq_len::Ptr{UInt64}
    uniform_len::UInt64
    uniform_stride_words::UInt64
    src_bits::UInt32
    first_symbol_offset::UInt32
end

struct KmcOut
    a::Ptr{UInt64}
    b::Ptr{UInt64}
    hash::Ptr{UInt64}
    index::Ptr{Int64}
    seq_out_offset::Ptr{UInt64}
    capacity::UInt64
    index_base::Int64
end

mutable struct KmcResult
    n_written::UInt64
    err_seq::UInt64
    err_pos::UInt64
    err_sym::UInt32
    kernel_ms::Float32
    digest::NTuple{4, UInt64}
    KmcResult() = new(0, 0, 0, 0, 0.0f0, (0, 0, 0, 0))
end

mutable struct Context
    handle::Ptr{Cvoid}
    owned::Bool
    function Context(device::Integer = 0)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        st = ccall((:kmc_ctx_create, LIB[]), Int32, (Int32, Ptr{Ptr{Cvoid}}), device, h)
        st == KMC_OK || error("KmersCUDA: kmc_ctx_create failed ($(status_string(st))); a CUDA device is required, there is no CPU fallback")
        ctx = new(h[], true)
        finalizer(c -> c.owned && ccall((:kmc_ctx_destroy, LIB[]), Int32, (Ptr{Cvoid},), c.handle), ctx)
        return ctx
    end
    Context(handle::Ptr{Cvoid}, owned::Bool) = new(handle, owned)   # a context that belongs to a Group
end

status_string(st::Int32) = unsafe_string(ccall((:kmc_status_string, LIB[]), Cstring, (Int32,), st))
last_error(ctx::Context) = unsafe_string(ccall((:kmc_last_error, LIB[]), Cstring, (Ptr{Cvoid},), ctx.handle))

"Every `ccall` status goes through here: anything but KMC_OK throws."
function check(ctx::Context, st::Int32)
    st == KMC_OK && return nothing
    msg = last_error(ctx)
    error("libkmerscuda status $st: $(isempty(msg) ? status_string(st) : msg)")
end

const DEFAULT_CTX = Ref{Union{Nothing, Context}}(nothing)
default_context() = something(DEFAULT_CTX[], (DEFAULT_CTX[] = Context(0)))

# ---------------------------------------------------------------------------------------------
# device memory owned by the library
# ---------------------------------------------------------------------------------------------
"""
    DeviceVector{T}

`n` elements of isbits type `T` in the memory of the context's GPU (`kmc_malloc`).  `Array(dv)` copies them to the
host; `free!(dv)` (or the finalizer) releases them.  `Kmer{A,K,N}` and `Tuple{Kmer,Kmer}` / `Tuple{Kmer,Int}` are
isbits, so a `DeviceVector{eltype(it)}` holds exactly what `collect(it)` would.
"""
mutable struct DeviceVector{T}
    ctx::Context
    ptr::Ptr{T}
    len::Int
    function DeviceVector{T}(ctx::Context, n::Integer) where {T}
        isbitstype(T) || throw(ArgumentError("DeviceVector needs an isbits element type"))
        p = Ref{Ptr{Cvoid}}(C_NULL)
        check(ctx, ccall((:kmc_malloc, LIB[]), Int32, (Ptr{Cvoid}, UInt64, Ptr{Ptr{Cvoid}}), ctx.handle, max(1, n * sizeof(T)), p))
        dv = new{T}(ctx, Ptr{T}(p[]), Int(n))
        finalizer(free!, dv)
        return dv
    end
end
Base.length(dv::DeviceVector) = dv.len
Base.eltype(::Type{DeviceVector{T}}) where {T} = T
Base.pointer(dv::DeviceVector) = dv.ptr
function free!(dv::DeviceVector)
    if dv.ptr != C_NULL
        ccall((:kmc_free, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), dv.ctx.handle, dv.ptr)
        dv.ptr = C_NULL
        dv.len = 0
    end
    return nothing
end
function Base.Array(dv::DeviceVector{T}) where {T}
    out = Vector{T}(undef, dv.len)
    GC.@preserve out check(dv.ctx, ccall((:kmc_download, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, UInt64),
        dv.ctx.handle, pointer(out), dv.ptr, dv.len * sizeof(T)))
    return out
end
"Shrink the logical length (the memory stays): used when fewer elements were written than allocated."
truncate!(dv::DeviceVector, n::Integer) = (dv.len = Int(n); dv)

function upload(ctx::Context, v::AbstractVector{T}) where {T}
    dv = DeviceVector{T}(ctx, length(v))
    GC.@preserve v begin
        check(ctx, ccall((:kmc_upload, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, UInt64), ctx.handle, dv.ptr, pointer(v), sizeof(T) * length(v)))
        check(ctx, ccall((:kmc_sync, LIB[]), Int32, (Ptr{Cvoid},), ctx.handle))
    end
    return dv
end
zero!(dv::DeviceVector{T}, byte::Integer = 0) where {T} =
    check(dv.ctx, ccall((:kmc_memset, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int32, UInt64), dv.ctx.handle, dv.ptr, byte, dv.len * sizeof(T)))

# Pin a host vector for the duration of `f` (kmc_host_register): a pageable destination makes every chunk of a large
# `collect` go through a staging copy inside the driver.  Registration costs about a millisecond per GB, so small
# vectors are left alone.
const PIN_THRESHOLD = 64 << 20
function with_pinned(f, ctx::Context, v::Vector)
    bytes = sizeof(v)
    if bytes < PIN_THRESHOLD
        return f()
    end
    GC.@preserve v begin
        st = ccall((:kmc_host_register, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, UInt64), ctx.handle, pointer(v), bytes)
        try
            return f()
        finally
            st == KMC_OK && ccall((:kmc_host_unregister, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), ctx.handle, pointer(v))
        end
    end
end

# ---------------------------------------------------------------------------------------------
# type parameters -> runtime integers; sources -> (pointer, words, length, bits, first symbol)
# ---------------------------------------------------------------------------------------------
const NucSeq{B} = Union{LongSequence{<:NucleicAcidAlphabet{B}}, LongSubSeq{<:NucleicAcidAlphabet{B}}}
src_bits(::Type{<:NucSeq{2}}) = UInt32(2)
src_bits(::Type{<:NucSeq{4}}) = UInt32(4)

mode_of(::FwKmers) = KMC_FW
mode_of(::FwRvIterator) = KMC_FWRV
mode_of(::CanonicalKmers) = KMC_CANON
mode_of(::UnambiguousKmers) = KMC_UNAMBIG

source(it::Union{FwKmers, FwRvIterator}) = it.seq
source(it::CanonicalKmers) = it.it.seq
source(it::UnambiguousKmers) = it.it.seq

# FwRvIterator and UnambiguousKmers are not AbstractKmerIterators in the reference
# (CanonicalKmers.jl:25, UnambiguousKmers.jl:29), so the parameters are read per type.
const AnyIter{A, K} = Union{FwKmers{A, K}, FwRvIterator{A, K}, CanonicalKmers{A, K}, UnambiguousKmers{A, K}}
ksize_of(::AnyIter{A, K}) where {A, K} = K
ksize_of(::Type{<:AnyIter{A, K}}) where {A, K} = K
alphabet_of(::Type{<:AnyIter{A, K}}) where {A, K} = A
mode_of(::Type{<:FwKmers}) = KMC_FW
mode_of(::Type{<:FwRvIterator}) = KMC_FWRV
mode_of(::Type{<:CanonicalKmers}) = KMC_CANON
mode_of(::Type{<:UnambiguousKmers}) = KMC_UNAMBIG

"""
What the library needs to know about one nucleotide sequence: the `Vector{UInt64}` that must stay alive, the first
word, the number of addressable words from there, the length in symbols and the offset of the first symbol inside
the first word.  A `LongSubSeq` (`view(seq, a:b)`, tested by the reference at test/runtests.jl:154-169) shares its
parent's `data`; the view starts `first(part) - 1` symbols in, which is a word offset plus `first_symbol_offset`.
"""
function seq_words(seq::LongSequence)
    return seq.data, pointer(seq.data), length(seq.data), length(seq), UInt32(0)
end
function seq_words(seq::LongSubSeq)
    spw = 64 ÷ Int(src_bits(typeof(seq)))
    skip = first(seq.part) - 1
    w0 = skip ÷ spw
    return seq.data, pointer(seq.data, w0 + 1), length(seq.data) - w0, length(seq), UInt32(skip % spw)
end

function throw_status(ctx::Context, st::Int32, res::KmcResult, ::Type{A}) where {A}
    if st == KMC_E_AMBIGUOUS
        # what src/construction.jl:108-110 throws: EncodeError(Alphabet, symbol)
        sym = A <: RNAAlphabet ? reinterpret(RNA, UInt8(res.err_sym)) : reinterpret(DNA, UInt8(res.err_sym))
        throw(BioSequences.EncodeError(A(), sym))
    elseif st == KMC_E_BAD_K
        error("K must be at least 1")            # src/iterators/FwKmers.jl:32-33
    else
        check(ctx, st)
    end
end

extract_host!(ctx, s, K, mode, flags, o, res) = ccall((:kmc_extract_host, LIB[]), Int32,
    (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, UInt32, Ptr{KmcOut}, Ref{KmcResult}), ctx.handle, s, K, mode, flags, o, res)

# ---------------------------------------------------------------------------------------------
# collect(it): one kmc_extract_host call straight into the memory of the result Vector
# ---------------------------------------------------------------------------------------------
"""
    KmersCUDA.collect(it) -> Vector{eltype}

Same result as `Base.collect(it)` for `FwKmers`, `FwRvIterator`, `CanonicalKmers` and
`UnambiguousKmers` whose source is a `LongSequence` / `LongSubSeq` over a 2- or 4-bit nucleotide alphabet or an
ASCII source.  The k-mer alphabet may be 2-bit (Copyable / FourToTwo / AsciiEncode) or, for the first three
iterators over a `LongSequence`, 4-bit (Copyable 4 -> 4 and TwoToFour: `KMC_KMER4`, K <= 64).  `Kmer{A,K,N}` and
tuples of `Kmer`/`Int` are isbits, so the device writes the Julia element layout directly into the vector (KMC_AOS).
"""
function collect(it::Union{FwKmers{A, K}, FwRvIterator{A, K}, CanonicalKmers{A, K}};
        ctx::Context = default_context()) where {A <: NucleicAcidAlphabet{4}, K}
    seq = source(it)
    seq isa NucSeq || throw(ArgumentError("4-bit k-mers are accelerated for LongSequence / LongSubSeq sources"))
    K <= 64 || throw(ArgumentError("KmersCUDA handles K <= 64 for k-mers over a 4-bit alphabet"))
    T = derive_type(Kmer{A, K})
    mode = mode_of(it)
    data, wptr, nwords, len, first = seq_words(seq)
    nwin = max(0, len - K + 1)
    ET = mode == KMC_FWRV ? Tuple{T, T} : T
    out = Vector{ET}(undef, nwin)
    res = KmcResult()
    GC.@preserve data out with_pinned(ctx, out) do
        s = Ref(KmcSeqs(wptr, nwords, 1, C_NULL, C_NULL, len, nwords, src_bits(typeof(seq)), first))
        o = Ref(KmcOut(Ptr{UInt64}(pointer(out)), C_NULL, C_NULL, C_NULL, C_NULL, nwin, 0))
        st = extract_host!(ctx, s, K, mode, KMC_AOS | KMC_KMER4, o, res)
        st == KMC_OK || throw_status(ctx, st, res, A)
    end
    return out
end

function collect(it::Union{FwKmers{A, K}, FwRvIterator{A, K}, CanonicalKmers{A, K}, UnambiguousKmers{A, K}};
        ctx::Context = default_context()) where {A <: NucleicAcidAlphabet{2}, K}
    seq = source(it)
    seq isa NucSeq || return collect_ascii(it, ascii_source(seq); ctx)
    T = derive_type(Kmer{A, K})
    mode = mode_of(it)
    data, wptr, nwords, len, first = seq_words(seq)
    bits = src_bits(typeof(seq))
    ET = mode == KMC_FWRV ? Tuple{T, T} : mode == KMC_UNAMBIG ? Tuple{T, Int} : T
    cap = max(0, len - K + 1)
    if mode == KMC_UNAMBIG && bits == UInt32(4)
        cap = count(it; ctx)   # Base.IteratorSize is SizeUnknown (UnambiguousKmers.jl:33-37)
    end
    out = Vector{ET}(undef, cap)
    res = KmcResult()
    GC.@preserve data out with_pinned(ctx, out) do
        s = Ref(KmcSeqs(wptr, nwords, 1, C_NULL, C_NULL, len, nwords, bits, first))
        o = Ref(KmcOut(Ptr{UInt64}(pointer(out)), C_NULL, C_NULL, C_NULL, C_NULL, cap, 0))
        st = extract_host!(ctx, s, K, mode, KMC_AOS, o, res)
        st == KMC_OK || throw_status(ctx, st, res, A)
    end
    resize!(out, res.n_written)
    return out
end

# ASCII sources (the AsciiEncode scheme, src/construction.jl:95-96): String, SubString{String}, codeunits, byte
# vectors -- and StringView (what FASTX hands over; the reference enables it in ext/StringViewsExt.jl:9 and tests it
# at test/runtests.jl:892-899) -- go to the device as they are (src_bits = 8); nothing is packed on the host.
# Anything whose code units are a dense byte array is passed by pointer; other AbstractStrings / byte vectors are
# copied into a Vector{UInt8} first.  (StringViews.jl is not a dependency: a StringView is an AbstractString whose
# `codeunits` is the wrapped array, which is all that is used here.)
const DenseBytes = Union{Vector{UInt8}, Base.CodeUnits{UInt8, String}, Base.CodeUnits{UInt8, SubString{String}},
    SubArray{UInt8, 1, Vector{UInt8}, <:Tuple{UnitRange}, true}}
ascii_source(s::Union{String, SubString{String}}) = codeunits(s)
ascii_source(s::AbstractString) = (cu = codeunits(s); cu isa DenseBytes ? cu : Vector{UInt8}(cu))
ascii_source(v::DenseBytes) = v
ascii_source(v::AbstractVector{UInt8}) = Vector{UInt8}(v)
ascii_source(x) = throw(ArgumentError("KmersCUDA accelerates LongSequence / LongSubSeq and ASCII sources, not $(typeof(x))"))

function collect_ascii(it::AnyIter{A, K}, bytes::DenseBytes; ctx::Context = default_context()) where {A <: NucleicAcidAlphabet{2}, K}
    T = derive_type(Kmer{A, K})
    mode = mode_of(it)
    len = length(bytes)
    ET = mode == KMC_FWRV ? Tuple{T, T} : mode == KMC_UNAMBIG ? Tuple{T, Int} : T
    out = Vector{ET}(undef, max(0, len - K + 1))     # upper bound; UnambiguousKmers may return fewer
    res = KmcResult()
    flags = KMC_AOS | (A <: RNAAlphabet ? KMC_RNA : UInt32(0))
    GC.@preserve bytes out with_pinned(ctx, out) do
        s = Ref(KmcSeqs(Ptr{UInt64}(pointer(bytes)), len, 1, C_NULL, C_NULL, len, max(len, 1), UInt32(8), 0))
        o = Ref(KmcOut(Ptr{UInt64}(pointer(out)), C_NULL, C_NULL, C_NULL, C_NULL, length(out), 0))
        st = extract_host!(ctx, s, K, mode, flags, o, res)
        if st == KMC_E_AMBIGUOUS   # FwKmers.jl:124-126 / UnambiguousKmers.jl:123-124
            throw(BioSequences.EncodeError(A(), repr(UInt8(res.err_sym))))
        end
        st == KMC_OK || throw_status(ctx, st, res, A)
    end
    resize!(out, res.n_written)
    return out
end

"""
    KmersCUDA.collect(it::SpacedKmers{A,K,J}) -> Vector{Kmer{A,K,N}}

`collect(SpacedKmers{A,K,J}(seq))` / `collect(each_codon(seq))` (src/iterators/SpacedKmers.jl:22-139): the k-mers at the
starts 1, 1+J, 1+2J, ... through `kmc_extract_spaced`, for 2-bit and 4-bit k-mer alphabets over `LongSequence`,
`LongSubSeq` and ASCII sources.  A symbol that cannot be encoded inside a sampled window throws the reference's
`EncodeError`; symbols between the windows of a step J > K are never read (test/runtests.jl:866-867).
"""
function collect(it::SpacedKmers{A, K, J}; ctx::Context = default_context()) where {A <: NucleicAcidAlphabet, K, J}
    T = derive_type(Kmer{A, K})
    seq = it.seq
    flags = (A <: NucleicAcidAlphabet{4} ? KMC_KMER4 : UInt32(0)) | (A <: RNAAlphabet ? KMC_RNA : UInt32(0))
    res = KmcResult()
    if seq isa NucSeq
        data, wptr, nwords, len, first = seq_words(seq)
        bits = src_bits(typeof(seq))
        keep, host, unit_count = data, unsafe_wrap(Array, wptr, nwords), nwords
    else
        bytes = ascii_source(seq)
        len, first, bits = length(bytes), UInt32(0), UInt32(8)
        keep, host, unit_count = bytes, bytes, length(bytes)
    end
    n = len < K ? 0 : (len - K) ÷ J + 1                      # SpacedKmers.jl:36-40
    out = DeviceVector{T}(ctx, n)
    GC.@preserve keep begin
        dsrc = upload(ctx, host isa Vector ? host : Vector{UInt8}(host))
        try
            s = Ref(KmcSeqs(Ptr{UInt64}(dsrc.ptr), unit_count, 1, C_NULL, C_NULL, len, max(unit_count, 1), bits, first))
            o = Ref(KmcOut(Ptr{UInt64}(out.ptr), C_NULL, C_NULL, C_NULL, C_NULL, n, 0))
            st = ccall((:kmc_extract_spaced, LIB[]), Int32,
                (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, UInt32, Ptr{KmcOut}, Ref{KmcResult}), ctx.handle, s, K, J, flags, o, res)
            if st == KMC_E_AMBIGUOUS && bits == UInt32(8)
                throw(BioSequences.EncodeError(A(), repr(UInt8(res.err_sym))))
            end
            st == KMC_OK || throw_status(ctx, st, res, A)
        finally
            free!(dsrc)
        end
    end
    v = Array(truncate!(out, res.n_written))
    free!(out)
    return v
end

"Number of elements `collect(it)` returns (runs the device count pass for 4-bit UnambiguousKmers)."
function count(it; ctx::Context = default_context())
    seq = source(it)
    data, wptr, nwords, len, first = seq_words(seq)
    n = Ref{UInt64}(0)
    GC.@preserve data begin
        dw = upload(ctx, unsafe_wrap(Array, wptr, nwords))
        try
            s = Ref(KmcSeqs(dw.ptr, nwords, 1, C_NULL, C_NULL, len, nwords, src_bits(typeof(seq)), first))
            check(ctx, ccall((:kmc_count, LIB[]), Int32, (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, Ptr{UInt64}),
                ctx.handle, s, ksize_of(it), mode_of(it), n))
        finally
            free!(dw)
        end
    end
    return Int(n[])
end

# ---------------------------------------------------------------------------------------------
# batched extraction over a read set: what `[collect(Iter(r)) for r in reads]` concatenates to
# ---------------------------------------------------------------------------------------------
"One word-aligned CSR buffer for a vector of reads (multithreaded gather on the host)."
struct PackedReads
    words::Vector{UInt64}
    woff::Vector{UInt64}   # first word of every read (n + 1 entries)
    lens::Vector{UInt64}
    bits::UInt32
end
function pack_reads(reads::AbstractVector{S}) where {S <: LongSequence}
    n = length(reads)
    lens = UInt64[length(r) for r in reads]
    nw = UInt64[length(r.data) for r in reads]
    woff = cumsum(vcat(UInt64(0), nw))
    words = Vector{UInt64}(undef, woff[end] + 1)
    words[end] = 0
    Threads.@threads for i in 1:n
        copyto!(words, woff[i] + 1, reads[i].data, 1, nw[i])
    end
    return PackedReads(words, woff, lens, src_bits(S))
end
windows(p::PackedReads, K::Integer) = sum(l -> l >= K ? Int(l) - K + 1 : 0, p.lens; init = 0)

"""
    extract(Iter, reads::Vector{<:LongSequence}; hash = false, device = false, group = nothing)

`Iter` is e.g. `CanonicalDNAMers{31}`.  Packs the reads into one word-aligned CSR buffer and makes ONE library call.

  * default: `(elements::Vector{eltype(Iter)}, hashes::Vector{UInt64}, offsets::Vector{UInt64})` in host memory;
    `offsets[i]+1 : offsets[i+1]` are the elements of read `i`;
  * `device = true`: `(elements::DeviceVector, hashes::DeviceVector)` -- the streams stay in HBM (KMC_OUT_DEVICE), only
    the reads cross PCIe; this is the path that runs at the speed of the GPU;
  * `group = Group(...)`: the reads are sharded over the group's GPUs by sequence (contiguous ranges, balanced by
    symbols) and extracted side by side; returns one `(elements, hashes, offsets)` per device, whose concatenation in
    device order is the single-GPU result.
"""
function extract(::Type{I}, reads::AbstractVector{S}; hash::Bool = false, device::Bool = false, group = nothing,
        ctx::Context = default_context()) where {I <: AnyIter, S <: LongSequence}
    group === nothing || return extract_group(I, reads, group; hash)
    A, K, mode = alphabet_of(I), ksize_of(I), mode_of(I)
    T = derive_type(Kmer{A, K})
    ET = mode == KMC_FWRV ? Tuple{T, T} : mode == KMC_UNAMBIG ? Tuple{T, Int} : T
    pk = pack_reads(reads)
    n = length(reads)
    cap = windows(pk, K)
    flags = KMC_AOS | (hash ? KMC_HASH_FX : UInt32(0))
    res = KmcResult()
    if device
        out = DeviceVector{ET}(ctx, cap)
        hashes = DeviceVector{UInt64}(ctx, hash ? cap : 0)
        GC.@preserve pk begin
            s = Ref(KmcSeqs(pointer(pk.words), length(pk.words), n, pointer(pk.woff), pointer(pk.lens), 0, 0, pk.bits, 0))
            o = Ref(KmcOut(Ptr{UInt64}(out.ptr), C_NULL, hash ? hashes.ptr : C_NULL, C_NULL, C_NULL, cap, 0))
            st = with_pinned(ctx, pk.words) do
                extract_host!(ctx, s, K, mode, flags | KMC_OUT_DEVICE, o, res)
            end
            st == KMC_OK || throw_status(ctx, st, res, A)
        end
        truncate!(out, res.n_written)
        hash && truncate!(hashes, res.n_written)
        return out, hashes
    end
    out = Vector{ET}(undef, cap)
    hashes = hash ? Vector{UInt64}(undef, cap) : UInt64[]
    offsets = Vector{UInt64}(undef, n + 1)
    GC.@preserve pk out hashes offsets with_pinned(ctx, out) do
        s = Ref(KmcSeqs(pointer(pk.words), length(pk.words), n, pointer(pk.woff), pointer(pk.lens), 0, 0, pk.bits, 0))
        o = Ref(KmcOut(Ptr{UInt64}(pointer(out)), C_NULL, hash ? pointer(hashes) : C_NULL, C_NULL, pointer(offsets), cap, 0))
        st = extract_host!(ctx, s, K, mode, flags, o, res)
        st == KMC_OK || throw_status(ctx, st, res, A)
    end
    resize!(out, res.n_written)
    hash && resize!(hashes, res.n_written)
    return out, hashes, offsets
end

# ---------------------------------------------------------------------------------------------
# several GPUs from one Julia process (kmc_group: a context per device + one NCCL communicator)
# ---------------------------------------------------------------------------------------------
"""
    Group(devices = 0:n-1)

One process driving several GPUs.  Reads shard by sequence and no stream ever crosses GPUs; the only collective is
the sum of the per-GPU count tables (`bucket_count(...; group)`), done by NCCL inside the library.
"""
mutable struct Group
    handle::Ptr{Cvoid}
    ctx::Vector{Context}
    function Group(devices = nothing)
        if devices === nothing
            n = Ref{Int32}(0)
            ccall((:kmc_device_count, LIB[]), Int32, (Ptr{Int32},), n)
            devices = 0:(n[] - 1)
        end
        devs = Int32[d for d in devices]
        h = Ref{Ptr{Cvoid}}(C_NULL)
        st = ccall((:kmc_group_create, LIB[]), Int32, (Int32, Ptr{Int32}, Ptr{Ptr{Cvoid}}), length(devs), devs, h)
        st == KMC_OK || error("KmersCUDA: kmc_group_create failed ($(status_string(st)))")
        ctxs = Context[]
        for i in 0:(length(devs) - 1)
            c = Ref{Ptr{Cvoid}}(C_NULL)
            ccall((:kmc_group_ctx, LIB[]), Int32, (Ptr{Cvoid}, Int32, Ptr{Ptr{Cvoid}}), h[], i, c)
            push!(ctxs, Context(c[], false))
        end
        g = new(h[], ctxs)
        finalizer(x -> ccall((:kmc_group_destroy, LIB[]), Int32, (Ptr{Cvoid},), x.handle), g)
        return g
    end
end
Base.length(g::Group) = length(g.ctx)

"Contiguous read ranges, balanced by symbols; reads are never split (the planner of kmerscuda/sharding.py)."
function shard_ranges(lens::Vector{<:Integer}, parts::Integer)
    total = sum(lens; init = 0)
    bounds = Int[0]
    acc, g = 0, 1
    for (i, l) in enumerate(lens)
        while g < parts && acc >= total * g / parts
            push!(bounds, i - 1)
            g += 1
        end
        acc += l
    end
    while length(bounds) < parts
        push!(bounds, length(lens))
    end
    push!(bounds, length(lens))
    return [(bounds[i] + 1):bounds[i + 1] for i in 1:parts]
end

function extract_group(::Type{I}, reads::AbstractVector{S}, g::Group; hash::Bool = false) where {I <: AnyIter, S <: LongSequence}
    A, K, mode = alphabet_of(I), ksize_of(I), mode_of(I)
    T = derive_type(Kmer{A, K})
    ET = mode == KMC_FWRV ? Tuple{T, T} : mode == KMC_UNAMBIG ? Tuple{T, Int} : T
    nd = length(g)
    ranges = shard_ranges([length(r) for r in reads], nd)
    packs = [pack_reads(view(reads, r)) for r in ranges]
    caps = [windows(pk, K) for pk in packs]
    outs = [Vector{ET}(undef, c) for c in caps]
    hashes = [hash ? Vector{UInt64}(undef, c) : UInt64[] for c in caps]
    offs = [Vector{UInt64}(undef, length(r) + 1) for r in ranges]
    seqs = [KmcSeqs(pointer(pk.words), length(pk.words), length(pk.lens), pointer(pk.woff), pointer(pk.lens), 0, 0, pk.bits, 0) for pk in packs]
    kouts = [KmcOut(Ptr{UInt64}(pointer(outs[i])), C_NULL, hash ? pointer(hashes[i]) : C_NULL, C_NULL, pointer(offs[i]), caps[i], 0) for i in 1:nd]
    results = [KmcResult() for _ in 1:nd]
    # kmc_result is a plain C struct: an array of them is one block of nd * sizeof(KmcResult) bytes
    rbuf = zeros(UInt8, nd * sizeof(KmcResult))
    GC.@preserve packs outs hashes offs seqs kouts rbuf begin
        st = ccall((:kmc_group_extract_host, LIB[]), Int32,
            (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, UInt32, Ptr{KmcOut}, Ptr{UInt8}),
            g.handle, seqs, K, mode, KMC_AOS | (hash ? KMC_HASH_FX : UInt32(0)), kouts, rbuf)
        for i in 1:nd
            unsafe_copyto!(Ptr{UInt8}(pointer_from_objref(results[i])), pointer(rbuf, (i - 1) * sizeof(KmcResult) + 1), sizeof(KmcResult))
        end
        if st != KMC_OK
            bad = findfirst(r -> r.err_pos != 0, results)
            throw_status(g.ctx[something(bad, 1)], st, results[something(bad, 1)], A)
        end
    end
    for i in 1:nd
        resize!(outs[i], results[i].n_written)
        hash && resize!(hashes[i], results[i].n_written)
    end
    return [(outs[i], hashes[i], offs[i]) for i in 1:nd]
end

# ---------------------------------------------------------------------------------------------
# fx_hash.(v) on the device (src/kmer.jl:255-261)
# ---------------------------------------------------------------------------------------------
function fx_hash_device(v::Vector{Kmer{A, K, N}}, h::UInt64 = UInt64(0); ctx::Context = default_context()) where {A, K, N}
    isempty(v) && return UInt64[]
    dk = upload(ctx, v)
    out = fx_hash_device(dk, h)
    free!(dk)
    r = Array(out)
    free!(out)
    return r
end
"`fx_hash.(v, h)` of a device-resident k-mer stream; the hashes stay on the device."
function fx_hash_device(dk::DeviceVector{Kmer{A, K, N}}, h::UInt64 = UInt64(0)) where {A, K, N}
    ctx = dk.ctx
    out = DeviceVector{UInt64}(ctx, length(dk))
    check(ctx, ccall((:kmc_fx_hash, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, UInt64, Int32, UInt64, Ptr{Cvoid}),
        ctx.handle, dk.ptr, length(dk), N, h, out.ptr))
    return out
end

# Base.hash(kmer, h) = hash(kmer.data, h ⊻ K) (src/kmer.jl:206) depends on the Julia version's tuple
# and integer hashing.  libkmerscuda implements the Julia 1.10 / 1.11 definition (kmc_base_hash); it
# reproduces the reference's documented hash(mer"UGCUGUAC"r) == 0xe5057d38c8907b22
# (docs/src/hashing.md:18-20).  Whether THIS Julia agrees is checked once, on the host, before the
# device path is trusted; otherwise Base.hash is evaluated on the returned k-mers by Julia itself.
const BASE_HASH_ON_DEVICE = Ref{Union{Nothing, Bool}}(nothing)
function base_hash_matches()
    if BASE_HASH_ON_DEVICE[] === nothing
        p1, p2 = [mer"UGCUGUAC"r], [mer"TAGCTAGGACATTTTAAACCCGGGTAGCTAGGACATTTTAAACC"d]   # one limb, two limbs
        BASE_HASH_ON_DEVICE[] = _hash_device(p1, UInt(0)) == hash.(p1) && _hash_device(p2, UInt(7)) == hash.(p2, UInt(7))
    end
    return BASE_HASH_ON_DEVICE[]::Bool
end

function _hash_device(v::Vector{Kmer{A, K, N}}, h::UInt; ctx::Context = default_context()) where {A, K, N}
    isempty(v) && return UInt64[]
    dk = upload(ctx, v)
    out = DeviceVector{UInt64}(ctx, length(v))
    check(ctx, ccall((:kmc_base_hash, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, UInt64, Int32, Int32, UInt64, Ptr{Cvoid}),
        ctx.handle, dk.ptr, length(v), N, K, h, out.ptr))
    r = Array(out)
    free!(dk)
    free!(out)
    return r
end

"`hash.(v, h)` (Base.hash of k-mers): on the device when this Julia's hashing matches, else on the host."
hash_device(v::Vector{<:Kmer}, h::UInt = UInt(0); ctx::Context = default_context()) =
    base_hash_matches() ? _hash_device(v, h; ctx) : hash.(v, h)

# ---------------------------------------------------------------------------------------------
# consumers of the stream that never materialise it (device-resident sequence, small results)
# ---------------------------------------------------------------------------------------------
function with_device_sequence(f, ctx::Context, seq::NucSeq)
    data, wptr, nwords, len, first = seq_words(seq)
    GC.@preserve data begin
        dw = upload(ctx, unsafe_wrap(Array, wptr, nwords))
        try
            s = Ref(KmcSeqs(dw.ptr, nwords, 1, C_NULL, C_NULL, len, nwords, src_bits(typeof(seq)), first))
            return f(s)
        finally
            free!(dw)
        end
    end
end

"""
    minhash_sketch(CanonicalKmers{A,K}(seq) | FwKmers{A,K}(seq), s) -> Vector{UInt64}

Bottom-`s` MinHash sketch under `fx_hash` -- `sketch(fx_hash, CanonicalDNAMers{K}(seq), s)` of
docs/src/minhash.md:31-36 -- the `s` smallest distinct hash values, ascending (`kmc_minhash_sketch`).
"""
function minhash_sketch(it::Union{FwKmers{A, K}, CanonicalKmers{A, K}}, s::Integer;
        ctx::Context = default_context()) where {A <: NucleicAcidAlphabet{2}, K}
    res = KmcResult()
    dout = DeviceVector{UInt64}(ctx, s)
    with_device_sequence(ctx, source(it)) do d
        st = ccall((:kmc_minhash_sketch, LIB[]), Int32,
            (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, UInt64, Ptr{Cvoid}, Ref{KmcResult}),
            ctx.handle, d, K, mode_of(typeof(it)), s, dout.ptr, res)
        st == KMC_OK || throw_status(ctx, st, res, A)
    end
    out = Array(truncate!(dout, res.n_written))
    free!(dout)
    return out
end

"""
    minhash_sketches(seqs::AbstractVector{<:LongSequence}, K, s; canonical = true) -> Vector{Vector{UInt64}}

The bottom-`s` sketch of every sequence on its own, in one call (`kmc_minhash_sketch_each`): element `i` is what
`minhash_sketch(CanonicalKmers{A,K}(seqs[i]), s)` returns (`FwKmers` with `canonical = false`).
"""
function minhash_sketches(seqs::AbstractVector{S}, K::Integer, s::Integer; canonical::Bool = true,
        ctx::Context = default_context()) where {S <: LongSequence{<:NucleicAcidAlphabet{2}}}
    n = length(seqs)
    n == 0 && return Vector{UInt64}[]
    pk = pack_reads(seqs)
    dw, doff, dlen = upload(ctx, pk.words), upload(ctx, pk.woff), upload(ctx, pk.lens)
    drows = DeviceVector{UInt64}(ctx, n * s)
    dn = DeviceVector{UInt32}(ctx, n)
    res = KmcResult()
    d = Ref(KmcSeqs(dw.ptr, length(pk.words), n, doff.ptr, dlen.ptr, 0, 0, UInt32(2), 0))
    st = ccall((:kmc_minhash_sketch_each, LIB[]), Int32,
        (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, UInt64, Ptr{Cvoid}, Ptr{Cvoid}, Ref{KmcResult}),
        ctx.handle, d, K, canonical ? KMC_CANON : KMC_FW, s, drows.ptr, dn.ptr, res)
    st == KMC_OK || throw_status(ctx, st, res, eltype(S))
    rows, lens = reshape(Array(drows), Int(s), n), Array(dn)
    foreach(free!, (dw, doff, dlen, drows, dn))
    return [rows[1:lens[i], i] for i in 1:n]
end

"""
    minhash_compare(a::Vector{Vector{UInt64}}, b = a, s) -> (shared::Matrix{UInt32}, shared_bottom::Matrix{UInt32})

Every sketch of `a` against every sketch of `b` (`kmc_minhash_compare`): `shared[i, j] = |a[i] ∩ b[j]|` and
`shared_bottom[i, j]` = how many of those are among the `s` smallest values of `a[i] ∪ b[j]`.  The Mash Jaccard
estimate is `shared_bottom / min(s, length(a[i]) + length(b[j]) - shared)`; sketches are ascending and distinct, as
`minhash_sketches` returns them, and are read up to `s` values.
"""
function minhash_compare(a::AbstractVector{<:AbstractVector{UInt64}}, b::AbstractVector{<:AbstractVector{UInt64}}, s::Integer;
        ctx::Context = default_context())
    na, nb = length(a), length(b)
    (na == 0 || nb == 0) && return (zeros(UInt32, na, nb), zeros(UInt32, na, nb))
    pack(v) = (m = fill(typemax(UInt64), Int(s), length(v));
               for (i, x) in enumerate(v); k = min(length(x), s); m[1:k, i] .= x[1:k]; end;
               (vec(m), UInt32[min(length(x), s) for x in v]))
    ra, la = pack(a)
    rb, lb = pack(b)
    da, dla, db, dlb = upload(ctx, ra), upload(ctx, la), upload(ctx, rb), upload(ctx, lb)
    dsh, dbt = DeviceVector{UInt32}(ctx, na * nb), DeviceVector{UInt32}(ctx, na * nb)
    check(ctx, ccall((:kmc_minhash_compare, LIB[]), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, UInt64, Ptr{Cvoid}, Ptr{Cvoid}, UInt64, UInt64, Ptr{Cvoid}, Ptr{Cvoid}),
        ctx.handle, da.ptr, dla.ptr, na, db.ptr, dlb.ptr, nb, s, dsh.ptr, dbt.ptr))
    # the library writes pair (i, j) at i * nb + j: row-major, so the column-major result is transposed
    shared = permutedims(reshape(Array(dsh), nb, na))
    bottom = permutedims(reshape(Array(dbt), nb, na))
    foreach(free!, (da, dla, db, dlb, dsh, dbt))
    return shared, bottom
end
minhash_compare(a::AbstractVector{<:AbstractVector{UInt64}}, s::Integer; kw...) = minhash_compare(a, a, s; kw...)

"""
    composition(FwKmers{A,K}(seq) | CanonicalKmers{A,K}(seq)) -> Vector{UInt32}  (length 4^K, K <= 14)

`counts[as_integer(kmer) + 1] += 1` for every k-mer (docs/src/composition.md:28-39), `kmc_composition`.
"""
function composition(it::Union{FwKmers{A, K}, CanonicalKmers{A, K}};
        ctx::Context = default_context()) where {A <: NucleicAcidAlphabet{2}, K}
    res = KmcResult()
    dt = DeviceVector{UInt32}(ctx, 4^K)
    zero!(dt)
    with_device_sequence(ctx, source(it)) do d
        st = ccall((:kmc_composition, LIB[]), Int32,
            (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, Ptr{Cvoid}, Ref{KmcResult}),
            ctx.handle, d, K, mode_of(typeof(it)), dt.ptr, res)
        st == KMC_OK || throw_status(ctx, st, res, A)
    end
    counts = Array(dt)
    free!(dt)
    return counts
end

"""
    minimizers(FwKmers{A,K}(seq) | CanonicalKmers{A,K}(seq), W; step = 1) -> (Vector{Kmer}, Vector{Int})

For every window start 1, 1+step, ...: the k-mer with the smallest `fx_hash` among `W` consecutive
k-mers and its 1-based start (docs/src/replacements.md:28-58), `kmc_minimizers`; K <= 32, K + W - 1 <= 64.
"""
function minimizers(it::Union{FwKmers{A, K}, CanonicalKmers{A, K}}, W::Integer; step::Integer = 1,
        ctx::Context = default_context()) where {A <: NucleicAcidAlphabet{2}, K}
    seq = source(it)
    T = derive_type(Kmer{A, K})
    span = K + W - 1
    n = length(seq) >= span ? (length(seq) - span) ÷ step + 1 : 0
    res = KmcResult()
    dk, di = DeviceVector{T}(ctx, n), DeviceVector{Int}(ctx, n)
    with_device_sequence(ctx, seq) do d
        o = Ref(KmcOut(Ptr{UInt64}(dk.ptr), C_NULL, C_NULL, Ptr{Int64}(di.ptr), C_NULL, n, 0))
        st = ccall((:kmc_minimizers, LIB[]), Int32,
            (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, Int32, Int32, UInt32, Ptr{KmcOut}, Ref{KmcResult}),
            ctx.handle, d, K, W, step, mode_of(typeof(it)), UInt32(0), o, res)
        st == KMC_OK || throw_status(ctx, st, res, A)
    end
    kmers, starts = Array(dk), Array(di)
    free!(dk)
    free!(di)
    return kmers, starts
end

"""
    count_kmers(FwKmers{A,K}(seq) | CanonicalKmers{A,K}(seq); log2_capacity) -> Dict{Kmer{A,K,N}, Int}

Exact k-mer counts -- the `Dict` a loop over the iterator would build -- through `kmc_kmer_count` (open addressing
in device memory keyed by the k-mer, K <= 31, or K = 32 for canonical k-mers) and `kmc_kmer_table_export`; two-limb
k-mers (K = 33..63, or K = 64 for canonical k-mers) through `kmc_kmer_count2` and `kmc_kmer_table2_export`.
`log2_capacity` defaults to twice the number of windows, rounded up to a power of two.
"""
function count_kmers(it::Union{FwKmers{A, K}, CanonicalKmers{A, K}};
        log2_capacity::Integer = max(10, ceil(Int, log2(2 * max(1, length(source(it)))))),
        ctx::Context = default_context()) where {A <: NucleicAcidAlphabet{2}, K}
    K <= 64 || throw(ArgumentError("count_kmers handles k-mers of one or two limbs (K <= 64)"))
    T = derive_type(Kmer{A, K})
    N = K <= 32 ? 1 : 2                         # UInt64 limbs per key
    slots = 1 << log2_capacity
    res = KmcResult()
    dk, dv = DeviceVector{UInt64}(ctx, N * slots), DeviceVector{UInt32}(ctx, slots)
    zero!(dk, 0xff)   # free slot = ~0 in every limb
    zero!(dv)
    with_device_sequence(ctx, source(it)) do d
        st = N == 1 ?
            ccall((:kmc_kmer_count, LIB[]), Int32,
                (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, Ptr{Cvoid}, Ptr{Cvoid}, UInt32, Ref{KmcResult}),
                ctx.handle, d, K, mode_of(typeof(it)), dk.ptr, dv.ptr, UInt32(log2_capacity), res) :
            ccall((:kmc_kmer_count2, LIB[]), Int32,
                (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, Ptr{Cvoid}, Ptr{Cvoid}, UInt32, Ref{KmcResult}),
                ctx.handle, d, K, mode_of(typeof(it)), dk.ptr, dv.ptr, UInt32(log2_capacity), res)
        st == KMC_OK || throw_status(ctx, st, res, A)
    end
    n = Int(res.digest[1])                      # keys this call added = every key of a fresh table
    ok, ov, nout = DeviceVector{UInt64}(ctx, N * n), DeviceVector{UInt32}(ctx, n), Ref{UInt64}(0)
    check(ctx, N == 1 ?
        ccall((:kmc_kmer_table_export, LIB[]), Int32,
            (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, UInt32, Ptr{Cvoid}, Ptr{Cvoid}, UInt64, Ptr{UInt64}),
            ctx.handle, dk.ptr, dv.ptr, UInt32(log2_capacity), ok.ptr, ov.ptr, n, nout) :
        ccall((:kmc_kmer_table2_export, LIB[]), Int32,
            (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, UInt32, Ptr{Cvoid}, Ptr{Cvoid}, UInt64, Ptr{UInt64}),
            ctx.handle, dk.ptr, dv.ptr, UInt32(log2_capacity), ok.ptr, ov.ptr, n, nout))
    keys, vals = Array(ok), Array(ov)
    foreach(free!, (dk, dv, ok, ov))
    # Kmer{A,K,N} is N UInt64 limbs, head first: the [N, n] export is a vector of n k-mers
    kmers = reinterpret(T, keys)
    return Dict{T, Int}(kmers[i] => Int(vals[i]) for i in eachindex(vals))
end

"""
    t = KmerCountTable(Kmer{A,K}, log2_capacity)
    count!(t, FwKmers{A,K}(seq) | CanonicalKmers{A,K}(seq))     # adds every k-mer (kmc_kmer_count / _count2)
    counts(t, it) -> Vector{UInt32}                             # the count of every k-mer of `it`, in iteration order
    get(t, kmers::Vector{<:Kmer}) -> Vector{UInt32}             # the count of each k-mer, 0 when absent
    spectrum(t, n_bins) -> Vector{UInt64}                       # bin c + 1 = keys with count c, the last bin the rest
    Dict(t; min_count = 1, max_count = typemax(UInt32))         # the keys whose count lies in [min_count, max_count]

An exact k-mer count table that stays in device memory, so that it can be queried without copying it out: the second
pass of a k-mer-spectrum error corrector (`counts`), the trusted / solid k-mers (`Dict` with bounds) and the count
spectrum.  One limb for K <= 32, two for K = 33..64.  Every iterator counted into or looked up in one table must be
of the same kind (forward or canonical).
"""
mutable struct KmerCountTable{T <: Kmer}
    ctx::Context
    log2_capacity::Int
    keys::DeviceVector{UInt64}
    vals::DeviceVector{UInt32}
    mode::Int32                                  # the iterator kind counted so far, -1 before the first count!
    n_keys::Int
end

function KmerCountTable(::Type{Kmer{A, K}}, log2_capacity::Integer; ctx::Context = default_context()) where {A <: NucleicAcidAlphabet{2}, K}
    K <= 64 || throw(ArgumentError("KmerCountTable holds k-mers of one or two limbs (K <= 64)"))
    T = derive_type(Kmer{A, K})
    N = K <= 32 ? 1 : 2
    dk, dv = DeviceVector{UInt64}(ctx, N << log2_capacity), DeviceVector{UInt32}(ctx, 1 << log2_capacity)
    zero!(dk, 0xff)
    zero!(dv)
    return KmerCountTable{T}(ctx, Int(log2_capacity), dk, dv, Int32(-1), 0)   # (the DeviceVectors free themselves)
end

limbs(::KmerCountTable{Kmer{A, K, N}}) where {A, K, N} = N

function check_mode!(t::KmerCountTable, mode::Int32)
    t.mode == -1 && (t.mode = mode)
    t.mode == mode || throw(ArgumentError("the table was counted from $(t.mode == KMC_CANON ? "canonical" : "forward") k-mers"))
end

function Base.count!(t::KmerCountTable{Kmer{A, K, N}}, it::Union{FwKmers{A, K}, CanonicalKmers{A, K}}) where {A, K, N}
    mode = Int32(mode_of(typeof(it)))
    check_mode!(t, mode)
    res, ctx = KmcResult(), t.ctx
    with_device_sequence(ctx, source(it)) do d
        st = limbs(t) == 1 ?
            ccall((:kmc_kmer_count, LIB[]), Int32, (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, Ptr{Cvoid}, Ptr{Cvoid}, UInt32, Ref{KmcResult}),
                ctx.handle, d, K, mode, t.keys.ptr, t.vals.ptr, UInt32(t.log2_capacity), res) :
            ccall((:kmc_kmer_count2, LIB[]), Int32, (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, Ptr{Cvoid}, Ptr{Cvoid}, UInt32, Ref{KmcResult}),
                ctx.handle, d, K, mode, t.keys.ptr, t.vals.ptr, UInt32(t.log2_capacity), res)
        st == KMC_OK || throw_status(ctx, st, res, A)
    end
    t.n_keys += Int(res.digest[1])
    return t
end

function counts(t::KmerCountTable{Kmer{A, K, N}}, it::Union{FwKmers{A, K}, CanonicalKmers{A, K}}) where {A, K, N}
    mode = Int32(mode_of(typeof(it)))
    check_mode!(t, mode)
    seq, res, ctx = source(it), KmcResult(), t.ctx
    n = max(0, length(seq) - K + 1)
    dout = DeviceVector{UInt32}(ctx, n)
    with_device_sequence(ctx, seq) do d
        st = limbs(t) == 1 ?
            ccall((:kmc_kmer_lookup, LIB[]), Int32,
                (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, Ptr{Cvoid}, Ptr{Cvoid}, UInt32, Ptr{Cvoid}, UInt64, Ref{KmcResult}),
                ctx.handle, d, K, mode, t.keys.ptr, t.vals.ptr, UInt32(t.log2_capacity), dout.ptr, n, res) :
            ccall((:kmc_kmer_lookup2, LIB[]), Int32,
                (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, Ptr{Cvoid}, Ptr{Cvoid}, UInt32, Ptr{Cvoid}, UInt64, Ref{KmcResult}),
                ctx.handle, d, K, mode, t.keys.ptr, t.vals.ptr, UInt32(t.log2_capacity), dout.ptr, n, res)
        st == KMC_OK || throw_status(ctx, st, res, A)
    end
    out = Array(dout)
    free!(dout)
    return out
end

function Base.get(t::KmerCountTable{T}, kmers::Vector{T}) where {T <: Kmer}
    ctx = t.ctx
    dq, dout = upload(ctx, reinterpret(UInt64, kmers)), DeviceVector{UInt32}(ctx, length(kmers))
    check(ctx, limbs(t) == 1 ?
        ccall((:kmc_kmer_table_get, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, UInt32, Ptr{Cvoid}, UInt64, Ptr{Cvoid}),
            ctx.handle, t.keys.ptr, t.vals.ptr, UInt32(t.log2_capacity), dq.ptr, UInt64(length(kmers)), dout.ptr) :
        ccall((:kmc_kmer_table2_get, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, UInt32, Ptr{Cvoid}, UInt64, Ptr{Cvoid}),
            ctx.handle, t.keys.ptr, t.vals.ptr, UInt32(t.log2_capacity), dq.ptr, UInt64(length(kmers)), dout.ptr))
    out = Array(dout)
    free!(dq)
    free!(dout)
    return out
end

function spectrum(t::KmerCountTable, n_bins::Integer)
    ctx = t.ctx
    dh = DeviceVector{UInt64}(ctx, n_bins)
    zero!(dh)
    check(ctx, limbs(t) == 1 ?
        ccall((:kmc_kmer_table_histogram, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, UInt32, Ptr{Cvoid}, UInt32),
            ctx.handle, t.keys.ptr, t.vals.ptr, UInt32(t.log2_capacity), dh.ptr, UInt32(n_bins)) :
        ccall((:kmc_kmer_table2_histogram, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, UInt32, Ptr{Cvoid}, UInt32),
            ctx.handle, t.keys.ptr, t.vals.ptr, UInt32(t.log2_capacity), dh.ptr, UInt32(n_bins)))
    out = Array(dh)
    free!(dh)
    return out
end

function Base.Dict(t::KmerCountTable{T}; min_count::Integer = 1, max_count::Integer = typemax(UInt32)) where {T <: Kmer}
    ctx, N, n = t.ctx, limbs(t), max(1, t.n_keys)
    ok, ov, nout = DeviceVector{UInt64}(ctx, N * n), DeviceVector{UInt32}(ctx, n), Ref{UInt64}(0)
    check(ctx, limbs(t) == 1 ?
        ccall((:kmc_kmer_table_export_range, LIB[]), Int32,
            (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, UInt32, UInt32, UInt32, Ptr{Cvoid}, Ptr{Cvoid}, UInt64, Ptr{UInt64}),
            ctx.handle, t.keys.ptr, t.vals.ptr, UInt32(t.log2_capacity), UInt32(min_count), UInt32(max_count), ok.ptr, ov.ptr, UInt64(n), nout) :
        ccall((:kmc_kmer_table2_export_range, LIB[]), Int32,
            (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, UInt32, UInt32, UInt32, Ptr{Cvoid}, Ptr{Cvoid}, UInt64, Ptr{UInt64}),
            ctx.handle, t.keys.ptr, t.vals.ptr, UInt32(t.log2_capacity), UInt32(min_count), UInt32(max_count), ok.ptr, ov.ptr, UInt64(n), nout))
    m = Int(nout[])
    keys, vals = Array(truncate!(ok, N * m)), Array(truncate!(ov, m))
    free!(ok)
    free!(ov)
    kmers = reinterpret(T, keys)
    return Dict{T, Int}(kmers[i] => Int(vals[i]) for i in eachindex(vals))
end

"""
    bucket_count(CanonicalKmers{A,K}(seq), bits) -> Vector{UInt32}   (length 2^bits)
    bucket_count(CanonicalDNAMers{K}, reads, bits; group) -> Vector{UInt32}

`table[fx_hash(canonical k-mer) >> (64 - bits) + 1] += 1` for every window (`kmc_bucket_count`).  With a `Group` the
reads are sharded over its GPUs, every GPU counts its shard and the tables are summed by NCCL inside the library, the
merge overlapping the count (`kmc_group_bucket_count`: north_star's count table and its only collective).
"""
function bucket_count(it::CanonicalKmers{A, K}, bits::Integer;
        ctx::Context = default_context()) where {A <: NucleicAcidAlphabet{2}, K}
    res = KmcResult()
    dt = DeviceVector{UInt32}(ctx, 1 << bits)
    zero!(dt)
    with_device_sequence(ctx, source(it)) do d
        st = ccall((:kmc_bucket_count, LIB[]), Int32,
            (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, Ptr{Cvoid}, Ref{KmcResult}),
            ctx.handle, d, K, bits, dt.ptr, res)
        st == KMC_OK || throw_status(ctx, st, res, A)
    end
    table = Array(dt)
    free!(dt)
    return table
end

function bucket_count(::Type{I}, reads::AbstractVector{S}, bits::Integer; group::Group) where {I <: CanonicalKmers, S <: LongSequence{<:NucleicAcidAlphabet{2}}}
    K = ksize_of(I)
    nd = length(group)
    ranges = shard_ranges([length(r) for r in reads], nd)
    packs = [pack_reads(view(reads, r)) for r in ranges]
    dwords = [upload(group.ctx[i], packs[i].words) for i in 1:nd]
    doff = [upload(group.ctx[i], packs[i].woff) for i in 1:nd]
    dlen = [upload(group.ctx[i], packs[i].lens) for i in 1:nd]
    tables = [DeviceVector{UInt32}(group.ctx[i], 1 << bits) for i in 1:nd]
    foreach(zero!, tables)
    seqs = [KmcSeqs(dwords[i].ptr, length(packs[i].words), length(packs[i].lens), doff[i].ptr, dlen[i].ptr, 0, 0, UInt32(2), 0) for i in 1:nd]
    tptr = Ptr{UInt32}[t.ptr for t in tables]
    rbuf = zeros(UInt8, nd * sizeof(KmcResult))
    GC.@preserve seqs tptr rbuf begin
        st = ccall((:kmc_group_bucket_count, LIB[]), Int32, (Ptr{Cvoid}, Ptr{KmcSeqs}, Int32, Int32, Ptr{Ptr{UInt32}}, Ptr{UInt8}),
            group.handle, seqs, K, bits, tptr, rbuf)
        check(group.ctx[1], st)
    end
    merged = Array(tables[1])   # every device holds the merged table
    foreach(free!, vcat(dwords, doff, dlen))
    foreach(free!, tables)
    return merged
end

end # module
