# Parity of KmersCUDA.collect against the reference's own iterators (run where Julia, Kmers.jl,
# BioSequences.jl, libkmerscuda.so and a B200 are all present; not runnable in the build image).
using Test, BioSequences, Kmers, KmersCUDA, StableRNGs

const RNG = StableRNG(0xccfb2d5055d8c990)   # the reference's test seed, test/runtests.jl:11

@testset "collect == reference" begin
    for len in (0, 30, 31, 32, 150, 10_007), K in (1, 5, 31, 32, 33, 63, 64)
        s2 = randdnaseq(RNG, len); s2 = LongDNA{2}(s2)
        for I in (FwDNAMers{K}, CanonicalDNAMers{K}, FwRvIterator{DNAAlphabet{2}, K}, UnambiguousDNAMers{K})
            @test KmersCUDA.collect(I(s2)) == collect(I(s2))
        end
        s4 = LongDNA{4}(s2)
        len > 3 && (s4[len ÷ 2] = DNA_N)
        @test KmersCUDA.collect(UnambiguousDNAMers{K}(s4)) == collect(UnambiguousDNAMers{K}(s4))
        if len >= K && len > 3
            @test_throws BioSequences.EncodeError KmersCUDA.collect(FwDNAMers{K}(s4))
        end
    end
end

@testset "fx_hash" begin
    v = collect(CanonicalDNAMers{31}(LongDNA{2}(randdnaseq(RNG, 1000))))
    @test KmersCUDA.fx_hash_device(v) == fx_hash.(v)
    @test KmersCUDA.fx_hash_device([mer"TAGCTAG"d])[1] == 0xa76409341339d05a   # test/runtests.jl:907
end

@testset "count_kmers == Dict loop" begin
    s = LongDNA{2}(randdnaseq(RNG, 5_000))
    want = Dict{eltype(CanonicalDNAMers{11}(s)), Int}()
    for m in CanonicalDNAMers{11}(s)
        want[m] = get(want, m, 0) + 1
    end
    @test KmersCUDA.count_kmers(CanonicalDNAMers{11}(s)) == want
    t = KmersCUDA.bucket_count(CanonicalDNAMers{11}(s), 12)
    @test sum(t) == length(s) - 10
end

@testset "count_kmers of two-limb k-mers (K = 33..64) == Dict loop" begin
    genome = randdnaseq(RNG, 2_000)
    s = LongDNA{2}(reduce(*, [genome[i:i+299] for i in rand(RNG, 1:1700, 20)]))   # repeated k-mers
    for (K, canonical) in ((33, false), (47, true), (63, false), (63, true), (64, true))
        it = canonical ? CanonicalDNAMers{K}(s) : FwDNAMers{K}(s)
        want = Dict{eltype(it), Int}()
        for m in it
            want[m] = get(want, m, 0) + 1
        end
        got = KmersCUDA.count_kmers(it)
        @test got == want
        @test keytype(got) == Kmer{DNAAlphabet{2}, K, 2}
    end
    pal = LongDNA{2}("T"^32 * "A"^32)                  # its own reverse complement, head limb all ones
    @test KmersCUDA.count_kmers(CanonicalDNAMers{64}(pal)) == Dict(first(CanonicalDNAMers{64}(pal)) => 1)
    @test_throws ErrorException KmersCUDA.count_kmers(FwDNAMers{64}(s))   # KMC_E_UNSUPPORTED: all-T is {~0, ~0}
    @test_throws ArgumentError KmersCUDA.count_kmers(CanonicalDNAMers{65}(s))
end

@testset "KmerCountTable: per-window counts, get, spectrum, solid k-mers" begin
    genome = randdnaseq(RNG, 3_000)
    s = LongDNA{2}(reduce(*, [genome[i:i+299] for i in rand(RNG, 1:2700, 30)]))
    q = LongDNA{2}(genome[1:1000] * randdnaseq(RNG, 1000))      # half of its k-mers are absent
    for (K, canonical) in ((21, true), (31, false), (47, true), (63, false))
        it(x) = canonical ? CanonicalDNAMers{K}(x) : FwDNAMers{K}(x)
        want = Dict{eltype(it(s)), Int}()
        for m in it(s)
            want[m] = get(want, m, 0) + 1
        end
        t = KmerCountTable(Kmer{DNAAlphabet{2}, K}, 14)
        count!(t, it(s))
        @test counts(t, it(q)) == [get(want, m, 0) for m in it(q)]
        ks = collect(it(q))
        @test get(t, ks) == [get(want, m, 0) for m in ks]
        h = spectrum(t, 8)
        @test h == [Base.count(c -> min(c, 7) == b, values(want)) for b in 0:7]
        @test Dict(t) == want
        @test Dict(t; min_count = 2, max_count = 5) == filter(p -> 2 <= p.second <= 5, want)
        @test_throws ArgumentError counts(t, canonical ? FwDNAMers{K}(q) : CanonicalDNAMers{K}(q))
    end
end

@testset "LongSubSeq views (reference: test/runtests.jl:154-169)" begin
    s2 = LongDNA{2}(randdnaseq(RNG, 1000))
    s4 = LongDNA{4}(s2); s4[500] = DNA_N
    for rng in (2:1000, 33:900, 65:64, 17:48), K in (5, 31, 33)
        v2, v4 = view(s2, rng), view(s4, rng)
        @test KmersCUDA.collect(FwDNAMers{K}(v2)) == collect(FwDNAMers{K}(v2))
        @test KmersCUDA.collect(CanonicalDNAMers{K}(v2)) == collect(CanonicalDNAMers{K}(v2))
        @test KmersCUDA.collect(UnambiguousDNAMers{K}(v4)) == collect(UnambiguousDNAMers{K}(v4))
    end
end

@testset "ASCII sources incl. StringView (reference: test/runtests.jl:892-899)" begin
    str = "ATGCTGATGATCGTATGATGTCGAAA"
    for src in (str, SubString(str, 3:20), codeunits(str), collect(codeunits(str)))
        @test KmersCUDA.collect(FwRvIterator{DNAAlphabet{2}, 9}(src)) == collect(FwRvIterator{DNAAlphabet{2}, 9}(src))
    end
    if Base.find_package("StringViews") !== nothing
        @eval using StringViews
        sv = StringView(collect(codeunits(str)))
        @test KmersCUDA.collect(FwRvIterator{DNAAlphabet{2}, 9}(sv)) == collect(FwRvIterator{DNAAlphabet{2}, 9}(sv))
    end
end

@testset "device-resident extraction and groups" begin
    reads = [LongDNA{2}(randdnaseq(RNG, rand(RNG, 0:300))) for _ in 1:2000]
    want = reduce(vcat, [collect(CanonicalDNAMers{31}(r)) for r in reads])
    km, h, off = KmersCUDA.extract(CanonicalDNAMers{31}, reads; hash = true)
    @test km == want && h == fx_hash.(want) && off[end] == length(want)
    dk, dh = KmersCUDA.extract(CanonicalDNAMers{31}, reads; hash = true, device = true)
    @test Array(dk) == want && Array(dh) == fx_hash.(want)
    @test Array(KmersCUDA.fx_hash_device(dk)) == fx_hash.(want)
    g = KmersCUDA.Group()
    parts = KmersCUDA.extract(CanonicalDNAMers{31}, reads; hash = true, group = g)
    @test reduce(vcat, [p[1] for p in parts]) == want
    t = KmersCUDA.bucket_count(CanonicalDNAMers{31}, reads, 16; group = g)
    ref = zeros(UInt32, 1 << 16)
    for m in want
        ref[(fx_hash(m) >> 48) + 1] += 1
    end
    @test t == ref
end

@testset "LongSequence.data layout (what the device assumes; tests/golden pins it for the oracle)" begin
    @test LongDNA{2}("TAGCTAGGACA").data == [0x000000000004a363]
end

@testset "SpacedKmers / each_codon (reference: test/runtests.jl:849-889)" begin
    for (s, A) in Any[("TA-NGAKATCGAWTAGA", DNAAlphabet{4}), ("AUGCUGAUGAGUCGUAG", RNAAlphabet{2})]
        for (k, j) in ((3, 2), (2, 4), (3, 3)), src in (s, codeunits(s))
            @test KmersCUDA.collect(SpacedKmers{A, k, j}(src)) == collect(SpacedKmers{A, k, j}(src))
        end
    end
    @test KmersCUDA.collect(SpacedKmers{DNAAlphabet{2}, 4, 3}(rna"UAGUCGUAGUAG")) == collect(SpacedKmers{DNAAlphabet{2}, 4, 3}(rna"UAGUCGUAGUAG"))
    @test KmersCUDA.collect(SpacedKmers{RNAAlphabet{4}, 2, 3}(dna"TAGCCWKMMNAGCTV")) == collect(SpacedKmers{RNAAlphabet{4}, 2, 3}(dna"TAGCCWKMMNAGCTV"))
    @test_throws BioSequences.EncodeError KmersCUDA.collect(SpacedDNAMers{3, 4}("TAGAWWWW"))
    @test KmersCUDA.collect(each_codon(DNA, "TGACGATCGAC")) == collect(each_codon(DNA, "TGACGATCGAC"))
end

@testset "minhash_sketches == minhash_sketch per sequence; minhash_compare == set definitions" begin
    seqs = [LongDNA{2}(randdnaseq(RNG, len)) for len in (0, 10, 20, 21, 500, 5_000, 50_000)]
    for canonical in (true, false), s in (1, 10, 1000)
        rows = KmersCUDA.minhash_sketches(seqs, 21, s; canonical)
        for (i, q) in enumerate(seqs)
            it = canonical ? CanonicalDNAMers{21}(q) : FwDNAMers{21}(q)
            @test rows[i] == KmersCUDA.minhash_sketch(it, s)
            @test rows[i] == first(sort!(unique(fx_hash.(collect(it)))), s)
        end
        shared, bottom = KmersCUDA.minhash_compare(rows, s)
        for i in eachindex(rows), j in eachindex(rows)
            x, y = Set(rows[i]), Set(rows[j])
            @test shared[i, j] == length(x ∩ y)
            @test bottom[i, j] == length(Set(first(sort!(collect(x ∪ y)), s)) ∩ x ∩ y)
        end
    end
end
