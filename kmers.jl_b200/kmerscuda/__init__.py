"""KmersCUDA host mirror: the Kmers.jl iterator interface over libkmerscuda.so (sm_100a).

Importing this package dlopen()s the in-tree CUDA library immediately, so a missing build is an
ImportError here and never a silent fallback.
"""
from . import _abi

_abi.load()

from .api import (  # noqa: E402
    Alphabet, CanonicalDNAMers, CanonicalKmers, CanonicalRNAMers, Context, DeviceBuffer, DeviceReadSet,
    DNAAlphabet2, DNAAlphabet4, EncodeError, Extracted, FwDNAMers, FwKmers, FwRNAMers, FwRvDNAIterator,
    FwRvIterator, KmersCUDAError, LongDNA2, LongDNA4, LongSequence, ReadSet, RNAAlphabet2, RNAAlphabet4,
    UnambiguousDNAMers, UnambiguousKmers, UnambiguousRNAMers, base_hash, bucket_count, default_context, extract, fx_hash,
    SpacedDNAMers, SpacedKmers, SpacedRNAMers, each_codon, extract_spaced, minimizers, minhash_sketch, minhash_sketches, minhash_compare, mash_jaccard, mash_distance, composition, KmerTable, Group, n_limbs)
from ._abi import (KMC_AOS, KMC_CANON, KMC_FW, KMC_FWRV, KMC_HASH_FX, KMC_MAX_K, KMC_NO_SYNC,  # noqa: E402
                   KMC_OUT_DEVICE, KMC_UNAMBIG)
