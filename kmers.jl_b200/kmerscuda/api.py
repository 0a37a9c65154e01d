"""Host-side mirror of the reference's iterator interface for the k-mer extraction path.

Same names, argument meaning and error behaviour as Kmers.jl (paths relative to the reference):

  FwKmers(A, K, seq)            src/iterators/FwKmers.jl:28-59
  FwRvIterator(A, K, seq)       src/iterators/CanonicalKmers.jl:25-56
  CanonicalKmers(A, K, seq)     src/iterators/CanonicalKmers.jl:199-225
  UnambiguousKmers(A, K, seq)   src/iterators/UnambiguousKmers.jl:29-62
  fx_hash(kmers, h)             src/kmer.jl:255-261
  LongSequence                  BioSequences.LongSequence{A}(data::Vector{UInt64}, len) (L0 substrate)

`collect(it)` returns what Julia's `collect` would hold in memory: an array of `Kmer{A,K,N}.data`
limbs (`NTuple{N,UInt64}`, head first), tuples in the Julia element layout.  All arithmetic happens
in libkmerscuda.so on the GPU; this module only maps types to integers and owns buffers.  There
is no CPU fallback: without the library or a CUDA device every call raises.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from . import _abi
from ._abi import (KMC_AOS, KMC_CANON, KMC_E_AMBIGUOUS, KMC_E_BAD_K, KMC_FW, KMC_FWRV, KMC_HASH_FX, KMC_KMER4, KMC_MAX_K,
                   KMC_MAX_K4, KMC_NO_SYNC, KMC_OK, KMC_OUT_DEVICE, KMC_RNA, KMC_UNAMBIG, kmc_out, kmc_result, kmc_seqs)

# ----------------------------------------------------------------------------------------------
# alphabets (only what the path needs: the 2- and 4-bit nucleic acid alphabets)
# ----------------------------------------------------------------------------------------------


@dataclass(frozen=True)
class Alphabet:
    name: str
    bits: int


DNAAlphabet2 = Alphabet("DNAAlphabet{2}", 2)
RNAAlphabet2 = Alphabet("RNAAlphabet{2}", 2)
DNAAlphabet4 = Alphabet("DNAAlphabet{4}", 4)
RNAAlphabet4 = Alphabet("RNAAlphabet{4}", 4)

_CODE2 = {"A": 0, "C": 1, "G": 2, "T": 3, "U": 3}
_CODE4 = {"-": 0, "A": 1, "C": 2, "M": 3, "G": 4, "R": 5, "S": 6, "V": 7, "T": 8, "U": 8, "W": 9, "Y": 10,
          "H": 11, "K": 12, "D": 13, "B": 14, "N": 15}
_SYM4_DNA = "-ACMGRSVTWYHKDBN"


class EncodeError(Exception):
    """BioSequences.EncodeError as thrown through src/construction.jl:108-110."""

    def __init__(self, alphabet: Alphabet, symbol: str, seq_index: int = 0, position: int = 0):
        super().__init__(f"cannot encode {symbol} in {alphabet.name}")
        self.alphabet, self.symbol, self.seq_index, self.position = alphabet, symbol, seq_index, position


class KmersCUDAError(RuntimeError):
    pass


def n_limbs(K: int, bits: int = 2) -> int:
    """N of Kmer{A,K,N} (src/kmer.jl:97-111): cld(K * bits per symbol, 64)."""
    return (bits * K + 63) // 64


def _check_K(K):
    # FwKmers.jl:31-33
    if not isinstance(K, (int, np.integer)) or isinstance(K, bool):
        raise TypeError("K must be an Int")
    if K < 1:
        raise ValueError("K must be at least 1")


# ----------------------------------------------------------------------------------------------
# sequences
# ----------------------------------------------------------------------------------------------


class LongSequence:
    """LongSequence{A}: `data` are the packed UInt64 words, `len` the number of symbols."""

    def __init__(self, alphabet: Alphabet, data: np.ndarray, length: int):
        self.alphabet = alphabet
        self.data = np.ascontiguousarray(data, dtype=np.uint64)
        self.len = int(length)
        need = (self.len * alphabet.bits + 63) // 64
        if self.data.size < need:
            raise ValueError("data holds fewer words than `length` symbols need")

    def __len__(self):
        return self.len

    @classmethod
    def from_string(cls, alphabet: Alphabet, s: str) -> "LongSequence":
        table = _CODE2 if alphabet.bits == 2 else _CODE4
        try:
            codes = np.fromiter((table[c] for c in s.upper()), dtype=np.uint64, count=len(s))
        except KeyError as e:  # what LongDNA{2}("...N...") does
            raise EncodeError(alphabet, e.args[0]) from None
        per = 64 // alphabet.bits
        nw = (len(s) + per - 1) // per
        padded = np.zeros(nw * per, dtype=np.uint64)
        padded[: len(s)] = codes
        shifts = np.arange(per, dtype=np.uint64) * np.uint64(alphabet.bits)
        data = np.bitwise_or.reduce(padded.reshape(nw, per) << shifts, axis=1) if nw else np.zeros(0, np.uint64)
        return cls(alphabet, data.astype(np.uint64), len(s))


def LongDNA2(s: str) -> LongSequence:
    return LongSequence.from_string(DNAAlphabet2, s)


def LongDNA4(s: str) -> LongSequence:
    return LongSequence.from_string(DNAAlphabet4, s)


class ReadSet:
    """A batch of LongSequences in one word-aligned CSR buffer (what `Vector{LongDNA{2}}` becomes).

    Either ragged (`seq_word_offset`, `seq_len` arrays) or uniform (`uniform_len`, `uniform_stride_words`).
    bits = 8 is a set of ASCII sources (`Vector{String}`): `words` are the concatenated BYTES and the
    offsets / strides count bytes.
    """

    def __init__(self, bits: int, words: np.ndarray, n_seqs: int, *, seq_word_offset=None, seq_len=None,
                 uniform_len: int = 0, uniform_stride_words: int = 0, first_symbol_offset: int = 0):
        self.bits = bits
        self.words = np.ascontiguousarray(words, dtype=np.uint8 if bits == 8 else np.uint64)
        self.n_seqs = int(n_seqs)
        self.seq_word_offset = None if seq_word_offset is None else np.ascontiguousarray(seq_word_offset, np.uint64)
        self.seq_len = None if seq_len is None else np.ascontiguousarray(seq_len, np.uint64)
        self.uniform_len = int(uniform_len)
        self.uniform_stride_words = int(uniform_stride_words)
        self.first_symbol_offset = int(first_symbol_offset)

    @classmethod
    def from_sequences(cls, seqs: Sequence[LongSequence]) -> "ReadSet":
        bits = seqs[0].alphabet.bits if seqs else 2
        need = [(len(s) * bits + 63) // 64 for s in seqs]
        off = np.zeros(len(seqs) + 1, dtype=np.uint64)
        off[1:] = np.cumsum(need)
        words = np.zeros(int(off[-1]), dtype=np.uint64)
        for s, o, n in zip(seqs, off[:-1], need):
            words[int(o): int(o) + n] = s.data[:n]
        return cls(bits, words, len(seqs), seq_word_offset=off[:-1].copy(),
                   seq_len=np.array([len(s) for s in seqs], dtype=np.uint64))

    @classmethod
    def from_strings(cls, strs) -> "ReadSet":
        """ASCII sources (str / bytes), concatenated without separators."""
        raw = [x.encode("latin-1") if isinstance(x, str) else bytes(x) for x in strs]
        lens = np.array([len(r) for r in raw], dtype=np.uint64)
        off = np.zeros(len(raw) + 1, dtype=np.uint64)
        off[1:] = np.cumsum(lens)
        data = np.frombuffer(b"".join(raw) + b"\0", dtype=np.uint8).copy()
        return cls(8, data, len(raw), seq_word_offset=off[:-1].copy(), seq_len=lens)

    @classmethod
    def ascii(cls, src, first_symbol_offset: int = 0, length: Optional[int] = None) -> "ReadSet":
        """One ASCII source (String, SubString, codeunits, Vector{UInt8})."""
        if isinstance(src, str):
            src = src.encode("latin-1")
        data = np.frombuffer(bytes(src), dtype=np.uint8) if not isinstance(src, np.ndarray) else np.ascontiguousarray(src, np.uint8)
        n = int(data.size) - first_symbol_offset if length is None else length
        if data.size == 0:
            data = np.zeros(1, np.uint8)
        return cls(8, data, 1, uniform_len=n, uniform_stride_words=int(data.size), first_symbol_offset=first_symbol_offset)

    @classmethod
    def single(cls, seq: LongSequence, first_symbol_offset: int = 0, length: Optional[int] = None) -> "ReadSet":
        n = len(seq) if length is None else length
        return cls(seq.alphabet.bits, seq.data, 1, uniform_len=n, uniform_stride_words=seq.data.size,
                   first_symbol_offset=first_symbol_offset)

    def window_counts(self, K: int) -> np.ndarray:
        if self.seq_len is None:
            return np.full(self.n_seqs, max(0, self.uniform_len - K + 1), dtype=np.uint64)
        return np.where(self.seq_len >= K, self.seq_len - np.uint64(K) + np.uint64(1), np.uint64(0)).astype(np.uint64)


# ----------------------------------------------------------------------------------------------
# device context
# ----------------------------------------------------------------------------------------------


class DeviceBuffer:
    """Device memory owned by the library (kmc_malloc / kmc_free)."""

    def __init__(self, ctx: "Context", nbytes: int):
        self.ctx = ctx
        self.nbytes = int(nbytes)
        p = C.c_void_p()
        ctx._check(ctx.lib.kmc_malloc(ctx.handle, max(self.nbytes, 1), C.byref(p)))
        self.ptr = p.value

    def upload(self, arr: np.ndarray):
        arr = np.ascontiguousarray(arr)
        assert arr.nbytes <= self.nbytes
        if arr.nbytes:
            self.ctx._check(self.ctx.lib.kmc_upload(self.ctx.handle, self.ptr, arr.ctypes.data, arr.nbytes))
            self.ctx.sync()  # `arr` may be a temporary
        return self

    def download(self, dtype, count: int, offset_bytes: int = 0) -> np.ndarray:
        out = np.empty(count, dtype=dtype)
        self.ctx._check(self.ctx.lib.kmc_download(self.ctx.handle, out.ctypes.data, self.ptr + offset_bytes, out.nbytes))
        return out

    def free(self):
        if self.ptr:
            self.ctx.lib.kmc_free(self.ctx.handle, self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    """One kmc_ctx: a device, a stream, scratch.  Not thread-safe (one caller at a time)."""

    def __init__(self, device: int = 0, _borrowed=None):
        self.lib = _abi.load()
        self.device = device
        self._owned = _borrowed is None
        if _borrowed is not None:  # a context that belongs to a Group
            self.handle = _borrowed
            return
        h = C.c_void_p()
        st = self.lib.kmc_ctx_create(device, C.byref(h))
        if st != KMC_OK:
            raise KmersCUDAError(
                f"kmc_ctx_create(device={device}) failed: {self.lib.kmc_status_string(st).decode()} "
                "-- KmersCUDA needs a CUDA device; there is no CPU fallback")
        self.handle = h

    def close(self):
        if self.handle and self._owned:
            self.lib.kmc_ctx_destroy(self.handle)
        self.handle = None

    # ---- one process per GPU: an NCCL communicator attached to this context (comm.cu) --------------
    @staticmethod
    def comm_unique_id() -> bytes:
        """128 bytes made by rank 0 and broadcast by the launcher (torch.distributed, MPI, a file)."""
        lib = _abi.load()
        buf = C.create_string_buffer(_abi.KMC_COMM_ID_BYTES)
        st = lib.kmc_comm_unique_id(buf)
        if st != KMC_OK:
            raise KmersCUDAError(f"kmc_comm_unique_id: {lib.kmc_status_string(st).decode()}")
        return buf.raw

    def comm_init(self, n_ranks: int, rank: int, unique_id: bytes):
        assert len(unique_id) == _abi.KMC_COMM_ID_BYTES
        self._check(self.lib.kmc_comm_init_rank(self.handle, n_ranks, rank, C.c_char_p(unique_id)))

    def comm_init_torch(self, group=None):
        """Attach a communicator whose ranks are the ranks of an initialised torch.distributed group: the id
        travels by broadcast_object_list; the collectives themselves then run inside libkmerscuda."""
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        box = [Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        self.comm_init(world, rank, box[0])

    def comm_info(self):
        r, n = C.c_int32(), C.c_int32()
        self._check(self.lib.kmc_comm_info(self.handle, C.byref(r), C.byref(n)))
        return r.value, n.value

    def comm_destroy(self):
        self._check(self.lib.kmc_comm_destroy(self.handle))

    def allreduce(self, dptr: int, n: int, dtype=np.uint32):
        fn = self.lib.kmc_allreduce_u32 if np.dtype(dtype).itemsize == 4 else self.lib.kmc_allreduce_u64
        self._check(fn(self.handle, dptr, n))

    def bucket_count_merge(self, desc, K: int, bucket_bits: int, table_ptr: int):
        """Count this rank's reads and sum the tables of all ranks, the merge overlapping the count
        (kmc_bucket_count_merge).  Returns (k-mers this rank counted, device ms)."""
        res = kmc_result()
        self._check(self.lib.kmc_bucket_count_merge(self.handle, C.byref(desc), K, bucket_bits, table_ptr, C.byref(res)))
        return int(res.n_written), float(res.kernel_ms)

    def trim(self):
        self._check(self.lib.kmc_trim(self.handle))

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st: int):
        if st != KMC_OK:
            msg = self.lib.kmc_last_error(self.handle).decode() or self.lib.kmc_status_string(st).decode()
            raise KmersCUDAError(f"libkmerscuda status {st}: {msg}")

    def sync(self):
        self._check(self.lib.kmc_sync(self.handle))

    def set_stream(self, cuda_stream: Optional[int]):
        self._check(self.lib.kmc_ctx_set_stream(self.handle, cuda_stream))

    def device_info(self):
        sm, mem, name = C.c_int32(), C.c_uint64(), C.create_string_buffer(128)
        self._check(self.lib.kmc_device_info(self.handle, C.byref(sm), C.byref(mem), name, 128))
        return {"sm_count": sm.value, "total_mem": mem.value, "name": name.value.decode()}

    def alloc(self, nbytes: int) -> DeviceBuffer:
        return DeviceBuffer(self, nbytes)

    def to_device(self, arr: np.ndarray) -> DeviceBuffer:
        arr = np.ascontiguousarray(arr)
        return DeviceBuffer(self, arr.nbytes).upload(arr)

    def pinned(self, nbytes: int, dtype=np.uint8) -> np.ndarray:
        """numpy view of pinned host memory (kmc_host_alloc); keep the returned array alive."""
        p = C.c_void_p()
        self._check(self.lib.kmc_host_alloc(self.handle, max(int(nbytes), 1), C.byref(p)))
        buf = (C.c_uint8 * max(int(nbytes), 1)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=np.uint8, count=int(nbytes)).view(dtype)
        _PINNED[arr.ctypes.data] = (self, p.value)
        return arr

    def digest(self, dptr: int, n_words: int):
        """(xor, wrapping sum) of n_words u64 in device memory (kmc_digest)."""
        out = (C.c_uint64 * 2)()
        self._check(self.lib.kmc_digest(self.handle, dptr, n_words, out))
        return int(out[0]), int(out[1])

    def timer_begin(self):
        self._check(self.lib.kmc_timer_begin(self.handle))

    def timer_end(self) -> float:
        ms = C.c_float()
        self._check(self.lib.kmc_timer_end(self.handle, C.byref(ms)))
        return ms.value


_PINNED: dict = {}
_DEFAULT: dict = {}


def default_context(device: int = 0) -> Context:
    if device not in _DEFAULT:
        _DEFAULT[device] = Context(device)
    return _DEFAULT[device]


# ----------------------------------------------------------------------------------------------
# device-resident read sets and results
# ----------------------------------------------------------------------------------------------


class DeviceReadSet:
    """A ReadSet uploaded once; the kmc_seqs descriptor points at device memory."""

    def __init__(self, ctx: Context, rs: ReadSet):
        self.ctx, self.host = ctx, rs
        self.words = ctx.to_device(rs.words)
        self.off = None if rs.seq_word_offset is None else ctx.to_device(rs.seq_word_offset)
        self.len = None if rs.seq_len is None else ctx.to_device(rs.seq_len)
        self.desc = kmc_seqs(self.words.ptr, rs.words.size, rs.n_seqs, self.off.ptr if self.off else None,
                             self.len.ptr if self.len else None, rs.uniform_len, rs.uniform_stride_words, rs.bits,
                             rs.first_symbol_offset)


def _host_desc(rs: ReadSet) -> kmc_seqs:
    return kmc_seqs(rs.words.ctypes.data if rs.words.size else None, rs.words.size, rs.n_seqs,
                    None if rs.seq_word_offset is None else rs.seq_word_offset.ctypes.data,
                    None if rs.seq_len is None else rs.seq_len.ctypes.data, rs.uniform_len, rs.uniform_stride_words,
                    rs.bits, rs.first_symbol_offset)


@dataclass
class Extracted:
    """Result of one extraction (host arrays).  Shapes follow the Julia element layout."""
    kmers: np.ndarray                 # [n, N]  (FWRV + aos: [n, 2, N])
    rv: Optional[np.ndarray] = None   # FWRV SoA: [n, N]
    hash: Optional[np.ndarray] = None
    index: Optional[np.ndarray] = None
    seq_out_offset: Optional[np.ndarray] = None
    n: int = 0
    kernel_ms: float = 0.0


_MODE_NAMES = {KMC_FW: "FwKmers", KMC_FWRV: "FwRvIterator", KMC_CANON: "CanonicalKmers", KMC_UNAMBIG: "UnambiguousKmers"}


def _raise_ambiguous(rs_bits: int, A: Alphabet, res: kmc_result):
    if rs_bits == 8:  # ASCII source: the offending byte
        raise EncodeError(A, chr(res.err_sym & 0xFF), int(res.err_seq), int(res.err_pos))
    sym = _SYM4_DNA[res.err_sym & 15]
    if A.name.startswith("RNA") and sym == "T":
        sym = "U"
    raise EncodeError(A, sym, int(res.err_seq), int(res.err_pos))


def _upper_bound(ctx: Context, desc: kmc_seqs, rs: ReadSet, K: int, mode: int) -> int:
    return int(rs.window_counts(K).sum())


def extract(mode: int, rs, K: int, *, A: Alphabet = DNAAlphabet2, hash: bool = False, aos: bool = False,
            want_seq_offsets: bool = False, ctx: Optional[Context] = None, host_path: bool = False,
            index_base: int = 0, device_out: bool = False) -> Extracted:
    """Batched `collect` of one iterator type over a ReadSet / DeviceReadSet.

    host_path=False: descriptors are uploaded (or already resident), kmc_extract runs on device
    buffers and the outputs are downloaded.  host_path=True: one kmc_extract_host call on host
    buffers (the pipelined entry point a Julia `collect` replacement uses); with device_out=True the
    sequences come from the host but the outputs are written to device buffers (KMC_OUT_DEVICE) and
    only downloaded afterwards.
    """
    _check_K(K)
    if K > (KMC_MAX_K if A.bits == 2 else KMC_MAX_K4):
        raise ValueError(f"K must be at most {KMC_MAX_K if A.bits == 2 else KMC_MAX_K4} for {A.name}")
    if A.bits == 4 and mode == KMC_UNAMBIG:
        raise TypeError("UnambiguousKmers{A<:TwoBit}: the k-mer alphabet must be a 2-bit alphabet")  # UnambiguousKmers.jl:29
    ctx = ctx or default_context()
    lib = ctx.lib
    N = n_limbs(K, A.bits)
    if isinstance(rs, DeviceReadSet):
        drs, hrs = rs, rs.host
    else:
        drs, hrs = None, rs
    cap = _upper_bound(ctx, None, hrs, K, mode)
    two = mode == KMC_FWRV
    want_index = mode == KMC_UNAMBIG
    a_elems = (2 * N if two else N + 1 if want_index else N) if aos else N
    flags = (KMC_HASH_FX if hash else 0) | (KMC_AOS if aos else 0) | (KMC_RNA if A.name.startswith("RNA") else 0)
    if A.bits == 4:
        flags |= KMC_KMER4  # Copyable (4-bit source) or TwoToFour (2-bit source): construction.jl:75-100
    res = kmc_result()

    if host_path and device_out:
        da = ctx.alloc(max(cap, 1) * a_elems * 8)
        db = ctx.alloc(max(cap, 1) * N * 8) if (two and not aos) else None
        dh = ctx.alloc(max(cap, 1) * 8) if hash else None
        di = ctx.alloc(max(cap, 1) * 8) if (want_index and not aos) else None
        dso = None
        out = kmc_out(da.ptr, db.ptr if db else None, dh.ptr if dh else None, di.ptr if di else None, None, cap,
                      index_base)
        desc = _host_desc(hrs)
        st = lib.kmc_extract_host(ctx.handle, C.byref(desc), K, mode, flags | KMC_OUT_DEVICE, C.byref(out), C.byref(res))
        host_path = False  # results are on the device: take the download branch below
    elif host_path:
        a = np.zeros(max(cap, 1) * a_elems, dtype=np.uint64)
        b = np.zeros(max(cap, 1) * N, dtype=np.uint64) if (two and not aos) else None
        h = np.zeros(max(cap, 1), dtype=np.uint64) if hash else None
        ix = np.zeros(max(cap, 1), dtype=np.int64) if (want_index and not aos) else None
        so = np.zeros(hrs.n_seqs + 1, dtype=np.uint64) if want_seq_offsets else None
        out = kmc_out(a.ctypes.data, None if b is None else b.ctypes.data, None if h is None else h.ctypes.data,
                      None if ix is None else ix.ctypes.data, None if so is None else so.ctypes.data, cap, index_base)
        desc = _host_desc(hrs)
        st = lib.kmc_extract_host(ctx.handle, C.byref(desc), K, mode, flags, C.byref(out), C.byref(res))
    else:
        if drs is None:
            drs = DeviceReadSet(ctx, hrs)
        da = ctx.alloc(max(cap, 1) * a_elems * 8)
        db = ctx.alloc(max(cap, 1) * N * 8) if (two and not aos) else None
        dh = ctx.alloc(max(cap, 1) * 8) if hash else None
        di = ctx.alloc(max(cap, 1) * 8) if (want_index and not aos) else None
        dso = ctx.alloc((hrs.n_seqs + 1) * 8) if want_seq_offsets else None
        out = kmc_out(da.ptr, db.ptr if db else None, dh.ptr if dh else None, di.ptr if di else None,
                      dso.ptr if dso else None, cap, index_base)
        st = lib.kmc_extract(ctx.handle, C.byref(drs.desc), K, mode, flags, C.byref(out), C.byref(res))
    if st == KMC_E_AMBIGUOUS:
        _raise_ambiguous(hrs.bits, A, res)
    ctx._check(st)
    n = int(res.n_written)
    if not host_path:
        a = da.download(np.uint64, n * a_elems)
        b = db.download(np.uint64, n * N) if db else None
        h = dh.download(np.uint64, n) if dh else None
        ix = di.download(np.int64, n) if di else None
        so = dso.download(np.uint64, hrs.n_seqs + 1) if dso else None
        for d in (da, db, dh, di, dso):
            if d:
                d.free()
    a = a[: n * a_elems]
    if aos and two:
        kmers = a.reshape(n, 2, N)
    elif aos and want_index:
        kmers = a.reshape(n, N + 1)
    else:
        kmers = a.reshape(n, N)
    return Extracted(kmers=kmers, rv=None if b is None else b[: n * N].reshape(n, N),
                     hash=None if h is None else h[:n], index=None if ix is None else ix[:n],
                     seq_out_offset=so, n=n, kernel_ms=float(res.kernel_ms))


# ----------------------------------------------------------------------------------------------
# the four iterator types
# ----------------------------------------------------------------------------------------------


class _KmerIterator:
    mode = KMC_FW

    def __init__(self, A: Alphabet, K: int, seq):
        _check_K(K)
        # RecodingScheme(A, S) (construction.jl:75-100): LongSequence -> Copyable / FourToTwo,
        # str / bytes / uint8 arrays -> AsciiEncode
        if not isinstance(seq, (LongSequence, str, bytes, bytearray, np.ndarray)):
            raise TypeError("sources are LongSequence (2- or 4-bit) or ASCII (str, bytes, uint8 array)")
        self.A, self.K, self.seq = A, K, seq
        self.is_ascii = not isinstance(seq, LongSequence)

    def __len__(self):
        # FwKmers.jl:40-43
        return max(0, len(self.seq) - self.K + 1)

    def _extract(self, **kw) -> Extracted:
        rs = ReadSet.ascii(self.seq) if self.is_ascii else ReadSet.single(self.seq)
        return extract(self.mode, rs, self.K, A=self.A, **kw)


class FwKmers(_KmerIterator):
    """Every k-mer of `seq`, in order.  collect() -> u64[n, N]."""
    mode = KMC_FW

    def collect(self, **kw) -> np.ndarray:
        return self._extract(**kw).kmers


class FwRvIterator(_KmerIterator):
    """(kmer, reverse_complement(kmer)) for every window.  collect() -> u64[n, 2, N] (Tuple{Kmer,Kmer})."""
    mode = KMC_FWRV

    def collect(self, **kw) -> np.ndarray:
        return self._extract(aos=True, **kw).kmers


class CanonicalKmers(_KmerIterator):
    """min(kmer, reverse_complement(kmer)) for every window.  collect() -> u64[n, N]."""
    mode = KMC_CANON

    def collect(self, **kw) -> np.ndarray:
        return self._extract(**kw).kmers


class UnambiguousKmers(_KmerIterator):
    """(kmer, start) for every window without ambiguous symbols.  collect() -> (u64[n, N], i64[n])."""
    mode = KMC_UNAMBIG

    def __len__(self):
        # IteratorSize is SizeUnknown unless the source is 2-bit (UnambiguousKmers.jl:33-37)
        if self.is_ascii or self.seq.alphabet.bits != 2:
            raise TypeError("length is unknown unless the source is a 2-bit sequence (Base.SizeUnknown)")
        return super().__len__()

    def collect(self, **kw):
        e = self._extract(**kw)
        return e.kmers, e.index


class SpacedKmers(_KmerIterator):
    """Every J-th k-mer: SpacedKmers{A,K,J} (src/iterators/SpacedKmers.jl:22-139), starts 1, 1+J, 1+2J, ...
    kmc_extract_spaced: 2- and 4-bit LongSequence sources and ASCII sources, k-mers over the 2- or the 4-bit
    alphabets (every recoding scheme of construction.jl:75-100), K <= 128 (64 for 4-bit k-mers).
    collect() -> u64[n, N]."""
    mode = KMC_FW

    def __init__(self, A: Alphabet, K: int, J: int, seq):
        super().__init__(A, K, seq)
        if not isinstance(J, (int, np.integer)) or isinstance(J, bool):
            raise TypeError("J must be an Int")
        if J < 1:
            raise ValueError("J must be at least 1")
        self.J = int(J)

    def __len__(self):
        # SpacedKmers.jl:36-40
        L = len(self.seq)
        return 0 if L < self.K else (L - self.K) // self.J + 1

    def collect(self, **kw) -> np.ndarray:
        rs = ReadSet.ascii(self.seq) if self.is_ascii else ReadSet.single(self.seq)
        return extract_spaced(rs, self.K, self.J, A=self.A, **kw).kmers


def extract_spaced(rs, K: int, J: int, *, A: Alphabet = DNAAlphabet2, hash: bool = False, want_seq_offsets: bool = False,
                   ctx: Optional[Context] = None) -> Extracted:
    """Batched collect(SpacedKmers{A,K,J}(seq)) over a ReadSet / DeviceReadSet (kmc_extract_spaced)."""
    _check_K(K)
    if K > (KMC_MAX_K if A.bits == 2 else KMC_MAX_K4):
        raise ValueError(f"K must be at most {KMC_MAX_K if A.bits == 2 else KMC_MAX_K4} for {A.name}")
    ctx = ctx or default_context()
    drs = rs if isinstance(rs, DeviceReadSet) else DeviceReadSet(ctx, rs)
    hrs = drs.host
    N = n_limbs(K, A.bits)
    if hrs.seq_len is None:
        cap = hrs.n_seqs * (0 if hrs.uniform_len < K else (hrs.uniform_len - K) // J + 1)
    else:
        ln = hrs.seq_len.astype(np.int64)
        cap = int(np.where(ln >= K, (ln - K) // J + 1, 0).sum())
    flags = (KMC_HASH_FX if hash else 0) | (KMC_RNA if A.name.startswith("RNA") else 0) | (KMC_KMER4 if A.bits == 4 else 0)
    da = ctx.alloc(max(cap, 1) * N * 8)
    dh = ctx.alloc(max(cap, 1) * 8) if hash else None
    dso = ctx.alloc((hrs.n_seqs + 1) * 8) if want_seq_offsets else None
    out = kmc_out(da.ptr, None, dh.ptr if dh else None, None, dso.ptr if dso else None, cap, 0)
    res = kmc_result()
    st = ctx.lib.kmc_extract_spaced(ctx.handle, C.byref(drs.desc), K, J, flags, C.byref(out), C.byref(res))
    if st == KMC_E_AMBIGUOUS:
        _raise_ambiguous(hrs.bits, A, res)
    ctx._check(st)
    n = int(res.n_written)
    e = Extracted(kmers=da.download(np.uint64, n * N).reshape(n, N), hash=dh.download(np.uint64, n) if dh else None,
                  seq_out_offset=dso.download(np.uint64, hrs.n_seqs + 1) if dso else None, n=n, kernel_ms=float(res.kernel_ms))
    for d in (da, dh, dso):
        if d:
            d.free()
    return e


def SpacedDNAMers(K, J, seq):
    return SpacedKmers(DNAAlphabet2, K, J, seq)


def SpacedRNAMers(K, J, seq):
    return SpacedKmers(RNAAlphabet2, K, J, seq)


def each_codon(seq, A: Optional[Alphabet] = None):
    """each_codon(s) = SpacedKmers{A,3,3}(s) (SpacedKmers.jl:57-82): 2-bit DNA / RNA 3-mers with step 3.  A BioSequence
    fixes DNA or RNA by its own alphabet; a byte-like source takes it from `A` (each_codon(DNA, s) / each_codon(RNA, s))."""
    if isinstance(seq, LongSequence):
        A = RNAAlphabet2 if seq.alphabet.name.startswith("RNA") else DNAAlphabet2
    return SpacedKmers(A or DNAAlphabet2, 3, 3, seq)


def FwDNAMers(K, seq):
    return FwKmers(DNAAlphabet2, K, seq)


def FwRNAMers(K, seq):
    return FwKmers(RNAAlphabet2, K, seq)


def FwRvDNAIterator(K, seq):
    return FwRvIterator(DNAAlphabet2, K, seq)


def CanonicalDNAMers(K, seq):
    return CanonicalKmers(DNAAlphabet2, K, seq)


def CanonicalRNAMers(K, seq):
    return CanonicalKmers(RNAAlphabet2, K, seq)


def UnambiguousDNAMers(K, seq):
    return UnambiguousKmers(DNAAlphabet2, K, seq)


def UnambiguousRNAMers(K, seq):
    return UnambiguousKmers(RNAAlphabet2, K, seq)


def fx_hash(kmers: np.ndarray, h: int = 0, ctx: Optional[Context] = None) -> np.ndarray:
    """fx_hash.(kmers, h) on the device; `kmers` is u64[n, N] (N may be 0: the empty k-mer)."""
    ctx = ctx or default_context()
    km = np.ascontiguousarray(kmers, dtype=np.uint64)
    if km.ndim == 1:
        km = km.reshape(-1, 1)
    n, N = km.shape
    dk = ctx.to_device(km) if km.size else None
    do = ctx.alloc(max(n, 1) * 8)
    ctx._check(ctx.lib.kmc_fx_hash(ctx.handle, dk.ptr if dk else None, n, N, h, do.ptr))
    out = do.download(np.uint64, n)
    if dk:
        dk.free()
    do.free()
    return out


def base_hash(kmers: np.ndarray, K: int, h: int = 0, ctx: Optional[Context] = None) -> np.ndarray:
    """Base.hash.(kmers, h) of Kmer{A,K,N} values (src/kmer.jl:206), Julia 1.10 / 1.11 hashing; `kmers` is u64[n, N]."""
    ctx = ctx or default_context()
    km = np.ascontiguousarray(kmers, dtype=np.uint64)
    if km.ndim == 1:
        km = km.reshape(-1, 1)
    n, N = km.shape
    dk = ctx.to_device(km) if km.size else None
    do = ctx.alloc(max(n, 1) * 8)
    ctx._check(ctx.lib.kmc_base_hash(ctx.handle, dk.ptr if dk else None, n, N, K, h, do.ptr))
    out = do.download(np.uint64, n)
    if dk:
        dk.free()
    do.free()
    return out


def minimizers(rs, K: int, W: int, step: int = 1, *, canonical: bool = False, hash: bool = False,
               ctx: Optional[Context] = None):
    """Minimizers under the fx_hash ordering (docs/src/replacements.md:28-58): for every window start
    1, 1+step, ... the k-mer with the smallest fx_hash among W consecutive k-mers.
    Returns (kmers u64[n], index i64[n] 1-based start of each minimizer, hash u64[n] or None, seq_out_offset)."""
    _check_K(K)
    ctx = ctx or default_context()
    drs = rs if isinstance(rs, DeviceReadSet) else DeviceReadSet(ctx, rs)
    h = drs.host
    span = K + W - 1
    lens = np.full(h.n_seqs, h.uniform_len, dtype=np.int64) if h.seq_len is None else h.seq_len.astype(np.int64)
    cap = int(np.where(lens >= span, (lens - span) // step + 1, 0).sum())
    da, di = ctx.alloc(max(cap, 1) * 8), ctx.alloc(max(cap, 1) * 8)
    dh = ctx.alloc(max(cap, 1) * 8) if hash else None
    dso = ctx.alloc((h.n_seqs + 1) * 8)
    out = kmc_out(da.ptr, None, dh.ptr if dh else None, di.ptr, dso.ptr, cap, 0)
    res = kmc_result()
    ctx._check(ctx.lib.kmc_minimizers(ctx.handle, C.byref(drs.desc), K, W, step, KMC_CANON if canonical else KMC_FW,
                                      KMC_HASH_FX if hash else 0, C.byref(out), C.byref(res)))
    n = int(res.n_written)
    r = (da.download(np.uint64, n), di.download(np.int64, n), dh.download(np.uint64, n) if dh else None,
         dso.download(np.uint64, h.n_seqs + 1))
    for d in (da, di, dh, dso):
        if d:
            d.free()
    return r


def minhash_sketch(rs, K: int, s: int, *, canonical: bool = True, ctx: Optional[Context] = None):
    """Bottom-s MinHash sketch under fx_hash -- `sketch(fx_hash, CanonicalDNAMers{K}(seq), s)` of the
    reference's example (docs/src/minhash.md:31-36): the s smallest distinct fx_hash values over the
    k-mers of the whole set, ascending (u64[<= s])."""
    _check_K(K)
    ctx = ctx or default_context()
    drs = rs if isinstance(rs, DeviceReadSet) else DeviceReadSet(ctx, rs)
    dh = ctx.alloc(max(int(s), 1) * 8)
    res = kmc_result()
    ctx._check(ctx.lib.kmc_minhash_sketch(ctx.handle, C.byref(drs.desc), K, KMC_CANON if canonical else KMC_FW, int(s), dh.ptr,
                                          C.byref(res)))
    out = dh.download(np.uint64, int(res.n_written))
    dh.free()
    return out


def minhash_sketches(rs, K: int, s: int, *, canonical: bool = True, ctx: Optional[Context] = None, stats: bool = False):
    """The bottom-s sketch of every sequence of the set on its own (kmc_minhash_sketch_each): row i of the u64[n_seqs, s]
    array is what `minhash_sketch` returns for sequence i alone, padded with ~0; the u32[n_seqs] array holds the row
    lengths.  stats=True adds a dict: device ms, rounds run past the first and sequences those rounds sketched again."""
    _check_K(K)
    ctx = ctx or default_context()
    drs = rs if isinstance(rs, DeviceReadSet) else DeviceReadSet(ctx, rs)
    n, s = drs.host.n_seqs, int(s)
    dh = ctx.alloc(max(n * max(s, 0), 1) * 8)
    dn = ctx.alloc(max(n, 1) * 4)
    res = kmc_result()
    try:
        ctx._check(ctx.lib.kmc_minhash_sketch_each(ctx.handle, C.byref(drs.desc), K, KMC_CANON if canonical else KMC_FW, s, dh.ptr,
                                                   dn.ptr, C.byref(res)))
        rows = dh.download(np.uint64, n * s).reshape(n, s)
        lens = dn.download(np.uint32, n)
    finally:
        dh.free()
        dn.free()
    if stats:
        return rows, lens, {"kernel_ms": float(res.kernel_ms), "extra_rounds": int(res.digest[0]), "resketched": int(res.digest[1]),
                            "n_written": int(res.n_written)}
    return rows, lens


def minhash_compare(a, a_n, b=None, b_n=None, *, ctx: Optional[Context] = None):
    """Every sketch of A against every sketch of B (kmc_minhash_compare).  a: u64[n_a, s] rows, ascending and distinct
    (as `minhash_sketches` returns them), a_n their lengths (a length above s is read as s); b=None compares A with
    itself.  Returns (shared, shared_bottom), u32[n_a, n_b]: |A_i ∩ B_j| and the number of those among the s smallest
    values of A_i ∪ B_j."""
    ctx = ctx or default_context()
    a = np.ascontiguousarray(a, dtype=np.uint64)
    a_n = np.ascontiguousarray(a_n, dtype=np.uint32)
    same = b is None
    if same:
        b, b_n = a, a_n
    b = np.ascontiguousarray(b, dtype=np.uint64)
    b_n = np.ascontiguousarray(b_n, dtype=np.uint32)
    if a.ndim != 2 or b.ndim != 2 or a.shape[1] != b.shape[1]:
        raise ValueError("a and b must be 2-D with the same sketch size s (columns)")
    if a_n.shape != (a.shape[0],) or b_n.shape != (b.shape[0],):
        raise ValueError("a_n / b_n must hold one length per row")
    n_a, n_b, s = a.shape[0], b.shape[0], a.shape[1]
    bufs = [ctx.to_device(a), ctx.to_device(a_n)]
    bufs += bufs if same else [ctx.to_device(b), ctx.to_device(b_n)]
    d_sh, d_bt = ctx.alloc(max(n_a * n_b, 1) * 4), ctx.alloc(max(n_a * n_b, 1) * 4)
    try:
        ctx._check(ctx.lib.kmc_minhash_compare(ctx.handle, bufs[0].ptr, bufs[1].ptr, n_a, bufs[2].ptr, bufs[3].ptr, n_b, s,
                                               d_sh.ptr, d_bt.ptr))
        shared = d_sh.download(np.uint32, n_a * n_b).reshape(n_a, n_b)
        bottom = d_bt.download(np.uint32, n_a * n_b).reshape(n_a, n_b)
    finally:
        for d in bufs + [d_sh, d_bt]:
            d.free()
    return shared, bottom


def mash_jaccard(shared, shared_bottom, a_n, b_n, s: int):
    """Mash's Jaccard estimate per pair: shared_bottom / min(s, n_A + n_B - shared), with the lengths read as at most s
    (0 where both sketches are empty).  Shapes as `minhash_compare` returns them."""
    na = np.minimum(np.asarray(a_n, dtype=np.int64), s)[:, None]
    nb = np.minimum(np.asarray(b_n, dtype=np.int64), s)[None, :]
    denom = np.minimum(s, na + nb - np.asarray(shared, dtype=np.int64))
    j = np.zeros(denom.shape, dtype=np.float64)
    np.divide(np.asarray(shared_bottom, dtype=np.float64), denom, out=j, where=denom > 0)
    return j


def mash_distance(j, K: int):
    """Mash distance from the Jaccard estimate: -ln(2j / (1 + j)) / K, and 1 where j = 0."""
    j = np.asarray(j, dtype=np.float64)
    d = np.ones(j.shape, dtype=np.float64)
    pos = j > 0
    d[pos] = -np.log(2.0 * j[pos] / (1.0 + j[pos])) / K
    return d


def composition(rs, K: int, *, canonical: bool = False, ctx: Optional[Context] = None, table: Optional[DeviceBuffer] = None):
    """k-mer composition vector: counts[as_integer(kmer)] over every k-mer of the set
    (docs/src/composition.md:28-39), u32[4^K], K <= 14."""
    _check_K(K)
    ctx = ctx or default_context()
    drs = rs if isinstance(rs, DeviceReadSet) else DeviceReadSet(ctx, rs)
    n = 1 << (2 * K)
    own = table is None
    if own:
        table = ctx.alloc(4 * n)
        ctx._check(ctx.lib.kmc_memset(ctx.handle, table.ptr, 0, 4 * n))
    res = kmc_result()
    ctx._check(ctx.lib.kmc_composition(ctx.handle, C.byref(drs.desc), K, KMC_CANON if canonical else KMC_FW, table.ptr,
                                       C.byref(res)))
    host = table.download(np.uint32, n)
    if own:
        table.free()
    return host, int(res.n_written), float(res.kernel_ms)


class KmerTable:
    """Exact k-mer counts on the device (kmc_kmer_count): an open-addressing table keyed by the k-mer,
    the `Dict{Kmer,Int}` a user of the reference's iterators builds.  K <= 31 (forward) / 32 (canonical).

    n_limbs=2 keys the table by two-limb k-mers (kmc_kmer_count2 and the other `*2` entry points): K = 33..63
    (forward) / 64 (canonical), 20 bytes per slot."""

    def __init__(self, log2_capacity: int, ctx: Optional[Context] = None, n_limbs: int = 1):
        if n_limbs not in (1, 2):
            raise ValueError(f"n_limbs must be 1 or 2, not {n_limbs}")
        self.ctx = ctx or default_context()
        self.log2_capacity = int(log2_capacity)
        self.n_limbs = n_limbs
        n = 1 << self.log2_capacity
        self.keys, self.vals = self.ctx.alloc(8 * n_limbs * n), self.ctx.alloc(4 * n)
        self.ctx._check(self.ctx.lib.kmc_memset(self.ctx.handle, self.keys.ptr, 0xFF, 8 * n_limbs * n))
        self.ctx._check(self.ctx.lib.kmc_memset(self.ctx.handle, self.vals.ptr, 0, 4 * n))
        self.n_keys = 0

    def _fn(self, name: str):
        """The entry point `name` of this table's key width (kmc_kmer_count -> kmc_kmer_count2, ...)."""
        if self.n_limbs == 2:
            name = (name.replace("kmc_kmer_table_", "kmc_kmer_table2_").replace("kmc_kmer_count", "kmc_kmer_count2")
                    .replace("kmc_kmer_lookup", "kmc_kmer_lookup2"))
        return getattr(self.ctx.lib, name)

    def _same_width(self, other: "KmerTable"):
        if other.n_limbs != self.n_limbs:
            raise ValueError(f"tables of {self.n_limbs} and {other.n_limbs} limbs cannot be combined")

    def count(self, rs, K: int, *, canonical: bool = True):
        """Adds every k-mer of the set.  Returns (k-mers counted, kernel_ms)."""
        _check_K(K)
        drs = rs if isinstance(rs, DeviceReadSet) else DeviceReadSet(self.ctx, rs)
        res = kmc_result()
        self.ctx._check(self._fn("kmc_kmer_count")(self.ctx.handle, C.byref(drs.desc), K, KMC_CANON if canonical else KMC_FW,
                                                   self.keys.ptr, self.vals.ptr, self.log2_capacity, C.byref(res)))
        self.n_keys += int(res.digest[0])
        return int(res.n_written), float(res.kernel_ms)

    def merge(self, other: "KmerTable"):
        """self[k] += other[k] for every key of `other` (same device): the merge step of a sharded count."""
        self._same_width(other)
        n_new = C.c_uint64(0)
        self.ctx._check(self._fn("kmc_kmer_table_merge")(self.ctx.handle, self.keys.ptr, self.vals.ptr, self.log2_capacity,
                                                         other.keys.ptr, other.vals.ptr, 1 << other.log2_capacity, C.byref(n_new)))
        self.n_keys += int(n_new.value)

    def exchange(self, owned_log2_capacity: int) -> "KmerTable":
        """One process per GPU: send every (key, count) to the rank that owns the key (kmc_kmer_table_exchange over the
        context's communicator) and return this rank's owned table.  Collective."""
        owned = KmerTable(owned_log2_capacity, ctx=self.ctx, n_limbs=self.n_limbs)
        self.ctx.sync()
        n_owned = C.c_uint64(0)
        self.ctx._check(self._fn("kmc_kmer_table_exchange")(self.ctx.handle, self.keys.ptr, self.vals.ptr, self.log2_capacity,
                                                            owned.keys.ptr, owned.vals.ptr, owned_log2_capacity, C.byref(n_owned)))
        owned.n_keys = int(n_owned.value)
        return owned

    def lookup(self, rs, K: int, *, canonical: bool = True, device_out: bool = False):
        """The count of every window of the set (kmc_kmer_lookup): u32[windows] in `extract` order, so element i is the
        count of extract(...).kmers[i] (0 for a k-mer the table does not hold).  Look up with the mode the table was
        counted with.  device_out=True leaves the counts on the device and returns their DeviceBuffer."""
        _check_K(K)
        drs = rs if isinstance(rs, DeviceReadSet) else DeviceReadSet(self.ctx, rs)
        n = int(drs.host.window_counts(K).sum())
        out = self.ctx.alloc(4 * max(n, 1))
        res = kmc_result()
        self.ctx._check(self._fn("kmc_kmer_lookup")(self.ctx.handle, C.byref(drs.desc), K, KMC_CANON if canonical else KMC_FW,
                                                    self.keys.ptr, self.vals.ptr, self.log2_capacity, out.ptr, n, C.byref(res)))
        if device_out:
            return out
        counts = out.download(np.uint32, n)
        out.free()
        return counts

    def get(self, keys: np.ndarray) -> np.ndarray:
        """table[key] for every key (kmc_kmer_table_get): keys u64[n] for one limb, u64[n, 2] for two; u32[n], 0 for a key
        that is not in the table."""
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        if keys.ndim != self.n_limbs or (self.n_limbs == 2 and keys.shape[1] != 2):
            raise ValueError(f"a table of {self.n_limbs} limbs takes keys of shape {'(n,)' if self.n_limbs == 1 else '(n, 2)'}")
        n = keys.shape[0]
        dq, dout = self.ctx.to_device(keys), self.ctx.alloc(4 * max(n, 1))
        self.ctx._check(self._fn("kmc_kmer_table_get")(self.ctx.handle, self.keys.ptr, self.vals.ptr, self.log2_capacity, dq.ptr, n,
                                                       dout.ptr))
        counts = dout.download(np.uint32, n)
        dq.free()
        dout.free()
        return counts

    def histogram(self, n_bins: int = 256) -> np.ndarray:
        """The count spectrum (kmc_kmer_table_histogram): u64[n_bins], bin c = keys with count c, the last bin every
        count of n_bins - 1 and more."""
        h = self.ctx.alloc(8 * n_bins)
        self.ctx._check(self.ctx.lib.kmc_memset(self.ctx.handle, h.ptr, 0, 8 * n_bins))
        self.ctx._check(self._fn("kmc_kmer_table_histogram")(self.ctx.handle, self.keys.ptr, self.vals.ptr, self.log2_capacity,
                                                             h.ptr, n_bins))
        out = h.download(np.uint64, n_bins)
        h.free()
        return out

    def items(self, min_count: Optional[int] = None, max_count: Optional[int] = None):
        """(keys, counts u32[n]) sorted by key: keys u64[n] for one limb; u64[n, 2] (limb 0 = head first) in Kmer order,
        lexicographic on (limb 0, limb 1), for two.  With min_count / max_count only the keys whose count lies in
        [min_count, max_count] (kmc_kmer_table_export_range; the solid k-mers)."""
        n = max(self.n_keys, 1)
        L = self.n_limbs
        dk, dv = self.ctx.alloc(8 * L * n), self.ctx.alloc(4 * n)
        n_out = C.c_uint64(0)
        if min_count is None and max_count is None:
            self.ctx._check(self._fn("kmc_kmer_table_export")(self.ctx.handle, self.keys.ptr, self.vals.ptr, self.log2_capacity,
                                                              dk.ptr, dv.ptr, n, C.byref(n_out)))
        else:
            lo, hi = 0 if min_count is None else int(min_count), 2**32 - 1 if max_count is None else int(max_count)
            self.ctx._check(self._fn("kmc_kmer_table_export_range")(self.ctx.handle, self.keys.ptr, self.vals.ptr,
                                                                    self.log2_capacity, lo, hi, dk.ptr, dv.ptr, n, C.byref(n_out)))
        m = int(n_out.value)
        k, v = dk.download(np.uint64, L * m), dv.download(np.uint32, m)
        dk.free()
        dv.free()
        if L == 1:
            order = np.argsort(k, kind="stable")
            return k[order], v[order]
        k = k.reshape(m, 2)
        order = np.lexsort((k[:, 1], k[:, 0]))
        return k[order], v[order]

    def free(self):
        self.keys.free()
        self.vals.free()


class Group:
    """One process driving several GPUs (kmc_group): a Context per device and one NCCL communicator over them.
    Shard i of the input goes to device i; outputs concatenate in device order (= the reference's order)."""

    def __init__(self, devices: Sequence[int]):
        self.lib = _abi.load()
        devs = (C.c_int32 * len(devices))(*devices)
        h = C.c_void_p()
        st = self.lib.kmc_group_create(len(devices), devs, C.byref(h))
        if st != KMC_OK:
            raise KmersCUDAError(f"kmc_group_create({list(devices)}) failed: {self.lib.kmc_status_string(st).decode()}")
        self.handle = h
        self.ctx = []
        for i, d in enumerate(devices):
            c = C.c_void_p()
            self.lib.kmc_group_ctx(self.handle, i, C.byref(c))
            self.ctx.append(Context(d, _borrowed=c))

    def __len__(self):
        return len(self.ctx)

    def close(self):
        if self.handle:
            for c in self.ctx:
                c.handle = None
            self.lib.kmc_group_destroy(self.handle)
            self.handle = None

    def _check(self, st: int):
        if st != KMC_OK:
            msgs = [self.lib.kmc_last_error(c.handle).decode() for c in self.ctx]
            raise KmersCUDAError(f"libkmerscuda status {st}: {self.lib.kmc_status_string(st).decode()} {[m for m in msgs if m]}")

    def sync(self):
        self._check(self.lib.kmc_group_sync(self.handle))

    def bucket_count(self, shards: Sequence["DeviceReadSet"], K: int, bucket_bits: int):
        """C5: count every shard on its device and merge the tables with NCCL (kmc_group_bucket_count).
        Returns (the merged table u32[2^bucket_bits] read from device 0, k-mers per device, device ms per device,
        the device tables)."""
        n = len(self.ctx)
        assert len(shards) == n
        tables = [c.alloc(4 << bucket_bits) for c in self.ctx]
        for c, t in zip(self.ctx, tables):
            c._check(self.lib.kmc_memset(c.handle, t.ptr, 0, 4 << bucket_bits))
        descs = (kmc_seqs * n)(*[sh.desc for sh in shards])
        ptrs = (C.c_void_p * n)(*[t.ptr for t in tables])
        res = (kmc_result * n)()
        self._check(self.lib.kmc_group_bucket_count(self.handle, descs, K, bucket_bits, ptrs, res))
        merged = tables[0].download(np.uint32, 1 << bucket_bits)
        return merged, [int(r.n_written) for r in res], [float(r.kernel_ms) for r in res], tables

    def extract_host(self, mode: int, shards: Sequence[ReadSet], K: int, *, hash: bool = False, aos: bool = False,
                     index_bases: Optional[Sequence[int]] = None):
        """`collect` over host shards on all devices side by side (kmc_group_extract_host); returns one Extracted
        per device (2-bit k-mer alphabets)."""
        n = len(self.ctx)
        assert len(shards) == n
        N = n_limbs(K)
        two, want_index = mode == KMC_FWRV, mode == KMC_UNAMBIG
        a_elems = (2 * N if two else N + 1 if want_index else N) if aos else N
        flags = (KMC_HASH_FX if hash else 0) | (KMC_AOS if aos else 0)
        bufs, outs = [], (kmc_out * n)()
        for i, rs in enumerate(shards):
            cap = max(int(rs.window_counts(K).sum()), 1)
            a = np.zeros(cap * a_elems, dtype=np.uint64)
            b = np.zeros(cap * N, dtype=np.uint64) if (two and not aos) else None
            h = np.zeros(cap, dtype=np.uint64) if hash else None
            ix = np.zeros(cap, dtype=np.int64) if (want_index and not aos) else None
            bufs.append((a, b, h, ix))
            outs[i] = kmc_out(a.ctypes.data, None if b is None else b.ctypes.data, None if h is None else h.ctypes.data,
                              None if ix is None else ix.ctypes.data, None, cap, 0 if index_bases is None else index_bases[i])
        descs = (kmc_seqs * n)(*[_host_desc(rs) for rs in shards])
        res = (kmc_result * n)()
        st = self.lib.kmc_group_extract_host(self.handle, descs, K, mode, flags, outs, res)
        self._check(st)
        out = []
        for (a, b, h, ix), r in zip(bufs, res):
            m = int(r.n_written)
            kmers = a[: m * a_elems].reshape(m, a_elems if aos else N)
            out.append(Extracted(kmers=kmers, rv=None if b is None else b[: m * N].reshape(m, N), hash=None if h is None else h[:m],
                                 index=None if ix is None else ix[:m], n=m, kernel_ms=float(r.kernel_ms)))
        return out

    def kmer_table_exchange(self, tables: Sequence["KmerTable"], owned_log2_capacity: int):
        """Every (key, count) of the per-device tables to its owner device (kmc_group_kmer_table_exchange);
        returns the owned tables, whose union is the count of the whole input."""
        n = len(self.ctx)
        n_limbs = tables[0].n_limbs
        for t in tables[1:]:
            tables[0]._same_width(t)
        owned = [KmerTable(owned_log2_capacity, ctx=c, n_limbs=n_limbs) for c in self.ctx]
        for c in self.ctx:
            c.sync()
        P = C.c_void_p * n
        n_owned = (C.c_uint64 * n)()
        fn = self.lib.kmc_group_kmer_table2_exchange if n_limbs == 2 else self.lib.kmc_group_kmer_table_exchange
        self._check(fn(
            self.handle, P(*[t.keys.ptr for t in tables]), P(*[t.vals.ptr for t in tables]), tables[0].log2_capacity,
            P(*[t.keys.ptr for t in owned]), P(*[t.vals.ptr for t in owned]), owned_log2_capacity, n_owned))
        for t, m in zip(owned, n_owned):
            t.n_keys = int(m)
        return owned


def bucket_count(rs, K: int, bucket_bits: int, ctx: Optional[Context] = None, table: Optional[DeviceBuffer] = None):
    """Histogram of fx_hash(canonical k-mer) >> (64 - bucket_bits) (north_star extension).
    Returns (table u32[2^bucket_bits] on the host, n_kmers, kernel_ms)."""
    _check_K(K)
    ctx = ctx or default_context()
    drs = rs if isinstance(rs, DeviceReadSet) else DeviceReadSet(ctx, rs)
    own = table is None
    if own:
        table = ctx.alloc(4 << bucket_bits)
        ctx._check(ctx.lib.kmc_memset(ctx.handle, table.ptr, 0, 4 << bucket_bits))
    res = kmc_result()
    ctx._check(ctx.lib.kmc_bucket_count(ctx.handle, C.byref(drs.desc), K, bucket_bits, table.ptr, C.byref(res)))
    host = table.download(np.uint32, 1 << bucket_bits)
    if own:
        table.free()
    return host, int(res.n_written), float(res.kernel_ms)
