"""Frames whose output reaches and passes 2^28 bytes, built cheaply, and the C references that check them.

Large outputs are made of RLE blocks (four bytes of frame each) with a Raw block now and then, so that building a frame of
2 GiB output costs milliseconds and a few hundred KiB of frame.  Offsets at the 2^28 - 1 seam sit in explicit-sequence
blocks (seqbuild.Seqs) after such a prefix.  Expected bytes come from libzstd (decoded into a numpy buffer) and expected
statuses from the oracle, both through pointers so that no Python bytes copy of an output is ever made.
"""
import ctypes as C
import hashlib
import struct

import numpy as np

import oracle_lib as O
import seqbuild as S
from cairo_zstd_b200 import workloads as W

M28 = 1 << 28
CLAMP = M28 - 1            # the largest offset a decoded sequence record holds exactly
MAX_OUT = (1 << 31) - 1    # CZB_MAX_FRAME_OUTPUT


class _Size:
    """Stands in for the content in seqbuild.build_frame when only its length is needed (checksum added separately)."""

    def __init__(self, n):
        self.n = n

    def __len__(self):
        return self.n


_oracle = None


def oracle():
    """The oracle's decode and XXH64 with pointer arguments (its own CDLL instance: oracle_lib's argtypes stay as they are)."""
    global _oracle
    if _oracle is None:
        L = C.CDLL(O.build())
        L.oracle_decode_frame.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_uint32,
                                          C.POINTER(O.OracleResult), C.c_void_p]
        L.oracle_decode_frame.restype = C.c_int
        L.oracle_xxh64.argtypes = [C.c_void_p, C.c_size_t, C.c_uint64]
        L.oracle_xxh64.restype = C.c_uint64
        _oracle = L
    return _oracle


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def xxh32_low(a):
    return oracle().oracle_xxh64(_ptr(a), a.size, 0) & 0xFFFFFFFF


def oracle_decode(frame, cap, keep_output=False):
    """(status, OracleResult[, output array]) of the oracle on `frame` with a dst span of `cap` bytes."""
    dst = np.empty(max(cap, 1), dtype=np.uint8)
    res = O.OracleResult()
    src = np.frombuffer(frame, dtype=np.uint8)
    st = oracle().oracle_decode_frame(_ptr(src), src.size, _ptr(dst), cap, 0, C.byref(res), None)
    if keep_output:
        return st, res, dst[:res.bytes_written] if st == 0 else None
    return st, res


def libzstd_decode(frame, size):
    """libzstd's output of a frame of `size` bytes of content, as a numpy array (asserts that libzstd accepts it)."""
    z = W.libzstd()
    out = np.empty(max(size, 1), dtype=np.uint8)
    src = np.frombuffer(frame, dtype=np.uint8)
    n = z.ZSTD_decompress(_ptr(out), out.size, _ptr(src), src.size)
    assert not z.ZSTD_isError(n), "libzstd rejects the frame"
    assert n == size, (n, size)
    return out[:size]


def digest(a):
    return hashlib.blake2b(memoryview(a), digest_size=32).hexdigest()


def fill_blocks(n, seed, raw_every=0):
    """Blocks regenerating n bytes: 128 KiB RLE blocks of varying bytes, every raw_every-th one a Raw block of random bytes
    (0: none), and a short Raw block at the start so that byte 0 is distinctive.  Returns (blocks, content array)."""
    rng = np.random.default_rng(seed)
    blocks, parts, pos, k = [], [], 0, 0
    head = rng.integers(0, 256, min(n, 61), dtype=np.uint8)
    blocks.append(S.Raw(head.tobytes())); parts.append(head); pos += head.size
    while pos < n:
        m = min(S.BLOCK_MAX, n - pos)
        if raw_every and k % raw_every == raw_every - 1:
            a = rng.integers(0, 256, m, dtype=np.uint8)
            blocks.append(S.Raw(a.tobytes())); parts.append(a)
        else:
            b = int(rng.integers(0, 256))
            blocks.append(S.Rle(b, m)); parts.append(np.full(m, b, dtype=np.uint8))
        pos += m; k += 1
    return blocks, np.concatenate(parts) if parts else np.zeros(0, np.uint8)


def rle_only(n, byte=0x5A):
    """n bytes of one value in RLE blocks: no content array needed to know the output."""
    return [S.Rle(byte, min(S.BLOCK_MAX, n - p)) for p in range(0, n, S.BLOCK_MAX)]


def frame(blocks, size, xxh=None, **kw):
    """seqbuild.build_frame for content of `size` bytes whose XXH64 low 32 bits are `xxh` (None: no checksum)."""
    f = S.build_frame(blocks, content=_Size(size), checksum=False, **kw)
    if xxh is None:
        return f
    f = bytearray(f)
    f[4] |= 4  # Content_Checksum_flag
    return bytes(f) + struct.pack("<I", xxh)


def seq_frame(prefix_n, seqs, lits=b"", window_log=None, seed=1, tail=None):
    """A prefix of prefix_n bytes (fill_blocks), then one Seqs block (the frame's first block with sequences), then the
    blocks of `tail` (seqbuild blocks).  The frame is built without a checksum: the content is what libzstd says, when it
    is valid.  window_log None: single segment (window = content size)."""
    blocks, _ = fill_blocks(prefix_n, seed)
    blocks.append(S.Seqs(lits, seqs))
    blocks += tail or []
    out = prefix_n + len(lits) + sum(ml for _, ml, _ in seqs) + sum(_block_out(b) for b in (tail or []))
    if window_log is None:
        return frame(blocks, out), out
    return frame(blocks, out, single_segment=False, window_log=window_log), out


def _block_out(b):
    if isinstance(b, S.Raw):
        return len(b.data)
    if isinstance(b, S.Rle):
        return b.n
    lits = b.literals[2] if isinstance(b.literals, tuple) else len(b.literals)
    return lits + sum(ml for _, ml, _ in b.seqs)


def text(n, seed=7, base_n=24 << 20):
    """n bytes of text: 1 MiB pieces of a 24 MiB synthetic text at random places, a byte in 4096 changed, so that matches
    reach back up to the whole output (far for a 2^27 window with long-distance matching, near for a 2^23 one)."""
    rng = np.random.default_rng(seed)
    base = np.frombuffer(W.synth_text(base_n, seed), dtype=np.uint8)
    out = np.empty(n, dtype=np.uint8)
    piece = 1 << 20
    for p in range(0, n, piece):
        m = min(piece, n - p)
        s = int(rng.integers(0, base_n - m))
        out[p:p + m] = base[s:s + m]
    flips = rng.integers(0, n, n >> 12)
    out[flips] ^= 0x20
    return out


def compress(data, window_log, ldm=False, level=1, content_size=True):
    """libzstd frame of a numpy array (checksum on)."""
    z = W.libzstd()
    cctx = z.ZSTD_createCCtx()
    try:
        # compressionLevel, windowLog, enableLongDistanceMatching, checksumFlag, contentSizeFlag
        for p, v in ((100, level), (101, window_log), (160, 1 if ldm else None), (201, 1), (200, None if content_size else 0)):
            if v is not None:
                assert not z.ZSTD_isError(z.ZSTD_CCtx_setParameter(cctx, p, v)), (p, v)
        bound = z.ZSTD_compressBound(data.size)
        buf = np.empty(bound, dtype=np.uint8)
        n = z.ZSTD_compress2(cctx, _ptr(buf), bound, _ptr(data), data.size)
        assert not z.ZSTD_isError(n)
        return buf[:n].tobytes()
    finally:
        z.ZSTD_freeCCtx(cctx)


class Case:
    def __init__(self, name, frame, out, gpu, cap=None, valid=True):
        self.name, self.frame, self.out, self.gpu, self.valid = name, frame, out, gpu, valid
        self.cap = out if cap is None else cap  # gpu: "exact" (libzstd's bytes), "oracle" (its status) or a status name


def seam_cases():
    """Offsets at the 2^28 - 1 seam.  `gpu` is what the decoder must report; "oracle" means exactly the oracle's result.
    A repeat code can only carry an offset of 2^28 - 1 or more into a later block after a direct one was coded, and that
    direct one is itself reported as CZS_UNSUPPORTED (far_then_repeat); the symbolic path beyond the seam is pinned with an
    offset just below the clamp (repeat_beyond_seam)."""
    off, rep, U = S.off, S.rep, "CZS_UNSUPPORTED"
    out = []

    def add(name, prefix, seqs, gpu, lits=b"", window_log=None, tail=None, cap_delta=0, valid=True):
        f, n = seq_frame(prefix, seqs, lits=lits, window_log=window_log, tail=tail)
        out.append(Case(name, f, n, gpu, cap=n + cap_delta, valid=valid))

    add("off_2^28-2_to_byte_0", M28 - 2, [(0, 64, off(M28 - 2))], "exact")
    add("off_2^28-2_after_2^28", M28, [(0, 64, off(M28 - 2))], "exact")
    add("far_2^28-1_at_2^28-1", CLAMP, [(0, 64, off(CLAMP))], U, window_log=29)           # valid: reaches byte 0
    add("far_2^28-1_wl29", M28 + (4 << 20), [(0, 64, off(CLAMP))], U, window_log=29)
    add("far_2^28+5_wl29", M28 + (4 << 20), [(0, 64, off(M28 + 5))], U, window_log=29)
    add("far_2^28+5_cap_short", M28 + (4 << 20), [(0, 64, off(M28 + 5))], U, window_log=29, cap_delta=-1)
    add("far_beyond_output", M28 + 16, [(0, 64, off(M28 + 1000))], U, window_log=29, valid=False)
    add("far_literal_overrun_first", M28 + 16, [(10, 64, off(M28 + 5))], "oracle", lits=b"abc", window_log=29, valid=False)
    add("far_2^28-1_at_2^28-2", CLAMP - 1, [(0, 64, off(CLAMP))], "oracle", window_log=29, valid=False)
    add("far_2^28+5_below_seam", M28 - 7, [(5, 64, off(M28 + 5))], "oracle", lits=b"hello", valid=False)
    add("far_2^28+5_small_window", 2 << 20, [(0, 64, off(M28 + 5))], "oracle", window_log=20, valid=False)
    add("repeat_beyond_seam", M28 - 2, [(0, 64, off(M28 - 2))], "exact",
        tail=[S.Rle(7, 1 << 17), S.Seqs(b"xy", [(2, 64, rep(1)), (0, 32, rep(3))])])
    add("far_then_repeat", M28 + 16, [(0, 64, off(M28 + 5))], U, window_log=29,
        tail=[S.Rle(7, 1 << 17), S.Seqs(b"xy", [(2, 64, rep(1))])])
    return out
