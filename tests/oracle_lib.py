"""ctypes binding of the CPU oracle (oracle/libzstd_oracle.so).

Test infrastructure only: imported by tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs.  Never by the product package.
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(os.path.dirname(_HERE), "oracle")
_LIB_PATH = os.path.join(ORACLE_DIR, "libzstd_oracle.so")

FLAG_NIBBLE_AS_WRITTEN = 1
FLAG_RESET_LIMIT = 2


class OracleResult(C.Structure):
    _fields_ = [
        ("status", C.c_int32),
        ("blocks_decoded", C.c_uint32),
        ("bytes_read", C.c_uint64),
        ("bytes_written", C.c_uint64),
        ("content_size", C.c_uint64),
        ("window_size", C.c_uint64),
        ("checksum_from_data", C.c_uint32),
        ("checksum_calculated", C.c_uint32),
        ("has_checksum", C.c_int32),
        ("finished", C.c_int32),
    ]


class DictInfo(C.Structure):
    _fields_ = [("id", C.c_uint32), ("huf_bytes", C.c_uint32), ("of_bytes", C.c_uint32), ("ml_bytes", C.c_uint32), ("ll_bytes", C.c_uint32),
                ("huf_max_bits", C.c_uint32), ("n_weights", C.c_uint32), ("of_log", C.c_uint32), ("ml_log", C.c_uint32),
                ("ll_log", C.c_uint32), ("offset_hist", C.c_uint32 * 3), ("table_hash", C.c_uint32), ("content_off", C.c_uint64),
                ("content_len", C.c_uint64)]


class BlockTrace(C.Structure):
    _fields_ = [
        ("block_type", C.c_uint8),
        ("lit_type", C.c_uint8),
        ("n_streams", C.c_uint8),
        ("modes", C.c_uint8),
        ("regen_size", C.c_uint32),
        ("n_seq", C.c_uint32),
        ("out_bytes", C.c_uint32),
        ("lit_off", C.c_uint64),
        ("seq_off", C.c_uint64),
    ]


class Trace(C.Structure):
    _fields_ = [
        ("blocks", C.POINTER(BlockTrace)),
        ("n_blocks", C.c_size_t),
        ("cap_blocks", C.c_size_t),
        ("lits", C.POINTER(C.c_uint8)),
        ("n_lits", C.c_size_t),
        ("cap_lits", C.c_size_t),
        ("seqs", C.POINTER(C.c_uint32)),
        ("n_seqs", C.c_size_t),
        ("cap_seqs", C.c_size_t),
    ]


def build(force=False):
    """Compile the oracle with gcc if the .so is missing or stale."""
    srcs = [os.path.join(ORACLE_DIR, f) for f in ("zstd_oracle.c", "zstd_oracle.h")]
    stale = (not os.path.exists(_LIB_PATH)) or any(
        os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in srcs
    )
    if force or stale:
        subprocess.check_call(["make", "-C", ORACLE_DIR, "-s"])
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB_PATH)
        u8p = C.POINTER(C.c_uint8)
        L.oracle_decode_frame.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_uint32,
                                          C.POINTER(OracleResult), C.POINTER(Trace)]
        L.oracle_decode_frame.restype = C.c_int
        L.oracle_decode_batch.argtypes = [C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                          C.POINTER(OracleResult), C.c_int]
        L.oracle_decode_batch.restype = C.c_int
        L.oracle_trace_free.argtypes = [C.POINTER(Trace)]
        L.oracle_xxh64.argtypes = [C.c_char_p, C.c_size_t, C.c_uint64]
        L.oracle_xxh64.restype = C.c_uint64
        L.oracle_xxh64_chunked.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t), C.c_size_t]
        L.oracle_xxh64_chunked.restype = C.c_uint64
        L.oracle_bitreader_reverse.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t,
                                               C.POINTER(C.c_uint64), C.POINTER(C.c_int64)]
        L.oracle_bitreader_forward.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.POINTER(C.c_uint64)]
        L.oracle_fse_predefined.argtypes = [C.c_int, C.POINTER(C.c_uint32), u8p, u8p, C.POINTER(C.c_uint32)]
        L.oracle_fse_build_from_probs.argtypes = [C.c_uint8, C.POINTER(C.c_int32), C.c_size_t,
                                                  C.POINTER(C.c_uint32), u8p, u8p]
        L.oracle_fse_build_decoder.argtypes = [C.c_char_p, C.c_size_t, C.c_uint8, C.POINTER(C.c_uint32), u8p, u8p,
                                               C.POINTER(C.c_uint32), C.POINTER(C.c_size_t)]
        L.oracle_huf_build_decoder.argtypes = [C.c_char_p, C.c_size_t, C.c_uint32, u8p, u8p, C.POINTER(C.c_uint32),
                                               C.POINTER(C.c_size_t), u8p, C.POINTER(C.c_uint32)]
        L.oracle_offset_history.argtypes = [C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32)]
        L.oracle_offset_history.restype = C.c_uint32
        L.oracle_dict_decode.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(DictInfo)]
        L.oracle_fd_new.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t), C.c_uint32, C.POINTER(C.c_int32)]
        L.oracle_fd_new.restype = C.c_void_p
        L.oracle_fd_reset.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.oracle_fd_reset.restype = C.c_int32
        L.oracle_fd_free.argtypes = [C.c_void_p]
        L.oracle_fd_decode_blocks.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t), C.c_int,
                                              C.c_uint32, C.POINTER(C.c_int32)]
        L.oracle_fd_decode_blocks.restype = C.c_int32
        L.oracle_fd_collect.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.oracle_fd_collect.restype = C.c_int
        L.oracle_fd_can_collect.argtypes = [C.c_void_p]
        L.oracle_fd_can_collect.restype = C.c_size_t
        L.oracle_fd_read.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.oracle_fd_read.restype = C.c_size_t
        L.oracle_fd_decode_from_to.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                               C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
        L.oracle_fd_decode_from_to.restype = C.c_int32
        L.oracle_fd_getters.argtypes = [C.c_void_p, C.POINTER(OracleResult)]
        L.oracle_fd_buffer_state.argtypes = [C.c_void_p, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
        _lib = L
    return _lib


def decode_frame(src: bytes, dst_cap: int = None, flags: int = 0, trace: bool = False):
    """_test_decode equivalent.  Returns (status, output bytes, OracleResult[, trace dict])."""
    L = lib()
    if dst_cap is None:
        dst_cap = max(1 << 16, 64 * len(src))
    dst = C.create_string_buffer(max(dst_cap, 1))
    res = OracleResult()
    tr = Trace() if trace else None
    st = L.oracle_decode_frame(src, len(src), dst, dst_cap, flags, C.byref(res), C.byref(tr) if trace else None)
    out = dst.raw[: res.bytes_written] if st == 0 else b""
    if not trace:
        return st, out, res
    blocks = []
    for i in range(tr.n_blocks):
        b = tr.blocks[i]
        nxt_lit = tr.blocks[i + 1].lit_off if i + 1 < tr.n_blocks else tr.n_lits
        nxt_seq = tr.blocks[i + 1].seq_off if i + 1 < tr.n_blocks else tr.n_seqs
        blocks.append(dict(
            block_type=b.block_type, lit_type=b.lit_type, n_streams=b.n_streams, modes=b.modes,
            regen_size=b.regen_size, n_seq=b.n_seq, out_bytes=b.out_bytes,
            lits=bytes(bytearray(tr.lits[b.lit_off:nxt_lit])) if nxt_lit > b.lit_off else b"",
            seqs=[tuple(tr.seqs[(b.seq_off + k) * 4 + j] for j in range(4)) for k in range(nxt_seq - b.seq_off)],
        ))
    L.oracle_trace_free(C.byref(tr))
    return st, out, res, blocks


def decode_batch(frames, dst_caps, n_threads=1, flags=0):
    """Decode a list of bytes objects; returns (outputs, results, failures)."""
    L = lib()
    n = len(frames)
    srcs = (C.c_char_p * n)(*frames)
    lens = (C.c_size_t * n)(*[len(f) for f in frames])
    bufs = [C.create_string_buffer(max(c, 1)) for c in dst_caps]
    dsts = (C.c_void_p * n)(*[C.addressof(b) for b in bufs])
    caps = (C.c_size_t * n)(*dst_caps)
    results = (OracleResult * n)()
    fails = L.oracle_decode_batch(n, srcs, lens, dsts, caps, flags, results, n_threads)
    outs = [bufs[i].raw[: results[i].bytes_written] if results[i].status == 0 else b"" for i in range(n)]
    return outs, results, fails
