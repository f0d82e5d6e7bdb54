"""ctypes binding of include/cairo_zstd_b200.h (libcairo_zstd_b200.so)."""
import ctypes as C
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("CZB_LIB") or os.path.join(_HERE, "libcairo_zstd_b200.so")  # CZB_LIB: a variant build, for A/B measurements
_INCLUDE = os.path.join(os.path.dirname(_HERE), "include")

FLAG_VERIFY_CHECKSUM = 1
MAX_FRAME_OUTPUT = (1 << 31) - 1  # CZB_MAX_FRAME_OUTPUT: larger frames get CZS_UNSUPPORTED (CZS_DST_TOO_SMALL below that dst_cap)


class CzbError(RuntimeError):
    pass


class FrameDesc(C.Structure):
    _fields_ = [("src", C.c_void_p), ("src_len", C.c_uint64), ("dst", C.c_void_p), ("dst_cap", C.c_uint64)]


class FrameResult(C.Structure):
    _fields_ = [
        ("status", C.c_int32), ("blocks_decoded", C.c_uint32), ("bytes_read", C.c_uint64), ("bytes_written", C.c_uint64),
        ("content_size", C.c_uint64), ("window_size", C.c_uint64), ("checksum_from_data", C.c_uint32),
        ("checksum_calculated", C.c_uint32), ("has_checksum", C.c_int32), ("finished", C.c_int32),
    ]


class FrameHeaderInfo(C.Structure):
    _fields_ = [
        ("status", C.c_int32), ("header_len", C.c_uint32), ("content_size", C.c_uint64), ("window_size", C.c_uint64),
        ("fcs_present", C.c_int32), ("has_checksum_flag", C.c_int32), ("single_segment", C.c_int32), ("dict_id", C.c_uint32),
    ]


class FrameSpan(C.Structure):
    _fields_ = [("offset", C.c_uint64), ("length", C.c_uint64), ("content_size", C.c_uint64), ("window_size", C.c_uint64),
                ("fcs_present", C.c_int32), ("has_checksum_flag", C.c_int32)]


class ShardStat(C.Structure):
    _fields_ = [("device", C.c_int32), ("pad", C.c_uint32), ("frames", C.c_uint64), ("bytes_in", C.c_uint64),
                ("bytes_out", C.c_uint64), ("ms", C.c_double)]


class DictionaryInfo(C.Structure):
    _fields_ = [("status", C.c_int32), ("id", C.c_uint32), ("huf_bytes", C.c_uint32), ("of_bytes", C.c_uint32), ("ml_bytes", C.c_uint32),
                ("ll_bytes", C.c_uint32), ("huf_max_bits", C.c_uint32), ("n_weights", C.c_uint32), ("of_log", C.c_uint32),
                ("ml_log", C.c_uint32), ("ll_log", C.c_uint32), ("offset_hist", C.c_uint32 * 3), ("table_hash", C.c_uint32),
                ("content_off", C.c_uint64), ("content_len", C.c_uint64)]


class DebugBlock(C.Structure):
    _fields_ = [
        ("frame", C.c_uint32), ("block_type", C.c_uint8), ("lit_type", C.c_uint8), ("n_streams", C.c_uint8), ("modes", C.c_uint8),
        ("regen_size", C.c_uint32), ("n_seq", C.c_uint32), ("status", C.c_int32), ("lit_off", C.c_uint64), ("seq_off", C.c_uint64),
    ]


class DebugWaveTotals(C.Structure):
    _fields_ = [("n_blocks", C.c_uint64), ("lit_bytes", C.c_uint64), ("n_seq", C.c_uint64), ("n_huf", C.c_uint64),
                ("n_fse", C.c_uint64), ("src_bytes", C.c_uint64), ("frame_cls", C.c_uint32 * 32), ("fse_cls", C.c_uint32 * 32)]


def _parse_status_names():
    names = {}
    try:
        text = open(os.path.join(_INCLUDE, "czstd_status.h")).read()
        for m in re.finditer(r"\b(CZS_[A-Z0-9_]+)\s*=\s*(\d+)", text):
            names[int(m.group(2))] = m.group(1)
    except OSError:
        pass
    return names


STATUS_NAMES = _parse_status_names()


def status_name(s):
    return STATUS_NAMES.get(int(s), f"CZS_UNKNOWN({s})")


# every symbol include/cairo_zstd_b200.h declares (checked by tests/test_abi.py)
EXPORTS = [
    "czb_abi_version", "czb_context_create", "czb_context_destroy", "czb_last_error", "czb_decode_batch_device",
    "czb_decode_batch_host", "czb_decode_batch_host_packed", "czb_frame_header_info_host", "czb_find_frame_end_host",
    "czb_fd_new", "czb_fd_reset", "czb_fd_free", "czb_fd_decode_blocks", "czb_fd_collect", "czb_fd_can_collect",
    "czb_fd_decode_from_to", "czb_fd_read", "czb_fd_content_size", "czb_fd_get_checksum_from_data",
    "czb_fd_get_calculated_checksum", "czb_fd_bytes_read_from_source", "czb_fd_is_finished", "czb_fd_blocks_decoded",
    "czb_debug_last_wave_counts", "czb_debug_copy_blocks", "czb_debug_copy_literals", "czb_debug_copy_sequences",
    "czb_kernel_launches", "czb_profile_enable", "czb_profile_collect", "czs_status_name",
    "czb_split_frames_host", "czb_split_frames_device", "czb_frame_sizes_device", "czb_frame_sizes_host",
    "czb_dictionary_parse_host", "czb_plan_batch_device", "czb_plan_destroy", "czb_decode_batch_device_planned", "czb_debug_fd_device_work", "czb_debug_guard_faults", "czb_debug_flow_watchdog", "czb_debug_plan_waves", "czb_partition_frames", "czb_multi_create", "czb_multi_destroy", "czb_decode_batch_multi", "czb_multi_last_error",
    "czb_verify_batch_device",
]

_lib = None


def load_library():
    """Load the CUDA library.  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise CzbError(f"{_LIB_PATH} is missing: run `python -m cairo_zstd_b200.build` (needs nvcc); "
                       "there is no CPU fallback")
    L = C.CDLL(_LIB_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32
    P = C.POINTER
    L.czb_abi_version.restype = C.c_int
    L.czb_context_create.argtypes = [C.c_int, u64, P(vp)]
    L.czb_context_destroy.argtypes = [vp]
    L.czb_last_error.argtypes = [vp]
    L.czb_last_error.restype = C.c_char_p
    L.czb_decode_batch_device.argtypes = [vp, vp, vp, u64, u32, vp]
    L.czb_verify_batch_device.argtypes = [vp, vp, vp, u64, vp]
    L.czb_decode_batch_host.argtypes = [vp, P(FrameDesc), P(FrameResult), u64, u32]
    L.czb_decode_batch_host_packed.argtypes = [vp, vp, vp, vp, vp, vp, u64, u32]
    L.czb_frame_header_info_host.argtypes = [C.c_char_p, u64, P(FrameHeaderInfo)]
    L.czb_find_frame_end_host.argtypes = [C.c_char_p, u64, P(u64)]
    L.czb_fd_new.argtypes = [vp, C.c_char_p, u64, P(u64), P(vp)]
    L.czb_fd_reset.argtypes = [vp, C.c_char_p, u64, P(u64)]
    L.czb_fd_free.argtypes = [vp]
    L.czb_fd_decode_blocks.argtypes = [vp, C.c_char_p, u64, P(u64), C.c_int, u32, P(i32)]
    L.czb_fd_collect.argtypes = [vp, vp, u64, P(u64)]
    L.czb_fd_can_collect.argtypes = [vp]
    L.czb_fd_can_collect.restype = u64
    L.czb_fd_decode_from_to.argtypes = [vp, C.c_char_p, u64, vp, u64, P(u64), P(u64)]
    L.czb_fd_read.argtypes = [vp, vp, u64]
    L.czb_fd_read.restype = C.c_int64
    L.czb_fd_content_size.argtypes = [vp]
    L.czb_fd_content_size.restype = u64
    L.czb_fd_get_checksum_from_data.argtypes = [vp, P(u32)]
    L.czb_fd_get_calculated_checksum.argtypes = [vp, P(u32)]
    L.czb_fd_bytes_read_from_source.argtypes = [vp]
    L.czb_fd_bytes_read_from_source.restype = u64
    L.czb_fd_is_finished.argtypes = [vp]
    L.czb_fd_blocks_decoded.argtypes = [vp]
    L.czb_fd_blocks_decoded.restype = u32
    L.czb_debug_last_wave_counts.argtypes = [vp, P(u64), P(u64), P(u64)]
    L.czb_debug_copy_blocks.argtypes = [vp, P(DebugBlock), u64]
    L.czb_debug_copy_literals.argtypes = [vp, vp, u64]
    L.czb_debug_copy_sequences.argtypes = [vp, vp, u64]
    L.czb_kernel_launches.argtypes = [vp]
    L.czb_kernel_launches.restype = u64
    L.czb_profile_enable.argtypes = [vp, C.c_int]
    L.czb_profile_collect.argtypes = [vp, P(C.c_double), P(u64)]
    L.czb_dictionary_parse_host.argtypes = [vp, C.c_char_p, u64, P(DictionaryInfo)]
    L.czb_plan_batch_device.argtypes = [vp, vp, u64, vp, P(vp)]
    L.czb_plan_destroy.argtypes = [vp]
    L.czb_decode_batch_device_planned.argtypes = [vp, vp, vp, vp, u64, u32, vp]
    L.czb_debug_fd_device_work.argtypes = [vp, P(u64), P(u64)]
    L.czb_debug_flow_watchdog.argtypes = [P(u32)]
    L.czb_debug_guard_faults.argtypes = [vp, P(u64)]
    L.czb_debug_plan_waves.argtypes = [vp, P(u64), P(u64), P(DebugWaveTotals), u64]
    L.czb_split_frames_host.argtypes = [C.c_char_p, u64, P(FrameSpan), u64, P(u64), P(u64), P(u64)]
    L.czb_split_frames_device.argtypes = [vp, vp, u64, vp, u64, vp, vp]
    L.czb_frame_sizes_device.argtypes = [vp, vp, vp, u64, vp]
    L.czb_frame_sizes_host.argtypes = [vp, P(FrameDesc), P(FrameResult), u64]
    L.czb_partition_frames.argtypes = [P(u64), u64, u32, P(u32), P(u64)]
    L.czb_multi_create.argtypes = [P(C.c_int), C.c_int, u64, P(vp)]
    L.czb_multi_destroy.argtypes = [vp]
    L.czb_decode_batch_multi.argtypes = [vp, P(FrameDesc), P(FrameResult), u64, u32, P(ShardStat)]
    L.czb_multi_last_error.argtypes = [vp, C.c_int]
    L.czb_multi_last_error.restype = C.c_char_p
    L.czs_status_name.argtypes = [C.c_int]
    L.czs_status_name.restype = C.c_char_p
    _lib = L
    return L


def frame_header_info(frame: bytes) -> FrameHeaderInfo:
    info = FrameHeaderInfo()
    load_library().czb_frame_header_info_host(frame, len(frame), C.byref(info))
    return info


def find_frame_end(data: bytes):
    n = C.c_uint64()
    st = load_library().czb_find_frame_end_host(data, len(data), C.byref(n))
    return st, n.value


def split_frames(buf: bytes, cap: int = None):
    """czb_split_frames_host: returns (status, [FrameSpan], n_skipped, consumed)."""
    L = load_library()
    cap = cap if cap is not None else max(1, len(buf) // 9 + 1)
    spans = (FrameSpan * cap)()
    n, sk, used = C.c_uint64(), C.c_uint64(), C.c_uint64()
    st = L.czb_split_frames_host(buf, len(buf), spans, cap, C.byref(n), C.byref(sk), C.byref(used))
    return st, [spans[i] for i in range(n.value)], sk.value, used.value


def partition_frames(costs, n_shards: int):
    """czb_partition_frames: greedy largest-first; returns (shard_of list, shard_load list)."""
    L = load_library()
    n = len(costs)
    c = (C.c_uint64 * max(n, 1))(*[int(x) for x in costs])
    so = (C.c_uint32 * max(n, 1))()
    load = (C.c_uint64 * n_shards)()
    rc = L.czb_partition_frames(c, n, n_shards, so, load)
    if rc != 0:
        raise CzbError(status_name(rc))
    return list(so[:n]), list(load)


class MultiContext:
    """czb_multi: one host batch decoded over several GPUs of this process (czb_decode_batch_multi)."""

    def __init__(self, devices, workspace_budget_bytes: int = 0):
        self._L = load_library()
        h = C.c_void_p()
        arr = (C.c_int * len(devices))(*devices)
        rc = self._L.czb_multi_create(arr, len(devices), workspace_budget_bytes, C.byref(h))
        if rc != 0:
            raise CzbError(f"czb_multi_create failed: {status_name(rc)}")
        self._h, self.devices = h, list(devices)

    def close(self):
        if getattr(self, "_h", None):
            self._L.czb_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def decode_batch(self, frames, dst_caps, flags: int = 0):
        n = len(frames)
        descs = (FrameDesc * n)()
        results = (FrameResult * n)()
        stats = (ShardStat * len(self.devices))()
        keep = []
        for i, (f, cap) in enumerate(zip(frames, dst_caps)):
            sb = C.create_string_buffer(f, len(f)) if len(f) else C.create_string_buffer(1)
            db = C.create_string_buffer(max(int(cap), 1))
            keep.append((sb, db))
            descs[i].src, descs[i].src_len, descs[i].dst, descs[i].dst_cap = C.addressof(sb), len(f), C.addressof(db), int(cap)
        rc = self._L.czb_decode_batch_multi(self._h, descs, results, n, flags, stats)
        if rc != 0:
            raise CzbError(status_name(rc))
        outs = [keep[i][1].raw[: results[i].bytes_written] if results[i].status == 0 else None for i in range(n)]
        return outs, results, list(stats)


class Context:
    """One decoder context on one CUDA device (czb_context)."""

    def __init__(self, device: int = 0, workspace_budget_bytes: int = 0):
        self._L = load_library()
        h = C.c_void_p()
        rc = self._L.czb_context_create(device, workspace_budget_bytes, C.byref(h))
        if rc != 0:
            raise CzbError(f"czb_context_create failed: {status_name(rc)} (is a CUDA device visible?)")
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            self._L.czb_context_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def last_error(self) -> str:
        return (self._L.czb_last_error(self._h) or b"").decode()

    def kernel_launches(self) -> int:
        return self._L.czb_kernel_launches(self._h)

    def _check(self, rc):
        if rc != 0:
            raise CzbError(f"{status_name(rc)}: {self.last_error()}")

    # ---- hot path, device-resident ----
    def decode_batch_device(self, descs_ptr: int, results_ptr: int, n: int, flags: int = 0, stream: int = 0):
        """descs_ptr/results_ptr: device addresses of czb_frame_desc[n] / czb_frame_result[n]."""
        self._check(self._L.czb_decode_batch_device(self._h, descs_ptr, results_ptr, n, flags, stream))

    def verify_batch_device(self, descs_ptr: int, results_ptr: int, n: int, stream: int = 0):
        """czb_verify_batch_device: decode into the context's scratch, XXH64 each output, keep only the results.
        descs_ptr/results_ptr: device addresses of czb_frame_desc[n] / czb_frame_result[n]; dst / dst_cap are ignored."""
        self._check(self._L.czb_verify_batch_device(self._h, descs_ptr, results_ptr, n, stream))

    def plan_batch_device(self, descs_ptr: int, n: int, stream: int = 0):
        """czb_plan_batch_device: returns an opaque plan handle (free with plan_destroy)."""
        h = C.c_void_p()
        self._check(self._L.czb_plan_batch_device(self._h, descs_ptr, n, stream, C.byref(h)))
        return h

    def plan_destroy(self, plan):
        self._L.czb_plan_destroy(plan)

    def decode_batch_device_planned(self, plan, descs_ptr: int, results_ptr: int, n: int, flags: int = 0, stream: int = 0):
        """No host synchronisation: every kernel is only enqueued (can be captured into a CUDA graph)."""
        self._check(self._L.czb_decode_batch_device_planned(self._h, plan, descs_ptr, results_ptr, n, flags, stream))

    # ---- host-pointer forms ----
    def decode_batch(self, frames, dst_caps, flags: int = 0):
        """frames: list of bytes; returns (list of output bytes or None, FrameResult array)."""
        n = len(frames)
        descs = (FrameDesc * n)()
        results = (FrameResult * n)()
        keep = []
        for i, (f, cap) in enumerate(zip(frames, dst_caps)):
            sb = C.create_string_buffer(f, len(f)) if len(f) else C.create_string_buffer(1)
            db = C.create_string_buffer(max(int(cap), 1))
            keep.append((sb, db))
            descs[i].src = C.addressof(sb)
            descs[i].src_len = len(f)
            descs[i].dst = C.addressof(db)
            descs[i].dst_cap = int(cap)
        self._check(self._L.czb_decode_batch_host(self._h, descs, results, n, flags))
        outs = [keep[i][1].raw[: results[i].bytes_written] if results[i].status == 0 else None for i in range(n)]
        return outs, results

    def decode_batch_packed(self, src_base: int, src_off, dst_base: int, dst_off, n: int, results_ptr: int, flags: int = 0):
        """Raw-pointer form: src_off/dst_off are ctypes/numpy uint64 arrays of n+1 entries (host)."""
        so = src_off.ctypes.data if hasattr(src_off, "ctypes") else C.addressof(src_off)
        do = dst_off.ctypes.data if hasattr(dst_off, "ctypes") else C.addressof(dst_off)
        self._check(self._L.czb_decode_batch_host_packed(self._h, src_base, so, dst_base, do, results_ptr, n, flags))

    def dictionary_parse(self, dict_bytes: bytes) -> DictionaryInfo:
        """czb_dictionary_parse_host: Dictionary::decode_dict (dictionary.cairo:35-90) on the device; status inside."""
        info = DictionaryInfo()
        self._L.czb_dictionary_parse_host(self._h, dict_bytes, len(dict_bytes), C.byref(info))
        return info

    def guard_faults(self) -> int:
        """CZB_GUARD=1 contexts: guard bytes behind the scratch buffers found overwritten so far (0 = clean)."""
        v = C.c_uint64()
        self._check(self._L.czb_debug_guard_faults(self._h, C.byref(v)))
        return v.value

    # ---- per-kernel timing ----
    KERNEL_CLASSES = ["scan", "fill", "huff", "fse", "exec", "xxh64", "header_results", "frame_sizes"]

    def frame_sizes(self, frames):
        """czb_frame_sizes_host: exact decoded size of every frame without executing it."""
        n = len(frames)
        descs = (FrameDesc * n)()
        results = (FrameResult * n)()
        keep = []
        for i, f in enumerate(frames):
            sb = C.create_string_buffer(f, len(f)) if len(f) else C.create_string_buffer(1)
            keep.append(sb)
            descs[i].src, descs[i].src_len = C.addressof(sb), len(f)
        self._check(self._L.czb_frame_sizes_host(self._h, descs, results, n))
        return results

    def profile_enable(self, on=True):
        self._check(self._L.czb_profile_enable(self._h, 1 if on else 0))

    def profile_collect(self):
        """Returns {class: (ms, launches)} accumulated since the last collect."""
        ms = (C.c_double * 8)()
        n = (C.c_uint64 * 8)()
        self._check(self._L.czb_profile_collect(self._h, ms, n))
        return {k: (ms[i], n[i]) for i, k in enumerate(self.KERNEL_CLASSES) if n[i]}

    # ---- debug taps ----
    def plan_waves(self, plan):
        """czb_debug_plan_waves: (frames per wave, [DebugWaveTotals] of every wave) of a plan from plan_batch_device."""
        w, nw = C.c_uint64(), C.c_uint64()
        self._check(self._L.czb_debug_plan_waves(plan, C.byref(w), C.byref(nw), None, 0))
        out = (DebugWaveTotals * max(nw.value, 1))()
        self._check(self._L.czb_debug_plan_waves(plan, None, None, out, nw.value))
        return w.value, [out[i] for i in range(nw.value)]

    def debug_last_wave(self):
        nb, lb, ns = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._L.czb_debug_last_wave_counts(self._h, C.byref(nb), C.byref(lb), C.byref(ns))
        blocks = (DebugBlock * max(nb.value, 1))()
        self._check(self._L.czb_debug_copy_blocks(self._h, blocks, nb.value))
        lits = C.create_string_buffer(max(lb.value, 1))
        self._check(self._L.czb_debug_copy_literals(self._h, lits, lb.value))
        seqs = (C.c_uint32 * max(3 * ns.value, 1))()
        self._check(self._L.czb_debug_copy_sequences(self._h, seqs, ns.value))
        return [blocks[i] for i in range(nb.value)], lits.raw[: lb.value], list(seqs[: 3 * ns.value])
