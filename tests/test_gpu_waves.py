"""-m gpu: batches split into many waves.

A batch call cuts its frames into waves of W frames; every wave gets its own scan totals, work lists, scratch offsets,
executor choice and checksum launch, and the kernels see frame indices relative to the wave.  W comes from
CZB_WAVE_FRAMES (rounded up to a multiple of 128), from the doubling that keeps the call at most 4096 waves, or from the
budget retry that halves W until a wave's scratch fits.  These tests decode batches that cross wave boundaries on purpose:
every frame kind on every seam, a different sequence executor in each wave, the budget retry, the two-stream overlap
(CZB_OVERLAP=1) with scratch guards, planned and graph-captured calls, back-to-back calls on two streams, 2049 waves of
tiny frames and the packed host path with several waves per chunk.

Every result field is compared with the oracle's (cached per distinct frame and capacity, so replicated frames cost
nothing), and outputs are compared with the same batch decoded in one wave.  czb_debug_plan_waves exposes a plan's wave
split, which is checked against totals computed on the CPU from the oracle's block trace."""
import ctypes as C
import struct

import numpy as np
import pytest

import handmade as H
import fsefamilies as X
import huffamilies as HF
import oracle_lib as O
import seqbuild as S
import seqfamilies as F
import cairo_zstd_b200 as czb
from cairo_zstd_b200 import api, workloads as WL
from seqbuild import Raw, Rle

pytestmark = pytest.mark.gpu

VERIFY = api.FLAG_VERIFY_CHECKSUM
PAT = 0xA5
GAP = 64
MODES = {   # the executor modes of test_gpu_seams.py
    "default": {},
    "flow-narrow": {"CZB_BIG_CLS": "0", "CZB_BIG_SEQ_BYTES": "0"},
    "flow-wide": {"CZB_BIG_CLS": "0", "CZB_BIG_SEQ_BYTES": "0", "CZB_FLOW_WIDE": "1"},
    "big": {"CZB_BIG_CLS": "0", "CZB_BIG_SEQ_BYTES": "0", "CZB_BIG_FLOW": "0"},
}
KNOBS = ("CZB_WAVE_FRAMES", "CZB_BUDGET_GB", "CZB_OVERLAP", "CZB_HOST_CHUNK_MB", "CZB_GUARD", "CZB_FLOW_WIDE", "CZB_BIG_FLOW",
         "CZB_BIG_CLS", "CZB_BIG_SEQ_BYTES", "CZB_SHARE_CLS", "CZB_BIG_SHARE", "CZB_FLOW_MAX")
KINDS = ["corpus", "seq", "seq-bad", "huf", "huf-bad", "weight", "synth", "mutant", "trunc", "header", "raw", "rle"]
LARGE = 1 << 15     # 2^share_cls: from this compressed size on a frame may get a CTA of its own


def _context(monkeypatch, env=None, budget=0):
    """A context created with exactly these knobs set (knobs are read at creation; every other knob is unset)."""
    with monkeypatch.context() as m:
        for k in KNOBS:
            m.delenv(k, raising=False)
        for k, v in (env or {}).items():
            m.setenv(k, v)
        return czb.Context(0, budget)


def _watchdog_clear():
    wd = (C.c_uint32 * 16)()
    czb.load_library().czb_debug_flow_watchdog(wd)
    assert wd[0] == 0, list(wd)


def size_class(v):
    c = 0
    while v > 1 and c < 31:
        v >>= 1
        c += 1
    return c


# ---------------------------------------------------------------------------------------------------------------------
# oracle, cached per (frame, capacity)
# ---------------------------------------------------------------------------------------------------------------------
_ORACLE = {}
FIELDS = ("bytes_written", "bytes_read", "blocks_decoded", "content_size", "window_size", "checksum_from_data",
          "checksum_calculated", "finished")


def oracle(frame, cap):
    key = (frame, cap)
    if key not in _ORACLE:
        st, out, r = O.decode_frame(frame, dst_cap=cap)
        _ORACLE[key] = (st, out, {f: getattr(r, f) for f in FIELDS}, bool(r.has_checksum))
    return _ORACLE[key]


def check(frames, caps, outs, res, label, ref=None):
    """Every result field equal to the oracle's; with ref = (outs, results) of the same batch decoded in one wave: valid
    frames byte-identical to it (output and the whole result record), failing frames with the same status."""
    for i, (f, cap) in enumerate(zip(frames, caps)):
        st, want, fields, has_ck = oracle(f, cap)
        r = res[i]
        tag = f"{label}[{i}] gpu={czb.status_name(r.status)} oracle={czb.status_name(st)}"
        if st == 0:
            assert r.status == 0, tag
            assert outs[i] == want, f"{tag}: output differs"
            for k in FIELDS:
                assert getattr(r, k) == fields[k], f"{tag}: {k} {getattr(r, k)} != {fields[k]}"
            assert bool(r.has_checksum) == has_ck and r.finished == 1, tag
        else:
            assert r.status == st, tag
        if ref is not None:
            if st == 0:
                assert outs[i] == ref[0][i] and bytes(r) == bytes(ref[1][i]), f"{tag}: differs from the single-wave decode"
            else:
                assert r.status == ref[1][i].status, f"{tag}: single-wave status {czb.status_name(ref[1][i].status)}"


# ---------------------------------------------------------------------------------------------------------------------
# device-resident batches
# ---------------------------------------------------------------------------------------------------------------------
class DevBatch:
    """Frames and outputs in device memory, descriptors and results too.  gaps=True: output spans with exact capacities,
    64-byte gaps at odd alignments between them, all filled with a pattern that must survive the decode."""

    def __init__(self, frames, caps, gaps=False):
        import torch
        self.frames, self.caps, self.n, self.gaps = list(frames), [int(c) for c in caps], len(frames), gaps
        n, dev = self.n, torch.device("cuda", 0)
        flens = np.array([len(f) for f in self.frames], dtype=np.int64)
        soff = np.concatenate([[0], np.cumsum((flens + 15) & ~15)])
        src_h = np.zeros(int(soff[-1]) + 16, dtype=np.uint8)
        for i, f in enumerate(self.frames):
            src_h[soff[i]:soff[i] + len(f)] = np.frombuffer(f, dtype=np.uint8)
        self.src = torch.from_numpy(src_h).to(dev)
        caps_a = np.array(self.caps, dtype=np.int64)
        if gaps:
            self.starts = GAP + np.concatenate([[0], np.cumsum(caps_a + GAP + np.arange(n) % 7)[:-1]])
            end = int(self.starts[-1] + caps_a[-1]) + GAP
        else:
            self.starts = np.concatenate([[0], np.cumsum((caps_a + 15) & ~15)[:-1]])
            end = int(self.starts[-1] + caps_a[-1]) + 64
        self.dst = torch.empty(end, dtype=torch.uint8, device=dev)
        d = np.zeros((n, 4), dtype=np.uint64)
        d[:, 0] = self.src.data_ptr() + soff[:-1]
        d[:, 1] = flens
        d[:, 2] = self.dst.data_ptr() + self.starts
        d[:, 3] = caps_a
        self.descs = torch.from_numpy(d.view(np.uint8).reshape(-1)).to(dev)
        self.results = torch.empty(n * C.sizeof(api.FrameResult), dtype=torch.uint8, device=dev)
        self.reset()

    def reset(self):
        self.dst.fill_(PAT if self.gaps else 0)
        self.results.zero_()

    def decode(self, ctx, stream, flags=VERIFY):
        ctx.decode_batch_device(self.descs.data_ptr(), self.results.data_ptr(), self.n, flags, stream)

    def plan(self, ctx, stream):
        return ctx.plan_batch_device(self.descs.data_ptr(), self.n, stream)

    def decode_planned(self, ctx, plan, stream, flags=VERIFY):
        ctx.decode_batch_device_planned(plan, self.descs.data_ptr(), self.results.data_ptr(), self.n, flags, stream)

    def fetch(self):
        """(outputs, results, raw results bytes, whole output buffer) after a device-wide synchronisation."""
        import torch
        torch.cuda.synchronize()
        raw = self.results.cpu().numpy().tobytes()
        res = (api.FrameResult * self.n).from_buffer_copy(raw)
        out = self.dst.cpu().numpy()
        outs = [out[s:s + r.bytes_written].tobytes() if r.status == 0 else None for s, r in zip(self.starts, res)]
        return outs, res, raw, out

    def spans_intact(self, out):
        mask = np.ones(out.size, dtype=bool)
        for s, c in zip(self.starts, self.caps):
            mask[s:s + c] = False
        return int((out[mask] != PAT).sum())


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def decode(ctx, frames, caps, label, ref_ctx=None, gaps=False):
    """Decode through the device entry point, check against the oracle and (ref_ctx) against the single-wave decode."""
    b = DevBatch(frames, caps, gaps=gaps)
    ref = None
    if ref_ctx is not None:
        b.decode(ref_ctx, _stream())
        ref = b.fetch()[:2]
        b.reset()
    b.decode(ctx, _stream())
    outs, res, _, out = b.fetch()
    check(frames, caps, outs, res, label, ref)
    if gaps:
        assert b.spans_intact(out) == 0, f"{label}: bytes outside the frames' spans were overwritten"
    return b


def plan_waves(ctx, frames, caps):
    b = DevBatch(frames, caps)
    plan = b.plan(ctx, _stream())
    try:
        return ctx.plan_waves(plan)
    finally:
        ctx.plan_destroy(plan)


# ---------------------------------------------------------------------------------------------------------------------
# the frame pool
# ---------------------------------------------------------------------------------------------------------------------
class Pool:
    def __init__(self):
        self.frames, self.caps, self.kinds = [], [], []
        self.scan = {}      # index of a valid frame -> what k_scan_frames counts for it, from the oracle's block trace

    def add(self, kind, frames, caps):
        for f, c in zip(frames, caps):
            self.frames.append(bytes(f)); self.caps.append(int(c)); self.kinds.append(kind)

    def finish(self):
        self.by_kind = {k: [i for i, kk in enumerate(self.kinds) if kk == k] for k in KINDS}
        assert all(self.by_kind[k] for k in KINDS), {k: len(v) for k, v in self.by_kind.items()}
        self.valid = [i for i in range(len(self.frames)) if oracle(self.frames[i], self.caps[i])[0] == 0]
        for k in ("seq-bad", "huf-bad", "header"):
            assert all(oracle(self.frames[i], self.caps[i])[0] != 0 for i in self.by_kind[k]), k
        assert all(czb.frame_header_info(self.frames[i]).status != 0 for i in self.by_kind["header"])
        for i in self.valid:
            _, _, _, blocks = O.decode_frame(self.frames[i], dst_cap=self.caps[i], trace=True)
            huf = [b for b in blocks if b["block_type"] == 2 and b["lit_type"] >= 2]
            seq = [b for b in blocks if b["block_type"] == 2 and b["n_seq"]]
            n_seq_true = sum(b["n_seq"] for b in seq)
            self.scan[i] = dict(n_blocks=len(blocks), lit_bytes=sum((b["regen_size"] + 16 + 15) & ~15 for b in huf),
                                n_seq=sum((b["n_seq"] + 3) & ~3 for b in seq), n_huf=len(huf), n_fse=len(seq),
                                src_bytes=len(self.frames[i]), fse_cls=size_class(n_seq_true // len(seq)) if seq else None)
        self.no_huf = [i for i in self.valid if self.scan[i]["n_huf"] == 0]
        self.no_seq = [i for i in self.valid if self.scan[i]["n_fse"] == 0]
        self.small = [i for i in range(len(self.frames)) if len(self.frames[i]) < LARGE]

    def batch(self, idx):
        return [self.frames[i] for i in idx], [self.caps[i] for i in idx]


def _weight_table_frames(n, seed):
    """Huffman weight descriptions with FSE accuracy log 10..20 (built in FseBigScratch, one warp at a time behind a lock),
    as in test_gpu_fuzz.py."""
    rng = np.random.default_rng(seed)
    frames = []
    for k in range(n):
        log = int(rng.choice([10, 11, 12, 13, 14, 16, 20]))
        nsym = int(rng.integers(2, 9))
        total = 1 << log
        cuts = np.sort(rng.choice(np.arange(1, total), size=nsym - 1, replace=False))
        probs = np.diff(np.concatenate([[0], cuts, [total]])).astype(int).tolist()
        if k % 5 == 0 and probs[-1] > 2:
            probs[-1] -= 2
            probs += [0, 0, -1, -1]
        ws = bytes(rng.integers(0, 256, size=int(rng.integers(1, 24)), dtype=np.uint8).tolist()[:-1] + [int(rng.integers(1, 256))])
        hs = bytes(rng.integers(0, 256, size=int(rng.integers(1, 40)), dtype=np.uint8).tolist()[:-1] + [int(rng.integers(1, 256))])
        frames.append(H.frame_with_weight_table(log, probs, ws, hs, int(rng.integers(1, 300))))
    return frames


def _raw_rle_frames():
    rng = np.random.default_rng(17)
    raw = [[Raw(rng.integers(0, 256, 1, dtype=np.uint8).tobytes())], [Raw(rng.integers(0, 256, 3000, dtype=np.uint8).tobytes())],
           [Raw(rng.integers(0, 256, 5000, dtype=np.uint8).tobytes()), Raw(b""), Raw(rng.integers(0, 256, 700, dtype=np.uint8).tobytes())]]
    rle = [[Rle(0x61, 1)], [Rle(0, 4000)], [Rle(0xFF, 70000), Rle(7, 3), Rle(0x20, 1000)]]
    build = lambda bl: S.build_frame(bl)
    return [build(b) for b in raw], [len(S.reference_decode(b)) for b in raw], [build(b) for b in rle], [len(S.reference_decode(b)) for b in rle]


def large_frames():
    """Three distinct ~128 KiB literal-heavy frames, each at least 32 KiB compressed."""
    cz = WL.Compressor()
    origs = [WL.skewed_bytes(128 << 10, 300 + k).tobytes() for k in range(3)]
    frames = [cz.compress(o) for o in origs]
    assert all(len(f) >= LARGE for f in frames), [len(f) for f in frames]
    return frames, [len(o) for o in origs]


def build_pool(corpus):
    p = Pool()
    p.add("corpus", [corpus.frame(i) for i in range(len(corpus))], [e["orig_len"] for e in corpus.index])
    for fam, mod in ((F, "seq"), (HF, "huf"), (X, "seq")):
        for name in sorted(fam.FAMILIES):
            for c in fam.cases(name):
                p.add(mod if isinstance(c.expected, bytes) else mod + "-bad", [c.frame], [c.cap])
    p.add("weight", _weight_table_frames(24, 7), [1024] * 24)
    for f, o in (WL.config2_text_frames(4, 65536), WL.config3_literal_heavy(1, frame_size=1 << 18),
                 WL.config5_mixed_sizes(6, hi=1 << 18), WL.small_alphabet_frames(4)):
        p.add("synth", f, [len(x) for x in o])
    rng = np.random.default_rng(5)   # as test_gpu_guard._frames: bit flips and truncations of corpus frames
    for i in (11, 33, 35, 97):
        b = bytearray(corpus.frame(i))
        for _ in range(3):
            b[int(rng.integers(8, len(b)))] ^= 1 << int(rng.integers(0, 8))
        p.add("mutant", [bytes(b)], [corpus.index[i]["orig_len"]])
        p.add("trunc", [corpus.frame(i)[: len(corpus.frame(i)) * 2 // 3]], [corpus.index[i]["orig_len"]])
    good = corpus.frame(0)
    # frames that fail in the header: empty, short magic, bad magic, truncated descriptor fields, a 2^41-byte window
    header = [b"", b"\x28\xb5\x2f", b"\x29" + good[1:], good[:5], struct.pack("<IB", 0xFD2FB528, 0xE0),
              good[:4] + b"\x00\xf8" + good[6:]]
    p.add("header", header, [4096] * len(header))
    # the reserved descriptor bit is not checked by the reference (frame.cairo): such a frame decodes
    p.add("mutant", [good[:4] + bytes([good[4] | 0x08]) + good[5:]], [corpus.index[0]["orig_len"]])
    rf, rc, lf, lc = _raw_rle_frames()
    p.add("raw", rf, rc)
    p.add("rle", lf, lc)
    p.finish()
    return p


@pytest.fixture(scope="module")
def pool(corpus):
    return build_pool(corpus)


def layout(p, n, W, r):
    """n pool indices: a fixed spread over the pool, with a frame of kind KINDS[(j + r) % len(KINDS)] on the j-th of the
    seam positions 0, W-1, W, 2W-1 and n-1 (rotating r over len(KINDS) puts every kind on every seam)."""
    P = len(p.frames)
    idx = [(i * 7919 + r * 131) % P for i in range(n)]
    seams = sorted({s for s in (0, W - 1, W, 2 * W - 1, n - 1) if 0 <= s < n})
    for j, s in enumerate(seams):
        members = p.by_kind[KINDS[(j + r) % len(KINDS)]]
        idx[s] = members[(r + 3 * j) % len(members)]
    return idx


def _cycle(members, n, start=0):
    return [members[(start + k) % len(members)] for k in range(n)]


# ---------------------------------------------------------------------------------------------------------------------
# 1. wave seams
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("W", [128, 384])
def test_every_frame_kind_on_every_wave_seam(pool, monkeypatch, W, mode):
    """CZB_WAVE_FRAMES = 128 and 384 (not a power of two: the scan's i / wave_frames and the per-CTA class histogram meet
    uneven boundaries), batch sizes around one and three waves, every frame kind at positions 0, W-1, W, 2W-1 and last."""
    ctx = _context(monkeypatch, dict(MODES[mode], CZB_WAVE_FRAMES=str(W)))
    ref = _context(monkeypatch, MODES[mode])
    sizes = sorted({127, 128, 129, W - 1, W, W + 1})
    for k, n in enumerate(sizes):
        frames, caps = pool.batch(layout(pool, n, W, k))
        decode(ctx, frames, caps, f"W={W}/{mode}/n={n}", ref)
    n = 3 * W + 5
    for r in range(len(KINDS)):
        frames, caps = pool.batch(layout(pool, n, W, r))
        decode(ctx, frames, caps, f"W={W}/{mode}/n={n}/r={r}", ref)
    _watchdog_clear()
    ctx.close(); ref.close()


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("W", [128, 384])
def test_waves_with_special_contents(pool, monkeypatch, W, mode):
    """Waves of header failures only (no frame to execute), without a Huffman section, without sequences, and the wave
    with the most scratch first, in the middle and last; the plan's totals confirm what each wave holds."""
    ctx = _context(monkeypatch, dict(MODES[mode], CZB_WAVE_FRAMES=str(W)))
    ref = _context(monkeypatch, MODES[mode])
    lf, lc = large_frames()
    base = len(pool.frames)
    frames_all, caps_all = pool.frames + lf, pool.caps + lc
    heavy = list(range(base, base + len(lf)))
    waves = {"header": _cycle(pool.by_kind["header"], W), "no-huf": _cycle(pool.no_huf, W, 1), "no-seq": _cycle(pool.no_seq, W, 2),
             "mixed": layout(pool, W, W, 4), "heavy": _cycle(heavy, W)}
    for order in (["heavy", "header", "no-huf", "no-seq", "mixed"], ["header", "no-huf", "heavy", "no-seq", "mixed"],
                  ["header", "no-huf", "no-seq", "mixed", "heavy"]):
        idx = [i for name in order for i in waves[name]][: 5 * W - 3]    # the last wave is three frames short
        frames, caps = [frames_all[i] for i in idx], [caps_all[i] for i in idx]
        label = f"W={W}/{mode}/{','.join(order)}"
        decode(ctx, frames, caps, label, ref)
        w, totals = plan_waves(ctx, frames, caps)
        assert w == W and len(totals) == 5, (w, len(totals))
        t = dict(zip(order, totals))
        assert sum(t["header"].frame_cls) == 0 and t["header"].n_blocks == 0 and t["header"].src_bytes == 0, label
        assert t["no-huf"].n_huf == 0 and t["no-huf"].lit_bytes == 0, label
        assert t["no-seq"].n_fse == 0 and t["no-seq"].n_seq == 0, label
        assert all(t["heavy"].lit_bytes > t[o].lit_bytes for o in order if o != "heavy"), label
    _watchdog_clear()
    ctx.close(); ref.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. a different executor in each wave
# ---------------------------------------------------------------------------------------------------------------------
def predicted_executor(t, count, sms):
    """The choice of czb_api.cu for one wave under the default rules (big_cls 19, share_cls 15, big_share 8192, seven
    k_exec_big CTAs per SM, flow_max = 2 x SMs), from the wave's totals."""
    share = t.src_bytes // 8192 + 1
    if count > 7 * sms:
        share = max(share, t.src_bytes * 3 // (2 * count) + 1)
    lo = min(19, max(15, size_class(share - 1) if share > 1 else 0))
    est = sum(t.frame_cls[lo:])
    if sum(t.frame_cls[15:]) == 0:
        return "k_exec"
    if est > 2 * sms:
        return "k_exec_big"
    return "k_exec_flow wide" if est <= sms else "k_exec_flow narrow"


def test_a_different_executor_in_each_wave(pool, monkeypatch):
    """CZB_WAVE_FRAMES=512: wave 0 holds one large frame (wide k_exec_flow), wave 1 between SMs+1 and 2 x SMs (narrow
    k_exec_flow), wave 2 more than 2 x SMs (k_exec_big), wave 3 none (k_exec alone)."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    W = 512
    n_large = [1, sms + sms // 2, 2 * sms + 16, 0]
    assert n_large[2] <= W
    lf, lc = large_frames()
    base = len(pool.frames)
    frames_all, caps_all = pool.frames + lf, pool.caps + lc
    small = pool.small
    idx = []
    for w, k in enumerate(n_large):
        step = W // k if k else 0
        for j in range(W):
            idx.append(base + (j // step) % 3 if k and j % step == 0 and j // step < k else small[(w * W + j * 31) % len(small)])
    frames, caps = [frames_all[i] for i in idx], [caps_all[i] for i in idx]
    ctx = _context(monkeypatch, {"CZB_WAVE_FRAMES": str(W)})
    ref = _context(monkeypatch)
    w, totals = plan_waves(ctx, frames, caps)
    assert w == W and len(totals) == 4
    for k, t in zip(n_large, totals):
        assert sum(t.frame_cls[15:]) == k, (k, list(t.frame_cls))
    assert [predicted_executor(t, W, sms) for t in totals] == ["k_exec_flow wide", "k_exec_flow narrow", "k_exec_big", "k_exec"]
    decode(ctx, frames, caps, "executor-per-wave", ref)
    _watchdog_clear()
    ctx.close(); ref.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. the budget retry
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["default", "flow-narrow"])
def test_budget_retry_decodes_like_one_wave(pool, monkeypatch, mode):
    """A 1-byte workspace budget: the planner halves W from 640 through 384 and 256 down to 128 (600 frames)."""
    ctx = _context(monkeypatch, MODES[mode], budget=1)
    ref = _context(monkeypatch, MODES[mode])
    frames, caps = pool.batch(layout(pool, 600, 128, 2))
    w, totals = plan_waves(ctx, frames, caps)
    assert w == 128 and len(totals) == 5
    decode(ctx, frames, caps, f"retry/{mode}", ref)
    _watchdog_clear()
    ctx.close(); ref.close()


def expected_totals(p, idx, W):
    """The per-wave totals of a batch of valid frames, from the oracle's block trace."""
    out = []
    for first in range(0, len(idx), W):
        t = dict(n_blocks=0, lit_bytes=0, n_seq=0, n_huf=0, n_fse=0, src_bytes=0, frame_cls=[0] * 32, fse_cls=[0] * 32)
        for i in idx[first:first + W]:
            s = p.scan[i]
            for k in ("n_blocks", "lit_bytes", "n_seq", "n_huf", "n_fse", "src_bytes"):
                t[k] += s[k]
            t["frame_cls"][size_class(s["src_bytes"])] += 1
            if s["fse_cls"] is not None:
                t["fse_cls"][s["fse_cls"]] += s["n_fse"]
        out.append(t)
    return out


def _as_dict(t):
    return dict(n_blocks=t.n_blocks, lit_bytes=t.lit_bytes, n_seq=t.n_seq, n_huf=t.n_huf, n_fse=t.n_fse, src_bytes=t.src_bytes,
                frame_cls=list(t.frame_cls), fse_cls=list(t.fse_cls))


def test_budget_retry_keeps_every_wave_total(pool, monkeypatch):
    """The plan after the retry holds the same wave split and the same totals, field for field, as the plan of a context
    that starts at 128 frames per wave; both equal the totals computed from the frames themselves (src_bytes: the sum of
    the frames' lengths, which the share rule of the CTA-per-frame executors divides)."""
    valid = pool.valid
    idx = [valid[(k * 37) % len(valid)] for k in range(600)]
    frames, caps = pool.batch(idx)
    retry = _context(monkeypatch, budget=1)
    w128 = _context(monkeypatch, {"CZB_WAVE_FRAMES": "128"})
    w_r, t_r = plan_waves(retry, frames, caps)
    w_1, t_1 = plan_waves(w128, frames, caps)
    assert (w_r, len(t_r)) == (w_1, len(t_1)) == (128, 5)
    want = expected_totals(pool, idx, 128)
    for k in range(5):
        assert _as_dict(t_1[k]) == want[k], (k, _as_dict(t_1[k]), want[k])
        assert _as_dict(t_r[k]) == want[k], (k, _as_dict(t_r[k]), want[k])
    retry.close(); w128.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4. two-stream overlap
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["default", "flow-narrow"])
def test_two_stream_overlap_reuses_both_scratch_sets(pool, monkeypatch, mode):
    """CZB_OVERLAP=1, CZB_WAVE_FRAMES=128, six waves: scratch set 0 is reused by waves 2 and 4, set 1 by waves 3 and 5.
    Guard zones behind the scratch (CZB_GUARD=1) and around every output span must stay intact.  The execution-free sizes
    of the same batch (k_frame_sizes runs on the exec stream) equal the oracle's."""
    env = dict(MODES[mode], CZB_OVERLAP="1", CZB_WAVE_FRAMES="128", CZB_GUARD="1")
    ctx = _context(monkeypatch, env)
    ref = _context(monkeypatch, MODES[mode])
    frames, caps = pool.batch(layout(pool, 5 * 128 + 37, 128, 6))
    for _ in range(2):  # twice: the second call reuses scratch that is exactly big enough
        decode(ctx, frames, caps, f"overlap/{mode}", ref, gaps=True)
    sizes = ctx.frame_sizes(frames)
    assert ctx.guard_faults() == 0
    for i, (f, cap) in enumerate(zip(frames, caps)):
        st, _, fields, _ = oracle(f, cap)
        if st == 0:
            r = sizes[i]
            assert r.status == 0 and (r.bytes_written, r.blocks_decoded, r.bytes_read) == \
                (fields["bytes_written"], fields["blocks_decoded"], fields["bytes_read"]), (i, czb.status_name(r.status))
    _watchdog_clear()
    ctx.close(); ref.close()


# ---------------------------------------------------------------------------------------------------------------------
# 5. planned and captured calls over many waves
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("setup", ["waves", "waves-overlap", "retry"])
def test_planned_and_captured_calls_over_many_waves(pool, monkeypatch, setup):
    """A plan of five waves (CZB_WAVE_FRAMES=128, with and without CZB_OVERLAP=1, or from the budget retry), decoded planned
    and then captured into a CUDA graph and replayed twice: outputs and results identical to the unplanned call's."""
    import torch
    env = {"waves": {"CZB_WAVE_FRAMES": "128"}, "waves-overlap": {"CZB_WAVE_FRAMES": "128", "CZB_OVERLAP": "1"}, "retry": {}}[setup]
    ctx = _context(monkeypatch, env, budget=1 if setup == "retry" else 0)
    frames, caps = pool.batch(layout(pool, 600, 128, 8))
    b = DevBatch(frames, caps)
    s = torch.cuda.Stream()
    b.decode(ctx, s.cuda_stream)
    outs, res, raw, _ = b.fetch()
    check(frames, caps, outs, res, f"unplanned/{setup}")
    plan = b.plan(ctx, s.cuda_stream)
    assert ctx.plan_waves(plan)[0] == 128 and len(ctx.plan_waves(plan)[1]) == 5
    b.reset()
    b.decode_planned(ctx, plan, s.cuda_stream)
    o2, _, raw2, _ = b.fetch()
    assert raw2 == raw and o2 == outs, f"planned/{setup}"
    g = torch.cuda.CUDAGraph()
    b.reset()
    torch.cuda.synchronize()
    with torch.cuda.graph(g, stream=s, capture_error_mode="relaxed"):
        b.decode_planned(ctx, plan, s.cuda_stream)
    for k in range(2):
        b.reset()
        g.replay()
        o3, _, raw3, _ = b.fetch()
        assert raw3 == raw and o3 == outs, f"replay {k}/{setup}"
    del g
    ctx.plan_destroy(plan)
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# 6. back-to-back calls on two streams
# ---------------------------------------------------------------------------------------------------------------------
def test_back_to_back_calls_on_two_streams(pool, monkeypatch):
    """A planned five-wave call on one stream, with no host synchronisation after it, then at once an ordinary call with a
    different batch on another stream: the second call must wait for the first one's kernels before it reuses the
    context's scratch, and both batches must decode correctly."""
    import torch
    ctx = _context(monkeypatch, {"CZB_WAVE_FRAMES": "128"})
    lf, lc = large_frames()
    fa, ca = pool.batch(layout(pool, 600, 128, 9))
    fa[::50], ca[::50] = lf * 4, lc * 4          # heavy frames through the first call's waves
    fb, cb = pool.batch(layout(pool, 300, 128, 10)[::-1])
    a, b = DevBatch(fa, ca), DevBatch(fb, cb)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    plan = a.plan(ctx, s1.cuda_stream)
    for k in range(2):
        a.reset(); b.reset()
        torch.cuda.synchronize()
        a.decode_planned(ctx, plan, s1.cuda_stream)
        b.decode(ctx, s2.cuda_stream)
        oa, ra, _, _ = a.fetch()
        ob, rb, _, _ = b.fetch()
        check(fa, ca, oa, ra, f"stream 1 [{k}]")
        check(fb, cb, ob, rb, f"stream 2 [{k}]")
    ctx.plan_destroy(plan)
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# 7. the kMaxWaves doubling
# ---------------------------------------------------------------------------------------------------------------------
RESULT_DTYPE = np.dtype([("status", "<i4"), ("blocks_decoded", "<u4"), ("bytes_read", "<u8"), ("bytes_written", "<u8"),
                         ("content_size", "<u8"), ("window_size", "<u8"), ("checksum_from_data", "<u4"),
                         ("checksum_calculated", "<u4"), ("has_checksum", "<i4"), ("finished", "<i4")])


def test_more_than_4096_waves_doubles_the_wave(monkeypatch):
    """4096 x 128 + 1 tiny frames with CZB_WAVE_FRAMES=128 would make 4097 waves: W doubles to 256 (2049 waves).  Raw, RLE,
    sequence and header-failure frames in a fixed pseudo-random order, checked kind by kind against the oracle."""
    import torch
    assert RESULT_DTYPE.itemsize == C.sizeof(api.FrameResult)
    small_seq = min((c for c in F.cases("repeat") if isinstance(c.expected, bytes)), key=lambda c: c.cap)
    kinds = [S.build_frame([Raw(bytes(range(40)))]), S.build_frame([Rle(0x33, 57)]), small_seq.frame,
             b"\x29" + small_seq.frame[1:]]
    caps = [40, 57, small_seq.cap, 64]
    slot = (max(caps) + 15) & ~15
    n = 4096 * 128 + 1
    kind = np.random.default_rng(23).integers(0, len(kinds), n)
    kind[:4] = [0, 1, 2, 3]
    dev = torch.device("cuda", 0)
    koff = np.concatenate([[0], np.cumsum([(len(f) + 15) & ~15 for f in kinds])])
    src_h = np.zeros(int(koff[-1]), dtype=np.uint8)
    for k, f in enumerate(kinds):
        src_h[koff[k]:koff[k] + len(f)] = np.frombuffer(f, dtype=np.uint8)
    src = torch.from_numpy(src_h).to(dev)
    dst = torch.zeros(n * slot, dtype=torch.uint8, device=dev)
    d = np.zeros((n, 4), dtype=np.uint64)
    d[:, 0] = src.data_ptr() + koff[kind]
    d[:, 1] = np.array([len(f) for f in kinds], dtype=np.uint64)[kind]
    d[:, 2] = dst.data_ptr() + np.arange(n, dtype=np.uint64) * slot
    d[:, 3] = np.array(caps, dtype=np.uint64)[kind]
    descs = torch.from_numpy(d.view(np.uint8).reshape(-1)).to(dev)
    results = torch.zeros(n * RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    ctx = _context(monkeypatch, {"CZB_WAVE_FRAMES": "128"})
    stream = _stream()
    plan = ctx.plan_batch_device(descs.data_ptr(), n, stream)
    w, totals = ctx.plan_waves(plan)
    ctx.plan_destroy(plan)
    assert w == 256 and len(totals) == 2049
    lens = np.where(kind == 3, 0, np.array([len(f) for f in kinds])[kind])     # the header failure is not walked
    want_src = np.add.reduceat(lens, np.arange(0, n, 256))
    assert [t.src_bytes for t in totals] == want_src.tolist()
    assert [sum(t.frame_cls) for t in totals] == np.add.reduceat((kind != 3).astype(np.int64), np.arange(0, n, 256)).tolist()
    ctx.decode_batch_device(descs.data_ptr(), results.data_ptr(), n, VERIFY, stream)
    torch.cuda.synchronize()
    res = np.frombuffer(results.cpu().numpy().tobytes(), dtype=RESULT_DTYPE)
    out = dst.cpu().numpy().reshape(n, slot)
    for k, (f, cap) in enumerate(zip(kinds, caps)):
        st, want, fields, has_ck = oracle(f, cap)
        m = kind == k
        assert (res["status"][m] == st).all(), (k, np.unique(res["status"][m]))
        if st == 0:
            for field in FIELDS:
                assert (res[field][m] == fields[field]).all(), (k, field)
            assert (res["has_checksum"][m] == int(has_ck)).all()
            assert (out[m, :len(want)] == np.frombuffer(want, dtype=np.uint8)).all(), k
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# 8. the packed host path with several waves per chunk
# ---------------------------------------------------------------------------------------------------------------------
def test_packed_host_path_several_waves_per_chunk(pool, monkeypatch):
    """CZB_HOST_CHUNK_MB=4 and CZB_WAVE_FRAMES=128 on small frames: each 4 MiB staging chunk holds several waves."""
    ctx = _context(monkeypatch, {"CZB_HOST_CHUNK_MB": "4", "CZB_WAVE_FRAMES": "128"})
    ref = _context(monkeypatch)
    cand = [i for i in pool.small if pool.caps[i] <= 8192]
    idx = [cand[(k * 13) % len(cand)] for k in range(2500)]
    frames, caps = pool.batch(idx)
    n = len(frames)
    src_off = np.zeros(n + 1, dtype=np.uint64); src_off[1:] = np.cumsum([len(f) for f in frames])
    dst_off = np.zeros(n + 1, dtype=np.uint64); dst_off[1:] = np.cumsum(caps)
    # the chunking rule of czb_decode_batch_host_packed: at most 4 MiB of source plus output per chunk
    cuts, i = [0], 0
    while i < n:
        j = i + 1
        while j < n and (src_off[j + 1] - src_off[i]) + (dst_off[j + 1] - dst_off[i]) <= 4 << 20:
            j += 1
        cuts.append(j); i = j
    assert len(cuts) >= 3 and min(b - a for a, b in zip(cuts[:-2], cuts[1:-1])) >= 3 * 128, cuts
    src = np.frombuffer(b"".join(frames), dtype=np.uint8).copy()
    dst = np.zeros(int(dst_off[-1]) + 1, dtype=np.uint8)
    results = (api.FrameResult * n)()
    ctx.decode_batch_packed(src.ctypes.data, src_off, dst.ctypes.data, dst_off, n, C.addressof(results), VERIFY)
    outs = [dst[int(dst_off[k]):int(dst_off[k]) + results[k].bytes_written].tobytes() if results[k].status == 0 else None
            for k in range(n)]
    ref_outs, ref_res = ref.decode_batch(frames, caps, VERIFY)
    check(frames, caps, outs, results, "packed", (ref_outs, ref_res))
    ctx.close(); ref.close()
