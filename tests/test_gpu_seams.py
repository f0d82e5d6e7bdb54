"""-m gpu: the frames of tests/seqfamilies.py -- matches, literal runs and repeat offsets placed on the seams of k_exec,
k_exec_big, k_exec_flow (both shapes) and k_fse -- decoded in one batch per family, through the default executor choice and
with every frame forced through each CTA-per-frame executor.  Every result field must equal the oracle's, the output must
equal the plain reference executor's, the device XXH64 must equal the trailer, and the flow executor's spin-limit safety net
must not have fired.  Also the GPU twin of the oracle's compression-level sweep (test_gpu_levels)."""
import ctypes as C

import numpy as np
import pytest

import gpu_common as G
import oracle_lib as O
import seqfamilies as F
import cairo_zstd_b200 as czb
from cairo_zstd_b200 import api, workloads as W

pytestmark = pytest.mark.gpu
MODES = ["default", "flow-narrow", "flow-wide", "big"]


def _context(monkeypatch, mode):
    if mode != "default":
        monkeypatch.setenv("CZB_BIG_CLS", "0"); monkeypatch.setenv("CZB_BIG_SEQ_BYTES", "0")
    if mode == "flow-wide":
        monkeypatch.setenv("CZB_FLOW_WIDE", "1")
    if mode == "big":
        monkeypatch.setenv("CZB_BIG_FLOW", "0")
    ctx = czb.Context(0)
    monkeypatch.setattr(G, "_ctx", ctx)   # gpu_common.compare_with_oracle decodes through this context
    return ctx


def _watchdog_clear():
    wd = (C.c_uint32 * 16)()
    czb.load_library().czb_debug_flow_watchdog(wd)
    assert wd[0] == 0, list(wd)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("family", sorted(F.FAMILIES))
def test_seam_families_match_reference_and_oracle(monkeypatch, family, mode):
    cases = F.cases(family)
    ctx = _context(monkeypatch, mode)
    frames, caps = [c.frame for c in cases], [c.cap for c in cases]
    outs, res = G.compare_with_oracle(frames, caps, label=f"{family}/{mode}")
    for c, o, r in zip(cases, outs, res):
        if isinstance(c.expected, bytes):
            assert o == c.expected, c.name
            assert bool(r.has_checksum) == bool(c.frame[4] & 4), c.name      # frames without the checksum flag: resume family
            assert not r.has_checksum or r.checksum_calculated == r.checksum_from_data, c.name
        else:
            assert czb.status_name(r.status) == c.expected, (c.name, czb.status_name(r.status))
    if mode != "default":
        _watchdog_clear()
    ctx.close()


GAP = 64
PAT = 0xA5


@pytest.mark.parametrize("mode", ["default", "big"])
def test_seam_frames_store_nothing_outside_their_spans(monkeypatch, mode):
    """The outputs laid out as in test_gpu_guard.py: exact capacities, 64-byte gaps at odd alignments filled with a pattern
    that must survive the decode (a failing frame must not scribble outside its span either)."""
    import torch
    cases = [c for f in ("chunks", "big", "invalid", "repeat") for c in F.cases(f)]
    ctx = _context(monkeypatch, mode)
    frames, caps = [c.frame for c in cases], [c.cap for c in cases]
    n = len(frames)
    dev = torch.device("cuda", 0)
    flens = np.array([len(f) for f in frames], dtype=np.int64)
    soff = np.concatenate([[0], np.cumsum((flens + 15) & ~15)])
    src_h = np.zeros(int(soff[-1]) + 16, dtype=np.uint8)
    for i, f in enumerate(frames):
        src_h[soff[i]:soff[i] + len(f)] = np.frombuffer(f, dtype=np.uint8)
    src = torch.from_numpy(src_h).to(dev)
    starts = np.zeros(n, dtype=np.int64)
    pos = GAP
    for i in range(n):
        starts[i] = pos
        pos += caps[i] + GAP + (i % 7)
    dst = torch.full((pos + GAP,), PAT, dtype=torch.uint8, device=dev)
    d = np.zeros((n, 4), dtype=np.uint64)
    d[:, 0] = src.data_ptr() + soff[:-1]
    d[:, 1] = flens
    d[:, 2] = dst.data_ptr() + starts
    d[:, 3] = np.array(caps, dtype=np.int64)
    descs = torch.from_numpy(d.view(np.uint8).reshape(-1)).to(dev)
    results = torch.zeros(n * C.sizeof(api.FrameResult), dtype=torch.uint8, device=dev)
    ctx.decode_batch_device(descs.data_ptr(), results.data_ptr(), n, api.FLAG_VERIFY_CHECKSUM, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    out = dst.cpu().numpy()
    res = (api.FrameResult * n).from_buffer_copy(results.cpu().numpy().tobytes())
    mask = np.ones(out.size, dtype=bool)
    for i, c in enumerate(cases):
        st, _, _ = O.decode_frame(c.frame, dst_cap=c.cap)
        assert res[i].status == st, (c.name, czb.status_name(st), czb.status_name(res[i].status))
        if isinstance(c.expected, bytes):
            assert out[starts[i]:starts[i] + len(c.expected)].tobytes() == c.expected, c.name
        mask[starts[i]:starts[i] + caps[i]] = False
    assert (out[mask] == PAT).all(), f"{int((out[mask] != PAT).sum())} bytes outside the frames' spans were overwritten"
    ctx.close()


# ---------------------------------------------------------------------------
# compression levels, strategies and minimum match lengths (libzstd as the encoder)
# ---------------------------------------------------------------------------
ZSTD_c_compressionLevel, ZSTD_c_minMatch, ZSTD_c_strategy, ZSTD_c_checksumFlag, ZSTD_c_contentSizeFlag = 100, 105, 107, 201, 200
LEVELS = [-5, -1, 1, 2, 5, 9, 13, 16, 19, 22]


def _compress(data, level, strategy=None, min_match=None, content_size=True):
    z = W.libzstd()
    cctx = z.ZSTD_createCCtx()
    try:
        for p, v in ((ZSTD_c_compressionLevel, level), (ZSTD_c_checksumFlag, 1), (ZSTD_c_strategy, strategy),
                     (ZSTD_c_minMatch, min_match), (ZSTD_c_contentSizeFlag, None if content_size else 0)):
            if v is not None:
                assert not z.ZSTD_isError(z.ZSTD_CCtx_setParameter(cctx, p, v)), (p, v)
        bound = z.ZSTD_compressBound(len(data))
        buf = C.create_string_buffer(bound)
        n = z.ZSTD_compress2(cctx, buf, bound, data, len(data))
        assert not z.ZSTD_isError(n)
        frame = buf.raw[:n]
    finally:
        z.ZSTD_freeCCtx(cctx)
    assert W.libzstd_decompress(frame, len(data)) == data   # the parameter set round-trips before the GPU sees it
    return frame


def _level_frames():
    texts = [W.synth_text(96 << 10, 11), W.skewed_bytes(96 << 10, 12).tobytes(), bytes(np.random.default_rng(13).integers(0, 2, 64 << 10, dtype=np.uint8))]
    frames, origs = [], []
    for lv in LEVELS:
        for t in texts:
            frames.append(_compress(t, lv)); origs.append(t)
    for strategy in range(1, 10):
        frames.append(_compress(texts[0], 3, strategy=strategy)); origs.append(texts[0])
    for mm in (3, 4, 5, 6, 7):
        frames.append(_compress(texts[1], 6, min_match=mm)); origs.append(texts[1])
    frames.append(_compress(texts[0], 3, content_size=False)); origs.append(texts[0])
    return frames, origs


@pytest.mark.parametrize("mode", ["default", "flow-narrow"])
def test_gpu_levels(monkeypatch, mode):
    """GPU twin of test_oracle.py's level sweep: frames from libzstd at levels -5..22, every strategy, minimum match lengths
    3..7 and without the content-size field; output and every result field equal to the oracle's, output equal to the input."""
    frames, origs = _level_frames()
    ctx = _context(monkeypatch, mode)
    outs, res = G.compare_with_oracle(frames, [len(o) for o in origs], label=mode)
    for o, g in zip(origs, outs):
        assert g == o
    if mode != "default":
        _watchdog_clear()
    ctx.close()
