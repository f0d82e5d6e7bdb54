"""-m gpu: czb_verify_batch_device against czb_decode_batch_device (CZB_FLAG_VERIFY_CHECKSUM) on the same frames.  Every
result field must be equal, for valid and malformed frames alike, in the four executor modes of test_gpu_large_frames.py.
The decode runs with dst_cap = the frame's known output size or a generous capacity (never reached), or CZB_MAX_FRAME_OUTPUT
for frames at the limit.  The descs given to the verify call point into a pattern-filled buffer that must stay untouched."""
import ctypes as C

import numpy as np
import pytest

import fsefamilies as XF
import huffamilies as HF
import largeframes as LF
import seqfamilies as SF
import cairo_zstd_b200 as czb
from cairo_zstd_b200 import api
from cairo_zstd_b200 import workloads as W
from test_gpu_fuzz import _mutants

pytestmark = pytest.mark.gpu
MODES = ["default", "flow-narrow", "flow-wide", "big"]
FIELDS = ("status", "blocks_decoded", "bytes_read", "bytes_written", "content_size", "window_size", "checksum_from_data",
          "checksum_calculated", "has_checksum", "finished")
PAT = 0x3C
UNSUPPORTED = "CZS_UNSUPPORTED"


def _env(monkeypatch, mode, **knobs):
    if mode == "warp":
        monkeypatch.setenv("CZB_BIG_CLS", "31"); monkeypatch.setenv("CZB_SHARE_CLS", "31")
    elif mode != "default":
        monkeypatch.setenv("CZB_BIG_CLS", "0"); monkeypatch.setenv("CZB_BIG_SEQ_BYTES", "0")
    if mode == "flow-wide":
        monkeypatch.setenv("CZB_FLOW_WIDE", "1")
    if mode == "big":
        monkeypatch.setenv("CZB_BIG_FLOW", "0")
    for k, v in knobs.items():
        monkeypatch.setenv(k, str(v))
    return czb.Context(0)


@pytest.fixture
def ctx(monkeypatch, request):
    c = _env(monkeypatch, request.param)
    yield c
    c.close()


def _results(t, n):
    return (api.FrameResult * n).from_buffer_copy(t.cpu().numpy().tobytes())


def verify_and_decode(ctx, frames, caps, decode=True):
    """Verify `frames` (descs whose dst points into a pattern buffer), then decode them with dst_cap = caps; assert equal
    results field for field and the pattern intact.  Returns the verify results."""
    import torch
    dev = torch.device("cuda", 0)
    n = len(frames)
    flens = np.array([len(f) for f in frames], dtype=np.int64)
    soff = np.concatenate([[0], np.cumsum((flens + 15) & ~15)])
    src_h = np.zeros(int(soff[-1]) + 16, dtype=np.uint8)
    for i, f in enumerate(frames):
        src_h[soff[i]:soff[i] + len(f)] = np.frombuffer(f, dtype=np.uint8)
    src = torch.from_numpy(src_h).to(dev)
    stream = torch.cuda.current_stream().cuda_stream
    rsize = C.sizeof(api.FrameResult)

    pattern = torch.full((4096,), PAT, dtype=torch.uint8, device=dev)
    d = np.zeros((n, 4), dtype=np.uint64)
    d[:, 0] = src.data_ptr() + soff[:-1]
    d[:, 1] = flens
    d[:, 2] = pattern.data_ptr() + (np.arange(n, dtype=np.uint64) % 64) * 64
    d[:, 3] = np.arange(n, dtype=np.uint64) % 3 * 32  # ignored: 0, 32 or 64 bytes "available"
    vdescs = torch.from_numpy(d.view(np.uint8).reshape(-1).copy()).to(dev)
    vres = torch.full((n * rsize,), 0xEE, dtype=torch.uint8, device=dev)
    ctx.verify_batch_device(vdescs.data_ptr(), vres.data_ptr(), n, stream)
    torch.cuda.synchronize()
    got = _results(vres, n)
    assert bool((pattern == PAT).all()), "verify wrote through a desc's dst"
    assert np.array_equal(vdescs.cpu().numpy().view(np.uint64).reshape(n, 4), d), "verify changed the caller's descs"
    if not decode:
        return got

    caps = np.array(caps, dtype=np.uint64)
    doff = np.concatenate([[0], np.cumsum((caps + 15) & ~np.uint64(15))]).astype(np.uint64)
    dst = torch.empty((int(doff[-1]) + 16,), dtype=torch.uint8, device=dev)
    d[:, 2] = dst.data_ptr() + doff[:-1]
    d[:, 3] = caps
    ddescs = torch.from_numpy(d.view(np.uint8).reshape(-1).copy()).to(dev)
    dres = torch.zeros((n * rsize,), dtype=torch.uint8, device=dev)
    ctx.decode_batch_device(ddescs.data_ptr(), dres.data_ptr(), n, api.FLAG_VERIFY_CHECKSUM, stream)
    torch.cuda.synchronize()
    want = _results(dres, n)
    del dst
    # a frame whose output passed its capacity: decode it again alone at the largest capacity
    again = [i for i in range(n) if czb.status_name(want[i].status) == "CZS_DST_TOO_SMALL"]
    if again:
        dst = torch.empty((LF.MAX_OUT + 16,), dtype=torch.uint8, device=dev)
        for i in again:
            one = d[i:i + 1].copy()
            one[0, 2], one[0, 3] = dst.data_ptr(), LF.MAX_OUT
            od = torch.from_numpy(one.view(np.uint8).reshape(-1)).to(dev)
            ores = torch.zeros((rsize,), dtype=torch.uint8, device=dev)
            ctx.decode_batch_device(od.data_ptr(), ores.data_ptr(), 1, api.FLAG_VERIFY_CHECKSUM, stream)
            torch.cuda.synchronize()
            want[i] = _results(ores, 1)[0]
        del dst
    for i in range(n):
        for k in FIELDS:
            assert getattr(got[i], k) == getattr(want[i], k), (i, k, getattr(got[i], k), getattr(want[i], k),
                                                               czb.status_name(got[i].status), czb.status_name(want[i].status))
    return got


# ---- frame sets -------------------------------------------------------------------------------------------------------

def _corpus(corpus):
    return [corpus.frame(i) for i in range(len(corpus.index))], [e["orig_len"] for e in corpus.index]


def _configs():
    frames, caps = [], []
    for f, o in [W.config2_text_frames(6, 65536, seed=5), W.config3_literal_heavy(2, seed=6),
                 W.config4_long_window(1, total=8 << 20, seed=7), W.config5_mixed_sizes(12, seed=8, hi=1 << 20)]:
        frames += list(f); caps += [len(x) for x in o]
    return frames, caps


def _families():
    frames, caps = [], []
    for mod in (SF, HF, XF):
        for name in mod.FAMILIES:
            for c in mod.cases(name):
                frames.append(c.frame)
                caps.append((len(c.expected) if isinstance(c.expected, bytes) else max(c.cap, 1 << 20)) + 4096)
    return frames, caps


def _no_content_size():
    frames, caps = [], []
    for k, n in enumerate((1000, 70000, 300000, 1 << 20)):
        data = W.synth_text(n, seed=40 + k)
        frames.append(LF.compress(np.frombuffer(data, dtype=np.uint8), 22, content_size=False)); caps.append(n)
    blocks, _ = LF.fill_blocks(5 << 20, seed=3, raw_every=8)
    frames.append(LF.frame(blocks, 5 << 20, fcs_width=0, single_segment=False, window_log=23)); caps.append(5 << 20)
    for f in frames:
        assert czb.frame_header_info(f).fcs_present == 0
    return frames, caps


def _fcs_too_small():
    """Frame_Content_Size below what the blocks produce (the field is not checked against the output, in the reference
    either): the output bound must come from the blocks."""
    frames, caps = [], []
    for n, claim in ((1000, 10), (300000, 1000), (3 << 20, 1 << 16)):
        blocks, content = LF.fill_blocks(n, seed=n & 0xFF, raw_every=3)
        frames.append(LF.frame(blocks, claim, xxh=LF.xxh32_low(content), single_segment=False, window_log=23, fcs_width=4))
        caps.append(n)
    return frames, caps


# ---- tests ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("ctx", MODES, indirect=True)
def test_corpus_configs_families_and_fuzz(ctx, corpus):
    for label, (frames, caps) in [("corpus", _corpus(corpus)), ("configs", _configs()), ("families", _families()),
                                  ("no-fcs", _no_content_size()), ("fcs-too-small", _fcs_too_small())]:
        res = verify_and_decode(ctx, frames, caps)
        assert all(czb.status_name(r.status) != "CZS_DST_TOO_SMALL" for r in res), label  # the decode capacities were never reached
    for seed in (7, 8, 20261018):
        frames, caps = _mutants(corpus, seed)
        verify_and_decode(ctx, frames, caps)


def test_valid_frames_verify_their_checksums(corpus):
    c = czb.Context(0)
    frames, caps = _corpus(corpus)
    res = verify_and_decode(c, frames, caps, decode=False)
    for r, n in zip(res, caps):
        assert r.status == 0 and r.bytes_written == n and r.finished == 1
        if r.has_checksum:
            assert r.checksum_calculated == r.checksum_from_data
    c.close()


@pytest.fixture(scope="module")
def large():
    """The large frames of largeframes.py: 2^28 - 1, 2^28 + 1 and 300 MiB (RLE/Raw and libzstd text), the 2^28 - 1 offset
    seam cases, 2^31 - 1 bytes with a checksum and 2^31 bytes."""
    frames, caps = [], []
    data = LF.text(300 << 20)
    for n in (LF.M28 - 1, LF.M28 + 1, 300 << 20):
        blocks, content = LF.fill_blocks(n, seed=n & 0xFFFF, raw_every=256)
        frames.append(LF.frame(blocks, n, xxh=LF.xxh32_low(content))); caps.append(n)
        del content
        frames.append(LF.compress(data[:n], 27, ldm=True)); caps.append(n)
    del data
    for c in LF.seam_cases():
        frames.append(c.frame); caps.append(max(c.cap, c.out) + 4096 if c.valid else c.cap)
    top = np.full(LF.MAX_OUT, 0x5A, dtype=np.uint8)
    xxh = LF.xxh32_low(top)
    del top
    frames.append(LF.frame(LF.rle_only(LF.MAX_OUT), LF.MAX_OUT, xxh=xxh)); caps.append(LF.MAX_OUT)
    frames.append(LF.frame(LF.rle_only(LF.MAX_OUT + 1), LF.MAX_OUT + 1)); caps.append(LF.MAX_OUT)
    return frames, caps


@pytest.mark.parametrize("ctx", MODES, indirect=True)
def test_large_frames_and_the_limit(ctx, large):
    frames, caps = large
    res = verify_and_decode(ctx, frames, caps)
    top, over = res[-2], res[-1]
    assert top.status == 0 and top.bytes_written == LF.MAX_OUT and top.checksum_calculated == top.checksum_from_data
    assert czb.status_name(over.status) == UNSUPPORTED
    assert any(czb.status_name(r.status) == UNSUPPORTED for r in res[6:-2])  # far offsets


def _waves(ctx):
    ctx.profile_enable(False)
    return ctx.profile_collect()["fill"][1]


def test_output_bound_forces_small_waves(monkeypatch, corpus):
    """Eight frames of 2^28 + 7 bytes (tiny compressed, 256 MiB of output bound each) with a 1 GiB budget: the retry halves the
    wave below 128 frames until the bound fits (two frames per wave).  The decode path does not count outputs: one wave."""
    c = _env(monkeypatch, "default", CZB_BUDGET_GB=1)
    n = LF.M28 + 7
    frames = [LF.frame(LF.rle_only(n, byte=0x40 + k), n) for k in range(8)]
    c.profile_enable(True)
    res = verify_and_decode(c, frames, [n] * 8, decode=False)
    assert _waves(c) == 4
    assert all(r.status == 0 and r.bytes_written == n for r in res)
    verify_and_decode(c, frames, [n] * 8)
    c.close()


def test_frame_over_the_budget_alone_is_unsupported(monkeypatch, corpus):
    big = (5 << 28) + 3  # 1.25 GiB of output: its bound alone exceeds a 1 GiB budget
    frames, caps = _corpus(corpus)
    frames = frames[:20] + [LF.frame(LF.rle_only(big), big)] + frames[20:40]
    caps = caps[:20] + [big] + caps[20:40]
    c = _env(monkeypatch, "default", CZB_BUDGET_GB=1)
    res = verify_and_decode(c, frames, caps, decode=False)
    assert czb.status_name(res[20].status) == UNSUPPORTED and res[20].content_size == big
    c.close()
    ref = czb.Context(0)  # the neighbours verify as the decode path decodes them
    want = verify_and_decode(ref, frames[:20] + frames[21:], caps[:20] + caps[21:])
    ref.close()
    for a, b in zip(list(res[:20]) + list(res[21:]), want):
        for k in FIELDS:
            assert getattr(a, k) == getattr(b, k), k


@pytest.mark.parametrize("knobs", [dict(CZB_WAVE_FRAMES=128), dict(CZB_WAVE_FRAMES=128, CZB_OVERLAP=1),
                                   dict(CZB_GUARD=1), dict(CZB_GUARD=1, CZB_WAVE_FRAMES=128, CZB_OVERLAP=1)],
                         ids=["waves", "waves-overlap", "guard", "guard-waves-overlap"])
def test_many_waves_overlap_and_guard(monkeypatch, corpus, knobs):
    frames, caps = _corpus(corpus)
    f2, c2 = _families()
    frames, caps = frames * 4 + f2, caps * 4 + c2
    order = np.random.default_rng(3).permutation(len(frames))
    frames, caps = [frames[i] for i in order], [caps[i] for i in order]
    c = _env(monkeypatch, "default", **knobs)
    c.profile_enable(True)
    verify_and_decode(c, frames, caps, decode=False)
    waves = _waves(c)
    if "CZB_WAVE_FRAMES" in knobs:
        assert waves == (len(frames) + 127) // 128
    verify_and_decode(c, frames, caps)
    if "CZB_GUARD" in knobs:
        assert c.guard_faults() == 0
    c.close()
