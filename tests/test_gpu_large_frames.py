"""-m gpu: frames whose output reaches and passes 2^28 bytes (tests/largeframes.py), in the four executor modes of
test_gpu_seams.py.  Outputs must equal libzstd's, every result field the oracle's, the device XXH64 the trailer; offsets at the
2^28 - 1 seam give the exact bytes, the oracle's status or CZS_UNSUPPORTED as include/cairo_zstd_b200.h states; frames of
2^31 - 1 bytes decode and larger ones are refused.  Frames go through device pointers, and every output is laid out between
64-byte guard gaps that must stay untouched."""
import ctypes as C

import numpy as np
import pytest

import largeframes as LF
import cairo_zstd_b200 as czb
from cairo_zstd_b200 import api
from cairo_zstd_b200.frame_decoder import ByteSlice

pytestmark = pytest.mark.gpu
MODES = ["default", "flow-narrow", "flow-wide", "big"]
SIZES = [LF.M28 - 2, LF.M28 - 1, LF.M28, 300 << 20]
GAP, PAT = 64, 0xA5
FIELDS = ("blocks_decoded", "bytes_read", "bytes_written", "content_size", "window_size", "checksum_from_data",
          "checksum_calculated", "has_checksum", "finished")


@pytest.fixture
def ctx(monkeypatch, request):
    """A context in the executor mode `request.param` (the knobs of test_gpu_seams.py)."""
    mode = request.param
    if mode == "warp":  # no frame is given a CTA: k_exec alone
        monkeypatch.setenv("CZB_BIG_CLS", "31"); monkeypatch.setenv("CZB_SHARE_CLS", "31")
    elif mode != "default":
        monkeypatch.setenv("CZB_BIG_CLS", "0"); monkeypatch.setenv("CZB_BIG_SEQ_BYTES", "0")
    if mode == "flow-wide":
        monkeypatch.setenv("CZB_FLOW_WIDE", "1")
    if mode == "big":
        monkeypatch.setenv("CZB_BIG_FLOW", "0")
    c = czb.Context(0)
    yield c
    if mode not in ("default", "warp"):
        wd = (C.c_uint32 * 16)()
        czb.load_library().czb_debug_flow_watchdog(wd)
        assert wd[0] == 0, list(wd)
    c.close()


def decode(ctx, frames, caps):
    """Decode through device pointers, outputs at odd offsets between 64-byte gaps of PAT.  Returns (dst tensor, starts,
    results); asserts that no gap byte changed."""
    import torch
    dev = torch.device("cuda", 0)
    n = len(frames)
    flens = np.array([len(f) for f in frames], dtype=np.int64)
    soff = np.concatenate([[0], np.cumsum((flens + 15) & ~15)])
    src_h = np.zeros(int(soff[-1]) + 16, dtype=np.uint8)
    for i, f in enumerate(frames):
        src_h[soff[i]:soff[i] + len(f)] = np.frombuffer(f, dtype=np.uint8)
    src = torch.from_numpy(src_h).to(dev)
    starts, pos = [], GAP
    for i in range(n):
        starts.append(pos)
        pos += caps[i] + GAP + (i % 7) + 1
    dst = torch.full((pos + GAP,), PAT, dtype=torch.uint8, device=dev)
    d = np.zeros((n, 4), dtype=np.uint64)
    d[:, 0] = src.data_ptr() + soff[:-1]
    d[:, 1] = flens
    d[:, 2] = dst.data_ptr() + np.array(starts, dtype=np.uint64)
    d[:, 3] = np.array(caps, dtype=np.uint64)
    descs = torch.from_numpy(d.view(np.uint8).reshape(-1)).to(dev)
    results = torch.zeros(n * C.sizeof(api.FrameResult), dtype=torch.uint8, device=dev)
    ctx.decode_batch_device(descs.data_ptr(), results.data_ptr(), n, api.FLAG_VERIFY_CHECKSUM, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    res = (api.FrameResult * n).from_buffer_copy(results.cpu().numpy().tobytes())
    for i in range(n):
        lo, hi = starts[i], starts[i] + caps[i]
        assert bool((dst[lo - GAP:lo] == PAT).all()) and bool((dst[hi:hi + GAP] == PAT).all()), f"frame {i}: guard gap overwritten"
    del src, descs, results
    return dst, starts, res


def out_digest(dst, start, n):
    return LF.digest(dst[start:start + n].cpu().numpy())


@pytest.fixture(scope="module")
def sized():
    """[(name, frame, size, libzstd digest, oracle status, oracle result)]: RLE/Raw and libzstd text (windowLog 23; windowLog 27
    with long-distance matching) at every size of SIZES."""
    out = []
    for n in SIZES:
        # pure RLE (a few KiB of frame: one warp in the default mode) and RLE with Raw blocks (a CTA)
        blocks, content = LF.fill_blocks(n, seed=n & 0xFFFF, raw_every=256 if n in (LF.M28 - 1, 300 << 20) else 0)
        out.append((f"fill_{n}", LF.frame(blocks, n, xxh=LF.xxh32_low(content)), n))
        del content
    data = LF.text(max(SIZES))
    for wl, ldm in ((23, False), (27, True)):
        for n in SIZES:
            out.append((f"text_wl{wl}_{n}", LF.compress(data[:n], wl, ldm=ldm), n))
    del data
    rows = []
    for name, f, n in out:
        st, res = LF.oracle_decode(f, n)
        assert st == 0, name
        rows.append((name, f, n, LF.digest(LF.libzstd_decode(f, n)), res))
    return rows


def _fields_equal(r, o, tag):
    for k in FIELDS:
        assert getattr(r, k) == getattr(o, k), (tag, k, getattr(r, k), getattr(o, k))


@pytest.mark.parametrize("ctx", MODES, indirect=True)
def test_sizes_around_2_28_match_libzstd_and_oracle(ctx, sized):
    dst, starts, res = decode(ctx, [s[1] for s in sized], [s[2] for s in sized])
    for (name, f, n, dig, ores), r, st in zip(sized, res, starts):
        assert r.status == 0, (name, czb.status_name(r.status))
        _fields_equal(r, ores, name)
        assert r.checksum_calculated == r.checksum_from_data, name
        assert out_digest(dst, st, n) == dig, name


@pytest.fixture(scope="module")
def seams():
    rows = []
    for c in LF.seam_cases():
        st, res = LF.oracle_decode(c.frame, c.cap)
        dig = LF.digest(LF.libzstd_decode(c.frame, c.out)) if c.gpu == "exact" else None
        rows.append((c, st, res, dig))
    return rows


@pytest.mark.parametrize("ctx", MODES, indirect=True)
def test_offsets_at_the_2_28_seam(ctx, seams):
    dst, starts, res = decode(ctx, [s[0].frame for s in seams], [s[0].cap for s in seams])
    for (c, ost, ores, dig), r, st in zip(seams, res, starts):
        tag = (c.name, czb.status_name(r.status), czb.status_name(ost))
        if c.gpu == "exact":
            assert r.status == 0 and ost == 0, tag
            _fields_equal(r, ores, c.name)
            assert out_digest(dst, st, c.out) == dig, c.name
        elif c.gpu == "oracle":
            assert r.status == ost, tag
        else:
            assert czb.status_name(r.status) == c.gpu, tag


@pytest.fixture(scope="module")
def limit_frames():
    """2^31 - 1 bytes (with checksum), 2^31 bytes, in RLE blocks of one value."""
    content = np.full(LF.MAX_OUT, 0x5A, dtype=np.uint8)
    xxh = LF.xxh32_low(content)
    del content
    return LF.frame(LF.rle_only(LF.MAX_OUT), LF.MAX_OUT, xxh=xxh), LF.frame(LF.rle_only(LF.MAX_OUT + 1), LF.MAX_OUT + 1)


@pytest.mark.parametrize("ctx", MODES + ["warp"], indirect=True)
def test_the_2_31_limit(ctx, limit_frames):
    top, over = limit_frames
    dst, starts, res = decode(ctx, [top, over, top], [LF.MAX_OUT, LF.MAX_OUT + 1, LF.MAX_OUT - 1])
    assert res[0].status == 0 and res[0].bytes_written == LF.MAX_OUT and res[0].finished == 1
    assert res[0].checksum_calculated == res[0].checksum_from_data
    assert bool((dst[starts[0]:starts[0] + LF.MAX_OUT] == 0x5A).all())
    assert czb.status_name(res[1].status) == "CZS_UNSUPPORTED"
    assert czb.status_name(res[2].status) == "CZS_DST_TOO_SMALL"


@pytest.mark.parametrize("ctx", ["default"], indirect=True)
def test_frame_sizes_without_content_size(ctx, sized):
    frames, sizes = [], []
    for n in SIZES:
        blocks, _ = LF.fill_blocks(n, seed=3, raw_every=256)
        frames.append(LF.frame(blocks, n, fcs_width=0, single_segment=False, window_log=27)); sizes.append(n)
    frames.append(LF.compress(LF.text(LF.M28, seed=11), 27, ldm=True, content_size=False)); sizes.append(LF.M28)
    for f in frames:
        assert czb.frame_header_info(f).fcs_present == 0
    res = ctx.frame_sizes(frames)
    for r, n in zip(res, sizes):
        assert r.status == 0 and r.bytes_written == n, (r.status, r.bytes_written, n)


@pytest.mark.parametrize("ctx", ["default"], indirect=True)
def test_handle_decodes_a_large_frame(ctx, sized):
    name, f, n, dig, ores = next(s for s in sized if s[0] == f"fill_{LF.M28}")
    source = ByteSlice(f)
    dec = czb.FrameDecoder.new(czb.FrameDecoderState.new(source, ctx))
    assert dec.decode_blocks(source, czb.BlockDecodingStrategy.All()) is True
    got = dec.collect()
    assert len(got) == n and LF.digest(np.frombuffer(got, dtype=np.uint8)) == dig
    assert dec.get_checksum_from_data() == ores.checksum_from_data
