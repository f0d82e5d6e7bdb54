"""-m gpu: the Huffman literals families of tests/huffamilies.py -- both k_huff table classes, every stream layout and head length,
the loop thresholds of k_huff's decode loop, Treeless chains, layouts only the reference accepts and sections that are invalid
by construction -- decoded in one batch per family, through the default executor choice and with every frame forced through each
CTA-per-frame executor.  Every result field must equal the oracle's, the output the reference's, the device XXH64 the trailer,
and the flow executor's spin-limit safety net must not have fired.  Beyond the frame results: the literal scratch of every
Huffman section that must decode equals the builder's literals (a k_huff fault shows there even when a later stage fails the
frame), the scratch guards stay intact, and a Treeless block decodes in a later handle call than its tree."""
import ctypes as C
import random

import numpy as np
import pytest

import gpu_common as G
import hufbuild as H
import huffamilies as HF
import oracle_lib as O
import seqbuild as S
import cairo_zstd_b200 as czb
from cairo_zstd_b200 import api
from cairo_zstd_b200.frame_decoder import ByteSlice
from hufbuild import Huf, Treeless

pytestmark = pytest.mark.gpu
MODES = ["default", "flow-narrow", "flow-wide", "big"]


def _context(monkeypatch, mode, guard=False):
    if guard:
        monkeypatch.setenv("CZB_GUARD", "1")
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


def _check_results(cases, outs, res):
    for c, o, r in zip(cases, outs, res):
        if isinstance(c.expected, bytes):
            assert o == c.expected, c.name
            assert r.checksum_calculated == r.checksum_from_data, c.name
        else:
            assert czb.status_name(r.status) == c.expected, (c.name, czb.status_name(r.status))


def _check_literal_scratch(ctx, cases):
    """Every Huffman section that must decode (no declared failure, and a tree in its frame) has status 0 in the last wave's
    block table and its literals in the literal scratch.  The batch must have been one wave."""
    blocks, lits, _ = ctx.debug_last_wave()
    per_frame = {}
    for b in blocks:
        per_frame.setdefault(b.frame, []).append(b)
    checked = 0
    for i, c in enumerate(cases):
        dbg = per_frame.get(i, [])
        assert len(dbg) >= len(c.blocks), (c.name, len(dbg), len(c.blocks))
        have_tree = False
        for spec, d in zip(c.blocks, dbg):
            h = getattr(spec, "literals", None)
            if not isinstance(h, Huf):
                continue
            if h.expect is None and (h.tree is not None or have_tree):
                assert d.status == 0, (c.name, czb.status_name(d.status))
                got = lits[d.lit_off:d.lit_off + d.regen_size]
                assert got == h.data, (c.name, d.lit_off, next((k for k in range(len(got)) if got[k] != h.data[k]), -1))
                checked += 1
            have_tree = have_tree or (h.tree is not None and h.expect is None)
    return checked


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("family", sorted(HF.FAMILIES))
def test_huffman_families_match_reference_and_oracle(monkeypatch, family, mode):
    cases = HF.cases(family)
    assert len(cases) <= 128   # one wave, so that the debug taps see the whole batch
    ctx = _context(monkeypatch, mode)
    outs, res = G.compare_with_oracle([c.frame for c in cases], [c.cap for c in cases], label=f"{family}/{mode}")
    _check_results(cases, outs, res)
    if mode == "default":
        assert _check_literal_scratch(ctx, cases) > 0
    else:
        _watchdog_clear()
    ctx.close()


def test_all_families_shuffled_into_one_batch(monkeypatch):
    """k_huff's warps take 8 sections each: here they mix 1- and 4-stream sections, both classes, failing and good sections;
    the number of Huffman sections is not a multiple of 8."""
    cases = [c for f in sorted(HF.FAMILIES) for c in HF.cases(f)]
    random.Random(41).shuffle(cases)
    n_huf = lambda cs: sum(isinstance(getattr(b, "literals", None), Huf) for c in cs for b in c.blocks)
    while n_huf(cases) % 8 == 0:
        cases.pop()
    ctx = _context(monkeypatch, "default")
    outs, res = G.compare_with_oracle([c.frame for c in cases], [c.cap for c in cases], label="shuffled")
    _check_results(cases, outs, res)
    ctx.close()


GAP = 64
PAT = 0xA5


@pytest.mark.parametrize("mode", ["default", "big"])
def test_huffman_frames_stay_inside_their_spans_and_scratch(monkeypatch, mode):
    """CZB_GUARD=1 and the outputs laid out with exact capacities and 64-byte gaps at odd alignments: no byte outside a
    frame's span changes, and the guard bytes behind the literal scratch (k_huff's 16-byte stores) stay intact, oversized
    sections included."""
    import torch
    cases = [c for f in ("refonly", "streams", "invalid", "treeless") for c in HF.cases(f)]
    ctx = _context(monkeypatch, mode, guard=True)
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
    assert ctx.guard_faults() == 0
    ctx.close()


def _getters_equal(dec, ofd):
    r = O.OracleResult()
    O.lib().oracle_fd_getters(ofd, C.byref(r))
    assert dec.blocks_decoded() == r.blocks_decoded
    assert dec.bytes_read_from_source() == r.bytes_read
    assert dec.is_finished() == bool(r.finished)
    assert dec.get_calculated_checksum() == r.checksum_calculated


def test_treeless_block_in_a_later_handle_call_than_its_tree():
    """Compressed -> Raw -> Treeless (1 and 4 streams, one with sequences) -> Compressed in the other class -> Treeless, one
    block per decode_from_to call: each Treeless section's tree belongs to a block an earlier device call executed."""
    rng = random.Random(42)
    nrng = np.random.default_rng(42)
    l8 = H.complete_lengths(list(range(97, 123)), 8)
    l11 = H.complete_lengths(list(range(60, 72)), 11)
    d = [HF.draw(nrng, l8, n) for n in (3000, 900, 2000)] + [HF.draw(nrng, l11, n) for n in (2500, 800)]
    seqs = HF.with_seqs(rng, len(d[2]), 3000 + 500 + 900)
    blocks = [S.Seqs(Huf(d[0], H.weights_of(l8), 8, ("fse", 6), 4), []), S.Raw(bytes(rng.getrandbits(8) for _ in range(500))),
              S.Seqs(Treeless(d[1], 1), []), S.Seqs(Treeless(d[2], 4), seqs),
              S.Seqs(Huf(d[3], H.weights_of(l11), 11, "direct", 4), []), S.Rle(0x44, 100), S.Seqs(Treeless(d[4], 4), [])]
    c = HF.case("handle-treeless", blocks, single_segment=False, window_log=17)
    f = c.frame
    L = O.lib()
    source = ByteSlice(f)
    dec = czb.FrameDecoder.new(czb.FrameDecoderState.new(source))
    used, st = C.c_size_t(), C.c_int32()
    ofd = L.oracle_fd_new(f, len(f), C.byref(used), 0, C.byref(st))
    assert st.value == 0 and source.pos == used.value
    pos = used.value
    obuf = C.create_string_buffer(len(c.expected) + 64)
    total = bytearray()
    for k in range(len(blocks)):
        bh = int.from_bytes(f[pos:pos + 3], "little")
        end = pos + 3 + (1 if (bh >> 1) & 3 == 1 else bh >> 3)
        chunk = f[pos:] if k == len(blocks) - 1 else f[pos:end]
        target = bytearray()
        C.memset(obuf, 0, len(obuf))
        rl, wr = dec.decode_from_to(chunk, target, cap=len(obuf))
        orl, owr = C.c_size_t(), C.c_size_t()
        assert L.oracle_fd_decode_from_to(ofd, chunk, len(chunk), obuf, len(obuf), C.byref(orl), C.byref(owr)) == 0
        assert (rl, wr) == (orl.value, owr.value) and rl == len(chunk), (k, rl, wr, orl.value, owr.value)
        assert bytes(target) == obuf.raw[:owr.value], k
        total += target
        _getters_equal(dec, ofd)
        pos += rl
    assert dec.is_finished()
    for _ in range(2):
        t = bytearray()
        C.memset(obuf, 0, len(obuf))
        n = dec.read(t, cap=len(obuf))
        assert n == L.oracle_fd_read(ofd, obuf, len(obuf)) and bytes(t) == obuf.raw[:n]
        total += t
    L.oracle_fd_free(ofd)
    assert bytes(total[:len(c.expected)]) == c.expected
    runs, executed = dec.device_work()
    assert executed == dec.blocks_decoded() == len(blocks) and runs >= 2, (runs, executed)
