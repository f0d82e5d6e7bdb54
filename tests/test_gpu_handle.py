"""-m gpu parity tests for the rest of the FrameDecoder handle surface (SURVEY.md section 8 rows a2, a4, f3):
FrameDecoderStateTrait::reset incl. the 100 MiB WindowSizeTooBig check (src/frame_decoder.cairo:78-105, :92-94),
FrameDecoderTrait::read (:328-334) and decode_from_to (:245-326) with small feeds, including the
RingBuffer::len quirk (src/decoding/ring_buffer.cairo:20-22), call by call against the oracle's restatement
of the same state machine (oracle_fd_*).  Everything goes through the C ABI (czb_fd_*).

The tests after those run tests/fdscript.py's scripts on the handle and the oracle call by call: every device run of the
handle RESUMES after the blocks earlier runs executed (FrameResume), under each executor: k_exec ("default", "warp": every
frame on the per-warp path), k_exec_flow narrow and wide, k_exec_big.  Every case of every seqfamilies / huffamilies family
block by block (the seams scripts), ragged / chunked / shrink / reset scripts over samples of them, corpus frames and libzstd
frames, and the handle's behaviour on failing calls."""
import ctypes as C
import struct

import pytest

import fdscript as D
import oracle_lib as O
import seqfamilies as F
import cairo_zstd_b200 as czb
from cairo_zstd_b200.frame_decoder import ByteSlice
from gpu_common import sha

pytestmark = pytest.mark.gpu

CZS_WINDOW_SIZE_TOO_BIG = 11


def _idx(corpus, name):
    return next(k for k, e in enumerate(corpus.index) if e["name"] == name)


def _oracle_new(f, flags=0):
    L = O.lib()
    used, st = C.c_size_t(), C.c_int32()
    h = L.oracle_fd_new(f, len(f), C.byref(used), flags, C.byref(st))
    return h, used.value, st.value


def _getters_equal(dec, ofd):
    r = O.OracleResult()
    O.lib().oracle_fd_getters(ofd, C.byref(r))
    assert dec.blocks_decoded() == r.blocks_decoded
    assert dec.bytes_read_from_source() == r.bytes_read
    assert dec.content_size() == r.content_size
    assert dec.is_finished() == bool(r.finished)
    got = dec.get_checksum_from_data()
    assert (got is not None) == bool(r.has_checksum)
    if got is not None:
        assert got == r.checksum_from_data
    assert dec.get_calculated_checksum() == r.checksum_calculated


def test_fd_reset_reuses_the_handle_like_the_reference(corpus):
    """new(A) -> decode -> reset(B) -> decode -> reset(A) ...: every getter equals the oracle's after each call."""
    L = O.lib()
    names = ["z000001", "z000033", "z000062", "z000009", "z000035"]  # incl. an empty original and a single-segment frame
    frames = [corpus.frame(_idx(corpus, n)) for n in names]
    source = ByteSlice(frames[0])
    state = czb.FrameDecoderState.new(source)
    dec = czb.FrameDecoder.new(state)
    ofd, opos, st = _oracle_new(frames[0])
    assert st == 0 and source.pos == opos
    obuf = C.create_string_buffer(1 << 21)
    for k, f in enumerate(frames):
        if k:
            source = ByteSlice(f)
            state.reset(source)
            dec.reset(state)
            used = C.c_size_t()
            assert L.oracle_fd_reset(ofd, f, len(f), C.byref(used)) == 0
            opos = used.value
            assert source.pos == opos
            _getters_equal(dec, ofd)  # counters cleared by reset (:78-105)
        fin = dec.decode_blocks(source, czb.BlockDecodingStrategy.All())
        ofin, oused = C.c_int32(), C.c_size_t()
        assert L.oracle_fd_decode_blocks(ofd, f[opos:], len(f) - opos, C.byref(oused), 0, 0, C.byref(ofin)) == 0
        assert fin == bool(ofin.value) and source.pos == opos + oused.value
        assert dec.can_collect() == L.oracle_fd_can_collect(ofd)
        got = dec.collect()
        wrote = C.c_size_t()
        assert L.oracle_fd_collect(ofd, obuf, len(obuf), C.byref(wrote)) == 1
        assert got == obuf.raw[:wrote.value]
        assert sha(got) == corpus.index[_idx(corpus, names[k])]["orig_sha256"]
        _getters_equal(dec, ofd)
    L.oracle_fd_free(ofd)


def test_fd_reset_rejects_windows_above_100_mib_but_new_accepts_them(corpus):
    """frame_decoder.cairo:92-94: only `reset` has the 100 MiB limit; `new` (:54-76) does not."""
    L = O.lib()
    good = corpus.frame(_idx(corpus, "z000001"))
    # magic, descriptor 0 (no single segment, no checksum, no FCS field), window descriptor exponent 17 -> 128 MiB
    big = struct.pack("<IBB", 0xFD2FB528, 0x00, 17 << 3) + b"\x01\x00\x00"
    just_ok = struct.pack("<IBB", 0xFD2FB528, 0x00, (16 << 3) | 4) + b"\x01\x00\x00"  # 64 MiB * 1.5 = 96 MiB <= 100 MiB
    # new accepts both
    for f in (big, just_ok):
        s = ByteSlice(f)
        czb.FrameDecoderState.new(s)
        h, used, st = _oracle_new(f)
        assert st == 0 and s.pos == used == 6
        L.oracle_fd_free(h)
    # reset: too big -> WindowSizeTooBig on both sides; 96 MiB passes
    source = ByteSlice(good)
    state = czb.FrameDecoderState.new(source)
    ofd, _, st = _oracle_new(good)
    assert st == 0
    with pytest.raises(czb.FrameDecoderError) as ei:
        state.reset(ByteSlice(big))
    used = C.c_size_t()
    ost = L.oracle_fd_reset(ofd, big, len(big), C.byref(used))
    assert ei.value.status == ost == CZS_WINDOW_SIZE_TOO_BIG
    s2 = ByteSlice(just_ok)
    state.reset(s2)
    assert L.oracle_fd_reset(ofd, just_ok, len(just_ok), C.byref(used)) == 0 and s2.pos == used.value
    # every other header-level error comes out of reset exactly as out of new
    for bad in (b"", b"\x28\xb5\x2f", struct.pack("<I", 0x184D2A50) + b"\x04\x00\x00\x00abcd", struct.pack("<IB", 0xFD2FB528, 0x00),
                struct.pack("<IBB", 0xFD2FB528, 0xC0, 0x00)):
        with pytest.raises(czb.FrameDecoderError) as ei:
            state.reset(ByteSlice(bad))
        assert ei.value.status == L.oracle_fd_reset(ofd, bad, len(bad), C.byref(used))
    L.oracle_fd_free(ofd)


@pytest.mark.parametrize("name,feed", [("z000033", 4096), ("z000035", 20000), ("z000011", 1 << 20), ("z000001", 7)])
def test_decode_from_to_with_small_feeds_matches_oracle(corpus, name, feed):
    """decode_from_to (:245-326): the caller hands over whatever source bytes it has; the decoder consumes whole blocks
    only, appends what may leave the window to `target` and reports (bytes read, bytes written)."""
    L = O.lib()
    i = _idx(corpus, name)
    f = corpus.frame(i)
    source = ByteSlice(f)
    dec = czb.FrameDecoder.new(czb.FrameDecoderState.new(source))
    ofd, opos, st = _oracle_new(f)
    assert st == 0 and source.pos == opos
    pos = opos
    obuf = C.create_string_buffer(corpus.index[i]["orig_len"] + 64)
    total, ototal = bytearray(), bytearray()
    window = feed
    for _ in range(200000):
        chunk = f[pos:pos + window]
        target = bytearray()
        C.memset(obuf, 0, len(obuf))
        rl, wr = dec.decode_from_to(chunk, target, cap=len(obuf))
        orl, owr = C.c_size_t(), C.c_size_t()
        assert L.oracle_fd_decode_from_to(ofd, chunk, len(chunk), obuf, len(obuf), C.byref(orl), C.byref(owr)) == 0
        assert (rl, wr) == (orl.value, owr.value), (name, pos, rl, wr, orl.value, owr.value)
        # `read` reports the amount it asked for (RingBuffer::len ignores head): the bytes really drained can be fewer, so
        # both sides start from zeroed buffers and the whole reported span is compared
        assert bytes(target) == obuf.raw[:owr.value], (name, pos)
        total += target
        _getters_equal(dec, ofd)
        assert dec.can_collect() == L.oracle_fd_can_collect(ofd)
        pos += rl
        if dec.is_finished() and pos >= len(f):
            break
        if rl == 0:
            assert window < len(f) * 2 + 16, "no progress"
            window *= 2  # not even one whole block in the feed: hand over more
        else:
            window = feed
    assert pos == len(f)
    # incremental, not quadratic: however small the feeds, every block is executed on the device exactly once
    runs, blocks = dec.device_work()
    assert blocks == dec.blocks_decoded(), (runs, blocks, dec.blocks_decoded())
    # drain the rest the way a caller would: read() until nothing comes
    for _ in range(4):
        t = bytearray()
        C.memset(obuf, 0, len(obuf))
        n = dec.read(t, cap=len(obuf))
        on = L.oracle_fd_read(ofd, obuf, len(obuf))
        assert n == on and bytes(t) == obuf.raw[:on]
        total += t
        _getters_equal(dec, ofd)
    L.oracle_fd_free(ofd)
    if name == "z000001":  # output smaller than the window: nothing leaves before the end, then everything at once, in order
        assert sha(bytes(total[:corpus.index[i]["orig_len"]])) == corpus.index[i]["orig_sha256"]


def test_read_after_partial_decode_follows_the_ring_buffer_len_quirk(corpus):
    """read (:328-334) after UptoBlocks: drains only what lies beyond the window until the frame is finished; because
    RingBuffer::len ignores `head` (ring_buffer.cairo:20-22) a second read() asks for the same amount again."""
    L = O.lib()
    i = _idx(corpus, "z000033")  # 986 blocks, window smaller than the output
    f = corpus.frame(i)
    source = ByteSlice(f)
    dec = czb.FrameDecoder.new(czb.FrameDecoderState.new(source))
    ofd, opos, st = _oracle_new(f)
    obuf = C.create_string_buffer(corpus.index[i]["orig_len"] + 64)
    total = bytearray()
    strat = czb.BlockDecodingStrategy.UptoBlocks(97)
    for _ in range(100):
        fin = dec.decode_blocks(source, strat)
        ofin, oused = C.c_int32(), C.c_size_t()
        assert L.oracle_fd_decode_blocks(ofd, f[opos:], len(f) - opos, C.byref(oused), 1, 97, C.byref(ofin)) == 0
        opos += oused.value
        assert source.pos == opos and fin == bool(ofin.value)
        for _ in range(2):  # twice: the second call exercises the quirk
            t = bytearray()
            C.memset(obuf, 0, len(obuf))
            n = dec.read(t, cap=len(obuf))
            on = L.oracle_fd_read(ofd, obuf, len(obuf))
            assert n == on and bytes(t) == obuf.raw[:on]
            total += t
            _getters_equal(dec, ofd)
        if fin:
            break
    assert dec.is_finished()
    L.oracle_fd_free(ofd)


# ---------------------------------------------------------------------------
# scripts, side by side with the oracle, under every executor
# ---------------------------------------------------------------------------
MODES = ["default", "warp", "flow-narrow", "flow-wide", "big"]


def _env(monkeypatch, mode, **knobs):
    """A context whose executor choice is forced (as test_gpu_verify.py's _env)."""
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


def _watchdog_clear():
    wd = (C.c_uint32 * 16)()
    czb.load_library().czb_debug_flow_watchdog(wd)
    assert wd[0] == 0, list(wd)


def _seams(ctx, c, label):
    lay = D.layout(c.frame)
    res = D.run(c.frame, D.seams(lay), ctx, label=f"{c.name}/{label}")
    D.check(c, "seams", res.epochs[0])
    if not lay.failing:   # one device run per block, and every block executed once
        assert res.device_work == (len(lay.blocks), len(lay.blocks)), (c.name, res.device_work, len(lay.blocks))
    return res


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("kind,name", D.family_names())
def test_seams_every_family_case(monkeypatch, kind, name, mode):
    """Every case, valid and invalid, decode_blocks(UptoBlocks(1)) per block with the span ending on that block's end: each
    device run executes one block on the output, history and counters of the runs before it."""
    ctx = _env(monkeypatch, mode)
    for c in D.family_cases(kind, name):
        _seams(ctx, c, mode)
    if mode != "default":
        _watchdog_clear()
    ctx.close()


def _script_frames(corpus):
    """(case, seed) of the ragged / chunked / shrink scripts: a fixed sample of each family, corpus frames, libzstd frames."""
    out = []
    for kind, name in D.family_names():
        out += [(c, k) for k, c in enumerate(D.sample(D.family_cases(kind, name)))]
    for name in D.CORPUS:
        i = _idx(corpus, name)
        f = corpus.frame(i)
        out.append((F.Case(name, f, O.decode_frame(f, dst_cap=corpus.index[i]["orig_len"] + 64)[1], 0), i))
    for wl, (f, data) in D.libzstd_frames().items():
        out.append((F.Case(f"libzstd-wl{wl}", f, data, len(data)), wl))
    return out


@pytest.mark.parametrize("mode", ["default", "warp"])
def test_ragged_chunked_shrink_scripts(monkeypatch, corpus, mode):
    """Span ends inside headers, bodies and the trailer under every strategy form; decode_from_to in chunks of 1, 3, 7, 4096
    bytes and a mix; spans that end before blocks the device already ran (the call fails as the oracle's does).  Under the
    two k_exec forms only (about 40 s each); the seams scripts cover every executor."""
    ctx = _env(monkeypatch, mode)
    for c, seed in _script_frames(corpus):
        lay = D.layout(c.frame)
        for sname, script in D.scripts(lay, seed):
            if sname == "chunked1" and len(c.frame) > 40000:
                continue
            res = D.run(c.frame, script, ctx, label=f"{c.name}/{sname}/{mode}")
            D.check(c, sname, res.epochs[0])
    if mode != "default":
        _watchdog_clear()
    ctx.close()


@pytest.mark.parametrize("mode", ["default", "big"])
def test_reset_in_the_middle_of_a_frame(monkeypatch, corpus, mode):
    """reset after a device run that executed blocks beyond block_counter, the other frame, then the first again block by
    block."""
    ctx = _env(monkeypatch, mode)
    pairs = [(F.cases("resume")[0], F.cases("repeat")[3]), (F.cases("resume")[-1], F.cases("resume")[17])]
    z = corpus.frame(_idx(corpus, "z000033"))
    pairs.append((F.cases("reach")[5], F.Case("z000033", z, O.decode_frame(z, dst_cap=1 << 24)[1], 0)))
    for a, b in pairs:
        res = D.run([a.frame, b.frame], D.reset(D.layout(a.frame)), ctx, label=f"reset {a.name} {b.name}")
        assert [e.frame for e in res.epochs] == [0, 1, 0]
        assert bytes(res.epochs[1].drained) == D.expected_output(b) and bytes(res.epochs[2].drained) == a.expected
    ctx.close()


@pytest.mark.parametrize("knob", ["CZB_OVERLAP", "CZB_GUARD"])
def test_resume_scripts_with_overlap_and_guard(monkeypatch, corpus, knob):
    ctx = _env(monkeypatch, "default", **{knob: 1})
    for c in F.cases("resume"):
        _seams(ctx, c, knob)
    f = corpus.frame(_idx(corpus, "z000033"))
    res = D.run(f, D.ragged(D.layout(f), __import__("random").Random(5)), ctx, label=f"z000033/ragged/{knob}")
    assert res.epochs[0].finished
    if knob == "CZB_GUARD":
        assert ctx.guard_faults() == 0
    ctx.close()


def test_failing_calls_consume_what_the_oracle_consumes():
    """A header error or a truncated body moves the caller's span 3 bytes on, a Compressed block whose body fails 3 +
    Block_Size; bytes_read_from_source counts 3 for a failing body, nothing for a header error.  Both call forms."""
    ctx = czb.Context(0)
    for frame, _, status, _, _ in D.failing_frames():
        for script in ([("blocks", None, D.ALL, 0), ("read",), ("collect",), ("blocks", None, D.ALL, 0), ("fromto", 64)],
                       [("blocks", None, D.UPTO_BLOCKS, 1), ("blocks", None, D.UPTO_BYTES, 1), ("read",)],
                       [("fromto*", [1, 5, 4096])]):
            res = D.run(frame, script, ctx, label=status)
            if script[0][0] != "fromto*" or status != "CZS_PANIC_TRUNCATED":   # decode_from_to waits for a truncated body
                assert czb.status_name(res.epochs[0].status) == status, (status, script[0])
    ctx.close()


def test_block_failing_in_execution_leaves_its_partial_output():
    """execute_sequences appends each sequence's literals before its offset checks, and the matches before the failing one:
    after the offset check fails the 300-byte Raw block is followed by 3 literals, a 4-byte match and 2 more literals
    (309 bytes), in collect(), read() and get_calculated_checksum alike."""
    ctx = czb.Context(0)
    c = next(c for c in F.cases("invalid") if c.name == "invalid-offset-past-start")
    for script in ([("fromto*", [4096]), ("collect",)], D.seams(D.layout(c.frame)),
                   [("blocks", None, D.ALL, 0), ("read",), ("read",), ("collect",)]):
        ep = D.run(c.frame, script, ctx, label=c.name).epochs[0]
        assert czb.status_name(ep.status) == c.expected == "CZS_OFFSET_TOO_BIG"
        assert len(ep.drained) == 309
    ctx.close()


def test_decode_calls_after_an_error_change_nothing():
    """After a failing call every later decode_blocks / decode_from_to returns the same status, consumes nothing and changes
    no getter, whatever span it is given; read, collect and the getters keep working (DESIGN.md section 6)."""
    ctx = czb.Context(0)
    for c in F.cases("invalid"):
        if D.expected_output(c) is not None:
            continue
        script = [("fromto", 1 << 20), ("blocks", None, D.ALL, 0), ("blocks", None, D.UPTO_BLOCKS, 1), ("fromto", 1 << 20),
                  ("read",), ("can_collect",), ("blocks", 0, D.ALL, 0), ("collect",), ("fromto", 3), ("read",)]
        ep = D.run(c.frame, script, ctx, label=c.name).epochs[0]
        assert czb.status_name(ep.status) == c.expected
    ctx.close()
