"""Scripts of FrameDecoder calls, run on the handle (czb_fd_*, cairo_zstd_b200.FrameDecoder) and on the oracle's restatement
of the same state machine (oracle_fd_*) side by side, call by call.

A script is a list of calls on one frame (`frames[0]`; `reset` switches between `frames`):

  ("blocks", end, kind, n)   decode_blocks over frame[pos:end] (end None: the rest), kind ALL / UPTO_BLOCKS / UPTO_BYTES
  ("fromto", size)           decode_from_to over frame[pos:pos + size]
  ("fromto*", sizes)         decode_from_to repeated, chunk sizes cycling through `sizes`, until an error or the end of the
                             frame (a call that reads nothing doubles the next chunk, as a caller would)
  ("read",) ("collect",) ("can_collect",)
  ("reset", k)               FrameDecoderState.reset on frames[k]

`pos` is the caller's position in the frame: ByteSlice.pos for decode_blocks, advanced by read_len for decode_from_to.
After every call the status, the consumed bytes (pos), `finished`, (read_len, written), the drained bytes, every getter and
can_collect() must be equal on both sides.  Drains start from zeroed buffers on both sides: `read` reports the amount it asked
for (RingBuffer::len ignores head), which can be more than it drained.

Once a decode call has failed, the handle refuses every later decode_blocks / decode_from_to with the same status and
changes nothing, where the oracle would read on from wherever the caller's span now starts with half-updated scratch
(DESIGN.md section 6).  From then on decode calls run on the handle only and must leave every getter as the oracle's stayed;
read, collect and the getters keep being compared.

The generators below build scripts from a frame's block layout (`layout`), seeded."""
import ctypes as C
import random
import struct
from dataclasses import dataclass, field

import oracle_lib as O

ALL, UPTO_BLOCKS, UPTO_BYTES = 0, 1, 2


def status_name(s):
    from cairo_zstd_b200.api import status_name as name
    return name(s)


# ---------------------------------------------------------------------------
# block layout of a frame
# ---------------------------------------------------------------------------
@dataclass
class Block:
    start: int          # first byte of the block header
    end: int            # first byte after the block content
    last: bool
    out: int            # bytes the block appends to the output; None: the oracle fails on this block
    status: int = 0


@dataclass
class Layout:
    hdr_len: int
    checksum: bool
    blocks: list
    frame_len: int
    total_out: int      # output of the blocks that decode

    @property
    def failing(self):
        return self.blocks and self.blocks[-1].out is None


def layout(frame):
    """Blocks of `frame` as the oracle decodes them one at a time: where each lies and what it appends."""
    L = O.lib()
    used, st = C.c_size_t(), C.c_int32()
    ofd = L.oracle_fd_new(frame, len(frame), C.byref(used), 0, C.byref(st))
    assert st.value == 0, status_name(st.value)
    pos = used.value
    checksum = bool((frame[4] >> 2) & 1)
    blocks, total = [], 0
    ln, hd = C.c_size_t(), C.c_size_t()
    try:
        while True:
            start = pos
            end = len(frame)
            if len(frame) - pos >= 3:
                a = frame[pos] | frame[pos + 1] << 8 | frame[pos + 2] << 16
                t, size = (a >> 1) & 3, a >> 3
                if t != 3 and size <= 1 << 17:
                    end = min(len(frame), pos + 3 + (1 if t == 1 else size))
            L.oracle_fd_buffer_state(ofd, C.byref(ln), C.byref(hd))
            before = ln.value
            cons, fin = C.c_size_t(), C.c_int32()
            s = L.oracle_fd_decode_blocks(ofd, frame[pos:], len(frame) - pos, C.byref(cons), UPTO_BLOCKS, 1, C.byref(fin))
            L.oracle_fd_buffer_state(ofd, C.byref(ln), C.byref(hd))
            last = bool(fin.value)
            if s != 0 and not (last and checksum and len(frame) - end < 4):
                blocks.append(Block(start, end, last, None, s))
                break
            blocks.append(Block(start, end, last, ln.value - before, s))
            total += ln.value - before
            pos += cons.value
            if last:
                break
    finally:
        L.oracle_fd_free(ofd)
    return Layout(used.value, checksum, blocks, len(frame), total)


# ---------------------------------------------------------------------------
# the two sides
# ---------------------------------------------------------------------------
class _OracleSide:
    def __init__(self, cap):
        self.L, self.fd = O.lib(), None
        self.buf = C.create_string_buffer(cap)

    def setup(self, frame, reset):
        used = C.c_size_t()
        if reset and self.fd:
            st = self.L.oracle_fd_reset(self.fd, frame, len(frame), C.byref(used))
        else:
            if self.fd:
                self.L.oracle_fd_free(self.fd)
            s = C.c_int32()
            self.fd = self.L.oracle_fd_new(frame, len(frame), C.byref(used), 0, C.byref(s))
            st = s.value
        return dict(status=st, consumed=used.value if st == 0 else 0)

    def _state(self):
        ln, hd = C.c_size_t(), C.c_size_t()
        self.L.oracle_fd_buffer_state(self.fd, C.byref(ln), C.byref(hd))
        return ln.value, hd.value

    def _zero(self):
        C.memset(self.buf, 0, len(self.buf))

    def decode_blocks(self, span, kind, n):
        used, fin = C.c_size_t(), C.c_int32()
        st = self.L.oracle_fd_decode_blocks(self.fd, span, len(span), C.byref(used), kind, n, C.byref(fin))
        return dict(status=st, consumed=used.value, finished=bool(fin.value) if st == 0 else None)

    def decode_from_to(self, span):
        self._zero()
        _, h0 = self._state()
        rl, wr = C.c_size_t(), C.c_size_t()
        st = self.L.oracle_fd_decode_from_to(self.fd, span, len(span), self.buf, len(self.buf), C.byref(rl), C.byref(wr))
        if st:
            return dict(status=st), b""
        _, h1 = self._state()
        return dict(status=0, read_len=rl.value, written=wr.value, data=self.buf.raw[:wr.value]), self.buf.raw[:h1 - h0]

    def read(self):
        self._zero()
        _, h0 = self._state()
        n = self.L.oracle_fd_read(self.fd, self.buf, len(self.buf))
        _, h1 = self._state()
        return dict(amount=n, data=self.buf.raw[:n]), self.buf.raw[:h1 - h0]

    def collect(self):
        self._zero()
        wr = C.c_size_t()
        rc = self.L.oracle_fd_collect(self.fd, self.buf, len(self.buf), C.byref(wr))
        data = self.buf.raw[:wr.value] if rc == 1 else None
        return dict(rc=rc, data=data), data or b""

    def can_collect(self):
        return self.L.oracle_fd_can_collect(self.fd)

    def getters(self):
        r = O.OracleResult()
        self.L.oracle_fd_getters(self.fd, C.byref(r))
        return dict(blocks_decoded=r.blocks_decoded, bytes_read=r.bytes_read, content_size=r.content_size,
                    finished=bool(r.finished), checksum_from_data=r.checksum_from_data if r.has_checksum else None,
                    calculated_checksum=r.checksum_calculated, can_collect=self.can_collect())

    def close(self):
        if self.fd:
            self.L.oracle_fd_free(self.fd)
            self.fd = None


class _HandleSide:
    def __init__(self, cap, ctx):
        import cairo_zstd_b200 as czb
        from cairo_zstd_b200.frame_decoder import ByteSlice
        self.czb, self.slice, self.ctx, self.cap = czb, ByteSlice, ctx, cap
        self.state = self.dec = None

    def setup(self, frame, reset):
        src = self.slice(frame)
        try:
            if reset and self.state:
                self.state.reset(src)
                self.dec.reset(self.state)
            else:
                self.state = self.czb.FrameDecoderState.new(src, self.ctx)
                self.dec = self.czb.FrameDecoder.new(self.state)
        except self.czb.FrameDecoderError as e:
            return dict(status=e.status, consumed=0)
        return dict(status=0, consumed=src.pos)

    def decode_blocks(self, span, kind, n):
        src = self.slice(span)
        try:
            fin = self.dec.decode_blocks(src, self.czb.BlockDecodingStrategy(kind, n))
            st = 0
        except self.czb.FrameDecoderError as e:
            fin, st = None, e.status
        return dict(status=st, consumed=src.pos, finished=fin)

    def decode_from_to(self, span):
        t = bytearray()
        try:
            rl, wr = self.dec.decode_from_to(span, t, cap=self.cap)
        except self.czb.FrameDecoderError as e:
            return dict(status=e.status)
        return dict(status=0, read_len=rl, written=wr, data=bytes(t))

    def read(self):
        t = bytearray()
        n = self.dec.read(t, cap=self.cap)
        return dict(amount=n, data=bytes(t))

    def collect(self):
        d = self.dec.collect()
        return dict(rc=1 if d is not None else 0, data=d)

    def can_collect(self):
        return self.dec.can_collect()

    def getters(self):
        d = self.dec
        return dict(blocks_decoded=d.blocks_decoded(), bytes_read=d.bytes_read_from_source(), content_size=d.content_size(),
                    finished=d.is_finished(), checksum_from_data=d.get_checksum_from_data(),
                    calculated_checksum=d.get_calculated_checksum(), can_collect=d.can_collect())


# ---------------------------------------------------------------------------
# the driver
# ---------------------------------------------------------------------------
@dataclass
class Epoch:
    """What one frame (from new / reset to the next reset) gave the caller."""
    frame: int
    drained: bytearray = field(default_factory=bytearray)
    status: int = 0     # first decode error, 0 if none
    finished: bool = False


@dataclass
class Result:
    epochs: list
    calls: int
    device_work: tuple  # the handle's (device runs, blocks executed on the device) at the end (None on the oracle alone)


def _show(v):
    if isinstance(v, (bytes, bytearray)):
        return f"<{len(v)} bytes {bytes(v[:16]).hex()}...>"
    return repr(v)


def _differ(a, b):
    if isinstance(a, (bytes, bytearray)) and isinstance(b, (bytes, bytearray)):
        k = next((i for i in range(min(len(a), len(b))) if a[i] != b[i]), min(len(a), len(b)))
        return f" (lengths {len(a)} / {len(b)}, first difference at {k})"
    return ""


def run(frames, script, ctx=None, label="", oracle_only=False, max_calls=1 << 20):
    """Run `script` on frames[0] (reset switches frames); returns a Result.  With oracle_only the handle is not touched."""
    if isinstance(frames, (bytes, bytearray)):
        frames = [bytes(frames)]
    # drains never exceed a frame's output; a failing block's partial output stays under a block's worth of matches
    cap = max(layout(f).total_out for f in frames) + (1 << 20)
    orc = _OracleSide(cap)
    hnd = None if oracle_only else _HandleSide(cap, ctx)
    where = [None]

    def eq(fld, h, o):
        assert h == o, f"{label}: call {where[0]}: {fld}: handle {_show(h)} oracle {_show(o)}{_differ(h, o)}"

    def both(fn, *a):
        o = getattr(orc, fn)(*a)
        od, drained = o if isinstance(o, tuple) else (o, None)
        if hnd is not None:
            h = getattr(hnd, fn)(*a)
            for k in set(od) | set(h):
                eq(f"{fn}.{k}", h.get(k), od.get(k))
        return od, drained

    cur = 0
    o = orc.setup(frames[0], False)
    assert o["status"] == 0, f"{label}: frame header: {status_name(o['status'])}"
    if hnd is not None:
        where[0] = "new"
        eq("new", hnd.setup(frames[0], False), o)
    pos = o["consumed"]
    ep = Epoch(0)
    epochs = [ep]
    calls = 0
    mult = 1

    def check_getters():
        if hnd is not None:
            hg, og = hnd.getters(), orc.getters()
            for k in og:
                eq(k, hg[k], og[k])

    def step(call):
        nonlocal pos, cur, ep, mult, calls
        calls += 1
        assert calls <= max_calls, f"{label}: more than {max_calls} calls"
        f = frames[cur]
        op = call[0]
        where[0] = f"{calls - 1} {call[0]}{call[1:]}"
        if op in ("blocks", "fromto"):
            if op == "blocks":
                end = len(f) if call[1] is None else max(pos, min(call[1], len(f)))
                span, args = f[pos:end], (call[2], call[3])
            else:
                assert mult <= 8 * len(f) + 64, f"{label}: decode_from_to makes no progress at {pos}"
                span, args = f[pos:pos + call[1] * mult], ()
            fn = "decode_blocks" if op == "blocks" else "decode_from_to"
            if ep.status:
                # a decode after an error: the handle returns the same status and changes nothing; the oracle is not asked
                if hnd is not None:
                    before = hnd.getters()
                    h = getattr(hnd, fn)(span, *args)
                    eq(f"{fn}.status after {status_name(ep.status)}", h["status"], ep.status)
                    if op == "blocks":
                        eq(f"{fn}.consumed after an error", h["consumed"], 0)
                    eq("getters after a refused call", hnd.getters(), before)
                    check_getters()
                return
            od, drained = both(fn, span, *args)
            if od["status"]:
                ep.status = od["status"]
                if op == "blocks":
                    pos += od["consumed"]
            elif op == "blocks":
                pos += od["consumed"]
            else:
                pos += od["read_len"]
                ep.drained += drained
                mult = 1 if od["read_len"] else mult * 2
        elif op in ("read", "collect"):
            _, drained = both(op)
            ep.drained += drained
        elif op == "can_collect":
            o = orc.can_collect()
            if hnd is not None:
                eq("can_collect", hnd.can_collect(), o)
        elif op == "reset":
            cur = call[1]
            o = orc.setup(frames[cur], True)
            if hnd is not None:
                eq("reset", hnd.setup(frames[cur], True), o)
            assert o["status"] == 0, f"{label}: reset: {status_name(o['status'])}"
            pos = o["consumed"]
            ep = Epoch(cur)
            epochs.append(ep)
            mult = 1
        else:
            raise ValueError(call)
        check_getters()
        ep.finished = orc.getters()["finished"]

    for call in script:
        if call[0] == "fromto*":
            sizes = call[1]
            k = 0
            # until an error or the end of the frame (a trailer fed in pieces of fewer than 4 bytes is never read: decode_from_to
            # reports 4 bytes read without taking the checksum, frame_decoder.cairo:256-267)
            while not ep.status and pos < len(frames[cur]):
                size, before = sizes[k % len(sizes)], pos
                whole = pos + size * mult >= len(frames[cur])
                step(("fromto", size))
                k += 1
                if whole and pos == before:     # the rest of the frame holds no whole block (a truncated frame)
                    break
        else:
            step(call)
    orc.close()
    return Result(epochs, calls, hnd.dec.device_work() if hnd is not None else None)


# ---------------------------------------------------------------------------
# script generators
# ---------------------------------------------------------------------------
def _end_with_trailer(lay, b):
    return b.end + (4 if b.last and lay.checksum else 0)


def seams(lay):
    """One decode_blocks(UptoBlocks(1)) per block, the span ending exactly at that block's end (the last block's with the
    checksum trailer): every device run executes one block.  A frame that fails gets one more decode call."""
    calls = []
    for i, b in enumerate(lay.blocks):
        calls.append(("blocks", _end_with_trailer(lay, b), UPTO_BLOCKS, 1))
        calls.append(("read",) if i % 2 else ("collect",))
    if lay.failing:
        calls.append(("blocks", None, ALL, 0))
    calls.append(("collect",))
    return calls


def _stop(lay, b, kind, n):
    """Index after the last block a decode_blocks call starting at block b reaches (the block loop of decode_blocks)."""
    produced, k = 0, b
    while k < len(lay.blocks):
        blk = lay.blocks[k]
        k += 1
        if blk.out is None or blk.last:
            return k
        produced += blk.out
        if kind == UPTO_BLOCKS and k - b >= n:
            return k
        if kind == UPTO_BYTES and produced >= n:
            return k
    return k


def ragged(lay, rng):
    """decode_blocks with span ends inside a block header, inside a body, on a block end and 0-3 bytes into the checksum
    trailer, under UptoBlocks(1..3), UptoBytes(1), UptoBytes(a block's exact output) and that output minus 1; each call's
    strategy stops before the first block its span does not hold (a frame that fails does fail, on its failing block)."""
    bl = lay.blocks
    calls, b = [], 0
    while b < len(bl):
        opts = []
        for j in range(b, min(len(bl), b + 6)):
            blk = bl[j]
            opts.append(blk.end)
            if j > b:
                opts += [blk.start + 1, blk.start + 2]
                if blk.end - blk.start > 3:
                    opts.append(blk.start + 3 + rng.randrange(blk.end - blk.start - 3))
            if blk.last and lay.checksum:
                opts += [blk.end + d for d in range(4)]
        for _ in range(50):
            end = rng.choice(opts)
            w = b
            while w < len(bl) and _end_with_trailer(lay, bl[w]) <= end:
                w += 1
            out = bl[b].out or 0
            strat = [(UPTO_BLOCKS, k) for k in (1, 2, 3)] + [(UPTO_BYTES, 1), (UPTO_BYTES, out)] + ([(UPTO_BYTES, out - 1)] if out > 1 else [])
            ok = [s for s in strat if _stop(lay, b, *s) <= w]
            if ok:
                break
        else:
            end, ok = _end_with_trailer(lay, bl[b]), [(UPTO_BLOCKS, 1)]
        kind, n = rng.choice(ok)
        calls.append(("blocks", end, kind, n))
        b = _stop(lay, b, kind, n)
        r = rng.random()
        if r < 0.3:
            calls.append(("read",))
        elif r < 0.6:
            calls.append(("collect",))
    calls += [("read",), ("collect",)]
    return calls


CHUNKS = (1, 3, 7, 4096)


def chunked(rng=None, size=None):
    """decode_from_to with one chunk size, or (rng) a random mix of sizes."""
    sizes = [size] if size is not None else [rng.choice([1, 2, 3, 5, 7, 16, 100, 700, 4096, 20000, 1 << 17]) for _ in range(61)]
    return [("fromto*", sizes), ("read",), ("read",)]


def shrink(lay, rng):
    """UptoBlocks(1) over the whole remainder (the device runs every block), a few calls whose span ends on the next block's
    end, then a span that ends inside a block the device already ran, header or body, under a strategy that reaches it: the
    call fails as the oracle does.  None for a frame of fewer than two blocks."""
    bl = lay.blocks
    if len(bl) < 2 or bl[0].out is None:
        return None
    calls = [("blocks", None, UPTO_BLOCKS, 1)]
    b = 1
    while b < len(bl) - 1 and bl[b].out is not None and rng.random() < 0.5:
        calls.append(("blocks", bl[b].end, UPTO_BLOCKS, 1))
        b += 1
    j = b + rng.randrange(len(bl) - b)
    blk = bl[j]
    ends = [blk.start, blk.start + 1, blk.start + 2]
    if blk.end - blk.start > 4:
        ends.append(blk.start + 3 + rng.randrange(blk.end - blk.start - 4))
    calls.append(("blocks", rng.choice(ends), UPTO_BLOCKS, j - b + 2))
    calls += [("read",), ("can_collect",), ("collect",), ("blocks", None, ALL, 0), ("fromto", 4096), ("read",)]
    return calls


def shrink_from_to(lay, rng):
    """UptoBlocks(1) over the whole remainder, then decode_from_to over short chunks: decode_from_to asks "enough bytes?"
    of the new span before it uses a block the device already ran."""
    if len(lay.blocks) < 2 or lay.blocks[0].out is None:
        return None
    return [("blocks", None, UPTO_BLOCKS, 1)] + chunked(rng)


def reset(lay):
    """reset in the middle of the frame after a device run past block_counter, then the other frame, then this frame again
    block by block."""
    return ([("blocks", None, UPTO_BLOCKS, 1), ("read",), ("reset", 1), ("blocks", None, ALL, 0), ("collect",), ("reset", 0)]
            + seams(lay))


def scripts(lay, seed, other=None):
    """The ragged, chunked, shrink (and, with another frame, reset) scripts of one frame: (name, script, frames index list)."""
    rng = random.Random(seed)
    out = [("ragged", ragged(lay, rng))]
    out += [(f"chunked{s}", chunked(size=s)) for s in CHUNKS]
    out.append(("chunked-mix", chunked(rng)))
    for name, s in (("shrink", shrink(lay, rng)), ("shrink-fromto", shrink_from_to(lay, rng))):
        if s is not None:
            out.append((name, s))
    if other is not None:
        out.append(("reset", reset(lay)))
    return out


# ---------------------------------------------------------------------------
# frames, and what the caller must get from them
# ---------------------------------------------------------------------------
def family_names():
    import huffamilies as HF
    import seqfamilies as F
    return [("seq", n) for n in sorted(F.FAMILIES)] + [("huf", n) for n in sorted(HF.FAMILIES)]


def family_cases(kind, name):
    import huffamilies as HF
    import seqfamilies as F
    return (F if kind == "seq" else HF).cases(name)


def sample(cases, n=4):
    """A fixed sample of about n cases of a family."""
    return cases[::max(1, len(cases) // n)]


def expected_output(c):
    """What the FrameDecoder drains from case c: its expected bytes; a frame that fails only for want of capacity decodes
    whole (the decoder's buffer grows); None for a frame that fails."""
    if isinstance(c.expected, bytes):
        return c.expected
    if c.expected == "CZS_DST_TOO_SMALL":
        st, out, _ = O.decode_frame(c.frame, dst_cap=1 << 24)
        assert st == 0
        return out
    return None


def check(c, script_name, ep):
    """A valid frame drains its output (a prefix of it when it did not finish); a failing frame fails with its status.
    Only the shrink scripts fail on a valid frame: their span ends before a block the call reaches."""
    want = expected_output(c)
    tag = (c.name, script_name, status_name(ep.status))
    if want is None:
        assert status_name(ep.status) == c.expected or script_name == "shrink", tag
        return
    if script_name == "shrink":
        assert status_name(ep.status) == "CZS_PANIC_TRUNCATED", tag
    else:
        assert ep.status == 0, tag
    if ep.finished:
        assert bytes(ep.drained) == want, tag
    else:   # a trailer fed in pieces of fewer than 4 bytes, or a shrink script
        assert script_name in ("shrink", "chunked1", "chunked3", "chunked-mix", "shrink-fromto"), tag
        assert want.startswith(bytes(ep.drained)), tag


CORPUS = ("z000033", "z000035")      # 986 blocks with a window smaller than the output; a large single-block-class frame
RAW0 = 103                           # bytes of the Raw block failing_frames() put first


def failing_frames():
    """(frame, span end, status, bytes a decode_blocks call over frame[header:span end] consumes after the Raw block in
    front, bytes it counts in bytes_read_from_source): block-header errors, truncated bodies and a compressed body that fails."""
    hdr = struct.pack("<IBB", 0xFD2FB528, 0x00, 0x00)        # no checksum, no content size, 1 KiB window
    raw = (100 << 3).to_bytes(3, "little") + bytes(range(100))

    def bh(last, t, size):
        return (last | t << 1 | size << 3).to_bytes(3, "little")
    bad_lits = bytes([20 << 3]) + b"abcd"                    # a Raw literals section of 20 bytes in a 5-byte block
    out = [
        (hdr + raw + bh(1, 3, 0), None, "CZS_FOUND_RESERVED_BLOCK", 3, 0),
        (hdr + raw + bh(1, 0, (1 << 17) + 1) + b"x" * 8, None, "CZS_BLOCK_SIZE_TOO_LARGE", 3, 0),
        (hdr + raw + bh(1, 0, 50) + b"y" * 20, None, "CZS_PANIC_TRUNCATED", 3, 3),
        (hdr + raw + bh(1, 1, 50), None, "CZS_PANIC_TRUNCATED", 3, 3),
        (hdr + raw + bh(1, 2, 50) + b"z" * 20, None, "CZS_PANIC_TRUNCATED", 3, 3),
        (hdr + raw + bh(1, 2, 5) + bad_lits, None, "CZS_MALFORMED_SECTION_HEADER", 8, 3),
        (hdr + raw + bh(1, 0, 10)[:2], None, "CZS_PANIC_TRUNCATED", 0, 0),
    ]
    return [(f, len(f) if e is None else e, s, c, n) for f, e, s, c, n in out]


_libzstd_frames = None


def libzstd_frames():
    """{window_log: (frame, data)} for window logs 10..17: libzstd frames of 300 KiB of text, with a checksum, with and
    without the content size."""
    global _libzstd_frames
    if _libzstd_frames is None:
        from cairo_zstd_b200 import workloads as W
        z = W.libzstd()
        _libzstd_frames = {}
        for wl in range(10, 18):
            data = W.synth_text(300 << 10, 40 + wl)
            cctx = z.ZSTD_createCCtx()
            try:
                for p, v in ((100, 3), (101, wl), (201, 1), (200, wl % 2)):   # level, windowLog, checksum, content size
                    assert not z.ZSTD_isError(z.ZSTD_CCtx_setParameter(cctx, p, v)), (p, v)
                bound = z.ZSTD_compressBound(len(data))
                buf = C.create_string_buffer(bound)
                n = z.ZSTD_compress2(cctx, buf, bound, data, len(data))
                assert not z.ZSTD_isError(n)
            finally:
                z.ZSTD_freeCCtx(cctx)
            _libzstd_frames[wl] = (buf.raw[:n], data)
    return _libzstd_frames
