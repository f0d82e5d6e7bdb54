"""A zstd frame builder driven by explicit sequences (RFC 8878), and a plain reference executor for what it builds.

Where an encoder decides what a frame contains, this module takes it from the caller: every block is given as
`Raw(bytes)`, `Rle(byte, n)` or `Seqs(literals, seqs, tables=...)` with `seqs` a list of `(ll, ml, ofv)` triples, so that a
test can put a match, a literal run or a repeat code exactly where a decoder changes its behaviour.  `ofv` is zstd's offset
value: 1..3 name the repeat offsets, anything larger is the offset + 3 (`off(n)`, `rep(k)`).

Table spec per stream (LL, OF, ML): "predefined", ("rle", code), ("fse", log), ("fse", log, probs) or "repeat" (the
previous block's table for that stream).  ("fse", log) derives normalized counts from the block's own code histogram.

The sequence bitstream is encoded backwards over each stream's decoding table: for the last sequence any state of its
symbol will do; for each earlier one, the unique state of its symbol whose [baseline, baseline + 2^nb) holds the next
state, the state bits being the difference.  Decoding tables come from the oracle's FSE table builder (the same
construction the decoder uses); libzstd decoding the frames is the independent check of the whole (tests/test_seqbuild.py).
"""
import struct
from dataclasses import dataclass

import handmade
import oracle_lib as O

MAGIC = struct.pack("<I", 0xFD2FB528)
BLOCK_MAX = 1 << 17

# RFC 8878 3.1.1.3.2.1.1: extra bits per literal-length / match-length code; baselines are the running sums of 2^bits
LL_BITS = [0] * 16 + [1, 1, 1, 1, 2, 2, 3, 3, 4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16]
ML_BITS = [0] * 32 + [1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16]


def _baselines(bits, first):
    out, b = [], first
    for n in bits:
        out.append(b)
        b += 1 << n
    return out


LL_BASE = _baselines(LL_BITS, 0)
ML_BASE = _baselines(ML_BITS, 3)
assert LL_BASE[35] == 65536 and ML_BASE[52] == 65539 and ML_BASE[43] == 131
MAX_LOG = (9, 8, 9)          # LL, OF, ML accuracy log limits
PREDEF_LOG = (6, 5, 6)


def off(n):
    """Offset value of a plain offset n >= 1."""
    assert n >= 1
    return n + 3


def rep(k):
    """Offset value of repeat code k (1..3)."""
    assert 1 <= k <= 3
    return k


def _code(value, base):
    c = 0
    while c + 1 < len(base) and base[c + 1] <= value:
        c += 1
    return c


def ll_code(ll):
    assert 0 <= ll <= LL_BASE[35] + (1 << 16) - 1, ll
    return ll if ll < 16 else _code(ll, LL_BASE)


def ml_code(ml):
    assert 3 <= ml <= ML_BASE[52] + (1 << 16) - 1, ml
    return ml - 3 if ml < 35 else _code(ml, ML_BASE)


def of_code(ofv):
    assert 1 <= ofv < (1 << 32), ofv
    return ofv.bit_length() - 1


@dataclass
class Raw:
    data: bytes


@dataclass
class Rle:
    byte: int
    n: int


@dataclass
class Seqs:
    """A compressed block.  literals: bytes (Raw literals section), ("rle", byte, n) or a Huffman section spec
    (tests/hufbuild.py: Huf, Treeless).  seqs: [(ll, ml, ofv)].
    tables: (LL, OF, ML) specs.  nbseq_form: 1, 2 or 3 forces that number-of-sequences header form."""
    literals: object
    seqs: list
    tables: tuple = ("predefined", "predefined", "predefined")
    nbseq_form: int = None


def _lit_bytes(lits):
    if isinstance(lits, tuple):
        assert lits[0] == "rle"
        return bytes([lits[1]]) * lits[2]
    return bytes(getattr(lits, "data", lits))


# ---------------------------------------------------------------------------
# reference executor
# ---------------------------------------------------------------------------
def reference_decode(blocks, window=None):
    """Execute the blocks byte by byte.  Returns the output, or the status name of the first failure (the oracle's leaf
    status: zstd_oracle.c execute_sequences / buf_repeat).  `window` only picks between the two names of a too-large offset."""
    out = bytearray()
    hist = [1, 4, 8]
    for b in blocks:
        if isinstance(b, Raw):
            out += b.data
        elif isinstance(b, Rle):
            out += bytes([b.byte]) * b.n
        else:
            lits = _lit_bytes(b.literals)
            pos = 0
            for ll, ml, ofv in b.seqs:
                if pos + ll > len(lits):
                    return "CZS_EXEC_NOT_ENOUGH_BYTES_FOR_SEQUENCE"
                out += lits[pos:pos + ll]
                pos += ll
                if ofv > 3:
                    o = ofv - 3
                    hist = [o, hist[0], hist[1]]
                elif ll > 0:
                    o = hist[ofv - 1]
                    if ofv == 2:
                        hist = [o, hist[0], hist[2]]
                    elif ofv == 3:
                        hist = [o, hist[0], hist[1]]
                else:
                    o = hist[1] if ofv == 1 else hist[2] if ofv == 2 else (hist[0] - 1) & 0xFFFFFFFF
                    hist = [o, hist[0], hist[2]] if ofv == 1 else [o, hist[0], hist[1]]
                if o == 0:
                    return "CZS_EXEC_ZERO_OFFSET"
                if o > len(out):
                    return "CZS_NOT_ENOUGH_BYTES_IN_DICTIONARY" if window is None or len(out) <= window else "CZS_OFFSET_TOO_BIG"
                start = len(out) - o
                if o >= ml:
                    out += out[start:start + ml]
                else:  # self-overlap: the match repeats the o bytes it starts on
                    out += (out[start:] * (ml // o + 1))[:ml]
            out += lits[pos:]
    return bytes(out)


# ---------------------------------------------------------------------------
# FSE tables
# ---------------------------------------------------------------------------
_table_cache = {}


def decoding_table(kind, log, probs):
    """(symbol, num_bits, baseline) per state, from the oracle's table builder.  kind 0/1/2 = LL/OF/ML; probs None = predefined."""
    import ctypes as C
    key = (kind, log, tuple(probs) if probs is not None else None)
    if key in _table_cache:
        return _table_cache[key]
    L = O.lib()
    n = 1 << 12
    bl = (C.c_uint32 * n)(); nb = (C.c_uint8 * n)(); sym = (C.c_uint8 * n)()
    if probs is None:
        size = C.c_uint32()
        assert L.oracle_fse_predefined(kind, bl, nb, sym, C.byref(size)) == 0
        size = size.value
    else:
        p = (C.c_int32 * len(probs))(*probs)
        assert L.oracle_fse_build_from_probs(log, p, len(probs), bl, nb, sym) == 0
        size = 1 << log
    t = [(sym[i], nb[i], bl[i]) for i in range(size)]
    _table_cache[key] = t
    return t


def normalized_counts(codes, log, extra=(), lt1=False):
    """Normalized counts summing to 2^log for the histogram of `codes`: every used code gets >= 1 (or -1, "less than one",
    when lt1 and its share is under one cell); `extra` symbols that are not used get one cell each (-1 when lt1)."""
    hist = {}
    for c in codes:
        hist[c] = hist.get(c, 0) + 1
    for c in extra:
        hist.setdefault(c, 0)
    total = 1 << log
    n = max(hist) + 1
    probs = [0] * n
    used = sum(hist.values())
    for c, k in hist.items():
        share = k * total // used if used else 0
        probs[c] = -1 if lt1 and share == 0 else max(1, share)
    assert sum(1 for p in probs if p) <= total, "more symbols than cells"
    while True:
        s = sum(abs(p) for p in probs)
        if s == total:
            return probs
        big = max(range(n), key=lambda c: probs[c])
        if s < total:
            probs[big] += total - s
        else:
            cut = min(s - total, probs[big] - 1)
            assert cut > 0, "cannot fit the histogram into the table"
            probs[big] -= cut


class _Stream:
    """One stream's table for a block: either an RLE code or a decoding table with a backwards state chooser."""

    def __init__(self, kind, spec, codes, prev):
        self.mode, self.desc, self.rle, self.table = None, b"", None, None
        if spec == "repeat":
            assert prev is not None, "repeat mode needs an earlier table"
            self.mode = 3
            self.rle, self.table = prev.rle, prev.table
        elif spec == "predefined":
            self.mode = 0
            self.table = decoding_table(kind, PREDEF_LOG[kind], None)
        elif spec[0] == "rle":
            self.mode, self.rle, self.desc = 1, spec[1], bytes([spec[1]])
        else:
            assert spec[0] == "fse"
            log = spec[1]
            probs = list(spec[2]) if len(spec) > 2 else normalized_counts(codes, log)
            self.mode = 2
            self.desc = handmade.fse_normalized_counts(log, probs)
            self.table = decoding_table(kind, log, probs)
        if self.table is not None:
            self.log = (len(self.table) - 1).bit_length()
            # pick[s][x] = the state of symbol s whose range holds next state x
            self.pick = {}
            for st, (s, nb, base) in enumerate(self.table):
                row = self.pick.setdefault(s, [None] * len(self.table))
                for x in range(base, base + (1 << nb)):
                    row[x] = st
        if self.rle is not None:
            assert all(c == self.rle for c in codes), "RLE table for a stream with several codes"

    def states(self, codes):
        """Decoder states for the sequence of symbols `codes` and the update bits (value, nb) between them."""
        n = len(codes)
        st = [0] * n
        row = self.pick.get(codes[-1])
        assert row is not None, f"symbol {codes[-1]} not in table"
        st[-1] = next(s for s in row if s is not None)
        ups = [None] * n
        for i in range(n - 2, -1, -1):
            row = self.pick.get(codes[i])
            assert row is not None, f"symbol {codes[i]} not in table"
            s = row[st[i + 1]]
            _, nb, base = self.table[s]
            st[i] = s
            ups[i] = (st[i + 1] - base, nb)
        return st, ups


def _block_header(last, btype, size):
    return (last | (btype << 1) | (size << 3)).to_bytes(3, "little")


def _lit_header(ltype, n):
    if n < 32:
        return bytes([ltype | (n << 3)])
    if n < 4096:
        return (ltype | (1 << 2) | (n << 4)).to_bytes(2, "little")
    assert n < (1 << 20)
    return (ltype | (3 << 2) | (n << 4)).to_bytes(3, "little")


def _nbseq_header(n, form):
    form = form or (1 if n < 128 else 2 if n < 0x7F00 else 3)
    if form == 1:
        assert n < 128
        return bytes([n])
    if form == 2:
        assert n < 0x7F00
        return bytes([(n >> 8) + 128, n & 255])
    assert 0x7F00 <= n < 0x7F00 + 0x10000
    return bytes([255]) + struct.pack("<H", n - 0x7F00)


def encode_seqs_block(b, prev, lit_state=None):
    """Body of one compressed block; `prev` = the (LL, OF, ML) streams of the last block that had sequences (for "repeat");
    `lit_state` = what the frame's Huffman sections so far left behind (the tree a Treeless section reuses)."""
    if isinstance(b.literals, tuple):
        lit = _lit_header(1, b.literals[2]) + bytes([b.literals[1]])
    elif hasattr(b.literals, "section"):
        lit = b.literals.section({} if lit_state is None else lit_state)
    else:
        lit = _lit_header(0, len(b.literals)) + bytes(b.literals)
    n = len(b.seqs)
    if n == 0:
        return lit + b"\x00", prev
    llc = [ll_code(ll) for ll, _, _ in b.seqs]
    ofc = [of_code(v) for _, _, v in b.seqs]
    mlc = [ml_code(ml) for _, ml, _ in b.seqs]
    streams = [_Stream(k, b.tables[k], codes, prev[k] if prev else None) for k, codes in enumerate((llc, ofc, mlc))]
    modes = (streams[0].mode << 6) | (streams[1].mode << 4) | (streams[2].mode << 2)
    hdr = _nbseq_header(n, b.nbseq_form) + bytes([modes]) + b"".join(s.desc for s in streams)
    sv = [s.states(c) if s.rle is None else (None, None) for s, c in zip(streams, (llc, ofc, mlc))]
    bits = []

    def put(v, nb):
        bits.extend((v >> (nb - 1 - k)) & 1 for k in range(nb))
    for k in (0, 1, 2):  # initial states: LL, OF, ML
        if sv[k][0] is not None:
            put(sv[k][0][0], streams[k].log)
    for i, (ll, ml, v) in enumerate(b.seqs):
        put(v - (1 << ofc[i]), ofc[i])                 # extra bits: OF, ML, LL
        put(ml - ML_BASE[mlc[i]], ML_BITS[mlc[i]])
        put(ll - LL_BASE[llc[i]], LL_BITS[llc[i]])
        if i + 1 < n:
            for k in (0, 2, 1):                        # state updates: LL, ML, OF
                if sv[k][1] is not None:
                    put(*sv[k][1][i])
    return lit + hdr + handmade.rev_stream(bits), streams


def build_frame(blocks, single_segment=True, window_log=None, fcs_width=None, checksum=True, content=None, body_hook=None):
    """The frame's bytes.  single_segment: window = frame content size; else window_log (10..30) sets the window
    descriptor.  fcs_width: 0, 1 (single segment only), 2, 4 or 8 bytes of frame content size (None: the smallest).
    content: the decoded bytes, for the checksum and the content size (default: reference_decode(blocks))."""
    if content is None:
        content = reference_decode(blocks)
        assert isinstance(content, bytes), content
    fcs = len(content)
    if fcs_width is None:
        fcs_width = 1 if single_segment and fcs < 256 else 2 if 256 <= fcs < 65536 + 256 else 4 if fcs < (1 << 32) else 8
        if not single_segment and fcs_width == 1:
            fcs_width = 0
    flag = {0: 0, 1: 0, 2: 1, 4: 2, 8: 3}[fcs_width]
    assert not (fcs_width == 1 and not single_segment) and not (fcs_width == 0 and single_segment)
    desc = (flag << 6) | (int(single_segment) << 5) | (int(checksum) << 2)
    hdr = MAGIC + bytes([desc])
    if not single_segment:
        assert window_log is not None and 10 <= window_log <= 41
        hdr += bytes([(window_log - 10) << 3])
    if fcs_width == 1:
        hdr += bytes([fcs])
    elif fcs_width == 2:
        hdr += struct.pack("<H", fcs - 256)
    elif fcs_width == 4:
        hdr += struct.pack("<I", fcs)
    elif fcs_width == 8:
        hdr += struct.pack("<Q", fcs)
    body = b""
    prev = None
    lit_state = {}
    for i, b in enumerate(blocks):
        last = int(i == len(blocks) - 1)
        if isinstance(b, Raw):
            body += _block_header(last, 0, len(b.data)) + b.data
        elif isinstance(b, Rle):
            body += _block_header(last, 1, b.n) + bytes([b.byte])
        else:
            blk, prev = encode_seqs_block(b, prev, lit_state)
            if body_hook:
                blk = body_hook(i, blk)
            assert len(blk) <= BLOCK_MAX
            body += _block_header(last, 2, len(blk)) + blk
    out = hdr + body
    if checksum:
        out += struct.pack("<I", O.lib().oracle_xxh64(content, len(content), 0) & 0xFFFFFFFF)
    return out
