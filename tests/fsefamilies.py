"""Sequence sections built field by field: FSE table descriptions, state walks and sequence counts chosen by the test, for
the parts of k_fse that exist for speed:

  phase 1a     fse_read_probabilities, one thread per block (lane * 4 + warp), counts parked in the table's own region;
  phase 1b     fse_build_table_warp: "less than one" cells by ballot over 32-symbol chunks, the spread walk, next-state
               numbering with __match_any_sync;
  lean loop    no data-dependent branches (num_bits from clz, next state from funnel shifts, two windows picked on
               extras & 32), rem looked at once at the end;
  exact loop   the blocks the lean loop refuses (a declared code beyond the code tables, offset code 31, anything that
               went wrong), and the first error in the reference's order;
  Repeat mode  the table re-derived from the block that set it, skipping the earlier streams' descriptions there.

Where tests/seqbuild.py chooses decoder states for given sequences, this module chooses the states: every compressed block
is written from one state walk per stream (the next state always inside the range the current state's bits can name), so
that a walk can visit every cell of a table, reach a cell of a code the reference refuses, or stop anywhere in the stream.
Frames are assembled by seqbuild.build_frame (body_hook puts the bodies written here in place).

Families (cases are seqfamilies.Case, with `blocks` = the Blk list of the frame):
  desc     valid descriptions of every stream at every accuracy log and symbol layout; every cell of every FSE table is the
           state of at least one decoded sequence (offset codes above OFFSET_CAP only in frames that fail in execution);
  repeat   Repeat chains: 1, 2 and 5 blocks after an FSE, RLE or predefined table, over Raw / RLE / zero-sequence blocks,
           each stream from another source block, source blocks where the stream's description follows others;
  counts   n_seq 1..9 on both loops, 0x7F01, 0xFFFF and NSEQ_MAX = 98047, with zero-bit streams and with streams of a few bits;
  cta      frames of 26, 27, 28 and 55 compressed blocks of mixed layouts (blocks of one frame share k_fse CTAs), and a batch
           of single-block frames of one sequence-count class alternating valid frames with every malformed kind;
  invalid  every sequence-stage error the reference can raise, as the only block and after valid blocks, and the quirks it
           accepts.
Each case's `expected` is reference_decode's output or the oracle's status name; `libzstd` is "ok", "reject" or None (a block
that regenerates more than 128 KiB, which libzstd 1.5 refuses and the reference accepts)."""
import random
from collections import deque
from dataclasses import dataclass

import handmade
import seqbuild as S
import seqfamilies as F
from seqbuild import Raw, Rle, Seqs

LL, OF, ML = 0, 1, 2
N_CODES = (36, 32, 53)       # codes each stream's code table knows (OF 31 is valid but k_fse decodes it in the exact loop)
OFFSET_CAP = 14              # highest offset code of a valid frame here: offsets up to 2^15 - 4 need that much output before
NSEQ_MAX = 0x7F00 + 0xFFFF   # the largest number of sequences the header can state (form 3)
BIG = 1 << 17                # a block regenerating more than this is refused by libzstd 1.5 (not by the reference)


# ---------------------------------------------------------------------------
# table descriptions (RFC 8878 4.1.1), with the encodings an encoder does not produce
# ---------------------------------------------------------------------------
def describe(log, probs, explicit_zero=(), pad=0, info=None):
    """The description of `probs` (-1 = "less than one"; they sum to 2^log counting -1 as 1).  explicit_zero: indices of
    zero-probability symbols written as a value of their own right after a zero run that ended with flag 0 (instead of being
    counted in that run); pad: the unused high bits of the last byte.  info (dict): receives nbits, and last = (bit position,
    short form, width) of the last value."""
    w = handmade.BitWriter()
    w.put(log - 5, 4)
    remaining, i, last = 1 << log, 0, None
    while remaining > 0:
        p = probs[i]
        value, max_remaining = p + 1, remaining + 1
        bits = max_remaining.bit_length()
        low = ((1 << bits) - 1) - max_remaining
        mask = (1 << (bits - 1)) - 1
        last = (w.n, value < low, bits)
        if value < low:
            w.put(value, bits - 1)
        elif value <= mask:
            w.put(value, bits)
        else:
            w.put(value + low, bits)
        remaining -= p if p > 0 else (1 if p == -1 else 0)
        i += 1
        if p == 0:
            run = 0
            while i + run < len(probs) and probs[i + run] == 0 and i + run not in explicit_zero:
                run += 1
            i += run
            while run >= 3:
                w.put(3, 2)
                run -= 3
            w.put(run, 2)
    assert remaining == 0 and i == len(probs), (remaining, i, len(probs))
    n = w.n
    if n % 8:
        w.v |= (pad & ((1 << (8 - n % 8)) - 1)) << n
    if info is not None:
        info.update(nbits=n, last=last)
    return w.bytes()


def spread(log, used, lt1=(), cheap=None):
    """Counts for symbols `used` (>= 1 each) and `lt1` ("less than one"), the cells left over going to the cheap symbols."""
    n = max(list(used) + list(lt1)) + 1
    p = [0] * n
    for s in lt1:
        p[s] = -1
    for s in used:
        p[s] = 1
    rest = (1 << log) - sum(abs(x) for x in p)
    assert rest >= 0, (log, len(used), len(lt1))
    cheap = list(cheap if cheap is not None else sorted(used)[:4])
    for k, s in enumerate(cheap):
        p[s] += rest // len(cheap) + (1 if k < rest % len(cheap) else 0)
    return p


# ---------------------------------------------------------------------------
# streams and state walks
# ---------------------------------------------------------------------------
@dataclass
class St:
    """One stream's table in one block.  mode: 0 predefined, 1 RLE, 2 FSE, 3 Repeat."""
    mode: int
    table: list = None      # [(symbol, num_bits, baseline)] per state; None for RLE
    rle: int = None
    desc: bytes = b""
    key: tuple = None       # (stream, log, probs) of an FSE table: what cell coverage is counted over


def pre(kind):
    return St(0, S.decoding_table(kind, S.PREDEF_LOG[kind], None))


def rle(code):
    return St(1, rle=code, desc=bytes([code]))


def fse(kind, log, probs, desc=None, **opts):
    return St(2, S.decoding_table(kind, log, probs), desc=desc if desc is not None else describe(log, probs, **opts),
              key=(kind, log, tuple(probs)))


def code_cost(kind, c):
    """What visiting a cell of code c adds to a block (literal bytes, match bytes, offset size); codes the reference refuses
    are never chosen by a walk that has any other cell to go to."""
    if c >= N_CODES[kind] or (kind == OF and c > OFFSET_CAP):
        return 1 << 40
    return S.LL_BASE[c] if kind == LL else S.ML_BASE[c] if kind == ML else 1 << c


CHEAP = (16, 1 << 5, 16)
_cheap_cache = {}


def _cheap(kind, t):
    """Per state: the cells of its range a filler walk may go to (the cheap ones, else the cheapest)."""
    key = (kind, id(t))
    if key not in _cheap_cache:
        rows = []
        for _, nb, b in t:
            r = range(b, b + (1 << nb))
            ok = [x for x in r if code_cost(kind, t[x][0]) <= CHEAP[kind]]
            rows.append(ok or [min(r, key=lambda x: code_cost(kind, t[x][0]))])
        _cheap_cache[key] = (t, rows)
    return _cheap_cache[key][1]


def extend(kind, t, w, n, rng):
    rows = _cheap(kind, t)
    if not w:
        w.append(rng.choice(min((r for r in rows), key=len)))
    while len(w) < n:
        w.append(rng.choice(rows[w[-1]]))
    return w


def cover_walks(kind, t, rng):
    """Walks that together visit every cell of table t, cheap cells first; a new walk (the next block) starts where no
    path leads on to a cell not yet visited (a single-symbol table: every state is its own successor)."""
    left = set(range(len(t)))
    cost = lambda s: code_cost(kind, t[s][0])
    walks = []
    while left:
        cur = min(left, key=lambda s: (cost(s), s))
        w = [cur]
        left.discard(cur)
        while left:
            _, nb, b = t[cur]
            cand = [x for x in range(b, b + (1 << nb)) if x in left]
            if cand:
                cur = min(cand, key=lambda s: (cost(s), rng.random()))
                w.append(cur)
                left.discard(cur)
                continue
            path = _path_to(t, cur, left)
            if path is None:
                break
            w += path
            left.difference_update(path)
            cur = w[-1]
        walks.append(w)
    return walks


def _path_to(t, start, targets):
    prev = {start: None}
    q = deque([start])
    while q:
        s = q.popleft()
        _, nb, b = t[s]
        for x in range(b, b + (1 << nb)):
            if x in prev:
                continue
            prev[x] = s
            if x in targets:
                path = [x]
                while prev[path[-1]] != start:
                    path.append(prev[path[-1]])
                return path[::-1]
            q.append(x)
    return None


# ---------------------------------------------------------------------------
# blocks and frames
# ---------------------------------------------------------------------------
@dataclass
class Blk:
    spec: object             # Raw / Rle / Seqs as seqbuild.reference_decode takes it (Seqs.seqs: [(ll, ml, ofv)])
    body: bytes = None       # the compressed block's body (None: Raw / Rle)
    streams: tuple = None    # (LL, OF, ML) St
    walks: tuple = None      # per stream: the state of every decoded sequence (None: RLE)
    status: str = None       # the sequence-stage status this block fails with (None: it decodes)
    risky: bool = False      # k_fse decodes the block in its exact loop (a declared code beyond the tables, offset code 31)
    beyond: bool = False     # a table declares a code beyond the code tables (libzstd refuses the frame)


def lit_section(lits):
    if isinstance(lits, tuple):
        return S._lit_header(1, lits[2]) + bytes([lits[1]])
    return S._lit_header(0, len(lits)) + bytes(lits)


class Bits:
    """Fields in the order the decoder reads them; rev() = the backward bitstream with its end marker."""

    def __init__(self):
        self.parts, self.ends, self.n = [], [], 0

    def put(self, v, nb):
        if nb:
            assert 0 <= v < (1 << nb), (v, nb)
            self.parts.append(format(v, f"0{nb}b"))
            self.n += nb

    def mark(self):
        self.ends.append(self.n)

    def rev(self, keep=None):
        s = "".join(self.parts)
        if keep is not None:
            s = s[:keep]
        v = int("1" + s, 2)
        return v.to_bytes((v.bit_length() + 7) // 8, "little")


def _extras(codes, seq):
    cl, co, cm = codes
    ll, ml, v = seq
    return [(v - (1 << co), co), (ml - S.ML_BASE[cm], S.ML_BITS[cm]), (ll - S.LL_BASE[cl], S.LL_BITS[cl])]


class Frame:
    """Blocks of one frame in order; tracks the tables a Repeat stream takes and the output so far."""

    def __init__(self, rng, pre_bytes=0):
        self.rng, self.blocks, self.prev, self.produced = rng, [], [None, None, None], 0
        if pre_bytes:
            self.raw(pre_bytes)

    def raw(self, n):
        self.blocks.append(Blk(Raw(self.rng.randbytes(n))))
        self.produced += n

    def rle(self, n):
        self.blocks.append(Blk(Rle(self.rng.randrange(256), n)))
        self.produced += n

    def empty(self, n_lits=0, trailing=b""):
        """A compressed block without sequences (number of sequences 0, then `trailing`)."""
        lits = self.rng.randbytes(n_lits)
        self.blocks.append(Blk(Seqs(lits, []), lit_section(lits) + b"\x00" + trailing))
        self.produced += n_lits

    def streams(self, specs):
        out = []
        for k, s in enumerate(specs):
            if s == "repeat":
                p = self.prev[k]
                s = St(3, p.table, p.rle, b"", p.key) if p is not None else St(3)
            elif s == "pre":
                s = pre(k)
            out.append(s)
        return out

    def seqs(self, specs, n=None, walks=None, lits_rle=None, tail=0, status=None, patch=None, keep_bits=None, nbseq=None,
             nbseq_form=None, modes_or=0):
        """A compressed block.  specs: (LL, OF, ML) St, "pre" or "repeat"; walks: per stream a state list (extended with cheap
        cells to n, or to the longest walk) or None; status: the sequence-stage failure the block is built to raise (its
        sequences are then not executed); patch(parts) edits the body's parts (lit, nbseq, modes, descs, bits);
        keep_bits: keep only the first so many bits of the bitstream, in reading order."""
        st = self.streams(specs)
        walks = [list(w) if w is not None else None for w in (walks or (None, None, None))]
        if n is None:
            n = max(len(w) for w in walks if w is not None)
        for k in range(3):
            if st[k].rle is None and st[k].table is not None:
                walks[k] = extend(k, st[k].table, walks[k] or [], n, self.rng)
            else:
                walks[k] = None
        codes = [[st[k].rle if walks[k] is None else st[k].table[walks[k][i]][0] for k in range(3)] for i in range(n)]
        if any(s.table is None and s.rle is None for s in st):   # Repeat with no table before it
            codes = [[99, 99, 99]] * n
        beyond = any((s.rle is not None and s.rle >= N_CODES[k]) or (s.key is not None and len(s.key[2]) > N_CODES[k])
                     for k, s in enumerate(st))
        risky = beyond or (st[OF].rle == 31) or (st[OF].key is not None and len(st[OF].key[2]) > 31)
        seqs = []
        for cl, co, cm in codes:
            if cl >= 36 or cm >= 53 or co >= 32:
                seqs.append(None)      # the reference stops here: no extra bits are read
                continue
            rng = self.rng
            ll = S.LL_BASE[cl] + (rng.randrange(1 << S.LL_BITS[cl]) if S.LL_BASE[cl] < 64 else 0)
            ml = S.ML_BASE[cm] + (rng.randrange(1 << S.ML_BITS[cm]) if S.ML_BASE[cm] < 131 else 0)
            v = 1 if co == 0 else 2 if co == 1 else (1 << co) + rng.randrange(1 << co)   # (repeat 3 with ll = 0 may be 0)
            seqs.append((ll, ml, v))
        n_lits = sum(s[0] for s in seqs if s) + tail
        lits = ("rle", lits_rle, n_lits) if lits_rle is not None else self.rng.randbytes(n_lits) if n_lits <= 4096 else \
            ("rle", self.rng.randrange(256), n_lits)
        bits = Bits()
        for k in (0, 1, 2):   # initial states: LL, OF, ML
            if walks[k] is not None:
                bits.put(walks[k][0], (len(st[k].table) - 1).bit_length())
        for i in range(n):
            if seqs[i] is not None:
                for v, nb in _extras(codes[i], seqs[i]):
                    bits.put(v, nb)
            if i + 1 < n:
                for k in (0, 2, 1):   # state updates: LL, ML, OF
                    if walks[k] is not None:
                        _, nb, b = st[k].table[walks[k][i]]
                        nxt = walks[k][i + 1]
                        assert b <= nxt < b + (1 << nb), (k, i, walks[k][i], nxt)
                        bits.put(nxt - b, nb)
            bits.mark()
        modes = (st[0].mode << 6) | (st[1].mode << 4) | (st[2].mode << 2) | modes_or
        parts = dict(lit=lit_section(lits), nbseq=S._nbseq_header(n if nbseq is None else nbseq, nbseq_form), modes=bytes([modes]),
                     descs=[s.desc for s in st], bits=bits.rev(keep_bits))
        if patch:
            patch(parts)
        body = parts["lit"] + parts["nbseq"] + parts["modes"] + b"".join(parts["descs"]) + parts["bits"]
        assert len(body) <= S.BLOCK_MAX, len(body)
        blk = Blk(Seqs(lits, seqs), body, tuple(st), tuple(walks), status, risky, beyond)
        blk.ends = bits.ends
        self.blocks.append(blk)
        if status is None:
            assert all(s is not None for s in seqs)
            self.produced += n_lits + sum(s[1] for s in seqs)
        for k in range(3):
            if st[k].mode != 3:
                self.prev[k] = st[k]
        return blk


def block_output(b):
    """Bytes a block regenerates."""
    if isinstance(b.spec, Raw):
        return len(b.spec.data)
    if isinstance(b.spec, Rle):
        return b.spec.n
    lits = b.spec.literals
    return (lits[2] if isinstance(lits, tuple) else len(lits)) + sum(s[1] for s in b.spec.seqs if s)


def case(name, fr, libzstd="ok", cap=None, **opts):
    blocks = fr.blocks
    bad = next((i for i, b in enumerate(blocks) if b.status), None)
    specs = [b.spec for b in blocks]
    window = (1 << opts["window_log"]) if not opts.get("single_segment", True) else None
    if bad is None:
        exp = S.reference_decode(specs, window)
        if not isinstance(exp, bytes) and window is None:
            exp = S.reference_decode(specs, 0)   # a failing single-segment frame is built with content size 0, so window 0
    else:
        exp = blocks[bad].status
    content = exp if isinstance(exp, bytes) else b""
    bodies = {i: b.body for i, b in enumerate(blocks) if b.body is not None}
    holders = [Seqs(b"", []) if b.body is not None else b.spec for b in blocks]
    frame = S.build_frame(holders, content=content, body_hook=lambda i, _: bodies[i], **opts)
    if cap is None:
        cap = len(exp) if isinstance(exp, bytes) else 1 << 20
    if isinstance(exp, bytes):
        if any(b.beyond for b in blocks):
            libzstd = "reject"        # libzstd refuses a table that declares a code beyond the code tables
        elif any(block_output(b) > BIG for b in blocks if b.body is not None):
            libzstd = None
    else:
        libzstd = "reject"
    c = F.Case(name, frame, exp, cap, libzstd)
    c.blocks = blocks
    c.fail_block = bad
    return c


# ---------------------------------------------------------------------------
# 1. descriptions
# ---------------------------------------------------------------------------
HI = (35, OFFSET_CAP, 52)                        # highest code of a valid frame's table


def _expensive(kind, c):
    return code_cost(kind, c) > CHEAP[kind] * 4


def _layouts(kind, log, rng):
    """{name: probs} of one stream at one accuracy log (the ones that fit 2^log cells and the stream's valid codes)."""
    size, hi = 1 << log, HI[kind]
    out = {}
    codes = list(range(hi + 1))
    if hi + 1 <= size:
        out["full"] = spread(log, [c for c in codes if not _expensive(kind, c)], [c for c in codes if _expensive(kind, c)])
    c0 = (1, 2, 2)[kind]
    out["single"] = [0] * c0 + [size]
    out["lt1-top"] = spread(log, [0, 1, 2, 3], [min(hi, 9)])
    for k in (32, 33, 40):
        if k < hi + 1 and k + 2 <= size:
            out[f"lt1-{k}"] = spread(log, [0, 1], list(range(hi + 1 - k, hi + 1)) if k > 32 else list(range(2, 2 + k)))
    if hi + 1 <= size:
        out["lt1-all-but-one"] = [size - hi] + [-1] * hi
    for r in (1, 2, 3, 4, 6, 34):
        if r + 2 <= hi:
            used = [0, r + 1] + ([r + 2] if r + 2 <= hi else [])
            out[f"zeros{r}"] = spread(log, used)
    return out


def _threshold_layouts(log):
    """Counts whose second value lies on each side of low_threshold and of the mask, with 2^k - 1, 2^k and 2^k + 1 cells
    remaining before it."""
    out = {}
    for k in sorted({2, log - 1}):
        for R in ((1 << k) - 1, 1 << k, (1 << k) + 1):
            bits = (R + 1).bit_length()
            low, mask = ((1 << bits) - 1) - (R + 1), (1 << (bits - 1)) - 1
            for v in sorted({0, 1, low - 1, low, mask, mask + 1, R + 1}):
                if not 0 <= v <= R + 1 or (v == 1 and R == 0):
                    continue
                p1 = v - 1
                rest = R - (1 if p1 == -1 else max(p1, 0))
                probs = [(1 << log) - R, p1] + ([rest] if rest else [])
                if probs[-1] == 0:
                    continue
                out[f"thr-k{k}-r{R}-v{v}"] = probs
    return out


def _boundary_layouts(kind, log, rng):
    """Descriptions that end on a byte boundary and one bit before one."""
    out = {}
    for want in (0, 7):
        for _ in range(500):
            used = sorted(rng.sample(range(HI[kind] + 1), rng.randrange(2, min(8, HI[kind] + 1))))
            lt1 = [c for c in rng.sample(range(HI[kind] + 1), 2) if c not in used]
            p = spread(log, used, lt1, cheap=[rng.choice(used)])
            info = {}
            describe(log, p, info=info)
            if info["nbits"] % 8 == want:
                out[f"end{want}"] = p
                break
    return out


def _noncanonical(log):
    """(probs, describe options): an explicit zero after a run ended with flag 0, runs of 3 and 6 (flags 3, 0 and 3, 3, 0),
    nonzero padding."""
    size = 1 << log
    return {
        "explicit-zero": ([size - 3, 0, 0, 1, 0, 1, 1], dict(explicit_zero=(2, 4))),
        "run3": ([size - 2, 0, 0, 0, 0, 1, 1], {}),
        "run6": ([size - 2, 0, 0, 0, 0, 0, 0, 0, 1, 1], {}),
        "pad": ([size - 5, 2, 0, 1, 1, -1], dict(pad=0xFF)),
    }


def _desc_frame(name, rng, tables, exec_fail=False):
    """One frame covering every cell of the given FSE tables: block 0 sets them, later blocks Repeat them (a walk that
    cannot go on starts the next block)."""
    segs = [cover_walks(k, st.table, rng) if st.mode == 2 else [] for k, st in enumerate(tables)]
    n_blocks = max(1, max(len(s) for s in segs))
    pre_bytes = 64 if exec_fail else (1 << (OFFSET_CAP + 1)) + 64
    fr = Frame(rng, pre_bytes)
    for j in range(n_blocks):
        specs = tables if j == 0 else ["repeat"] * 3
        walks = [s[j] if j < len(s) else None for s in segs]
        n = max([len(w) for w in walks if w is not None] + [1])
        fr.seqs(specs, n=n, walks=walks)
    return case(name, fr)


def family_desc(seed=11):
    rng = random.Random(seed)
    cases = []
    for log in range(5, 10):
        ologs = min(log, 8)
        lay = [_layouts(LL, log, rng), _layouts(OF, ologs, rng), _layouts(ML, log, rng)]
        names = sorted(set(lay[0]) | set(lay[1]) | set(lay[2]))
        for nm in names:
            tables = [fse(k, (log, ologs, log)[k], lay[k][nm]) if nm in lay[k] else rle((1, 2, 3)[k]) for k in range(3)]
            cases.append(_desc_frame(f"desc-{nm}-log{log}", rng, tables))
        thr = [_threshold_layouts(log), _threshold_layouts(ologs), _threshold_layouts(log)]
        for nm in sorted(thr[0]):
            tables = [fse(k, (log, ologs, log)[k], thr[k][nm]) if nm in thr[k] else pre(k) for k in range(3)]
            cases.append(_desc_frame(f"desc-{nm}-log{log}", rng, tables))
        bnd = [_boundary_layouts(k, (log, ologs, log)[k], rng) for k in range(3)]
        for nm in ("end0", "end7"):
            tables = [fse(k, (log, ologs, log)[k], bnd[k][nm]) for k in range(3)]
            cases.append(_desc_frame(f"desc-{nm}-log{log}", rng, tables))
        for nm, (p, opts) in _noncanonical(log).items():
            op, oo = _noncanonical(ologs)[nm]
            tables = [fse(LL, log, p, **opts), fse(OF, ologs, op, **oo), fse(ML, log, p, **opts)]
            cases.append(_desc_frame(f"desc-{nm}-log{log}", rng, tables))
    # offset codes above OFFSET_CAP: the whole code range, code 31 (exact loop), all codes but one "less than one"; the
    # frames fail in execution (an offset beyond the output), after k_fse decoded every block
    for log in range(5, 9):
        size = 1 << log
        full = spread(log, list(range(min(31, size))))
        layouts = {"of-full": full, "of-31": spread(log, list(range(32)), cheap=[0])}
        if size > 31:
            layouts["of-lt1-all-but-one"] = [size - 30] + [-1] * 30
        for nm, p in layouts.items():
            tables = [rle(0), fse(OF, log, p), rle(1)]
            c = _desc_frame(f"desc-{nm}-log{log}", rng, tables, exec_fail=True)
            assert c.expected in ("CZS_OFFSET_TOO_BIG", "CZS_NOT_ENOUGH_BYTES_IN_DICTIONARY"), (c.name, c.expected)
            cases.append(c)
    return cases


def coverage(c):
    """{table key: cells never the state of a decoded sequence} over the frame's blocks (FSE tables only)."""
    seen = {}
    for b in c.blocks:
        if b.walks is None:
            continue
        for st, w in zip(b.streams, b.walks):
            if st.key is not None and w is not None:
                seen.setdefault(st.key, set()).update(w)
    return {k: set(range(1 << k[1])) - v for k, v in seen.items()}


# ---------------------------------------------------------------------------
# 2. Repeat chains
# ---------------------------------------------------------------------------
def _small_fse(kind, rng, log=None):
    log = log or rng.choice((5, 6, S.MAX_LOG[kind]))
    hi = min(HI[kind], 6 if kind == OF else 10)        # offsets up to 124: every frame here has that much output first
    used = sorted(rng.sample(range(hi + 1), rng.randrange(2, hi + 1)))
    return fse(kind, log, spread(log, used, cheap=used[:2]))


def _source(kind_of_source, rng):
    if kind_of_source == "fse":
        return [_small_fse(k, rng) for k in range(3)]
    if kind_of_source == "rle":
        return [rle(rng.randrange(4)), rle(rng.randrange(2, 5)), rle(rng.randrange(6))]
    return ["pre"] * 3


def _gap(fr, rng, j):
    """A block that leaves the tables alone: Raw, RLE, or a compressed block without sequences."""
    [lambda: fr.raw(1 + rng.randrange(40)), lambda: fr.rle(1 + rng.randrange(40)), lambda: fr.empty(rng.randrange(5))][j % 3]()


def family_repeat(seed=12):
    rng = random.Random(seed)
    cases = []
    for src in ("fse", "rle", "pre"):
        for dist in (1, 2, 5):
            for chained in (False, True):
                fr = Frame(rng, 300)
                fr.seqs(_source(src, rng), n=1 + rng.randrange(40))
                for j in range(dist - 1):
                    if chained:
                        fr.seqs(["repeat"] * 3, n=1 + rng.randrange(20))
                    else:
                        _gap(fr, rng, j)
                fr.seqs(["repeat"] * 3, n=1 + rng.randrange(60))
                _gap(fr, rng, dist)
                fr.seqs(["repeat"] * 3, n=4 + rng.randrange(9))
                cases.append(case(f"repeat-{src}-{dist}{'-chain' if chained else ''}", fr))
    # each stream repeats another source block: LL from A, OF from B, ML from C
    fr = Frame(rng, 300)
    fr.seqs([_small_fse(k, rng) for k in range(3)], n=30)
    _gap(fr, rng, 0)
    fr.seqs(["repeat", _small_fse(OF, rng), _small_fse(ML, rng)], n=20)
    _gap(fr, rng, 2)
    fr.seqs(["repeat", "repeat", rle(5)], n=9)
    for j in range(3):
        fr.seqs(["repeat"] * 3, n=5 + 7 * j)
        _gap(fr, rng, j)
    cases.append(case("repeat-three-sources", fr))
    # the repeated stream's description follows one or two others in its source block: an RLE byte, FSE descriptions that
    # end mid-byte
    for variant in range(4):
        fr = Frame(rng, 300)
        for _ in range(50):
            tabs = [_small_fse(k, rng) for k in range(3)]
            info = {}
            describe(tabs[0].key[1], list(tabs[0].key[2]), info=info)
            if info["nbits"] % 8:
                break
        if variant == 0:
            src = [rle(2), tabs[1], tabs[2]]
        elif variant == 1:
            src = [tabs[0], rle(3), tabs[2]]
        elif variant == 2:
            src = [tabs[0], tabs[1], tabs[2]]
        else:
            src = [rle(1), rle(2), tabs[2]]
        fr.seqs(src, n=25)
        fr.empty(3)
        fr.seqs(["pre", "pre", "repeat"], n=12)
        fr.seqs([rle(0), "repeat", "repeat"], n=12)
        fr.rle(10)
        fr.seqs(["repeat", "repeat", "repeat"], n=7)
        cases.append(case(f"repeat-after-descs-{variant}", fr))
    # Repeat with no table before it: in the first block with sequences, and after zero-sequence blocks only
    for k in range(3):
        for lead in (0, 1, 3):
            fr = Frame(rng, 64 if lead else 0)
            for j in range(lead):
                fr.empty(rng.randrange(4))
            specs = ["pre", "pre", "pre"]
            specs[k] = "repeat"
            fr.seqs(specs, n=3, status="CZS_FSE_TABLE_IS_UNINITIALIZED")
            cases.append(case(f"repeat-uninitialized-{'LOM'[k]}-{lead}", fr))
    return cases


# ---------------------------------------------------------------------------
# 3. sequence counts
# ---------------------------------------------------------------------------
def _zero_bit(kind):
    return [0, 0, 31][kind]                      # ll 0, offset value 1 (repeat), ml 34: no extra bits


def family_counts(seed=13):
    rng = random.Random(seed)
    cases = []
    for n in list(range(1, 10)) + [0x7F01, 0xFFFF, NSEQ_MAX]:
        variants = {
            "rle0": [rle(_zero_bit(k)) for k in range(3)],
            "fse0": [fse(k, 5 + k, [0] * _zero_bit(k) + [1 << (5 + k)]) for k in range(3)],
            "bits": [fse(LL, 5, [20, 12]), fse(OF, 5, [0, 0, 16, 16]), fse(ML, 6, [16, 16, 16, 16])],
        }
        if n < 10:
            variants["bits-risky"] = [fse(LL, 5, [20, 11, 0, 0] + [0] * 36 + [-1]), fse(OF, 5, [0, 0, 16, 16]), fse(ML, 6, [16] * 4)]
            variants["bits-of31"] = [fse(LL, 5, [20, 12]), fse(OF, 5, [0, 0, 15, 16] + [0] * 27 + [1]), fse(ML, 6, [16] * 4)]
        for nm, tabs in variants.items():
            fr = Frame(rng, 64)
            walks = [None] * 3
            if nm.startswith("fse0"):
                walks = [[rng.randrange(1 << (5 + k))] * n for k in range(3)]   # num_bits 0: the state never moves
            fr.seqs(tabs, n=n, walks=walks, lits_rle=0x2E)
            cases.append(case(f"counts-{n}-{nm}", fr))
    return cases


# ---------------------------------------------------------------------------
# 4. malformed sections
# ---------------------------------------------------------------------------
def _valid(fr, rng, n):
    fr.seqs([_small_fse(k, rng) for k in range(3)], n=n)


def _cut_bits(blk_ends, j):
    """Bits to keep so that the stream runs short during sequence j (after sequence j - 1 decoded whole)."""
    lo = blk_ends[j - 1] if j else 0
    assert blk_ends[j] > lo
    return blk_ends[j] - 1


def _short(fr, rng, n, j, with_rle):
    st = "CZS_SEQ_NOT_ENOUGH_BYTES_FOR_NUM_SEQUENCES" if with_rle else "CZS_PANIC_INTERNAL"
    while True:
        tabs = [rle(1) if with_rle else _small_fse(LL, rng), _small_fse(OF, rng), _small_fse(ML, rng)]
        state = rng.getstate()
        probe = fr.seqs(tabs, n=n)
        fr.blocks.pop()
        if probe.ends[j] > (probe.ends[j - 1] if j else 0):
            break
    rng.setstate(state)
    fr.seqs(tabs, n=n, status=st, keep_bits=_cut_bits(probe.ends, j))


def _walk_to(kind, t, cell, j, rng):
    """A walk of cheap states whose state j is `cell`, built backwards: every cell lies in the range of one state of each
    symbol."""
    w = [cell]
    for _ in range(j):
        w.insert(0, rng.choice([s for s, (sym, nb, b) in enumerate(t) if b <= w[0] < b + (1 << nb) and code_cost(kind, sym) <= CHEAP[kind]]))
    return w


def _bad_code(fr, rng, n, kind, code, via, j=0, keep=None):
    st = "CZS_SEQ_UNSUPPORTED_OFFSET" if kind == OF and code >= 32 else "CZS_SEQ_GET_BITS_ERROR"
    tabs = [rle(1), rle(2), rle(3)] if via == "rle" else [_small_fse(k, rng, 6) for k in range(3)]
    walks = [None] * 3
    if via == "rle":
        tabs[kind] = rle(code)
    else:
        log = 6
        tabs[kind] = fse(kind, log, spread(log, [0, 1, 2], [code]))
        walks[kind] = _walk_to(kind, tabs[kind].table, (1 << log) - 1, j, rng)
    if keep is None:
        fr.seqs(tabs, n=n, walks=walks, status=st)
        return
    state = rng.getstate()
    probe = fr.seqs(tabs, n=n, walks=walks, status=st)
    fr.blocks.pop()
    rng.setstate(state)
    fr.seqs(tabs, n=n, walks=walks, status=keep[1], keep_bits=_cut_bits(probe.ends, keep[0]))


def _patched(fr, rng, n, status, patch, tabs=None, **kw):
    fr.seqs(tabs or [_small_fse(k, rng) for k in range(3)], n=n, status=status, patch=patch, **kw)


def _cut_desc(k, keep_bytes):
    def patch(p):
        p["descs"][k] = p["descs"][k][:keep_bytes]
        del p["descs"][k + 1:]
        p["bits"] = b""
    return patch


def malformed(rng, n):
    """(name, maker(fr)) of every malformed kind at n sequences; maker adds the failing block to frame fr."""
    out = []
    for extra in (1, 5):
        out.append((f"nseq+{extra}-pre", lambda fr, e=extra: fr.seqs(["pre"] * 3, n=n, nbseq=n + e, status="CZS_PANIC_INTERNAL")))
        out.append((f"nseq+{extra}-rle", lambda fr, e=extra: fr.seqs([rle(1), "pre", "pre"], n=n, nbseq=n + e,
                                                                       status="CZS_SEQ_NOT_ENOUGH_BYTES_FOR_NUM_SEQUENCES")))
    if n > 1:
        out.append(("nseq-1", lambda fr: fr.seqs(["pre"] * 3, n=n, nbseq=n - 1, status="CZS_SEQ_EXTRA_BITS")))
    pad = "CZS_SEQ_EXTRA_PADDING"
    out.append(("last-byte-0", lambda fr: _patched(fr, rng, n, pad, lambda p: p.update(bits=p["bits"][:-1] + b"\x00"))))
    out.append(("extra-zero-byte", lambda fr: _patched(fr, rng, n, pad, lambda p: p.update(bits=p["bits"] + b"\x00"))))
    out.append(("empty-bitstream", lambda fr: _patched(fr, rng, n, pad, lambda p: p.update(bits=b""))))
    for code in (32, 63, 64, 200):
        out.append((f"rle-of-{code}", lambda fr, c=code: _bad_code(fr, rng, n, OF, c, "rle")))
    for code in (32, 63, 64):
        out.append((f"fse-of-{code}", lambda fr, c=code: _bad_code(fr, rng, n, OF, c, "fse", j=min(n - 1, 2))))
    for code in (36, 63, 64, 255):
        out.append((f"rle-ll-{code}", lambda fr, c=code: _bad_code(fr, rng, n, LL, c, "rle")))
        out.append((f"fse-ll-{code}", lambda fr, c=code: _bad_code(fr, rng, n, LL, c, "fse", j=n - 1)))
    for code in (53, 63, 64):
        out.append((f"rle-ml-{code}", lambda fr, c=code: _bad_code(fr, rng, n, ML, c, "rle")))
        out.append((f"fse-ml-{code}", lambda fr, c=code: _bad_code(fr, rng, n, ML, c, "fse", j=0)))
    big = "CZS_FSE_ACC_LOG_TOO_BIG"
    for k, where in ((LL, 0), (OF, 1), (ML, 2)):
        def acc(fr, k=k):
            tabs = [_small_fse(q, rng) for q in range(3)]
            tabs[k] = St(2, tabs[k].table, desc=bytes([(S.MAX_LOG[k] + 1 - 5) | (tabs[k].desc[0] & 0xF0)]) + tabs[k].desc[1:], key=tabs[k].key)
            if k == ML:
                tabs[0] = rle(1)
            fr.seqs(tabs, n=n, status=big)
        out.append((f"acc-log-{'LOM'[k]}", acc))
    out.append(("modes-missing", lambda fr: _patched(fr, rng, n, "CZS_SEQ_HDR_NOT_ENOUGH_BYTES",
                                                     lambda p: p.update(modes=b"", descs=[], bits=b""))))
    out.append(("nbseq-form2-cut", lambda fr: _patched(fr, rng, n, "CZS_SEQ_HDR_NOT_ENOUGH_BYTES",
                                                       lambda p: p.update(nbseq=p["nbseq"][:1], modes=b"", descs=[], bits=b""), nbseq_form=2)
                if n < 0x7F00 else None))
    out.append(("nbseq-form3-cut", lambda fr: _patched(fr, rng, n, "CZS_SEQ_HDR_NOT_ENOUGH_BYTES",
                                                       lambda p: p.update(nbseq=b"\xff\x01", modes=b"", descs=[], bits=b""))))
    for k in range(3):
        def rle_missing(fr, k=k):
            tabs = ["pre", "pre", "pre"]
            tabs[k] = rle(1)
            fr.seqs(tabs, n=n, status=("CZS_MISSING_BYTE_FOR_RLE_LL_TABLE", "CZS_MISSING_BYTE_FOR_RLE_OF_TABLE",
                                       "CZS_MISSING_BYTE_FOR_RLE_ML_TABLE")[k], patch=lambda p: p.update(descs=[], bits=b""))
        out.append((f"rle-byte-missing-{'LOM'[k]}", rle_missing))
    for nsym in (257, 300):
        def many(fr, nsym=nsym):
            probs = [63] + [0] * (nsym - 2) + [1]
            d = describe(6, probs)
            fr.seqs([fse(LL, 6, [63, 1], desc=d), "pre", "pre"], n=n, status="CZS_FSE_TOO_MANY_SYMBOLS")
        out.append((f"symbols-{nsym}", many))
    t255 = S.decoding_table(LL, 6, [63] + [0] * 254 + [1])
    out.append(("symbol-255-used", lambda fr: fr.seqs([fse(LL, 6, [63] + [0] * 254 + [1]), "pre", "pre"], n=n,
                                                      walks=[_walk_to(LL, t255, [x[0] for x in t255].index(255), n // 2, rng), None, None],
                                                      status="CZS_SEQ_GET_BITS_ERROR")))
    return [(nm, mk) for nm, mk in out]


def family_invalid(seed=14):
    rng = random.Random(seed)
    cases = []
    n = 10
    for name, mk in malformed(rng, n):
        for lead in (False, True):
            fr = Frame(rng, 200 if lead else 0)
            if lead:
                _valid(fr, rng, 12)
                fr.rle(30)
                _valid(fr, rng, 7)
            mk(fr)
            if fr.blocks and fr.blocks[-1].status:
                fr.raw(10)     # a block after the failing one is never reached
                cases.append(case(f"invalid-{name}{'-after' if lead else ''}", fr))
    # descriptions cut inside their last value, for each stream's description last in the section
    for k in range(3):
        for log in (5, 6, S.MAX_LOG[k]):
            for trial in range(6):
                used = sorted(rng.sample(range(min(HI[k], 12) + 1), rng.randrange(2, 6)))
                p = spread(log, used, cheap=[used[0]])
                info = {}
                d = describe(log, p, info=info)
                start, short, width = info["last"]
                tabs = ["pre", "pre", "pre"]
                tabs[k] = fse(k, log, p)
                for cut in sorted({start // 8, (start + width - 1) // 8}):
                    if cut >= len(d):
                        continue
                    fr = Frame(rng, 200)
                    _valid(fr, rng, 5)
                    fr.seqs(tabs, n=4, status="CZS_FSE_GET_BITS_ERROR", patch=_cut_desc(k, cut))
                    cases.append(case(f"invalid-cut-{'LOM'[k]}-log{log}-{trial}-{cut}of{len(d)}", fr))
                if short and (start + width - 1) % 8 == 0:
                    # the given-back bit of a short-form last value lies just past the end: the value reads `width` bits
                    fr = Frame(rng, 0)
                    fr.seqs(tabs, n=4, status="CZS_FSE_GET_BITS_ERROR", patch=_cut_desc(k, (start + width - 1) // 8))
                    cases.append(case(f"invalid-cut-short-{'LOM'[k]}-log{log}-{trial}", fr))
    # running short at the first sequence, inside a group of four, in the tail and at the last sequence
    for with_rle in (False, True):
        for j in (0, 2, 5, 8, 9):
            fr = Frame(rng, 200)
            _short(fr, rng, 10, j, with_rle)
            cases.append(case(f"invalid-short-at-{j}-{'rle' if with_rle else 'fse'}", fr))
    # two errors in one block: a bad code, then running short (the bad code wins); running short, then a bad code
    fr = Frame(rng, 200)
    _bad_code(fr, rng, 12, LL, 40, "fse", j=3, keep=(7, "CZS_SEQ_GET_BITS_ERROR"))
    cases.append(case("invalid-bad-code-then-short", fr))
    fr = Frame(rng, 200)
    _bad_code(fr, rng, 12, LL, 40, "fse", j=9, keep=(5, "CZS_PANIC_INTERNAL"))
    cases.append(case("invalid-short-then-bad-code", fr))
    # accepted: trailing bytes after n_seq = 0, reserved bits of the modes byte, declared codes beyond the tables (unused)
    fr = Frame(rng, 50)
    fr.empty(5, trailing=b"\x9c\x01")
    cases.append(case("quirk-nseq0-trailing-bytes", fr, libzstd="reject"))
    fr = Frame(rng, 50)
    fr.seqs([_small_fse(k, rng) for k in range(3)], n=20, modes_or=3)
    cases.append(case("quirk-reserved-modes-bits", fr))
    for k, code in ((OF, 40), (ML, 60), (LL, 50)):
        for other in ("fse", "rle"):
            fr = Frame(rng, 300)
            tabs = [_small_fse(q, rng) for q in range(3)] if other == "fse" else [rle(1), rle(2), rle(3)]
            used = list(range(4))
            tabs[k] = fse(k, 6, spread(6, used, [code]))
            fr.seqs(tabs, n=30)
            cases.append(case(f"quirk-unused-{'LOM'[k]}{code}-{other}", fr))
    return cases


# ---------------------------------------------------------------------------
# 5. blocks sharing a k_fse CTA
# ---------------------------------------------------------------------------
def _mixed_block(fr, rng, j):
    kind = j % 7
    n = rng.choice((1, 3, 4, 5, 8, 9, 17, 40, 130))
    if kind == 0:
        fr.seqs([_small_fse(k, rng) for k in range(3)], n=n)                                         # lean
    elif kind == 1:
        fr.seqs([fse(LL, 6, spread(6, [0, 1, 2, 3], [44])), _small_fse(OF, rng), "pre"], n=n)     # exact (declared LL 44)
    elif kind == 2:
        fr.seqs([rle(rng.randrange(4)), rle(2), rle(rng.randrange(5))], n=n)                        # RLE, zero-bit-ish
    elif kind == 3:
        fr.seqs(["pre"] * 3, n=n)
    elif kind == 4:
        fr.seqs(["repeat", "repeat", "repeat"] if fr.prev[0] is not None else ["pre"] * 3, n=n)
    elif kind == 5:
        fr.empty(rng.randrange(3))
    else:
        fr.seqs([fse(k, 5, [0] * _zero_bit(k) + [32]) for k in range(3)], n=n, walks=[[rng.randrange(32)] * n for _ in range(3)])


def family_cta(seed=15):
    rng = random.Random(seed)
    cases = []
    for n_blocks in (26, 27, 28, 55):
        for fail in (False, True):
            fr = Frame(rng, 500)
            while sum(1 for b in fr.blocks if b.body is not None) < n_blocks - (1 if fail else 0):
                _mixed_block(fr, rng, len(fr.blocks))
            if fail:
                fr.seqs(["pre"] * 3, n=6, nbseq=5, status="CZS_SEQ_EXTRA_BITS")
            cases.append(case(f"cta-{n_blocks}{'-fail' if fail else ''}", fr, single_segment=False, window_log=20))
    # single-block frames of one sequence-count class (64..127): frames whose sequence section is valid alternate with every
    # malformed kind.  Without output before them, most of the former fail in execution in their first chunk of 32 sequences,
    # with matches of the next chunk reaching back into it (k_exec_flow once waited for those bytes until its spin limit)
    kinds = malformed(rng, 100)
    for i, (name, mk) in enumerate(kinds):
        fr = Frame(rng, 0)
        fr.seqs([_small_fse(k, rng) for k in range(3)] if i % 2 else ["pre"] * 3, n=64 + rng.randrange(64))
        cases.append(case(f"cta-class6-seq-ok-{i}", fr))
        fr = Frame(rng, 0)
        mk(fr)
        if fr.blocks:
            cases.append(case(f"cta-class6-{name}", fr))
    return cases


FAMILIES = {"desc": family_desc, "repeat": family_repeat, "counts": family_counts, "invalid": family_invalid, "cta": family_cta}
_cache = {}


def cases(name):
    if name not in _cache:
        _cache[name] = FAMILIES[name]()
    return _cache[name]
