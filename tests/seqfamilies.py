"""Frames built sequence by sequence (tests/seqbuild.py) that put matches, literal runs and repeat offsets on the seams where
the sequence executors and k_fse change their behaviour:

  k_exec       32 sequences per chunk (lane = sequence); tile path up to EXEC_TILE = 1024 bytes of chunk span, row path
               above; first 16 bytes of a segment per lane, longer tails by the warp; self-overlapping matches whose source
               starts before the chunk; RLE literal sections.
  k_exec_big   BIG_WIN = 16384 bytes of window trusted BIG_WIN_REACH = 8128 bytes back, 1 KiB slices, chunks longer than a
               slice, batches of BIG_BATCH = 1024 chunks.
  k_exec_flow  64 KiB / 4096-byte slices / reach 36864 (narrow), 128 KiB / 8192 / 73728 (wide), 256 completion slots,
               batches of 1024 chunks.
  k_fse        four steps per group plus a tail, lean and exact loops, symbolic offset history for blocks that are not first
               in their frame, every table mode, the three number-of-sequences header forms.

Each family returns Cases; a case's `expected` is reference_decode's output (or the oracle's status name of the failure)
and `libzstd` says whether libzstd must accept the frame ("ok"), must reject it ("reject"), or is not asked (None)."""
import random
from dataclasses import dataclass

import seqbuild as S
from seqbuild import Raw, Rle, Seqs, off, rep


@dataclass
class Case:
    name: str
    frame: bytes
    expected: object        # bytes, or the oracle's status name
    cap: int
    libzstd: str = "ok"


def _rb(rng, n):
    return bytes(rng.getrandbits(8) for _ in range(n))


def case(name, blocks, libzstd="ok", cap=None, **opts):
    window = (1 << opts["window_log"]) if not opts.get("single_segment", True) else None
    exp = S.reference_decode(blocks, window)
    if not isinstance(exp, bytes) and window is None:
        exp = S.reference_decode(blocks, 0)   # a failing single-segment frame is built with content size 0, so window 0
    content = exp if isinstance(exp, bytes) else b""
    frame = S.build_frame(blocks, content=content, **opts)
    if cap is None:
        cap = len(exp) if isinstance(exp, bytes) else 1 << 20
    return Case(name, frame, exp, cap, libzstd if isinstance(exp, bytes) else "reject")


def lits_for(seqs, rng, tail=0, rle=None):
    n = sum(s[0] for s in seqs) + tail
    return ("rle", rle, n) if rle is not None else _rb(rng, n)


class _Hist:
    """Offset history of the sequences appended so far, so that a generator can pick repeat codes that resolve to a valid
    offset."""

    def __init__(self, produced=0):
        self.h, self.produced = [1, 4, 8], produced

    def resolve(self, ll, ofv):
        h = self.h
        if ofv > 3:
            return ofv - 3, [ofv - 3, h[0], h[1]]
        if ll > 0:
            o = h[ofv - 1]
            return o, (h if ofv == 1 else [o, h[0], h[2]] if ofv == 2 else [o, h[0], h[1]])
        o = h[1] if ofv == 1 else h[2] if ofv == 2 else h[0] - 1
        return o, ([o, h[0], h[2]] if ofv == 1 else [o, h[0], h[1]])

    def ok(self, ll, ofv):
        o, _ = self.resolve(ll, ofv)
        return 1 <= o <= self.produced + ll

    def add(self, ll, ml, ofv):
        o, self.h = self.resolve(ll, ofv)
        assert 1 <= o <= self.produced + ll, (ll, ml, ofv, o, self.produced)
        self.produced += ll + ml
        return (ll, ml, ofv)

    def skip(self, n):
        self.produced += n


# ---------------------------------------------------------------------------
# 1. chunk and tile seams (k_exec)
# ---------------------------------------------------------------------------
LIT_RUNS = [0, 1, 15, 16, 17, 31, 32, 33]
NSEQ = [1, 2, 3, 4, 5, 31, 32, 33, 63, 64, 65, 127, 128]


def _small_seqs(rng, n, hist, lit_runs=LIT_RUNS, max_ml=40, max_off=40):
    out = []
    for i in range(n):
        ll = lit_runs[i % len(lit_runs)]
        ml = 3 + rng.randrange(max_ml - 2)
        while True:
            ofv = rng.choice([1, 2, 3]) if rng.random() < 0.25 else off(1 + rng.randrange(max_off))
            if hist.ok(ll, ofv):
                break
        out.append(hist.add(ll, ml, ofv))
    return out


def _span_chunk(rng, hist, span):
    """32 sequences whose ll + ml add up to `span` bytes."""
    seqs = []
    left = span
    for i in range(32):
        rest = 31 - i
        if rest == 0:
            ll, ml = (left - 3, 3) if left - 3 < 64 else (32, left - 32)
        else:
            seg = max(3, min(left - 3 * rest, left // (rest + 1) + rng.randrange(-3, 4)))
            ll = min(seg - 3, rng.choice(LIT_RUNS))
            ml = seg - ll
        left -= ll + ml
        seqs.append(hist.add(ll, ml, off(1 + rng.randrange(min(40, hist.produced + ll)))))
    assert left == 0
    return seqs


def family_chunks(seed=1):
    rng = random.Random(seed)
    cases = []
    pre = _rb(rng, 64)
    for n in NSEQ:
        for rle in (None, 0x5A):
            h = _Hist(len(pre))
            seqs = _small_seqs(rng, n, h)
            tables = ("predefined",) * 3 if n % 2 else (("fse", 5), ("fse", 5), ("fse", 6))
            cases.append(case(f"nseq{n}-{'rle' if rle else 'raw'}", [Raw(pre), Seqs(lits_for(seqs, rng, n % 7, rle), seqs, tables)]))
    # every ml 3..40 at every offset 1..40, literal runs cycling through the per-lane / warp seams
    for rle in (None, 0xC3):
        h = _Hist(len(pre))
        seqs = [h.add(LIT_RUNS[(ml * 41 + o) % 8], ml, off(o)) for ml in range(3, 41) for o in range(1, 41)]
        cases.append(case(f"ml-x-off-{'rle' if rle else 'raw'}", [Raw(pre), Seqs(lits_for(seqs, rng, 5, rle), seqs, (("fse", 9), ("fse", 8), ("fse", 9)))]))
    # chunk spans around EXEC_TILE, as the first and as a later chunk of a block
    for span in (1023, 1024, 1025):
        for rle in (None, 0x11):
            h = _Hist(len(pre))
            seqs = _small_seqs(rng, 32, h) + _span_chunk(rng, h, span) + _small_seqs(rng, 7, h)
            h2 = _Hist(len(pre))
            first = _span_chunk(rng, h2, span) + _small_seqs(rng, 40, h2)
            cases.append(case(f"span{span}-{'rle' if rle else 'raw'}",
                              [Raw(pre), Seqs(lits_for(seqs, rng, 3, rle), seqs), Seqs(lits_for(first, rng, 0, rle), first)]))
    # self-overlapping matches whose source starts d = 1..15 bytes before the chunk: at sequence 0 and at sequence 31
    for rle in (None, 0x77):
        h = _Hist(len(pre))
        seqs = []
        for d in range(1, 16):
            seqs.append(h.add(0, d + 1 + rng.randrange(40), off(d)))                # sequence 0: ll = 0, source at -d
            seqs += [h.add(LIT_RUNS[k % 8] if k % 3 else 0, 3, off(1 + rng.randrange(30))) for k in range(1, 31)]
            seg_m = sum(a + b for a, b, _ in seqs[-31:]) + 2                         # chunk-relative start of sequence 31's match
            seqs.append(h.add(2, seg_m + d + 20 + rng.randrange(40), off(seg_m + d)))
        cases.append(case(f"overlap-before-chunk-{'rle' if rle else 'raw'}", [Raw(pre), Seqs(lits_for(seqs, rng, 9, rle), seqs)]))
    # chains: match j reads match j-1's output, inside one chunk (and across into the next)
    for rle in (None, 0x3C):
        h = _Hist(len(pre))
        seqs = []
        prev_ml = None
        for j in range(96):
            ll = LIT_RUNS[j % 8]
            ml = 3 + rng.randrange(30)
            o = off(prev_ml + ll) if prev_ml else off(7)
            seqs.append(h.add(ll, ml, o))
            prev_ml = ml
        cases.append(case(f"chain-{'rle' if rle else 'raw'}", [Raw(pre), Seqs(lits_for(seqs, rng, 0, rle), seqs)]))
    # last-literal tails of 0..33 bytes
    for tail in range(34):
        h = _Hist(len(pre))
        seqs = _small_seqs(rng, 5 + tail % 3, h)
        cases.append(case(f"tail{tail}", [Raw(pre), Seqs(lits_for(seqs, rng, tail, 0x42 if tail % 2 else None), seqs)]))
    return cases


# ---------------------------------------------------------------------------
# 2. offset reach: matches that reach back to the first byte of the frame
# ---------------------------------------------------------------------------
def _reach_blocks(rng, total):
    """Blocks of <= min(total, 128 KiB) each, a Raw and an RLE block first, then compressed ones whose matches reach back to
    byte 0, into the Raw block, into the RLE block and across the boundaries between them."""
    bmax = min(total, S.BLOCK_MAX)
    raw_n = min(bmax, total // 4)
    rle_n = min(bmax, total // 8)
    blocks = [Raw(_rb(rng, raw_n)), Rle(0x9E, rle_n)]
    h = _Hist(raw_n + rle_n)
    while total - h.produced > 100:
        room = min(bmax, total - h.produced)
        seqs = []
        out = 0
        while out + 80 < room:
            ll = rng.choice([0, 1, 5, 16])
            before = h.produced + ll
            pick = rng.randrange(5)
            if pick == 0:
                o = before                                  # the first byte of the frame
            elif pick == 1:
                o = before - raw_n + rng.randrange(1, 9)    # straddles Raw -> RLE
            elif pick == 2:
                o = before - raw_n - rng.randrange(rle_n)   # inside the RLE block
            elif pick == 3:
                o = before - (raw_n + rle_n) + rng.randrange(1, 9)  # straddles RLE -> the first compressed block
            else:
                o = 1 + rng.randrange(before)
            o = max(1, min(o, before))
            ml = min(3 + rng.randrange(40), room - out - ll)
            if ml < 3:
                break
            seqs.append(h.add(ll, ml, off(o)))
            out += ll + ml
        blocks.append(Seqs(lits_for(seqs, rng, 0), seqs))
    return blocks


def family_reach(seed=2):
    rng = random.Random(seed)
    cases = []
    for wl in range(10, 24):
        total = min(1 << wl, 300 << 10)
        cases.append(case(f"reach-wl{wl}", _reach_blocks(rng, total), single_segment=False, window_log=wl))
    for total in (1000, 70000, 300 << 10):
        cases.append(case(f"reach-ss{total}", _reach_blocks(rng, total)))
    # a source that straddles the boundary of two 128 KiB blocks
    a, b = _rb(rng, S.BLOCK_MAX), _rb(rng, S.BLOCK_MAX)
    h = _Hist(2 * S.BLOCK_MAX)
    seqs = [h.add(0, 200, off(S.BLOCK_MAX + 100)), h.add(3, 64, off(2 * S.BLOCK_MAX + 203 - 10)), h.add(1, 500, off(S.BLOCK_MAX + 7))]
    cases.append(case("reach-straddle-128k", [Raw(a), Raw(b), Seqs(lits_for(seqs, rng, 2), seqs)], single_segment=False, window_log=19))
    return cases


# ---------------------------------------------------------------------------
# 3. repeat offsets and symbolic history
# ---------------------------------------------------------------------------
REP_COMBOS = [(ll, v) for ll in (0, 1) for v in (1, 2, 3)]


def _rep_seqs(rng, h, n, only_rep=False):
    seqs = []
    for i in range(n):
        for _ in range(100):
            ll0, v = REP_COMBOS[(i + rng.randrange(2)) % 6] if only_rep or i % 3 else (rng.choice([0, 2]), off(1 + rng.randrange(60)))
            ll = ll0 * (1 + rng.randrange(4)) if ll0 else 0
            if h.ok(ll, v):
                break
        else:
            ll, v = 1, rep(1)
        seqs.append(h.add(ll, 3 + rng.randrange(20), v))
    return seqs


def family_repeat(seed=3):
    rng = random.Random(seed)
    cases = []
    # the first block's repeat codes run on the initial history (1, 4, 8)
    for v in (1, 2, 3):
        for ll in (0, 9):
            h = _Hist()
            seqs = [h.add(9, 3, rep(1)) if not (ll == 9 and v == 1) else h.add(9, 4, rep(1))]
            if h.ok(ll, v):
                seqs.append(h.add(ll, 5, v))
            seqs += _rep_seqs(rng, h, 12)
            cases.append(case(f"rep-initial-ll{ll}-v{v}", [Seqs(lits_for(seqs, rng, 4), seqs)]))
    # chains across >= 6 compressed blocks with Raw, RLE and zero-sequence blocks between them
    for variant in range(4):
        pre = _rb(rng, 100)
        blocks = [Raw(pre)]
        h = _Hist(len(pre))
        for k in range(8):
            seqs = _rep_seqs(rng, h, 1 + rng.randrange(70), only_rep=(k % 2 == 1))
            tbl = ("predefined", "predefined", "predefined") if k == 0 or variant % 2 else ("repeat", "repeat", "repeat")
            blocks.append(Seqs(lits_for(seqs, rng, k % 3, 0x61 if (variant + k) % 3 == 0 else None), seqs, tbl))
            gap = (k + variant) % 3
            if gap == 0:
                blocks.append(Raw(_rb(rng, 1 + rng.randrange(50)))); h.skip(len(blocks[-1].data))
            elif gap == 1:
                blocks.append(Rle(0x33, 1 + rng.randrange(50))); h.skip(blocks[-1].n)
            else:
                t = _rb(rng, rng.randrange(20))
                blocks.append(Seqs(t, [])); h.skip(len(t))
        cases.append(case(f"rep-chain{variant}", blocks, single_segment=bool(variant % 2), window_log=17))
    # blocks made only of repeat codes, after blocks that set the history with plain offsets
    pre = _rb(rng, 500)
    h = _Hist(len(pre))
    b1 = [h.add(5, 4, off(o)) for o in (17, 101, 333)]
    blocks = [Raw(pre), Seqs(lits_for(b1, rng, 0), b1)]
    for k in range(6):
        s = _rep_seqs(rng, h, 6 + 13 * k, only_rep=True)
        blocks.append(Seqs(lits_for(s, rng, 1), s))
    cases.append(case("rep-only-blocks", blocks))
    return cases


# ---------------------------------------------------------------------------
# 4. k_exec_big window
# ---------------------------------------------------------------------------
BIG_OFFS = [8127, 8128, 8129, 12287, 12288, 16383, 16384, 16385]
BIG_MLS = [3, 16, 17, 64, 1500]


def _filler(rng, h, n_chunks, ll=24, ml=8):
    """Chunks of 32 sequences of ll literals + a short match each: 32 * (ll + ml) bytes per chunk."""
    return [h.add(ll, ml, off(1 + rng.randrange(40))) for _ in range(32 * n_chunks)]


def family_big(seed=4):
    rng = random.Random(seed)
    cases = []
    for o in BIG_OFFS:
        h = _Hist()
        seqs = [h.add(40, 3, off(1 + rng.randrange(40)))] + _filler(rng, h, 24)[1:]   # 24 KiB of window chunks
        for ml in BIG_MLS:
            # align the match's source so that it crosses a multiple of 16384 (the window wraps there when dst is aligned)
            chunk = _filler(rng, h, 1, ll=8, ml=4)[:20]
            pos = h.produced + 8
            src = pos - o
            want = ((src // 16384) + 1) * 16384 - min(ml // 2, 8)
            pad = (want - src) % 16384 if ml < 1500 else 0
            pad = pad if pad < 2000 else pad % 700
            chunk.append(h.add(8 + pad, ml, off(o)))
            chunk += _filler(rng, h, 1, ll=8, ml=4)[:11]
            seqs += chunk
        cases.append(case(f"big-off{o}", [Seqs(lits_for(seqs, rng, 3), seqs, (("fse", 9), ("fse", 8), ("fse", 9)))]))
    # chunks of exactly 1024 / 1025 bytes in a long run
    h = _Hist()
    seqs = _filler(rng, h, 20)
    for span in (1024, 1025, 1024, 1023, 1025):
        seqs += _span_chunk(rng, h, span)
    seqs += [h.add(3, 64, off(o)) for o in (8127, 8128, 12288, 16383, 16384)]
    cases.append(case("big-spans", [Seqs(lits_for(seqs, rng, 0), seqs)]))
    # one 20 KiB sequence (straight to dst), then short-offset matches that read it
    h = _Hist()
    seqs = _filler(rng, h, 3) + [h.add(20480, 3, off(50)), h.add(0, 64, off(100)), h.add(5, 40, off(2000))]
    seqs += [h.add(3, 20480, off(7)), h.add(0, 64, off(30)), h.add(2, 100, off(19000))] + _filler(rng, h, 2)
    cases.append(case("big-single-20k", [Seqs(lits_for(seqs, rng, 1), seqs)]))
    return cases


# ---------------------------------------------------------------------------
# 5. k_exec_flow windows, both shapes
# ---------------------------------------------------------------------------
FLOW_SHAPES = {"narrow": (65536, 4096), "wide": (131072, 8192)}


def family_flow(seed=5):
    rng = random.Random(seed)
    cases = []
    for shape, (win, sl) in FLOW_SHAPES.items():
        reach = win // 2 + sl
        offs = [reach - 1, reach, reach + 1, win - 1, win, win + 1, 2 * win - 1, 2 * win + 1]
        pre = [Raw(_rb(rng, S.BLOCK_MAX)), Raw(_rb(rng, S.BLOCK_MAX))]
        h = _Hist(2 * S.BLOCK_MAX)
        seqs = _filler(rng, h, 80, ll=16, ml=16)  # 80 KiB of 1 KiB chunks in this block
        for o in offs:
            if o < h.produced - 2 * S.BLOCK_MAX or o > 2 * S.BLOCK_MAX:
                seqs += _filler(rng, h, 1, ll=16, ml=16)[:13] + [h.add(4, 40, off(o))] + _filler(rng, h, 1, ll=16, ml=16)[:18]
        cases.append(case(f"flow-{shape}-offs", pre + [Seqs(lits_for(seqs, rng, 0), seqs)], single_segment=False, window_log=20))
        # chunk spans of SLICE and SLICE + 1
        h = _Hist(2 * S.BLOCK_MAX)
        seqs = _filler(rng, h, 4, ll=16, ml=16)
        for span in (sl, sl + 1, sl, sl - 1, sl + 1):
            seqs += _span_chunk(rng, h, span)
        seqs += _filler(rng, h, 4, ll=16, ml=16)
        cases.append(case(f"flow-{shape}-slice", pre + [Seqs(lits_for(seqs, rng, 0), seqs)], single_segment=False, window_log=20))
    # long dependency chains: every chunk's last match copies the previous chunk's last match
    h = _Hist(1024)
    seqs, last_at, last_ml = [], None, None
    for c in range(200):
        chunk = [h.add(2, 3 + rng.randrange(8), off(1 + rng.randrange(30))) for _ in range(31)]
        at = h.produced + 1
        ml = 40 + rng.randrange(40)
        chunk.append(h.add(1, ml, off(at - last_at) if last_at else off(900)))
        last_at = at
        seqs += chunk
    cases.append(case("flow-chain", [Raw(_rb(rng, 1024)), Seqs(lits_for(seqs, rng, 0), seqs)]))
    # more than 256 small chunks in flight: 400 chunks of 96 bytes
    h = _Hist(64)
    seqs = [h.add(0, 3, off(1 + rng.randrange(60))) for _ in range(32 * 400)]
    cases.append(case("flow-many-chunks", [Raw(_rb(rng, 64)), Seqs(lits_for(seqs, rng, 5), seqs)]))
    return cases


# ---------------------------------------------------------------------------
# 6. batch seams and the number-of-sequences header forms
# ---------------------------------------------------------------------------
def _dense(rng, h, n):
    out = []
    for i in range(n):
        ll = 1 if i % 23 == 0 else 0
        v = off(1 + rng.randrange(64)) if i % 5 else rep(1 + i % 3) if h.ok(ll, rep(1 + i % 3)) else off(9)
        out.append(h.add(ll, 3, v))
    return out


def family_batch(seed=6):
    rng = random.Random(seed)
    cases = []
    for n in (32767, 32768, 32769, 43000):
        h = _Hist(64)
        seqs = _dense(rng, h, n)
        cases.append(case(f"batch-n{n}", [Raw(_rb(rng, 64)), Seqs(lits_for(seqs, rng, 0), seqs, (("fse", 6), ("fse", 8), "predefined"))]))
    for n, form in ((127, 1), (127, 2), (128, 2), (0x7EFF, 2), (0x7F00, 3)):
        h = _Hist(64)
        seqs = _dense(rng, h, n)
        cases.append(case(f"nbseq{n}-form{form}", [Raw(_rb(rng, 64)), Seqs(lits_for(seqs, rng, 2), seqs, nbseq_form=form)]))
    return cases


# ---------------------------------------------------------------------------
# 7. table modes side by side
# ---------------------------------------------------------------------------
POOLS = (list(range(0, 20)), list(range(0, 16)), list(range(0, 25)))   # LL, OF, ML codes an FSE / predefined table is used with
MODES = ["predefined", "rle", "fse5", "fsemax", "repeat"]


def _spec(kind, mode, rng):
    if mode == "predefined":
        return "predefined", POOLS[kind]
    if mode == "rle":
        c = rng.choice(POOLS[kind][2:])
        return ("rle", c), [c]
    log = 5 if mode == "fse5" else S.MAX_LOG[kind]
    return ("fse", log, S.normalized_counts(POOLS[kind], log, lt1=(mode == "fsemax"))), POOLS[kind]


def _value(kind, code, rng):
    if kind == 0:
        return S.LL_BASE[code] + rng.randrange(1 << S.LL_BITS[code])
    if kind == 2:
        return S.ML_BASE[code] + rng.randrange(1 << S.ML_BITS[code])
    return (1 << code) + rng.randrange(1 << code)


def _table_block(rng, h, specs_pools, n):
    seqs = []
    (_, llp), (_, ofp), (_, mlp) = specs_pools
    while len(seqs) < n:
        ll = _value(0, rng.choice(llp), rng)
        ml = _value(2, rng.choice(mlp), rng)
        for _ in range(50):
            v = _value(1, rng.choice(ofp), rng)
            if h.ok(ll, v):
                break
        else:
            if len(ofp) == 1:
                return None
            continue
        seqs.append(h.add(ll, ml, v))
    return seqs


def family_tables(seed=7):
    rng = random.Random(seed)
    cases = []
    combos = [(a, b, c) for a in MODES for b in MODES for c in MODES]
    rng.shuffle(combos)
    for f in range(0, len(combos), 5):
        pre = _rb(rng, 1 << 16)
        blocks = [Raw(pre)]
        h = _Hist(len(pre))
        prev = None
        for combo in combos[f:f + 5]:
            sp = []
            for kind, mode in enumerate(combo):
                if mode == "repeat":
                    sp.append(("repeat", prev[kind][1]) if prev else _spec(kind, "predefined", rng))
                else:
                    sp.append(_spec(kind, mode, rng))
            for _ in range(20):
                trial = _Hist(h.produced); trial.h = list(h.h)
                seqs = _table_block(rng, trial, sp, 1 + rng.randrange(90))
                if seqs is not None:
                    break
            h = trial
            blocks.append(Seqs(lits_for(seqs, rng, rng.randrange(4)), seqs, tuple(s for s, _ in sp)))
            prev = [(s, p) if s != "repeat" else prev[k] for k, (s, p) in enumerate(sp)]
        cases.append(case("tables-" + "|".join(",".join(c) for c in combos[f:f + 5]), blocks))
    return cases


def risky_pair(seed=8):
    """The same sequences under an LL table that declares an unused symbol above code 35 (so k_fse takes the exact loop) and
    under a plain one.  libzstd rejects a literal-length table with a symbol above 35, so the first frame is pinned by the
    oracle and by the plain twin only."""
    rng = random.Random(seed)
    h = _Hist(256)
    seqs = _small_seqs(rng, 70, h)
    codes = [S.ll_code(ll) for ll, _, _ in seqs]
    plain = S.normalized_counts(codes, 7)
    risky = S.normalized_counts(codes, 7, extra=(40,))
    pre = _rb(rng, 256)
    lits = lits_for(seqs, rng, 3)
    a = case("risky-ll-table", [Raw(pre), Seqs(lits, seqs, (("fse", 7, risky), "predefined", "predefined"))], libzstd="reject")
    b = case("risky-twin", [Raw(pre), Seqs(lits, seqs, (("fse", 7, plain), "predefined", "predefined"))])
    return [a, b]


# ---------------------------------------------------------------------------
# 8. invalid by construction
# ---------------------------------------------------------------------------
def family_invalid(seed=9):
    rng = random.Random(seed)
    cases = []
    pre = _rb(rng, 300)
    # offset = produced + 1 (in a block after the first, and across a Raw block)
    s = [(3, 4, off(100)), (2, 5, off(300 + 3 + 4 + 2 + 1))]
    cases.append(case("invalid-offset-past-start", [Raw(pre), Seqs(lits_for(s, rng, 0), s)]))
    # rep0 - 1 resolving to 0: history starts at (1, 4, 8); ll = 0 and repeat code 3 names h0 - 1
    s = [(0, 4, rep(3))]
    cases.append(case("invalid-rep0-minus-1", [Raw(pre), Seqs(b"", s)]))
    s = [(2, 4, off(1)), (0, 5, rep(3))]
    cases.append(case("invalid-rep0-minus-1-later", [Raw(pre), Seqs(lits_for(s, rng, 0), s)]))
    # the sequences consume more literals than the section holds
    s = [(10, 4, off(5)), (20, 4, off(9))]
    cases.append(case("invalid-ll-past-literals", [Raw(pre), Seqs(_rb(rng, 25), s)]))
    # exact capacity minus one
    h = _Hist(len(pre))
    s = _small_seqs(rng, 40, h)
    c = case("invalid-capacity-minus-1", [Raw(pre), Seqs(lits_for(s, rng, 3), s)])
    c.cap -= 1
    c.expected, c.libzstd = "CZS_DST_TOO_SMALL", "reject"
    cases.append(c)
    # a block whose regen + sum(ml) exceeds 128 KiB: neither the reference semantics nor libzstd 1.5 limit a block's output
    h = _Hist(64)
    s = [h.add(0, 1000 + rng.randrange(40), off(1 + rng.randrange(64))) for _ in range(140)]
    cases.append(case("block-output-over-128k", [Raw(_rb(rng, 64)), Seqs(b"", s)], libzstd=None))
    return cases


# ---------------------------------------------------------------------------
# 9. resume points of the FrameDecoder handle
# ---------------------------------------------------------------------------
RESUME_OPTS = [dict(), dict(single_segment=False, window_log=10), dict(single_segment=False, window_log=10, checksum=False, fcs_width=0),
               dict(checksum=False)]


def family_resume(seed=10):
    """Frames for the FrameDecoder handle fed block by block, where every device run starts after the blocks earlier runs
    executed (FrameResume): a Raw / RLE prefix before each compressed block puts a resume point right in front of it.
      - output before the resume point at every residue mod 16;
      - the first sequence after it with offset 1 (a self-overlapping match starting on the resume point), 2..15, the first
        byte of the frame (out0), out0 - 1 and the window;
      - repeat codes first after it (ll = 0 and ll > 0, repeat 3 with ll = 0 = h0 - 1) on a history set before it;
      - Repeat-mode tables whose FSE / RLE definition lies 1, 2 and 50 blocks back, over zero-output blocks (Raw(b""),
        Rle(x, 0), a literals-only block of 0 bytes);
    with window_log 10 (collect and read drain many windows) or single segment, with and without checksum and content size."""
    rng = random.Random(seed)
    cases = []

    def gap(blocks, h, n):
        blocks.append(Raw(_rb(rng, n)) if rng.random() < 0.5 else Rle(rng.randrange(256), n))
        h.skip(n)

    for r in range(16):
        opts = RESUME_OPTS[r % 4]
        window = 1 << 10 if "window_log" in opts else None
        blocks, h = [], _Hist()
        gap(blocks, h, 1024 + 16 * rng.randrange(8) + r)           # out0 = r (mod 16)
        for k in range(4):
            out0 = h.produced
            o = [1 + (r + k) % 15, out0, out0 - 1, window or out0 - 2][k]
            seqs = [h.add(0, o + 3 + rng.randrange(30) if k == 0 else 3 + rng.randrange(40), off(o))]
            seqs += _rep_seqs(rng, h, 4 + rng.randrange(30))
            tbl = ("predefined",) * 3 if k % 2 else (("fse", 6), ("fse", 5), ("fse", 6))
            blocks.append(Seqs(lits_for(seqs, rng, rng.randrange(3)), seqs, tbl))
            gap(blocks, h, 16 * rng.randrange(1, 40) + (r + 5 * k) % 16)
        cases.append(case(f"resume-first-seq-r{r}", blocks, **opts))
    # repeat codes first after the resume point, on a history the block before it set
    for variant in range(4):
        opts = RESUME_OPTS[variant]
        blocks, h = [], _Hist()
        gap(blocks, h, 700 + variant)
        for ll0, v in REP_COMBOS:
            setter = [h.add(2, 4, off(2 + rng.randrange(300))) for _ in range(3)]
            blocks.append(Seqs(lits_for(setter, rng, 1), setter))
            gap(blocks, h, 1 + rng.randrange(90))
            ll = ll0 * (1 + rng.randrange(3))
            if not h.ok(ll, v):
                ll = 1
            seqs = [h.add(ll, 3 + rng.randrange(20), v)] + _rep_seqs(rng, h, 3 + rng.randrange(10), only_rep=True)
            blocks.append(Seqs(lits_for(seqs, rng, 0), seqs))
            if variant % 2:
                gap(blocks, h, rng.randrange(40))
        cases.append(case(f"resume-rep-first-v{variant}", blocks, **opts))
    # Repeat-mode tables defined 1, 2 and 50 blocks earlier, FSE and RLE definitions, zero-output blocks between
    lls, mls, offs = (1, 2, 5, 9), (3, 4, 7, 10), range(5, 29)     # offsets 5..28: offset codes 3 and 4

    def table_block(h, rle):
        if rle:
            seqs = [h.add(5, 7, off(rng.choice(offs))) for _ in range(12)]
            return Seqs(lits_for(seqs, rng, 2), seqs, (("rle", S.ll_code(5)), ("fse", 5), ("rle", S.ml_code(7))))
        seqs = [h.add(a, b, off(o)) for a in lls for b in mls for o in (6, 20)]
        rng.shuffle(seqs)
        return Seqs(lits_for(seqs, rng, 1), seqs, (("fse", 6), ("fse", 5), ("fse", 6)))

    for n_between in (1, 2, 50):
        for rle in (False, True):
            opts = RESUME_OPTS[(n_between + rle) % 4]
            blocks, h = [], _Hist()
            gap(blocks, h, 512 + n_between)
            for _ in range(2):
                blocks.append(table_block(h, rle))
                for j in range(n_between):
                    z = j % 4
                    if z == 0:
                        blocks.append(Raw(b""))
                    elif z == 1:
                        blocks.append(Rle(0x5C, 0))
                    elif z == 2:
                        blocks.append(Seqs(b"", []))
                    else:
                        gap(blocks, h, 1 + rng.randrange(60))
                if rle:
                    seqs = [h.add(5, 7, off(rng.choice(offs))) for _ in range(9)]
                else:
                    seqs = [h.add(rng.choice(lls), rng.choice(mls), off(rng.choice((6, 20)))) for _ in range(20)]
                blocks.append(Seqs(lits_for(seqs, rng, 3), seqs, ("repeat", "repeat", "repeat")))
                blocks.append(Seqs(b"", []))
            cases.append(case(f"resume-repeat-tables-{n_between}-{'rle' if rle else 'fse'}", blocks, **opts))
    # no content size, and a late block that regenerates more than 128 KiB: the handle's output bound for the blocks it has
    # not run is too small in the middle of the frame; the next block matches into output written before that
    h = _Hist()
    blocks = [Raw(_rb(rng, 3000)), Rle(0x21, 5000)]
    h.skip(8000)
    s = [h.add(0, 1000 + rng.randrange(40), off(1 + rng.randrange(7000))) for _ in range(140)]
    blocks += [Seqs(b"", s), Raw(_rb(rng, 100))]
    h.skip(100)
    s = [h.add(1, 200, off(h.produced + 1 - rng.randrange(1, 2000))) for _ in range(5)]
    blocks.append(Seqs(lits_for(s, rng, 2), s))
    cases.append(case("resume-late-block-over-128k", blocks, libzstd=None, single_segment=False, window_log=20, fcs_width=0))
    return cases


FAMILIES = {
    "chunks": family_chunks, "reach": family_reach, "repeat": family_repeat, "big": family_big, "flow": family_flow,
    "batch": family_batch, "tables": lambda: family_tables() + risky_pair(), "invalid": family_invalid,
    "resume": family_resume,
}

_cache = {}


def cases(name):
    if name not in _cache:
        _cache[name] = FAMILIES[name]()
    return _cache[name]
