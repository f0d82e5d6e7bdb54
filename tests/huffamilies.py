"""Frames whose literals are Huffman sections built from explicit codes (tests/hufbuild.py), placed where k_huff_prep and k_huff
change their behaviour:

  tables     max_bits <= 9 decodes from 1 KiB tables (k_huff<9>), 10 and 11 from 4 KiB tables (k_huff<11>); direct weights
             (<= 128) or FSE-coded ones (<= 255); the implicit last weight; sparse alphabets.
  streams    lane = section * 4 + stream; stream k writes from k * ceil(regen / 4) in the 16-byte aligned literal scratch: single
             literals until the write pointer is aligned (head 0..15), then 16 literals per iteration while >= 176 bits remain and
             16 more are expected, then 4 while >= 44 bits remain, then single literals; four() decodes 4 codes from one 64-bit
             window.  1-stream sections have no end check, 4-stream sections not split as RFC 8878 says are decoded again
             serially (huf_decode_concatenated).
  chains     Treeless sections re-derive the tree of the block k_fill_blocks names (last_huf).

Each family returns seqfamilies.Case objects (plus the block list, for the literal-scratch check of tests/test_gpu_huff.py);
`expected` is hufbuild.reference_decode's output or the oracle status name of the failure, `libzstd` says whether libzstd must
accept the frame ("ok"), must reject it ("reject") or is not asked (None: layouts only the reference accepts)."""
import random

import numpy as np

import hufbuild as H
import seqbuild as S
import seqfamilies as F
from hufbuild import Huf, Treeless
from seqbuild import Raw, Rle, Seqs, off


def case(name, blocks, libzstd="ok", cap=None, **opts):
    window = (1 << opts["window_log"]) if not opts.get("single_segment", True) else None
    exp = H.reference_decode(blocks, window)
    if not isinstance(exp, bytes) and window is None:
        exp = H.reference_decode(blocks, 0)
    content = exp if isinstance(exp, bytes) else b""
    frame = S.build_frame(blocks, content=content, **opts)
    if cap is None:
        cap = len(exp) if isinstance(exp, bytes) else 1 << 20
    c = F.Case(name, frame, exp, cap, libzstd if isinstance(exp, bytes) else "reject")
    c.blocks = blocks
    return c


def draw(rng, lengths, n, every=True):
    """n literals over the alphabet of `lengths` ({symbol: code length}), symbol s with probability ~ 2^-len(s); with `every`
    each symbol occurs at least once (when n allows)."""
    syms = sorted(lengths)
    p = np.array([2.0 ** -lengths[s] for s in syms])
    out = rng.choice(np.array(syms, dtype=np.uint8), size=n, p=p / p.sum())
    if every and n >= len(syms):
        out[rng.choice(n, size=len(syms), replace=False)] = syms
    return out.tobytes()


def with_seqs(rng, lits_len, produced):
    """Sequences that consume the first part of a literals section of lits_len bytes (offsets into `produced` bytes of
    history plus what they add), leaving a tail of literals."""
    h = F._Hist(produced)
    seqs, used = [], 0
    while used + 40 < lits_len * 3 // 4:
        ll = rng.choice(F.LIT_RUNS)
        seqs.append(h.add(ll, 3 + rng.randrange(30), off(1 + rng.randrange(min(60, h.produced + ll)))))
        used += ll
    return seqs


def _alphabet(rng, n, hi):
    return sorted(rng.sample(range(hi), n))


# ---------------------------------------------------------------------------
# 1. code lengths and table classes
# ---------------------------------------------------------------------------
def family_tables(seed=21):
    rng = random.Random(seed)
    nrng = np.random.default_rng(seed)
    pre = bytes(rng.getrandbits(8) for _ in range(64))
    cases = []
    for L in range(1, 12):
        for streams in (1, 4):
            for tree in ("direct", "fse"):
                hi = 129 if tree == "direct" else 256
                n = rng.randrange(L + 1, min(1 << L, hi) + 1) if L > 1 else 2
                alpha = _alphabet(rng, n, hi)
                if tree == "fse" and alpha[-1] < 2:
                    alpha[-1] = 2 + rng.randrange(200)   # FSE weights: two states, so at least two explicit weights
                lens = H.complete_lengths(rng.sample(alpha, n), L)
                spec = "direct" if tree == "direct" else ("fse", 5 + L % 2)
                nl = rng.randrange(200, 1000) if streams == 1 else rng.randrange(1200, 6000)
                lits = draw(nrng, lens, nl)
                blocks = [Raw(pre)]
                if L % 3 == 0:
                    blocks.append(Seqs(Huf(lits, H.weights_of(lens), L, spec, streams), with_seqs(rng, nl, len(pre))))
                else:
                    blocks.append(Seqs(Huf(lits, H.weights_of(lens), L, spec, streams), []))
                cases.append(case(f"mb{L}-{streams}s-{tree}-{n}sym", blocks))
    # every code length 1..11 at once; alphabets of 2, 3, 128, 129, 256 symbols; sparse ones (the last is the implicit weight)
    shapes = [("len1to11", list(range(40, 52)), 11), ("2sym", [7, 9], 1), ("3sym", [0, 1, 2], 2), ("128sym", list(range(128)), 8),
              ("129sym", list(range(129)), 9), ("256sym", list(range(256)), 11), ("256sym-flat", list(range(256)), 8),
              ("sparse-0-200-255", [0, 200, 255], 2), ("sparse-0-100-127", [0, 100, 127], 2), ("sparse-255-only-high", [250, 255], 1)]
    for name, alpha, L in shapes:
        lens = H.complete_lengths(alpha, L)
        for streams in (1, 4):
            for spec in ("direct", ("fse", 6)):
                if spec == "direct" and max(alpha) > 128:
                    continue
                if spec != "direct" and max(alpha) < 2:
                    continue
                nl = 900 if streams == 1 else 5000
                lits = draw(nrng, lens, nl)
                cases.append(case(f"{name}-{streams}s-{'direct' if spec == 'direct' else 'fse'}",
                                  [Seqs(Huf(lits, H.weights_of(lens), L, spec, streams), [])]))
    # FSE weight tables with accuracy logs libzstd does not take (7..9 from shared memory, 10 through k_huff_prep's global table)
    for log in (7, 9, 10):
        lens = H.complete_lengths(list(range(30)), 7)
        lits = draw(nrng, lens, 3000)
        cases.append(case(f"fse-log{log}", [Seqs(Huf(lits, H.weights_of(lens), 7, ("fse", log), 4), [])], libzstd=None))
    # both classes back to back in one frame: max_bits 9, 10, 9, 11, 1, 10 (with sequences in between)
    blocks, produced = [Raw(pre)], len(pre)
    for k, L in enumerate((9, 10, 9, 11, 1, 10)):
        lens = H.complete_lengths(_alphabet(rng, min(1 << L, L + 1 + rng.randrange(60)), 256), L)
        lits = draw(nrng, lens, 4000)
        seqs = with_seqs(rng, len(lits), produced) if k % 2 else []
        blocks.append(Seqs(Huf(lits, H.weights_of(lens), L, ("fse", 6), 4 if k % 3 else 1 if len(lits) < 1024 else 4), seqs))
        produced += len(lits) + sum(m for _, m, _ in seqs)
    cases.append(case("classes-9-10-9-11-1-10", blocks))
    return cases


# ---------------------------------------------------------------------------
# 2. stream geometry
# ---------------------------------------------------------------------------
LONG = H.complete_lengths(list(range(60, 72)), 11)        # every length 1..11: symbols 60..69 have 1..10 bits, 70 and 71 have 11
BIT1 = {0x30: 1, 0x31: 1}


def _for_bits(nbits, lens):
    """Symbols whose codes add up to exactly nbits: as many of the longest codes as fit, then one code of the rest."""
    by_len = {}
    for s, l in sorted(lens.items()):
        by_len.setdefault(l, s)
    top = max(by_len)
    q, r = divmod(nbits, top)
    out = [by_len[top]] * q + ([by_len[r]] if r else [])
    assert sum(lens[s] for s in out) == nbits
    return bytes(out)


def family_streams(seed=22):
    rng = random.Random(seed)
    nrng = np.random.default_rng(seed)
    cases = []
    mid = H.complete_lengths(list(range(32, 32 + 40)), 8)
    w_mid = H.weights_of(mid)
    # regen 1..80, 121..132 (stream sizes 15, 16, 17, 31, 32, 33) and 4 * seg - r for seg 200..215: every stream start mod 16
    regens = list(range(1, 81)) + list(range(121, 133)) + [4 * seg - (seg % 4) for seg in range(200, 216)]
    for i in range(0, len(regens), 8):
        blocks = []
        for regen in regens[i:i + 8]:
            lits = draw(nrng, mid, regen, every=False)
            blocks.append(Seqs(Huf(lits, w_mid, 8, ("fse", 6), 4), []))
        small = min(regens[i:i + 8]) < 6   # libzstd takes 4-stream sections of 6 literals or more only
        cases.append(case(f"regen{regens[i]}-{regens[min(i + 7, len(regens) - 1)]}", blocks, libzstd=None if small else "ok"))
    # streams of 43 / 44 / 45 and 175 / 176 / 177 bits: 11-bit codes (plus one shorter code) and 1-bit codes
    for lname, lens in (("11bit", LONG), ("1bit", BIT1)):
        w = H.weights_of(lens)
        for nbits in (43, 44, 45, 175, 176, 177):
            one = _for_bits(nbits, lens)
            blocks = [Seqs(Huf(one, w, max(lens.values()), "direct", 1), []),
                      Seqs(Huf(one * 4, w, max(lens.values()), "direct", 4), [])]
            cases.append(case(f"bits{nbits}-{lname}", blocks))
    # 4-literal groups of the longest codes (44 bits each), long and mixed 10/11-bit streams
    w = H.weights_of(LONG)
    for n, mix in ((3000, (70, 71)), (2003, (69, 70, 71)), (777, (70, 71, 60))):
        lits = bytes(rng.choice(mix) for _ in range(n))
        cases.append(case(f"wide-groups-{n}", [Seqs(Huf(lits, w, 11, "direct", 4), []), Seqs(Huf(lits[:600], w, 11, "direct", 1), [])]))
    # the limits of each literals header form (1-stream 10-bit; 4-stream 10 / 14 / 18-bit) and a 128 KiB section
    small = H.complete_lengths(list(range(65, 81)), 4)
    ws = H.weights_of(small)
    for regen, streams, sf in ((1023, 1, 0), (1023, 4, 1), (1024, 4, 2), (16383, 4, 2), (16384, 4, 3), (S.BLOCK_MAX, 4, 3)):
        lits = draw(nrng, small, regen)
        h = Huf(lits, ws, 4, ("fse", 6), streams)
        h.section({})
        assert h.info["sf"] == sf, (regen, h.info["sf"])
        cases.append(case(f"form{sf}-regen{regen}", [Seqs(h, [])]))
    # a larger form than the sizes need
    lits = draw(nrng, small, 300)
    cases.append(case("form3-regen300", [Seqs(Huf(lits, ws, 4, ("fse", 6), 4, size_format=3), [])]))
    return cases


# ---------------------------------------------------------------------------
# 3. Treeless chains
# ---------------------------------------------------------------------------
def family_treeless(seed=23):
    rng = random.Random(seed)
    nrng = np.random.default_rng(seed)
    cases = []
    l8 = H.complete_lengths(list(range(97, 123)) + [32, 46], 8)    # small class
    l10 = H.complete_lengths(list(range(40, 140)), 10)             # large class
    w8, w10 = H.weights_of(l8), H.weights_of(l10)
    pre = bytes(rng.getrandbits(8) for _ in range(100))
    d = [draw(nrng, l8, n) for n in (3000, 700, 5000)] + [draw(nrng, l10, n) for n in (4000, 900)]
    blocks = [Raw(pre), Seqs(Huf(d[0], w8, 8, ("fse", 6), 4), with_seqs(rng, len(d[0]), 100)),
              Seqs(Treeless(d[1], 1), []),
              Seqs(("rle", 0x5F, 300), []),
              Raw(b"raw block"), Rle(0x21, 77),
              Seqs(bytes(rng.getrandbits(8) for _ in range(50)), []),
              Seqs(Treeless(d[2], 4), []),
              Seqs(Huf(d[3], w10, 10, ("fse", 6), 4), []),
              Seqs(Treeless(d[4], 1), [])]
    cases.append(case("chain", blocks))
    # the same with sequences behind every section
    blocks2, produced = [Raw(pre)], len(pre)
    for k, b in enumerate(blocks[1:]):
        if isinstance(b, Seqs) and k % 2 == 0:
            n = len(S._lit_bytes(b.literals))
            seqs = with_seqs(rng, n, produced) if n > 60 else []
            b = Seqs(b.literals, seqs)
            produced += sum(m for _, m, _ in seqs)
        produced += len(S._lit_bytes(b.literals)) if isinstance(b, Seqs) else len(b.data) if isinstance(b, Raw) else b.n
        blocks2.append(b)
    cases.append(case("chain-with-seqs", blocks2))
    # a Treeless section before any tree of the frame: first section, and after Raw / RLE literals only
    cases.append(case("treeless-first", [Seqs(Treeless(d[1], 1, weights=w8), [])]))
    cases.append(case("treeless-after-raw-lits", [Raw(pre), Seqs(b"abc", []), Seqs(("rle", 1, 40), []), Seqs(Treeless(d[2], 4, weights=w8), [])]))
    # two frames: the second starts with a Treeless section coded with the first frame's tree, and must not find it
    cases.append(case("tree-owner", [Seqs(Huf(d[0], w8, 8, ("fse", 6), 4), [])]))
    cases.append(case("treeless-next-frame", [Seqs(Treeless(d[1], 1, weights=w8), [])]))
    return cases


# ---------------------------------------------------------------------------
# 4. layouts only the reference accepts
# ---------------------------------------------------------------------------
def family_refonly(seed=24):
    rng = random.Random(seed)
    nrng = np.random.default_rng(seed)
    cases = []
    l6 = H.complete_lengths(list(range(50, 90)), 6)
    w6 = H.weights_of(l6)
    w11 = H.weights_of(LONG)
    for n, split in ((2000, [0, 700, 5, 1295]), (2000, [2000, 0, 0, 0]), (2000, [1, 2, 3, 1994]), (601, [200, 200, 201, 0]),
                     (3333, [833, 834, 834, 832]), (300, [0, 0, 0, 300])):
        lits = draw(nrng, l6, n)
        cases.append(case(f"split-{'-'.join(map(str, split))}", [Seqs(Huf(lits, w6, 6, ("fse", 6), 4, split=split), [])], libzstd=None))
    lits = bytes(rng.choice((70, 71, 69)) for _ in range(1999))
    cases.append(case("split-11bit", [Seqs(Huf(lits, w11, 11, "direct", 4, split=[3, 1000, 990, 6]), [])], libzstd=None))
    # 1-stream over-read: the last code's trailing zero bits are not in the stream (symbol 70 has the all-zero 11-bit code)
    for nbits in (1, 5, 10):
        lits = bytes(rng.choice((60, 61, 70, 71)) for _ in range(500)) + bytes([70])
        cases.append(case(f"overread-1s-{nbits}", [Seqs(Huf(lits, w11, 11, "direct", 1, damage=("overread", 0, nbits)), [])], libzstd=None))
    # oversized sections: Huffman regen 200 000 and 2^18 - 1 (18-bit form), RLE literals 2^20 - 1; alone and with sequences in
    # front of a trailing literal run of more than 2^17 bytes
    l2 = H.complete_lengths([0x41, 0x42, 0x43, 0x44], 3)
    for regen in (200000, (1 << 18) - 1):
        lits = draw(nrng, l2, regen)
        cases.append(case(f"huf-regen{regen}", [Seqs(Huf(lits, H.weights_of(l2), 3, "direct", 4), [])], libzstd=None))
        h = F._Hist(0)
        seqs = [h.add(5, 4, off(3)), h.add(40000, 100, off(1000)), h.add(3, 3000, off(7))]
        cases.append(case(f"huf-regen{regen}-seqs", [Seqs(Huf(lits, H.weights_of(l2), 3, "direct", 4), seqs)], libzstd=None))
    n = (1 << 20) - 1
    cases.append(case("rle-lits-2^20-1", [Seqs(("rle", 0x41, n), [])], libzstd=None))
    h = F._Hist(0)
    seqs = [h.add(100, 50, off(1)), h.add(131071, 4, off(90000)), h.add(0, 3, F.rep(1))]
    cases.append(case("rle-lits-2^20-1-seqs", [Seqs(("rle", 0x41, n), seqs)], libzstd=None))
    return cases


# ---------------------------------------------------------------------------
# 5. invalid by construction
# ---------------------------------------------------------------------------
def _zero_ended(lits, zero_sym, streams):
    """The same literals with the last symbol of every stream replaced by zero_sym (whose code is all zero bits)."""
    b = bytearray(lits)
    counts = H.rfc_split(len(b)) if streams == 4 else [len(b)]
    pos = 0
    for c in counts:
        pos += c
        if c:
            b[pos - 1] = zero_sym
    return bytes(b)


def _weight_errors():
    fse_ok = H.fse_tree([3, 2, 2, 1, 0, 1, 1], 6)
    return [
        ("weight12", ("raw", H.direct_tree([12, 1, 1])), None, "CZS_HUF_WEIGHT_BIGGER_THAN_MAX_NUM_BITS"),
        ("all-zero", ("raw", H.direct_tree([0, 0, 0])), None, "CZS_HUF_MISSING_WEIGHTS"),
        ("leftover-3", ("raw", H.direct_tree([2, 2, 1])), None, "CZS_HUF_LEFTOVER_NOT_POWER_OF_2"),
        ("max-bits-12", ("raw", H.direct_tree([11, 11])), None, "CZS_HUF_MAX_BITS_TOO_HIGH"),
        ("direct-truncated", ("raw", H.direct_tree([1] * 9)), ("truncate", 3), "CZS_HUF_NOT_ENOUGH_BYTES_IN_SOURCE"),
        ("fse-desc-over-header", ("raw", bytes([1]) + fse_ok[1:]), None, "CZS_HUF_FSE_TABLE_USED_TOO_MANY_BYTES"),
        ("fse-header-over-payload", ("raw", fse_ok), ("truncate", 3), "CZS_HUF_NOT_ENOUGH_BYTES_FOR_WEIGHTS"),
        ("fse-zero-last", ("raw", fse_ok), ("tree_zero_last",), "CZS_HUF_EXTRA_PADDING"),
        ("256-weights", ("raw", H.fse_tree([1] * 256, 6)), None, "CZS_PANIC_INTERNAL"),
        ("258-weights", ("raw", H.fse_tree([1] * 258, 6)), None, "CZS_HUF_TOO_MANY_WEIGHTS"),
    ]


def family_invalid(seed=25):
    rng = random.Random(seed)
    nrng = np.random.default_rng(seed)
    cases = []
    l7 = H.complete_lengths(list(range(40, 100)), 7)
    w7 = H.weights_of(l7)
    zero_sym = H.read_tree(H.direct_tree(w7[:-1])).symbol[0]
    lits4 = _zero_ended(draw(nrng, l7, 2000), zero_sym, 4)
    lits1 = _zero_ended(draw(nrng, l7, 600), zero_sym, 1)
    bad = [("jump-header", Huf(lits4, w7, 7, "direct", 4, damage=("truncate", len(H.direct_tree(w7[:-1])) + 5), expect="CZS_MISSING_BYTES_FOR_JUMP_HEADER")),
           ("jump-past-end", Huf(lits4, w7, 7, "direct", 4, damage=("jump", (0xFFFF, 0xFFFF, 0xFFFF)), expect="CZS_MISSING_BYTES_FOR_LITERALS"))]
    for k in range(4):
        bad.append((f"empty-stream{k}", Huf(lits4, w7, 7, "direct", 4, damage=("empty", k), expect="CZS_LIT_EXTRA_PADDING")))
        bad.append((f"zero-last-stream{k}", Huf(lits4, w7, 7, "direct", 4, damage=("zero_last", k), expect="CZS_LIT_EXTRA_PADDING")))
        bad.append((f"overread-stream{k}", Huf(lits4, w7, 7, "direct", 4, damage=("overread", k, 1), expect="CZS_BITSTREAM_READ_MISMATCH")))
        # the cut lands on a code boundary of stream 1: that stream then ends cleanly, one literal short
        bad.append((f"cut-stream{k}", Huf(lits4, w7, 7, "direct", 4, damage=("cut", k, 3),
                                          expect="CZS_DECODED_LITERAL_COUNT_MISMATCH" if k == 1 else "CZS_BITSTREAM_READ_MISMATCH")))
    bad.append(("zero-last-1s", Huf(lits1, w7, 7, "direct", 1, damage=("zero_last", 0), expect="CZS_LIT_EXTRA_PADDING")))
    for streams, lits in ((1, lits1), (4, lits4)):
        for dn in (1, -1):
            bad.append((f"count{'+' if dn > 0 else '-'}1-{streams}s", Huf(lits, w7, 7, "direct", streams, regen=len(lits) + dn,
                                                                         expect="CZS_DECODED_LITERAL_COUNT_MISMATCH")))
    for name, tree, dmg, st in _weight_errors():
        bad.append((name, Huf(b"\x00\x01" * 20, tree=tree, damage=dmg, expect=st)))
    good = Huf(draw(nrng, l7, 1500), w7, 7, ("fse", 6), 4)
    pre = bytes(rng.getrandbits(8) for _ in range(40))
    for name, h in bad:
        cases.append(case(f"bad-{name}", [Seqs(h, [])]))
        cases.append(case(f"bad-{name}-block2", [Seqs(good, []), Seqs(h, [])]))
        # behind an earlier error of the frame: block 1 matches 100 bytes back with 40 + 2 produced
        cases.append(case(f"bad-{name}-behind", [Raw(pre), Seqs(b"xy", [(2, 4, off(100))]), Seqs(h, [])]))
    return cases


# ---------------------------------------------------------------------------
# 6. the seam families of seqfamilies.py with Huffman literals
# ---------------------------------------------------------------------------
def _as_huf(lits, k):
    data = S._lit_bytes(lits)
    if len(set(data)) < 2:
        return lits
    streams = 1 if len(data) < 6 or (len(data) < 700 and k % 2) else 4
    tree = ("fse", 6) if k % 3 else "direct"
    if tree == "direct" and max(data) > 128:
        tree = ("fse", 6)
    for spec in (tree, ("fse", 5), ("fse", 6)):
        try:
            h = Huf(data, max_bits=(9, 10, 11, 8)[k % 4], tree=spec, streams=streams)
            h.section({})
            return h
        except (ValueError, AssertionError):
            continue
    return lits


def family_seams(name):
    """seqfamilies' family `name` with every literals section of two or more distinct bytes re-encoded as Huffman: the
    same output, but the executors now take literals from the literal scratch."""
    orig = F.case
    counter = [0]

    def huf_case(cname, blocks, libzstd="ok", cap=None, **opts):
        out = []
        for b in blocks:
            if isinstance(b, Seqs):
                counter[0] += 1
                b = Seqs(_as_huf(b.literals, counter[0]), b.seqs, b.tables, b.nbseq_form)
            out.append(b)
        try:
            return case("huf-" + cname, out, libzstd, cap, **opts)
        except AssertionError:      # a block grew past 128 KiB: keep the Raw literals of that frame
            return case("raw-" + cname, blocks, libzstd, cap, **opts)
    F.case = huf_case
    try:
        return F.FAMILIES[name]()
    finally:
        F.case = orig


FAMILIES = {
    "tables": family_tables, "streams": family_streams, "treeless": family_treeless, "refonly": family_refonly,
    "invalid": family_invalid, "seam-chunks": lambda: family_seams("chunks"), "seam-repeat": lambda: family_seams("repeat"),
    "seam-flow": lambda: family_seams("flow"),
}

_cache = {}


def cases(name):
    if name not in _cache:
        _cache[name] = FAMILIES[name]()
    return _cache[name]
