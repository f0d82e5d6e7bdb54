"""Huffman literals sections (RFC 8878 3.1.1.3.1 and 4.2) built from explicit codes, as literals specs for seqbuild.Seqs.

`Huf(data, ...)` is a Compressed_Literals section, `Treeless(data, ...)` a Treeless_Literals_Section that reuses the last
tree of the frame; both go where seqbuild.Seqs takes its literals:

    Seqs(Huf(lits, max_bits=9, tree=("fse", 6), streams=4), seqs)

Weights are given per symbol (index = byte value, 0 = not present; the last non-zero one is the implicit weight) or derived
from the histogram of `data` with the code lengths limited to `max_bits`.  The tree description is either direct 4-bit weights
(up to 128 explicit weights) or FSE-compressed weights, two interleaved states chosen backwards over the table the way
seqbuild._Stream chooses sequence states.  Every description is read back through the oracle's Huffman table builder, which
must return exactly the intended weights; the codes come from the table it builds: the code of a symbol is its first table
index >> (max_bits - num_bits).  Codes are written MSB-first in decode order into a backward stream (handmade.rev_stream's
layout), with numpy, so that sections of 2^18 literals build quickly.

`split` gives per-stream symbol counts for 4-stream layouts other than RFC 8878's ceil(regen / 4); `size_format` forces the
literals header form (0: 1 stream, 10-bit sizes; 1 / 2 / 3: 4 streams, 10 / 14 / 18-bit sizes); `regen` overrides the
regenerated size written in the header.  `damage` breaks a built section on purpose, and `expect` is then the oracle status
of the frame:

    ("zero_last", k)      the last byte of stream k becomes 0 (no end marker)
    ("jump", (a, b, c))   the jump table says a, b, c instead of the stream sizes
    ("empty", k)          stream k has no bytes at all
    ("cut", k, n)         the first n bytes of stream k are gone (the bits decoded last)
    ("overread", k, n)    the last n bits of stream k, all of them zero bits of its last code, are dropped: the decoder then
                          reads that code partly from below the stream start, where the reference reads zeros
    ("truncate", n)       the section payload (tree, jump table, streams) is cut to n bytes
    ("tree_zero_last",)   the last byte of an FSE weight description becomes 0
`tree=("raw", bytes)` writes the given tree description as it is (the weight-error cases) and fills the streams with 1-bit
codes that no decoder reaches."""
import ctypes as C
import heapq
from dataclasses import dataclass

import numpy as np

import handmade
import oracle_lib as O
import seqbuild as S

MAX_BITS = 11


# ---------------------------------------------------------------------------
# tables and code lengths
# ---------------------------------------------------------------------------
@dataclass
class HufTable:
    status: int
    max_bits: int
    tree_bytes: int
    weights: list     # as read from the description (explicit weights only)
    symbol: list      # per table cell
    num_bits: list

    def codes(self):
        """{symbol: (code, num_bits)}: a symbol's cells are consecutive, the first one names its code."""
        out = {}
        for i in range(1 << self.max_bits):
            s, nb = self.symbol[i], self.num_bits[i]
            if s not in out:
                out[s] = (i >> (self.max_bits - nb), nb)
        return out


def read_tree(tree: bytes) -> HufTable:
    """The oracle's Huffman table builder on a tree description (huff0_decoder.cairo build_decoder)."""
    L = O.lib()
    sym, nb = (C.c_uint8 * 2048)(), (C.c_uint8 * 2048)()
    mb, used, w, nw = C.c_uint32(), C.c_size_t(), (C.c_uint8 * 260)(), C.c_uint32()
    st = L.oracle_huf_build_decoder(tree, len(tree), 0, sym, nb, C.byref(mb), C.byref(used), w, C.byref(nw))
    size = 1 << mb.value if st == 0 else 0
    return HufTable(st, mb.value if st == 0 else 0, used.value, list(w[:min(nw.value, 258)]), list(sym[:size]), list(nb[:size]))


def complete_lengths(alphabet, max_bits):
    """{symbol: code length} of a complete prefix code over `alphabet` whose longest code has exactly max_bits bits (needs
    max_bits + 1 <= len(alphabet) <= 2^max_bits): a chain 1, 2, .., max_bits, max_bits, then the shortest leaf split in two
    until every symbol has a code.  The lengths go to the symbols in the order given."""
    n = len(alphabet)
    assert 1 <= max_bits <= MAX_BITS and max_bits + 1 <= n <= (1 << max_bits), (n, max_bits)
    lens = list(range(1, max_bits)) + [max_bits, max_bits]
    heap = [l for l in lens if l < max_bits]
    heapq.heapify(heap)
    full = [l for l in lens if l == max_bits]
    while len(heap) + len(full) < n:
        l = heapq.heappop(heap)
        for _ in range(2):
            (heapq.heappush(heap, l + 1) if l + 1 < max_bits else full.append(l + 1))
    lens = sorted(heap) + full
    return dict(zip(alphabet, lens))


def limited_lengths(data, max_bits):
    """{symbol: code length}: Huffman code lengths of the histogram of `data`, limited to max_bits (lengths above the limit
    are clamped, then the least frequent short codes are lengthened until the code fits, then the longest codes shortened
    until it is complete)."""
    hist = np.bincount(np.frombuffer(bytes(data), dtype=np.uint8), minlength=256)
    syms = [s for s in range(256) if hist[s]]
    assert len(syms) >= 2, "a Huffman section needs two symbols"
    assert len(syms) <= (1 << max_bits), (len(syms), max_bits)
    heap = [(int(hist[s]), s, (s,)) for s in syms]
    heapq.heapify(heap)
    depth = dict.fromkeys(syms, 0)
    while len(heap) > 1:
        a, b = heapq.heappop(heap), heapq.heappop(heap)
        for s in a[2] + b[2]:
            depth[s] += 1
        heapq.heappush(heap, (a[0] + b[0], min(a[1], b[1]), a[2] + b[2]))
    lens = {s: min(d, max_bits) for s, d in depth.items()}
    one = 1 << max_bits
    kraft = sum(one >> l for l in lens.values())
    by_rarity = sorted(syms, key=lambda s: (hist[s], s))
    while kraft > one:
        s = next(s for s in by_rarity if lens[s] < max_bits)
        kraft -= one >> (lens[s] + 1)
        lens[s] += 1
    while kraft < one:
        s = max((s for s in syms if lens[s] > 1 and (one >> lens[s]) <= one - kraft), key=lambda s: (lens[s], hist[s]))
        kraft += one >> lens[s]
        lens[s] -= 1
    return lens


def weights_of(lengths):
    """Weights indexed by symbol (0 = not present), from {symbol: code length}; the last entry is the implicit weight."""
    mb = max(lengths.values())
    assert sum(1 << (mb - l) for l in lengths.values()) == 1 << mb, "not a complete prefix code"
    w = [0] * (max(lengths) + 1)
    for s, l in lengths.items():
        w[s] = mb + 1 - l
    return w


# ---------------------------------------------------------------------------
# tree descriptions
# ---------------------------------------------------------------------------
def direct_tree(explicit):
    nw = len(explicit)
    assert 1 <= nw <= 128, nw
    b = bytearray([127 + nw])
    for i in range(0, nw, 2):
        b.append((explicit[i] << 4) | (explicit[i + 1] if i + 1 < nw else 0))
    return bytes(b)


def fse_tree(explicit, log, probs=None):
    """FSE-compressed weights (RFC 8878 4.2.1.2): the normalized counts, then a backward stream with two interleaved states
    that decodes to `explicit`.  The decoder stops when a state update reads past the stream start, and then emits the other
    state's symbol: so the last weight but one must sit in a state that reads at least one bit."""
    n = len(explicit)
    assert n >= 2, "two states give at least two weights"
    if probs is None:
        extra = () if len(set(explicit)) > 1 else ((explicit[0] + 1) % 12,)   # one symbol alone has states of 0 bits only
        probs = S.normalized_counts(explicit, log, extra=extra)
    st = S._Stream(0, ("fse", log, probs), explicit, None)
    table, pick = st.table, st.pick
    chains = [explicit[0::2], explicit[1::2]]
    states, ups = [], []
    for c, chain in enumerate(chains):
        last_reads = (n - 2) % 2 == c      # this chain holds the last weight but one
        row = pick[chain[-1]]
        cand = [s for s in sorted(set(x for x in row if x is not None)) if table[s][1] >= 1 or not last_reads]
        assert cand, "no state of the last weight but one reads a bit"
        sts = [0] * len(chain)
        up = [None] * len(chain)
        sts[-1] = cand[0]
        for i in range(len(chain) - 2, -1, -1):
            s = pick[chain[i]][sts[i + 1]]
            _, nb, base = table[s]
            sts[i] = s
            up[i] = (sts[i + 1] - base, nb)
        states.append(sts)
        ups.append(up)
    bits = []

    def put(v, nb):
        bits.extend((v >> (nb - 1 - k)) & 1 for k in range(nb))
    put(states[0][0], log)
    put(states[1][0], log)
    for k in range(n - 2):                  # the update after weight k moves its chain on to weight k + 2
        put(*ups[k % 2][k // 2])
    body = st.desc + handmade.rev_stream(bits)
    assert len(body) <= 127, f"FSE weight description of {len(body)} bytes"
    return bytes([len(body)]) + body


# ---------------------------------------------------------------------------
# streams
# ---------------------------------------------------------------------------
def pack_codes(values, lengths):
    """Backward stream of the given codes, first decoded first: [1][code 0][code 1]..., MSB-first, little-endian bytes."""
    values = np.asarray(values, dtype=np.int64)
    lengths = np.asarray(lengths, dtype=np.int64)
    total = 1 + int(lengths.sum())
    idx = np.repeat(np.arange(len(lengths)), lengths)
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]]) if len(lengths) else np.zeros(0, np.int64)
    j = np.arange(total - 1) - starts[idx]
    bits = np.concatenate([[1], (values[idx] >> (lengths[idx] - 1 - j)) & 1]).astype(np.uint8)
    pad = (-total) % 8
    return np.packbits(np.concatenate([np.zeros(pad, np.uint8), bits]))[::-1].tobytes()


def _lit_header(ltype, sf, regen, comp):
    if sf <= 1:
        assert regen < 1024 and comp < 1024, (regen, comp)
        return (ltype | (sf << 2) | (regen << 4) | (comp << 14)).to_bytes(3, "little")
    if sf == 2:
        assert regen < 16384 and comp < 16384, (regen, comp)
        return (ltype | (sf << 2) | (regen << 4) | (comp << 18)).to_bytes(4, "little")
    assert regen < (1 << 18) and comp < (1 << 18), (regen, comp)
    return (ltype | (sf << 2) | (regen << 4) | (comp << 22)).to_bytes(5, "little")


def rfc_split(regen):
    seg = (regen + 3) // 4
    return [max(0, min(seg, regen - k * seg)) for k in range(4)]


@dataclass
class Huf:
    data: bytes
    weights: list = None
    max_bits: int = None
    tree: object = "direct"
    streams: int = 1
    split: list = None
    size_format: int = None
    regen: int = None
    damage: tuple = None
    expect: str = None

    def __post_init__(self):
        self.data = bytes(self.data)
        self.derived = self.weights is None and self.tree is not None and not (isinstance(self.tree, tuple) and self.tree[0] == "raw")
        if self.derived:    # max_bits is then a limit, not the exact table size
            self.weights = weights_of(limited_lengths(self.data, self.max_bits or MAX_BITS))
        assert self.streams in (1, 4)

    def tree_bytes(self):
        nz = [s for s, w in enumerate(self.weights) if w]
        explicit = list(self.weights[:nz[-1]])
        if self.tree == "direct":
            t = direct_tree(explicit)
        else:
            assert self.tree[0] == "fse", self.tree
            t = fse_tree(explicit, self.tree[1], self.tree[2] if len(self.tree) > 2 else None)
        got = read_tree(t)
        if got.status or got.weights != explicit or got.tree_bytes != len(t):
            raise ValueError(f"tree description reads back as status {got.status}, {got.weights[:8]}.. ({len(got.weights)} weights)")
        if self.max_bits is not None and (got.max_bits > self.max_bits or (not self.derived and got.max_bits != self.max_bits)):
            raise ValueError(f"max_bits {got.max_bits}, not {self.max_bits}")
        return t, got

    def section(self, state):
        """The literals section's bytes (header included); records the tree in `state` and the layout in self.info."""
        ltype = 3 if self.tree is None else 2
        if ltype == 3:
            tree = b""
            codes, mb = state.get("tree") or self._fallback()
        elif isinstance(self.tree, tuple) and self.tree[0] == "raw":
            tree, codes, mb = bytes(self.tree[1]), {0: (0, 1), 1: (1, 1)}, 1
        else:
            tree, table = self.tree_bytes()
            codes, mb = table.codes(), table.max_bits
            state["tree"] = (codes, mb)
        data = self.data if not isinstance(self.tree, tuple) or self.tree[0] != "raw" else bytes(b & 1 for b in self.data)
        regen = len(data) if self.regen is None else self.regen
        if self.streams == 1:
            counts = [len(data)]
        else:
            counts = list(self.split) if self.split is not None else rfc_split(len(data))
        assert sum(counts) == len(data) and len(counts) == self.streams, (counts, len(data))
        sym = np.frombuffer(data, dtype=np.uint8)
        cv = np.zeros(256, np.int64); cl = np.zeros(256, np.int64)
        for s, (v, nb) in codes.items():
            cv[s], cl[s] = v, nb
        assert all(cl[s] for s in set(data)), "a symbol without a code"
        streams, lens, pos = [], [], 0
        for n in counts:
            part = sym[pos:pos + n]; pos += n
            lens.append(cl[part])
            streams.append(bytearray(pack_codes(cv[part], cl[part])))
        jump = None
        dmg = self.damage or ()
        kind = dmg[0] if dmg else None
        if kind == "zero_last":
            streams[dmg[1]][-1] = 0
        elif kind == "empty":
            streams[dmg[1]] = bytearray()
        elif kind == "cut":
            streams[dmg[1]] = streams[dmg[1]][dmg[2]:]
        elif kind == "overread":
            k, nbits = dmg[1], dmg[2]
            x = int.from_bytes(streams[k], "little")
            last_v, last_n = int(cv[sym[sum(counts[:k + 1]) - 1]]), int(lens[k][-1])
            assert nbits <= last_n and last_v & ((1 << nbits) - 1) == 0, "only zero bits of the last code may go"
            x >>= nbits
            streams[k] = bytearray(x.to_bytes((x.bit_length() + 7) // 8, "little"))
        elif kind == "jump":
            jump = dmg[1]
        if self.streams == 4:
            jump = jump or [len(s) for s in streams[:3]]
            body = bytes(tree) + b"".join(x.to_bytes(2, "little") for x in jump) + b"".join(bytes(s) for s in streams)
        else:
            body = bytes(tree) + bytes(streams[0])
        if kind == "truncate":
            body = body[:dmg[1]]
        elif kind == "tree_zero_last":
            body = body[:len(tree) - 1] + b"\x00" + body[len(tree):]
        comp = len(body)
        sf = self.size_format
        if sf is None:
            sf = 0 if self.streams == 1 else 1 if max(regen, comp) < 1024 else 2 if max(regen, comp) < 16384 else 3
        self.info = dict(ltype=ltype, sf=sf, regen=regen, streams=self.streams, counts=counts, lens=lens, max_bits=mb,
                         bits=[int(l.sum()) for l in lens])
        return _lit_header(ltype, sf, regen, comp) + body

    def _fallback(self):
        t = read_tree(direct_tree(self.weights[:max(s for s, w in enumerate(self.weights) if w)]))
        return t.codes(), t.max_bits


class Treeless(Huf):
    """Treeless_Literals_Section: the streams are coded with the frame's last tree.  `weights` only serve when the frame has
    no tree yet (the section must then fail, but its streams are still real codes of that table)."""

    def __init__(self, data, streams=1, split=None, size_format=None, weights=None, regen=None, damage=None, expect=None):
        super().__init__(data, weights=weights, tree=None, streams=streams, split=split, size_format=size_format, regen=regen,
                         damage=damage, expect=expect)


# ---------------------------------------------------------------------------
# reference
# ---------------------------------------------------------------------------
def reference_decode(blocks, window=None):
    """seqbuild.reference_decode with the literals stage in front: a damaged section gives its declared status, a Treeless
    section before any Huffman tree of the frame gives CZS_UNINITIALIZED_HUFFMAN_TABLE.  Errors come in block order."""
    have_tree = False
    for i, b in enumerate(blocks):
        lits = getattr(b, "literals", None)
        if not isinstance(lits, Huf):
            continue
        err = lits.expect
        if err is None and lits.tree is None and not have_tree:
            err = "CZS_UNINITIALIZED_HUFFMAN_TABLE"
        if err is not None:
            before = S.reference_decode(blocks[:i], window)
            return before if isinstance(before, str) else err
        have_tree = have_tree or lits.tree is not None
    return S.reference_decode(blocks, window)


def kernel_walk(info, dst_base=0):
    """What k_huff's decode loop does with each stream of a built section (its head, 16-literal, 4-literal and per-literal
    loops): per stream the head length, the (loop, bits remaining, taken) checks where a loop's bit threshold decided, and the
    number of 4-literal groups of more than 32 bits.  dst_base: the section's literal scratch offset (16-byte aligned)."""
    out = []
    regen = info["regen"]
    seg = (regen + 3) // 4
    for k in range(info["streams"]):
        if info["streams"] == 4:
            start = k * seg
            expect = 0 if start >= regen else min(seg, regen - start)
        else:
            start, expect = 0, regen
        lens = [int(x) for x in info["lens"][k]]
        rem, n, i = info["bits"][k], 0, 0
        head = (-(dst_base + start)) % 16
        checks, wide = [], 0

        def take(c):
            nonlocal rem, n, i
            rem -= sum(lens[i:i + c]); n += c; i += c
        while rem > 0 and n < head and i < len(lens):
            take(1)
        while True:
            ok_n = n + 16 <= expect
            if ok_n and rem in (175, 176, 177):
                checks.append((16, rem, rem >= 176))
            if not (rem >= 176 and ok_n):
                break
            wide += sum(1 for g in range(4) if sum(lens[i + 4 * g:i + 4 * g + 4]) > 32)
            take(16)
        while True:
            ok_n = n + 4 <= expect
            if ok_n and rem in (43, 44, 45):
                checks.append((4, rem, rem >= 44))
            if not (rem >= 44 and ok_n):
                break
            wide += sum(lens[i:i + 4]) > 32
            take(4)
        out.append(dict(head=head, expect=expect, checks=checks, wide=wide))
    return out
