"""The Huffman literals builder (tests/hufbuild.py) against two decoders: every frame of tests/huffamilies.py must decode to
hufbuild.reference_decode's output in the oracle (status 0, the whole frame read, the checksum matching) and, where flagged,
in libzstd; frames that are invalid by construction must fail with their declared oracle status.  Also: FSE weight
descriptions read back as the intended weights, and the families really reach k_huff's seams (checked on the built
sections, through a model of k_huff's decode loop)."""
import random

import numpy as np
import pytest

import hufbuild as H
import huffamilies as HF
import oracle_lib as O
import cairo_zstd_b200 as czb
from cairo_zstd_b200 import workloads as W


@pytest.mark.parametrize("family", sorted(HF.FAMILIES))
def test_family_frames_decode_to_the_reference_in_the_oracle_and_libzstd(family):
    cases = HF.cases(family)
    assert cases
    for c in cases:
        st, out, r = O.decode_frame(c.frame, dst_cap=c.cap)
        if isinstance(c.expected, bytes):
            assert st == 0, (c.name, czb.status_name(st))
            assert out == c.expected, c.name
            assert r.bytes_read == len(c.frame), c.name
            assert r.has_checksum and r.checksum_calculated == r.checksum_from_data, c.name
        else:
            assert czb.status_name(st) == c.expected, (c.name, czb.status_name(st))
        if c.libzstd == "ok":
            assert W.libzstd_decompress(c.frame, c.cap) == c.expected, c.name
        elif c.libzstd == "reject":
            with pytest.raises(RuntimeError):
                W.libzstd_decompress(c.frame, c.cap)


def test_fse_weight_descriptions_read_back_as_the_intended_weights():
    rng = random.Random(31)
    for _ in range(300):
        nw = rng.randrange(2, 256)
        top = rng.randrange(1, 12)
        explicit = [rng.choice([0, 0, 1, top, rng.randrange(12)]) for _ in range(nw)]
        log = rng.choice([5, 6, 7, 9, 10])
        try:
            t = H.fse_tree(explicit, log)
        except AssertionError:     # longer than the 127 bytes a description may have, or more weight symbols than cells
            continue
        got = H.read_tree(t)
        assert got.tree_bytes == len(t) and got.weights[:nw] == explicit, (explicit, log)
    # and every FSE description the families use
    n = 0
    for fam in HF.FAMILIES:
        for c in HF.cases(fam):
            for b in c.blocks:
                h = getattr(b, "literals", None)
                if isinstance(h, H.Huf) and isinstance(h.tree, tuple) and h.tree[0] == "fse":
                    t, table = h.tree_bytes()
                    assert H.read_tree(t).weights == table.weights
                    n += 1
    assert n > 100


def test_complete_lengths_and_limited_lengths_give_complete_codes():
    rng = np.random.default_rng(32)
    for L in range(1, 12):
        for n in sorted({L + 1, min(1 << L, 256), min(1 << L, L + 7)}):
            lens = H.complete_lengths(list(range(n)), L)
            assert max(lens.values()) == L and sum(2.0 ** -l for l in lens.values()) == 1.0
        data = rng.geometric(0.3, 5000).clip(0, 255).astype(np.uint8).tobytes()
        if len(set(data)) <= (1 << L):
            lens = H.limited_lengths(data, L)
            assert max(lens.values()) <= L and sum(2.0 ** -l for l in lens.values()) == 1.0


def _sections():
    """(case, block index, Huf spec, oracle trace of the block) for every Huffman section of every valid frame."""
    out = []
    for fam in HF.FAMILIES:
        for c in HF.cases(fam):
            if not isinstance(c.expected, bytes):
                continue
            st, _, _, trace = O.decode_frame(c.frame, dst_cap=c.cap, trace=True)
            assert st == 0
            for i, (b, t) in enumerate(zip(c.blocks, trace)):
                h = getattr(b, "literals", None)
                if isinstance(h, H.Huf):
                    assert t["lit_type"] == h.info["ltype"] and t["n_streams"] == h.streams and t["regen_size"] == h.info["regen"]
                    out.append((c, i, h, t))
    return out


def test_families_reach_the_seams_of_k_huff():
    secs = _sections()
    classes, heads, checks, forms = set(), set(), set(), set()
    wide = 0
    non_rfc = 0
    for c, i, h, t in secs:
        classes.add(h.info["max_bits"])
        forms.add(h.info["sf"])
        if h.streams == 4 and h.info["counts"] != H.rfc_split(t["regen_size"]):
            non_rfc += 1
        for k, s in enumerate(H.kernel_walk(h.info)):
            if k >= 1 and s["expect"]:
                heads.add(s["head"])
            checks.update(s["checks"])
            wide += s["wide"]
    assert {9, 10} <= classes and classes == set(range(1, 12)), classes          # both k_huff table classes, every max_bits
    assert heads == set(range(16)), sorted(heads)                                  # streams 1..3: every head length
    for loop, at in ((16, 176), (4, 44)):                                          # each loop's bit threshold, both ways
        assert (loop, at, True) in checks and (loop, at - 1, False) in checks, (loop, sorted(checks))
    assert wide > 1000                                                             # 4-literal groups of more than 32 bits
    assert forms == {0, 1, 2, 3}                                                   # all four literals header forms
    assert non_rfc >= 5                                                            # 4-stream splits other than RFC 8878's
    # a Treeless section whose nearest earlier literals section is a Raw / RLE one
    after_plain = 0
    for fam in HF.FAMILIES:
        for c in HF.cases(fam):
            last = None
            for b in c.blocks:
                lits = getattr(b, "literals", None)
                if lits is None:
                    continue
                if isinstance(lits, H.Treeless) and last == "plain" and isinstance(c.expected, bytes):
                    after_plain += 1
                last = "huf" if isinstance(lits, H.Huf) else "plain"
    assert after_plain >= 1


def test_overread_keeps_the_output_and_the_cut_lands_on_a_code_boundary():
    c = next(c for c in HF.cases("refonly") if c.name == "overread-1s-10")
    h = c.blocks[0].literals
    assert h.damage == ("overread", 0, 10) and c.expected == h.data     # 10 of the last code's 11 bits lie below the stream
    c = next(c for c in HF.cases("invalid") if c.name == "bad-cut-stream1")
    h = c.blocks[0].literals
    lens = [int(x) for x in h.info["lens"][1]]
    cut_bits = 24
    assert cut_bits in np.cumsum(lens[::-1]).tolist()                   # the 24 bits decoded last are whole codes
