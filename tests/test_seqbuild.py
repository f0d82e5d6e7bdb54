"""The sequence-driven frame builder (tests/seqbuild.py) against two decoders: every frame of every family in
tests/seqfamilies.py must decode to reference_decode's output in libzstd and in the oracle (status 0, the whole frame read,
the checksum matching), and the frames that are invalid by construction must fail with the oracle status named by the
reference executor.  The builder takes its FSE decoding tables from the oracle; libzstd is the independent check."""
import pytest

import oracle_lib as O
import seqbuild as S
import seqfamilies as F
import cairo_zstd_b200 as czb
from cairo_zstd_b200 import workloads as W


def test_code_tables_follow_rfc_8878():
    assert S.LL_BASE[16:26] == [16, 18, 20, 22, 24, 28, 32, 40, 48, 64] and S.LL_BASE[35] == 65536
    assert S.ML_BASE[32:44] == [35, 37, 39, 41, 43, 47, 51, 59, 67, 83, 99, 131] and S.ML_BASE[52] == 65539
    for ll in list(range(300)) + [65535, 65536, 131071]:
        c = S.ll_code(ll)
        assert S.LL_BASE[c] <= ll < S.LL_BASE[c] + (1 << S.LL_BITS[c])
    for ml in list(range(3, 300)) + [65538, 65539, 131074]:
        c = S.ml_code(ml)
        assert S.ML_BASE[c] <= ml < S.ML_BASE[c] + (1 << S.ML_BITS[c])


def test_reference_decode_offset_history():
    pre = bytes(range(100))
    # ll > 0: repeat 1 keeps the history; ll = 0: repeat 1 is h1, repeat 3 is h0 - 1
    out = S.reference_decode([S.Raw(pre), S.Seqs(b"ab", [(1, 3, S.rep(1)), (0, 3, S.rep(1)), (0, 3, S.rep(3)), (1, 3, S.rep(3))])])
    want = bytearray(pre)
    for ll_lit, o in ((b"a", 1), (b"", 4), (b"", 3), (b"b", 1)):
        want += ll_lit
        for _ in range(3):
            want.append(want[-o])
    assert out == bytes(want)
    assert S.reference_decode([S.Raw(pre), S.Seqs(b"", [(0, 3, S.rep(3))])]) == "CZS_EXEC_ZERO_OFFSET"


@pytest.mark.parametrize("family", sorted(F.FAMILIES))
def test_family_frames_decode_to_the_reference_in_libzstd_and_the_oracle(family):
    cases = F.cases(family)
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


def test_risky_table_frame_equals_its_plain_twin():
    risky, plain = F.risky_pair()
    assert risky.expected == plain.expected
    assert O.decode_frame(risky.frame, dst_cap=risky.cap)[1] == O.decode_frame(plain.frame, dst_cap=plain.cap)[1] == plain.expected


def test_nbseq_header_forms():
    seqs = [(1, 3, S.off(1))] * 127
    lits = b"x" * 127
    for form in (1, 2):
        blk, _ = S.encode_seqs_block(S.Seqs(lits, seqs, nbseq_form=form), None)
        hdr = blk[len(S._lit_header(0, 127)) + 127:]
        assert (hdr[0] == 127) if form == 1 else (hdr[0] == 128 and hdr[1] == 127)
    blk, _ = S.encode_seqs_block(S.Seqs(b"", [(0, 3, S.off(1))] * 0x7F00), None)
    assert blk[1:4] == b"\xff\x00\x00"
