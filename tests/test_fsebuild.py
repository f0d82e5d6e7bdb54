"""The field-by-field sequence sections of tests/fsefamilies.py against the oracle and libzstd: valid frames decode to the
reference executor's output (libzstd too where its block limit allows), every malformed frame fails with the sequence-stage
status it was built for, every description reads back to the table its counts give and uses exactly its bytes, and every
cell of every FSE table of a desc frame is the state of a decoded sequence."""
import ctypes as C

import pytest

import fsefamilies as X
import oracle_lib as O
import seqbuild as S
import cairo_zstd_b200 as czb
from cairo_zstd_b200 import workloads as W

# the statuses of the sequence stage, each of which some case must be built to raise
SEQ_STATUSES = {"CZS_PANIC_INTERNAL", "CZS_SEQ_NOT_ENOUGH_BYTES_FOR_NUM_SEQUENCES", "CZS_SEQ_EXTRA_BITS", "CZS_SEQ_EXTRA_PADDING",
                "CZS_SEQ_UNSUPPORTED_OFFSET", "CZS_FSE_TABLE_IS_UNINITIALIZED", "CZS_FSE_ACC_LOG_TOO_BIG", "CZS_FSE_GET_BITS_ERROR",
                "CZS_SEQ_HDR_NOT_ENOUGH_BYTES", "CZS_MISSING_BYTE_FOR_RLE_LL_TABLE", "CZS_MISSING_BYTE_FOR_RLE_OF_TABLE",
                "CZS_MISSING_BYTE_FOR_RLE_ML_TABLE", "CZS_FSE_TOO_MANY_SYMBOLS", "CZS_SEQ_GET_BITS_ERROR"}


@pytest.mark.parametrize("family", sorted(X.FAMILIES))
def test_fse_family_frames_against_the_oracle_and_libzstd(family):
    cases = X.cases(family)
    assert cases
    for c in cases:
        st, out, r = O.decode_frame(c.frame, dst_cap=c.cap)
        if isinstance(c.expected, bytes):
            assert st == 0, (c.name, czb.status_name(st))
            assert out == c.expected and r.bytes_read == len(c.frame), c.name
            assert r.checksum_calculated == r.checksum_from_data, c.name
        else:
            assert czb.status_name(st) == c.expected, (c.name, czb.status_name(st))
            if c.fail_block is not None:     # the blocks before the failing one decoded
                assert r.blocks_decoded == c.fail_block, (c.name, r.blocks_decoded)
        if c.libzstd == "ok":
            assert W.libzstd_decompress(c.frame, c.cap) == c.expected, c.name
        elif c.libzstd == "reject":
            with pytest.raises(RuntimeError):
                W.libzstd_decompress(c.frame, c.cap)


def test_every_sequence_stage_status_is_built():
    built = {c.expected for f in X.FAMILIES for c in X.cases(f) if c.fail_block is not None}
    assert SEQ_STATUSES <= built, SEQ_STATUSES - built
    names = {c.name for f in X.FAMILIES for c in X.cases(f)}
    for n in ("invalid-bad-code-then-short", "invalid-short-then-bad-code", "quirk-nseq0-trailing-bytes", "quirk-reserved-modes-bits",
              "counts-98047-rle0", "counts-98047-fse0", "counts-98047-bits", "cta-55-fail"):
        assert n in names, n


def _read_back(desc, log, kind):
    L = O.lib()
    n = 1 << 12
    bl = (C.c_uint32 * n)(); nb = (C.c_uint8 * n)(); sym = (C.c_uint8 * n)()
    size, used = C.c_uint32(), C.c_size_t()
    st = L.oracle_fse_build_decoder(desc + b"\xa5" * 8, len(desc) + 8, S.MAX_LOG[kind], bl, nb, sym, C.byref(size), C.byref(used))
    assert st == 0, czb.status_name(st)
    return [(sym[i], nb[i], bl[i]) for i in range(size.value)], used.value


def test_descriptions_read_back_to_their_tables():
    seen = 0
    for f in X.FAMILIES:
        for c in X.cases(f):
            for b in c.blocks:
                for k, st in enumerate(b.streams or ()):
                    if st.mode != 2 or b.status:
                        continue
                    kind, log, probs = st.key
                    table, used = _read_back(st.desc, log, kind)
                    assert used == len(st.desc), (c.name, k, used, len(st.desc))
                    assert table == S.decoding_table(kind, log, list(probs)), (c.name, k)
                    seen += 1
    assert seen > 500


def test_noncanonical_descriptions():
    d = X.describe(6, [61, 0, 0, 1, 0, 1, 1], explicit_zero=(2, 4))
    assert d != X.describe(6, [61, 0, 0, 1, 0, 1, 1])
    assert _read_back(d, 6, 0) == (S.decoding_table(0, 6, [61, 0, 0, 1, 0, 1, 1]), len(d))
    p = X.describe(6, [59, 2, 0, 1, 1, -1], pad=0xFF)
    assert p[:-1] == X.describe(6, [59, 2, 0, 1, 1, -1])[:-1] and p[-1] != X.describe(6, [59, 2, 0, 1, 1, -1])[-1]


def test_every_cell_of_every_table_is_decoded():
    """The walks are what the decoder goes through: the oracle's sequences (trace) have the walks' codes; and the walks of
    a desc frame visit every cell of its FSE tables."""
    for c in X.cases("desc"):
        assert not any(X.coverage(c).values()), (c.name, {k[:2]: len(v) for k, v in X.coverage(c).items() if v})
        _, _, _, trace = O.decode_frame(c.frame, dst_cap=c.cap, trace=True)
        comp = [b for b in c.blocks if b.body is not None]
        tr = [t for t in trace if t["block_type"] == 2]
        assert len(tr) == len(comp), c.name
        for b, t in zip(comp, tr):
            assert [tuple(s[:3]) for s in t["seqs"]] == b.spec.seqs, c.name
            for k, (st, w) in enumerate(zip(b.streams, b.walks)):
                if w is not None:
                    codes = [S.ll_code(s[0]) if k == 0 else S.of_code(s[2]) if k == 1 else S.ml_code(s[1]) for s in b.spec.seqs]
                    assert [st.table[x][0] for x in w] == codes, (c.name, k)
