"""-m gpu: the field-by-field sequence sections of tests/fsefamilies.py on the device.  Every family is decoded in one batch
per executor mode against the oracle and the reference executor; k_fse's own output (block statuses and the sequence records
of the last wave) is compared with the sequences the builder wrote, so that a wrong table cell, a wrong state step or a
mix-up between the lean and the exact loop shows even where the frame fails later; the execution-free sizes and the verify
call agree with the decode; guard zones behind the scratch stay intact."""
import ctypes as C

import pytest

import fsefamilies as X
import gpu_common as G
import oracle_lib as O
import cairo_zstd_b200 as czb
from test_gpu_seams import MODES, _context, _watchdog_clear
from test_gpu_verify import verify_and_decode

pytestmark = pytest.mark.gpu
OFF29_CLAMP = (1 << 28) - 1


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("family", sorted(X.FAMILIES))
def test_fse_families_match_reference_and_oracle(monkeypatch, family, mode):
    cases = X.cases(family)
    ctx = _context(monkeypatch, mode)
    outs, res = G.compare_with_oracle([c.frame for c in cases], [c.cap for c in cases], label=f"{family}/{mode}")
    for c, o, r in zip(cases, outs, res):
        if isinstance(c.expected, bytes):
            assert o == c.expected, c.name
            assert r.checksum_calculated == r.checksum_from_data, c.name
        else:
            assert czb.status_name(r.status) == c.expected, (c.name, czb.status_name(r.status))
    if mode != "default":
        _watchdog_clear()
    ctx.close()


def _resolve(h, ll, v):
    """do_offset_history: the offset of value v after ll literals, and the new history."""
    if v > 3:
        return v - 3, [v - 3, h[0], h[1]]
    if ll > 0:
        o = h[v - 1]
        return o, (h if v == 1 else [o, h[0], h[2]] if v == 2 else [o, h[0], h[1]])
    o = h[1] if v == 1 else h[2] if v == 2 else (h[0] - 1) & 0xFFFFFFFF
    return o, ([o, h[0], h[2]] if v == 1 else [o, h[0], h[1]])


@pytest.mark.parametrize("family", sorted(X.FAMILIES))
def test_k_fse_records_equal_the_built_sequences(monkeypatch, family):
    """One wave: every compressed block up to the frame's failing one has stage status OK and records (ll, ml) equal to the
    builder's sequences, offsets equal to the resolved ones where the record is not symbolic (a block that is not first
    in its frame refers to the history before it symbolically; a plain offset never does); the failing block has its
    status."""
    cases = X.cases(family)
    ctx = _context(monkeypatch, "default")
    G.gpu_decode([c.frame for c in cases], [c.cap for c in cases])
    blocks, _, recs = ctx.debug_last_wave()
    per_frame = {}
    for b in blocks:
        per_frame.setdefault(b.frame, []).append(b)
    assert len(per_frame) == len(cases)
    checked = 0
    for i, c in enumerate(cases):
        dbg = per_frame[i]
        hist = [1, 4, 8]
        for j, blk in enumerate(c.blocks):
            if j == c.fail_block:
                assert czb.status_name(dbg[j].status) == blk.status, (c.name, j, czb.status_name(dbg[j].status))
                break
            if blk.body is None:
                continue
            d = dbg[j]
            assert d.block_type == 2 and d.status == 0, (c.name, j, czb.status_name(d.status))
            seqs = blk.spec.seqs
            assert d.n_seq == len(seqs), (c.name, j, d.n_seq, len(seqs))
            for k, (ll, ml, v) in enumerate(seqs):
                r = recs[3 * (d.seq_off + k):3 * (d.seq_off + k) + 3]
                assert (r[0], r[1]) == (ll, ml), (c.name, j, k, r, (ll, ml, v))
                o, hist = _resolve(hist, ll, v)
                symbolic = r[2] >> 28 == 0xF
                assert not (symbolic and v > 3), (c.name, j, k, hex(r[2]), v)
                if not symbolic:
                    assert r[2] == min(o, OFF29_CLAMP), (c.name, j, k, r[2], o, v)
                checked += 1
    assert checked > 0
    ctx.close()


@pytest.mark.parametrize("family", sorted(X.FAMILIES))
def test_execution_free_sizes(family):
    """czb_frame_sizes: a valid frame's decoded size; a sequence-stage failure's status; a frame that fails only in execution
    (offsets beyond the output) OK and the regenerated sizes plus the match lengths."""
    cases = X.cases(family)
    res = G.ctx().frame_sizes([c.frame for c in cases])
    for c, r in zip(cases, res):
        if c.fail_block is not None:
            assert czb.status_name(r.status) == c.expected, (c.name, czb.status_name(r.status))
            continue
        assert r.status == 0, (c.name, czb.status_name(r.status))
        assert r.bytes_written == sum(X.block_output(b) for b in c.blocks), c.name
        if isinstance(c.expected, bytes):
            assert r.bytes_written == len(c.expected), c.name


def _big(c):
    return any(X.block_output(b) > X.BIG for b in c.blocks if b.body is not None)


@pytest.mark.parametrize("family", sorted(X.FAMILIES))
def test_verify_equals_decode(monkeypatch, family):
    """czb_verify_batch_device reports every field as the decode call does; a frame with a block regenerating more than
    128 KiB may instead be CZS_UNSUPPORTED when its wave's output scratch cannot hold it (cairo_zstd_b200.h, rule c)."""
    cases = X.cases(family)
    ctx = _context(monkeypatch, "default")
    small = [c for c in cases if not _big(c)]
    verify_and_decode(ctx, [c.frame for c in small],
                      [(len(c.expected) if isinstance(c.expected, bytes) else c.cap) + 4096 for c in small])
    big = [c for c in cases if _big(c)]
    if big:
        got = verify_and_decode(ctx, [c.frame for c in big], [0] * len(big), decode=False)
        for c, r in zip(big, got):
            st = czb.status_name(r.status)
            want = "CZS_OK" if isinstance(c.expected, bytes) else c.expected
            assert st in (want, "CZS_UNSUPPORTED"), (c.name, st)
            if st == "CZS_OK":
                assert r.bytes_written == len(c.expected) and r.checksum_calculated == r.checksum_from_data, c.name
    ctx.close()


def test_guard_zones_stay_intact(monkeypatch):
    """CZB_GUARD=1 over every family in one batch: nothing is written behind the used part of the literal, sequence and
    block scratch (the NSEQ_MAX-record blocks size the sequence scratch exactly)."""
    monkeypatch.setenv("CZB_GUARD", "1")
    cases = [c for f in sorted(X.FAMILIES) for c in X.cases(f)]
    ctx = _context(monkeypatch, "default")
    G.compare_with_oracle([c.frame for c in cases], [c.cap for c in cases], label="guard")
    assert ctx.guard_faults() == 0
    ctx.close()
