"""The FrameDecoder scripts of tests/fdscript.py on the oracle alone (no GPU): every script of every family frame drains the
frame's expected output, or fails with the frame's expected status, and the seams scripts put a span end on every block end.
The -m gpu tests in test_gpu_handle.py run the same scripts on the handle and the oracle side by side."""
import ctypes as C
import random

import pytest

import fdscript as D
import oracle_lib as O
import seqfamilies as F
import cairo_zstd_b200 as czb

FAMILIES = D.family_names()
family_cases, expected_output, check, sample = D.family_cases, D.expected_output, D.check, D.sample


def test_seqfamilies_have_the_resume_family():
    names = [c.name for c in F.cases("resume")]
    assert len([n for n in names if n.startswith("resume-first-seq-r")]) == 16
    assert "resume-late-block-over-128k" in names


@pytest.mark.parametrize("kind,name", FAMILIES)
def test_seams_scripts_on_the_oracle(kind, name):
    for c in family_cases(kind, name):
        lay = D.layout(c.frame)
        script = D.seams(lay)
        ends = [s[1] for s in script if s[0] == "blocks" and s[1] is not None]
        want = [b.end + (4 if b.last and lay.checksum else 0) for b in lay.blocks]
        assert ends == want, c.name
        if expected_output(c) is not None:      # the seams cover the whole frame: every block end, then the trailer
            assert ends[-1] == len(c.frame) and lay.blocks[-1].last, c.name
            assert all(lay.blocks[k].end == lay.blocks[k + 1].start for k in range(len(lay.blocks) - 1)), c.name
        res = D.run(c.frame, script, label=c.name, oracle_only=True)
        check(c, "seams", res.epochs[0])


@pytest.mark.parametrize("kind,name", FAMILIES)
def test_ragged_chunked_shrink_scripts_on_the_oracle(kind, name):
    cases = family_cases(kind, name)
    for k, c in enumerate(sample(cases)):
        lay = D.layout(c.frame)
        for sname, script in D.scripts(lay, seed=k):
            if sname == "chunked1" and len(c.frame) > 40000:
                continue
            res = D.run(c.frame, script, label=f"{c.name}/{sname}", oracle_only=True)
            check(c, sname, res.epochs[0])


def test_reset_script_on_the_oracle():
    a, b = F.cases("resume")[0], F.cases("repeat")[3]
    lay = D.layout(a.frame)
    res = D.run([a.frame, b.frame], D.reset(lay), label="reset", oracle_only=True)
    assert [e.frame for e in res.epochs] == [0, 1, 0]
    assert bytes(res.epochs[1].drained) == b.expected and bytes(res.epochs[2].drained) == a.expected


def test_scripts_on_corpus_and_libzstd_frames(corpus):
    for name in D.CORPUS:
        i = next(k for k, e in enumerate(corpus.index) if e["name"] == name)
        f = corpus.frame(i)
        want = O.decode_frame(f, dst_cap=corpus.index[i]["orig_len"] + 64)[1]
        lay = D.layout(f)
        for sname, script in D.scripts(lay, seed=i):
            if sname == "chunked1" and name == "z000033":
                continue
            ep = D.run(f, script, label=f"{name}/{sname}", oracle_only=True).epochs[0]
            check(F.Case(name, f, want, len(want)), sname, ep)
    for wl, (f, data) in D.libzstd_frames().items():
        lay = D.layout(f)
        assert len(lay.blocks) >= 3, wl
        for sname, script in D.scripts(lay, seed=wl):
            if sname == "chunked1":
                continue
            ep = D.run(f, script, label=f"wl{wl}/{sname}", oracle_only=True).epochs[0]
            check(F.Case(f"wl{wl}", f, data, len(data)), sname, ep)


def test_ragged_scripts_cover_every_kind_of_span_end():
    """Over the resume family, the ragged scripts end spans inside headers, inside bodies, on block ends and inside the
    checksum trailer, and use every strategy form."""
    seen, strat = set(), set()
    for k, c in enumerate(F.cases("resume")):
        lay = D.layout(c.frame)
        starts = {b.start for b in lay.blocks}
        ends = {b.end for b in lay.blocks}
        last = lay.blocks[-1]
        rng = random.Random(k)
        for call in D.ragged(lay, rng):
            if call[0] != "blocks":
                continue
            e = call[1]
            outs = {b.out for b in lay.blocks}
            strat.add((call[2], call[3] if call[2] == D.UPTO_BLOCKS or call[3] <= 1 else "out" if call[3] in outs else "out-1"))
            if e in ends:
                seen.add("end")
            elif e - 1 in starts or e - 2 in starts:
                seen.add("header")
            elif last.end < e < last.end + 4:
                seen.add("trailer")
            else:
                seen.add("body")
    assert seen == {"end", "header", "body", "trailer"}, seen
    assert {(D.UPTO_BLOCKS, 1), (D.UPTO_BLOCKS, 2), (D.UPTO_BLOCKS, 3), (D.UPTO_BYTES, 1), (D.UPTO_BYTES, "out"),
            (D.UPTO_BYTES, "out-1")} <= strat, strat


def test_oracle_fails_truncated_and_bad_blocks_the_reference_way():
    """What a failing decode_blocks call consumes in the oracle (block_decoder.cairo via read_block_header, which advances
    before it checks, and decompress_block, which slices the content off before it parses): 3 bytes for a header error or a
    truncated body, 3 + Block_Size for a compressed block whose body fails; bytes_read_from_source counts nothing for a
    header error and 3 for a block whose body fails."""
    L = O.lib()
    for frame, span_end, want_status, want_consumed, want_counted in D.failing_frames():
        used, st = C.c_size_t(), C.c_int32()
        fd = L.oracle_fd_new(frame, len(frame), C.byref(used), 0, C.byref(st))
        pos = used.value
        cons, fin = C.c_size_t(), C.c_int32()
        s = L.oracle_fd_decode_blocks(fd, frame[pos:span_end], span_end - pos, C.byref(cons), D.ALL, 0, C.byref(fin))
        r = O.OracleResult()
        L.oracle_fd_getters(fd, C.byref(r))
        L.oracle_fd_free(fd)
        assert czb.status_name(s) == want_status, (want_status, czb.status_name(s))
        assert cons.value == D.RAW0 + want_consumed, (want_status, cons.value)      # after the Raw block in front
        assert r.bytes_read == pos + D.RAW0 + want_counted, want_status
