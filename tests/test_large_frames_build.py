"""CPU: the frames of tests/largeframes.py that test_gpu_large_frames.py decodes.  Valid ones round-trip through libzstd and
the oracle; invalid ones fail in the oracle with the expected status (a far offset beyond the output: the reference's
offset errors).  Also: the Python mirror of CZB_MAX_FRAME_OUTPUT equals the header's."""
import os
import re

import numpy as np
import pytest

import largeframes as LF
import cairo_zstd_b200 as czb
from cairo_zstd_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_max_frame_output_mirrors_header():
    h = open(os.path.join(ROOT, "include", "cairo_zstd_b200.h")).read()
    m = re.search(r"#define CZB_MAX_FRAME_OUTPUT (0x[0-9A-Fa-f]+)ull", h)
    assert m and int(m.group(1), 16) == api.MAX_FRAME_OUTPUT == czb.MAX_FRAME_OUTPUT == (1 << 31) - 1


ORACLE_STATUS = {
    "far_beyond_output": "CZS_NOT_ENOUGH_BYTES_IN_DICTIONARY",
    "far_literal_overrun_first": "CZS_EXEC_NOT_ENOUGH_BYTES_FOR_SEQUENCE",
    "far_2^28-1_at_2^28-2": "CZS_NOT_ENOUGH_BYTES_IN_DICTIONARY",
    "far_2^28+5_below_seam": "CZS_NOT_ENOUGH_BYTES_IN_DICTIONARY",
    "far_2^28+5_small_window": "CZS_OFFSET_TOO_BIG",
    "far_2^28+5_cap_short": "CZS_DST_TOO_SMALL",
}


@pytest.fixture(scope="module")
def cases():
    return LF.seam_cases()


def test_seam_frames_in_libzstd_and_oracle(cases):
    assert {c.name for c in cases} >= set(ORACLE_STATUS)
    for c in cases:
        st, res, out = LF.oracle_decode(c.frame, c.cap, keep_output=True)
        want = ORACLE_STATUS.get(c.name, "CZS_OK")
        assert czb.status_name(st) == want, (c.name, czb.status_name(st))
        if c.valid:
            ref = LF.libzstd_decode(c.frame, c.out)
            if st == 0:
                assert res.bytes_written == c.out and np.array_equal(out, ref), c.name
        del out


@pytest.mark.parametrize("n", [LF.M28 - 2, LF.M28 - 1, LF.M28])
def test_fill_frames_round_trip(n):
    blocks, content = LF.fill_blocks(n, seed=n & 0xFFFF, raw_every=256)
    f = LF.frame(blocks, n, xxh=LF.xxh32_low(content))
    assert np.array_equal(LF.libzstd_decode(f, n), content)
    st, res, out = LF.oracle_decode(f, n, keep_output=True)
    assert st == 0 and res.bytes_written == n and res.checksum_from_data == res.checksum_calculated
    assert np.array_equal(out, content)


def test_text_frames_round_trip():
    data = LF.text(40 << 20)
    for wl, ldm in ((23, False), (27, True)):
        f = LF.compress(data, wl, ldm=ldm)
        assert np.array_equal(LF.libzstd_decode(f, data.size), data)
        st, res = LF.oracle_decode(f, data.size)
        assert st == 0 and res.bytes_written == data.size and res.window_size == min(1 << wl, data.size)
