"""The shared-memory layout of the rescoring kernels (csrc/stage_window.h) compiled for the HOST, over every shape the
API accepts: rows of 2, 4 and 8 bytes per element, every dim from 1 to 4096, every candidate count kp the scans use,
and every key source (the tcgen05 scan's union buffer, its dumped tiles, the CUDA-core scan's per-CTA lists).  The
layout must fit shared memory, leave room for a band of 1 024 to 2 048 rows, and its column chunks must tile each row
and land in three disjoint slots of the staged-row window -- stage_and_chain indexes them with the same formulas."""
import numpy as np
import pytest

from stage_window_lib import ELEM_BYTES, KP_SIMT, KP_TC, SLAB, SM_COUNT, Harness

FITS, GPR, PITCH, CHUNKS, BAND_CAP, SMEM = range(6)


@pytest.fixture(scope="module")
def H(tmp_path_factory):
    return Harness(tmp_path_factory.mktemp("stage_window"))


def _key_sources(H, kp, scan):
    """(name, lists, list_len) of every key source the select kernel sees for candidate count kp."""
    if scan == "tc":
        yield "slab", 0, 0
        for tiles in range(1, H.SCAN_DUMP_MAX_KEYS // H.SCAN_DUMP_TILE + 1):   # dump mode: 1 to 74 tiles of 128 keys
            yield f"dump{tiles}", tiles, H.SCAN_DUMP_TILE
    else:
        for lists in range(1, 2 * SM_COUNT + 1):                                # min(ceil(n / 32), 2 x 148) lists of kp keys
            yield f"lists{lists}", lists, kp


def _shapes():
    for dt in ELEM_BYTES:
        for kp in KP_TC:
            yield dt, kp, "tc"
        for kp in KP_SIMT:
            yield dt, kp, "simt"


def _check_windows(H, gpr, pitch, chunks, what):
    """Every distinct (gpr, pitch, chunks) walked once with the kernel's chunk and slot formulas."""
    for g, p, c in sorted(set(zip(gpr.tolist(), pitch.tolist(), chunks.tolist()))):
        rc, lo, slot = H.walk(g, p, c)
        rule = {1: "chunks do not tile the row", 2: "a chunk is wider than its slot", 3: "slots overlap or leave the window",
                4: "whole rows are not staged in their own columns"}.get(rc)
        assert rc == 0, (what, g, p, c, rule, lo.tolist(), slot.tolist())


def _check_pitch(gpr, pitch, chunks, elem_bytes, what):
    """The staged-row pitch is an odd number of 16-byte groups (chains walking their own rows at the same column hit
    different banks).  The one exception: whole bf16 rows with an odd number of groups, staged as they are."""
    odd = (pitch // 16) % 2 == 1
    whole = (chunks == 3) & (pitch // 16 == gpr + 1)
    exception = whole & (gpr % 2 == 1)
    assert not exception.any() or elem_bytes == 2, what
    assert (pitch % 16 == 0).all(), what
    assert odd[~exception].all(), (what, np.nonzero(~odd & ~exception)[0][:5] + 1)


@pytest.mark.parametrize("dt,kp,scan", list(_shapes()))
def test_select_layout_every_shape(H, dt, kp, scan):
    eb = ELEM_BYTES[dt]
    for name, lists, list_len in _key_sources(H, kp, scan):
        what = (dt, kp, name)
        a = H.select(eb, kp, lists, list_len)
        assert a[:, FITS].all(), (what, "does not fit at dim", int(np.argmin(a[:, FITS])) + 1)
        assert (a[:, SMEM] <= 180 * 1024).all() and H.SR_SMEM_LIMIT == 180 * 1024, what
        cap = a[:, BAND_CAP]
        assert ((cap >= 1024) & (cap <= 2048) & (cap % 64 == 0)).all(), (what, cap.min(), cap.max())
        assert (a[:, CHUNKS] >= 3).all() and (a[:, CHUNKS] <= np.maximum(a[:, GPR], 3)).all(), what
        # the band arrays fill what the window leaves: one more 64-row step of band would not fit
        assert ((a[:, SMEM] + 64 * 12 > H.SR_SMEM_LIMIT) | (cap == 2048)).all(), what
        _check_pitch(a[:, GPR], a[:, PITCH], a[:, CHUNKS], eb, what)
        _check_windows(H, a[:, GPR], a[:, PITCH], a[:, CHUNKS], what)


@pytest.mark.parametrize("dt", list(ELEM_BYTES))
def test_collect_layout_every_dim(H, dt):
    eb = ELEM_BYTES[dt]
    a = H.collect(eb)
    assert H.CR_ROWS == 32 and (a[:, 0] == 32).all()
    assert (a[:, 3] >= 3).all(), "collect pass does not fit"
    assert (a[:, 4] <= 200 * 1024).all() and H.CR_SMEM_LIMIT == 200 * 1024
    _check_pitch(a[:, 1], a[:, 2], a[:, 3], eb, ("collect", dt))
    _check_windows(H, a[:, 1], a[:, 2], a[:, 3], ("collect", dt))


def test_whole_bf16_rows_with_odd_groups_are_the_pitch_exception(H):
    """A 1000-d bf16 row is 125 groups: staged whole, its pitch is 126 groups -- even, and the only kind of even pitch."""
    a = H.select(2, 32, dims=(1000, 1001))[0]
    assert a[GPR] == 125 and a[CHUNKS] == 3 and a[PITCH] == 126 * 16


def test_regimes_the_gpu_tests_rely_on(H):
    """Windowed and whole-row regimes at the shape edges, and band capacities below the 2 048-row maximum."""
    # last whole-row dim and first windowed dim of the candidate window (slab mode)
    for eb, kp, last_whole in [(4, 32, 1016), (4, 64, 520), (2, 32, 1920), (2, 64, 1016), (8, 32, 520), (8, 64, 264)]:
        assert H.stage_regime(eb, last_whole, kp)[0] == 3
        assert H.stage_regime(eb, last_whole + 1, kp)[0] > 3
    assert [H.stage_regime(eb, 4096, kp)[0] for eb, kp in [(4, 32), (4, 64), (2, 32), (2, 64), (8, 32), (8, 64)]] == [16, 31, 8, 16, 31, 61]
    for eb, last_whole, chunks_4096 in [(4, 1136, 13), (2, 2152, 7), (8, 584, 26)]:
        assert H.collect_regime(eb, last_whole)[0] == 3 and H.collect_regime(eb, last_whole + 1)[0] > 3
        assert H.collect_regime(eb, 4096)[0] == chunks_4096
    # the adapters' default store (binary64, 384-d) with 17 <= k <= 48 in dump mode, and other capacities below 2 048
    assert H.stage_regime(8, 384, 64, H.dump_tiles(9472)) == (7, 1360, 1472)
    assert H.stage_regime(8, 1920, 64)[2] == 1152
    assert H.stage_regime(8, 4096, 64, H.dump_tiles(9472)) == (103, 976, 1024)
    assert H.stage_regime(8, 4096, 64)[2] == 1088
    assert H.dump_tiles(9472) == (74, 128) and H.dump_tiles(9473) is None and SLAB == 0
