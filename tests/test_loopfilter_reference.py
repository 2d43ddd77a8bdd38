"""The in-loop filters without a GPU: the numpy restatement of deblocking and SAO (tests/loopfilter_ref.py) against the CPU
oracle's `deblocked` and final planes on every synthetic stream over more seeds than the FFmpeg-pinned two, on fixture
tiles and on the random configuration sweep (tests/synth/sweep.py); the oracle against FFmpeg, live, on the whole sweep
and on the CTB-16 streams; and coverage assertions over the reference's counters, so that none of this, nor the GPU
tests on the same streams (tests/test_gpu_loopfilter.py), can pass without reaching every filter decision and SAO class.

FFmpeg is not the referee everywhere.  The bundled FFmpeg deviates from H.265 in two places, both characterised by
the reference (DESIGN.md section 4), and an oracle/FFmpeg mismatch passes only where the oracle equals the reference and
the sample lies inside one of these two patterns:
- FFMPEG_CTB16_SAO_CORNER: with 16x16 CTBs (8x8 chroma CTBs), FFmpeg's SAO of the right column of a chroma CTB reads
  the next CTB's first column before that column's horizontal chroma edge is deblocked.  8.7.3 takes the deblocked
  picture.  Affected: chroma samples at x % 8 == 7 with a right neighbour, in rows y % 8 in {6, 7, 0, 1}.
- FFMPEG_CHROMA_QPI_CLIP: FFmpeg clips the chroma deblocking index qPi to 57 (the clip 8.6.1 applies to dequantisation);
  8.7.2.5.5 has no clip, Table 8-10 gives QpC = qPi - 6 above 42.  Affected: the two samples either side of a chroma
  edge segment whose qPi exceeds 57 where the two tC differ, and the samples next to them that SAO reads them from.
"""
from collections import Counter

import numpy as np
import pytest

from oracle import oracle_py as O
from oracle.ffmpeg_oracle import FFmpegHevc
from tests import loopfilter_ref as L
from tests.synth import synth
from tests.synth.configs import CONFIGS, EXTREME_CONFIGS
from tests.synth.sweep import SWEEP

SEEDS = range(4)
_CTB16 = dict(log2_ctb=4, log2_max_tb=4, width=96, height=80)
# the CTB-16 streams on which the oracle and FFmpeg were first seen to disagree
CTB16_STREAMS = [
    ("ctb16", dict(CONFIGS)["ctb16"]),
    ("big_qp51_ctb16", dict(EXTREME_CONFIGS)["big_qp51_ctb16"]),
    ("ctb16_96x80_qp30", dict(_CTB16, init_qp_minus26=4)),
    ("ctb16_96x80_qp51", dict(_CTB16, init_qp_minus26=25)),
]
CTB16_SEEDS = range(16)


def _oracle(pic):
    t = pic.tile
    return O.decode_picture(pic.sps, pic.pps, t.header, (t.rbsp, t.rbsp_len))


def _ffmpeg(pic):
    # a fresh context per picture: one context carried state from a 4:2:0 picture into a following 4:0:0 one
    dec = FFmpegHevc()
    try:
        return dec.decode_picture(pic.annexb())
    finally:
        dec.close()


def _reference(sps, pps, sh, ref, stats=None):
    return L.loop_filter(sps, pps, sh, ref["recon"], ref["tu_map"], ref["qp_map"], ref["sao"], stats)


def _assert_reference_matches(pic, ref, stats=None):
    deblocked, final, stats = _reference(pic.sps, pic.pps, pic.tile.header, ref, stats)
    for key, planes in (("deblocked", deblocked), ("plane", final)):
        for c, (a, b) in enumerate(zip(planes, ref[key])):
            assert np.array_equal(a, b), f"{key} {c}: {int((a != b).sum())} samples differ"
    return stats


# ---- the two FFmpeg deviations -------------------------------------------------------------------------------------
def _ctb16_sao_corner(pic, c, shape):
    log2_ctb = pic.sps.log2_min_luma_coding_block_size_minus3 + 3 + pic.sps.log2_diff_max_min_luma_coding_block_size
    mask = np.zeros(shape, bool)
    if c == 0 or log2_ctb != 4:
        return mask
    h, w = shape
    ys, xs = np.arange(h)[:, None], np.arange(w)[None, :]
    return (xs % 8 == 7) & (xs + 1 < w) & np.isin(ys % 8, (6, 7, 0, 1))


def _qpi_clip_vertical(a_shape, edges, qp, qp_offset, tc_off):
    """Samples of a chroma plane (vertical-edge orientation) next to a chroma edge segment whose tC changes when qPi is
    clipped to 57: p1 .. q1 over the segment's lines and one line either side."""
    mask = np.zeros(a_shape, bool)
    ce = edges[0::2, 0::2].copy()
    ce[:, 0] = False
    for seg, col in zip(*np.nonzero(ce)):
        qpi = ((int(qp[seg, 2 * col]) + int(qp[seg, 2 * col - 1]) + 1) >> 1) + qp_offset
        tc = [L.TC_TABLE[min(53, max(0, L.qpc_from_qpi(q) + 2 + 2 * tc_off))] for q in (qpi, min(qpi, 57))]
        if qpi > 57 and tc[0] != tc[1]:
            mask[max(0, 4 * seg - 1):4 * seg + 5, 8 * col - 2:8 * col + 2] = True
    return mask


def _chroma_qpi_clip(pic, ref, c):
    if c == 0 or pic.tile.header.slice_deblocking_filter_disabled_flag:
        return np.zeros(ref["plane"][c].shape, bool)
    ver, hor = L.transform_edges(pic.sps, ref["tu_map"])
    off = pic.pps.pps_cb_qp_offset if c == 1 else pic.pps.pps_cr_qp_offset
    tc_off = pic.tile.header.slice_tc_offset_div2
    shape = ref["plane"][c].shape
    return (_qpi_clip_vertical(shape, ver, ref["qp_map"], off, tc_off)
            | _qpi_clip_vertical(shape[::-1], hor.T, ref["qp_map"].T, off, tc_off).T)


def assert_oracle_matches_ffmpeg(pic, ref, hits: Counter):
    """Oracle final planes == FFmpeg's, except at the two characterised FFmpeg deviations (counted into `hits`).  The
    callers have checked the oracle against the reference, so every exempted sample is one where they agree."""
    got = _ffmpeg(pic)
    assert len(got) == len(ref["plane"])
    for c, (f, o) in enumerate(zip(got, ref["plane"])):
        bad = f != o
        if not bad.any():
            continue
        corner, clip = _ctb16_sao_corner(pic, c, o.shape), _chroma_qpi_clip(pic, ref, c)
        rest = bad & ~corner & ~clip
        assert not rest.any(), f"component {c}: {int(rest.sum())} samples differ from FFmpeg, e.g. (y, x) {np.argwhere(rest)[:4].tolist()}"
        hits["ctb16_sao_corner"] += int((bad & corner).sum())
        hits["chroma_qpi_clip"] += int((bad & clip & ~corner).sum())


# ---- tests ---------------------------------------------------------------------------------------------------------
def test_tables_follow_the_standard():
    assert L.BETA_TABLE[15:19] == (0, 6, 7, 8) and L.BETA_TABLE[28:31] == (18, 20, 22) and L.BETA_TABLE[51] == 64
    assert L.TC_TABLE[17:19] == (0, 1) and L.TC_TABLE[26:28] == (1, 2) and L.TC_TABLE[37:54:4] == (4, 6, 10, 16, 24)
    assert all(a <= b for a, b in zip(L.BETA_TABLE, L.BETA_TABLE[1:])) and all(a <= b for a, b in zip(L.TC_TABLE, L.TC_TABLE[1:]))
    assert [L.qpc_from_qpi(q) for q in (-12, 29, 30, 34, 35, 42, 43, 57, 63)] == [-12, 29, 29, 33, 33, 37, 37, 51, 57]


@pytest.mark.parametrize("name,cfg", CONFIGS, ids=[n for n, _ in CONFIGS])
def test_reference_matches_oracle_on_synthetic_streams(built, name, cfg):
    for seed in SEEDS:
        pic = synth.encode(seed, **cfg)
        _assert_reference_matches(pic, _oracle(pic))


@pytest.mark.parametrize("name,cfg", EXTREME_CONFIGS, ids=[n for n, _ in EXTREME_CONFIGS])
def test_reference_matches_oracle_on_extreme_streams(built, name, cfg):
    for seed in SEEDS:
        pic = synth.encode(seed, **cfg)
        _assert_reference_matches(pic, _oracle(pic))


@pytest.mark.parametrize("tile", [0, 17, 47])
def test_reference_matches_oracle_on_fixture_tiles(heic_file, oracle_tiles, tile):
    img = heic_file.primary
    ref = oracle_tiles(tile)
    deblocked, final, _ = _reference(img.sps, img.pps, img.tiles[tile].header, ref)
    for c in range(3):
        assert np.array_equal(deblocked[c], ref["deblocked"][c]), c
        assert np.array_equal(final[c], ref["plane"][c]), c


@pytest.fixture(scope="module")
def sweep_set(built):
    """Every sweep picture: reference == oracle, oracle == FFmpeg within the exemption; counters per CTB size."""
    stats = {k: L.new_stats() for k in (4, 5, 6)}
    hits = Counter()
    for name, cfg, seed in SWEEP:
        pic = synth.encode(seed, **cfg)
        ref = _oracle(pic)
        _assert_reference_matches(pic, ref, stats[cfg["log2_ctb"]])
        assert_oracle_matches_ffmpeg(pic, ref, hits)
    return stats, hits


def test_reference_matches_oracle_on_the_sweep(sweep_set):
    """Reported on its own; sweep_set asserts the reference against the oracle picture by picture."""
    stats, _ = sweep_set
    assert sum(s["luma"]["skipped"] + s["luma"]["strong"] + s["luma"]["normal"] for s in stats.values()) > 0


def test_oracle_matches_ffmpeg_on_the_sweep(sweep_set):
    _, hits = sweep_set
    # both deviations turn up in the sweep: it has CTB-16 pictures with SAO and chroma offsets that push qPi over 57
    assert hits["ctb16_sao_corner"] > 0 and hits["chroma_qpi_clip"] > 0, hits


@pytest.mark.parametrize("name,cfg", CTB16_STREAMS, ids=[n for n, _ in CTB16_STREAMS])
def test_ctb16_streams_follow_the_reference_not_ffmpeg(built, name, cfg):
    """The CTB-16 disagreement: the oracle equals the reference on every picture, and every sample where FFmpeg differs
    is an SAO sample at a chroma CTB corner."""
    hits = Counter()
    for seed in CTB16_SEEDS:
        pic = synth.encode(seed, **cfg)
        ref = _oracle(pic)
        _assert_reference_matches(pic, ref)
        assert_oracle_matches_ffmpeg(pic, ref, hits)
    assert hits["ctb16_sao_corner"] > 0 and hits["chroma_qpi_clip"] == 0, hits


def test_sweep_reaches_every_decision(sweep_set):
    stats, _ = sweep_set
    total = L.new_stats()
    for s in stats.values():
        total["luma"].update(s["luma"])
        total["chroma_filtered"] += s["chroma_filtered"]
        total["chroma_tc0"] += s["chroma_tc0"]
        for c in range(3):
            total["sao"][c].update(s["sao"][c])
    for k in ("skipped", "strong", "normal", "dEp", "dEq"):
        assert total["luma"][k] > 0, total["luma"]
    assert total["luma"]["normal"] > total["luma"]["dEp"] and total["luma"]["normal"] > total["luma"]["dEq"]  # both ways
    assert total["chroma_filtered"] > 0 and total["chroma_tc0"] > 0
    for c in range(3):
        for k in ("band", "eo0", "eo1", "eo2", "eo3"):
            assert total["sao"][c][k] > 0, (c, total["sao"][c])
    # for every CTB size and component, SAO results that depend on a neighbour in another CTB which deblocking changed,
    # and SAO changing samples on CTB borders
    for log2_ctb, s in stats.items():
        for c in range(3):
            assert s["sao_reads_deblocked_across_ctb"][c] > 0, (log2_ctb, c, s["sao_reads_deblocked_across_ctb"])
            assert s["sao_boundary_changed"][c] > 0, (log2_ctb, c, s["sao_boundary_changed"])


def test_sweep_is_deterministic_and_varied():
    from tests.synth.sweep import cases

    assert cases() == SWEEP and cases(1) != SWEEP
    cfgs = [cfg for _, cfg, _ in SWEEP]
    assert {c["log2_ctb"] for c in cfgs} == {4, 5, 6} and {c["chroma_format_idc"] for c in cfgs} == {0, 1}
    assert {c["wpp"] for c in cfgs} == {0, 1} and {c["scaling_list_mode"] for c in cfgs} == {0, 1, 2, 3}
    assert any(c.get("deblocking_disabled") for c in cfgs) and any(c["sao"] == 0 for c in cfgs)
    assert any(c.get("slice_sao_luma") == 0 for c in cfgs) and any(c.get("slice_sao_chroma") == 0 for c in cfgs)
    assert any(c["width"] <= 1 << c["log2_ctb"] for c in cfgs) and any(c["height"] <= 1 << c["log2_ctb"] for c in cfgs)
    for c in cfgs:
        assert c["width"] % (1 << c["log2_min_cb"]) == 0 and c["height"] % (1 << c["log2_min_cb"]) == 0
        assert c["log2_min_tb"] < c["log2_min_cb"] <= c["log2_ctb"] and c["log2_max_tb"] <= min(5, c["log2_ctb"])
        assert 0 <= 26 + c["init_qp_minus26"] + c["slice_qp_delta"] <= 51
        for k in ("cb", "cr"):
            assert abs(c[f"{k}_qp_offset"]) <= 12 and abs(c[f"{k}_qp_offset"] + c[f"slice_{k}_qp_offset"]) <= 12
