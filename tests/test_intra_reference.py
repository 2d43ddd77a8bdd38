"""Intra prediction without a GPU: the numpy restatement of 8.4.4.2 (tests/intra_ref.py) against the CPU oracle's `recon`
on every synthetic stream, the value-range extremes, the random configuration sweep (tests/synth/sweep.py), the directed
INTRA_CONFIGS streams and fixture tiles; the oracle against FFmpeg, live, on every INTRA_CONFIGS stream (exactly where
deblocking and SAO are off, so that FFmpeg's output is the intra reconstruction itself); and coverage assertions over the
reference's counters, so that none of this, nor the GPU tests on the same streams (tests/test_gpu_intra.py), can pass
without reaching every mode, size, filter decision and availability case."""
import hashlib
from collections import Counter

import numpy as np
import pytest

from oracle import oracle_py as O
from tests import intra_ref as I
from tests import loopfilter_ref as L
from tests.synth import synth
from tests.synth.configs import CONFIGS, EXTREME_CONFIGS, EXTREME_SEEDS, INTRA_CONFIGS, INTRA_SEEDS, SEEDS
from tests.synth.sweep import SWEEP
from tests.test_loopfilter_reference import _ffmpeg, assert_oracle_matches_ffmpeg

INTRA_STREAMS = [(name, cfg, seed) for name, cfg in INTRA_CONFIGS for seed in INTRA_SEEDS]
# sha256 over the four NAL units of every INTRA_STREAMS picture, in order: the coverage below is asserted for these streams
INTRA_STREAMS_SHA256 = "06c5fcca943be2edf88fb12bafffcb2402acf252cd2c6a1a624a8e922a72d0c5"
SIZES = (("Y", 4), ("Y", 8), ("Y", 16), ("Y", 32), ("C", 4), ("C", 8), ("C", 16))
MIN_PER_MODE = 8
MIN_PER_CLASS = 10


def _oracle(pic):
    t = pic.tile
    return O.decode_picture(pic.sps, pic.pps, t.header, (t.rbsp, t.rbsp_len))


def assert_reference_matches(pic, ref, stats=None):
    planes, stats = I.reconstruct(pic.sps, ref["tu_map"], ref["resid"], stats)
    for c, (a, b) in enumerate(zip(planes, ref["recon"])):
        assert np.array_equal(a, b), f"recon {c}: {int((a != b).sum())} samples differ, e.g. (y, x) {np.argwhere(a != b)[:4].tolist()}"
    return planes, stats


def test_tables_follow_the_standard():
    A = I.INTRA_PRED_ANGLE
    assert A[2:11] == (32, 26, 21, 17, 13, 9, 5, 2, 0) and A[18] == -32 and A[26] == 0 and A[34] == 32
    assert all(A[m] == A[36 - m] for m in range(2, 35)) and all(A[m] == -A[20 - m] for m in range(2, 10))
    assert [I.INV_ANGLE[m] for m in (11, 12, 13, 14, 15, 16, 17, 18)] == [-4096, -1638, -910, -630, -482, -390, -315, -256]
    assert all(I.INV_ANGLE[m] == I.INV_ANGLE[36 - m] for m in range(11, 26))
    # invAngle is 256 * 32 / intraPredAngle, rounded
    assert all(I.INV_ANGLE[m] == round(8192 / A[m]) for m in range(11, 26))
    assert I.INTRA_HOR_VER_DIST_THRES == {8: 7, 16: 1, 32: 0}


@pytest.mark.parametrize("name,cfg", CONFIGS, ids=[n for n, _ in CONFIGS])
def test_reference_matches_oracle_on_synthetic_streams(built, name, cfg):
    for seed in SEEDS:
        pic = synth.encode(seed, **cfg)
        assert_reference_matches(pic, _oracle(pic))


@pytest.mark.parametrize("name,cfg", EXTREME_CONFIGS, ids=[n for n, _ in EXTREME_CONFIGS])
def test_reference_matches_oracle_on_extreme_streams(built, name, cfg):
    for seed in EXTREME_SEEDS:
        pic = synth.encode(seed, **cfg)
        assert_reference_matches(pic, _oracle(pic))


@pytest.mark.parametrize("tile", range(48))
def test_reference_matches_oracle_on_fixture_tiles(heic_file, oracle_tiles, tile):
    img = heic_file.primary
    ref = oracle_tiles(tile)
    planes, _ = I.reconstruct(img.sps, ref["tu_map"], ref["resid"])
    for c in range(3):
        assert np.array_equal(planes[c], ref["recon"][c]), c


@pytest.fixture(scope="module")
def sweep_stats(built):
    """Every sweep picture: reference == oracle; the counters."""
    stats = I.new_stats()
    for name, cfg, seed in SWEEP:
        pic = synth.encode(seed, **cfg)
        assert_reference_matches(pic, _oracle(pic), stats)
    return stats


@pytest.fixture(scope="module")
def intra_set(built):
    """Every INTRA_CONFIGS picture: reference == oracle, oracle == FFmpeg; the counters, the reconstructions by stream and
    the FFmpeg deviations met."""
    stats, recon, hits = I.new_stats(), {}, Counter()
    for name, cfg, seed in INTRA_STREAMS:
        pic = synth.encode(seed, **cfg)
        ref = _oracle(pic)
        planes, _ = assert_reference_matches(pic, ref, stats)
        recon[name, seed] = planes
        sh = pic.tile.header
        if sh.slice_deblocking_filter_disabled_flag and not pic.sps.sample_adaptive_offset_enabled_flag:
            got = _ffmpeg(pic)
            assert len(got) == len(planes)
            for c, (f, o) in enumerate(zip(got, planes)):
                assert np.array_equal(f, o), (name, seed, c, int((f != o).sum()))
        else:
            deblocked, final, _ = L.loop_filter(pic.sps, pic.pps, sh, ref["recon"], ref["tu_map"], ref["qp_map"], ref["sao"])
            for c in range(len(final)):
                assert np.array_equal(deblocked[c], ref["deblocked"][c]) and np.array_equal(final[c], ref["plane"][c]), c
            assert_oracle_matches_ffmpeg(pic, ref, hits)
    return stats, recon, hits


def test_reference_matches_oracle_on_the_sweep(sweep_stats):
    """Reported on its own; sweep_stats asserts the reference against the oracle picture by picture."""
    assert sum(sweep_stats[k][("mode", 0)] for k in SIZES) > 0


def test_oracle_matches_ffmpeg_on_intra_streams(intra_set):
    """intra_set compares every picture: exactly with the loop filters off, else outside the two FFmpeg deviations of
    DESIGN.md section 4.  Half the streams run with the loop filters off."""
    n_off = sum(cfg.get("deblocking_disabled", 0) and not cfg.get("sao", 1) for _, cfg in INTRA_CONFIGS)
    assert 0.4 * len(INTRA_CONFIGS) <= n_off <= 0.6 * len(INTRA_CONFIGS)


def test_strong_smoothing_flag_changes_the_reconstruction(intra_set):
    """The smooth streams run twice with the same slice data, strong intra smoothing on and off: the flag must matter."""
    _, recon, _ = intra_set
    pairs = [(n, n.replace("_strong", "_no_strong")) for n, _ in INTRA_CONFIGS if "_strong" in n and "_no_strong" not in n
             and n.replace("_strong", "_no_strong") in dict(INTRA_CONFIGS)]
    assert len(pairs) == 2
    for on, off in pairs:
        for seed in INTRA_SEEDS:
            assert not np.array_equal(recon[on, seed][0], recon[off, seed][0]), (on, seed)


def test_directed_streams_reach_every_case(sweep_stats, intra_set):
    """Coverage over the union of the sweep and INTRA_CONFIGS, per component and block size."""
    total = I.new_stats()
    for s in (sweep_stats, intra_set[0]):
        for k, v in s.items():
            total[k].update(v)
    for k in SIZES:
        c = total[k]
        modes = [c[("mode", m)] for m in range(35)]
        assert min(modes) >= MIN_PER_MODE, (k, modes)
        # the interval assumption of the kernel's availability (one clamp of the scan position) holds everywhere
        assert c["not_one_interval"] == 0 and c["bl_partial_order"] == 0 and c["tr_partial_order"] == 0, (k, c)
        # partial bottom-left / above-right availability needs the picture edge through a neighbour block of N > 8
        # samples: picture sizes are multiples of MinCb >= 8, so it cannot happen for luma 4 / 8 and chroma 4
        classes = ("none", "full", "partial", "partial_edge") if k[1] > (4 if k[0] == "C" else 8) else ("none", "full")
        for side in ("bl", "tr"):
            for cls in classes:
                assert c[f"{side}_{cls}"] >= MIN_PER_CLASS, (k, side, cls, c)
        for key in ("left_missing", "top_missing", "none_available", "negative_angle_extended", "partial_ctb"):
            assert c[key] > 0, (k, key, c)
    assert total[("C", 4)]["split_chroma_4x4"] >= MIN_PER_CLASS
    for n in (8, 16, 32):
        c = total[("Y", n)]
        assert c["filter_none"] >= MIN_PER_CLASS and c["filter_121"] >= MIN_PER_CLASS, (n, c)
    c = total[("Y", 32)]
    assert c["filter_strong"] >= 10 * MIN_PER_CLASS, c
    for key in ("filter_strong_rejected", "reject_bl", "reject_tr", "reject_both"):
        assert c[key] >= MIN_PER_CLASS, (key, c)
    # flatness exactly at 1 << (BitDepth - 5): the strict comparison decides these
    assert c["reject_at_threshold"] >= 5, c


def test_intra_streams_are_deterministic():
    assert len({n for n, _ in INTRA_CONFIGS}) == len(INTRA_CONFIGS)
    digest = hashlib.sha256()
    for _, cfg, seed in INTRA_STREAMS:
        for nal in synth.encode_nals(seed, **cfg):
            digest.update(nal)
    assert digest.hexdigest() == INTRA_STREAMS_SHA256
