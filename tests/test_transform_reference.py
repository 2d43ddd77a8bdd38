"""Value-range extremes without a GPU: the numpy restatement of scaling + inverse transform (tests/transform_ref.py)
against the CPU oracle on the extreme synthetic streams (escape-coded levels up to 32767, saturating scaling, QP 0 / 51,
scaling lists over 1..255), the ordinary ones and fixture tiles; the escape code of coeff_abs_level_remaining through the
arithmetic coder for every value and cRiceParam; and coverage assertions, so that the GPU tests on the same streams
(tests/test_gpu_extremes.py) cannot pass without reaching the limits they are about."""
from collections import Counter

import numpy as np
import pytest

from oracle import oracle_py as O
from tests import transform_ref as R
from tests.synth import synth
from tests.synth.configs import CONFIGS, EXTREME_CONFIGS, EXTREME_SEEDS, SEEDS


def _oracle(pic):
    t = pic.tile
    return O.decode_picture(pic.sps, pic.pps, t.header, (t.rbsp, t.rbsp_len))


def _assert_reference_matches(pic, ref, stats=None):
    res, stats = R.residuals(pic.sps, pic.pps, pic.tile.header, ref["tu_map"], ref["level"], stats)
    assert len(res) == len(ref["resid"])
    for c, (a, b) in enumerate(zip(res, ref["resid"])):
        assert np.array_equal(a, b), f"residual {c}: {int((a != b).sum())} samples differ"
    return stats


def test_matrices_follow_the_standard():
    # the 4 / 8 / 16 point DCTs are the 32-point matrix's rows 0, 32/n, 2*32/n, ... cut to n columns
    for n in (4, 8, 16):
        assert np.array_equal(R.dct_matrix(n), R.DCT32[:: 32 // n, :n]), n
    # nearly orthogonal with norm 64^2 * n: a wrong magnitude or sign anywhere breaks this
    for m in (R.DCT4, R.DCT8, R.DCT16, R.DCT32, R.DST4):
        n = m.shape[0]
        p = m @ m.T
        diag = np.diag(p)
        assert np.all(np.abs(diag - 4096 * n) <= 0.005 * 4096 * n), n
        assert np.abs(p - np.diag(diag)).max() <= 0.005 * 4096 * n, n
    # the even rows of the 32-point matrix are symmetric, the odd ones antisymmetric
    assert np.array_equal(R.DCT32[0::2], R.DCT32[0::2, ::-1]) and np.array_equal(R.DCT32[1::2], -R.DCT32[1::2, ::-1])
    assert list(R.DCT32[1, :16]) == [90, 90, 88, 85, 82, 78, 73, 67, 61, 54, 46, 38, 31, 22, 13, 4]


def test_chroma_qp_table():
    assert [R.chroma_qp(q, 0) for q in range(28, 46)] == [28, 29, 29, 30, 31, 32, 33, 33, 34, 34, 35, 35, 36, 36, 37, 37, 38, 39]
    assert R.chroma_qp(51, 12) == 51 and R.chroma_qp(0, -12) == 0 and R.chroma_qp(51, -12) == 35


@pytest.mark.parametrize("name,cfg", EXTREME_CONFIGS, ids=[n for n, _ in EXTREME_CONFIGS])
def test_reference_matches_oracle_on_extreme_streams(built, name, cfg):
    for seed in EXTREME_SEEDS:
        pic = synth.encode(seed, **cfg)
        _assert_reference_matches(pic, _oracle(pic))


@pytest.mark.parametrize("name,cfg", CONFIGS, ids=[n for n, _ in CONFIGS])
def test_reference_matches_oracle_on_synthetic_streams(built, name, cfg):
    for seed in SEEDS:
        pic = synth.encode(seed, **cfg)
        _assert_reference_matches(pic, _oracle(pic))


@pytest.mark.parametrize("tile", [0, 17, 47])
def test_reference_matches_oracle_on_fixture_tiles(heic_file, oracle_tiles, tile):
    img = heic_file.primary
    ref = oracle_tiles(tile)
    res, _ = R.residuals(img.sps, img.pps, img.tiles[tile].header, ref["tu_map"], ref["level"])
    for c in range(3):
        assert np.array_equal(res[c], ref["resid"][c]), c


@pytest.mark.parametrize("rice", range(5))
def test_level_remaining_round_trip_is_exhaustive(built, rice):
    """Every coeff_abs_level_remaining value 0..32767 at cRiceParam 0..4, each at four seeded ivlCurrRange / bit / byte
    phases: the device routine (7-bin division steps), the bin-by-bin loop and the encoder agree on value and bins."""
    bad = []
    for value in range(32768):
        for phase in range(4):
            rc, dev, loop, n_bins = synth.level_remaining_roundtrip(rice, value, value * 4 + phase)
            if rc != 0 or dev != (value, n_bins) or loop != (value, n_bins):
                bad.append((value, phase, rc, dev, loop, n_bins))
    assert not bad, bad[:8]


def _escape_bins(rice, value):  # 9.3.3.11 bin count, restated
    if value < 4 << rice:
        return (value >> rice) + 1 + rice
    u, k, ones = value - (4 << rice), rice + 1, 0
    while u >= 1 << k:
        u -= 1 << k
        k += 1
        ones += 1
    return 4 + ones + 1 + k


def test_level_remaining_bin_counts(built):
    for rice in range(5):
        for value in (0, 1, 3, 4, 5, 15, 16, 63, 64, 65, 1000, 8193, 8194, 32767):
            _, _, _, n_bins = synth.level_remaining_roundtrip(rice, value, 1)
            assert n_bins == _escape_bins(rice, value), (rice, value)


@pytest.fixture(scope="module")
def extreme_set(built):
    """Oracle decodes and reference counters of every extreme stream, both seeds."""
    stats = R.new_stats()
    qps, samples, max_level = Counter(), Counter(), 0
    for name, cfg in EXTREME_CONFIGS:
        for seed in EXTREME_SEEDS:
            pic = synth.encode(seed, **cfg)
            ref = _oracle(pic)
            _assert_reference_matches(pic, ref, stats)
            tu = ref["tu_map"]
            qps.update(((tu[(tu & 1) == 1] >> 19) & 63).tolist())
            for p in ref["plane"]:
                samples[0] += int((p == 0).sum())
                samples[255] += int((p == 255).sum())
            max_level = max(max_level, max(int(np.abs(l.astype(np.int32)).max()) for l in ref["level"]))
    return stats, qps, samples, max_level


def test_extreme_set_reaches_the_limits(extreme_set):
    stats, qps, samples, max_level = extreme_set
    assert max_level == 32767
    assert sum(v for k, v in stats["prefix"].items() if k >= 12) > 0, stats["prefix"]  # long EG(k) escape prefixes
    assert stats["wide_blocks"] > 0 and stats["wide_unsaturated_blocks"] > 0  # the kernels' 64-bit scaling branch
    assert stats["big_level_4x4_blocks"] > 0  # |level| > 255 in 4x4 blocks: the 64-bit branch of the 4x4 kernel
    for cls in R.CLASSES:
        assert stats["sat_pos"][cls] > 0 and stats["sat_neg"][cls] > 0, (cls, stats["sat_pos"], stats["sat_neg"])
    for cls in ("4y", "4c", "8", "16", "32"):
        assert stats["first_clip"][cls] > 0, (cls, stats["first_clip"])
    assert stats["second_clip"] == 0  # |r| <= 32768 * 2880 >> 12 cannot leave int16
    assert min(qps) <= 2 and max(qps) >= 49 and 0 in qps and 51 in qps, sorted(qps)
    assert samples[0] > 0 and samples[255] > 0
