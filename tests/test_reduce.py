"""The box reduction's definition on the host (no GPU): the fixed-point formula of include/heic_b200.h
(heic_b200_decode_grids_reduced) is what the installed Pillow's Image.reduce computes, for every block shape and every
block sum, and on random images with partial blocks; and the Python size helper gives the reduced output size."""
import numpy as np
import pytest
from PIL import Image

import heif_b200 as H
from heif_b200 import _capi as K


def multiplier(n):
    """M(n) = trunc(float32(2^32) / float32(256 n))."""
    return np.uint32(np.float32(2.0 ** 32) / np.float32(256 * n))


def reduce_formula(a, k):
    """out = (((S + n // 2) * M(n)) mod 2^32) >> 24 over the blocks of k x k pixels (fewer in the last row and column) of an
    (H, W) or (H, W, C) uint8 array."""
    h, w = a.shape[:2]
    ys, xs = np.arange(0, h, k), np.arange(0, w, k)
    s = np.add.reduceat(np.add.reduceat(a.astype(np.uint64), ys, axis=0), xs, axis=1)
    n = np.outer(np.minimum(ys + k, h) - ys, np.minimum(xs + k, w) - xs).astype(np.uint64)
    m = np.vectorize(multiplier, otypes=[np.uint64])(n)
    if a.ndim == 3:
        n, m = n[..., None], m[..., None]
    return ((((s + n // 2) * m) & 0xFFFFFFFF) >> 24).astype(np.uint8)


@pytest.mark.parametrize("rows", range(1, 17))
def test_every_block_shape_and_every_sum(rows):
    """Blocks of rows x cols pixels (cols = 1..16) in an L image reduced by (cols, rows): one block per sum 0..255 n,
    the block's pixels filled with 255 up to the sum."""
    for cols in range(1, 17):
        n = rows * cols
        sums = np.arange(255 * n + 1, dtype=np.int64)
        per_row = 256
        n_blocks = -(-len(sums) // per_row) * per_row
        s = np.zeros(n_blocks, np.int64)
        s[:len(sums)] = sums
        j = np.arange(n)
        px = np.clip(s[:, None] - 255 * j[None, :], 0, 255).astype(np.uint8)  # (block, pixel of the block)
        img = px.reshape(n_blocks // per_row, per_row, rows, cols).transpose(0, 2, 1, 3).reshape(n_blocks // per_row * rows, per_row * cols)
        got = np.asarray(Image.fromarray(img, "L").reduce((cols, rows))).ravel()[:len(sums)]
        exp = ((((sums.astype(np.uint64) + n // 2) * np.uint64(multiplier(n))) & 0xFFFFFFFF) >> 24).astype(np.uint8)
        assert np.array_equal(got, exp), (rows, cols, int(np.flatnonzero(got != exp)[0]))


def test_rounded_mean_is_not_the_definition():
    """The exact rounded mean differs at ties for n not a power of two (k = 3: 255 sums)."""
    n = 9
    sums = np.arange(255 * n + 1, dtype=np.uint64)
    fixed = (((sums + n // 2) * np.uint64(multiplier(n))) & 0xFFFFFFFF) >> 24
    assert int(np.count_nonzero(fixed != (sums + n // 2) // n)) == 255


@pytest.mark.parametrize("mode", ["RGB", "L"])
def test_random_images_with_partial_blocks(mode):
    rng = np.random.default_rng(7)
    for i in range(60):
        h, w = (int(v) | 1 for v in rng.integers(1, 90, 2))
        shape = (h, w, 3) if mode == "RGB" else (h, w)
        a = rng.integers(0, 256, shape, dtype=np.uint8)
        if i % 3 == 0:
            a = np.where(a > 40, 255, a).astype(np.uint8)  # near saturation: the largest sums
        for k in range(1, 17):
            got = np.asarray(Image.fromarray(a, mode).reduce(k))
            exp = reduce_formula(a, k)
            assert got.shape == exp.shape == (-(-h // k), -(-w // k)) + shape[2:]
            assert np.array_equal(got, exp), (mode, h, w, k)


@pytest.mark.parametrize("orientation", range(8))
def test_output_size_is_ceil_after_the_turn(orientation):
    for crop in ((0, 0, 4032, 3024), (333, 217, 1001, 777), (1999, 0, 1, 3024), (500, 490, 30, 41)):
        t = K.ImageTransform(*crop, orientation)
        w, h = (crop[3], crop[2]) if orientation & 1 else (crop[2], crop[3])
        for k in range(1, 17):
            assert H._canvas(None, transform=t, reduce=k) == (-(-w // k), -(-h // k))


def test_output_size_of_the_file_canvas(heic_file):
    img = heic_file.primary
    assert H._canvas(img, reduce=3) == (1344, 1008)
    assert H._canvas(img, apply_transforms=True, reduce=7) == (-(-3024 // 7), -(-4032 // 7))


def test_reduction_factors_per_image():
    assert H._reduce_list(4, 3) == [4, 4, 4]
    assert H._reduce_list([1, 2, 16], 3) == [1, 2, 16]
    with pytest.raises(ValueError):
        H._reduce_list([2, 2], 3)
