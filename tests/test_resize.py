"""The resize's definition on the host (no GPU): the fixed-point tables of heic_b200_resample_coeffs, fed to a numpy
restatement of the two integer passes of include/heic_b200.h (heic_b200_decode_grids_resized), give what the installed
Pillow's Image.resize gives -- all five filters, RGB and L, random sizes up- and downscaling, one axis unchanged and
extreme ratios.  Three mistakes in the restatement each break that agreement: the vertical pass first, no uint8 clip
between the passes, float32 coefficients.  Plus the ABI details: sizeof(heic_resize), the new exports, the Python size
helper."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest
from PIL import Image

import heif_b200 as H
from heif_b200 import _capi as K

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILTERS = {"LANCZOS": 1, "BILINEAR": 2, "BICUBIC": 3, "BOX": 4, "HAMMING": 5}
PIL_FILTERS = {1: Image.Resampling.LANCZOS, 2: Image.Resampling.BILINEAR, 3: Image.Resampling.BICUBIC, 4: Image.Resampling.BOX,
               5: Image.Resampling.HAMMING}


# ---- the coefficients, restated (for the float32 mistake and as a cross-check of the library's tables) ------------------
def _filters(dt):
    pi, half, one = dt(math.pi), dt(0.5), dt(1.0)
    sin, cos = (math.sin, math.cos) if dt is float else (lambda v: dt(np.sin(v)), lambda v: dt(np.cos(v)))

    def box(x):
        return one if -half < x <= half else dt(0.0)

    def bilinear(x):
        x = abs(x)
        return one - x if x < one else dt(0.0)

    def hamming(x):
        x = abs(x)
        if x == 0:
            return one
        if x >= one:
            return dt(0.0)
        x = x * pi
        return sin(x) / x * (dt(np.float32(0.54)) + dt(np.float32(0.46)) * cos(x))  # Pillow's 0.54f and 0.46f

    def bicubic(x):
        a = dt(-0.5)
        x = abs(x)
        if x < one:
            return ((a + dt(2.0)) * x - (a + dt(3.0))) * x * x + one
        if x < dt(2.0):
            return (((x - dt(5)) * x + dt(8)) * x - dt(4)) * a
        return dt(0.0)

    def sinc(x):
        if x == 0:
            return one
        x = x * pi
        return sin(x) / x

    def lanczos(x):
        return sinc(x) * sinc(x / dt(3)) if dt(-3.0) <= x < dt(3.0) else dt(0.0)

    return {1: (lanczos, 3.0), 2: (bilinear, 1.0), 3: (bicubic, 2.0), 4: (box, 0.5), 5: (hamming, 1.0)}


def coeffs_restated(n_in, n_out, f, dt=float):
    fn, sup = _filters(dt)[f]
    scale = dt(n_in) / dt(n_out)
    fs = max(scale, dt(1.0))
    support = dt(sup) * fs
    ss = dt(1.0) / fs
    bounds, coeffs = [], []
    for xx in range(n_out):
        center = (dt(xx) + dt(0.5)) * scale
        xmin = max(int(center - support + dt(0.5)), 0)
        xmax = min(int(center + support + dt(0.5)), n_in) - xmin
        w = [fn((dt(x + xmin) - center + dt(0.5)) * ss) for x in range(xmax)]
        ww = dt(0.0)
        for v in w:
            ww += v
        if ww != 0:
            w = [v / ww for v in w]
        bounds.append((xmin, xmax))
        coeffs += [int(dt(-0.5) + v * dt(1 << 22)) if v < 0 else int(dt(0.5) + v * dt(1 << 22)) for v in w]
    return np.array(bounds, np.int32).reshape(n_out, 2), np.array(coeffs, np.int32)


# ---- the two integer passes ------------------------------------------------------------------------------------------------
def _dense(bounds, coeffs, n_in):
    m = np.zeros((len(bounds), n_in), np.int64)
    off = 0
    for j, (xmin, n) in enumerate(bounds):
        m[j, xmin:xmin + n] = coeffs[off:off + n]
        off += n
    return m


def _pass(a, m, axis, clip=True):
    """s = 2^21 + sum in * k in int32 along `axis` of an (h, w, c) array, then s >> 22 clamped to 0..255."""
    s = np.einsum("hwc,ow->hoc", a, m) if axis == 1 else np.einsum("hwc,oh->owc", a, m)
    s = s + (1 << 21)
    assert np.abs(s).max(initial=0) < 2 ** 31  # int32 arithmetic, as the kernels and Pillow do it
    s = s >> 22
    return np.clip(s, 0, 255) if clip else s


def resize_restated(img, size, f, mistake=None):
    W, Hh = size
    h, w = img.shape[:2]
    a = img.reshape(h, w, -1).astype(np.int64)
    if (W, Hh) == (w, h):
        return img.copy()
    tab = (lambda n_in, n_out: coeffs_restated(n_in, n_out, f, np.float32)) if mistake == "float32" else \
        (lambda n_in, n_out: H.resample_coeffs(n_in, n_out, f))
    bh, kh = tab(w, W)
    bv, kv = tab(h, Hh)
    if mistake == "vertical_first":
        if Hh != h:
            a = _pass(a, _dense(bv, kv, h), 0)
        if W != w:
            a = _pass(a, _dense(bh, kh, w), 1)
    else:
        if W != w:
            row0, row1 = int(bv[0, 0]), int(bv[-1, 0] + bv[-1, 1])
            a = _pass(a[row0:row1], _dense(bh, kh, w), 1, clip=mistake != "no_clip")
            bv = bv.copy()
            bv[:, 0] -= row0
        if Hh != h:
            a = _pass(a, _dense(bv, kv, a.shape[0]), 0)
    return np.clip(a, 0, 255).astype(np.uint8).reshape((Hh, W) + img.shape[2:])


def pillow(img, size, f):
    return np.asarray(Image.fromarray(img).resize(size, PIL_FILTERS[f], reducing_gap=None))


def random_cases(seed, n):
    """(h, w, W, H) with sizes 1..400, about a third with one axis unchanged."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        h, w, W, Hh = (int(v) for v in rng.integers(1, 401, 4))
        if i % 3 == 1:
            W = w
        elif i % 3 == 2:
            Hh = h
        out.append((h, w, W, Hh))
    return out


def image(rng, h, w, mode):
    a = rng.integers(0, 256, (h, w, 3) if mode == "RGB" else (h, w), dtype=np.uint8)
    return np.where(a > 200, 255, np.where(a < 40, 0, a)).astype(np.uint8)  # hard edges: ringing that overshoots 0..255


EXTREME = [(3, 4032, 1, 3), (4032, 3, 3, 1), (2, 1, 300, 2), (1, 2, 2, 300), (1, 1, 300, 300), (3, 3024, 3, 3), (3024, 3, 3, 3),
           (7, 4032, 1, 1)]


@pytest.mark.parametrize("mode", ["RGB", "L"])
@pytest.mark.parametrize("name", list(FILTERS))
def test_restatement_with_library_tables_equals_pillow(name, mode):
    f = FILTERS[name]
    rng = np.random.default_rng(f * 10 + (mode == "L"))
    for h, w, W, Hh in random_cases(f + 100 * (mode == "L"), 40) + EXTREME:
        a = image(rng, h, w, mode)
        got, exp = resize_restated(a, (W, Hh), f), pillow(a, (W, Hh), f)
        assert got.shape == exp.shape and np.array_equal(got, exp), (name, mode, (w, h), (W, Hh))


@pytest.mark.parametrize("name", list(FILTERS))
def test_library_tables_equal_the_double_restatement(name):
    f = FILTERS[name]
    for n_in, n_out in [(c[1], c[2]) for c in random_cases(f, 30)] + [(4032, 1), (1, 300), (3024, 3), (4032, 224), (3024, 168),
                                                                      (4032, 5000), (17, 17)]:
        b, k = H.resample_coeffs(n_in, n_out, f)
        rb, rk = coeffs_restated(n_in, n_out, f)
        assert np.array_equal(b, rb) and np.array_equal(k, rk), (name, n_in, n_out)
        assert b[:, 1].sum() == len(k) and (b[:, 0] >= 0).all() and (b[:, 0] + b[:, 1] <= n_in).all()


@pytest.mark.parametrize("name", list(FILTERS))
def test_first_used_row_of_a_whole_image_is_zero(name):
    """With the whole image as the source box, output 0 always starts at input 0 ((int)(center - support + 0.5) < 1), so the
    shift of the vertical bounds by the first used row is 0 and the horizontal pass always starts at row 0; the kernels
    keep the shift because the definition has it."""
    f = FILTERS[name]
    for n_in in (1, 2, 3, 17, 224, 3024, 4032):
        for n_out in (1, 2, 3, 5, 224, 1000, 3023, 5000):
            assert H.resample_coeffs(n_in, n_out, f)[0][0, 0] == 0, (name, n_in, n_out)


@pytest.mark.parametrize("mistake", ["vertical_first", "no_clip", "float32"])
def test_each_mistake_in_the_restatement_is_caught(mistake):
    """Over the cases of the test above (RGB), each mistake makes some output differ from Pillow."""
    caught = 0
    for name, f in FILTERS.items():
        rng = np.random.default_rng(f * 10)
        for h, w, W, Hh in random_cases(f, 40):
            a = image(rng, h, w, "RGB")
            if not np.array_equal(resize_restated(a, (W, Hh), f, mistake), pillow(a, (W, Hh), f)):
                caught += 1
    assert caught > 0, mistake


def test_pillow_4032x3024_axes_to_224x168():
    """The two axes of the serving-size downscale 4032 x 3024 -> 224 x 168 (bicubic and Lanczos), on strips of a 12 MP
    image, through the library's tables."""
    rng = np.random.default_rng(5)
    for f in (3, 1):
        for shape, size in (((24, 4032, 3), (224, 24)), ((3024, 24, 3), (24, 168)), ((300, 4032, 3), (224, 17))):
            a = image(rng, shape[0], shape[1], "RGB")
            assert np.array_equal(resize_restated(a, size, f), pillow(a, size, f)), (f, shape, size)


def test_invalid_tables_are_rejected():
    lib = K.load()
    for n_in, n_out, f in [(0, 5, 3), (5, 0, 3), (5, 32769, 3), (5, 5, 0), (5, 5, 6)]:
        assert lib.heic_b200_resample_coeffs(n_in, n_out, f, None, None, 0) == K.HEIC_E_INVALID_ARG, (n_in, n_out, f)
    assert lib.heic_b200_resample_coeffs(5, 32768, 3, None, None, 0) > 0
    small = (K.i32 * 1)()
    assert lib.heic_b200_resample_coeffs(100, 10, 3, None, small, 1) == K.HEIC_E_INVALID_ARG


def test_resize_struct_and_exports(built):
    src = r'''
#include <stdio.h>
#include "heic_b200.h"
int main(void) { printf("%zu %d %d %d %d %d\n", sizeof(heic_resize), HEIC_RESAMPLE_LANCZOS, HEIC_RESAMPLE_BILINEAR,
  HEIC_RESAMPLE_BICUBIC, HEIC_RESAMPLE_BOX, HEIC_RESAMPLE_HAMMING); return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "s.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I" + os.path.join(ROOT, "include"), "-o", os.path.join(d, "s"), os.path.join(d, "s.c")])
        vals = [int(x) for x in subprocess.check_output([os.path.join(d, "s")]).split()]
    assert vals == [C.sizeof(K.Resize), 1, 2, 3, 4, 5] and vals[0] == 12
    assert {name: int(getattr(Image.Resampling, name)) for name in FILTERS} == FILTERS  # Pillow's numbers
    lib = C.CDLL(K.LIB_PATH)
    for n in ("heic_b200_decode_grids_resized", "heic_b200_decode_grids_submit_resized", "heic_b200_batch_create_resized",
              "heic_b200_resample_coeffs"):
        assert hasattr(lib, n), n


def test_output_size_helper(heic_file):
    img = heic_file.primary
    assert H._canvas(img, resize=(224, 224)) == (224, 224)
    assert H._canvas(img, reduce=4, resize=(1000, 750)) == (1000, 750)
    assert H._canvas(img, resize=None, reduce=4) == (1008, 756)
    assert H._canvas(None, transform=K.ImageTransform(0, 0, 4032, 3024, 1), resize=(5000, 3000)) == (5000, 3000)
    assert H._resize_list((224, 224), 2) == [(224, 224)] * 2
    assert H._resize_list([None, (3, 4)], 2) == [None, (3, 4)]
    assert H._resize_list(None, 3) == [None] * 3
    with pytest.raises(ValueError):
        H._resize_list([(3, 4)], 2)
    assert H._resample_list(Image.Resampling.LANCZOS, 2) == [1, 1]
    assert H._resample_list([Image.Resampling.BOX, 5], 2) == [4, 5]
