"""Box-reduced RGB on the GPU, byte-equal to Pillow: every output is Image.fromarray(T).reduce(k) of the oracle's RGB T
under the same transform.  The fixture under every orientation and several crops through the three entry points,
conformance-cropped grids, the monochrome auxiliary image, a batch that mixes factors and geometries, invalid factors, a
bench-scale resident batch, and the whole file with SAO applied outside the colour kernel."""
import os
import subprocess
import sys

import numpy as np
import pytest
from PIL import Image

import heif_b200 as H
from heif_b200 import _capi as K
from oracle import oracle_py as O
from tests.test_geometry import apply_transform
from tests.test_gpu_geometry import CONF_WINDOWS, Grid, _conf_pics, expected_grid, fixture_rgb  # noqa: F401

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CROPS = {
    "canvas": (0, 0, 4032, 3024),
    "odd_origin": (333, 217, 1001, 777),
    "four_tiles": (500, 490, 30, 41),
    "column": (1999, 0, 1, 3024),
}
FACTORS = (2, 3, 4, 7, 8, 16)


def reduced(rgb, t, k):
    return np.asarray(Image.fromarray(np.ascontiguousarray(apply_transform(rgb, t))).reduce(k))


@pytest.fixture(scope="module")
def expected(fixture_rgb):
    cache = {}

    def get(crop, o, k):
        if (crop, o, k) not in cache:
            cache[(crop, o, k)] = reduced(fixture_rgb, K.ImageTransform(*CROPS[crop], o), k)
        return cache[(crop, o, k)]

    return get


@pytest.mark.parametrize("crop", list(CROPS), ids=list(CROPS))
def test_fixture_orientations_crops_and_factors(decoder, heic_file, expected, crop):
    img = heic_file.primary
    xfs = [K.ImageTransform(*CROPS[crop], o) for o in range(8)]
    for k in FACTORS:
        # decode_grids: one call per output shape
        for parity in (0, 1):
            sel = [o for o in range(8) if (o & 1) == parity]
            got = decoder.decode_grids([img] * 4, transforms=[xfs[o] for o in sel], reduce=k)
            for i, o in enumerate(sel):
                assert np.array_equal(got[i], expected(crop, o, k)), (crop, o, k)
        # the submit path
        out = np.empty((4,) + expected(crop, 0, k).shape, np.uint8)
        decoder.wait_job(decoder.submit_grids([img] * 4, out, transforms=[xfs[o] for o in (0, 2, 4, 6)], reduce=k))
        for i, o in enumerate((0, 2, 4, 6)):
            assert np.array_equal(out[i], expected(crop, o, k)), (crop, o, k)
    # a resident batch of every orientation and factor
    items = [(o, k) for k in FACTORS for o in range(8)]
    with decoder.batch([img] * len(items), transforms=[xfs[o] for o, _ in items], reduce=[k for _, k in items]) as b:
        b.decode()
        for i, (o, k) in enumerate(items):
            assert np.array_equal(b.download_image(i), expected(crop, o, k)), (crop, o, k)
    # download_rgb of a batch of equal output shapes
    with decoder.batch([img] * 4, transforms=[xfs[o] for o in (1, 3, 5, 7)], reduce=3) as b:
        b.decode()
        got = b.download_rgb()
        for i, o in enumerate((1, 3, 5, 7)):
            assert np.array_equal(got[i], expected(crop, o, 3)), (crop, o)


@pytest.mark.parametrize("chroma", [1, 0], ids=["420", "400"])
def test_conformance_cropped_grids(decoder, chroma):
    pics = _conf_pics(chroma, CONF_WINDOWS["all"], 6, seed0=60)
    tw, th = H.tile_size(pics[0].desc)
    canvas = (3 * tw - 5, 2 * th - 3)
    grid = Grid(pics, 2, 3, canvas)
    _, rgb = expected_grid(pics, 2, 3, canvas)
    for k in (2, 5):
        for t in (K.ImageTransform(0, 0, *canvas, 0), K.ImageTransform(1, 2, canvas[0] - 4, canvas[1] - 3, 5),
                  K.ImageTransform(3, 1, canvas[0] - 7, canvas[1] - 2, 2)):
            exp = reduced(rgb, t, k)
            assert np.array_equal(decoder.decode_grids([grid.desc], transforms=[t], reduce=k)[0], exp), (k, t.orientation)
            with decoder.batch([grid.desc], transforms=[t], reduce=k) as b:
                b.decode()
                assert np.array_equal(b.download_image(0), exp), (k, t.orientation)


def test_monochrome_aux_image(decoder, heic_file):
    img = heic_file.aux_images[0]
    assert img.sps.chroma_format_idc == 0
    td = img.tiles[0]
    y = O.decode_picture(img.sps, img.pps, td.header, (td.rbsp, td.rbsp_len), intermediates=False)["plane"][0]
    w, h = img.output_width, img.output_height
    ye = np.zeros(((h + 1) & ~1, (w + 1) & ~1), np.uint8)
    ye[:h, :w] = y[:h, :w]
    neutral = np.full(ye.size // 4, 128, np.uint8)
    rgb = O.color_stitch(np.concatenate([ye.ravel(), neutral, neutral]), 1, 1, ye.shape[1], ye.shape[0], w, h,
                         img.sps.video_full_range_flag, img.sps.matrix_coeffs)
    for k in (2, 5):
        for o in (0, 3):
            t = K.ImageTransform(0, 0, w, h, o)
            assert np.array_equal(decoder.decode_grids([img], transforms=[t], reduce=k)[0], reduced(rgb, t, k)), (k, o)


def test_mixed_factors_in_one_batch(decoder, heic_file, fixture_rgb):
    """Factors 1 (the _transformed output, byte for byte), 2, 4, 5 and 16 with different geometries in one resident batch
    and one submitted call: the colour stage groups images only when their factor is equal."""
    img = heic_file.primary
    pics = _conf_pics(1, CONF_WINDOWS["all"], 6, seed0=70)
    tw, th = H.tile_size(pics[0].desc)
    canvas = (3 * tw - 5, 2 * th - 3)
    grid = Grid(pics, 2, 3, canvas)
    _, grid_rgb = expected_grid(pics, 2, 3, canvas)
    full = K.ImageTransform(0, 0, 4032, 3024, 0)
    items = [(img, full, 1), (img, full, 2), (img, full, 2), (img, full, 4), (img, K.ImageTransform(333, 217, 1001, 777, 6), 5),
             (grid.desc, K.ImageTransform(0, 0, *canvas, 0), 2), (img, K.ImageTransform(0, 0, 4032, 3024, 1), 1),
             (img, K.ImageTransform(8, 2, 4000, 3000, 7), 16), (grid.desc, K.ImageTransform(1, 1, canvas[0] - 2, canvas[1] - 2, 3), 1),
             (img, full, 1)]
    exps = [reduced(fixture_rgb if d is img else grid_rgb, t, k) for d, t, k in items]
    with decoder.batch([d for d, _, _ in items], transforms=[t for _, t, _ in items], reduce=[k for _, _, k in items]) as b:
        b.decode()
        for i, e in enumerate(exps):
            assert np.array_equal(b.download_image(i), e), i
    # factor 1 is today's transformed output
    plain = decoder.decode_grids([img, img], transforms=[full, full])
    assert np.array_equal(plain[0], exps[0])
    # one call whose outputs share a shape: 4032 x 3024 by 2 and 2016 x 1512 as it is
    aux = heic_file.aux_images[0]
    aux_id = K.ImageTransform(0, 0, aux.output_width, aux.output_height, 0)
    out = np.empty((3, 1512, 2016, 3), np.uint8)
    decoder.wait_job(decoder.submit_grids([img, aux, img], out, transforms=[full, aux_id, full], reduce=[2, 1, 2]))
    assert np.array_equal(out[0], exps[1]) and np.array_equal(out[2], exps[1])
    assert np.array_equal(out[1], decoder.decode_grids([aux])[0])


def test_invalid_factor_is_rejected_before_anything_runs(decoder, heic_file):
    img = heic_file.primary
    full = K.ImageTransform(0, 0, 4032, 3024, 0)
    for bad in (0, 17):
        n = decoder.launch_count()
        out = np.full((2, 1512, 2016, 3), 7, np.uint8)
        with pytest.raises(H.HeicError) as e:
            decoder.decode_grids([img, img], out=out, transforms=[full, full], reduce=bad)
        assert e.value.code == K.HEIC_E_INVALID_ARG
        with pytest.raises(H.HeicError) as e:
            decoder.submit_grids([img, img], out, transforms=[full, full], reduce=[2, bad])
        assert e.value.code == K.HEIC_E_INVALID_ARG
        with pytest.raises(H.HeicError) as e:
            decoder.batch([img, img], transforms=[full, full], reduce=[2, bad])
        assert e.value.code == K.HEIC_E_INVALID_ARG
        assert decoder.launch_count() == n
        assert (out == 7).all()


def test_rgb_layout_of_a_reduced_batch(decoder, heic_file):
    img = heic_file.primary
    with decoder.batch([img] * 3, transforms=[(0, 0, 4032, 3024, 0), (0, 0, 4032, 3024, 1), (5, 0, 1001, 777, 0)],
                       reduce=[4, 4, 3]) as b:
        _, pitch, stride = b.rgb_layout()
        # widest reduced row (1008 x 3 bytes, to 16) and tallest reduced image (1008 rows of the turned one)
        assert pitch == 3024 and stride == (3024 * 1008 + 255) // 256 * 256
    with decoder.batch([img], transforms=[(0, 0, 4032, 3024, 0)], reduce=7) as b:
        _, pitch, stride = b.rgb_layout()
        assert pitch == (576 * 3 + 15) // 16 * 16 and stride == (pitch * 432 + 255) // 256 * 256


def test_bench_scale_batch_reduced(built, heic_file):
    """64 pool images (3072 tiles) through the throughput path at k = 4; 8 random images against the oracle."""
    import bench
    from tests.synth import pool as P

    pool = P.build_pool(heic_file, 128)
    n_img = 64
    images, keep, ids = P.compose_images(pool, heic_file.primary, range(n_img), 1)
    chk = np.sort(np.random.default_rng(4).choice(n_img, 8, replace=False))
    planes = np.zeros((len(chk), 48, bench.TILE_BYTES), np.uint8)
    rgb = np.zeros((len(chk), bench.OUT_H, bench.OUT_W, 3), np.uint8)
    bench.CpuDecoder(pool, heic_file.primary, 8).decode(ids[chk], planes, rgb)
    full = K.ImageTransform(0, 0, 4032, 3024, 0)
    with H.HeicDecoder(device=0) as dec:
        with dec.batch(images, transforms=[full] * n_img, reduce=4) as b:
            b.decode()
            b.sync()
            st = b.status()
            assert all(st[i].code == 0 for i in range(b.n_tiles))
            for j, i in enumerate(chk):
                assert np.array_equal(b.download_image(int(i)), reduced(rgb[j], full, 4)), f"image {i}"


def test_reduction_without_fused_sao(built):
    """The same with SAO written to its own planes before the colour kernel (HEIC_B200_FUSE_SAO=0, read once per process,
    hence the subprocess)."""
    e = dict(os.environ)
    e["HEIC_B200_FUSE_SAO"] = "0"
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_reduce.py", "-x", "-q", "-m", "gpu", "-p", "no:cacheprovider",
                        "-k", "not without_fused_sao and not bench_scale"], cwd=ROOT, env=e, capture_output=True, text=True,
                       timeout=1800)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
