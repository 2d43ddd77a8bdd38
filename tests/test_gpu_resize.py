"""Resized RGB on the GPU, byte-equal to Pillow: every output is Image.fromarray(T).resize(size, f, reducing_gap=None) of
the oracle's RGB T under the same transform and box reduction.  The fixture under four orientations with the whole canvas
and an odd-origin crop at down-, up- and one-axis sizes, all five filters through decode_grids, submit_grids and a
resident batch, reduce(k) then resize, conformance-cropped 4:2:0 / 4:0:0 grids, the monochrome auxiliary image, calls that
mix sizes, filters, factors, transforms and unresized images, a call cut into several pipeline chunks, a bench-scale
batch, invalid resizes, and the whole file with SAO applied outside the colour kernel."""
import ctypes as C
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

LANCZOS, BILINEAR, BICUBIC, BOX, HAMMING = 1, 2, 3, 4, 5
FILTERS = (LANCZOS, BILINEAR, BICUBIC, BOX, HAMMING)
CROPS = {"canvas": (0, 0, 4032, 3024), "odd_origin": (333, 217, 1001, 777)}
ORIENTATIONS = (0, 1, 5, 6)


def resized(rgb, t, size, f, k=1):
    a = Image.fromarray(np.ascontiguousarray(apply_transform(rgb, t)))
    if k > 1:
        a = a.reduce(k)
    return np.asarray(a.resize(tuple(size), Image.Resampling(f), reducing_gap=None))


def size_of(t, k=1):
    w, h = (t.crop_h, t.crop_w) if t.orientation & 1 else (t.crop_w, t.crop_h)
    return -(-w // k), -(-h // k)


@pytest.mark.parametrize("crop", list(CROPS), ids=list(CROPS))
def test_fixture_orientations_and_sizes(decoder, heic_file, fixture_rgb, crop):
    """decode_grids, one call per output size with the four orientations: downscales, an upscale, a 1-pixel-high strip,
    one side equal to the source and the source size (which is the unresized output)."""
    img = heic_file.primary
    xfs = [K.ImageTransform(*CROPS[crop], o) for o in ORIENTATIONS]
    for size, f in (((224, 224), BICUBIC), ((1000, 750), LANCZOS), ((4031, 1), BILINEAR), ((5000, 3000), HAMMING)):
        got = decoder.decode_grids([img] * 4, transforms=xfs, resize=size, resample=f)
        for i, t in enumerate(xfs):
            assert np.array_equal(got[i], resized(fixture_rgb, t, size, f)), (crop, t.orientation, size, f)
    for parity in (0, 1):
        sel = [t for t in xfs if (t.orientation & 1) == parity]
        w, h = size_of(sel[0])
        for size, f in (((w, 500), BOX), ((640, h), LANCZOS), ((w, h), BICUBIC)):
            got = decoder.decode_grids([img] * 2, transforms=sel, resize=size, resample=f)
            for i, t in enumerate(sel):
                assert np.array_equal(got[i], resized(fixture_rgb, t, size, f)), (crop, t.orientation, size, f)
        plain = decoder.decode_grids([img] * 2, transforms=sel)
        assert np.array_equal(got, plain)  # resize to the source size = no resize


def test_wide_horizontal_spans(decoder, heic_file, fixture_rgb):
    """Horizontal downscales whose band of 32 outputs needs more shared memory than resample_h_kernel takes (4032 -> 1 and
    4032 -> 16 under Lanczos: resample_h_wide_kernel) and ones just under the limit (4032 -> 32 Lanczos, ~197 KB;
    4032 -> 48 bicubic, ~108 KB)."""
    img = heic_file.primary
    xfs = [K.ImageTransform(0, 0, 4032, 3024, o) for o in (0, 6)]
    for size, f in (((1, 64), LANCZOS), ((16, 300), LANCZOS), ((32, 24), LANCZOS), ((48, 36), BICUBIC), ((1, 3024), BOX)):
        got = decoder.decode_grids([img] * 2, transforms=xfs, resize=size, resample=f)
        for i, t in enumerate(xfs):
            assert np.array_equal(got[i], resized(fixture_rgb, t, size, f)), (t.orientation, size, f)


def test_all_filters_through_every_entry_point(decoder, heic_file, fixture_rgb):
    img = heic_file.primary
    xfs = [K.ImageTransform(*CROPS["odd_origin"], o) for o in (0, 6)]
    for f in FILTERS:
        exp = [resized(fixture_rgb, t, (224, 160), f) for t in xfs]
        got = decoder.decode_grids([img] * 2, transforms=xfs, resize=(224, 160), resample=f)
        assert all(np.array_equal(g, e) for g, e in zip(got, exp)), f
        out = np.empty((2, 160, 224, 3), np.uint8)
        decoder.wait_job(decoder.submit_grids([img] * 2, out, transforms=xfs, resize=(224, 160), resample=f))
        assert all(np.array_equal(g, e) for g, e in zip(out, exp)), f
        with decoder.batch([img] * 2, transforms=xfs, resize=(224, 160), resample=Image.Resampling(f)) as b:
            b.decode()
            assert np.array_equal(b.download_image(1), exp[1]), f
            got = b.download_rgb()
            assert all(np.array_equal(g, e) for g, e in zip(got, exp)), f
    # the HeicFile convenience call
    assert np.array_equal(decoder.decode(heic_file, resize=(300, 200), resample=LANCZOS),
                          resized(fixture_rgb, K.ImageTransform(0, 0, 4032, 3024, 0), (300, 200), LANCZOS))


def test_reduce_then_resize(decoder, heic_file, fixture_rgb):
    img = heic_file.primary
    for k in (2, 4):
        for t, size, f in ((K.ImageTransform(0, 0, 4032, 3024, 1), (224, 224), BICUBIC),
                           (K.ImageTransform(*CROPS["odd_origin"], 5), (301, 199), LANCZOS),
                           (K.ImageTransform(0, 0, 4032, 3024, 0), (1500, 1100), BILINEAR)):
            exp = resized(fixture_rgb, t, size, f, k)
            assert np.array_equal(decoder.decode_grids([img], transforms=[t], reduce=k, resize=size, resample=f)[0], exp), (k, size)
            with decoder.batch([img], transforms=[t], reduce=k, resize=size, resample=f) as b:
                b.decode()
                assert np.array_equal(b.download_image(0), exp), (k, size)


@pytest.mark.parametrize("chroma", [1, 0], ids=["420", "400"])
def test_conformance_cropped_grids(decoder, chroma):
    pics = _conf_pics(chroma, CONF_WINDOWS["all"], 6, seed0=80)
    tw, th = H.tile_size(pics[0].desc)
    canvas = (3 * tw - 5, 2 * th - 3)
    grid = Grid(pics, 2, 3, canvas)
    _, rgb = expected_grid(pics, 2, 3, canvas)
    for t in (K.ImageTransform(0, 0, *canvas, 0), K.ImageTransform(1, 2, canvas[0] - 4, canvas[1] - 3, 5)):
        for k, size, f in ((1, (37, 23), LANCZOS), (1, (500, 301), BICUBIC), (2, (40, 90), HAMMING), (1, (canvas[1], 7), BOX)):
            exp = resized(rgb, t, size, f, k)
            assert np.array_equal(decoder.decode_grids([grid.desc], transforms=[t], reduce=k, resize=size, resample=f)[0], exp), (k, size)
            with decoder.batch([grid.desc], transforms=[t], reduce=k, resize=size, resample=f) as b:
                b.decode()
                assert np.array_equal(b.download_image(0), exp), (k, size)


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
    for o, k, size, f in ((0, 1, (224, 224), BICUBIC), (3, 2, (100, 333), LANCZOS), (0, 1, (3000, 2000), BILINEAR)):
        t = K.ImageTransform(0, 0, w, h, o)
        got = decoder.decode_grids([img], transforms=[t], reduce=k, resize=size, resample=f)[0]
        assert np.array_equal(got, resized(rgb, t, size, f, k)), (o, k, size)


def _mixed_items(img, grid_desc, canvas):
    full = K.ImageTransform(0, 0, 4032, 3024, 0)
    return [(img, full, 1, None, BICUBIC), (img, full, 1, (224, 224), BICUBIC), (img, full, 1, (224, 224), BICUBIC),
            (img, K.ImageTransform(0, 0, 4032, 3024, 1), 4, (224, 224), LANCZOS), (img, full, 2, None, BICUBIC),
            (grid_desc, K.ImageTransform(0, 0, *canvas, 0), 1, (64, 48), HAMMING), (img, full, 1, (4032, 17), BOX),
            (img, K.ImageTransform(333, 217, 1001, 777, 6), 1, (1000, 750), BILINEAR), (img, full, 1, (224, 224), LANCZOS),
            (grid_desc, K.ImageTransform(1, 1, canvas[0] - 2, canvas[1] - 2, 3), 1, None, BICUBIC), (img, full, 1, (224, 224), BICUBIC)]


def test_mixed_batch_and_call(decoder, heic_file, fixture_rgb):
    """Sizes, filters, factors, transforms and unresized images in one resident batch; then one submitted call whose outputs
    share a shape (224 x 224 from different sources, filters and factors, and an image that is 224 x 224 unresized)."""
    img = heic_file.primary
    pics = _conf_pics(1, CONF_WINDOWS["all"], 6, seed0=90)
    tw, th = H.tile_size(pics[0].desc)
    canvas = (3 * tw - 5, 2 * th - 3)
    grid = Grid(pics, 2, 3, canvas)
    _, grid_rgb = expected_grid(pics, 2, 3, canvas)
    items = _mixed_items(img, grid.desc, canvas)

    def expect(d, t, k, size, f):
        src = fixture_rgb if d is img else grid_rgb
        if size is None:
            a = Image.fromarray(np.ascontiguousarray(apply_transform(src, t)))
            return np.asarray(a.reduce(k) if k > 1 else a)
        return resized(src, t, size, f, k)

    exps = [expect(*it) for it in items]
    with decoder.batch([d for d, *_ in items], transforms=[t for _, t, *_ in items], reduce=[k for _, _, k, _, _ in items],
                       resize=[s for *_, s, _ in items], resample=[f for *_, f in items]) as b:
        b.decode()
        for i, e in enumerate(exps):
            assert np.array_equal(b.download_image(i), e), i
    sel = [1, 3, 8, 10]
    out = np.empty((len(sel), 224, 224, 3), np.uint8)
    decoder.wait_job(decoder.submit_grids([items[i][0] for i in sel], out, transforms=[items[i][1] for i in sel],
                                          reduce=[items[i][2] for i in sel], resize=[items[i][3] for i in sel],
                                          resample=[items[i][4] for i in sel]))
    for j, i in enumerate(sel):
        assert np.array_equal(out[j], exps[i]), i


def test_call_cut_into_chunks(built, heic_file, fixture_rgb):
    """Nine images through a context that cuts calls into chunks of two images (HEIC_B200_PIPE_CHUNK, read when the context
    is created): resized and unresized images share chunks, and the chunks reuse their slots' buffers."""
    img = heic_file.primary
    old = os.environ.get("HEIC_B200_PIPE_CHUNK")
    os.environ["HEIC_B200_PIPE_CHUNK"] = "2"
    try:
        dec = H.HeicDecoder(device=0)
    finally:
        if old is None:
            os.environ.pop("HEIC_B200_PIPE_CHUNK")
        else:
            os.environ["HEIC_B200_PIPE_CHUNK"] = old
    with dec:
        xfs = [K.ImageTransform(0, 0, 4032, 3024, o) for o in (0, 1, 5, 6, 0, 1, 5, 6, 0)]
        ks = [1, 2, 1, 4, 1, 1, 2, 1, 1]
        filters = [BICUBIC, LANCZOS, BOX, HAMMING, BILINEAR, BICUBIC, LANCZOS, BICUBIC, BICUBIC]
        sizes = [(320, 240)] * 9
        sizes[4] = None
        xfs[4] = K.ImageTransform(1000, 1000, 320, 240, 0)  # 320 x 240 without a resize
        for _ in range(2):
            got = dec.decode_grids([img] * 9, transforms=xfs, reduce=ks, resize=sizes, resample=filters)
            for i in range(9):
                exp = np.asarray(Image.fromarray(np.ascontiguousarray(apply_transform(fixture_rgb, xfs[i])))) if sizes[i] is None \
                    else resized(fixture_rgb, xfs[i], sizes[i], filters[i], ks[i])
                assert np.array_equal(got[i], exp), i


def test_invalid_resize_is_rejected_before_anything_runs(decoder, heic_file):
    img = heic_file.primary
    full = K.ImageTransform(0, 0, 4032, 3024, 0)
    arr = H._desc_array([img, img])
    st = (K.TileStatus * (2 * img.n_tiles))()
    for bad, f in (((0, 224), BICUBIC), ((224, 0), BICUBIC), ((32769, 224), BICUBIC), ((224, 32769), LANCZOS), ((224, 224), 0),
                   ((224, 224), 6)):
        n = decoder.launch_count()
        out = np.full((2, 224, 224, 3), 7, np.uint8)
        # the C ABI directly: the Python size helper would refuse the mismatched output shapes first
        rs = H._resize_array([(224, 224), bad], [BICUBIC, f])
        xf, ks = H._transform_array([full, full], 2), H._reduce_array([1, 1])
        rc = decoder._lib.heic_b200_decode_grids_resized(decoder._h, arr, xf, ks, rs, 2, out.ctypes.data, out.strides[1],
                                                         out.strides[0], st)
        assert rc == K.HEIC_E_INVALID_ARG, (bad, f)
        job = C.c_void_p()
        rc = decoder._lib.heic_b200_decode_grids_submit_resized(decoder._h, arr, xf, ks, rs, 2, out.ctypes.data, out.strides[1],
                                                                out.strides[0], st, C.byref(job))
        assert rc == K.HEIC_E_INVALID_ARG, (bad, f)
        if bad == (224, 224):
            with pytest.raises(H.HeicError) as e:
                decoder.decode_grids([img, img], out=out, transforms=[full, full], resize=(224, 224), resample=[BICUBIC, f])
            assert e.value.code == K.HEIC_E_INVALID_ARG
        with pytest.raises(H.HeicError) as e:
            decoder.batch([img, img], transforms=[full, full], resize=[(224, 224), bad], resample=[BICUBIC, f])
        assert e.value.code == K.HEIC_E_INVALID_ARG
        assert decoder.launch_count() == n
        assert (out == 7).all()


def test_rgb_layout_of_a_resized_batch(decoder, heic_file):
    img = heic_file.primary
    with decoder.batch([img] * 3, transforms=[(0, 0, 4032, 3024, 0)] * 3, resize=[(224, 224), (100, 300), None]) as b:
        _, pitch, stride = b.rgb_layout()
        assert pitch == (4032 * 3 + 15) // 16 * 16 and stride == (pitch * 3024 + 255) // 256 * 256  # the unresized image
    with decoder.batch([img] * 2, transforms=[(0, 0, 4032, 3024, 0)] * 2, resize=(224, 224)) as b:
        _, pitch, stride = b.rgb_layout()
        assert pitch == 672 and stride == 672 * 224


def test_bench_scale_batch_resized(built, heic_file):
    """64 pool images (3072 tiles) through the throughput path at 224 x 224 BICUBIC; 8 random images against the oracle."""
    import bench
    from tests.synth import pool as P

    pool = P.build_pool(heic_file, 128)
    n_img = 64
    images, keep, ids = P.compose_images(pool, heic_file.primary, range(n_img), 1)
    chk = np.sort(np.random.default_rng(5).choice(n_img, 8, replace=False))
    planes = np.zeros((len(chk), 48, bench.TILE_BYTES), np.uint8)
    rgb = np.zeros((len(chk), bench.OUT_H, bench.OUT_W, 3), np.uint8)
    bench.CpuDecoder(pool, heic_file.primary, 8).decode(ids[chk], planes, rgb)
    full = K.ImageTransform(0, 0, 4032, 3024, 0)
    with H.HeicDecoder(device=0) as dec:
        with dec.batch(images, transforms=[full] * n_img, resize=(224, 224), resample=BICUBIC) as b:
            b.decode()
            b.sync()
            st = b.status()
            assert all(st[i].code == 0 for i in range(b.n_tiles))
            for j, i in enumerate(chk):
                assert np.array_equal(b.download_image(int(i)), resized(rgb[j], full, (224, 224), BICUBIC)), f"image {i}"


def test_resize_without_fused_sao(built):
    """The same with SAO written to its own planes before the colour kernel (HEIC_B200_FUSE_SAO=0, read once per process,
    hence the subprocess)."""
    e = dict(os.environ)
    e["HEIC_B200_FUSE_SAO"] = "0"
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_resize.py", "-x", "-q", "-m", "gpu", "-p", "no:cacheprovider",
                        "-k", "not without_fused_sao and not bench_scale"], cwd=ROOT, env=e, capture_output=True, text=True,
                       timeout=2400)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
