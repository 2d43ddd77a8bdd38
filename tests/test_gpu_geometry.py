"""Output geometry on the GPU, bit-exact: the fixture under every orientation and several crops (three entry points),
conformance-cropped synthetic pictures and grids (RGB and planar), a batch that mixes geometries, and HEIF files with
clap / irot / imir in different orders.  Also the whole file with SAO applied outside the colour kernel."""
import os
import subprocess
import sys

import numpy as np
import pytest

import heif_b200 as H
from heif_b200 import _capi as K
from oracle import oracle_py as O
from tests.synth import conf_window
from tests.synth import heif_writer as W
from tests.synth import synth
from tests.test_geometry import apply_property, apply_transform

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CROPS = {
    "canvas": None,
    "inset_1": (1, 1, 4031, 3023),
    "odd_origin": (333, 217, 1001, 777),      # width not a multiple of 8
    "column": (1999, 0, 1, 3024),
    "four_tiles": (500, 490, 30, 41),         # straddles the corner of four 512 x 512 tiles
}


@pytest.fixture(scope="module")
def fixture_rgb(heic_file):
    img = heic_file.primary
    planes = []
    for t in range(img.n_tiles):
        td = img.tiles[t]
        r = O.decode_picture(img.sps, img.pps, td.header, (td.rbsp, td.rbsp_len), intermediates=False)
        planes.append(np.concatenate([p.ravel() for p in r["plane"]]))
    return O.color_stitch(np.concatenate(planes), img.grid_rows, img.grid_cols, 512, 512, img.output_width, img.output_height,
                          img.sps.video_full_range_flag, img.sps.matrix_coeffs)


def _xf(crop, o):
    return K.ImageTransform(*(crop or (0, 0, 4032, 3024)), o)


@pytest.mark.parametrize("crop", list(CROPS), ids=list(CROPS))
def test_fixture_orientations_and_crops(decoder, heic_file, fixture_rgb, crop):
    img = heic_file.primary
    xfs = [_xf(CROPS[crop], o) for o in range(8)]
    exp = [apply_transform(fixture_rgb, t) for t in xfs]
    # decode_grids_transformed: one call per output shape
    for parity in (0, 1):
        sel = [o for o in range(8) if (o & 1) == parity]
        got = decoder.decode_grids([img] * len(sel), transforms=[xfs[o] for o in sel])
        for k, o in enumerate(sel):
            assert np.array_equal(got[k], exp[o]), (crop, o)
    # the submit path
    out = np.empty((4,) + exp[1].shape, np.uint8)
    job = decoder.submit_grids([img] * 4, out, transforms=[xfs[o] for o in (1, 3, 5, 7)])
    decoder.wait_job(job)
    for k, o in enumerate((1, 3, 5, 7)):
        assert np.array_equal(out[k], exp[o]), (crop, o)
    # a resident batch
    with decoder.batch([img] * 8, transforms=xfs) as b:
        b.decode()
        b.sync()
        for o in range(8):
            assert np.array_equal(b.download_image(o), exp[o]), (crop, o)


def test_invalid_transform_is_rejected_before_anything_runs(decoder, heic_file):
    img = heic_file.primary
    for t in ((0, 0, 4033, 3024, 0), (1, 0, 4032, 3024, 0), (0, 0, 4032, 3024, 8), (0, 0, 0, 3024, 0)):
        with pytest.raises(H.HeicError) as e:
            decoder.decode_grids([img], transforms=[t])
        assert e.value.code == K.HEIC_E_INVALID_ARG
        with pytest.raises(H.HeicError) as e:
            decoder.batch([img], transforms=[t])
        assert e.value.code == K.HEIC_E_INVALID_ARG


CONF_WINDOWS = {"left": (1, 0, 0, 0), "right": (0, 3, 0, 0), "right_by_8": (0, 4, 0, 0), "top": (0, 0, 1, 0),
                "bottom": (0, 0, 0, 3), "all": (1, 2, 3, 1)}


class Grid:
    """rows x cols synthetic pictures of one configuration (so one SPS / PPS) as a grid image with a given canvas."""

    def __init__(self, pics, rows, cols, canvas):
        self.pics = pics
        self._tiles = (K.TileDesc * len(pics))()
        for i, p in enumerate(pics):
            self._tiles[i] = p.tile
        d = K.ImageDesc()
        d.sps, d.pps = pics[0].sps, pics[0].pps
        d.grid_rows, d.grid_cols = rows, cols
        d.output_width, d.output_height = canvas
        d.n_tiles = len(pics)
        d.tiles = K.C.cast(self._tiles, K.C.POINTER(K.TileDesc))
        self.desc = d


def _planes(pic):
    t = pic.tile
    return O.decode_picture(pic.sps, pic.pps, t.header, (t.rbsp, t.rbsp_len), intermediates=False)["plane"]


def expected_grid(pics, rows, cols, canvas):
    """Oracle planes cut to each tile's conformance window, stitched in numpy and cropped to the canvas: (Y, Cb, Cr)
    (chroma None for 4:0:0), and the RGB of O.color_stitch over them."""
    s = pics[0].sps
    sub = 2 if s.chroma_format_idc == 1 else 1
    l, t = sub * s.conf_win_left_offset, sub * s.conf_win_top_offset
    tw, th = H.tile_size(pics[0].desc)
    cw, ch = canvas
    planes = [_planes(p) for p in pics]
    y = np.block([[planes[r * cols + c][0][t:t + th, l:l + tw] for c in range(cols)] for r in range(rows)])[:ch, :cw]
    fr, mc = s.video_full_range_flag, s.matrix_coeffs
    if sub == 1:  # monochrome: one even-sized tile of the stitched luma with neutral chroma
        ye = np.zeros(((ch + 1) & ~1, (cw + 1) & ~1), np.uint8)
        ye[:ch, :cw] = y
        neutral = np.full(ye.size // 4, 128, np.uint8)
        rgb = O.color_stitch(np.concatenate([ye.ravel(), neutral, neutral]), 1, 1, ye.shape[1], ye.shape[0], cw, ch, fr, mc)
        return (y, None, None), rgb
    cut = [[pl[0][t:t + th, l:l + tw]] + [pl[c][t // 2:t // 2 + th // 2, l // 2:l // 2 + tw // 2] for c in (1, 2)] for pl in planes]
    rgb = O.color_stitch(np.concatenate([np.concatenate([a.ravel() for a in tile]) for tile in cut]), rows, cols, tw, th, cw, ch, fr, mc)
    chroma = [np.block([[cut[r * cols + c][k] for c in range(cols)] for r in range(rows)])[:(ch + 1) // 2, :(cw + 1) // 2] for k in (1, 2)]
    return (y, chroma[0], chroma[1]), rgb


def _conf_pics(chroma, win, n, seed0=20):
    return [conf_window.encode(seed0 + i, win, width=96, height=64, chroma_format_idc=chroma) for i in range(n)]


@pytest.mark.parametrize("chroma", [1, 0], ids=["420", "400"])
@pytest.mark.parametrize("win", list(CONF_WINDOWS), ids=list(CONF_WINDOWS))
def test_conformance_windows(decoder, chroma, win):
    pics = _conf_pics(chroma, CONF_WINDOWS[win], 6)
    tw, th = H.tile_size(pics[0].desc)
    grid = Grid(pics, 2, 3, (3 * tw - 5, 2 * th - 3))  # ragged canvas: the last column and row of tiles are cut
    cases = [(p.desc, [p], 1, 1, (tw, th)) for p in pics[:2]] + [(grid.desc, pics, 2, 3, (3 * tw - 5, 2 * th - 3))]
    for desc, ps, rows, cols, canvas in cases:
        (y, cb, cr), rgb = expected_grid(ps, rows, cols, canvas)
        assert np.array_equal(decoder.decode_grids([desc])[0], rgb), (win, rows)
        with decoder.batch([desc]) as b:
            b.decode()
            assert np.array_equal(b.download_image(0), rgb)
        gy, gcb, gcr = decoder.decode_grids_yuv([desc])[0]
        assert np.array_equal(gy, y)
        if chroma:
            assert np.array_equal(gcb, cb) and np.array_equal(gcr, cr)
        # with a crop and a turn on top of the window
        t = K.ImageTransform(1, 2, canvas[0] - 4, canvas[1] - 3, 5)
        assert np.array_equal(decoder.decode_grids([desc], transforms=[t])[0], apply_transform(rgb, t))


def test_mixed_geometries_in_one_batch(decoder, heic_file, fixture_rgb):
    """Old-geometry and new-geometry images in one resident batch and in one decode_grids call: the colour stage groups
    consecutive images of equal geometry into one launch, and each output must still be exact."""
    img = heic_file.primary
    pics = _conf_pics(1, CONF_WINDOWS["all"], 6, seed0=40)
    tw, th = H.tile_size(pics[0].desc)
    grid = Grid(pics, 2, 3, (3 * tw - 5, 2 * th - 3))
    _, grid_rgb = expected_grid(pics, 2, 3, (3 * tw - 5, 2 * th - 3))
    plain = synth.encode(50, width=128, height=64)
    _, plain_rgb = expected_grid([plain], 1, 1, (128, 64))
    full = K.ImageTransform(0, 0, 4032, 3024, 0)
    g_id = K.ImageTransform(0, 0, 3 * tw - 5, 2 * th - 3, 0)
    items = [(img, full, fixture_rgb), (img, full, fixture_rgb), (img, K.ImageTransform(8, 2, 4000, 3000, 0), None),
             (img, K.ImageTransform(8, 2, 4000, 3000, 0), None), (img, K.ImageTransform(0, 0, 4032, 3024, 1), None),
             (grid.desc, g_id, grid_rgb), (img, K.ImageTransform(333, 217, 1001, 777, 6), None), (plain.desc, K.ImageTransform(0, 0, 128, 64, 0), plain_rgb),
             (grid.desc, K.ImageTransform(1, 1, 3 * tw - 6, 2 * th - 4, 3), None), (img, full, fixture_rgb)]
    exps = []
    for desc, t, base in items:
        src = base if base is not None else (fixture_rgb if desc is img else grid_rgb)
        exps.append(apply_transform(src, t))
    with decoder.batch([d for d, _, _ in items], transforms=[t for _, t, _ in items]) as b:
        b.decode()
        for i, e in enumerate(exps):
            assert np.array_equal(b.download_image(i), e), i


def _fixture_file(heic_file, props):
    img = heic_file.primary
    tiles = [heic_file.tile_nal(t) for t in range(img.n_tiles)]
    ps = [heic_file.parameter_set_nal(k) for k in (32, 33, 34)]
    return W.write_heif(*ps, tiles, (512, 512), grid=(img.grid_rows, img.grid_cols), canvas=(img.output_width, img.output_height),
                        props=props)


FILE_PROPS = {
    "clap_irot_imir": [W.clap(4001, 1, 2999, 1, -7, 2, 5, 1), W.irot(1), W.imir(0)],
    "imir_clap_irot": [W.imir(1), W.clap(4020, 1, 3000, 1, 3, 1, -1, 2), W.irot(3)],
    "irot_imir_clap": [W.irot(2), W.imir(1), W.clap(1001, 1, 513, 1, -101, 1, 77, 1)],
    "irot_clap": [W.irot(1), W.clap(3000, 1, 4000, 1, 1, 1, 1, 1)],
    "imir_only": [W.imir(0)],
}


@pytest.mark.parametrize("name", list(FILE_PROPS), ids=list(FILE_PROPS))
def test_files_with_geometry_properties(decoder, heic_file, fixture_rgb, name):
    data = _fixture_file(heic_file, FILE_PROPS[name])
    exp = fixture_rgb
    for p in FILE_PROPS[name]:
        exp = apply_property(exp, p)
    got = decoder.decode(data, apply_transforms=True)
    assert got.shape == exp.shape and np.array_equal(got, exp)
    assert np.array_equal(decoder.decode(data), fixture_rgb)  # without transforms: the canvas


def test_geometry_without_fused_sao(built):
    """The same file with SAO written to its own planes before the colour kernel (HEIC_B200_FUSE_SAO=0, read once per
    process, hence the subprocess)."""
    e = dict(os.environ)
    e["HEIC_B200_FUSE_SAO"] = "0"
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_geometry.py", "-x", "-q", "-m", "gpu", "-p", "no:cacheprovider",
                        "-k", "not without_fused_sao"], cwd=ROOT, env=e, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
