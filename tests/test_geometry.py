"""Output geometry on the host: the clap / irot / imir composition, the transform and file info of HEIF files written by
tests/synth/heif_writer.py, and SPS conformance windows from the synthetic encoder (no GPU)."""
import itertools
import math
from fractions import Fraction

import numpy as np
import pytest

import heif_b200 as H
from heif_b200 import _capi as K
from tests.synth import conf_window
from tests.synth import heif_writer as W
from tests.synth import synth

# imir axis -> normal-form orientation: 0 mirrors top <-> bottom, 1 left <-> right (heif_reader.h kImirOrientation).  If
# the axis turns out to be read the other way round, this table and kImirOrientation change together.
IMIR_ORIENTATION = {0: 6, 1: 4}


def _clap_rect(v, w, h):
    """The clean aperture of an image of w x h as (left, top, width, height): left and top rounded down, the size
    rounded to the nearest integer (halves up)."""
    wn, wd, hn, hd, xn, xd, yn, yd = v
    cw, ch = Fraction(wn, wd), Fraction(hn, hd)
    left = math.floor(Fraction(xn, xd) + (w - cw) / 2)
    top = math.floor(Fraction(yn, yd) + (h - ch) / 2)
    return left, top, math.floor(cw + Fraction(1, 2)), math.floor(ch + Fraction(1, 2))


def apply_property(a, p):
    kind, v = p
    if kind == "irot":
        return np.rot90(a, v)
    if kind == "imir":
        return a[::-1, :] if v == 0 else a[:, ::-1]
    left, top, cw, ch = _clap_rect(v, a.shape[1], a.shape[0])
    return a[top:top + ch, left:left + cw]


def apply_transform(a, t):
    out = np.rot90(a[t.crop_y:t.crop_y + t.crop_h, t.crop_x:t.crop_x + t.crop_w], t.orientation & 3)
    return out[:, ::-1] if t.orientation & 4 else out


# clap symbols, each a function of the current image size: an integral inset, odd (half-pixel) offsets, a size that is
# not integral
CLAPS = {
    "clap_inset": lambda w, h: W.clap(w - 2, 1, h - 2, 1, 0, 1, 0, 1),
    "clap_odd": lambda w, h: W.clap(w - 3, 1, h - 5, 1, -1, 2, 3, 2),
    "clap_frac": lambda w, h: W.clap(2 * w - 3, 2, h, 2, 0, 1, -h, 4),
}
SYMBOLS = list(CLAPS) + ["irot1", "irot2", "irot3", "imir0", "imir1"]


def _props_for(seq, w, h):
    """The property list of a symbol sequence, each clap sized for the image as it stands when it applies."""
    a = np.zeros((h, w), np.uint8)
    props = []
    for s in seq:
        if s in CLAPS:
            p = CLAPS[s](a.shape[1], a.shape[0])
        elif s.startswith("irot"):
            p = W.irot(int(s[-1]))
        else:
            p = W.imir(int(s[-1]))
        props.append(p)
        a = apply_property(a, p)
    return props


@pytest.fixture(scope="module")
def pictures(built):
    """Single-item canvases: 64 x 48, 72 x 40, and 64 x 48 cut to 62 x 44 by a conformance window."""
    return [synth.encode(3, width=64, height=48), synth.encode(4, width=72, height=40),
            conf_window.encode(5, (0, 1, 0, 2), width=64, height=48)]


def _file(pic, props):
    return W.write_heif(pic.vps, pic.sps_nal, pic.pps_nal, [pic.slice_nal], H.tile_size(pic.desc), props=props)


def test_canvas_sizes(pictures):
    assert [H.tile_size(p.desc) for p in pictures] == [(64, 48), (72, 40), (62, 44)]


def test_composed_normal_form_equals_the_properties_one_by_one(pictures):
    """Every sequence of up to three clap / irot / imir properties, on three canvas sizes: the file's transform applied to
    an index array equals the properties applied in ipma order.  Covers claps after turns and mirrors, odd and
    non-integral claps, and mirrors that cancel."""
    n = 0
    for pic in pictures:
        w, h = H.tile_size(pic.desc)
        idx = np.arange(w * h).reshape(h, w)
        for k in range(1, 4):
            for seq in itertools.product(SYMBOLS, repeat=k):
                props = _props_for(seq, w, h)
                f = H.HeicFile(_file(pic, props))
                t = f.transform()
                exp = idx
                for p in props:
                    exp = apply_property(exp, p)
                got = apply_transform(idx, t)
                assert got.shape == exp.shape and np.array_equal(got, exp), (w, h, seq, (t.crop_x, t.crop_y, t.crop_w, t.crop_h, t.orientation))
                info = f.info
                assert (info.rotated_height, info.rotated_width) == exp.shape
                f.close()
                n += 1
    assert n == 3 * (8 + 64 + 512)


def test_imir_axis_mapping_is_the_named_constant(pictures):
    pic = pictures[0]
    for axis, o in IMIR_ORIENTATION.items():
        t = H.HeicFile(_file(pic, [W.imir(axis)])).transform()
        assert (t.crop_x, t.crop_y, t.crop_w, t.crop_h, t.orientation) == (0, 0, 64, 48, o)
    t = H.HeicFile(_file(pic, [W.imir(0), W.imir(0)])).transform()
    assert t.orientation == 0


def test_file_without_geometry_properties_has_the_identity(pictures):
    f = H.HeicFile(_file(pictures[2], []))
    t = f.transform()
    assert (t.crop_x, t.crop_y, t.crop_w, t.crop_h, t.orientation) == (0, 0, 62, 44, 0)
    assert (f.info.rotated_width, f.info.rotated_height) == (62, 44)


def test_fixture_transform_is_its_irot(heic_file):
    t = heic_file.transform()
    info = heic_file.info
    assert (t.crop_x, t.crop_y, t.crop_w, t.crop_h) == (0, 0, heic_file.primary.output_width, heic_file.primary.output_height)
    assert t.orientation == info.rotation_ccw_quarter_turns
    assert (info.rotated_width, info.rotated_height) == (3024, 4032)


@pytest.mark.parametrize("prop", [
    W.clap(32, 0, 32, 1, 0, 1, 0, 1), W.clap(32, 1, 32, 0, 0, 1, 0, 1), W.clap(32, 1, 32, 1, 0, 0, 0, 1),
    W.clap(32, 1, 32, 1, 0, 1, 0, 0),
    W.clap(65, 1, 48, 1, 0, 1, 0, 1), W.clap(32, 1, 32, 1, 17, 1, 0, 1), W.clap(32, 1, 32, 1, 0, 1, -9, 1),
    W.clap(0, 1, 32, 1, 0, 1, 0, 1), W.clap(1, 4, 32, 1, 0, 1, 0, 1),
], ids=["width_d0", "height_d0", "horiz_d0", "vert_d0", "too_wide", "right_of_image", "above_image", "empty", "rounds_to_empty"])
def test_bad_clap_is_a_bitstream_error(pictures, prop):
    with pytest.raises(H.HeicError) as e:
        H.HeicFile(_file(pictures[0], [prop]))
    assert e.value.code == K.HEIC_E_BITSTREAM


def test_clap_after_a_turn_is_checked_against_the_turned_image(pictures):
    """64 x 48 turned once is 48 x 64: a 60-pixel-high aperture fits only after the turn."""
    H.HeicFile(_file(pictures[0], [W.irot(1), W.clap(40, 1, 60, 1, 0, 1, 0, 1)]))
    with pytest.raises(H.HeicError):
        H.HeicFile(_file(pictures[0], [W.clap(40, 1, 60, 1, 0, 1, 0, 1), W.irot(1)]))


def test_fixture_grid_rewritten_with_geometry_properties(heic_file):
    """The fixture's own 48 tiles and parameter sets in a file of the test writer: clap, irot and imir on the grid item."""
    img = heic_file.primary
    tiles = [heic_file.tile_nal(t) for t in range(img.n_tiles)]
    ps = [heic_file.parameter_set_nal(k) for k in (32, 33, 34)]
    cw, ch = img.output_width, img.output_height
    data = W.write_heif(*ps, tiles, (512, 512), grid=(img.grid_rows, img.grid_cols), canvas=(cw, ch),
                        props=[W.imir(1), W.clap(cw - 100, 1, ch - 50, 1, 11, 1, -7, 1), W.irot(1)])
    f = H.HeicFile(data)
    t = f.transform()
    left, top = 11 + 50, -7 + 25
    # mirrored first: the aperture's left edge in the mirrored image is the canvas column cw - 1 - (left + width - 1); a
    # quarter turn after the mirror is the mirror after three quarter turns (orientation 3 | 4)
    assert (t.crop_x, t.crop_y, t.crop_w, t.crop_h, t.orientation) == (cw - left - (cw - 100), top, cw - 100, ch - 50, 7)
    assert (f.info.rotated_width, f.info.rotated_height) == (ch - 50, cw - 100)
    assert f.primary.n_tiles == img.n_tiles


CONF_WINDOWS = [(1, 0, 0, 0), (0, 3, 0, 0), (0, 0, 1, 0), (0, 0, 0, 3), (1, 2, 3, 1)]


@pytest.mark.parametrize("chroma", [1, 0], ids=["420", "400"])
@pytest.mark.parametrize("win", CONF_WINDOWS, ids=["left", "right", "top", "bottom", "all"])
def test_conformance_window_parses_back(built, chroma, win):
    pic = conf_window.encode(7, win, width=96, height=64, chroma_format_idc=chroma)
    plain = synth.encode(7, width=96, height=64, chroma_format_idc=chroma)
    assert pic.vps == plain.vps and pic.pps_nal == plain.pps_nal and pic.slice_nal == plain.slice_nal
    s = pic.sps
    assert s.conformance_window_flag == 1
    assert (s.conf_win_left_offset, s.conf_win_right_offset, s.conf_win_top_offset, s.conf_win_bottom_offset) == win
    sub = 2 if chroma else 1
    assert H.tile_size(pic.desc) == (96 - sub * (win[0] + win[1]), 64 - sub * (win[2] + win[3]))
    assert (pic.desc.output_width, pic.desc.output_height) == H.tile_size(pic.desc)


@pytest.mark.parametrize("chroma", [1, 0], ids=["420", "400"])
@pytest.mark.parametrize("win", [(0, 3, 0, 0), (0, 0, 0, 3), (0, 2, 0, 1)], ids=["right", "bottom", "right_bottom"])
def test_ffmpeg_crops_what_the_oracle_decodes(built, chroma, win):
    """FFmpeg's cropped planes are the oracle's full planes cut by the window.  Only right / bottom offsets are compared:
    without AV_CODEC_FLAG_UNALIGNED (not set by the FFmpeg test oracle) FFmpeg may align a left crop down."""
    from oracle import ffmpeg_oracle
    from oracle import oracle_py as O

    pic = conf_window.encode(8, win, width=96, height=64, chroma_format_idc=chroma)
    t = pic.tile
    ref = O.decode_picture(pic.sps, pic.pps, t.header, (t.rbsp, t.rbsp_len), intermediates=False)["plane"]
    dec = ffmpeg_oracle.FFmpegHevc()
    try:
        got = dec.decode_picture(pic.annexb())
    finally:
        dec.close()
    w, h = H.tile_size(pic.desc)
    assert np.array_equal(got[0], ref[0][:h, :w])
    if chroma:
        for c in (1, 2):
            assert np.array_equal(got[c], ref[c][:h // 2, :w // 2])
