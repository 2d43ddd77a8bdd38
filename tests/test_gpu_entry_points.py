"""The narrow C entry points are the _resized calls with default arguments: for the fixture under a few output specs, each
of decode_grids{,_transformed,_reduced} and their _submit forms, batch_create{,_ex,_transformed,_reduced} and
decode_file, called through ctypes, writes the same bytes and launches the same number of kernels as its _resized
equivalent.  Every call that takes xforms, reduce or resize rejects NULL for it.  And the plain size sort of the CABAC
grouping (HEIC_B200_CABAC_PLAIN_SORT) changes the launch order only, not the RGB."""
import ctypes as C
import os

import numpy as np
import pytest

import heif_b200 as H
from heif_b200 import _capi as K

pytestmark = pytest.mark.gpu
N = 2  # images per call


def _specs(img):
    """name -> (transform, reduction factor, apply_transforms of the calls without arrays that mean the same, or None)."""
    w, h = img.output_width, img.output_height
    rot = img.rotation_ccw_quarter_turns & 3
    assert rot, "the fixture has an irot: the 'irot' spec differs from the identity"
    return {
        "identity": (K.ImageTransform(0, 0, w, h, 0), 1, 0),
        "irot": (K.ImageTransform(0, 0, w, h, rot), 1, 1),
        "odd_crop_o5": (K.ImageTransform(333, 217, 1001, 777, 5), 1, None),
        "factor2": (K.ImageTransform(0, 0, w, h, 0), 2, None),
    }


SPEC_NAMES = ["identity", "irot", "odd_crop_o5", "factor2"]


def _arrays(t, k, n=N):
    return H._transform_array([t] * n, n), H._reduce_array([k] * n), (K.Resize * n)()


def _shape(img, t, k, n=N):
    w, h = H._canvas(img, transform=t, reduce=k)
    return (n, h, w, 3)


def _run(dec, fn, shape, n_tiles):
    """fn(rgb_out, pitch, image_stride, status) -> (return code, RGB, status tuples, kernel launches)."""
    out = np.full(shape, 7, np.uint8)
    st = (K.TileStatus * n_tiles)()
    n0 = dec.launch_count()
    rc = fn(out.ctypes.data, out.strides[1], out.strides[0], st)
    return rc, out, [(s.code, s.bins_decoded, s.ctus_decoded) for s in st], dec.launch_count() - n0


def _submitted(lib, fn):
    """A _submit form as a synchronous call: fn(rgb_out, pitch, image_stride, status, out_job), then the wait."""
    def call(o, p, s, st):
        job = C.c_void_p()
        rc = fn(o, p, s, st, C.byref(job))
        return rc if rc else lib.heic_b200_job_wait(job)
    return call


@pytest.mark.parametrize("spec", SPEC_NAMES)
def test_decode_grids_forms_match_resized(decoder, heic_file, spec):
    img = heic_file.primary
    t, k, apply = _specs(img)[spec]
    lib, h = decoder._lib, decoder._h
    arr = H._desc_array([img] * N)
    xf, ks, rs = _arrays(t, k)
    shape, n_tiles = _shape(img, t, k), N * img.n_tiles
    ref = _run(decoder, lambda o, p, s, st: lib.heic_b200_decode_grids_resized(h, arr, xf, ks, rs, N, o, p, s, st), shape, n_tiles)
    assert ref[0] == 0
    calls = {
        "submit_resized": _submitted(lib, lambda *a: lib.heic_b200_decode_grids_submit_resized(h, arr, xf, ks, rs, N, *a)),
        "reduced": lambda *a: lib.heic_b200_decode_grids_reduced(h, arr, xf, ks, N, *a),
        "submit_reduced": _submitted(lib, lambda *a: lib.heic_b200_decode_grids_submit_reduced(h, arr, xf, ks, N, *a)),
    }
    if k == 1:
        calls["transformed"] = lambda *a: lib.heic_b200_decode_grids_transformed(h, arr, xf, N, *a)
        calls["submit_transformed"] = _submitted(lib, lambda *a: lib.heic_b200_decode_grids_submit_transformed(h, arr, xf, N, *a))
    if apply is not None:
        calls["decode_grids"] = lambda o, p, s, st: lib.heic_b200_decode_grids(h, arr, N, o, p, s, apply, st)
        calls["submit"] = _submitted(lib, lambda o, p, s, st, j: lib.heic_b200_decode_grids_submit(h, arr, N, o, p, s, apply, st, j))
    for name, fn in calls.items():
        rc, out, st, launches = _run(decoder, fn, shape, n_tiles)
        assert rc == 0, name
        assert np.array_equal(out, ref[1]), name
        assert st == ref[2], name
        assert launches == ref[3], name


def _batch(dec, create, shape):
    """create(out_batch) -> (RGB of download_rgb after a decode, heic_b200_batch_rgb's pitch and stride, kernel launches)."""
    lib = dec._lib
    b = C.c_void_p()
    n0 = dec.launch_count()
    K.check(create(C.byref(b)))
    try:
        K.check(lib.heic_b200_batch_decode(b))
        ptr, pitch, stride = C.c_void_p(), C.c_size_t(), C.c_size_t()
        K.check(lib.heic_b200_batch_rgb(b, C.byref(ptr), C.byref(pitch), C.byref(stride)))
        out = np.full(shape, 7, np.uint8)
        K.check(lib.heic_b200_batch_download_rgb(b, out.ctypes.data, out.strides[1], out.strides[0]))
        return out, pitch.value, stride.value, dec.launch_count() - n0
    finally:
        lib.heic_b200_batch_destroy(b)


@pytest.mark.parametrize("spec", SPEC_NAMES)
def test_batch_create_forms_match_resized(decoder, heic_file, spec):
    img = heic_file.primary
    t, k, apply = _specs(img)[spec]
    lib, h = decoder._lib, decoder._h
    arr = H._desc_array([img] * N)
    xf, ks, rs = _arrays(t, k)
    shape = _shape(img, t, k)
    ref = _batch(decoder, lambda b: lib.heic_b200_batch_create_resized(h, arr, xf, ks, rs, N, b), shape)
    calls = {"reduced": lambda b: lib.heic_b200_batch_create_reduced(h, arr, xf, ks, N, b)}
    if k == 1:
        calls["transformed"] = lambda b: lib.heic_b200_batch_create_transformed(h, arr, xf, N, b)
    if apply is not None:
        calls["ex"] = lambda b: lib.heic_b200_batch_create_ex(h, arr, N, apply, b)
    if apply == 0:
        calls["create"] = lambda b: lib.heic_b200_batch_create(h, arr, N, b)
    for name, create in calls.items():
        out, pitch, stride, launches = _batch(decoder, create, shape)
        assert np.array_equal(out, ref[0]), name
        assert (pitch, stride) == ref[1:3], name
        assert launches == ref[3], name


def test_decode_file_matches_resized(decoder, heic_file, fixture_bytes):
    img = heic_file.primary
    lib, h = decoder._lib, decoder._h
    arr = H._desc_array([img])
    for apply, t in ((0, _specs(img)["identity"][0]), (1, heic_file.transform())):
        xf, ks, rs = _arrays(t, 1, 1)
        shape = _shape(img, t, 1, 1)
        ref = _run(decoder, lambda o, p, s, st: lib.heic_b200_decode_grids_resized(h, arr, xf, ks, rs, 1, o, p, s, st), shape,
                   img.n_tiles)
        assert ref[0] == 0
        rc, out, _, launches = _run(decoder, lambda o, p, s, st: lib.heic_b200_decode_file(h, fixture_bytes, len(fixture_bytes), o, p,
                                                                                          apply), shape, img.n_tiles)
        assert rc == 0, apply
        assert np.array_equal(out, ref[1]), apply
        assert launches == ref[3], apply


def test_null_arrays_are_rejected(decoder, heic_file):
    img = heic_file.primary
    lib, h = decoder._lib, decoder._h
    arr = H._desc_array([img] * N)
    t, k, _ = _specs(img)["identity"]
    xf, ks, rs = _arrays(t, k)
    shape, n_tiles = _shape(img, t, k), N * img.n_tiles
    job = C.byref(C.c_void_p())
    grids = {  # name -> (call taking (xforms, reduce, resize, rgb_out, pitch, image_stride, status), arrays it takes)
        "decode_grids_transformed": (lambda x, r, z, *a: lib.heic_b200_decode_grids_transformed(h, arr, x, N, *a), "x"),
        "decode_grids_submit_transformed":
            (lambda x, r, z, *a: lib.heic_b200_decode_grids_submit_transformed(h, arr, x, N, *a, job), "x"),
        "decode_grids_reduced": (lambda x, r, z, *a: lib.heic_b200_decode_grids_reduced(h, arr, x, r, N, *a), "xr"),
        "decode_grids_submit_reduced":
            (lambda x, r, z, *a: lib.heic_b200_decode_grids_submit_reduced(h, arr, x, r, N, *a, job), "xr"),
        "decode_grids_resized": (lambda x, r, z, *a: lib.heic_b200_decode_grids_resized(h, arr, x, r, z, N, *a), "xrz"),
        "decode_grids_submit_resized":
            (lambda x, r, z, *a: lib.heic_b200_decode_grids_submit_resized(h, arr, x, r, z, N, *a, job), "xrz"),
    }
    batches = {  # name -> (call taking (xforms, reduce, resize, out_batch), arrays it takes)
        "batch_create_transformed": (lambda x, r, z, b: lib.heic_b200_batch_create_transformed(h, arr, x, N, b), "x"),
        "batch_create_reduced": (lambda x, r, z, b: lib.heic_b200_batch_create_reduced(h, arr, x, r, N, b), "xr"),
        "batch_create_resized": (lambda x, r, z, b: lib.heic_b200_batch_create_resized(h, arr, x, r, z, N, b), "xrz"),
    }

    def args(null):
        return tuple(None if a == null else v for a, v in (("x", xf), ("r", ks), ("z", rs)))

    for name, (fn, takes) in grids.items():
        for null in takes:
            rc, out, _, launches = _run(decoder, lambda *a: fn(*args(null), *a), shape, n_tiles)
            assert rc == K.HEIC_E_INVALID_ARG, (name, null)
            assert launches == 0 and (out == 7).all(), (name, null)
    for name, (fn, takes) in batches.items():
        for null in takes:
            b = C.c_void_p()
            n0 = decoder.launch_count()
            assert fn(*args(null), C.byref(b)) == K.HEIC_E_INVALID_ARG, (name, null)
            assert not b.value and decoder.launch_count() == n0, (name, null)


def test_plain_sort_gives_the_same_rgb(decoder, heic_file):
    """HEIC_B200_CABAC_PLAIN_SORT (read when the context is created) with the thread-per-substream mapping: copies of a tile
    may share a warp, which they never do otherwise, and the RGB is the same."""
    img = heic_file.primary
    knobs = {"HEIC_B200_CABAC_PLAIN_SORT": "1", "HEIC_B200_LOW_LATENCY_TILES": "0"}
    old = {k: os.environ.get(k) for k in knobs}
    os.environ.update(knobs)
    try:
        dec = H.HeicDecoder(device=0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    with dec:
        with dec.batch([img] * N) as b:
            order, per_group = b.cabac_order()
            assert per_group == 32
            groups = [[int(t) % img.n_tiles for t in order[g:g + 32] if t != 0xFFFFFFFF] for g in range(0, len(order), 32)]
            assert any(len(set(g)) < len(g) for g in groups)
        got = dec.decode_grids([img] * N, transforms=[(333, 217, 1001, 777, 5)] * N)
    assert np.array_equal(got, decoder.decode_grids([img] * N, transforms=[(333, 217, 1001, 777, 5)] * N))
