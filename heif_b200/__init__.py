"""heif_b200 — B200-native HEIC image reconstruction behind the decode API of friendlymatthew/heif.

Host-side mirror of the reference's public interface (names follow the crate):

    HeifReader(data).read()          src/heif/reader.rs:25,59     -> HeicFile (container + parameter sets + slice headers)
    HeicDecoder().decode(data)       src/heic/decoder.rs:12       -> RGB image (the reference returns ())

Everything here is ctypes plumbing over the C ABI in include/heic_b200.h (heif_b200/libheic_b200.so, built by
``__graft_entry__.build()``).  All computation happens in the library's sm_100a kernels; there is no Python or
CPU fallback — without the library, or without a CUDA device, the calls raise.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi as K
from ._capi import HeicError, STAGE_ALL, STAGE_CABAC, STAGE_COLOR, STAGE_DEBLOCK, STAGE_INTRA, STAGE_SAO, STAGE_TRANSFORM

__all__ = [
    "HeicDecoder", "HeicFile", "HeifReader", "Batch", "HeicError", "remove_emulation_prevention", "parse_sps", "parse_pps",
    "parse_slice_header", "parse_slice_header_raw", "read_ue", "read_se", "STAGE_ALL", "STAGE_CABAC", "STAGE_TRANSFORM", "STAGE_INTRA", "STAGE_DEBLOCK", "STAGE_SAO",
    "STAGE_COLOR",
]


def _lib():
    return K.load()


# ---- host parse layer (reference: src/hevc/rbsp_reader.rs, parameter_set_reader.rs, slice.rs:44-204) --------------
def remove_emulation_prevention(data: bytes, with_positions: bool = False):
    """RbspReader::remove_emulation_prevention (rbsp_reader.rs:11-39)."""
    lib = _lib()
    out = (K.u8 * max(len(data), 1))()
    pos = (K.u32 * max(len(data) // 3 + 1, 1))()
    n_epb = C.c_size_t()
    n = lib.heic_b200_remove_emulation_prevention(bytes(data), len(data), out, pos, len(pos), C.byref(n_epb))
    K.check(int(n))
    res = bytes(out[: int(n)])
    if with_positions:
        return res, [int(pos[i]) for i in range(n_epb.value)]
    return res


def read_ue(data: bytes, bit_pos: int = 0):
    """RbspReader::read_ue (rbsp_reader.rs:87) -> (value, new bit position)."""
    pos, out = C.c_size_t(bit_pos), K.u32()
    K.check(_lib().heic_b200_rbsp_read_ue(bytes(data), len(data), C.byref(pos), C.byref(out)))
    return out.value, pos.value


def read_se(data: bytes, bit_pos: int = 0):
    """RbspReader::read_se (rbsp_reader.rs:101) -> (value, new bit position)."""
    pos, out = C.c_size_t(bit_pos), K.i32()
    K.check(_lib().heic_b200_rbsp_read_se(bytes(data), len(data), C.byref(pos), C.byref(out)))
    return out.value, pos.value


def parse_sps(rbsp: bytes) -> K.Sps:
    """sequence_parameter_set_rbsp (parameter_set_reader.rs:36); input without the 2-byte NAL header."""
    out = K.Sps()
    K.check(_lib().heic_b200_parse_sps(bytes(rbsp), len(rbsp), C.byref(out)))
    return out


def parse_pps(rbsp: bytes) -> K.Pps:
    """picture_parameter_set_rbsp (parameter_set_reader.rs:351)."""
    out = K.Pps()
    K.check(_lib().heic_b200_parse_pps(bytes(rbsp), len(rbsp), C.byref(out)))
    return out


def parse_slice_header(rbsp: bytes, nal_unit_type: int, sps: K.Sps, pps: K.Pps, epb_pos=()) -> K.SliceHeader:
    """SliceSegmentReader::read_header (slice.rs:44-204) + un-escaped substream offsets."""
    out = K.SliceHeader()
    arr = (K.u32 * max(len(epb_pos), 1))(*epb_pos)
    K.check(_lib().heic_b200_parse_slice_header(bytes(rbsp), len(rbsp), nal_unit_type, C.byref(sps), C.byref(pps), arr,
                                                len(epb_pos), C.byref(out)))
    return out


def parse_slice_header_raw(nal_payload: bytes, nal_unit_type: int, sps: K.Sps, pps: K.Pps) -> K.SliceHeader:
    """The slice header read from a raw NAL payload; offsets stay in raw byte counts (TileDesc.escaped = 1)."""
    out = K.SliceHeader()
    K.check(_lib().heic_b200_parse_slice_header_raw(bytes(nal_payload), len(nal_payload), nal_unit_type, C.byref(sps), C.byref(pps),
                                                    C.byref(out)))
    return out


class HeicFile:
    """A parsed HEIC file: HeifReader::read + the item walk of HeicDecoder::decode up to the slice headers."""

    def __init__(self, data: bytes):
        self._lib = _lib()
        self._data = bytes(data)
        self._h = C.c_void_p()
        K.check(self._lib.heic_b200_file_open(self._data, len(self._data), C.byref(self._h)))

    def close(self):
        if self._h:
            self._lib.heic_b200_file_close(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def primary(self) -> K.ImageDesc:
        return self._lib.heic_b200_file_primary_image(self._h).contents

    @property
    def aux_images(self):
        n = self._lib.heic_b200_file_aux_image_count(self._h)
        return [self._lib.heic_b200_file_aux_image(self._h, i).contents for i in range(n)]

    @property
    def primary_raw(self) -> K.ImageDesc:
        """The primary image with raw tile payloads: emulation prevention removal happens on the GPU."""
        return self._lib.heic_b200_file_primary_image_raw(self._h).contents

    @property
    def aux_images_raw(self):
        n = self._lib.heic_b200_file_aux_image_count(self._h)
        return [self._lib.heic_b200_file_aux_image_raw(self._h, i).contents for i in range(n)]

    @property
    def info(self) -> K.FileInfo:
        out = K.FileInfo()
        K.check(self._lib.heic_b200_file_info(self._h, C.byref(out)))
        return out

    def transform(self, image: int = -1) -> K.ImageTransform:
        """The image item's clap / irot / imir properties in normal form (image = -1: primary, >= 0: auxiliary)."""
        out = K.ImageTransform()
        K.check(self._lib.heic_b200_file_image_transform(self._h, image, C.byref(out)))
        return out

    def parameter_set_nal(self, nal_unit_type: int, image: int = -1) -> bytes:
        p, n = C.POINTER(K.u8)(), C.c_size_t()
        K.check(self._lib.heic_b200_file_parameter_set_nal(self._h, image, nal_unit_type, C.byref(p), C.byref(n)))
        return bytes(p[: n.value])

    def tile_nal(self, tile: int, image: int = -1) -> bytes:
        p, n = C.POINTER(K.u8)(), C.c_size_t()
        K.check(self._lib.heic_b200_file_tile_nal(self._h, image, tile, C.byref(p), C.byref(n)))
        return bytes(p[: n.value])


class HeifReader:
    """Name-compatible wrapper: ``HeifReader(data).read()`` (src/heif/reader.rs:25,59)."""

    def __init__(self, data: bytes):
        self._data = data

    def read(self) -> HeicFile:
        return HeicFile(self._data)


def tile_size(img: K.ImageDesc):
    """(width, height) at which the grid stitches a tile: the SPS conformance window of its decoded picture."""
    sps = img.sps
    w, h = sps.pic_width_in_luma_samples, sps.pic_height_in_luma_samples
    if sps.conformance_window_flag:
        sub = 2 if sps.chroma_format_idc == 1 else 1
        w -= sub * (sps.conf_win_left_offset + sps.conf_win_right_offset)
        h -= sub * (sps.conf_win_top_offset + sps.conf_win_bottom_offset)
    return w, h


def canvas_transform(img: K.ImageDesc, apply_transforms: bool = False) -> K.ImageTransform:
    """What the calls without transforms apply: the whole canvas, turned by irot when apply_transforms is set."""
    tw, th = tile_size(img)
    w = img.output_width or img.grid_cols * tw
    h = img.output_height or img.grid_rows * th
    return K.ImageTransform(0, 0, w, h, (img.rotation_ccw_quarter_turns & 3) if apply_transforms else 0)


def _transform(t) -> K.ImageTransform:
    return t if isinstance(t, K.ImageTransform) else K.ImageTransform(*t)


def _canvas(img: K.ImageDesc, apply_transforms: bool = False, transform=None, reduce: int = 1):
    """(width, height) of an image's output: the transform's crop, turned for odd quarter turns, then reduced by the box
    reduction factor to ceil(w / reduce) x ceil(h / reduce).  (A factor outside 1..16 is left for the library to reject.)"""
    t = _transform(transform) if transform is not None else canvas_transform(img, apply_transforms)
    w, h = (t.crop_h, t.crop_w) if t.orientation & 1 else (t.crop_w, t.crop_h)
    k = max(int(reduce), 1)
    return -(-w // k), -(-h // k)


def _reduce_list(reduce, n: int):
    """One box reduction factor per image from an int or a sequence."""
    ks = [int(reduce)] * n if isinstance(reduce, (int, np.integer)) else [int(k) for k in reduce]
    if len(ks) != n:
        raise ValueError("one reduction factor per image")
    return ks


def _reduce_array(ks):
    return (K.u32 * len(ks))(*[k & 0xFFFFFFFF for k in ks])


def _transform_array(transforms, n: int):
    transforms = [_transform(t) for t in transforms]
    if len(transforms) != n:
        raise ValueError("one transform per image")
    arr = (K.ImageTransform * n)()
    for i, t in enumerate(transforms):
        arr[i] = t
    return arr


def _desc_array(images):
    arr = (K.ImageDesc * len(images))()
    for i, im in enumerate(images):
        C.memmove(C.byref(arr, i * C.sizeof(K.ImageDesc)), C.byref(im), C.sizeof(K.ImageDesc))
    return arr


class Batch:
    """A resident batch: bitstreams, descriptors and every intermediate live in HBM (heic_b200_batch_*)."""

    def __init__(self, dec: "HeicDecoder", images, apply_transforms: bool = False, transforms=None, reduce=1):
        """transforms: one heic_image_transform (K.ImageTransform or (x, y, w, h, orientation)) per image; when None,
        apply_transforms selects the irot turn of every image or none.  reduce: box reduction factor (1..16), one int for
        every image or one per image: image i is PIL.Image.reduce(reduce[i]) of its transformed RGB (heic_b200.h,
        heic_b200_decode_grids_reduced)."""
        self._lib = dec._lib
        self._dec = dec
        self.images = list(images)
        self.apply_transforms = bool(apply_transforms)
        self.reduce = _reduce_list(reduce, len(self.images))
        self._arr = _desc_array(self.images)
        self._h = C.c_void_p()
        if any(k != 1 for k in self.reduce):
            xf = transforms if transforms is not None else [canvas_transform(im, self.apply_transforms) for im in self.images]
            self._xf = _transform_array(xf, len(self.images))
            self.transforms = list(self._xf)
            K.check(self._lib.heic_b200_batch_create_reduced(dec._h, self._arr, self._xf, _reduce_array(self.reduce), len(self.images),
                                                             C.byref(self._h)))
        elif transforms is None:
            self.transforms = [canvas_transform(im, self.apply_transforms) for im in self.images]
            K.check(self._lib.heic_b200_batch_create_ex(dec._h, self._arr, len(self.images), int(self.apply_transforms), C.byref(self._h)))
        else:
            self._xf = _transform_array(transforms, len(self.images))
            self.transforms = list(self._xf)
            K.check(self._lib.heic_b200_batch_create_transformed(dec._h, self._arr, self._xf, len(self.images), C.byref(self._h)))

    def close(self):
        if self._h:
            self._lib.heic_b200_batch_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def n_tiles(self) -> int:
        return self._lib.heic_b200_batch_tile_count(self._h)

    def cabac_order(self):
        """(tile indices in CABAC launch order with 0xffffffff for idle lanes, tiles per warp-group)."""
        tpg = C.c_uint32()
        n = self._lib.heic_b200_batch_cabac_order(self._h, None, 0, C.byref(tpg))
        out = np.zeros(n, np.uint32)
        self._lib.heic_b200_batch_cabac_order(self._h, out.ctypes.data_as(C.POINTER(C.c_uint32)), n, C.byref(tpg))
        return out, int(tpg.value)

    @property
    def stream(self) -> int:
        return int(self._lib.heic_b200_batch_stream(self._h) or 0)

    def run(self, stage_mask: int = STAGE_ALL):
        K.check(self._lib.heic_b200_batch_run_stages(self._h, stage_mask))

    def decode(self):
        K.check(self._lib.heic_b200_batch_decode(self._h))

    def sync(self):
        K.check(self._lib.heic_b200_batch_sync(self._h))

    def rgb_layout(self):
        p, pitch, stride = C.c_void_p(), C.c_size_t(), C.c_size_t()
        K.check(self._lib.heic_b200_batch_rgb(self._h, C.byref(p), C.byref(pitch), C.byref(stride)))
        return int(p.value or 0), pitch.value, stride.value

    def download_rgb(self, out: np.ndarray | None = None) -> np.ndarray:
        w, h = _canvas(self.images[0], transform=self.transforms[0], reduce=self.reduce[0])
        if out is None:
            out = np.empty((len(self.images), h, w, 3), np.uint8)
        K.check(self._lib.heic_b200_batch_download_rgb(self._h, out.ctypes.data, out.strides[1], out.strides[0]))
        return out

    def download_image(self, index: int) -> np.ndarray:
        """RGB of one image of the batch (H, W, 3)."""
        w, h = _canvas(self.images[index], transform=self.transforms[index], reduce=self.reduce[index])
        out = np.empty((h, w, 3), np.uint8)
        K.check(self._lib.heic_b200_batch_download_image(self._h, index, out.ctypes.data, out.strides[0]))
        return out

    def status(self):
        st = (K.TileStatus * self.n_tiles)()
        K.check(self._lib.heic_b200_batch_status(self._h, st))
        return st

    def dump_tile(self, tile: int, image: int = 0) -> dict:
        """Intermediate buffers of one tile (layouts: DESIGN.md 'Data layout in HBM')."""
        img = self.images[image]
        sps = img.sps
        w, h = sps.pic_width_in_luma_samples, sps.pic_height_in_luma_samples
        log2_ctb = sps.log2_min_luma_coding_block_size_minus3 + 3 + sps.log2_diff_max_min_luma_coding_block_size
        ctb = 1 << log2_ctb
        n_ctb = -(-w // ctb) * -(-h // ctb)
        n_tu = n_ctb * (ctb // 4) ** 2
        chroma = sps.chroma_format_idc == 1
        d = K.TileDump()
        res = {"tu_map": np.zeros(n_tu, np.uint32), "qp_map": np.zeros((h // 8, w // 8), np.uint8),
               "sao": np.zeros(n_ctb * 4, np.uint32), "coeff": [], "plane": []}
        d.tu_map = res["tu_map"].ctypes.data_as(C.POINTER(K.u32))
        d.tu_map_len = n_tu
        d.qp_map = res["qp_map"].ctypes.data_as(C.POINTER(K.u8))
        d.qp_map_len = res["qp_map"].size
        d.sao = res["sao"].ctypes.data_as(C.POINTER(K.u32))
        d.sao_len = res["sao"].size
        for c in range(3 if chroma else 1):
            a = np.zeros(n_tu * (4 if c else 16), np.int16)
            res["coeff"].append(a)
            d.coeff[c] = a.ctypes.data_as(C.POINTER(C.c_int16))
            d.coeff_len[c] = a.size
            p = np.zeros((h >> (1 if c else 0), w >> (1 if c else 0)), np.uint8)
            res["plane"].append(p)
            d.plane[c] = p.ctypes.data_as(C.POINTER(K.u8))
            d.plane_len[c] = p.size
        first = sum(im.n_tiles for im in self.images[:image])
        K.check(self._lib.heic_b200_batch_dump_tile(self._h, first + tile, C.byref(d)))
        return res


class HeicDecoder:
    """HeicDecoder::decode (src/heic/decoder.rs:12) with the image it never returned.

    One decoder = one heic_b200_ctx = one CUDA stream on one device."""

    def __init__(self, device: int = -1):
        self._lib = _lib()
        self._h = C.c_void_p()
        K.check(self._lib.heic_b200_create(device, C.byref(self._h)))

    def close(self):
        if self._h:
            self._lib.heic_b200_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def launch_count(self) -> int:
        return int(self._lib.heic_b200_launch_count(self._h))

    def decode(self, data, apply_transforms: bool = False, reduce: int = 1) -> np.ndarray:
        """bytes | HeicFile -> (H, W, 3) uint8 RGB of the primary item; apply_transforms: with the file's clap / irot / imir;
        reduce: box reduction factor 1..16 (see Batch)."""
        f = data if isinstance(data, HeicFile) else HeicFile(data)
        if apply_transforms:
            return self.decode_grids([f.primary], transforms=[f.transform()], reduce=reduce)[0]
        return self.decode_grids([f.primary], reduce=reduce)[0]

    def decode_grids(self, images, out: np.ndarray | None = None, apply_transforms: bool = False, return_status: bool = False,
                     transforms=None, reduce=1):
        """Batch of image descriptors (host) -> (n, H, W, 3) uint8 RGB (host).  All outputs must share one size.
        transforms: one heic_image_transform per image (see Batch); when None, apply_transforms selects irot or nothing.
        reduce: box reduction factor (1..16), one for every image or one per image (see Batch)."""
        images = list(images)
        arr = _desc_array(images)
        xf = [None] * len(images) if transforms is None else list(transforms)
        ks = _reduce_list(reduce, len(images))
        sizes = [_canvas(im, apply_transforms, t, k) for im, t, k in zip(images, xf, ks)]
        w, h = sizes[0]
        if any(s != (w, h) for s in sizes[1:]):
            raise ValueError("decode_grids packs the images into one (n, H, W, 3) array: all outputs (after the transform) must be equal")
        if out is None:
            out = np.empty((len(images), h, w, 3), np.uint8)
        n_tiles = sum(im.n_tiles for im in images)
        st = (K.TileStatus * n_tiles)()
        if any(k != 1 for k in ks):
            xf = [canvas_transform(im, apply_transforms) if t is None else t for im, t in zip(images, xf)]
            rc = self._lib.heic_b200_decode_grids_reduced(self._h, arr, _transform_array(xf, len(images)), _reduce_array(ks), len(images),
                                                          out.ctypes.data, out.strides[1], out.strides[0], st)
        elif transforms is None:
            rc = self._lib.heic_b200_decode_grids(self._h, arr, len(images), out.ctypes.data, out.strides[1], out.strides[0],
                                                  1 if apply_transforms else 0, st)
        else:
            rc = self._lib.heic_b200_decode_grids_transformed(self._h, arr, _transform_array(xf, len(images)), len(images),
                                                              out.ctypes.data, out.strides[1], out.strides[0], st)
        if return_status:
            return out, rc, st
        K.check(rc)
        return out

    def submit_grids(self, images, out: np.ndarray, apply_transforms: bool = False, transforms=None, reduce=1):
        """Asynchronous decode_grids: returns a job; call ``wait_job(job)`` before reading ``out``."""
        images = list(images)
        arr = _desc_array(images)
        n_tiles = sum(im.n_tiles for im in images)
        st = (K.TileStatus * n_tiles)()
        job = C.c_void_p()
        ks = _reduce_list(reduce, len(images))
        if any(k != 1 for k in ks):
            xf = transforms if transforms is not None else [canvas_transform(im, apply_transforms) for im in images]
            K.check(self._lib.heic_b200_decode_grids_submit_reduced(self._h, arr, _transform_array(xf, len(images)), _reduce_array(ks),
                                                                    len(images), out.ctypes.data, out.strides[1], out.strides[0], st,
                                                                    C.byref(job)))
        elif transforms is None:
            K.check(self._lib.heic_b200_decode_grids_submit(self._h, arr, len(images), out.ctypes.data, out.strides[1], out.strides[0],
                                                            1 if apply_transforms else 0, st, C.byref(job)))
        else:
            K.check(self._lib.heic_b200_decode_grids_submit_transformed(self._h, arr, _transform_array(transforms, len(images)),
                                                                        len(images), out.ctypes.data, out.strides[1],
                                                                        out.strides[0], st, C.byref(job)))
        return (job, st, out)

    def unescape(self, nal_payload: bytes, data_offset: int = 0, substream_offsets=()):
        """GPU emulation-prevention removal of one raw NAL payload -> (rbsp, data_offset, substream_offsets) re-based."""
        n = len(substream_offsets)
        sub = (K.u32 * max(n, 1))(*substream_offsets)
        sub_out = (K.u32 * max(n, 1))()
        out = (K.u8 * max(len(nal_payload), 1))()
        out_len, off = C.c_size_t(), K.u32()
        K.check(self._lib.heic_b200_unescape(self._h, bytes(nal_payload), len(nal_payload), data_offset, sub, n, out, C.byref(out_len),
                                             C.byref(off), sub_out))
        return bytes(out[: out_len.value]), off.value, list(sub_out[:n])

    def wait_job(self, job) -> np.ndarray:
        h, st, out = job
        K.check(self._lib.heic_b200_job_wait(h))
        return out

    def decode_grids_yuv(self, images):
        """Batch -> list of (Y, Cb, Cr) planes cropped to the canvas (no colour conversion)."""
        images = list(images)
        arr = _desc_array(images)
        sizes = [_canvas(im, False) for im in images]
        ny = sum(w * h for w, h in sizes)
        nc = sum(((w + 1) // 2) * ((h + 1) // 2) for w, h in sizes)
        y, cb, cr = np.zeros(ny, np.uint8), np.zeros(nc, np.uint8), np.zeros(nc, np.uint8)
        K.check(self._lib.heic_b200_decode_grids_yuv(self._h, arr, len(images), y.ctypes.data, cb.ctypes.data, cr.ctypes.data, None))
        res, yo, co = [], 0, 0
        for w, h in sizes:
            cw, ch = (w + 1) // 2, (h + 1) // 2
            res.append((y[yo:yo + w * h].reshape(h, w), cb[co:co + cw * ch].reshape(ch, cw), cr[co:co + cw * ch].reshape(ch, cw)))
            yo += w * h
            co += cw * ch
        return res

    def batch(self, images, apply_transforms: bool = False, transforms=None, reduce=1) -> Batch:
        return Batch(self, images, apply_transforms, transforms, reduce)

    def color_stitch(self, dev_planes: int, n_images, grid_rows, grid_cols, tile_w, tile_h, out_w, out_h, dev_rgb: int,
                     pitch: int, image_stride: int, full_range: int = 1, matrix_coeffs: int = 6):
        """Stand-alone colour + stitch stage on caller-owned DEVICE buffers (raw device pointers)."""
        K.check(self._lib.heic_b200_color_stitch(self._h, dev_planes, n_images, grid_rows, grid_cols, tile_w, tile_h, out_w,
                                                 out_h, full_range, matrix_coeffs, dev_rgb, pitch, image_stride))
