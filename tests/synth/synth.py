"""Python face of the synthetic HEVC intra bitstream generator (tests/synth/hevc_synth.cc).  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import heif_b200 as H
from heif_b200 import _capi as K

HERE = os.path.dirname(os.path.abspath(__file__))


class Config(C.Structure):
    _fields_ = [
        ("width", C.c_uint32), ("height", C.c_uint32), ("chroma_format_idc", C.c_uint32), ("log2_min_cb", C.c_uint32),
        ("log2_ctb", C.c_uint32), ("log2_min_tb", C.c_uint32), ("log2_max_tb", C.c_uint32),
        ("max_transform_hierarchy_depth_intra", C.c_uint32), ("scaling_list_mode", C.c_uint32), ("sao", C.c_uint32),
        ("strong_intra_smoothing", C.c_uint32), ("sign_data_hiding", C.c_uint32), ("transform_skip", C.c_uint32),
        ("cu_qp_delta", C.c_uint32), ("diff_cu_qp_delta_depth", C.c_uint32), ("init_qp_minus26", C.c_int32),
        ("slice_qp_delta", C.c_int32), ("cb_qp_offset", C.c_int32), ("cr_qp_offset", C.c_int32),
        ("slice_cb_qp_offset", C.c_int32), ("slice_cr_qp_offset", C.c_int32), ("wpp", C.c_uint32),
        ("deblocking_disabled", C.c_uint32), ("beta_offset_div2", C.c_int32), ("tc_offset_div2", C.c_int32),
        ("slice_sao_luma", C.c_uint32), ("slice_sao_chroma", C.c_uint32), ("full_range", C.c_uint32),
        ("matrix_coeffs", C.c_uint32), ("lps_gain", C.c_double), ("max_bypass_ones", C.c_uint32),
        ("sao_on_prob", C.c_double), ("split_cu_prob", C.c_double), ("big_level_prob", C.c_double),
        ("scaling_list_min", C.c_uint32), ("scaling_list_max", C.c_uint32), ("cbf_prob", C.c_double),
        ("prev_intra_prob", C.c_double),
    ]


DEFAULTS = dict(width=128, height=128, chroma_format_idc=1, log2_min_cb=3, log2_ctb=5, log2_min_tb=2, log2_max_tb=5,
                max_transform_hierarchy_depth_intra=0, scaling_list_mode=0, sao=1, strong_intra_smoothing=0, sign_data_hiding=0,
                transform_skip=0, cu_qp_delta=0, diff_cu_qp_delta_depth=0, init_qp_minus26=0, slice_qp_delta=0, cb_qp_offset=0,
                cr_qp_offset=0, slice_cb_qp_offset=0, slice_cr_qp_offset=0, wpp=1, deblocking_disabled=0, beta_offset_div2=0,
                tc_offset_div2=0, slice_sao_luma=1, slice_sao_chroma=1, full_range=1, matrix_coeffs=6, lps_gain=1.0,
                max_bypass_ones=0, sao_on_prob=-1.0, split_cu_prob=-1.0, big_level_prob=0.0, scaling_list_min=8, scaling_list_max=63,
                cbf_prob=-1.0, prev_intra_prob=-1.0)

_lib = None


def _load():
    global _lib
    if _lib is None:
        subprocess.check_call(["make", "-s", "-C", HERE])
        _lib = C.CDLL(os.path.join(HERE, "_build", "libhevc_synth.so"))
        _lib.synth_encode_picture.argtypes = [C.POINTER(Config), C.c_uint64] + [C.c_void_p] * 4 + [C.c_size_t, C.POINTER(C.c_size_t)]
        _lib.synth_level_remaining_roundtrip.argtypes = [C.c_int, C.c_uint32, C.c_uint64, C.POINTER(C.c_uint32)]
    return _lib


def level_remaining_roundtrip(rice: int, value: int, seed: int):
    """coeff_abs_level_remaining `value` encoded as bypass bins and decoded by the device routine and by the bin-by-bin
    loop (see hevc_synth.cc).  Returns (flags, (device value, device bins), (loop value, loop bins), encoded bins)."""
    out = (C.c_uint32 * 5)()
    rc = _load().synth_level_remaining_roundtrip(rice, value, seed, out)
    return rc, (out[0], out[1]), (out[2], out[3]), out[4]


class Picture:
    """One synthetic coded picture: NAL units + the host-parsed descriptor the decode API takes."""

    def __init__(self, nals, cfg):
        self.vps, self.sps_nal, self.pps_nal, self.slice_nal = nals
        self.cfg = cfg
        self.sps = H.parse_sps(H.remove_emulation_prevention(self.sps_nal[2:]))
        self.pps = H.parse_pps(H.remove_emulation_prevention(self.pps_nal[2:]))
        rbsp, epb = H.remove_emulation_prevention(self.slice_nal[2:], with_positions=True)
        self._rbsp = (K.u8 * len(rbsp)).from_buffer_copy(rbsp)
        self.header = H.parse_slice_header(rbsp, 20, self.sps, self.pps, epb)
        self._tiles = (K.TileDesc * 1)()
        self._tiles[0].rbsp = C.cast(self._rbsp, C.POINTER(K.u8))
        self._tiles[0].rbsp_len = len(rbsp)
        self._tiles[0].nal_unit_type = 20
        self._tiles[0].header = self.header
        d = K.ImageDesc()
        d.sps, d.pps = self.sps, self.pps
        d.grid_rows = d.grid_cols = 1
        d.output_width, d.output_height = self.sps.pic_width_in_luma_samples, self.sps.pic_height_in_luma_samples
        d.n_tiles = 1
        d.tiles = C.cast(self._tiles, C.POINTER(K.TileDesc))
        self.desc = d
        self.n_epb = len(epb)
        # the same picture as a raw NAL payload: emulation prevention removal and entry-point re-basing happen on the GPU
        payload = self.slice_nal[2:]
        self._raw = (K.u8 * len(payload)).from_buffer_copy(payload)
        self._tiles_raw = (K.TileDesc * 1)()
        self._tiles_raw[0].rbsp = C.cast(self._raw, C.POINTER(K.u8))
        self._tiles_raw[0].rbsp_len = len(payload)
        self._tiles_raw[0].nal_unit_type = 20
        self._tiles_raw[0].escaped = 1
        self._tiles_raw[0].header = H.parse_slice_header_raw(payload, 20, self.sps, self.pps)
        r = K.ImageDesc()
        C.memmove(C.byref(r), C.byref(d), C.sizeof(K.ImageDesc))
        r.tiles = C.cast(self._tiles_raw, C.POINTER(K.TileDesc))
        self.desc_raw = r

    @property
    def tile(self):
        return self._tiles[0]

    def annexb(self) -> bytes:
        return b"".join(b"\x00\x00\x00\x01" + n for n in (self.vps, self.sps_nal, self.pps_nal, self.slice_nal))


def encode(seed: int, **kw) -> Picture:
    """Deterministic: the same (seed, config) always yields the same bytes.  Retries the seed when the random walk hits a
    non-conformant value (rare; e.g. CuQpDeltaVal out of range)."""
    nals, vals = _encode(seed, kw)
    return Picture(nals, vals)


def encode_nals(seed: int, **kw):
    """The four NAL units (VPS, SPS, PPS, slice) of encode(seed, **kw) without parsing them; safe to call from threads."""
    return _encode(seed, kw)[0]


def _encode(seed: int, kw):
    lib = _load()
    vals = dict(DEFAULTS)
    vals.update(kw)
    if vals["cu_qp_delta"] and not vals["max_bypass_ones"]:
        vals["max_bypass_ones"] = 3
    cfg = Config(**vals)
    cap = (1 << 20) if vals["width"] * vals["height"] <= 512 * 512 else (8 << 20)  # four output buffers of this size per call
    bufs = [C.create_string_buffer(cap) for _ in range(4)]
    lens = (C.c_size_t * 4)()
    for attempt in range(64):
        rc = lib.synth_encode_picture(C.byref(cfg), seed + 1000003 * attempt, *[C.cast(b, C.c_void_p) for b in bufs], cap, lens)
        if rc == 0:
            return [bufs[i].raw[: lens[i]] for i in range(4)], vals
        if rc != -3:
            raise ValueError(f"synth_encode_picture rejected the configuration (rc={rc}): {vals}")
    raise RuntimeError("no conformant random walk found in 64 attempts")
