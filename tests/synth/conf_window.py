"""Synthetic pictures with an SPS conformance window.  TEST INFRASTRUCTURE ONLY.

The encoder (hevc_synth.cc) writes conformance_window_flag = 0.  A conformance window changes nothing the slice data
depends on, so a windowed picture is the encoder's picture with its SPS rewritten: conformance_window_flag = 1 and the
four conf_win_*_offset values inserted (7.3.2.2), the RBSP trailing bits redone and emulation prevention re-applied.
The pictures without a window, and their bytes, stay exactly what synth.encode makes."""
from __future__ import annotations

import heif_b200 as H
from tests.synth import synth


class _Bits:
    def __init__(self, data: bytes):
        self.bits = "".join(f"{b:08b}" for b in data)
        self.pos = 0

    def u(self, n: int) -> int:
        v = int(self.bits[self.pos:self.pos + n], 2) if n else 0
        self.pos += n
        return v

    def ue(self) -> int:
        z = 0
        while self.bits[self.pos] == "0":
            z += 1
            self.pos += 1
        self.pos += 1
        return (1 << z) - 1 + self.u(z)


def _ue(v: int) -> str:
    b = f"{v + 1:b}"
    return "0" * (len(b) - 1) + b


def _escape(rbsp: bytes) -> bytes:
    out, zeros = bytearray(), 0
    for b in rbsp:
        if zeros >= 2 and b <= 3:
            out.append(3)
            zeros = 0
        out.append(b)
        zeros = zeros + 1 if b == 0 else 0
    return bytes(out)


def add_conformance_window(sps_nal: bytes, left: int, right: int, top: int, bottom: int) -> bytes:
    """The SPS NAL unit (2-byte header + escaped payload) with the given conformance window offsets (in chroma units:
    SubWidthC / SubHeightC luma samples each).  The input must have conformance_window_flag = 0 and one sub-layer."""
    r = _Bits(H.remove_emulation_prevention(sps_nal[2:]))
    r.u(4)                                      # sps_video_parameter_set_id
    if r.u(3) != 0:                             # sps_max_sub_layers_minus1
        raise ValueError("only single-layer SPS are rewritten")
    r.u(1)                                      # sps_temporal_id_nesting_flag
    r.u(2 + 1 + 5 + 32 + 4 + 43 + 1 + 8)        # profile_tier_level(1, 0)
    r.ue()                                      # sps_seq_parameter_set_id
    if r.ue() == 3:                             # chroma_format_idc
        r.u(1)
    r.ue()
    r.ue()                                      # pic_width / pic_height_in_luma_samples
    at = r.pos
    if r.u(1):
        raise ValueError("the SPS already has a conformance window")
    body = r.bits[:at] + "1" + "".join(_ue(v) for v in (left, right, top, bottom)) + r.bits[at + 1:]
    body = body[:body.rindex("1")] + "1"        # rbsp_stop_one_bit, then byte alignment
    body += "0" * (-len(body) % 8)
    rbsp = bytes(int(body[i:i + 8], 2) for i in range(0, len(body), 8))
    return bytes(sps_nal[:2]) + _escape(rbsp)


def encode(seed: int, window=(0, 0, 0, 0), **cfg) -> synth.Picture:
    """synth.encode(seed, **cfg) with the conformance window (left, right, top, bottom); the descriptor's canvas is the
    window's size, as a HEIF reader sets it for a single item."""
    vps, sps, pps, slice_nal = synth.encode_nals(seed, **cfg)
    if any(window):
        sps = add_conformance_window(sps, *window)
    vals = dict(synth.DEFAULTS)
    vals.update(cfg)
    pic = synth.Picture((vps, sps, pps, slice_nal), vals)
    for d in (pic.desc, pic.desc_raw):
        d.output_width, d.output_height = H.tile_size(d)
    return pic
