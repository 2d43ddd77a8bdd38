"""Plain int64 numpy restatement of H.265 scaling and inverse transform for 8-bit 4:2:0 / 4:0:0 intra pictures:
chroma QP (8.6.1, Table 8-10), ScalingFactor (7.4.5 with the Table 7-5 / 7-6 defaults), scaling with the int16 clip,
transform skip, the 4x4 DST-VII and the 4..32 point DCTs as straight matrix products (8.6.4.2).  TEST INFRASTRUCTURE ONLY.

Independent of oracle/ and of the kernels: the matrices and default lists are typed here from the standard.  Input and
output use the decoder's dump layout: `tu_map` words (heif_b200/csrc/cuda/dev_types.h) and z-ordered, TU-contiguous
int16 coefficient arrays (a luma TU at tu_map index t owns the n*n slots from 16*t, raster inside the TU; its chroma
blocks sit at 16*(t >> 2) of the chroma arrays).  Besides the residuals, `residuals()` counts what the value-range tests
need to show they reached: escape-code prefix lengths, blocks on the kernels' 64-bit scaling path, saturated
coefficients, and first- and second-stage clips of the inverse transform.
"""
from __future__ import annotations

from collections import Counter

import numpy as np

# ---- 8.6.4.2 transform matrices --------------------------------------------------------------------------------------
DST4 = np.array([[29, 55, 74, 84],
                 [74, 74, 0, -74],
                 [84, -29, -74, 55],
                 [55, -84, 74, -29]], np.int64)
DCT4 = np.array([[64, 64, 64, 64],
                 [83, 36, -36, -83],
                 [64, -64, -64, 64],
                 [36, -83, 83, -36]], np.int64)
DCT8 = np.array([[64, 64, 64, 64, 64, 64, 64, 64],
                 [89, 75, 50, 18, -18, -50, -75, -89],
                 [83, 36, -36, -83, -83, -36, 36, 83],
                 [75, -18, -89, -50, 50, 89, 18, -75],
                 [64, -64, -64, 64, 64, -64, -64, 64],
                 [50, -89, 18, 75, -75, -18, 89, -50],
                 [36, -83, 83, -36, -36, 83, -83, 36],
                 [18, -50, 75, -89, 89, -75, 50, -18]], np.int64)
# The 32-point matrix: row k, column n is 64 * sqrt(2) * cos(pi * (2n + 1) * k / 64), rounded the way the standard's table
# is.  Its distinct magnitudes, by the angle a = (2n + 1) k mod 128 in units of pi / 64 (a = 0 only for the DC row):
_ODD32 = (90, 90, 88, 85, 82, 78, 73, 67, 61, 54, 46, 38, 31, 22, 13, 4)  # a = 1, 3, .., 31 (odd rows of the 32-point)
_ODD16 = (90, 87, 80, 70, 57, 43, 25, 9)                                  # a = 2, 6, .., 30
_ODD8 = (89, 75, 50, 18)                                                  # a = 4, 12, 20, 28
_ODD4 = (83, 36)                                                          # a = 8, 24


def _dct32():
    mag = np.zeros(33, np.int64)
    mag[0] = mag[16] = 64
    mag[1:32:2] = _ODD32
    mag[2:32:4] = _ODD16
    mag[4:32:8] = _ODD8
    mag[8:32:16] = _ODD4
    m = np.zeros((32, 32), np.int64)
    for k in range(32):
        for n in range(32):
            a = (2 * n + 1) * k % 128
            m[k, n] = mag[a] if a <= 32 else -mag[64 - a] if a <= 64 else -mag[a - 64] if a <= 96 else mag[128 - a]
    return m


DCT32 = _dct32()
DCT16 = DCT32[::2, :16]


def dct_matrix(n: int) -> np.ndarray:
    return {4: DCT4, 8: DCT8, 16: DCT16, 32: DCT32}[n]


# ---- 7.4.5 scaling factors ------------------------------------------------------------------------------------------
# Table 7-6, intra (matrixId 0..2) default for sizeId 1..3, in coded (up-right diagonal) order; Table 7-5: 4x4 all 16
DEFAULT_INTRA_8 = (16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 17, 16, 17, 16, 17, 18,
                   17, 18, 18, 17, 18, 21, 19, 20, 21, 20, 19, 21, 24, 22, 22, 24,
                   24, 22, 22, 24, 25, 25, 27, 30, 27, 25, 25, 29, 31, 35, 35, 31,
                   29, 36, 41, 44, 41, 36, 47, 54, 54, 47, 65, 70, 65, 88, 88, 115)
LEVEL_SCALE = (40, 45, 51, 57, 64, 72)
CHROMA_QP_30_42 = (29, 30, 31, 32, 33, 33, 34, 34, 35, 35, 36, 36, 37)  # Table 8-10, qPi = 30..42


def diag_scan(n: int):
    """6.5.3 up-right diagonal scan: list of (x, y)."""
    out, x, y = [], 0, 0
    while len(out) < n * n:
        while y >= 0:
            if x < n and y < n:
                out.append((x, y))
            y -= 1
            x += 1
        y, x = x, 0
    return out


def scan4(scan_idx: int):
    """ScanOrder[2][scanIdx]: (x, y) of the 16 positions of a 4x4 sub-block (diagonal, horizontal, vertical)."""
    if scan_idx == 0:
        return diag_scan(4)
    if scan_idx == 1:
        return [(i & 3, i >> 2) for i in range(16)]
    return [(i >> 2, i & 3) for i in range(16)]


def scaling_factors(sps, pps):
    """ScalingFactor per (log2 size, cIdx) as (n, n) int64 arrays indexed [y, x]; None when scaling lists are off (m = 16)."""
    if not sps.scaling_list_enabled_flag:
        return None
    if pps.pps_scaling_list_data_present_flag:
        sl = pps.scaling_list
    elif sps.sps_scaling_list_data_present_flag:
        sl = sps.scaling_list
    else:
        sl = None
    out = {}
    for size_id in range(4):
        n = 4 << size_id
        coded = diag_scan(4 if size_id == 0 else 8)
        for c in range(3):
            matrix_id = 0 if size_id == 3 else c  # intra; 32x32 blocks are luma only here
            if sl is None:
                lst = [16] * 16 if size_id == 0 else list(DEFAULT_INTRA_8)
                dc = 16
            else:
                lst = [sl.list[size_id][matrix_id][i] for i in range(16 if size_id == 0 else 64)]
                dc = sl.dc[size_id - 2][matrix_id] if size_id >= 2 else None
            f = np.zeros((n, n), np.int64)
            rep = max(1, n // 8)
            for i, (x, y) in enumerate(coded):
                f[y * rep:(y + 1) * rep, x * rep:(x + 1) * rep] = lst[i]
            if size_id >= 2:
                f[0, 0] = dc
            out[(size_id + 2, c)] = f
    return out


def chroma_qp(qp_y: int, offset: int) -> int:
    """8.6.1 for ChromaArrayType 1, 8-bit: Table 8-10 applied to qPi = Clip3(0, 57, QpY + offsets)."""
    qpi = min(57, max(0, qp_y + offset))
    if qpi < 30:
        return qpi
    if qpi > 42:
        return qpi - 6
    return CHROMA_QP_30_42[qpi - 30]


# ---- block-level scaling + transform -------------------------------------------------------------------------------
CLASSES = ("4y", "4c", "8", "16", "32", "tskip")  # the kernels' transform classes, transform-skip blocks apart


def block_class(log2: int, c_idx: int, tskip: bool) -> str:
    if tskip:
        return "tskip"
    if log2 == 2:
        return "4y" if c_idx == 0 else "4c"
    return str(1 << log2)


def _bits(v: int) -> int:
    return int(v).bit_length()


def scale_and_transform(lvl: np.ndarray, qp: int, m, log2: int, c_idx: int, tskip: bool, stats: dict) -> np.ndarray:
    """One n x n block of TransCoeffLevel -> residual (both int64 [y, x]); adds to `stats`."""
    n = 1 << log2
    cls = block_class(log2, c_idx, tskip)
    lvl = lvl.astype(np.int64)
    mm = np.full((n, n), 16, np.int64) if m is None or (tskip and n > 4) else m
    scale = LEVEL_SCALE[qp % 6] << (qp // 6)
    bd_shift = 8 + log2 - 5  # BitDepth + Log2(nTbS) - 5
    d = (lvl * mm * scale + (1 << (bd_shift - 1))) >> bd_shift
    stats["sat_pos"][cls] += int((d > 32767).sum())
    stats["sat_neg"][cls] += int((d < -32768).sum())
    d = np.clip(d, -32768, 32767)
    # the kernels' choice of a 32-bit product (8x8 .. 32x32): bits of the OR of the magnitudes (complements for negative
    # levels) plus bits of the largest factor * levelScale must stay <= 30; otherwise the 64-bit branch runs
    if log2 > 2 and not tskip:
        mag = int(np.bitwise_or.reduce((lvl ^ (lvl >> 63)).ravel()))
        if _bits(mag) + _bits((255 if m is not None else 16) * scale) > 30:
            stats["wide_blocks"] += 1
            if not (d.min() == -32768 or d.max() == 32767):
                stats["wide_unsaturated_blocks"] += 1
    if log2 == 2 and np.abs(lvl).max() > 255:
        stats["big_level_4x4_blocks"] += 1
    if tskip:
        ts_shift = 5 + log2
        return ((d << ts_shift) + (1 << 11)) >> 12  # bdShift = 20 - BitDepth
    mat = DST4 if (log2 == 2 and c_idx == 0) else dct_matrix(n)
    e = mat.T @ d                        # columns: y[i] = sum_j M[j][i] x[j]
    g = (e + 64) >> 7
    stats["first_clip"][cls] += int(((g > 32767) | (g < -32768)).sum())
    g = np.clip(g, -32768, 32767)
    r = (g @ mat + (1 << 11)) >> 12      # rows
    stats["second_clip"] += int(((r > 32767) | (r < -32768)).sum())
    return np.clip(r, -32768, 32767)


def _scan_idx(log2: int, c_idx: int, mode: int) -> int:
    if log2 == 2 or (log2 == 3 and c_idx == 0):
        if 6 <= mode <= 14:
            return 2
        if 22 <= mode <= 30:
            return 1
    return 0


def escape_prefixes(lvl: np.ndarray, log2: int, scan_idx: int, hist: Counter) -> None:
    """EG(k) prefix length of every coeff_abs_level_remaining of one block, rederived from its levels (7.3.8.11: which
    coefficients carry one and their baseLevel; 9.3.3.11: cRiceParam, reset per sub-block).  TR-only values count as -1."""
    order = scan4(scan_idx)[::-1]
    for ys in range(0, 1 << log2, 4):
        for xs in range(0, 1 << log2, 4):
            vals = [abs(int(lvl[ys + y, xs + x])) for x, y in order]
            vals = [v for v in vals if v]
            first_g1 = next((i for i, v in enumerate(vals[:8]) if v > 1), -1)
            rice = 0
            for i, v in enumerate(vals):
                if i < 8:
                    base = 1 + (v > 1) + (i == first_g1 and v > 2)
                    if base != (3 if i == first_g1 else 2):
                        continue
                else:
                    base = 1
                rem = v - base
                if rem < (4 << rice):
                    hist[-1] += 1
                else:
                    u, k, ones = rem - (4 << rice), rice + 1, 0
                    while u >= (1 << k):
                        u -= 1 << k
                        k += 1
                        ones += 1
                    hist[ones] += 1
                if v > 3 * (1 << rice):
                    rice = min(rice + 1, 4)


def new_stats() -> dict:
    return dict(prefix=Counter(), wide_blocks=0, wide_unsaturated_blocks=0, big_level_4x4_blocks=0,
                sat_pos=Counter({c: 0 for c in CLASSES}), sat_neg=Counter({c: 0 for c in CLASSES}),
                first_clip=Counter({c: 0 for c in CLASSES}), second_clip=0)


def residuals(sps, pps, sh, tu_map: np.ndarray, levels, stats: dict | None = None):
    """Residual arrays (int16, the layout of `levels`) of one picture; returns (residuals, stats)."""
    stats = new_stats() if stats is None else stats
    chroma = sps.chroma_format_idc == 1
    factors = scaling_factors(sps, pps)
    offsets = (0, pps.pps_cb_qp_offset + sh.slice_cb_qp_offset, pps.pps_cr_qp_offset + sh.slice_cr_qp_offset)
    out = [np.zeros_like(l) for l in levels]
    for t in np.flatnonzero(tu_map & 1):
        w = int(tu_map[t])
        log2 = ((w >> 1) & 3) + 2
        qp_y = (w >> 19) & 63
        blocks = []
        if w & (1 << 3):
            blocks.append((0, log2, 16 * int(t), (w >> 7) & 63))
        if chroma and w & (1 << 6):
            log2c = max(log2 - 1, 2)
            for c in (1, 2):
                if w & (1 << (3 + c)):
                    blocks.append((c, log2c, 16 * (int(t) >> 2), (w >> 13) & 63))
        for c, lg, off, mode in blocks:
            n = 1 << lg
            lvl = levels[c][off:off + n * n].reshape(n, n)
            tskip = bool((w >> (25 + c)) & 1)
            qp = qp_y if c == 0 else chroma_qp(qp_y, offsets[c])
            m = None if factors is None else factors[(lg, c)]
            res = scale_and_transform(lvl, qp, m, lg, c, tskip, stats)
            out[c][off:off + n * n] = res.astype(np.int16).ravel()
            escape_prefixes(lvl, lg, _scan_idx(lg, c, mode), stats["prefix"])
    return out, stats
