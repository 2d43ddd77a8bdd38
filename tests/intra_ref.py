"""Plain numpy restatement of H.265 intra sample prediction (8.4.4.2.1 .. 8.4.4.2.6) and reconstruction for 8-bit
4:2:0 / 4:0:0 all-intra, single-slice pictures.  TEST INFRASTRUCTURE ONLY.

Independent of oracle/ and of the kernels: Tables 8-4 and 8-5 are typed here from the standard and every step follows its
text.  Input uses the decoder's dump layout: the `tu_map` words (heif_b200/csrc/cuda/dev_types.h: bit 0 marks a
transform unit origin, bits 1..2 its log2 size - 2, bits 3..5 cbf Y / Cb / Cr, bit 6 "carries the chroma blocks",
bits 7..12 IntraPredModeY, bits 13..18 IntraPredModeC; the index is the z-order 4x4 position inside the CTB, CTBs in
raster order) and the residuals, z-ordered and TU-contiguous (DESIGN.md section 2: a luma block whose first 4x4 unit has
index t owns the N * N values from 16 t, raster inside the block; a chroma block the n * n values from 4 t, t the index of
the 4x4 luma unit at its luma origin).

Decoding order is the tu_map walk: CTBs in raster order, transform units in z-order inside each CTB; luma, then the
chroma blocks of the unit.  The chroma blocks of an 8x8 luma block split into four 4x4 units are decoded with the fourth
unit (blkIdx 3).  A sample is available (6.4.1) iff it lies inside the picture and its z-scan address (MinTbAddrZs at 4x4
granularity: CTB raster address, then z-order inside the CTB -- the tu_map index) is below that of the current block.
Nothing here assumes that the available samples form one interval of the scan: the counters record any block where they
do not.

`reconstruct()` also counts, per component ("Y" / "C") and block size N, what the tests need to show they reached: modes,
filter decisions, bottom-left / above-right availability classes, missing left column / top row / everything,
negative-angle reference extension, chroma 4x4 blocks of split 8x8 units and blocks in partial CTBs.
"""
from __future__ import annotations

from collections import Counter, defaultdict
from functools import lru_cache

import numpy as np

BIT_DEPTH = 8
# Table 8-4: intraPredAngle for predModeIntra 2..34 (index = mode; planar and DC have none)
INTRA_PRED_ANGLE = (None, None, 32, 26, 21, 17, 13, 9, 5, 2, 0, -2, -5, -9, -13, -17, -21, -26,
                    -32, -26, -21, -17, -13, -9, -5, -2, 0, 2, 5, 9, 13, 17, 21, 26, 32)
# Table 8-5: invAngle for predModeIntra 11..25
INV_ANGLE = dict(zip(range(11, 26), (-4096, -1638, -910, -630, -482, -390, -315, -256, -315, -390, -482, -630, -910,
                                     -1638, -4096)))
# 8.4.4.2.3: intraHorVerDistThres[nTbS]
INTRA_HOR_VER_DIST_THRES = {8: 7, 16: 1, 32: 0}
assert len(INTRA_PRED_ANGLE) == 35


def new_stats():
    """Counters keyed by (component "Y" / "C", block size N)."""
    return defaultdict(Counter)


def _morton(z: int):
    return (sum(((z >> (2 * b)) & 1) << b for b in range(8)), sum(((z >> (2 * b + 1)) & 1) << b for b in range(8)))


# ---- 8.4.4.2.2: the reference sample scan ----------------------------------------------------------------------------
# The substitution process visits p[-1][2N-1] up to p[-1][-1], then p[0][-1] to p[2N-1][-1]: scan position s = 0 .. 4N.
# p[-1][y] is at s = 2N - 1 - y, the corner p[-1][-1] at s = 2N, p[x][-1] at s = 2N + 1 + x.
@lru_cache(maxsize=None)
def _scan(n: int):
    s = np.arange(4 * n + 1)
    dx = np.where(s <= 2 * n, -1, s - 2 * n - 1)
    dy = np.where(s <= 2 * n, 2 * n - 1 - s, -1)
    return dx, dy


def left(n, y):
    return 2 * n - 1 - y


def top(n, x):
    return 2 * n + 1 + x


def corner(n):
    return 2 * n


def substitute(avail: np.ndarray, samples: np.ndarray) -> np.ndarray:
    """8.4.4.2.2 over the scan: nothing available -> 1 << (BitDepth - 1) everywhere; else an unavailable p[-1][2N-1] takes
    the first available sample met going up and then right, and every later unavailable sample the one before it."""
    if not avail.any():
        return np.full(samples.shape, 1 << (BIT_DEPTH - 1), np.int32)
    pos = np.where(avail, np.arange(avail.size), -1)
    if not avail[0]:
        pos[0] = int(np.argmax(avail))
    pos = np.maximum.accumulate(pos)
    return samples[..., pos]


# ---- 8.4.4.2.6: angular prediction as taps into the scan ---------------------------------------------------------------
@lru_cache(maxsize=None)
def angular_taps(mode: int, n: int):
    """(a, b, fact, extended): predSamples[x][y] = ((32 - fact) * p[a] + fact * p[b] + 16) >> 5 for the scan array p,
    as [y, x] arrays; `extended`: the reference array was extended by invAngle projections.  ref[] is built exactly as
    8.4.4.2.6 builds it, holding scan positions instead of sample values."""
    angle = INTRA_PRED_ANGLE[mode]
    vertical = mode >= 18
    if vertical:  # ref[x] = p[-1 + x][-1]; the projection reads p[-1][-1 + k]
        main, side = (lambda i: corner(n) if i == 0 else top(n, i - 1)), (lambda k: corner(n) if k == 0 else left(n, k - 1))
    else:         # ref[x] = p[-1][-1 + x]; the projection reads p[-1 + k][-1]
        main, side = (lambda i: corner(n) if i == 0 else left(n, i - 1)), (lambda k: corner(n) if k == 0 else top(n, k - 1))
    ref = {x: main(x) for x in range(n + 1)}
    extended = False
    if angle < 0:
        if (n * angle) >> 5 < -1:
            extended = True
            for x in range((n * angle) >> 5, 0):
                ref[x] = side((x * INV_ANGLE[mode] + 128) >> 8)
    else:
        for x in range(n + 1, 2 * n + 1):
            ref[x] = main(x)
    a = np.zeros((n, n), np.intp)
    b = np.zeros((n, n), np.intp)
    fact = np.zeros((n, n), np.int32)
    for j in range(n):          # y for vertical modes, x for horizontal ones
        i_idx, i_fact = ((j + 1) * angle) >> 5, ((j + 1) * angle) & 31
        for i in range(n):
            yx = (j, i) if vertical else (i, j)
            a[yx] = ref[i + i_idx + 1]
            b[yx] = ref[i + i_idx + 2] if i_fact else a[yx]
            fact[yx] = i_fact
    return a, b, fact, extended


def predict(p: np.ndarray, n: int, mode: int, luma: bool) -> np.ndarray:
    """8.4.4.2.4 .. 8.4.4.2.6 from the (filtered) scan array p (shape [..., 4N + 1]): predSamples as [..., y, x]."""
    log2 = n.bit_length() - 1
    ys, xs = np.arange(n)[:, None], np.arange(n)[None, :]
    pl = p[..., left(n, np.arange(n))]    # p[-1][y]
    pt = p[..., top(n, np.arange(n))]     # p[x][-1]
    if mode == 0:  # planar
        return (((n - 1 - xs) * pl[..., :, None] + (xs + 1) * p[..., top(n, n), None, None]
                 + (n - 1 - ys) * pt[..., None, :] + (ys + 1) * p[..., left(n, n), None, None] + n) >> (log2 + 1))
    if mode == 1:  # DC
        dc = (pl.sum(-1) + pt.sum(-1) + n) >> (log2 + 1)
        pred = np.broadcast_to(dc[..., None, None], p.shape[:-1] + (n, n)).copy()
        if luma and n < 32:
            pred[..., 0, 0] = (p[..., left(n, 0)] + 2 * dc + p[..., top(n, 0)] + 2) >> 2
            pred[..., 0, 1:] = (pt[..., 1:] + 3 * dc[..., None] + 2) >> 2
            pred[..., 1:, 0] = (pl[..., 1:] + 3 * dc[..., None] + 2) >> 2
        return pred
    a, b, fact, _ = angular_taps(mode, n)
    pred = ((32 - fact) * p[..., a] + fact * p[..., b] + 16) >> 5
    if luma and n < 32:
        clip = (0, (1 << BIT_DEPTH) - 1)
        if mode == 26:
            pred[..., :, 0] = np.clip(p[..., top(n, 0), None] + ((pl - p[..., corner(n), None]) >> 1), *clip)
        elif mode == 10:
            pred[..., 0, :] = np.clip(p[..., left(n, 0), None] + ((pt - p[..., corner(n), None]) >> 1), *clip)
    return pred


def filter_samples(p: np.ndarray, n: int, mode: int, strong_enabled: bool, counts: Counter) -> np.ndarray:
    """8.4.4.2.3 on the luma scan array p (1-D): the filtered array, with the decision counted."""
    if mode == 1 or n == 4 or min(abs(mode - 26), abs(mode - 10)) <= INTRA_HOR_VER_DIST_THRES[n]:
        counts["filter_none"] += 1
        return p
    if strong_enabled and n == 32:
        c0, bl, tr = int(p[corner(n)]), int(p[left(n, 2 * n - 1)]), int(p[top(n, 2 * n - 1)])
        dev_tr = abs(c0 + tr - 2 * int(p[top(n, n - 1)]))
        dev_bl = abs(c0 + bl - 2 * int(p[left(n, n - 1)]))
        thres = 1 << (BIT_DEPTH - 5)
        if dev_tr < thres and dev_bl < thres:  # biIntFlag: bilinear between the corner and the two far ends
            counts["filter_strong"] += 1
            pf = p.copy()
            for i in range(2 * n - 1):
                pf[left(n, i)] = ((63 - i) * c0 + (i + 1) * bl + 32) >> 6
                pf[top(n, i)] = ((63 - i) * c0 + (i + 1) * tr + 32) >> 6
            return pf
        counts["filter_strong_rejected"] += 1
        counts["reject_" + ("both" if min(dev_tr, dev_bl) >= thres else "bl" if dev_bl >= thres else "tr")] += 1
        if max(dev_tr, dev_bl) == thres:
            counts["reject_at_threshold"] += 1  # every failing test fails by equality: "<=" would have taken it
    else:
        counts["filter_121"] += 1
    pf = p.copy()  # [1 2 1] along the scan; its two ends are kept
    pf[1:-1] = (p[:-2] + 2 * p[1:-1] + p[2:] + 2) >> 2
    return pf


def _count_availability(counts: Counter, n: int, avail: np.ndarray, inside: np.ndarray) -> None:
    for name, seg in (("bl", slice(0, n)), ("tr", slice(3 * n + 1, 4 * n + 1))):
        got, pic = int(avail[seg].sum()), int(inside[seg].sum())
        cls = "none" if got == 0 else "full" if got == n else "partial"
        counts[f"{name}_{cls}"] += 1
        if cls == "partial":
            counts[f"{name}_partial_{'edge' if got == pic else 'order'}"] += 1
    left_col, top_row = avail[n:2 * n].any(), avail[2 * n + 1:3 * n + 1].any()
    if not avail.any():
        counts["none_available"] += 1
    elif not left_col and top_row:
        counts["left_missing"] += 1
    elif left_col and not top_row:
        counts["top_missing"] += 1
    runs = np.count_nonzero(np.diff(np.concatenate(([0], avail.astype(np.int8), [0]))) == 1)
    if runs > 1:
        counts["not_one_interval"] += 1


def reconstruct(sps, tu_map, resid, stats=None):
    """The reconstructed planes (uint8, before the loop filters) of one picture, and the counters."""
    stats = new_stats() if stats is None else stats
    w, h = sps.pic_width_in_luma_samples, sps.pic_height_in_luma_samples
    log2_ctb = sps.log2_min_luma_coding_block_size_minus3 + 3 + sps.log2_diff_max_min_luma_coding_block_size
    ctb, ctb4 = 1 << log2_ctb, 1 << (log2_ctb - 2)
    wctb, hctb = -(-w >> log2_ctb), -(-h >> log2_ctb)
    chroma = sps.chroma_format_idc == 1
    strong_enabled = bool(sps.strong_intra_smoothing_enabled_flag)
    tu_map = np.asarray(tu_map)
    # z-scan address of every 4x4 luma unit of the CTB grid (6.5.2 at 4x4 granularity): the tu_map index
    zaddr = np.zeros((hctb * ctb4, wctb * ctb4), np.int64)
    for z in range(ctb4 * ctb4):
        x4, y4 = _morton(z)
        zaddr[y4::ctb4, x4::ctb4] = np.arange(hctb * wctb).reshape(hctb, wctb) * ctb4 * ctb4 + z
    rec_y = np.zeros((hctb * ctb, wctb * ctb), np.int32)
    rec_c = np.zeros((2, hctb * ctb // 2, wctb * ctb // 2), np.int32)
    res = [np.asarray(r, np.int32) for r in resid]

    def block(rec, sub, x0, y0, n, mode, addr, cbfs, offs, split_chroma):
        luma = sub == 0
        counts = stats[("Y" if luma else "C", n)]
        counts[("mode", mode)] += 1
        if split_chroma:
            counts["split_chroma_4x4"] += 1
        if (((x0 << sub) >> log2_ctb) + 1) * ctb > w or (((y0 << sub) >> log2_ctb) + 1) * ctb > h:
            counts["partial_ctb"] += 1
        dx, dy = _scan(n)
        xs, ys = x0 + dx, y0 + dy
        inside = (xs >= 0) & (ys >= 0) & (xs < (w >> sub)) & (ys < (h >> sub))
        xi, yi = np.clip(xs, 0, (w >> sub) - 1), np.clip(ys, 0, (h >> sub) - 1)
        avail = inside & (zaddr[(yi << sub) >> 2, (xi << sub) >> 2] < addr)
        _count_availability(counts, n, avail, inside)
        p = substitute(avail, rec[..., yi, xi])
        if luma:
            p = filter_samples(p, n, mode, strong_enabled, counts)
        if mode >= 2 and angular_taps(mode, n)[3]:
            counts["negative_angle_extended"] += 1
        pred = predict(p, n, mode, luma)
        out = rec[..., y0:y0 + n, x0:x0 + n]
        for k, (cbf, off) in enumerate(zip(cbfs, offs)):
            blk = pred if luma else pred[k]
            dst = out if luma else out[k]
            dst[...] = np.clip(blk + res[off[0]][off[1]:off[1] + n * n].reshape(n, n), 0, 255) if cbf else blk

    for t in np.flatnonzero(tu_map & 1):
        word = int(tu_map[t])
        n = 4 << ((word >> 1) & 3)
        ctb_addr, z = divmod(int(t), ctb4 * ctb4)
        x4, y4 = _morton(z)
        x0, y0 = ((ctb_addr % wctb) << log2_ctb) + 4 * x4, ((ctb_addr // wctb) << log2_ctb) + 4 * y4
        block(rec_y, 0, x0, y0, n, (word >> 7) & 63, int(t), [(word >> 3) & 1], [(0, 16 * int(t))], False)
        if chroma and word & (1 << 6):
            split = n == 4  # the chroma 4x4 of an 8x8 split into four luma 4x4 units: at the 8x8's origin
            xl, yl = (x0 - 4, y0 - 4) if split else (x0, y0)
            base = int(zaddr[yl >> 2, xl >> 2])
            block(rec_c, 1, xl >> 1, yl >> 1, 4 if split else n >> 1, (word >> 13) & 63, int(t),
                  [(word >> 4) & 1, (word >> 5) & 1], [(1, 4 * base), (2, 4 * base)], split)
    planes = [rec_y[:h, :w].astype(np.uint8)]
    if chroma:
        planes += [rec_c[k, :h // 2, :w // 2].astype(np.uint8) for k in range(2)]
    return planes, stats
