"""Plain numpy restatement of the H.265 in-loop filters for 8-bit 4:2:0 / 4:0:0 intra pictures: deblocking (8.7.2) and
sample adaptive offset (8.7.3).  TEST INFRASTRUCTURE ONLY.

Independent of oracle/ and of the kernels: the tables are typed here from the standard and every step follows its text.
Input uses the decoder's dump layout: the reconstructed planes, `tu_map` words (heif_b200/csrc/cuda/dev_types.h; bit 0
marks a transform block origin, bits 1..2 its log2 size - 2; the index is the z-order 4x4 position inside the CTB, CTBs
in raster order), the 8x8 `qp_map` of QpY and the four SAO words per CTB (Y, Cb, Cr, unused: bits 0..1 SaoTypeIdx,
bits 2..6 sao_band_position or SaoEoClass, 4-bit two's-complement SaoOffsetVal[1..4] from bit 8).

Intra pictures keep this simple: every coding block is intra, so bS is 2 on every transform-block edge of the 8x8 grid
(8.7.2.4) and 0 elsewhere; coding-block edges are transform-block edges (the transform tree's root is the coding block);
one slice, no tiles, no PCM and no transquant bypass.  Vertical edges never share a sample they write with another
vertical edge 8 samples away, so all vertical edges of the picture are filtered at once from the reconstructed picture,
then all horizontal edges from that result: the order 8.7.2 prescribes.  SAO reads the fully deblocked picture only.

`loop_filter()` also counts what the tests need to show they reached: luma segments per decision (skipped by dE = 0,
strong, normal, and normal with dEp / dEq), chroma segments filtered, SAO CTBs per type and edge class per component,
and SAO at CTB boundaries: samples changed there, and samples whose result depends on a neighbour in another CTB that
deblocking changed (so reading the neighbour before deblocking would give another value).
"""
from __future__ import annotations

from collections import Counter

import numpy as np

# Table 8-11: beta' for Q = 0..51
BETA_TABLE = (0,) * 16 + (6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18) + tuple(range(20, 65, 2))
# Table 8-12: tC' for Q = 0..53
TC_TABLE = (0,) * 18 + (1,) * 9 + (2,) * 4 + (3,) * 4 + (4,) * 3 + (5, 5, 6, 6, 7, 8, 9, 10, 11, 13, 14, 16, 18, 20, 22, 24)
# Table 8-10: QpC for qPi = 30..42 (qPi < 30: QpC = qPi; qPi > 42: QpC = qPi - 6)
QPC_30_42 = (29, 30, 31, 32, 33, 33, 34, 34, 35, 35, 36, 36, 37)
# Table 8-13 (8.7.3.2): hPos / vPos of the two neighbours per SaoEoClass
EO_NEIGHBOURS = (((-1, 0), (1, 0)), ((0, -1), (0, 1)), ((-1, -1), (1, 1)), ((1, -1), (-1, 1)))  # ((dx, dy) a, (dx, dy) b)
assert len(BETA_TABLE) == 52 and len(TC_TABLE) == 54


def qpc_from_qpi(qpi: int) -> int:
    if qpi < 30:
        return qpi
    if qpi > 42:
        return qpi - 6
    return QPC_30_42[qpi - 30]


def new_stats() -> dict:
    return dict(luma=Counter(skipped=0, strong=0, normal=0, dEp=0, dEq=0), chroma_filtered=0, chroma_tc0=0,
                sao={c: Counter(band=0, eo0=0, eo1=0, eo2=0, eo3=0) for c in range(3)},
                sao_boundary_changed=Counter({c: 0 for c in range(3)}),
                sao_reads_deblocked_across_ctb=Counter({c: 0 for c in range(3)}))


def _geometry(sps):
    log2_ctb = sps.log2_min_luma_coding_block_size_minus3 + 3 + sps.log2_diff_max_min_luma_coding_block_size
    return sps.pic_width_in_luma_samples, sps.pic_height_in_luma_samples, log2_ctb


def transform_edges(sps, tu_map: np.ndarray):
    """edgeFlags of 8.7.2.3 on the 8x8 grid, picture boundary excluded: (vertical [y4, x8], horizontal [y8, x4]).
    vertical[j, i] is the edge at luma x = 8 i over rows 4 j .. 4 j + 3; horizontal[j, i] the edge at y = 8 j over
    columns 4 i .. 4 i + 3."""
    w, h, log2_ctb = _geometry(sps)
    ctb4 = 1 << (log2_ctb - 2)
    wctb = -(-w >> log2_ctb)
    ver = np.zeros((h >> 2, w >> 3), bool)
    hor = np.zeros((h >> 3, w >> 2), bool)
    for t in np.flatnonzero(tu_map & 1):
        word = int(tu_map[t])
        n = 4 << ((word >> 1) & 3)
        ctb, z = divmod(int(t), ctb4 * ctb4)
        x4 = sum(((z >> (2 * b)) & 1) << b for b in range(4))
        y4 = sum(((z >> (2 * b + 1)) & 1) << b for b in range(4))
        x0 = ((ctb % wctb) << log2_ctb) + 4 * x4
        y0 = ((ctb // wctb) << log2_ctb) + 4 * y4
        if x0 > 0 and x0 % 8 == 0:
            ver[y0 >> 2:(y0 + n) >> 2, x0 >> 3] = True
        if y0 > 0 and y0 % 8 == 0:
            hor[y0 >> 3, x0 >> 2:(x0 + n) >> 2] = True
    return ver, hor


def _luma_edges(a: np.ndarray, edges: np.ndarray, qp: np.ndarray, beta_off: int, tc_off: int, stats: dict) -> None:
    """8.7.2.5.3 + 8.7.2.5.6 / 8.7.2.5.7 on the vertical edges of `a` (int32, modified in place).  edges[j, i]: the
    segment of rows 4 j .. 4 j + 3 at x = 8 i, bS 2.  qp: QpY per 8x8 block, same orientation as `a`."""
    seg, col = np.nonzero(edges)
    if not len(seg):
        return
    lines = 4 * seg[:, None] + np.arange(4)                      # [n, line]
    taps = np.arange(4)
    xq = 8 * col
    rows = lines[:, :, None]
    p = a[rows, (xq[:, None] - 1 - taps)[:, None, :]]            # p[n, line, i] = p_i of that line
    q = a[rows, (xq[:, None] + taps)[:, None, :]]
    qp_p = qp[seg >> 1, col - 1].astype(np.int64)                # the CUs holding p0,0 and q0,0
    qp_q = qp[seg >> 1, col].astype(np.int64)
    qpl = (qp_q + qp_p + 1) >> 1
    beta = np.array(BETA_TABLE)[np.clip(qpl + 2 * beta_off, 0, 51)]
    tc = np.array(TC_TABLE)[np.clip(qpl + 2 * (2 - 1) + 2 * tc_off, 0, 53)]
    dp_l = np.abs(p[:, :, 2] - 2 * p[:, :, 1] + p[:, :, 0])      # per line; only lines 0 and 3 decide
    dq_l = np.abs(q[:, :, 2] - 2 * q[:, :, 1] + q[:, :, 0])
    dpq0, dpq3 = dp_l[:, 0] + dq_l[:, 0], dp_l[:, 3] + dq_l[:, 3]
    dp, dq = dp_l[:, 0] + dp_l[:, 3], dq_l[:, 0] + dq_l[:, 3]
    d = dpq0 + dpq3

    def dsam(k, dpq):  # 8.7.2.5.6
        return ((2 * dpq < (beta >> 2)) & (np.abs(p[:, k, 3] - p[:, k, 0]) + np.abs(q[:, k, 0] - q[:, k, 3]) < (beta >> 3))
                & (np.abs(p[:, k, 0] - q[:, k, 0]) < ((5 * tc + 1) >> 1)))

    on = d < beta
    strong = on & dsam(0, dpq0) & dsam(3, dpq3)                  # dE = 2
    normal = on & ~strong                                        # dE = 1
    dep = normal & (dp < ((beta + (beta >> 1)) >> 3))
    deq = normal & (dq < ((beta + (beta >> 1)) >> 3))
    stats["luma"].update(skipped=int((~on).sum()), strong=int(strong.sum()), normal=int(normal.sum()),
                         dEp=int(dep.sum()), dEq=int(deq.sum()))
    t = tc[:, None]
    p0, p1, p2, p3 = (p[:, :, i] for i in range(4))
    q0, q1, q2, q3 = (q[:, :, i] for i in range(4))
    newp, newq = p.copy(), q.copy()
    # strong (8-339 .. 8-344)
    s = strong[:, None] & np.ones((1, 4), bool)
    sp = [np.clip((p2 + 2 * p1 + 2 * p0 + 2 * q0 + q1 + 4) >> 3, p0 - 2 * t, p0 + 2 * t),
          np.clip((p2 + p1 + p0 + q0 + 2) >> 2, p1 - 2 * t, p1 + 2 * t),
          np.clip((2 * p3 + 3 * p2 + p1 + p0 + q0 + 4) >> 3, p2 - 2 * t, p2 + 2 * t)]
    sq = [np.clip((p1 + 2 * p0 + 2 * q0 + 2 * q1 + q2 + 4) >> 3, q0 - 2 * t, q0 + 2 * t),
          np.clip((p0 + q0 + q1 + q2 + 2) >> 2, q1 - 2 * t, q1 + 2 * t),
          np.clip((p0 + q0 + q1 + 3 * q2 + 2 * q3 + 4) >> 3, q2 - 2 * t, q2 + 2 * t)]
    for i in range(3):
        newp[:, :, i] = np.where(s, sp[i], newp[:, :, i])
        newq[:, :, i] = np.where(s, sq[i], newq[:, :, i])
    # normal (8-345 .. 8-354), per line: nothing changes where abs(delta) >= tC * 10
    delta = (9 * (q0 - p0) - 3 * (q1 - p1) + 8) >> 4
    n = normal[:, None] & (np.abs(delta) < t * 10)
    delta = np.clip(delta, -t, t)
    newp[:, :, 0] = np.where(n, np.clip(p0 + delta, 0, 255), newp[:, :, 0])
    newq[:, :, 0] = np.where(n, np.clip(q0 - delta, 0, 255), newq[:, :, 0])
    dlt_p = np.clip((((p2 + p0 + 1) >> 1) - p1 + delta) >> 1, -(t >> 1), t >> 1)
    dlt_q = np.clip((((q2 + q0 + 1) >> 1) - q1 - delta) >> 1, -(t >> 1), t >> 1)
    newp[:, :, 1] = np.where(n & dep[:, None], np.clip(p1 + dlt_p, 0, 255), newp[:, :, 1])
    newq[:, :, 1] = np.where(n & deq[:, None], np.clip(q1 + dlt_q, 0, 255), newq[:, :, 1])
    a[rows, (xq[:, None] - 1 - taps)[:, None, :]] = newp
    a[rows, (xq[:, None] + taps)[:, None, :]] = newq


def _chroma_edges(a: np.ndarray, edges: np.ndarray, qp: np.ndarray, qp_offset: int, tc_off: int, stats: dict) -> None:
    """8.7.2.5.5 on the vertical edges of chroma plane `a` (int32, in place).  edges / qp: the luma edge flags
    [y4, x8] and QpY per luma 8x8 block, same orientation.  Chroma edges lie on the 8-sample chroma grid (16 luma),
    one segment is 4 chroma lines, its bS is the luma one at the segment's first line."""
    ce = edges[0::2, 0::2].copy()                                # [chroma 4-line segment, chroma x / 8]
    ce[:, 0] = False
    seg, col = np.nonzero(ce)
    if not len(seg):
        return
    rows = 4 * seg[:, None] + np.arange(4)
    xq = 8 * col[:, None]
    qp_p = qp[seg, 2 * col - 1].astype(np.int64)                 # luma of p0,0 is (16 col - 2, 8 seg)
    qp_q = qp[seg, 2 * col].astype(np.int64)
    qpi = ((qp_q + qp_p + 1) >> 1) + qp_offset                   # cQpPicOffset: the PPS offset only
    qpc = np.array([qpc_from_qpi(int(v)) for v in qpi], np.int64)
    tc = np.array(TC_TABLE)[np.clip(qpc + 2 * (2 - 1) + 2 * tc_off, 0, 53)][:, None]
    stats["chroma_filtered"] += int((tc > 0).sum())
    stats["chroma_tc0"] += int((tc == 0).sum())
    p0, p1, q0, q1 = a[rows, xq - 1], a[rows, xq - 2], a[rows, xq], a[rows, xq + 1]
    delta = np.clip((((q0 - p0) << 2) + p1 - q1 + 4) >> 3, -tc, tc)
    a[rows, xq - 1] = np.clip(p0 + delta, 0, 255)
    a[rows, xq] = np.clip(q0 - delta, 0, 255)


def deblock(sps, pps, sh, recon, tu_map, qp_map, stats: dict | None = None):
    """8.7.2: the deblocked planes (uint8) of one picture."""
    stats = new_stats() if stats is None else stats
    if sh.slice_deblocking_filter_disabled_flag:
        return [np.array(p, np.uint8) for p in recon], stats
    ver, hor = transform_edges(sps, tu_map)
    out = [np.array(p, np.int32) for p in recon]
    qp = np.asarray(qp_map)
    offsets = (0, pps.pps_cb_qp_offset, pps.pps_cr_qp_offset)
    beta_off, tc_off = sh.slice_beta_offset_div2, sh.slice_tc_offset_div2
    # EDGE_VER over the whole picture, then EDGE_HOR on its result; horizontal edges are the vertical ones of the
    # transposed picture
    _luma_edges(out[0], ver, qp, beta_off, tc_off, stats)
    for c in range(1, len(out)):
        _chroma_edges(out[c], ver, qp, offsets[c], tc_off, stats)
    t = [np.ascontiguousarray(p.T) for p in out]
    _luma_edges(t[0], hor.T, qp.T, beta_off, tc_off, stats)
    for c in range(1, len(out)):
        _chroma_edges(t[c], hor.T, qp.T, offsets[c], tc_off, stats)
    return [np.ascontiguousarray(p.T).astype(np.uint8) for p in t], stats


def unpack_sao(word: int):
    """(SaoTypeIdx, band position or EO class, SaoOffsetVal[0..4]) of one SAO word."""
    offs = [0]
    for k in range(4):
        o = (word >> (8 + 4 * k)) & 15
        offs.append(o - 16 if o >= 8 else o)
    return word & 3, (word >> 2) & 31, offs


def edge_idx(plane: np.ndarray, cls: int):
    """8.7.3.2 edgeIdx (after the remap, 0..4) of every sample for one SaoEoClass, and whether both neighbours lie in
    the picture (elsewhere the sample is left unchanged)."""
    h, w = plane.shape
    v = plane.astype(np.int32)
    pad = np.pad(v, 1, mode="edge")
    valid = np.ones((h, w), bool)
    e = np.full((h, w), 2, np.int32)
    for dx, dy in EO_NEIGHBOURS[cls]:
        nb = pad[1 + dy:1 + dy + h, 1 + dx:1 + dx + w]
        e += np.sign(v - nb)
        ys, xs = np.arange(h)[:, None] + dy, np.arange(w)[None, :] + dx
        valid &= (ys >= 0) & (ys < h) & (xs >= 0) & (xs < w)
    e = np.where(e == 0, 1, np.where(e == 1, 2, np.where(e == 2, 0, e)))  # edgeIdx 0, 1, 2 -> 1, 2, 0
    return e, valid


def sao(sps, sh, deblocked, recon, sao_words, stats: dict | None = None):
    """8.7.3: the final planes (uint8).  `recon` is only used to count samples whose result depends on deblocking of a
    neighbour in another CTB."""
    stats = new_stats() if stats is None else stats
    w, h, log2_ctb = _geometry(sps)
    wctb, hctb = -(-w >> log2_ctb), -(-h >> log2_ctb)
    words = np.asarray(sao_words).reshape(-1, 4)
    out = []
    for c, plane in enumerate(deblocked):
        src = plane.astype(np.int32)
        dst = src.copy()
        enabled = sps.sample_adaptive_offset_enabled_flag and (sh.slice_sao_chroma_flag if c else sh.slice_sao_luma_flag)
        if not enabled:
            out.append(dst.astype(np.uint8))
            continue
        cs = (1 << log2_ctb) >> (1 if c else 0)
        ph, pw = src.shape
        eo = [edge_idx(src, k) for k in range(4)]
        pre = np.asarray(recon[c]).astype(np.int32)
        ctb_x = np.arange(pw) // cs
        ctb_y = np.arange(ph) // cs
        for ry in range(hctb):
            for rx in range(wctb):
                wd = words[ry * wctb + rx]
                _, pos, offs = unpack_sao(int(wd[c]))
                # Cr takes Cb's SaoTypeIdx and SaoEoClass (7.4.9.3.2); its offsets and band position are its own
                typ, cls = unpack_sao(int(wd[1 if c == 2 else c]))[:2]
                if typ == 0:
                    continue
                ys, xs = slice(ry * cs, min((ry + 1) * cs, ph)), slice(rx * cs, min((rx + 1) * cs, pw))
                s = src[ys, xs]
                offs = np.array(offs, np.int32)
                if typ == 1:  # band offset: bandShift = bitDepth - 5
                    table = np.zeros(32, np.int32)
                    for k in range(4):
                        table[(k + pos) & 31] = k + 1
                    dst[ys, xs] = np.clip(s + offs[table[s >> 3]], 0, 255)
                    stats["sao"][c]["band"] += 1
                    continue
                e, valid = eo[cls][0][ys, xs], eo[cls][1][ys, xs]
                dst[ys, xs] = np.where(valid, np.clip(s + offs[e], 0, 255), s)
                stats["sao"][c][f"eo{cls}"] += 1
                # samples whose result would differ had SAO read their neighbours in other CTBs before deblocking
                yy, xx = np.mgrid[ys, xs]
                e_alt = np.full(e.shape, 2, np.int32)
                for dx, dy in EO_NEIGHBOURS[cls]:
                    ny, nx = np.clip(yy + dy, 0, ph - 1), np.clip(xx + dx, 0, pw - 1)
                    other = (ctb_y[ny] != ry) | (ctb_x[nx] != rx)
                    e_alt += np.sign(s - np.where(other, pre[ny, nx], src[ny, nx]))
                e_alt = np.where(e_alt == 0, 1, np.where(e_alt == 1, 2, np.where(e_alt == 2, 0, e_alt)))
                stats["sao_reads_deblocked_across_ctb"][c] += int((valid & (offs[e] != offs[e_alt])).sum())
        border = np.zeros(src.shape, bool)
        border[:, 0::cs] = border[:, cs - 1::cs] = True
        border[0::cs, :] = border[cs - 1::cs, :] = True
        stats["sao_boundary_changed"][c] += int(((dst != src) & border).sum())
        out.append(dst.astype(np.uint8))
    return out, stats


def loop_filter(sps, pps, sh, recon, tu_map, qp_map, sao_words, stats: dict | None = None):
    """Deblocking then SAO of one picture: (deblocked planes, final planes, stats)."""
    stats = new_stats() if stats is None else stats
    deblocked, stats = deblock(sps, pps, sh, recon, tu_map, qp_map, stats)
    final, stats = sao(sps, sh, deblocked, recon, sao_words, stats)
    return deblocked, final, stats
