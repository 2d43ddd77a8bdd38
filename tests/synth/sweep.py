"""A seeded random sweep over the synthetic encoder's configuration space (tests/synth/synth.py), next to the hand-picked
CONFIGS / EXTREME_CONFIGS.  TEST INFRASTRUCTURE ONLY.

Every case is a legal combination: CTB 16 / 32 / 64 with min CB 8 .. CTB, MinTb < MinCb, MaxTb <= min(CTB, 32), any
transform hierarchy depth the sizes allow; picture sizes that are multiples of MinCb up to 256 x 256, a quarter of
them one CTB wide or high; 4:2:0 or 4:0:0; WPP on or off; SAO off, on, luma only or chroma only, with a random share of
CTBs that code it; deblocking off or on with beta / tC offsets -6..6; SliceQpY 0..51 through init_qp_minus26 -26..25
and slice_qp_delta; cu_qp_delta at any depth; PPS and slice chroma QP offsets whose sums stay within +-12; every scaling
list mode with random entry ranges; transform skip, sign data hiding, strong intra smoothing; large escape-coded levels,
CU split bias, full / limited range and BT.601 / BT.709.

cases() is a pure function of its seed: the same seed gives the same list, configurations and stream seeds alike.
Budget: encoding the default SWEEP (SWEEP_CASES pictures), decoding it with the CPU oracle and FFmpeg and running
tests/loopfilter_ref.py over it takes a few seconds of one CPU core; the CPU tests built on it
(tests/test_loopfilter_reference.py) must stay within two minutes on one core.  Raise SWEEP_CASES only within that.
"""
from __future__ import annotations

import random

SWEEP_SEED = 20261021
SWEEP_CASES = 120
MAX_SIDE = 256


def _case(r: random.Random) -> dict:
    log2_ctb = r.choice((4, 5, 6))
    log2_min_cb = r.randint(3, log2_ctb)
    log2_min_tb = r.randint(2, log2_min_cb - 1)
    log2_max_tb = r.randint(log2_min_tb, min(5, log2_ctb))
    cb, ctb = 1 << log2_min_cb, 1 << log2_ctb
    shape = r.random()
    if shape < 0.12:    # one CTB row
        width, height = cb * r.randint(1, MAX_SIDE // cb), cb * r.randint(1, ctb // cb)
    elif shape < 0.24:  # one CTB column
        width, height = cb * r.randint(1, ctb // cb), cb * r.randint(1, MAX_SIDE // cb)
    else:
        width, height = cb * r.randint(1, MAX_SIDE // cb), cb * r.randint(1, MAX_SIDE // cb)
    init_qp_minus26 = r.randint(-26, 25)
    slice_qp = r.choice((26 + init_qp_minus26, r.randint(0, 51)))
    cfg = dict(width=width, height=height, log2_ctb=log2_ctb, log2_min_cb=log2_min_cb, log2_min_tb=log2_min_tb,
               log2_max_tb=log2_max_tb, max_transform_hierarchy_depth_intra=r.randint(0, log2_ctb - log2_min_tb),
               chroma_format_idc=0 if r.random() < 0.15 else 1, wpp=r.randint(0, 1),
               init_qp_minus26=init_qp_minus26, slice_qp_delta=slice_qp - 26 - init_qp_minus26,
               transform_skip=r.randint(0, 1), sign_data_hiding=r.randint(0, 1), strong_intra_smoothing=r.randint(0, 1),
               full_range=r.randint(0, 1), matrix_coeffs=r.choice((1, 6)), lps_gain=round(r.uniform(0.5, 2.0), 2))
    sao = r.random()
    if sao < 0.15:
        cfg.update(sao=0)
    else:
        cfg.update(sao=1, slice_sao_luma=int(sao >= 0.3), slice_sao_chroma=int(sao < 0.3 or sao >= 0.45))
        if r.random() < 0.5:
            cfg.update(sao_on_prob=round(r.uniform(0.05, 0.95), 2))
    if r.random() < 0.15:
        cfg.update(deblocking_disabled=1)
    else:
        cfg.update(beta_offset_div2=r.randint(-6, 6), tc_offset_div2=r.randint(-6, 6))
    if r.random() < 0.5:
        cfg.update(cu_qp_delta=1, diff_cu_qp_delta_depth=r.randint(0, log2_ctb - log2_min_cb))
    for c in ("cb", "cr"):
        pps = r.randint(-12, 12)
        cfg[f"{c}_qp_offset"] = pps
        cfg[f"slice_{c}_qp_offset"] = r.randint(-12 - min(pps, 0), 12 - max(pps, 0)) if r.random() < 0.5 else 0
    cfg["scaling_list_mode"] = r.randint(0, 3)
    if cfg["scaling_list_mode"] >= 2 and r.random() < 0.5:
        lo, hi = sorted((r.randint(1, 255), r.randint(1, 255)))
        cfg.update(scaling_list_min=lo, scaling_list_max=hi)
    if r.random() < 0.25:
        cfg.update(big_level_prob=round(r.uniform(0.02, 0.3), 3))
    if r.random() < 0.5:
        cfg.update(split_cu_prob=round(r.uniform(0.1, 0.9), 2))
    return cfg


def cases(seed: int = SWEEP_SEED, n: int = SWEEP_CASES) -> list[tuple[str, dict, int]]:
    """(name, encoder config, stream seed) of n random legal configurations."""
    r = random.Random(seed)
    out = []
    for i in range(n):
        cfg = _case(r)
        name = (f"s{i:03d}_ctb{1 << cfg['log2_ctb']}_{cfg['width']}x{cfg['height']}"
                f"{'_400' if cfg['chroma_format_idc'] == 0 else ''}")
        out.append((name, cfg, r.randrange(1 << 20)))
    return out


SWEEP = cases()
