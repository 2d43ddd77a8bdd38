"""Colour-stage cost of each output geometry: STAGE_SAO | STAGE_COLOR on a resident batch of pool images (the fixture's
12 MP grid geometry, tiles drawn from the fixture and the synthetic pool as bench.py does), timed with CUDA events.

Geometries: identity (color_stitch_kernel), orientations 1..7 and an odd-origin crop (color_geom_kernel), and a grid of
conformance-cropped tiles (the same tiles with a conformance window in their SPS: 502 x 504 of every 512 x 512 picture).
Reports us per image and GB/s on the algorithmic traffic of 1.5 B in + 3 B out per output pixel, with the GPU's name and
power limit.  The rounds alternate the geometries, and the median round is reported.

    python tools/geometry_bench.py [--images 64] [--reps 10] [--rounds 3] [--out results/geometry_bench.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_description() -> str:
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True).strip()
    except (OSError, subprocess.CalledProcessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=64)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import ctypes as C

    import numpy as np
    import torch

    import heif_b200 as H
    from heif_b200 import _capi as K
    from tests.synth import pool as P

    data = open(os.path.join(ROOT, "tests", "golden", "halfmoonbay.heic"), "rb").read()
    f = H.HeicFile(data)
    pool = P.build_pool(f, n_synth=256)
    images, keep, _ = P.compose_images(pool, f.primary, range(args.images))
    W, Hh = f.primary.output_width, f.primary.output_height
    cropped = []
    for im in images:  # conformance window 3 / 2 / 1 / 3 (x2 luma samples): 502 x 504 tiles, canvas 8 x 502 - 9 by 6 x 504 - 5
        c = K.ImageDesc()
        C.memmove(C.byref(c), C.byref(im), C.sizeof(K.ImageDesc))
        c.sps.conformance_window_flag = 1
        c.sps.conf_win_left_offset, c.sps.conf_win_right_offset, c.sps.conf_win_top_offset, c.sps.conf_win_bottom_offset = 3, 2, 1, 3
        c.output_width, c.output_height = 8 * 502 - 9, 6 * 504 - 5
        cropped.append(c)
    cases = {"identity": (images, (0, 0, W, Hh, 0))}
    for o in range(1, 8):
        cases[f"orientation_{o}"] = (images, (0, 0, W, Hh, o))
    cases["odd_origin_crop"] = (images, (3, 5, W - 11, Hh - 7, 0))
    cases["conformance_cropped_grid"] = (cropped, (0, 0, 8 * 502 - 9, 6 * 504 - 5, 0))

    dec = H.HeicDecoder(device=0)
    batches = {}
    for name, (imgs, t) in cases.items():
        b = dec.batch(imgs, transforms=[t] * len(imgs))
        b.decode()
        b.sync()
        batches[name] = b
    times = {name: [] for name in cases}
    for _ in range(args.rounds):
        for name, b in batches.items():
            s = torch.cuda.ExternalStream(b.stream, device=torch.device("cuda", 0))
            b.run(H.STAGE_SAO | H.STAGE_COLOR)  # warm
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s)
            for _ in range(args.reps):
                b.run(H.STAGE_SAO | H.STAGE_COLOR)
            e1.record(s)
            b.sync()
            times[name].append(e0.elapsed_time(e1) / args.reps / args.images * 1e3)  # us per image
    res = {"gpu": gpu_description(), "images": args.images, "reps": args.reps, "rounds": args.rounds, "cases": {}}
    base = float(np.median(times["identity"]))
    for name, (imgs, t) in cases.items():
        us = float(np.median(times[name]))
        px = t[2] * t[3]
        res["cases"][name] = {"us_per_image": round(us, 2), "GB_per_s": round(4.5 * px / (us * 1e-6) / 1e9, 1),
                              "vs_identity": round(us / base, 3), "rounds_us": [round(x, 2) for x in times[name]]}
    for b in batches.values():
        b.close()
    dec.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
