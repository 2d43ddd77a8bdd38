"""Cost and benefit of the box reduction (heic_b200_decode_grids_reduced), on pool images of the fixture's 12 MP grid
geometry (tiles drawn from the fixture and the synthetic pool as bench.py does).

1. Colour stage: STAGE_SAO | STAGE_COLOR on a resident batch, timed with CUDA events, for k in {1, 2, 4, 8} x
   orientations {0, 1, 6} (k = 1 is color_stitch_kernel / color_geom_kernel, k > 1 color_reduce_kernel).  Reports us per
   image and GB/s on the algorithmic traffic of 1.5 B in + 3 / k^2 B out per canvas pixel.  The rounds alternate the cases,
   and the median round is reported.
2. Serving loop: calls of --call-images images through HeicDecoder.submit_grids / wait_job with 3 calls in
   flight (pinned host RGB, as bench.py's e2e), and the synchronous call one at a time, for k in {1, 2, 4, 8}: canvas MP/s
   (12.19 MP per image, whatever k) and the device->host bytes per call.  The rounds alternate the factors.

The GPU's name and power limit are read in the same run.

    python tools/reduce_bench.py [--images 64] [--reps 10] [--rounds 3] [--call-images 296] [--calls 8] [--out results/reduce_bench.json]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

FACTORS = (1, 2, 4, 8)
ORIENTATIONS = (0, 1, 6)
N_BUF = 3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=64)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--call-images", type=int, default=296)
    ap.add_argument("--calls", type=int, default=8)
    ap.add_argument("--serving-rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch

    import bench
    import heif_b200 as H
    from geometry_bench import gpu_description
    from tests.synth import pool as P

    gpu = gpu_description()
    data = open(os.path.join(ROOT, "tests", "golden", "halfmoonbay.heic"), "rb").read()
    f = H.HeicFile(data)
    pool = P.build_pool(f, n_synth=256)
    W, Hh = f.primary.output_width, f.primary.output_height
    mp = W * Hh / 1e6
    dec = H.HeicDecoder(device=0)

    # ---- 1. colour stage ----------------------------------------------------------------------------------
    images, keep, _ = P.compose_images(pool, f.primary, range(args.images))
    cases = {(k, o): None for k in FACTORS for o in ORIENTATIONS}
    for k, o in cases:
        b = dec.batch(images, transforms=[(0, 0, W, Hh, o)] * len(images), reduce=k)
        b.decode()
        b.sync()
        cases[(k, o)] = b
    times = {c: [] for c in cases}
    for _ in range(args.rounds):
        for c, b in cases.items():
            s = torch.cuda.ExternalStream(b.stream, device=torch.device("cuda", 0))
            b.run(H.STAGE_SAO | H.STAGE_COLOR)  # warm
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s)
            for _ in range(args.reps):
                b.run(H.STAGE_SAO | H.STAGE_COLOR)
            e1.record(s)
            b.sync()
            times[c].append(e0.elapsed_time(e1) / args.reps / args.images * 1e3)  # us per image
    stage = {}
    for (k, o), b in cases.items():
        us = float(np.median(times[(k, o)]))
        traffic = W * Hh * (1.5 + 3.0 / (k * k))
        stage[f"k{k}_orientation_{o}"] = {"us_per_image": round(us, 2), "GB_per_s": round(traffic / (us * 1e-6) / 1e9, 1),
                                          "out_bytes_per_image": int(b.rgb_layout()[2]),
                                          "rounds_us": [round(x, 2) for x in times[(k, o)]]}
        b.close()
    del cases

    # ---- 2. serving loop ----------------------------------------------------------------------------------
    n = args.call_images
    fit = int(0.4 * bench.host_memory_available() / (N_BUF * W * Hh * 3))  # pinned buffers of the k = 1 case
    n = max(8, min(n, fit // 8 * 8)) if fit < n else n
    images, keep, _ = P.compose_images(pool, f.primary, range(n))
    full = [(0, 0, W, Hh, 0)] * n
    serving = {k: {"pipelined_s": [], "sync_s": []} for k in FACTORS}
    for _ in range(args.serving_rounds):
        for k in FACTORS:
            ow, oh = -(-W // k), -(-Hh // k)
            bufs = [torch.empty((n, oh, ow, 3), dtype=torch.uint8, pin_memory=True) for _ in range(N_BUF)]
            outs = [x.numpy() for x in bufs]
            for i in range(2 * N_BUF):  # every pipeline slot and every buffer touched before the timed region
                dec.decode_grids(images, out=outs[i % N_BUF], transforms=full, reduce=k)
            t0 = time.perf_counter()
            jobs = []
            for i in range(args.calls):
                if len(jobs) >= N_BUF:
                    dec.wait_job(jobs.pop(0))
                jobs.append(dec.submit_grids(images, outs[i % N_BUF], transforms=full, reduce=k))
            for j in jobs:
                dec.wait_job(j)
            serving[k]["pipelined_s"].append((time.perf_counter() - t0) / args.calls)
            t0 = time.perf_counter()
            for _ in range(2):
                dec.decode_grids(images, out=outs[0], transforms=full, reduce=k)
            serving[k]["sync_s"].append((time.perf_counter() - t0) / 2)
            del outs, bufs
    serve = {}
    for k in FACTORS:
        pipe, sync = float(np.median(serving[k]["pipelined_s"])), float(np.median(serving[k]["sync_s"]))
        serve[f"k{k}"] = {"d2h_bytes_per_call": n * -(-W // k) * -(-Hh // k) * 3,
                          "pipelined_3_in_flight_MPps": round(n * mp / pipe, 1), "sync_MPps": round(n * mp / sync, 1),
                          "pipelined_ms_per_call": [round(x * 1e3, 1) for x in serving[k]["pipelined_s"]],
                          "sync_ms_per_call": [round(x * 1e3, 1) for x in serving[k]["sync_s"]]}
    dec.close()
    res = {"gpu": gpu, "colour_stage": {"images": args.images, "reps": args.reps, "rounds": args.rounds, "cases": stage},
           "serving": {"images_per_call": n, "calls": args.calls, "rounds": args.serving_rounds, "MP_per_image": round(mp, 3),
                       "factors": serve}}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
