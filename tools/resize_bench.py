"""Cost and benefit of the resize (heic_b200_decode_grids_resized), on pool images of the fixture's 12 MP grid geometry
(tiles drawn from the fixture and the synthetic pool as bench.py does).

1. Stage time: STAGE_SAO | STAGE_COLOR on a resident batch (SAO + colour + the resampling passes), timed with CUDA
   events, for sizes (224, 224), (1024, 768), (2016, 1512) x {BILINEAR, BICUBIC, LANCZOS}, each without and with
   reduce=4 first, against k = 1 with no resize.  Reports us per 12 MP image.  The rounds alternate the cases, and the
   median round is reported.
2. Serving loop: calls of --call-images images through heic_b200_decode_grids_submit_resized / _job_wait with 3 calls in
   flight (pinned host RGB, as bench.py's e2e), and the synchronous call one at a time, at 224 x 224 BICUBIC against the
   full-size call: canvas MP/s (12.19 MP per image, whatever the output size) and the device->host bytes per call.

The GPU's name and power limit are read in the same run.

    python tools/resize_bench.py [--images 32] [--reps 10] [--rounds 3] [--call-images 296] [--calls 8] [--out results/resize_bench.json]
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

SIZES = ((224, 224), (1024, 768), (2016, 1512))
FILTERS = {"BILINEAR": 2, "BICUBIC": 3, "LANCZOS": 1}
N_BUF = 3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=32)
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
    full = [(0, 0, W, Hh, 0)]

    # ---- 1. stage time ------------------------------------------------------------------------------------
    images, keep, _ = P.compose_images(pool, f.primary, range(args.images))
    cases = {("none", "-", 1): None}
    for size in SIZES:
        for name in FILTERS:
            for k in (1, 4):
                cases[(f"{size[0]}x{size[1]}", name, k)] = None
    for key in cases:
        size, name, k = key
        rs = None if size == "none" else tuple(int(v) for v in size.split("x"))
        b = dec.batch(images, transforms=full * len(images), reduce=k, resize=rs, resample=FILTERS.get(name, 3))
        b.decode()
        b.sync()
        cases[key] = b
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
    base = float(np.median(times[("none", "-", 1)]))
    for (size, name, k), b in cases.items():
        us = float(np.median(times[(size, name, k)]))
        stage[f"{size}_{name}_k{k}"] = {"us_per_image": round(us, 2), "over_unresized_us": round(us - base, 2),
                                        "rounds_us": [round(x, 2) for x in times[(size, name, k)]]}
        b.close()
    del cases

    # ---- 2. serving loop ----------------------------------------------------------------------------------
    n = args.call_images
    fit = int(0.4 * bench.host_memory_available() / (N_BUF * W * Hh * 3))  # pinned buffers of the full-size case
    n = max(8, min(n, fit // 8 * 8)) if fit < n else n
    images, keep, _ = P.compose_images(pool, f.primary, range(n))
    modes = {"full": None, "224x224_BICUBIC": (224, 224)}
    serving = {m: {"pipelined_s": [], "sync_s": []} for m in modes}
    for _ in range(args.serving_rounds):
        for m, rs in modes.items():
            ow, oh = rs if rs else (W, Hh)
            bufs = [torch.empty((n, oh, ow, 3), dtype=torch.uint8, pin_memory=True) for _ in range(N_BUF)]
            outs = [x.numpy() for x in bufs]
            kw = dict(transforms=full * n, resize=rs, resample=3)
            for i in range(2 * N_BUF):  # every pipeline slot and every buffer touched before the timed region
                dec.decode_grids(images, out=outs[i % N_BUF], **kw)
            t0 = time.perf_counter()
            jobs = []
            for i in range(args.calls):
                if len(jobs) >= N_BUF:
                    dec.wait_job(jobs.pop(0))
                jobs.append(dec.submit_grids(images, outs[i % N_BUF], **kw))
            for j in jobs:
                dec.wait_job(j)
            serving[m]["pipelined_s"].append((time.perf_counter() - t0) / args.calls)
            t0 = time.perf_counter()
            for _ in range(2):
                dec.decode_grids(images, out=outs[0], **kw)
            serving[m]["sync_s"].append((time.perf_counter() - t0) / 2)
            del outs, bufs
    serve = {}
    for m, rs in modes.items():
        ow, oh = rs if rs else (W, Hh)
        pipe, sync = float(np.median(serving[m]["pipelined_s"])), float(np.median(serving[m]["sync_s"]))
        serve[m] = {"d2h_bytes_per_call": n * ow * oh * 3,
                    "pipelined_3_in_flight_MPps": round(n * mp / pipe, 1), "sync_MPps": round(n * mp / sync, 1),
                    "pipelined_ms_per_call": [round(x * 1e3, 1) for x in serving[m]["pipelined_s"]],
                    "sync_ms_per_call": [round(x * 1e3, 1) for x in serving[m]["sync_s"]]}
    dec.close()
    res = {"gpu": gpu, "stage": {"images": args.images, "reps": args.reps, "rounds": args.rounds, "cases": stage},
           "serving": {"images_per_call": n, "calls": args.calls, "rounds": args.serving_rounds, "MP_per_image": round(mp, 3),
                       "modes": serve}}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
