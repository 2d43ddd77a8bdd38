#!/usr/bin/env python
"""bench.py — decoded MP/s of the HEIC hot path (slice data -> RGB) on a batch of 12 MP 8x6 grid images.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference ...                      (CPU arm: the oracle port on all host cores)

Workload = SURVEY section 8(d) config 5: images composed by rng(seed=1) from a pool of 48 real tiles (halfmoonbay.heic)
+ 512 synthetic 512x512 WPP tiles (tests/synth: the in-repo CABAC encoder, under the fixture's own SPS/PPS), sharded
image_idx % n_gpus (heif_b200/sharding.py).  A step = one decode of one resident batch of --batch images per GPU.  `value`
times K steps with the batch already in HBM (CUDA events on the library's stream); `e2e` times the reference-facing C-ABI
call heic_b200_decode_grids_submit/_job_wait with HOST descriptors/bitstreams in and pinned HOST RGB out.  No data-path
collective (weak scaling).  The run FAILS on a wrong pixel: after warm-up, random images of the resident batch and of the
e2e output are compared with the CPU oracle, and every 32-lane CABAC group is checked to hold 32 different tiles.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FIXTURE = os.path.join(ROOT, "tests", "golden", "halfmoonbay.heic")
OUT_W, OUT_H = 4032, 3024
MP_PER_IMAGE = OUT_W * OUT_H / 1e6
TILE_W = TILE_H = 512
TILE_BYTES = TILE_W * TILE_H * 3 // 2
CODED_SAMPLES_PER_IMAGE = 48 * TILE_BYTES
SEED = 1


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.p = [], None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0: float, t1: float):
        if not self.p:
            return None
        time.sleep(0.15)
        self.p.terminate()
        rows = [r for ts, r in self.rows if t0 - 0.05 <= ts <= t1 + 0.15 and len(r) >= 6] or [r for _, r in self.rows if len(r) >= 6]
        if not rows:
            return None
        try:
            sm = sorted(float(r[0]) for r in rows)
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            reasons = sorted({n for r in rows for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
            return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "reasons": reasons, "samples": len(rows)}
        except ValueError:
            return None


def host_memory_available() -> int:
    """Bytes of host memory this process may still use: MemAvailable, capped by the cgroup limit if there is one."""
    avail = 64 << 30
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                avail = int(line.split()[1]) * 1024
    except OSError:
        pass
    for lim, cur in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                     ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            m = open(lim).read().strip()
            if m != "max" and int(m) < (1 << 60):
                avail = min(avail, int(m) - int(open(cur).read().strip()))
        except (OSError, ValueError):
            pass
    return max(avail, 0)


def bind_to_gpu_numa_node(index: int) -> str:
    """CPU affinity of this process := the CPUs NVML names as closest to GPU `index`.  Best effort; says what it did."""
    try:
        import pynvml

        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = index
        if vis:
            ent = vis.split(",")[index].strip()
            if ent.isdigit():
                phys = int(ent)
            else:
                return f"not bound (CUDA_VISIBLE_DEVICES={vis})"
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = {64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "not bound (NVML reports no local CPUs)"
        os.sched_setaffinity(0, cpus)
        return f"{len(cpus)} CPUs local to GPU {phys}"
    except Exception as e:  # noqa: BLE001 - any failure leaves the default affinity
        return f"not bound ({type(e).__name__}: {e})"


# ---------------------------------------------------------------------------------------------------------
# CPU side: the oracle port (oracle/hevc_oracle.c) on the host cores.  kind = "port": the reference is Rust, there is no
# cargo/rustc in the image, and its slice decoder ends in todo!() anyway (DESIGN.md, "Oracle").  It serves twice: as the
# checker of the GPU pixels and as the timed CPU baseline / reference arm.
# ---------------------------------------------------------------------------------------------------------
class CpuDecoder:
    """Decodes images of the job with the oracle.  All buffers are allocated up front; the timed part is C calls only
    (hevc_oracle_decode_picture per tile, hevc_oracle_color_stitch per grid row), spread over `threads` host threads."""

    def __init__(self, pool, base_image, threads: int):
        from concurrent.futures import ThreadPoolExecutor

        from oracle import oracle_py

        oracle_py.load()
        self.O = oracle_py
        self.pool, self.img, self.threads = pool, base_image, threads
        self.ex = ThreadPoolExecutor(threads)

    def decode(self, ids: np.ndarray, planes: np.ndarray, rgb: np.ndarray) -> float:
        """ids [n, 48] pool entries -> planes [n, 48, TILE_BYTES], rgb [n, OUT_H, OUT_W, 3]; returns seconds."""
        O, pool, img = self.O, self.pool, self.img
        n, nt = ids.shape
        cols, rows = img.grid_cols, img.grid_rows
        fr, mc = img.sps.video_full_range_flag, img.sps.matrix_coeffs

        def tile(k):
            i, t = divmod(k, nt)
            td = pool.descs[int(ids[i, t])]
            O.decode_picture_into(pool.sps, pool.pps, td.header, td.rbsp, td.rbsp_len, planes[i, t])

        def row(k):  # colour + stitch of one grid row (the last row is cropped by the canvas height)
            i, r = divmod(k, rows)
            O.color_stitch_into(planes[i, r * cols].ctypes.data, 1, cols, TILE_W, TILE_H, OUT_W, min(TILE_H, OUT_H - r * TILE_H),
                                fr, mc, rgb[i, r * TILE_H].ctypes.data, OUT_W * 3)

        t0 = time.perf_counter()
        list(self.ex.map(tile, range(n * nt)))
        list(self.ex.map(row, range(n * rows)))
        return time.perf_counter() - t0


def ffmpeg_decode_images(heic_file, n_images: int, threads: int):
    """FFmpeg's native HEVC decoder (planes only, no colour conversion) on the fixture's real tiles, one decoder per thread.
    Extra context next to the oracle port: 'what a CPU does today'.  Returns seconds, or None when FFmpeg is absent."""
    try:
        from concurrent.futures import ThreadPoolExecutor

        from oracle.ffmpeg_oracle import FFmpegHevc, annexb
    except Exception:
        return None
    try:
        ps = [heic_file.parameter_set_nal(t) for t in (32, 33, 34)]
        aus = [annexb(ps + [heic_file.tile_nal(t)]) for t in range(heic_file.primary.n_tiles)]
        local = threading.local()

        def one(i):
            if not hasattr(local, "dec"):
                local.dec = FFmpegHevc()
            local.dec.decode_picture(aus[i % len(aus)])

        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(one, range(threads)))  # warm up: one decoder per thread
            t0 = time.perf_counter()
            list(ex.map(one, range(n_images * len(aus))))
            return time.perf_counter() - t0
    except Exception:
        return None


# the workload both arms name in `config` (BASELINE.json configs[4], image-sharded)
WORKLOAD = ("configs[4] sharded: 12 MP 8x6 grid images of 512x512 HEVC intra tiles (WPP, SAO, deblock, scaling lists) -> RGB 4032x3024; "
            "tiles drawn by rng(seed=1) from a pool of 48 real + 512 synthetic tiles (SURVEY 8(d) config 5)")


def data_note(pool):
    c = pool.composition()
    return (f"pool of {c['real_tiles']} real tiles (halfmoonbay.heic) + {c['synthetic_tiles']} synthetic 512x512 WPP tiles (in-repo CABAC "
            f"encoder, QP / lps_gain sweep; slice bytes min/quartiles/max real {c['slice_bytes_quartiles_real']}, synthetic "
            f"{c['slice_bytes_quartiles_synthetic']}); every image = 48 distinct pool tiles by rng(seed={SEED}, image_idx)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # The CPU arm reads its inputs through a host-only build of the repo's parse layer (oracle/_build/libheic_host.so):
    # the product library libheic_b200.so is never mapped into this process.
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])
    from heif_b200 import _capi

    _capi.load(os.path.join(ROOT, "oracle", "_build", "libheic_host.so"), host_only=True)
    import heif_b200
    from tests.synth import pool as P

    f = heif_b200.HeicFile(open(FIXTURE, "rb").read())
    cores = os.cpu_count() or 1
    pool = P.build_pool(f, args.pool)
    n_img = max(1, args.ref_images)
    ids = np.stack([P.image_tile_ids(len(pool), i, f.primary.n_tiles, SEED) for i in range(n_img)])
    cpu = CpuDecoder(pool, f.primary, cores)
    planes = np.zeros((n_img, 48, TILE_BYTES), np.uint8)
    rgb = np.zeros((n_img, OUT_H, OUT_W, 3), np.uint8)
    for _ in range(args.warmup):
        cpu.decode(ids, planes, rgb)
    dt = sum(cpu.decode(ids, planes, rgb) for _ in range(args.steps))
    value = args.steps * n_img * MP_PER_IMAGE / dt
    sample = f"images 0..{n_img - 1} of the job = {48 * n_img} tiles per step, oracle port (C, -O3), {cores} threads"
    print(json.dumps({
        "impl": "reference", "metric": "decoded MP/s (12MP HEIC grid batch)", "value": round(value, 3), "unit": "MP/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": data_note(pool) + ", CPU",
        "config": {"workload": WORKLOAD, "images_per_step": n_img, "note": "bounded CPU sample of the same workload"},
        "cpu_baseline": {"value": round(value, 3), "unit": "MP/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": round(value, 3), "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def check_groups_distinct(batch, ids_flat: np.ndarray) -> dict:
    """Every CABAC warp-group must hold different pool tiles (copies of one tile in a warp would run converged)."""
    order, tpg = batch.cabac_order()
    if tpg != 32:
        return {"tiles_per_group": tpg}
    g = order.reshape(-1, 32)
    valid = g != 0xFFFFFFFF
    pid = np.where(valid, ids_flat[np.where(valid, g, 0)], -1 - np.arange(32)[None, :])  # idle lanes: unique dummies
    s = np.sort(pid, axis=1)
    dup = int((s[:, 1:] == s[:, :-1]).any(axis=1).sum())
    if dup:
        raise SystemExit(f"{dup} CABAC groups hold two copies of one tile: the batch would measure converged warps")
    return {"tiles_per_group": 32, "groups": int(g.shape[0]), "lane_fill": round(float(valid.mean()), 4), "groups_with_duplicates": 0}


def dump_outputs(batch, out_dir: str, n_images: int = 16, n_pixels: int = 1 << 18):
    """The RGB the last decode left in the resident batch, as .npy files that two builds can be compared by (about 55 MB):
        rgb_tile_sums.npy      float64 [images, 6, 8, 3]  sum of each channel over each 512x512 grid cell, every image (exact)
        rgb_sample.npy         float32 [n_images, n_pixels, 3]  RGB of the sampled pixels of the sampled images
        rgb_sample_images.npy  float64 [n_images]  batch indices of the sampled images
        rgb_sample_pixels.npy  float64 [n_pixels, 2]  (row, column) of the sampled pixels
    The sample is drawn by rng(SEED): the same arguments give the same sample."""
    import torch

    n = len(batch.images)
    ptr, pitch, stride = batch.rgb_layout()

    class DeviceRgb:  # the batch's RGB in HBM, summed where it is (a host pass over every image takes minutes)
        __cuda_array_interface__ = {"shape": (n, OUT_H, OUT_W * 3), "strides": (stride, pitch, 1), "typestr": "|u1",
                                    "data": (ptr, False), "version": 2}

    rgb = torch.as_tensor(DeviceRgb(), device="cuda").view(n, OUT_H, OUT_W, 3)
    gh, gw = -(-OUT_H // TILE_H), -(-OUT_W // TILE_W)
    cells = torch.zeros((gh * TILE_H, gw * TILE_W, 3), dtype=torch.int32, device="cuda")
    sums = torch.zeros((n, gh, gw, 3), dtype=torch.float64, device="cuda")
    for i in range(n):
        cells[:OUT_H, :OUT_W] = rgb[i]
        sums[i] = cells.view(gh, TILE_H, gw, TILE_W, 3).sum((1, 3))
    rng = np.random.default_rng(SEED)
    images = np.sort(rng.choice(n, size=min(n_images, n), replace=False))
    rows, cols = rng.integers(0, OUT_H, n_pixels), rng.integers(0, OUT_W, n_pixels)
    sample = np.stack([batch.download_image(int(i))[rows, cols] for i in images]).astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "rgb_tile_sums.npy"), sums.cpu().numpy())
    np.save(os.path.join(out_dir, "rgb_sample.npy"), sample)
    np.save(os.path.join(out_dir, "rgb_sample_images.npy"), images.astype(np.float64))
    np.save(os.path.join(out_dir, "rgb_sample_pixels.npy"), np.stack([rows, cols], axis=1).astype(np.float64))


# ---------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed decodes of the resident batch (`value`); the e2e serving loop makes max(12, min(steps, 32)) calls")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=int(os.environ.get("HEIC_BENCH_BATCH", "592")), help="images per GPU per step")
    ap.add_argument("--pool", type=int, default=512, help="synthetic tiles in the pool (beside the 48 real ones)")
    ap.add_argument("--e2e-batch", type=int, default=int(os.environ.get("HEIC_BENCH_E2E_BATCH", "296")),
                    help="images per reference-facing call (296 images = 444 CABAC groups = one resident wave of CTAs)")
    ap.add_argument("--ref-images", type=int, default=64, help="images per step of the CPU arm")
    ap.add_argument("--cpu-images", type=int, default=128, help="images in the cpu_baseline sample")
    ap.add_argument("--check-images", type=int, default=8, help="images compared pixel by pixel with the oracle")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-converged", action="store_true", help="skip the copies-of-one-tile-per-warp upper bound")
    ap.add_argument("--stages", action="store_true", help="also print a per-stage table to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write (rank 0's) RGB of the last step to DIR/*.npy: see dump_outputs()")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch

    import heif_b200 as H
    from heif_b200 import sharding
    from tests.synth import pool as P

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    # One process per GPU on a multi-socket box: run on (and first-touch the pinned staging buffers from) the CPUs next to
    # this rank's GPU, so that the device->host RGB copies of all ranks do not cross the socket interconnect.
    affinity = bind_to_gpu_numa_node(local) if world > 1 else "not bound (single process)"
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    f = H.HeicFile(open(FIXTURE, "rb").read())
    dec = H.HeicDecoder(device=local)
    pool = P.build_pool(f, args.pool, threads=max(2, (os.cpu_count() or 2) // world))
    # the job: world * batch images, image i on rank i % world (SURVEY 8(e))
    n_job = world * args.batch
    my_images = list(sharding.shard_modulo(n_job, rank, world))
    images, keep, ids = P.compose_images(pool, f.primary, my_images, SEED)
    batch = dec.batch(images)
    groups = check_groups_distinct(batch, ids.reshape(-1))
    stream = torch.cuda.ExternalStream(batch.stream, device=torch.device("cuda", local))
    hbm_peak, peak_src = peaks()

    def ev():
        return torch.cuda.Event(enable_timing=True)

    # ---- warm-up, then the pixel check: random images of the resident batch against the CPU oracle ------------------
    for _ in range(max(args.warmup, 3)):
        batch.decode()
    batch.sync()
    st = batch.status()
    bad = [i for i in range(batch.n_tiles) if st[i].code != 0]
    if bad:
        raise SystemExit(f"{len(bad)} tiles failed to decode")
    bins_per_step = sum(st[i].bins_decoded for i in range(batch.n_tiles))
    n_chk = min(args.check_images, args.batch)
    cpu_threads = max(1, (os.cpu_count() or 1) // world)
    cpu_dec = CpuDecoder(pool, f.primary, cpu_threads)
    chk = np.sort(np.random.default_rng(1234 + rank).choice(args.batch, size=n_chk, replace=False))
    eb = min(args.e2e_batch, args.batch)
    chk[0] = min(int(chk[0]), eb - 1)  # at least one of them also lies inside the e2e call
    chk = np.unique(chk)
    ref_planes = np.zeros((len(chk), 48, TILE_BYTES), np.uint8)
    ref_rgb = np.zeros((len(chk), OUT_H, OUT_W, 3), np.uint8)
    cpu_dec.decode(ids[chk], ref_planes, ref_rgb)
    for k, i in enumerate(chk):
        got = batch.download_image(int(i))
        if not np.array_equal(got, ref_rgb[k]):
            raise SystemExit(f"resident batch, image {int(i)}: {int((got != ref_rgb[k]).sum())} RGB bytes differ from the oracle")
    pixel_check = {"resident_images_checked": [int(i) for i in chk], "vs": "CPU oracle (decode + the frozen colour definition), bit-exact"}

    # ---- value: K steps, batch resident in HBM -----------------------------------------------------------
    barrier()
    clocks = ClockSampler(local) if rank == 0 else None
    l0 = dec.launch_count()
    e0, e1 = ev(), ev()
    t_wall0 = time.time()
    e0.record(stream)
    for _ in range(args.steps):
        batch.decode()
    e1.record(stream)
    batch.sync()
    barrier()
    t_wall1 = time.time()
    launches = dec.launch_count() - l0
    ms = e0.elapsed_time(e1)
    clk = clocks.stop(t_wall0, t_wall1) if clocks else None
    if args.dump_outputs and rank == 0:
        dump_outputs(batch, args.dump_outputs)

    # ---- per-stage device times (same batch, one stage per event pair) -------------------------------------
    stage_defs = [("cabac", H.STAGE_CABAC), ("transform", H.STAGE_TRANSFORM), ("intra", H.STAGE_INTRA),
                  ("deblock", H.STAGE_DEBLOCK), ("sao", H.STAGE_SAO), ("color_stitch", H.STAGE_COLOR)]
    stage_ms = {n: 0.0 for n, _ in stage_defs}
    reps = 2
    for _ in range(reps):
        evs = [ev() for _ in range(len(stage_defs) + 1)]
        evs[0].record(stream)
        for i, (n, m) in enumerate(stage_defs):
            batch.run(m)
            evs[i + 1].record(stream)
        batch.sync()
        for i, (n, _) in enumerate(stage_defs):
            stage_ms[n] += evs[i].elapsed_time(evs[i + 1]) / reps

    # SAO applied inside the colour kernel: what a full decode (`value`) runs instead of the two separate stages above
    fe = [ev() for _ in range(reps + 1)]
    fe[0].record(stream)
    for i in range(reps):
        batch.run(H.STAGE_SAO | H.STAGE_COLOR)
        fe[i + 1].record(stream)
    batch.sync()
    fused_ms = fe[0].elapsed_time(fe[reps]) / reps

    # coded samples (cbf = 1) per pool tile, for the algorithmic bytes of the transform / intra stages: measured on the
    # first tile of every pool entry that occurs in this rank's batch
    flat = ids.reshape(-1)
    first_of = {}
    for t, pid in enumerate(flat):
        first_of.setdefault(int(pid), t)
    coded_of = {}
    for pid, t in first_of.items():
        m = batch.dump_tile(t)["tu_map"]
        o = m[(m & 1) == 1]
        n2 = (4 << ((o >> 1) & 3)).astype(np.int64) ** 2
        c = int((n2 * ((o >> 3) & 1)).sum())
        nc = np.where(((o >> 1) & 3) == 0, 16, n2 // 4)
        c += int((nc * ((o >> 6) & 1) * (((o >> 4) & 1) + ((o >> 5) & 1))).sum())
        coded_of[pid] = c
    n_img = args.batch
    coded_total = int(sum(coded_of[int(pid)] for pid in flat))
    slice_bytes_total = int(sum(pool.descs[int(pid)].rbsp_len for pid in flat))
    a_c = CODED_SAMPLES_PER_IMAGE
    alg_bytes = {  # per step (whole batch), SURVEY.md section 8(d)
        "cabac": slice_bytes_total + 2 * coded_total,        # slice data in + TransCoeffLevel out (dense int16 of coded blocks)
        "transform": 4 * coded_total,                        # 2 B in + 2 B out per coded sample
        "intra": 2 * coded_total + a_c * n_img,              # residual in + reconstructed planes out
        "deblock": 2 * a_c * n_img,                          # planes in + out
        "sao": 2 * a_c * n_img,
        "color_stitch": int(4.5 * OUT_W * OUT_H) * n_img,    # 1.5 B in + 3 B out per output pixel
    }
    stages = []
    for n, _ in stage_defs:
        gbs = alg_bytes[n] / (stage_ms[n] * 1e-3) / 1e9 if stage_ms[n] > 0 else 0.0
        stages.append({"kernel": n, "ms": round(stage_ms[n], 4), "alg_GB": round(alg_bytes[n] / 1e9, 4),
                       "achieved_GBps": round(gbs, 1), "frac_of_hbm_peak": round(gbs / hbm_peak, 4)})
    dom = max(stages, key=lambda s: s["ms"])
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "dram_traffic_per_image.json")
    if os.path.exists(tpath):  # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture, per image
        per_image = json.load(open(tpath)).get(dom["kernel"])
        if per_image:
            traffic = int(per_image * n_img)
    n_sm = torch.cuda.get_device_properties(local).multi_processor_count
    cabac_bins = bins_per_step / (stage_ms["cabac"] * 1e-3)

    # the resident batch has served (76 GB of intermediates): its memory goes to the pipeline slots of the e2e path
    batch.close()
    batch = None

    # ---- e2e: host descriptors + bitstreams in, pinned host RGB out, through heic_b200_decode_grids ----------
    # A serving loop over the asynchronous form of the C-ABI call (heic_b200_decode_grids_submit / heic_b200_job_wait) with
    # N_BUF calls in flight: while call k's RGB travels to the host, call k+1 runs its kernels and call k+2 is being staged
    # by the host (with two in flight the GPU idled ~100 ms per call behind "wait for the copy, then stage the next call").
    # Every call carries all of its own copies; N_BUF pinned output buffers rotate.
    N_BUF = 3
    # pinned host RGB: N_BUF x 36.6 MB per image per rank; all ranks together may pin 40 % of the host memory that is free
    fit = torch.tensor([int(0.4 * host_memory_available() / world / (N_BUF * OUT_H * OUT_W * 3))], device="cuda", dtype=torch.int64)
    if dist is not None:
        dist.all_reduce(fit, op=dist.ReduceOp.MIN)  # the same call size on every rank
    if int(fit[0]) < eb:
        eb = max(32, int(fit[0]) // 8 * 8)
    bufs = [torch.empty((eb, OUT_H, OUT_W, 3), dtype=torch.uint8, pin_memory=True) for _ in range(N_BUF)]
    outs = [b_.numpy() for b_ in bufs]
    out_np = outs[0]
    h2d = sum(images[i].tiles[t].rbsp_len for i in range(eb) for t in range(48)) + eb * 48 * (C.sizeof(H._capi.TileDesc) // 8)
    d2h = eb * OUT_H * OUT_W * 3
    # warm-up: the library's pipeline slots allocate their arenas on first use, so run enough calls to have touched every
    # slot (and every output buffer) before the timed region
    for k in range(2 * N_BUF):
        dec.decode_grids(images[:eb], out=outs[k % N_BUF])
    for k, i in enumerate(chk):  # pixels of the reference-facing call as well
        if i < eb:
            for o in outs:  # the warm-up wrote every buffer
                if not np.array_equal(o[int(i)], ref_rgb[k]):
                    raise SystemExit(f"decode_grids, image {int(i)}: RGB differs from the oracle")
    pixel_check["e2e_images_checked"] = [int(i) for i in chk if i < eb]
    barrier()
    e2e_steps = max(12, min(args.steps, 32))  # enough calls that the pipeline's fill and drain are amortised
    t0 = time.perf_counter()
    jobs = []
    submit_s = 0.0
    for k in range(e2e_steps):
        if len(jobs) >= N_BUF:  # the buffer this call writes must have been handed back
            dec.wait_job(jobs.pop(0))
        ts = time.perf_counter()
        jobs.append(dec.submit_grids(images[:eb], outs[k % N_BUF]))
        submit_s += time.perf_counter() - ts
    for j in jobs:
        dec.wait_job(j)
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    # The plain synchronous call, one at a time: the other serving mode.  On one GPU it loses (nothing overlaps the copy); with
    # all 8 ranks of a box copying at once it WINS, because the box's host memory system, not the GPUs, is the limit there
    # (DESIGN 6: 94-121 GB/s for eight concurrent device->host streams) and fewer concurrent DMA streams contend less.
    barrier()
    n_sync = 2 if world == 1 else 6
    t0 = time.perf_counter()
    for _ in range(n_sync):
        dec.decode_grids(images[:eb], out=out_np)
    sync_s = (time.perf_counter() - t0) / n_sync
    e2e_val = eb * MP_PER_IMAGE / e2e_s

    # ---- aggregate over ranks: max time --------------------------------------------------------------------
    ms, sums = sharding.reduce_timing(dist, torch.device("cuda", local), ms, {"bins": float(bins_per_step)})
    if dist is not None:
        t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t[0])
        e2e_val = eb * MP_PER_IMAGE / e2e_s
        t = torch.tensor([sync_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sync_s = float(t[0])
    value = world * args.steps * n_img * MP_PER_IMAGE / (ms * 1e-3)
    # e2e = the better of the two serving modes measured in this run (both through the C-ABI call with host buffers, both
    # max over ranks); the line says which, and carries both figures
    pipelined_total = world * e2e_val
    sync_total = world * eb * MP_PER_IMAGE / sync_s
    e2e_mode = "3 calls in flight: heic_b200_decode_grids_submit/_job_wait, pinned host RGB"
    e2e_total = pipelined_total
    if sync_total > pipelined_total:
        e2e_total = sync_total
        e2e_s = sync_s
        e2e_mode = "one synchronous heic_b200_decode_grids call at a time per rank, pinned host RGB (faster than 3 calls in flight on this box)"

    # ---- the same colour stage with the irot rotation applied (apply_transforms = 1; every iPhone portrait has one) ------------
    rotated = None
    if world == 1:
        n_rot = min(128, args.batch)
        rb = dec.batch(images[:n_rot], apply_transforms=True)
        rs = torch.cuda.ExternalStream(rb.stream, device=torch.device("cuda", local))
        rb.decode()
        rb.sync()
        turns = int(images[0].rotation_ccw_quarter_turns) & 3
        k0 = int(np.argmax(chk < n_rot)) if (chk < n_rot).any() else None
        if k0 is not None:
            got = rb.download_image(int(chk[k0]))
            if not np.array_equal(got, np.rot90(ref_rgb[k0], turns)):
                raise SystemExit(f"rotated output, image {int(chk[k0])}: differs from the rotated oracle image")
        r0, r1 = ev(), ev()
        r0.record(rs)
        for _ in range(4):
            rb.run(H.STAGE_SAO | H.STAGE_COLOR)
        r1.record(rs)
        rb.sync()
        rot_ms = r0.elapsed_time(r1) / 4 / n_rot
        rotated = {"quarter_turns_ccw": turns, "us_per_image": round(rot_ms * 1e3, 2), "us_per_image_unrotated": round(fused_ms / n_img * 1e3, 2),
                   "ratio": round(rot_ms / (fused_ms / n_img), 3), "images": n_rot,
                   "pixel_check": None if k0 is None else f"image {int(chk[k0])} == rot90(oracle image, {turns})"}
        rb.close()

    # ---- upper bound for context: copies of ONE tile in every CABAC warp (what a batch of 48 repeated tiles measures) ----
    converged = None
    if world == 1 and not args.no_converged:
        dec.close()  # hands back the pipeline slots (3 x 38 GB): the next batch needs 76 GB
        dec = None
        rng = np.random.default_rng(SEED)
        perm_ids = np.stack([rng.permutation(48) for _ in range(args.batch)])  # real tiles only, 592 copies of each
        os.environ["HEIC_B200_CABAC_PLAIN_SORT"] = "1"  # plain size sort: the copies of a tile land in the same warps
        dec2 = H.HeicDecoder(device=local)
        del os.environ["HEIC_B200_CABAC_PLAIN_SORT"]
        imgs2, keep2 = [], []
        tsize = C.sizeof(H._capi.TileDesc)
        for i in range(args.batch):
            tiles = (H._capi.TileDesc * 48)()
            for d, s in enumerate(perm_ids[i]):
                C.memmove(C.byref(tiles, d * tsize), C.byref(pool.descs[int(s)]), tsize)
            im = H._capi.ImageDesc()
            C.memmove(C.byref(im), C.byref(f.primary), C.sizeof(H._capi.ImageDesc))
            im.tiles = C.cast(tiles, C.POINTER(H._capi.TileDesc))
            keep2.append(tiles)
            imgs2.append(im)
        b2 = dec2.batch(imgs2)
        s2 = torch.cuda.ExternalStream(b2.stream, device=torch.device("cuda", local))
        for _ in range(2):
            b2.decode()
        b2.sync()
        m0, m1, m2 = ev(), ev(), ev()
        m0.record(s2)
        for _ in range(2):
            b2.decode()
        m1.record(s2)
        b2.run(H.STAGE_CABAC)
        m2.record(s2)
        b2.sync()
        c_ms = m0.elapsed_time(m1) / 2
        converged = {"value": round(n_img * MP_PER_IMAGE / (c_ms * 1e-3), 2), "unit": "MP/s", "ms_per_step": round(c_ms, 4),
                     "cabac_ms": round(m1.elapsed_time(m2), 4),
                     "note": "UPPER BOUND, not the workload: a batch that repeats the fixture's 48 real tiles, size-sorted so that "
                             "every CABAC warp holds 32 copies of one tile and never diverges (round 1's headline)"}
        b2.close()
        dec2.close()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        n_cpu = args.cpu_images
        cids = np.stack([P.image_tile_ids(len(pool), i, 48, SEED) for i in range(n_cpu)])
        cpl = np.zeros((n_cpu, 48, TILE_BYTES), np.uint8)
        crgb = np.zeros((n_cpu, OUT_H, OUT_W, 3), np.uint8)
        dt = CpuDecoder(pool, f.primary, cores).decode(cids, cpl, crgb)
        cpu = {"value": round(n_cpu * MP_PER_IMAGE / dt, 3), "unit": "MP/s", "cores": cores, "kind": "port",
               "sample": f"images 0..{n_cpu - 1} of the job = {48 * n_cpu} tiles, oracle port (C -O3), {cores} threads, {dt:.1f} s"}
        del cpl, crgb
        fdt = ffmpeg_decode_images(f, 64, cores)
        if fdt:
            cpu["ffmpeg_hevc"] = {"value": round(64 * MP_PER_IMAGE / fdt, 3), "unit": "MP/s", "cores": cores,
                                  "note": "FFmpeg native hevc decoder, YCbCr planes only (no colour conversion), the 48 real tiles; context, not the reference"}

    if rank == 0:
        line = {
            "metric": "decoded MP/s (12MP HEIC grid batch)", "value": round(value, 2), "unit": "MP/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic batch: " + data_note(pool),
            "config": {"workload": WORKLOAD,
                       "images_per_gpu_per_step": n_img, "tiles_per_step_per_gpu": n_img * 48, "images_in_job": n_job,
                       "parallelism": f"image_idx % {world} (heif_b200/sharding.py), no collective",
                       "l2": "working set per step >> 126 MB L2 (inputs larger than L2)",
                       "cabac_groups": groups},
            "roofline": {"kernel": dom["kernel"], "bound": "latency" if dom["kernel"] == "cabac" else "hbm",
                         "achieved": round(cabac_bins / n_sm / 1e9, 4) if dom["kernel"] == "cabac" else dom["achieved_GBps"],
                         "peak": None if dom["kernel"] == "cabac" else hbm_peak,
                         "unit": "Gbin/s/SM" if dom["kernel"] == "cabac" else "GB/s",
                         "frac": None if dom["kernel"] == "cabac" else dom["frac_of_hbm_peak"],
                         "hbm": {"achieved": dom["achieved_GBps"], "peak": hbm_peak, "unit": "GB/s", "frac": dom["frac_of_hbm_peak"]},
                         "traffic": traffic, "peak_source": peak_src,
                         "note": "dominant kernel by time.  CABAC is bound by the serial bin chain, not by a throughput roofline: "
                                 "`achieved` is bins/s/SM (SURVEY 8(d)); its HBM figure is under `hbm`; per-kernel rooflines in `stages`"},
            "stages": stages,
            "fused_sao_color": {"ms": round(fused_ms, 4), "alg_GB": round(alg_bytes["color_stitch"] / 1e9, 4),
                                "achieved_GBps": round(alg_bytes["color_stitch"] / (fused_ms * 1e-3) / 1e9, 1),
                                "frac_of_hbm_peak": round(alg_bytes["color_stitch"] / (fused_ms * 1e-3) / 1e9 / hbm_peak, 4),
                                "note": "a full decode applies SAO inside the colour kernel (1.5 B in + 3 B out per output pixel); "
                                        "`sao` and `color_stitch` above are the stand-alone stages"},
            "cabac_bins_per_s_per_sm": round(cabac_bins / n_sm, 1), "cabac_bins_per_image": int(sums["bins"] / world) // n_img,
            "coded_mp_per_s": round(value * (48 * 512 * 512) / (OUT_W * OUT_H), 2),
            "pixel_check": pixel_check,
            "cpu_baseline": cpu,
            "e2e": {"value": round(e2e_total, 2), "unit": "MP/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "images_per_call": eb, "host_affinity": affinity, "ms_per_call": round(e2e_s * 1e3, 3), "host_submit_ms_per_call": round(submit_s / e2e_steps * 1e3, 3),
                    "mode": e2e_mode, "pipelined_3_in_flight_MPps": round(pipelined_total, 2),
                    "synchronous_call_MPps": round(sync_total, 2)},
            "rotated_color": rotated,
            "copies_per_warp_upper_bound": converged,
            "gpu_launches": int(launches),
            "clocks": clk,
        }
        print(json.dumps(line))
        if args.stages:
            for s in stages:
                print(s, file=sys.stderr)
    if batch is not None:
        batch.close()
    if dec is not None:
        dec.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
