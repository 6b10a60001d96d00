#!/usr/bin/env python
"""bench.py — the lens-warp benchmark (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

metric   lens-warp Mpixels/s (output pixels, W*H per frame) on the headline workload of
         BASELINE.json: 3840x2160 screen, cube globe of 6x2048^2 8-bit faces, panini lens.
step     one pass of the hot path over one batch of FRAMES distinct synthetic frames per GPU
         (one kernel launch).  The frames of a batch are 16 x 25 MB = 403 MB of faces, larger
         than the 126 MB L2, so every step streams its faces from HBM; the lensmap (static per
         lens, like the reference's) is reused by all frames and stays L2-resident.
value    N = 1: throughput with inputs resident in HBM (CUDA events on the launch stream).  N > 1: frames are
         independent — rank r warps its own batch, no collective on the data path ("weak" scaling;
         `value_warp_only` is that aggregate) — and the reference topology's last step, finished frames to the
         one display, is a gather to rank 0 through the C ABI (blinky_shard_warp_gather: NCCL send/recv,
         copy-engine peer copies or in-kernel peer stores, overlapped with the warp): `value` is the
         DELIVERED-TO-RANK-0 rate of the fastest transport (all three are timed and compared, key "gather"),
         max over ranks.
e2e      the same metric through the C ABI's host entry point blinky_warp_host: pinned host
         faces -> batched async copies -> warp -> copy back, all inside the timed region.
roofline frac = SURVEY 8(d) algorithmic bytes / launch time / measured HBM peak; compulsory_frac = bytes the
         launch cannot avoid (counted from the lensmap in this run); dram_frac = ncu-measured DRAM bytes of
         this workload's launch (profiles/traffic_r2.json) / this run's launch time.
secondary  every other BASELINE configuration (C2, C3, the C4 lenses, C5 trism/cube): batched and single
         cold frame, same three fractions.
--impl reference   the reference's own CPU loop (oracle/_ref = unmodified fisheye.c compiled
         headless; else the oracle port) on the host cores, same workload, bounded sample.
--dump-outputs DIR  after the timed steps, rank 0's output batch of the last step as a fixed, seeded sample
         (see dump_outputs); the inputs are seeded too, so two builds can be compared output for output.

The oracle (oracle/) is only ever the thing TIMED BESIDE or CHECKED AGAINST — never the
product path, which raises if libblinky_b200.so is missing.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (W, H, platesize, globe, lens, zoom command, rubix)
    "4k-cube-panini": (3840, 2160, 2048, "cube", "panini", "f_fov 180", False),           # headline (metric)
    "1080p-cube-panini170": (1920, 1080, 1024, "cube", "panini", "f_fov 170", False),     # BASELINE configs[1]
    "4k-cube-quincuncial-rubix": (3840, 2160, 2048, "cube", "quincuncial", "f_cover", True),  # configs[2]
    "4k-trism-stereographic": (3840, 2160, 2048, "trism", "stereographic", "f_fov 180", False),  # configs[4]
    "4k-cube-stereographic": (3840, 2160, 2048, "cube", "stereographic", "f_fov 180", False),
    "4k-cube-equirect": (3840, 2160, 2048, "cube", "equirect", "f_contain", False),
    "4k-cube-hammer": (3840, 2160, 2048, "cube", "hammer", "f_contain", False),
    "4k-cube-fisheye1": (3840, 2160, 2048, "cube", "fisheye1", "f_contain", False),
    "c1-640x480": (640, 480, 256, "cube", "panini", "f_fov 180", False),                  # configs[0]
}
OUT = sys.stdout
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md, used only if MEASURED_PEAKS.json is absent


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    except Exception:  # noqa: BLE001
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons, sampled with NVML while the load runs"""

    def __init__(self, index: int):
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.004)

    def start(self):
        if self.nv:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        if self._thread:
            self._stop.set()
            self._thread.join()

    def summary(self, note: str):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "NVML unavailable"}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples), "note": note}


def cpu_baseline(workload, threads_all: bool = False):
    """The reference's CPU loop on this box: oracle/_ref (kind 'reference') when it was built,
    else the plain-C port (kind 'port').  Bounded sample: a few seconds of render_lensmap."""
    import blinky_b200 as bb
    from oracle.pyoracle import RefOracle, Restatement

    W, H, PS, globe, lens, zoom, rubix = workload
    pal = bb.synthetic_palette()
    faces = bb.synthetic_faces(6 if globe != "trism" else 5, PS, 0)
    out = {}
    if RefOracle.available():
        R = RefOracle.get(bb.SCRIPT_DIR, pal)
        R.set_screen(W, H)
        R.command(f"f_globe {globe}")
        R.command(f"f_lens {lens}")
        R.command(zoom)
        if R.rubix_enabled != rubix:
            R.command("f_rubix")
        t0 = time.time()
        R.build(W, H, PS)
        build_s = time.time() - t0
        R.render(faces, None)  # loads the faces into globe.pixels
        best1, _ = R.time_render(1)
        reps = int(max(3, min(200, 4.0 / max(best1, 1e-4))))
        best, total = R.time_render(reps)
        out = {"value": round(W * H / best / 1e6, 1), "unit": "Mpixels/s", "cores": 1, "kind": "reference",
               "sample": f"{reps} x render_lensmap() of one {W}x{H} frame, unmodified fisheye.c compiled -O2 (oracle/_ref), "
                         f"single thread as in the engine; best call; lensmap build {build_s:.1f} s not counted",
               "mean_value": round(W * H * reps / total / 1e6, 1),
               "lensmap_build_s": round(build_s, 2)}  # the reference's create_lensmap (Lua VM per pixel), same map
        idx, tint = R.lensmap()
    else:
        with bb.Fisheye(device=None, palette=pal) as fe:
            fe.command(f"f_globe {globe}")
            fe.command(f"f_lens {lens}")
            fe.command(zoom)
            fe.build_lensmap(W, H, PS, bb.usable_cpus())
            idx, tint = fe.lensmap()
    O = Restatement()
    pm = O.palmaps(pal)
    if not out:
        best1, _ = O.time_render(idx, tint, faces, pm, rubix, 1, 1)
        reps = int(max(3, min(200, 4.0 / max(best1, 1e-4))))
        best, total = O.time_render(idx, tint, faces, pm, rubix, 1, reps)
        out = {"value": round(W * H / best / 1e6, 1), "unit": "Mpixels/s", "cores": 1, "kind": "port",
               "sample": f"{reps} x restated render_lensmap (oracle/blinky_oracle.c) of one {W}x{H} frame, single thread; best call",
               "mean_value": round(W * H * reps / total / 1e6, 1)}
    nthreads = min(O.max_threads(), bb.usable_cpus())  # the cgroup quota, not the 128 cores the box shows
    bestn, _ = O.time_render(idx, tint, faces, pm, rubix, nthreads, 20)
    out["all_cores_port"] = {"value": round(W * H / bestn / 1e6, 1), "unit": "Mpixels/s", "cores": nthreads,
                             "note": "same loop, rows split over all host threads (oracle port; the reference itself is single-threaded)"}
    return out


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation, same metric/config/unit."""
    if rank != 0:
        return
    workload = WORKLOADS[args.workload]
    W, H, PS, globe, lens, zoom, rubix = workload
    import blinky_b200 as bb
    from oracle.pyoracle import RefOracle, Restatement

    pal = bb.synthetic_palette()
    P = 5 if globe == "trism" else 6
    frames_per_step = 4
    faces = [bb.synthetic_faces(P, PS, f) for f in range(frames_per_step)]
    if RefOracle.available():
        R = RefOracle.get(bb.SCRIPT_DIR, pal)
        R.set_screen(W, H)
        for c in (f"f_globe {globe}", f"f_lens {lens}", zoom):
            R.command(c)
        if R.rubix_enabled != rubix:
            R.command("f_rubix")
        R.build(W, H, PS)
        kind, cores = "reference", 1

        def step():
            for f in faces:
                R.render(f, None)  # memcpy of the plates into globe.pixels (render_plate's job) + render_lensmap
    else:
        with bb.Fisheye(device=None, palette=pal) as fe:
            for c in (f"f_globe {globe}", f"f_lens {lens}", zoom):
                fe.command(c)
            fe.build_lensmap(W, H, PS, bb.usable_cpus())
            idx, tint = fe.lensmap()
        O = Restatement()
        pm = O.palmaps(pal)
        kind, cores = "port", 1

        def step():
            for f in faces:
                O.render(idx, tint, f, pm, rubix)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = W * H * frames_per_step * args.steps / dt / 1e6
    line = {"impl": "reference", "metric": "lens-warp Mpixels/s", "value": round(value, 1), "unit": "Mpixels/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": args.workload, "screen": [W, H], "globe": globe, "platesize": PS, "lens": lens, "zoom": zoom,
                       "rubix": rubix, "frames_per_step": frames_per_step},
            "cpu_baseline": {"value": round(value, 1), "unit": "Mpixels/s", "cores": cores, "kind": kind,
                             "sample": f"{frames_per_step} frames per step: plate copy into globe.pixels + render_lensmap, "
                                       f"single thread (the reference's loop has no threading)"},
            "e2e": {"value": round(value, 1), "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), file=OUT, flush=True)


def claim_stdout():
    """stdout carries exactly one JSON line.  Native libraries print there too (NCCL's version banner
    under NCCL_DEBUG=VERSION, for one), so fd 1 is pointed at stderr and the line goes out through a
    private duplicate of the original stdout."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def setup_workload(fe, name):
    W, H, PS, globe, lens, zoom, rubix = WORKLOADS[name]
    for c in (f"f_globe {globe}", f"f_lens {lens}", zoom):
        fe.command(c)
    fe.set_rubix(rubix)
    t0 = time.time()
    fe.build_lensmap(W, H, PS, threads=0)  # GPU build (translated lens); every rank rebuilds deterministically: nothing to broadcast
    return time.time() - t0


def compulsory_bytes(fe, frames):
    """Bytes a launch cannot avoid moving through HBM: every 32-byte sector of the faces the lensmap reads
    (once per frame), the output (once per frame) and the tile plan's entry blocks + descriptors (once per
    launch: they stay in L2 across the frames of a batch)."""
    idx, _ = fe.lensmap()
    v = idx[idx >= 0].astype(np.int64)
    sectors = np.unique(v >> 5).size
    tiles, entries = fe.tile_plan()
    per_frame = sectors * 32 + fe.width * fe.height
    return int(per_frame * frames + entries.size + tiles.nbytes), int(sectors * 32)


def time_device(torch, fe, d_faces, d_out, frames, steps, warmup, stream, flush=None):
    """CUDA-event time of `steps` launches (seconds per launch); flush = a >L2 buffer rewritten before every
    launch (cold single-frame case) — then each launch is timed on its own"""
    for _ in range(warmup):
        fe.warp(d_faces, d_out, nframes=frames, stream=stream)
    torch.cuda.synchronize()
    if flush is None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fe.warp(d_faces, d_out, nframes=frames, stream=stream)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3 / steps
    ts = []
    for _ in range(steps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fe.warp(d_faces, d_out, nframes=frames, stream=stream)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e-3)
    return float(np.median(ts))


def time_single_frame_stream(torch, fe, d_faces, d_out, stream, rounds=3):
    """seconds per single-frame launch when every launch warps a different frame (the engine's call pattern)"""
    F = d_faces.shape[0]
    for i in range(F):  # warm-up: builds the per-pointer TMA descriptors
        fe.warp(d_faces[i:], d_out[i:], nframes=1, stream=stream)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(rounds):
        for i in range(F):
            fe.warp(d_faces[i:], d_out[i:], nframes=1, stream=stream)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / (rounds * F)


def roofline_entry(fe, launch_s, frames, peak, traffic):
    npix, M = fe.width * fe.height, fe.mapped_pixels
    alg = (5 * npix + M) * frames  # SURVEY section 8d: 4 B lensmap entry + 1 B source (mapped) + 1 B output per pixel
    comp, face_sector_bytes = compulsory_bytes(fe, frames)
    out = {"achieved": round(alg / launch_s / 1e9, 1), "frac": round(alg / launch_s / 1e9 / peak, 4),
           "algorithmic_bytes_per_launch": int(alg), "launch_us": round(launch_s * 1e6, 2),
           "compulsory_bytes_per_launch": comp, "compulsory_frac": round(comp / launch_s / 1e9 / peak, 4),
           "face_sector_bytes_per_frame": face_sector_bytes}
    if traffic:
        # the contract's `traffic`: dram__bytes_read.sum + dram__bytes_write.sum of this workload's launch (one ncu --set full capture)
        out["traffic"] = int(traffic["dram_bytes_per_launch"])
        out["traffic_detail"] = traffic
        out["dram_frac"] = round(traffic["dram_bytes_per_launch"] / launch_s / 1e9 / peak, 4)
    else:
        out["traffic"] = None
        out["dram_frac"] = None
    return out


DUMP_SAMPLE = 1 << 22  # drawn pixel positions: <= 16 MB of float32 values + 32 MB of float64 indices


def dump_outputs(directory, d_out):
    """What a caller of the timed path receives, d_out [frames][H][W] uint8, sampled at a fixed seeded set of
    positions (the whole batch is 531 MB as float32): out.npy holds the pixel values as float32, out_index.npy
    their flat indices into d_out as float64, both in ascending index order."""
    import torch

    os.makedirs(directory, exist_ok=True)
    flat = d_out.reshape(-1)
    idx = np.unique(np.random.default_rng(0).integers(0, flat.numel(), DUMP_SAMPLE))
    vals = flat[torch.from_numpy(idx).to(flat.device)].cpu().numpy()
    np.save(os.path.join(directory, "out.npy"), vals.astype(np.float32))
    np.save(os.path.join(directory, "out_index.npy"), idx.astype(np.float64))


def load_traffic():
    """measured DRAM bytes per launch (ncu, this round) per workload: profiles/traffic_r2.json, written by
    scripts/ncu_traffic.py from the committed .ncu-rep summaries"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic_r2.json")))
    except Exception:  # noqa: BLE001
        return {}


def main():
    global OUT
    OUT = claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="4k-cube-panini", choices=sorted(WORKLOADS))
    ap.add_argument("--frames", type=int, default=16, help="distinct frames per GPU per step")
    ap.add_argument("--kernel", type=int, default=0, help="0 auto (ring kernel, TMA-staged boxes), 1 flat gather")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the other BASELINE configurations")
    ap.add_argument("--gather-mode", default="best", choices=["best", "nccl", "peer_copy", "peer_store"],
                    help="N > 1: which transport's delivered rate is `value` (best = the fastest of the three measured)")
    ap.add_argument("--chunk", type=int, default=4, help="frames per gather chunk (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's output to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's output; the reference arm keeps none")
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    bind_to_gpu_numa_node(local_rank)
    import torch
    import torch.distributed as dist

    import blinky_b200 as bb  # raises if the CUDA extension is missing — there is no fallback

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    W, H, PS, globe, lens, zoom, rubix = WORKLOADS[args.workload]
    F = args.frames
    fe = bb.Fisheye(device=local_rank, palette=bb.synthetic_palette())
    build_s = setup_workload(fe, args.workload)
    build_info = fe.build_info
    fe.set_kernel(args.kernel)
    P, M, npix = fe.numplates, fe.mapped_pixels, W * H
    gen = torch.Generator(device="cuda").manual_seed(1000 + rank)
    d_faces = torch.randint(0, 256, (F, P, PS, PS), dtype=torch.uint8, device="cuda", generator=gen)
    d_out = torch.zeros((F, H, W), dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    peak, peak_src = hbm_peak()
    traffic_db = load_traffic()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        fe.warp(d_faces, d_out, nframes=F, stream=stream)

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident warp: every rank its own batch, nothing exchanged ---------------------
    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = fe.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    launches = fe.launch_count - launches0
    elapsed = max_over_ranks(e0.elapsed_time(e1) * 1e-3)
    kernel_name = fe.last_kernel
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_out)
    # the timed region is a few milliseconds: keep the identical load running so that NVML
    # (which refreshes every few ms) actually sees the clocks this kernel runs at
    t_end = time.time() + 1.0
    while time.time() < t_end:
        for _ in range(20):
            step()
        torch.cuda.synchronize()
    sampler.stop()
    warp_value = world * F * args.steps * npix / elapsed / 1e6

    # ---- end to end through the C ABI's host entry point ------------------------------------------
    h_faces = fe.alloc_pinned(F * P * PS * PS)
    h_out = fe.alloc_pinned(F * npix)
    h_faces[:] = d_faces.cpu().numpy().reshape(-1)
    e2e_steps = max(2, min(args.steps, 6))
    fe.warp_host(h_faces, h_out.reshape(F, H, W))  # warm-up (allocates the frame ring)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        fe.warp_host(h_faces, h_out.reshape(F, H, W))
    torch.cuda.synchronize()
    e2e_t = max_over_ranks(time.perf_counter() - t0)
    same = bool(np.array_equal(h_out.reshape(F, H, W)[F - 1], d_out[F - 1].cpu().numpy()))
    e2e_value = world * F * e2e_steps * npix / e2e_t / 1e6
    upload_bytes = int(fe.upload_bytes_per_frame * F)
    fe.free_pinned(h_faces)
    fe.free_pinned(h_out)

    # ---- N > 1: the reference topology — finished frames reach rank 0 (C ABI: blinky_shard_*) --------
    gather = None
    value = warp_value
    if world > 1:
        gather = run_sharded(args, torch, dist, bb, fe, d_faces, rank, world, barrier, max_over_ranks, stream)
        value = gather["value"]

    if rank == 0:
        launch_s = elapsed / args.steps
        roof = roofline_entry(fe, launch_s, F, peak, traffic_db.get(args.workload))
        roof.update({"bound": "hbm", "peak": peak, "unit": "GB/s", "peak_source": peak_src,
                     "kernels_per_step": int(launches // max(1, args.steps)),
                     "note": "frac = SURVEY 8(d) algorithmic bytes (5*W*H + M per frame) / CUDA-event launch time / peak; "
                             "compulsory_frac = bytes the launch cannot avoid (sampled 32-byte face sectors + output per frame, "
                             "tile plan once per launch) / time / peak — computed in this run; dram_frac = DRAM bytes per launch "
                             "measured by ncu this round (profiles/traffic_r2.json) / this run's launch time / peak"})
        line = {
            "metric": "lens-warp Mpixels/s", "value": round(value, 1), "unit": "Mpixels/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(elapsed / args.steps * 1e3, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": args.workload, "screen": [W, H], "globe": globe, "numplates": P, "platesize": PS, "lens": lens,
                       "zoom": zoom, "rubix": rubix, "frames_per_gpu_per_step": F, "global_batch_frames": F * world,
                       "parallelism": f"frames sharded over {world} GPU(s), no data-path collective"
                                      + ("; finished frames gathered on rank 0 (value = delivered rate)" if world > 1 else ""),
                       "l2": "inputs larger than L2 (403 MB of distinct faces per step); lensmap reused across frames by design",
                       "mapped_pixel_fraction": round(M / npix, 4), "lensmap_build_s": round(build_s, 3), "lensmap_build": build_info,
                       "tiling": fe.plan_summary},
            "kernel": kernel_name, "gpu_launches": int(launches),
            "value_warp_only": round(warp_value, 1),
            "roofline": roof,
            "e2e": {"value": round(e2e_value, 1), "unit": "Mpixels/s", "h2d_bytes_per_step": upload_bytes,
                    "d2h_bytes_per_step": int(npix * F), "steps": e2e_steps, "matches_device_path": same,
                    "how": "blinky_warp_host: pinned host faces -> async copies of the texel rectangle each shown plate is sampled in -> "
                           "kernel -> copy back, multi-slot stream pipeline; wall clock around synchronous calls"},
            "clocks": sampler.summary("sampled by NVML over the timed region plus 1 s of the identical load"),
        }
        if gather:
            line["gather"] = gather
            # N > 1: `value` is what reaches rank 0, so the step time that goes with it is the gathered step's
            line["ms_per_step_warp_only"] = line["ms_per_step"]
            line["ms_per_step"] = gather["ms"]
    # ---- the other BASELINE configurations (device-resident; every rank runs them, rank 0 reports) ----
    if world == 1 and not args.no_secondary:
        secondary = run_secondary(args, torch, bb, fe, peak, traffic_db, stream)
        if rank == 0:
            line["secondary"] = secondary
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(WORKLOADS[args.workload])
        print(json.dumps(line), file=OUT, flush=True)
    fe.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def bind_to_gpu_numa_node(local_rank):
    """One process per GPU: keep the process (and therefore its pinned allocations, first-touch) on the
    NUMA node its GPU hangs off, so that 8 ranks do not push their PCIe traffic through one socket."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        node = None
        try:
            node = pynvml.nvmlDeviceGetNumaNodeId(h)
        except Exception:  # noqa: BLE001
            bus = pynvml.nvmlDeviceGetPciInfo(h).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
            path = f"/sys/bus/pci/devices/{bus[-12:].lower()}/numa_node"
            if os.path.exists(path):
                node = int(open(path).read())
        if node is None or node < 0:
            return
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
    except Exception:  # noqa: BLE001
        pass


def run_sharded(args, torch, dist, bb, fe, d_faces, rank, world, barrier, max_over_ranks, stream):
    """N > 1: blinky_shard_warp_gather — every rank warps its block of the global batch, finished frames
    are gathered on rank 0 chunk by chunk, overlapped with the warp of the next chunk.  All three
    transports are timed and reported; `value` is the delivered rate of the fastest (or of --gather-mode)."""
    from oracle.pyoracle import Restatement

    F = d_faces.shape[0]
    W, H = fe.width, fe.height
    npix = W * H
    total = F * world
    uid = [bb.shard_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    fe.shard_init(rank, world, uid[0])
    root = fe.shard_buffer(total)
    modes = {"nccl": bb.GATHER_NCCL, "peer_copy": bb.GATHER_PEER_COPY, "peer_store": bb.GATHER_PEER_STORE}
    out = {"chunk_frames": args.chunk, "bytes_into_rank0_per_step": (world - 1) * F * npix, "modes": {}}
    gathered = None
    if rank == 0:
        class _Raw:
            __cuda_array_interface__ = {"shape": (total, H, W), "typestr": "|u1", "data": (root, False), "version": 2}

        gathered = torch.as_tensor(_Raw(), device="cuda")
    reference = None
    for name, mode in modes.items():
        if rank == 0:
            gathered.fill_(0xEE)  # a frame that never lands shows up
        barrier()
        for _ in range(3):
            fe.shard_warp_gather(d_faces, total, mode, args.chunk, stream=stream)
        barrier()
        steps = max(5, min(args.steps, 20))
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(steps):
            fe.shard_warp_gather(d_faces, total, mode, args.chunk, stream=stream)
        g1.record()
        barrier()
        sec = max_over_ranks(g0.elapsed_time(g1) * 1e-3 / steps)
        entry = {"ms_per_step": round(sec * 1e3, 4), "value": round(total * npix / sec / 1e6, 1),
                 "GBs_into_rank0": round((world - 1) * F * npix / sec / 1e9, 1)}
        if rank == 0:
            if reference is None:
                reference = gathered.clone()
                entry["bytes_equal_first_mode"] = True
            else:
                entry["bytes_equal_first_mode"] = bool(torch.equal(gathered, reference))
        out["modes"][name] = entry
    # one gathered frame per rank against the oracle (restated render_lensmap on the product's lensmap,
    # which the GPU suite compares with the oracle's own build)
    if rank == 0:
        orc = Restatement()
        idx, tint = fe.lensmap()
        pm = orc.palmaps(bb.synthetic_palette())
        checked = []
        for r in range(world):
            gen_r = torch.Generator(device="cuda").manual_seed(1000 + r)
            faces_r = torch.randint(0, 256, tuple(d_faces.shape), dtype=torch.uint8, device="cuda", generator=gen_r)
            k = (r * 7 + 3) % F
            want = orc.render(idx, tint, faces_r[k].cpu().numpy(), pm, fe.rubix_enabled, background=np.zeros((H, W), np.uint8),
                              threads=bb.usable_cpus())
            got = reference[r * F + k].cpu().numpy()
            checked.append(bool(np.array_equal(got, want)))
        out["oracle_check"] = {"frames_checked": world, "all_equal": all(checked),
                               "how": "one gathered frame per rank vs oracle.render (restated render_lensmap, engine/NQ/fisheye.c:2406-2424)"}
        if not all(checked):
            print(f"[bench] gathered frames differ from the oracle: {checked}", file=sys.stderr)
    mode = args.gather_mode if args.gather_mode != "best" else max(out["modes"], key=lambda m: out["modes"][m]["value"])
    chosen = out["modes"][mode]
    out.update({"mode": mode, "ms": chosen["ms_per_step"], "value": chosen["value"], "included_in_value": True,
                "how": "blinky_shard_warp_gather (C ABI): per rank a compute stream warps chunk k+1 while a communication stream moves "
                       "chunk k to rank 0 (ncclSend/ncclRecv, copy-engine peer copies, or in-kernel peer stores)"})
    fe.shard_close()
    return out


SECONDARY = ["1080p-cube-panini170", "4k-cube-quincuncial-rubix", "4k-cube-stereographic", "4k-cube-equirect", "4k-cube-hammer",
             "4k-cube-fisheye1", "4k-trism-stereographic"]


def run_secondary(args, torch, bb, fe, peak, traffic_db, stream):
    """every other BASELINE configuration, device-resident: batched launch (16 frames) and a single cold frame
    (L2 flushed before each launch — the in-engine shape), both fractions of the HBM roofline"""
    rows = []
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    names = [args.workload] + [n for n in SECONDARY if n != args.workload]
    for name in names:
        W, H, PS = WORKLOADS[name][:3]
        F = args.frames
        build_s = setup_workload(fe, name)
        P = fe.numplates
        gen = torch.Generator(device="cuda").manual_seed(2000)
        d_faces = torch.randint(0, 256, (F, P, PS, PS), dtype=torch.uint8, device="cuda", generator=gen)
        d_out = torch.zeros((F, H, W), dtype=torch.uint8, device="cuda")
        row = {"workload": name, "lensmap_build_s": round(build_s, 3), "tiling": fe.plan_summary, "frames_per_launch": F}
        if name != args.workload:
            t = time_device(torch, fe, d_faces, d_out, F, 10, 3, stream)
            row.update({"us_per_frame": round(t * 1e6 / F, 2), "value": round(W * H * F / t / 1e6, 1), "kernel": fe.last_kernel,
                        "roofline": roofline_entry(fe, t, F, peak, traffic_db.get(name))})
        tc = time_device(torch, fe, d_faces, d_out, 1, 7, 3, stream, flush=flush)
        row["single_frame_cold"] = {"us": round(tc * 1e6, 2), "value": round(W * H / tc / 1e6, 1),
                                    "roofline": roofline_entry(fe, tc, 1, peak, None)}
        ts = time_single_frame_stream(torch, fe, d_faces, d_out, stream)
        row["single_frame_stream"] = {"us": round(ts * 1e6, 2), "value": round(W * H / ts / 1e6, 1),
                                      "roofline": roofline_entry(fe, ts, 1, peak, None),
                                      "how": "single-frame launches back to back, each on a different frame of the batch: the faces miss "
                                             "L2 (F x 25 MB > 126 MB), the tile plan stays resident — the in-engine shape"}
        rows.append(row)
        del d_faces, d_out
    return rows


if __name__ == "__main__":
    main()
