#!/usr/bin/env python
"""bench.py — embed+detect FPS of the watermark hot path on B200 (BASELINE.json metric), one JSON line.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload video4k|image1080p|image4k|image8k|batch256|image512|all] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...      # the reference path on the host CPU cores (oracle port, all threads)

Default workload: `video4k` — BASELINE configs[2], the configuration the north-star target ("at 4K", "video FPS from 1 to 8 GPUs") is
stated on: synthetic 3840x2160 u8 Y planes, watermark_interval 1, ME embed + ME detect per frame through the video driver
(`wm_process_frames`, main.cpp:343-410).  A default N = 1 run appends the record of BASELINE configs[1] (`image1080p`: NVF embed, ME embed, NVF
detect, ME detect per frame — the reference's testForImage protocol, main.cpp:167-223 — plus its literal one-image synchronous-call loop)
under the key `image1080p`; `--workload all` appends every other configuration, each with its own parity gate.

A "step" is one pass of the hot path over one batch of synthetic frames that are resident in HBM before the timed region.  The frames of a
step are generated on the device from their GLOBAL frame index, so rank r of a multi-GPU run holds exactly the contiguous chunk
`wm_shard_frames(F, r, world)` of one global frame set and processes it with `first_index = first` (the interval gate sees the global index,
main.cpp:346,395); only per-frame scalars are gathered.
`value` = frames/s over all ranks (device-timed with CUDA events, max over ranks); `e2e` = the same metric through the host-buffer entry
points (`wm_process_frames` with frames in pinned HOST memory, row padding included; `wm_*_host_batch` for images), H2D and D2H copies inside
the timed region.  Every step streams more bytes than the 126 MB L2 holds.

Roofline accounting (per kernel family, per timed bracket = one op call): algorithmic bytes = every image byte the call must read or write
once per frame + the watermark W ONCE per call (one operand per launch, shared by all its frames) — `frac`; and the DRAM bytes ncu counted
for the same kernels (profiles/r2_traffic.json, per frame x frames per call) — `frac_dram`.  A fraction above 1.05 is flagged as an
accounting error.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    # name: (rows, cols, frames per API call, calls per step, kind, dtype).  Frames per call divide the resident CTA counts of a launch
    # (4 x 148 for the sweep and the u8 kernels, 3 x 148 / 2 x 148 for f32 stats / apply / detector); frames and calls per step make the timed
    # region of a default run (20 steps) >= 1 s.
    "video4k": (2160, 3840, 1332, 1, "video", "u8"),      # one wm_process_frames call over the rank's whole chunk (79 runs of 16-17 frames inside)
    "image1080p": (1080, 1920, 148, 12, "image", "f32"),
    "image4k": (2160, 3840, 37, 12, "image", "f32"),
    "image8k": (4320, 7680, 4, 28, "image", "f32"),
    "image512": (512, 512, 296, 24, "image", "f32"),
    "batch256": (256, 256, 4096, 4, "image", "f32"),
}
# algorithmic (compulsory) bytes per pixel of ONE frame in each kernel family: image bytes read + output bytes written; W (4 B/px) is
# added once per call, not per frame (DESIGN.md section 5)
IMG_BYTES = {
    "f32": {"rx_sweep": 4, "me_stats": 4, "nvf_stats": 4, "me_apply": 8, "nvf_apply": 8, "me_detect": 4, "nvf_detect": 4},
    "u8": {"rx_sweep": 1, "me_stats": 1, "nvf_stats": 1, "me_apply": 2, "nvf_apply": 2, "me_detect": 1, "nvf_detect": 1},
}
USES_W = {"rx_sweep": 0, "me_stats": 1, "nvf_stats": 1, "me_apply": 1, "nvf_apply": 1, "me_detect": 1, "nvf_detect": 1}
# compulsory bytes per pixel of one frame's embed + detect pair: embed reads I, writes out; detect reads the marked frame
PAIR_IMG_BYTES = {"f32": 12, "u8": 3}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdin=subprocess.DEVNULL, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                mx = float(f[1])
                if t0 - 0.05 <= ts <= t1 + 0.15:
                    sm.append(float(f[0]))
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
            except ValueError:
                continue
        if not sm:  # region shorter than the sampling period: take whatever was seen
            for ts, line in self.rows:
                try:
                    sm.append(float(line.split(",")[0]))
                except ValueError:
                    pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_inputs(rows, cols, n, dtype):
    """numpy frames for the CPU arm (same recipe as the device generator: shifted natural image + light noise)."""
    import util
    base = util.natural_image(rows, cols, seed=1)
    rng = np.random.default_rng(7)
    out = np.empty((n, rows, cols), np.uint8 if dtype == "u8" else np.float32)
    for i in range(n):
        f = np.roll(base, (3 * i + 1, 5 * i + 2), (0, 1)) + rng.uniform(-2, 2, base.shape).astype(np.float32)
        f = np.clip(f, 0, 255)
        out[i] = np.rint(f) if dtype == "u8" else f
    W = util.normal_w(rows, cols, seed=28390211)
    return out, W


def device_frames(torch, dev, base_t, first, count, dtype, out=None):
    """Frames [first, first + count) of the GLOBAL synthetic stream, generated on the device: frame i = the natural base image shifted
    cyclically by (3i+1, 5i+2) + uniform noise in [-2, 2) from a generator seeded by i, clipped to 0..255 (u8: rounded).  A frame
    depends on its global index only, so every sharding of the stream sees the same frames."""
    rows, cols = base_t.shape
    tdt = torch.uint8 if dtype == "u8" else torch.float32
    if out is None:
        out = torch.empty((count, rows, cols), dtype=tdt, device=dev)
    g = torch.Generator(device=dev)
    for j in range(count):
        i = first + j
        g.manual_seed(7919 * i + 13)
        f = torch.roll(base_t, shifts=((3 * i + 1) % rows, (5 * i + 2) % cols), dims=(0, 1))
        f = f + (torch.rand((rows, cols), generator=g, device=dev, dtype=torch.float32) * 4.0 - 2.0)
        f.clamp_(0.0, 255.0)
        out[j] = torch.round(f).to(tdt) if dtype == "u8" else f
    return out


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_frame(oracle, img, W, kind):
    """one frame through the same ops as the GPU step"""
    if kind == "video":
        st, out, a = oracle.embed_frame_u8(img, W, 40.0, oracle.ME)
        oracle.detect_frame_u8(out, W, oracle.ME)
        return
    for mask in (oracle.NVF, oracle.ME):
        o = oracle.embed(img, W, 40.0, mask)
        oracle.detect(o["out"], W, mask)


def cpu_baseline(oracle, frames, W, kind, budget_s=12.0):
    t = time.perf_counter()
    cpu_frame(oracle, frames[0], W, kind)  # warm-up + calibration
    t1 = time.perf_counter() - t
    n = int(max(2, min(64, round(budget_s / max(t1, 1e-3)))))
    t = time.perf_counter()
    for i in range(n):
        cpu_frame(oracle, frames[i % len(frames)], W, kind)
    dt = time.perf_counter() - t
    return n / dt, n


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core (libgomp reads this at load)."""
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    try:  # undo bind_to_gpu_numa_node: the CPU arm uses every core of the box
        os.sched_setaffinity(0, range(os.cpu_count() or 1))
    except OSError:
        pass


METRIC = {"image": "embed+detect FPS (NVF & PE masks)", "video": "embed+detect FPS (PE mask, 4K u8 video frames)"}
OPS = {"image": "NVF embed, ME embed, NVF detect, ME detect", "video": "ME embed, ME detect"}
CPU_NOTE = ("OpenMP port restating Watermark.cpp + the kernels op for op (the reference's ArrayFire/OpenCL stack cannot be built offline); "
            "a naive port: every tap clamps its coordinates, one pass per ArrayFire op")


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    use_all_host_threads()
    from oracle import oracle
    rows, cols, nfr, ncalls, kind, dtype = WORKLOADS[wl]
    frames, W = make_inputs(rows, cols, 4, dtype)
    # bounded sample per step so the whole run ends within minutes
    t = time.perf_counter()
    cpu_frame(oracle, frames[0], W, kind)
    t1 = time.perf_counter() - t
    per_step = int(max(1, min(8, round(3.0 / max(t1, 1e-3)))))
    for _ in range(args.warmup):
        cpu_frame(oracle, frames[0], W, kind)
    t = time.perf_counter()
    for s in range(args.steps):
        for i in range(per_step):
            cpu_frame(oracle, frames[(s * per_step + i) % len(frames)], W, kind)
    dt = time.perf_counter() - t
    fps = args.steps * per_step / dt
    line = {
        "impl": "reference", "metric": METRIC[kind],
        "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if dtype == "f32" else "u8->f32", "data": "synthetic",
        "config": {"workload": wl, "rows": rows, "cols": cols, "frames_per_step": per_step, "p": 3, "psnr": 40.0, "ops_per_frame": OPS[kind]},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": oracle.num_threads(), "kind": "port",
                         "sample": "%d frame(s) per step x %d steps of %s on the host CPU; %s" % (per_step, args.steps, wl, CPU_NOTE)},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="video4k", choices=sorted(WORKLOADS) + ["all"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the image1080p record a default (video4k, N = 1) run appends")
    ap.add_argument("--no-sync-proto", action="store_true", help="skip the single-image synchronous-call measurement (keeps ncu launch lists to the timed region)")
    ap.add_argument("--exact", action="store_true", help="f32 products in Rx/rx instead of the reference's fp16 rounding")
    ap.add_argument("--frames", type=int, default=0, help="frames per API call (0 = the workload's own count)")
    ap.add_argument("--calls", type=int, default=0, help="API calls per step (0 = the workload's own count)")
    ap.add_argument("--no-tma", action="store_true", help="plain register-prefetched tile loaders instead of TMA (A/B)")
    ap.add_argument("--split-cost", type=int, default=None, help="WM_OPT_SPLIT_COST (A/B: -1 = never partition an unbalanced batch)")
    ap.add_argument("--fhadd", action="store_true", help="sum the rounded Rx/rx products with the FHADD chain instead of HMMA (A/B)")
    ap.add_argument("--no-tma-store", action="store_true", help="WM_OPT_TMA_STORE = 0: apply kernel output through per-thread vector stores (A/B)")
    ap.add_argument("--no-narrow", action="store_true", help="WM_OPT_NARROW_U8 = 0: u8 stats / apply on 256-thread CTAs (A/B)")
    ap.add_argument("--run-mb", type=int, default=0, help="WM_OPT_RUN_MB: MB of device frames per run of the video driver (A/B)")
    ap.add_argument("--host-run", type=int, default=0, help="WM_OPT_HOST_RUN_FRAMES for the e2e video path (A/B)")
    ap.add_argument("--e2e-frames", type=int, default=0, help="frames per e2e pass (0 = 128 for video, 96 for images)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of each workload computed (rank 0's frames) as "
                    "DIR/<workload>_<array>.npy in float32: per frame a and correlation of each mask type, and a fixed sample of "
                    "%d watermarked pixels per mask type (all of them when fewer)" % DUMP_PIXELS)
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args, "video4k" if args.workload == "all" else args.workload)

    import torch
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    bind_to_gpu_numa_node(torch, local_rank)
    primary = "video4k" if args.workload == "all" else args.workload
    line = run_workload(args, primary, torch, dist, dev, rank, local_rank, world)
    extra = []
    if args.workload == "all":
        extra = [w for w in ("image1080p", "image4k", "image8k", "batch256", "image512")]
    elif args.workload == "video4k" and world == 1 and not args.no_secondary:
        extra = ["image1080p"]
    for w in extra:
        torch.cuda.empty_cache()
        sec = run_workload(args, w, torch, dist, dev, rank, local_rank, world, secondary=True)
        if line is not None and sec is not None:
            keep = ("metric", "value", "unit", "ms_per_step", "steps", "dtype", "config", "step_frac_of_peak", "step_frac_sweeps", "roofline",
                    "kernels", "e2e", "gpu_launches", "sync_single_image", "parity", "cpu_baseline", "results")
            line[w] = {k: sec[k] for k in keep if k in sec}
    if line is not None:
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


NUMA_NOTE = None


def bind_to_gpu_numa_node(torch, index):
    """Pin this rank's host threads to the CPUs next to its GPU BEFORE any pinned buffer is allocated (first touch puts the pages
    on that NUMA node), so the e2e copies of several ranks do not all cross one socket's memory controllers / the inter-socket
    link.  Best effort: NVML may be missing or the box may have one node."""
    global NUMA_NOTE
    if os.environ.get("WM_BENCH_NO_AFFINITY"):
        NUMA_NOTE = "affinity off (WM_BENCH_NO_AFFINITY)"
        return
    try:
        import pynvml
        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(index)
        bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode() if bytes is str else bus)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        cpus = sorted(os.sched_getaffinity(0))
        NUMA_NOTE = "host threads bound to the %d CPUs next to GPU %s (%d..%d)" % (len(cpus), bus, cpus[0], cpus[-1])
    except Exception as e:  # noqa: BLE001
        NUMA_NOTE = "no NUMA binding (%s)" % (str(e)[:80],)


def load_traffic():
    for name in ("r2_traffic.json", "traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            try:
                return json.load(open(p)), "profiles/" + name
            except Exception:
                pass
    return {}, None


def run_workload(args, wl, torch, dist, dev, rank, local_rank, world, secondary=False):
    """One workload through warm-up, the timed region, e2e and the CPU baseline / parity gate; returns the JSON record on rank 0."""
    import util
    pkg = importlib.import_module("watermarking-gpu_b200")
    C = pkg.C

    rows, cols, nfr, ncalls, kind, dtype = WORKLOADS[wl]
    if args.frames:
        nfr = args.frames
    if args.calls:
        ncalls = args.calls
    npx = rows * cols
    per_rank = nfr * ncalls                      # frames of this rank per step
    total = per_rank * world                     # frames of the global stream per step
    first, count = pkg.shard_frames(total, rank, world)
    assert count == per_rank
    W = util.normal_w(rows, cols, seed=28390211)
    stream = torch.cuda.Stream(device=dev)
    wm = pkg.Watermark(rows, cols, W, 3, 40.0, device=local_rank, stream=stream.cuda_stream)
    if args.exact:
        wm.set_option(pkg.OPT_FP16_PRODUCTS, 0)
    if args.fhadd:
        wm.set_option(pkg.OPT_MMA_ACCUM, 0)
    if args.no_tma:
        wm.set_option(pkg.OPT_USE_TMA, 0)
    if args.split_cost is not None:
        wm.set_option(pkg.OPT_SPLIT_COST, args.split_cost)
    if args.host_run:
        wm.set_option(pkg.OPT_HOST_RUN_FRAMES, args.host_run)
    if args.no_tma_store:
        wm.set_option(pkg.OPT_TMA_STORE, 0)
    if args.no_narrow:
        wm.set_option(pkg.OPT_NARROW_U8, 0)
    if args.run_mb:
        wm.set_option(pkg.OPT_RUN_MB, args.run_mb)
    dt_code = pkg.U8 if dtype == "u8" else pkg.F32
    esz = 1 if dtype == "u8" else 4
    # image workloads: ArrayFire layout (column-major); video: row-major Y planes
    layout = pkg.ROW_MAJOR if kind == "video" else pkg.COL_MAJOR
    base_np = util.natural_image(rows, cols, seed=1)
    base_t = torch.from_numpy(base_np if layout == pkg.ROW_MAJOR else np.ascontiguousarray(base_np.T)).to(dev)
    # the device generator works in MEMORY order: for column-major images the base is transposed first, so frame i of the stream is the
    # same logical image whatever the layout
    d_in = device_frames(torch, dev, base_t, first, count, dtype)
    nout = 1 if kind == "video" else 2
    d_out = [torch.empty_like(d_in) for _ in range(nout)]  # video: ME-marked; images: NVF-marked, ME-marked
    a_host = [np.zeros(count, np.float32) for _ in range(2)]
    c_host = [np.zeros(count, np.float32) for _ in range(2)]
    st_host = np.zeros(count, np.int32)

    def logical(mem):  # memory-order frame -> logical (rows, cols)
        return mem if layout == pkg.ROW_MAJOR else np.ascontiguousarray(mem.T)

    vctx = pkg.VideoProcessingContext(wm, rows, cols, 1, linesize=cols, frames_on_device=True)

    def step():
        if kind == "video":
            for c in range(ncalls):
                o = c * nfr
                pkg.process_frames(vctx, pkg.VIDEO_EMBED, d_in[o].data_ptr(), d_out[0][o].data_ptr(), first + o, nfr, a_host[1][o:o + nfr])
                pkg.process_frames(vctx, pkg.VIDEO_DETECT, d_out[0][o].data_ptr(), None, first + o, nfr, c_host[1][o:o + nfr])
            return
        for c in range(ncalls):
            o = c * nfr
            di = pkg.image_desc(d_in[o].data_ptr(), rows, cols, layout, dt_code)
            for k, mask in enumerate((pkg.NVF, pkg.ME)):
                do = pkg.image_desc(d_out[k][o].data_ptr(), rows, cols, layout, dt_code)
                wm.embed_batch(0, di, di, do, npx, npx, npx, nfr, mask, a_host[k][o:o + nfr], st_host[o:o + nfr])
                wm.detect_batch(0, do, npx, nfr, mask, c_host[k][o:o + nfr], st_host[o:o + nfr])
        wm.sync(0)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    with torch.cuda.stream(stream):
        sampler = ClockSampler(local_rank) if rank == 0 else None
        t_warm = time.time()
        for _ in range(args.warmup):
            step()
        while time.time() - t_warm < 0.5:  # keep the GPU under the same load until the sampler has a few readings
            step()
        barrier()
        l0 = wm.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record(stream)
        for _ in range(args.steps):
            step()
        e1.record(stream)
        barrier()
        t1 = time.time()
        ms = e0.elapsed_time(e1)
        launches = wm.launch_count - l0
        # before anything else runs on the frames: the passes below recompute or overwrite the outputs
        outputs = last_step_outputs(torch, dev, d_out, a_host, c_host, kind, layout == pkg.ROW_MAJOR, rows, cols) \
            if args.dump_outputs and rank == 0 else None
        # per-kernel durations for the roofline: one more pass with CUDA-event brackets around every kernel family of every call, the video
        # driver's slots serialised (wm option 4) so that a bracket holds one kernel family and nothing else
        if kind == "video":
            wm.set_option(pkg.OPT_SERIAL_SLOTS, 1)
        wm.set_option(pkg.OPT_KERNEL_TIMING, 1)
        wm.kernel_times(reset=True)
        k_steps = max(1, min(args.steps, 3))
        for _ in range(k_steps):
            step()
        torch.cuda.synchronize(dev)
        ktimes = wm.kernel_times(reset=True)
        wm.set_option(pkg.OPT_KERNEL_TIMING, 0)
        wm.set_option(pkg.OPT_SERIAL_SLOTS, 0)
    clocks = sampler.stop(t_warm + 0.2, t1) if sampler else None
    if dist is not None:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    fps = total * args.steps / (ms * 1e-3)

    # ---- e2e through the host-buffer entry points: frames start in pinned HOST memory, results end there ----
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, pkg, torch, dist, dev, wm, wl, d_in, a_host, c_host, first, world)

    # the reference's literal protocol for the image configs (main.cpp:167-223): ONE image, synchronous calls, mean over loops
    sync_proto = None
    if kind == "image" and rank == 0 and not args.no_sync_proto:
        one_in = pkg.image_desc(d_in.data_ptr(), rows, cols, layout, dt_code)
        one_out = pkg.image_desc(d_out[0].data_ptr(), rows, cols, layout, dt_code)
        av, cv = C.c_float(0), C.c_float(0)
        L_ = pkg.lib()
        loops = 200 if npx <= 4 * 2073600 else 50

        def four_ops():
            for mask in (pkg.NVF, pkg.ME):
                L_.wm_embed(wm._h, C.byref(one_in), C.byref(one_in), C.byref(one_out), mask, C.byref(av))
                L_.wm_detect(wm._h, C.byref(one_out), mask, C.byref(cv))

        for _ in range(3):
            four_ops()
        tt = time.perf_counter()
        for _ in range(loops):
            four_ops()
        dt_s = time.perf_counter() - tt
        sync_proto = {"value": loops / dt_s, "unit": "frames/s", "us_per_frame": 1e6 * dt_s / loops, "loops": loops,
                      "what": "the reference's literal loops_for_test protocol: one resident image, synchronous wm_embed / wm_detect calls (4 per frame), CUDA-graph replay"}
        step()  # the four ops above overwrote frame 0's scalars / outputs: restore the batch results the parity gate reads
        torch.cuda.synchronize(dev)

    # ---- multi-GPU: the only data that crosses ranks are per-frame scalars (SURVEY.md 8e), gathered after the timed region ----
    shard = None
    if dist is not None:
        shard = check_sharding(pkg, torch, dist, dev, wm, vctx if kind == "video" else None, base_t, dtype, kind, layout, dt_code, rows, cols,
                               first, count, total, world, rank, a_host[1], c_host[1], d_out)
    if rank != 0:
        return None

    # ---- roofline per kernel family ----
    peak, peak_src = peaks()
    traffic, traffic_src = load_traffic()
    tr_frame = traffic.get(wl, {}).get("per_frame", {})
    in_frame = traffic.get(wl, {}).get("warp_instr_per_frame", {})
    # the bound the kernels actually sit on: warp-instruction issue.  Peak = 4 schedulers x SMs x SM clock (one warp instruction per
    # scheduler per clock); achieved = warp instructions ncu counted per frame x frames per launch / the launch's CUDA-event time
    props = torch.cuda.get_device_properties(dev)
    sm_mhz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz") or 1965.0
    issue_peak = 4.0 * props.multi_processor_count * sm_mhz * 1e6
    kern = []
    calls_frames = per_rank * k_steps            # frames one kernel family covered per op kind in the bracketed passes
    for name, (n, tot_ms) in ktimes.items():
        if n == 0:
            continue
        ops = 1
        if name == "rx_sweep":
            ops = 3 if kind == "image" else 2     # ME embed, NVF detect, ME detect / ME embed, ME detect
        frames_per_launch = calls_frames * ops / n
        alg = IMG_BYTES[dtype][name] * npx * frames_per_launch + USES_W[name] * 4 * npx
        avg_ms = tot_ms / n
        rec = {"kernel": name, "launches": n, "avg_ms": avg_ms, "total_ms": tot_ms, "frames_per_launch": frames_per_launch,
               "alg_bytes_per_launch": alg, "achieved_gbs": alg / (avg_ms * 1e-3) / 1e9, "frac": alg / (avg_ms * 1e-3) / 1e9 / peak}
        if name in tr_frame:
            rec["traffic"] = tr_frame[name] * frames_per_launch
            rec["frac_dram"] = rec["traffic"] / (avg_ms * 1e-3) / 1e9 / peak
        if name in in_frame:
            rec["warp_instr_per_launch"] = in_frame[name] * frames_per_launch
            rec["issue_frac"] = rec["warp_instr_per_launch"] / (avg_ms * 1e-3) / issue_peak
            rec["instr_per_px"] = in_frame[name] * 32.0 / npx
        if rec["frac"] > 1.05:
            rec["accounting_error"] = "fraction above the HBM peak: the byte count is wrong"
        kern.append(rec)
    kern.sort(key=lambda k: -k["total_ms"])
    dom = kern[0] if kern else None
    roof = None
    if dom:
        roof = {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved_gbs"], "peak": peak, "unit": "GB/s",
                "frac": dom["frac"], "traffic": dom.get("traffic"), "frac_dram": dom.get("frac_dram"), "peak_source": peak_src,
                "issue_frac": dom.get("issue_frac"), "instr_per_px": dom.get("instr_per_px"),
                "issue_peak_winst_per_s": issue_peak,
                "alg_bytes_per_launch": dom["alg_bytes_per_launch"], "avg_launch_ms": dom["avg_ms"], "frames_per_launch": dom["frames_per_launch"],
                "traffic_source": traffic_src and traffic_src + " (ncu dram__bytes_read.sum + dram__bytes_write.sum per frame x frames per launch)",
                "accounting": "image bytes once per frame + W once per launch; kernel time = CUDA-event bracket of one op call",
                "issue_bound_note": "the path is instruction-issue bound, not HBM bound (profiles/r2_README.md): the reference's arithmetic costs more issue slots "
                                    "per pixel than an HBM-rate stream leaves time for"}
    # whole step: compulsory bytes of the embed + detect pairs (image once in, once out, marked image once in; W once per op call),
    # and the sum of the per-kernel algorithmic bytes (every dependence-mandated sweep streams its image)
    pairs = 2 if kind == "image" else 1
    op_calls = sum(k["launches"] for k in kern if k["kernel"] in ("me_apply", "nvf_apply", "me_detect", "nvf_detect")) / k_steps  # embed / detect calls per step
    step_bytes = PAIR_IMG_BYTES[dtype] * npx * per_rank * pairs + op_calls * 4 * npx
    sweeps_bytes = sum(k["alg_bytes_per_launch"] * k["launches"] for k in kern) / k_steps
    step_s = ms / args.steps * 1e-3

    cb = None
    parity = None
    if not args.no_cpu_baseline and world == 1:  # rank 0 at N = 1 only
        use_all_host_threads()
        from oracle import oracle
        nh = min(count, 4)
        frames_np = np.stack([logical(d_in[i].cpu().numpy()) for i in range(nh)])
        v, n = cpu_baseline(oracle, frames_np, W, kind, budget_s=12.0 if not secondary else 6.0)
        # parity gate in the same job (SURVEY.md 8d): frame 0 through the oracle against the scalars the timed region produced
        if kind == "image":
            chk = {}
            for k2, mask in enumerate((oracle.NVF, oracle.ME)):
                o = oracle.embed(frames_np[0], W, 40.0, mask)
                od = oracle.detect(o["out"], W, mask)
                got = logical(d_out[k2][0].cpu().numpy())
                chk["a_%s_rel" % ("nvf", "me")[k2]] = abs(float(a_host[k2][0]) - o["a"]) / abs(o["a"])
                chk["corr_%s_rel" % ("nvf", "me")[k2]] = abs(float(c_host[k2][0]) - od["corr"]) / abs(od["corr"])
                chk["pixels_%s_maxabs" % ("nvf", "me")[k2]] = float(np.abs(got - o["out"]).max())
            ok = all(v_ <= 1e-3 for k_, v_ in chk.items() if k_.endswith("_rel")) and all(v_ <= 1e-4 * 255 for k_, v_ in chk.items() if k_.endswith("_maxabs"))
        else:
            st_, out_, a_ = oracle.embed_frame_u8(frames_np[0], W, 40.0, oracle.ME)
            corr_ = oracle.detect_frame_u8(out_, W, oracle.ME)[1]
            got = d_out[0][0].cpu().numpy()
            chk = {"a_me_rel": abs(float(a_host[1][0]) - a_) / abs(a_), "corr_me_rel": abs(float(c_host[1][0]) - corr_) / abs(corr_),
                   "pixels_max_lsb": int(np.abs(got.astype(np.int32) - out_.astype(np.int32)).max())}
            ok = chk["a_me_rel"] <= 1e-3 and chk["corr_me_rel"] <= 1e-3 and chk["pixels_max_lsb"] <= 1
        parity = dict(chk, tolerance="a, corr 1e-3 relative; f32 pixels 1e-4 x 255; u8 pixels 1 LSB", ok=bool(ok),
                      what="frame 0: scalars and output pixels of the timed region vs the CPU oracle")
        cb = {"value": v, "unit": "frames/s", "cores": oracle.num_threads(), "kind": "port",
              "sample": "%d frames of %s, same ops per frame; %s" % (n, wl, CPU_NOTE)}
    line = {
        "metric": METRIC[kind],
        "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "wall_ms_per_step": (t1 - t0) * 1e3 / args.steps, "timed_region_s": ms * 1e-3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if dtype == "f32" else "u8->f32", "data": "synthetic",
        "config": {"workload": wl, "rows": rows, "cols": cols, "frames_per_step": total, "frames_per_step_per_gpu": per_rank,
                   "frames_per_call": nfr, "calls_per_step": ncalls, "p": 3, "psnr": 40.0,
                   "layout": "col-major (ArrayFire)" if layout == pkg.COL_MAJOR else "row-major Y plane",
                   "ops_per_frame": OPS[kind], "fp16_products": not args.exact,
                   "l2": "inputs larger than L2: %.0f MB of frames + W per step per GPU" % ((d_in.numel() * esz + W.nbytes) / 1e6),
                   "sharding": "one global frame stream generated from the global frame index; rank r holds chunk wm_shard_frames(F, r, world) and "
                               "processes it with first_index = first; no collective on the data path",
                   "first_index": first},
        "step_effective_gbs": step_bytes / step_s / 1e9, "step_frac_of_peak": step_bytes / step_s / 1e9 / peak,
        "step_frac_sweeps": sweeps_bytes / step_s / 1e9 / peak,
        "roofline": roof, "kernels": kern, "cpu_baseline": cb, "e2e": e2e, "gpu_launches": int(launches),
        "sync_single_image": sync_proto, "parity": parity, "sharding_check": shard,
        "clocks": clocks,
        "results": {"a_nvf": float(a_host[0][0]), "a_me": float(a_host[1][0]), "corr_nvf": float(c_host[0][0]), "corr_me": float(c_host[1][0])},
    }
    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in outputs.items():
            np.save(os.path.join(args.dump_outputs, "%s_%s.npy" % (wl, name)), arr)
    return line


DUMP_PIXELS = 1 << 20  # per mask type: the dumps of a `--workload all` run (11 outputs) stay under 64 MB


def last_step_outputs(torch, dev, d_out, a_host, c_host, kind, row_major, rows, cols):
    """What a caller of the timed path holds after its last step, as float32 arrays: per frame the strength factor `a` and the
    correlation of each mask type, and the watermarked frames as a seeded sample of logical (frame, row, col) positions that is the
    same in every run with the same frame count and shape."""
    count = d_out[0].shape[0]
    npx = rows * cols
    n = count * npx
    pick = np.arange(n) if n <= DUMP_PIXELS else np.sort(np.random.default_rng(28390211).choice(n, DUMP_PIXELS, replace=False))
    f, r, c = pick // npx, pick % npx // cols, pick % cols
    idx = torch.from_numpy(f * npx + (r * cols + c if row_major else c * rows + r)).to(dev)
    masks = [("me", 0, 1)] if kind == "video" else [("nvf", 0, 0), ("me", 1, 1)]  # (name, index in d_out, index in a_host / c_host)
    out = {}
    for name, k, s in masks:
        out[name + "_a"] = a_host[s].astype(np.float32)
        out[name + "_corr"] = c_host[s].astype(np.float32)
        out[name + "_out_sample"] = d_out[k].reshape(-1).index_select(0, idx).float().cpu().numpy()
    return out


def run_e2e(args, pkg, torch, dist, dev, wm, wl, d_in, a_host, c_host, first, world):
    """Frames/s through the host-buffer entry points, copies inside the timed region (wall clock around whole passes, max over ranks)."""
    rows, cols, nfr, ncalls, kind, dtype = WORKLOADS[wl]
    esz = 1 if dtype == "u8" else 4
    dt_code = pkg.U8 if dtype == "u8" else pkg.F32
    layout = pkg.ROW_MAJOR if kind == "video" else pkg.COL_MAJOR
    n = args.e2e_frames or (128 if kind == "video" else 96)
    n = min(n, d_in.shape[0])
    L_, P_ = d_in.shape[1], d_in.shape[2]
    if kind == "video":
        # decoded frames as ffmpeg hands them over: rows padded to `linesize` > width (main.cpp:348-353 repacks them)
        linesize = cols + 64
        pin_in = torch.zeros((n, rows, linesize), dtype=torch.uint8).pin_memory()
        pin_in[:, :, :cols].copy_(d_in[:n].cpu())
        pin_out = torch.empty((n, rows, cols), dtype=torch.uint8).pin_memory()
        sc = np.zeros(2 * n, np.float32)
        vh = pkg.VideoProcessingContext(wm, rows, cols, 1, linesize=linesize, frames_on_device=False)

        def one_pass():
            pkg.process_frames(vh, pkg.VIDEO_EMBED_VERIFY, pin_in.data_ptr(), pin_out.data_ptr(), first, n, sc)

        h2d, d2h = n * rows * cols, n * rows * cols + 2 * 4 * n
        api = "wm_process_frames(WM_VIDEO_EMBED_VERIFY, frames_on_device = 0): pinned host frames with linesize = width + 64 in, watermarked frames + a + correlation out"
        same = lambda: bool(np.allclose(sc[:n], a_host[1][:n], rtol=1e-6, equal_nan=True) and np.allclose(sc[n:], c_host[1][:n], rtol=1e-5, atol=1e-7, equal_nan=True))
    else:
        npx = rows * cols
        pin_in = d_in[:n].cpu().pin_memory()
        pin_out = [torch.empty_like(pin_in).pin_memory() for _ in range(2)]
        a_e = [np.zeros(n, np.float32) for _ in range(2)]
        c_e = [np.zeros(n, np.float32) for _ in range(2)]
        chunk = 4 if npx * esz <= (40 << 20) else 1
        NS = wm.num_slots

        def one_pass():
            for ci, o in enumerate(range(0, n, chunk)):
                nb = min(chunk, n - o)
                hin = pkg.image_desc(pin_in[o].data_ptr(), rows, cols, layout, dt_code)
                for k2, mask in enumerate((pkg.NVF, pkg.ME)):
                    # consecutive calls go to different slots (streams): on one slot the second upload would queue behind the first
                    # call's download and detector, and the copy engines (FIFO in submission order) would alternate instead of overlapping
                    sl = (2 * ci + k2) % NS
                    hout = pkg.image_desc(pin_out[k2][o].data_ptr(), rows, cols, layout, dt_code)
                    # embed, download the watermarked images, detect on them where they lie on the device (main.cpp:178-217)
                    wm.embed_verify_host_batch(sl, hin, hin, hout, npx, npx, npx, nb, mask, a_e[k2][o:o + nb], c_e[k2][o:o + nb])
            wm.sync(-1)

        h2d, d2h = 2 * n * npx * esz, 2 * n * npx * esz + 4 * 4 * n
        api = ("wm_embed_verify_host_batch on rotating slots (%d frames per call): pinned host images in (once per mask type), watermarked "
               "images + strengths + correlations out" % chunk)
        same = lambda: bool(np.allclose(a_e[1], a_host[1][:n], rtol=1e-6) and np.allclose(c_e[1], c_host[1][:n], rtol=1e-5, atol=1e-7))
    one_pass()  # warm-up: staging buffers, pinned result rings
    torch.cuda.synchronize(dev)
    if dist is not None:
        dist.barrier()
    reps = max(2, min(args.steps, 8))
    tt = time.perf_counter()
    for _ in range(reps):
        one_pass()
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - tt
    if dist is not None:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    v = world * reps * n / e2e_s
    return {"value": v, "unit": "frames/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "frames_per_step": n, "passes": reps, "matches_resident_path": same(),
            "h2d_gbs": v * h2d / n / 1e9, "d2h_gbs": v * d2h / n / 1e9, "host_affinity": NUMA_NOTE,
            "pcie_note": "tools/pcie_bw.py on this pool's boxes (profiles/r1_pcie_bw.txt): one GPU copies 55 GB/s one way, 46 GB/s each way when both "
                         "directions run; all 8 GPUs together get 118 GB/s D2H / 77 GB/s each way, which caps e2e at N = 8",
            "api": api}


def check_sharding(pkg, torch, dist, dev, wm, vctx, base_t, dtype, kind, layout, dt_code, rows, cols, first, count, total, world, rank,
                   a_mine, c_mine, d_out):
    """After the timed region: gather the per-frame scalars of all ranks into one array indexed by GLOBAL frame, then prove the sharding:
    (1) rank 0 regenerates the first two frames of every other rank's chunk from their global indices, runs them itself and must get the
    same scalars (to 1e-6 relative: two frames per launch get a different CTA split than a run of eleven, so the f64 sums of the
    second stage are added in another order); (2) video: a detect pass with watermark_interval = 2 must gate on the GLOBAL index across chunk boundaries."""
    npx = rows * cols
    mine = torch.from_numpy(np.stack([a_mine, c_mine])).to(dev)
    parts = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(parts, mine)
    glob = torch.cat(parts, dim=1).cpu().numpy()  # [(a, corr), global frame]
    res = {"ranks": world, "frames_total": int(total), "first_index": int(first), "gathered": int(glob.shape[1])}
    gate = None
    if vctx is not None:
        v2 = pkg.VideoProcessingContext(wm, rows, cols, 2, linesize=cols, frames_on_device=True)
        c2 = np.zeros(count, np.float32)
        pkg.process_frames(v2, pkg.VIDEO_DETECT, d_out[0].data_ptr(), None, first, count, c2)
        t2 = torch.from_numpy(c2).to(dev)
        p2 = [torch.empty_like(t2) for _ in range(world)]
        dist.all_gather(p2, t2)
        g2 = torch.cat(p2).cpu().numpy()
        idx = np.arange(total)
        gate = bool(np.all(np.isnan(g2[idx % 2 == 1])) and np.array_equal(g2[idx % 2 == 0], glob[1][idx % 2 == 0]))
        res["interval2_gates_on_global_index"] = gate
    if rank == 0:
        worst = 0.0
        checked = 0
        for r in range(1, world):
            f_r, _ = pkg.shard_frames(total, r, world)
            fr = device_frames(torch, dev, base_t, f_r, 2, dtype)
            out = torch.empty_like(fr)
            torch.cuda.synchronize(dev)  # the frames are generated on torch's stream, the library runs on its own (non-blocking) streams
            a2, c2 = np.zeros(2, np.float32), np.zeros(2, np.float32)
            if vctx is not None:
                pkg.process_frames(vctx, pkg.VIDEO_EMBED, fr.data_ptr(), out.data_ptr(), f_r, 2, a2)
                pkg.process_frames(vctx, pkg.VIDEO_DETECT, out.data_ptr(), None, f_r, 2, c2)
            else:
                di = pkg.image_desc(fr.data_ptr(), rows, cols, layout, dt_code)
                do = pkg.image_desc(out.data_ptr(), rows, cols, layout, dt_code)
                wm.embed_batch(0, di, di, do, npx, npx, npx, 2, pkg.ME, a2)
                wm.detect_batch(0, do, npx, 2, pkg.ME, c2)
                wm.sync(0)
            for got, want in ((a2, glob[0][f_r:f_r + 2]), (c2, glob[1][f_r:f_r + 2])):
                worst = max(worst, float(np.max(np.abs(got - want) / np.abs(want))))
            checked += 2
        res["other_ranks_frames_rerun_on_rank0"] = checked
        res["rerun_max_rel_diff"] = worst
        res["gathered_scalars_match_single_rank_run"] = bool(worst <= 1e-6)
        res["a_me_mean"] = float(np.nanmean(glob[0]))
        res["corr_me_mean"] = float(np.nanmean(glob[1]))
    return res


if __name__ == "__main__":
    sys.exit(main())
