"""v210 frames (WM_PACKED_V210: DeckLink / ffmpeg 10-bit 4:2:2) through the video driver, against what a caller composes today.  Prints one
JSON line.

Workloads (ME mask, WM_VIDEO_EMBED_VERIFY with every frame gated; frame sets larger than the 126 MB of L2; widths multiples of 48, so a
row is whole groups):
  driver : frames and output on the device, 1080p x 48 and 4K x 12, in three arms that alternate in one process, each for at least
           --seconds per run, two runs, bracketed by CUDA events (every arm returns after its work has completed):
    v210     : (a) the v210 frames handed over as they are
    composed : (b) what a caller writes without WM_PACKED_V210: torch unpacks the luma into WM_Y10 words, wm_embed_batch / WM_Y10,
               torch repacks the output words into the input's groups, wm_detect_batch / WM_Y10 on the output words; the torch work
               runs on the library's slot stream, so nothing waits between the steps
    y10      : (c) the WM_Y10 driver on the same luma, for context
  e2e    : pinned host frames with 64 bytes of row padding, v210 and y10 arms, host clock
After the timed region frame 0 of every arm is checked against the CPU oracle on x = v / 4 (a and the correlation within 1e-3 relative,
samples within one code), and the bytes of arm (a) against arm (b).
--profile: a separate run of arm (a) under torch.profiler, reporting the mean CUDA time of each kernel per launch (extraction and pack
kernels included), instead of the timed workloads.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import packed_rgb_bench as rb  # noqa: E402  (gpu_info; puts the repository and tests/ on sys.path)
import util  # noqa: E402
from y10_bench import gate10, timed_runs  # noqa: E402
from test_gpu_v210 import pack, pitch, unpack_luma  # noqa: E402

wmb = rb.wmb
PSNR = rb.PSNR
KEEP = (~(0x3FF << 10), ~(0x3FF | 0x3FF << 20), ~(0x3FF << 10), ~(0x3FF | 0x3FF << 20))  # the non-luma bits of the words of a group


def frames(rows, cols, n):
    """(n, rows) luma samples and v210 frames (n, rows, pitch) uint8 around them, with random chroma and bits 30-31"""
    rng = np.random.default_rng(7)
    base = [np.clip(np.rint(util.natural_image(rows, cols, seed=13 * j) * 4.0 + rng.integers(-2, 3, (rows, cols))), 0, 1023) for j in range(4)]
    v = np.stack([np.roll(base[i % 4], 6 * i, axis=1) for i in range(n)]).astype(np.uint16)
    f = np.stack([pack(v[i], seed=100 + i) for i in range(n)])
    return v, f


def rates(per_call, n):
    r = {}
    for a, ts in per_call.items():
        fps = [n / t for t in ts]
        r[a] = {"frames_per_s": [round(x, 1) for x in fps], "spread_pct": round(100.0 * (max(fps) - min(fps)) / min(fps), 2)}
    if "composed" in r:
        r["v210_over_composed"] = round(min(r["v210"]["frames_per_s"]) / max(r["composed"]["frames_per_s"]), 3)
    r["v210_over_y10"] = round(np.mean(r["v210"]["frames_per_s"]) / np.mean(r["y10"]["frames_per_s"]), 3)
    return r


def driver_workload(rows, cols, n, seconds, oracle):
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    v, f = frames(rows, cols, n)
    ng = cols // 6
    dv = torch.from_numpy(f).cuda()  # v210 frames
    dvo = torch.empty_like(dv)
    dy = torch.from_numpy(v.view(np.int16)).cuda()  # the same luma as WM_Y10 words
    dyo = torch.empty_like(dy)
    w10, o10 = torch.empty((n, rows, cols), dtype=torch.int16, device="cuda"), torch.empty((n, rows, cols), dtype=torch.int16, device="cuda")
    cvo = torch.empty_like(dv)
    keep = torch.tensor(KEEP, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    sv, sy = np.zeros(2 * n, np.float32), np.zeros(2 * n, np.float32)
    ac, sc, cc, scc = np.zeros(n, np.float32), np.zeros(n, np.int32), np.zeros(n, np.float32), np.zeros(n, np.int32)
    vv = wmb.VideoProcessingContext(wm, rows, cols, 1, frames_on_device=True, layout=wmb.PACKED_V210)
    vy = wmb.VideoProcessingContext(wm, rows, cols, 1, frames_on_device=True, layout=wmb.Y10)
    slot = torch.cuda.ExternalStream(wm.stream(0))
    d10 = lambda t: wmb.image_desc(t.data_ptr(), rows, cols, wmb.Y10, wmb.U8, 0, 2)

    def v210():
        wmb.process_frames(vv, wmb.VIDEO_EMBED_VERIFY, dv.data_ptr(), dvo.data_ptr(), 0, n, sv)

    def composed():
        with torch.cuda.stream(slot):
            g = dv.view(torch.int32).view(n, rows, ng, 4)
            y = torch.stack([g[..., 0] >> 10, g[..., 1], g[..., 1] >> 20, g[..., 2] >> 10, g[..., 3], g[..., 3] >> 20], -1) & 1023
            w10.copy_(y.view(n, rows, cols))
            wm.embed_batch(0, d10(w10), d10(w10), d10(o10), 0, 0, 0, n, wmb.ME, ac, sc)
            q = o10.view(n, rows, ng, 6).to(torch.int32)
            out = cvo.view(torch.int32).view(n, rows, ng, 4)
            torch.bitwise_and(g, keep, out=out)
            out[..., 0] |= q[..., 0] << 10
            out[..., 1] |= q[..., 1] | q[..., 2] << 20
            out[..., 2] |= q[..., 3] << 10
            out[..., 3] |= q[..., 4] | q[..., 5] << 20
            wm.detect_batch(0, d10(o10), 0, n, wmb.ME, cc, scc)
        wm.sync(0)

    def y10():
        wmb.process_frames(vy, wmb.VIDEO_EMBED_VERIFY, dy.data_ptr(), dyo.data_ptr(), 0, n, sy)

    r = rates(timed_runs({"v210": v210, "composed": composed, "y10": y10}, seconds), n)
    v210()
    composed()
    y10()
    torch.cuda.synchronize()
    ov, oc = dvo.cpu().numpy(), cvo.cpu().numpy()
    r["gate"] = {"v210": gate10(oracle, W, v[0], unpack_luma(ov[0], cols), sv[0], sv[n]),
                 "composed": gate10(oracle, W, v[0], unpack_luma(oc[0], cols), ac[0], cc[0]),
                 "y10": gate10(oracle, W, v[0], dyo[0].cpu().numpy().view(np.uint16), sy[0], sy[n])}
    r["v210_equals_composed_bytes"] = bool(np.array_equal(ov, oc))
    r["gate"]["v210"]["ok"] = r["gate"]["v210"]["ok"] and r["v210_equals_composed_bytes"]
    wm.close()
    return {"workload": "driver", "rows": rows, "cols": cols, "frames": n, "frame_set_mb": round(f.nbytes / 2**20, 1), **r}


def e2e_workload(rows, cols, n, seconds, oracle):
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    v, f = frames(rows, cols, n)
    pb = pitch(cols)
    ls, ls10 = pb + 64, 2 * cols + 64
    hin = torch.zeros((n, rows, ls), dtype=torch.uint8).pin_memory()
    hin[:, :, :pb] = torch.from_numpy(f)
    hout = torch.empty((n, rows, pb), dtype=torch.uint8).pin_memory()
    h10 = torch.zeros((n, rows, ls10), dtype=torch.uint8).pin_memory()
    h10[:, :, :2 * cols] = torch.from_numpy(v.view(np.uint8).reshape(n, rows, 2 * cols))
    h10o = torch.empty((n, rows, 2 * cols), dtype=torch.uint8).pin_memory()
    sv, sy = np.zeros(2 * n, np.float32), np.zeros(2 * n, np.float32)
    vv = wmb.VideoProcessingContext(wm, rows, cols, 1, linesize=ls, layout=wmb.PACKED_V210)
    vy = wmb.VideoProcessingContext(wm, rows, cols, 1, linesize=ls10, layout=wmb.Y10)

    def v210():
        wmb.process_frames(vv, wmb.VIDEO_EMBED_VERIFY, hin.data_ptr(), hout.data_ptr(), 0, n, sv)

    def y10():
        wmb.process_frames(vy, wmb.VIDEO_EMBED_VERIFY, h10.data_ptr(), h10o.data_ptr(), 0, n, sy)

    r = rates(timed_runs({"v210": v210, "y10": y10}, seconds, host_clock=True), n)
    r["v210"]["linesize"] = ls
    v210()
    y10()
    r["gate"] = {"v210": gate10(oracle, W, v[0], unpack_luma(hout[0].numpy(), cols), sv[0], sv[n]),
                 "y10": gate10(oracle, W, v[0], h10o[0].numpy().view(np.uint16), sy[0], sy[n])}
    wm.close()
    return {"workload": "e2e", "rows": rows, "cols": cols, "frames": n, **r}


def profile(rows, cols, n, out_dir):
    """arm (a) under torch.profiler -> {kernel name: mean us per launch}"""
    from torch.profiler import ProfilerActivity, profile as tprofile
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    _, f = frames(rows, cols, n)
    dv, dvo = torch.from_numpy(f).cuda(), torch.empty((n, rows, pitch(cols)), dtype=torch.uint8, device="cuda")
    sv = np.zeros(2 * n, np.float32)
    vv = wmb.VideoProcessingContext(wm, rows, cols, 1, frames_on_device=True, layout=wmb.PACKED_V210)
    run = lambda: wmb.process_frames(vv, wmb.VIDEO_EMBED_VERIFY, dv.data_ptr(), dvo.data_ptr(), 0, n, sv)
    run()
    torch.cuda.synchronize()
    with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            run()
        torch.cuda.synchronize()
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        prof.export_chrome_trace(os.path.join(out_dir, "v210_%dx%d.json" % (rows, cols)))
    k = {}
    for e in prof.key_averages():
        if e.device_type == torch.autograd.DeviceType.CUDA and e.count:
            name = e.key.split("(")[0].split("<")[0].replace("void ", "").replace("wm::", "")
            t = k.setdefault(name, [0.0, 0])
            t[0] += e.device_time_total
            t[1] += e.count
    wm.close()
    return {"rows": rows, "cols": cols, "frames_per_call": n, "calls": 5,
            "kernels_us_per_launch": {a: round(t / c, 1) for a, (t, c) in sorted(k.items(), key=lambda x: -x[1][0])},
            "kernels_us_per_frame": {a: round(t / (5 * n), 1) for a, (t, c) in sorted(k.items(), key=lambda x: -x[1][0])}}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--seconds", type=float, default=1.0, help="timed work per arm and run (at least)")
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    ap.add_argument("--profile", action="store_true", help="kernel times of arm (a) under torch.profiler instead of the timed workloads")
    ap.add_argument("--trace-dir", default="", help="--profile: also write the chrome traces here")
    args = ap.parse_args()
    if not torch.cuda.is_available() or wmb.device_count() < 1:
        sys.exit("v210_bench: no CUDA device (this measurement has no CPU fallback)")
    name, power = rb.gpu_info()
    if args.profile:
        sizes = [(270, 480, 8)] if args.quick else [(1080, 1920, 48), (2160, 3840, 12)]
        print(json.dumps({"tool": "v210_bench", "gpu": name, "power_limit": power, "profile": [profile(r, c, n, args.trace_dir) for r, c, n in sizes]}))
        return
    from oracle import oracle
    oracle.lib()
    if args.quick:
        res = [driver_workload(270, 480, 8, args.seconds, oracle), e2e_workload(270, 480, 8, args.seconds, oracle)]
    else:
        res = [driver_workload(1080, 1920, 48, args.seconds, oracle), driver_workload(2160, 3840, 12, args.seconds, oracle),
               e2e_workload(1080, 1920, 48, args.seconds, oracle), e2e_workload(2160, 3840, 12, args.seconds, oracle)]
    ok = all(g["ok"] for w in res for g in w["gate"].values())
    bar = all(w["v210_over_composed"] > 1.0 for w in res if "v210_over_composed" in w)
    print(json.dumps({"tool": "v210_bench", "gpu": name, "power_limit": power, "mask": "ME", "mode": "EMBED_VERIFY", "interval": 1,
                      "workloads": res, "parity_ok": ok, "faster_than_composed_everywhere": bar}))
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
