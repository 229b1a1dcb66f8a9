"""10-bit luma frames (WM_Y10: yuv420p10le Y planes) through the video driver, against what a caller composes today.  Prints one JSON line.

Workloads (ME mask, wm_process_frames in WM_VIDEO_EMBED_VERIFY with every frame gated; frame sets larger than the 126 MB of L2):
  driver : frames and output on the device, 1080p x 64 and 4K x 16, in three arms that alternate in one process, each for at least
           --seconds per run, two runs, bracketed by CUDA events (every arm returns after its work has completed):
    y10      : (a) the Y10 frames handed over as they are
    composed : (b) what a caller writes without WM_Y10: torch (w & 1023) * 0.25 into f32 planes, wm_embed_batch (f32, base = in), torch
               quantise to words (clamp(4 y, 0, 1023)), torch * 0.25 of the result, wm_detect_batch; the torch work runs on the library's
               slot stream, so nothing waits between the steps
    y8       : (c) the 8-bit Y-plane driver on u8 frames of the same size, for context
  e2e    : pinned host frames with 64 bytes of row padding (linesize = 2 * width + 64; Y planes: width + 64), y10 and y8 arms, host clock
After the timed region frame 0 of every arm is checked against the CPU oracle on x = v / 4 (8-bit arm: on its u8 frame): a and the
correlation within 1e-3 relative, words within one code.
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

wmb = rb.wmb
PSNR = rb.PSNR


def samples(rows, cols, n):
    """(n, rows, cols) uint16 10-bit samples with natural statistics; bits 10-15 seeded random (ignored by WM_Y10)"""
    rng = np.random.default_rng(7)
    base = [np.clip(np.rint(util.natural_image(rows, cols, seed=13 * j) * 4.0 + rng.integers(-2, 3, (rows, cols))), 0, 1023) for j in range(4)]
    v = np.stack([np.roll(base[i % 4], 5 * i, axis=1) for i in range(n)]).astype(np.uint16)
    return v, v | (rng.integers(0, 64, v.shape, dtype=np.uint16) << 10)


def timed_runs(arms, seconds, runs=2, host_clock=False):
    """every arm alternately for at least `seconds` per run -> {arm: [seconds per call of run 1, run 2, ...]}"""
    for f in arms.values():  # warm-up of every shape the timed region uses
        f()
        f()
    out = {a: [] for a in arms}
    for _ in range(runs):
        state = {a: [0.0, 0] for a in arms}
        while any(v[0] < seconds for v in state.values()):
            for a, f in arms.items():
                if state[a][0] >= seconds:
                    continue
                if host_clock:
                    t0 = time.perf_counter()
                    f()
                    state[a][0] += time.perf_counter() - t0
                else:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    f()
                    e1.record()
                    e1.synchronize()
                    state[a][0] += e0.elapsed_time(e1) / 1e3
                state[a][1] += 1
        for a, (t, reps) in state.items():
            out[a].append(t / reps)
    return out


def rates(per_call, n):
    r = {}
    for a, ts in per_call.items():
        fps = [n / t for t in ts]
        r[a] = {"frames_per_s": [round(x, 1) for x in fps], "spread_pct": round(100.0 * (max(fps) - min(fps)) / min(fps), 2)}
    if "composed" in r:
        r["y10_over_composed"] = round(min(r["y10"]["frames_per_s"]) / max(r["composed"]["frames_per_s"]), 3)
    r["y10_over_y8"] = round(np.mean(r["y10"]["frames_per_s"]) / np.mean(r["y8"]["frames_per_s"]), 3)
    return r


def gate10(oracle, W, v0, words0, a, corr, shift=0):
    x = v0.astype(np.float32) * np.float32(0.25)
    e = oracle.embed(x, W, PSNR, oracle.ME)
    ref = np.clip(4.0 * e["out"].astype(np.float64), 0, 1023).astype(np.int64)
    got = (words0.astype(np.int64) >> shift) & 1023
    d = oracle.detect(got.astype(np.float32) * np.float32(0.25), W, oracle.ME)
    g = {"a_rel": util.rel(a, e["a"]), "corr_rel": util.rel(corr, d["corr"]), "max_code_diff": int(np.abs(got - ref).max())}
    g["ok"] = bool(e["status"] == 0 and g["a_rel"] <= 1e-3 and g["corr_rel"] <= 1e-3 and g["max_code_diff"] <= 1)
    return g


def gate8(oracle, W, y0, out0, a, corr):
    st, eo, ea = oracle.embed_frame_u8(y0, W, PSNR, oracle.ME)
    _, ec = oracle.detect_frame_u8(eo, W, oracle.ME)
    g = {"a_rel": util.rel(a, ea), "corr_rel": util.rel(corr, ec), "max_code_diff": int(np.abs(out0.astype(int) - eo.astype(int)).max())}
    g["ok"] = bool(st == 0 and g["a_rel"] <= 1e-3 and g["corr_rel"] <= 1e-3 and g["max_code_diff"] <= 1)
    return g


def driver_workload(rows, cols, n, seconds, oracle):
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    v, w = samples(rows, cols, n)
    y8 = (v >> 2).astype(np.uint8)
    dw = torch.from_numpy(w.view(np.int16)).cuda()  # the words, as int16 (torch's bitwise ops on int16 read the same bits)
    dwo = torch.empty_like(dw)
    d8, d8o = torch.from_numpy(y8).cuda(), torch.empty((n, rows, cols), dtype=torch.uint8, device="cuda")
    x = torch.empty((n, rows, cols), dtype=torch.float32, device="cuda")
    y, xq = torch.empty_like(x), torch.empty_like(x)
    q = torch.empty_like(dw)
    torch.cuda.synchronize()
    s10, s8 = np.zeros(2 * n, np.float32), np.zeros(2 * n, np.float32)
    ac, sc, cc, scc = np.zeros(n, np.float32), np.zeros(n, np.int32), np.zeros(n, np.float32), np.zeros(n, np.int32)
    v10 = wmb.VideoProcessingContext(wm, rows, cols, 1, frames_on_device=True, layout=wmb.Y10)
    v8 = wmb.VideoProcessingContext(wm, rows, cols, 1, frames_on_device=True)
    slot = torch.cuda.ExternalStream(wm.stream(0))
    desc = lambda t: wmb.image_desc(t.data_ptr(), rows, cols, wmb.ROW_MAJOR, wmb.F32, 0, 1)

    def y10():
        wmb.process_frames(v10, wmb.VIDEO_EMBED_VERIFY, dw.data_ptr(), dwo.data_ptr(), 0, n, s10)

    def composed():
        with torch.cuda.stream(slot):
            torch.mul(torch.bitwise_and(dw, 1023), 0.25, out=x)
            wm.embed_batch(0, desc(x), desc(x), desc(y), 0, 0, 0, n, wmb.ME, ac, sc)
            q.copy_(torch.clamp(y * 4.0, 0, 1023))  # float -> int16 truncates
            torch.mul(q, 0.25, out=xq)
            wm.detect_batch(0, desc(xq), 0, n, wmb.ME, cc, scc)
        wm.sync(0)

    def eight():
        wmb.process_frames(v8, wmb.VIDEO_EMBED_VERIFY, d8.data_ptr(), d8o.data_ptr(), 0, n, s8)

    r = rates(timed_runs({"y10": y10, "composed": composed, "y8": eight}, seconds), n)
    y10()
    composed()
    eight()
    torch.cuda.synchronize()
    o10, oc, o8 = dwo[0].cpu().numpy().view(np.uint16), q[0].cpu().numpy().view(np.uint16), d8o[0].cpu().numpy()
    r["gate"] = {"y10": gate10(oracle, W, v[0], o10, s10[0], s10[n]), "composed": gate10(oracle, W, v[0], oc, ac[0], cc[0]),
                 "y8": gate8(oracle, W, y8[0], o8, s8[0], s8[n])}
    r["y10_vs_composed_max_code_diff"] = int(np.abs(dwo.cpu().numpy().astype(np.int64) - q.cpu().numpy().astype(np.int64)).max())
    wm.close()
    return {"workload": "driver", "rows": rows, "cols": cols, "frames": n, "frame_set_mb": round(w.nbytes / 2**20, 1), **r}


def e2e_workload(rows, cols, n, seconds, oracle):
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    v, w = samples(rows, cols, n)
    y8 = (v >> 2).astype(np.uint8)
    ls, ls8 = 2 * cols + 64, cols + 64
    hin = torch.zeros((n, rows, ls), dtype=torch.uint8).pin_memory()
    hin[:, :, :2 * cols] = torch.from_numpy(w.view(np.uint8).reshape(n, rows, 2 * cols))
    hout = torch.empty((n, rows, 2 * cols), dtype=torch.uint8).pin_memory()
    h8 = torch.zeros((n, rows, ls8), dtype=torch.uint8).pin_memory()
    h8[:, :, :cols] = torch.from_numpy(y8)
    h8o = torch.empty((n, rows, cols), dtype=torch.uint8).pin_memory()
    s10, s8 = np.zeros(2 * n, np.float32), np.zeros(2 * n, np.float32)
    v10 = wmb.VideoProcessingContext(wm, rows, cols, 1, linesize=ls, layout=wmb.Y10)
    v8 = wmb.VideoProcessingContext(wm, rows, cols, 1, linesize=ls8)

    def y10():
        wmb.process_frames(v10, wmb.VIDEO_EMBED_VERIFY, hin.data_ptr(), hout.data_ptr(), 0, n, s10)

    def eight():
        wmb.process_frames(v8, wmb.VIDEO_EMBED_VERIFY, h8.data_ptr(), h8o.data_ptr(), 0, n, s8)

    r = rates(timed_runs({"y10": y10, "y8": eight}, seconds, host_clock=True), n)
    r["y10"]["linesize"] = ls
    y10()
    eight()
    r["gate"] = {"y10": gate10(oracle, W, v[0], hout[0].numpy().view(np.uint16), s10[0], s10[n]),
                 "y8": gate8(oracle, W, y8[0], h8o[0].numpy(), s8[0], s8[n])}
    wm.close()
    return {"workload": "e2e", "rows": rows, "cols": cols, "frames": n, **r}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--seconds", type=float, default=1.0, help="timed work per arm and run (at least)")
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    if not torch.cuda.is_available() or wmb.device_count() < 1:
        sys.exit("y10_bench: no CUDA device (this measurement has no CPU fallback)")
    from oracle import oracle
    oracle.lib()
    name, power = rb.gpu_info()
    if args.quick:
        res = [driver_workload(270, 480, 8, args.seconds, oracle), e2e_workload(270, 480, 8, args.seconds, oracle)]
    else:
        res = [driver_workload(1080, 1920, 64, args.seconds, oracle), driver_workload(2160, 3840, 16, args.seconds, oracle),
               e2e_workload(1080, 1920, 64, args.seconds, oracle), e2e_workload(2160, 3840, 16, args.seconds, oracle)]
    ok = all(g["ok"] for w in res for g in w["gate"].values())
    bar = all(w["y10_over_composed"] > 1.0 for w in res if "y10_over_composed" in w)
    print(json.dumps({"tool": "y10_bench", "gpu": name, "power_limit": power, "mask": "ME", "mode": "EMBED_VERIFY", "interval": 1,
                      "workloads": res, "parity_ok": ok, "faster_than_composed_everywhere": bar}))
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
