"""Packed colour frames (BGR / BGRA) through the video driver, wm_process_frames in WM_VIDEO_EMBED_VERIFY mode.  Prints one JSON line.

Per workload (1080p and 4K, BGR and BGRA; every frame gated, a frame set larger than the 126 MB of L2):
  device arms (frames and output in device memory), frames/s of embed + detect:
    driver       : wm_process_frames, run size counted on the packed bytes of a frame (the default rule)
    driver_gray  : wm_process_frames with WM_OPT_RUN_MB lowered so that a run holds as many frames as a count of packed + f32 gray bytes
                   per frame (4 B/px more) would give: the other run-size rule
    loop         : the same runs written by hand: wm_embed_batch + wm_detect_batch per run (the driver's run sizes), slots in rotation
    y_driver     : the driver on Y planes of the same size (1 B/px), for scale
  end to end (pinned host frames, linesize = row bytes + 64): the driver with host frames; frames/s and GB/s of frame bytes each way.
Arms of a workload alternate in one process; each gets at least --seconds of timed work.  The driver returns after all its slots'
work has completed, so one call is bracketed by CUDA events recorded before and after it (the same for the loop, which ends in wm_sync).
After the timed region a parity gate compares frame 0 of every packed arm with the CPU oracle (a and corr within 1e-3 relative, colour
bytes within 1 LSB, the fourth byte exact), and checks that the driver's output and scalars equal the hand-written loop's.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import packed_rgb_bench as rb  # noqa: E402  (gpu_info, color_images, oracle_ref; puts the repository and tests/ on sys.path)
import util  # noqa: E402

wmb = rb.wmb
PSNR = rb.PSNR
NSLOTS = 8
RUN_MB = 136  # the driver's default WM_OPT_RUN_MB


def frames_of(rows, cols, n, bpp):
    """(n, rows, cols, bpp) BGR(A) frames: the colour images of packed_rgb_bench with B and R swapped, seeded alpha"""
    rgb = rb.color_images(rows, cols, n)
    out = np.empty((n, rows, cols, bpp), np.uint8)
    out[..., :3] = rgb[..., ::-1]
    if bpp == 4:
        out[..., 3] = np.random.default_rng(77).integers(0, 256, (n, rows, cols), dtype=np.uint8)
    return out


def run_sizes(n, B):
    """the driver's even runs of at most B frames"""
    nruns = (n + B - 1) // B
    base, extra = n // nruns, n % nruns
    return [base + (1 if r < extra else 0) for r in range(nruns)]


def timed_call(fn, state):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    state[0] += e0.elapsed_time(e1) / 1e3
    state[1] += 1


def alternate(arms, seconds):
    for f in arms.values():  # warm-up of every shape the timed region uses
        f()
        f()
    state = {k: [0.0, 0] for k in arms}
    while any(v[0] < seconds for v in state.values()):
        for k, f in arms.items():
            if state[k][0] < seconds:
                timed_call(f, state[k])
    return state


def gate(ref, out0, in0, a, corr):
    ro, ra, rc = ref
    dpx = int(np.abs(out0[..., 2::-1].astype(int) - ro.astype(int)).max())
    g = {"a_rel": util.rel(a, ra), "corr_rel": util.rel(corr, rc), "max_px": dpx}
    g["fourth_byte_exact"] = bool(in0.shape[-1] == 3 or np.array_equal(out0[..., 3], in0[..., 3]))
    g["ok"] = bool(g["a_rel"] <= 1e-3 and g["corr_rel"] <= 1e-3 and dpx <= 1 and g["fourth_byte_exact"])
    return g


def workload(rows, cols, bpp, n, seconds, oracle):
    layout = wmb.PACKED_BGR if bpp == 3 else wmb.PACKED_BGRA
    npx = rows * cols
    fbytes, rowb = bpp * npx, bpp * cols
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    imgs = frames_of(rows, cols, n, bpp)
    x = torch.from_numpy(imgs).cuda()
    o = torch.empty_like(x)
    y = x[..., 1].contiguous()  # Y-plane frames of the same size (the green byte)
    yo = torch.empty_like(y)
    torch.cuda.synchronize()
    s = np.zeros(2 * n, np.float32)
    a_loop, c_loop = np.zeros(n, np.float32), np.zeros(n, np.float32)
    B = min(32, (RUN_MB << 20) // fbytes)
    B_gray = min(32, (RUN_MB << 20) // (fbytes + 4 * npx))
    mb_gray = -(-B_gray * fbytes // (1 << 20))  # the smallest WM_OPT_RUN_MB that gives runs of B_gray frames with the packed-bytes rule
    assert min(32, (mb_gray << 20) // fbytes) == B_gray
    v = wmb.VideoProcessingContext(wm, rows, cols, 1, frames_on_device=True, layout=layout)
    vy = wmb.VideoProcessingContext(wm, rows, cols, 1, frames_on_device=True)
    desc = lambda p: wmb.image_desc(p, rows, cols, layout, wmb.U8, 0, bpp)
    sizes = run_sizes(n, B)

    def driver(mb):
        def f():
            wm.set_option(wmb.OPT_RUN_MB, mb)
            wmb.process_frames(v, wmb.VIDEO_EMBED_VERIFY, x.data_ptr(), o.data_ptr(), 0, n, s)
        return f

    def loop():
        g = 0
        for r, nb in enumerate(sizes):
            slot = r % NSLOTS
            pi, po = x.data_ptr() + g * fbytes, o.data_ptr() + g * fbytes
            wm.embed_batch(slot, desc(pi), desc(pi), desc(po), 0, 0, 0, nb, wmb.ME, a_loop[g:g + nb])
            wm.detect_batch(slot, desc(po), 0, nb, wmb.ME, c_loop[g:g + nb])
            g += nb
        wm.sync(-1)

    def y_driver():
        wm.set_option(wmb.OPT_RUN_MB, RUN_MB)
        wmb.process_frames(vy, wmb.VIDEO_EMBED_VERIFY, y.data_ptr(), yo.data_ptr(), 0, n, s)

    arms = {"driver": driver(RUN_MB), "driver_gray": driver(mb_gray), "loop": loop, "y_driver": y_driver}
    state = alternate(arms, seconds)
    dev = {k: {"frames_per_s": round(n * r / t, 1), "us_per_frame": round(t / (n * r) * 1e6, 2), "reps": r} for k, (t, r) in state.items()}
    dev["driver"]["frames_per_run"] = B
    dev["driver_gray"].update({"frames_per_run": B_gray, "run_mb": mb_gray})
    dev["loop"]["frames_per_run"] = B
    dev["y_driver"]["frames_per_run"] = min(32, (RUN_MB << 20) // npx)
    dev["driver_over_loop"] = round(dev["driver"]["frames_per_s"] / dev["loop"]["frames_per_s"], 3)
    dev["driver_gray_over_driver"] = round(dev["driver_gray"]["frames_per_s"] / dev["driver"]["frames_per_s"], 3)
    # parity, after the timed region
    ref = rb.oracle_ref(oracle, np.ascontiguousarray(imgs[0, ..., 2::-1]), W, wmb.ME)
    loop()
    lo = o.cpu().numpy()
    dev["loop"]["gate"] = gate(ref, lo[0], imgs[0], float(a_loop[0]), float(c_loop[0]))
    for k in ("driver", "driver_gray"):
        o.zero_()
        arms[k]()
        do = o.cpu().numpy()
        dev[k]["gate"] = gate(ref, do[0], imgs[0], float(s[0]), float(s[n]))
        dev[k]["equals_loop"] = bool(np.array_equal(do, lo) and np.array_equal(s[:n].view(np.uint32), a_loop.view(np.uint32)) and
                                     float(np.max(np.abs(s[n:].astype(np.float64) - c_loop) / np.abs(c_loop))) <= 1e-6)
        dev[k]["gate"]["ok"] = dev[k]["gate"]["ok"] and dev[k]["equals_loop"]
    del x, o, y, yo
    torch.cuda.empty_cache()

    # end to end: pinned host frames with 64 bytes of row padding
    ls = rowb + 64
    hin = torch.zeros((n, rows, ls), dtype=torch.uint8).pin_memory()
    hin[:, :, :rowb] = torch.from_numpy(imgs.reshape(n, rows, rowb))
    hout = torch.empty((n, rows, rowb), dtype=torch.uint8).pin_memory()
    vh = wmb.VideoProcessingContext(wm, rows, cols, 1, linesize=ls, layout=layout)
    wm.set_option(wmb.OPT_RUN_MB, RUN_MB)

    def host():
        wmb.process_frames(vh, wmb.VIDEO_EMBED_VERIFY, hin.data_ptr(), hout.data_ptr(), 0, n, s)

    host()
    t0, reps = time.perf_counter(), 0
    while time.perf_counter() - t0 < seconds:
        host()  # synchronous: every copy and kernel of the call is complete when it returns
        reps += 1
    fps = n * reps / (time.perf_counter() - t0)
    e2e = {"frames_per_s": round(fps, 1), "linesize": ls, "bytes_up_per_frame": rows * ls, "bytes_down_per_frame": fbytes,
           "gb_s_up": round(fps * rows * ls / 1e9, 2), "gb_s_down": round(fps * fbytes / 1e9, 2), "reps": reps,
           "frames_per_run": 4}  # the default WM_OPT_HOST_RUN_FRAMES
    e2e["gate"] = gate(ref, hout[0].numpy().reshape(rows, cols, bpp), imgs[0], float(s[0]), float(s[n]))
    wm.close()
    return {"rows": rows, "cols": cols, "layout": "BGR" if bpp == 3 else "BGRA", "frames": n, "frame_set_mb": round(n * fbytes / 2**20, 1),
            "device": dev, "end_to_end": e2e}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--seconds", type=float, default=1.0, help="timed work per arm (at least)")
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    if not torch.cuda.is_available() or wmb.device_count() < 1:
        sys.exit("packed_video_bench: no CUDA device (this measurement has no CPU fallback)")
    from oracle import oracle
    oracle.lib()
    name, power = rb.gpu_info()
    if args.quick:
        cases = [(540, 960, 3, 12), (540, 960, 4, 12)]
    else:
        cases = [(1080, 1920, 3, 64), (1080, 1920, 4, 64), (2160, 3840, 3, 16), (2160, 3840, 4, 16)]
    res = [workload(r, c, bpp, n, args.seconds, oracle) for r, c, bpp, n in cases]
    ok = all(w["end_to_end"]["gate"]["ok"] and all(v["gate"]["ok"] for k, v in w["device"].items() if isinstance(v, dict) and "gate" in v)
             for w in res)
    print(json.dumps({"tool": "packed_video_bench", "gpu": name, "power_limit": power, "mask": "ME", "mode": "EMBED_VERIFY", "interval": 1,
                      "workloads": res, "parity_ok": ok}))
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
