"""Packed 4:2:2 frames (YUYV / UYVY) through the video driver and the image entry points.  Prints one JSON line.

Every workload is timed in three arms that alternate in one process, each for at least --seconds, bracketed by CUDA events (the driver
returns after all its slots' work has completed; the batch calls end in wm_sync):
  packed   : the 4:2:2 frames handed over as they are (WM_PACKED_YUYV / UYVY)
  y_plane  : (a) the Y-plane path on the same luma frames (u8 planes at a pitch of round_up(width, 16)): the speed the 4:2:2 path aims at
  composed : (b) what a caller writes without the 4:2:2 layouts: a torch de-interleave (frames[..., k].contiguous()), the Y-plane path,
             then a re-interleave of the result into a copy of the frames
Workloads (ME mask; frame sets larger than the 126 MB of L2):
  driver : wm_process_frames, WM_VIDEO_EMBED_VERIFY, every frame gated, frames and output on the device; 1080p and 4K, YUYV and UYVY
  images : wm_embed_batch + wm_detect_batch; 148 x 1080p and 16 x 4K, YUYV
  e2e    : wm_process_frames with pinned host frames, linesize = row bytes + 64 (Y planes: width + 64); 1080p and 4K, YUYV
After the timed region a parity gate compares frame 0 of every arm with the CPU oracle (oracle.embed_frame_u8 / detect_frame_u8 on the
luma: a and corr within 1e-3 relative, luma within 1 LSB, chroma exact) and checks, in every workload, that the packed arm's luma bytes
and `a` equal the Y-plane arm's and its correlations are within 1e-6 relative.
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


def round16(n):
    return (n + 15) // 16 * 16


def frames_of(rows, cols, n, k):
    """(n, rows, cols, 2) 4:2:2 frames: natural lumas at byte k, seeded random chroma in the other byte"""
    base = [util.natural_image(rows, cols, seed=13 * j, integer=True) for j in range(4)]
    out = np.empty((n, rows, cols, 2), np.uint8)
    for i in range(n):
        out[i, ..., k] = np.roll(base[i % 4], 5 * i, axis=1)
    out[..., 1 - k] = np.random.default_rng(77).integers(0, 256, (n, rows, cols), dtype=np.uint8)
    return out


def alternate(arms, seconds):
    for f in arms.values():  # warm-up of every shape the timed region uses
        f()
        f()
    state = {a: [0.0, 0] for a in arms}
    while any(v[0] < seconds for v in state.values()):
        for a, f in arms.items():
            if state[a][0] < seconds:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                f()
                e1.record()
                e1.synchronize()
                state[a][0] += e0.elapsed_time(e1) / 1e3
                state[a][1] += 1
    return state


def rates(state, n):
    r = {a: {"frames_per_s": round(n * reps / t, 1), "reps": reps} for a, (t, reps) in state.items()}
    r["packed_over_y_plane"] = round(r["packed"]["frames_per_s"] / r["y_plane"]["frames_per_s"], 3)
    r["packed_over_composed"] = round(r["packed"]["frames_per_s"] / r["composed"]["frames_per_s"], 3)
    return r


def oracle_ref(oracle, W, frame0, k):
    st, eo, ea = oracle.embed_frame_u8(np.ascontiguousarray(frame0[..., k]), W, PSNR, oracle.ME)
    _, ec = oracle.detect_frame_u8(eo, W, oracle.ME)
    return st, eo, ea, ec


def oracle_gate(ref, luma0, a, corr):
    st, eo, ea, ec = ref
    dpx = int(np.abs(luma0.astype(int) - eo.astype(int)).max())
    g = {"a_rel": util.rel(a, ea), "corr_rel": util.rel(corr, ec), "max_luma": dpx}
    g["ok"] = bool(st == 0 and g["a_rel"] <= 1e-3 and g["corr_rel"] <= 1e-3 and dpx <= 1)
    return g


def same_as_y(lp, ap, cp, ly, ay, cy):
    """packed arm vs Y-plane arm: luma bytes and `a` identical, correlations within 1e-6 relative"""
    cp, cy = np.asarray(cp, np.float64), np.asarray(cy, np.float64)
    return bool(np.array_equal(lp, ly) and np.array_equal(np.asarray(ap, np.float32).view(np.uint32), np.asarray(ay, np.float32).view(np.uint32))
                and np.max(np.abs(cp - cy) / np.abs(cy)) <= 1e-6)


def driver_workload(rows, cols, layout, n, seconds, oracle):
    k = 0 if layout == wmb.PACKED_YUYV else 1
    lp = round16(cols)
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    imgs = frames_of(rows, cols, n, k)
    x = torch.from_numpy(imgs).cuda()
    o = torch.empty_like(x)
    y = torch.zeros((n, rows, lp), dtype=torch.uint8, device="cuda")
    y[..., :cols] = x[..., k]
    yo = torch.empty((n, rows, cols), dtype=torch.uint8, device="cuda")
    oc = torch.empty_like(x)
    torch.cuda.synchronize()
    s, sy, sc = (np.zeros(2 * n, np.float32) for _ in range(3))
    v = wmb.VideoProcessingContext(wm, rows, cols, 1, frames_on_device=True, layout=layout)
    vy = wmb.VideoProcessingContext(wm, rows, cols, 1, linesize=lp, frames_on_device=True)
    vd = wmb.VideoProcessingContext(wm, rows, cols, 1, frames_on_device=True)  # dense Y planes of the de-interleave

    def packed():
        wmb.process_frames(v, wmb.VIDEO_EMBED_VERIFY, x.data_ptr(), o.data_ptr(), 0, n, s)

    def y_plane():
        wmb.process_frames(vy, wmb.VIDEO_EMBED_VERIFY, y.data_ptr(), yo.data_ptr(), 0, n, sy)

    def composed():
        yd = x[..., k].contiguous()
        torch.cuda.current_stream().synchronize()  # the driver's slot streams do not order after torch's stream
        wmb.process_frames(vd, wmb.VIDEO_EMBED_VERIFY, yd.data_ptr(), yo.data_ptr(), 0, n, sc)
        oc.copy_(x)
        oc[..., k] = yo

    dev = rates(alternate({"packed": packed, "y_plane": y_plane, "composed": composed}, seconds), n)
    packed()
    y_plane()
    po, yl = o.cpu().numpy(), yo.cpu().numpy()
    composed()
    co = oc.cpu().numpy()
    torch.cuda.synchronize()
    ref = oracle_ref(oracle, W, imgs[0], k)
    gates = {"packed": oracle_gate(ref, po[0, ..., k], s[0], s[n]),
             "y_plane": oracle_gate(ref, yl[0], sy[0], sy[n]),
             "composed": oracle_gate(ref, co[0, ..., k], sc[0], sc[n])}
    gates["packed"]["chroma_exact"] = bool(np.array_equal(po[..., 1 - k], imgs[..., 1 - k]))
    gates["packed"]["equals_y_plane"] = same_as_y(po[..., k], s[:n], s[n:], yl, sy[:n], sy[n:])
    gates["packed"]["ok"] = gates["packed"]["ok"] and gates["packed"]["chroma_exact"] and gates["packed"]["equals_y_plane"]
    dev["gate"] = gates
    wm.close()
    return {"workload": "driver", "rows": rows, "cols": cols, "layout": "YUYV" if k == 0 else "UYVY", "frames": n,
            "frame_set_mb": round(imgs.nbytes / 2**20, 1), **dev}


def images_workload(rows, cols, batch, seconds, oracle):
    k, layout = 0, wmb.PACKED_YUYV
    lp = round16(cols)
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    imgs = frames_of(rows, cols, batch, k)
    x = torch.from_numpy(imgs).cuda()
    o = torch.empty_like(x)
    y = torch.zeros((batch, rows, lp), dtype=torch.uint8, device="cuda")
    y[..., :cols] = x[..., k]
    yo = torch.empty_like(y)
    oc, yco = torch.empty_like(x), torch.empty((batch, rows, cols), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    res = {arm: (np.zeros(batch, np.float32), np.zeros(batch, np.float32)) for arm in ("packed", "y_plane", "composed")}
    pdesc = lambda p: wmb.image_desc(p, rows, cols, layout, wmb.U8, 0, 2)
    ydesc = lambda p, ld: wmb.image_desc(p, rows, cols, wmb.ROW_MAJOR, wmb.U8, ld, 1)

    def packed():
        a, c = res["packed"]
        wm.embed_batch(0, pdesc(x.data_ptr()), pdesc(x.data_ptr()), pdesc(o.data_ptr()), 0, 0, 0, batch, wmb.ME, a)
        wm.detect_batch(0, pdesc(o.data_ptr()), 0, batch, wmb.ME, c)
        wm.sync(0)

    def y_plane():
        a, c = res["y_plane"]
        wm.embed_batch(0, ydesc(y.data_ptr(), lp), ydesc(y.data_ptr(), lp), ydesc(yo.data_ptr(), lp), 0, 0, 0, batch, wmb.ME, a)
        wm.detect_batch(0, ydesc(yo.data_ptr(), lp), 0, batch, wmb.ME, c)
        wm.sync(0)

    def composed():
        a, c = res["composed"]
        yd = x[..., k].contiguous()
        torch.cuda.current_stream().synchronize()
        wm.embed_batch(0, ydesc(yd.data_ptr(), 0), ydesc(yd.data_ptr(), 0), ydesc(yco.data_ptr(), 0), 0, 0, 0, batch, wmb.ME, a)
        wm.detect_batch(0, ydesc(yco.data_ptr(), 0), 0, batch, wmb.ME, c)
        wm.sync(0)
        oc.copy_(x)
        oc[..., k] = yco

    r = rates(alternate({"packed": packed, "y_plane": y_plane, "composed": composed}, seconds), batch)
    for f in (packed, y_plane, composed):
        f()
    torch.cuda.synchronize()
    po, yl, co = o.cpu().numpy(), yo[..., :cols].cpu().numpy(), oc.cpu().numpy()
    ref = oracle_ref(oracle, W, imgs[0], k)
    gates = {"packed": oracle_gate(ref, po[0, ..., k], res["packed"][0][0], res["packed"][1][0]),
             "y_plane": oracle_gate(ref, yl[0], res["y_plane"][0][0], res["y_plane"][1][0]),
             "composed": oracle_gate(ref, co[0, ..., k], res["composed"][0][0], res["composed"][1][0])}
    gates["packed"]["chroma_exact"] = bool(np.array_equal(po[..., 1 - k], imgs[..., 1 - k]))
    gates["packed"]["equals_y_plane"] = same_as_y(po[..., k], res["packed"][0], res["packed"][1], yl, res["y_plane"][0], res["y_plane"][1])
    gates["packed"]["ok"] = gates["packed"]["ok"] and gates["packed"]["chroma_exact"] and gates["packed"]["equals_y_plane"]
    r["gate"] = gates
    wm.close()
    return {"workload": "images", "rows": rows, "cols": cols, "layout": "YUYV", "batch": batch, "batch_mb": round(imgs.nbytes / 2**20, 1), **r}


def e2e_workload(rows, cols, n, seconds, oracle):
    k, layout = 0, wmb.PACKED_YUYV
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    imgs = frames_of(rows, cols, n, k)
    ls, lsy = 2 * cols + 64, cols + 64
    hin = torch.zeros((n, rows, ls), dtype=torch.uint8).pin_memory()
    hin[:, :, :2 * cols] = torch.from_numpy(imgs.reshape(n, rows, 2 * cols))
    hout = torch.empty((n, rows, cols, 2), dtype=torch.uint8).pin_memory()
    hy = torch.zeros((n, rows, lsy), dtype=torch.uint8).pin_memory()
    hy[..., :cols] = torch.from_numpy(imgs[..., k])
    hyo = torch.empty((n, rows, cols), dtype=torch.uint8).pin_memory()
    hc, hco = torch.empty((n, rows, cols), dtype=torch.uint8).pin_memory(), torch.empty((n, rows, cols, 2), dtype=torch.uint8).pin_memory()
    s, sy, sc = (np.zeros(2 * n, np.float32) for _ in range(3))
    v = wmb.VideoProcessingContext(wm, rows, cols, 1, linesize=ls, layout=layout)
    vy = wmb.VideoProcessingContext(wm, rows, cols, 1, linesize=lsy)
    vd = wmb.VideoProcessingContext(wm, rows, cols, 1)
    hin4 = hin[:, :, :2 * cols].view(n, rows, cols, 2)

    def packed():
        wmb.process_frames(v, wmb.VIDEO_EMBED_VERIFY, hin.data_ptr(), hout.data_ptr(), 0, n, s)

    def y_plane():
        wmb.process_frames(vy, wmb.VIDEO_EMBED_VERIFY, hy.data_ptr(), hyo.data_ptr(), 0, n, sy)

    def composed():  # the de-interleave and re-interleave run on the host, as a caller of the host-frame driver would write them
        hc.copy_(hin4[..., k])
        wmb.process_frames(vd, wmb.VIDEO_EMBED_VERIFY, hc.data_ptr(), hyo.data_ptr(), 0, n, sc)
        hco.copy_(hin4)
        hco[..., k] = hyo

    # host-synchronous calls: timed with the host clock
    arms = {"packed": packed, "y_plane": y_plane, "composed": composed}
    for f in arms.values():
        f()
    state = {a: [0.0, 0] for a in arms}
    while any(t < seconds for t, _ in state.values()):
        for a, f in arms.items():
            if state[a][0] < seconds:
                t0 = time.perf_counter()
                f()
                state[a][0] += time.perf_counter() - t0
                state[a][1] += 1
    r = rates(state, n)
    r["packed"].update({"linesize": ls, "gb_s_up": round(r["packed"]["frames_per_s"] * rows * ls / 1e9, 2),
                        "gb_s_down": round(r["packed"]["frames_per_s"] * rows * 2 * cols / 1e9, 2)})
    packed()
    po = hout.numpy().copy()
    y_plane()
    yl = hyo.numpy().copy()
    composed()
    co = hco.numpy().copy()
    ref = oracle_ref(oracle, W, imgs[0], k)
    gates = {"packed": oracle_gate(ref, po[0, ..., k], s[0], s[n]),
             "y_plane": oracle_gate(ref, yl[0], sy[0], sy[n]),
             "composed": oracle_gate(ref, co[0, ..., k], sc[0], sc[n])}
    gates["packed"]["chroma_exact"] = bool(np.array_equal(po[..., 1 - k], imgs[..., 1 - k]))
    gates["packed"]["equals_y_plane"] = same_as_y(po[..., k], s[:n], s[n:], yl, sy[:n], sy[n:])
    gates["packed"]["ok"] = gates["packed"]["ok"] and gates["packed"]["chroma_exact"] and gates["packed"]["equals_y_plane"]
    r["gate"] = gates
    wm.close()
    return {"workload": "e2e", "rows": rows, "cols": cols, "layout": "YUYV", "frames": n, **r}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--seconds", type=float, default=1.0, help="timed work per arm (at least)")
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    if not torch.cuda.is_available() or wmb.device_count() < 1:
        sys.exit("packed_yuv422_bench: no CUDA device (this measurement has no CPU fallback)")
    from oracle import oracle
    oracle.lib()
    name, power = rb.gpu_info()
    Y, U = wmb.PACKED_YUYV, wmb.PACKED_UYVY
    if args.quick:
        res = [driver_workload(270, 480, Y, 8, args.seconds, oracle), images_workload(270, 480, 8, args.seconds, oracle),
               e2e_workload(270, 480, 8, args.seconds, oracle)]
    else:
        res = [driver_workload(1080, 1920, Y, 64, args.seconds, oracle), driver_workload(1080, 1920, U, 64, args.seconds, oracle),
               driver_workload(2160, 3840, Y, 16, args.seconds, oracle), driver_workload(2160, 3840, U, 16, args.seconds, oracle),
               images_workload(1080, 1920, 148, args.seconds, oracle), images_workload(2160, 3840, 16, args.seconds, oracle),
               e2e_workload(1080, 1920, 64, args.seconds, oracle), e2e_workload(2160, 3840, 16, args.seconds, oracle)]
    ok = all(g["ok"] for w in res for g in w["gate"].values())
    bar = all(w["packed_over_composed"] > 1.0 for w in res)
    print(json.dumps({"tool": "packed_yuv422_bench", "gpu": name, "power_limit": power, "mask": "ME", "mode": "EMBED_VERIFY", "interval": 1,
                      "workloads": res, "parity_ok": ok, "faster_than_composed_everywhere": bar}))
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
