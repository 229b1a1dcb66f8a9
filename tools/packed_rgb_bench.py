"""Packed 8-bit RGB images (WM_PACKED_RGB) against the composed planar path a caller has without them.  Prints one JSON line.

Device-resident arms, per image of a batch (148 x 1080p, 16 x 4K: both more than the 126 MB of L2 as packed u8):
  packed   : wm_embed_batch on the packed batch (gray computed on load, packed u8 out), wm_detect_batch on the packed output
  composed : torch de-interleave + widen to planar f32, wm_rgb2gray per image, wm_embed_batch with the 3-plane f32 base and u8 planar
             out, torch re-interleave, then widen + wm_rgb2gray + wm_detect_batch for the detection
  for the ME and the NVF mask (embed + detect of that mask).  Every arm runs on slot 0's stream; CUDA events bracket each repetition,
  arms alternate in the same process, each is timed for at least --seconds.
End to end through the host-buffer entry points (pinned memory, 1080p):
  packed : wm_embed_verify_host_batch on packed u8 host images (3 B/px up, 3 B/px down)
  planar : wm_embed_host_batch (gray f32 + 3-plane f32 base up, 3-plane u8 down) + wm_detect_host_batch on the gray f32 of the output
           (the host-side gray of the output is prepared outside the timed region, which favours this arm)
A parity gate compares image 0 of every arm with the CPU oracle (oracle.rgb2gray -> oracle.embed(base=rgb) -> truncate ->
oracle.rgb2gray -> oracle.detect) after the timed region: a and corr within 1e-3 relative, pixels within 1 LSB.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import util  # noqa: E402

wmb = importlib.import_module("watermarking-gpu_b200")
PSNR = 40.0


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001
        return torch.cuda.get_device_name(0), "unknown (%s)" % e


def color_images(rows, cols, n):
    base = []
    for k in range(4):
        base.append(np.stack([util.natural_image(rows, cols, seed=31 * k + c, integer=True) for c in range(3)], -1))
    return np.stack([np.roll(base[b % 4], 5 * b, axis=1) for b in range(n)])


def oracle_ref(oracle, img, W, mask):
    rgb = np.ascontiguousarray(img.transpose(2, 0, 1)).astype(np.float32)
    e = oracle.embed(oracle.rgb2gray(rgb), W, PSNR, mask, base=rgb)
    trunc = e["out"].astype(np.uint8)
    corr = oracle.detect(oracle.rgb2gray(trunc.astype(np.float32)), W, mask)["corr"]
    return np.ascontiguousarray(trunc.transpose(1, 2, 0)), e["a"], corr


def gate(oracle, img, W, mask, out, a, corr):
    ro, ra, rc = oracle_ref(oracle, img, W, mask)
    dpx = int(np.abs(out.astype(int) - ro.astype(int)).max())
    rel_a, rel_c = util.rel(a, ra), util.rel(corr, rc)
    return {"a_rel": rel_a, "corr_rel": rel_c, "max_px": dpx, "ok": bool(rel_a <= 1e-3 and rel_c <= 1e-3 and dpx <= 1)}


def timed(stream, fn, seconds, state):
    """one repetition bracketed by CUDA events on `stream`; accumulates into state = [total_s, reps]"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    fn()
    e1.record(stream)
    e1.synchronize()
    state[0] += e0.elapsed_time(e1) / 1e3
    state[1] += 1
    return state[0] >= seconds


def device_case(rows, cols, batch, seconds, oracle):
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    st = torch.cuda.ExternalStream(wm.stream(0))
    imgs = color_images(rows, cols, batch)
    npx = rows * cols
    with torch.cuda.stream(st):
        x = torch.from_numpy(imgs).cuda()                              # (B, rows, cols, 3) u8, packed
        pout = torch.empty_like(x)
        planar = torch.empty((batch, 3, rows, cols), dtype=torch.float32, device="cuda")
        gray = torch.empty((batch, rows, cols), dtype=torch.float32, device="cuda")
        uout = torch.empty((batch, 3, rows, cols), dtype=torch.uint8, device="cuda")
        st.synchronize()
    a = np.zeros(batch, np.float32)
    c = np.zeros(batch, np.float32)
    pk = lambda t: wmb.image_desc(t.data_ptr(), rows, cols, wmb.PACKED_RGB, wmb.U8, 0, 3)
    g1 = lambda t, b: wmb.image_desc(t[b].data_ptr(), rows, cols, wmb.ROW_MAJOR, wmb.F32, 0, 1)
    p3 = lambda t, dt, b=0: wmb.image_desc(t[b].data_ptr(), rows, cols, wmb.ROW_MAJOR, dt, 0, 3, npx)

    def rgb2gray_all():
        for b in range(batch):
            d_in, d_out = p3(planar, wmb.F32, b), g1(gray, b)
            wm._check(wmb.lib().wm_rgb2gray(wm._h, wmb.C.byref(d_in), wmb.C.byref(d_out), 0.299, 0.587, 0.114))

    def packed_arm(mask):
        wm.embed_batch(0, pk(x), pk(x), pk(pout), 0, 0, 0, batch, mask, a)
        wm.detect_batch(0, pk(pout), 0, batch, mask, c)
        wm.sync(0)

    def composed_arm(mask):
        with torch.cuda.stream(st):
            planar.copy_(x.permute(0, 3, 1, 2))
            rgb2gray_all()
            wm.embed_batch(0, g1(gray, 0), p3(planar, wmb.F32), p3(uout, wmb.U8), npx, 3 * npx, 3 * npx, batch, mask, a)
            pout.copy_(uout.permute(0, 2, 3, 1))
            planar.copy_(pout.permute(0, 3, 1, 2))
            rgb2gray_all()
            wm.detect_batch(0, g1(gray, 0), npx, batch, mask, c)
            wm.sync(0)

    arms = {}
    for mname, mask in (("me", wmb.ME), ("nvf", wmb.NVF)):
        for aname, fn in (("packed", packed_arm), ("composed", composed_arm)):
            arms["%s_%s" % (mname, aname)] = (lambda f=fn, m=mask: f(m))
    for f in arms.values():  # warm-up of every shape the timed region uses
        f()
        f()
    state = {k: [0.0, 0] for k in arms}
    done = set()
    while len(done) < len(arms):  # arms alternate until each has `seconds` of timed work
        for k, f in arms.items():
            if k not in done and timed(st, f, seconds, state[k]):
                done.add(k)
    res = {k: {"images_per_s": round(batch * v[1] / v[0], 1), "us_per_image": round(v[0] / (batch * v[1]) * 1e6, 2), "reps": v[1]}
           for k, v in state.items()}
    for mname, mask in (("me", wmb.ME), ("nvf", wmb.NVF)):
        res["%s_speedup" % mname] = round(res["%s_packed" % mname]["images_per_s"] / res["%s_composed" % mname]["images_per_s"], 2)
        for aname, fn in (("packed", packed_arm), ("composed", composed_arm)):
            fn(mask)
            res["%s_%s" % (mname, aname)]["gate"] = gate(oracle, imgs[0], W, mask, pout[0].cpu().numpy(), float(a[0]), float(c[0]))
    wm.close()
    return {"rows": rows, "cols": cols, "batch": batch, "packed_mb_per_batch": round(imgs.nbytes / 2**20, 1), "arms": res}


def e2e_case(rows, cols, batch, chunk, seconds, oracle):
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    imgs = color_images(rows, cols, batch)
    npx = rows * cols
    h_in = torch.from_numpy(imgs).pin_memory()
    h_out = torch.empty_like(h_in).pin_memory()
    rgb = torch.from_numpy(imgs).permute(0, 3, 1, 2).float().contiguous().pin_memory()
    gray = torch.from_numpy(np.stack([util_gray(rgb[b].numpy()) for b in range(batch)])).pin_memory()
    u_out = torch.empty((batch, 3, rows, cols), dtype=torch.uint8).pin_memory()
    gray_out = gray.clone().pin_memory()  # stands in for the gray of the output, prepared outside the timed region
    a = np.zeros(batch, np.float32)
    c = np.zeros(batch, np.float32)
    NS = wm.num_slots

    def packed_arm(mask):
        for k, o in enumerate(range(0, batch, chunk)):
            nb = min(chunk, batch - o)
            d_in = wmb.image_desc(h_in[o].data_ptr(), rows, cols, wmb.PACKED_RGB, wmb.U8, 0, 3)
            d_out = wmb.image_desc(h_out[o].data_ptr(), rows, cols, wmb.PACKED_RGB, wmb.U8, 0, 3)
            wm.embed_verify_host_batch(k % NS, d_in, d_in, d_out, 0, 0, 0, nb, mask, a[o:o + nb], c[o:o + nb])
        wm.sync(-1)

    def planar_arm(mask):
        for k, o in enumerate(range(0, batch, chunk)):
            nb = min(chunk, batch - o)
            d_in = wmb.image_desc(gray[o].data_ptr(), rows, cols, wmb.ROW_MAJOR, wmb.F32, 0, 1)
            d_base = wmb.image_desc(rgb[o].data_ptr(), rows, cols, wmb.ROW_MAJOR, wmb.F32, 0, 3, npx)
            d_out = wmb.image_desc(u_out[o].data_ptr(), rows, cols, wmb.ROW_MAJOR, wmb.U8, 0, 3, npx)
            d_g = wmb.image_desc(gray_out[o].data_ptr(), rows, cols, wmb.ROW_MAJOR, wmb.F32, 0, 1)
            wm.embed_host_batch(k % NS, d_in, d_base, d_out, npx, 3 * npx, 3 * npx, nb, mask, a[o:o + nb])
            wm.detect_host_batch(k % NS, d_g, npx, nb, mask, c[o:o + nb])
        wm.sync(-1)

    arms = {"packed": packed_arm, "planar": planar_arm}
    for f in arms.values():
        f(wmb.ME)
    import time
    state = {k: [0.0, 0] for k in arms}
    done = set()
    while len(done) < len(arms):
        for k, f in arms.items():
            if k in done:
                continue
            t = time.perf_counter()
            f(wmb.ME)  # ends in wm_sync: every copy and kernel of the pass is complete
            state[k][0] += time.perf_counter() - t
            state[k][1] += 1
            if state[k][0] >= seconds:
                done.add(k)
    bytes_px = {"packed": (3, 3), "planar": (4 + 12 + 4, 3)}  # (up, down) per pixel
    res = {}
    for k, (tot, reps) in state.items():
        ips = batch * reps / tot
        up, down = bytes_px[k]
        res[k] = {"images_per_s": round(ips, 1), "bytes_up_per_image": up * npx, "bytes_down_per_image": down * npx,
                  "gb_s_up": round(ips * up * npx / 1e9, 2), "gb_s_down": round(ips * down * npx / 1e9, 2), "reps": reps}
    res["speedup"] = round(res["packed"]["images_per_s"] / res["planar"]["images_per_s"], 2)
    packed_arm(wmb.ME)
    res["packed"]["gate"] = gate(oracle, imgs[0], W, wmb.ME, h_out[0].numpy(), float(a[0]), float(c[0]))
    wm.close()
    return {"rows": rows, "cols": cols, "batch": batch, "images_per_call": chunk, "mask": "ME", "arms": res}


def util_gray(rgb):
    return ((np.float32(0.299) * rgb[0] + np.float32(0.587) * rgb[1]) + np.float32(0.114) * rgb[2]).astype(np.float32)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--seconds", type=float, default=1.0, help="timed work per arm (at least)")
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    if not torch.cuda.is_available() or wmb.device_count() < 1:
        sys.exit("packed_rgb_bench: no CUDA device (this measurement has no CPU fallback)")
    from oracle import oracle
    oracle.lib()
    name, power = gpu_info()
    if args.quick:
        dev = [device_case(270, 480, 8, args.seconds, oracle)]
        e2e = e2e_case(270, 480, 16, 4, args.seconds, oracle)
    else:
        dev = [device_case(1080, 1920, 148, args.seconds, oracle), device_case(2160, 3840, 16, args.seconds, oracle)]
        e2e = e2e_case(1080, 1920, 48, 4, args.seconds, oracle)
    ok = all(v["gate"]["ok"] for d in dev for k, v in d["arms"].items() if isinstance(v, dict)) and e2e["arms"]["packed"]["gate"]["ok"]
    print(json.dumps({"tool": "packed_rgb_bench", "gpu": name, "power_limit": power, "device": dev, "end_to_end": e2e, "parity_ok": ok}))
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
