"""Packed 8-bit RGBA images (WM_PACKED_RGBA) against splitting off the alpha byte, the way a caller handles them without it.  Prints one JSON line.

Device-resident arms, per image of a batch (148 x 1080p, 16 x 4K: both more than the 126 MB of L2 as packed u8):
  rgba  : wm_embed_batch on the packed RGBA batch (alpha copied through), wm_detect_batch on the RGBA output
  split : torch copies the RGB bytes into a packed RGB buffer, the packed RGB path runs (embed + detect), then torch writes the RGB
          result and the input's alpha back into a 4-byte output buffer
  rgb   : the packed RGB path alone on the same pixels without alpha (what the fourth byte costs)
  for the ME and the NVF mask (embed + detect of that mask).  Every arm runs on slot 0's stream; CUDA events bracket each repetition,
  arms alternate in the same process, each is timed for at least --seconds.
End to end at 1080p (pinned host memory): wm_embed_verify_host_batch on RGBA host images (4 B/px up, 4 B/px down), alternated with the
same on RGB host images (3 B/px each way).
A parity gate compares image 0 of every arm with the CPU oracle after the timed region (tools/packed_rgb_bench.py: a and corr within 1e-3
relative, colour bytes within 1 LSB) and requires the output's alpha to equal the input's, byte for byte.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import packed_rgb_bench as rb  # noqa: E402  (gpu_info, timed, gate, color_images; puts the repository and tests/ on sys.path)
import util  # noqa: E402

wmb = rb.wmb
PSNR = rb.PSNR


def alphas(rows, cols, n):
    a = np.random.default_rng(77).integers(0, 256, (rows, cols), dtype=np.uint8)
    a[0, 0], a[-1, -1] = 0, 255
    return np.stack([np.roll(a, 3 * b, axis=0) for b in range(n)])


def gate4(oracle, img4, W, mask, out4, a, corr):
    g = rb.gate(oracle, img4[..., :3], W, mask, out4[..., :3], a, corr)
    g["alpha_exact"] = bool(np.array_equal(out4[..., 3], img4[..., 3]))
    g["ok"] = g["ok"] and g["alpha_exact"]
    return g


def run_arms(arms, st, seconds, batch):
    for f in arms.values():  # warm-up of every shape the timed region uses
        f()
        f()
    state = {k: [0.0, 0] for k in arms}
    done = set()
    while len(done) < len(arms):  # arms alternate until each has `seconds` of timed work
        for k, f in arms.items():
            if k not in done and rb.timed(st, f, seconds, state[k]):
                done.add(k)
    return {k: {"images_per_s": round(batch * v[1] / v[0], 1), "us_per_image": round(v[0] / (batch * v[1]) * 1e6, 2), "reps": v[1]}
            for k, v in state.items()}


def device_case(rows, cols, batch, seconds, oracle):
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    st = torch.cuda.ExternalStream(wm.stream(0))
    rgb = rb.color_images(rows, cols, batch)
    imgs = np.concatenate([rgb, alphas(rows, cols, batch)[..., None]], -1)
    with torch.cuda.stream(st):
        x4 = torch.from_numpy(imgs).cuda()                   # (B, rows, cols, 4) u8, packed RGBA
        o4 = torch.empty_like(x4)
        x3 = torch.from_numpy(np.ascontiguousarray(rgb)).cuda()  # the same pixels without alpha
        s3 = torch.empty_like(x3)                            # split arm's RGB scratch
        o3 = torch.empty_like(x3)
        st.synchronize()
    a = np.zeros(batch, np.float32)
    c = np.zeros(batch, np.float32)
    d4 = lambda t: wmb.image_desc(t.data_ptr(), rows, cols, wmb.PACKED_RGBA, wmb.U8, 0, 4)
    d3 = lambda t: wmb.image_desc(t.data_ptr(), rows, cols, wmb.PACKED_RGB, wmb.U8, 0, 3)

    def rgba_arm(mask):
        wm.embed_batch(0, d4(x4), d4(x4), d4(o4), 0, 0, 0, batch, mask, a)
        wm.detect_batch(0, d4(o4), 0, batch, mask, c)
        wm.sync(0)

    def split_arm(mask):
        with torch.cuda.stream(st):
            s3.copy_(x4[..., :3])
            wm.embed_batch(0, d3(s3), d3(s3), d3(o3), 0, 0, 0, batch, mask, a)
            wm.detect_batch(0, d3(o3), 0, batch, mask, c)
            o4[..., :3].copy_(o3)
            o4[..., 3].copy_(x4[..., 3])
            wm.sync(0)

    def rgb_arm(mask):
        wm.embed_batch(0, d3(x3), d3(x3), d3(o3), 0, 0, 0, batch, mask, a)
        wm.detect_batch(0, d3(o3), 0, batch, mask, c)
        wm.sync(0)

    fns = {"rgba": rgba_arm, "split": split_arm, "rgb": rgb_arm}
    arms = {"%s_%s" % (m, k): (lambda f=f, mask=mask: f(mask)) for m, mask in (("me", wmb.ME), ("nvf", wmb.NVF)) for k, f in fns.items()}
    res = run_arms(arms, st, seconds, batch)
    for m, mask in (("me", wmb.ME), ("nvf", wmb.NVF)):
        res["%s_rgba_over_split" % m] = round(res["%s_rgba" % m]["images_per_s"] / res["%s_split" % m]["images_per_s"], 2)
        res["%s_rgba_over_rgb" % m] = round(res["%s_rgba" % m]["images_per_s"] / res["%s_rgb" % m]["images_per_s"], 2)
        for k, f in fns.items():
            f(mask)
            if k == "rgb":
                g = rb.gate(oracle, rgb[0], W, mask, o3[0].cpu().numpy(), float(a[0]), float(c[0]))
            else:
                g = gate4(oracle, imgs[0], W, mask, o4[0].cpu().numpy(), float(a[0]), float(c[0]))
            res["%s_%s" % (m, k)]["gate"] = g
    wm.close()
    return {"rows": rows, "cols": cols, "batch": batch, "rgba_mb_per_batch": round(imgs.nbytes / 2**20, 1), "arms": res}


def e2e_case(rows, cols, batch, chunk, seconds, oracle):
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    rgb = rb.color_images(rows, cols, batch)
    imgs = np.concatenate([rgb, alphas(rows, cols, batch)[..., None]], -1)
    npx = rows * cols
    h4, h3 = torch.from_numpy(imgs).pin_memory(), torch.from_numpy(np.ascontiguousarray(rgb)).pin_memory()
    o4, o3 = torch.empty_like(h4).pin_memory(), torch.empty_like(h3).pin_memory()
    a = np.zeros(batch, np.float32)
    c = np.zeros(batch, np.float32)
    NS = wm.num_slots

    def arm(hin, hout, layout, n):
        def run(mask):
            for k, o in enumerate(range(0, batch, chunk)):
                nb = min(chunk, batch - o)
                d_in = wmb.image_desc(hin[o].data_ptr(), rows, cols, layout, wmb.U8, 0, n)
                d_out = wmb.image_desc(hout[o].data_ptr(), rows, cols, layout, wmb.U8, 0, n)
                wm.embed_verify_host_batch(k % NS, d_in, d_in, d_out, 0, 0, 0, nb, mask, a[o:o + nb], c[o:o + nb])
            wm.sync(-1)
        return run

    arms = {"rgba": arm(h4, o4, wmb.PACKED_RGBA, 4), "rgb": arm(h3, o3, wmb.PACKED_RGB, 3)}
    for f in arms.values():
        f(wmb.ME)
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
    res = {}
    for k, (tot, reps) in state.items():
        ips = batch * reps / tot
        bpp = 4 if k == "rgba" else 3  # bytes per pixel up, and the same down
        res[k] = {"images_per_s": round(ips, 1), "bytes_up_per_image": bpp * npx, "bytes_down_per_image": bpp * npx,
                  "gb_s_up": round(ips * bpp * npx / 1e9, 2), "gb_s_down": round(ips * bpp * npx / 1e9, 2), "reps": reps}
    arms["rgba"](wmb.ME)
    res["rgba"]["gate"] = gate4(oracle, imgs[0], W, wmb.ME, o4[0].numpy(), float(a[0]), float(c[0]))
    arms["rgb"](wmb.ME)
    res["rgb"]["gate"] = rb.gate(oracle, rgb[0], W, wmb.ME, o3[0].numpy(), float(a[0]), float(c[0]))
    wm.close()
    return {"rows": rows, "cols": cols, "batch": batch, "images_per_call": chunk, "mask": "ME", "arms": res}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--seconds", type=float, default=1.0, help="timed work per arm (at least)")
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    if not torch.cuda.is_available() or wmb.device_count() < 1:
        sys.exit("packed_rgba_bench: no CUDA device (this measurement has no CPU fallback)")
    from oracle import oracle
    oracle.lib()
    name, power = rb.gpu_info()
    if args.quick:
        dev = [device_case(270, 480, 8, args.seconds, oracle)]
        e2e = e2e_case(270, 480, 16, 4, args.seconds, oracle)
    else:
        dev = [device_case(1080, 1920, 148, args.seconds, oracle), device_case(2160, 3840, 16, args.seconds, oracle)]
        e2e = e2e_case(1080, 1920, 48, 4, args.seconds, oracle)
    ok = all(v["gate"]["ok"] for d in dev for v in d["arms"].values() if isinstance(v, dict)) and \
        all(v["gate"]["ok"] for v in e2e["arms"].values())
    print(json.dumps({"tool": "packed_rgba_bench", "gpu": name, "power_limit": power, "device": dev, "end_to_end": e2e, "parity_ok": ok}))
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
