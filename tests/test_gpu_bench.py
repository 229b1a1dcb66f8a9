"""bench.py --dump-outputs on the GPU: what it writes is what the timed path computed, checked against the CPU oracle on the
benchmark's own synthetic frames."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import util

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs_match_oracle(oracle, tmp_path):
    import torch
    import bench
    rows, cols, nfr = 512, 512, 2  # 2 column-major frames: fewer pixels than the sample, so every pixel is written, in logical order
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "image512", "--frames", str(nfr), "--calls", "1",
                        "--steps", "2", "--warmup", "0", "--no-cpu-baseline", "--no-e2e", "--no-sync-proto", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == 2
    names = sorted(os.listdir(tmp_path))
    assert names == sorted("image512_%s_%s.npy" % (m, k) for m in ("nvf", "me") for k in ("a", "corr", "out_sample"))
    got = {n[len("image512_"):-len(".npy")]: np.load(tmp_path / n) for n in names}
    assert all(a.dtype == np.float32 for a in got.values())
    assert got["me_a"][0] == np.float32(line["results"]["a_me"]) and got["nvf_corr"][0] == np.float32(line["results"]["corr_nvf"])
    # the benchmark's frames, regenerated the way it makes them (column-major: generated from the transposed base)
    dev = torch.device("cuda", 0)
    base_t = torch.from_numpy(np.ascontiguousarray(util.natural_image(rows, cols, seed=1).T)).to(dev)
    frames = [f.cpu().numpy().T for f in bench.device_frames(torch, dev, base_t, 0, nfr, "f32")]
    W = util.normal_w(rows, cols, seed=28390211)
    for name, mask in (("nvf", oracle.NVF), ("me", oracle.ME)):
        out = got[name + "_out_sample"].reshape(nfr, rows, cols)
        for i in range(nfr):
            o = oracle.embed(frames[i], W, 40.0, mask)
            od = oracle.detect(o["out"], W, mask)
            assert abs(got[name + "_a"][i] - o["a"]) / o["a"] <= 1e-3
            assert abs(got[name + "_corr"][i] - od["corr"]) / abs(od["corr"]) <= 1e-3
            assert np.abs(out[i] - o["out"]).max() <= 1e-4 * 255
