"""Regenerates tests/golden/ref_kernels.json: what the reference's three OpenCL kernels (nvf, scaled_neighbors_p3, me)
compute on the inputs of tests/test_oracle_vs_reference_kernels.py, so that the test pins the C restatement
(oracle/wm_oracle.c) without the reference's source tree.

  python tests/golden/make_ref_kernels_golden.py                      # from oracle/_ref (make -C oracle REF=<reference checkout>)
  python tests/golden/make_ref_kernels_golden.py --from-restatement   # from oracle/wm_oracle.c

Image outputs are stored as the SHA-256 of their float32 bytes (row-major, little-endian) plus a seeded sample of 32
values for diagnostics; the 8x8 Rx and 8-vector rx in full.  --from-restatement is only valid for a restatement that
has passed the pin against the reference's kernel text and not changed since.  The stored file was made that way:
oracle/ is unchanged since commit bcf514d, and the pin passed against oracle/_ref built from the reference after it.
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import util  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_kernels.json")
SHAPES = [(64, 64), (48, 80), (67, 131), (130, 70), (512, 512)]
WIDE = [(64, 64), (67, 131), (130, 70)]
COEF = np.array([-0.21, 0.47, -0.18, 0.49, 0.52, -0.2, 0.45, -0.24], np.float32)
NSAMPLE = 32


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a, "<f4").tobytes()).hexdigest()


def image_record(a):
    idx = np.sort(np.random.default_rng(a.size).choice(a.size, NSAMPLE, replace=False))
    return {"shape": list(a.shape), "sha256": sha256(a), "index": idx.tolist(), "values": [float(v) for v in a.ravel()[idx]]}


def image(oracle, rows, cols, seed, integer=False):
    if rows == 512 and not integer:
        return util.load_512_gray(oracle)
    img = util.natural_image(rows, cols, seed=seed, integer=integer)
    return img.astype(np.float32)


class FromReference:
    """the reference's own kernel text, compiled for the CPU under oracle/clshim"""
    source = "the reference's kernel text under oracle/clshim (oracle/_ref)"

    def __init__(self):
        from oracle import ref_kernels
        if not ref_kernels.available():
            raise SystemExit("oracle/_ref is not built: run `make -C oracle REF=<reference checkout>` first")
        self.r = ref_kernels

    def nvf(self, img, p):
        return self.r.nvf(img, fma=False, p=p)

    def scaled_neighbors(self, img, fma):
        return self.r.scaled_neighbors(img, COEF, fma=fma)

    def rx(self, img):
        Rx, rx = self.r.rx(img, fma=False)
        Rx2, rx2 = self.r.rx(img, fma=True)  # products are stored to fp16 before any add: contraction cannot change them
        assert np.array_equal(Rx, Rx2) and np.array_equal(rx, rx2)
        return Rx, rx


class FromRestatement:
    source = ("oracle/wm_oracle.c (contraction off for nvf and the unfused scaled_neighbors, on for the fused one; FAITHFUL for "
              "Rx / rx), unchanged since its pin last passed bit for bit against the reference's kernel text")

    def __init__(self, oracle):
        self.o = oracle

    def nvf(self, img, p):
        return self.o.nvf(img, self.o.opts(contract=0, p=p))

    def scaled_neighbors(self, img, fma):
        return self.o.scaled_neighbors(img, COEF, self.o.opts(contract=int(fma)))

    def rx(self, img):
        return self.o.rx(img, self.o.FAITHFUL)


def main():
    from oracle import oracle
    oracle.lib()
    ref = FromRestatement(oracle) if "--from-restatement" in sys.argv else FromReference()
    cases = {}
    for rows, cols in SHAPES:
        cases["nvf/%dx%d/p3" % (rows, cols)] = image_record(ref.nvf(image(oracle, rows, cols, 1), 3))
    for rows, cols in WIDE:
        for p in (5, 7, 9):
            cases["nvf/%dx%d/p%d" % (rows, cols, p)] = image_record(ref.nvf(image(oracle, rows, cols, 10 + p), p))
    for rows, cols in SHAPES:
        img = image(oracle, rows, cols, 2)
        for fma in (False, True):
            cases["scaled_neighbors/%dx%d/%s" % (rows, cols, "fma" if fma else "nofma")] = image_record(ref.scaled_neighbors(img, fma))
    for rows, cols in SHAPES:
        for kind, img in (("natural", image(oracle, rows, cols, 3)), ("integer", image(oracle, rows, cols, 4, integer=True))):
            Rx, rx = ref.rx(img)
            cases["me/%dx%d/%s" % (rows, cols, kind)] = {"Rx": np.asarray(Rx, np.float64).ravel().tolist(),
                                                         "rx": np.asarray(rx, np.float64).tolist()}
    with open(OUT, "w") as f:
        json.dump({"source": ref.source, "coef": [float(c) for c in COEF], "cases": cases}, f, indent=0)
        f.write("\n")
    print("wrote %s: %d cases from %s" % (OUT, len(cases), ref.source))


if __name__ == "__main__":
    main()
