"""Pins the C restatement (oracle/wm_oracle.c) against what the reference's own kernel source computes
(tests/golden/ref_kernels.json, made by tests/golden/make_ref_kernels_golden.py from that source run on the CPU under
oracle/clshim).  The reference ships no golden vectors (SURVEY.md §4), so this is the pin for the three OpenCL kernels;
the ArrayFire calls between them stay a restatement of documented semantics."""
import hashlib
import json
import os

import numpy as np
import pytest

import util

SHAPES = [(64, 64), (48, 80), (67, 131), (130, 70), (512, 512)]
REF = json.load(open(os.path.join(util.GOLDEN, "ref_kernels.json")))["cases"]


def assert_ref_image(got, key):
    """bit for bit: the stored sample first (it shows where a difference is), then the digest of the whole image"""
    want = REF[key]
    assert list(got.shape) == want["shape"]
    sample = np.ascontiguousarray(got, np.float32).ravel()[want["index"]]
    assert np.array_equal(sample, np.array(want["values"], np.float32)), (key, sample, want["values"])
    assert hashlib.sha256(np.ascontiguousarray(got, "<f4").tobytes()).hexdigest() == want["sha256"], key


def ref_rx(key):
    want = REF[key]
    return np.array(want["Rx"], np.float64).reshape(8, 8), np.array(want["rx"], np.float64)


@pytest.mark.parametrize("rows,cols", SHAPES)
def test_nvf_kernel(oracle, rows, cols):
    img = util.natural_image(rows, cols, seed=1) if rows != 512 else util.load_512_gray(oracle)
    unfused = oracle.nvf(img, oracle.opts(contract=0))
    assert_ref_image(unfused, "nvf/%dx%d/p3" % (rows, cols))
    # with contraction allowed (-cl-mad-enable, main.cpp:106) WHICH mul+add pairs fuse is the compiler's choice, and
    # the naive variance amplifies it (SURVEY.md H2: 8.6e-3 max abs between contraction choices): the fused restatement
    # is bounded against the reference's unfused output (`unfused` equals it), not equal to it
    assert np.abs(oracle.nvf(img, oracle.opts(contract=1)) - unfused).max() <= 1e-2


@pytest.mark.parametrize("p", [5, 7, 9])
@pytest.mark.parametrize("rows,cols", [(64, 64), (67, 131), (130, 70)])
def test_nvf_kernel_larger_windows(oracle, rows, cols, p):
    """The class accepts p in {3, 5, 7, 9} (Watermark.cpp:24); the nvf kernel is generic in p (kernels/nvf.hpp:14-17)."""
    img = util.natural_image(rows, cols, seed=10 + p)
    unfused = oracle.nvf(img, oracle.opts(contract=0, p=p))
    assert_ref_image(unfused, "nvf/%dx%d/p%d" % (rows, cols, p))
    assert np.abs(oracle.nvf(img, oracle.opts(contract=1, p=p)) - unfused).max() <= 2e-2


@pytest.mark.parametrize("rows,cols", SHAPES)
def test_scaled_neighbors_kernel(oracle, rows, cols):
    img = util.natural_image(rows, cols, seed=2) if rows != 512 else util.load_512_gray(oracle)
    coef = np.array([-0.21, 0.47, -0.18, 0.49, 0.52, -0.2, 0.45, -0.24], np.float32)
    assert_ref_image(oracle.scaled_neighbors(img, coef, oracle.opts(contract=0)), "scaled_neighbors/%dx%d/nofma" % (rows, cols))
    assert_ref_image(oracle.scaled_neighbors(img, coef, oracle.opts(contract=1)), "scaled_neighbors/%dx%d/fma" % (rows, cols))


@pytest.mark.parametrize("rows,cols", SHAPES)
def test_me_kernel(oracle, rows, cols):
    """fp16-rounded products, 64-wide sequential f32 group sums, padded columns contributing 0 (the same Rx / rx with
    and without contraction: products are stored to fp16 before any add)."""
    img = util.natural_image(rows, cols, seed=3) if rows != 512 else util.load_512_gray(oracle)
    Rx, rx = oracle.rx(img, oracle.FAITHFUL)
    rRx, rrx = ref_rx("me/%dx%d/natural" % (rows, cols))
    assert np.array_equal(Rx, rRx)
    assert np.array_equal(rx, rrx)
    # integer-valued frames
    y = util.natural_image(rows, cols, seed=4, integer=True).astype(np.float32)
    Rx, rx = oracle.rx(y, oracle.FAITHFUL)
    rRx, rrx = ref_rx("me/%dx%d/integer" % (rows, cols))
    assert np.array_equal(Rx, rRx) and np.array_equal(rx, rrx)
    assert np.array_equal(Rx, Rx.T)
