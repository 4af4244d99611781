"""CPU-only: pin the CFAR oracle (oracle/cfar_ref.c) against the reference.

 * against tests/golden/cfar_reference.npz, what the UNMODIFIED reference cfar.cpp
   (oracle/_ref/libcfar_ref.so) returned on the inputs below (tools/make_golden.py);
 * against tests/golden/cfar_masks.npz, produced by running the reference's own CFAR class
   (tools/make_golden.py).
"""
import hashlib

import numpy as np
import pytest

from oracle import oracle as orc
from sonar_slam_b200 import synth

TAU = {"CA": 2.3701490070915554, "SOCA": 2.749063720096473, "GOCA": 2.121926842646487, "OS": 9.137608674642355}
ALGS = ["CA", "SOCA", "GOCA", "OS"]


def _inputs():
    rng = np.random.default_rng(7)
    yield "u8frame", synth.make_frame(3).astype(np.float32), 20, 5, 10
    yield "fractional", (rng.rayleigh(18.0, (96, 40)) + rng.random((96, 40))).astype(np.float32), 20, 5, 7
    yield "small_window", rng.integers(0, 255, (64, 33)).astype(np.float32), 4, 2, 3
    yield "too_short", rng.random((30, 8)).astype(np.float32), 20, 5, 0
    yield "negative_and_big", (rng.normal(0, 1e6, (80, 17))).astype(np.float32), 6, 1, 11


def _sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.mark.parametrize("alg", ALGS)
def test_port_equals_unmodified_reference(alg, golden_dir):
    g = np.load(f"{golden_dir}/cfar_reference.npz")
    for name, img, T, G, k in _inputs():
        assert _sha256(img) == str(g[name + "_input_sha256"]), name  # the inputs the fixture was made from
        for i, tau in enumerate((TAU[alg], 0.37)):
            key = f"{name}_{alg}_{i}"
            m1, t1 = orc.cfar(alg, img, T, G, k, tau, want_thr=True)
            assert np.array_equal(np.packbits(np.ascontiguousarray(m1)), g[key + "_mask"]), key
            t1 = np.ascontiguousarray(t1)
            assert np.array_equal(t1[::7, ::5].view(np.uint32), g[key + "_thr_sample"].view(np.uint32)), key
            assert _sha256(t1) == str(g[key + "_thr_sha256"]), key  # bit-exact thresholds
            m2, _ = orc.cfar(alg, img, T, G, k, tau, want_thr=False)
            assert np.array_equal(m1, m2), key


@pytest.mark.parametrize("alg", ALGS)
def test_port_equals_golden_masks(alg, golden_dir):
    g = np.load(f"{golden_dir}/cfar_masks.npz")
    img = synth.make_frame(seed=1)
    m, thr = orc.cfar(alg, img, 20, 5, 10, TAU[alg], want_thr=True)
    assert m.flags["F_CONTIGUOUS"] and m.dtype == np.uint8
    assert int(m.sum()) == int(g[alg + "_count"])
    assert np.array_equal(np.packbits(np.ascontiguousarray(m)), g[alg])
    thr_c = np.ascontiguousarray(thr)
    assert hashlib.sha256(thr_c.tobytes()).hexdigest() == str(g[alg + "_thr_sha256"])
    assert np.array_equal(thr_c[::37, ::41], g[alg + "_thr_sample"])


def test_u8_entry_equals_float_entry_plus_gate():
    img = synth.make_frame(5)
    for alg in ALGS:
        m, _ = orc.cfar(alg, img, 20, 5, 10, TAU[alg])
        want = np.ascontiguousarray(m) & (img > 65)
        assert np.array_equal(orc.cfar_u8(alg, img, 20, 5, 10, TAU[alg], 65), want)
        assert np.array_equal(orc.cfar_u8(alg, img, 20, 5, 10, TAU[alg], -1), np.ascontiguousarray(m))
