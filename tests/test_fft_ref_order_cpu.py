"""opensmile_b200/csrc/fft_ref_order.cuh (the 512-point real FFT of the formant branch, reference rounding order) compiled for
the host (tests/native/fft_ref_order_host.cpp) against the reference's own transform (its rdft's outputs and work table in
tests/golden/reference_fft512.npz, scripts/make_golden_reference_runs.py).  Bit-for-bit equality is the bar -- this transform
exists because order-11 LPC amplifies 2e-7 of spectral noise into 1e-2 of the formants (DESIGN.md 3.6)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


@pytest.fixture(scope="module")
def libs():
    so = "/tmp/osm_ro_host_%d.so" % os.getuid()
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-I/usr/local/cuda/include", "-o", so,
                           os.path.join(HERE, "native", "fft_ref_order_host.cpp"), os.path.join(ROOT, "opensmile_b200", "csrc", "tables.cpp")])
    return C.CDLL(so)


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(HERE, "golden", "reference_fft512.npz"))


def fft_cases():
    rng = np.random.default_rng(5)
    cases = [rng.standard_normal(512).astype(np.float32) * s for s in (1.0, 1e-3, 3e4) for _ in range(40)]
    imp = np.zeros(512, np.float32); imp[3] = 1.0
    n = np.arange(320)
    frame = np.zeros(512, np.float32)                                  # a windowed, zero padded frame like the kernel's input
    frame[96:416] = (np.sin(0.07 * n) * np.exp(-0.5 * ((n - 159.5) / 64.0) ** 2)).astype(np.float32)
    cases += [imp, np.ones(512, np.float32), frame, np.zeros(512, np.float32)]
    return cases


def test_twiddle_tables_equal_the_reference(libs, ref):
    wc = np.zeros(256, np.float32)
    libs.roh_tables(_fp(wc))
    assert np.array_equal(wc, ref["w"][:256])


def test_transform_is_bit_identical(libs, ref):
    cases = fft_cases()
    out = np.zeros(512, np.float32)
    assert len(ref["case_index"]) == 28
    for i, r in zip(ref["case_index"], ref["rdft"]):
        x = cases[i]
        for scramble in (0, 1):                                        # order of the work items inside a phase is free
            libs.roh_rdft512(_fp(x), _fp(out), scramble)
            assert np.array_equal(out.view(np.uint32), r.view(np.uint32))
