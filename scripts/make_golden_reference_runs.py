"""Generate tests/golden/reference_rows.npz and tests/golden/reference_fft512.npz with the UNMODIFIED reference
(oracle/_ref/SMILExtract and oracle/_ref/libfftsg.so, built by `make -C oracle ref`):
    python scripts/make_golden_reference_runs.py

reference_rows.npz     the reference's LLD rows for the seeded inputs of tests/test_oracle_cpu.py
  mfcc_<sr>_<n>_<seed>[_<nch>ch]   config/mfcc/MFCC12_0_D_A.conf on voiced_pcm(n, sr, seed=seed, n_chan=nch) [T, 39]
  plp_<sr>_<n>_<seed>_<nch>ch      config/plp/PLP_0_D_A.conf on the same kind of input [T, 18]
  crc_<key>                        sum of the input samples (detects a drift of the synthetic generator)
reference_fft512.npz   the reference's rdft(512) for the inputs of tests/test_fft_ref_order_cpu.py
  w            the work table rdft leaves behind (twiddle factors w[0:256], then the cosine table)
  case_index   which of the test's inputs are stored: 8 of the 40 random vectors at each of the three scales and the four
               structured ones (a full copy of the 120 random outputs would be 250 KB of incompressible floats)
  rdft         the reference's packed output for each stored input [len(case_index), 512]
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import refrun  # noqa: E402
from opensmile_b200.synth import voiced_pcm  # noqa: E402
from test_fft_ref_order_cpu import fft_cases  # noqa: E402
from test_oracle_cpu import MFCC_CASES, PLP_CASES, mfcc_key, plp_key  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def reference_rows():
    out = {}
    for sr, n, seed, nch in MFCC_CASES:
        pcm = voiced_pcm(n, sr, seed=seed, n_chan=nch)
        k = mfcc_key(sr, n, seed, nch)
        out[k] = refrun.extract("mfcc/MFCC12_0_D_A.conf", pcm, sr, n_chan=nch)
        out["crc_" + k] = np.int64(pcm.astype(np.int64).sum())
    for sr, n, seed, nch in PLP_CASES:
        pcm = voiced_pcm(n, sr, seed=seed, n_chan=nch)
        k = plp_key(sr, n, seed, nch)
        out[k] = refrun.extract("plp/PLP_0_D_A.conf", pcm, sr, n_chan=nch)
        out["crc_" + k] = np.int64(pcm.astype(np.int64).sum())
    np.savez_compressed(os.path.join(GOLD, "reference_rows.npz"), **out)


def reference_fft512():
    F = C.CDLL(os.path.join(refrun.REF_DIR, "libfftsg.so"))

    def rdft(x):
        ip = np.zeros(64, np.int32)
        w = np.zeros(512, np.float32)
        a = x.copy()
        F.rdft(512, 1, a.ctypes.data_as(C.POINTER(C.c_float)), ip.ctypes.data_as(C.POINTER(C.c_int)), w.ctypes.data_as(C.POINTER(C.c_float)))
        return a, w

    cases = fft_cases()
    idx = [s * 40 + i for s in range(3) for i in range(8)] + list(range(120, len(cases)))
    np.savez_compressed(os.path.join(GOLD, "reference_fft512.npz"), w=rdft(np.zeros(512, np.float32))[1],
                        case_index=np.array(idx, np.int64), rdft=np.stack([rdft(cases[i])[0] for i in idx]))


if __name__ == "__main__":
    assert refrun.available() and os.path.exists(os.path.join(refrun.REF_DIR, "libfftsg.so")), "build the reference first: make -C oracle ref"
    reference_rows()
    reference_fft512()
