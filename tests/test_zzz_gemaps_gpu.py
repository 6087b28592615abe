"""The shipped GeMAPSv01a/b.conf, eGeMAPSv01a/b.conf, eGeMAPSv02.conf (BASELINE configs[2]) end to end on the GPU against the
reference's LLD files: EVERY column -- including the formant frequencies / bandwidths / amplitudes and H1-A3 that read the
order-11 LPC chain -- within 1e-5 of the column's scale on every row (north_star's bar).  The formant branch gets there
through the reference-order FFT of fft_ref_order.cuh; scripts/parity_report.py prints the per-column table."""
import json
import os

import numpy as np
import pytest

from opensmile_b200.synth import mixed_pcm

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(HERE, "golden", "config")
TOL = 1e-5


def _percol(got, ref):
    return np.abs(got - ref) / (np.abs(ref).max(axis=0) + 1e-30)


@pytest.mark.parametrize("conf,opts,key", [("gemaps/v01b/GeMAPSv01b.conf", {"lldhtkoutput": "x.htk"}, "gemaps_lld"),
                                           ("egemaps/v02/eGeMAPSv02.conf", {"lldcsvoutput": "x.csv"}, "egemaps_lld")])
def test_shipped_configuration_rows(conf, opts, key):
    from opensmile_b200.session import Session
    G = np.load(os.path.join(HERE, "golden", "formant_goldens.npz"))
    pcms = [mixed_pcm(24000, 16000, seed=3), mixed_pcm(40000, 16000, seed=5)]
    off = np.concatenate([[0], np.cumsum([len(x) for x in pcms])]).astype(np.int64)
    s = Session(os.path.join(REF, conf), options=opts, device=0)
    names = s.element_names()
    rows, fo = s.extract_pcm(np.concatenate(pcms + [np.zeros(8, np.int16)]), off, 16000.0, 1)
    s.close()
    for i, k in enumerate((key + "_m24k", key + "_m40k")):
        got, ref = rows[fo[i]:fo[i + 1]], G[k]
        assert got.shape == ref.shape
        err = _percol(got, ref)
        worst = {names[j]: float(err[:, j].max()) for j in range(len(names)) if err[:, j].max() >= TOL}
        assert not worst, worst


def test_all_shipped_gemaps_family_rows():
    """the five shipped feature-set files (v01a / v01b / v02) against the reference's LLD rows (tests/golden/gemaps_family.npz)"""
    from opensmile_b200.session import Session
    gold = json.load(open(os.path.join(HERE, "golden", "gemaps_headers.json")))
    R = np.load(os.path.join(HERE, "golden", "gemaps_family.npz"))
    pcm = mixed_pcm(24000, 16000, seed=3)
    for conf, g in gold.items():
        s = Session(os.path.join(REF, conf), options={"lldcsvoutput": "x.csv"}, device=0)
        names = s.element_names()
        rows, fo = s.extract_pcm(np.concatenate([pcm, np.zeros(8, np.int16)]), np.array([0, len(pcm)], np.int64), 16000.0, 1)
        s.close()
        ref = R[os.path.splitext(os.path.basename(conf))[0]]
        assert names == g["names"] and rows.shape == ref.shape
        err = _percol(rows, ref)
        worst = {names[j]: float(err[:, j].max()) for j in range(len(names)) if err[:, j].max() >= TOL}
        assert not worst, (conf, worst)
