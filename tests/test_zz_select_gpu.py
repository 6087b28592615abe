"""tests/configs/gemaps_sel.conf (cDataSelector over the pitch and jitter / shimmer levels of the reference's shipped GeMAPS
graph + the shipped selector gemapsv01b_lldsetE) on the GPU against the reference's CSV rows.  The selector only regroups
columns of kernels the other GPU tests cover."""
import os

import numpy as np
import pytest

from opensmile_b200.synth import mixed_pcm, voiced_pcm

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REFCONF = os.path.join(HERE, "golden", "config")


def test_selector_configuration_rows(tmp_path):
    from opensmile_b200.session import Session
    G = np.load(os.path.join(HERE, "golden", "select_goldens.npz"))
    conf = tmp_path / "gsel.conf"
    conf.write_text(open(os.path.join(HERE, "configs", "gemaps_sel.conf")).read().replace("REFCONF", REFCONF))
    pcms = [mixed_pcm(24000, 16000, seed=3), voiced_pcm(32000, 16000, seed=7)]
    off = np.concatenate([[0], np.cumsum([len(x) for x in pcms])]).astype(np.int64)
    s = Session(str(conf), device=0)
    rows, fo = s.extract_pcm(np.concatenate(pcms + [np.zeros(8, np.int16)]), off, 16000.0, 1)
    s.close()
    for i, key in enumerate(("gsel_m24k", "gsel_v32k")):
        got, ref = rows[fo[i]:fo[i + 1]], G[key]
        assert got.shape == ref.shape
        assert (np.abs(got - ref) / (np.abs(ref).max(axis=0) + 1e-30)).max() < 1e-5
