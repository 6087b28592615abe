"""ComParE_2016 full LLD set (BASELINE configs[3]) on the GPU: the shipped configuration file runs unchanged
through the C ABI (session layer) and is compared with the UNMODIFIED reference's LLD output
(tests/golden/pitch_goldens.npz, scripts/make_golden_pitch.py)."""
import os

import numpy as np
import pytest

from opensmile_b200.synth import mixed_pcm, voiced_pcm

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
G = np.load(os.path.join(HERE, "golden", "pitch_goldens.npz"))
CONF = os.path.join(HERE, "golden", "config", "compare16", "ComParE_2016.conf")

CASES = {
    "v32k": lambda: voiced_pcm(32000, 16000, seed=7),
    "m48k": lambda: mixed_pcm(48000, 16000, seed=2),
    "m30k": lambda: mixed_pcm(30000, 16000, seed=4),
    "m64k": lambda: mixed_pcm(64000, 16000, seed=3),
    "short_960": lambda: voiced_pcm(960, 16000, seed=7),
    "short_1600": lambda: voiced_pcm(1600, 16000, seed=7),
    "short_2400": lambda: voiced_pcm(2400, 16000, seed=7),
}


@pytest.fixture(scope="module")
def session():
    from opensmile_b200.session import Session
    s = Session(CONF, options={"lldcsvoutput": "x.csv"}, device=0)
    yield s
    s.close()


def _check(got, ref, names):
    assert got.shape == ref.shape
    # tolerance: 1e-5 of each column's largest magnitude (columns mix Hz, ratios and dB); the magnitude is taken
    # from a long utterance so that one- and two-row outputs are not judged against their own near-zero deltas
    sc = np.maximum(np.abs(ref).max(axis=0), np.abs(G["v32k_lld"]).max(axis=0)) + 1e-30
    err = np.abs(got - ref) / sc
    bad = np.argwhere(err > 1e-5)
    assert bad.size == 0, [(names[c], int(r), float(got[r, c]), float(ref[r, c])) for r, c in bad[:8]]


def test_compare16_full_lld_batch(session):
    """all cases as ONE ragged batch"""
    keys = sorted(CASES)
    pcms = [CASES[k]() for k in keys]
    off = np.cumsum([0] + [p.size for p in pcms]).astype(np.int64)
    rows, fo = session.extract_pcm(np.concatenate(pcms), off, 16000.0, 1)
    names = session.element_names(16000.0, 1)
    assert list(names) == [str(x) for x in G["names_lld"]]
    for i, k in enumerate(keys):
        _check(rows[fo[i]:fo[i + 1]], G[k + "_lld"], names)


def test_compare16_44k(session):
    """the same configuration file at 44.1 kHz: 2646-sample frames, FFT 4096 (2049-point spline), 882-sample frames, FFT 1024"""
    pcm = mixed_pcm(60000, 16000, seed=5)
    rows, _ = session.extract_pcm(pcm, np.array([0, pcm.size], np.int64), 44100.0, 1)
    ref = G["m60k_44k_lld"]
    assert rows.shape == ref.shape
    sc = np.abs(ref).max(axis=0) + 1e-30
    err = np.abs(rows - ref) / sc
    names = session.element_names(44100.0, 1)
    bad = np.argwhere(err > 1e-5)
    assert bad.size == 0, [(names[c], int(r), float(rows[r, c]), float(ref[r, c])) for r, c in bad[:8]]


def test_compare16_stereo(session):
    """two channels, mono mixdown in the wave source (every kernel that reads PCM averages the channels itself)"""
    from opensmile_b200.synth import stereo_mixed_pcm
    pcm = stereo_mixed_pcm(40000, 16000, seed=9)
    rows, _ = session.extract_pcm(pcm, np.array([0, 40000], np.int64), 16000.0, 2)
    _check(rows, G["m40k_stereo_lld"], session.element_names(16000.0, 2))


def test_compare16_single_and_repeatable(session):
    pcm = CASES["m30k"]()
    off = np.array([0, pcm.size], np.int64)
    a, _ = session.extract_pcm(pcm, off, 16000.0, 1)
    b, _ = session.extract_pcm(pcm, off, 16000.0, 1)
    assert np.array_equal(a, b)
    _check(a, G["m30k_lld"], session.element_names(16000.0, 1))


def test_pitch_variant_switches():
    """tests/configs/pitch_variants.conf (see tests/test_pitch_cpu.py::test_variant_switches) vs the reference"""
    from opensmile_b200.session import Session
    s = Session(os.path.join(HERE, "configs", "pitch_variants.conf"), options={"O": "x.htk"}, device=0)
    pcms = [mixed_pcm(48000, 16000, seed=6), mixed_pcm(40000, 16000, seed=8)]
    off = np.cumsum([0] + [p.size for p in pcms]).astype(np.int64)
    rows, fo = s.extract_pcm(np.concatenate(pcms), off, 16000.0, 1)
    names = s.element_names(16000.0, 1)
    for i, case in enumerate(("var_m48k", "var_m40k")):
        got, ref = rows[fo[i]:fo[i + 1]], G[case + "_lld"]
        assert got.shape == ref.shape
        sc = np.abs(ref).max(axis=0) + 1e-30
        bad = np.argwhere(np.abs(got - ref) / sc > 1e-5)
        assert bad.size == 0, [(names[c], int(r), float(got[r, c]), float(ref[r, c])) for r, c in bad[:8]]
    s.close()


def test_compare16_empty_and_too_short_utterances(session):
    """utterances with no 60 ms frame (0 and 500 samples) inside a batch yield no rows and leave their neighbours alone"""
    a, b = CASES["m30k"](), CASES["short_2400"]()
    pcm = np.concatenate([a, np.zeros(0, np.int16), voiced_pcm(500, 16000, seed=1), b])
    off = np.cumsum([0, a.size, 0, 500, b.size]).astype(np.int64)
    rows, fo = session.extract_pcm(pcm, off, 16000.0, 1)
    assert list(np.diff(fo)) == [G["m30k_lld"].shape[0], 0, 0, G["short_2400_lld"].shape[0]]
    names = session.element_names(16000.0, 1)
    _check(rows[fo[0]:fo[1]], G["m30k_lld"], names)
    _check(rows[fo[3]:fo[4]], G["short_2400_lld"], names)
