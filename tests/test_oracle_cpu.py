"""CPU tests: the oracle (plain-C restatement) against the golden vectors produced by the
unmodified reference."""
import os

import numpy as np
import pytest

from conftest import GOLD, rel_to_frame_scale
from opensmile_b200.synth import voiced_pcm
from oracle import oracle

TOL = 1e-5   # of the per-frame vector scale (north_star: 1e-5 relative, float32)
# (sample rate, samples, seed, channels) of the inputs whose reference rows tests/golden/reference_rows.npz holds
# (scripts/make_golden_reference_runs.py)
MFCC_CASES = [(16000, 40000, 3, 1), (44100, 30000, 4, 1), (16000, 400, 5, 1), (16000, 561, 6, 1), (16000, 20000, 7, 2)]
PLP_CASES = [(16000, 30000, 11, 1), (44100, 20000, 12, 2), (16000, 560, 13, 1)]


def mfcc_key(sr, n, seed, nch):
    return "mfcc_%d_%d_%d" % (sr, n, seed) + ("_%dch" % nch if nch > 1 else "")


def plp_key(sr, n, seed, nch):
    return "plp_%d_%d_%d_%dch" % (sr, n, seed, nch)


def reference_rows(key, pcm):
    """the unmodified reference's rows for `pcm`, stored under `key`"""
    g = np.load(os.path.join(GOLD, "reference_rows.npz"))
    assert int(pcm.astype(np.int64).sum()) == int(g["crc_" + key]), "synthetic generator drifted"
    return g[key]


def test_geometry_known_answers():
    # SURVEY.md 8(a'): frame-count known answers measured on the reference
    fe, _, _ = oracle.mfcc12_0_d_a(16000.0)
    assert oracle.geometry(fe, 80000) == (400, 160, 512, 498)
    assert oracle.geometry(fe, 9600000)[3] == 59998
    fe, _, _ = oracle.mfcc12_0_d_a(44100.0)
    assert oracle.geometry(fe, 90112) == (1103, 441, 2048, 202)
    assert oracle.geometry(fe, 1102)[3] == 0
    assert oracle.geometry(fe, 1103)[3] == 1


def test_oracle_vs_golden_example_wav():
    g = np.load(os.path.join(GOLD, "mfcc_example_44k1.npz"))
    out = oracle.mfcc_d_a(g["pcm"], float(g["sample_rate"]))
    assert out.shape == g["lld"].shape == (202, 39)
    assert rel_to_frame_scale(out, g["lld"]) < TOL


def test_oracle_vs_golden_synth16k():
    g = np.load(os.path.join(GOLD, "mfcc_synth16k_s0.npz"))
    pcm = voiced_pcm(80000, 16000, seed=0)
    assert int(pcm.astype(np.int64).sum()) == int(g["crc"]), "synthetic generator drifted"
    out = oracle.mfcc_d_a(pcm, 16000.0)
    assert out.shape == g["lld"].shape == (498, 39)
    assert rel_to_frame_scale(out, g["lld"]) < TOL


def test_oracle_taps_vs_golden():
    g = np.load(os.path.join(GOLD, "mfcc_taps16k_s1.npz"))
    pcm = voiced_pcm(16000, 16000, seed=1)
    out, mag, mel = oracle.mfcc_d_a(pcm, 16000.0, taps=True)
    assert mag.shape[0] == int(g["n_frames"])
    n = g["fftmag"].shape[0]
    assert rel_to_frame_scale(mag[:n], g["fftmag"]) < 2e-6
    assert rel_to_frame_scale(mel[:n], g["melspec"]) < 2e-6
    assert rel_to_frame_scale(out[:n, :13], g["ft0"]) < TOL


def test_delta_is_bit_exact_on_reference_statics():
    # the regression stages are float arithmetic in a fixed order: given the reference's own
    # static features the oracle must reproduce delta / delta-delta bit for bit, including
    # the phantom frames at the end (SURVEY.md H3)
    for name in ("mfcc_example_44k1.npz", "mfcc_synth16k_s0.npz"):
        lld = np.load(os.path.join(GOLD, name))["lld"]
        T = lld.shape[0]
        d = oracle.delta(lld[:, :13], 2)
        dd = oracle.delta(d, 2)
        assert d.shape[0] == T + 2 and dd.shape[0] == T + 4
        assert np.array_equal(d[:T], lld[:, 13:26])
        assert np.array_equal(dd[:T], lld[:, 26:39])


@pytest.mark.parametrize("sr,n,seed", [(16000, 40000, 3), (44100, 30000, 4), (16000, 400, 5), (16000, 561, 6)])
def test_oracle_vs_live_reference(sr, n, seed):
    pcm = voiced_pcm(n, sr, seed=seed)
    ref = reference_rows(mfcc_key(sr, n, seed, 1), pcm)
    out = oracle.mfcc_d_a(pcm, float(sr))
    assert out.shape == ref.shape
    assert rel_to_frame_scale(out, ref) < TOL


def test_oracle_vs_live_reference_stereo():
    pcm = voiced_pcm(20000, 16000, seed=7, n_chan=2)
    ref = reference_rows(mfcc_key(16000, 20000, 7, 2), pcm)
    out = oracle.mfcc_d_a(pcm, 16000.0, n_chan=2)
    assert out.shape == ref.shape
    assert rel_to_frame_scale(out, ref) < TOL


def test_plp_oracle_vs_golden():
    g = np.load(os.path.join(GOLD, "plp_goldens.npz"))
    ex = np.load(os.path.join(GOLD, "mfcc_example_44k1.npz"))
    out = oracle.plp_d_a(ex["pcm"], float(ex["sample_rate"]))
    assert out.shape == g["example_lld"].shape == (202, 18)
    assert rel_to_frame_scale(out, g["example_lld"]) < TOL
    pcm2 = voiced_pcm(44100, 44100, seed=2, n_chan=2)
    assert int(pcm2.astype(np.int64).sum()) == int(g["stereo_crc"])
    out2 = oracle.plp_d_a(pcm2, 44100.0, n_chan=2)
    assert out2.shape == g["stereo44k1_lld"].shape
    assert rel_to_frame_scale(out2, g["stereo44k1_lld"]) < TOL


@pytest.mark.parametrize("sr,n,seed,nch", PLP_CASES)
def test_plp_oracle_vs_live_reference(sr, n, seed, nch):
    pcm = voiced_pcm(n, sr, seed=seed, n_chan=nch)
    ref = reference_rows(plp_key(sr, n, seed, nch), pcm)
    out = oracle.plp_d_a(pcm, float(sr), n_chan=nch)
    assert out.shape == ref.shape
    assert rel_to_frame_scale(out, ref) < TOL


def test_rasta_oracle_vs_golden():
    """cPlp with RASTA / newRASTA and cVectorOperation(ll1): oracle restatement against outputs of the
    unmodified reference (tests/golden/conf_goldens.npz, scripts/make_golden_conf.py)."""
    g = np.load(os.path.join(GOLD, "conf_goldens.npz"))
    # tests/configs/rasta_plp.conf: RASTA-PLP cepstra 0..8 on the HTK-style front end
    fe = oracle.Frontend(16000.0, 0.025, 0.010, 1, 0.97, oracle.WIN["ham"], 0.4, 1.0, 0.0, 0)
    ms = oracle.Melspec(26, 0.0, 8000.0, 1, 1)
    pl = oracle.Plp(8, 0, -1, 1, 1, 1, 1, 1, 1, 1, 0, 29.0, 1.0, 22.0, 0.33, 1e-6, 0)
    st = oracle.plp_static(voiced_pcm(16000, 16000, seed=9), 16000.0, (fe, ms, pl))
    ref = g["rasta_plp"]
    assert st.shape == (ref.shape[0], 9)
    assert rel_to_frame_scale(st, ref[:, :9]) < TOL
    assert np.array_equal(oracle.delta(ref[:, :9], 2)[:ref.shape[0]], ref[:, 9:])
    # tests/configs/compare_ns.conf taps: newRASTA-filtered auditory bands and the two band sums
    fe = oracle.Frontend(16000.0, 0.020, 0.010, 0, 0.0, oracle.WIN["ham"], 0.4, 1.0, 0.0, 1)
    ms = oracle.Melspec(26, 20.0, 8000.0, 1, 0)
    pcm = voiced_pcm(16000, 16000, seed=7)
    aud, audR = (oracle.plp_static(pcm, 16000.0, (fe, ms, oracle.Plp(5, 0, -1, 0, 1, 0, 0, 0, 0, 0, nr, 29.0, 1.0, 22.0, 0.33, 9.3e-10, 0)))
                 for nr in (0, 1))
    tap = g["cmp_taps"]
    assert tap.shape == (aud.shape[0], 28)
    assert rel_to_frame_scale(audR, tap[:, :26]) < TOL
    assert np.abs(oracle.ll1(aud) - tap[:, 26]).max() < TOL * np.abs(tap[:, 26]).max()
    assert np.abs(oracle.ll1(audR) - tap[:, 27]).max() < TOL * np.abs(tap[:, 27]).max()
    assert np.array_equal(oracle.ll1(tap[:, :26]), tap[:, 27])       # ll1 itself is bit-exact given its input


def test_cms_oracle_bit_exact_given_reference_statics():
    """cFullinputMean (cepstral mean subtraction): float sum in frame order / (float)T, subtracted --
    bit-exact against the reference given the reference's own statics; deltas are taken from the
    un-normalised coefficients and stay untouched."""
    g = np.load(os.path.join(GOLD, "conf_goldens.npz"))
    z, plain = g["mfcc_z"], g["mfcc_z_plain"]
    assert z.shape == plain.shape == (73, 39)
    assert np.array_equal(oracle.cms(plain[:, :13]), z[:, :13])
    assert np.array_equal(plain[:, 13:], z[:, 13:])


def test_intensity_oracle_bit_exact_vs_reference():
    """cIntensity loudness of config/prosody/prosodyAcf.conf (third column of its lld level, after sma3):
    restated with the reference's own loop bound (only the first sample(s) of a frame enter the sum)."""
    g = np.load(os.path.join(GOLD, "conf_goldens.npz"))
    ref = g["ref_prosody_acf"]
    fe = oracle.Frontend(16000.0, 0.050, 0.010, 0, 0.0, oracle.WIN["gau"], 0.4, 1.0, 0.0, 0)
    loud = oracle.intensity(voiced_pcm(12000, 16000, seed=11), fe, oracle.Intensity(0, 1))
    assert np.array_equal(oracle.sma(loud, 3)[:ref.shape[0], 0], ref[:, 2])
