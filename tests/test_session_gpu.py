"""GPU tests of the conf front end: whole configuration files through libosm_b200.so (parser ->
plan -> CUDA kernels -> HTK / CSV writers) against outputs of the UNMODIFIED reference for the same
files (tests/golden/conf_goldens.npz, scripts/make_golden_conf.py).

Tolerance: float32 path, |got - ref| <= 1e-5 * (largest magnitude of that element over the
utterance) per element -- BASELINE's 1e-5 relative bound taken per output column, because one row
mixes quantities of very different scale (spectral variance ~1e6 Hz^2 next to a zero-crossing rate)."""
import os
import struct
import subprocess
import wave

import numpy as np
import pytest

from conftest import ROOT
from opensmile_b200 import Session, pack_utterances
from opensmile_b200.synth import voiced_pcm

pytestmark = pytest.mark.gpu
CONF = os.path.join(ROOT, "tests", "configs")
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "conf_goldens.npz"))
REFCONF = os.path.join(ROOT, "tests", "golden", "config")


def col_err(got, ref):
    scale = np.maximum(np.abs(ref).max(axis=0), 1e-30)
    return (np.abs(got.astype(np.float64) - ref) / scale).max(axis=0)


def write_wav(path, pcm, sr, nch=1):
    with wave.open(str(path), "wb") as w:
        w.setnchannels(nch)
        w.setsampwidth(2)
        w.setframerate(sr)
        w.writeframes(np.ascontiguousarray(pcm, dtype="<i2").tobytes())


def read_htk(path):
    raw = open(path, "rb").read()
    n, period, size, kind = struct.unpack(">iihh", raw[:12])
    return np.frombuffer(raw[12:], dtype=">f4").astype(np.float32).reshape(n, size // 4), period, kind


def test_mfcc_e_d_a_conf_batch_with_short_utterances():
    pcm = voiced_pcm(12000, 16000, seed=5)
    utts = [pcm, pcm[:400], pcm[:560], pcm[:720], pcm[:880]]
    packed, off = pack_utterances(utts)
    s = Session(os.path.join(CONF, "mfcc_e_d_a.conf"))
    rows, fo = s.extract_pcm(packed, off, 16000, 1)
    refs = [GOLD["mfcc_e"]] + [GOLD["mfcc_e_short_%d" % n] for n in (400, 560, 720, 880)]
    assert list(np.diff(fo)) == [r.shape[0] for r in refs]
    for u, ref in enumerate(refs):
        got = rows[fo[u]:fo[u + 1]]
        scale = np.abs(ref).max(axis=1, keepdims=True)
        assert (np.abs(got - ref) / scale).max() < 1e-5, u


def test_plp_e_d_a_conf():
    pcm = voiced_pcm(12000, 16000, seed=6)
    s = Session(os.path.join(CONF, "plp_e_d_a.conf"))
    rows, fo = s.extract_pcm(pcm, [0, 12000], 16000, 1)
    ref = GOLD["plp_e"]
    assert rows.shape == ref.shape
    assert (np.abs(rows - ref) / np.abs(ref).max(axis=1, keepdims=True)).max() < 1e-5


@pytest.mark.parametrize("key,n,sr,nch,seed", [("mix16k", 16000, 16000, 1, 3), ("mix32k_stereo", 16000, 32000, 2, 4)])
def test_mixed_lld_conf_two_streams(key, n, sr, nch, seed):
    pcm = voiced_pcm(n, sr, seed=seed, n_chan=nch)
    s = Session(os.path.join(CONF, "lld_mix.conf"))
    names = s.element_names(sr, nch)
    rows, fo = s.extract_pcm(pcm, [0, n], sr, nch)
    ref = GOLD[key]
    assert rows.shape == ref.shape
    err = col_err(rows, ref)
    # F0 / F0env follow an arg-max over ACF lags: exact lag or a different peak, never "close"
    lagcols = [i for i, nm in enumerate(names) if nm.startswith("F0")]
    others = [i for i in range(len(names)) if i not in lagcols]
    bad = [(names[i], float(err[i])) for i in others if err[i] > 1e-5]
    assert not bad, bad
    for i in lagcols:
        assert (np.abs(rows[:, i] - ref[:, i]) <= 1e-5 * np.abs(ref[:, i]).max()).mean() > 0.98, names[i]


def test_extract_files_writes_reference_formats(tmp_path):
    pcm = voiced_pcm(12000, 16000, seed=5)
    write_wav(tmp_path / "a.wav", pcm, 16000)
    write_wav(tmp_path / "b.wav", pcm[:880], 16000)
    s = Session(os.path.join(CONF, "mfcc_e_d_a.conf"), options={"instname": "utt7"})
    frames = s.extract_files([str(tmp_path / "a.wav"), str(tmp_path / "b.wav")],
                             [str(tmp_path / "a.htk"), str(tmp_path / "b.htk")], [str(tmp_path / "a.csv"), None])
    assert list(frames) == [73, 4]
    got, period, kind = read_htk(tmp_path / "a.htk")
    assert (period, kind) == (100000, 9)
    ref = GOLD["mfcc_e"]
    assert (np.abs(got - ref) / np.abs(ref).max(axis=1, keepdims=True)).max() < 1e-5
    gotb, _, _ = read_htk(tmp_path / "b.htk")
    assert np.abs(gotb - GOLD["mfcc_e_short_880"]).max() < 1e-5 * np.abs(GOLD["mfcc_e_short_880"]).max()
    lines = (tmp_path / "a.csv").read_text().splitlines()
    ref_lines = GOLD["csv_bytes"].tobytes().decode().splitlines()
    assert lines[0] == ref_lines[0] and len(lines) == len(ref_lines)
    for a, b in zip(lines[1:], ref_lines[1:]):
        fa, fb = a.split(";"), b.split(";")
        assert fa[:2] == fb[:2]                      # 'utt7' and the %f time stamp
        va, vb = np.array(fa[2:], float), np.array(fb[2:], float)
        assert np.abs(va - vb).max() <= 2e-5 * np.abs(vb).max()
    assert not (tmp_path / "b.csv").exists()


def test_command_line_front_end(tmp_path):
    exe = os.path.join(ROOT, "opensmile_b200", "SMILExtract_b200")
    pcm = voiced_pcm(12000, 16000, seed=6)
    write_wav(tmp_path / "in.wav", pcm, 16000)
    r = subprocess.run([exe, "-C", os.path.join(CONF, "plp_e_d_a.conf"), "-I", str(tmp_path / "in.wav"),
                        "-O", str(tmp_path / "out.htk"), "-csvoutput", str(tmp_path / "out.csv")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got, _, _ = read_htk(tmp_path / "out.htk")
    ref = GOLD["plp_e"]
    assert (np.abs(got - ref) / np.abs(ref).max(axis=1, keepdims=True)).max() < 1e-5
    hdr = (tmp_path / "out.csv").read_text().splitlines()[0].split(";")
    assert hdr[:2] == ["name", "frameTime"] and hdr[2:] == [str(x) for x in GOLD["names_plp_e"]]
    # errors are loud and non-zero
    r = subprocess.run([exe, "-C", os.path.join(CONF, "does_not_exist.conf"), "-I", str(tmp_path / "in.wav")], capture_output=True, text=True)
    assert r.returncode != 0 and "cannot open" in r.stderr


def _check_columns(rows, ref, names, tol=1e-5):
    assert rows.shape == ref.shape
    err = col_err(rows, ref)
    bad = [(names[i], float(err[i])) for i in range(len(names)) if err[i] > tol]
    assert not bad, bad


def test_compare_ns_conf_three_band_ops_rasta_and_truncating_reader():
    """ComParE_2016's LLD-path columns: three band ops on one FFT chain (auditory spectrum, its
    newRASTA-filtered variant, MFCC 1-14), band sums (ll1), cSpectral, RMS energy, a 60 ms zcr stream,
    sma3 over multi-level readers that truncate to the shorter stream, delta regression."""
    s = Session(os.path.join(CONF, "compare_ns.conf"))
    pcm = voiced_pcm(16000, 16000, seed=7)
    utts = [pcm, pcm[:960], pcm[:1100], pcm[:1300], pcm[:2000]]
    packed, off = pack_utterances(utts)
    names = s.element_names(16000, 1)
    rows, fo = s.extract_pcm(packed, off, 16000, 1)
    refs = [GOLD["cmp_ns"]] + [GOLD["cmp_ns_short_%d" % n] for n in (960, 1100, 1300, 2000)]
    assert list(np.diff(fo)) == [r.shape[0] for r in refs]
    _check_columns(rows[fo[0]:fo[1]], refs[0], names)
    for u in range(1, 5):     # 2..8-row utterances: per-column scales are not meaningful, use the long utterance's
        scale = np.abs(refs[0]).max(axis=0)
        assert (np.abs(rows[fo[u]:fo[u + 1]] - refs[u]) <= 1e-5 * scale).all(), u


def test_compare_ns_conf_44k():
    s = Session(os.path.join(CONF, "compare_ns.conf"))
    pcm = voiced_pcm(30000, 44100, seed=8)
    rows, fo = s.extract_pcm(pcm, [0, 30000], 44100, 1)
    _check_columns(rows, GOLD["cmp_ns_44k"], s.element_names(44100, 1))


def test_rasta_plp_conf():
    s = Session(os.path.join(CONF, "rasta_plp.conf"))
    pcm = voiced_pcm(16000, 16000, seed=9)
    rows, fo = s.extract_pcm(pcm, [0, 16000], 16000, 1)
    ref = GOLD["rasta_plp"]
    assert rows.shape == ref.shape
    assert (np.abs(rows - ref) / np.abs(ref).max(axis=1, keepdims=True)).max() < 1e-5
    assert s.element_names()[:2] == ["RASTAPlpCC[0]", "RASTAPlpCC[1]"]


def test_gemaps_ns_conf():
    """eGeMAPSv02's LLD-path columns: loudness, log-spectral slopes / alpha ratio / Hammarberg index,
    flux, MFCC 1-4, sma3.  The two log-spectral slopes are least-squares fits over a handful of dB
    values of low-energy bins -> ill-conditioned, checked at 1e-4 of the column scale (see
    test_spectral_compare16_and_gemaps_vs_oracle)."""
    s = Session(os.path.join(CONF, "gemaps_ns.conf"))
    pcm = voiced_pcm(16000, 16000, seed=10)
    rows, fo = s.extract_pcm(pcm, [0, 16000], 16000, 1)
    ref = GOLD["gemaps_ns"]
    names = s.element_names()
    assert rows.shape == ref.shape and names == [str(x) for x in GOLD["names_gemaps_ns"]]
    err = col_err(rows, ref)
    for i, nm in enumerate(names):
        assert err[i] < (1e-4 if "Slope" in nm else 1e-5), (nm, float(err[i]))


def test_mfcc_and_plp_0_d_a_confs_match_reference_goldens():
    """tests/configs/{mfcc,plp}_0_d_a.conf carry the parameters of the reference's MFCC12_0_D_A / PLP_0_D_A
    configurations: their output must equal the goldens the reference produced with its own files."""
    ex = np.load(os.path.join(ROOT, "tests", "golden", "mfcc_example_44k1.npz"))
    pcm, sr = ex["pcm"], int(ex["sample_rate"])
    s = Session(os.path.join(CONF, "mfcc_0_d_a.conf"))
    rows, _ = s.extract_pcm(pcm, [0, len(pcm)], sr, 1)
    ref = ex["lld"]
    assert rows.shape == ref.shape == (202, 39)
    assert (np.abs(rows - ref) / np.abs(ref).max(axis=1, keepdims=True)).max() < 1e-5
    assert s.element_names(sr, 1)[0] == "pcm_fftMag_mfcc[0]"
    g = np.load(os.path.join(ROOT, "tests", "golden", "plp_goldens.npz"))
    s = Session(os.path.join(CONF, "plp_0_d_a.conf"))
    rows, _ = s.extract_pcm(pcm, [0, len(pcm)], sr, 1)
    ref = g["example_lld"]
    assert rows.shape == ref.shape == (202, 18)
    assert (np.abs(rows - ref) / np.abs(ref).max(axis=1, keepdims=True)).max() < 1e-5


def test_cepstral_mean_subtraction_confs():
    """cFullinputMean: per-utterance mean of the static coefficients (float sum in frame order) subtracted;
    own configuration and -- when the build copied them -- the reference's four shipped *_Z files."""
    pcm = voiced_pcm(12000, 16000, seed=11)
    utts = [pcm, pcm[:4000], pcm]                    # the mean is per utterance: neighbours must not leak
    packed, off = pack_utterances(utts)
    s = Session(os.path.join(CONF, "mfcc_0_d_a_z.conf"))
    rows, fo = s.extract_pcm(packed, off, 16000, 1)
    ref = GOLD["mfcc_z"]
    for u in (0, 2):
        got = rows[fo[u]:fo[u + 1]]
        assert got.shape == ref.shape
        assert (np.abs(got - ref) / np.abs(GOLD["mfcc_z_plain"]).max(axis=1, keepdims=True)).max() < 1e-5
    assert np.array_equal(rows[fo[0]:fo[1]], rows[fo[2]:fo[3]])
    for key, rel in (("ref_mfcc_0_z", "mfcc/MFCC12_0_D_A_Z.conf"), ("ref_mfcc_e_z", "mfcc/MFCC12_E_D_A_Z.conf"),
                     ("ref_plp_0_z", "plp/PLP_0_D_A_Z.conf"), ("ref_plp_e_z", "plp/PLP_E_D_A_Z.conf")):
        s = Session(os.path.join(REFCONF, rel))
        got, _ = s.extract_pcm(pcm, [0, 12000], 16000, 1)
        ref = GOLD[key]
        assert got.shape == ref.shape, key
        # scale: the un-normalised statics are ~1e1, mean-subtracted columns can be ~0 in a whole row
        assert np.abs(got - ref).max() < 1e-5 * np.abs(ref).max(), key


def test_more_shipped_configs_audspec_spectrogram_demo1(tmp_path):
    """config/audspec/*.conf (auditory spectrum + deltas), config/spectrum/spectrogram.conf (the magnitude
    level itself as output) and config/demo/demo1_energy.conf (CSV sink with a frame index column), unchanged."""
    pcm = voiced_pcm(12000, 16000, seed=11)
    for key, rel in (("ref_audspec", "audspec/audspec.conf"), ("ref_audspec_compat", "audspec/audspec_compat.conf")):
        got, _ = Session(os.path.join(REFCONF, rel)).extract_pcm(pcm, [0, 12000], 16000, 1)
        ref = GOLD[key]
        assert got.shape == ref.shape, key
        assert (np.abs(got - ref) / np.abs(ref).max(axis=1, keepdims=True)).max() < 1e-5, key
    s = Session(os.path.join(REFCONF, "spectrum", "spectrogram.conf"))
    got, _ = s.extract_pcm(pcm[:4000], [0, 4000], 16000, 1)
    ref = GOLD["ref_spectrogram"]
    assert got.shape == ref.shape == (23, 257)
    assert (np.abs(got - ref) / np.abs(ref).max(axis=1, keepdims=True)).max() < 1e-5
    assert s.element_names()[256] == "pcm_fftMag[256]"
    # prosodyAcf: ACF / cepstrum pitch + cIntensity loudness, smoothed
    s = Session(os.path.join(REFCONF, "prosody", "prosodyAcf.conf"))
    got, _ = s.extract_pcm(pcm, [0, 12000], 16000, 1)
    ref = GOLD["ref_prosody_acf"]
    assert got.shape == ref.shape and s.element_names() == [str(x) for x in GOLD["names_ref_prosody_acf"]]
    assert np.abs(got[:, 0] - ref[:, 0]).max() < 1e-5 and np.abs(got[:, 2] - ref[:, 2]).max() <= 1e-6 * np.abs(ref[:, 2]).max()
    assert (np.abs(got[:, 1] - ref[:, 1]) <= 1e-5 * np.abs(ref[:, 1]).max()).mean() > 0.98      # F0: lag-valued
    # demo1: the csv file is named by -O (the config's own option), one row per frame: index;time;value
    write_wav(tmp_path / "in.wav", pcm, 16000)
    s = Session(os.path.join(REFCONF, "demo", "demo1_energy.conf"), options={"O": str(tmp_path / "unused.csv")})
    s.extract_files([str(tmp_path / "in.wav")], None, [str(tmp_path / "out.csv")])
    lines = (tmp_path / "out.csv").read_text().splitlines()
    ref_lines = GOLD["ref_demo1_energy_csv"].tobytes().decode().splitlines()
    assert lines[0] == ref_lines[0] == "frameIndex;frameTime;pcm_LOGenergy" and len(lines) == len(ref_lines)
    for a, b in zip(lines[1:], ref_lines[1:]):
        fa, fb = a.split(";"), b.split(";")
        assert fa[:2] == fb[:2] and abs(float(fa[2]) - float(fb[2])) <= 2e-6 * abs(float(fb[2]))
