"""The arithmetic of the formant kernel (opensmile_b200/csrc/formant.cu) held against level taps of the UNMODIFIED
reference without a GPU: formant_math.cuh and the table builder are compiled for the host (tests/formant_harness.py),
the lanes of a warp become loops.  Stage by stage, each on the reference's own input level:
  cSpecResample level -> cLpc coefficients      bit-identical
  cLpc level -> cFormantLpc frequencies / bandwidths   bit-identical
  windower level -> cSpecResample level         within 2e-6 of the frame scale (one rounding per product instead of the
                                                reference's float FFT + float inverse sum)
and the graph side: element names, defaults, refusals."""
import os

import numpy as np
import pytest

import formant_harness as fh
from opensmile_b200.session import Session, SessionError
from opensmile_b200.synth import mixed_pcm

HERE = os.path.dirname(os.path.abspath(__file__))
G = np.load(os.path.join(HERE, "golden", "formant_goldens.npz"))
CONF = os.path.join(HERE, "configs", "formant_taps.conf")


def test_lpc_bit_identical_on_the_reference_resampled_level():
    a = np.stack([fh.lpc(x, 11) for x in G["res"]])
    assert np.array_equal(a, G["lpc"])


def test_formants_bit_identical_on_the_reference_lpc_level():
    f = np.stack([fh.formants(a, 1.0 / 11000.0, 5, 50.0, 5450.0) for a in G["lpc"]])
    assert np.array_equal(f, G["fmt"])


def test_root_finder_against_lapack():
    """simultaneous iteration vs numpy (companion matrix eigenvalues) on LPC-like polynomials incl. poles next to the
    unit circle; bounded sweep count"""
    rng = np.random.default_rng(0)
    worst, sweeps = 0.0, 0
    for _ in range(400):
        r = []
        for k in range(5):
            m, th = rng.uniform(0.3, 0.9999), rng.uniform(0.01, 3.13)
            r += [m * np.exp(1j * th), m * np.exp(-1j * th)]
        r.append(rng.uniform(-0.99, 0.99))
        c = np.poly(r).real[::-1][:11].copy()
        z, it = fh.roots(c)
        ref = np.roots(np.concatenate([c, [1.0]])[::-1])
        worst = max(worst, np.abs(z[:, None] - ref[None, :]).min(axis=1).max())
        sweeps = max(sweeps, it)
    assert worst < 1e-8 and sweeps < 40


def test_degenerate_frames():
    assert not fh.lpc(np.zeros(220, np.float32), 11).any()                        # silence: r[0] == 0 -> a = 0
    assert not fh.formants(np.zeros(11, np.float32), 1.0 / 11000.0, 5, 50.0, 5450.0).any()   # all roots at the origin
    a = np.zeros(11, np.float32)
    a[0] = -0.9                                                                   # one real pole, ten roots at the origin
    assert not fh.formants(a, 1.0 / 11000.0, 5, 50.0, 5450.0).any()
    a[:2] = [-1.2, -0.81]                                                         # a conjugate pair: radius 0.9, angle acos(-2/3)
    f = fh.formants(a, 1.0 / 11000.0, 5, 50.0, 5450.0)
    ang = np.arccos(-1.2 / (2 * 0.9))
    assert abs(f[0] - ang / (2 * np.pi) * 11000.0) < 1e-2 and abs(f[5] - (-np.log(0.9) * 11000.0 / np.pi)) < 1e-2 and not f[1:5].any()


def test_resampled_frames_are_bit_identical_to_the_reference_level():
    """FFT size 512: the kernel's statements (reference-order FFT, fft_ref_order.cuh, + the float inverse sum in the reference's
    order) reproduce the reference's cSpecResample level bit for bit"""
    pcm = mixed_pcm(24000, 16000, seed=3)
    xw, nfft = fh.windowed_frames(pcm)
    res, per = fh.resample(xw, 16000.0, nfft, 0.020, 11000.0)
    assert res.shape == G["res"].shape and per == 1.0 / 11000.0
    assert np.array_equal(res.view(np.uint32), G["res"].view(np.uint32))


def test_composed_table_path_against_the_reference_level(monkeypatch):
    """other FFT sizes use the composed table (zero padding, FFT and inverse sum folded into one matrix in double): 2e-6"""
    monkeypatch.setenv("OSM_B200_FORMANT_COMPOSED", "1")
    pcm = mixed_pcm(24000, 16000, seed=3)
    xw, nfft = fh.windowed_frames(pcm)
    res, per = fh.resample(xw, 16000.0, nfft, 0.020, 11000.0)
    assert res.shape == G["res"].shape and per == 1.0 / 11000.0
    err = np.abs(res - G["res"]).max() / np.abs(G["res"]).max()
    assert 0 < err < 2e-6


def test_end_to_end_formants_equal_the_reference_level():
    """PCM -> formant frequencies / bandwidths through the kernel's statements: equal to the reference's cFormantLpc level on
    every frame (the reference-order FFT removed the 1e-3 .. 1e-2 deviations that order-11 LPC made of 2e-7 spectral noise)"""
    got = fh.formant_chain(mixed_pcm(24000, 16000, seed=3))
    ref = G["fmt"]
    assert got.shape == ref.shape
    assert (np.abs(got - ref) / np.abs(ref).max(axis=0)).max() < 1e-6


def test_composed_path_deviation_is_the_conditioning_of_lpc(monkeypatch):
    """kept for the FFT sizes without a reference-order transform: a 1e-6 difference of the resampled frames reaches the
    formants through an order-11 float Durbin recursion -- typical rows agree to 1e-5, rows with poles next to each other move
    by percents"""
    monkeypatch.setenv("OSM_B200_FORMANT_COMPOSED", "1")
    got = fh.formant_chain(mixed_pcm(24000, 16000, seed=3))
    ref = G["fmt"]
    err = np.abs(got - ref) / np.abs(ref).max(axis=0)
    assert np.median(err) < 1e-4
    assert (err.max(axis=1) > 1e-3).mean() < 0.25


def test_graph_names_and_refusals(tmp_path):
    s = Session(CONF, output_level="formants", device=-1)
    assert s.element_names() == ["formantFreqLpc[%d]" % i for i in range(1, 6)] + ["formantBandwidthLpc[%d]" % i for i in range(1, 6)]
    text = open(CONF).read()
    for old, new, needle in (("method=acf", "method=burg", "method=acf"), ("nFormants=5", "nFormants=3", "nFormants < p/2"),
                             ("medianFilter=0", "medianFilter=5", "medianFilter"), ("residual=0", "residual=1", "residual")):
        assert old in text
        p = tmp_path / "c.conf"
        p.write_text(text.replace(old, new))
        with pytest.raises(SessionError, match=needle):
            Session(str(p), output_level="formants", device=-1)


# ------------------------------------------------------------------------------------------------------------------
# cHarmonics (opensmile_b200/csrc/harmonics_math.cuh, kernel harmonics.cu) and the shipped GeMAPS graphs

def test_harmonics_on_the_reference_input_levels():
    """host build of the kernel's statements on the reference's own F0 / formant / magnitude levels
    (tests/configs/harmonics_taps.conf): every decision (harmonic peaks, formant-range maxima, ACF peak) reproduced,
    values within 1e-5 dB (log10f / log10 of another libm)"""
    f0, fmt, mag, harm = G["h_f0"], G["h_fmt"], G["h_mag"], G["h_harm"]
    T = min(len(f0), len(fmt), len(mag), len(harm))
    nfft = (mag.shape[1] - 1) * 2
    bin_hz = 1.0 / (0.060 * nfft / 960)
    out = np.stack([fh.harmonics(f0[t, 0], fmt[t, :5], mag[t], bin_hz) for t in range(T)])
    assert (f0[:T, 0] > 0).sum() > 50
    assert np.abs(out - harm[:T]).max() < 1e-5


def test_harmonics_unvoiced_and_edge_frames():
    mag = np.abs(np.random.default_rng(0).standard_normal(513)).astype(np.float32)
    out = fh.harmonics(0.0, [500.0, 1500.0, 2500.0], mag, 16000.0 / 1024)
    assert list(out) == [0.0, 0.0, 0.0, -201.0, -201.0, -201.0]                  # F0 = 0: HNR 0, differences 0, amplitudes at the floor
    out = fh.harmonics(7900.0, [500.0, 1500.0, 2500.0], mag, 16000.0 / 1024)    # first harmonic next to Nyquist
    assert np.isfinite(out).all()
    out = fh.harmonics(120.0, [500.0, 1500.0, 2500.0], np.zeros(513, np.float32), 16000.0 / 1024)   # silence
    assert np.isfinite(out).all()
    out = fh.harmonics(1e-3, [500.0, 1500.0, 2500.0], mag, 16000.0 / 1024)      # F0 far below the pitch range: lag beyond the ACF, bounded search
    assert np.isfinite(out).all()


@pytest.mark.parametrize("conf,opts,key,n", [("gemaps/v01b/GeMAPSv01b.conf", {"lldhtkoutput": "x.htk"}, "gemaps_lld", 18),
                                             ("egemaps/v02/eGeMAPSv02.conf", {"lldcsvoutput": "x.csv"}, "egemaps_lld", 25)])
def test_shipped_gemaps_configurations_open(conf, opts, key, n):
    """the shipped GeMAPSv01b.conf / eGeMAPSv02.conf (BASELINE configs[2]) compile unchanged: cDataSelector scopes, cHarmonics
    field lookup by name, the lagging selector over pitch / jitter / harmonics / formant levels; element names and frame
    counts against the reference's LLD files"""
    ref = os.path.join(HERE, "golden", "config")
    from oracle import formant_oracle as fo
    s = Session(os.path.join(ref, conf), options=opts, device=-1)
    names = s.element_names()
    assert len(names) == n
    if key == "egemaps_lld":
        assert names == list(G["names_egemaps_lld"]) == fo.EGEMAPS_LLD_NAMES
    else:
        assert names[:5] == fo.EGEMAPS_LLD_NAMES[:5] and names[5] == "F0semitoneFrom27.5Hz_sma3nz" and names[-1] == "F3amplitudeLogRelF0_sma3nz"
    fo_ = s.frame_offsets(np.array([0, 24000, 64000], np.int64), 16000.0, 1)
    assert list(np.diff(fo_)) == [G[key + "_m24k"].shape[0], G[key + "_m40k"].shape[0]]


@pytest.mark.parametrize("sr,target", [(44100.0, 11000.0), (8000.0, 11000.0), (8000.0, 16000.0), (16000.0, 32000.0), (22050.0, 22050.0)])
def test_resampling_table_other_rates(sr, target):
    """the composed table (zero padding + FFT + inverse DFT of the low bins in one matrix) against the literal restatement
    FFT -> cSpecResample of the oracle at other sample rates, incl. up-sampling (the branch with the Nyquist term, I >= K)"""
    import ctypes as C
    from oracle import oracle, formant_oracle as fo
    pcm = mixed_pcm(int(sr * 0.3), int(sr), seed=4)
    fe = oracle.frontend(sr, 0.020, 0.010, win="ham", zero_pad_symmetric=1)
    spec = fo.fft_frames(pcm, fe)
    N, H, nfft, T = oracle.geometry(fe, len(pcm))
    rs = fo.SpecResample(nfft, sr, target, oracle.lib().osm_or_fft_frame_size_sec(C.byref(fe)), 0.020)
    ref = np.stack([rs(a) for a in spec])
    xw, nfft2 = fh.windowed_frames(pcm, sr)
    res, per = fh.resample(xw, sr, nfft2, 0.020, target)
    assert nfft2 == nfft and res.shape == ref.shape and per == rs.base_period_out
    assert np.abs(res - ref).max() / np.abs(ref).max() < 3e-6


def test_all_shipped_gemaps_family_configurations_compile_unchanged():
    """the five shipped feature-set files of the GeMAPS family (-lldcsvoutput): element names and row counts equal the
    reference's CSV files (tests/golden/gemaps_headers.json, written by running oracle/_ref/SMILExtract on
    mixed_pcm(24000, seed=3))"""
    import json
    ref = os.path.join(HERE, "golden", "config")
    gold = json.load(open(os.path.join(HERE, "golden", "gemaps_headers.json")))
    assert len(gold) == 5
    for conf, g in gold.items():
        s = Session(os.path.join(ref, conf), options={"lldcsvoutput": "x.csv"}, device=-1)
        assert s.element_names() == g["names"]
        assert int(s.frame_offsets(np.array([0, 24000], np.int64), 16000.0, 1)[-1]) == g["rows_m24k"]


def test_formants_at_the_nyquist_edge():
    """GeMAPSv01a searches up to maxF = 5500 Hz = the Nyquist frequency of the resampled frames, where real negative roots
    sit: the kernel statements (roots with rounding-noise imaginary parts snapped to the real axis) take the same decisions
    as the oracle's LAPACK roots on every frame"""
    from oracle import formant_oracle as fo
    if not fo.ref_fft_available():
        pytest.skip("oracle/_ref/libfftsg.so not built (make -C oracle ref)")
    fmt, res, lpcs = fo.gemaps_formant_chain(mixed_pcm(24000, 16000, seed=3), taps=True, exact_fft=True, v01a=True)
    got = np.stack([fh.formants(a, 1.0 / 11000.0, 5, 50.0, 5500.0) for a in lpcs])
    assert np.abs(got - fmt).max() < 1e-2
