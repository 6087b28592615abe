"""cFunctionals on the GPU (opensmile_b200/csrc/functionals.cu) through the C ABI: the kernel on the reference's own LLD rows
against the reference's functionals rows and the pinned oracle; the shipped IS09_emotion.conf end to end from PCM (LLD plan ->
rows resident in HBM -> summary -> one row per utterance) against the reference's -csvoutput row."""
import os

import numpy as np
import pytest

from oracle import functionals_oracle as fo
from opensmile_b200 import functionals as F
from opensmile_b200.synth import mixed_pcm, voiced_pcm
from test_functionals_cpu import G, G2, G3, LEVELS, LEVELS2, LEVELS3, REFCONF, contour_rows, to_c_spec

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _cspec(spec):
    """oracle Spec -> ctypes spec"""
    return to_c_spec(spec)


def _close(got, ref, rtol):
    # a summary value is compared relative to its own magnitude, with the magnitude of the largest value of the row's
    # functional family as floor for values near zero (a skewness of 1e-4 next to one of 1.0)
    return np.abs(got - ref) <= rtol * (np.abs(ref) + 1e-3 * np.abs(ref).max()) + 1e-12


@pytest.mark.parametrize("key", ["m24k", "v32k", "rec"])
def test_kernel_on_the_reference_lld_rows(key):
    lld = G["is09_lld_" + key]
    names = list(G["is09_lld_names"])
    for tag, spec, cols, dn, gk in LEVELS:
        rows = np.ascontiguousarray(contour_rows(lld, dn)[:, cols])
        f = F.Functionals(_cspec(spec), names[cols], 0.01, device=0)
        assert f.element_names() == list(G["is09_func_names"] if tag == "is09" else G[gk + "_names"])
        got = f.run_host(rows, [0], [rows.shape[0]])[0]
        f.close()
        ora = fo.functionals(spec, rows, 0.01)
        assert np.all(np.abs(got - ora) <= 2e-6 * np.abs(ora) + 1e-9), tag       # double reductions in another order, float log10 / exp
        ref = G["%s_%s" % (gk, key)][0]
        assert np.all(np.abs(got - ref) <= 2e-6 * np.abs(ref) + 1e-9), tag       # the reference's CSV: 7 significant digits


@pytest.mark.parametrize("key", ["m24k", "v32k", "rec"])
def test_times_lpc_segments_peaks2_on_the_reference_lld_rows(key):
    """tests/configs/func_variants2.conf (the ComParE_2016 / GeMAPS option sets): float statements in the reference's order -> equal
    to the oracle bit for bit except where a double reduction feeds them (the contour mean), and to the reference's CSV digits"""
    lld = G["is09_lld_" + key]
    names = list(G["is09_lld_names"])
    for tag, spec, cols, dn in LEVELS2:
        rows = np.ascontiguousarray(contour_rows(lld, dn)[:, cols])
        f = F.Functionals(to_c_spec(spec), names[cols], 0.01, device=0)
        assert f.element_names() == list(G2["var%s_names" % tag])
        got = f.run_host(rows, [0], [rows.shape[0]])[0]
        f.close()
        ora = fo.functionals(spec, rows, 0.01)
        assert np.all(np.abs(got - ora) <= 2e-6 * np.abs(ora) + 1e-9), (tag, np.nonzero(~(np.abs(got - ora) <= 2e-6 * np.abs(ora) + 1e-9))[0][:8])
        ref = G2["var%s_%s" % (tag, key)][0]
        assert np.all(np.abs(got - ref) <= 2e-6 * np.abs(ref) + 1e-9), tag


@pytest.mark.parametrize("key", ["m24k", "v32k", "rec"])
def test_onset_peaks_crossings_on_the_reference_lld_rows(key):
    """tests/configs/func_variants3.conf (cFunctionalOnset / cFunctionalPeaks / cFunctionalCrossings with the IS10_paraling and emo_large
    option sets and their other norms): equal to the oracle and to the reference's CSV digits"""
    lld = G["is09_lld_" + key]
    names = list(G["is09_lld_names"])
    for tag, spec, cols, dn in LEVELS3:
        rows = np.ascontiguousarray(contour_rows(lld, dn)[:, cols])
        f = F.Functionals(to_c_spec(spec), names[cols], 0.01, device=0)
        assert f.element_names() == list(G3["var%s_names" % tag])
        got = f.run_host(rows, [0], [rows.shape[0]])[0]
        f.close()
        ora = fo.functionals(spec, rows, 0.01)
        assert np.all(np.abs(got - ora) <= 2e-6 * np.abs(ora) + 1e-9), (tag, np.nonzero(~(np.abs(got - ora) <= 2e-6 * np.abs(ora) + 1e-9))[0][:8])
        ref = G3["var%s_%s" % (tag, key)][0]
        assert np.all(np.abs(got - ref) <= 2e-6 * np.abs(ref) + 1e-9), tag


def test_sequential_functionals_on_ragged_and_degenerate_contours():
    rng = np.random.default_rng(11)
    lens = [300, 1, 2, 0, 5, 33, 64, 2500]
    K = 6
    rows = np.cumsum(rng.standard_normal((sum(lens), K)), axis=0).astype(np.float32)
    rows[:, 1] = 0
    rows[::3, 2] = 0
    rows[:, 3] = 2.5
    rows[:, 4] = np.where(rng.random(sum(lens)) > 0.6, 0, rows[:, 4])           # pauses for nonX / eqX
    rows[:, 5] = np.round(rows[:, 5])                                            # plateaus
    off = np.concatenate([[0], np.cumsum(lens)])[:-1]
    pk = {k: 1 for k in fo.PEAKS2_NAMES}
    specs = [fo.Spec(["Times", "Lpc", "Segments", "Peaks2", "Percentiles"], non_zero=nz, master_norm=mn, percentiles=dict(quartile2=1),
                     times=dict(buggySecNorm=bs), lpc=dict(lpGain=1, order=od),
                     segments=dict(segmentationAlgorithm=al, thresholds=[0.3, 0.6], maxNumSeg=50, numSegments=1, meanSegLen=1, maxSegLen=1,
                                   minSegLen=1, segLenStddev=1),
                     peaks2=dict(pk, relThresh=rt, dynRelThresh=dy, doRatioLimit=rl))
             for nz, mn, bs, od, al, rt, dy, rl in ((0, fo.SEGMENT, 0, 5, "relTh", 0.1, 0, 1), (1, fo.SECOND, 1, 8, "nonX", 0.35, 1, 0),
                                                    (0, fo.FRAME, 0, 3, "eqX", 0.0, 0, 1))]
    specs += [fo.Spec(["Onset", "Peaks", "Crossings", "Percentiles"], non_zero=nz, master_norm=mn, percentiles=dict(quartile2=1),
                      onset=dict(threshold=th, useAbsVal=ab, onsetPos=1, offsetPos=1, numOnsets=1, numOffsets=1, onsetRate=1),
                      peaks=dict(peakDistStddev=1), crossings=dict(amean=1))
              for nz, mn, th, ab in ((0, fo.SEGMENT, 0.0, 0), (1, fo.SECOND, 1.5, 1), (0, fo.FRAME, -2.0, 0))]
    for spec in specs:
        f = F.Functionals(to_c_spec(spec), ["c%d" % i for i in range(K)], 0.01, device=0)
        got = f.run_host(rows, off, lens)
        f.close()
        for u, (o, n) in enumerate(zip(off, lens)):
            ora = fo.functionals(spec, rows[o:o + n], 0.01) if n else np.zeros(got.shape[1], np.float32)
            ok = (np.abs(got[u] - ora) <= 2e-6 * np.abs(ora) + 1e-9) | (np.isnan(got[u]) & np.isnan(ora))
            assert np.all(ok), (spec.enabled, spec.segments["segmentationAlgorithm"], u, np.nonzero(~ok)[0][:8], got[u][~ok][:4], ora[~ok][:4])


def test_ragged_batch_and_degenerate_contours():
    rng = np.random.default_rng(3)
    lens = [300, 1, 2, 0, 33, 64, 4097]
    K = 5
    rows = rng.standard_normal((sum(lens), K)).astype(np.float32)
    rows[:, 1] = 0                                    # a contour without any non-zero value
    rows[::3, 2] = 0                                  # zeros spread over a contour
    rows[:, 3] = 2.5                                  # a constant contour
    off = np.concatenate([[0], np.cumsum(lens)])[:-1]
    for spec in (fo.Spec(["Extremes", "Means", "Moments", "Percentiles", "Regression"], non_zero=nz, master_norm=fo.SEGMENT,
                         percentiles=dict(quartile1=1, quartile2=1, quartile3=1, iqr13=1, percentile=[0.05, 0.95], pctlrange=[(0, 1)], interp=ip),
                         regression=dict(centroidUseAbsValues=ab), moments=dict(stddevNorm=1, amean=1))
                 for nz, ip, ab in ((0, 1, 1), (1, 0, 0), (2, 1, 1))):
        f = F.Functionals(_cspec(spec), ["c%d" % i for i in range(K)], 0.01, device=0)
        got = f.run_host(rows, off, lens)
        f.close()
        for u, (o, n) in enumerate(zip(off, lens)):
            ora = fo.functionals(spec, rows[o:o + n], 0.01) if n else np.zeros(got.shape[1], np.float32)
            assert np.all(_close(got[u], ora, 1e-5)), (spec.non_zero, u)


def test_shipped_is09_configuration_end_to_end():
    from opensmile_b200.session import Session
    rec = np.load(os.path.join(HERE, "golden", "egemaps_recordings.npz"))["pcm_opensmile_16k"]
    pcms = [mixed_pcm(24000, 16000, seed=3), np.zeros(100, np.int16), voiced_pcm(32000, 16000, seed=7), rec]
    off = np.concatenate([[0], np.cumsum([len(x) for x in pcms])]).astype(np.int64)
    s = Session(os.path.join(REFCONF, "is09-13", "IS09_emotion.conf"), options={"csvoutput": "f.csv"}, device=0)
    assert s.element_names() == list(G["is09_func_names"])
    rows, fo_ = s.extract_pcm(np.concatenate(pcms + [np.zeros(8, np.int16)]), off, 16000.0, 1)
    s.close()
    assert list(fo_) == [0, 1, 1, 2, 3] and rows.shape == (3, 384)
    names = list(G["is09_func_names"])
    for r, key in enumerate(("m24k", "v32k", "rec")):
        ref = G["is09_func_" + key][0]
        # Per functional family (12 values per contour): 1e-5 of the family's largest magnitude over the 32 contours.
        fam = np.abs(ref).reshape(32, 12).max(axis=0)
        err = (np.abs(rows[r] - ref).reshape(32, 12) / (fam + 1e-12))
        worst = {names[int(i) * 12 + int(j)]: float(err[i, j]) for i, j in zip(*np.nonzero(err >= 1e-5))}
        assert not worst, (key, worst)


def test_shipped_compare16_functionals_end_to_end():
    """config/compare16/ComParE_2016.conf -csvoutput unchanged: 6373 features = six cFunctionals instances (Extremes, Percentiles,
    Moments, Segments, Times, Lpc, Means, Regression, Peaks2) on column subsets of the 130 LLD columns, from PCM, against the
    reference's row.  Per functional value (name suffix): 1e-5 of that value's largest magnitude over the contours; the few
    discontinuous ones (positions, counts, percentile picks on plateaus) may flip on single contours and are counted (<= 0.5 %).
    Exception, stated: cFunctionalLpc.  Its order-5 float Durbin recursion on the autocorrelation of a smooth contour is ill
    conditioned -- the 1e-7 differences between the LLD rows here and the reference's (different FFT) come out as up to 3e-3 of the
    coefficients' scale, while the same kernel on the reference's own LLD rows is exact (test_times_lpc_segments_peaks2_...): the lpc /
    lpgain values are held to 2e-2."""
    from opensmile_b200.session import Session
    GC = np.load(os.path.join(HERE, "golden", "compare16_func.npz"))
    names = list(GC["names"])
    rec = np.load(os.path.join(HERE, "golden", "egemaps_recordings.npz"))["pcm_opensmile_16k"]
    pcms = [mixed_pcm(24000, 16000, seed=3), voiced_pcm(32000, 16000, seed=7), rec]
    off = np.concatenate([[0], np.cumsum([len(x) for x in pcms])]).astype(np.int64)
    s = Session(os.path.join(REFCONF, "compare16", "ComParE_2016.conf"), options={"csvoutput": "f.csv"}, device=0)
    assert s.element_names() == names
    rows, fo_ = s.extract_pcm(np.concatenate(pcms), off, 16000.0, 1)
    s.close()
    assert list(fo_) == [0, 1, 2, 3] and rows.shape == (3, 6373)
    suffix = np.array([n.rsplit("_", 1)[1] for n in names])
    report = {}
    for r, key in enumerate(("m24k", "v32k", "rec")):
        ref = GC["func_" + key][0]
        bad_total = 0
        for sfx in np.unique(suffix):
            idx = np.nonzero(suffix == sfx)[0]
            scale = np.abs(ref[idx]).max() + 1e-12
            err = np.abs(rows[r, idx] - ref[idx]) / scale
            if sfx.startswith("lpc") or sfx == "lpgain":
                assert err.max() < 2e-2, (key, sfx, float(err.max()))
                continue
            bad = idx[err > 1e-5]
            if bad.size:
                report[(key, sfx)] = (int(bad.size), float(err.max()), names[int(bad[0])])
                bad_total += int(bad.size)
        assert bad_total <= 0.005 * len(names), (key, bad_total, sorted(report.items(), key=lambda kv: -kv[1][0])[:12])
    print("compare16 functionals: values beyond 1e-5 of their family's scale:", report)


def _gemaps_inputs():
    rec = np.load(os.path.join(HERE, "golden", "egemaps_recordings.npz"))["pcm_opensmile_16k"]
    pcms = [mixed_pcm(24000, 16000, seed=3), voiced_pcm(32000, 16000, seed=7), rec]
    off = np.concatenate([[0], np.cumsum([len(x) for x in pcms])]).astype(np.int64)
    return np.concatenate(pcms), off


def test_gemaps_functionals_input_levels_equal_the_reference():
    """the seven levels the eGeMAPSv02 functionals read -- smoothed F0 / loudness, the cValbasedSelector-gated voiced / unvoiced
    parameter sets behind cDataSelector + cContourSmoother, the frame energy -- row by row against the unmodified reference's dumps
    (tests/golden/gemaps_func_levels.npz): same row counts, every column within 1e-5 of its scale"""
    from opensmile_b200.session import Session
    GL = np.load(os.path.join(HERE, "golden", "gemaps_func_levels.npz"))
    pcm, off = _gemaps_inputs()
    conf = os.path.join(REFCONF, "egemaps", "v02", "eGeMAPSv02.conf")
    for lv in sorted({k.split("_", 1)[1] for k in GL.files if not k.startswith("names_")}):
        s = Session(conf, output_level=lv, device=0)
        assert s.element_names() == [str(x) for x in GL["names_" + lv]]
        rows, fo_ = s.extract_pcm(pcm, off, 16000.0, 1)
        s.close()
        for u, key in enumerate(("m24k", "v32k", "rec")):
            ref = GL["%s_%s" % (key, lv)]
            got = rows[fo_[u]:fo_[u + 1]]
            assert got.shape == ref.shape, (lv, key, got.shape, ref.shape)
            err = np.abs(got - ref) / (np.abs(ref).max(axis=0) + 1e-12)
            assert err.max() < 1e-5, (lv, key, float(err.max()))


@pytest.mark.parametrize("conf,tag,n", [("egemaps/v02/eGeMAPSv02.conf", "egemaps", 88), ("gemaps/v01b/GeMAPSv01b.conf", "gemaps", 62)])
def test_shipped_gemaps_summaries_end_to_end(conf, tag, n):
    """config/egemaps/v02/eGeMAPSv02.conf and config/gemaps/v01b/GeMAPSv01b.conf -csvoutput unchanged, from PCM, three utterances in
    one batch, against the reference's rows: nine (seven) cFunctionals instances on the gated / smoothed levels, cDataSelector
    renaming, cVectorOperation dBp, cVectorConcat order.  Every value within 1e-4 of its own magnitude (the reference's CSV row
    carries 7 digits; the summaries amplify the 1e-6 LLD differences: stddevNorm, slopes)."""
    from opensmile_b200.session import Session
    GF = np.load(os.path.join(HERE, "golden", "gemaps_func.npz"))
    pcm, off = _gemaps_inputs()
    s = Session(os.path.join(REFCONF, conf), options={"csvoutput": "f.csv"}, device=0)
    names = s.element_names()
    assert names == [str(x) for x in GF["names_" + tag]] and len(names) == n
    rows, fo_ = s.extract_pcm(pcm, off, 16000.0, 1)
    s.close()
    assert list(fo_) == [0, 1, 2, 3] and rows.shape == (3, n)
    for u, key in enumerate(("m24k", "v32k", "rec")):
        ref = GF["%s_%s" % (tag, key)][0]
        rel = np.abs(rows[u] - ref) / (np.abs(ref) + 1e-6)
        assert rel.max() < 1e-4, (key, names[int(np.argmax(rel))], float(rows[u][int(np.argmax(rel))]), float(ref[int(np.argmax(rel))]))


@pytest.mark.parametrize("conf,tag", [("egemaps/v02/eGeMAPSv02.conf", "egemaps"), ("gemaps/v01b/GeMAPSv01b.conf", "gemaps")])
def test_gemaps_summaries_on_degenerate_inputs(conf, tag):
    """digital silence, unvoiced noise, an utterance shorter than the Viterbi buffer (the smoother never emits before end of input:
    V = 0), one voiced burst between silence -- ragged batch, against the reference's rows (empty voiced sets: the non-zero filter
    leaves nothing, functionals.cpp:286-330 then writes zeros; no voiced / unvoiced segment at all)"""
    from opensmile_b200.session import Session
    GF = np.load(os.path.join(HERE, "golden", "gemaps_func.npz"))
    rng = np.random.RandomState(11)
    burst = np.zeros(20000, np.int16)
    burst[6000:12000] = voiced_pcm(6000, 16000, seed=5)
    sig = {"silence": np.zeros(16000, np.int16), "noise": (rng.randn(16000) * 800).astype(np.int16), "short": voiced_pcm(4000, 16000, seed=9),
           "burst": burst}
    keys = ["silence", "noise", "short", "burst"]
    sig["tiny"] = voiced_pcm(300, 16000, seed=2)          # shorter than one 20 ms frame: no frame, hence no summary row for this input
    order = ["silence", "noise", "tiny", "short", "burst"]
    off = np.concatenate([[0], np.cumsum([len(sig[k]) for k in order])]).astype(np.int64)
    s = Session(os.path.join(REFCONF, conf), options={"csvoutput": "f.csv"}, device=0)
    names = s.element_names()
    rows, fo_ = s.extract_pcm(np.concatenate([sig[k] for k in order]), off, 16000.0, 1)
    s.close()
    assert list(fo_) == [0, 1, 2, 2, 3, 4]
    for u, key in enumerate(keys):
        ref = GF["%s_%s" % (tag, key)][0]
        assert np.all(np.isfinite(rows[u]))
        err = np.abs(rows[u] - ref) / (np.abs(ref) + 1e-4)
        i = int(np.argmax(err))
        assert err[i] < 2e-4, (key, names[i], float(rows[u][i]), float(ref[i]))


def test_summary_configuration_from_wav_files_to_csv(tmp_path):
    """the file route of a summary configuration (what the command line front end runs): WAV files in, one CSV per input with the
    reference sink's layout and the reference's values (eGeMAPSv02.conf -I x.wav -csvoutput x.csv)"""
    from oracle import refrun
    from opensmile_b200.session import Session
    from test_functionals_cpu import _csv_close
    GF = np.load(os.path.join(HERE, "golden", "gemaps_func.npz"))
    wavs, outs = [], []
    for i, pcm in enumerate((mixed_pcm(24000, 16000, seed=3), voiced_pcm(32000, 16000, seed=7))):
        wavs.append(str(tmp_path / ("in%d.wav" % i)))
        outs.append(str(tmp_path / ("out%d.csv" % i)))
        refrun.write_wav(wavs[-1], pcm, 16000, 1)
    s = Session(os.path.join(REFCONF, "egemaps", "v02", "eGeMAPSv02.conf"), options={"csvoutput": "f.csv"}, device=0)
    frames = s.extract_files(wavs, csv_paths=outs)
    s.close()
    assert list(frames) == [1, 1]
    _csv_close(open(outs[0]).read(), GF["csv_egemaps_m24k"].tobytes().decode(), 1e-4)
    head = open(outs[1]).read().split("\n")
    assert head[0] == GF["csv_egemaps_m24k"].tobytes().decode().split("\n")[0] and head[1].startswith("'unknown';0.000000;")
    vals = np.array(head[1].split(";")[2:], np.float64)
    ref = GF["egemaps_v32k"][0]
    assert np.all(np.abs(vals - ref) <= 1e-4 * (np.abs(ref) + 1e-6))


GMS = np.load(os.path.join(HERE, "golden", "more_summaries.npz"))


@pytest.mark.parametrize("conf,tag", [("egemaps/v01a/eGeMAPSv01a.conf", "eGeMAPSv01a"), ("egemaps/v01b/eGeMAPSv01b.conf", "eGeMAPSv01b"),
                                      ("gemaps/v01a/GeMAPSv01a.conf", "GeMAPSv01a")])
def test_earlier_gemaps_versions_end_to_end(conf, tag):
    """the other shipped members of the GeMAPS family (same graphs as v01b / v02 with fewer parameters) against the reference's row for
    one utterance: every value within 1e-4 of its own magnitude"""
    from opensmile_b200.session import Session
    pcm = mixed_pcm(24000, 16000, seed=3)
    s = Session(os.path.join(REFCONF, conf), options={"csvoutput": "f.csv"}, device=0)
    assert s.element_names() == [str(x) for x in GMS["names_" + tag]]
    rows, fo_ = s.extract_pcm(pcm, np.array([0, pcm.size], np.int64), 16000.0, 1)
    s.close()
    ref = GMS["row_" + tag][0]
    assert rows.shape == (1, len(ref))
    rel = np.abs(rows[0] - ref) / (np.abs(ref) + 1e-6)
    assert rel.max() < 1e-4, (s and None, str(GMS["names_" + tag][int(np.argmax(rel))]), float(rows[0][int(np.argmax(rel))]), float(ref[int(np.argmax(rel))]))
