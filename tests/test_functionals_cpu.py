"""cFunctionals (SURVEY.md 8f-3): the CPU restatement (oracle/functionals_oracle.py) against rows of the UNMODIFIED reference
(tests/golden/functionals_goldens.npz, scripts/make_golden_functionals.py), and the host side of the product -- the shipped
config/is09-13/IS09_emotion.conf (384 features) and tests/configs/func_variants.conf open unchanged with the reference's element
names; functionals the GPU path does not implement are refused loudly."""
import os

import numpy as np
import pytest

from oracle import functionals_oracle as fo

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REFCONF = os.path.join(HERE, "golden", "config")
G = np.load(os.path.join(HERE, "golden", "functionals_goldens.npz"))
G2 = np.load(os.path.join(HERE, "golden", "functionals_goldens2.npz"))
S, SEC, FR = fo.SEGMENT, fo.SECOND, fo.FRAME

SPEC_A = fo.Spec(["Means"], master_norm=SEC, means=dict(flatness=1, posamean=1, negamean=1, posqmean=1, posrqmean=1, negqmean=1, negrqmean=1,
                                                            rqmean=1, nzrqmean=1))
SPEC_B = fo.Spec(["Percentiles", "Moments", "Extremes"], non_zero=1, master_norm=S,
                 percentiles=dict(quartile1=1, quartile2=1, quartile3=1, iqr12=1, iqr23=1, iqr13=1, percentile=[0.2, 0.5, 0.8], pctlrange=[(0, 2)], interp=1),
                 moments=dict(variance=1, stddev=0, skewness=0, kurtosis=0, amean=1, stddevNorm=2),
                 extremes=dict(max=0, min=0, range=1, maxpos=1, minpos=1, amean=0, maxameandist=1, minameandist=1))
SPEC_C = fo.Spec(["Regression", "Percentiles", "Means"], non_zero=2, name_append="x",
                 regression=dict(centroidNorm=SEC, centroidUseAbsValues=1, centroidRatioLimit=0, normRegCoeff=1, normInputs=1, oldBuggyQerr=0),
                 percentiles=dict(quartile1=1, quartile2=1, quartile3=1, interp=0),
                 means=dict(amean=1, absmean=0, qmean=0, nzamean=0, nzabsmean=0, nzqmean=0, nzgmean=0, nnz=1, norm=S, norm_set=True))
# second set (tests/configs/func_variants2.conf): the Times / Lpc / Segments / Peaks2 option sets of the shipped ComParE_2016 and
# GeMAPS functionals blocks
_CMP_PEAKS = ["meanPeakDist", "peakDistStddev", "peakRangeAbs", "peakRangeRel", "peakMeanAbs", "peakMeanMeanDist", "peakMeanRel", "minRangeRel",
              "meanRisingSlope", "stddevRisingSlope", "meanFallingSlope", "stddevFallingSlope"]
SPEC_D = fo.Spec(["Extremes", "Segments", "Times", "Lpc"], master_norm=S,
                 extremes=dict(max=0, min=0, range=1, maxpos=1, minpos=1, amean=0, maxameandist=0, minameandist=0),
                 segments=dict(maxNumSeg=100, segmentationAlgorithm="relTh", thresholds=[0.25, 0.75], meanSegLen=1, maxSegLen=1, minSegLen=1,
                               segLenStddev=1, norm=SEC, norm_set=True),
                 times=dict(downleveltime25=0, downleveltime50=0, downleveltime75=0, downleveltime90=0, falltime=0, rightctime=0, duration=0,
                            buggySecNorm=0, norm=S, norm_set=True),
                 lpc=dict(lpGain=1, lpc=1, firstCoeff=0, order=5))
SPEC_E = fo.Spec(["Means", "Segments", "Peaks2"], master_norm=S,
                 means=dict(amean=0, absmean=0, qmean=0, nzamean=0, nzabsmean=0, nzqmean=0, nzgmean=0, nnz=1, norm=S, norm_set=True),
                 segments=dict(maxNumSeg=100, segmentationAlgorithm="nonX", X=0.0, numSegments=1, meanSegLen=1, maxSegLen=1, minSegLen=1,
                               segLenStddev=1, norm=SEC, norm_set=True),
                 peaks2=dict(numPeaks=1, norm=SEC, norm_set=True, relThresh=0.1))
SPEC_F = fo.Spec(["Peaks2", "Times"], master_norm=SEC, peaks2=dict({k: 1 for k in _CMP_PEAKS}, norm=SEC, norm_set=True, relThresh=0.1, doRatioLimit=1),
                 times=dict(norm=SEC, norm_set=True))
SPEC_G = fo.Spec(["Segments", "Peaks2", "Times"], master_norm=SEC, name_append="g",
                 segments=dict(maxNumSeg=1000, segmentationAlgorithm="eqX", X=0.0, numSegments=1, meanSegLen=1, segLenStddev=1, norm=SEC, norm_set=True),
                 peaks2=dict({k: 1 for k in fo.PEAKS2_NAMES}, norm=FR, norm_set=True, relThresh=0.35, dynRelThresh=1, doRatioLimit=0),
                 times=dict(norm=FR, norm_set=True, buggySecNorm=0))
SPEC_H = fo.Spec(["Regression", "Moments"], master_norm=S,
                 regression=dict(linregerrA=0, qregerrA=0, centroid=1, centroidUseAbsValues=1, centroidRatioLimit=1, normRegCoeff=2, normInputs=1,
                                 oldBuggyQerr=0, doRatioLimit=1),
                 moments=dict(variance=0, stddev=1, skewness=0, kurtosis=0, amean=0, stddevNorm=1, doRatioLimit=1))
# tests/configs/func_variants3.conf: Onset / Peaks / Crossings
SPEC_I = fo.Spec(["Onset", "Times", "Peaks", "Crossings"], name_append="Turn",
                 onset=dict(threshold=0.0, thresholdOnset=0.0, thresholdOffset=0.0, numOnsets=1),
                 times=dict({k: 0 for k in fo.TIMES_NAMES}, duration=1, norm=SEC, norm_set=True), peaks=dict(), crossings=dict())
SPEC_J = fo.Spec(["Crossings", "Peaks", "Onset", "Segments"], master_norm=SEC,
                 segments=dict(maxNumSeg=100, segmentationAlgorithm="NArelTh", thresholds=[0.25, 0.5, 0.75], numSegments=1, meanSegLen=1, maxSegLen=1,
                               minSegLen=1, segLenStddev=1),
                 onset=dict(threshold=0.05, thresholdOffset=0.01, useAbsVal=1, onsetPos=1, offsetPos=1, numOnsets=1, numOffsets=1, onsetRate=1),
                 peaks=dict(peakDistStddev=1), crossings=dict(amean=1))
SPEC_K = fo.Spec(["Peaks", "Onset", "Crossings"], non_zero=1, master_norm=SEC,
                 onset=dict(threshold=0.2, onsetPos=1, offsetPos=1, numOnsets=1, onsetRate=1, norm=FR, norm_set=True),
                 peaks=dict(peakMean=0, peakMeanMeanDist=0, peakDistStddev=1, norm=S, norm_set=True), crossings=dict(zcr=0, mcr=1, amean=1))
SPEC_L = fo.Spec(["Samples", "Moments", "DCT"], samples=dict(samplepos=[0, 0.1, 0.33, 0.5, 0.999, 1.0, 1.0]),
                 moments=dict(variance=0, stddev=1, skewness=0, kurtosis=0, amean=0), dct=dict(firstCoeff=0, lastCoeff=8))
LEVELS3 = [("I", SPEC_I, slice(0, 32), -2), ("J", SPEC_J, slice(0, 16), 0), ("K", SPEC_K, slice(0, 16), 0), ("L", SPEC_L, slice(0, 16), 0)]
G3 = np.load(os.path.join(HERE, "golden", "functionals_goldens3.npz"))
LEVELS2 = [("D", SPEC_D, slice(0, 32), -2), ("E", SPEC_E, slice(0, 16), 0), ("F", SPEC_F, slice(0, 32), -2), ("G", SPEC_G, slice(0, 16), 0),
           ("H", SPEC_H, slice(0, 32), -2)]

# (tag, spec, columns of the 32-column lld;lld_de level, frames the functionals see relative to T = static frames)
LEVELS = [("is09", fo.IS09, slice(0, 32), -2, "is09_func"), ("A", SPEC_A, slice(0, 32), -2, "varA"), ("B", SPEC_B, slice(0, 16), 0, "varB"),
          ("C", SPEC_C, slice(16, 32), -2, "varC")]


def contour_rows(lld, dn):
    """the rows a full-input reader sees when it first ticks at end of input (graph.cpp:desc_num_frames_first_eoi): the smoothed
    level (T + 1 rows in the end) holds T rows then, the delta level behind it T - 2"""
    T = lld.shape[0] - 1                      # the lld;lld_de sink level has T + 1 rows
    return lld[:T + dn]


@pytest.mark.parametrize("key", ["m24k", "v32k", "rec"])
def test_oracle_reproduces_the_reference_rows(key):
    lld = G["is09_lld_" + key]
    names = list(G["is09_lld_names"])
    for tag, spec, cols, dn, gk in LEVELS:
        got = fo.functionals(spec, contour_rows(lld, dn)[:, cols], 0.01)
        ref = G["%s_%s" % (gk, key)][0]
        assert fo.element_names(spec, names[cols]) == list(G["is09_func_names"] if tag == "is09" else G[gk + "_names"])
        # the reference's CSV prints 7 significant digits
        assert np.all(np.abs(got - ref) <= 1e-6 * np.abs(ref) + 1e-12), tag


@pytest.mark.parametrize("key", ["m24k", "v32k", "rec"])
def test_oracle_reproduces_the_reference_rows_times_lpc_segments_peaks2(key):
    lld = G["is09_lld_" + key]
    names = list(G["is09_lld_names"])
    for tag, spec, cols, dn in LEVELS2:
        got = fo.functionals(spec, contour_rows(lld, dn)[:, cols], 0.01)
        ref = G2["var%s_%s" % (tag, key)][0]
        assert fo.element_names(spec, names[cols]) == list(G2["var%s_names" % tag])
        assert np.all(np.abs(got - ref) <= 1e-6 * np.abs(ref) + 1e-12), tag


@pytest.mark.parametrize("key", ["m24k", "v32k", "rec"])
def test_oracle_reproduces_the_reference_rows_onset_peaks_crossings(key):
    lld = G["is09_lld_" + key]
    names = list(G["is09_lld_names"])
    for tag, spec, cols, dn in LEVELS3:
        got = fo.functionals(spec, contour_rows(lld, dn)[:, cols], 0.01)
        ref = G3["var%s_%s" % (tag, key)][0]
        assert fo.element_names(spec, names[cols]) == list(G3["var%s_names" % tag])
        assert np.all(np.abs(got - ref) <= 1e-6 * np.abs(ref) + 1e-12), (tag, [(n, a, b) for n, a, b in zip(G3["var%s_names" % tag], got, ref) if abs(a - b) > 1e-6 * abs(b) + 1e-12][:5])


def to_c_spec(spec):
    """oracle Spec -> ctypes mirror of osm_b200_functionals_spec"""
    from opensmile_b200 import functionals as F
    norm = lambda d: dict(norm=d["norm"], normIsSet=int(d["norm_set"]))
    sub = {}
    sub["extremes"] = {k: v for k, v in spec.extremes.items() if k not in ("norm", "norm_set")} | norm(spec.extremes)
    sub["means"] = {k: v for k, v in spec.means.items() if k not in ("norm", "norm_set")} | norm(spec.means)
    sub["moments"] = dict(spec.moments)
    sub["percentiles"] = dict(spec.percentiles)
    sub["regression"] = dict(spec.regression)
    sub["times"] = {k: v for k, v in spec.times.items() if k not in ("norm", "norm_set")} | norm(spec.times)
    sub["lpc"] = dict(spec.lpc)
    g = spec.segments
    sub["segments"] = dict(numSegments=g["numSegments"], meanSegLen=g["meanSegLen"], maxSegLen=g["maxSegLen"], minSegLen=g["minSegLen"],
                           segLenStddev=g["segLenStddev"], maxNumSeg=g["maxNumSeg"], X=g["X"], XisRel=g["XisRel"], segMinLng=g["segMinLng"],
                           segMinLngIsSet=int(g["segMinLng_set"]), pauseMinLng=g["pauseMinLng"], **norm(g))
    if g["segmentationAlgorithm"] in F.SEG_BY_NAME:
        sub["segments"]["segmentationAlgorithm"] = g["segmentationAlgorithm"]
        sub["segments"]["thresholds"] = list(g["thresholds"])
    c = spec.peaks2
    sub["peaks2"] = {k: c[k] for k in fo.PEAKS2_NAMES} | dict(relThresh=c["relThresh"], dynRelThresh=c["dynRelThresh"], doRatioLimit=c["doRatioLimit"],
                                                              useAbsThresh=int(c["absThresh"] is not None), absThresh=c["absThresh"] or 0.0, **norm(c))
    o = spec.onset
    sub["onset"] = dict(onsetPos=o["onsetPos"], offsetPos=o["offsetPos"], numOnsets=o["numOnsets"], numOffsets=o["numOffsets"], onsetRate=o["onsetRate"],
                        thresholdOnset=o["threshold"] if o["thresholdOnset"] is None else o["thresholdOnset"],
                        thresholdOffset=o["threshold"] if o["thresholdOffset"] is None else o["thresholdOffset"], useAbsVal=o["useAbsVal"], **norm(o))
    sub["peaks"] = {k: spec.peaks[k] for k in fo.PEAKS_NAMES} | norm(spec.peaks)
    sub["crossings"] = dict(spec.crossings)
    sub["samples"] = dict(samplepos=[float(x) for x in spec.samples["samplepos"]])
    sub["dct"] = dict(spec.dct)
    return F.spec(spec.enabled, non_zero=spec.non_zero, master_norm=-1 if spec.master_norm is None else spec.master_norm,
                  name_append=spec.name_append or "", **sub)


def test_device_statements_of_the_sequential_functionals_on_the_host():
    """opensmile_b200/csrc/functionals_seq.cuh compiled for the host: bit-identical to the oracle on the reference's contours and on
    random ones (zigzags, plateaus, constant and very short contours)"""
    import functionals_harness as fh
    rng = np.random.RandomState(5)
    contours = [G["is09_lld_rec"][:-1, c] for c in range(16)]
    contours += [np.cumsum(rng.randn(n)).astype(np.float32) for n in (5, 6, 9, 40, 300, 1200)]
    contours += [np.round(rng.rand(200) * 4).astype(np.float32), np.zeros(50, np.float32), np.ones(7, np.float32),
                 (rng.rand(300) > 0.5).astype(np.float32) * rng.rand(300).astype(np.float32), np.array([1, 3, 2, 4, 1, 5, 0, 6, 2, 7, 1], np.float32)]
    for spec in (SPEC_D, SPEC_E, SPEC_F, SPEC_G):
        cs = to_c_spec(spec)
        for x in contours:
            mn, mx = np.float32(x.min()), np.float32(x.max())
            mean = np.float32(x.astype(np.float64).sum() / len(x))
            if "Segments" in spec.enabled:
                nrm = fo._norm(spec.segments["norm"], spec.segments["norm_set"], spec.master_norm)
                assert np.array_equal(fh.segments(cs, x, 0.01, nrm), np.array(fo._segments(spec, x, mn, mx, mean, 0.01), np.float32))
            if "Peaks2" in spec.enabled:
                nrm = fo._norm(spec.peaks2["norm"], spec.peaks2["norm_set"], spec.master_norm)
                a, b = fh.peaks2(cs, x, 0.01, nrm), np.array(fo._peaks2(spec, x, mn, mx, mean, 0.01), np.float32)
                assert np.array_equal(a, b, equal_nan=True), (a, b)
            if "Lpc" in spec.enabled:
                a, b = fh.lpc(cs, x), np.array(fo._lpc(spec, x), np.float32)
                assert np.array_equal(a, b, equal_nan=True), (a, b)
    for spec in (SPEC_I, SPEC_J, SPEC_K):
        cs = to_c_spec(spec)
        for x in contours:
            nrm = fo._norm(spec.onset["norm"], spec.onset["norm_set"], spec.master_norm)
            a, b = fh.onset(cs, x, 0.01, nrm), np.array(fo._onset(spec, x, 0.01), np.float32)
            assert np.array_equal(a, b, equal_nan=True), (a, b)
            nrm = fo._norm(spec.peaks["norm"], spec.peaks["norm_set"], spec.master_norm)
            a, b = fh.peaks(cs, x, 0.01, nrm), np.array(fo._peaks_old(spec, x, 0.01), np.float32)
            assert np.array_equal(a, b, equal_nan=True), (a, b)
            a, b = fh.crossings(cs, x), np.array(fo._crossings(spec, x), np.float32)
            assert np.array_equal(a, b, equal_nan=True), (a, b)


def test_zero_and_single_value_contours():
    spec = fo.Spec(["Extremes", "Moments", "Regression", "Percentiles"], non_zero=1, percentiles=dict(quartile2=1),
                   regression=dict(centroid=0))
    assert not np.any(fo.functionals(spec, np.zeros((20, 2), np.float32), 0.01))        # nothing survives the filter: zero fill
    x = np.zeros((9, 1), np.float32); x[4] = 3.5
    v = dict(zip(fo.value_names(spec), fo.functionals(spec, x, 0.01)))
    assert v["max"] == v["min"] == v["quartile2"] == v["linregc2"] == np.float32(3.5) and v["linregc1"] == 0 and v["stddev"] == 0 and v["maxPos"] == 0


def _session(conf, opts):
    from opensmile_b200.session import Session
    return Session(conf, options=opts, device=-1)


def test_shipped_is09_configuration_opens_unchanged():
    s = _session(os.path.join(REFCONF, "is09-13", "IS09_emotion.conf"), {"csvoutput": "f.csv"})
    assert s.element_names() == list(G["is09_func_names"])                              # 384 features, the reference's header
    # one summary row per utterance with at least one frame
    fo_ = s.frame_offsets(np.array([0, 24000, 24100, 24100 + 32000, 24100 + 32000 + 400], np.int64), 16000.0, 1)
    assert list(fo_) == [0, 1, 1, 2, 3]
    s.close()
    s = _session(os.path.join(REFCONF, "is09-13", "IS09_emotion.conf"), {"lldcsvoutput": "l.csv"})   # the LLD sinks still work
    assert s.element_names() == list(G["is09_lld_names"])
    s.close()


def test_variant_configuration_names(tmp_path):
    conf = tmp_path / "v.conf"
    conf.write_text(open(os.path.join(HERE, "configs", "func_variants.conf")).read().replace("REFCONF", REFCONF))
    for opt, key in (("outA", "varA"), ("outB", "varB"), ("outC", "varC")):
        s = _session(str(conf), {opt: "x.csv"})
        assert s.element_names() == list(G[key + "_names"])
        s.close()


def test_second_variant_configuration_names(tmp_path):
    conf = tmp_path / "v.conf"
    conf.write_text(open(os.path.join(HERE, "configs", "func_variants2.conf")).read().replace("REFCONF", REFCONF))
    for lv in "DEFGH":
        s = _session(str(conf), {"out" + lv: "x.csv"})
        assert s.element_names() == list(G2["var%s_names" % lv])
        s.close()


def test_unimplemented_functionals_are_refused_loudly(tmp_path):
    from opensmile_b200.session import SessionError
    from opensmile_b200 import capi
    txt = open(os.path.join(HERE, "configs", "func_variants.conf")).read().replace("REFCONF", REFCONF)
    bad = tmp_path / "bad.conf"
    bad.write_text(txt.replace("functionalsEnabled = Means\n", "functionalsEnabled = Means ; Modulation\n"))
    with pytest.raises(SessionError) as e:
        _session(str(bad), {"outA": "x.csv"})
    assert e.value.status == capi.ERR_UNSUPPORTED and "cFunctionalModulation" in str(e.value)
    bad.write_text(txt.replace("nonZeroFuncts = 0\n", "nonZeroFuncts = 0\nbogusField = 1\n"))
    with pytest.raises(SessionError) as e:
        _session(str(bad), {"outA": "x.csv"})
    assert "bogusField" in str(e.value)
    # glue the summary graphs do not use stays refused: another cVectorOperation behind the functionals, a concat that drops the fields
    ege = open(os.path.join(REFCONF, "egemaps", "v02", "eGeMAPSv02.conf")).read()
    for a, b, needle in (("includeSingleElementFields = 1\n\n\\{../../shared/standard_data_output_no_lld_de", "includeSingleElementFields = 0\n\n\\{../../shared/standard_data_output_no_lld_de", "drops single-element fields"),):
        assert a in ege
        d = tmp_path / "egemaps" / "v02"
        d.mkdir(parents=True, exist_ok=True)
        (d / "bad.conf").write_text(ege.replace(a, b).replace("\\{../../", "\\{" + REFCONF + "/").replace("\\{eGeMAPSv02_core", "\\{" + REFCONF + "/egemaps/v02/eGeMAPSv02_core"))
        with pytest.raises(SessionError) as e:
            _session(str(d / "bad.conf"), {"csvoutput": "x.csv"})
        assert e.value.status == capi.ERR_UNSUPPORTED and needle in str(e.value)


GGF = np.load(os.path.join(HERE, "golden", "gemaps_func.npz"))


@pytest.mark.parametrize("conf,tag", [("egemaps/v02/eGeMAPSv02.conf", "egemaps"), ("gemaps/v01b/GeMAPSv01b.conf", "gemaps")])
def test_gemaps_summary_names(conf, tag):
    """the shipped GeMAPS / eGeMAPS files open unchanged with -csvoutput: cVectorConcat / cDataSelector (newNames) / cVectorOperation
    (dBp) behind eight cFunctionals instances, cValbasedSelector gates in front of them -- the reference's 62 / 88 names"""
    s = _session(os.path.join(REFCONF, conf), {"csvoutput": "x.csv"})
    assert s.element_names() == [str(x) for x in GGF["names_" + tag]]
    s.close()


def test_spec_mirror_and_descriptions():
    from opensmile_b200 import functionals as F
    sp = F.spec(["Extremes", "Regression", "Moments"], extremes=dict(amean=1, maxameandist=0, minameandist=0, norm=2, normIsSet=1),
                regression=dict(linregerrA=0, qregc1=0, qregc2=0, qregc3=0, qregerrA=0, qregerrQ=0, centroid=0), moments=dict(variance=0))
    f = F.Functionals(sp, list(G["is09_lld_names"]), 0.01, device=-1)
    assert f.num_values == 12 and f.element_names() == list(G["is09_func_names"])
    with pytest.raises(RuntimeError):                                                   # description-only objects never compute
        f.run_host(np.zeros((4, 32), np.float32), [0], [4])
    f.close()


def test_gemaps_summary_oracle_on_the_reference_levels():
    """oracle/gemaps_summary_oracle.py (eight cFunctionals instances + cDataSelector renaming + dBp) on the reference's own dumps of the
    seven input levels reproduces the reference's 88-value eGeMAPSv02 row.  The rows every instance sees at the first end-of-input
    tick (graph.cpp:desc_num_frames_first_eoi): static level T, smoothed level T (of T + 1), levels behind the Viterbi smoother V =
    143 / 193 / 198 -- the same lags the ComParE_2016 rows pin (tests/golden/compare16_func.npz)."""
    from oracle import gemaps_summary_oracle as go
    GL = np.load(os.path.join(HERE, "golden", "gemaps_func_levels.npz"))
    lvls = sorted({k.split("_", 1)[1] for k in GL.files if not k.startswith("names_")})
    names = {l: [str(x) for x in GL["names_" + l]] for l in lvls}
    for key, V in (("m24k", 143), ("v32k", 193), ("rec", 198)):
        lv = {}
        for l in lvls:
            full = GL["%s_%s" % (key, l)]
            if l.endswith("energyRMS"): n = len(full)
            elif l in ("gemapsv01b_loudness_smo", "egemapsv02_lldSetNoF0AndLoudnessZ_smo"): n = len(full) - 1
            else: n = min(V, len(full))
            lv[l] = full[:n]
        nm, val = go.egemaps_summary(lv, names)
        ref = GGF["egemaps_" + key][0]
        assert nm == [str(x) for x in GGF["names_egemaps"]]
        rel = np.abs(val - ref) / (np.abs(ref) + 1e-6)
        assert rel.max() < 2e-5, (key, nm[int(np.argmax(rel))], float(rel.max()))   # the CSV rows carry 7 significant digits


def test_valbased_gate_oracle_on_the_reference_levels():
    """the voiced / unvoiced gates (other/valbasedSelector.cpp:195-233): in the reference's dumps a frame of the smoothed F0 level that
    is zero together with its neighbours has all-zero voiced parameters; the unvoiced spectral parameters are zero where F0 and its
    neighbours are voiced -- the gate oracle on the F0 contour predicts both supports"""
    from oracle import gemaps_summary_oracle as go
    GL = np.load(os.path.join(HERE, "golden", "gemaps_func_levels.npz"))
    for key in ("m24k", "v32k", "rec"):
        f0 = GL[key + "_gemapsv01b_lld_single_logF0_smo"][:, 0]
        snz = GL[key + "_egemapsv02_lldSetSpectralNz_smo"]
        sz = GL[key + "_egemapsv02_lldSetSpectralZ_smo"]
        n = min(len(f0), len(snz), len(sz))
        voiced = go.valbased_gate(f0[:n], np.ones((n, 1), np.float32))[:, 0] > 0          # smoothed F0 > 0 <=> raw F0 > 0 (noZeroSma)
        assert np.all(snz[:n][~voiced] == 0) and np.all(sz[:n][voiced] == 0)
        inv = go.valbased_gate(f0[:n], np.ones((n, 1), np.float32), invert=True)[:, 0] > 0
        assert np.array_equal(inv, ~voiced)


def _csv_close(got_text, ref_text, rtol):
    """same header line, same row prefix (instance name ; time stamp), values equal within rtol of their magnitude"""
    g, r = got_text.strip().split("\n"), ref_text.strip().split("\n")
    assert g[0] == r[0] and len(g) == len(r)
    for a, b in zip(g[1:], r[1:]):
        fa, fb = a.split(";"), b.split(";")
        assert fa[:2] == fb[:2] and len(fa) == len(fb)
        va, vb = np.array(fa[2:], np.float64), np.array(fb[2:], np.float64)
        assert np.all(np.abs(va - vb) <= rtol * (np.abs(vb) + 1e-6)), (a[:80], b[:80])


def test_summary_rows_are_written_like_the_reference_sink(tmp_path):
    """osm_b200_session_write_files on a cFunctionals session: the sink's file has the summary's names, one row per input,
    `'unknown';0.000000;values` -- the reference's file for the same input (the values here are the reference's own, re-printed)"""
    s = _session(os.path.join(REFCONF, "egemaps", "v02", "eGeMAPSv02.conf"), {"csvoutput": "x.csv"})
    out = tmp_path / "f.csv"
    s.write_files(GGF["egemaps_m24k"], [0, 1], 16000.0, 1, n_samples=[24000], csv_paths=[str(out)])
    s.close()
    _csv_close(out.read_text(), GGF["csv_egemaps_m24k"].tobytes().decode(), 2e-7)


GMS = np.load(os.path.join(HERE, "golden", "more_summaries.npz"))
MORE = [("is09-13/IS12_speaker_trait.conf", "IS12_speaker_trait", 5757), ("is09-13/IS13_ComParE.conf", "IS13_ComParE", 6373),
        ("egemaps/v01a/eGeMAPSv01a.conf", "eGeMAPSv01a", 88), ("egemaps/v01b/eGeMAPSv01b.conf", "eGeMAPSv01b", 88),
        ("gemaps/v01a/GeMAPSv01a.conf", "GeMAPSv01a", 62)]


@pytest.mark.parametrize("conf,tag,n", MORE)
def test_more_shipped_summary_configurations_open_with_the_reference_names(conf, tag, n):
    s = _session(os.path.join(REFCONF, conf), {"csvoutput": "x.csv"})
    assert s.element_names() == [str(x) for x in GMS["names_" + tag]] and len(s.element_names()) == n
    s.close()


def test_sub_window_functionals_are_refused(tmp_path):
    """the reference's default frameMode is "fixed": a cFunctionals section without frameMode = full summarises sub-windows (the
    MediaEval configurations: frameSize = 2.0) -- refused by name instead of silently summarising the whole input"""
    from opensmile_b200.session import SessionError
    from opensmile_b200 import capi
    txt = open(os.path.join(HERE, "configs", "func_variants.conf")).read().replace("REFCONF", REFCONF)
    inc = "\\{REFCONF/shared/FrameModeFunctionals.conf.inc}".replace("REFCONF", REFCONF)
    assert inc in txt
    bad = tmp_path / "sub.conf"
    bad.write_text(txt.replace(inc, "frameSize = 2.0\nframeStep = 2.0"))
    with pytest.raises(SessionError) as e:
        _session(str(bad), {"outA": "x.csv"})
    assert e.value.status == capi.ERR_UNSUPPORTED and "frameMode = fixed" in str(e.value)
    # EOIlevel > 0 would let the summary see the rows the window processors append in later end-of-input passes
    bad.write_text(txt.replace("functionalsEnabled = Means\n", "functionalsEnabled = Means\nEOIlevel = 1\n"))
    with pytest.raises(SessionError) as e:
        _session(str(bad), {"outA": "x.csv"})
    assert e.value.status == capi.ERR_UNSUPPORTED and "EOIlevel" in str(e.value)
