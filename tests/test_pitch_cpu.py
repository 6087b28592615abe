"""SHS pitch chain (SURVEY.md 8f-1): the CPU restatement (oracle/osm_oracle_pitch.c + the end-of-input lag
model in oracle/oracle.py) against level taps of the UNMODIFIED reference (tests/golden/pitch_goldens.npz,
scripts/make_golden_pitch.py), and the description-only view of the shipped ComParE_2016 configuration."""
import os

import numpy as np
import pytest

from opensmile_b200.synth import mixed_pcm, voiced_pcm
from oracle import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
G = np.load(os.path.join(HERE, "golden", "pitch_goldens.npz"))
SINKS = np.load(os.path.join(HERE, "golden", "lld_sink_files.npz"))

CASES = {
    "v32k": lambda: voiced_pcm(32000, 16000, seed=7),
    "m48k": lambda: mixed_pcm(48000, 16000, seed=2),
    "m30k": lambda: mixed_pcm(30000, 16000, seed=4),
    "m64k": lambda: mixed_pcm(64000, 16000, seed=3),
}


def _rel(a, b):
    sc = np.abs(b).max(axis=0) + 1e-30
    return float((np.abs(a - b) / sc).max())


@pytest.mark.parametrize("case", sorted(CASES))
def test_shs_level(case):
    fe, sc, ps, vc, jc = oracle.compare16_pitch_cfg()
    shs = oracle.pitch_shs(CASES[case](), fe, sc, ps)
    ref = G[case + "_shs"]
    assert shs.shape == ref.shape
    assert np.array_equal(shs[:, 0], ref[:, 0])                 # number of candidates
    assert _rel(shs, ref) < 2e-6


@pytest.mark.parametrize("case", sorted(CASES))
def test_viterbi_selector_jitter_exact_given_inputs(case):
    """Given the reference's own input levels the sequential stages reproduce it bit for bit."""
    fe, sc, ps, vc, jc = oracle.compare16_pitch_cfg()
    vit = oracle.viterbi(G[case + "_shs"], ps, vc)
    assert np.array_equal(vit, G[case + "_vit"])
    sel = oracle.valbased_select(G[case + "_e60"][:, 0], G[case + "_vit"], 0.001)
    assert np.array_equal(sel, G[case + "_sel"])
    jit = oracle.pitch_jitter(CASES[case](), fe, jc, G[case + "_sel"][:, 0])
    assert np.array_equal(jit, G[case + "_jit"])


@pytest.mark.parametrize("case", sorted(CASES))
def test_whole_chain_and_eoi_lag_model(case):
    """PCM -> smoothed level and its onlyInSegments delta, including the rows the reference computes
    while its jitter level lags behind the flushed Viterbi level."""
    pcm = CASES[case]()
    nz, lag = oracle.compare16_pitch(pcm, with_lag=True)
    ref = np.concatenate([G[case + "_sel"], G[case + "_jit"]], axis=1)
    assert nz.shape == ref.shape
    assert _rel(nz, ref) < 2e-6
    sm, de = oracle.compare16_nz_lld(pcm)
    assert sm.shape == G[case + "_nz"].shape and de.shape == G[case + "_nzde"].shape
    assert _rel(sm, G[case + "_nz"]) < 2e-6
    assert _rel(de, G[case + "_nzde"]) < 1e-5
    # the lag model is exact on the reference's own statics
    assert np.array_equal(oracle.sma_nz_lagged(ref, lag, {2, 3, 4, 5}), G[case + "_nz"])
    assert np.array_equal(oracle.delta_segments_lagged(G[case + "_nz"], lag, 2), G[case + "_nzde"])


def test_whole_chain_44k():
    """same graph at 44.1 kHz (FFT 4096: 2049-point spline) against the reference's LLD file"""
    pcm = mixed_pcm(60000, 16000, seed=5)
    sm, de = oracle.compare16_nz_lld(pcm, sample_rate=44100.0)
    ref = G["m60k_44k_lld"]
    R = ref.shape[0]
    sc = np.abs(ref).max(axis=0) + 1e-30
    assert (np.abs(sm[:R] - ref[:, :6]) / sc[:6]).max() < 2e-6
    assert (np.abs(de[:R] - ref[:, 65:71]) / sc[65:71]).max() < 1e-5


def test_whole_chain_stereo():
    from opensmile_b200.synth import stereo_mixed_pcm
    sm, de = oracle.compare16_nz_lld(stereo_mixed_pcm(40000, 16000, seed=9), n_chan=2)
    ref = G["m40k_stereo_lld"]
    R = ref.shape[0]
    sc = np.abs(ref).max(axis=0) + 1e-30
    assert (np.abs(sm[:R] - ref[:, :6]) / sc[:6]).max() < 2e-6
    assert (np.abs(de[:R] - ref[:, 65:71]) / sc[65:71]).max() < 1e-5


def test_lagged_cases_cover_both_lags():
    fe, sc, ps, vc, jc = oracle.compare16_pitch_cfg()
    lags = {c: oracle.viterbi(G[c + "_shs"], ps, vc, with_lag=True)[1] - G[c + "_shs"].shape[0] for c in CASES}
    assert set(lags.values()) >= {-1, -2}, lags


def test_compare16_conf_description():
    """The shipped ComParE_2016.conf opens unchanged (sinks without a file name and the functionals they feed
    stay idle); element names and row counts equal the reference's LLD file."""
    from opensmile_b200.session import Session
    conf = _compare16_conf()
    s = Session(conf, options={"lldcsvoutput": "x.csv"}, device=-1)
    assert list(s.element_names(16000.0, 1)) == [str(x) for x in G["names_lld"]]
    off = s.frame_offsets(np.array([0, 32000, 32000 + 48000, 32000 + 48000 + 960]), 16000.0)
    assert list(np.diff(off)) == [G["v32k_lld"].shape[0], G["m48k_lld"].shape[0], G["short_960_lld"].shape[0]]
    s.close()


@pytest.mark.parametrize("case,seed,n", [("var_m48k", 6, 48000), ("var_m40k", 8, 40000)])
def test_variant_switches(case, seed, n):
    """tests/configs/pitch_variants.conf: non-greedy peak picker, octave correction, forced Viterbi decisions,
    envelope / clipped outputs, every cPitchJitter output incl. the 2.2-compatible threshold, plain smoother
    (the 40 000-sample case ends with a Viterbi lag of 7 frames)"""
    got, lag = oracle.pitch_variants_lld(mixed_pcm(n, 16000, seed=seed))
    ref = G[case + "_lld"]
    assert got.shape == ref.shape
    assert _rel(got, ref) < 1e-5


def test_variant_conf_description():
    from opensmile_b200.session import Session
    s = Session(os.path.join(HERE, "configs", "pitch_variants.conf"), options={"O": "x.htk"}, device=-1)
    assert list(s.element_names(16000.0, 1)) == [str(x) for x in G["names_var"]]
    off = s.frame_offsets(np.array([0, 48000, 88000]), 16000.0)
    assert list(np.diff(off)) == [G["var_m48k_lld"].shape[0], G["var_m40k_lld"].shape[0]]
    s.close()


def _compare16_conf():
    return os.path.join(HERE, "golden", "config", "compare16", "ComParE_2016.conf")


def test_compare16_sink_selection():
    """Which sink is active decides the plan: the LLD sinks read lld;lld_de (130 columns, both give the same
    plan); the summary sinks (-O / -csvoutput) read the concatenation of the six cFunctionals levels: 6373 features on the
    union of their input levels; without any file name there is nothing to compute."""
    from opensmile_b200 import capi
    from opensmile_b200.session import Session, SessionError
    conf = _compare16_conf()
    a = Session(conf, options={"lldcsvoutput": "x.csv"}, device=-1)
    b = Session(conf, options={"lldhtkoutput": "x.htk"}, device=-1)
    assert list(a.element_names(16000.0, 1)) == list(b.element_names(16000.0, 1))
    assert len(a.element_names(16000.0, 1)) == 130
    # the same level at 44.1 kHz: frame geometry changes, names and columns do not
    assert list(a.element_names(44100.0, 1)) == list(a.element_names(16000.0, 1))
    a.close()
    b.close()
    c = Session(conf, options={"lldarffoutput": "x.arff"}, device=-1)      # the LLD ARFF sink reads the same levels
    assert len(c.element_names(16000.0, 1)) == 130
    c.close()
    for opts in ({"csvoutput": "x.csv"}, {"O": "x.arff"}):   # summaries: six cFunctionals instances behind a cVectorConcat
        d = Session(conf, options=opts, device=-1)
        assert len(d.element_names(16000.0, 1)) == 6373
        d.close()
    with pytest.raises(SessionError) as e:               # nothing requested
        Session(conf, device=-1)
    assert "no active sink" in str(e.value)


def test_compare16_component_mapping_and_baseline_geometry():
    """the conf front end hands the pitch chain's sections over with the reference's values
    (ComParE_2016_core.lld.conf.inc:62-190), and BASELINE configs[3]'s shard (125 000 utterances x 3.0 s) has the
    row counts of SURVEY.md 8a' (296 per utterance) -- description only, no device"""
    from opensmile_b200 import capi
    from opensmile_b200.session import Session
    s = Session(_compare16_conf(), options={"lldcsvoutput": "x.csv"}, device=-1)
    comps, level = s.components(16000.0, 1)
    by_type = {}
    for c in comps:
        by_type.setdefault(c.type, []).append(c)
    assert not by_type.get(-1)
    sc = by_type[capi.C_SPECSCALE][0].u.specscale
    assert (sc.scaleOctave, sc.sourceLin, sc.splineInterp, sc.specSmooth, sc.specEnhance, sc.auditoryWeighting) == (1, 1, 1, 1, 1, 1)
    assert (sc.minF, sc.maxF, sc.nPointsTarget) == (25.0, -1.0, 0)
    ps = by_type[capi.C_PITCHSHS][0].u.pitchshs
    assert (ps.nCandidates, ps.greedyPeakAlgo, ps.nHarmonics, ps.F0raw, ps.voicingClip) == (6, 1, 15, 1, 1)
    assert (ps.maxPitch, ps.minPitch) == (620.0, 52.0) and abs(ps.voicingCutoff - 0.7) < 1e-12 and abs(ps.compressionFactor - 0.85) < 1e-12
    vt = by_type[capi.C_PITCHSMOOTHERVITERBI][0].u.pitchsmootherviterbi
    assert (vt.bufferLength, vt.F0final, vt.voicingFinalUnclipped, vt.voicingFinalClipped) == (30, 1, 1, 0)
    assert (vt.wTvv, vt.wTvvd, vt.wTvuv, vt.wThr, vt.wLocal, vt.wRange, vt.wTuu) == (10.0, 5.0, 10.0, 4.0, 2.0, 1.0, 0.0)
    vs = by_type[capi.C_VALBASEDSELECTOR][0]
    assert (vs.u.valbasedselector.idx, vs.u.valbasedselector.removeIdx, vs.u.valbasedselector.zeroVec) == (0, 1, 1)
    assert abs(vs.u.valbasedselector.threshold - 0.001) < 1e-12 and vs.n_inputs == 2
    pj = by_type[capi.C_PITCHJITTER][0].u.pitchjitter
    assert pj.F0reader_dmLevel == b"is13_pitchG60" and pj.F0field == b"F0final"
    assert (pj.jitterLocal, pj.jitterDDP, pj.shimmerLocal, pj.logHNR, pj.useBrokenJitterThresh) == (1, 1, 1, 1, 0)
    assert abs(pj.searchRangeRel - 0.25) < 1e-12
    # functionals and their sinks are not part of the plan
    assert capi.C_VECTORCONCAT in by_type and len(comps) < 50
    n = 1000                                            # (frame_offsets is linear in the number of utterances)
    off = np.arange(n + 1, dtype=np.int64) * 48000
    fo = s.frame_offsets(off, 16000.0)
    assert int(fo[-1]) == 296 * n and set(np.diff(fo)) == {296}
    s.close()


def test_one_pass_cross_correlation_matches_the_two_pass_form():
    """jitter_kernel evaluates the normalised cross correlation of a candidate period in its one-pass form
    (window sums from prefix sums, DESIGN.md 3.5); the reference's two-pass loop (lld/pitchJitter.cpp:339-413)
    gives the same value to ~1e-15 and the same peak decision on every window tried"""
    rng = np.random.default_rng(0)

    def two_pass(x, y):
        n = len(x)
        mx = my = 0.0
        for a, b in zip(x, y):
            mx += float(a)
            my += float(b)
        mx /= n
        my /= n
        cc = nx = ny = 0.0
        for a, b in zip(x, y):
            dx, dy = float(a) - mx, float(b) - my
            cc += dx * dy
            nx += dx * dx
            ny += dy * dy
        return cc / (np.sqrt(nx) * np.sqrt(ny))

    def one_pass(w, tf):
        x, y = w[:tf].astype(np.float64), w[tf:2 * tf].astype(np.float64)
        n = float(tf)
        sx, sy = x.sum(), y.sum()
        return ((x * y).sum() - sx * sy / n) / (np.sqrt((x * x).sum() - sx * sx / n) * np.sqrt((y * y).sum() - sy * sy / n))

    def pick(c):
        best, mx = -1, None
        for i in range(1, len(c) - 2):
            if c[i - 1] < c[i] and c[i] > c[i + 1] and (best == -1 or c[i] > mx):
                best, mx = i, c[i]
        return best

    worst, n_win = 0.0, 0
    for seed in range(4):
        pcm = (mixed_pcm(24000, 16000, seed=seed) if seed % 2 else voiced_pcm(24000, 16000, seed=seed)).astype(np.float32) / np.float32(32767.0)
        for _ in range(12):
            start, tf0 = int(rng.integers(0, 22000)), int(rng.integers(60, 300))
            tmin, tmax = int(0.75 * tf0), int(np.ceil(1.25 * tf0))
            if start + 2 * tmax + 1 >= len(pcm):
                continue
            w = pcm[start:]
            a = np.array([two_pass(w[:tf], w[tf:2 * tf]) for tf in range(tmin, tmax + 1)])
            b = np.array([one_pass(w, tf) for tf in range(tmin, tmax + 1)])
            ok = np.isfinite(a) & np.isfinite(b)
            worst = max(worst, float(np.abs(a[ok] - b[ok]).max()))
            assert pick(a) == pick(b)
            n_win += 1
    assert n_win > 30 and worst < 1e-12


def test_compare16_lld_csv_file_is_byte_identical():
    """cCsvSink file of the lld;lld_de reader (instance name, frameTime, 130 values per row): written from the
    reference's rows it equals the reference's file byte for byte -- including the last row, which a window
    processor appended at the end of input and which repeats the time stamp of the last real frame"""
    import tempfile
    from opensmile_b200 import Plan, write_csv
    from opensmile_b200.session import Session
    s = Session(_compare16_conf(), options={"lldcsvoutput": "x.csv"}, device=-1)
    comps, level = s.components(16000.0, 1)
    p = Plan(list(comps), level, device=-1)
    assert (p.num_frames(32000), p.num_time_frames(32000)) == (196, 195)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "lld.csv")
        write_csv(path, G["v32k_lld"], [str(x) for x in G["names_lld"]], 0.01, instance_name="utt7", frame_index=False,
                  frame_time=True, n_time_frames=p.num_time_frames(32000))
        assert open(path, "rb").read() == SINKS["v32k_lld_csv"].tobytes()
    p.close()
    s.close()


def test_compare16_lld_arff_file_is_byte_identical(tmp_path):
    """cArffSink file of the LLD reader (-lldarffoutput, -instname utt7; relation, attributes, the class attribute of
    the included targets file, %e values, '?' target): written from the reference's rows it equals the reference's
    file byte for byte; with append=1 a second call adds rows without repeating the header (iocore/arffSink.cpp:244-256)"""
    from opensmile_b200 import write_arff
    names = [str(x) for x in G["names_lld"]]
    p = tmp_path / "lld.arff"
    write_arff(p, G["v32k_lld"], names, 0.01, relation="openSMILE_features", instance_name="utt7", frame_index=False,
               frame_time=True, classes=(("class", "numeric", "?"),), n_time_frames=195)
    ref = SINKS["v32k_lld_arff"].tobytes()
    assert p.read_bytes() == ref
    write_arff(p, G["v32k_lld"][:3], names, 0.01, relation="openSMILE_features", instance_name="utt8", frame_index=False,
               frame_time=True, classes=(("class", "numeric", "?"),), append=True)
    lines = p.read_bytes().split(b"\n")
    assert lines[: len(ref.split(b"\n")) - 1] == ref.split(b"\n")[:-1] and lines[-2].startswith(b"utt8,0.020000,") and lines.count(b"@data") == 1


def test_compare16_sink_options_from_the_configuration():
    """formatting options of the active sinks as the session took them from the shipped configuration: CSV without
    frame index, instance name from -instname; ARFF relation / class attribute / target of the included targets file
    (config/shared/arff_targets.conf.inc) incl. its command line options, append = 1 for the LLD ARFF sink"""
    from opensmile_b200.session import Session
    conf = _compare16_conf()
    s = Session(conf, options={"lldcsvoutput": "x.csv", "lldarffoutput": "x.arff", "lldhtkoutput": "x.htk", "instname": "utt7"}, device=-1)
    o = s.sink_options().splitlines()
    assert o[0] == "csv: header=1 time=1 index=0 name=1:'utt7' delim=;"
    assert o[1] == "htk: parmKind=9"
    assert o[2] == "arff: relation='openSMILE_features' time=1 index=0 name=1:'utt7' append=1 dummy=1 classes=class:numeric:?"
    s.close()
    s = Session(conf, options={"lldarffoutput": "x.arff", "class": "happy", "classtype": "{happy,sad}", "relation": "my set"}, device=-1)
    assert s.sink_options().splitlines()[2] == "arff: relation='my set' time=1 index=0 name=1:'unknown' append=1 dummy=1 classes=class:{happy,sad}:happy"
    s.close()
