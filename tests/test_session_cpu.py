"""CPU tests of the host front end (include/osm_b200_host.h): the reference's .conf syntax is parsed
into the same component graph, element names and frame counts as the reference produces (golden
vectors from the unmodified reference, scripts/make_golden_conf.py), and the HTK / CSV writers are
byte-identical to the reference's sinks.  Description-only sessions (device = -1): no compute."""
import os

import numpy as np
import pytest

from conftest import ROOT
from opensmile_b200 import Session, SessionError, capi, write_csv, write_htk

CONF = os.path.join(ROOT, "tests", "configs")
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "conf_goldens.npz"))
REF_CONF = os.path.join(ROOT, "tests", "golden", "config")


@pytest.mark.parametrize("conf,key", [("lld_mix.conf", "mix"), ("mfcc_e_d_a.conf", "mfcc_e"), ("plp_e_d_a.conf", "plp_e"),
                                      ("compare_ns.conf", "cmp_ns"), ("gemaps_ns.conf", "gemaps_ns"),
                                      ("mfcc_0_d_a_z.conf", "mfcc_z")])
def test_element_names_match_reference_csv_header(conf, key):
    s = Session(os.path.join(CONF, conf), device=-1)
    assert s.element_names(16000, 1) == [str(x) for x in GOLD["names_" + key]]


def test_frame_counts_match_reference():
    s = Session(os.path.join(CONF, "mfcc_e_d_a.conf"), device=-1)
    lens = [12000, 400, 560, 720, 880, 399, 0]
    off = np.concatenate([[0], np.cumsum(lens)])
    fo = s.frame_offsets(off, 16000, 1)
    want = [GOLD["mfcc_e"].shape[0]] + [GOLD["mfcc_e_short_%d" % n].shape[0] for n in (400, 560, 720, 880)] + [0, 0]
    assert list(np.diff(fo)) == want
    m = Session(os.path.join(CONF, "lld_mix.conf"), device=-1)
    assert m.frame_offsets([0, 16000], 16000, 1)[-1] == GOLD["mix16k"].shape[0]          # min over the three levels
    assert m.frame_offsets([0, 16000], 32000, 2)[-1] == GOLD["mix32k_stereo"].shape[0]


def test_truncating_multi_level_reader_frame_counts():
    # compare_ns.conf: cContourSmoother reads levels of the 20 ms and the 60 ms stream at once -> the
    # reader delivers min over them (core/dataReader.cpp:375-380); the reference's row counts:
    s = Session(os.path.join(CONF, "compare_ns.conf"), device=-1)
    lens = [16000, 960, 1100, 1300, 2000, 959]
    fo = s.frame_offsets(np.concatenate([[0], np.cumsum(lens)]), 16000, 1)
    want = [GOLD["cmp_ns"].shape[0]] + [GOLD["cmp_ns_short_%d" % n].shape[0] for n in (960, 1100, 1300, 2000)] + [0]
    assert list(np.diff(fo)) == want
    assert s.frame_offsets([0, 30000], 44100, 1)[-1] == GOLD["cmp_ns_44k"].shape[0]
    names = s.element_names()
    assert names[:4] == ["audspec_lengthL1norm_sma", "audspecRasta_lengthL1norm_sma", "pcm_RMSenergy_sma", "pcm_zcr_sma"]
    assert names[4] == "audSpec_Rfilt_sma[0]" and names[59] == "audspec_lengthL1norm_sma_de"


def test_parsed_components_carry_config_values():
    s = Session(os.path.join(CONF, "lld_mix.conf"), device=-1)
    comps, level = s.components(16000, 1)
    by = {c.name.decode(): c for c in comps}
    assert level == "_sinkconcat"                        # the sink reads three levels -> implicit concat
    assert [by["_sinkconcat"].reader_dmLevel[i].value.decode() for i in range(3)] == ["lld", "lld_de", "pitch_sma"]
    assert by["waveIn"].u.wavesource.sampleRate == 16000 and by["waveIn"].u.wavesource.monoMixdown == 1
    assert (by["fr25"].u.framer.frameSize, by["fr25"].u.framer.frameStep) == (0.025, 0.010)
    assert by["fr50"].u.framer.frameSize == 0.050
    assert by["win25"].u.windower.winFunc == capi.WIN_BY_NAME["ham"] and by["win50"].u.windower.winFunc == capi.WIN_BY_NAME["gau"]
    sp = by["spec"].u.spectral
    assert (sp.nBands, sp.bandLo[0], sp.bandHi[0], sp.bandLo[1], sp.bandHi[1]) == (2, 250, 650, 1000, 4000)
    assert (sp.nRollOff, sp.rollOff[0], sp.rollOff[1]) == (2, 0.25, 0.90)
    assert by["cep"].u.acf.cepstrum == 1 and by["cep"].u.acf.usePower == 0      # dspcore/acf.cpp:91-99
    assert by["acf"].u.acf.usePower == 1
    assert by["cat"].u.vectorconcat.includeSingleElementFields == 1
    assert by["pitch"].n_inputs == 2 and by["sm"].u.contoursmoother.smaWin == 3


def test_command_line_options_substitute():
    s = Session(os.path.join(CONF, "lld_mix.conf"), options={"step": "0.020"}, device=-1)
    comps, _ = s.components(16000, 1)
    by = {c.name.decode(): c for c in comps}
    assert by["fr25"].u.framer.frameStep == 0.020 and by["fr50"].u.framer.frameStep == 0.020   # \cm[step] reuse
    assert s.frame_offsets([0, 16000], 16000, 1)[-1] == (16000 - 800) // 320 + 1 + 1


def test_concat_drops_single_element_fields_by_default(tmp_path):
    # cVectorProcessor's processArrayFields=1 default (core/vectorProcessor.cpp:196-243): the
    # reference writes 36 columns for this variant (energy dropped), cf. tests/configs/inc/ft0_d_a_out.conf.inc
    inc = open(os.path.join(CONF, "inc", "ft0_d_a_out.conf.inc")).read().replace("includeSingleElementFields = 1", "")
    os.makedirs(tmp_path / "inc")
    (tmp_path / "inc" / "ft0_d_a_out.conf.inc").write_text(inc)
    (tmp_path / "inc" / "htk_frontend.conf.inc").write_text(open(os.path.join(CONF, "inc", "htk_frontend.conf.inc")).read())
    (tmp_path / "c.conf").write_text(open(os.path.join(CONF, "mfcc_e_d_a.conf")).read())
    names = Session(str(tmp_path / "c.conf"), device=-1).element_names()
    assert len(names) == 36 and not any("energy" in n for n in names)


@pytest.mark.parametrize("text,status,needle", [
    ("[frame:cFramer]\nreader.dmLevel=wave\nwriter.dmLevel=frames\nframeSizee = 0.025\n", capi.ERR_INVALID, "unknown field"),
    ("[x:cChroma]\nreader.dmLevel=wave\nwriter.dmLevel=func\n", capi.ERR_UNSUPPORTED, "cChroma"),
    ("[x:cFunctionals]\nreader.dmLevel=wave\nwriter.dmLevel=func\n", capi.ERR_INVALID, "functionalsEnabled"),
    ("[frame:cFramer]\nreader.dmLevel=wave\nwriter.dmLevel=frames\nframeSize = \\cm[fs:frame size]\n", capi.ERR_INVALID, "no value"),
    ("\\{does_not_exist.conf.inc}\n", capi.ERR_INVALID, "cannot open"),
    ("[frame:cFramer]\nreader.dmLevel=wave\nwriter.dmLevel=frames\nframeMode = list\n", capi.ERR_INVALID, "frameMode"),
])
def test_config_errors_are_loud(tmp_path, text, status, needle):
    head = ("[componentInstances:cComponentManager]\ninstance[dataMemory].type=cDataMemory\ninstance[waveIn].type=cWaveSource\n"
            "instance[frame].type=cFramer\ninstance[x].type=%s\n[waveIn:cWaveSource]\nwriter.dmLevel=wave\n")
    xt = "cChroma" if "cChroma" in text else "cFunctionals"
    head = head % xt
    if "[x:" not in text:
        head = head.replace("instance[x].type=%s\n" % xt, "")
    if "[frame:" not in text:
        head = head.replace("instance[frame].type=cFramer\n", "")
    (tmp_path / "bad.conf").write_text(head + text)
    with pytest.raises(SessionError) as e:
        # a component off the supported LLD path is rejected when the requested level depends on it (components
        # the output level does not depend on stay idle, like the reference's sinks without a file name)
        Session(str(tmp_path / "bad.conf"), output_level="func" if "[x:" in text else "frames", device=-1)
    assert e.value.status == status and needle in str(e.value), str(e.value)


def test_writers_are_byte_identical_to_reference_sinks(tmp_path):
    rows, names = GOLD["mfcc_e"], [str(x) for x in GOLD["names_mfcc_e"]]
    write_htk(tmp_path / "a.htk", rows, 0.01, 9)
    assert (tmp_path / "a.htk").read_bytes() == GOLD["htk_bytes"].tobytes()
    write_csv(tmp_path / "a.csv", rows, names, 0.01, instance_name="utt7", frame_index=False)
    assert (tmp_path / "a.csv").read_bytes() == GOLD["csv_bytes"].tobytes()


def test_description_only_session_refuses_to_compute():
    s = Session(os.path.join(CONF, "mfcc_e_d_a.conf"), device=-1)
    with pytest.raises(SessionError) as e:
        s.extract_pcm(np.zeros(16000, np.int16), [0, 16000], 16000, 1)
    assert e.value.status == capi.ERR_CUDA            # no CPU fallback


@pytest.mark.parametrize("conf,n", [("mfcc/MFCC12_0_D_A.conf", 39), ("mfcc/MFCC12_E_D_A.conf", 39),
                                    ("plp/PLP_0_D_A.conf", 18), ("plp/PLP_E_D_A.conf", 18),
                                    ("mfcc/MFCC12_0_D_A_Z.conf", 39), ("mfcc/MFCC12_E_D_A_Z.conf", 39),
                                    ("plp/PLP_0_D_A_Z.conf", 18), ("plp/PLP_E_D_A_Z.conf", 18),
                                    ("audspec/audspec.conf", 78), ("audspec/audspec_compat.conf", 78),
                                    ("spectrum/spectrogram.conf", 257), ("demo/demo1_energy.conf", 1),
                                    ("prosody/prosodyAcf.conf", 3)])
def test_reference_standard_configs_parse(conf, n):
    s = Session(os.path.join(REF_CONF, conf), device=-1)
    names = s.element_names(16000, 1)
    assert len(names) == n
    if conf.endswith("MFCC12_E_D_A.conf"):
        assert names == [str(x) for x in GOLD["names_mfcc_e"]]
    if conf.endswith("PLP_E_D_A.conf"):
        assert names == [str(x) for x in GOLD["names_plp_e"]]


def test_cli_fails_loudly_without_a_gpu(tmp_path):
    """No CPU fallback anywhere: on a box without a CUDA device the command line front end parses the
    configuration, then refuses to compute (non-zero exit, no output file)."""
    import subprocess
    import wave
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    exe = os.path.join(ROOT, "opensmile_b200", "SMILExtract_b200")
    pcm = (np.random.default_rng(0).standard_normal(8000) * 1000).astype("<i2")
    with wave.open(str(tmp_path / "t.wav"), "wb") as w:
        w.setnchannels(1); w.setsampwidth(2); w.setframerate(16000); w.writeframes(pcm.tobytes())
    r = subprocess.run([exe, "-C", os.path.join(CONF, "mfcc_e_d_a.conf"), "-I", str(tmp_path / "t.wav"), "-O", str(tmp_path / "o.htk")],
                       capture_output=True, text=True)
    assert r.returncode != 0 and "CUDA" in r.stderr and not (tmp_path / "o.htk").exists()
    # the reference's value-less switches (SMILExtract.cpp:60-72) do not swallow the argument behind them: the run gets just as far
    r = subprocess.run([exe, "-nologfile", "-C", os.path.join(CONF, "mfcc_e_d_a.conf"), "-noconsoleoutput", "-I", str(tmp_path / "t.wav"), "-l", "0",
                        "-appendLogfile", "1", "-O", str(tmp_path / "o.htk")], capture_output=True, text=True)
    assert r.returncode != 0 and "CUDA" in r.stderr and "required" not in r.stderr


def _conf_with(tmp_path, extra_instances, extra_sections, level):
    """htk front end + extra sections, HTK sink on `level`"""
    inc = tmp_path / "inc"
    inc.mkdir(exist_ok=True)
    (inc / "htk_frontend.conf.inc").write_text(open(os.path.join(CONF, "inc", "htk_frontend.conf.inc")).read())
    text = "\\{inc/htk_frontend.conf.inc}\n[componentInstances:cComponentManager]\n"
    text += "".join("instance[%s].type = %s\n" % kv for kv in extra_instances) + "instance[out].type = cHtkSink\n"
    text += extra_sections + "\n[out:cHtkSink]\nreader.dmLevel = %s\nfilename = o.htk\n" % level
    (tmp_path / "c.conf").write_text(text)
    return str(tmp_path / "c.conf")


def test_graph_rules_of_the_wider_component_set(tmp_path):
    # the magnitude level itself as output (spectrogram): one array field of nBins elements
    c = _conf_with(tmp_path, [], "", "fftmag")
    names = Session(c, device=-1).element_names(16000, 1)
    assert len(names) == 257 and names[0] == "pcm_fftMag[0]"
    assert len(Session(c, device=-1).element_names(44100, 1)) == 1025          # 1103-sample frames -> FFT 2048
    # mean subtraction must be the last stage of its branch
    secs = ("[mfcc:cMfcc]\nreader.dmLevel = melspec\nwriter.dmLevel = mfcc\n[cms:cFullinputMean]\nreader.dmLevel = mfcc\nwriter.dmLevel = mfccM\n"
            "[de:cDeltaRegression]\nreader.dmLevel = mfccM\nwriter.dmLevel = mfccMde\n")
    c = _conf_with(tmp_path, [("mfcc", "cMfcc"), ("cms", "cFullinputMean"), ("de", "cDeltaRegression")], secs, "mfccMde")
    with pytest.raises(SessionError) as e:
        Session(c, device=-1)
    assert e.value.status == capi.ERR_UNSUPPORTED and "cFullinputMean" in str(e.value)
    c = _conf_with(tmp_path, [("mfcc", "cMfcc"), ("cms", "cFullinputMean")], secs.split("[de:")[0], "mfccM")
    assert Session(c, device=-1).element_names()[0] == "pcm_fftMag_mfcc[1]"
    # cVectorOperation: only the n -> 1 mean (ll1) is on the path
    secs = ("[mfcc:cMfcc]\nreader.dmLevel = melspec\nwriter.dmLevel = mfcc\n[vo:cVectorOperation]\nreader.dmLevel = mfcc\nwriter.dmLevel = vo\n"
            "operation = %s\nnameBase = cepsum\n")
    c = _conf_with(tmp_path, [("mfcc", "cMfcc"), ("vo", "cVectorOperation")], secs % "ll1", "vo")
    assert Session(c, device=-1).element_names() == ["cepsum_lengthL1norm"]
    c = _conf_with(tmp_path, [("mfcc", "cMfcc"), ("vo", "cVectorOperation")], secs % "norm", "vo")
    with pytest.raises(SessionError) as e:
        Session(c, device=-1)
    assert "ll1" in str(e.value)
    # two cepstral ops on one FFT chain + RASTA naming
    secs = ("[mfcc:cMfcc]\nreader.dmLevel = melspec\nwriter.dmLevel = mfcc\n[rp:cPlp]\nreader.dmLevel = melspec\nwriter.dmLevel = rp\n"
            "RASTA = 1\nhtkcompatible = 0\n[cat:cVectorConcat]\nreader.dmLevel = mfcc;rp\nwriter.dmLevel = both\n")
    c = _conf_with(tmp_path, [("mfcc", "cMfcc"), ("rp", "cPlp"), ("cat", "cVectorConcat")], secs, "both")
    names = Session(c, device=-1).element_names()
    assert names[0] == "pcm_fftMag_mfcc[1]" and names[12] == "RASTAPlpCC[0]" and len(names) == 12 + 5   # cPlp defaults: firstCC = 1, lpOrder = 5


def test_parallel_file_sinks_equal_the_single_file_writers(tmp_path):
    """osm_b200_session_write_files (the sink half of extract_files: files formatted on host threads) against the single-file
    writers that are pinned byte for byte to the reference's sinks; incl. an empty file and the repeated time stamp of rows a
    window processor appends at the end of input"""
    from opensmile_b200 import write_csv, write_htk
    s = Session(os.path.join(CONF, "mfcc_e_d_a.conf"), device=-1)
    names = s.element_names()
    K = len(names)
    n_samples = np.array([16000, 400, 0, 48000] + [8000 + 160 * i for i in range(36)], np.int64)
    off = np.concatenate([[0], np.cumsum(n_samples)])
    fo = s.frame_offsets(off, 16000.0, 1)
    rows = np.random.default_rng(0).standard_normal((int(fo[-1]), K)).astype(np.float32)
    rows[::7, 3] = 0.0
    rows[5, 1] = 42.0
    assert "index=0 name=1:'unknown'" in s.sink_options()
    n = len(n_samples)
    htk = [str(tmp_path / ("p%d.htk" % i)) for i in range(n)]
    csv = [str(tmp_path / ("p%d.csv" % i)) for i in range(n)]
    s.write_files(rows, fo, 16000.0, 1, n_samples=n_samples, htk_paths=htk, csv_paths=csv)
    comps, level = s.components(16000.0, 1)
    from opensmile_b200 import Plan
    plan = Plan(list(comps), level, device=-1)
    for i in range(n):
        r = rows[fo[i]:fo[i + 1]]
        write_htk(str(tmp_path / "a.htk"), r, 0.01)
        write_csv(str(tmp_path / "a.csv"), r, names, 0.01, instance_name="unknown", frame_index=False,      # the configuration's sink options
                  n_time_frames=plan.num_time_frames(int(n_samples[i])))
        assert open(htk[i], "rb").read() == open(tmp_path / "a.htk", "rb").read()
        assert open(csv[i], "rb").read() == open(tmp_path / "a.csv", "rb").read()
    os.environ["OSM_B200_IO_THREADS"] = "1"                       # serial path
    try:
        s.write_files(rows, fo, 16000.0, 1, n_samples=n_samples, csv_paths=[str(tmp_path / ("q%d.csv" % i)) for i in range(n)])
    finally:
        del os.environ["OSM_B200_IO_THREADS"]
    assert all(open(csv[i], "rb").read() == open(tmp_path / ("q%d.csv" % i), "rb").read() for i in range(n))
    with pytest.raises(Exception, match="cannot write"):
        s.write_files(rows, fo, 16000.0, 1, csv_paths=[str(tmp_path / "nodir" / "x.csv")] * n)


def test_inputs_sharing_one_output_file_are_written_in_order(tmp_path):
    """the LLD ARFF sink of the feature-set configurations appends (append = 1): several inputs naming the same file must be
    written one after the other in input order, not by the parallel writers"""
    ref = os.path.join(REF_CONF, "compare16", "ComParE_2016.conf")
    s = Session(ref, options={"lldarffoutput": "x.arff", "instname": "u"}, device=-1)
    assert "append=1" in s.sink_options()
    K = len(s.element_names())
    n_samples = np.array([16000 + 1600 * i for i in range(12)], np.int64)
    fo = s.frame_offsets(np.concatenate([[0], np.cumsum(n_samples)]), 16000.0, 1)
    rows = np.zeros((int(fo[-1]), K), np.float32)
    for i in range(len(n_samples)):
        rows[fo[i]:fo[i + 1], 0] = i + 1                            # first column = 1-based file index
    out = str(tmp_path / "all.arff")
    s.write_files(rows, fo, 16000.0, 1, n_samples=n_samples, arff_paths=[out] * len(n_samples))
    data = open(out).read().split("@data")[1].strip().splitlines()
    assert len(data) == int(fo[-1])
    first = [int(float(ln.split(",")[2])) for ln in data]          # name, frameTime, then the values
    assert first == sorted(first) and first[0] == 1 and first[-1] == len(n_samples)


@pytest.mark.parametrize("case", ["bla", "bla_alpha", "bla_a012", "blh", "bah", "lac", "han_sqrt", "ham_fade", "blh_gain_sqrt_fade", "gau", "tri"])
def test_window_tables_equal_the_reference(tmp_path, case):
    """cWindower's table through the conf front end (names, defaults and coefficient rules of dspcore/windower.cpp:60-113) and the
    table builder, against the reference's cWindower level of a constant signal (tests/golden/window_goldens.npz,
    scripts/make_golden_windows.py): Blackman, Blackman-Harris, Bartlett-Hann, Lanczos, squareRoot, fade, custom coefficients"""
    import ctypes as C
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "window_goldens.npz"))
    (tmp_path / "inc").mkdir()
    inc = open(os.path.join(CONF, "inc", "htk_frontend.conf.inc")).read().replace("winFunc = ham\n", str(g[case + "_conf"]) + "\n")
    (tmp_path / "inc" / "htk_frontend.conf.inc").write_text(inc)
    (tmp_path / "inc" / "ft0_d_a_out.conf.inc").write_text(open(os.path.join(CONF, "inc", "ft0_d_a_out.conf.inc")).read())
    (tmp_path / "c.conf").write_text(open(os.path.join(CONF, "mfcc_0_d_a.conf")).read())
    s = Session(str(tmp_path / "c.conf"), device=-1)
    comps, _ = s.components(16000.0, 1)
    win = [c for c in comps if c.type == capi.C_WINDOWER][0]
    out = np.zeros(400, np.float32)
    assert capi.lib().osm_b200_window_table(C.byref(win.u.windower), 400, out.ctypes.data_as(C.POINTER(C.c_float))) == 0
    s.close()
    ref = g[case]
    # the reference's CSV prints 7 significant digits of the float product 1.0 * (float)w
    assert np.all(np.abs(out - ref) <= 1e-6 * np.abs(ref) + 1e-12), (case, float(np.abs(out - ref).max()))


def test_partial_file_options_are_refused_not_ignored():
    """cWaveSource.start / end / endrel select a part of the input file in the reference (iocore/waveSource.cpp:48-58); whole files
    are read here, so any value but the defaults is an error instead of a silently different result"""
    conf = os.path.join(REF_CONF, "mfcc", "MFCC12_0_D_A.conf")
    Session(conf, options={"O": "x.htk", "start": "0", "end": "-1"}, device=-1).close()
    for opts, needle in (({"start": "1.5"}, "start"), ({"end": "2.0"}, "end")):
        with pytest.raises(SessionError) as e:
            Session(conf, options=dict(opts, O="x.htk"), device=-1)
        assert e.value.status == capi.ERR_UNSUPPORTED or e.value.status == capi.ERR_INVALID
        assert needle in str(e.value)
