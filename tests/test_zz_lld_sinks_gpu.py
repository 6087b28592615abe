"""The three LLD sinks of the shipped ComParE_2016 configuration (-lldhtkoutput / -lldcsvoutput / -lldarffoutput)
through osm_b200_session_extract_files_arff on the GPU: file structure identical to the reference's files
(headers, instance name, time stamps incl. the repeated one of the appended last row), values within 1e-5 of each
column's scale.  (Named to run last: it exercises file I/O on top of paths the other GPU tests already cover.)
The writers themselves are pinned byte for byte on the CPU (tests/test_pitch_cpu.py)."""
import os

import numpy as np
import pytest

from opensmile_b200.synth import voiced_pcm

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
G = np.load(os.path.join(HERE, "golden", "pitch_goldens.npz"))
SINKS = np.load(os.path.join(HERE, "golden", "lld_sink_files.npz"))
CONF = os.path.join(HERE, "golden", "config", "compare16", "ComParE_2016.conf")


def _write_wav(path, pcm, sr):
    import wave
    with wave.open(str(path), "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(sr)
        w.writeframes(np.ascontiguousarray(pcm, dtype="<i2").tobytes())


def test_compare16_three_lld_sinks(tmp_path):
    from opensmile_b200.session import Session
    wav = tmp_path / "in.wav"
    _write_wav(wav, voiced_pcm(32000, 16000, seed=7), 16000)
    s = Session(CONF, options={"lldcsvoutput": "x.csv", "lldarffoutput": "x.arff", "lldhtkoutput": "x.htk", "instname": "utt7"}, device=0)
    frames = s.extract_files([str(wav)], [str(tmp_path / "o.htk")], [str(tmp_path / "o.csv")], [str(tmp_path / "o.arff")])
    s.close()
    ref = G["v32k_lld"]
    assert list(frames) == [ref.shape[0]]
    scale = np.abs(ref).max(axis=0) + 1e-30

    # CSV: same header, same name / time columns, values within tolerance (printed with 7 significant digits)
    got = (tmp_path / "o.csv").read_text().splitlines()
    exp = SINKS["v32k_lld_csv"].tobytes().decode().splitlines()
    assert got[0] == exp[0] and len(got) == len(exp)
    for a, b in zip(got[1:], exp[1:]):
        fa, fb = a.split(";"), b.split(";")
        assert fa[:2] == fb[:2]
        assert (np.abs(np.array(fa[2:], float) - np.array(fb[2:], float)) / scale < 2e-5).all()

    # ARFF: identical header block, identical name / time / target fields
    got = (tmp_path / "o.arff").read_text().split("\n")
    exp = SINKS["v32k_lld_arff"].tobytes().decode().split("\n")
    n_hdr = exp.index("@data") + 2
    assert got[:n_hdr] == exp[:n_hdr] and len(got) == len(exp)
    for a, b in zip(got[n_hdr:-1], exp[n_hdr:-1]):
        fa, fb = a.split(","), b.split(",")
        assert fa[:2] == fb[:2] and fa[-1] == fb[-1] == "?"
        assert (np.abs(np.array(fa[2:-1], float) - np.array(fb[2:-1], float)) / scale < 2e-5).all()

    # HTK: header (rows, 10 ms period in 100 ns units, 130 * 4 bytes, parmKind 9) + big-endian floats
    raw = (tmp_path / "o.htk").read_bytes()
    n, period, size, kind = np.frombuffer(raw[:12], dtype=">i4,>i4,>i2,>i2")[0]
    assert (int(n), int(period), int(size), int(kind)) == (ref.shape[0], 100000, 520, 9)
    rows = np.frombuffer(raw[12:], dtype=">f4").reshape(ref.shape).astype(np.float32)
    assert (np.abs(rows - ref) / scale < 1e-5).all()
