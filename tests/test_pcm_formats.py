"""SURVEY.md 8(a) row a-1 for every sample format cWaveSource accepts (smileutil/smileUtil.c:2500-2680): 8 / 24 / 32 bit integer,
24 valid bits in a 32-bit container (the reference masks without sign extension), 32-bit float, mono and stereo mixdown.
Goldens: the unmodified reference's `wave` level and MFCC12_0_D_A rows (scripts/make_golden_pcm_formats.py).
CPU: the oracle's conversion equals the reference's samples bit for bit.  GPU: pcm_convert_kernel + the plan, through the C ABI."""
import os
import struct

import numpy as np
import pytest

from oracle import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
G = np.load(os.path.join(HERE, "golden", "pcm_formats.npz"))
# name -> (osm_b200_pcm_format, WAV format tag, bits, bytes per sample, channels)
VARIANTS = {"s8_mono": (2, 1, 8, 1, 1), "s8_stereo": (2, 1, 8, 1, 2), "s24_mono": (3, 1, 24, 3, 1), "s24_stereo": (3, 1, 24, 3, 2),
            "s24in32_mono": (4, 1, 24, 4, 1), "s32_mono": (5, 1, 32, 4, 1), "s32_stereo": (5, 1, 32, 4, 2),
            "f32_mono": (1, 3, 32, 4, 1), "f32_stereo": (1, 3, 32, 4, 2)}


@pytest.mark.parametrize("name", list(VARIANTS))
def test_oracle_conversion_equals_the_reference_wave_level(name):
    fmt, _, _, _, nchan = VARIANTS[name]
    got = oracle.pcm_to_float(G["data_" + name].tobytes(), fmt, nchan)
    ref = G["wave_" + name]
    assert got.shape == ref.shape and np.array_equal(got.view(np.uint32), ref.view(np.uint32))


def test_oracle_int16_path_agrees_with_the_generic_one():
    rng = np.random.RandomState(3)
    x = rng.randint(-32768, 32768, size=6000).astype(np.int16)
    for nchan in (1, 2, 3):
        a = oracle.pcm_to_float(x.tobytes(), 0, nchan)
        L = oracle.lib()
        b = np.empty(len(x) // nchan, np.float32)
        L.osm_or_pcm16_to_float.argtypes = [oracle.C.c_void_p, oracle.C.c_long, oracle.C.c_int, oracle.C.c_void_p]
        L.osm_or_pcm16_to_float(x.ctypes.data, len(x) // nchan, nchan, b.ctypes.data)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _close(rows, ref):
    """the MFCC rule of conftest.column_scale_report on a 23-frame sample: nothing beyond 5e-5 of a column's scale; the isolated
    values between 1e-5 and 5e-5 (log of weak bands through the delta regression) are counted in values, not in per mille"""
    from conftest import column_scale_report
    worst, share = column_scale_report(rows, ref)
    assert worst < 5e-5 and share * rows.size <= max(6, 1e-3 * rows.size), (worst, share * rows.size)


def _write_wav(path, data, tag, bits, bps, nchan, sr=16000):
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", 36 + len(data)) + b"WAVE")
        f.write(b"fmt " + struct.pack("<IHHIIHH", 16, tag, nchan, sr, sr * bps * nchan, bps * nchan, bits))
        f.write(b"data" + struct.pack("<I", len(data)) + data)


def test_unsupported_sample_formats_are_refused_by_the_file_reader(tmp_path):
    """what the reference refuses (smileUtil.c:2445-2449: anything but integer PCM and IEEE float; :2573 unknown widths) is refused
    here before any device work: A-law, 64-bit float, 16 valid bits in a 32-bit container"""
    from opensmile_b200.session import Session, SessionError
    conf = os.path.join(HERE, "configs", "mfcc_e_d_a.conf")
    s = Session(conf, device=-1)
    for tag, bits, bps in ((6, 8, 1), (3, 64, 8), (1, 16, 4)):
        p = tmp_path / ("bad_%d_%d.wav" % (tag, bits))
        _write_wav(str(p), b"\0" * (bps * 4000), tag, bits, bps, 1)
        with pytest.raises(SessionError) as e:
            s.extract_files([str(p)], htk_paths=[str(tmp_path / "o.htk")])
        assert "unsupported sample format" in str(e.value)
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(VARIANTS))
def test_plan_on_every_sample_format_equals_the_reference(name):
    """MFCC12_0_D_A rows from the raw bytes of each format through osm_b200_plan_run_host (pcm_convert_kernel in front of the
    kernels): every column within 1e-5 of its scale, same frame count"""
    from opensmile_b200 import Plan, components_mfcc12_0_d_a
    fmt, _, _, bps, nchan = VARIANTS[name]
    data = np.ascontiguousarray(G["data_" + name])
    plan = Plan(components_mfcc12_0_d_a(16000.0, nchan, pcm_format=fmt), "lld", device=0)
    assert plan.sample_frame_bytes == bps * nchan
    n = data.size // (bps * nchan)
    rows = plan.run_host(data, np.array([0, n], np.int64))
    ref = G["mfcc_" + name]
    assert rows.shape == ref.shape
    _close(rows, ref)


@pytest.mark.gpu
def test_formats_mix_in_one_file_batch(tmp_path):
    """files of different sample formats in one osm_b200_session_extract_files call: grouped by (rate, channels, format), each group
    one plan run, every HTK file equal to the reference's rows"""
    from oracle import refrun
    from opensmile_b200.session import Session
    conf = os.path.join(HERE, "golden", "config", "mfcc", "MFCC12_0_D_A.conf")
    names = ["s8_stereo", "s24_mono", "f32_stereo", "s32_mono", "s24in32_mono"]
    wavs, outs = [], []
    for nm in names:
        fmt, tag, bits, bps, nchan = VARIANTS[nm]
        wavs.append(str(tmp_path / (nm + ".wav")))
        outs.append(str(tmp_path / (nm + ".htk")))
        _write_wav(wavs[-1], G["data_" + nm].tobytes(), tag, bits, bps, nchan)
    s = Session(conf, options={"O": "x.htk"}, device=0)
    frames = s.extract_files(wavs, htk_paths=outs)
    s.close()
    for nm, o, fr in zip(names, outs, frames):
        rows, _ = refrun.read_htk(o)
        assert fr == len(G["mfcc_" + nm]) and rows.shape == G["mfcc_" + nm].shape
        _close(rows, G["mfcc_" + nm])
