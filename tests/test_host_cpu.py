"""CPU tests of the host side: the C-ABI library loads, exports every declared symbol, and the
graph compiler reproduces the reference's geometry / naming / frame-count rules.  No compute
calls (there is no GPU here and the library has no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from opensmile_b200 import Plan, capi, components_mfcc12_0_d_a
from opensmile_b200.plan import _comp


def test_library_exports_every_declared_symbol():
    inc = os.path.join(ROOT, "include")
    hdr = "".join(open(os.path.join(inc, f)).read() for f in sorted(os.listdir(inc)) if f.endswith(".h"))
    declared = set(re.findall(r"OSM_B200_API[^;]*?\b(osm_b200_\w+)\s*\(", hdr))
    assert declared == set(capi.EXPORTS), declared ^ set(capi.EXPORTS)
    L = C.CDLL(capi.LIB_PATH)
    for sym in declared:
        assert hasattr(L, sym), sym
    assert capi.lib().osm_b200_abi_version() == 3


def test_struct_mirror_matches_library():
    assert capi.lib().osm_b200_sizeof_component() == C.sizeof(capi.Component)


def test_defaults_follow_reference_schema():
    # SURVEY.md Appendix A (dumped from the reference with -configDflt)
    L = capi.lib()
    c = capi.Component()
    assert L.osm_b200_component_defaults(capi.C_MELSPEC, C.byref(c)) == 0
    assert (c.u.melspec.nBands, c.u.melspec.lofreq, c.u.melspec.hifreq, c.u.melspec.usePower,
            c.u.melspec.htkcompatible) == (26, 20.0, 8000.0, 0, 1)
    L.osm_b200_component_defaults(capi.C_MFCC, C.byref(c))
    assert (c.u.mfcc.firstMfcc, c.u.mfcc.lastMfcc, c.u.mfcc.cepLifter, c.u.mfcc.melfloor) == (1, 12, 22.0, 1e-8)
    L.osm_b200_component_defaults(capi.C_TRANSFORMFFT, C.byref(c))
    assert c.u.transformfft.zeroPadSymmetric == 1
    L.osm_b200_component_defaults(capi.C_DELTAREGRESSION, C.byref(c))
    assert c.u.deltaregression.deltawin == 2
    L.osm_b200_component_defaults(capi.C_FRAMER, C.byref(c))
    assert (c.u.framer.frameSize, c.u.framer.noPostEOIprocessing) == (0.025, 1)


def test_plan_geometry_names_and_frame_counts():
    p = Plan(components_mfcc12_0_d_a(44100.0), "lld", device=-1)
    assert (p.num_elements, p.frame_size, p.frame_step, p.fft_size) == (39, 1103, 441, 2048)
    names = p.element_names
    assert names[0] == "pcm_fftMag_mfcc[0]" and names[12] == "pcm_fftMag_mfcc[12]"
    assert names[13] == "pcm_fftMag_mfcc_de[0]" and names[38] == "pcm_fftMag_mfcc_de_de[12]"
    assert p.num_frames(90112) == 202 and p.num_frames(1102) == 0 and p.num_frames(1103) == 1
    p16 = Plan(components_mfcc12_0_d_a(16000.0), "lld", device=-1)
    assert (p16.frame_size, p16.frame_step, p16.fft_size) == (400, 160, 512)
    assert p16.num_frames(80000) == 498 and p16.num_frames(9600000) == 59998 and p16.num_frames(0) == 0
    off = np.array([0, 80000, 80399, 80799, 180799], np.int64)
    assert p16.frame_offsets(off).tolist() == [0, 498, 498, 499, 499 + 623]
    assert abs(p16.frame_period - 0.010) < 1e-15


def test_description_plan_cannot_run_and_errors_are_reported():
    p = Plan(components_mfcc12_0_d_a(16000.0), "lld", device=-1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        p.run_host(np.zeros(1000, np.int16), np.array([0, 1000], np.int64))


def test_graph_errors():
    comps = components_mfcc12_0_d_a(16000.0)
    with pytest.raises(RuntimeError, match="no writer"):
        Plan(comps, "nonexistent", device=-1)
    with pytest.raises(RuntimeError, match="exactly one cWaveSource"):
        Plan(comps[1:], "lld", device=-1)
    bad = components_mfcc12_0_d_a(16000.0)
    bad[8] = _comp(capi.C_DELTAREGRESSION, "delta", "ft0", "ft0de", deltawin=2, relativeDelta=1, onlyInSegments=1)
    with pytest.raises(RuntimeError, match="not supported"):
        Plan(bad, "lld", device=-1)
    bad[8] = _comp(capi.C_DELTAREGRESSION, "delta", "ft0", "ft0de", deltawin=0)          # simple difference: refused
    with pytest.raises(RuntimeError, match="deltawin"):
        Plan(bad, "lld", device=-1)


def test_no_gpu_means_loud_failure_not_fallback():
    if capi.lib().osm_b200_device_count() > 0:
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no usable CUDA device"):
        Plan(components_mfcc12_0_d_a(16000.0), "lld", device=0)


def test_fft_butterflies_host_build(tmp_path):
    """fft_radix.cuh compiled for the host and checked against a naive DFT."""
    exe = str(tmp_path / "test_fft_radix")
    subprocess.check_call(["nvcc", "-std=c++17", "-O2", "-Wno-deprecated-gpu-targets", "-o", exe,
                           os.path.join(ROOT, "tests", "native", "test_fft_radix.cu")])
    subprocess.check_call([exe])


def test_div32767_trick():
    """kernels.cu::div32767 (reciprocal multiply + two FMAs) must equal IEEE x / 32767.0f for
    every value the PCM conversion can produce: all int16 (mono) and all half-integers k/2,
    |k| <= 65536 (stereo mixdown).  Exact rational arithmetic, no GPU needed."""
    import struct
    from fractions import Fraction

    def f32(fr):
        if fr == 0:
            return 0.0
        y = np.float32(float(fr))
        c = [np.nextafter(y, np.float32(-np.inf)), y, np.nextafter(y, np.float32(np.inf))]
        ds = sorted(c, key=lambda v: abs(Fraction(float(v)) - fr))
        if abs(Fraction(float(ds[0])) - fr) == abs(Fraction(float(ds[1])) - fr):
            for v in ds[:2]:
                if (struct.unpack("I", struct.pack("f", float(v)))[0] & 1) == 0:
                    return float(v)
        return float(ds[0])

    D = Fraction(32767)
    rc = f32(Fraction(1) / D)
    assert rc == float(np.float32(3.0518509447574615e-05))
    for k in list(range(-65536, 65535, 7)) + list(range(-65536, -65400)) + list(range(65400, 65535)) + list(range(-64, 64)):
        x = Fraction(k, 2)
        q0 = f32(x * Fraction(rc))
        r = f32(x - Fraction(q0) * D)
        q1 = f32(Fraction(q0) + Fraction(r) * Fraction(rc))
        assert q1 == f32(x / D), k


def test_text_sink_number_formatting_equals_printf(tmp_path):
    """the text sinks format values with std::to_chars into a buffer (opensmile_b200/host/front.cpp TextBuf); for finite
    floats that is byte-identical to the reference's fprintf("%e") / ("%.0f"): 40 M values incl. random bit patterns"""
    exe = str(tmp_path / "fmt_check")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "native", "fmt_check.cpp")])
    subprocess.check_call([exe], stdout=subprocess.DEVNULL)


def test_device_text_formatter_equals_printf():
    """opensmile_b200/csrc/text_format.cuh (the cCsvSink value format of the device sinks) compiled for the host: identical to printf
    on millions of values -- random bit patterns, LLD-sized decimals and their neighbours, dyadic ties, powers of ten, integers --
    and it leaves at most ~1e-6 of the in-range values to the host formatter"""
    exe = "/tmp/osm_fmt_device_check_%d" % os.getuid()
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-o", exe, os.path.join(ROOT, "tests", "native", "fmt_device_check.cpp")])
    out = subprocess.run([exe, "3000000"], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    checked, bad, uncertain = (int(x) for x in out.stdout.split())
    assert bad == 0 and checked > 5000000 and uncertain <= checked * 2e-6, out.stdout
