"""cDataSelector (core/dataSelector.cpp, elementMode = 1) in the graph compiler: tests/configs/gemaps_sel.conf puts a selector
on top of the reference's shipped GeMAPS graph (pitch + jitter / shimmer levels) next to the shipped selector
gemapsv01b_lldsetE.  Element names, order and frame counts against the reference's CSV file
(tests/golden/select_goldens.npz, scripts/make_golden_select.py); the oracle's rows (incl. the rule that every column of a
selector reading the cPitchJitter level lags at the end of input) against the same file; refusals."""
import os

import numpy as np
import pytest

from opensmile_b200.session import Session, SessionError
from opensmile_b200.synth import mixed_pcm, voiced_pcm

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
G = np.load(os.path.join(HERE, "golden", "select_goldens.npz"))
REFCONF = os.path.join(HERE, "golden", "config")


def _conf(tmp_path, edit=None):
    text = open(os.path.join(HERE, "configs", "gemaps_sel.conf")).read().replace("REFCONF", REFCONF)
    if edit:
        assert edit[0] in text
        text = text.replace(edit[0], edit[1])
    p = tmp_path / "gsel.conf"
    p.write_text(text)
    return str(p)


def test_names_order_and_frame_counts(tmp_path):
    s = Session(_conf(tmp_path), device=-1)
    assert s.element_names() == list(G["gsel_names"])
    fo = s.frame_offsets(np.array([0, 24000, 56000], np.int64), 16000.0, 1)
    assert list(np.diff(fo)) == [G["gsel_m24k"].shape[0], G["gsel_v32k"].shape[0]]


def test_oracle_rows_of_the_selector_configuration():
    from oracle import formant_oracle as fo
    for key, pcm in (("gsel_m24k", mixed_pcm(24000, 16000, seed=3)), ("gsel_v32k", voiced_pcm(32000, 16000, seed=7))):
        got, ref = fo.gemaps_sel_lld(pcm), G[key]
        assert got.shape == ref.shape
        assert (np.abs(got - ref) / (np.abs(ref).max(axis=0) + 1e-30)).max() < 5e-6     # the CSV file holds 7 digits


@pytest.mark.parametrize("edit,needle", [
    (("selected = shimmerLocalDB;F0finalLog;jitterLocal", "selected = shimmerLocalDB;F0finalLogX;jitterLocal"), "not found"),
    (("selected = shimmerLocalDB;F0finalLog;jitterLocal", "selected = jitterLocal;F0finalLog;jitterLocal"), "selected twice"),
    (("newNames = shimmerLocaldB;F0semitoneFrom27.5Hz", "elementMode = 0"), "elementMode"),
    (("[smoF:cContourSmoother]\nreader.dmLevel = selF\n",
      "[componentInstances:cComponentManager]\ninstance[selF2].type=cDataSelector\n[selF2:cDataSelector]\nreader.dmLevel = selF\n"
      "writer.dmLevel = selF2\nselected = jitterLocal\n[smoF:cContourSmoother]\nreader.dmLevel = selF2\n"), "nested"),
])
def test_refusals(tmp_path, edit, needle):
    with pytest.raises(SessionError, match=needle):
        Session(_conf(tmp_path, edit), device=-1)


def test_names_without_new_names(tmp_path):
    s = Session(_conf(tmp_path, ("newNames = shimmerLocaldB;F0semitoneFrom27.5Hz", "nameAppend = sel")), device=-1)
    assert s.element_names()[5:] == ["shimmerLocalDB_sel_sma3nz", "F0finalLog_sel_sma3nz", "jitterLocal_sel_sma3nz"]


_BASE = """[componentInstances:cComponentManager]
instance[dataMemory].type=cDataMemory
instance[waveIn].type=cWaveSource
instance[fr].type=cFramer
instance[win].type=cWindower
instance[fft].type=cTransformFFT
instance[mag].type=cFFTmagphase
instance[mel].type=cMelspec
instance[mfcc].type=cMfcc
instance[en].type=cEnergy
instance[sel].type=cDataSelector
instance[sink].type=cCsvSink
[waveIn:cWaveSource]
writer.dmLevel=wave
filename=\\cm[inputfile(I){in.wav}:input]
monoMixdown=1
[fr:cFramer]
reader.dmLevel=wave
writer.dmLevel=frames
frameSize=0.025
frameStep=0.010
frameCenterSpecial=left
[win:cWindower]
reader.dmLevel=frames
writer.dmLevel=win
winFunc=ham
[fft:cTransformFFT]
reader.dmLevel=win
writer.dmLevel=fft
[mag:cFFTmagphase]
reader.dmLevel=fft
writer.dmLevel=mag
[mel:cMelspec]
reader.dmLevel=mag
writer.dmLevel=mel
nBands=26
[mfcc:cMfcc]
reader.dmLevel=mel
writer.dmLevel=mfcc
firstMfcc=0
lastMfcc=12
[en:cEnergy]
reader.dmLevel=frames
writer.dmLevel=energy
rms=1
log=1
[sel:cDataSelector]
reader.dmLevel=mfcc;energy
writer.dmLevel=out
SELECTED
[sink:cCsvSink]
reader.dmLevel=out
filename=\\cm[outputfile(O){out.csv}:output]
"""


def test_selector_on_array_elements_and_plain_fields(tmp_path):
    """elements of an array field (mfcc[3]) and single-element fields (pcm_LOGenergy) through one selector at the top of the
    graph: order of `selected`, contiguous elements merged into one group, nameAppend when no new name is given"""
    p = tmp_path / "s.conf"
    p.write_text(_BASE.replace("SELECTED", "selected = pcm_LOGenergy;pcm_fftMag_mfcc[3];pcm_fftMag_mfcc[4];pcm_fftMag_mfcc[1]\nnewNames = E;c3"))
    s = Session(str(p), device=-1)
    assert s.element_names() == ["E", "c3", "pcm_fftMag_mfcc[4]", "pcm_fftMag_mfcc[1]"]
    assert int(s.frame_offsets(np.array([0, 16000], np.int64), 16000.0, 1)[-1]) == 98
    p.write_text(_BASE.replace("SELECTED", "selected = pcm_fftMag_mfcc[12];pcm_RMSenergy\nnameAppend = x"))
    assert Session(str(p), device=-1).element_names() == ["pcm_fftMag_mfcc[12]_x", "pcm_RMSenergy_x"]
    p.write_text(_BASE.replace("SELECTED", "selected[0] = pcm_RMSenergy\nselected[1] = pcm_fftMag_mfcc[0]\nnewNames[1] = c0"))   # indexed array syntax
    assert Session(str(p), device=-1).element_names() == ["pcm_RMSenergy", "c0"]
    p.write_text(_BASE.replace("SELECTED", "selected = pcm_fftMag_mfcc"))          # a field name is not an element name (elementMode = 1)
    with pytest.raises(SessionError, match="not found"):
        Session(str(p), device=-1)
