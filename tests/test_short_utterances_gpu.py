"""Very short utterances (0 .. 26 output rows) on the shipped ComParE_2016 / eGeMAPSv02 LLD graphs against the unmodified reference's
rows (tests/golden/short_utterances.npz): row counts for every length, values per column.

Stated exception (DESIGN.md section 5): ComParE_2016 utterances with 2 .. 4 frames of the 60 ms level (3 .. 5 output rows, i.e. shorter
than 0.1 s) -- the six onlyInSegments delta columns behind the pitch chain (`*_sma_de` of F0final, voicingFinalUnclipped, jitterLocal,
jitterDDP, shimmerLocal, logHNR) follow a tick order at end of input that the model of seq_post_kernel does not cover; all other 124
columns and all lengths from 5 frames on are equal.  eGeMAPSv02 (no segment deltas) is equal for every length."""
import os

import numpy as np
import pytest

from opensmile_b200.synth import voiced_pcm

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
REFCONF = os.path.join(HERE, "golden", "config")
G = np.load(os.path.join(HERE, "golden", "short_utterances.npz"))
LENS = (900, 1000, 1130, 1290, 1450, 1610, 2000, 3000, 4800)
SEG_DE = ["F0final_sma_de", "voicingFinalUnclipped_sma_de", "jitterLocal_sma_de", "jitterDDP_sma_de", "shimmerLocal_sma_de", "logHNR_sma_de"]


@pytest.mark.parametrize("conf,tag", [("compare16/ComParE_2016.conf", "c16"), ("egemaps/v02/eGeMAPSv02.conf", "ege")])
def test_short_utterances(conf, tag):
    from opensmile_b200.session import Session
    s = Session(os.path.join(REFCONF, conf), options={"lldcsvoutput": "x.csv"}, device=0)
    names = s.element_names()
    off = np.concatenate([[0], np.cumsum(LENS)]).astype(np.int64)
    rows, fo = s.extract_pcm(np.concatenate([voiced_pcm(n, 16000, seed=n) for n in LENS]), off, 16000.0, 1)
    s.close()
    scale = np.abs(G["%s_4800" % tag]).max(axis=0) + 1e-9
    for u, n in enumerate(LENS):
        ref = G["%s_%d" % (tag, n)]
        got = rows[fo[u]:fo[u + 1]]
        assert got.shape[0] == ref.shape[0], (tag, n, got.shape, ref.shape)          # 0 rows below one 60 ms frame
        if ref.size == 0:
            continue
        cols = np.ones(len(names), bool)
        if tag == "c16" and 3 <= len(ref) <= 5:
            cols = np.array([nm not in SEG_DE for nm in names])                      # the stated exception
        err = np.abs(got - ref)[:, cols] / scale[cols]
        assert err.max() < 1e-4, (tag, n, float(err.max()), np.array(names)[cols][int(np.argmax(err.max(axis=0)))])
