"""Generate tests/golden/pitch_goldens.npz with the UNMODIFIED reference (oracle/_ref/SMILExtract):

    python scripts/make_golden_pitch.py        # needs `make -C oracle ref` (build container only)

For each case (inputs are regenerated in the tests from opensmile_b200.synth):
  <case>_lld      config/compare16/ComParE_2016.conf -lldhtkoutput: the full ComParE_2016 LLD set [rows, 130]
                  (level lld ; lld_de, float32 exact)
  <case>_shs/_vit/_sel/_jit/_nz/_nzde/_e60   level taps of tests/configs/compare_pitch_taps.conf (cPitchShs,
                  cPitchSmootherViterbi, cValbasedSelector, cPitchJitter, smoothed level and its delta, rms energy)
  names_lld       element names of the LLD CSV header; v32k_lld_csv / v32k_lld_arff = the reference's -lldcsvoutput / -lldarffoutput files (-instname utt7) as bytes,
                  stored in tests/golden/lld_sink_files.npz
Cases: v32k = voiced_pcm(32000, seed=7); m48k = mixed_pcm(48000, seed=2) (Viterbi lag 1); m30k = mixed_pcm(30000, seed=4);
       m64k = mixed_pcm(64000, seed=3); m60k_44k = mixed_pcm(60000, seed=5) written as a 44.1 kHz file (FFT 4096 / 1024,
       _lld only); m40k_stereo = stereo_mixed_pcm(40000, seed=9), 16 kHz, 2 channels (_lld only); var_m48k / var_m40k = tests/configs/pitch_variants.conf on mixed_pcm(48000, seed=6) / mixed_pcm(40000, seed=8)
       (Viterbi lags 1 and 7), names_var its element names; short_<n> = voiced_pcm(n, seed=7) for n = 960, 1120, 1600, 2400 (1, 2, 5, 10 frames of 60 ms)
"""
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import refrun  # noqa: E402
from opensmile_b200.synth import mixed_pcm, voiced_pcm  # noqa: E402

CASES = {
    "v32k": lambda: voiced_pcm(32000, 16000, seed=7),
    "m48k": lambda: mixed_pcm(48000, 16000, seed=2),
    "m30k": lambda: mixed_pcm(30000, 16000, seed=4),
    "m64k": lambda: mixed_pcm(64000, 16000, seed=3),
    "short_960": lambda: voiced_pcm(960, 16000, seed=7),
    "short_1120": lambda: voiced_pcm(1120, 16000, seed=7),
    "short_1600": lambda: voiced_pcm(1600, 16000, seed=7),
    "short_2400": lambda: voiced_pcm(2400, 16000, seed=7),
}


def main():
    assert refrun.available(), "build the reference first: make -C oracle ref"
    out = {}
    taps_src = open(os.path.join(ROOT, "tests", "configs", "compare_pitch_taps.conf")).read().replace("REFCONF", refrun.CONFIG_DIR)
    full = os.path.join(refrun.CONFIG_DIR, "compare16", "ComParE_2016.conf")
    for name, gen in CASES.items():
        pcm = gen()
        with tempfile.TemporaryDirectory() as d:
            wav = os.path.join(d, "in.wav")
            refrun.write_wav(wav, pcm, 16000, 1)
            with open(os.path.join(d, "taps.conf"), "w") as f:
                f.write(taps_src)
            subprocess.run([refrun.SMILEXTRACT, "-C", "taps.conf", "-I", "in.wav", "-l", "0"], cwd=d, check=True,
                           stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            for k in ("shs", "vit", "sel", "jit", "nz", "nzde", "e60"):
                p = os.path.join(d, k + ".htk")
                if os.path.exists(p) and os.path.getsize(p) > 12:
                    out["%s_%s" % (name, k)] = refrun.read_htk(p)[0]
            subprocess.run([refrun.SMILEXTRACT, "-C", full, "-I", wav, "-lldhtkoutput", os.path.join(d, "lld.htk"),
                            "-lldcsvoutput", os.path.join(d, "lld.csv"), "-l", "0"], check=True,
                           stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            p = os.path.join(d, "lld.htk")
            if os.path.exists(p) and os.path.getsize(p) > 12:
                out["%s_lld" % name] = refrun.read_htk(p)[0]
            if name == "v32k":                       # the LLD CSV file itself (instance name utt7), for the writer test
                subprocess.run([refrun.SMILEXTRACT, "-C", full, "-I", wav, "-lldcsvoutput", os.path.join(d, "utt7.csv"),
                                "-instname", "utt7", "-l", "0"], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                out["v32k_lld_csv"] = np.frombuffer(open(os.path.join(d, "utt7.csv"), "rb").read(), dtype=np.uint8)
                subprocess.run([refrun.SMILEXTRACT, "-C", full, "-I", wav, "-lldarffoutput", os.path.join(d, "utt7.arff"),
                                "-instname", "utt7", "-l", "0"], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                out["v32k_lld_arff"] = np.frombuffer(open(os.path.join(d, "utt7.arff"), "rb").read(), dtype=np.uint8)
            if "names_lld" not in out and os.path.exists(os.path.join(d, "lld.csv")):
                hdr = open(os.path.join(d, "lld.csv")).readline().strip().split(";")
                out["names_lld"] = np.array([h for h in hdr if h not in ("name", "frameIndex", "frameTime")])
        print(name, {k[len(name) + 1:]: v.shape for k, v in out.items() if k.startswith(name + "_")})
    with tempfile.TemporaryDirectory() as d:            # the same configuration at 44.1 kHz
        wav = os.path.join(d, "in.wav")
        refrun.write_wav(wav, mixed_pcm(60000, 16000, seed=5), 44100, 1)
        subprocess.run([refrun.SMILEXTRACT, "-C", full, "-I", wav, "-lldhtkoutput", os.path.join(d, "lld.htk"), "-l", "0"],
                       check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        out["m60k_44k_lld"] = refrun.read_htk(os.path.join(d, "lld.htk"))[0]
    with tempfile.TemporaryDirectory() as d:            # stereo input (mono mixdown in the wave source)
        from opensmile_b200.synth import stereo_mixed_pcm
        wav = os.path.join(d, "in.wav")
        refrun.write_wav(wav, stereo_mixed_pcm(40000, 16000, seed=9), 16000, 2)
        subprocess.run([refrun.SMILEXTRACT, "-C", full, "-I", wav, "-lldhtkoutput", os.path.join(d, "lld.htk"), "-l", "0"],
                       check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        out["m40k_stereo_lld"] = refrun.read_htk(os.path.join(d, "lld.htk"))[0]
    var = os.path.join(ROOT, "tests", "configs", "pitch_variants.conf")     # the chain's other switches
    for name, pcm in (("var_m48k", mixed_pcm(48000, 16000, seed=6)), ("var_m40k", mixed_pcm(40000, 16000, seed=8))):
        with tempfile.TemporaryDirectory() as d:
            wav = os.path.join(d, "in.wav")
            refrun.write_wav(wav, pcm, 16000, 1)
            subprocess.run([refrun.SMILEXTRACT, "-C", var, "-I", wav, "-O", os.path.join(d, "o.htk"), "-csvoutput", os.path.join(d, "o.csv"),
                            "-l", "0"], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            out[name + "_lld"] = refrun.read_htk(os.path.join(d, "o.htk"))[0]
            hdr = open(os.path.join(d, "o.csv")).readline().strip().split(";")
            out["names_var"] = np.array([h for h in hdr if h not in ("name", "frameIndex", "frameTime")])
    # the two sink files go to an archive of their own: each file under tests/golden/ stays below 1 MB
    sinks = {k: out.pop(k) for k in ("v32k_lld_csv", "v32k_lld_arff")}
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "pitch_goldens.npz"), **out)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "lld_sink_files.npz"), **sinks)


if __name__ == "__main__":
    main()
