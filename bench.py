#!/usr/bin/env python
"""bench.py -- LLD frames/s of the B200 path on the BASELINE.json configurations.

A "step" is one pass of the hot path over one batch of synthetic utterances (weak scaling: every rank owns its own batch; the
path has no data-path collective, NCCL only carries the timing / counter reduction).

  workloads (--workload, or OSM_BENCH_WORKLOAD for a driver that passes no flags):
    mfcc12    BASELINE configs[1]  MFCC12_0_D_A, 16 kHz mono, 2000 utterances x 500 frames = 1 M frames per GPU   (default,
              the configuration the metric is quoted on)
    egemaps   configs[2]  the shipped eGeMAPSv02.conf (25 LLD columns), 16 kHz mono, 3 s utterances
    compare16 configs[3]  the shipped ComParE_2016.conf (130 LLD columns), 16 kHz mono, 3 s utterances
    plp44k    configs[4]  PLP_0_D_A, 44.1 kHz STEREO streams (monoMixdown), 1836 algorithmic bytes per frame
  The default run prints ONE JSON line for mfcc12 and, inside it under "other_workloads", a short measurement of the other
  three configurations (device-resident value, e2e, per-kernel split, parity check) so that a flag-less driver run records all
  four; --no-others switches that off.

  value : frames/s with PCM already resident in HBM (osm_b200_plan_run_device), CUDA events, barrier + synchronize on both
          sides, max over ranks
  e2e   : the same metric through the C ABI's host entry point (osm_b200_plan_run_host) with pinned HOST buffers allocated on
          the GPU's NUMA node: H2D of the PCM + kernels + D2H of the LLD rows inside the timed region, every step
  roofline     : algorithmic bytes (SURVEY.md 8d) over the measured time vs the measured HBM copy bandwidth -- for mfcc12 of
                 the one fused kernel, for the multi-kernel workloads of the WHOLE step, naming the dominant kernel and its share
                 (per-kernel CUDA events, osm_b200_plan_set_profiling)
  summaries    : (default run, one GPU) the shipped summary configurations end to end -- eGeMAPSv02.conf / ComParE_2016.conf with
                 -csvoutput, 1 000 utterances x 3 s from host PCM to one row of 88 / 6 373 values each (utterances/s); an extra,
                 not a headline number
  parity       : rows of bench utterances (200 for mfcc12) taken from the e2e run's output are compared with the UNMODIFIED
                 reference's rows for the same PCM (per column, 1e-5 of the column scale)
  cpu_baseline : the UNMODIFIED reference on the box's host cores on a bounded sample of the same workload.  Two legs:
                 "value" = start-up free (one smile_initialize per core through the reference's own C API, then smile_run +
                 smile_reset per utterance, oracle/refapi.py), "per_process_value" = one SMILExtract process per utterance
                 (what a shell loop over files gets; dominated by process start-up and component registration).

`--impl reference` times the reference's own CPU implementation as its own line (same legs).
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "LLD frames/sec (16kHz, 25ms/10ms)"
# the shipped openSMILE configurations the workloads run unchanged, stored with the test fixtures
CONFIG_DIR = os.path.join(ROOT, "tests", "golden", "config")
DUMP_BYTES = 8 << 20          # --dump-outputs: at most this many bytes per array (6 arrays stay below 64 MB)


class Workload:
    def __init__(self, key, conf, out_opt, sr, nchan, n_utt, utt_len, rows_per_utt, cols, title, parity_utts):
        self.key, self.conf, self.out_opt, self.sr, self.nchan = key, conf, out_opt, sr, nchan
        self.n_utt, self.utt_len, self.rows_per_utt, self.cols = n_utt, utt_len, rows_per_utt, cols
        self.parity_utts = parity_utts
        hop = sr // 100
        self.bytes_per_frame = hop * nchan * 2 + cols * 4      # each PCM sample read once, each LLD value written once (SURVEY 8d)
        self.title = title % dict(n=n_utt, rows=n_utt * rows_per_utt)


def workload(key):
    n = int(os.environ.get("OSM_BENCH_N_UTT", "0"))
    if key == "mfcc12":
        return Workload(key, "mfcc/MFCC12_0_D_A.conf", "-O", 16000, 1, n or 2000, 400 + 160 * 499, 500, 39,
                        "MFCC12_0_D_A, synthetic 16 kHz mono int16, %(n)d utterances x 500 frames = %(rows)d frames per GPU", 200)
    if key == "egemaps":
        return Workload(key, "egemaps/v02/eGeMAPSv02.conf", "-lldhtkoutput", 16000, 1, n or 10000, 48000, 296, 25,
                        "eGeMAPSv02 LLD set (config/egemaps/v02/eGeMAPSv02.conf unchanged, 25 columns), synthetic 16 kHz mono int16, "
                        "%(n)d utterances x 3.0 s = %(rows)d rows per GPU", 32)
    if key == "compare16":
        return Workload(key, "compare16/ComParE_2016.conf", "-lldhtkoutput", 16000, 1, n or 10000, 48000, 296, 130,
                        "ComParE_2016 full LLD set (config/compare16/ComParE_2016.conf unchanged, 130 columns), synthetic 16 kHz mono "
                        "int16, %(n)d utterances x 3.0 s = %(rows)d rows per GPU", 32)
    if key == "plp44k":
        T = 5000                                   # 50 s streams: 1103 + 441 * 4999 sample frames
        return Workload(key, "plp/PLP_0_D_A.conf", "-O", 44100, 2, n or 100, 1103 + 441 * (T - 1), T, 18,
                        "PLP_0_D_A, synthetic 44.1 kHz STEREO int16 streams (monoMixdown), %(n)d streams x 50 s = %(rows)d frames per GPU", 8)
    raise SystemExit("unknown workload " + key)


# ------------------------------------------------------------------------------------------
def synth_batch_torch(w, device, seed):
    """Voiced-like harmonic source + noise (SURVEY.md 8d formula), generated on the device; stereo = the same source
    with independent noise per channel, the right channel scaled by 0.8."""
    import torch
    g = torch.Generator(device=device).manual_seed(1234 + seed)
    out = torch.empty(w.n_utt * w.utt_len * w.nchan, dtype=torch.int16, device=device)
    chunk = max(1, min(100, (8 << 20) // w.utt_len))            # utterances per chunk (bounds temporaries)
    t = torch.arange(w.utt_len, device=device, dtype=torch.float32) / w.sr
    for u0 in range(0, w.n_utt, chunk):
        n = min(chunk, w.n_utt - u0)
        ph0 = torch.rand(n, 1, device=device, generator=g) * 6.2831853
        f0 = 120.0 + 30.0 * torch.sin(6.2831853 * 0.5 * t[None, :] + ph0)
        phi = 6.2831853 * torch.cumsum(f0, dim=1) / w.sr
        x = torch.zeros(n, w.utt_len, device=device)
        for k in range(1, 20):
            x += torch.sin(k * phi) / k
        chans = []
        for c in range(w.nchan):
            y = (0.1 if c == 0 else 0.08) * x + 0.02 * torch.randn(n, w.utt_len, device=device, generator=g)
            chans.append((y.clamp(-1, 1) * 32767.0).round().to(torch.int16))
        y = chans[0] if w.nchan == 1 else torch.stack(chans, dim=2)
        out[u0 * w.utt_len * w.nchan:(u0 + n) * w.utt_len * w.nchan] = y.reshape(-1)
    return out


class ClockSampler:
    """nvidia-smi clock / throttle sampling during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        self.lines = []
        self.idx = gpu_index

    def start(self):
        if shutil.which("nvidia-smi") is None:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.03)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profile_traffic():
    """dram bytes per launch of the fused kernel from the committed ncu capture, if any."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("lld_kernel_dram_bytes_per_launch")
        except Exception:
            return None
    return None


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank (and therefore its first-touch pinned host buffers and the copy threads of the driver) to the CPUs of
    the NUMA node the GPU hangs off (VERDICT r01 weak #5: at 8 ranks unbound buffers cost 34 % of the e2e rate).
    Returns a description for the JSON line."""
    try:
        import torch
        prop = torch.cuda.get_device_properties(local_rank)
        bus = "%04x:%02x:%02x.0" % (getattr(prop, "pci_domain_id", 0), prop.pci_bus_id, prop.pci_device_id)
        base = "/sys/bus/pci/devices/" + bus
        node = int(open(base + "/numa_node").read().strip())
        cpus = open(base + "/local_cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        ids &= set(os.sched_getaffinity(0))
        if ids:
            os.sched_setaffinity(0, ids)
        return {"pci": bus, "numa_node": node, "cpus": cpus, "bound": bool(ids)}
    except Exception as e:      # no sysfs entry (container) -> run unbound, say so
        return {"bound": False, "why": str(e)[:80]}


def dump_rows(dump_dir, name, rows):
    """Writes rows ([n, k] float32, a torch tensor or a numpy array) as dump_dir/<name>.npy and the numbers of the rows written as
    dump_dir/<name>_row_index.npy (float64).  Above DUMP_BYTES a fixed, seeded sample of rows is written, the same rows in every
    run with the same arguments, so that the outputs of two builds can be compared."""
    n, k = rows.shape
    m = min(n, max(1, DUMP_BYTES // (4 * max(k, 1))))
    idx = np.sort(np.random.default_rng(0).choice(n, size=m, replace=False)) if m < n else np.arange(n)
    if isinstance(rows, np.ndarray):
        sample = rows[idx]
    else:
        import torch
        sample = rows[torch.as_tensor(idx, device=rows.device)].cpu().numpy()
    np.save(os.path.join(dump_dir, name + ".npy"), np.ascontiguousarray(sample, dtype=np.float32))
    np.save(os.path.join(dump_dir, name + "_row_index.npy"), idx.astype(np.float64))


# ------------------------------------------------------------------------------------------
# the unmodified reference on the host cores
# ------------------------------------------------------------------------------------------
def _exec_worker(args):
    """one SMILExtract process per file; returns rows (and the rows themselves when keep=True)"""
    from oracle import refrun
    files, outdir, conf, out_opt, keep = args
    n, rows = 0, []
    for wav in files:
        out = os.path.join(outdir, "%s.%d.htk" % (os.path.basename(wav), os.getpid()))
        subprocess.run([refrun.SMILEXTRACT, "-C", os.path.join(refrun.CONFIG_DIR, conf), "-I", wav, out_opt, out,
                        "-l", "0"], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        if keep:
            rows.append(refrun.read_htk(out)[0])
        else:
            n += refrun.read_htk(out)[1]["n"]
        os.remove(out)
    return rows if keep else n


def _write_wavs(w, n_files, tmpdir, seed):
    from opensmile_b200.synth import voiced_pcm
    from oracle import refrun
    base = [voiced_pcm(w.utt_len, w.sr, seed=seed + i, n_chan=w.nchan) for i in range(min(8, n_files))]
    files = []
    for i in range(n_files):
        p = os.path.join(tmpdir, "u%05d.wav" % i)
        refrun.write_wav(p, base[i % len(base)], w.sr, w.nchan)
        files.append(p)
    return files


def reference_per_process(w, n_files, workers, tmpdir, seed=0):
    """one SMILExtract exec per utterance, `workers` at a time.  (rows, seconds)"""
    from concurrent.futures import ProcessPoolExecutor
    files = _write_wavs(w, n_files, tmpdir, seed)
    shards = [s for s in (files[i::workers] for i in range(workers)) if s]
    with ProcessPoolExecutor(max_workers=len(shards)) as ex:
        list(ex.map(_exec_worker, [([files[0]], tmpdir, w.conf, w.out_opt, False)] * len(shards)))       # warm page cache / binaries
        t0 = time.perf_counter()
        rows = sum(ex.map(_exec_worker, [(s, tmpdir, w.conf, w.out_opt, False) for s in shards]))
        dt = time.perf_counter() - t0
    for p in files:
        os.remove(p)
    return rows, dt


def reference_in_process(w, n_files, workers, tmpdir, seed=0):
    """start-up free: one smile_initialize per worker, smile_run + smile_reset per utterance (oracle/refapi.py).
    (rows, seconds = the slowest worker's timed loop, wall seconds incl. the one-time initialisation)"""
    from concurrent.futures import ProcessPoolExecutor
    from oracle import refapi
    files = _write_wavs(w, n_files, tmpdir, seed)
    shards = [s for s in (files[i::workers] for i in range(workers)) if s]
    t0 = time.perf_counter()
    with ProcessPoolExecutor(max_workers=len(shards)) as ex:
        res = list(ex.map(refapi.worker, [(s, w.conf, w.out_opt, tmpdir, w.rows_per_utt, 1) for s in shards]))
    wall = time.perf_counter() - t0
    for p in files:
        os.remove(p)
    for rows, dt, n_last in res:
        assert n_last == w.rows_per_utt, "reference wrote %d rows per utterance, the workload assumes %d" % (n_last, w.rows_per_utt)
    return sum(r[0] for r in res), max(r[1] for r in res), wall


def sample_sizes(w, cores):
    """bounded samples (about 10-30 s of CPU work over all cores)"""
    per_utt_s = w.rows_per_utt / {"mfcc12": 55e3, "plp44k": 15e3, "egemaps": 4.4e3, "compare16": 5.5e3}[w.key]
    n_in = int(max(2 * cores, min(w.n_utt, 12.0 * cores / (per_utt_s + 0.004))))
    n_in = max(cores, n_in // cores * cores)
    n_ex = max(cores, min(n_in, 4 * cores))
    return n_in, n_ex


def cpu_baseline(w, with_per_process=True, seed=0):
    from oracle import refapi, refrun
    cores = os.cpu_count() or 1
    tmp = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        if refapi.available() and refrun.available():
            n_in, n_ex = sample_sizes(w, cores)
            rows, dt, wall = reference_in_process(w, n_in, cores, tmp, seed)
            cb = {"value": rows / dt, "unit": "frames/s", "cores": cores, "kind": "reference",
                  "sample": "%d of the %d utterances (%d rows) through oracle/_ref/libSMILEapi.so -C %s: one smile_initialize per core, "
                            "smile_run + smile_reset per utterance, WAV in /dev/shm -> HTK out; slowest worker %.2f s (wall incl. "
                            "initialisation %.2f s)" % (n_in, w.n_utt, rows, w.conf, dt, wall),
                  "per_core_value": rows / dt / cores}
            if with_per_process:
                r2, d2 = reference_per_process(w, n_ex, cores, tmp, seed)
                cb["per_process_value"] = r2 / d2
                cb["per_process_sample"] = "%d utterances, one SMILExtract process each (start-up bound), %.2f s" % (n_ex, d2)
            return cb
        # the reference binary did not travel: time the C restatement instead (single thread, MFCC only)
        from opensmile_b200.synth import voiced_pcm
        from oracle import oracle
        pcm = voiced_pcm(80240, 16000, seed=0)
        n = 40
        t0 = time.perf_counter()
        for _ in range(n):
            oracle.mfcc_d_a(pcm, 16000.0)
        dt = time.perf_counter() - t0
        return {"value": n * 500 / dt, "unit": "frames/s", "cores": 1, "kind": "port",
                "sample": "%d MFCC12_0_D_A utterances through oracle/liboracle.so (double-precision FFT restatement), %.2f s" % (n, dt)}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def reference_rows_for(w, pcms):
    """rows of the unmodified reference for a list of int16 utterances (parity check inside the bench)"""
    from concurrent.futures import ProcessPoolExecutor
    from oracle import refrun
    tmp = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        files = []
        for i, x in enumerate(pcms):
            p = os.path.join(tmp, "p%05d.wav" % i)
            refrun.write_wav(p, x, w.sr, w.nchan)
            files.append(p)
        workers = min(len(files), os.cpu_count() or 1)
        shards = [files[i::workers] for i in range(workers)]
        with ProcessPoolExecutor(max_workers=workers) as ex:
            res = list(ex.map(_exec_worker, [(s, tmp, w.conf, w.out_opt, True) for s in shards]))
        out = [None] * len(files)
        for k, rows in enumerate(res):
            for j, r in enumerate(rows):
                out[k + j * workers] = r
        return out
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def parity_check(w, h_pcm, h_out, fo):
    """rows of `parity_utts` utterances spread over the batch vs the unmodified reference; per column, relative to the
    column's scale over the checked rows"""
    from oracle import refrun
    if not refrun.available():
        return {"checked": 0, "why": "reference binary not present"}
    idx = np.unique(np.linspace(0, w.n_utt - 1, w.parity_utts).astype(np.int64))
    L = w.utt_len * w.nchan
    pcms = [np.array(h_pcm[i * L:(i + 1) * L]) for i in idx]
    ref = np.concatenate(reference_rows_for(w, pcms), axis=0)
    got = np.concatenate([np.array(h_out[fo[i]:fo[i + 1]]) for i in idx], axis=0)
    if got.shape != ref.shape:
        return {"checked": int(len(idx)), "ok": False, "why": "shape %s vs reference %s" % (got.shape, ref.shape)}
    err = np.abs(got - ref) / (np.abs(ref).max(axis=0) + 1e-30)
    bad = float((err > 1e-5).mean())
    # Rules.  MFCC / PLP: the only difference to the reference is the FFT's float rounding (2e-7 of a frame's spectral peak, the
    # same distance the reference's own FFT has from the exact transform); on the delta columns, whose scale is 10-20x below the
    # statics', single values reach 1-2e-5 of the column scale: at most 0.01 % of the values may pass 1e-5 and none 5e-5.
    # Feature sets with discontinuous descriptors (arg-max lags, roll-off bins, harmonic picks; SURVEY.md H9): single-row flips
    # are counted, at most 0.2 % of the values.
    if w.key in ("mfcc12", "plp44k"):
        ok = bool(bad <= 1e-4 and err.max() <= 5e-5)
        rule = "<= 0.01 % of the values beyond 1e-5 of their column's scale, none beyond 5e-5"
    else:
        ok = bool(bad <= 2e-3)
        rule = "values beyond 1e-5 of their column's scale (single-row flips of discontinuous descriptors, SURVEY.md H9) counted, <= 0.2 %"
    return {"utterances": int(len(idx)), "rows": int(ref.shape[0]), "columns": int(ref.shape[1]), "tolerance": 1e-5,
            "max_err_of_column_scale": float(err.max()), "share_of_values_beyond_tolerance": bad, "ok": ok, "rule": rule}


# ------------------------------------------------------------------------------------------
def run_reference(args, w, rank, world):
    if rank != 0:
        return
    from oracle import refapi, refrun
    cores = os.cpu_count() or 1
    tmp = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        if not (refapi.available() and refrun.available()):
            cb = cpu_baseline(w)
            v = cb["value"]
            ms = w.rows_per_utt * 1e3 / v
        else:
            n_in, n_ex = sample_sizes(w, cores)
            for _ in range(min(args.warmup, 1)):
                reference_in_process(w, cores, cores, tmp)
            tot_f, tot_t, walls = 0, 0.0, 0.0
            for s in range(args.steps):
                fr, dt, wall = reference_in_process(w, n_in, cores, tmp, seed=s)
                tot_f += fr; tot_t += dt; walls += wall
            v = tot_f / tot_t
            ms = tot_t / args.steps * 1e3
            r2, d2 = reference_per_process(w, n_ex, cores, tmp)
            cb = {"value": v, "unit": "frames/s", "cores": cores, "kind": "reference",
                  "sample": "per step %d of the %d utterances (%d rows) through oracle/_ref/libSMILEapi.so (the reference's own C API: "
                            "smile_initialize once per core, smile_run + smile_reset per utterance), one worker per host core; "
                            "wall incl. per-step initialisation %.2f s per step" % (n_in, w.n_utt, n_in * w.rows_per_utt, walls / args.steps),
                  "per_core_value": v / cores,
                  "per_process_value": r2 / d2,
                  "per_process_sample": "%d utterances, one SMILExtract process each (start-up bound), %.2f s" % (n_ex, d2)}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w.title, "note": "reference is single-threaded per process; %d workers" % cores},
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def make_plan(w, local_rank):
    from opensmile_b200 import Plan, Session, components_mfcc12_0_d_a
    if w.key == "mfcc12":
        return Plan(components_mfcc12_0_d_a(float(w.sr)), "lld", device=local_rank)
    conf = os.path.join(CONFIG_DIR, *w.conf.split("/"))
    opt = {w.out_opt.lstrip("-"): "x.htk"}
    sess = Session(conf, options=opt, device=-1)             # conf front end only; the plan below computes
    comps, level = sess.components(float(w.sr), w.nchan)
    return Plan(list(comps), level, device=local_rank)


def measure(w, args, rank, world, local_rank, dist, steps, with_cpu, sampler=None):
    """one workload on this rank's GPU; returns the JSON-able result dict (rank 0) or None"""
    import torch
    from opensmile_b200.dist import reduce_counters
    dev = torch.device("cuda", local_rank)
    plan = make_plan(w, local_rank)
    off = np.arange(w.n_utt + 1, dtype=np.int64) * w.utt_len
    fo = plan.frame_offsets(off)
    rows = int(fo[-1])
    assert rows == w.n_utt * w.rows_per_utt, (rows, w.n_utt * w.rows_per_utt)
    assert plan.num_elements == w.cols, (plan.num_elements, w.cols)
    d_pcm = synth_batch_torch(w, dev, seed=rank)
    d_out = torch.empty((rows, plan.num_elements), dtype=torch.float32, device=dev)
    h_pcm = torch.empty(w.n_utt * w.utt_len * w.nchan, dtype=torch.int16).pin_memory()
    h_pcm.copy_(d_pcm)
    h_out = torch.empty((rows, plan.num_elements), dtype=torch.float32).pin_memory()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ----
    for _ in range(args.warmup):
        plan.run_device(d_pcm, off, d_out=d_out, frame_offsets=fo)
    barrier()
    if sampler is not None:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    ev0.record()
    for _ in range(steps):
        plan.run_device(d_pcm, off, d_out=d_out, frame_offsets=fo)
        launches += plan.last_launch_count()
    ev1.record()
    barrier()
    dt_ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_rows(args.dump_outputs, w.key + "_lld", d_out)          # the rows of the last timed step
    # kernel times need a sync per step: taken in a separate pass so the timed loop stays free of host synchronisation
    lld_ms, post_ms = [], []
    for _ in range(min(steps, 10)):
        plan.run_device(d_pcm, off, d_out=d_out, frame_offsets=fo)
        a, b = plan.last_kernel_times()
        lld_ms.append(a); post_ms.append(b)
    # per-kernel split of a step (events after every launch, one stream)
    plan.set_profiling(True)
    prof = {}
    for _ in range(3):
        plan.run_device(d_pcm, off, d_out=d_out, frame_offsets=fo)
        torch.cuda.synchronize()
        for nm, ms in plan.kernel_profile():
            prof.setdefault(nm, []).append(ms)
    plan.set_profiling(False)
    n_prof = 3
    kernels = {nm: sum(v) / n_prof for nm, v in prof.items()}

    # ---- end to end through the host entry point (pinned host buffers); the clock sampler keeps running ----
    for _ in range(max(1, min(args.warmup, 3))):
        plan.run_host(h_pcm, off, out=h_out, frame_offsets=fo)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        plan.run_host(h_pcm, off, out=h_out, frame_offsets=fo)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop() if sampler is not None else None

    frames_all, dt_s = reduce_counters(rows * steps, dt_ms * 1e-3, dist, dev)
    frames_e2e, e2e_s = reduce_counters(rows * steps, e2e_s, dist, dev)
    res = None
    if rank == 0:
        value = frames_all / dt_s
        e2e_value = frames_e2e / e2e_s
        ms_step = dt_s * 1e3 / steps
        peak, peak_src = measured_peak_hbm()
        alg = rows * w.bytes_per_frame
        h2d, d2h = int(h_pcm.numel() * 2), int(h_out.numel() * 4)
        dom = max(kernels, key=kernels.get) if kernels else None
        ksum = sum(kernels.values()) or 1.0
        if w.key == "mfcc12":
            k_ms = statistics.mean(lld_ms)
            roof = {"bound": "hbm", "achieved": alg / (k_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                    "traffic": profile_traffic(),
                    "kernel": "lld_kernel<256,32,256,2,VEC2,MFCC>" if os.environ.get("OSM_B200_LLD_FAST", "1")[:1] == "0" else "lld512_kernel<13>",
                    "kernel_ms": k_ms,
                    "post_kernel_ms": statistics.mean(post_ms), "algorithmic_bytes_per_launch": alg, "peak_source": peak_src}
        else:
            roof = {"bound": "hbm", "achieved": alg / (ms_step * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "traffic": None,
                    "kernel": "whole step (%d launches); dominant kernel %s = %.1f %% of the summed kernel time"
                              % (launches // max(steps, 1), dom, 100.0 * kernels[dom] / ksum),
                    "kernel_ms": ms_step, "algorithmic_bytes_per_launch": alg, "peak_source": peak_src,
                    "note": "algorithmic bytes of the WHOLE step over the step's device time"}
        roof["frac"] = roof["achieved"] / peak
        roof["kernels_ms"] = {k: round(v, 4) for k, v in sorted(kernels.items(), key=lambda kv: -kv[1])}
        res = {
            "metric": METRIC, "value": value, "unit": "frames/s",
            "n_gpus": world, "steps": steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": w.title, "frames_per_gpu_per_step": rows,
                       "l2": "no flush needed: per step %d MB PCM in + %d MB rows out exceed the 126 MB L2" % (h2d // 1000000, d2h // 1000000),
                       "parallelism": "utterance shards, one rank per GPU, no data-path collective"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": steps,
                    "api": "osm_b200_plan_run_host (pinned host buffers on the GPU's NUMA node)",
                    "pcie_gbs_per_rank": {"h2d": h2d * steps / e2e_s / 1e9, "d2h": d2h * steps / e2e_s / 1e9}},
            "gpu_launches": launches,
            "roofline": roof,
        }
        res["parity"] = parity_check(w, h_pcm.numpy(), h_out.numpy(), fo)
        if with_cpu:
            res["cpu_baseline"] = cpu_baseline(w, with_per_process=(w.key == "mfcc12"))
    plan.close()
    del d_pcm, d_out, h_pcm, h_out
    torch.cuda.empty_cache()
    return res


def measure_summaries(n_utt=1000, dump_dir=None):
    """SURVEY.md 8(f)-3, reported beside the LLD workloads (not a headline number): the shipped summary configurations end to end
    through the session API from host PCM -- LLD plan, rows resident in HBM, cFunctionals instances + glue, one row per utterance
    copied back.  Wall clock around the blocking call (it synchronises), after one warm-up call on the same batch."""
    import time
    import numpy as np
    from opensmile_b200 import Session
    from opensmile_b200.synth import mixed_pcm
    out = []
    base = [mixed_pcm(48000, 16000, seed=s) for s in range(8)]
    pcm = np.concatenate([base[i % 8] for i in range(n_utt)])
    off = np.arange(n_utt + 1, dtype=np.int64) * 48000
    for rel, tag, key in (("egemaps/v02/eGeMAPSv02.conf", "eGeMAPSv02.conf -csvoutput", "egemaps"),
                          ("compare16/ComParE_2016.conf", "ComParE_2016.conf -csvoutput", "compare16")):
        conf = os.path.join(CONFIG_DIR, rel)
        try:
            s = Session(conf, options={"csvoutput": "x.csv"}, device=0)
            s.extract_pcm(pcm, off, 16000.0, 1)                  # warm-up with the same batch: buffers sized, modules loaded
            t0 = time.perf_counter()
            rows, _ = s.extract_pcm(pcm, off, 16000.0, 1)
            dt = time.perf_counter() - t0
            s.close()
            if dump_dir:
                dump_rows(dump_dir, "summary_" + key, rows)
            out.append({"config": tag, "utterances": n_utt, "seconds_of_audio": 3.0 * n_utt, "values_per_utterance": int(rows.shape[1]),
                        "wall_s": dt, "utterances_per_s": n_utt / dt, "api": "osm_b200_session_extract_pcm (host PCM in, summary rows out)"})
        except Exception as e:      # a reported extra: never takes the bench line down
            out.append({"config": tag, "error": str(e)[:200]})
    return out


def run_ours(args, rank, world, local_rank):
    import torch
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))
    w = workload(args.workload)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    line = measure(w, args, rank, world, local_rank, dist, args.steps, with_cpu=(world == 1), sampler=sampler)
    others = []
    if not args.no_others and args.workload == "mfcc12":
        for key in ("egemaps", "compare16", "plp44k"):
            r = measure(workload(key), args, rank, world, local_rank, dist, max(3, min(args.steps, 5)), with_cpu=(world == 1))
            if r is not None:
                others.append({k: r[k] for k in ("value", "unit", "ms_per_step", "steps", "config", "e2e", "gpu_launches", "roofline",
                                                 "parity", "cpu_baseline") if k in r})
    summaries = measure_summaries(dump_dir=args.dump_outputs) if (world == 1 and not args.no_others and args.workload == "mfcc12") else []
    if rank == 0:
        line["config"]["numa"] = numa
        if others:
            line["other_workloads"] = others
        if summaries:
            line["summaries"] = summaries
        if line.get("parity", {}).get("ok") is False or any(o.get("parity", {}).get("ok") is False for o in others):
            line["parity_failed"] = True
        print(json.dumps(line))
        if line.get("parity_failed"):
            sys.stderr.write("bench.py: PARITY CHECK FAILED -- the numbers above are not valid\n")
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0 and line.get("parity_failed"):
        sys.exit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("OSM_BENCH_WORKLOAD", "mfcc12"), choices=["mfcc12", "egemaps", "compare16", "plp44k"],
                    help="mfcc12 = BASELINE configs[1] (default, the quoted metric); egemaps = configs[2]; compare16 = configs[3]; "
                         "plp44k = configs[4] (44.1 kHz stereo)")
    ap.add_argument("--no-others", action="store_true", default=os.environ.get("OSM_BENCH_NO_OTHERS") == "1",
                    help="mfcc12 only: do not append the short measurements of the other three configurations")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the rows the timed path computed in its last step as DIR/<workload>_lld.npy (float32; a fixed, "
                         "seeded sample of at most 8 MB per array, row numbers in DIR/<name>_row_index.npy) and the summary rows "
                         "as DIR/summary_<config>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, workload(args.workload), rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
