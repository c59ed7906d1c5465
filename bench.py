#!/usr/bin/env python
"""bench.py -- CPI frames/s of the passive-radar hot path (clutter filter -> fast_xambg) on B200.

    python bench.py --gpus N --steps K --warmup W                     # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W    # the reference's CPU path on the host cores
    python bench.py --config c4                                       # NLMS_filter -> fast_xambg, 2M-sample CPI, 512 x 400
    python bench.py --config c5                                       # sweep CPI 256k..4M x Doppler 64..1024 (one line, "sweep": [...])
    python bench.py --dump-outputs DIR                                # also write the maps of the last timed step to DIR

One "step" = ``--frames-per-step`` CPI frames pushed through the frame pipeline: the rank's resident set of
``--resident`` DISTINCT frames (default 125 = BASELINE config 3's 1000-frame stream over 8 GPUs; 2.1 GB, far larger
than the 126 MB L2, so no pass finds its inputs cached) is walked as many times as the step needs.  With the defaults
the timed region is 20 steps x 4000 frames = a few seconds; the SM clocks in the line are sampled INSIDE it.
``value`` = frames/s with the frames already resident in HBM; ``e2e`` = the same through
``FramePipeline.run_host`` with pinned HOST buffers, H2D of both channels and D2H of the map inside the timed region;
``e2e_dropin`` = the reference's own call signatures (LS_Filter -> fast_xambg on pageable numpy arrays) driven from a
thread pool the way main.py's dask scheduler does.  Rank r processes its own frames (weak scaling, no data-path
collective); time = max over ranks.  With N > 1 the line also carries ``config3_stream``: the 1000-frame stream held by
rank 0 and staged to the other ranks over NCCL (double buffered against compute).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIGS = {
    # BASELINE.json configs[1] / [2]: the configuration the metric is quoted on
    "c2": dict(n=2 ** 20, F=256, R=300, filter_len=300, peek=10, reg=1.0, clutter="ls",
               name="1M-sample CPI (2^20), 256 Doppler x 300 range, LS_Filter(filterLen=300, reg=1, peek=10) -> fast_xambg(kaiser 5.0)"),
    # BASELINE.json configs[0]: the reference's CPU-runnable plumbing case
    "c1": dict(n=200_000, F=64, R=100, filter_len=100, peek=10, reg=1.0, clutter="ls",
               name="200k-sample CPI, 64 Doppler x 100 range, LS_Filter -> fast_xambg"),
    # BASELINE.json configs[3]: NLMS clutter variant (block_len 1 = the reference's NLMS_filter; --nlms-block B = block_NLMS)
    "c4": dict(n=2 ** 21, F=512, R=400, filter_len=400, peek=10, mu=0.05, clutter="nlms",
               name="2M-sample CPI (2^21), 512 Doppler x 400 range, NLMS_filter(filterLen=400, mu=0.05, peek=10) -> fast_xambg(kaiser 5.0)"),
}
# not a BASELINE config: the chunk main.py really processes with the shipped PRconfig.yaml (config.py:13-59 -> N = 524 288,
# F = 1024, R = 175; clutter filter main.py:169-176 = LS_Filter_Multiple over five Doppler bins at the IF rate)
CONFIGS["main"] = dict(n=524288, F=1024, R=175, filter_len=175, peek=10, clutter="multi", bins=[0.0, 1.0, -1.0, 2.0, -2.0],
                       fs=2.4e6 * 13 / 119,
                       name="PRconfig.yaml chunk: 524288-sample CPI, 1024 Doppler x 175 range, LS_Filter_Multiple(175, [0,1,-1,2,-2]) -> fast_xambg(kaiser 5.0)")
SWEEP_N = [2 ** 18, 2 ** 19, 2 ** 20, 2 ** 21, 2 ** 22]
SWEEP_F = [64, 256, 1024]
METRIC = "CPI frames/sec (1M-sample CPI, 256 Doppler x 300 range)"
UNIT = "frames/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS) + ["c5"])
    ap.add_argument("--resident", type=int, default=0, help="distinct frames resident in HBM per GPU (0 = per config)")
    ap.add_argument("--frames-per-step", type=int, default=0, help="frames per step per GPU (0 = per config)")
    ap.add_argument("--batch", type=int, default=25, help="frames per library call (one launch of each kernel); 125 resident frames = 5 calls")
    ap.add_argument("--slots", type=int, default=5, help="concurrent CUDA streams of the frame pipeline (measured: 25 x 5 38.2k, 16 x 3 34.9k frames/s)")
    ap.add_argument("--profile", default="P1", choices=["P0", "P1"])
    ap.add_argument("--nlms-block", type=int, default=1, help="config c4: block_len of block_NLMS (1 = NLMS_filter)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stream", action="store_true", help="skip the config-3 NCCL staging measurement at N > 1")
    ap.add_argument("--cpu-procs", type=int, default=0, help="worker processes of the CPU arm (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the range-Doppler maps of the last timed step to DIR/*.npy (see dump_maps)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.config == "c5"):
        ap.error("--dump-outputs writes the maps of the GPU arm of one configuration (not --impl reference or --config c5)")
    return args


def config_dict(cfg, args, world):
    """The `config` object of the JSON line -- identical on both arms."""
    return {"workload": cfg["name"], "profile": args.profile, "n": cfg["n"], "doppler_bins": cfg["F"], "range_bins": cfg["R"],
            "clutter_filter": {"ls": "LS_Filter", "multi": "LS_Filter_Multiple"}.get(cfg["clutter"]) or ("NLMS_filter" if args.nlms_block == 1 else f"block_NLMS(blockLen={args.nlms_block})"),
            "parallelism": f"frames sharded over {world} GPU(s), no collective on the data path"}


# ----------------------------------------------------------------------------- bytes
def bytes_frame(n, F, R):
    """Compulsory HBM bytes per frame (SURVEY.md 8d): read ref+srv once, write the map once."""
    return 2 * 8 * n + 8 * F * (R + 1)


def kernel_alg_bytes(cfg):
    """Algorithmic bytes per FRAME for each kernel of the frame (DESIGN.md section 4)."""
    n, F, R = cfg["n"], cfg["F"], cfg["R"]
    M = cfg["filter_len"] + cfg["peek"]
    nb = len(cfg.get("bins", [0]))
    return {
        "lagcorr_ls": nb * (2 * 8 * n + 2 * 8 * M), # read ref, srv; write 2 x M correlation lags (per Doppler bin of LS_Filter_Multiple)
        "levinson": 2 * 8 * M + 8 * M,
        "fir_apply": nb * 3 * 8 * n,                # read ref, srv; write cleaned srv
        "lagcorr_caf": 2 * 8 * n + 4 * n + 8 * F * (R + 1),   # ref, srv, f32 window; block sums
        "doppler_fft": 2 * 8 * F * (R + 1),
        "nlms": 3 * 8 * n,
    }


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin=None, t_end=None):
        """Summary of the samples taken in [t_begin, t_end] (perf_counter seconds); all samples when None."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, r in self.rows:
            if t_begin is not None and not (t_begin <= ts <= t_end):
                continue
            parts = [x.strip() for x in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
                power.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(smax)) if smax else None,
                "power_w_max": float(max(power)) if power else None,
                "samples": len(sm), "sampled": "inside the timed region", "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- CPU arm
def _ref_modules():
    """(LS_Filter, NLMS_filter, fast_xambg, kind): the UNMODIFIED reference functions from baseline/_ref when the
    recipe baseline/install_ref.py has been run (kind "reference"), else the oracle port (kind "port")."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(os.path.join(ref_dir, "passiveRadar")):
        if ref_dir not in sys.path:
            sys.path.insert(0, ref_dir)
        from passiveRadar.clutter_removal import LS_Filter, NLMS_filter, LS_Filter_Multiple
        from passiveRadar.range_doppler_processing import fast_xambg
        _ref_modules.multi = LS_Filter_Multiple
        return LS_Filter, NLMS_filter, fast_xambg, "reference"
    from oracle import clutter_oracle as co
    from oracle import xambg_oracle as xo
    _ref_modules.multi = co.ls_filter_multiple_oracle
    return co.ls_filter_oracle, co.nlms_filter_oracle, xo.fast_xambg_oracle, "port"


def _install_decimate_shim():
    """SciPy >= 1.12's decimate(ftype=dlti) detours through dlti._as_zpk() -> np.roots of degree n/F PER RANGE LAG
    (46 s per lag at 4096) before doing the FIR it was asked for; route FIR dlti straight to resample_poly, which is
    what decimate ends up calling -- bit-identical output (tests/test_oracle_golden.py::test_shim_is_bit_identical...).
    This patches a SciPy function for the CPU arm; the reference's own code is untouched."""
    import scipy.signal as signal
    if getattr(signal.decimate, "_prc_shim", False):
        return
    real = signal.decimate

    def patched(x, q, n=None, ftype='iir', axis=-1, zero_phase=True):
        if isinstance(ftype, signal.dlti) and zero_phase:
            tf = ftype._as_tf()
            den = np.atleast_1d(tf.den)
            if den.shape[0] == 1:
                return signal.resample_poly(x, 1, q, axis=axis, window=tf.num / tf.den)
        return real(x, q, n=n, ftype=ftype, axis=axis, zero_phase=zero_phase)

    patched._prc_shim = True
    signal.decimate = patched


def _cpu_sample_worker(job):
    """One bounded sample of a frame on the CPU: the clutter filter on n/div samples with the full tap count (its cost
    is linear in n: data matrix, Gram and solve for LS_Filter, the recurrence for NLMS_filter) and fast_xambg on the
    FULL frame with all range lags.  Returns (estimated seconds for one whole frame, filter seconds, xambg seconds)."""
    cfg, seed_frame, div, profile, nlms_block, lag_div = job
    import scipy.signal as signal
    from passiveradar_b200 import synth
    LS_Filter, NLMS_filter, fast_xambg, kind = _ref_modules()
    _install_decimate_shim()
    n, F, R = cfg["n"], cfg["F"], cfg["R"]
    ref, srv = synth.make_frame(n, profile, seed_frame)
    w = signal.get_window(("kaiser", 5.0), n)
    ns = n // div
    t0 = time.perf_counter()
    if cfg["clutter"] == "ls":
        LS_Filter(ref[:ns], srv[:ns], cfg["filter_len"], cfg["reg"], cfg["peek"])
    elif cfg["clutter"] == "multi":
        _ref_modules.multi(ref[:ns], srv[:ns], cfg["filter_len"], cfg["fs"], cfg["bins"])
    else:
        NLMS_filter(ref[:ns], srv[:ns], cfg["filter_len"], cfg["mu"], cfg["peek"])
    t_f = time.perf_counter() - t0
    t0 = time.perf_counter()
    Rs = (R + 1) // lag_div - 1                      # lag_div > 1: a subset of the range lags (every lag costs the same)
    fast_xambg(ref, srv, Rs, F, n, w)
    t_x = time.perf_counter() - t0
    return t_f * div + t_x * (R + 1) / (Rs + 1), t_f, t_x


def cpu_full_frame(cfg, profile, timeout=240):
    """ONE whole frame through the reference's own functions in one process with all BLAS threads: nothing sampled,
    nothing extrapolated.  It checks the scaling of the pool's bounded sample (one frame takes about a minute and 8 GB,
    which is why the pool does not do this in every worker).  Returns a dict or None."""
    code = (
        "import json, sys, time, numpy as np\n"
        f"sys.path.insert(0, {ROOT!r})\n"
        "import bench\n"
        "import scipy.signal as signal\n"
        "from passiveradar_b200 import synth\n"
        f"cfg = {cfg!r}\n"
        "LS_Filter, NLMS_filter, fast_xambg, kind = bench._ref_modules()\n"
        "bench._install_decimate_shim()\n"
        f"ref, srv = synth.make_frame(cfg['n'], {profile!r}, 999)\n"
        "w = signal.get_window(('kaiser', 5.0), cfg['n'])\n"
        "t0 = time.perf_counter()\n"
        "clean = LS_Filter(ref, srv, cfg['filter_len'], cfg['reg'], cfg['peek'])\n"
        "t1 = time.perf_counter()\n"
        "fast_xambg(ref, clean, cfg['R'], cfg['F'], cfg['n'], w)\n"
        "t2 = time.perf_counter()\n"
        "print(json.dumps({'ls_seconds': t1 - t0, 'xambg_seconds': t2 - t1, 'kind': kind}))\n")
    env = dict(os.environ)
    for k in ("OPENBLAS_NUM_THREADS", "OMP_NUM_THREADS", "MKL_NUM_THREADS"):
        env.pop(k, None)
    try:
        res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=timeout, env=env)
        if res.returncode != 0:
            return None
        out = json.loads(res.stdout.strip().splitlines()[-1])
        out["frames_per_s_one_process"] = 1.0 / (out["ls_seconds"] + out["xambg_seconds"])
        out["note"] = "one whole frame, LS_Filter -> fast_xambg, one process, default BLAS threads, no sampling"
        return out
    except Exception:
        return None


class CpuArm:
    """Frame-parallel pool, one process per host core (1 BLAS thread each), as SURVEY 8d asks."""

    def __init__(self, cfg, procs, profile, nlms_block=1, bounded=False, blas_threads=0):
        """bounded=False: the sample of `cpu_baseline` (one round: fast_xambg on the whole frame, every lag measured).
        bounded=True: the reference arm's step, repeated steps + warmup times, so a step is cut to a few seconds
        (fast_xambg on 1/8 of the range lags, clutter filter on a shorter piece)."""
        import multiprocessing as mp
        self.bounded = bounded
        self.cfg = cfg
        self.profile = profile
        self.nlms_block = nlms_block
        ncpu = os.cpu_count() or 1
        try:
            ncpu = len(os.sched_getaffinity(0))
        except (AttributeError, OSError):
            pass
        # bounded sample: LS_Filter at full size builds a 2.6 GB data matrix twice over (33-62 s, 8 GB RSS per frame);
        # n/8 keeps a worker at ~1 GB and a few seconds.  NLMS_filter is a Python loop of 8.8 us per sample: n/32.
        big = cfg["n"] >= 2 ** 19
        self.div = {"ls": 8, "multi": 1}.get(cfg["clutter"], 32) if big else 1      # LS_Filter_Multiple: Toeplitz filters, whole frame measured
        self.lag_div = 1
        if bounded and big:
            self.div *= 4
            self.lag_div = 8
        try:
            mem_gb = os.sysconf("SC_PHYS_PAGES") * os.sysconf("SC_PAGE_SIZE") / 2 ** 30
        except (ValueError, OSError):
            mem_gb = 16
        # measured on the GPU box's host (128 logical CPUs, profiles/r02_cpu_pool.log): the workers are memory-bandwidth
        # bound; 32 workers x 4 BLAS threads give the best whole-pool rate (0.51 frames/s; 64 x 2: 0.47, 16 x 8: 0.44,
        # 8 x 16: 0.27), so the arm uses one worker per four logical CPUs
        self.procs = procs if procs > 0 else max(1, min(ncpu // 4 if ncpu >= 8 else ncpu, int(mem_gb // 3), 64))
        self.blas_threads = blas_threads if blas_threads > 0 else max(1, ncpu // self.procs)
        for k in ("OPENBLAS_NUM_THREADS", "OMP_NUM_THREADS", "MKL_NUM_THREADS"):
            os.environ[k] = str(self.blas_threads)
        self.kind = _ref_modules()[3]
        self.pool = mp.get_context("spawn").Pool(self.procs)
        self.round = 0

    def step(self):
        """One round: every worker processes one bounded sample.  Returns (frames/s, wall seconds, est s/frame)."""
        jobs = [(self.cfg, 1000 + self.round * self.procs + i, self.div, self.profile, self.nlms_block, self.lag_div)
                for i in range(self.procs)]
        self.round += 1
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_sample_worker, jobs)
        wall = time.perf_counter() - t0
        est = [r[0] for r in res]
        sampled = [r[1] + r[2] for r in res]
        # whole-frame throughput of the pool = procs / (mean estimated whole-frame seconds), corrected by how much
        # slower the round ran than its slowest worker's own compute (pool overhead)
        eff = max(sampled) / wall if wall > 0 else 1.0
        fps = self.procs / float(np.mean(est)) * min(1.0, eff)
        return fps, wall, float(np.mean(est)), float(np.mean([r[1] for r in res])), float(np.mean([r[2] for r in res]))

    def sample_text(self):
        c = self.cfg
        flt = {"ls": "LS_Filter", "multi": "LS_Filter_Multiple"}.get(c["clutter"], "NLMS_filter")
        src = "the reference's own functions (baseline/_ref, unmodified)" if self.kind == "reference" else "the oracle port"
        ext = (f"{flt} on n/{self.div} = {c['n'] // self.div} samples with all {c['filter_len'] + c['peek']} taps, time x{self.div} "
               f"(EXTRAPOLATED: cost linear in n)") if self.div > 1 else f"{flt} on the full frame"
        lags = (f"all {c['R'] + 1} range lags (measured" if self.lag_div == 1 else
                f"{(c['R'] + 1) // self.lag_div} of {c['R'] + 1} range lags, time x{(c['R'] + 1) / ((c['R'] + 1) // self.lag_div):.2f} (EXTRAPOLATED: every lag costs the same")
        return (f"per worker, {src}: {ext} + fast_xambg on the FULL {c['n']}-sample frame, {lags}; scipy.signal.decimate's np.roots "
                f"detour bypassed bit-identically); {self.procs} workers in parallel, {self.blas_threads} BLAS thread(s) each")

    def close(self):
        self.pool.terminate()
        self.pool.join()


def run_reference(args, cfg, rank, world):
    if rank != 0:
        return
    arm = CpuArm(cfg, args.cpu_procs, args.profile, args.nlms_block, bounded=(args.steps + args.warmup) > 3)
    try:
        for _ in range(args.warmup):
            arm.step()
        fps_list = []
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fps_list.append(arm.step()[0])
        total = time.perf_counter() - t0
    finally:
        arm.close()
    value = float(np.mean(fps_list))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "c64 (f32 pairs; f64 block sums)",
        "data": "synthetic", "config": config_dict(cfg, args, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.procs * arm.blas_threads, "workers": arm.procs, "kind": arm.kind,
                         "sample": arm.sample_text(), "filter_extrapolated": arm.div > 1, "xambg_extrapolated": arm.lag_div > 1},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU arm helpers
def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "sm_max_mhz": float(p.get("sm_max_mhz", 1965.0)),
                "source": "MEASURED_PEAKS.json (measured copy bandwidth)", "of": "of measured"}
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "source": "fallback (B200_PROFILING.md)", "of": "of fallback"}


def make_resident(torch, dev, n, profile, count, rank, base=8):
    """`count` DISTINCT frames on the device: `base` frames from the seeded host generator (the ones the parity tests
    use), the rest derived on the device by a circular roll of both channels (different per frame) and a unit phasor --
    same statistics, same clutter geometry (the LS model is circular), different samples."""
    from passiveradar_b200 import synth
    base = min(base, count)
    refs, srvs = zip(*[synth.make_frame(n, profile, rank * 1000 + i) for i in range(base)])
    bref = torch.from_numpy(np.stack(refs)).to(dev)
    bsrv = torch.from_numpy(np.stack(srvs)).to(dev)
    ref_d = torch.empty((count, n), dtype=torch.complex64, device=dev)
    srv_d = torch.empty((count, n), dtype=torch.complex64, device=dev)
    for i in range(count):
        k, g = i % base, i // base
        if g == 0:
            ref_d[i] = bref[k]
            srv_d[i] = bsrv[k]
        else:
            ph = complex(np.exp(2j * np.pi * (0.137 * g + 0.011 * k)))
            sh = (7919 * g + 104729 * k) % n
            ref_d[i] = torch.roll(bref[k], sh) * ph
            srv_d[i] = torch.roll(bsrv[k], sh) * ph
    return ref_d, srv_d, np.stack(refs), np.stack(srvs)


DUMP_BYTES = 64 * 10 ** 6


def dump_maps(out_dir, maps_d, rank, world):
    """Write the maps the last timed step computed (`maps_d`, one per resident frame it covered) so that two builds can be
    compared map for map on the same seeded inputs: maps[.npy] = float32 (frames, F, R+1, 2) real/imaginary pairs, and
    frame_index[.npy] = which resident frames they are (float64).  All frames when they fit in DUMP_BYTES over all ranks,
    else a fixed seeded sample of frames.  With N > 1 each rank writes its own pair of files (suffix _rank<r>)."""
    import torch
    count = maps_d.shape[0]
    keep = min(count, DUMP_BYTES // world // (maps_d[0].numel() * 8 + 8))
    idx = np.arange(count) if keep == count else np.sort(np.random.default_rng(0).choice(count, keep, replace=False))
    maps = torch.view_as_real(maps_d[torch.from_numpy(idx).to(maps_d.device)]).cpu().numpy()
    suffix = f"_rank{rank}" if world > 1 else ""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"maps{suffix}.npy"), maps)
    np.save(os.path.join(out_dir, f"frame_index{suffix}.npy"), idx.astype(np.float64))


class Workload:
    """What one step runs, per config: c2/c1 the fused LS frame pipeline; c4 NLMS_filter (one CTA per frame, the batch
    fills the GPU) followed by the batched CAF of the cleaned channels."""

    def __init__(self, args, cfg, torch, dev, local_rank):
        from passiveradar_b200 import _lib
        from passiveradar_b200.frames import FramePipeline
        self.args, self.cfg, self.torch, self.dev = args, cfg, torch, dev
        self.lib = _lib.load()
        self._lib = _lib
        n, F, R = cfg["n"], cfg["F"], cfg["R"]
        self.n, self.F, self.R = n, F, R
        self.local_rank = local_rank
        self.bins = np.ascontiguousarray(cfg.get("bins", [0.0]), dtype=np.float64)
        if cfg["clutter"] == "ls":
            self.pipe = FramePipeline(n, R, F, filter_len=cfg["filter_len"], reg=cfg["reg"], peek=cfg["peek"],
                                      window=("kaiser", 5.0), device=local_rank, nslots=args.slots, batch=args.batch)
        else:
            import scipy.signal as signal
            self.window = torch.from_numpy(signal.get_window(("kaiser", 5.0), n).astype(np.float32)).to(dev)
            self.clean = None
            self.stream = torch.cuda.Stream(device=dev)       # the library keeps one workspace per caller stream

    def run_device(self, ref_d, srv_d, maps_d):
        if self.cfg["clutter"] == "ls":
            self.pipe.run_device(ref_d, srv_d, maps_d)
            return
        torch, _lib, c = self.torch, self._lib, self.cfg
        nf = ref_d.shape[0]
        if self.clean is None or self.clean.shape[0] < nf:
            self.clean = torch.empty((nf, self.n), dtype=torch.complex64, device=self.dev)
        cur = torch.cuda.current_stream(self.dev)
        self.stream.wait_stream(cur)
        st = self.stream.cuda_stream
        flags = _lib.FLAG_ASYNC | _lib.FLAG_WINDOW_F32
        if c["clutter"] == "multi":
            stride = ref_d.stride(0) if nf > 1 else self.n
            assert stride == self.n, "bench frames are contiguous"
            _lib.check(self.lib.prc_ls_multiple_frames_c64(ref_d.data_ptr(), srv_d.data_ptr(), self.n, nf, stride, c["filter_len"], c["peek"],
                                                           c["fs"], self.bins.ctypes.data, len(self.bins), self.clean.data_ptr(),
                                                           _lib.MEM_DEVICE, self.local_rank, st, _lib.FLAG_ASYNC))
            _lib.check(self.lib.prc_xambg_frames_c64(ref_d.data_ptr(), self.clean.data_ptr(), self.n, nf, stride, self.R, self.F,
                                                     self.window.data_ptr(), maps_d.data_ptr(), _lib.MEM_DEVICE, self.local_rank, st, flags))
            cur.wait_stream(self.stream)
            return
        _lib.check(self.lib.prc_nlms_frames_c64(ref_d.data_ptr(), srv_d.data_ptr(), self.n, nf, ref_d.stride(0) if nf > 1 else self.n,
                                                c["filter_len"], c["peek"], c["mu"], self.args.nlms_block, None,
                                                self.clean.data_ptr(), None, _lib.MEM_DEVICE, self.local_rank, st, _lib.FLAG_ASYNC))
        _lib.check(self.lib.prc_xambg_frames_c64(ref_d.data_ptr(), self.clean.data_ptr(), self.n, nf, self.n, self.R, self.F,
                                                 self.window.data_ptr(), maps_d.data_ptr(), _lib.MEM_DEVICE, self.local_rank, st, flags))
        cur.wait_stream(self.stream)

    def run_host(self, ref_h, srv_h, maps_h, stage):
        if self.cfg["clutter"] == "ls":
            self.pipe.run_host(ref_h, srv_h, maps_h)
            return
        torch = self.torch
        rd, sd, md = stage
        nf = ref_h.shape[0]
        rd[:nf].copy_(torch.from_numpy(ref_h), non_blocking=True)
        sd[:nf].copy_(torch.from_numpy(srv_h), non_blocking=True)
        self.run_device(rd[:nf], sd[:nf], md[:nf])
        torch.from_numpy(maps_h.reshape(nf, self.F, self.R + 1)).copy_(md[:nf], non_blocking=True)
        torch.cuda.synchronize(self.dev)


def time_passes(torch, dev, work, ref_d, srv_d, maps_d, frames):
    """Walk the resident set until `frames` frames have been processed (enqueue only)."""
    res = ref_d.shape[0]
    done = 0
    while done < frames:
        m = min(res, frames - done)
        work.run_device(ref_d[:m], srv_d[:m], maps_d[:m])
        done += m


def run_b200(args, cfg, rank, world, local_rank, quiet=False):
    import torch
    import torch.distributed as dist
    from passiveradar_b200 import _lib
    from passiveradar_b200.frames import pinned_empty

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: libprcore has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)

    n, F, R = cfg["n"], cfg["F"], cfg["R"]
    nlms = cfg["clutter"] == "nlms"
    direct = cfg["clutter"] != "ls"          # clutter filter and CAF as two batched library calls (no FramePipeline)
    resident = args.resident or (444 if nlms else 125)
    fps_guess = 450.0 if nlms else 25000.0
    frames_per_step = args.frames_per_step or (resident if nlms else 4000)
    work = Workload(args, cfg, torch, dev, local_rank)
    ref_d, srv_d, ref_base, srv_base = make_resident(torch, dev, n, args.profile, resident, rank)
    maps_d = torch.empty((resident, F, R + 1), dtype=torch.complex64, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput (headline `value`)
    warm = max(args.warmup, 3)
    for _ in range(warm):
        time_passes(torch, dev, work, ref_d, srv_d, maps_d, min(frames_per_step, 2 * resident))
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        time_passes(torch, dev, work, ref_d, srv_d, maps_d, frames_per_step)
    e1.record()
    barrier()
    t_end = time.perf_counter()
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
    frames_total = frames_per_step * args.steps * world
    value = frames_total / (ms * 1e-3)
    if args.dump_outputs:
        # a step walks the resident set from frame 0, so the last one wrote the maps of its first min(resident, frames) frames
        dump_maps(args.dump_outputs, maps_d[:min(resident, frames_per_step)], rank, world)

    # ---- end to end through the public API with host buffers (pinned), copies inside the timed region
    nb_host = ref_base.shape[0]
    if nlms:
        nb_host = 148                # NLMS runs one CTA per frame: a call must carry enough frames to use the GPU
    ref_h = pinned_empty((nb_host, n))
    srv_h = pinned_empty((nb_host, n))
    for i in range(nb_host):
        ref_h[i] = ref_base[i % ref_base.shape[0]]
        srv_h[i] = srv_base[i % srv_base.shape[0]]
    maps_h = pinned_empty((nb_host, F, R + 1, 1))
    stage = None
    if direct:
        stage = (torch.empty((nb_host, n), dtype=torch.complex64, device=dev), torch.empty((nb_host, n), dtype=torch.complex64, device=dev),
                 torch.empty((nb_host, F, R + 1), dtype=torch.complex64, device=dev))
    e2e_frames_per_step = max(nb_host, int(round((148 if nlms else 640) / nb_host)) * nb_host)
    passes = e2e_frames_per_step // nb_host
    for _ in range(2):
        work.run_host(ref_h, srv_h, maps_h, stage)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for _ in range(passes):
            work.run_host(ref_h, srv_h, maps_h, stage)      # synchronises before returning
    torch.cuda.synchronize(dev)
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_total = e2e_frames_per_step * args.steps * world
    e2e_value = e2e_total / e2e_s

    # ---- the reference's own call signatures from a thread pool (main.py:169-194 under dask's threaded scheduler):
    # pageable numpy arrays in, numpy arrays out, one library workspace per calling thread
    dropin = None
    if rank == 0 and not direct and not quiet:
        import concurrent.futures as cf
        import scipy.signal as signal
        import passiveradar_b200 as prb
        w64 = signal.get_window(("kaiser", 5.0), n)
        pairs = [(np.array(ref_base[i % ref_base.shape[0]]), np.array(srv_base[i % srv_base.shape[0]])) for i in range(8)]

        def one(i):
            r, s = pairs[i % 8]
            cleaned = prb.LS_Filter(r, s, cfg["filter_len"], cfg["reg"], cfg["peek"])
            return prb.fast_xambg(r, cleaned, R, F, n, w64)

        nthr, ncall = 8, 48
        with cf.ThreadPoolExecutor(nthr) as ex:
            list(ex.map(one, range(nthr)))
            t0 = time.perf_counter()
            list(ex.map(one, range(ncall)))
            dt = time.perf_counter() - t0
        dropin = {"value": ncall / dt, "unit": UNIT, "threads": nthr, "calls": ncall,
                  "api": "passiveradar_b200.LS_Filter -> passiveradar_b200.fast_xambg (reference signatures, pageable numpy in/out, float64 window)"}

    # ---- what the host link can carry: plain pinned-memory H2D copies of the same buffers, nothing else running
    h2d_peak = None
    try:
        if rank == 0 and not quiet:
            src = torch.from_numpy(ref_h.reshape(-1).view(np.float32))
            dst = torch.empty_like(src, device=dev)
            dst.copy_(src, non_blocking=True)
            torch.cuda.synchronize(dev)
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for _ in range(4):
                dst.copy_(src, non_blocking=True)
            c1.record()
            torch.cuda.synchronize(dev)
            h2d_peak = 4 * src.numel() * 4 / (c0.elapsed_time(c1) * 1e-3) / 1e9
            del dst
    except Exception:       # context only: never let it break the bench line
        h2d_peak = None

    # ---- per-kernel durations (CUDA events on the launching stream around every launch, one stream, the same batch
    # size as the timed region, walking the resident set: inputs > L2) and single-frame latency
    roofline, per_kernel, latency_us = None, {}, None
    if rank == 0:
        peaks = load_peaks()
        args1 = argparse.Namespace(**vars(args))
        args1.slots = 1
        single = Workload(args1, cfg, torch, dev, local_rank)
        m = min(resident, 4 * args.batch) if not nlms else resident
        single.run_device(ref_d[:m], srv_d[:m], maps_d[:m])
        torch.cuda.synchronize(dev)
        _lib.profile_reset()
        _lib.profile(True)
        reps = 2 if nlms else 8
        for r in range(reps):
            o = (r * m) % max(1, resident - m + 1)
            single.run_device(ref_d[o:o + m], srv_d[o:o + m], maps_d[o:o + m])
        torch.cuda.synchronize(dev)
        prof = _lib.profile_read()
        _lib.profile(False)
        frames_prof = reps * m
        algb = kernel_alg_bytes(cfg)
        tot = sum(v[0] for v in prof.values())
        for name, (tms, cnt) in prof.items():
            if cnt == 0:
                continue
            us_frame = 1e3 * tms / frames_prof
            per_kernel[name] = {"us_per_frame": round(us_frame, 3), "avg_launch_us": round(1e3 * tms / cnt, 2), "launches": cnt,
                                "frames_per_launch": round(frames_prof / cnt, 2), "share": round(tms / tot, 4) if tot else None,
                                "alg_GBps": round(algb[name] / (us_frame * 1e-6) / 1e9, 1) if name in algb else None}
        # dominant kernel = largest share of the serialised kernel time, whatever it is
        dom = max(per_kernel, key=lambda k: prof[k][0])
        fpl = per_kernel[dom]["frames_per_launch"]
        traffic, traffic_note = None, None
        tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            ent = tj.get(args.config, {}).get(dom)
            if ent:
                traffic = ent["dram_bytes_per_frame"] * fpl
                traffic_note = ent.get("note")
        ach = per_kernel[dom]["alg_GBps"]
        frame_gbps = bytes_frame(n, F, R) * value / world / 1e9
        roofline = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": round(ach / peaks["hbm_gbs"], 5) if ach else None, "traffic": traffic,
                    "algorithmic_bytes_per_launch": algb.get(dom, 0) * fpl, "avg_launch_us": per_kernel[dom]["avg_launch_us"],
                    "frames_per_launch": fpl, "traffic_note": traffic_note,
                    "frame_GBps": round(frame_gbps, 1), "frame_frac": round(frame_gbps / peaks["hbm_gbs"], 5),
                    "note": "frac: the dominant kernel's algorithmic bytes over its CUDA-event duration (timed inside a run of back-to-back "
                            "launches) against the measured HBM copy bandwidth; frame_frac: the whole frame's compulsory bytes "
                            "(2*8*n + 8*F*(R+1)) x the headline frames/s against the same peak. Kernels named by stage: lagcorr_ls = "
                            "LS lag sums, levinson = float64 Toeplitz solve (one CTA per frame, latency-bound), lagcorr_caf = CAF block "
                            "sums (clutter filter fused in), doppler_fft, misc = taps spectrum.",
                    "peak_source": peaks["source"] + ", " + peaks["of"],
                    "path": "fft" if _lib.get_option("fft") else "direct (tcgen05 / FP32)"}
        # single-frame latency: one frame, one stream, synchronised
        if not direct:
            lat = Workload(args1, cfg, torch, dev, local_rank)
            lat.pipe.batch = 1
            for _ in range(3):
                lat.run_device(ref_d[:1], srv_d[:1], maps_d[:1])
            torch.cuda.synchronize(dev)
            l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0.record()
            for i in range(20):
                lat.run_device(ref_d[i:i + 1], srv_d[i:i + 1], maps_d[i:i + 1])
            l1.record()
            torch.cuda.synchronize(dev)
            latency_us = round(1e3 * l0.elapsed_time(l1) / 20, 1)

    # ---- config 3: the 1000-frame stream held by rank 0, staged over NCCL, double buffered against compute
    stream = None
    if world > 1 and not args.no_stream and not direct:
        from passiveradar_b200 import distributed as pd
        stream = pd.stream_benchmark(work.pipe, ref_d, srv_d, maps_d, nframes_total=1000, chunk=args.batch, rank=rank, world=world,
                                     device=dev)

    # ---- CPU baseline beside it (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        arm = CpuArm(cfg, args.cpu_procs, args.profile, args.nlms_block)
        try:
            fps, wall, est, t_f, t_x = arm.step()
            cpu = {"value": fps, "unit": UNIT, "cores": arm.procs * arm.blas_threads, "workers": arm.procs, "kind": arm.kind, "sample": arm.sample_text(),
                   "est_seconds_per_frame_per_core": est, "filter_seconds_sampled": t_f, "xambg_seconds_full_frame": t_x,
                   "filter_extrapolated": arm.div > 1, "wall_s": wall}
        finally:
            arm.close()
        if cfg["clutter"] == "ls":
            cpu["full_frame_check"] = cpu_full_frame(cfg, args.profile)

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "c64 (f32 pairs: FP32 FFT-domain block correlations; f64 Toeplitz solve)" if not nlms else "c64 (f32 pairs)",
            "metric_note": None if args.config in ("c2", "c3") else f"frames/s of config {args.config!r}, not of the headline configuration",
            "data": "synthetic", "config": config_dict(cfg, args, world),
            "run": {"frames_per_step_per_gpu": frames_per_step, "resident_distinct_frames_per_gpu": resident,
                    "frames_per_call": args.batch, "slots": args.slots, "timed_region_s": round(ms * 1e-3, 3),
                    "cache": f"resident set {resident * 2 * n * 8 / 2 ** 20:.0f} MiB per GPU > 126 MB L2 (no flush needed)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": e2e_frames_per_step * 2 * n * 8,
                    "d2h_bytes_per_step": e2e_frames_per_step * F * (R + 1) * 8, "frames_per_step_per_gpu": e2e_frames_per_step,
                    "api": "passiveradar_b200.frames.FramePipeline.run_host (pinned host ndarrays)" if not direct else
                           "clutter-filter + prc_xambg_frames_c64 batched calls around pinned host ndarrays",
                    "h2d_GBps": round(e2e_frames_per_step * 2 * n * 8 * args.steps / e2e_s / 1e9, 2),
                    "h2d_link_GBps": round(h2d_peak, 2) if h2d_peak else None,
                    "note": "h2d_GBps = input bytes per second per GPU through the timed region; h2d_link_GBps = plain "
                            "pinned-memory cudaMemcpy of the same buffers measured beside it (the PCIe ceiling of e2e)"},
            "e2e_dropin": dropin,
            "latency_us": latency_us,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofline,
            "kernels": per_kernel,
            "config3_stream": stream,
            "cpu_baseline": cpu,
        }
        if not quiet:
            print(json.dumps(line), flush=True)
    if world > 1 and not quiet:
        dist.barrier()
        dist.destroy_process_group()
    return line


def run_sweep(args, rank, world, local_rank):
    """BASELINE config 5: CPI 256k -> 4M samples x Doppler 64 -> 1024, LS frame, distinct frames, HBM GB/s vs roofline."""
    import torch
    import torch.distributed as dist
    rows = []
    base_steps = args.steps
    for n in SWEEP_N:
        for F in SWEEP_F:
            cfg = dict(n=n, F=F, R=300, filter_len=300, peek=10, reg=1.0, clutter="ls", name=f"sweep n={n} F={F} R=300")
            a = argparse.Namespace(**vars(args))
            a.resident = max(20, min(125, (2 ** 31) // (16 * n))) // 5 * 5
            a.batch = a.resident // 5                      # five even calls per pass, one per slot
            a.steps = min(base_steps, 5)
            a.frames_per_step = max(a.resident, int(8000 * 2 ** 20 / n / a.steps))      # ~0.3 s of GPU time per point
            a.no_cpu_baseline = True
            a.no_stream = True
            line = run_b200(a, cfg, rank, world, local_rank, quiet=True)
            if rank == 0:
                rows.append({"n": n, "F": F, "R": 300, "frames_per_s": round(line["value"], 1),
                             "frame_GBps": line["roofline"]["frame_GBps"], "frame_frac": line["roofline"]["frame_frac"],
                             "e2e_frames_per_s": round(line["e2e"]["value"], 1), "latency_us": line["latency_us"],
                             "dominant": line["roofline"]["kernel"]})
            torch.cuda.empty_cache()
    if rank == 0:
        c2 = [r for r in rows if r["n"] == 2 ** 20 and r["F"] == 256][0]
        out = {"metric": METRIC, "value": c2["frames_per_s"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "c64", "data": "synthetic",
               "config": {"workload": "sweep CPI 256k..4M samples x Doppler 64..1024 (R=300, LS_Filter(300) -> fast_xambg); value = the n=2^20, F=256 row",
                          "profile": args.profile}, "sweep": rows}
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.config == "c5":
        if args.impl == "reference":
            raise SystemExit("the sweep has no CPU arm")
        run_sweep(args, rank, world, local_rank)
        return
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
        return
    run_b200(args, cfg, rank, world, local_rank)


if __name__ == "__main__":
    main()
