#!/usr/bin/env python
"""bench.py -- audio-seconds separated per second.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path (STFT -> encoder/decoder -> soft mask + cross-fade ->
iSTFT/OLA) over one batch of synthetic mono 44.1 kHz mixtures per GPU.  `--config` picks the workload:
  dsd2048 (default)  BASELINE.json configs[1] (and, under torchrun with 8 ranks, literally configs[3]: 256 three-minute
                     mixtures sharded over 8 GPUs): DSD100 4 sources, frameSize 2048, hop 512, time_context 30,
                     overlap 25, 32 clips x 180 s per step per GPU
  dsd1024            the same net at the frame size the reference's DSD100 scripts really use
  bach10             configs[2]: Bach10 4 instruments, frameSize 4096, blackmanharris, 8 x 30 s
  bach10_score       configs[4]: score-informed Bach10 (4-channel input from score filters), 4 x 30 s
  ikala              configs[0]'s network (iKala, max-pool) on the GPU, 8 x 30 s
`value`   : whole-job audio-s/s with the inputs already resident in HBM (CUDA events, max over ranks);
`e2e`     : the same metric through the C-ABI host-buffer call with pinned host memory, H2D and D2H
            inside the timed region (DSD100/iKala/Bach10: int16 wav samples in / int16 stems out,
            train_auto's contract, dcs_separate_pcm16_host; score-informed: float32 + filters);
`roofline`: dominant kernel, timed live with CUDA events on its own stream (dcs_profile); `traffic` =
            dram bytes of that kernel captured live with one short ncu pass AFTER the timing;
`parity`  : one clip of this run checked against stems the float64 oracle produced (tests/golden/bench_check_*.npz);
`cpu_baseline`: the float64 numpy oracle (the restated reference path) on a bounded sample.
`--impl reference` times that CPU path on the host cores this process may really use (the reference itself --
Python 2 + Theano 0.9 + Lasagne -- cannot be installed here; see DESIGN.md).
`--dump-outputs DIR` writes the stems the last timed step computed to DIR/stems.npy (float32), so that two builds
can be compared output for output: the inputs depend on the command line only.  Stems of more than
DUMP_SAMPLES values (the default workload's are 4 GB) are written as the values at a fixed seeded sample of
positions instead (`dump_positions`).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SR = 44100
DUMP_SAMPLES = 8_000_000          # float32 values in a sampled dump: 32 MB
METRIC = "audio_seconds_separated_per_second"
_emit = print
UNIT = "audio-s/s"

CONFIGS = {
    "dsd2048": dict(arch="dsd", N=2048, window="hanning", overlap=25, patcher="standalone", scale=0.3, seconds=180.0, clips=32,
                    nsrc=4, baseline="BASELINE configs[1]: DSD100 4-source separation"),
    "dsd1024": dict(arch="dsd", N=1024, window="hanning", overlap=25, patcher="standalone", scale=0.3, seconds=180.0, clips=32,
                    nsrc=4, baseline="BASELINE configs[1] at the frame size of the reference's own DSD100 scripts"),
    "bach10": dict(arch="bach10", N=4096, window="blackmanharris", overlap=25, patcher="standalone", scale=0.3, seconds=30.0,
                   clips=8, nsrc=4, baseline="BASELINE configs[2]: Bach10 4-instrument separation"),
    "bach10_score": dict(arch="bach10_score", N=4096, window="blackmanharris", overlap=25, patcher="util", scale=0.2,
                         seconds=30.0, clips=4, nsrc=4, baseline="BASELINE configs[4]: Bach10 score-informed separation"),
    "ikala": dict(arch="ikala", N=1024, window="hanning", overlap=20, patcher="standalone", scale=0.3, seconds=30.0, clips=8,
                  nsrc=2, baseline="BASELINE configs[0]'s network (iKala 2-source, max-pool) on the GPU"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="dsd2048", choices=sorted(CONFIGS))
    ap.add_argument("--clips", type=int, default=None, help="clips per step per GPU (default: the config's)")
    ap.add_argument("--seconds", type=float, default=None)
    ap.add_argument("--frame-size", type=int, default=None, help="(dsd configs) overrides the config's frame size")
    ap.add_argument("--e2e-streams", type=int, default=3)
    ap.add_argument("--device-streams", type=int, default=3,
                    help="contexts / CUDA streams the device-resident loop spreads a step's clips over (kernels of "
                         "different clips overlap: single-wave kernels leave tails); per-stage timing stays single-stream")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--traffic", default="live", choices=["live", "off"],
                    help="live: one ncu pass over one clip after the timing (dram bytes of the dominant kernel)")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--ref-clip-seconds", type=float, default=None, help="reference arm: clip length (default: sized to the run)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the stems of the last timed step (or a fixed sample of them) to DIR/stems.npy")
    ap.add_argument("--traffic-probe", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = dict(CONFIGS[a.config])
    if a.frame_size is not None:
        if cfg["arch"] != "dsd":
            ap.error("--frame-size only applies to the dsd configs")
        cfg["N"] = a.frame_size
    a.cfg = cfg
    a.clips = a.clips if a.clips is not None else cfg["clips"]
    a.seconds = a.seconds if a.seconds is not None else cfg["seconds"]
    a.frame_size = cfg["N"]
    return a


# ------------------------------------------------------------------------------------------ shapes
def arch_dims(arch, F, tc=30):
    """Layer sizes of the reference's build_ca() variants (SURVEY.md App. A.3)."""
    if arch == "dsd":
        kh2 = tc // 2
        return dict(f1=50, nch=1, kw1=F, sw1=1, J=1, WP=1, pool=0, f2=50, kh2=kh2, kw2=1, h2=tc - kh2 + 1, w2=1, nfc=128,
                    ndec=3, ndec_live=3, nout=4)
    sw1 = 3 if arch.startswith("ikala") else 4
    pool = 4 if arch == "ikala" else 0
    J = (F - 30) // sw1 + 1
    WP = J // pool if pool else J
    if arch.startswith("ikala"):
        kh2, kw2, ndec, nout, nch = 10, 20, 2, 2, 1
    else:
        kh2, kw2, ndec, nch = int(2 * tc / 3), 1, 4, (4 if arch == "bach10_score" else 1)
        nout = 4 * nch
    return dict(f1=30, nch=nch, kw1=30, sw1=sw1, J=J, WP=WP, pool=pool, f2=30, kh2=kh2, kw2=kw2, h2=tc - kh2 + 1,
                w2=WP - kw2 + 1, nfc=256, ndec=ndec, ndec_live=1 if arch == "bach10_score" else ndec, nout=nout)


def param_shapes(arch, F, tc=30):
    d = arch_dims(arch, F, tc)
    flat = d["f2"] * d["h2"] * d["w2"]
    shp = [(d["f1"], d["nch"], 1, d["kw1"]), (d["f1"],), (d["f1"],), (d["f2"], d["f1"], d["kh2"], d["kw2"]), (d["f2"],),
           (d["f2"],), (flat, d["nfc"]), (d["nfc"],)]
    for _ in range(d["ndec"]):
        shp += [(d["nfc"], flat), (flat,)]
    shp.append((d["nout"],))
    return shp


def synthetic_params(arch, F, seed=0):
    """Random-init weights of the named architecture (Lasagne GlorotUniform; output bias scaled so that the
    masks vary) -- the same stream as oracle.nets.make_synthetic_params (tests/test_bench_host.py)."""
    import numpy as np
    rng = np.random.default_rng(seed)
    shapes = param_shapes(arch, F)
    out = []
    for i, s in enumerate(shapes):
        if len(s) == 4:
            a = np.sqrt(6.0 / ((s[0] + s[1]) * s[2] * s[3]))
        elif len(s) == 2:
            a = np.sqrt(6.0 / (s[0] + s[1]))
        else:
            a = 0.002 if i == len(shapes) - 1 else 0.1
        out.append(rng.uniform(-a, a, size=s).astype(np.float32))
    return out


def synthetic_filters(T, F, seed=4):
    """Score filters with the structure LargeDatasetMask2.filterSpec produces (dataset.py:839-862): 1 on the
    harmonic bins of sounding notes, 1e-18 elsewhere, normalised over the four instruments."""
    import numpy as np
    rng = np.random.default_rng(seed)
    raw = np.full((4, T, F), 1e-18, dtype=np.float32)
    for j in range(4):
        for _ in range(max(4, T // 40)):
            t0, dur = int(rng.integers(0, max(1, T - 60))), int(rng.integers(20, 60))
            f0 = int(rng.integers(8, 60))
            for h in range(1, 20):
                b = f0 * h
                if b + 2 < F:
                    raw[j, t0:t0 + dur, b - 1:b + 2] = 1.0
    return (raw / raw.sum(axis=0)).astype(np.float32)


def synth_clip_device(L, seed, device):
    """Synthetic 4-stem mixture generated on the device: harmonic tone with vibrato, gated low
    sine, decaying noise bursts, broadband noise; int16-quantised like a wav file."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    t = torch.arange(L, device=device, dtype=torch.float32) / SR
    r = torch.rand(8, generator=g, device=device)
    f0 = 110 + 330 * r[0]
    ph = 2 * math.pi * f0 * t * (1 + 0.01 * torch.sin(2 * math.pi * 5 * t))
    s1 = sum(torch.sin(ph * h + 6.28 * r[1] * h) / h for h in range(1, 11))
    fb = 55 + 55 * r[2]
    s2 = torch.sin(2 * math.pi * fb * t) * (torch.sin(2 * math.pi * (1 + r[3]) * t) > 0)
    rate = 2 + 2 * r[4]
    env = torch.exp(-((t * rate) % 1.0) / (rate * 0.010))
    s3 = torch.randn(L, generator=g, device=device) * env
    s4 = torch.randn(L, generator=g, device=device)
    mix = torch.zeros(L, device=device)
    for s in (s1, s2, s3, s4):
        mix += 0.2 * s / s.abs().max().clamp_min(1e-9)
    return torch.round(mix * 32767).clamp(-32768, 32767) / 32767.0


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.perf_counter(), ln.strip()))

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if t0 is not None and not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p.get("bf16_tflops", 1590.0)), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


def stage_work(cfg, stage, L, hop=512, tc=30):
    """Algorithmic (bytes, flops) of one launch group of a pipeline stage for one clip (DESIGN.md 4)."""
    N, ov, arch, nsrc = cfg["N"], cfg["overlap"], cfg["arch"], cfg["nsrc"]
    F = N // 2 + 1
    T = -(-L // hop) + 2
    step = tc - ov
    lim = tc if cfg["patcher"] == "standalone" else ov
    P = max(0, (T - lim - 1) // step + 1)
    fft = 2.5 * N * math.log2(N)
    d = arch_dims(arch, F, tc)
    w = {"stft_fwd": (L * 4 + T * F * 12, T * fft),
         "istft_ola": (nsrc * T * F * 8 + nsrc * L * 4, nsrc * T * fft),
         "score_channels": (T * F * 4 * 9, T * F * 4.0)}
    if arch == "dsd":
        w.update({
            "enc_conv1_gemm": (T * F * 4 + T * 50 * 4 + F * 50 * 4, 2.0 * T * F * 50),
            "enc_conv2_gemm": (T * 50 * 8, 2.0 * (T - 14) * 750 * 50),
            "bottleneck_gemm": (T * 50 * 4 + P * 128 * 4 + 800 * 128 * 4, 2.0 * P * 800 * 128),
            "dec_dense_gemm": (P * 128 * 4 + P * 2400 * 4 + 128 * 2400 * 4, 2.0 * P * 128 * 2400),
            "dec_convT2_gemm": (P * 3 * 44 * 50 * 4 + P * 90 * 50 * 4, 2.0 * P * 90 * 750 * 50),
            "dec_convT1_mask_xfade": (T * F * 8 + P * 90 * 50 * 4 + 4 * T * F * 8, 2.0 * P * 90 * 50 * F),
        })
    else:
        J, WP, kh2, kw2, h2, w2, nd = d["J"], d["WP"], d["kh2"], d["kw2"], d["h2"], d["w2"], d["ndec_live"]
        flat = 30 * h2 * w2
        conv2 = 2.0 * 30 * 30 * kh2 * kw2        # flops per conv2 output position
        w.update({
            "enc_conv1_gemm": (d["nch"] * T * F * 4 + T * J * 32 * 4, 2.0 * T * J * 30 * 30 * d["nch"]),
            "enc_maxpool": (T * J * 32 * 4 + T * WP * 32 * 5, T * J * 32.0),
            "enc_conv2_gemm": (T * WP * 32 * 4 + (T - kh2 + 1) * w2 * 32 * 4, conv2 * (T - kh2 + 1) * w2),
            "bottleneck_gemm": (flat * 256 * 4 + (T - kh2 + 1) * w2 * 32 * 4 + P * 256 * 4, 2.0 * P * flat * 256),
            "dec_dense_gemm": (nd * flat * 256 * 4 + P * nd * flat * 4, 2.0 * P * nd * flat * 256),
            "dec_convT2_gemm": (P * nd * (flat + tc * WP * 32) * 4, conv2 * P * nd * h2 * w2),
            "dec_convT1_mask_xfade": (P * nd * tc * WP * 32 * 4 + T * F * 8 + nsrc * T * F * 8 + (T * WP * 32 if d["pool"] else 0),
                                      2.0 * P * nd * tc * F * (30.0 / d["sw1"]) * 30 * d["nch"]),
        })
    return w[stage]


# kernels behind each stage (names as ncu prints them), for the live traffic capture
STAGE_KERNELS = {"stft_fwd": "stft_", "istft_ola": "istft_", "dec_convT1_mask_xfade": "_mask_", "enc_maxpool": "pool4",
                 "score_channels": "channel_mul"}


def workload_config(args):
    """The `config` of the JSON line: a function of the command line and WORLD_SIZE only, so that both arms
    (`--impl ours`, `--impl reference`) print the SAME object for the same invocation.  What differs between
    the arms (the reference arm's bounded sample; this arm's placement) goes into their own top-level keys."""
    c = args.cfg
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return {"workload": "%s, mono 44.1 kHz, frameSize=%d hop=512 time_context=30 overlap=%d, %d clips x %.0f s per step per GPU" % (
                c["baseline"], c["N"], c["overlap"], args.clips, args.seconds),
            "name": args.config, "arch": c["arch"], "frame_size": c["N"], "hop": 512, "time_context": 30, "overlap": c["overlap"],
            "window": c["window"], "patcher": c["patcher"], "nsrc": c["nsrc"],
            "clips_per_step_per_gpu": args.clips, "clip_seconds": args.seconds,
            "l2_policy": "inputs larger than L2 (%.0f MB of audio per step, intermediates of one clip exceed 126 MB)" % (
                args.clips * args.seconds * SR * 4 / 1e6),
            "parallelism": "clips sharded over %d GPU(s) (sharding.shard_clips), no data-path collective" % args.gpus,
            "device_streams": max(1, args.device_streams),
            "job": "%d clips sharded over %d rank(s)" % (world * args.clips, world)}


# ------------------------------------------------------------------------------------------ CPU arm
def _oracle_separate(cfg, mix, params, filters=None):
    import numpy as np
    from oracle import dsp, pipeline
    win = np.hanning if cfg["window"] == "hanning" else dsp.blackmanharris
    if cfg["arch"] == "bach10_score":
        return pipeline.separate_score(mix, filters, params, frameSize=cfg["N"], hopSize=512, window=win,
                                       scale_factor=cfg["scale"], overlap=cfg["overlap"])
    return pipeline.separate(mix, params, cfg["arch"], frameSize=cfg["N"], hopSize=512, window=win,
                             scale_factor=cfg["scale"], overlap=cfg["overlap"], patcher=cfg["patcher"])


_worker_state = {}


def _cpu_worker(job):
    """One single-threaded worker: the restated reference path on one clip (params are made once per process)."""
    cfg, seconds, seed = job
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=1)
    except Exception:
        pass
    from oracle import pipeline
    key = (cfg["arch"], cfg["N"])
    if key not in _worker_state:
        _worker_state[key] = synthetic_params(cfg["arch"], cfg["N"] // 2 + 1, 0)
    params = _worker_state[key]
    mix, _ = pipeline.synth_mixture(seconds, seed)
    filters = None
    if cfg["arch"] == "bach10_score":
        filters = synthetic_filters(-(-mix.size // 512) + 2, cfg["N"] // 2 + 1)
    t = time.perf_counter()
    out = _oracle_separate(cfg, mix, params, filters)
    dt = time.perf_counter() - t
    assert out.shape[0] == cfg["nsrc"]
    return dt


def run_reference(args):
    """The reference's CPU path (oracle port) on the host threads this process may use.  Each step = `procs`
    single-threaded workers (BLAS pinned to 1 thread each) x one clip; --steps / --warmup are honoured; the
    clip length is the longest of (180, 60, 30, 10) s for which the whole run fits ~4 minutes, judged from a
    short calibration pass that also finds the worker count with the best throughput (a hidden CPU quota or a
    memory-bound box saturates below the visible core count)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    from deepconvsep_b200.sharding import effective_cores
    cfg = args.cfg
    cores = effective_cores()
    K, W = max(1, args.steps), max(0, args.warmup)
    ctx = mp.get_context("spawn")
    cal_s = 4.0 if cfg["arch"] == "dsd" else 2.0
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker, [(cfg, 1.0, 7000 + i) for i in range(cores)], chunksize=1)   # imports, params, page-in
        single = cal_s / _cpu_single(cfg, cal_s)                                       # single process, 1 BLAS thread
        cands, best, p = [], None, cores
        while p >= 1:
            cands.append(p)
            p //= 2
        for p in cands:          # all usable threads first; fewer workers only if that is measurably faster
            t = time.perf_counter()
            pool.map(_cpu_worker, [(cfg, cal_s, 7100 + i) for i in range(p)], chunksize=1)
            thr = p * cal_s / (time.perf_counter() - t)
            if best is None or thr > best[1] * 1.05:
                best = (p, thr)
        procs, cal_thr = best
        budget = 240.0
        clip_s = args.ref_clip_seconds
        if clip_s is None:
            clip_s = 10.0
            for c in (180.0, 60.0, 30.0):
                if (K + W) * (c * procs / cal_thr) <= budget:
                    clip_s = c
                    break
        for w in range(W):
            pool.map(_cpu_worker, [(cfg, clip_s, 7200 + w * procs + i) for i in range(procs)], chunksize=1)
        t0 = time.perf_counter()
        for s in range(K):
            pool.map(_cpu_worker, [(cfg, clip_s, 1000 + s * procs + i) for i in range(procs)], chunksize=1)
        dt = time.perf_counter() - t0
    value = K * procs * clip_s / dt
    sample = ("%d steps (+%d warm-up) x %d single-threaded workers x one %.0f s clip each; float64 numpy restatement of the "
              "reference's separate path, BLAS 1 thread/worker; %d usable host threads (affinity + cgroup quota; os.cpu_count()=%d), "
              "worker count chosen by calibration; single process: %.1f audio-s/s" % (
                  K, W, procs, clip_s, cores, os.cpu_count() or 0, single))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": K,
        "warmup": W, "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "reference_sample": {"clip_seconds": clip_s, "workers": procs, "clips_per_step": procs,
                             "what": "each step is a bounded sample of the workload in `config`: one clip per worker"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": "port", "sample": sample,
                         "single_process_value": single, "usable_host_threads": cores},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "the reference's own runtime (Python 2.7 + Theano 0.9 + Lasagne) is not installable here; this is "
                "the oracle port of its CPU path",
    }
    _emit(json.dumps(line))


def _cpu_single(cfg, seconds):
    try:
        from threadpoolctl import threadpool_limits
        with threadpool_limits(limits=1):
            return _cpu_worker((cfg, seconds, 7050))
    except ImportError:
        return _cpu_worker((cfg, seconds, 7050))


# ------------------------------------------------------------------------------------------ GPU arm
def make_separator(cfg, params, device):
    from deepconvsep_b200.engine import Separator
    return Separator(params, arch=cfg["arch"], frame_size=cfg["N"], hop=512, window=cfg["window"], overlap=cfg["overlap"],
                     patcher=cfg["patcher"], scale_factor=cfg["scale"], feat_size=cfg["N"] // 2 + 1, device=device)


def dump_positions(total):
    """Sorted flat positions of the sampled dump of `total` output values: the same for the same shape."""
    import numpy as np
    return np.unique(np.random.default_rng(0).integers(0, total, size=DUMP_SAMPLES))


def dump_outputs(path, outs):
    """outs: float32 cuda [clips, sources, samples], the stems as a caller of the timed path receives them."""
    import numpy as np
    import torch
    if outs.numel() > DUMP_SAMPLES:
        idx = torch.from_numpy(dump_positions(outs.numel())).to(outs.device)
        outs = outs.reshape(-1)[idx]
    os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
    np.save(path, outs.cpu().numpy())


def parity_check(args, sep):
    """One clip of this very run against stems the float64 oracle produced for it (committed fixture made by
    tools/make_bench_check.py).  Plain 1e-4 per stem; the few time-frequency bins the ORACLE flagged as
    sitting on the soft mask's discontinuity are taken out bin by bin exactly like tests/parity.py does (the
    oracle spectrum adopts the device's value there; the inverse STFT is linear, so that is a correction of the
    expected waveform by istft(D), D non-zero at the flagged bins only).  No oracle code runs here."""
    import numpy as np
    path = os.path.join(ROOT, "tests", "golden", "bench_check_%s.npz" % args.config)
    if args.frame_size != CONFIGS[args.config]["N"] or not os.path.exists(path):
        return {"checked": False, "why": "no oracle fixture for this configuration"}
    g = np.load(path)
    N, hop, win = int(g["N"]), int(g["hop"]), g["window"]
    mix = g["mix"].astype(np.float64) / 32767.0
    filters = synthetic_filters(-(-mix.size // hop) + 2, N // 2 + 1) if args.cfg["arch"] == "bach10_score" else None
    got, S = sep.separate_tapped(mix, filters)
    want = g["stems"].astype(np.float64)
    tt, ff, S_or = g["flag_t"], g["flag_f"], g["S_or_flag"]
    T, L = S.shape[1], mix.size
    corr = np.zeros_like(want)
    if tt.size:
        total = hop * (T - 1) + N
        norm = np.zeros(total)
        for n in range(T):
            norm[n * hop:n * hop + N] += win * win
        norm = norm[N // 2:]
        norm[norm == 0] = 1.0
        for s in range(want.shape[0]):
            data = np.zeros(total)
            for n in sorted(set(int(t) for t in tt)):
                row = np.zeros(N // 2 + 1, dtype=np.complex128)
                sel = tt == n
                row[ff[sel]] = S[s][n, ff[sel]].astype(np.complex128) - S_or[s][sel]
                data[n * hop:n * hop + N] += win * np.fft.irfft(row, N)
            corr[s] = (data[N // 2:] / norm)[:L]
    errs = [float(np.linalg.norm(got[s] - (want[s] + corr[s])) / np.linalg.norm(want[s])) for s in range(want.shape[0])]
    raw = [float(np.linalg.norm(got[s] - want[s]) / np.linalg.norm(want[s])) for s in range(want.shape[0])]
    return {"checked": True, "fixture": os.path.relpath(path, ROOT), "clip_seconds": mix.size / SR, "rel_l2_per_stem": errs,
            "rel_l2_unmodified": raw, "flagged_bins_excluded": int(tt.size), "max_rel_l2": max(errs), "tol": 1e-4,
            "ok": bool(max(errs) <= 1e-4)}


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from deepconvsep_b200 import sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this framework has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity0 = os.sched_getaffinity(0)
    numa = {"numa_node": None} if args.no_numa else sharding.bind_to_gpu_numa(local)   # before any pinned allocation
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    cfg = args.cfg
    N, B, K, W = cfg["N"], args.clips, args.steps, max(args.warmup, 3)
    F = N // 2 + 1
    L = int(round(args.seconds * SR))
    score = cfg["arch"] == "bach10_score"
    nsrc = cfg["nsrc"]
    params = synthetic_params(cfg["arch"], F, 0)
    sep = make_separator(cfg, params, local)
    # the literal sharded job: world*B clips, longest-first greedy assignment (all equal here), clip seeds by global index
    lengths = [L] * (world * B)
    mine = sharding.shard_clips(lengths, world, rank)
    assert len(mine) == B
    clips = [synth_clip_device(L, 1000 + g, dev) for g in mine]
    outs = torch.empty((B, nsrc, L), dtype=torch.float32, device=dev)
    filt_h = filt_d = None
    if score:
        T = sep.stft.num_frames(L)
        filt_h = synthetic_filters(T, F)
        filt_d = torch.zeros((4, T, sep.stft.ldf), dtype=torch.float32, device=dev)
        filt_d[:, :, :F] = torch.as_tensor(filt_h, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    parity = parity_check(args, sep) if (rank == 0 and not args.traffic_probe) else None

    nd = max(1, args.device_streams)
    dworkers = [sep] + [make_separator(cfg, params, local) for _ in range(nd - 1)]
    dstreams = [torch.cuda.Stream(device=dev) for _ in range(nd)] if nd > 1 else []

    def one_clip(w, i, stream=None):
        if score:
            w.separate_score(clips[i], filt_d, out=outs[i], stream=stream)
        else:
            w.separate_device(clips[i], outs[i], stream=stream)

    def step_device():
        if nd == 1:
            for i in range(B):
                one_clip(sep, i)
            return
        cur = torch.cuda.current_stream()
        for s_ in dstreams:
            s_.wait_stream(cur)
        for i in range(B):
            one_clip(dworkers[i % nd], i, dstreams[i % nd])
        for s_ in dstreams:
            cur.wait_stream(s_)

    if args.traffic_probe:          # child of the live traffic capture: one warm clip, one measured clip, nothing else
        one_clip(sep, 0)
        torch.cuda.synchronize()
        one_clip(sep, 0)
        torch.cuda.synchronize()
        return

    # ---- device-resident throughput -------------------------------------------------------
    for _ in range(W):
        step_device()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.25)
    launches0 = sum(w.ctx.launch_count() for w in dworkers)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_host0 = time.perf_counter()
    e0.record()
    for _ in range(K):
        step_device()
    e1.record()
    barrier()
    t_host1 = time.perf_counter()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    launches = sum(w.ctx.launch_count() for w in dworkers) - launches0
    clocks = sampler.stop(t_host0, t_host1)
    if args.dump_outputs:
        dump_outputs(os.path.join(args.dump_outputs, "stems.npy" if world == 1 else "stems_rank%d.npy" % rank), outs)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    audio_s = world * B * K * args.seconds
    value = audio_s / (ms * 1e-3)
    finite = bool(torch.isfinite(outs).all().item())

    # ---- per-stage timing (CUDA events inside libdcs, on the launching stream) --------------
    sep.ctx.profile(True)
    for _ in range(2):     # one stream: stage times must not include the overlap with other clips
        for i in range(B):
            one_clip(sep, i)
    torch.cuda.synchronize()
    recs = sep.ctx.profile_read()
    sep.ctx.profile(False)
    stages = {}
    for name, t in recs:
        stages.setdefault(name, []).append(t)
    stage_ms = {k: sum(v) / len(v) for k, v in stages.items()}
    tot = sum(stage_ms.values())
    dom = max(stage_ms, key=stage_ms.get)
    hbm_peak, tensor_peak, peak_src = measured_peaks()
    by, fl = stage_work(cfg, dom, L)

    def roof(stage):
        b_, f_ = stage_work(cfg, stage, L)
        t_ = stage_ms[stage] * 1e-3
        if stage.endswith("_gemm"):   # dense contractions: tensor pipe (3xTF32 = 3 MMAs at half the bf16 rate)
            a_ = f_ / t_ / 1e12
            return {"kernel": stage, "bound": "tensor", "achieved": a_, "peak": tensor_peak, "unit": "TFLOP/s",
                    "frac": a_ / tensor_peak, "note": "fp32-accurate 3xTF32: the ceiling of this arithmetic is peak/6"}
        a_ = b_ / t_ / 1e9
        return {"kernel": stage, "bound": "hbm", "achieved": a_, "peak": hbm_peak, "unit": "GB/s", "frac": a_ / hbm_peak}
    roofline = roof(dom)
    # whole pipeline against the governing roofline of SURVEY 8(d): max(compulsory bytes / HBM, tensor flops / (bf16 peak / 6))
    tflops = sum(stage_work(cfg, k, L)[1] for k in stage_ms if k.endswith("_gemm") or k == "dec_convT1_mask_xfade")
    t_hbm, t_tensor = (L * 4 + nsrc * L * 4) / (hbm_peak * 1e9), tflops / (tensor_peak * 1e12 / 6.0)
    t_roof = max(t_hbm, t_tensor)
    roofline.update({"traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": by,
                     "algorithmic_flops_per_launch": fl, "launch_ms": stage_ms[dom],
                     "share_of_step": stage_ms[dom] / tot,
                     "pipeline": {"ms_per_clip_single_stream": tot, "ms_per_clip_timed_loop": ms / K / B,
                                  "roofline_ms_per_clip": t_roof * 1e3, "frac": t_roof * 1e3 / (ms / K / B),
                                  "governing": "tensor pipe, 3xTF32 (bf16 peak / 6)" if t_tensor > t_hbm else "HBM, compulsory bytes"},
                     "all_stages": [dict(roof(k), share_of_step=stage_ms[k] / tot) for k in stage_ms]})
    stage_table = {k: {"ms": v, "share": v / tot, "gbps": stage_work(cfg, k, L)[0] / (v * 1e-3) / 1e9,
                       "tflops": stage_work(cfg, k, L)[1] / (v * 1e-3) / 1e12} for k, v in stage_ms.items()}

    # ---- end to end through the host-buffer C-ABI call --------------------------------------
    ns = max(1, args.e2e_streams)
    workers = dworkers[:ns] + [make_separator(cfg, params, local) for _ in range(ns - len(dworkers))]
    streams = [torch.cuda.Stream(device=dev) for _ in range(ns)]
    pcm = not score
    # (a) the wav contract of train_auto (separate_dsd.py:275-287,307-309): int16 samples in, int16 stems out
    # (b) float32 host buffers (dcs_separate_host; the score-informed path: float32 audio + the filter planes)
    h_in16 = [torch.empty(L, dtype=torch.int16).pin_memory() for _ in range(B)]
    h_out16 = [torch.empty((nsrc, L), dtype=torch.int16).pin_memory() for _ in range(B)]
    h_in = [torch.empty(L, dtype=torch.float32).pin_memory() for _ in range(B)]
    h_out = [torch.empty((nsrc, L), dtype=torch.float32).pin_memory() for _ in range(B)]
    for i in range(B):
        h_in[i].copy_(clips[i].cpu())
        h_in16[i].copy_(torch.round(clips[i].cpu() * 32767).to(torch.int16))
    np_in, np_out = [t.numpy() for t in h_in], [t.numpy() for t in h_out]
    np_in16, np_out16 = [t.numpy() for t in h_in16], [t.numpy() for t in h_out16]
    filt_pinned = torch.as_tensor(filt_h).pin_memory() if score else None

    def e2e_worker(w, nsteps, use_pcm):
        torch.cuda.set_device(local)
        with torch.cuda.stream(streams[w]):
            for _ in range(nsteps):
                for i in range(w, B, ns):
                    if score:
                        fd = torch.zeros((4, filt_d.shape[1], filt_d.shape[2]), dtype=torch.float32, device=dev)
                        fd[:, :, :F].copy_(filt_pinned, non_blocking=True)
                        x = torch.empty(L, dtype=torch.float32, device=dev)
                        x.copy_(h_in[i], non_blocking=True)
                        y = workers[w].separate_score(x, fd)
                        h_out[i].copy_(y, non_blocking=True)
                        torch.cuda.current_stream().synchronize()
                    elif use_pcm:
                        workers[w].separate_pcm16(np_in16[i], out=np_out16[i])
                    else:
                        workers[w].separate(np_in[i], out=np_out[i])

    def e2e_run(nsteps, use_pcm):
        ths = [threading.Thread(target=e2e_worker, args=(w, nsteps, use_pcm)) for w in range(ns)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()

    def e2e_measure(use_pcm):
        e2e_run(2, use_pcm)
        barrier()
        l0 = sum(w.ctx.launch_count() for w in workers)
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        e2e_run(K, use_pcm)
        for s in streams:
            torch.cuda.current_stream().wait_stream(s)
        f1.record()
        barrier()
        nl = sum(w.ctx.launch_count() for w in workers) - l0
        t = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), nl

    ems_f32, l_f32 = e2e_measure(False)
    if pcm:
        ems, e2e_launches = e2e_measure(True)
        h2d, d2h = B * L * 2, B * nsrc * L * 2
        api = "dcs_separate_pcm16_host: pinned int16 wav samples in, int16 stems out (train_auto's wav contract)"
    else:
        ems, e2e_launches = ems_f32, l_f32
        h2d, d2h = B * (L * 4 + int(filt_pinned.numel()) * 4), B * nsrc * L * 4
        api = "dcs_separate_audio_score behind Separator.separate_score: pinned float32 audio + 4 filter planes in, float32 stems out"
    e2e_value = audio_s / (ems * 1e-3)
    # the same contract through the library's own multi-clip scheduler (one context, one call per step:
    # dcs_separate_batch_pcm16_host pipelines H2D | kernels | D2H over the clips)
    batch = None
    if pcm:
        sep.separate_pcm16_batch(np_in16, outs=np_out16)
        barrier()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record()
        for _ in range(K):
            sep.separate_pcm16_batch(np_in16, outs=np_out16)
        b1.record()
        barrier()
        tb = torch.tensor([b0.elapsed_time(b1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tb, op=dist.ReduceOp.MAX)
        batch = {"value": audio_s / (float(tb.item()) * 1e-3), "ms_per_step": float(tb.item()) / K,
                 "api": "dcs_separate_batch_pcm16_host: one context, one call per step, three-stage pipeline inside the library"}
    # result checks on the host copies: where masks cover it the stems add up to the mixture (DSD/iKala mask rule)
    chk = float(np.abs(np_out[0][:, 44100:88200].sum(0) - np_in[0][44100:88200]).max())
    chk16 = int(np.abs(np_out16[0][:, 44100:88200].astype(np.int32).sum(0) - np_in16[0][44100:88200]).max()) if pcm else None

    # ---- live DRAM traffic of the dominant kernel: one ncu pass over one clip, after all timing -------------
    traffic_note = None
    if rank == 0 and world == 1 and args.traffic == "live":
        roofline["traffic"], traffic_note = live_traffic(args, dom)
    roofline["traffic_source"] = traffic_note

    # ---- CPU baseline (rank 0, N=1 only): the oracle on a bounded sample --------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, affinity0)
        secs = 20.0 if cfg["arch"] == "dsd" else 5.0
        t0 = time.perf_counter()
        dt = _cpu_worker_threads(cfg, secs)
        cpu = {"value": secs / dt, "unit": UNIT, "cores": sharding.effective_cores(), "kind": "port",
               "sample": "one %.0f s clip, frameSize=%d, float64 numpy oracle (per-frame FFT loops, batches of 32 "
                         "patches, BLAS threads = usable host threads), %.1f s of CPU time" % (secs, N, time.perf_counter() - t0)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(args), "placement": {"numa": numa},
            "x_realtime": value, "gpu_launches": int(launches), "outputs_finite": finite,
            "clocks": clocks, "parity": parity,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ems / K, "streams": ns, "gpu_launches": int(e2e_launches), "api": api,
                    "d2h_gbs_per_gpu": d2h / (ems / K * 1e-3) / 1e9, "h2d_gbs_per_gpu": h2d / (ems / K * 1e-3) / 1e9,
                    "bound": "PCIe: the copies of a step take longer than its kernels" if ems > 1.15 * ms else "kernels",
                    "stem_sum_max_abs_err_lsb": chk16, "batch_api": batch,
                    "float32_buffers": {"value": audio_s / (ems_f32 * 1e-3), "ms_per_step": ems_f32 / K,
                                        "h2d_bytes_per_step": B * L * 4, "d2h_bytes_per_step": B * nsrc * L * 4,
                                        "api": "dcs_separate_host", "stem_sum_max_abs_err": chk}},
            "roofline": roofline, "stages": stage_table, "cpu_baseline": cpu,
        }
        _emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def live_traffic(args, dom):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant stage's kernel(s) for ONE clip, from a
    short ncu pass over a child process (never the timed process).  Returns (bytes | None, note)."""
    import csv
    import shutil
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None, "ncu not found"
    pat = STAGE_KERNELS.get(dom)
    if pat is None:
        return None, "stage %s shares its kernel with other stages; no per-stage capture" % dom
    out = "/tmp/dcs_traffic_%d.csv" % os.getpid()
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "-k", "regex:" + pat,
           "--csv", "--log-file", out, sys.executable, os.path.abspath(__file__), "--traffic-probe", "--config", args.config,
           "--seconds", str(args.seconds), "--clips", "1", "--no-numa", "--device-streams", "1"]
    if args.cfg["arch"] == "dsd":
        cmd += ["--frame-size", str(args.frame_size)]
    try:
        subprocess.run(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=240, check=False)
        rows = []
        with open(out) as f:
            lines = [ln for ln in f if not ln.startswith("==")]
        for r in csv.DictReader(lines):
            if r.get("Metric Name", "").startswith("dram__bytes"):
                v = float(r["Metric Value"].replace(",", ""))
                u = r.get("Metric Unit", "byte").lower()
                v *= {"byte": 1, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(u, 1)
                rows.append((int(r["ID"]), v))
        if not rows:
            return None, "ncu produced no dram metrics"
        ids = sorted({i for i, _ in rows})
        half = set(ids[len(ids) // 2:])     # the probe runs the clip twice: keep the second (warm) pass
        total = sum(v for i, v in rows if i in half)
        return int(total), ("ncu dram__bytes_read.sum + dram__bytes_write.sum, kernels matching '%s', one clip, "
                            "captured live by this run after the timing" % pat)
    except Exception as e:  # noqa: BLE001
        return None, "live capture failed: %r" % (e,)
    finally:
        try:
            os.remove(out)
        except OSError:
            pass


def _cpu_worker_threads(cfg, seconds):
    from oracle import pipeline
    params = synthetic_params(cfg["arch"], cfg["N"] // 2 + 1, 0)
    mix, _ = pipeline.synth_mixture(seconds, 1000)
    filters = synthetic_filters(-(-mix.size // 512) + 2, cfg["N"] // 2 + 1) if cfg["arch"] == "bach10_score" else None
    t = time.perf_counter()
    _oracle_separate(cfg, mix, params, filters)
    return time.perf_counter() - t


def main():
    args = parse_args()
    # stdout must carry exactly ONE JSON line: NCCL / torchrun / libraries print banners to fd 1
    # ("NCCL version ..."), so everything else is sent to stderr and the line is written to the
    # original descriptor at the end.
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    out = os.fdopen(real, "w")
    global _emit
    _emit = lambda line: (out.write(line + "\n"), out.flush())
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
