#!/usr/bin/env python
"""Make the fixtures bench.py's `parity` leg checks one clip against (tests/golden/bench_check_<config>.npz).

For each bench configuration: the float64 oracle (oracle/pipeline.py, the restated reference path) separates one
short seeded clip with the very weights bench.py uses (bench.synthetic_params(arch, F, 0)); the fixture holds the
int16 clip, the oracle stems (float32), and -- for the time-frequency bins the oracle flags as sitting on the
soft mask's discontinuity (oracle.nets.near_kink) -- their coordinates and the oracle's spectrum values there,
so that bench.py can take exactly those bins out of the comparison the way tests/parity.py does, without
importing the oracle on the GPU box's timed path.

    python tools/make_bench_check.py [config ...]
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from oracle import dsp, pipeline  # noqa: E402

SECONDS = {"dsd2048": 1.0, "dsd1024": 1.0, "ikala": 1.5, "bach10": 1.0, "bach10_score": 1.0}   # each fixture under 1 MB


def make(name):
    cfg = bench.CONFIGS[name]
    N, F = cfg["N"], cfg["N"] // 2 + 1
    params = bench.synthetic_params(cfg["arch"], F, 0)
    mix, _ = pipeline.synth_mixture(SECONDS[name], 5000 + N)
    pcm = np.round(mix * 32767).astype(np.int16)
    mix = pcm.astype(np.float64) / 32767.0
    win = np.hanning if cfg["window"] == "hanning" else dsp.blackmanharris
    if cfg["arch"] == "bach10_score":
        T = dsp.num_frames(mix.size, 512)
        filters = bench.synthetic_filters(T, F)
        want, mag, ph, mm = pipeline.separate_score(mix, filters, params, frameSize=N, hopSize=512, window=win,
                                                    scale_factor=cfg["scale"], overlap=cfg["overlap"], count_kinks=True,
                                                    return_spec=True)
        kmap = pipeline.separate_score.last_kink_map
    else:
        want, mag, ph, mm = pipeline.separate(mix, params, cfg["arch"], frameSize=N, hopSize=512, window=win,
                                              scale_factor=cfg["scale"], overlap=cfg["overlap"], patcher=cfg["patcher"],
                                              count_kinks=True, return_spec=True)
        kmap = pipeline.separate.last_kink_map
    T = ph.shape[0]
    tt, ff = np.nonzero(kmap)
    S_or = (mm[:, :T] / cfg["scale"]) * np.sqrt(N) * np.exp(1j * ph)[None]
    out = os.path.join(ROOT, "tests", "golden", "bench_check_%s.npz" % name)
    np.savez(out, mix=pcm, stems=want.astype(np.float32), flag_t=tt.astype(np.int32), flag_f=ff.astype(np.int32),
             S_or_flag=S_or[:, tt, ff], window=win(N), N=N, hop=512)
    print(name, "clip %.1f s" % SECONDS[name], "flagged bins", tt.size, "of", kmap.size, "->", out, "%.2f MB" % (os.path.getsize(out) / 1e6))


if __name__ == "__main__":
    for n in (sys.argv[1:] or sorted(SECONDS)):
        make(n)
