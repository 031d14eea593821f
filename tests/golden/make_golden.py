#!/usr/bin/env python
"""Generate tests/golden/*.npz by EXECUTING THE REFERENCE'S OWN FUNCTION BODIES.

Run in the build container only (needs /root/reference).  The reference files are Python 2
(print statements) and cannot be imported, but the hot-path functions themselves are valid
Python 3: their source text is sliced out of the reference files at run time (nothing is
copied into this repo), exec'd with numpy in scope, and run on seeded inputs.  The outputs
pin oracle/dsp.py and oracle/patch.py (tests/test_oracle_golden.py); tests/dspgolden.py makes the
inputs and says how dsp_golden.npz stores the outputs.

The network (Theano/Lasagne) cannot be executed here -> no golden for it (parity unpinned).
"""
import os
import re
import sys
import numpy as np

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import dspgolden  # noqa: E402


def grab(path, names):
    """Return {name: function} for top-level `def name(` blocks in a reference file."""
    src = open(os.path.join(REF, path)).read()
    ns = {"np": np, "numpy": np}
    for name in names:
        m = re.search(r"^def %s\(.*?(?=^(?:def |class |if __name__)|\Z)" % re.escape(name), src, re.S | re.M)
        assert m, (path, name)
        exec(compile(m.group(0), path + ":" + name, "exec"), ns)
    return ns


def main():
    tr = grab("transform.py", ["sinebell", "stft_norm", "istft_norm"])
    sd = grab("examples/dsd100/separate_dsd.py",
              ["sinebell", "stft_norm", "istft_norm", "compute_file", "compute_inverse",
               "generate_overlapadd", "overlapadd_multi"])
    ik = grab("examples/ikala/separate_ikala.py", ["overlapadd"])
    ut = grab("util.py", ["generate_overlapadd", "overlapadd_multi"])

    out = {}
    stream = iter(range(2000, 3000))        # sample positions of each stored output

    def keep(key, a):
        out.update(dspgolden.record(key, a, next(stream)))
    # --- STFT / iSTFT (transform.py) for the three frame sizes and three windows
    from scipy.signal import windows
    for ci, (N, H, wname, L) in enumerate(dspgolden.STFT_CASES):
        w = {"hanning": np.hanning, "blackmanharris": windows.blackmanharris,
             "sinebell": tr["sinebell"]}[wname](N)
        x, Z = dspgolden.stft_inputs(ci)
        X = tr["stft_norm"](x, window=w, hopsize=float(H), nfft=float(N), fs=44100.0)
        assert X.shape == Z.shape
        out.update({"stft%d_w" % ci: w, "stft%d_NH" % ci: np.array([N, H])})
        keep("stft%d_X" % ci, X)
        keep("stft%d_y" % ci, tr["istft_norm"](X, window=w, analysisWindow=w, hopsize=float(H), nfft=float(N)))
        keep("stft%d_y2" % ci, tr["istft_norm"](Z, window=w, analysisWindow=w, hopsize=float(H), nfft=float(N)))
    out["n_stft"] = np.array(len(dspgolden.STFT_CASES))
    # --- compute_file / compute_inverse of the stand-alone script (hanning 1024/512 defaults)
    mag, ph = sd["compute_file"](dspgolden.cf_input(), phase=True)
    keep("cf_mag", mag)
    keep("cf_ph", ph)
    keep("cf_inv", sd["compute_inverse"](mag * 0.7, ph))
    # --- patchers + cross-fade
    for ci, (T, F, tc, ov, bs) in enumerate(dspgolden.PATCH_CASES):
        m = dspgolden.patch_input(ci)
        fb, n = sd["generate_overlapadd"](m, input_size=F, time_context=tc, overlap=ov, batch_size=bs)
        if n:
            fb[int((n - 1) / bs), int((n - 1) % bs) + 1:] = 0   # np.empty tail -> deterministic
        fbu, nu = ut["generate_overlapadd"](m, input_size=F, time_context=tc, overlap=ov, batch_size=bs)
        out.update({"pat%d_cfg" % ci: np.array([tc, ov, bs]), "pat%d_n" % ci: np.array(n), "pat%d_nu" % ci: np.array(nu)})
        keep("pat%d_fb" % ci, fb)
        keep("pat%d_fbu" % ci, fbu)
        if n:
            pred = dspgolden.patch_pred(ci, n)
            assert pred.shape[0] == fb.shape[0]
            keep("pat%d_sep" % ci, sd["overlapadd_multi"](pred, fb, n, overlap=ov))
            keep("pat%d_sepu" % ci, ut["overlapadd_multi"](pred, fb, n, overlap=ov))
            s1, s2 = ik["overlapadd"](pred[:, :2], fb, n, overlap=ov)
            keep("pat%d_sep2" % ci, np.stack([s1, s2]))
    out["n_pat"] = np.array(len(dspgolden.PATCH_CASES))
    # 3-D (channel) input through util's patcher (score-informed path)
    fb3, n3 = ut["generate_overlapadd"](dspgolden.pat3d_input(), input_size=11, time_context=30, overlap=25, batch_size=8)
    out["pat3d_n"] = np.array(n3)
    keep("pat3d_fb", fb3)
    np.savez_compressed(os.path.join(HERE, "dsp_golden.npz"), **out)
    print("wrote", os.path.join(HERE, "dsp_golden.npz"), len(out), "arrays")


# ---------------------------------------------------------------------------------------------
# score prelude of the score-informed path: util.getMidiNum / expandMidi / slicefft_slices / str2midi
# and LargeDatasetMask2.filterSpec, executed from the reference source (Python-2 idioms shimmed:
# `filter` returns a list, note names read as bytes are decoded before str2midi).
def grab_method(path, cls_marker, name):
    src = open(os.path.join(REF, path)).read()
    i = src.index(cls_marker)
    m = re.search(r"^    def %s\(.*?(?=^    def |\Z)" % re.escape(name), src[i:], re.S | re.M)
    assert m, (path, name)
    import textwrap
    return textwrap.dedent(m.group(0))


SCORES = {
    "bassoon_b": "0.10,0.80,C3\n0.90,1.60,E3\n1.70,2.90,G2\n3.00,3.02,A2\n3.10,3.90,C#3\n",
    "clarinet_b": "0.00,0.70,E4\n0.75,1.50,G4\n1.50,2.20,Bb4\n2.60,3.80,A4\n",
    "saxophone_b": "0.20,1.00,G3\n1.00,2.00,B3\n2.10,2.80,D4\n2.80,3.95,F#3\n",
    "violin_b": "0.05,0.60,C5\n0.60,1.20,D5\n1.25,2.40,E5\n2.40,3.00,F5\n3.20,3.90,G5\n",
}


def score_golden():
    import itertools
    import tempfile
    import builtins
    from bisect import bisect_left, bisect_right
    src = open(os.path.join(REF, "util.py")).read()
    ns = {"np": np, "os": os, "it": itertools, "bisect_left": bisect_left, "bisect_right": bisect_right,
          "nan": float("nan"), "filter": lambda f, l: list(builtins.filter(f, l)), "MIDI_A4": 69}
    for name in ["midi2freq", "getfreqs", "remove_overlap", "slicefft_slices", "str2midi", "getMidiNum", "expandMidi"]:
        m = re.search(r"^def %s\(.*?(?=^(?:def |class |#+ )|\Z)" % re.escape(name), src, re.S | re.M)
        assert m, name
        exec(compile(m.group(0), "util.py:" + name, "exec"), ns)
    orig = ns["str2midi"]
    ns["str2midi"] = lambda n: orig(n.decode("ascii") if isinstance(n, bytes) else n)
    fs_src = grab_method("dataset.py", "class LargeDatasetMask2", "filterSpec")
    fns = {"np": np}
    exec(compile(fs_src, "dataset.py:filterSpec", "exec"), fns)

    class Dummy(object):
        tensortype = np.float32
        timbre_model_path = None
    out = {}
    d = tempfile.mkdtemp()
    for k, v in SCORES.items():
        open(os.path.join(d, k + ".txt"), "w").write(v)
        out["txt_" + k] = np.frombuffer(v.encode("ascii"), dtype=np.uint8)
    insts = ["bassoon_b", "clarinet_b", "saxophone_b", "violin_b"]
    nharm, frameSize, hop, sr = 20, 4096, 512, 44100
    nframes = int(np.ceil(4.0 * sr / float(hop))) + 2
    nelem = 1
    for i, inst in enumerate(insts):
        ng = ns["getMidiNum"](inst, d, 0, 40.0)
        out["num_%d" % i] = np.array(ng)
        nelem = max(nelem, ng)
    melody = np.zeros((4, nelem, 2 * nharm + 3))
    for i, inst in enumerate(insts):
        tmp = ns["expandMidi"](inst, d, 0, 40.0, 50, 440, nharm, sr, hop, frameSize, 0.2, 0.2, nframes, 0.5)
        out["exp_%d" % i] = tmp
        melody[i, :tmp.shape[0], :] = tmp
    rng = np.random.default_rng(5)
    mag = (0.3 * np.abs(rng.standard_normal((nframes, frameSize // 2 + 1)))).astype(np.float32)
    mask = fns["filterSpec"](Dummy(), mag, melody, 0, nframes)
    out["melody"] = melody
    out["mask"] = mask
    out["nframes"] = np.array(nframes)
    out["str2midi"] = np.array([ns["str2midi"](s) for s in ["C3", "Bb4", "F#3", "C#5", "A4", "Ebb2", "Gx6"]], dtype=np.float64)
    np.savez_compressed(os.path.join(HERE, "score_golden.npz"), **out)
    print("wrote score_golden.npz", len(out), "arrays; mask", mask.shape, "ones", int((mask > 0.99).sum()))


if __name__ == "__main__":
    if "--score" in sys.argv:
        score_golden()
    else:
        main()
        score_golden()
