"""Pin the oracle's DSP / patcher / cross-fade against vectors produced by the reference's
own function bodies (tests/golden/make_golden.py)."""
import numpy as np
from dspgolden import check
from oracle import dsp, patch


def test_stft_istft_match_reference(golden):
    g = golden
    for ci in range(int(g["n_stft"])):
        N, H = (int(v) for v in g["stft%d_NH" % ci])
        x, w = g["stft%d_x" % ci], g["stft%d_w" % ci]
        X = dsp.stft_norm(x, window=w, hopsize=float(H), nfft=float(N))
        assert X.shape[0] == dsp.num_frames(x.size, H)
        check(g, "stft%d_X" % ci, X)
        y = dsp.istft_norm(X, window=w, analysisWindow=w, hopsize=float(H), nfft=float(N))
        check(g, "stft%d_y" % ci, y)
        assert y.size == (X.shape[0] - 1) * H + N - N // 2
        y2 = dsp.istft_norm(g["stft%d_Z" % ci], window=w, analysisWindow=w, hopsize=float(H), nfft=float(N))
        check(g, "stft%d_y2" % ci, y2)
        # perfect reconstruction of the analysed signal (property, SURVEY App. C)
        err = np.linalg.norm(y[:x.size] - x) / np.linalg.norm(x)
        assert err < 1e-14


def test_compute_file_inverse(golden):
    g = golden
    mag, ph = dsp.compute_file(g["cf_x"], phase=True)
    check(g, "cf_mag", mag)
    check(g, "cf_ph", ph)
    check(g, "cf_inv", dsp.compute_inverse(mag * 0.7, ph))


def test_patchers_and_crossfade(golden):
    g = golden
    for ci in range(int(g["n_pat"])):
        tc, ov, bs = (int(v) for v in g["pat%d_cfg" % ci])
        m = g["pat%d_m" % ci]
        fb, n = patch.generate_overlapadd(m, input_size=m.shape[1], time_context=tc, overlap=ov, batch_size=bs)
        assert n == int(g["pat%d_n" % ci]) == patch.num_patches(m.shape[0], tc, ov, "standalone")
        check(g, "pat%d_fb" % ci, fb)
        fbu, nu = patch.generate_overlapadd_util(m, input_size=m.shape[1], time_context=tc, overlap=ov, batch_size=bs)
        assert nu == int(g["pat%d_nu" % ci]) == patch.num_patches(m.shape[0], tc, ov, "util")
        check(g, "pat%d_fbu" % ci, fbu)
        if n:
            pred = g["pat%d_pred" % ci]
            sep = patch.overlapadd_multi(pred, fb, n, overlap=ov)
            check(g, "pat%d_sep" % ci, sep)
            check(g, "pat%d_sepu" % ci, sep)   # util copy is identical
            s1, s2 = patch.overlapadd(pred[:, :2], fb, n, overlap=ov)
            check(g, "pat%d_sep2" % ci, np.stack([s1, s2]))
            # output length >= T for the stand-alone patcher (separate_dsd.py:304 relies on it)
            assert sep.shape[1] >= m.shape[0]
    fb3, n3 = patch.generate_overlapadd_util(g["pat3d_m"], input_size=11, time_context=30, overlap=25, batch_size=8)
    assert n3 == int(g["pat3d_n"])
    check(g, "pat3d_fb", fb3)


def test_crossfade_closed_form(golden):
    """Closed-form weights (SURVEY App. A.5) == the sequential recurrence, and sum to 1."""
    g = golden
    for ci in range(int(g["n_pat"])):
        tc, ov, bs = (int(v) for v in g["pat%d_cfg" % ci])
        n = int(g["pat%d_n" % ci])
        if not n:
            continue
        pred, m = g["pat%d_pred" % ci], g["pat%d_m" % ci]
        fb, _ = patch.generate_overlapadd(m, input_size=m.shape[1], time_context=tc, overlap=ov, batch_size=bs)
        sep = patch.overlapadd_multi(pred, fb, n, overlap=ov)
        check(g, "pat%d_sep" % ci, sep)
        flat = pred.transpose(1, 0, 2, 3, 4, 5).reshape(4, -1, tc, pred.shape[-1])  # [src, patch, tc, F]
        for t in range(sep.shape[1]):
            ws = patch.crossfade_weights(t, n, tc, ov)
            if not ws:
                assert np.all(sep[:, t] == 0)
                continue
            assert abs(sum(w for _, w in ws) - 1) < 1e-12
            acc = sum(w * flat[:, k, t - k * (tc - ov)] for k, w in ws)
            np.testing.assert_allclose(acc, sep[:, t], rtol=0, atol=1e-14)
