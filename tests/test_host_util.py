"""Host-side mirror of the reference interface (no GPU): util drop-ins == oracle (which is
pinned to the reference's own functions), tensor-dump format, wav helpers, CLI plumbing."""
import os
import numpy as np
import pytest

from deepconvsep_b200 import util
from dspgolden import check
from oracle import patch


def test_util_patchers_and_crossfade_equal_oracle():
    rng = np.random.default_rng(0)
    for T, F, tc, ov, bs in [(100, 7, 30, 25, 32), (64, 5, 30, 20, 8), (30, 5, 30, 25, 4), (31, 3, 30, 25, 4),
                             (203, 4, 20, 15, 16), (9, 3, 30, 25, 4), (40, 3, 30, 0, 4)]:
        m = rng.random((T, F))
        a, n = util.generate_overlapadd(m, F, tc, ov, bs)
        b, n2 = patch.generate_overlapadd_util(m, F, tc, ov, bs)
        assert n == n2 and np.array_equal(a, b)
        a, n = util.generate_overlapadd_standalone(m, F, tc, ov, bs)
        b, n2 = patch.generate_overlapadd(m, F, tc, ov, bs)
        assert n == n2 and np.array_equal(a, b)
        if n:
            pred = rng.random((a.shape[0], 4, bs, 1, tc, F))
            assert np.array_equal(util.overlapadd_multi(pred, a, n, ov), patch.overlapadd_multi(pred, a, n, ov))
            s1, s2 = util.overlapadd(pred, a, n, ov)
            t1, t2 = patch.overlapadd(pred[:, :2], a, n, ov)
            assert np.array_equal(s1, t1) and np.array_equal(s2, t2)
    m3 = rng.random((4, 57, 11))
    a, n = util.generate_overlapadd(m3, 11, 30, 25, 8)
    b, n2 = patch.generate_overlapadd_util(m3, 11, 30, 25, 8)
    assert n == n2 and np.array_equal(a, b)
    with pytest.raises(AssertionError):
        util.generate_overlapadd(m3, 12, 30, 25, 8)


def test_golden_patchers(golden):
    """...and directly against the vectors produced by the reference's own functions."""
    g = golden
    for ci in range(int(g["n_pat"])):
        tc, ov, bs = (int(v) for v in g["pat%d_cfg" % ci])
        m = g["pat%d_m" % ci]
        fb, n = util.generate_overlapadd_standalone(m, m.shape[1], tc, ov, bs)
        assert n == int(g["pat%d_n" % ci])
        check(g, "pat%d_fb" % ci, fb)
        fbu, nu = util.generate_overlapadd(m, m.shape[1], tc, ov, bs)
        assert nu == int(g["pat%d_nu" % ci])
        check(g, "pat%d_fbu" % ci, fbu)
        if n:
            check(g, "pat%d_sep" % ci, util.overlapadd_multi(g["pat%d_pred" % ci], fb, n, ov))


def test_wav_helpers_and_tensor_dump(tmp_path):
    from deepconvsep_b200.transform import Transforms
    rng = np.random.default_rng(1)
    x = (rng.standard_normal(1000) * 0.1)
    fn = str(tmp_path / "a.wav")
    util.writeAudioScipy(fn, x, 44100, "int16")
    y, sr, dt = util.readAudioScipy(fn)
    assert sr == 44100 and dt == np.int16
    assert np.array_equal((x * 32767).astype("int16"), np.round(y * 32767).astype("int16"))
    assert util.infoAudioScipy(fn) == (1000, 44100, np.dtype("int16"))
    # .data / .shape dumps (transform.py:159-185): raw float64 + '#a\tb\tc'
    t = Transforms(frameSize=256)
    t.out_path = str(tmp_path / "feat.data")
    arr = rng.random((2, 5, 7))
    t.saveTensor(arr, "_x_m_")
    assert open(str(tmp_path / "feat_x_m_.shape")).read() == "#2\t5\t7\n"
    assert os.path.getsize(str(tmp_path / "feat_x_m_.data")) == arr.size * 8
    np.testing.assert_array_equal(t.loadTensor("_x_m_"), arr)


def test_cli_usage_and_descriptors(capsys):
    import deepconvsep_b200.examples.dsd100.separate_dsd as sd
    import deepconvsep_b200.examples.hiphopss.separate_hhds as sh
    import deepconvsep_b200.examples.ikala.separate_ikala as si
    import deepconvsep_b200.examples.bach10.separate_bach10 as sb
    import deepconvsep_b200.examples.bach10_scoreinformed.separate_bach10 as ss
    assert ss.build_ca()["nchannels"] == 4
    for mod in (sd, sh, si, sb, ss):
        with pytest.raises(SystemExit):
            mod.main(["-h"])
        assert "-i <inputfile> -o <outputdir> -m <path_to_model.pkl>" in capsys.readouterr().out
        with pytest.raises(SystemExit) as e:
            mod.main(["--bogus"])
        assert e.value.code == 2
        capsys.readouterr()
    assert sd.build_ca(None, 32, 30, 513)["nsources"] == 4 and si.build_ca()["nsources"] == 2


def test_cli_parse_long_options(tmp_path):
    """`-i -o -m` as the reference scripts take them, plus the long options of SURVEY.md 5 (host logic only)"""
    from deepconvsep_b200.examples import _common
    o = _common.parse_cli(["-i", "a.wav", "-o", "out", "-m", "m.pkl"], "usage")
    assert (o["inputfile"], o["outdir"], o["model"]) == ("a.wav", "out", "m.pkl")
    assert o["frame_size"] is None and o["window"] is None and o["devices"] is None and o["batch_clips"] == 1
    o = _common.parse_cli(["--ifile", "d", "--odir", "o", "--mfile", "m", "--frame-size", "2048", "--window", "blackmanharris",
                           "--devices", "0,3", "--batch-clips", "4"], "usage")
    assert o["frame_size"] == 2048 and o["window"] == "blackmanharris" and o["devices"] == [0, 3] and o["batch_clips"] == 4
    import pytest
    with pytest.raises(SystemExit):
        _common.parse_cli(["-i", "a.wav"], "usage")            # -o / -m missing: usage + exit 2, like the reference
    with pytest.raises(SystemExit):
        _common.parse_cli(["--no-such-flag"], "usage")
