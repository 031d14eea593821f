"""Host-side pieces of bench.py and of the multi-GPU plumbing that need no GPU."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from oracle import nets  # noqa: E402
from deepconvsep_b200 import sharding  # noqa: E402


@pytest.mark.parametrize("arch,F", [("dsd", 513), ("dsd", 1025), ("ikala", 513), ("bach10", 257), ("bach10_score", 257)])
def test_bench_weights_are_the_oracles(arch, F):
    """bench.py may not import the oracle on the timed path, so it carries its own shape table: same stream
    of numbers as oracle.nets.make_synthetic_params (the fixtures of tools/make_bench_check.py depend on it)."""
    assert bench.param_shapes(arch, F) == [tuple(s) for s in nets.param_shapes(arch, F)]
    a, b = bench.synthetic_params(arch, F, 0), nets.make_synthetic_params(arch, F, seed=0)
    assert len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))


def test_stage_work_covers_every_stage_of_every_config():
    stages = ["stft_fwd", "enc_conv1_gemm", "enc_conv2_gemm", "bottleneck_gemm", "dec_dense_gemm", "dec_convT2_gemm",
              "dec_convT1_mask_xfade", "istft_ola"]
    for name, cfg in bench.CONFIGS.items():
        L = int(cfg["seconds"] * 44100)
        extra = (["enc_maxpool"] if cfg["arch"] == "ikala" else []) + (["score_channels"] if cfg["arch"] == "bach10_score" else [])
        for st in stages + extra:
            by, fl = bench.stage_work(cfg, st, L)
            assert by > 0 and fl > 0, (name, st)
    # SURVEY 8(d): 264.5 MFLOP of tensor work per audio-second for DSD100 at N=2048 (de-duplicated)
    cfg, L = bench.CONFIGS["dsd2048"], 180 * 44100
    tens = sum(bench.stage_work(cfg, s, L)[1] for s in stages[1:7]) / 180.0
    assert 2.5e8 < tens < 3.4e8


def test_synthetic_filters_are_normalised():
    f = bench.synthetic_filters(120, 257)
    assert f.shape == (4, 120, 257) and f.dtype == np.float32
    np.testing.assert_allclose(f.sum(axis=0), 1.0, atol=3e-7)
    assert (f.max(axis=(1, 2)) > 0.9).all()


def test_effective_cores_and_cpulist():
    n = sharding.effective_cores()
    assert 1 <= n <= (os.cpu_count() or 1)
    assert sharding._parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    assert sharding.gpu_numa_node("0000:ff:1f.7-not-a-device") is None
    info = sharding.bind_to_gpu_numa(0)          # no GPU here: must be a harmless no-op
    assert info["numa_node"] is None or isinstance(info["numa_node"], int)


def test_bench_check_fixtures_are_consistent():
    for name in bench.CONFIGS:
        p = os.path.join(ROOT, "tests", "golden", "bench_check_%s.npz" % name)
        assert os.path.exists(p), "run tools/make_bench_check.py"
        g = np.load(p)
        assert g["mix"].dtype == np.int16 and g["stems"].shape == (bench.CONFIGS[name]["nsrc"], g["mix"].size)
        assert int(g["N"]) == bench.CONFIGS[name]["N"] and g["flag_t"].shape == g["flag_f"].shape
        assert g["S_or_flag"].shape == (bench.CONFIGS[name]["nsrc"], g["flag_t"].size)


def test_steps_must_be_positive(monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit):
        bench.parse_args()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "7", "--dump-outputs", "out"])
    a = bench.parse_args()
    assert a.steps == 7 and a.dump_outputs == "out"


def test_dump_outputs_whole_or_a_fixed_sample(tmp_path):
    import torch
    small = torch.arange(24, dtype=torch.float32).reshape(2, 3, 4)
    bench.dump_outputs(str(tmp_path / "a" / "stems.npy"), small)
    np.testing.assert_array_equal(np.load(str(tmp_path / "a" / "stems.npy")), small.numpy())
    big = torch.rand((2, 4, 1500000), generator=torch.Generator().manual_seed(0))
    pos = bench.dump_positions(big.numel())
    assert np.array_equal(pos, bench.dump_positions(big.numel())) and np.all(np.diff(pos) > 0)
    assert 0 <= pos[0] and pos[-1] < big.numel()
    bench.dump_outputs(str(tmp_path / "b" / "stems.npy"), big)
    got = np.load(str(tmp_path / "b" / "stems.npy"))
    assert got.dtype == np.float32 and got.nbytes <= 64 * 10 ** 6
    np.testing.assert_array_equal(got, big.numpy().reshape(-1)[pos])


def test_both_arms_print_the_same_config(monkeypatch):
    """`config` is a function of the command line and WORLD_SIZE only: the reference arm (launched by the driver
    with the same flags, torchrun included) names the same workload as this arm; its bounded sample lives elsewhere."""
    for extra, world in (([], "1"), (["--config", "bach10"], "1"), (["--gpus", "8"], "8")):
        monkeypatch.setenv("WORLD_SIZE", world)
        cfgs = []
        for impl in ("ours", "reference"):
            monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", impl, "--steps", "20", "--warmup", "5"] + extra)
            cfgs.append(bench.workload_config(bench.parse_args()))
        assert cfgs[0] == cfgs[1]
        assert cfgs[0]["job"] == "%d clips sharded over %s rank(s)" % (int(world) * cfgs[0]["clips_per_step_per_gpu"], world)
        assert "L2" in cfgs[0]["l2_policy"] and "numa" not in cfgs[0]
