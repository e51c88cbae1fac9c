"""Host tests of emission saliency: the stratified timestep schedule, the saliency noise draw ids, saliency.py's
argument checks and the NetCDF writer.  The kernels, the engine and the CLI run are tests/test_saliency_gpu.py's."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_ema_host import _tiny_checkpoint  # noqa: E402


@pytest.mark.parametrize("T,D", [(1000, 1), (1000, 16), (1000, 3), (1000, 1000), (7, 7), (10, 4)])
def test_stratified_timesteps(T, D):
    from cesm_emulator_b200.engine import saliency_timesteps
    t = saliency_timesteps(T, D)
    assert t.dtype == torch.int64 and t.shape == (D,)
    assert t.tolist() == [int(np.floor((d + 0.5) * T / D)) for d in range(D)]
    assert int(t.min()) >= 0 and int(t.max()) < T and len(set(t.tolist())) == D  # distinct, inside the schedule
    for d, v in enumerate(t.tolist()):  # the midpoint of stratum d
        assert d * T / D <= v < (d + 1) * T / D


def test_stratified_timesteps_examples():
    from cesm_emulator_b200.engine import saliency_timesteps
    assert saliency_timesteps(1000, 1).tolist() == [500]
    assert saliency_timesteps(1000, 4).tolist() == [125, 375, 625, 875]
    assert saliency_timesteps(1000, 1000).tolist() == list(range(1000))


@pytest.mark.parametrize("D", [0, -1, 1001, 2.0, True, "4", None])
def test_stratified_timesteps_bounds(D):
    from cesm_emulator_b200.engine import saliency_timesteps
    with pytest.raises(ValueError):
        saliency_timesteps(1000, D)


def test_saliency_draw_ids_are_disjoint_from_the_samplers():
    from cesm_emulator_b200 import kernels as K
    first, last = K.SALIENCY_DRAW_BASE, K.SALIENCY_DRAW_BASE + K.SALIENCY_MAX_DRAWS - 1
    # sampler draws: timesteps 0..T-1 (any T < 2^31) and X_T_DRAW
    assert first >= 1 << 31 and last < K.X_T_DRAW and last <= 0xFFFFFFFF
    assert not first <= K.X_T_DRAW <= last


@pytest.mark.parametrize("argv", [["--draws", "0"], ["--draws", "-3"], ["--seed", "-1"], ["--seed", str(1 << 64)],
                                  ["--batch_size", "0"]])
def test_cli_argument_errors(argv, capsys):
    import saliency
    with pytest.raises(SystemExit) as e:
        saliency._parse_args(["--ckpt", "x.pt", *argv])
    assert e.value.code == 2
    assert "error" in capsys.readouterr().err


def test_cli_accepts_the_seed_range():
    import saliency
    assert saliency._parse_args(["--ckpt", "x.pt", "--seed", str((1 << 64) - 1)]).seed == (1 << 64) - 1
    a = saliency._parse_args(["--ckpt", "x.pt"])
    assert (a.draws, a.seed, a.batch_size, a.members, a.times, a.ema) == (16, None, 8, 2, 8, False)


def test_cli_ema_on_a_checkpoint_without_one(tmp_path):
    import saliency
    path, _, _, _ = _tiny_checkpoint(tmp_path, with_ema=False)
    with pytest.raises(SystemExit) as e:
        saliency.main(["--ckpt", path, "--ema", "--out", str(tmp_path / "s.npy")])
    assert '"ema"' in str(e.value.code)
    assert not os.path.exists(tmp_path / "s.npy")


def test_netcdf_writer_round_trip(tmp_path):
    from scipy.io import netcdf_file
    import saliency
    sal = np.random.default_rng(0).standard_normal((3, 2, 3, 4, 5)).astype(np.float32)
    path = str(tmp_path / "out" / "sal.nc")
    attrs = {"checkpoint": "/x/final.pt", "cond_var": "synthetic", "draws": 16, "seed": "7", "ema": 1}
    saliency.write_saliency_netcdf(path, sal, lat=np.linspace(-1, 1, 4), attrs=attrs)
    with netcdf_file(path, "r", mmap=False) as f:
        v = f.variables["saliency"]
        assert v.dimensions == ("window", "member_id", "frame", "lat", "lon")
        assert np.array_equal(np.array(v[:]), sal)
        assert (v.checkpoint, v.cond_var, v.draws, v.seed, v.ema) == (b"/x/final.pt", b"synthetic", 16, b"7", 1)
        assert np.allclose(f.variables["lat"][:], np.linspace(-1, 1, 4))
        assert list(f.variables["window"][:]) == [0, 1, 2] and list(f.variables["frame"][:]) == [0, 1, 2]
    with pytest.raises(ValueError):
        saliency.write_saliency_netcdf(str(tmp_path / "bad.nc"), sal, lat=np.zeros(3))
