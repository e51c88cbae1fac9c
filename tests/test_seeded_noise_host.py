"""CPU tests of seeded, shard-invariant ensemble generation: the numpy Philox4x32-10 oracle against the Random123
known-answer vectors, the oracle's Box-Muller normals, seed and field-id validation, and inference.py's --seed."""
import numpy as np
import pytest
import torch

import philox_oracle as PO


@pytest.mark.parametrize("ctr, key, expect", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, expect):
    assert tuple(int(w) for w in PO.philox4x32_10(ctr, key)) == expect


def test_uniform_is_exact_in_fp32_and_open():
    w = np.array([0, 1, 511, 512, 1 << 31, 0xFFFFFDFF, 0xFFFFFE00, 0xFFFFFFFF], dtype=np.uint32)
    u = PO.uniform(w)
    u32 = ((w >> np.uint32(9)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -23)   # the kernel's arithmetic
    assert np.array_equal(u32.astype(np.float64), u)
    assert u.min() == 2.0 ** -24 and u.max() == 1 - 2.0 ** -24


def test_oracle_normals_are_per_field_and_standard():
    a = PO.field_normal(7, 3, 0, 4 * 50_000)
    assert abs(a.mean()) < 5 / np.sqrt(a.size) and abs(a.var() - 1) < 5 * np.sqrt(2 / a.size)
    assert np.array_equal(PO.field_normal(7, 3, 0, 13), a[:13])          # a prefix does not depend on the size
    assert not np.allclose(PO.field_normal(7, 4, 0, 16), a[:16])          # other field, other draw, other seed
    assert not np.allclose(PO.field_normal(7, 3, 1, 16), a[:16])
    assert not np.allclose(PO.field_normal(8, 3, 0, 16), a[:16])
    big = PO.field_normal(7, 3 + (1 << 32), 0, 16)                        # the high word of the id counts
    assert not np.allclose(big, a[:16])


@pytest.mark.parametrize("bad", [-1, 1 << 64, True, False, 1.0, "3", None])
def test_split_seed_rejects(bad):
    from cesm_emulator_b200 import kernels as K
    with pytest.raises(ValueError):
        K.split_seed(bad)


def test_split_seed_words():
    from cesm_emulator_b200 import kernels as K
    assert K.split_seed(0) == (0, 0)
    assert K.split_seed((1 << 64) - 1) == (0xFFFFFFFF, 0xFFFFFFFF)
    assert K.split_seed(np.uint64(5 << 32 | 9)) == (9, 5)


def test_field_id_vector():
    from cesm_emulator_b200 import kernels as K
    assert K.field_id_vector(None, 3, "cpu").tolist() == [0, 1, 2]
    assert K.field_id_vector([4, 4, 1 << 40], 3, "cpu").tolist() == [4, 4, 1 << 40]   # repeats are padding rows
    for bad in ([0, -1, 2], [0, 1], [[0, 1, 2]], [0.0, 1.0, 2.0], [True, False, True]):
        with pytest.raises(ValueError):
            K.field_id_vector(bad, 3, "cpu")


def test_unseeded_paths_reject_field_ids_and_bad_seeds():
    """Checked before any device work, so no GPU is needed."""
    from torch import nn

    from cesm_emulator_b200.engine import SampleEngine
    from cesm_emulator_b200.model import Diffusion
    d = Diffusion(nn.Linear(1, 1))
    with pytest.raises(ValueError):
        d.sample(None, (2, 1, 4, 4), "cpu", field_ids=[0, 1])
    with pytest.raises(ValueError):
        d.ddim_sample(None, (2, 1, 4, 4), "cpu", steps=5, field_ids=[0, 1])
    with pytest.raises(ValueError):
        d.dpm_sample(None, (2, 1, 4, 4), "cpu", steps=5, seed=-3)
    with pytest.raises(ValueError):
        SampleEngine(d, (2, 1, 4, 4), seed=True)
    with pytest.raises(ValueError):
        SampleEngine(d, (2, 1, 4, 4), ddim_steps=5, seed=1 << 64)
    with pytest.raises(ValueError):
        SampleEngine(d, (2, 1, 4, 4)).sample(torch.zeros(2, 1, 4, 4), field_ids=[0, 1])


def test_cli_seed():
    import inference
    assert inference._parse_args(["--ckpt", "c.pt"]).seed is None
    assert inference._parse_args(["--ckpt", "c.pt", "--seed", "7"]).seed == 7
    assert inference._parse_args(["--ckpt", "c.pt", "--seed", str((1 << 64) - 1)]).seed == (1 << 64) - 1
    for bad in ("-1", str(1 << 64), "1.5"):
        with pytest.raises(SystemExit):
            inference._parse_args(["--ckpt", "c.pt", "--seed", bad])
