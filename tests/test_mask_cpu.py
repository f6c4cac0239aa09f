"""CPU: vampnet_b200.mask against outputs of the reference's vampnet/mask.py under the same torch seed (stored in
tests/golden/vs_reference_mask.npz), plus checks that need no reference output (including the reference's only fixture
for this code, scratch/rms_mask.txt: period 7, 3 unmasked-able codebooks)."""
import os

import numpy as np
import pytest
import torch

from vampnet_b200 import mask as pm


def test_periodic_and_codebook_mask_shape_of_fixture():
    z = torch.zeros(1, 14, 100, dtype=torch.long)
    m = pm.mask_and(pm.linear_random(z, 1.0), pm.periodic_mask(z, 7, 1, random_roll=False))
    m = pm.codebook_mask(pm.codebook_unmask(m, 0), 3)
    assert m.shape == (1, 14, 100)
    assert (m[0, 3:] == 1).all()
    assert (m[0, :3, ::7] == 0).all() and m[0, :3].sum() == 3 * (100 - 15)


def test_apply_mask_and_inpaint():
    x = torch.randint(0, 1024, (2, 4, 20))
    m = pm.inpaint(x, 3, 5)
    assert (m[:, :, :3] == 0).all() and (m[:, :, -5:] == 0).all() and (m[:, :, 3:-5] == 1).all()
    y, _ = pm.apply_mask(x, m, 1024)
    assert torch.equal(y[:, :, :3], x[:, :, :3]) and (y[:, :, 3:-5] == 1024).all()
    with pytest.raises(AssertionError):
        pm.apply_mask(x, m * 2, 1024)
    with pytest.raises(AssertionError):
        pm.apply_mask(x, m.int(), 1024)


MASK_X_SEED, BUILD_X_SEED = 0, 1
MASK_CASES = [
    lambda M, x: M.linear_random(x, 0.7),
    lambda M, x: M.random(x, 0.3),
    lambda M, x: M.inpaint(x, 4, 9),
    lambda M, x: M.inpaint(x, 0, 0),
    lambda M, x: M.periodic_mask(x, 7, 1, random_roll=True),
    lambda M, x: M.periodic_mask(x, 5, 3, random_roll=True),
    lambda M, x: M.periodic_mask(x, 0, 1),
    lambda M, x: M.codebook_mask(M.codebook_unmask(M.full_mask(x), 2), 5),
    lambda M, x: M.dropout(M.periodic_mask(x, 3, 1), 0.3),
    lambda M, x: M.mask_or(M.inpaint(x, 2, 2), M.periodic_mask(x, 4, 1)),
    lambda M, x: M.time_stretch_mask(x, 3),
    lambda M, x: M.apply_mask(x, M.periodic_mask(x, 7, 1), 1024)[0],
    lambda M, x: M._gamma(torch.linspace(0, 1, 13)),
]


def mask_case(M, i):
    """Case i of MASK_CASES run with the mask module M (ours, or the reference's when the golden file is written)."""
    x = torch.randint(0, 1024, (3, 9, 57), generator=torch.Generator().manual_seed(MASK_X_SEED))
    torch.manual_seed(123 + i)
    return MASK_CASES[i](M, x)


def build_mask_stream(M):
    """Interface.build_mask's composition of the pieces under torch.manual_seed(7), and the next draws after it."""
    x = torch.randint(0, 1024, (2, 14, 100), generator=torch.Generator().manual_seed(BUILD_X_SEED))
    torch.manual_seed(7)
    m = M.linear_random(x, 1.0)
    m = M.mask_and(m, M.inpaint(x, 0, 0))
    m = M.mask_and(m, M.periodic_mask(x, 7, 1, random_roll=True))
    m = M.dropout(m, 0.1)
    m = M.codebook_unmask(m, 0)
    return M.codebook_mask(m, 3, None), torch.rand(4)


def _golden(golden_dir):
    return np.load(os.path.join(golden_dir, "vs_reference_mask.npz"), allow_pickle=False)


def test_against_reference_mask_module(golden_dir):
    """Every piece of vampnet/mask.py against the reference's own outputs under the same torch seed
    (tests/golden/vs_reference_mask.npz, written by ``python -m oracle.gen_golden vs_reference``)."""
    g = _golden(golden_dir)
    for i in range(len(MASK_CASES)):
        got = mask_case(pm, i)
        want = torch.from_numpy(g[f"case_{i}"])
        assert got.dtype == want.dtype and torch.equal(got, want), f"case {i}"


def test_build_mask_rng_stream_matches_reference(golden_dir):
    """Interface.build_mask composes the pieces; same seed -> same mask AND same RNG state afterwards."""
    g = _golden(golden_dir)
    m, r = build_mask_stream(pm)
    assert torch.equal(m, torch.from_numpy(g["build_mask"])) and torch.equal(r, torch.from_numpy(g["build_mask_next_rand"]))
