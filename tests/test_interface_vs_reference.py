"""CPU: Interface orchestration (SURVEY.md §8 rows A1-A3 + build_mask) pinned against outputs of the REFERENCE'S OWN code.

``python -m oracle.gen_golden vs_reference`` gave a reference `Interface` object (its vampnet/interface.py, codec and
beat-tracker imports as name-only stubs) the stand-in models and the inputs defined here — `generate` is a
deterministic pure function of (start_tokens, mask) — and stored its results in tests/golden/vs_reference_interface.npz.
The outputs of `coarse_vamp`, `coarse_to_fine`, `vamp` and `build_mask`, and the generate calls behind them, must be
identical: chunking, edge anchors, padding, codebook stacking, time stretch, feedback passes, mask composition and
RNG consumption.  The oracle's restatement (oracle/vampnet_oracle.py) is checked in the same breath."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import vampnet_oracle as vo
from tests.test_interface_cpu import MASK_TOKEN, StubCodec, StubModel, fake_generate, rand_case

COARSE_S, C2F_S = 0.6, 0.25
COARSE_T = [1, 34, 35, 36, 83, 140]
C2F_CASES = [(15, 14), (29, 14), (30, 4), (47, 14), (1, 4)]
VAMP_CASES = [(1, 1, 1, 83), (3, 1, 1, 40), (2, 2, 1, 61), (2, 3, 2, 37), (1, 1, 3, 20)]
BUILD_MASK_KW = [
    dict(),
    dict(rand_mask_intensity=0.7, periodic_prompt=5, periodic_prompt_width=2, upper_codebook_mask=4),
    dict(prefix_s=0.3, suffix_s=0.2, periodic_prompt=0, _dropout=0.3, ncc=1),
    dict(rand_mask_intensity=0.0, periodic_prompt=3, upper_codebook_mask=14),
]
UNIT_SECONDS = (0.0, 0.1, 1.0, 3.0, 10.0, 13.37)


def stub_models():
    coarse, c2f = StubModel(4, 0, salt=5), StubModel(14, 4, salt=9)
    coarse.chunk_size_s, c2f.chunk_size_s = COARSE_S, C2F_S
    return coarse, c2f


def calls(model, keys):
    """The generate calls a stand-in model saw, as plain JSON data."""
    return json.dumps([{k: c[k] for k in keys} for c in model.calls])


# Each case runs one entry point on an Interface (ours, or the reference's when the golden file is written) and
# returns its results by name: token tensors, and the generate calls as JSON.
def coarse_vamp_case(iface, T):
    z, mask = rand_case(2, T, seed=T)
    if T > 70:
        mask[:, :, 70:] = 1
    out, start = iface.coarse_vamp(z, mask, return_mask=True, temperature=0.7)
    return dict(out=out, start=start, calls=calls(iface.coarse, ("kwargs", "shape")))


def coarse_to_fine_case(iface, T, n_in):
    z, mask = rand_case(2, T, seed=100 + T)
    z = z[:, :n_in]
    out, start = iface.coarse_to_fine(z, mask=mask, return_mask=True)
    no_mask = iface.coarse_to_fine(z, mask=None)
    return dict(out=out, start=start, no_mask=no_mask, calls=calls(iface.c2f, ("time_steps", "shape", "kwargs")))


def vamp_case(iface, batch, feedback, stretch, T):
    z, mask = rand_case(1, T, seed=7 * T + batch)
    out, out_mask = iface.vamp(z, mask, batch_size=batch, feedback_steps=feedback, time_stretch_factor=stretch,
                               return_mask=True, temperature=1.3)
    return dict(out=out, mask=out_mask, calls=calls(iface.c2f, ("kwargs",)))


def build_mask_case(iface, i):
    z, _ = rand_case(2, 97, seed=3)
    torch.manual_seed(11)
    mask = iface.build_mask(z, **BUILD_MASK_KW[i])
    return dict(mask=mask, rng=torch.get_rng_state())


def units(iface):
    return json.dumps([[iface.s2t(s), iface.s2t2s(s)] for s in UNIT_SECONDS] + [iface.t2s(575)])


def case_key(kind, *params):
    return "_".join([kind] + [str(p) for p in params])


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "vs_reference_interface.npz"), allow_pickle=False)


def ours():
    from vampnet_b200.interface import Interface
    return Interface.from_models(StubCodec(), *stub_models(), device="cpu", coarse_chunk_size_s=COARSE_S,
                                 coarse2fine_chunk_size_s=C2F_S)


def check(got, golden, key):
    for name, v in got.items():
        want = golden[f"{key}.{name}"]
        if isinstance(v, str):
            assert json.loads(v) == json.loads(str(want)), (key, name)
        else:
            assert torch.equal(v, torch.from_numpy(want).to(v.dtype)), (key, name)


@pytest.mark.parametrize("T", COARSE_T)
def test_coarse_vamp(golden, T):
    iface = ours()
    got = coarse_vamp_case(iface, T)
    check(got, golden, case_key("coarse_vamp", T))
    z, mask = rand_case(2, T, seed=T)
    if T > 70:
        mask[:, :, 70:] = 1
    o, o_start = vo.coarse_vamp(z, mask, 4, iface.s2t(COARSE_S), MASK_TOKEN, lambda s, m: fake_generate(s, m, 5))
    assert torch.equal(o, got["out"]) and torch.equal(o_start, got["start"])


@pytest.mark.parametrize("T,n_in", C2F_CASES)
def test_coarse_to_fine(golden, T, n_in):
    iface = ours()
    got = coarse_to_fine_case(iface, T, n_in)
    check(got, golden, case_key("coarse_to_fine", T, n_in))
    z, mask = rand_case(2, T, seed=100 + T)
    o, o_start = vo.coarse_to_fine(z[:, :n_in], mask, 14, 4, iface.s2t(C2F_S), MASK_TOKEN,
                                   lambda s, m: fake_generate(s, m, 9))
    assert torch.equal(o, got["out"]) and torch.equal(o_start, got["start"])


@pytest.mark.parametrize("batch,feedback,stretch,T", VAMP_CASES)
def test_vamp(golden, batch, feedback, stretch, T):
    iface = ours()
    got = vamp_case(iface, batch, feedback, stretch, T)
    check(got, golden, case_key("vamp", batch, feedback, stretch, T))
    z, mask = rand_case(1, T, seed=7 * T + batch)
    o, o_mask = vo.vamp(z, mask, batch, feedback, stretch, 4, 14, 4, iface.s2t(COARSE_S), iface.s2t(C2F_S), MASK_TOKEN,
                        lambda s, m: fake_generate(s, m, 5), lambda s, m: fake_generate(s, m, 9))
    assert torch.equal(o, got["out"]) and torch.equal(o_mask, got["mask"])


@pytest.mark.parametrize("kw", BUILD_MASK_KW)
def test_build_mask(golden, kw):
    # the mask and the global RNG state afterwards: the same draws were consumed in the same order
    check(build_mask_case(ours(), BUILD_MASK_KW.index(kw)), golden, case_key("build_mask", BUILD_MASK_KW.index(kw)))


def test_units(golden):
    assert json.loads(units(ours())) == json.loads(str(golden["units"]))
