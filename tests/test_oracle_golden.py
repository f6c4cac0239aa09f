"""CPU: the oracle restatement (oracle/vampnet_oracle.py) against the committed golden
vectors that were produced by the reference's own code (oracle/gen_golden.py)."""
import glob
import json
import os

import numpy as np
import pytest
import torch

from oracle import vampnet_oracle as vo
from oracle.gen_golden import load


def _load(golden_dir, name):
    return load(os.path.join(golden_dir, name))


def _model(g, mode="fp32"):
    cfg = vo.OracleConfig(**json.loads(str(g["cfg"])))
    sd = vo.make_state_dict(cfg, seed=int(g["weight_seed"]), lora=bool(int(g["lora"])) if "lora" in g else False)
    return cfg, vo.OracleVampNet(cfg, sd, mode)


def test_relbucket_lut(golden_dir):
    g = _load(golden_dir, "relbucket_lut_T3072.npz")
    lut = vo.relative_position_bucket_lut(3072)
    assert np.array_equal(lut.numpy().astype(np.int8), g["lut"])
    # SURVEY.md §A.3 spot checks (rel = key - query)
    T = 3072
    at = lambda rel: int(lut[rel + T - 1])
    assert at(0) == 0 and at(-7) == 7 and at(-8) == 8 and at(-91) == 15 and at(-3000) == 15
    assert at(1) == 17 and at(7) == 23 and at(8) == 24 and at(90) == 30 and at(91) == 31
    # Toeplitz: a shorter T is a centred slice of the long LUT
    short = vo.relative_position_bucket_lut(100)
    assert torch.equal(short, lut[T - 100: T + 99])


def test_gamma_schedule(golden_dir):
    rows = _load(golden_dir, "gamma_schedule.npz")["rows"]
    for steps, n0, i, n in rows.tolist():  # python ints: (i+1)/steps must be a python float -> fp32 tensor
        r = torch.tensor((i + 1) / steps).repeat(1)
        got = torch.floor(vo.gamma(r) * torch.tensor(int(n0))).long().item()
        assert got == n, (steps, n0, i, n, got)


@pytest.mark.parametrize("tag", ["coarse", "c2f", "coarse_lora"])
def test_forward_tiny(golden_dir, tag):
    g = _load(golden_dir, f"forward_tiny_{tag}.npz")
    cfg, orc = _model(g)
    cb = vo.make_codebooks(cfg.n_codebooks, seed=int(g["codebook_seed"]))
    lat = orc.from_codes(torch.from_numpy(g["codes"]), cb)
    assert np.array_equal(lat.numpy(), g["latents"])
    logits = orc.forward(lat)
    np.testing.assert_allclose(logits.numpy(), g["logits"], atol=2e-5, rtol=0)


def test_forward_tiny_bf16_mode_is_close(golden_dir):
    """The bf16-operand mode (the kernels' parity target) stays near the fp32 reference; the
    distance is the quantisation error we report, not a kernel bug."""
    g = _load(golden_dir, "forward_tiny_coarse.npz")
    cfg, orc = _model(g, "bf16")
    logits = orc.forward(torch.from_numpy(g["latents"]))
    err = np.abs(logits.numpy() - g["logits"])
    assert err.mean() < 2e-2 and err.max() < 0.25, (err.mean(), err.max())


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "generate_tiny_*.npz"))))
def test_generate_tiny(path):
    g = np.load(path, allow_pickle=False)
    cfg, orc = _model(g)
    cb = vo.make_codebooks(cfg.n_codebooks, seed=int(g["codebook_seed"]))
    kw = json.loads(str(g["kwargs"]))
    out = orc.generate(cb, torch.from_numpy(g["z"]), torch.from_numpy(g["mask"]), _sampling_steps=int(g["steps"]),
                       seed=int(g["seed"]), rng="torch", **kw)
    assert np.array_equal(out.numpy(), g["out"])
    assert not (out == cfg.mask_token).any()
    keep = torch.from_numpy(g["mask"]) == 0
    assert torch.equal(out[keep], torch.from_numpy(g["z"])[keep])  # unmasked inputs are preserved


def test_sampler_pieces(golden_dir):
    g = _load(golden_dir, "sampler_greedy.npz")
    cfg = vo.OracleConfig(n_heads=4, n_layers=0, n_codebooks=4, embedding_dim=256)
    orc = vo.OracleVampNet.__new__(vo.OracleVampNet)
    orc.cfg = cfg
    logits = torch.from_numpy(g["logits"])
    tok, p = orc.sample_from_logits(logits, sample=False, temperature=1.0)
    assert np.array_equal(tok.numpy(), g["tok"])
    np.testing.assert_allclose(p.numpy(), g["p"], rtol=1e-6)
    tok_t, p_t = orc.sample_from_logits(logits, sample=False, temperature=0.7)
    assert np.array_equal(tok_t.numpy(), g["tok_t"])
    np.testing.assert_allclose(p_t.numpy(), g["p_t"], rtol=1e-6)
    m, _ = vo.OracleVampNet.mask_by_random_topk(torch.from_numpy(g["n"]), torch.from_numpy(g["p_inf"]), torch.zeros(3))
    assert np.array_equal(m.numpy(), g["remask"])
    assert m.sum(-1).tolist() == g["n"].reshape(-1).tolist()


def test_forward_full_coarse_T100(golden_dir):
    """BASELINE.json configs[0]: random-init coarse VampNet (4 codebooks, d=1280, 20 layers), T=100, B=1, CPU."""
    g = _load(golden_dir, "forward_full_coarse_T100.npz")
    cfg = vo.OracleConfig(**json.loads(str(g["cfg"])))
    sd = vo.make_state_dict(cfg, seed=int(g["weight_seed"]))
    orc = vo.OracleVampNet(cfg, sd, "fp32")
    lat = torch.randn(1, 32, 100, generator=torch.Generator().manual_seed(int(g["latents_seed"])))
    logits = orc.forward(lat)
    assert logits.shape == (1, 1024, 400)
    np.testing.assert_allclose(logits[:, :, ::16].numpy(), g["logits_sub"], atol=5e-4, rtol=0)
    assert (logits.argmax(1).numpy() == g["argmax"]).mean() > 0.995


def test_philox_known_answer():
    """Random123 known-answer vectors for Philox4x32-10."""
    from oracle import philox
    o = philox.philox4x32_10(0, 0, 0, 0, 0, 0)
    assert [int(x) for x in o] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    o = philox.philox4x32_10(0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF)
    assert [int(x) for x in o] == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    o = philox.philox4x32_10(0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344, 0xA4093822, 0x299F31D0)
    assert [int(x) for x in o] == [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]
    u = philox.uniform_bsv((1, 2), 3, 2, 5, 1024)
    assert u.dtype == np.float32 and u.min() > 0 and u.max() < 1 and abs(u.mean() - 0.5) < 0.02
