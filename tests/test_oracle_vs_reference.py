"""CPU: the oracle restatement (oracle/vampnet_oracle.py) against outputs of the reference's own code.

The inputs are built here; ``python -m oracle.gen_golden vs_reference`` ran the reference on them and stored what it
returned in tests/golden/vs_reference_*.npz (logits and activations as a fixed strided sample, tokens in full)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import vampnet_oracle as vo
from oracle.gen_golden import strided_sample

CFGS = {
    "coarse": dict(n_heads=4, n_layers=2, n_codebooks=4, n_conditioning_codebooks=0, embedding_dim=256),
    "c2f": dict(n_heads=2, n_layers=1, n_codebooks=14, n_conditioning_codebooks=4, embedding_dim=128),
}
GEN_VARIANTS = (dict(sample_cutoff=-1.0, mask_temperature=0.0), dict(), dict(temperature=1.3, top_p=0.8),
                dict(sample_cutoff=0.4))
GEN_STEPS = (1, 2, 7)
GEN_SEED = 9


def forward_case(tag, lora):
    """(cfg, state_dict, codebooks, z, masked z, generate mask) of one forward/generate comparison."""
    cfg = vo.OracleConfig(**CFGS[tag])
    sd = vo.make_state_dict(cfg, seed=7, lora=lora)
    cb = vo.make_codebooks(cfg.n_codebooks, seed=2)
    z = torch.randint(0, 1024, (3, cfg.n_codebooks, 31), generator=torch.Generator().manual_seed(3))
    zm = z.clone()
    zm[:, cfg.n_conditioning_codebooks:, ::2] = 1024
    mask = torch.ones_like(z)
    mask[:, :, ::5] = 0
    return cfg, sd, cb, z, zm, mask


def typical_logits():
    return torch.randn(2, 9, 1024, generator=torch.Generator().manual_seed(0))


def default_mask_case():
    """(cfg, state_dict, codebooks, z, masks): generate with mask=None and with a 2-D (B, T) mask."""
    cfg = vo.OracleConfig(**CFGS["c2f"])
    sd = vo.make_state_dict(cfg, seed=4)
    cb = vo.make_codebooks(cfg.n_codebooks, seed=2)
    z = torch.randint(0, 1024, (2, 14, 12), generator=torch.Generator().manual_seed(1))
    m2 = torch.ones(2, 12, dtype=torch.long)
    m2[:, ::3] = 0
    return cfg, sd, cb, z, (None, m2)


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name), allow_pickle=False)


@pytest.mark.parametrize("tag", ["coarse", "c2f"])
@pytest.mark.parametrize("lora", [False, True])
def test_forward_and_generate_match_reference(golden_dir, tag, lora):
    g = _load(golden_dir, f"vs_reference_{tag}{'_lora' if lora else ''}.npz")
    cfg, sd, cb, z, zm, mask = forward_case(tag, lora)
    orc = vo.OracleVampNet(cfg, sd, "fp32")
    lat = orc.from_codes(zm, cb)
    assert torch.equal(strided_sample(lat), torch.from_numpy(g["latents"]))
    lo = orc.forward(lat)
    assert (strided_sample(lo) - torch.from_numpy(g["logits"])).abs().max() < 3e-5
    lo2, acts = orc.forward(lat, return_activations=True)  # residual stream after every layer (transformer.py:443-461)
    assert tuple(g["acts_shape"]) == acts.shape == (cfg.n_layers, 3, 31, cfg.embedding_dim)
    acts_ref = torch.from_numpy(g["acts"])
    assert (strided_sample(acts) - acts_ref).abs().max() < 3e-5 * max(1.0, float(g["acts_absmax"]))
    assert torch.equal(lo2, lo)
    assert json.loads(str(g["variants"])) == [dict(kw) for kw in GEN_VARIANTS] and tuple(g["steps"]) == GEN_STEPS
    want = torch.from_numpy(g["out"].astype(np.int64))
    i = 0
    for kw in GEN_VARIANTS:
        for steps in GEN_STEPS:
            zo = orc.generate(cb, z.clone(), mask.clone(), _sampling_steps=steps, seed=GEN_SEED, rng="torch", **kw)
            assert torch.equal(zo, want[i]), (kw, steps)
            i += 1


def test_typical_filter_is_a_noop_in_the_reference(golden_dir):
    """SURVEY.md §0.4: the reference discards typical_filter's result (transformer.py:989-993), so the oracle, which
    has no typical filter, draws what the reference draws with it on and off."""
    g = _load(golden_dir, "vs_reference_typical_filter.npz")
    a, b = (torch.from_numpy(g[k].astype(np.int64)) for k in ("typical_on", "typical_off"))
    assert torch.equal(a, b)
    cfg = vo.OracleConfig(**CFGS["coarse"])
    orc = vo.OracleVampNet.__new__(vo.OracleVampNet)
    orc.cfg = cfg
    torch.manual_seed(1)
    tok, _ = orc.sample_from_logits(typical_logits(), sample=True, temperature=1.0)
    assert torch.equal(tok, a)


def test_mask_2d_and_default_mask(golden_dir):
    g = _load(golden_dir, "vs_reference_default_mask.npz")
    cfg, sd, cb, z, masks = default_mask_case()
    orc = vo.OracleVampNet(cfg, sd, "fp32")
    for name, mask in zip(("mask_none", "mask_2d"), masks):
        zo = orc.generate(cb, z.clone(), None if mask is None else mask.clone(), _sampling_steps=3, seed=1)
        assert torch.equal(zo, torch.from_numpy(g[name].astype(np.int64))), name
