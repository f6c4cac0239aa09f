"""GPU: forward parity at the BENCHMARKED shapes and exact-decision tests that bite.

What can and cannot be asserted about logits computed with bf16 operands is measured in
tests/test_oracle_conditioning_cpu.py: the oracle's bf16 mode moves by ~1.5e-2 max / 2e-3 mean (2 layers) to
~3e-2 / 5e-3 (20 layers) when its activations are nudged by a relative 1e-7 before rounding.  The tests below
therefore (1) require the kernels to sit within 1.5x of that floor, measured on the SAME inputs by running the
oracle's jitter probe next to the comparison, (2) bound the distance to the fp32 reference by fixed numbers, and
(3) turn the bound into exact statements: wherever the fp32 reference's top-2 logit margin exceeds twice the bound,
the greedy decision (argmax) MUST equal the reference's — no agreement rates, no teacher forcing.

Fixed bounds vs the fp32 reference (logit std ~1): TOL32 = 0.09 max, 1.2e-2 mean (measured 2.5e-2..5.8e-2 max,
4e-3..8.3e-3 mean; the reference's own bf16-autocast path: 3.2e-2 / 5.6e-3, BASELINE.md §2)."""
import glob
import json
import os
import time

import numpy as np
import pytest
import torch

from oracle import vampnet_oracle as vo
from oracle.gen_golden import load
from tests.test_gpu_parity import TINY_C2F, TINY_COARSE, build

pytestmark = pytest.mark.gpu

TOL32_MAX, TOL32_MEAN = 0.09, 1.2e-2
FULL_COARSE = dict(n_heads=20, n_layers=20, n_codebooks=4, n_conditioning_codebooks=0, embedding_dim=1280)
FULL_C2F = dict(n_heads=20, n_layers=16, n_codebooks=14, n_conditioning_codebooks=4, embedding_dim=1280)


def margins(ref_logits_bsv):
    """top-1 minus top-2 logit per position of a (B, S, V) tensor, and the argmax."""
    top2 = ref_logits_bsv.topk(2, dim=-1)
    return top2.values[..., 0] - top2.values[..., 1], top2.indices[..., 0]


def assert_decisions_exact_where_margin_allows(got_bsv, ref32_bsv, tag):
    e = (got_bsv - ref32_bsv).abs()
    assert e.max() <= TOL32_MAX and e.mean() <= TOL32_MEAN, (tag, e.max().item(), e.mean().item())
    m, arg = margins(ref32_bsv)
    safe = m > 2 * TOL32_MAX
    got_arg = got_bsv.argmax(-1)
    wrong = (got_arg != arg) & safe
    print(f"[{tag}] vs fp32 reference: max {e.max():.3e} mean {e.mean():.3e}; margin > {2 * TOL32_MAX:.2f} at "
          f"{safe.float().mean():.1%} of {safe.numel()} positions, all decided identically; overall argmax agreement "
          f"{(got_arg == arg).float().mean():.4f}")
    assert safe.float().mean() > 0.2, "the margin test must cover a real share of the positions"
    assert not wrong.any(), f"{int(wrong.sum())} decisions with a safe margin differ from the reference"
    # and the tight form: a flipped decision is only possible where the measured errors can explain it
    flipped = got_arg != arg
    if flipped.any():
        assert (m[flipped] <= 2 * e.max()).all()


@pytest.mark.parametrize("tag,cfgd,lora", [("coarse", TINY_COARSE, False), ("c2f", TINY_C2F, False),
                                           ("coarse_lora", TINY_COARSE, True)])
def test_forward_decisions_vs_reference_golden(golden_dir, tag, cfgd, lora):
    g = load(os.path.join(golden_dir, f"forward_tiny_{tag}.npz"))
    cfg, sd, model, cb, codec = build(cfgd, seed=int(g["weight_seed"]), lora=lora, cb_seed=int(g["codebook_seed"]))
    got = model(torch.from_numpy(g["latents"]).cuda()).cpu()          # (B, V, S)
    ref32 = torch.from_numpy(g["logits"])                             # the reference's own fp32 output
    assert_decisions_exact_where_margin_allows(got.permute(0, 2, 1), ref32.permute(0, 2, 1), tag)


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden",
                                                                "generate_tiny_*_greedy_s1.npz"))))
def test_greedy_generate_one_step_exact_where_margin_allows(path):
    """One greedy sampling iteration (sample_cutoff < 0, mask_temperature = 0) END TO END against the reference's own
    output tokens: every masked position whose fp32 margin is safe must carry the reference's token.  No teacher
    forcing: the product computes its own logits."""
    g = np.load(path)
    cfgd = json.loads(str(g["cfg"]))
    cfg, sd, model, cb, codec = build(cfgd, seed=int(g["weight_seed"]), lora=bool(int(g["lora"])),
                                      cb_seed=int(g["codebook_seed"]))
    kw = json.loads(str(g["kwargs"]))
    z, mask = torch.from_numpy(g["z"]), torch.from_numpy(g["mask"])
    got = model.generate(codec, start_tokens=z.cuda(), mask=mask.cuda(), _sampling_steps=1, seed=5,
                         return_signal=False, **kw).cpu()
    want = torch.from_numpy(g["out"])
    # margins from the fp32 oracle (pinned bit-for-bit to the reference's generate by tests/test_oracle_vs_reference.py)
    orc = vo.OracleVampNet(cfg, sd, "fp32")
    zm = z.masked_fill(mask.bool(), cfg.mask_token)
    ref32 = orc.forward(orc.from_codes(zm, cb)).permute(0, 2, 1)      # (B, S, V), s = t*Cp + c
    m, arg = margins(ref32)
    ncc, Cp = cfg.n_conditioning_codebooks, cfg.n_predict_codebooks
    m_bct = vo.codebook_unflatten(m, Cp)
    safe = torch.zeros_like(mask, dtype=torch.bool)
    safe[:, ncc:] = (m_bct > 2 * TOL32_MAX) & mask[:, ncc:].bool()
    assert torch.equal(vo.codebook_unflatten(arg, Cp)[mask[:, ncc:].bool()], want[:, ncc:][mask[:, ncc:].bool()])  # oracle == golden
    n_safe, n_masked = int(safe.sum()), int(mask[:, ncc:].sum())
    print(f"{os.path.basename(path)}: {n_safe}/{n_masked} masked positions have a safe margin; agreement overall "
          f"{(got == want).float().mean():.4f}")
    assert n_safe > 0.2 * n_masked
    assert torch.equal(got[safe], want[safe])
    assert torch.equal(got[mask == 0], z[mask == 0])


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden",
                                                                "generate_tiny_*_greedy_s6.npz"))))
def test_greedy_generate_six_steps_agreement_floor(path):
    """Six iterations: one early low-margin flip changes every later input, so this stays an agreement rate — with the
    floor at what a correct bf16 implementation measures (0.878 .. 1.000 in round 1), not at 0.5."""
    g = np.load(path)
    cfgd = json.loads(str(g["cfg"]))
    cfg, sd, model, cb, codec = build(cfgd, seed=int(g["weight_seed"]), lora=bool(int(g["lora"])),
                                      cb_seed=int(g["codebook_seed"]))
    kw = json.loads(str(g["kwargs"]))
    z, mask = torch.from_numpy(g["z"]), torch.from_numpy(g["mask"])
    got = model.generate(codec, start_tokens=z.cuda(), mask=mask.cuda(), _sampling_steps=6, seed=5,
                         return_signal=False, **kw).cpu()
    agree = (got.numpy() == g["out"]).mean()
    print(f"{os.path.basename(path)}: token agreement with the fp32 reference {agree:.4f}")
    assert agree >= 0.85


def _calibrated_compare(cfg, sd, got_rows, lat_rows, tag, floor_caps=None):
    """got_rows[i] (V, S) from the GPU for latents lat_rows[i] (1, K, T): distance to the bf16 oracle, required to be
    within 1.5x of the oracle's own jitter floor on the same inputs (or, with floor_caps = (max, mean), of the floor
    measured for this model at shorter T: saves the third 25 s oracle forward at T = 3072); decisions exact where the
    fp32 margin is safe."""
    orc_bf16 = vo.OracleVampNet(cfg, sd, "bf16")
    orc_jit = vo.OracleVampNet(cfg, sd, "bf16", jitter=1e-6, jitter_seed=1) if floor_caps is None else None
    orc_32 = vo.OracleVampNet(cfg, sd, "fp32")
    for i, (got, lat) in enumerate(zip(got_rows, lat_rows)):
        t0 = time.time()
        ref = orc_bf16.forward(lat)[0]
        ref32 = orc_32.forward(lat)[0]
        e = (got - ref).abs()
        if orc_jit is not None:
            floor = (orc_jit.forward(lat)[0] - ref).abs()
            fmax, fmean = floor.max().item(), floor.mean().item()
        else:
            fmax, fmean = floor_caps
        print(f"[{tag} row {i}] vs bf16 oracle: max {e.max():.3e} mean {e.mean():.3e}; oracle jitter floor: max "
              f"{fmax:.3e} mean {fmean:.3e}  (oracle forwards: {time.time() - t0:.1f} s)")
        assert e.mean() <= 1.5 * fmean and e.max() <= 1.5 * fmax + 5e-3
        assert_decisions_exact_where_margin_allows(got.t()[None], ref32.t()[None], f"{tag} row {i}")


@pytest.mark.parametrize("B", [8, 32])
def test_full_coarse_forward_at_the_benchmarked_shape(B):
    """BASELINE.json configs[1] / configs[2], coarse stage: d=1280, 20 layers, T=768, B=8 and B=32 (random-init
    weights, random codes with every 3rd frame masked).  The whole batch runs on the GPU; the first and last batch
    rows are compared with B=1 oracle runs; every row must equal its own B=1 GPU run bit for bit."""
    cfg, sd, model, cb, codec = build(FULL_COARSE, seed=0)
    T = 768
    g = torch.Generator().manual_seed(B)
    z = torch.randint(0, 1024, (B, 4, T), generator=g)
    z[:, :, ::3] = 1024
    got = model.forward_codes(z.cuda(), codec)                        # (B, S, V)
    for b in (0, B // 2, B - 1):
        alone = model.forward_codes(z[b:b + 1].cuda(), codec)
        assert torch.equal(alone[0], got[b]), f"row {b} of the batch differs from its B=1 run"
    orc = vo.OracleVampNet(cfg, sd, "fp32")
    rows = (0, B - 1)
    _calibrated_compare(cfg, sd, [got[b].t().cpu() for b in rows], [orc.from_codes(z[b:b + 1], cb) for b in rows],
                        f"coarse B={B} T={T}")


def test_full_c2f_forward_at_the_benchmarked_shape():
    """configs[2], coarse-to-fine stage: 14 codebooks (4 conditioning), 16 layers, d=1280, T=768, B=32."""
    cfg, sd, model, cb, codec = build(FULL_C2F, seed=1)
    B, T = 32, 768
    g = torch.Generator().manual_seed(7)
    z = torch.randint(0, 1024, (B, 14, T), generator=g)
    z[:, 4:, :] = 1024
    z[:, 4:8, ::5] = 7
    got = model.forward_codes(z.cuda(), codec)
    alone = model.forward_codes(z[5:6].cuda(), codec)
    assert torch.equal(alone[0], got[5])
    orc = vo.OracleVampNet(cfg, sd, "fp32")
    _calibrated_compare(cfg, sd, [got[31].t().cpu()], [orc.from_codes(z[31:32], cb)], f"c2f B={B} T={T}")


def test_full_coarse_forward_long_context():
    """configs[4]: T=3072 at full width (B=2 on the GPU, one row against the oracle)."""
    cfg, sd, model, cb, codec = build(FULL_COARSE, seed=0)
    B, T = 2, 3072
    g = torch.Generator().manual_seed(11)
    z = torch.randint(0, 1024, (B, 4, T), generator=g)
    z[:, :, ::4] = 1024
    got = model.forward_codes(z.cuda(), codec)
    orc = vo.OracleVampNet(cfg, sd, "fp32")
    # jitter floor of this model measured at T=768 (3.2-3.6e-2 max / 4.4-4.5e-3 mean) and at T=3072 (3.8e-2 / 4.8e-3)
    _calibrated_compare(cfg, sd, [got[1].t().cpu()], [orc.from_codes(z[1:2], cb)], f"coarse B={B} T={T}",
                        floor_caps=(3.8e-2, 4.8e-3))
