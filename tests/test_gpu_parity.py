"""GPU parity tests proper: the CUDA path (through the C ABI, via the VampNet host mirror) against
the CPU oracle on the same seeded inputs, and against the committed golden fixtures.

Tolerances (stated here, per the north-star):
  * integer outputs (tokens, masks) — bit-exact given identical logits; END-TO-END exactness of greedy decisions
    wherever the fp32 reference's top-2 margin allows it is in tests/test_gpu_parity_shapes.py;
  * logits — the kernels compute with bf16 operands / fp32 accumulation, so the target is the oracle's "bf16" mode
    (same rounding points).  That function is chaotic at the rounding level (tests/test_oracle_conditioning_cpu.py: a
    relative 1e-7 nudge of the activations moves the logits by 1.4e-2 max / 1.8e-3 mean on these tiny models), so the
    assertion is "within 1.5x of the oracle's own jitter floor on the same inputs", plus the absolute caps 2e-2 / 3e-3;
  * the distance to the fp32 reference is bounded separately (0.09 max / 1.2e-2 mean on logits of std ~1); the
    reference's own bf16-autocast GPU path sits 3.2e-2 max / 5.6e-3 mean from its fp32 CPU path (BASELINE.md §2).
"""
import ctypes as C
import glob
import json
import os

import numpy as np
import pytest
import torch

from oracle import vampnet_oracle as vo
from oracle.gen_golden import load

pytestmark = pytest.mark.gpu

TINY_COARSE = dict(n_heads=4, n_layers=2, n_codebooks=4, n_conditioning_codebooks=0, embedding_dim=256)
TINY_C2F = dict(n_heads=4, n_layers=2, n_codebooks=14, n_conditioning_codebooks=4, embedding_dim=256)


class StubCodec:
    def __init__(self, codebooks):
        import types
        self.quantizer = types.SimpleNamespace(
            quantizers=[types.SimpleNamespace(codebook=types.SimpleNamespace(weight=codebooks[i]))
                        for i in range(codebooks.shape[0])])
        self.sample_rate = 44100
        self.hop_length = 768


def build(cfgd, seed=0, lora=False, cb_seed=1):
    from vampnet_b200.modules.transformer import VampNet
    cfg = vo.OracleConfig(**cfgd)
    sd = vo.make_state_dict(cfg, seed=seed, lora=lora)
    model = VampNet(**cfgd)
    res = model.load_state_dict(sd, strict=False)
    assert not res.unexpected_keys, res.unexpected_keys
    assert all("lora" in k for k in res.missing_keys), res.missing_keys
    model = model.to("cuda")
    cb = vo.make_codebooks(cfg.n_codebooks, seed=cb_seed)
    return cfg, sd, model, cb, StubCodec(cb.cuda())


@pytest.mark.parametrize("tag,cfgd,lora", [("coarse", TINY_COARSE, False), ("c2f", TINY_C2F, False),
                                           ("coarse_lora", TINY_COARSE, True)])
def test_forward_vs_oracle_and_golden(golden_dir, tag, cfgd, lora):
    g = load(os.path.join(golden_dir, f"forward_tiny_{tag}.npz"))
    cfg, sd, model, cb, codec = build(cfgd, seed=int(g["weight_seed"]), lora=lora, cb_seed=int(g["codebook_seed"]))
    lat = torch.from_numpy(g["latents"])
    got = model(lat.cuda()).cpu()  # (B, V, S)
    assert got.shape == g["logits"].shape
    ref_bf16 = vo.OracleVampNet(cfg, sd, "bf16").forward(lat)
    floor = (vo.OracleVampNet(cfg, sd, "bf16", jitter=1e-6, jitter_seed=1).forward(lat) - ref_bf16).abs()
    e = (got - ref_bf16).abs()
    print(f"[{tag}] vs oracle-bf16: max {e.max():.3e} mean {e.mean():.3e} (oracle jitter floor: max {floor.max():.3e} "
          f"mean {floor.mean():.3e})")
    assert e.max() < 2e-2 and e.mean() < 3e-3
    assert e.mean() <= 1.5 * floor.mean() and e.max() <= 1.5 * floor.max() + 5e-3
    e32 = (got - torch.from_numpy(g["logits"])).abs()
    print(f"[{tag}] vs reference fp32 golden: max {e32.max():.3e} mean {e32.mean():.3e}")
    assert e32.mean() < 1.2e-2 and e32.max() < 0.09
    # codes entry point == from_codes + forward
    got2 = model.forward_codes(torch.from_numpy(g["codes"]).cuda(), codec).permute(0, 2, 1).cpu()
    assert torch.equal(got, got2)


@pytest.mark.parametrize("tag,cfgd", [("coarse", TINY_COARSE), ("c2f", TINY_C2F)])
@pytest.mark.parametrize("kw", [dict(), dict(temperature=0.7, sample_cutoff=0.5), dict(sample_cutoff=-1.0, mask_temperature=0.0)])
def test_fused_sampler_equals_materialised_sampler(tag, cfgd, kw):
    """vnb_set_option("fused_sampler"): sampling inside the classifier GEMM's epilogue (default) and sampling from the
    materialised logits tensor draw with the same two-level inverse CDF from the same Philox stream, so the tokens are
    the same (they could differ only where a uniform lands within rounding of a CDF step).  T = 150 gives two row tiles
    with a ragged tail; the batch of 3 exercises the (b, t) -> Philox counter mapping."""
    from vampnet_b200 import _lib as L
    import ctypes
    cfg, sd, model, cb, codec = build(cfgd)
    g = torch.Generator().manual_seed(23)
    z = torch.randint(0, 1024, (3, cfg.n_codebooks, 150), generator=g).cuda()
    mask = torch.ones_like(z)
    mask[:, :, ::5] = 0
    prev = ctypes.c_int32(0)
    L.check(L.lib().vnb_get_option(b"fused_sampler", ctypes.byref(prev)))
    outs = []
    try:
        for fused in (1, 0):
            L.check(L.lib().vnb_set_option(b"fused_sampler", fused))
            for graph in (False, True):
                model.use_cuda_graph = graph
                outs.append(model.generate(codec, start_tokens=z, mask=mask, _sampling_steps=5, seed=17,
                                           return_signal=False, **kw).cpu())
    finally:
        L.check(L.lib().vnb_set_option(b"fused_sampler", prev.value))
    assert not (outs[0] == cfg.mask_token).any()
    for o in outs[1:]:
        assert torch.equal(outs[0], o), f"{(outs[0] != o).sum().item()} of {o.numel()} tokens differ"


def _teacher_forced(model, codec):
    """logits_fn for the oracle loop: the product's own forward on the oracle's current state, so both
    samplers see bit-identical logits."""
    def fn(i, z_masked):
        return model.forward_codes(z_masked.cuda(), codec).permute(0, 2, 1).cpu()
    return fn


@pytest.mark.parametrize("tag,cfgd", [("coarse", TINY_COARSE), ("c2f", TINY_C2F)])
@pytest.mark.parametrize("steps", [1, 6])
@pytest.mark.parametrize("graph", [False, True])
def test_generate_greedy_bit_exact_given_logits(tag, cfgd, steps, graph):
    cfg, sd, model, cb, codec = build(cfgd)
    model.use_cuda_graph = graph
    orc = vo.OracleVampNet(cfg, sd, "bf16")
    g = torch.Generator().manual_seed(11)
    z = torch.randint(0, 1024, (3, cfg.n_codebooks, 40), generator=g)
    mask = torch.ones_like(z)
    mask[:, :, ::7] = 0
    mask[:, :cfg.n_conditioning_codebooks, :] = 0
    kw = dict(sample_cutoff=-1.0, mask_temperature=0.0)
    want = orc.generate(cb, z.clone(), mask.clone(), _sampling_steps=steps, rng="philox", philox_key=(5, 0),
                        logits_fn=_teacher_forced(model, codec), **kw)
    for _ in range(2):  # second call replays the captured graph
        got = model.generate(codec, start_tokens=z.cuda(), mask=mask.cuda(), _sampling_steps=steps, seed=5,
                             return_signal=False, **kw).cpu()
        assert torch.equal(got, want), f"{(got != want).sum().item()} of {got.numel()} tokens differ"
    assert not (got == cfg.mask_token).any()
    assert torch.equal(got[mask == 0], z[mask == 0])


@pytest.mark.parametrize("tag,cfgd", [("coarse", TINY_COARSE), ("c2f", TINY_C2F)])
@pytest.mark.parametrize("kw", [dict(), dict(temperature=0.8), dict(sample_cutoff=0.5, mask_temperature=3.0),
                                dict(temperature=0.9, top_p=0.85), dict(top_p=0.5, sample_cutoff=-1.0, mask_temperature=0.0)])
def test_generate_sampled_matches_oracle_with_shared_noise(tag, cfgd, kw):
    """Sampling parity under the shared Philox stream: identical tokens except where the oracle's own
    decision margin is a numerical near-tie (libm vs CUDA logf/expf differ by ulps)."""
    cfg, sd, model, cb, codec = build(cfgd)
    orc = vo.OracleVampNet(cfg, sd, "bf16")
    g = torch.Generator().manual_seed(12)
    z = torch.randint(0, 1024, (2, cfg.n_codebooks, 33), generator=g)
    mask = torch.ones_like(z)
    mask[:, :, ::5] = 0
    mask[:, :cfg.n_conditioning_codebooks, :] = 0
    seed = 1234567
    want = orc.generate(cb, z.clone(), mask.clone(), _sampling_steps=6, rng="philox", philox_key=(seed, 0),
                        logits_fn=_teacher_forced(model, codec), **kw)
    got = model.generate(codec, start_tokens=z.cuda(), mask=mask.cuda(), _sampling_steps=6, seed=seed,
                         return_signal=False, **kw).cpu()
    diff = (got != want).float().mean().item()
    print(f"[{tag} {kw}] sampled-token mismatch fraction {diff:.5f}")
    assert diff <= 0.002
    assert torch.equal(got[mask == 0], z[mask == 0])


def test_sample_step_unit_vs_oracle(golden_dir):
    """vnb_sample_step on the golden logits of tests/golden/sampler_greedy.npz (reference outputs)."""
    from vampnet_b200 import _lib as L
    g = np.load(os.path.join(golden_dir, "sampler_greedy.npz"))
    logits = torch.from_numpy(g["logits"]).cuda().contiguous()
    B, S, V = logits.shape
    zflat = torch.full((B, S), 1024, dtype=torch.int32, device="cuda")
    tokens = torch.empty((B, S), dtype=torch.int32, device="cuda")
    conf = torch.empty((B, S), dtype=torch.float32, device="cuda")
    n0 = torch.tensor([17], dtype=torch.int32, device="cuda")
    L.check(L.lib().vnb_sample_step(L.ptr(logits), L.ptr(zflat), L.ptr(tokens), L.ptr(conf), L.ptr(n0), B, S, V, 1024,
                                    0, 0, 0, 1.0, 1.0, 0.0, 1, 2, L.stream_ptr()))
    torch.cuda.synchronize()
    assert np.array_equal(tokens.cpu().numpy(), g["tok"])
    np.testing.assert_allclose(conf.cpu().numpy(), np.log(g["p"]), rtol=0, atol=2e-5)
    # gamma=1, n0=17, not last: 17 tokens re-masked per row (cut = 17th smallest confidence)
    assert ((zflat == 1024).sum(-1) == 17).all()
    srt = np.sort(np.log(g["p"]), axis=-1)
    want = np.log(g["p"]) < srt[:, 17:18]
    assert (want != (zflat.cpu().numpy() == 1024)).sum() <= 2  # ties at the cut only


def test_full_size_forward_cfg1(golden_dir):
    """BASELINE.json configs[0] shape (random-init coarse, d=1280, 20 layers, T=100, B=1) against the
    reference's fp32 CPU logits."""
    g = np.load(os.path.join(golden_dir, "forward_full_coarse_T100.npz"))
    cfgd = json.loads(str(g["cfg"]))
    cfg, sd, model, cb, codec = build(cfgd, seed=int(g["weight_seed"]))
    lat = torch.randn(1, 32, 100, generator=torch.Generator().manual_seed(int(g["latents_seed"])))
    got = model(lat.cuda()).cpu()
    e = (got[:, :, ::16] - torch.from_numpy(g["logits_sub"])).abs()
    agree = (got.argmax(1).numpy() == g["argmax"]).mean()
    print(f"full coarse T=100: vs fp32 reference max {e.max():.3e} mean {e.mean():.3e}; argmax agreement {agree:.4f}")
    assert e.mean() < 1.2e-2 and e.max() < 0.09 and agree > 0.95


def test_cpu_model_raises():
    from vampnet_b200.modules.transformer import VampNet
    m = VampNet(**TINY_COARSE)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 32, 8))


def test_workspace_eviction_many_shapes():
    """More distinct (B, T) shapes than the library keeps workspaces for: results stay correct after eviction."""
    cfg, sd, model, cb, codec = build(TINY_COARSE)
    g = torch.Generator().manual_seed(5)
    first = None
    for T in (16, 24, 32, 40, 48, 56, 64, 72, 16):
        z = torch.randint(0, 1024, (1, 4, T), generator=torch.Generator().manual_seed(T)).cuda()
        out = model.generate(codec, start_tokens=z, _sampling_steps=2, seed=3, return_signal=False,
                             sample_cutoff=-1.0, mask_temperature=0.0)
        assert out.shape == z.shape and not (out == 1024).any()
        if T == 16:
            if first is None:
                first = out.clone()
            else:
                assert torch.equal(first, out)  # same answer before and after its workspace was evicted


def test_hot_swap_keeps_handle_and_graphs():
    """f-4: load_state_dict on a LIVE model rewrites the packed device buffers in place — the handle, workspaces and
    captured generate graphs survive (no new capture) and the next generate equals a freshly built model's."""
    from vampnet_b200 import _lib as L
    cfg, sd_a, model, cb, codec = build(TINY_COARSE, seed=0, lora=False)
    _, sd_b, fresh_b, _, _ = build(TINY_COARSE, seed=7, lora=True)
    z = torch.randint(0, 1024, (2, 4, 40), generator=torch.Generator().manual_seed(2)).cuda()
    kw = dict(start_tokens=z, _sampling_steps=3, seed=5, return_signal=False, sample_cutoff=-1.0, mask_temperature=0.0)
    out_a = model.generate(codec, **kw)
    want_b = fresh_b.generate(codec, **kw)
    assert not torch.equal(out_a, want_b)
    handle, ptrs = model._handle.value, {k: v.data_ptr() for k, v in model._packed.items()}
    captures = L.lib().vnb_graph_capture_count()
    model.load_state_dict(sd_b, strict=False)
    assert model._handle.value == handle and ptrs == {k: v.data_ptr() for k, v in model._packed.items()}
    assert torch.equal(model.generate(codec, **kw), want_b)
    assert L.lib().vnb_graph_capture_count() == captures  # replayed the graph captured for model A
    # and back again, dropping the adapter: a plain checkpoint must not inherit lora_B (swap_checkpoint semantics)
    import os
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "a.pth")
        torch.save({"state_dict": sd_a, "metadata": {"kwargs": dict(TINY_COARSE)}}, path)
        assert model.swap_checkpoint(path) is True
    assert torch.equal(model.generate(codec, **kw), out_a)
    assert model._handle.value == handle and L.lib().vnb_graph_capture_count() == captures


def test_sampler_distribution_chi_square():
    """RNG parity with torch.multinomial is distributional by construction (DESIGN.md §2): with the same logits in
    40 000 positions the empirical token histogram of the CUDA sampler must match softmax(logits / T)."""
    from vampnet_b200 import _lib as L
    g = torch.Generator().manual_seed(0)
    V, S, T = 1024, 40000, 0.7
    row = torch.full((V,), -30.0)
    support = torch.randperm(V, generator=g)[:40]
    row[support] = torch.randn(40, generator=g) * 1.5
    logits = row[None, None, :].expand(1, S, V).contiguous().cuda()
    zflat = torch.full((1, S), 1024, dtype=torch.int32, device="cuda")
    tokens = torch.empty((1, S), dtype=torch.int32, device="cuda")
    conf = torch.empty((1, S), dtype=torch.float32, device="cuda")
    n0 = torch.tensor([S], dtype=torch.int32, device="cuda")
    L.check(L.lib().vnb_sample_step(L.ptr(logits), L.ptr(zflat), L.ptr(tokens), L.ptr(conf), L.ptr(n0), 1, S, V, 1024,
                                    0, 1, 1, T, 1.0, 0.0, 12345, 678, L.stream_ptr()))
    torch.cuda.synchronize()
    p = torch.softmax(row / T, 0).double()
    counts = torch.bincount(tokens.cpu().flatten().long(), minlength=V).double()
    assert counts[p < 1e-9].sum() == 0  # nothing outside the support
    keep = p * S >= 5
    chi2 = (((counts - p * S) ** 2) / (p * S))[keep].sum().item()
    dof = int(keep.sum()) - 1
    print(f"chi2 = {chi2:.1f} with {dof} dof")
    assert chi2 < dof + 5 * (2 * dof) ** 0.5  # ~5 sigma
    # the reported probability is softmax(logits / T)[token]
    got_p = torch.exp(conf.cpu().flatten().double())
    assert torch.allclose(got_p, p[tokens.cpu().flatten().long()], rtol=1e-4, atol=1e-9)


@pytest.mark.parametrize("case", ["default_mask", "mask_2d", "nothing_masked", "everything_masked", "tiny_T", "one_step"])
def test_generate_edge_cases_vs_oracle(case):
    """Edge cases of VampNet.generate (reference transformer.py:749-753, 766, 906-913): default mask, 2-D mask,
    N0 == 0, fully masked input, sequences shorter than any tile, a single sampling step."""
    cfgd = TINY_C2F if case in ("default_mask", "mask_2d") else TINY_COARSE
    cfg, sd, model, cb, codec = build(cfgd)
    orc = vo.OracleVampNet(cfg, sd, "bf16")
    g = torch.Generator().manual_seed(21)
    B, T, steps = 2, 29, 4
    if case == "tiny_T":
        T = 3
    if case == "one_step":
        steps = 1
    z = torch.randint(0, 1024, (B, cfg.n_codebooks, T), generator=g)
    if case == "default_mask":
        mask = None
    elif case == "mask_2d":
        mask = torch.ones(B, T, dtype=torch.long)
        mask[:, ::4] = 0
    elif case == "nothing_masked":
        mask = torch.zeros_like(z)
    elif case == "everything_masked":
        mask = torch.ones_like(z)
    else:
        mask = torch.ones_like(z)
        mask[:, :, ::3] = 0
    kw = dict(sample_cutoff=-1.0, mask_temperature=0.0)
    want = orc.generate(cb, z.clone(), None if mask is None else mask.clone(), _sampling_steps=steps, rng="philox",
                        philox_key=(9, 0), logits_fn=_teacher_forced(model, codec), **kw)
    got = model.generate(codec, start_tokens=z.cuda(), mask=None if mask is None else mask.cuda(), _sampling_steps=steps,
                         seed=9, return_signal=False, **kw).cpu()
    assert torch.equal(got, want)
    if case == "nothing_masked":
        assert torch.equal(got, z)
    assert not (got == cfg.mask_token).any()


def test_long_context_forward_T3072():
    """BASELINE.json configs[4] sequence length (T = 3072) on a narrow model: attention tiling, the constant-bias
    fast path far from the diagonal and the Toeplitz lookups near it, against the bf16-operand oracle."""
    cfgd = dict(n_heads=4, n_layers=1, n_codebooks=4, n_conditioning_codebooks=0, embedding_dim=256)
    cfg, sd, model, cb, codec = build(cfgd)
    z = torch.randint(0, 1025, (1, 4, 3072), generator=torch.Generator().manual_seed(4))
    got = model.forward_codes(z.cuda(), codec).cpu()  # (B, S, V)
    orc = vo.OracleVampNet(cfg, sd, "bf16")
    ref = orc.forward(orc.from_codes(z, cb)).permute(0, 2, 1)
    e = (got - ref).abs()
    print(f"T=3072: max {e.max():.3e} mean {e.mean():.3e}")
    assert e.max() < 2e-2 and e.mean() < 3e-3


def test_return_activations_matches_oracle():
    """VampNet.forward(return_activations=True) (reference transformer.py:617-639, 443-461; used by
    scripts/utils/gtzan_embeddings.py:123): logits unchanged, activations = the fp32 residual stream after every layer,
    the last one equal to the hidden-state tap, each within bf16-operand distance of the oracle's."""
    cfg, sd, model, cb, codec = build(TINY_COARSE)
    g = torch.Generator().manual_seed(2)
    z = torch.randint(0, 1025, (2, cfg.n_codebooks, 50), generator=g)
    orc = vo.OracleVampNet(cfg, sd, "bf16")
    lat = orc.from_codes(z, cb)
    plain = model(lat.cuda()).clone()
    logits, acts = model(lat.cuda(), return_activations=True)
    assert torch.equal(logits, plain)
    assert acts.shape == (cfg.n_layers, 2, 50, cfg.embedding_dim) and acts.dtype == torch.float32
    assert torch.equal(acts[-1], model.hidden_state(2, 50))
    _, want = orc.forward(lat, return_activations=True)
    for layer in range(cfg.n_layers):
        e = (acts[layer].cpu() - want[layer]).abs()
        scale = want[layer].abs().mean().item()
        assert e.max() < 0.05 * max(scale, 1.0) and e.mean() < 5e-3 * max(scale, 1.0), (layer, e.max().item(), scale)
    assert not torch.equal(acts[0], acts[1])


def test_broadcastable_mask_and_flash_checkpoint_rejected():
    """generate() accepts a (1, C, T) mask against B > 1 start tokens like the reference's masked_fill (:762); a
    flash_attn=True checkpoint (FlashMHA tensor names) is refused instead of silently leaving random projections."""
    cfg, sd, model, cb, codec = build(TINY_COARSE)
    g = torch.Generator().manual_seed(4)
    z = torch.randint(0, 1024, (3, cfg.n_codebooks, 30), generator=g).cuda()
    mask = torch.ones(1, cfg.n_codebooks, 30, dtype=torch.long).cuda()
    mask[:, :, ::3] = 0
    kw = dict(_sampling_steps=3, seed=2, return_signal=False, sample_cutoff=-1.0, mask_temperature=0.0)
    a = model.generate(codec, start_tokens=z, mask=mask, **kw)
    b = model.generate(codec, start_tokens=z, mask=mask.expand(3, -1, -1).contiguous(), **kw)
    assert torch.equal(a, b)
    bad = dict(sd)
    bad["transformer.layers.0.self_attn.Wqkv.weight"] = torch.zeros(3 * cfg.embedding_dim, cfg.embedding_dim)
    with pytest.raises(RuntimeError, match="FlashMHA"):
        model.load_state_dict(bad, strict=False)


def test_embedding_projection_is_fp32_grade():
    """CodebookEmbedding.from_codes + out_proj (reference layers.py:134-162) runs as a split-bf16 tensor-core
    contraction; with the transformer stack switched off (zero layers cannot be built, so: compare the residual stream
    tap of a model whose layers contribute exactly zero) it must match the fp32 einsum to ~1e-5 relative."""
    cfg, sd, model, cb, codec = build(TINY_C2F, seed=4)
    sd = dict(sd)
    for k in list(sd):  # zero every projection that feeds the residual stream: x stays the embedding
        if k.endswith("self_attn.fc.weight") or k.endswith("feed_forward.w_2.weight"):
            sd[k] = torch.zeros_like(sd[k])
    model.load_state_dict(sd, strict=False)
    g = torch.Generator().manual_seed(8)
    z = torch.randint(0, 1025, (2, cfg.n_codebooks, 37), generator=g)
    model.forward_codes(z.cuda(), codec)
    x = model.hidden_state(2, 37).cpu()
    orc = vo.OracleVampNet(cfg, sd, "fp32")
    lat = orc.from_codes(z, cb)
    want = torch.einsum("bkt,nk->btn", lat, orc.emb_w) + orc.emb_b
    err = (x - want).abs().max().item()
    print(f"embedding projection: max err {err:.2e} on values of magnitude {want.abs().max():.2f}")
    assert err < 3e-5 * max(1.0, want.abs().max().item())
    # the latents entry point shares the contraction: bit-identical
    model(lat.cuda())
    assert torch.equal(model.hidden_state(2, 37).cpu(), x)
