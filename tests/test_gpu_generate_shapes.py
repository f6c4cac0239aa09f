"""GPU: VampNet.generate at the benchmarked shapes (BASELINE.json configs[1] / configs[2]: d=1280, T=768, coarse B=32,
c2f B=8) against the oracle's sampler driven by the same Philox stream.

At T = 768 the classifier GEMM with the fused sampling epilogue (EPI_SAMPLE) runs about 21 tiles per CTA pair on the
coarse model and about 52 on the c2f model, so the TMEM accumulator phase flip, the double-buffered bias copy in shared
memory and long runs of skipped (fully unmasked) warps all run under a comparison.  The Philox counters reach row
t * Cp + cp = 7679 and batch index 31, and the sampled tests take their key from torch's generator the way
generate(seed=None) does, so the high key word is non-zero.

The oracle is teacher-forced with the product's own logits (tests/test_gpu_parity.py::_teacher_forced): those are the
logits the sampling epilogue sees, bit for bit.  What may still differ is rounding between the kernels' exp2 / log and
libm: a categorical draw whose threshold lies on a CDF step, a re-mask cut whose neighbouring confidence is within
rounding, a top-p cumulative mass on top_p.  near_ties() / cut_near_ties() flag exactly those, and every mismatch must
be flagged.  Thresholds were set from the first B200 run; the measured values are printed by each test."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import philox
from oracle import vampnet_oracle as vo
from tests.test_gpu_parity import _teacher_forced, build
from tests.test_gpu_parity_shapes import FULL_C2F, FULL_COARSE

T = 768
DELTA = 1e-6       # relative distance of a draw threshold from a CDF step (or of top_p from a cumulative mass)
CUT_TOL = 1e-5     # distance of the re-mask cut from its neighbour, relative for |cut| > 1
TILE = 128         # vocabulary entries per tile of the two-level draw


# ---------------------------------------------------------------------------------------------- near-tie helpers
def near_ties(logits, u1, u2, temperature, top_p=None, delta=DELTA):
    """Draws of the oracle's two-level inverse CDF (vo.OracleVampNet.sample_from_logits, rng="philox") that rounding
    could flip.  logits (B, S, V) fp32, u1 / u2 (B, S) the Philox uniforms.  Returns (flags (B, S) bool, the oracle's
    token (B, S)).  A draw is flagged when u1 * total lies within delta * total of a step of the tile CDF, when u2 * mass
    lies within delta * mass of a step of the chosen tile's CDF, or (top_p) when a sorted cumulative mass lies within
    delta of top_p."""
    x = torch.as_tensor(logits, dtype=torch.float32)
    B, S, V = x.shape
    flags = np.zeros((B, S), dtype=bool)
    if top_p is not None and top_p < 1.0:
        f, x = top_p_filter(x, top_p, delta)
        flags |= f
    inv_t = np.float32(1.0 / temperature) if temperature > 0 else np.float32(1.0)
    xs = (x.numpy() * inv_t).reshape(B, S, V // TILE, TILE)
    m_k = xs.max(-1)
    m_safe = np.where(np.isfinite(m_k), m_k, np.float32(0))                    # a tile removed entirely by top-p
    cdf_in = np.cumsum(np.exp(xs - m_safe[..., None], dtype=np.float32), axis=-1, dtype=np.float32)
    mass = cdf_in[..., -1] * np.exp(m_k - m_k.max(-1, keepdims=True), dtype=np.float32)
    cdf_t = np.cumsum(mass, axis=-1, dtype=np.float32)
    total = cdf_t[..., -1]
    t1 = u1 * total
    flags |= (np.abs(cdf_t.astype(np.float64) - t1[..., None]).min(-1) <= delta * total)
    hit_t = cdf_t > t1[..., None]
    k = np.where(hit_t.any(-1), hit_t.argmax(-1), m_k.argmax(-1))
    cdf_k = np.take_along_axis(cdf_in, k[..., None, None], axis=2)[:, :, 0, :]
    xs_k = np.take_along_axis(xs, k[..., None, None], axis=2)[:, :, 0, :]
    mass_k = cdf_k[..., -1]
    t2 = u2 * mass_k
    flags |= (np.abs(cdf_k.astype(np.float64) - t2[..., None]).min(-1) <= delta * mass_k)
    hit_v = cdf_k > t2[..., None]
    idx = np.where(hit_v.any(-1), hit_v.argmax(-1), xs_k.argmax(-1))
    return flags, k * TILE + idx


def top_p_filter(x, top_p, delta=DELTA):
    """The oracle's nucleus filter (transformer.py:1001-1016) on (B, S, V) logits: returns (rows whose sorted
    cumulative mass lies within delta of top_p, the filtered logits)."""
    v, si = x.sort(dim=-1, descending=True)
    cum = v.softmax(dim=-1).cumsum(dim=-1)
    flags = ((cum.double() - top_p).abs() <= delta).any(-1).numpy()
    rm = torch.nn.functional.pad(cum > top_p, (1, 0), value=False)[..., :-1]
    return flags, x.masked_fill(rm.scatter(-1, si, rm), -float("inf"))


def cut_near_ties(conf, num_to_mask, tol=CUT_TOL):
    """Rows whose re-mask cut (the num_to_mask-th smallest confidence; positions below it are re-masked) lies within
    tol (relative for |cut| > 1) of the largest confidence below it.  conf (B, S), num_to_mask (B, 1)."""
    srt = torch.as_tensor(conf).double().sort(dim=-1).values
    n = torch.as_tensor(num_to_mask).reshape(-1).long()
    S = srt.shape[-1]
    ok = (n >= 1) & (n < S)
    nc = n.clamp(1, S - 1)[:, None]
    cut = srt.gather(1, nc)[:, 0]
    below = srt.gather(1, nc - 1)[:, 0]
    return (ok & ((cut - below) <= tol * cut.abs().clamp(min=1.0))).numpy()


class _NoLogitsTrace(list):
    """Trace for multi-step oracle runs that only need confidences: drops each step's (B, S, V) logits copy."""
    def append(self, d):
        d.pop("logits", None)
        super().append(d)


def test_near_tie_helpers_on_synthetic_rows():
    """CPU: a threshold placed exactly on a CDF step is flagged at either level, one far from every step is not; the
    same for the re-mask cut and for top_p; and the helper's token is the oracle's."""
    V = 1024
    flat = torch.zeros(1, 4, V)  # e = 1 everywhere: tile CDF 128, 256, ..., 1024; in-tile CDF 1, 2, ..., 128
    u1 = np.array([[0.5, 0.5625, 0.5625, 0.5625]], dtype=np.float32)  # 0.5 * 1024 = 512 is a tile step; 576 is not
    u2 = np.array([[63.5 / 128, 0.5, 63.5 / 128, 63.75 / 128]], dtype=np.float32)  # 64 is an entry step; 63.5 is not
    f, tok = near_ties(flat, u1, u2, 1.0)
    assert f.tolist() == [[True, True, False, False]]
    assert tok[0, 2] == 4 * 128 + 63 and tok[0, 3] == 4 * 128 + 63
    # random rows: the first step after u1 = (exact mass of tiles 0..3) / total is flagged, the mid-point is not
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 3, V, generator=g) * 2
    p = torch.softmax(x.double(), -1)
    step = p[..., :4 * TILE].sum(-1)
    mid = step + 0.5 * p[..., 4 * TILE:5 * TILE].sum(-1)
    half = np.full((2, 3), 0.5, dtype=np.float32)
    f_on, _ = near_ties(x, step.float().numpy(), half, 1.0)
    f_off, tok = near_ties(x, mid.float().numpy(), half, 1.0)
    assert f_on.all() and not f_off.any()
    # the helper draws what the oracle draws (rng="philox", same uniforms)
    orc = vo.OracleVampNet.__new__(vo.OracleVampNet)
    for temp, top_p in ((1.0, None), (0.8, None), (1.0, 0.85)):
        want, _ = orc.sample_from_logits(x.clone(), True, temp, top_p, rng="philox", philox_key=(7, 3), step=2)
        _, tok = near_ties(x, philox.uniform_bs((7, 3), 2, 2, 3, stream=0, word=0),
                           philox.uniform_bs((7, 3), 2, 2, 3, stream=0, word=1), temp, top_p)
        assert np.array_equal(tok, want.numpy()), (temp, top_p)
    # top-p: with equal logits the sorted cumulative mass is k / 1024, so top_p = 0.5 sits on a step
    assert top_p_filter(flat, 0.5)[0].all() and not top_p_filter(flat, 0.5 + 0.5 / V)[0].any()
    assert near_ties(flat, u1, u2, 1.0, top_p=0.5)[0].all()
    # re-mask cut: rows 0 / 1 have the cut 1e-7 / 1e-1 above its neighbour; row 2 re-masks nothing (last step)
    conf = torch.tensor([[-3.0, -2.0, -2.0 + 1e-7, -1.0, float("inf")],
                         [-3.0, -2.0, -1.9, -1.0, float("inf")],
                         [-3.0, -3.0, -3.0, -1.0, float("inf")]])
    assert cut_near_ties(conf, torch.tensor([[2], [2], [0]])).tolist() == [True, False, False]
    assert cut_near_ties(conf * 100, torch.tensor([[2], [2], [0]])).tolist() == [True, False, False]


# ---------------------------------------------------------------------------------------------- GPU fixtures
def _option(name, value):
    """Sets a library option, returns the previous value."""
    from vampnet_b200 import _lib as L
    prev = ctypes.c_int32(0)
    L.check(L.lib().vnb_get_option(name, ctypes.byref(prev)))
    L.check(L.lib().vnb_set_option(name, value))
    return prev.value


def _production_key(seed):
    """The Philox key generate(seed=None) draws after torch.manual_seed(seed) (62 bits, high word non-zero).  An
    explicit seed cannot carry a high word: generate(seed=...) also seeds numpy, which accepts 32 bits only."""
    torch.manual_seed(seed)
    k = int(torch.randint(0, 2 ** 62, (1,)).item())
    assert k >> 32 != 0
    return k


@pytest.fixture(scope="module")
def coarse():
    cfg, sd, model, cb, codec = build(FULL_COARSE, seed=0)
    return cfg, model, cb, codec, vo.OracleVampNet(cfg, sd, "bf16")


@pytest.fixture(scope="module")
def c2f():
    cfg, sd, model, cb, codec = build(FULL_C2F, seed=1)
    return cfg, model, cb, codec, vo.OracleVampNet(cfg, sd, "bf16")


def _codes(cfg, B, seed, every=None, rate=None):
    """Random codes and a mask over the predicted codebooks: every `every`-th frame, or a random `rate` of positions."""
    g = torch.Generator().manual_seed(seed)
    z = torch.randint(0, 1024, (B, cfg.n_codebooks, T), generator=g)
    mask = torch.zeros_like(z)
    ncc = cfg.n_conditioning_codebooks
    if every is not None:
        mask[:, ncc:, ::every] = 1
    else:
        mask[:, ncc:] = (torch.rand(B, cfg.n_codebooks - ncc, T, generator=g) < rate).long()
    return z, mask


# ---------------------------------------------------------------------------------------------- 1. greedy, exact
@pytest.mark.gpu
@pytest.mark.parametrize("stage,B,steps", [("coarse", 32, 12), ("c2f", 8, 4)])
@pytest.mark.parametrize("mask_temperature", [0.0, 10.5])
def test_greedy_multistep_exact(request, stage, B, steps, mask_temperature):
    """Greedy decisions on bit-identical logits cannot differ; only the re-mask cut can, where two confidences are
    within rounding.  Every row with no flagged cut in any step equals the oracle bit for bit, and at least 75 % of
    the rows qualify (measured on a B200: 28/32 coarse rows at mask_temperature 0, every other case all rows; every
    row identical, flagged or not).  Every 3rd frame is masked: deep inside a long all-mask region, positions beyond
    the position bias saturation distance can have identical logits."""
    cfg, model, cb, codec, orc = request.getfixturevalue(stage)
    z, mask = _codes(cfg, B, seed=100 + B, every=3)
    kw = dict(sample_cutoff=-1.0, mask_temperature=mask_temperature)
    trace = _NoLogitsTrace()
    want = orc.generate(cb, z.clone(), mask.clone(), _sampling_steps=steps, rng="philox", philox_key=(77, 0),
                        trace=trace, logits_fn=_teacher_forced(model, codec), **kw)
    got = model.generate(codec, start_tokens=z.cuda(), mask=mask.cuda(), _sampling_steps=steps, seed=77,
                         return_signal=False, **kw).cpu()
    flagged = np.zeros(B, dtype=bool)
    for st in trace:
        flagged |= cut_near_ties(st["conf"], st["num_to_mask"])
    same = np.array([torch.equal(got[b], want[b]) for b in range(B)])
    print(f"[greedy {stage} B={B} steps={steps} mask_temperature={mask_temperature}] rows with a flagged cut "
          f"{int(flagged.sum())}/{B} ({int((flagged & same).sum())} of them identical anyway); rows identical "
          f"{int(same.sum())}/{B}; tokens differing {int((got != want).sum())} of {got.numel()}")
    assert same[~flagged].all(), f"rows {np.nonzero(~flagged & ~same)[0].tolist()} differ without a near-tie"
    assert (~flagged).mean() >= 0.75
    assert not (got == cfg.mask_token).any()
    assert torch.equal(got[mask == 0], z[mask == 0])


# ---------------------------------------------------------------------------------------------- 2./4. one sampled step
@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(temperature=1.0), dict(temperature=0.8), dict(temperature=1.0, top_p=0.85)],
                         ids=["t1.0", "t0.8", "top_p0.85"])
def test_sampled_one_step_exact_up_to_near_ties(coarse, kw):
    """One sampled iteration at coarse B = 32 with a 62-bit key: every mismatching position is a flagged near-tie and
    at most 1e-3 of the draws are flagged (1e-2 under top_p).  Both the fused sampler (epilogue + combine) and the
    materialised one (sample_rows_kernel; the only path under top_p) are held to this rule.  Measured on a B200 over
    32 768 draws: flagged 1.5e-4 (T = 1.0), 2.1e-4 (T = 0.8), 3.5e-3 (top_p); mismatches 0, 0 fused and 0, 1
    materialised, 0 under top_p."""
    cfg, model, cb, codec, orc = coarse
    B, seed = 32, 0x5EED
    key = _production_key(seed)
    pk = (key & 0xFFFFFFFF, key >> 32)
    z, mask = _codes(cfg, B, seed=200, every=3)
    trace = []
    want = orc.generate(cb, z.clone(), mask.clone(), _sampling_steps=1, rng="philox", philox_key=pk, trace=trace,
                        logits_fn=_teacher_forced(model, codec), **kw)
    S = T * cfg.n_predict_codebooks
    flags, tok = near_ties(trace[0]["logits"], philox.uniform_bs(pk, 0, B, S, stream=0, word=0),
                           philox.uniform_bs(pk, 0, B, S, stream=0, word=1), kw["temperature"], kw.get("top_p"))
    ncc = cfg.n_conditioning_codebooks
    drawn = mask[:, ncc:].bool()
    flags = vo.codebook_unflatten(torch.from_numpy(flags), cfg.n_predict_codebooks) & drawn
    assert torch.equal(vo.codebook_unflatten(torch.from_numpy(tok), cfg.n_predict_codebooks)[drawn],
                       want[:, ncc:][drawn])  # the helper draws what the oracle drew
    prev = _option(b"fused_sampler", 1)
    try:
        for fused in (1, 0):
            _option(b"fused_sampler", fused)
            torch.manual_seed(seed)
            got = model.generate(codec, start_tokens=z.cuda(), mask=mask.cuda(), _sampling_steps=1, seed=None,
                                 return_signal=False, **kw).cpu()
            mism = got[:, ncc:] != want[:, ncc:]
            print(f"[sampled 1 step {kw} fused={fused} key=0x{key:016x}] draws {int(drawn.sum())}; mismatches "
                  f"{int(mism.sum())}, flagged near-ties {int(flags.sum())} ({flags.sum().item() / drawn.sum().item():.2e}"
                  f" of the draws), mismatches not flagged {int((mism & ~flags).sum())}")
            assert not (mism & ~flags).any(), f"{int((mism & ~flags).sum())} tokens differ without a near-tie"
            assert torch.equal(got[mask == 0], z[mask == 0])
    finally:
        _option(b"fused_sampler", prev)
    # top-p adds a near-tie wherever one of ~1000 cumulative-mass steps falls within DELTA of top_p
    assert flags.sum() <= (1e-2 if "top_p" in kw else 1e-3) * drawn.sum()


# ---------------------------------------------------------------------------------------------- 3. sampled, many steps
@pytest.mark.gpu
@pytest.mark.parametrize("stage,steps,kw", [("coarse", 12, dict()), ("c2f", 6, dict(sample_cutoff=0.5))])
def test_sampled_multistep_rate(request, stage, steps, kw):
    """Several sampled iterations (c2f: sampled and greedy steps mixed) at B = 8 with about 1 in 16 positions masked, so
    few draws per row and many fully unmasked warps in the epilogue.  One near-tie changes every later input of its
    row, so this is a rate: at least half of the rows bit-identical and below 5 % of the masked positions different
    (measured on a B200: 8/8 rows, no mismatch, in both cases).  A wrong step counter, key word or (b, t, cp) ->
    counter mapping differs at about every drawn position."""
    cfg, model, cb, codec, orc = request.getfixturevalue(stage)
    B, seed = 8, 4242
    z, mask = _codes(cfg, B, seed=300, rate=1 / 16)
    want = orc.generate(cb, z.clone(), mask.clone(), _sampling_steps=steps, rng="philox", philox_key=(seed, 0),
                        logits_fn=_teacher_forced(model, codec), **kw)
    got = model.generate(codec, start_tokens=z.cuda(), mask=mask.cuda(), _sampling_steps=steps, seed=seed,
                         return_signal=False, **kw).cpu()
    same = np.array([torch.equal(got[b], want[b]) for b in range(B)])
    m = mask.bool()
    rate = (got[m] != want[m]).float().mean().item()
    print(f"[sampled {stage} B={B} steps={steps} {kw}] rows identical {int(same.sum())}/{B}; masked positions "
          f"{int(m.sum())}, mismatch {rate:.4f}")
    assert same.mean() >= 0.5
    assert rate < 0.05
    assert not (got == cfg.mask_token).any()
    assert torch.equal(got[mask == 0], z[mask == 0])


# ---------------------------------------------------------------------------------------------- 5. variants
@pytest.mark.gpu
def test_variants_identical_at_benchmarked_shape(coarse):
    """gemm_pair 0 / 1 and CUDA graph off / on give bit-identical tokens for a 12-step sampled coarse B = 32 run: the
    tile schedule and the graph change no element's arithmetic."""
    cfg, model, cb, codec, orc = coarse
    z, mask = _codes(cfg, 32, seed=400, every=3)
    prev_pair = _option(b"gemm_pair", 0)
    prev_graph = model.use_cuda_graph
    outs = {}
    try:
        for pair in (0, 1):
            _option(b"gemm_pair", pair)
            for graph in (False, True):
                model.use_cuda_graph = graph
                outs[pair, graph] = model.generate(codec, start_tokens=z.cuda(), mask=mask.cuda(), _sampling_steps=12,
                                                   seed=31, return_signal=False).cpu()
    finally:
        _option(b"gemm_pair", prev_pair)
        model.use_cuda_graph = prev_graph
    first = outs[0, False]
    assert not (first == cfg.mask_token).any()
    for k, o in outs.items():
        assert torch.equal(o, first), f"{k}: {int((o != first).sum())} of {o.numel()} tokens differ"
