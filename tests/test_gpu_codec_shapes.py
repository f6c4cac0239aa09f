"""GPU: the full-width codec (do.CodecConfig(): encoder 64..1024, decoder 1536..96) on 10 s clips, the length the
product is benchmarked at (BASELINE.json configs[3]).

tests/test_gpu_codec.py checks the full widths on 3 frames only, where no layer has more tiles than the B200 has SMs.
Here a 10 s clip gives every persistent CTA many tiles (about 23 per CTA on the decoder's 96-channel layers), so the
skip-row prefetch across tile boundaries, the second TMEM accumulator, the BN = 96 three-chunk epilogue and the
tile -> (batch item, row, column) mapping all run under a comparison.  The batch holds two clips: a 10 s clip
(441 000 samples, padded to 575 frames: not a multiple of 8, so the frame-rate layers end on a ragged tile) and a
7.3 s clip zero-padded to the same length.

Tolerances are those of tests/test_gpu_codec.py (fp32 on both sides, 2e-4 on O(1) activations, codes exact except
near-ties), plus the north-star bound on the decoded waveform: 1e-3 against the fp32 reference for the default
split-bf16 tensor-core path."""
import pytest
import torch

from oracle import dac_oracle as do
from tests.test_gpu_codec import PRECISIONS, build

pytestmark = pytest.mark.gpu

CFG = do.CodecConfig()
SR = 44100
LENGTHS = (10 * SR, 322_000)  # 10 s, and a 7.3 s clip whose last frame is partial


@pytest.fixture(scope="module")
def clips():
    """Seeded audio, the oracle's encoding of the batch and its decoding of the oracle's z; shared by both precisions."""
    g = torch.Generator().manual_seed(10)
    x = torch.zeros(len(LENGTHS), 1, max(LENGTHS))
    for b, n in enumerate(LENGTHS):
        x[b, :, :n] = torch.randn(1, n, generator=g) * 0.3
    xp, n = do.preprocess(x, CFG)
    assert xp.shape[-1] == 575 * CFG.hop_length
    w = do.make_codec_weights(CFG, seed=0)
    ref = do.encode(xp, w, CFG)
    audio_ref = do.decode(ref["z"], w, CFG)["audio"]
    return dict(x=x, xp=xp, ref=ref, audio_ref=audio_ref)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_encode_10s_batch(clips, precision):
    """Codes mismatch below 2 %; z within 2e-4 on frames where every level agrees; level-0 latents (values up to ~3)
    within 5e-4 for "tc" and 5e-5 for "fp32" everywhere (level 0 sees the encoder output itself).
    Measured on a B200 (1000 W): no code differs in either precision; z 1.8e-6 / 1.7e-6; latents 2.9e-4 ("tc": the
    split-bf16 error of the 1024-channel encoder output; 3-frame and small-width clips stay below 2e-4) / 1.2e-5."""
    _, m = build(CFG, precision=precision)
    xg, n = m.preprocess(clips["x"].cuda(), SR)
    assert torch.equal(xg.cpu(), clips["xp"])
    got = m.encode(xg, SR)
    ref = clips["ref"]
    assert got["codes"].shape == ref["codes"].shape == (2, CFG.n_codebooks, 575)
    mism = got["codes"].cpu() != ref["codes"]
    ok = ~mism.any(dim=1)
    ez = (got["z"].cpu() - ref["z"]).abs().permute(0, 2, 1)[ok]
    el = (got["latents"].cpu()[:, :CFG.codebook_dim] - ref["latents"][:, :CFG.codebook_dim]).abs()
    print(f"[{precision}] encode 2 x 575 frames: code mismatch {mism.float().mean().item():.5f} "
          f"({int(mism.sum())} of {mism.numel()}); z on {int(ok.sum())} agreeing frames max {ez.max():.3e}; "
          f"level-0 latents max {el.max():.3e}")
    assert mism.float().mean() < 0.02
    assert ok.float().mean() > 0.5
    assert ez.max() < 2e-4
    assert el.max() < (5e-4 if precision == "tc" else 5e-5)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_decode_10s_batch(clips, precision):
    """The oracle's z decoded by the product: max error <= 1e-3 for "tc" (the north-star bound) and <= 1e-4 for
    "fp32".  Measured on a B200 (1000 W), waveform of mean magnitude 0.53: "tc" max 5.0e-4, mean 5.2e-5; "fp32" max
    2.5e-5, mean 2.7e-6."""
    _, m = build(CFG, precision=precision)
    audio = m.decode(clips["ref"]["z"].cuda())["audio"].cpu()
    want = clips["audio_ref"]
    assert audio.shape == want.shape == (2, 1, 575 * CFG.hop_length)
    err = (audio - want).abs()
    print(f"[{precision}] decode 2 x 575 frames: max err {err.max():.3e} mean err {err.mean():.3e} "
          f"(reference absmean {want.abs().mean():.3e}); per item max {[f'{v:.3e}' for v in err.amax((1, 2))]}")
    assert err.max() <= (1e-3 if precision == "tc" else 1e-4)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_batch_item_equals_its_own_run(clips, precision):
    """Item 1 encoded and decoded alone equals item 1 of the batch bit for bit: which tile (and which CTA) computes an
    element may depend on the batch, its arithmetic may not."""
    _, m = build(CFG, precision=precision)
    xp = clips["xp"].cuda()
    both = m.encode(xp, SR)
    alone = m.encode(xp[1:2].contiguous(), SR)
    for k in ("codes", "z", "latents"):
        assert torch.equal(both[k][1:2], alone[k]), k
    z = clips["ref"]["z"].cuda()
    assert torch.equal(m.decode(z)["audio"][1:2], m.decode(z[1:2].contiguous())["audio"])
