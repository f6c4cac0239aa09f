"""CPU: the repository's ``vampnet`` package is a drop-in for the reference's import surface (SURVEY.md §8b).

The reference's OWN import lines are executed (its app.py:16-17, verbatim), then the hello.py:1-36 call sequence up
to the first device computation runs against a synthetic model cache written in the reference's on-disk layout, codec checkpoint in the lac /
descript-audio-codec key layout included.  Everything that computes needs the GPU and is covered by
tests/test_gpu_dropin.py; here a CPU-resident Interface must refuse to compute (there is no CPU fallback)."""
import sys

import pytest
import torch

APP_IMPORTS = ["from vampnet.interface import Interface, signal_concat", "from vampnet import mask as pmask"]  # app.py:16-17


@pytest.fixture()
def cache(tmp_path, monkeypatch):
    from tests.dropin_cache import write_cache
    root = tmp_path / "models" / "vampnet"
    codec, sds = write_cache(root)
    monkeypatch.setenv("VAMPNET_MODELS_DIR", str(root))
    for k in [k for k in sys.modules if k == "vampnet" or k.startswith("vampnet.")]:
        del sys.modules[k]   # import the package fresh (another test may have imported the reference under a shim)
    return root, codec, sds


def test_reference_import_lines_resolve_to_this_repository(cache):
    ns = {}
    for line in APP_IMPORTS:
        exec(line, ns)
    import vampnet_b200.interface
    import vampnet_b200.mask
    assert ns["Interface"] is vampnet_b200.interface.Interface
    assert ns["signal_concat"] is vampnet_b200.interface.signal_concat
    assert ns["pmask"].linear_random is vampnet_b200.mask.linear_random
    assert ns["pmask"].apply_mask is vampnet_b200.mask.apply_mask
    # the other import lines reference scripts use (train.py:20-23, hello.py:2, experiment.py:11-12)
    exec("import vampnet\nfrom vampnet.modules.transformer import VampNet\n"
         "from vampnet.util import codebook_unflatten, codebook_flatten, scalar_to_batch_tensor", ns)
    assert ns["vampnet"].interface.Interface is ns["Interface"] and ns["vampnet"].VampNet is ns["VampNet"]
    t = torch.arange(2 * 3 * 5).view(2, 3, 5)
    flat = ns["codebook_flatten"](t)
    assert flat.shape == (2, 15) and flat[0, 1] == t[0, 1, 0] and torch.equal(ns["codebook_unflatten"](flat, 3), t)
    assert torch.equal(ns["scalar_to_batch_tensor"](0.5, 3), torch.tensor(0.5).repeat(3))


def test_hello_sequence_up_to_the_device(cache):
    root, codec_ref, sds = cache
    import vampnet
    # hello.py:6-23
    interface = vampnet.interface.Interface.default()
    choices = interface.available_models()
    assert choices == ["opera", "default"]                       # "incomplete" has no c2f.pth
    assert vampnet.list_finetuned() == ["opera"]
    assert vampnet.download_default() == (str(root / "coarse.pth"), str(root / "c2f.pth"))
    assert vampnet.download_codec() == str(root / "codec.pth")
    interface.load_finetuned("default")
    # the checkpoints were ingested: reference key names (LoRA absent) and the lac-layout codec
    from tests.dropin_cache import C2F, COARSE, CODEC
    assert (interface.coarse.n_codebooks, interface.c2f.n_codebooks, interface.c2f.n_conditioning_codebooks) == (4, 14, 4)
    assert interface.codec.hop_length == CODEC.hop_length == 768 and interface.codec.sample_rate == 44100
    sd = interface.coarse.state_dict()
    assert all(torch.equal(sd[k], v) for k, v in sds["coarse"].items())
    want = codec_ref.state_dict()["quantizer.quantizers.3.codebook.weight"]
    assert torch.equal(interface.codec.quantizer.quantizers[3].codebook.weight, want)
    # fine-tuned swap and back (interface.py:134-174)
    interface.load_finetuned("opera")
    k = "transformer.layers.0.feed_forward.w_1.lora_B"
    assert torch.equal(interface.coarse.state_dict()[k], sds["lora_coarse"][k])
    interface.load_finetuned("default")
    # hello.py:27-36 needs audio -> tokens on the device; the mask algebra itself is device-agnostic
    codes = torch.randint(0, 1024, (1, 14, interface.s2t(2.0)))
    mask = interface.build_mask(codes, None, periodic_prompt=13, upper_codebook_mask=3)
    assert mask.shape == codes.shape and mask[:, 3:].all() and set(mask.unique().tolist()) <= {0, 1}
    assert mask[:, :3].sum() < mask[:, :3].numel()               # the periodic prompt keeps frames in the coarse books
    # no CPU fallback: computing on a CPU-resident Interface raises instead of running torch code
    with pytest.raises(RuntimeError, match="CUDA"):
        interface.vamp(codes, mask, _sampling_steps=2)
    from vampnet_b200.audio import AudioSignal
    with pytest.raises(RuntimeError, match="CUDA"):
        interface.encode(AudioSignal(torch.zeros(1, 1, 44100), 44100))


def test_missing_cache_entry_raises_instead_of_downloading(cache, monkeypatch):
    root, _, _ = cache
    import vampnet
    monkeypatch.setenv("VAMPNET_MODELS_DIR", str(root / "nowhere"))
    with pytest.raises(RuntimeError, match="local model cache"):
        vampnet.interface.Interface.default()
    with pytest.raises(RuntimeError, match="local model cache"):
        vampnet.download_finetuned("opera")
