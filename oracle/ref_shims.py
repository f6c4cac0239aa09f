"""TEST INFRASTRUCTURE — not product code.

Import the *unmodified* reference modules from a checkout of the reference
(VAMPNET_REFERENCE_ROOT) through two tiny shims, so that the reference's own code
can be executed as the ground truth when golden vectors are generated
(oracle/gen_golden.py).  The tests only read those stored vectors.

Nothing is copied: the reference files are imported from where they lie.
Nothing outside golden generation needs the checkout (``available()`` says
whether it is present).

Shims (SURVEY.md §8c):
  * ``audiotools``  -> ml.BaseModel = nn.Module subclass with a .device
    property; util.seed; a minimal AudioSignal (reference uses it in
    vampnet/mask.py:4 and transformer.py:670).
  * ``loralib``     -> Linear(in, out, r=...) implemented as W x + scaling * B A x
    (loralib semantics, lora_alpha=1 default => scaling = 1/r) so that LoRA
    folding in the product can be checked against an unfused evaluation.
  * the reference package itself is imported under the name ``vampnet_reference``: a synthetic
    package object whose __path__ points at /root/reference/vampnet, so vampnet/__init__.py (HF hub +
    lac + librosa imports) is skipped and the name ``vampnet`` stays free for this repository's own
    drop-in package (vampnet/ at the repo root).  The reference only uses relative imports inside
    its package, so the name it is imported under does not matter.
"""
from __future__ import annotations

import importlib
import math
import os
import random
import sys
import types

import numpy as np
import torch
import torch.nn as nn

REFERENCE_ROOT = os.environ.get("VAMPNET_REFERENCE_ROOT", "/root/reference")
PKG = "vampnet_reference"


def available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "vampnet", "modules", "transformer.py"))


class _BaseModel(nn.Module):
    INTERN: list = []
    EXTERN: list = []

    @property
    def device(self):
        return next(self.parameters()).device


class _AudioSignal:
    def __init__(self, audio_data, sample_rate):
        self.audio_data = audio_data
        self.sample_rate = sample_rate

    @property
    def samples(self):
        return self.audio_data


class _LoraLinear(nn.Linear):
    """loralib.Linear semantics for inference (PyPI loralib 0.1.x, unpinned in the
    reference's requirements.txt:4): y = x W^T + (x A^T B^T) * (lora_alpha / r)."""

    def __init__(self, in_features, out_features, r=0, lora_alpha=1, bias=True, **kw):
        super().__init__(in_features, out_features, bias=bias)
        self.r = r
        self.scaling = (lora_alpha / r) if r > 0 else 0.0
        if r > 0:
            self.lora_A = nn.Parameter(torch.zeros(r, in_features))
            self.lora_B = nn.Parameter(torch.zeros(out_features, r))
            nn.init.kaiming_uniform_(self.lora_A, a=math.sqrt(5))

    def forward(self, x):
        y = super().forward(x)
        if self.r > 0:
            y = y + (x @ self.lora_A.t() @ self.lora_B.t()) * self.scaling
        return y


def _seed(seed: int):
    random.seed(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)


def install():
    """Install the shims into sys.modules (idempotent)."""
    if PKG in sys.modules:
        return
    if not available():
        raise RuntimeError(f"reference not found under {REFERENCE_ROOT}")
    at = types.ModuleType("audiotools")
    at.ml = types.ModuleType("audiotools.ml")
    at.ml.BaseModel = _BaseModel
    at.util = types.ModuleType("audiotools.util")
    at.util.seed = _seed
    at.AudioSignal = _AudioSignal
    sys.modules["audiotools"] = at
    sys.modules["audiotools.ml"] = at.ml
    sys.modules["audiotools.util"] = at.util

    lora = types.ModuleType("loralib")
    lora.Linear = _LoraLinear
    sys.modules["loralib"] = lora

    pkg = types.ModuleType(PKG)
    pkg.__path__ = [os.path.join(REFERENCE_ROOT, "vampnet")]
    pkg._is_ref_shim = True
    sys.modules[PKG] = pkg
    mods = types.ModuleType(PKG + ".modules")
    mods.__path__ = [os.path.join(REFERENCE_ROOT, "vampnet", "modules")]
    sys.modules[PKG + ".modules"] = mods

    # vampnet/interface.py:12,16 imports the beat tracker (librosa) and the codec package (lac); neither is in this
    # image and neither is touched by the chunking / masking logic that the Interface tests pin, so both are
    # name-only stubs.
    beats = types.ModuleType(PKG + ".beats")
    beats.WaveBeat = type("WaveBeat", (), {})
    sys.modules[PKG + ".beats"] = beats
    for name in ("lac", "lac.model", "lac.model.lac"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m._is_ref_shim = True
            sys.modules[name] = m
    sys.modules["lac.model.lac"].LAC = type("LAC", (), {})
    sys.modules["lac"].model = sys.modules["lac.model"]
    sys.modules["lac.model"].lac = sys.modules["lac.model.lac"]


def uninstall():
    shim_names = ("audiotools", "audiotools.ml", "audiotools.util", "loralib")
    for k in list(sys.modules):
        if k == PKG or k.startswith(PKG + ".") or k in shim_names:
            del sys.modules[k]
        elif k in ("lac", "lac.model", "lac.model.lac") and getattr(sys.modules[k], "_is_ref_shim", False):
            del sys.modules[k]


def load_reference():
    """Return (transformer_module, mask_module, util_module) of the reference."""
    install()
    tr = importlib.import_module(PKG + ".modules.transformer")
    mk = importlib.import_module(PKG + ".mask")
    ut = importlib.import_module(PKG + ".util")
    return tr, mk, ut


def load_reference_interface():
    """The reference's vampnet/interface.py module (Interface with its own chunking / masking code)."""
    install()
    return importlib.import_module(PKG + ".interface")


class StubCodec:
    """The only thing VampNet.generate touches on the codec when
    return_signal=False: codec.quantizer.quantizers[i].codebook.weight
    (reference vampnet/modules/layers.py:145)."""

    def __init__(self, codebooks: torch.Tensor):
        # codebooks: (n_codebooks, 1024, 8)
        qs = []
        for i in range(codebooks.shape[0]):
            q = types.SimpleNamespace()
            q.codebook = types.SimpleNamespace(weight=codebooks[i])
            qs.append(q)
        self.quantizer = types.SimpleNamespace(quantizers=qs)
        self.sample_rate = 44100
        self.hop_length = 768
