"""Shared helpers for the parity tests."""
import hashlib
import json
import os
import tempfile

import numpy as np

from moonshine_b200.arch import ARCHS
from moonshine_b200.weights import pack_msw, synth_audio, synth_tokenizer_bin, synth_weights
from oracle.moonshine_oracle import Dims, Oracle

GOLD = os.path.join(os.path.dirname(__file__), "golden")
_cache = {}


def weights_for(arch, seed=0, init="scaled"):
    key = (arch, seed, init)
    if key not in _cache:
        _cache[key] = synth_weights(arch, seed, init)
    return _cache[key]


def oracle_for(arch, seed=0, init="scaled", **kw):
    return Oracle(Dims.from_product(ARCHS[arch]), weights_for(arch, seed, init), **kw)


def memory_files(arch, seed=0, init="scaled", tokenizer=None):
    d = ARCHS[arch]
    return {
        "model.msw": pack_msw(arch, weights_for(arch, seed, init)),
        "tokenizer.bin": tokenizer if tokenizer is not None else synth_tokenizer_bin(d.vocab),
    }


def beckett():
    return np.load(os.path.join(GOLD, "beckett_pcm16.npy")).astype(np.float32) / np.float32(32768.0)


def reference_golden(name):
    """Outputs of the original project's own code recorded by golden/make_golden_reference.py."""
    with open(os.path.join(GOLD, name), encoding="utf-8") as f:
        return json.load(f)


def digest(data):
    """SHA-256 of the exact bytes (of a numpy array's buffer, or of a bytes object): how bit-exact outputs too large
    to store are kept in the golden files."""
    return hashlib.sha256(data.tobytes() if isinstance(data, np.ndarray) else bytes(data)).hexdigest()


def rel_err(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max() / max(np.abs(b).max(), 1e-30))
