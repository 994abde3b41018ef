"""Shared test helpers: synthetic random-init Falcon models (SURVEY.md section 8d row 2) quantised by the oracle."""
import hashlib
import os
import sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import pyoracle as po  # noqa: E402
import ggllm_cpp_b200.ggcc as ggcc  # noqa: E402

TINY_40B = dict(n_vocab=512, n_embd=256, n_head=4, n_head_kv=2, n_layer=2, falcon_type=40)
TINY_7B = dict(n_vocab=512, n_embd=256, n_head=4, n_head_kv=1, n_layer=2, falcon_type=7)


def synth_model(hp, wtype, seed=1234, embed_type=None, overrides=None):
    """Random-init weights as SURVEY 8d specifies: 2-D weights N(0, 0.02), LN gamma = 1 + 0.1 N(0,1),
    beta = 0.01 N(0,1); every 2-D weight quantised row-wise to `wtype` with the oracle's
    quantize_row_q*_reference restatement (what falcon_quantize does, libfalcon.cpp:3606-3705).
    overrides: {substring of a tensor name: ggml type} for models that mix types; F16 / F32 stay unquantised (rounded to fp16 / as is)."""
    rng = np.random.default_rng(seed)
    o = po.orc()
    tensors = {}
    for name, ne in ggcc.falcon_shapes(hp).items():
        if len(ne) == 1:
            if name.endswith(".weight"):
                v = (1.0 + 0.1 * rng.standard_normal(ne[0])).astype(np.float32)
            else:
                v = (0.01 * rng.standard_normal(ne[0])).astype(np.float32)
            tensors[name] = (po.F32, ne, v)
        else:
            w = (0.02 * rng.standard_normal((ne[1], ne[0]))).astype(np.float32)
            t = embed_type if (embed_type is not None and "word_embeddings" in name) else wtype
            for key, ot in (overrides or {}).items():
                if key in name:
                    t = ot
            tensors[name] = (t, ne, w if t == po.F32 else w.astype(np.float16) if t == po.F16 else o.quantize(t, w))
    return tensors


def digest(a):
    """SHA-256 of an array's bytes: how tests/golden stores reference outputs that are compared bit for bit but too large to keep"""
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


# the sampler-chain cases of tests/test_sampling_gpu.py: (top_k, top_p, temp, repeat_penalty, repeat_last_n)
SAMPLER_CASES = [(40, 0.95, 0.8, 1.1, 64), (1, 1.0, 0.8, 1.0, 0), (200, 0.5, 1.3, 1.3, 16), (40, 1.0, 0.0, 1.2, 64), (7, 0.9, 0.7, 1.0, 0),
                 (1000, 0.999, 2.0, 1.05, 200)]


def codec_random_inputs(t):
    """-> [(scale, x)]: the random rows the codecs of type t are checked on, 8 x 2048 N(0, scale^2) per scale, the first 300 values of
    row 0 zero"""
    rng = np.random.default_rng(t)
    out = []
    for scale in (1.0, 0.02, 30.0):
        x = (rng.standard_normal((8, 2048)) * scale).astype(np.float32)
        x[0, :300] = 0
        out.append((scale, x))
    return out


def sampler_case(top_k, last_n, n_vocab=65024):
    """the seeded inputs of one sampler-chain case: (100-id history, next_logits(window) -> the next float32 logits row)"""
    rng = np.random.default_rng(top_k + last_n)
    history = [int(v) for v in rng.integers(0, n_vocab, size=100)]

    def next_logits(window):
        logits = (rng.standard_normal(n_vocab) * 3.0).astype(np.float32)
        logits[rng.integers(0, n_vocab, size=5)] += 6.0                      # a few dominant candidates, like real logits
        if window:
            logits[window[-1]] += 5.0                                       # make the penalty matter: the last id stays attractive
        return logits
    return history, next_logits


def write_synth(path, hp, wtype, seed=1234):
    tensors = synth_model(hp, wtype, seed)
    ggcc.write_ggcc(path, hp, tensors, ftype=ggcc.FTYPE_OF_TYPE.get(wtype, 0))
    return tensors
