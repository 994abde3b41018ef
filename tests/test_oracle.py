"""CPU tests (-m "not gpu"): the oracle restatement (oracle/ggml_oracle.c) pinned against
 (1) the committed golden vectors generated from the UNMODIFIED reference (tests/golden, made by tests/golden/make_golden.py):
     bit-exact codecs on fixed and on random rows, eval within fp tolerance,
 (2) the acceptance thresholds of the reference's own codec test (tests/test-quantize-fns.cpp:18-22, 129-152).
"""
import json
import os
import numpy as np
import pytest
import pyoracle as po
from helpers import TINY_40B, TINY_7B, synth_model, digest, codec_random_inputs

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(GOLD, "codecs.npz"))


@pytest.mark.parametrize("t", po.WEIGHT_TYPES)
def test_codecs_match_reference_golden_vectors(orc, gold, t):
    n = po.TYPE_NAMES[t]
    x, a = gold["x"], gold["a"]
    assert np.array_equal(orc.quantize(t, x), gold[n + "_q"])                                   # bit-exact blocks
    assert np.array_equal(orc.dequantize(t, gold[n + "_q"], 1024).view(np.uint32), gold[n + "_deq"].view(np.uint32))
    aq = orc.quantize_act(t, a)
    blk = po.BLOCK_BYTES[po.VEC_DOT_TYPE[t]]
    if po.VEC_DOT_TYPE[t] == po.Q8_K:
        assert np.array_equal(aq.reshape(4, -1, blk)[:, :, :292], gold[n + "_aq"].reshape(4, -1, blk)[:, :, :292])
    else:
        assert np.array_equal(aq, gold[n + "_aq"])
    dots = np.array([orc.vec_dot(t, 1024, gold[n + "_q"][i], gold[n + "_aq"][i]) for i in range(4)], np.float32)
    # integer block dots are exact; scalar vs AVX2 fp32 summation order: 1e-5 relative to sum |w x|
    wd, ad = orc.dequantize(t, gold[n + "_q"], 1024), a
    assert np.all(np.abs(dots - gold[n + "_dot"]) <= 1e-5 * np.sum(np.abs(wd * ad), axis=1))


@pytest.mark.parametrize("t", po.WEIGHT_TYPES)
def test_reference_acceptance_thresholds(orc, t):
    """tests/test-quantize-fns.cpp: round-trip RMSE/n < 0.002 (Q2_K 0.0075, Q3_K 0.0040), |vec_dot - fp32 dot|/n < 0.02"""
    x = po.synth_vector(4096)
    y = po.synth_vector(4096, offset=1.0)
    q = orc.quantize(t, x)
    d = orc.dequantize(t, q, 4096)
    rmse = np.sqrt(np.sum((x.astype(np.float64) - d) ** 2)) / 4096
    assert rmse < {po.Q2_K: 0.0075, po.Q3_K: 0.0040}.get(t, 0.002)
    dot = orc.vec_dot(t, 4096, q, orc.quantize_act(t, y))
    assert abs(dot - float(np.dot(x.astype(np.float64), y))) / 4096 < 0.02


def test_fp16_conversion_all_values(orc):
    h = np.arange(65536, dtype=np.uint16)
    f = h.view(np.float16).astype(np.float32)
    ok = ~np.isnan(f)
    mine = np.array([orc.L.orc_f16_to_f32(int(v)) for v in h[::7]], np.float32)
    assert np.array_equal(mine[~np.isnan(mine)].view(np.uint32), f[::7][~np.isnan(f[::7])].view(np.uint32))
    rng = np.random.default_rng(0)
    v = np.concatenate([rng.standard_normal(20000).astype(np.float32) * s for s in (1e-8, 1e-5, 1e-3, 1, 100, 7e4)] + [f[ok]])
    back = np.array([orc.L.orc_f32_to_f16(float(x)) for x in v], np.uint16)
    assert np.array_equal(back, v.astype(np.float16).view(np.uint16))          # numpy rounds to nearest even like F16C


def test_ops_against_numpy(orc):
    rng = np.random.default_rng(1)
    x = rng.standard_normal((3, 512)).astype(np.float32) * 4
    n = orc.norm(x)
    ref = (x - x.mean(1, keepdims=True)) / np.sqrt(x.var(1, keepdims=True) + 1e-5)
    assert np.allclose(n, ref, atol=1e-5)
    g = orc.gelu(x)
    gref = 0.5 * x * (1 + np.tanh(0.7978845608 * x * (1 + 0.044715 * x * x)))
    assert np.allclose(g, gref, rtol=2e-3, atol=1e-3)                            # fp16 LUT
    s = orc.soft_max(x)
    e = np.exp(x - x.max(1, keepdims=True))
    assert np.allclose(s, e / e.sum(1, keepdims=True), rtol=4e-3, atol=1e-6)     # fp16 LUT on (x - max)
    assert np.allclose(s.sum(1), 1, atol=1e-5)
    r = orc.rope_neox(x.reshape(3, 8, 64), n_past=5, n_ctx_rope=64)
    ts = 10000.0 ** (-2.0 / 64)
    for t in range(3):
        th = (5 + t) * ts ** np.arange(32)
        v = x.reshape(3, 8, 64)[t]
        assert np.allclose(r[t][:, :32], v[:, :32] * np.cos(th) - v[:, 32:] * np.sin(th), atol=2e-5)
        assert np.allclose(r[t][:, 32:], v[:, :32] * np.sin(th) + v[:, 32:] * np.cos(th), atol=2e-5)
    assert abs(orc.theta_scale(64, 8192) - (7.0 ** (64 / 62.0) * 10000.0) ** (-2.0 / 64)) < 1e-6


@pytest.mark.parametrize("name", ["tiny40b_q4_K", "tiny7b_q4_0"])
def test_falcon_eval_matches_reference_golden_logits(name):
    g = np.load(os.path.join(GOLD, name + ".npz"))
    hp = {k: int(g["hp_" + k]) for k in ("n_vocab", "n_embd", "n_head", "n_head_kv", "n_layer", "falcon_type")}
    tensors = synth_model(hp, int(g["wtype"]), seed=int(g["seed"]))
    o = po.OrcFalcon(hp, tensors, n_ctx=int(g["n_ctx"]))
    scale = np.abs(g["prompt_logits"]).max()
    got = o.eval(g["prompt"], 0, all_logits=True)
    assert np.abs(got - g["prompt_logits"]).max() <= 2e-2 * scale and np.median(np.abs(got - g["prompt_logits"])) <= 2e-5 * scale
    for i, tok in enumerate(g["decode_tokens"]):
        got = o.eval(np.array([tok], np.int32), len(g["prompt"]) + i)
        d = np.abs(got - g["decode_logits"][i:i + 1])
        assert d.max() <= 2e-2 * scale and np.median(d) <= 2e-5 * scale


def test_pipeline_stages_compose(orc):
    """layer-range evaluation (the unit of the multi-GPU pipeline) chained == whole-model evaluation, bit for bit"""
    hp = dict(TINY_40B, n_layer=4)
    tensors = synth_model(hp, po.Q4_K, seed=2)
    whole, a, b = (po.OrcFalcon(hp, tensors, n_ctx=32) for _ in range(3))
    toks = np.array([11, 30, 31, 32], np.int32)
    want = whole.eval(toks, 0, all_logits=True)
    resid = a.eval_range(toks, 0, 0, 2)
    got = b.eval_range(toks, 0, 2, 4, resid_in=resid, all_logits=True)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("t", po.WEIGHT_TYPES + [po.Q8_K])
def test_codecs_bit_exact_vs_reference_random(orc, t):
    """quantise / dequantise / activation quantisation of random rows at three scales (tests/helpers.codec_random_inputs) against
    the reference's outputs, stored as SHA-256 digests of their bytes (tests/golden/codecs_random.json)"""
    gold = json.load(open(os.path.join(GOLD, "codecs_random.json")))[po.TYPE_NAMES[t]]
    for scale, x in codec_random_inputs(t):
        want = gold[repr(scale)]
        q = orc.quantize(t, x)
        if t == po.Q8_K:
            assert digest(q.reshape(8, -1, 292)[:, 1:]) == want["q_blocks_1_on"], scale
            continue
        assert digest(q) == want["q"], scale
        assert digest(orc.dequantize(t, q, 2048)) == want["deq"], scale
        assert digest(orc.quantize_act(t, x)[..., :260]) == want["aq_260"], scale


def test_falcon_eval_vs_reference_live():
    """all-token logits of a 5-token prompt of the synthetic Q3_K model against the reference's falcon_eval (tests/golden/tiny40b_q3_K.npz)"""
    g = np.load(os.path.join(GOLD, "tiny40b_q3_K.npz"))
    hp = dict(TINY_40B)
    o = po.OrcFalcon(hp, synth_model(hp, po.Q3_K, seed=int(g["seed"])), n_ctx=int(g["n_ctx"]))
    a, b = g["logits"], o.eval(g["prompt"], 0, all_logits=True)
    scale = np.abs(a).max()
    assert np.abs(a - b).max() <= 2e-2 * scale and np.median(np.abs(a - b)) <= 2e-5 * scale
