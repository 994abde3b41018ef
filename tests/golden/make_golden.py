"""Generate the committed golden vectors from the UNMODIFIED reference (oracle/_ref, built from /root/reference).

Run here (where /root/reference exists):   python tests/golden/make_golden.py
Outputs (small, committed):
  codecs.npz          for every weight type: the reference's own test vector x[i] = 0.1 + 2 cos(i) (test-quantize-fns.cpp:26-30),
                      the reference's quantised bytes, its dequantised values, its Q8 activation bytes and vec_dot result
  tiny40b_q4_K.npz    logits of falcon_eval (CPU build) for the synthetic model recipe tests/helpers.synth_model
  tiny7b_q4_0.npz
  codecs_random.json  SHA-256 digests of the reference's quantised bytes, dequantised values and Q8 activation bytes for the random rows
                      of tests/helpers.codec_random_inputs (64 KB of output per case: the digest keeps the comparison bit-exact)
  tiny40b_q3_K.npz    all-token logits of falcon_eval (CPU build) for a 5-token prompt of the synthetic Q3_K model, seed 31
  sampling.npz        the ids the reference's sampling chain (falcon_main's order, std::mt19937 stream) draws for the seeded logits rows
                      of tests/helpers.SAMPLER_CASES, and a generation over the oracle's logits of the synthetic Q4_K model
Machines without the reference's sources run the tests against these files.  Arguments select outputs (default: all of them).
"""
import json
import os
import sys
import tempfile
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from helpers import po, ggcc, synth_model, digest, codec_random_inputs, sampler_case, SAMPLER_CASES, TINY_40B, TINY_7B  # noqa: E402


def codecs():
    r = po.ref()
    out = {}
    x = po.synth_vector(4096).reshape(4, 1024)
    a = po.synth_vector(4096, offset=1.0).reshape(4, 1024)
    out["x"], out["a"] = x, a
    for t in po.WEIGHT_TYPES:
        n = po.TYPE_NAMES[t]
        q = r.quantize(t, x)
        out[n + "_q"] = q
        out[n + "_deq"] = r.dequantize(t, q, 1024)
        aq = r.quantize_act(t, a)
        out[n + "_aq"] = aq
        out[n + "_dot"] = np.array([r.vec_dot(t, 1024, q[i], aq[i]) for i in range(4)], np.float32)
    np.savez_compressed(os.path.join(HERE, "codecs.npz"), **out)


def model(name, hp, wt, seed, n_ctx=64):
    tensors = synth_model(hp, wt, seed)
    path = os.path.join(tempfile.gettempdir(), name + ".ggcc")
    ggcc.write_ggcc(path, hp, tensors, ftype=ggcc.FTYPE_OF_TYPE[wt])
    ref = po.RefFalcon(path, n_ctx=n_ctx, n_batch=8, logits_all=True)
    prompt = np.array([11, 100, 101, 102, 103, 104, 105], np.int32)
    pl = ref.eval(prompt, 0, n_threads=4)
    dec = np.array([200, 17, 333, 42], np.int32)
    dl = np.concatenate([ref.eval(dec[i:i + 1], len(prompt) + i, n_threads=4) for i in range(len(dec))])
    ref.close()
    os.remove(path)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), prompt=prompt, prompt_logits=pl, decode_tokens=dec, decode_logits=dl,
                        wtype=wt, seed=seed, n_ctx=n_ctx, **{"hp_" + k: v for k, v in hp.items()})


def codecs_random():
    r = po.ref()
    out = {}
    for t in po.WEIGHT_TYPES + [po.Q8_K]:
        out[po.TYPE_NAMES[t]] = cases = {}
        for scale, x in codec_random_inputs(t):
            q = r.quantize(t, x)
            if t == po.Q8_K:                 # Q8_K is an activation format: its quantiser only, first block of each row excluded
                cases[repr(scale)] = {"q_blocks_1_on": digest(q.reshape(8, -1, 292)[:, 1:])}
                continue
            cases[repr(scale)] = {"q": digest(q), "deq": digest(r.dequantize(t, q, 2048)), "aq_260": digest(r.quantize_act(t, x)[..., :260])}
    with open(os.path.join(HERE, "codecs_random.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")


def model_q3_k():
    hp = dict(TINY_40B)
    tensors = synth_model(hp, po.Q3_K, seed=31)
    path = os.path.join(tempfile.gettempdir(), "tiny40b_q3_K.ggcc")
    ggcc.write_ggcc(path, hp, tensors, ftype=12)
    ref = po.RefFalcon(path, n_ctx=64, n_batch=8, logits_all=True)
    prompt = np.array([11, 70, 71, 72, 73], np.int32)
    logits = ref.eval(prompt, 0, n_threads=2)
    ref.close()
    os.remove(path)
    np.savez_compressed(os.path.join(HERE, "tiny40b_q3_K.npz"), prompt=prompt, logits=logits, seed=31, n_ctx=64)


def sampling():
    hp = dict(TINY_40B)
    tensors = synth_model(hp, po.Q4_K, seed=1234)
    path = os.path.join(tempfile.gettempdir(), "sampling.ggcc")
    ggcc.write_ggcc(path, hp, tensors, ftype=15)
    ref = po.RefFalcon(path, n_ctx=64, n_batch=8)          # a context for the sampling functions; its model is not evaluated
    out = {}
    for i, (top_k, top_p, temp, penalty, last_n) in enumerate(SAMPLER_CASES):
        history, next_logits = sampler_case(top_k, last_n)
        ref.set_seed(4242)
        win, ids = (history[-last_n:] if last_n > 0 else []), []
        for _ in range(48):
            ids.append(ref.sample(next_logits(win), win, top_k, top_p, temp, penalty))
            if last_n > 0:
                win = (win + [ids[-1]])[-last_n:]
        out["chain_%d" % i] = np.array(ids, np.int32)
    # falcon_main's loop over a model's logits (the oracle's): the first id at the seed, then the stream restarted at the seed for 20 steps
    o = po.OrcFalcon(hp, tensors, n_ctx=64)
    prompt = np.array([11, 100, 101, 102, 103], np.int32)
    lg0 = o.eval(prompt, 0)[0]
    ref.set_seed(77)
    first = ref.sample(lg0, prompt, 40, 0.95, 0.8, 1.1)
    ref.set_seed(77)
    win, rows, ids = [int(t) for t in prompt] + [first], [], []
    for i in range(20):
        rows.append(o.eval(np.array([win[-1]], np.int32), len(prompt) + i)[0])
        ids.append(ref.sample(rows[-1], win[-64:], 40, 0.95, 0.8, 1.1))
        win.append(ids[-1])
    ref.close()
    os.remove(path)
    np.savez_compressed(os.path.join(HERE, "sampling.npz"), gen_prompt=prompt, gen_prompt_logits=lg0, gen_first=first, gen_logits=np.array(rows),
                        gen_ids=np.array(ids, np.int32), **out)


if __name__ == "__main__":
    makers = {"codecs": codecs, "models": lambda: (model("tiny40b_q4_K", TINY_40B, po.Q4_K, 1234), model("tiny7b_q4_0", TINY_7B, po.Q4_0, 1234)),
              "codecs_random": codecs_random, "model_q3_k": model_q3_k, "sampling": sampling}
    for name in sys.argv[1:] or list(makers):
        makers[name]()
    print("golden vectors written to", HERE)
