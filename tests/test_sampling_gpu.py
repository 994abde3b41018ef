"""-m gpu: the device sampler (b200_sampler_*, b200_falcon_generate; sampling.cu) against the REFERENCE's own sampling functions
(llama_sample_repetition_penalty / top_k / top_p / temperature / token, called in falcon_main's order by oracle/ref_harness.cpp):
the same seed must sample the same token ids -- the MT19937 stream, libstdc++'s discrete_distribution table and every cut are
restated bit for bit.  The reference's ids for seeded logits rows are stored in tests/golden/sampling.npz (tests/golden/make_golden.py).
A draw can differ only when device expf and glibc expf differ by an ulp AND the uniform variate lands within ~1e-7 of a table
boundary; the sequences below are fixed and short enough that this does not occur (a failing id would be a real divergence)."""
import os
import numpy as np
import pytest
import pyoracle as po
from helpers import TINY_40B, SAMPLER_CASES, sampler_case, synth_model

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(GOLD, "sampling.npz"))


def sample_row(gpu, sampler, logits):
    d = gpu.DevBuf(src=np.ascontiguousarray(logits, np.float32))
    return sampler.sample(d.ptr, logits.size)


@pytest.mark.parametrize("top_k,top_p,temp,penalty,last_n", SAMPLER_CASES)
def test_sampler_matches_reference_chain(gpu, gold, top_k, top_p, temp, penalty, last_n):
    want = gold["chain_%d" % SAMPLER_CASES.index((top_k, top_p, temp, penalty, last_n))].tolist()
    history, next_logits = sampler_case(top_k, last_n)
    seed = 4242
    sp = gpu.SamplingParams(top_k=top_k, top_p=top_p, temp=temp, repeat_penalty=penalty, repeat_last_n=last_n, seed=seed)
    dev = gpu.Sampler(sp, history)
    got = []
    win = history[-last_n:] if last_n > 0 else []
    for s, w in enumerate(want):
        got.append(sample_row(gpu, dev, next_logits(win)))
        if last_n > 0:
            win = (win + [w])[-last_n:]
        assert got[-1] == w, (s, got, want)                                 # stop at the first divergence: the windows would differ afterwards
    assert got == want


def test_generate_with_sampler_equals_host_loop_with_reference_sampler(gpu, gold):
    """b200_falcon_generate (sampler inside the step graph, ids never leave the GPU) == eval -> sampling chain on the host -> eval.
    The host loop samples with the stand-alone device sampler, which is first held to the reference's own loop over a model's logits
    (falcon_main's order: the first id at the seed, then the stream restarted at the seed)."""
    hp = dict(TINY_40B)
    tensors = synth_model(hp, po.Q4_K, seed=1234)
    sp = gpu.SamplingParams(top_k=40, top_p=0.95, temp=0.8, repeat_penalty=1.1, repeat_last_n=64, seed=77)
    prompt = gold["gen_prompt"]
    # (1) the stand-alone sampler == the reference over the stored logits rows
    assert sample_row(gpu, gpu.Sampler(sp, prompt), gold["gen_prompt_logits"]) == int(gold["gen_first"])
    s = gpu.Sampler(sp, list(prompt) + [int(gold["gen_first"])])
    assert [sample_row(gpu, s, row) for row in gold["gen_logits"]] == gold["gen_ids"].tolist()
    # (2) generation on the device == the host loop over this engine's logits
    a, b = gpu.Falcon(hp, n_ctx=64, n_batch=8), gpu.Falcon(hp, n_ctx=64, n_batch=8)
    a.set_tensors(tensors); b.set_tensors(tensors)
    a.eval(prompt, 0); lg = b.eval(prompt, 0)
    steps = 20
    first = sample_row(gpu, gpu.Sampler(sp, prompt), lg[0])
    win = [int(t) for t in prompt] + [first]
    dev = a.generate(sp, win, first, len(prompt), steps)
    host_sampler = gpu.Sampler(sp, win)                                     # the device stream starts at the seed: the host loop's too
    host, tok = [], first
    for i in range(steps):
        lg = b.eval(np.array([tok], np.int32), len(prompt) + i)
        tok = sample_row(gpu, host_sampler, lg[0])
        host.append(tok)
    assert dev.tolist() == host
    # greedy generation still works afterwards (the step graph is rebuilt around the arg-max kernel)
    g1 = a.generate_greedy(first, len(prompt), 4)
    sp0 = gpu.SamplingParams(top_k=1, top_p=1.0, temp=0.0, repeat_penalty=1.0, repeat_last_n=0, seed=1)
    g2 = a.generate(sp0, [], first, len(prompt), 4)
    assert g1.tolist() == g2.tolist()
    with pytest.raises(RuntimeError):
        a.generate(gpu.SamplingParams(top_k=0), [], first, len(prompt), 2)      # "whole vocabulary" is not supported on the device
    a.free(); b.free()
