#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric (Falcon-40B Q4_K decode tokens/s on B200) and, beside it, every BASELINE config.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--config headline|1|2|3|4|5] [--no-extras] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...      (N > 1)

A "step" is one decode eval (one token, n_batch = 1) of a synthetic random-init Falcon model through the hot path; weights are
generated directly as well-formed quantised blocks on the device (SURVEY.md section 8d).  One JSON line is printed by rank 0.

Top level = the headline config (or the one --config selects):
  value   : decode tokens/s with token ids and logits resident in HBM, CUDA events on the eval stream.
            N = 1: K x b200_falcon_decode_dev.   N > 1 (layer-range pipeline): STRICT AUTOREGRESSIVE single stream -- the last rank
            takes the arg-max on the device and the id travels to rank 0 by ncclSend/ncclRecv inside the step graph
            (b200_falcon_generate_greedy); the teacher-forced figure, where consecutive tokens overlap across the stages, is reported
            separately as pipelined_tok_s and is NOT the value.
  e2e     : the same metric through the reference-facing C-ABI call b200_falcon_eval with HOST buffers (token id H2D + logits D2H
            inside the timed region; N > 1: the last rank's host arg-max is broadcast before the next step may start)
  roofline: the dominant kernel (decode mat-vec) timed alone with CUDA events over the model's own matrices; step_frac = the whole
            step's algorithmic bytes / time against the measured HBM peak (the number the north-star target is about)
  e2e_dropin: the same metric through the UNMODIFIED reference's own falcon_eval (libfalcon.cpp + ggml.c built with -DGGML_USE_CUBLAS)
            running on top of this library's ggml_cuda_* operator surface -- the drop-in number
  cpu_baseline / --impl reference: the UNMODIFIED reference's CPU path (oracle/_ref falcon_eval) on the box's host cores over the
            REAL full-size model file (written to /dev/shm; identical layer tensors repeated, CPU time does not depend on values)
  prompt  : BASELINE config 3 (2048-token prompt, n_batch 512) with its own tensor roofline
  configs : cfg1 (Q4_0 4096x4096x1 mat-vec: reference ggml.c on the host cores + its GPU twin), cfg2 (Falcon-7B Q4_0 decode, 128 tokens),
            cfg4 (Falcon-40B Q3_K decode, layer-split at N), cfg5 (Falcon-180B Q4_K decode at 8k context, KV pre-filled)
  pipeline_parity (N > 1): a small fixed model evaluated through the N-rank pipeline gives bit-identical logits / greedy tokens to
            the same model on one rank
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODELS = {
    "falcon40b": dict(n_vocab=65024, n_embd=8192, n_head=128, n_head_kv=8, n_layer=60, falcon_type=40),
    "falcon7b": dict(n_vocab=65024, n_embd=4544, n_head=71, n_head_kv=1, n_layer=32, falcon_type=7),
    "falcon180b": dict(n_vocab=65024, n_embd=14848, n_head=232, n_head_kv=8, n_layer=80, falcon_type=40),
}
Q4_0, Q3_K, Q4_K = 2, 11, 12
TYPE_NAME = {Q4_0: "Q4_0", Q3_K: "Q3_K", Q4_K: "Q4_K"}
BYTES_PER_WEIGHT = {Q4_0: 18 / 32, Q3_K: 110 / 256, Q4_K: 144 / 256}
# name -> (model, weight type, n_ctx, first timed position, metric)
DECODE_CONFIGS = {
    "headline": ("falcon40b", Q4_K, 2048, 0, "falcon40b_q4_k_decode_tokens_per_s"),
    "2": ("falcon7b", Q4_0, 2048, 0, "falcon7b_q4_0_decode_tokens_per_s"),
    "4": ("falcon40b", Q3_K, 2048, 0, "falcon40b_q3_k_decode_tokens_per_s"),
    "5": ("falcon180b", Q4_K, 8192, 8000, "falcon180b_q4_k_decode_8k_ctx_tokens_per_s"),
}
WORKLOAD = {
    "headline": "Falcon-40B Q4_K decode, n_batch=1, synthetic random-init GGCC-shaped weights",
    "1": "Q4_0 4096x4096x1 mat-vec (examples/benchmark matmult shape), 32 rotating matrices",
    "2": "Falcon-7B Q4_0 decode, n_batch=1, 128 tokens, random-init GGCC-shaped weights",
    "3": "Falcon-40B Q4_K prompt, n_batch=512, 2048 synthetic tokens",
    "4": "Falcon-40B Q3_K decode, n_batch=1, contiguous layer ranges per GPU",
    "5": "Falcon-180B Q4_K decode at 8k context (KV pre-filled to position 8000), contiguous layer ranges per GPU",
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", 1451.1)), "measured (MEASURED_PEAKS.json: hbm_gbs, bf16_tflops_sustained)"
    return 6650.0, 1450.0, "fallback (B200_PROFILING.md: 6.65 TB/s copy, 1.45 PFLOP/s sustained bf16)"


def weight_elems(hp):
    """elements of the 2-D weights a decode step streams (everything but the embedding matrix, which contributes one row)"""
    E, H, HKV, L, V = hp["n_embd"], hp["n_head"], hp["n_head_kv"], hp["n_layer"], hp["n_vocab"]
    D = E // H
    return L * (E * (H + 2 * HKV) * D + E * E + 8 * E * E) + E * V


def kv_bytes(hp, n_past):
    return hp["n_layer"] * 2 * n_past * hp["n_head_kv"] * (hp["n_embd"] // hp["n_head"]) * 4


def stage_ranges(hp, world):
    """contiguous layer ranges balanced by BYTES: the last rank also streams lm_head (worth V / (9 E + (H + 2 HKV) D) layers), so it
    gets correspondingly fewer layers; the other ranks share the rest evenly (replaces the VRAM-proportional tensor_split,
    ggml-cuda.cu:1999-2012).  Of the two candidate sizes of the last stage the one with the smaller maximum stage is taken."""
    E, H, HKV, L, V = hp["n_embd"], hp["n_head"], hp["n_head_kv"], hp["n_layer"], hp["n_vocab"]
    D = E // H
    if world == 1:
        return [(0, L)]
    head = V / float(9 * E + (H + 2 * HKV) * D)
    per = (L + head) / world
    best = None
    for n_last in {max(1, int(per - head)), max(1, int(per - head) + 1)}:
        rest = L - n_last
        if rest < world - 1:
            continue
        base, rem = divmod(rest, world - 1)
        sizes = [base + (1 if r < rem else 0) for r in range(world - 1)] + [n_last]
        loads = sizes[:-1] + [n_last + head]
        key = (max(loads), max(loads) - min(loads))                  # smallest maximum stage, then smallest spread
        if best is None or key < best[0]:
            best = (key, sizes)
    cuts = [0]
    for n in best[1]:
        cuts.append(cuts[-1] + n)
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled during the timed region (B200_PROFILING.md recipe)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(dev), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm = [float(r[1]) for r in rows if len(r) >= 9]
        busy = [v for v in sm if v > 0.6 * max(sm)] if sm else []
        reasons = set()
        for r in rows:
            if len(r) < 9:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": float(rows[0][2]) if rows else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ reference (CPU) arm
def _oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle as po
    return po


def _host_threads():
    return os.cpu_count() or 1


def write_full_model(path, hp, wtype, rng):
    """a GGCC v10 file of the FULL model: one random tensor per distinct shape, repeated for every layer (the CPU path's time does
    not depend on the weight values; the file is byte-for-byte a valid model the unmodified reference loads)"""
    import ggllm_cpp_b200.ggcc as ggcc
    cache, tensors = {}, {}
    for name, ne in ggcc.falcon_shapes(hp).items():
        key = (tuple(ne), name.endswith(".bias"))
        if key not in cache:
            if len(ne) == 1:
                cache[key] = (0, ne, (0.01 * rng.standard_normal(ne[0])).astype(np.float32) if name.endswith(".bias")
                              else (1.0 + 0.1 * rng.standard_normal(ne[0])).astype(np.float32))
            else:
                cache[key] = (wtype, ne, ggcc.random_blocks(wtype, ne[1], ne[0], rng))
        tensors[name] = cache[key]
    ggcc.write_ggcc(path, hp, tensors, ftype=ggcc.FTYPE_OF_TYPE.get(wtype, 0))
    return sum(ggcc.tensor_nbytes(t, ne) for n, (t, ne, _) in tensors.items() if len(ne) == 2 and "word_embeddings" not in n)


class FullModelFile:
    """the FULL-size random model as a GGCC file in /dev/shm for the reference-side arms (CPU baseline, drop-in run); falls back to a
    6-layer slice ("extrapolated": true, tok/s scaled by the weight-byte ratio) only when /dev/shm cannot hold it or is too slow"""

    def __init__(self, model, wtype):
        self.model, self.wtype = model, wtype
        hp_full = dict(MODELS[model])
        self.full_bytes = weight_elems(hp_full) * BYTES_PER_WEIGHT[wtype]
        need = self.full_bytes * 1.05 + hp_full["n_vocab"] * hp_full["n_embd"] * BYTES_PER_WEIGHT[wtype]
        shm = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
        st = os.statvfs(shm)
        self.extrapolated = st.f_bavail * st.f_frsize < need * 1.1
        if not self.extrapolated:                        # writing the file must stay a small part of a run that has to end within minutes
            probe_path = os.path.join(shm, "b200_bench_probe_%d" % os.getpid())
            t0 = time.time()
            np.zeros(1 << 28, np.uint8).tofile(probe_path)
            rate = (1 << 28) / max(time.time() - t0, 1e-3)
            os.unlink(probe_path)
            self.extrapolated = need / rate > float(os.environ.get("BENCH_REF_MAX_WRITE_S", "100"))
        self.hp = dict(hp_full, n_layer=6) if self.extrapolated else hp_full
        self.path = os.path.join(shm if not self.extrapolated else tempfile.gettempdir(), "b200_bench_ref_%d.ggcc" % os.getpid())
        t0 = time.time()
        self.sample_bytes = write_full_model(self.path, self.hp, wtype, np.random.default_rng(1))
        self.write_s = time.time() - t0
        self.scale = self.sample_bytes / self.full_bytes

    def what(self):
        return ("the %s random-init %s %s GGCC model (%.2f GB of weights, %s)"
                % ("FULL %d-layer" % self.hp["n_layer"] if not self.extrapolated else "%d-layer slice of the" % self.hp["n_layer"], self.model,
                   TYPE_NAME[self.wtype], self.sample_bytes / 1e9,
                   "no extrapolation" if not self.extrapolated else "tok/s scaled by the weight-byte ratio %.4f" % self.scale))

    def close(self):
        if os.path.exists(self.path):
            os.unlink(self.path)


def reference_cpu_decode(model, wtype, steps, warmup, n_ctx_rope=129, mf=None):
    """The UNMODIFIED reference's CPU path (falcon_eval from oracle/_ref/libfalcon_ref.so; the oracle port if that library is absent)
    decoding with n_batch = 1 over the full-size random model file."""
    po = _oracle()
    kind = "reference" if po.have_ref_falcon() else "port"
    own = mf is None
    if own:
        mf = FullModelFile(model, wtype)
    cores = _host_threads()
    t0 = time.time()
    try:
        if kind == "reference":
            eng = po.RefFalcon(mf.path, n_ctx=256, n_batch=1)
            run = lambda tok, pos, t: eng.eval(np.array([tok], np.int32), pos, n_threads=t, n_max_real_ctx=n_ctx_rope)
        else:
            import ggllm_cpp_b200.ggcc as ggcc
            _, tensors = ggcc.read_ggcc(mf.path)
            eng = po.OrcFalcon(mf.hp, tensors, n_ctx=256)
            run = lambda tok, pos, t: eng.eval(np.array([tok], np.int32), pos, n_ctx_rope=n_ctx_rope, nthreads=min(t, 64))
        run(11, 0, min(cores, 32))                      # the reference's own warm-up eval (falcon_main.cpp:662-673): also faults the file in
        # thread count: ggml's spin-barrier pool does not scale monotonically with threads (README.md:137) -- probe, keep the fastest
        pos, probe = 1, {}
        for t in sorted(set(min(cores, c) for c in (8, 16, 32, 64, 128))):
            t1 = time.time()
            run(50 + t, pos, t); pos += 1
            probe[t] = time.time() - t1
            if probe[t] > 1.5 * min(probe.values()):      # past the knee (128 spinning threads: 30 s per token): stop probing
                break
        best_t = min(probe, key=probe.get)
        for i in range(warmup):
            run(100 + i, pos, best_t); pos += 1
        t1 = time.time()
        for i in range(steps):
            run(200 + i, pos, best_t); pos += 1
        dt = time.time() - t1
        if kind == "reference":
            eng.close()
    finally:
        if own:
            mf.close()
    tps = steps / dt * mf.scale
    return dict(value=tps, unit="tok/s", cores=best_t, kind=kind, ms_per_step=1e3 / tps, steps=steps, extrapolated=bool(mf.extrapolated),
                sample=("%d decode tokens (after BOS + %d probe + %d warm-up evals) of %s through %s falcon_eval, -t %d (fastest of %s on %d host cores); "
                        "file written in %.0f s, load + evals %.0f s")
                       % (steps, len(probe), warmup, mf.what(), "the unmodified reference's (oracle/_ref)" if kind == "reference" else "the oracle port's", best_t,
                          {k: round(v, 3) for k, v in probe.items()}, cores, mf.write_s, time.time() - t0))


def dropin_decode(cx, mf, steps, warmup, n_ctx_rope=129):
    """The drop-in number: the UNMODIFIED reference (ggml.c + libfalcon.cpp built with -DGGML_USE_CUBLAS, oracle/_ref/libfalcon_hook.so) loads the
    same GGCC file with every layer offloaded and decodes through ITS OWN falcon_eval; the ggml_cuda_* symbols it calls are this
    library's.  After the first eval the operator hook recognises the Falcon graph and evaluates it whole on the device (ggml_surface.cu)."""
    po = _oracle()
    hook = os.path.join(po.HERE, "_ref", "libfalcon_hook.so")
    if not os.path.exists(hook):
        return {"unavailable": "oracle/_ref/libfalcon_hook.so not built (needs /root/reference at build time)"}
    L = cx.b.lib()                                      # libggml_b200.so in the global symbol scope: resolves the hook library's ggml_cuda_*
    t0 = time.time()
    eng = po.RefFalcon(mf.path, n_ctx=2048, n_batch=1, hook=True, n_gpu_layers=mf.hp["n_layer"] + 2)
    load_s = time.time() - t0
    taken0 = L.b200_surface_takeover_evals()
    eng.eval(np.array([11], np.int32), 0, n_threads=1, n_max_real_ctx=n_ctx_rope)      # falcon_main's BOS warm-up eval = the hook's learning eval (per-node path)
    pos = 1
    for i in range(warmup):
        eng.eval(np.array([100 + i], np.int32), pos, n_threads=1, n_max_real_ctx=n_ctx_rope); pos += 1
    t1 = time.perf_counter()
    for i in range(steps):
        eng.eval(np.array([200 + i], np.int32), pos, n_threads=1, n_max_real_ctx=n_ctx_rope); pos += 1
    dt = time.perf_counter() - t1
    taken = L.b200_surface_takeover_evals() - taken0
    eng.close()
    tps = steps / dt * mf.scale
    return {"value": tps, "unit": "tok/s", "ms_per_step": 1e3 / tps, "steps": steps, "engine_evals": int(taken), "extrapolated": bool(mf.extrapolated),
            "load_seconds": load_s, "h2d_bytes_per_step": 8, "d2h_bytes_per_step": mf.hp["n_vocab"] * 4,
            "api": "falcon_eval of the unmodified reference (-t 1, every layer offloaded) on top of libggml_b200.so's ggml_cuda_* surface",
            "what": "%d decode tokens of %s; %d of %d evals after the first ran as whole-graph device evaluations behind ggml_cuda_compute_forward"
                    % (steps, mf.what(), taken, steps + warmup)}


def reference_cpu_matvec(K=4096, M=4096, n_mats=32, iters=8):
    """BASELINE config 1 on the host cores: ggml_mul_mat + ggml_graph_compute of the unmodified reference over rotating Q4_0 matrices"""
    po = _oracle()
    import ggllm_cpp_b200.ggcc as ggcc
    rng = np.random.default_rng(5)
    blocks = ggcc.random_blocks(Q4_0, M * n_mats, K, rng)
    x = rng.standard_normal(K).astype(np.float32)
    y = np.zeros(M, np.float32)
    cores = _host_threads()
    out = {"shape": [K, M, 1], "n_mats": n_mats, "bytes_per_call": K * M * 18 // 32}
    if not po.have_ref_falcon():
        t0 = time.time()
        for i in range(4):
            y = po.orc().mul_mat(Q4_0, blocks[i * M:(i + 1) * M], K, M, x[None, :], nthreads=min(cores, 64))[0]
        out.update(kind="port", us_per_call=(time.time() - t0) / 4 * 1e6, cores=min(cores, 64))
    else:
        L = C.CDLL(os.path.join(po.HERE, "_ref", "libfalcon_ref.so"))
        L.refh_matvec_bench.restype = C.c_double
        L.refh_matvec_bench.argtypes = [C.c_int] * 5 + [C.c_void_p] * 4
        best = None
        for t in sorted(set(min(cores, c) for c in (4, 8, 16, 32))):      # a 9 MB mat-vec stops scaling early: keep the fastest thread count
            b_us = C.c_double()
            us = L.refh_matvec_bench(K, M, n_mats, iters, t, blocks.ctypes.data, x.ctypes.data, y.ctypes.data, C.byref(b_us))
            if best is None or us < best[0]:
                best = (us, b_us.value, t)
        out.update(kind="reference", us_per_call=best[0], best_us=best[1], cores=best[2])
    out["GBs"] = out["bytes_per_call"] / out["us_per_call"] / 1e3
    out["GFLOPs"] = 2.0 * K * M / out["us_per_call"] / 1e3
    return out, blocks, x, y


# ------------------------------------------------------------------------------------------------ GPU legs
class Ctx:
    """binding + (optional) torch.distributed for one bench process"""

    def __init__(self):
        self.rank, self.world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        import ggllm_cpp_b200.binding as b
        self.b = b
        self.dist = None
        if self.world > 1:
            import torch
            import torch.distributed as dist
            torch.cuda.set_device(self.local_rank)
            dist.init_process_group("nccl")
            self.dist, self.torch = dist, torch
        b.init(self.local_rank)
        self.L = b.lib()

    def barrier(self, stream=None):
        self.L.b200_stream_synchronize(stream)
        if self.dist is not None:
            self.dist.barrier()

    def max_over_ranks(self, vals):
        if self.dist is None:
            return [float(v) for v in vals]
        t = self.torch.tensor([float(v) for v in vals], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def sum_over_ranks(self, vals):
        if self.dist is None:
            return [float(v) for v in vals]
        t = self.torch.tensor([float(v) for v in vals], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    def make_model(self, hp, wtype, n_ctx, n_batch, seed=1234):
        import ggllm_cpp_b200.ggcc as ggcc
        lf, ll = stage_ranges(hp, self.world)[self.rank]
        f = self.b.Falcon(hp, n_ctx=n_ctx, n_batch=n_batch, rank=self.rank, world=self.world, layers=(lf, ll))
        f.set_random(ggcc.falcon_shapes(hp), wtype, seed=seed)
        if self.world > 1:
            ids = [self.b.Falcon.nccl_unique_id() if self.rank == 0 else None]
            self.dist.broadcast_object_list(ids, src=0)
            f.init_pipeline(ids[0])
        return f


def decode_leg(cx, f, hp, wtype, steps, warmup, pos0, rope, with_kernel_probe=True, keep_output=False):
    """-> dict of the decode figures of one model (see module docstring).  All ranks call it; figures are max-over-ranks times.
    keep_output (one GPU): "_output" holds the logits the last timed step left on the device."""
    L, b = cx.L, cx.b
    stream = f.stream()
    tok_dev = b.DevBuf(src=np.array([1234], np.int32))
    pos = pos0
    if pos0 == 0:
        f.eval(np.array([11], np.int32), 0, rope)        # the reference's own BOS warm-up eval at n_past = 0 (falcon_main.cpp:662-673)
        pos = 1
    else:
        f.kv_fill_random(0, pos0, seed=77)               # a long context without evaluating pos0 tokens first
    for _ in range(warmup):
        f.decode_dev(tok_dev.ptr, pos, rope); pos += 1
    for _ in range(3):
        f.eval(np.array([100 + pos % 1000], np.int32), pos, rope); pos += 1
    pos_start = pos
    cx.barrier(stream)

    # ---- (1) device-resident, teacher-forced: K x decode_dev, CUDA events on the eval stream
    e0, e1 = L.b200_event_create(), L.b200_event_create()
    cx.barrier(stream)
    t0 = time.perf_counter()
    L.b200_event_record(e0, stream)
    for _ in range(steps):
        f.decode_dev(tok_dev.ptr, pos, rope); pos += 1
    L.b200_event_record(e1, stream)
    cx.barrier(stream)
    wall_ms = (time.perf_counter() - t0) * 1e3
    tf_ms = L.b200_event_elapsed_ms(e0, e1)
    launches = f.last_launches() * steps
    output = None
    if keep_output:
        output = np.empty(hp["n_vocab"], np.float32)
        L.b200_memcpy_d2h(output.ctypes.data_as(C.c_void_p), f.logits_dev(), output.nbytes)

    # ---- (2) N > 1: strict autoregressive, device-side (arg-max on the last rank, id -> rank 0 over NCCL inside the step graph)
    auto_ms = None
    if cx.world > 1:
        f.generate_greedy(1234, pos, 4, rope); pos += 4              # builds the generation-step graphs
        cx.barrier(stream)
        f.generate_greedy(1234, pos, steps, rope); pos += steps
        auto_ms = f.last_ms()
        cx.barrier(stream)

    # ---- (3) end to end through the C ABI with host buffers (token H2D + logits D2H each step)
    cx.barrier(stream)
    t0 = time.perf_counter()
    if cx.world == 1:
        for i in range(steps):
            f.eval(np.array([300 + i], np.int32), pos, rope); pos += 1
    else:
        tok = cx.torch.zeros(1, dtype=cx.torch.int32, device="cuda")
        for i in range(steps):
            lg = f.eval(np.array([int(tok.item()) % hp["n_vocab"]], np.int32), pos, rope)
            if cx.rank == cx.world - 1:
                tok[0] = int(np.argmax(lg[0]))
            cx.dist.broadcast(tok, src=cx.world - 1)
            pos += 1
    cx.barrier(stream)
    e2e_ms = (time.perf_counter() - t0) * 1e3

    probe = None
    if with_kernel_probe:
        mv_ms, mv_n, mv_bytes = f.profile_matvec(reps=3)
        probe = (mv_ms, mv_n, mv_bytes)
    vals = cx.max_over_ranks([tf_ms, wall_ms, e2e_ms, auto_ms if auto_ms is not None else 0.0])
    tf_ms, wall_ms, e2e_ms, auto_max = vals
    wbytes, launches = cx.sum_over_ranks([float(f.weight_bytes()), float(launches)])
    dev_ms = auto_max if cx.world > 1 else tf_ms
    value = steps / (dev_ms / 1e3)
    n_past_mid = pos_start + steps // 2
    sbytes = wbytes + kv_bytes(hp, n_past_mid)
    peak, _, _ = peaks()
    out = {"tok_s": value, "ms_per_step": dev_ms / steps, "e2e_tok_s": steps / (e2e_ms / 1e3), "e2e_ms_per_step": e2e_ms / steps,
           "wall_ms_per_step": wall_ms / steps, "gpu_launches": int(launches), "weight_bytes": wbytes, "step_bytes": sbytes,
           "n_past": [pos_start, pos_start + steps],
           # one token stream walks the stages one after the other: per-GPU bandwidth while a stage is active = step bytes / step time
           "step_achieved_GBs": sbytes * value / 1e9, "step_frac": sbytes * value / 1e9 / peak, "roofline_tok_s": peak * 1e9 / sbytes}
    if cx.world > 1:
        out["pipelined_tok_s"] = steps / (tf_ms / 1e3)
        out["autoregressive_tok_s"] = value
    out["_probe"] = probe
    if keep_output:
        out["_output"] = output
    return out


def prompt_leg(cx, f, hp, n_tokens=2048, n_batch=512):
    """BASELINE config 3: n_tokens synthetic prompt tokens in chunks of n_batch through b200_falcon_eval (host token ids in, host logits
    of the last token out).  N > 1: chunk c+1 enters stage 0 while chunk c is in stage 1 -- legitimate for a prompt (the KV cache of a
    stage only depends on that stage's earlier chunks)."""
    toks = np.random.default_rng(7).integers(12, hp["n_vocab"], size=n_tokens).astype(np.int32)
    stream = f.stream()
    f.eval(toks[:n_batch], 0, 0)                     # warm-up (tensor maps, scratch)
    cx.barrier(stream)
    t0 = time.perf_counter()
    dev_ms = 0.0
    for c in range(n_tokens // n_batch):
        logits = f.eval(toks[n_batch * c: n_batch * (c + 1)], n_batch * c, 0)
        dev_ms += f.last_ms()
    cx.barrier(stream)
    wall_s = time.perf_counter() - t0
    wall_s, dev_ms = cx.max_over_ranks([wall_s, dev_ms])
    E, H, Lh, D = hp["n_embd"], hp["n_head"], hp["n_layer"], hp["n_embd"] // hp["n_head"]
    mm_flop = 2.0 * weight_elems(hp) * n_tokens - 2.0 * E * hp["n_vocab"] * (n_tokens - n_tokens // n_batch)     # lm_head: last token of each chunk only
    att_flop = sum(4.0 * n_batch * (n_batch * c + (n_batch + 1) / 2.0) * D * H * Lh for c in range(n_tokens // n_batch))     # causal: QK^T and PV over the visible keys
    _, tf_peak, _ = peaks()
    secs = wall_s if cx.world > 1 else dev_ms / 1e3
    return {"tok_s": n_tokens / wall_s, "tokens": n_tokens, "n_batch": n_batch, "seconds": wall_s, "device_seconds": dev_ms / 1e3 if cx.world == 1 else None,
            "device_tok_s": n_tokens / (dev_ms / 1e3) if cx.world == 1 else None,
            "matmul_TFLOP": mm_flop / 1e12, "attention_TFLOP": att_flop / 1e12,
            "roofline": {"bound": "tensor", "achieved": (mm_flop + att_flop) / secs / 1e12 / cx.world, "peak": tf_peak, "unit": "TFLOP/s",
                         "frac": (mm_flop + att_flop) / secs / 1e12 / cx.world / tf_peak, "traffic": None,
                         "what": "whole prompt (dequantising tcgen05 GEMMs + tcgen05 attention) per GPU against the sustained dense bf16 peak; "
                                 + ("device time (CUDA events per eval)" if cx.world == 1 else "wall clock (pipelined chunks)")},
            "roofline_tok_s": tf_peak * 1e12 * cx.world / ((mm_flop + att_flop) / n_tokens),
            "what": "%d x b200_falcon_eval of %d host tokens; tok_s = wall clock incl. H2D / D2H" % (n_tokens // n_batch, n_batch),
            "_output": logits[0]}


def matvec_leg(cx, K=4096, M=4096, n_mats=32, reps=20, cpu=True):
    """BASELINE config 1 on the GPU (+ the reference's ggml.c on the host cores): same blocks, same activation column.
    "_output" holds the result column of the last timed call."""
    L, b = cx.L, cx.b
    import ggllm_cpp_b200.ggcc as ggcc
    if cpu:
        ref, blocks, x, y_cpu = reference_cpu_matvec(K, M, n_mats)
    else:
        rng = np.random.default_rng(5)
        ref, blocks, x, y_cpu = None, ggcc.random_blocks(Q4_0, M * n_mats, K, rng), rng.standard_normal(K).astype(np.float32), None
    Ws = [b.Weight(Q4_0, K, M, blocks[i * M:(i + 1) * M]) for i in range(n_mats)]
    xd, yd = b.DevBuf(src=x[None, :]), b.DevBuf(M * 4)
    A = b.ActQ(Q4_0, K, 1)
    A.quantize(xd.ptr)
    for w in Ws:
        L.b200_mul_mat_vec_q(w.h, A.h, yd.ptr, M, 0, None, None)
    L.b200_synchronize()
    e0, e1 = L.b200_event_create(), L.b200_event_create()
    L.b200_event_record(e0, None)
    for _ in range(reps):
        for w in Ws:
            L.b200_mul_mat_vec_q(w.h, A.h, yd.ptr, M, 0, None, None)
    L.b200_event_record(e1, None)
    L.b200_event_synchronize(e1)
    us = L.b200_event_elapsed_ms(e0, e1) * 1e3 / (reps * n_mats)
    y_last = yd.download(np.float32, (M,))
    # end to end: host activation column in, host result out (H2D + quantise + mat-vec + D2H), what ggml_cuda_mul_mat's caller sees
    xh, yh = np.ascontiguousarray(x[None, :]), np.zeros((1, M), np.float32)
    t0 = time.perf_counter()
    for r in range(4):
        for w in Ws:
            L.b200_memcpy_h2d(xd.ptr, xh.ctypes.data_as(C.c_void_p), xh.nbytes)
            L.b200_mul_mat(w.h, xd.ptr, K, 1, yd.ptr, M)
            L.b200_memcpy_d2h(yh.ctypes.data_as(C.c_void_p), yd.ptr, yh.nbytes)
    e2e_us = (time.perf_counter() - t0) * 1e6 / (4 * n_mats)
    L.b200_mul_mat(Ws[0].h, xd.ptr, K, 1, yd.ptr, M)
    y_gpu = yd.download(np.float32, (M,))
    nbytes = K * M * 18 // 32
    peak, _, _ = peaks()
    out = {"shape": [K, M, 1], "n_mats": n_mats, "l2": "%d rotating matrices = %.0f MB > 126 MB L2" % (n_mats, n_mats * nbytes / 1e6),
           "gpu": {"us_per_call": us, "GBs": nbytes / us / 1e3, "frac_of_hbm_peak": nbytes / us / 1e3 / peak, "GFLOPs": 2.0 * K * M / us / 1e3,
                   "e2e_us_per_call": e2e_us, "e2e_bytes": {"h2d": K * 4, "d2h": M * 4}, "roofline_us": nbytes / peak / 1e3,
                   "note": "a 9.4 MB mat-vec lasts ~2 us: back-to-back launches are launch-latency bound, not HBM bound"},
           "cpu": ref, "_output": y_last}
    if y_cpu is not None:
        mag = float(np.abs(y_cpu).max())
        out["parity_max_abs_diff_over_max"] = float(np.abs(y_gpu - y_cpu).max() / mag)
    for w in Ws:
        w.free()
    return out


def pipeline_parity(cx):
    """a small fixed model through the N-rank pipeline vs the same model on ONE rank (the last rank holds both): logits of a prompt and of
    decode steps and the greedy token sequence must be bit-identical -- the residual crosses each boundary unchanged and every
    kernel is deterministic"""
    import ggllm_cpp_b200.ggcc as ggcc
    hp = dict(n_vocab=1024, n_embd=1024, n_head=16, n_head_kv=2, n_layer=max(8, 2 * cx.world), falcon_type=40)
    shapes = ggcc.falcon_shapes(hp)
    f = cx.make_model(hp, Q4_K, 128, 16, seed=4321)
    prompt = np.arange(12, 12 + 16, dtype=np.int32)
    outs = [f.eval(prompt, 0, 0, all_logits=True)]
    for i in range(4):
        outs.append(f.eval(np.array([100 + i], np.int32), 16 + i, 0))
    toks = f.generate_greedy(77, 20, 12, 0)
    ok = 1.0
    if cx.rank == cx.world - 1:
        g = cx.b.Falcon(hp, n_ctx=128, n_batch=16)
        g.set_random(shapes, Q4_K, seed=4321)
        want = [g.eval(prompt, 0, 0, all_logits=True)] + [g.eval(np.array([100 + i], np.int32), 16 + i, 0) for i in range(4)]
        wt = g.generate_greedy(77, 20, 12, 0)
        ok = float(all(np.array_equal(a, c) for a, c in zip(outs, want)) and np.array_equal(toks, wt))
        g.free()
    f.free()
    return {"bit_identical": bool(cx.sum_over_ranks([ok])[0] == cx.world), "model": hp,
            "checked": "16-token prompt (all logits) + 4 decode evals + 12 greedy tokens generated through the ring, last rank vs 1-rank engine"}


def dump_outputs(out_dir, arrays):
    """DIR/<name>.npy in float32, so that two builds run with the same arguments can be compared output for output (the inputs are
    seeded); the arrays here are a few hundred KB at most"""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="headline", choices=["headline", "1", "2", "3", "4", "5"])
    ap.add_argument("--no-extras", action="store_true", help="only the selected config (skip the other BASELINE configs and the CPU baseline)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--layers", type=int, default=0, help="debug: fewer layers than the real model (the result is then NOT a valid bench value)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy "
                                                          "(float32): the logits of a decode or prompt config, the result column of config 1")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (world > 1 or args.impl != "b200"):
        ap.error("--dump-outputs needs a single-GPU run of --impl b200")
    warmup = max(args.warmup, 3)
    sel = args.config
    dsel = sel if sel in DECODE_CONFIGS else "headline"
    model, wtype, n_ctx, pos0, metric = DECODE_CONFIGS[dsel]
    rope = 129 if pos0 == 0 else n_ctx               # falcon_main sets n_max_real_ctx = prompt + n_predict (falcon_main.cpp:835-836)
    config = {"workload": WORKLOAD[sel] + (", STRICT AUTOREGRESSIVE (device-side arg-max feeds the next step)" if world > 1 and sel != "3" else ""),
              "baseline_config": sel, "model_shape": MODELS[model], "weights": TYPE_NAME[wtype], "n_ctx": n_ctx, "n_ctx_rope": rope,
              "l2": "inputs (the weights streamed per step, GBs) are far larger than the 126 MB L2; no explicit flush needed",
              "parallelism": ("layer-range pipeline x%d (contiguous layers per GPU balanced by bytes, ncclSend/ncclRecv of the residual per boundary, "
                              "sampled id last rank -> rank 0)" % world) if world > 1 else "single GPU"}

    if args.impl == "reference":
        if rank != 0:
            return
        if sel == "1":
            r, _, _, _ = reference_cpu_matvec()
            line = {"impl": "reference", "metric": "q4_0_4096x4096_matvec_us", "value": r["us_per_call"], "unit": "us", "higher_is_better": False,
                    "ms_per_step": r["us_per_call"] / 1e3, "cpu_baseline": {"value": r["us_per_call"], "unit": "us", "cores": r["cores"], "kind": r["kind"],
                                                                           "sample": "%d rotating Q4_0 4096x4096 matrices x 8 passes through ggml_graph_compute" % r["n_mats"]}}
            steps_run = args.steps
        else:
            steps_run = max(1, min(args.steps, 32))
            r = reference_cpu_decode(model, wtype, steps=steps_run, warmup=min(warmup, 3), n_ctx_rope=rope)
            line = {"impl": "reference", "metric": metric, "value": r["value"], "unit": "tok/s", "higher_is_better": True, "ms_per_step": r["ms_per_step"],
                    "extrapolated": r["extrapolated"],
                    "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}}
        line.update({"n_gpus": args.gpus, "steps": steps_run, "warmup": min(warmup, 3) if sel != "1" else 0, "scaling": "strong", "vs_baseline": None,
                     "dtype": "int8 x int4 block dots, fp32 accumulate (CPU, AVX2)", "data": "synthetic", "config": config,
                     "e2e": {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        print(json.dumps(line))
        return

    cx = Ctx()
    hp = dict(MODELS[model])
    if args.layers:
        hp["n_layer"] = args.layers
        config["INVALID_debug_layers"] = args.layers
    peak, tf_peak, peak_src = peaks()
    extras = not args.no_extras and not args.layers
    out_extra = {}

    if sel == "1":
        r = matvec_leg(cx, reps=args.steps, cpu=not args.no_cpu_baseline) if cx.rank == 0 else None
        if cx.rank == 0:
            y = r.pop("_output")
            if args.dump_outputs:
                dump_outputs(args.dump_outputs, {"y": y})
            print(json.dumps({"metric": "q4_0_4096x4096_matvec_us", "value": r["gpu"]["us_per_call"], "unit": "us", "n_gpus": args.gpus, "steps": args.steps, "warmup": warmup,
                              "ms_per_step": r["gpu"]["us_per_call"] / 1e3, "higher_is_better": False, "scaling": "weak", "vs_baseline": None, "dtype": "int8 x int4 block dots (dp4a)",
                              "data": "synthetic", "config": config, "e2e": {"value": r["gpu"]["e2e_us_per_call"], "unit": "us", "h2d_bytes_per_step": 4096 * 4, "d2h_bytes_per_step": 4096 * 4},
                              "gpu_launches": args.steps * r["n_mats"], "roofline": {"bound": "hbm", "achieved": r["gpu"]["GBs"], "peak": peak, "unit": "GB/s", "frac": r["gpu"]["frac_of_hbm_peak"], "traffic": None},
                              "cpu_baseline": {"value": r["cpu"]["us_per_call"], "unit": "us", "cores": r["cpu"]["cores"], "kind": r["cpu"]["kind"], "sample": "32 rotating matrices x 8 passes"} if r["cpu"] else None,
                              "detail": r}))
        return

    n_batch = 512 if (sel in ("headline", "3") and extras or sel == "3") else 1
    sampler = ClockSampler(cx.local_rank)
    f = cx.make_model(hp, wtype, n_ctx, n_batch)
    d = decode_leg(cx, f, hp, wtype, args.steps, warmup, pos0, rope, keep_output=bool(args.dump_outputs) and sel != "3")
    clocks = sampler.stop()
    prompt, prompt_output = None, None
    if n_batch >= 512:
        prompt = prompt_leg(cx, f, hp)
        prompt_output = prompt.pop("_output", None)
    f.free()
    decode_output = d.pop("_output", None)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits": prompt_output if sel == "3" else decode_output})
    parity = pipeline_parity(cx) if cx.world > 1 else None

    if extras and sel == "headline":
        steps_x = max(8, min(args.steps, 64))
        for key in ("2", "4", "5"):
            m2, wt2, nctx2, pos2, metric2 = DECODE_CONFIGS[key]
            if key == "2" and cx.world > 1:
                continue                                  # BASELINE runs Falcon-7B on one GPU
            try:
                f2 = cx.make_model(MODELS[m2], wt2, nctx2, 1)
                r2 = decode_leg(cx, f2, MODELS[m2], wt2, 128 if key == "2" and cx.world == 1 else steps_x, warmup, pos2, 129 if pos2 == 0 else nctx2, with_kernel_probe=False)
                f2.free()
                r2.pop("_probe", None)
                r2.update(metric=metric2, workload=WORKLOAD[key], steps=128 if key == "2" and cx.world == 1 else steps_x)
                out_extra["cfg" + key] = r2
            except Exception as ex:                       # an extra config must never take the headline down
                out_extra["cfg" + key] = {"error": repr(ex)}
        if cx.rank == 0:
            try:
                out_extra["cfg1"] = matvec_leg(cx, cpu=not args.no_cpu_baseline)
                out_extra["cfg1"].pop("_output", None)
            except Exception as ex:
                out_extra["cfg1"] = {"error": repr(ex)}
    if cx.rank != 0:
        return

    mv_ms, mv_n, mv_bytes = d.pop("_probe")
    traffic, traffic_src = None, None
    for tname in ("r2_traffic.json", "r1_traffic.json"):          # ncu launch list of this command, summarised by tools/launch_list.py
        try:
            with open(os.path.join(ROOT, "profiles", tname)) as tf:
                tj = json.load(tf)
            traffic, traffic_src = float(tj["dram_bytes_per_matvec_launch"]), tj.get("source", tname)
            break
        except Exception:
            pass
    ach = mv_bytes / (mv_ms / 1e3) / 1e9
    if sel == "3":
        value, unit, metric_name, ms_step = prompt["tok_s"], "tok/s", "falcon40b_q4_k_prompt_tokens_per_s", prompt["seconds"] * 1e3 / 4
        e2e = {"value": prompt["tok_s"], "unit": "tok/s", "h2d_bytes_per_step": 512 * 4, "d2h_bytes_per_step": hp["n_vocab"] * 4, "api": "b200_falcon_eval (512 host token ids in, host logits out)"}
    else:
        value, unit, metric_name, ms_step = d["tok_s"], "tok/s", metric, d["ms_per_step"]
        e2e = {"value": d["e2e_tok_s"], "unit": "tok/s", "h2d_bytes_per_step": 8, "d2h_bytes_per_step": hp["n_vocab"] * 4, "ms_per_step": d["e2e_ms_per_step"],
               "api": "b200_falcon_eval (host token id in, host logits out)" + ("; last rank's host arg-max broadcast before the next step" if world > 1 else "")}
    out = {"metric": metric_name, "value": value, "unit": unit, "n_gpus": args.gpus, "steps": args.steps, "warmup": warmup, "ms_per_step": ms_step,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None,        # one token stream through the whole model: total work is fixed as GPUs are added
           "dtype": "int8 x int4 block dots (dp4a), fp32 accumulate; f32 KV/attention", "data": "synthetic", "config": config, "e2e": e2e,
           "gpu_launches": d["gpu_launches"], "clocks": clocks,
           "step_roofline_frac": d["step_frac"],
           "roofline": {"bound": "hbm", "kernel": "mmv_fast_kernel<%s> (register-resident fused dequantise + int8 dot mat-vec)" % TYPE_NAME[wtype], "achieved": ach, "peak": peak,
                        "unit": "GB/s", "frac": ach / peak, "peak_source": peak_src, "traffic": traffic,
                        "traffic_source": ("ncu dram__bytes_read.sum + dram__bytes_write.sum per mat-vec launch: " + traffic_src) if traffic else None,
                        "launches_timed": int(mv_n), "avg_launch_us": mv_ms * 1e3 / max(mv_n, 1), "algorithmic_bytes_per_launch": mv_bytes / max(mv_n, 1),
                        "how": "all resident mat-vecs of rank 0 (4 per layer + lm_head) launched back to back x3 on the eval stream, CUDA events around the region; "
                               "each launch reads a different matrix, one pass >> L2",
                        "step_frac": d["step_frac"], "step_achieved_GBs": d["step_achieved_GBs"], "step_bytes": d["step_bytes"], "step_roofline_tok_s": d["roofline_tok_s"],
                        "step_frac_what": "whole decode step: (weight bytes + KV bytes at the mid position) x tok/s against the measured HBM peak -- the north-star fraction"},
           "decode": {k: v for k, v in d.items()},
           "wall_ms_per_step": d["wall_ms_per_step"]}
    if world > 1:
        out["pipelined_tok_s"] = d["pipelined_tok_s"]
        out["autoregressive_tok_s"] = d["autoregressive_tok_s"]
        out["pipeline_parity"] = parity
        config["decode_dependency"] = ("value = strict autoregressive single stream, timed on the device; pipelined_tok_s = teacher-forced ids "
                                       "(consecutive tokens overlap across stages), reported for reference only")
    if prompt is not None:
        out["prompt"] = prompt
    if out_extra:
        out["configs"] = out_extra
    if world == 1 and extras and not args.no_cpu_baseline and sel in DECODE_CONFIGS:
        mf = None
        try:
            mf = FullModelFile(model, wtype)
            try:
                out["e2e_dropin"] = dropin_decode(cx, mf, steps=max(8, min(args.steps, 64)), warmup=3, n_ctx_rope=rope)
            except Exception as ex:
                out["e2e_dropin"] = {"error": repr(ex)}
            r = reference_cpu_decode(model, wtype, steps=8, warmup=2, n_ctx_rope=rope, mf=mf)
            out["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "extrapolated")}
        except Exception as ex:       # the baseline is reporting only; never let it take the GPU number down
            out["cpu_baseline"] = {"value": None, "unit": "tok/s", "cores": 0, "kind": "reference", "sample": "failed: %r" % (ex,)}
        finally:
            if mf is not None:
                mf.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
