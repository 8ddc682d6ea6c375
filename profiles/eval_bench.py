#!/usr/bin/env python
"""Evaluation (held-out validation) costs at B = 4096, C = 20 884, in the tf32 and bf16 modes.  Prints one JSON line:

* the fused 512 -> C BCE GEMM, loss only (cc_gemm_bce_tc_ex with dz = NULL) against the dlogit-writing training call;
* cc_softmax_kl_loss against cc_softmax_kl_fwd_bwd_metrics over 4096 rows of M-hat, with the algorithmic bytes
  (8 C per row read by the loss-only kernel: logits + target; 12 C by the training kernel, which also writes dlogits)
  over kernel time against the measured HBM rate of 6546.9 GB/s;
* ``evaluate`` throughput (cubes/s, noise kernel included) against the train step's.

Kernel times: CUDA events around single launches, L2 overwritten (256 MB) before each launch, median of ``REPS``.
Card name and power limit are read in the same run.

    python profiles/eval_bench.py > profiles/eval_bench.json
"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from cubecobrarecommender_b200 import _lib, graph as G  # noqa: E402
from cubecobrarecommender_b200.ml import engine as E, generator as GEN, model as M, tensorcore as TC, train as T  # noqa: E402
from cubecobrarecommender_b200.sparse import CubeCSR  # noqa: E402
from cubecobrarecommender_b200.synth import synth_cubes_csr  # noqa: E402

B, C, K = 4096, 20884, 512
CPAD = (C + 127) // 128 * 128
HBM_GBS = 6546.9
REPS = int(os.environ.get("EVAL_BENCH_REPS", 20))
call, ptr, stream_ptr = _lib.call, _lib.ptr, _lib.stream_ptr
dev = torch.device("cuda", 0)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, sm = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": sm}
    except Exception as e:           # the timings stand without it, but say why it is missing
        return {"name": torch.cuda.get_device_name(0), "power_limit": None, "error": repr(e)}


def timed(fn):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(REPS):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)) * 1e3, float(min(ts)) * 1e3          # microseconds


def bce_pass(precision):
    g = torch.Generator(device=dev).manual_seed(1)
    dt = torch.bfloat16 if precision == "bf16" else torch.float32
    a = torch.relu(torch.randn(B, K, device=dev, generator=g)).to(dt)
    w_pad = (torch.randn(K, CPAD, device=dev, generator=g) * 0.05).to(dt)   # rows padded to 16 bytes, as the engine keeps them
    if precision == "tf32":
        call("cc_round_tf32", ptr(a), ptr(a), a.numel(), stream_ptr())
        call("cc_round_tf32", ptr(w_pad), ptr(w_pad), w_pad.numel(), stream_ptr())
    w = w_pad[:, :C]
    bias = torch.randn(C, device=dev, generator=g) * 0.1 - 4
    yb = torch.randint(-2 ** 31, 2 ** 31 - 1, (B, CPAD // 32), dtype=torch.int32, device=dev, generator=g) \
        & torch.randint(-2 ** 31, 2 ** 31 - 1, (B, CPAD // 32), dtype=torch.int32, device=dev, generator=g)
    n = TC.bce_partial_count(B, CPAD)
    part, acc = (torch.zeros(n, dtype=torch.float64, device=dev) for _ in range(2))
    dz = torch.zeros(B, CPAD, dtype=dt, device=dev)
    dbias = torch.zeros(C, device=dev)
    train = timed(lambda: TC.gemm_bce(a, w, bias, yb, float(B * C), dz, part, precision=precision, dbias=dbias, acc_partial=acc))
    p_train = part.clone()
    loss = timed(lambda: TC.gemm_bce(a, w, bias, yb, float(B * C), None, part, precision=precision, acc_partial=acc,
                                     lddz=CPAD))
    return {"train_dlogits_us": train[0], "loss_only_us": loss[0], "train_min_us": train[1], "loss_only_min_us": loss[1],
            "speedup": train[0] / loss[0], "partials_bit_equal": bool(torch.equal(p_train, part)),
            "dlogit_bytes_not_written": B * CPAD * (2 if precision == "bf16" else 4)}


def kl_pass(mhat, fast=1):
    g = torch.Generator(device=dev).manual_seed(2)
    z = torch.zeros(B, CPAD, device=dev)
    z[:, :C] = torch.randn(B, C, device=dev, generator=g) * 2
    trow = torch.randint(0, C, (B,), dtype=torch.int32, device=dev, generator=g)
    tlogt = torch.zeros(C, dtype=torch.float64, device=dev)
    am = torch.zeros(C, dtype=torch.int32, device=dev)
    call("cc_kl_target_table", ptr(mhat), mhat.stride(0), C, C, ptr(tlogt), stream_ptr())
    call("cc_kl_target_argmax", ptr(mhat), mhat.stride(0), C, C, ptr(am), stream_ptr())
    loss = torch.zeros(B, dtype=torch.float64, device=dev); hit = torch.zeros(B, dtype=torch.int32, device=dev)
    dz = torch.empty_like(z); dbias = torch.zeros(C, device=dev)
    train = timed(lambda: call("cc_softmax_kl_fwd_bwd_metrics", ptr(z), z.stride(0), ptr(mhat), mhat.stride(0), ptr(trow), B,
                               C, CPAD, 1e-4, ptr(dz), dz.stride(0), ptr(loss), fast, ptr(dbias), None, 0, ptr(tlogt),
                               ptr(am), ptr(hit), stream_ptr()))
    ref = loss.clone()
    ev = timed(lambda: call("cc_softmax_kl_loss", ptr(z), z.stride(0), ptr(mhat), mhat.stride(0), ptr(trow), B, C, CPAD,
                            ptr(tlogt), ptr(am), ptr(loss), ptr(hit), fast, stream_ptr()))
    b_train, b_loss = B * C * 12, B * C * 8
    return {"train_us": train[0], "loss_only_us": ev[0], "train_min_us": train[1], "loss_only_min_us": ev[1],
            "train_GBps": b_train / train[0] / 1e3, "loss_only_GBps": b_loss / ev[0] / 1e3,
            "train_frac_of_hbm": b_train / train[0] / 1e3 / HBM_GBS, "loss_only_frac_of_hbm": b_loss / ev[0] / 1e3 / HBM_GBS,
            "row_loss_bit_equal": bool(torch.equal(ref, loss)), "bytes_per_row": {"train": 12 * C, "loss_only": 8 * C}}


def throughput(precision, csr, mhat):
    gen = GEN.DataGenerator(mhat, csr, batch_size=B, noise=0.2, seed=1)
    model = M.CC_Recommender(C, device=dev, seed=0, precision=precision)
    eng = E.DAEEngine(model, mhat, batch=B, reg_rows=B, reg=0.1, max_cube_size=max(csr.max_size, 1))
    steps = 10
    for i in range(3):
        eng.sample_batch(gen.indptr, gen.indices_dev, gen.batch_ids(i % len(gen)), gen.alias_prob, gen.alias_idx, seed=1)
        eng.train_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        eng.sample_batch(gen.indptr, gen.indices_dev, gen.batch_ids(i % len(gen)), gen.alias_prob, gen.alias_idx, seed=1)
        eng.train_step()
    torch.cuda.synchronize()
    step_ms = (time.perf_counter() - t0) * 1e3 / steps
    T.evaluate(model, gen, 0.1, engine=eng)                       # warm-up (and the fixed validation draws)
    ts = []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        T.evaluate(model, gen, 0.1, engine=eng)                   # ends in a host read of the sums
        ts.append(time.perf_counter() - t0)
    ev_s = float(np.median(ts))
    return {"train_step_ms": step_ms, "train_cubes_per_s": B / step_ms * 1e3, "evaluate_cubes": gen.N_cubes,
            "evaluate_ms": ev_s * 1e3, "evaluate_ms_per_batch": ev_s * 1e3 / (gen.N_cubes / B),
            "evaluate_cubes_per_s": gen.N_cubes / ev_s, "eval_batch_over_train_step": ev_s * 1e3 / (gen.N_cubes / B) / step_ms}


def main():
    torch.cuda.set_device(0)
    info = card()
    ip, ix = synth_cubes_csr(4 * B, C, seed=3)
    csr = CubeCSR(ip, ix, C)
    mhat = G.build_graph(csr, dev, want_m64=False).mhat
    out = {"card": info, "B": B, "C": C, "reps": REPS, "l2": "256 MB overwritten before every timed launch",
           "hbm_GBps_reference": HBM_GBS}
    out["kl"] = kl_pass(mhat)
    for precision in ("tf32", "bf16"):
        out[precision] = {"bce": bce_pass(precision), "throughput": throughput(precision, csr, mhat)}
    out["card_after"] = card()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
