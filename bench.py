#!/usr/bin/env python
"""Benchmark of the hot path: the regularised-DAE train step (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--precision P] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the train path over one batch of 4096 synthetic cubes per GPU:
noise function F + reg-row draw, both towers forward, BCE + 0.1*KLD, backward, (gradient
all_reduce when N > 1), TF-style Adam over all 32.6 M parameters.  Prints ONE JSON line.

* `value`  : cubes/s with cubes (CSR), M-hat and weights resident in HBM, CUDA-event timed.
* `e2e`    : the same step driven from HOST buffers through the package's host-fed trainer path
             (ml.engine.HostBatchStream): the batch's CSR is copied from pinned host memory every step
             (double-buffered on a copy stream) and every step's loss is copied back and read on the host.
* `roofline`: the dominant kernel (the 512<->C GEMM passes), timed with CUDA events inside the
             timed region, against MEASURED_PEAKS.json.
* `cpu_baseline`: the oracle port of the reference CPU path (reference DataGenerator restated
             + torch-CPU restatement of the Keras step) on a bounded sample, rank 0, N=1.
* `--impl reference`: that CPU path as its own arm (the reference is Python/TensorFlow 2.5.2,
             TensorFlow is not installable here, so the arm is the oracle port, kind "port").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

# torch.distributed.run exports OMP_NUM_THREADS=1 to its workers unless the variable is already set; the CPU arm is meant to
# use every host core it can, so the launcher's default is undone BEFORE numpy / torch load their OpenMP runtimes
_LAUNCHER_OMP = os.environ.get("OMP_NUM_THREADS")
if "reference" in sys.argv[1:] and "TORCHELASTIC_RUN_ID" in os.environ:
    for _k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        os.environ.pop(_k, None)

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

METRIC = "dae_train_cubes_per_s"
UNIT = "cubes/s"


def load_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], bf16_burst=p["bf16_tflops"], bf16_sustained=p["bf16_tflops_sustained"],
                    source="measured")
    return dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback")


def ncu_traffic(precision, kernel=None):
    """(dram__bytes_read.sum + dram__bytes_write.sum per launch, the capture it comes from) of a kernel, from the
    committed `ncu --set full` capture of this workload -- profiles/roofline_traffic.json, written by
    profiles/summarize_ncu.py from the raw capture it names; (None, None) when absent."""
    path = os.path.join(REPO, "profiles", "roofline_traffic.json")
    try:
        t = json.load(open(path))
        e = t.get(kernel or f"gemm_tc_kernel<{precision}>", {})
        return e.get("dram_bytes_per_launch"), e.get("source")
    except Exception:
        return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md).  The poller is
    started before warm-up (nvidia-smi needs a few hundred ms before its first sample); only samples whose
    timestamp falls between mark_begin() and mark_end() are reported."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []
        self.t0 = self.t1 = self.t2 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "10", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def mark_load_end(self):
        self.t2 = time.time()

    def samples_in_timed_region(self):
        """Samples with a timestamp inside [mark_begin, mark_end] so far (the poller may still be running)."""
        import datetime
        n = 0
        for ln in list(self.lines):
            try:
                ts = datetime.datetime.strptime(ln.split(",")[0].strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except ValueError:
                continue
            n += 1 if (self.t0 is not None and self.t1 is not None and self.t0 <= ts <= self.t1) else 0
        return n

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.thread.join(timeout=2)
        import datetime
        rows = []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(f[2]), float(f[3]), float(f[4]), f[5:9]))
            except ValueError:
                continue
        inside = [r for r in rows if self.t0 is not None and self.t1 is not None and self.t0 <= r[0] <= self.t1]
        window = "timed region"
        if len(inside) < 3 and self.t0 is not None and self.t2 is not None:
            # a region of a few sampling periods: add the instrumented pass behind it (the same K steps, the same load)
            inside = [r for r in rows if self.t0 <= r[0] <= self.t2]
            window = "timed region + the instrumented pass of the same K steps"
        if not inside:      # still nothing: everything sampled since the poller started
            inside, window = rows, "whole run"
        reasons = set()
        for r in inside:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm = [r[1] for r in inside]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(r[2] for r in inside) if inside else None,
                "power_w_max": max(r[3] for r in inside) if inside else None, "samples": len(inside), "window": window,
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------------ CPU comparator
REF_BATCH = 4096      # cubes per CPU step = the native arm's batch (halved only if the run would not fit REF_BUDGET_S;
                      # the CPU path gets faster with the batch -- 126 / 182 / 320 cubes/s at 64 / 256 / 1024 on 8 cores)


def host_threads():
    """Host threads this process may use (cgroup / affinity aware)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def use_all_host_threads():
    """Give torch's intra-op pool (and, through threadpoolctl, NumPy's BLAS) every host thread; returns the count."""
    import torch
    n = host_threads()
    torch.set_num_threads(n)
    try:
        import threadpoolctl
        threadpoolctl.threadpool_limits(limits=n)
    except Exception:
        pass
    return torch.get_num_threads()


REF_BUDGET_S = 170.0  # the whole --steps K --warmup W run of the CPU arm should end within a few minutes


def cpu_reference(num_cards, steps, warmup, batch=REF_BATCH, num_cubes=REF_BATCH, mhat64=None, log=None,
                  budget_s=None):
    """Oracle port of the reference CPU train path: DataGenerator (restated from
    src/ml/generator.py) + torch-CPU restatement of the Keras step.  Returns cubes/s.

    ``budget_s``: if the (warmup + steps) steps at ``batch`` cubes would take longer than this, the per-step sample is
    halved (down to the reference's default batch_size of 64) until they fit; the estimate comes from one calibration
    step at 64 cubes (after a cold one) and the measured scaling of the CPU path with the batch (cubes/s ~ batch^(1/3))."""
    import torch
    from cubecobrarecommender_b200.workload import TRAIN_STEP, make_cubes
    from oracle import dae as od, graph as og, noise as on
    use_all_host_threads()
    t0 = time.time()
    csr = make_cubes(num_cubes, num_cards, cfg=TRAIN_STEP["cfg"])
    dense = csr.to_dense(np.float64)
    if mhat64 is None:
        x32 = torch.from_numpy(dense.astype(np.float32))
        cnt = (x32.t() @ x32).double().numpy()           # exact: counts < 2^24
        mhat64 = og.m_hat(og.adjacency_from_counts(cnt))
        del cnt, x32
    np.random.seed(0)
    model = od.TorchDAE(od.init_params(num_cards, seed=0))
    if budget_s is not None and batch > 64:
        cal = on.DataGenerator(mhat64, dense, batch_size=64, noise=TRAIN_STEP["noise"])
        for _ in range(2):                                 # the second step is the estimate (the first one is cold)
            tc = time.perf_counter()
            (x, xr), (y, yr) = cal[0]
            model.train_step(torch.from_numpy(x.astype(np.float32)), torch.from_numpy(y.astype(np.float32)),
                             torch.from_numpy(np.argmax(xr, 1)), torch.from_numpy(yr.astype(np.float32)), TRAIN_STEP["reg"])
            cps64 = 64 / (time.perf_counter() - tc)
        while batch > 64 and (warmup + steps) * batch / (cps64 * (batch / 64.0) ** (1.0 / 3.0)) > budget_s:
            batch //= 2
        if log:
            log(f"cpu reference: {cps64:.0f} cubes/s at 64 cubes per step -> {batch} cubes per step for {warmup}+{steps} steps")
    gen = on.DataGenerator(mhat64, dense, batch_size=batch, noise=TRAIN_STEP["noise"])
    if log:
        log(f"cpu reference setup {time.time() - t0:.1f}s, threads={torch.get_num_threads()}")
    t_gen = t_model = 0.0
    for i in range(warmup + steps):
        a = time.perf_counter()
        (x, xr), (y, yr) = gen[i % len(gen)]
        b = time.perf_counter()
        rows = torch.from_numpy(np.argmax(xr, 1))
        model.train_step(torch.from_numpy(x.astype(np.float32)), torch.from_numpy(y.astype(np.float32)), rows,
                         torch.from_numpy(yr.astype(np.float32)), TRAIN_STEP["reg"])
        c = time.perf_counter()
        if i >= warmup:
            t_gen += b - a; t_model += c - b
    total = t_gen + t_model
    return dict(value=batch * steps / total, seconds=total, gen_seconds=t_gen, model_seconds=t_model,
                cores=torch.get_num_threads(), batch=batch)


def workload_config(world, batch, reg_rows, global_reg_rows, reg_mode, scaling):
    """The `config` object of the JSON line -- the SAME function for both arms, so that the reference arm is quoted on
    the native arm's configuration (precision is the line's `dtype`, not part of the workload)."""
    from cubecobrarecommender_b200.workload import TRAIN_STEP as W, train_step_flops
    C = W["num_cards"]
    return {"workload": W["workload"], "num_cards": C, "batch_per_gpu": batch, "reg_rows_per_gpu": reg_rows,
            "global_batch": batch * world, "dims": "C-512-256-128-64-128-256-512-C x2 decoders",
            "reg": W["reg"], "noise": W["noise"], "parallelism": f"dp{world}", "scaling": scaling,
            "reg_mode": "sampled rows (reference generator.py:47-51)" if reg_mode == "sampled"
                        else f"full identity: all {C} rows of I, {global_reg_rows // world} per rank",
            "l2": "working set per step (weights+Adam 0.52 GB, logits 0.69 GB, M-hat rows 0.34 GB) exceeds the 126 MB L2; no flush needed",
            "algorithmic_tflop_per_step": train_step_flops(batch, reg_rows, C) / 1e12}


def per_gpu_sizes(args, world, rank=0):
    """(B, R, global_R) per rank: weak scaling keeps 4096 cubes + 4096 reg rows per GPU, strong scaling keeps the GLOBAL
    batch at 4096 (BASELINE configs[2]); --reg-mode full shards all C rows of I over the ranks."""
    from cubecobrarecommender_b200.ml.engine import full_identity_shard
    from cubecobrarecommender_b200.workload import TRAIN_STEP as W
    B, R = W["batch"], W["reg_rows"]
    if args.scaling == "strong":
        if B % world or R % world:
            raise SystemExit(f"--scaling strong: {B} cubes do not divide over {world} ranks")
        B, R = B // world, R // world
    global_R = R * world
    if args.reg_mode == "full":
        lo_r, hi_r = full_identity_shard(W["num_cards"], rank, world)
        R, global_R = hi_r - lo_r, W["num_cards"]
    return B, R, global_R


def run_reference(args, rank, world):
    """The CPU arm: rank 0 alone (under torchrun the other ranks exit 0), every host thread, the native arm's config.
    One step = one batch of the native arm's size (4096 cubes; halved only when K+W such steps would overrun
    REF_BUDGET_S, and then the line's config says so)."""
    if rank != 0:
        return
    from cubecobrarecommender_b200.workload import TRAIN_STEP
    log = lambda m: print(m, file=sys.stderr, flush=True)
    threads = use_all_host_threads()
    log(f"cpu reference: {threads} torch threads (host threads available {host_threads()}, launcher OMP_NUM_THREADS="
        f"{_LAUNCHER_OMP!r})")
    B = TRAIN_STEP["batch"]       # the CPU arm is one process: it steps one GPU's share (weak) = the global batch (strong)
    r = cpu_reference(TRAIN_STEP["num_cards"], args.steps, args.warmup, batch=B, num_cubes=max(B, REF_BATCH), log=log,
                      budget_s=REF_BUDGET_S)
    sample = (f"{args.steps} steps x {r['batch']} cubes + {r['batch']} reg rows"
              + ("" if r["batch"] == B else f" (a bounded sample of the {B}-cube batch)")
              + f", C={TRAIN_STEP['num_cards']}; generator {r['gen_seconds']:.2f}s + model {r['model_seconds']:.2f}s; "
                f"{r['cores']} threads")
    cb, cr, cgr = per_gpu_sizes(args, args.gpus)
    shrink = r["batch"] / float(B)                          # 1.0 unless the budget forced a smaller CPU step
    cfg = workload_config(args.gpus, int(cb * shrink), int(cr * shrink), int(cgr * shrink), args.reg_mode, args.scaling)
    if args.gpus > 1:
        cfg["note"] = ("CPU arm: rank 0's host cores only, stepping " + ("the global batch" if args.scaling == "strong"
                       else "one GPU's share of the global batch"))
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * r["seconds"] / args.steps,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": sample,
                         "note": "oracle port of the reference CPU path (reference DataGenerator restated + torch-CPU "
                                 "restatement of the Keras step; TensorFlow 2.5.2 is not installable)"},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------ extras
def measure_extras(dev, peaks, log):
    """The other two sub-metrics BASELINE.json names, on one GPU: the co-occurrence graph build
    (configs[0]: 20k cubes x 21k cards) and batched top-50 ML recommendation (configs[3])."""
    import torch
    from cubecobrarecommender_b200 import _lib, graph as G
    from cubecobrarecommender_b200.ml import inference as INF, model as M
    from cubecobrarecommender_b200.workload import make_cubes
    from oracle import dae as od, graph as og
    out = {}
    # ---------------- graph build: K = 20 000 cubes, C = 21 000 cards ----------------
    K, C = 20000, 21000
    t0 = time.time()
    csr = make_cubes(K, C, cfg=1)
    log(f"extras: {K} synthetic cubes in {time.time() - t0:.1f}s")
    indptr, indices = G.upload_csr(csr, dev)
    lib = _lib.load()
    bits = torch.empty((lib.cc_bits_words(K), lib.cc_bits_cpad(C)), dtype=torch.int32, device=dev)
    ws = torch.empty(lib.cc_cooc_tc_workspace_bytes(K, C), dtype=torch.uint8, device=dev)
    counts = torch.empty((C, C), dtype=torch.int32, device=dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    times = {"tensor": [], "popcount": []}
    for method in ("popcount", "tensor"):          # "tensor" (tcgen05 kind::i8) last: it is the product path
        for it in range(3):
            ev[0].record()
            G.count_cooccurrence(indptr, indices, K, C, counts=counts, bits=bits, workspace=ws, method=method)
            ev[1].record()
            gr = G.normalise(counts)
            ev[2].record()
            torch.cuda.synchronize()
            times[method].append((ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])))
            del gr
    t_cnt, t_norm = min(t[0] for t in times["tensor"]), min(t[1] for t in times["tensor"])
    t_cnt_popc = min(t[0] for t in times["popcount"])
    algo_bytes = K * C / 8 + 4.0 * C * C + 4.0 * C * C + 8.0 * C * C          # SURVEY.md 8d config 1a: 7.11 GB
    pair_words = C * (C + 1) / 2 * (K / 32.0)                                  # AND+POPC word pairs (upper triangle)
    t1 = time.time()
    m_host = G.create_adjacency_matrix_host(csr)
    t_host = time.time() - t1
    del m_host
    # CPU comparator: line-by-line restatement of utils.create_adjacency_matrix on a cube subsample;
    # its cost is linear in nnz (SURVEY.md 3.1), so the full build is extrapolated by nnz
    ksub = 120
    sub = csr.rows(np.arange(ksub)).to_dense()
    t2 = time.time()
    og.create_adjacency_matrix_loop(sub)
    t_cpu_sub = time.time() - t2
    nnz_ratio = float(csr.indptr[-1]) / float(csr.indptr[ksub])
    out["graph_build"] = {
        "workload": f"create_mtx: K={K} cubes x C={C} cards, nnz={int(csr.indptr[-1])}",
        "count_ms": t_cnt, "count_kernel": "expand_cubes_u8 + gemm_tc_kernel<u8, kind::i8> (X^T X, upper triangle mirrored)",
        "count_tensor_top_per_s": 2.0 * K * C * C / (t_cnt * 1e-3) / 1e12,
        "count_popcount_ms": t_cnt_popc, "normalise_ms": t_norm, "device_seconds": (t_cnt + t_norm) / 1e3,
        "e2e_host_seconds": t_host, "e2e_note": "CSR H2D + kernels + 3.5 GB float64 M D2H through cc_create_adjacency_matrix_host",
        "roofline": {"kernel": "count (tcgen05 kind::i8) + row_normalise", "bound": "hbm", "achieved": algo_bytes / ((t_cnt + t_norm) * 1e-3) / 1e9,
                     "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": algo_bytes / ((t_cnt + t_norm) * 1e-3) / 1e9 / peaks["hbm_gbs"],
                     "traffic": None,
                     "note": "algorithmic bytes of SURVEY.md 8d (7.11 GB) over count + normalise; the count itself is a "
                             "2*K*C^2 contraction (tensor-bound at this K), the normalise pass is the HBM-bound part",
                     "normalise_GBps": 16.0 * C * C / (t_norm * 1e-3) / 1e9,
                     "popcount_kernel_word_pairs_per_s": pair_words / (t_cnt_popc * 1e-3)},
        "cpu_baseline": {"seconds_extrapolated": t_cpu_sub * nnz_ratio, "cores": 1, "kind": "port",
                         "sample": f"create_adjacency_matrix loop restatement on {ksub} cubes x {C} cards: {t_cpu_sub:.1f}s, scaled by nnz x{nnz_ratio:.0f}"},
        # the count as the tensor-bound kernel it is: executed int8 multiply-adds (upper triangle only) against the
        # nominal dense int8 rate of the part (MEASURED_PEAKS.json holds no int8 figure); ncu has the IMMA pipe 89% active
        "count_roofline": {"kernel": "gemm_tc_kernel<u8, kind::i8>", "bound": "tensor",
                           "achieved": K * C * (C + 256.0) / (t_cnt * 1e-3) / 1e12, "peak": 4500.0, "unit": "TOP/s",
                           "frac": K * C * (C + 256.0) / (t_cnt * 1e-3) / 1e12 / 4500.0,
                           "peak_source": "nominal dense int8 (4.5 POP/s); executed ops = 2 * K * C * (C + 256) / 2 (symmetry)",
                           "ncu_tensor_pipe_active_pct": 89.0,
                           "ncu_source": "profiles/r02x_step_kernels_ncu_full.csv"},
    }
    # the UNMODIFIED reference function timed on this very input in the build container (the reference tree does not
    # travel to the GPU box): profiles/reference_create_adjacency_cpu.py -> the committed JSON
    try:
        ref_json = json.load(open(os.path.join(REPO, "profiles", "r02_reference_create_adjacency_cpu.json")))
        out["graph_build"]["reference_measured"] = {**ref_json, "kind": "reference",
                                                    "note": "unmodified src/non_ml/utils.py:75-92, one thread, timed in the build "
                                                            "container on the same 20 000 x 21 000 input; output equals the oracle "
                                                            "(and hence this build) bit for bit"}
    except Exception:
        pass
    # ---------------- recommend.py top-50 (configs[0], second half): graph scoring + masked select ----------------
    try:
        G.count_cooccurrence(indptr, indices, K, C, counts=counts, workspace=ws, method="tensor")
        gr = G.normalise(counts, want_m64=True, want_mhat=False, want_neg=False)
        grec = G.GraphRecommender(gr.m64)
        one = csr.rows(np.arange(1))
        many = csr.rows(np.arange(256))
        grec.recs(one, 50); grec.recs(many, 50)
        torch.cuda.synchronize()
        t5 = time.time()
        ids1, _, _ = grec.recs(one, 50); ids1 = ids1.cpu().numpy()
        t_one = time.time() - t5
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); grec.recs(many, 50); e1.record(); torch.cuda.synchronize()
        t_many = e0.elapsed_time(e1) / 1e3
        nnz_many = int(many.indptr[-1])
        m_host = gr.m64.cpu().numpy()                       # the 3.5 GB matrix the reference np.load()s per invocation
        t6 = time.time()
        ref_ids = og.simple_recs(one.to_dense()[0], m_host)[:50]
        t_cpu_one = time.time() - t6
        out["graph_recommend"] = {
            "workload": f"recommend.py top-50: sum of the cube's rows of M (float64, C={C}) + masked select",
            "one_cube_seconds": t_one, "one_cube_note": "host CSR in, ids out, M resident on the GPU",
            "batch256_cubes_per_s": 256 / t_many,
            "roofline": {"kernel": "gather_leaf_kernel (+ combine, select)", "bound": "hbm",
                         "achieved": nnz_many * C * 8.0 / t_many / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": nnz_many * C * 8.0 / t_many / 1e9 / peaks["hbm_gbs"], "traffic": None,
                         "note": "algorithmic bytes s*C*8 per cube (SURVEY.md 8d config 1b) over the whole batched call"},
            "ids_equal_reference_ranking": bool(np.array_equal(ids1[0], np.asarray(ref_ids))),
            "cpu_baseline": {"seconds": t_cpu_one, "cores": 1, "kind": "port",
                             "sample": "simple_recs restatement on one cube, M already in host memory (the reference "
                                       "also np.load()s the 3.5 GB file on every invocation)"}}
        del gr, grec, m_host
    except Exception as e:  # side measurement: never take the headline down
        out["graph_recommend"] = {"error": repr(e)}
    del counts, bits, ws
    torch.cuda.empty_cache()
    # ---------------- batched ML recommend: top-50 with in-cube masking ----------------
    C2, K2 = 20884, 100000                      # configs[3]: 100k cubes, top-50, in-cube masking
    csr2 = make_cubes(K2, C2, cfg=4).pin_memory()           # the request batch sits in pinned host memory
    model = M.CC_Recommender(C2, device=dev, seed=0, precision="tf32")
    rec = INF.MLRecommender(model, chunk=8192)
    rec.recommend(csr2, 50, copy=False)                       # warm: allocator pools, copy stream, pinned result buffers
    torch.cuda.synchronize()
    t_runs = []
    for _ in range(3):                                        # median of three host-to-host calls
        t3 = time.time()
        ids, vals, cnt = rec.recommend(csr2, 50, copy=False)  # ids / scores / counts as views of pinned host buffers
        t_runs.append(time.time() - t3)
    t_rec = float(np.median(t_runs))
    t_dev_runs = []
    for _ in range(3):                                        # (a host hiccup between two chunks shows in the event span too)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rec.recommend_device(csr2, 50)
        e1.record()
        torch.cuda.synchronize()
        t_dev_runs.append(e0.elapsed_time(e1) / 1e3)
    t_rec_dev = float(np.median(t_dev_runs))
    params = model.get_weights_dict()
    nb = 32
    dense = csr2.rows(np.arange(nb)).to_dense()
    t4 = time.time()
    tm = od.TorchDAE(params)
    with torch.no_grad():
        probs = torch.sigmoid(tm.tower(torch.from_numpy(dense.astype(np.float32)), "main")).numpy()
    for r in range(nb):
        od.rank_additions(probs[r], dense[r], 50)
    t_cpu = time.time() - t4
    out["ml_recommend"] = {
        "workload": f"ml_recommend top-50, {K2} cubes, C={C2}, in-cube masking, pinned host CSR in / host ids out "
                    f"(median of three calls after a warm-up call)",
        "recs_per_s": K2 / t_rec, "seconds": t_rec, "seconds_runs": t_runs, "device_recs_per_s": K2 / t_rec_dev, "device_seconds_runs": t_dev_runs,
        "device_note": "CUDA-event time of the same call without the final D2H of ids/scores (CSR H2D included), median of three",
        "cpu_baseline": {"value": nb / t_cpu, "unit": "cubes/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": f"{nb} cubes: torch-CPU forward + argsort walk (model load excluded)"},
    }
    # ---------------- the masked top-50 select alone (the HBM-bound half of configs[3]) ----------------
    try:
        nb_sel = 4096
        ld = (C2 + 127) // 128 * 128                         # the row stride the decoder GEMM writes
        gsel = torch.Generator(device=dev).manual_seed(4)
        logits = torch.randn((nb_sel, ld), device=dev, generator=gsel) * 3 - 4
        sub = csr2.rows(np.arange(nb_sel))
        mp, mi = G.upload_csr(sub, dev)
        res = G.topn_masked(logits[:, :C2], mp, mi, 50, sigmoid=True)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # larger than the 126 MB L2
        ts = []
        for _ in range(10):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); G.topn_masked(logits[:, :C2], mp, mi, 50, sigmoid=True, out=res); e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        t_sel = float(np.median(ts)) * 1e-3
        sel_bytes = nb_sel * (4.0 * C2 + 8 * 50 + 4) + 4.0 * int(sub.indptr[-1])   # SURVEY.md 8d config 4: 4C + 4s + out
        # the committed ncu capture ranks `cubes` cubes per launch: its DRAM bytes scale with the cube count
        sel_traffic = ncu_traffic(None, "topn_rowselect_kernel")[0]
        try:
            cap_cubes = json.load(open(os.path.join(REPO, "profiles", "roofline_traffic.json")))["topn_rowselect_kernel"]["cubes"]
            sel_traffic = int(sel_traffic * nb_sel / cap_cubes)
        except Exception:
            pass
        out["ml_recommend"]["select_roofline"] = {
            "kernel": "topn_rowselect_kernel<sigmoid> (CTA per cube, row staged in shared memory by bulk copies)",
            "bound": "hbm", "achieved": sel_bytes / t_sel / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": sel_bytes / t_sel / 1e9 / peaks["hbm_gbs"], "traffic": sel_traffic,
            "traffic_source": ncu_traffic(None, "topn_rowselect_kernel")[1],
            "launch_us": t_sel * 1e6, "cubes": nb_sel,
            "note": "one launch over 4096 logit rows, L2 flushed between launches, median of 10; traffic = ncu "
                    "dram read + write of a 2048-cube launch of the same kernel, scaled by the cube count"}
        del logits, flush
    except Exception as e:  # side measurement: never take the headline down
        out["ml_recommend"]["select_roofline"] = {"error": repr(e)}
    return out


# ------------------------------------------------------------------------------ native
def oracle_loss_check(eng, csr, batch_ids, prob, alias, indptr, indices, W, log):
    """Step-1 loss of the benchmarked configuration against the float64 oracle (oracle/dae.py) on the SAME noise output,
    regulariser rows and weights.  The engine's buffers are left holding that batch; nothing is trained."""
    import torch
    from oracle import dae as od, graph as og
    t0 = time.time()
    use_all_host_threads()
    B, R, C = eng.B, eng.R, eng.C
    eng.sample_batch(indptr, indices, batch_ids, prob, alias, W["noise"], W["noise_std"], seed=1234)
    eng.check_overflow()
    eng.forward_backward()
    got = [float(v) for v in eng.loss3.cpu().numpy()]
    xl = eng.x_len.cpu().numpy(); xi = eng.x_idx.cpu().numpy()
    x = np.zeros((B, C))
    for i in range(B):
        x[i, xi[i, :xl[i]]] = 1
    bits = eng.y_bits.cpu().numpy().view(np.uint32)
    y = ((bits[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(B, -1)[:, :C].astype(np.float64)
    rows = eng.reg_rows[:R].cpu().numpy().astype(np.int64)
    t32 = og.m_hat_rows(csr.indptr, csr.indices, C, rows).astype(np.float32).astype(np.float64)
    p64 = {k: v.astype(np.float64) for k, v in eng.model.get_weights_dict().items()}
    (tot, bce, kl), _ = od.loss_and_grads_np(p64, x, y, rows, t32, eng.reg, onehot_rows_as_gather=True)
    if eng.global_R != R or eng.global_B != B:
        raise RuntimeError("oracle_loss_check is a single-GPU check")
    rel = {"bce": abs(got[0] - bce) / bce, "kl": abs(got[1] - kl) / kl, "total": abs(got[2] - tot) / tot}
    log(f"oracle loss check: native {got[2]:.8f} vs oracle {tot:.8f} (rel {rel['total']:.2e}) in {time.time() - t0:.1f}s")
    return {"loss_rel_err": rel["total"], "bce_rel_err": rel["bce"], "kl_rel_err": rel["kl"],
            "native": {"bce": got[0], "kl": got[1], "total": got[2]}, "oracle": {"bce": bce, "kl": kl, "total": tot},
            "what": "step-1 loss on the first timed-workload batch (noise output read back) vs oracle/dae.py float64, "
                    "M-hat rows from the oracle's own counts", "seconds": time.time() - t0}


DUMP_SAMPLE = 1 << 20      # entries kept of a larger weight tensor: the three C x 512 kernels are 128 MB in full


def dump_outputs(out_dir, loss, weights, log):
    """What a caller of the train step receives from the last timed step: loss3 = [bce, kl, total] (float64) and every
    weight tensor after its Adam update (float32, Keras names with '/' -> '.'), one <name>.npy each.  A tensor of more
    than DUMP_SAMPLE entries is written as `<name>.sampled.npy`: the same DUMP_SAMPLE flat positions in every run.
    The inputs are seeded, but the bias gradients and the first layer's backward sum with float atomics, and Adam's
    m / sqrt(v) turns those rounding differences of near-zero gradients into +-lr weight steps: two runs of one build
    agree on the first step's loss and drift apart from there (on a B200 after 25 steps: loss 1e-3 relative, weights up
    to 1.1e-2), so builds are compared with a tolerance, not bit for bit."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), loss.cpu().numpy().astype(np.float64))
    total = 0
    for key, w in weights.items():
        name = key.replace("/", ".")
        if w.size > DUMP_SAMPLE:
            pick = np.sort(np.random.default_rng(0).choice(w.size, DUMP_SAMPLE, replace=False))
            w, name = w.ravel()[pick], name + ".sampled"
        np.save(os.path.join(out_dir, name + ".npy"), w.astype(np.float32))
        total += w.nbytes
    log(f"outputs of the last timed step: {len(weights) + 1} arrays, {total / 2**20:.1f} MB -> {out_dir}")


def run_native(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from cubecobrarecommender_b200 import graph as G
    from cubecobrarecommender_b200.ml import engine as E, model as M
    from cubecobrarecommender_b200.workload import TRAIN_STEP, make_cubes, train_step_flops

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl native needs a CUDA device (there is no CPU fallback)")
    # stdout carries exactly one JSON line: anything a library prints there (NCCL's version banner)
    # is diverted to stderr, and the line is written to the saved descriptor at the end
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    log = (lambda m: print(f"[bench] {m}", file=sys.stderr, flush=True)) if rank == 0 else (lambda m: None)
    W = TRAIN_STEP
    C = W["num_cards"]
    B, R, global_R = per_gpu_sizes(args, world, rank)
    t0 = time.time()
    # every rank owns its own cubes (weak scaling: per-GPU batch fixed); the graph is the
    # all_reduce of the per-rank int32 counts, so M-hat is identical everywhere
    # the clock poller starts here: nvidia-smi takes a few hundred ms to print its first sample, and the warm-up plus the
    # timed region of the default run last ~50 ms
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    csr = make_cubes(W["num_cubes"], C, cfg=W["cfg"] * 1000 + rank)
    gr = G.build_graph(csr, dev, want_m64=False, want_mhat=True, want_neg=True)
    log(f"cubes + graph ready in {time.time() - t0:.1f}s")
    prob, alias = E.alias_table(gr.neg_sampler.cpu().numpy(), dev)
    model = M.CC_Recommender(C, device=dev, seed=0, precision=args.precision)
    eng = E.DAEEngine(model, gr.mhat, batch=B, reg_rows=R, reg=W["reg"], max_cube_size=720,
                      global_batch=B * world, global_reg_rows=global_R)
    if args.reg_mode == "full":
        eng.set_full_identity_rows(rank, world)
    del gr.counts
    indptr, indices = G.upload_csr(csr, dev)
    nb = csr.num_cubes // B
    batch_ids = [torch.arange(i * B, (i + 1) * B, dtype=torch.int32, device=dev) for i in range(nb)]
    # ---- parity of the very step that is about to be timed: the first batch's noise output is read back and the float64
    #      oracle evaluates the same (x, y, r, weights); `loss_rel_err` goes into the line (rank 0, N = 1) ----
    loss_check = None
    if world == 1 and not args.no_loss_check:
        loss_check = oracle_loss_check(eng, csr, batch_ids[0], prob, alias, indptr, indices, W, log)

    def batch_args(i):
        return dict(indptr=indptr, indices=indices, batch_ids=batch_ids[i % nb], alias_prob=prob, alias_idx=alias,
                    noise=W["noise"], noise_std=W["noise_std"], seed=1234 + rank)

    def step(i):
        # one step = noise F + reg-row draw for ITS batch, forward, losses, backward, exchange, Adam.  The engine draws
        # batch i+1 on a side stream under step i's optimiser (DAEEngine.train_step(next_batch=...)), so inside the timed
        # region every step still pays for exactly one noise launch: batch i+1's instead of its own
        if not eng.has_prefetched_batch():
            a = batch_args(i)
            eng.sample_batch(a["indptr"], a["indices"], a["batch_ids"], a["alias_prob"], a["alias_idx"], a["noise"],
                             a["noise_std"], seed=a["seed"])
        return eng.train_step(next_batch=batch_args(i + 1))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    eng.check_overflow()
    barrier()
    # ---- the timed region: exactly K steps, nothing but the step's own kernels on the stream ----
    eng.launches = 0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clocks.mark_begin()
    ev0.record()
    for i in range(args.steps):
        loss = step(args.warmup + i)
    ev1.record()
    barrier()
    clocks.mark_end()
    # the last timed step's results, held before the instrumented pass below trains the model further
    outputs = (loss.clone(), model.store.params.clone()) if args.dump_outputs and rank == 0 else None
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    launches = eng.launches
    # the poller is stopped here when the timed region already holds three samples: nvidia-smi queries take driver locks,
    # and the instrumented pass below is what the roofline numbers come from
    clock_info = None
    if rank == 0:
        time.sleep(0.05)                                   # (lets the reader thread catch up with the pipe)
        if clocks.samples_in_timed_region() >= 3:
            clock_info = clocks.stop()
    # ---- the same K steps again with a CUDA-event pair around every kernel of interest (the roofline leg).  The
    #      event records sit between consecutive GEMM launches and so defeat their programmatic dependent launch:
    #      this pass is a few percent slower than the timed region above, and is reported separately ----
    eng.enable_kernel_timing(True)
    evi0, evi1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    evi0.record()
    for i in range(args.steps):
        step(args.warmup + args.steps + i)
    evi1.record()
    barrier()
    ms_instr = evi0.elapsed_time(evi1)
    # clocks: the samples inside the timed region when there are at least three of them (10 ms period), else the
    # samples from its start to the end of the instrumented pass -- the same K steps under the same load
    clocks.mark_load_end()
    if rank == 0 and clock_info is None:
        clock_info = clocks.stop()
    ktimes = eng.kernel_times_ms()
    eng.enable_kernel_timing(False)
    loss_host = [float(v) for v in loss.cpu().numpy()]
    value = B * world * args.steps / (ms_total / 1e3)

    # ---- e2e: the package's host-fed trainer path (HostBatchStream): every step's batch CSR is copied from pinned
    #      host memory (double-buffered on a copy stream) and every step's loss is copied back to the host ----
    feed = E.HostBatchStream(eng, [csr.rows(np.arange(i * B, (i + 1) * B)) for i in range(nb)])
    e2e_losses = []
    for i in range(min(args.warmup, 3)):
        feed.step(i, prob, alias, W["noise"], W["noise_std"], seed=99 + rank)
    feed.drain()
    barrier()
    t_a = time.perf_counter()
    for i in range(args.steps):
        l = feed.step(3 + i, prob, alias, W["noise"], W["noise_std"], seed=99 + rank)
        if l is not None:
            e2e_losses.append(float(l[2]))
    e2e_losses.append(float(feed.drain()[2]))                       # K losses read on the host inside the region
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t_a], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    assert len(e2e_losses) == args.steps and all(np.isfinite(e2e_losses))
    e2e_value = B * world * args.steps / float(e2e_s.item())
    h2d = feed.h2d_bytes

    # ---- --check: N ranks on a fixed global batch reproduce the 1-GPU step (cubecobrarecommender_b200/dp_check.py) ----
    check = None
    if args.check and world > 1:
        from cubecobrarecommender_b200 import dp_check
        del feed
        torch.cuda.empty_cache()
        check = dp_check.run_check(args.precision, steps=3, log=log)
        check["violations"] = dp_check.verdict(check)
    elif args.check:
        check = {"skipped": "a single rank has nothing to exchange", "violations": []}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs[0], model.store.to_dict(outputs[1]), log)
    # ---- roofline of the dominant kernel: the eight 512<->C GEMM passes per step (seven with the gather first layer) ----
    peaks = load_peaks()
    n_big, ms_big = ktimes.get("big_gemm", (0, 0.0))
    n_dw1, ms_dw1 = ktimes.get("dw1_gemm", (0, 0.0))      # dW1 = x^T g1 is one more 2*B*512*C pass
    n_big, ms_big = n_big + n_dw1, ms_big + ms_dw1
    n_fw1, ms_fw1 = ktimes.get("fw1_gemm", (0, 0.0))      # x W1 on the tensor cores (when the engine takes that route)
    n_big, ms_big = n_big + n_fw1, ms_big + ms_fw1
    passes_b = 4.0 + (1.0 if n_fw1 else 0.0)
    # 512 <-> C passes per step: main tower fwd/dW/dX + dW1 (+ x W1) on B rows, reg tower fwd/dW/dX on R rows
    flops_per_launch = 2.0 * 512 * C * (passes_b * B + 3.0 * R) / (passes_b + 3.0)
    # fp32 / tf32 kinds run at half the bf16 tensor rate.  The timed region lasts K * 2.3 ms -- well under a second at the
    # default K -- so the denominator is the BURST figure of MEASURED_PEAKS.json (a kernel timed alone / a short region);
    # the fraction against the sustained figure (seconds-long, power-capped runs) is reported beside it
    kind_scale = 1.0 if args.precision == "bf16" else 0.5
    region_s = ms_total / 1e3
    peak_burst, peak_sust = peaks["bf16_burst"] * kind_scale, peaks["bf16_sustained"] * kind_scale
    tensor_peak = peak_burst if region_s < 2.0 else peak_sust
    achieved = flops_per_launch / (ms_big / n_big * 1e-3) / 1e12 if n_big else 0.0
    traffic, traffic_src = ncu_traffic(args.precision)
    roofline = {"kernel": {"fp32": "gemm_simt_kernel", "tf32": "gemm_tc_kernel<tf32>", "bf16": "gemm_tc_kernel<bf16>"}[args.precision],
                "bound": "tensor", "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s",
                "frac": achieved / tensor_peak, "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": 4.0 * (B * 512 + 512 * C + B * C) * (kind_scale if args.precision == "bf16" else 1.0),
                "peak_source": f"{peaks['source']} bf16 {'burst' if region_s < 2.0 else 'sustained'} x{kind_scale} "
                               f"({args.precision}; timed region {region_s:.2f} s)",
                "frac_of_burst": achieved / peak_burst, "frac_of_sustained": achieved / peak_sust,
                "launches_timed": n_big, "avg_launch_ms": ms_big / n_big if n_big else None,
                "share_of_step": ms_big / ms_instr if ms_instr else None,
                "instrumented_ms_per_step": ms_instr / args.steps,
                "note": "per-kernel CUDA events over a second pass of the same K steps (events between launches "
                        "disable programmatic dependent launch, hence the slower instrumented step)"}
    kernels = {k: {"launches": n, "ms_total": round(t, 3), "share": round(t / ms_instr, 4)} for k, (n, t) in ktimes.items()}
    # HBM-bound helpers, for the record: logical GB/s of the gather and Adam kernels
    if "bag_fwd" in ktimes and ktimes["bag_fwd"][1] > 0:
        n, t = ktimes["bag_fwd"]
        nnz_x = float(eng.x_len.sum().item())
        kernels["bag_fwd"]["logical_GBps"] = round((nnz_x * (4 + 2048) + B * 2048) / (t / n * 1e-3) / 1e9, 1)
    if "adam" in ktimes and ktimes["adam"][1] > 0:
        n, t = ktimes["adam"]
        kernels["adam"]["GBps"] = round(model.store.total * 4 * 7 / (t / n * 1e-3) / 1e9, 1)

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        log("timing the CPU comparator (oracle port) on a bounded sample ...")
        r = cpu_reference(C, steps=3, warmup=1, log=log, budget_s=40.0)
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
               "sample": f"3 steps x {r['batch']} cubes + {r['batch']} reg rows at C={C}: generator {r['gen_seconds']:.2f}s + "
                         f"torch-CPU step {r['model_seconds']:.2f}s (host has {os.cpu_count()} cpus, {r['cores']} threads used)"}
    extras = None
    if world == 1 and not args.no_extras:
        del eng, model
        torch.cuda.empty_cache()
        try:
            extras = measure_extras(dev, peaks, log)
        except Exception as e:  # the headline line must survive a failure in the side measurements
            extras = {"error": repr(e)}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": {"fp32": "f32", "tf32": "tf32", "bf16": "bf16"}[args.precision], "data": "synthetic",
        "config": {**workload_config(world, B, R, global_R, args.reg_mode, args.scaling),
                   **({"gradient_exchange": ("p2p_overlap" if eng.p2p_buckets else eng.dp_mode)
                       + (" (multimem)" if getattr(eng, "_multicast", False) else "")} if world > 1 else {})},
        **({"note": "non-headline configuration (--reg-mode full)"} if args.reg_mode == "full" else {}),
        "loss": {"bce": loss_host[0], "kl": loss_host[1], "total": loss_host[2]},
        "loss_rel_err": loss_check["loss_rel_err"] if loss_check else None, "loss_check": loss_check,
        **({"check": check} if check is not None else {}),
        "roofline": roofline, "kernels": kernels, "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 24,
                "ms_per_step": 1e3 * float(e2e_s.item()) / args.steps},
        "gpu_launches": launches, "clocks": clock_info, "extras": extras,
    }
    sys.stdout.flush()
    os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--precision", default=os.environ.get("CC_PRECISION", "tf32"), choices=["fp32", "tf32", "bf16"])
    ap.add_argument("--reg-mode", default="sampled", choices=["sampled", "full"],
                    help="regulariser rows per step: B sampled rows per rank (the reference's code path, the headline "
                         "config) or ALL rows of I sharded over the ranks (README formula, BASELINE configs[2])")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: 4096 cubes + 4096 reg rows PER GPU (the headline); strong: the GLOBAL batch stays 4096 "
                         "(BASELINE configs[2]: 512 per GPU at N = 8)")
    ap.add_argument("--check", action="store_true",
                    help="N > 1: also run the fixed-global-batch equality check against the 1-GPU step and add it to the line")
    ap.add_argument("--no-loss-check", action="store_true", help="N = 1: skip the float64 oracle comparison of the step-1 loss")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the graph-build and ml_recommend side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and the updated weights of the last timed step to DIR/<name>.npy (inputs are "
                         "seeded: two builds run with the same arguments can be compared array by array)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the outputs of the native train step (--impl native)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    args.warmup = max(args.warmup, 3) if args.impl == "native" else args.warmup
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_native(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
