#!/usr/bin/env python
"""Costs and results of the leave-k-out baselines at C = 20 884.  Prints one JSON line:

1. ``kernel``: cc_rank_targets_f64 on 4096 graph-score rows (float64, ld = C; scores of synthetic cubes of
   s ~ U{360..720} cards with 20% hidden, against M of 20 000 other cubes), next to the float64 top-50 select
   (cc_topn_masked_f64) on the same rows and cc_rank_targets_f32 on the same rows cast to float32; and the popularity
   form, cc_rank_targets_f64 over one shared row (ld = 0).  Algorithmic bytes (8 C for a score row, or 8 C once for the
   shared one, + 4 |visible| + 8 |hidden| per cube) over kernel time.
2. ``scoring``: cc_score_gather_f64 (the graph scores, NumPy's pairwise order) for the same 4096 cubes: time per cube
   and the M rows it reads (8 C |visible| bytes per cube) over that time.
3. ``end_to_end``: ``evaluate_recommendations`` for the graph baseline, the popularity baseline and the ML model
   (tf32) on the same 16 384 held-out cubes, in cubes/s.
4. ``metrics``: the three metric sets side by side, the ML model trained for a few epochs on the 20 000 training cubes.
   Synthetic cubes are independent draws from one popularity law, so co-occurrence carries little beyond popularity
   here; the numbers show the plumbing, not what real cubes give.

Kernel times: CUDA events around single launches, L2 overwritten (256 MB) before each launch, median of ``REPS``.
End-to-end times: host clock around calls that end in their host read, median of 3.  Card name and power limit are read
in the same run.

    python profiles/baseline_rank_bench.py > profiles/r05_baselines/baseline_rank_bench.json
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
from cubecobrarecommender_b200.ml import generator as GEN, model as M, ranking as R, train as T  # noqa: E402
from cubecobrarecommender_b200.sparse import CubeCSR  # noqa: E402
from cubecobrarecommender_b200.synth import synth_cubes_csr  # noqa: E402

B, C, N = 4096, 20884, 50
K_TRAIN, K_VAL = 20000, 16384
REPS = int(os.environ.get("RANK_BENCH_REPS", 20))
EPOCHS = int(os.environ.get("BASELINE_BENCH_EPOCHS", 10))
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


def clock(fn, reps=3):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def kernels_and_scoring(rec, pop):
    ip, ix = synth_cubes_csr(B, C, seed=51)
    vis, hid, _ = R.holdout_split(CubeCSR(ip, ix, C), 0.2, seed=9)
    mp, mi = (torch.from_numpy(a).to(dev) for a in (vis.indptr, vis.indices))
    tp, ti = (torch.from_numpy(a).to(dev) for a in (hid.indptr, hid.indices))
    nv, nh = len(vis.indices), len(hid.indices)
    out = {"hidden_per_cube": nh / B, "visible_per_cube": nv / B}

    # 2. graph scoring, with the plan built and uploaded beforehand
    lib = _lib.load()
    vp = vis.indptr.astype(np.int64)
    leaves = int(sum(lib.cc_pairwise_leaf_count(int(n)) for n in np.diff(vp) if n > 0))
    plan_h = np.zeros((leaves, 4), dtype=np.int32)
    leaf_ptr_h = np.zeros(B + 1, dtype=np.int32)
    _lib.call("cc_pairwise_plan_host", _lib.ptr(vp), B, _lib.ptr(plan_h), _lib.ptr(leaf_ptr_h))
    plan, leaf_ptr = torch.from_numpy(plan_h).to(dev), torch.from_numpy(leaf_ptr_h).to(dev)
    partial = torch.empty((leaves, C), dtype=torch.float64, device=dev)
    scores = torch.empty((B, C), dtype=torch.float64, device=dev)

    def score():
        _lib.call("cc_score_gather_f64", _lib.ptr(rec.m), rec.m.stride(0), C, _lib.ptr(mi), _lib.ptr(mp), B,
                  _lib.ptr(plan), _lib.ptr(leaf_ptr), leaves, 0, _lib.ptr(partial), _lib.ptr(scores), scores.stride(0),
                  _lib.stream_ptr())
    sc_us = timed(score)
    m_bytes = 8 * C * nv
    out["scoring"] = {"us_per_4096_cubes": sc_us[0], "min_us": sc_us[1], "us_per_cube": sc_us[0] / B,
                      "leaves": leaves, "m_row_bytes_per_cube": m_bytes / B,
                      "m_rows_GBps": m_bytes / sc_us[0] / 1e3, "partial_bytes": 8 * C * leaves}
    score()
    torch.cuda.synchronize()
    assert torch.equal(scores, rec.scores(vis)[0])            # the timed call is the recommender's scoring

    # 1. the rank kernels on those rows
    ranks = torch.empty(nh, dtype=torch.int32, device=dev)
    rank64 = timed(lambda: G.rank_targets(scores, mp, mi, tp, ti, out=ranks))
    r64 = ranks.cpu().numpy().copy()
    outs = (torch.empty(B, N, dtype=torch.int32, device=dev), torch.empty(B, N, dtype=torch.float64, device=dev),
            torch.empty(B, dtype=torch.int32, device=dev))
    sel64 = timed(lambda: G.topn_masked(scores, mp, mi, N, out=outs))
    s32 = scores.float()
    rank32 = timed(lambda: G.rank_targets(s32, mp, mi, tp, ti, out=ranks))
    r32 = ranks.cpu().numpy().copy()
    row = pop.scores.expand(B, C)
    rank_pop = timed(lambda: G.rank_targets(row, mp, mi, tp, ti, out=ranks))
    list_bytes = 4 * nv + 8 * nh
    out["kernel"] = {
        "rank_f64_us": rank64[0], "rank_f64_min_us": rank64[1],
        "rank_f64_GBps": (8 * C * B + list_bytes) / rank64[0] / 1e3,
        "top50_select_f64_us": sel64[0], "top50_select_f64_min_us": sel64[1],
        "rank_f32_cast_us": rank32[0], "rank_f32_cast_min_us": rank32[1],
        "rank_f32_cast_GBps": (4 * C * B + list_bytes) / rank32[0] / 1e3,
        "rank_popularity_ld0_us": rank_pop[0], "rank_popularity_ld0_min_us": rank_pop[1],
        "rank_f64_over_select_f64": rank64[0] / sel64[0], "rank_f64_over_rank_f32": rank64[0] / rank32[0],
        "rank_f64_over_scoring": rank64[0] / sc_us[0],
        "median_hidden_rank_f64": float(np.median(r64)), "recall_at_50_f64": float(np.mean(r64 < N)),
        "ranks_f32_cast_differ": float(np.mean(r64 != r32))}
    return out


def main():
    torch.cuda.set_device(0)
    out = {"card": card(), "B": B, "C": C, "reps": REPS, "l2": "256 MB overwritten before every timed kernel launch"}
    ip, ix = synth_cubes_csr(K_TRAIN + K_VAL, C, seed=53)
    csr = CubeCSR(ip, ix, C)
    mhat = G.build_graph(csr, dev, want_m64=False, want_neg=False).mhat
    gen = GEN.DataGenerator(mhat, csr, batch_size=4096, noise=0.2, seed=1)
    train, val = gen.split(K_VAL / (K_TRAIN + K_VAL))
    assert val.N_cubes == K_VAL
    g = G.build_graph(train.csr, dev, allreduce=False, want_m64=True, want_mhat=False, want_neg=False)
    rec, pop = G.GraphRecommender(g.m64), G.PopularityRecommender(train.csr, dev)
    del g
    out.update(kernels_and_scoring(rec, pop))

    # 3. evaluate_recommendations throughput on the same 16 384 held-out cubes
    model = M.CC_Recommender(C, device=dev, seed=0, precision="tf32")
    val.holdout_split(0.2)                                   # the split is drawn once per generator; not timed
    e2e = {"cubes": K_VAL}
    for name, m in (("graph", rec), ("popularity", pop), ("ml", model)):
        s = clock(lambda: T.evaluate_recommendations(m, val, at=(10, 50)))
        e2e[name] = {"seconds": s, "cubes_per_s": K_VAL / s}
    out["end_to_end"] = e2e

    # 4. the three metric sets, the model trained for a few epochs
    t0 = time.perf_counter()
    T.fit(model, train, epochs=EPOCHS, reg=0.1, log=lambda *_: None)
    torch.cuda.synchronize()
    out["metrics"] = {"ml_epochs": EPOCHS, "ml_train_seconds": time.perf_counter() - t0, "holdout": 0.2,
                      "ml": T.evaluate_recommendations(model, val, at=(10, 50)),
                      **T.ranking_baselines(train, val, at=(10, 50), holdout=0.2)}
    out["card_after"] = card()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
