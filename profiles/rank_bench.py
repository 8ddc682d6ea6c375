#!/usr/bin/env python
"""Leave-k-out ranking evaluation costs at C = 20 884.  Prints one JSON line:

* cc_rank_targets_f32 (fused sigmoid) on 4096 rows of logits, ld 20 884 (unpadded) and 20 992 (padded to 128),
  cubes of s ~ U{360..720} cards with 20% hidden, for two logit distributions: "untrained" (N(0, 1): about half of
  every row lies above the lowest target, the most elements the kernel keys and counts) and "trained" (the hidden
  cards lifted by +3.5, into the top few hundred).  Algorithmic bytes (4 C + 4 |visible| + 8 |hidden| per cube: the
  logit row, the mask list, the target list and the ranks) over kernel time against the 6546.9 GB/s HBM rate the
  project uses; the fused-sigmoid top-50 select (cc_topn_masked_sigmoid_f32) on the same rows in the same run.
* ``evaluate_recommendations`` throughput (cubes/s) on 16 384 held-out cubes against ``recommend_device`` top-50 on
  the same visible cubes (tf32 model), and ``target_ranks_device`` alone.

Kernel times: CUDA events around single launches, L2 overwritten (256 MB) before each launch, median of ``REPS``.
End-to-end times: host clock around calls that end in a device synchronise (evaluate_recommendations ends in its host
read), median of 5.  Card name and power limit are read in the same run.

    python profiles/rank_bench.py > profiles/r04_ranking/rank_bench.json
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
from cubecobrarecommender_b200 import graph as G  # noqa: E402
from cubecobrarecommender_b200.ml import generator as GEN, model as M, ranking as R, train as T  # noqa: E402
from cubecobrarecommender_b200.ml.inference import MLRecommender  # noqa: E402
from cubecobrarecommender_b200.sparse import CubeCSR  # noqa: E402
from cubecobrarecommender_b200.synth import synth_cubes_csr  # noqa: E402

B, C, N = 4096, 20884, 50
HBM_GBS = 6546.9
REPS = int(os.environ.get("RANK_BENCH_REPS", 30))
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


def kernels():
    ip, ix = synth_cubes_csr(B, C, seed=41)
    vis, hid, _ = R.holdout_split(CubeCSR(ip, ix, C), 0.2, seed=7)
    mp, mi = (torch.from_numpy(a).to(dev) for a in (vis.indptr, vis.indices))
    tp, ti = (torch.from_numpy(a).to(dev) for a in (hid.indptr, hid.indices))
    nbytes = B * 4 * C + 4 * len(vis.indices) + 8 * len(hid.indices)
    rows = np.repeat(np.arange(B), np.diff(hid.indptr))
    out = {"bytes": nbytes, "hidden_per_cube": float(len(hid.indices) / B), "visible_per_cube": float(len(vis.indices) / B)}
    for ld in (20884, 20992):
        g = torch.Generator(device=dev).manual_seed(ld)
        z = torch.randn(B, ld, device=dev, generator=g)[:, :C]
        for dist in ("untrained", "trained"):
            if dist == "trained":
                z[torch.from_numpy(rows).to(dev), ti.long()] += 3.5
            ranks = torch.empty(len(hid.indices), dtype=torch.int32, device=dev)
            rk = timed(lambda: G.rank_targets(z, mp, mi, tp, ti, sigmoid=True, out=ranks))
            outs = (torch.empty(B, N, dtype=torch.int32, device=dev), torch.empty(B, N, device=dev),
                    torch.empty(B, dtype=torch.int32, device=dev))
            sel = timed(lambda: G.topn_masked(z, mp, mi, N, sigmoid=True, out=outs))
            r = ranks.cpu().numpy()
            out[f"ld{ld}_{dist}"] = {
                "rank_us": rk[0], "rank_min_us": rk[1], "rank_GBps": nbytes / rk[0] / 1e3,
                "rank_frac_of_hbm": nbytes / rk[0] / 1e3 / HBM_GBS, "top50_select_us": sel[0],
                "top50_select_min_us": sel[1], "rank_over_select": rk[0] / sel[0],
                "median_hidden_rank": float(np.median(r)), "recall_at_50": float(np.mean(r < N))}
    return out


def end_to_end():
    k = 16384
    ip, ix = synth_cubes_csr(k, C, seed=43)
    csr = CubeCSR(ip, ix, C)
    mhat = G.build_graph(csr, dev, want_m64=False).mhat
    gen = GEN.DataGenerator(mhat, csr, batch_size=4096, noise=0.2, seed=1)
    model = M.CC_Recommender(C, device=dev, seed=0, precision="tf32")
    vis, hid, _ = gen.holdout_split(0.2)
    rec = MLRecommender(model)

    def clock(fn):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        return float(np.median(ts))
    ev = clock(lambda: T.evaluate_recommendations(model, gen, at=(10, 50)))
    rk = clock(lambda: rec.target_ranks_device(vis, hid))
    rd = clock(lambda: rec.recommend_device(vis, N))
    res = T.evaluate_recommendations(model, gen, at=(10, 50))
    return {"cubes": k, "evaluate_s": ev, "evaluate_cubes_per_s": k / ev, "target_ranks_device_s": rk,
            "target_ranks_cubes_per_s": k / rk, "recommend_device_top50_s": rd, "recommend_cubes_per_s": k / rd,
            "evaluate_over_recommend_throughput": rd / ev, "untrained_metrics": res}


def main():
    torch.cuda.set_device(0)
    out = {"card": card(), "B": B, "C": C, "reps": REPS, "l2": "256 MB overwritten before every timed kernel launch",
           "hbm_GBps_reference": HBM_GBS}
    out["kernel"] = kernels()
    out["end_to_end"] = end_to_end()
    out["card_after"] = card()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
