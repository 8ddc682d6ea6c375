#!/usr/bin/env python
"""Costs of similar cards and cubes at C = 20 884.  Prints one JSON line:

1. ``kernel``: cc_cosine_neg_many_f32 over all C x C card pairs (the embeddings of an untrained fp32 model, ReLU
   outputs with many zeros) into a (C, C) row-padded matrix: time, pairs/s, bytes written, and the FP32 issue floor
   -- pairs x FP32 instructions per pair (64 FFMA + 31 FADD + 2 FMUL + 1 negation = 98, from the SASS) over
   148 SMs x 128 lanes x the SM clock sampled by nvidia-smi while the kernel runs back to back.  Also the
   (4096, C) block the table computes at a time, and the row select on it (``topn_masked``, n = 50, ascending).
2. ``table``: ``similar_cards(None, 50, exclude_self=True)`` with its host read (card embeddings included), against
   the loop of one-card calls over every card: the route ``similar()`` took before (cc_cosine_neg_f32 + a batch-1
   select + host read per card) and ``similar()`` as it is now.  The table and the old route are checked equal.
3. ``cubes``: ``similar_cubes`` of 100 000 synthetic cubes (``synth_cubes_csr``) against each other, n = 50, with
   ``cube_embeddings`` included and the host read of the result, and ``cube_embeddings`` alone; tf32 model.

Kernel times: CUDA events around single launches, L2 overwritten (256 MB) before each, median of ``REPS``.  End-to-end
times: host clock around calls that end in their host read, median of 3.  Card name and power limit are read in the
same run.

    python profiles/similarity_bench.py > profiles/r08_similarity/similarity_bench.json
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
sys.path.insert(0, os.path.join(REPO, "profiles"))
from baseline_rank_bench import card, clock, timed  # noqa: E402
from cubecobrarecommender_b200 import _lib, graph as G  # noqa: E402
from cubecobrarecommender_b200.ml import model as M  # noqa: E402
from cubecobrarecommender_b200.ml.inference import MLRecommender  # noqa: E402
from cubecobrarecommender_b200.sparse import CubeCSR  # noqa: E402
from cubecobrarecommender_b200.synth import synth_cubes_csr  # noqa: E402

C, N, BLOCK, K_CUBES = 20884, 50, 4096, 100_000
FP32_PER_PAIR = 98
dev = torch.device("cuda", 0)


def many(q, c, out):
    _lib.call("cc_cosine_neg_many_f32", _lib.ptr(q), q.stride(0), q.shape[0], _lib.ptr(c), c.stride(0), c.shape[0], 64,
              _lib.ptr(out), out.stride(0), _lib.stream_ptr())


def sm_clock_during(fn, seconds=2.0):
    """Median SM clock (MHz) nvidia-smi reports while ``fn`` runs back to back for ``seconds``."""
    p = subprocess.Popen(["nvidia-smi", "-i", "0", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits",
                          "-lms", "100"], stdout=subprocess.PIPE, text=True)
    try:
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            for _ in range(20):
                fn()
            torch.cuda.synchronize()
    finally:
        p.terminate()
        out, _ = p.communicate(timeout=30)
    mhz = [float(s) for s in out.split() if s.replace(".", "", 1).isdigit()]
    return float(np.median(mhz[len(mhz) // 4:])) if mhz else None      # skip the samples taken before the loop


def kernel(emb):
    ldo = (C + 3) // 4 * 4
    out = torch.empty((C, ldo), dtype=torch.float32, device=dev)
    t = timed(lambda: many(emb, emb, out))
    mhz = sm_clock_during(lambda: many(emb, emb, out))
    pairs = C * C
    res = {"pairs": pairs, "all_pairs_us": t[0], "all_pairs_min_us": t[1], "pairs_per_s": pairs / (t[0] * 1e-6),
           "bytes_written": 4 * pairs, "write_GBps": 4 * pairs / t[0] / 1e3, "sm_clock_mhz_during": mhz,
           "fp32_instructions_per_pair": FP32_PER_PAIR}
    if mhz:
        floor_us = pairs * FP32_PER_PAIR / (148 * 128 * mhz * 1e6) * 1e6
        res.update({"fp32_issue_floor_us": floor_us, "share_of_fp32_issue_floor": floor_us / t[0]})
    blk = out[:BLOCK]
    tb = timed(lambda: many(emb[:BLOCK], emb, blk))
    mp = torch.zeros(BLOCK + 1, dtype=torch.int64, device=dev)
    mi = torch.zeros(1, dtype=torch.int32, device=dev)
    outs = (torch.empty(BLOCK, N, dtype=torch.int32, device=dev), torch.empty(BLOCK, N, device=dev),
            torch.empty(BLOCK, dtype=torch.int32, device=dev))
    ts = timed(lambda: G.topn_masked(blk[:, :C], mp, mi, N, descending=False, out=outs))
    res.update({"block_rows": BLOCK, "block_us": tb[0], "block_bytes_written": 4 * BLOCK * C,
                "block_select_n50_us": ts[0]})
    del out
    return res


def parent_similar(emb, q, n):
    dists = torch.empty((1, C), dtype=torch.float32, device=dev)
    _lib.call("cc_cosine_neg_f32", _lib.ptr(emb), emb.stride(0), C, 64, int(q), _lib.ptr(dists), _lib.stream_ptr())
    none_ptr = torch.zeros(2, dtype=torch.int64, device=dev)
    none_idx = torch.zeros(1, dtype=torch.int32, device=dev)
    ids, vals, _ = G.topn_masked(dists, none_ptr, none_idx, n, only_listed=False, descending=False)
    return ids[0].cpu().numpy(), vals[0].cpu().numpy()


def table(rec, emb):
    def run():
        ids, dists = rec.similar_cards(None, N, exclude_self=True)
        return ids.cpu().numpy(), dists.cpu().numpy()
    t = clock(run)
    ids, dists = run()
    old = [parent_similar(emb, q, N + 1) for q in range(C)]             # checked: the table is the old route minus self
    for q in range(C):
        keep = old[q][0] != q
        assert np.array_equal(ids[q], old[q][0][keep][:N]) and np.array_equal(dists[q], old[q][1][keep][:N]), q
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for q in range(C):
        parent_similar(emb, q, N)
    t_old = time.perf_counter() - t0
    t0 = time.perf_counter()
    for q in range(C):
        rec.similar(q, N, embeddings=emb)
    t_new_loop = time.perf_counter() - t0
    return {"n": N, "table_with_host_read_ms": t * 1e3, "old_route_loop_s": t_old, "similar_loop_s": t_new_loop,
            "old_route_loop_over_table": t_old / t, "similar_loop_over_table": t_new_loop / t, "equal_to_old_route": True}


def cubes():
    ip, ix = synth_cubes_csr(K_CUBES, C, seed=81)
    csr = CubeCSR(ip, ix, C)
    model = M.CC_Recommender(C, device=dev, seed=0, precision="tf32")
    rec = MLRecommender(model)

    def run():
        ids, dists = rec.similar_cubes(csr, N)
        return ids.cpu().numpy(), dists.cpu().numpy()
    t = clock(run)
    te = clock(lambda: rec.cube_embeddings(csr).cpu())
    return {"cubes": K_CUBES, "n": N, "mean_cube_size": float(np.diff(ip).mean()), "similar_cubes_with_host_read_ms": t * 1e3,
            "cube_embeddings_ms": te * 1e3, "pairs": K_CUBES * K_CUBES}


def main():
    torch.cuda.set_device(0)
    out = {"card": card(), "C": C, "l2": "256 MB overwritten before every timed kernel launch"}
    model = M.CC_Recommender(C, device=dev, seed=0, precision="fp32")
    rec = MLRecommender(model)
    emb = rec.card_embeddings()
    out["zero_fraction_of_embeddings"] = float((emb == 0).float().mean())
    out["kernel"] = kernel(emb)
    out["table"] = table(rec, emb)
    out["cubes"] = cubes()
    out["card_after"] = card()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
