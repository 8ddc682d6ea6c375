#!/usr/bin/env python
"""Costs of scoring the cut list at C = 20 884.  Prints one JSON line:

1. ``kernel_f32``: cc_rank_cuts_f32 with the fused sigmoid on 4096 logit rows (synthetic cubes of s ~ U{360..720}
   cards plus 20% intruders from ``ranking.intruder_split``), next to the only route the tree had to these ranks:
   cc_sigmoid_f32 over the rows, cc_topn_masked_f32(only_listed, ascending, n = largest corrupted cube), and the
   inverse permutation of the returned ids (torch scatter / gather).  Both give the same ranks (checked).  Bytes: the
   kernel gathers one 32-byte sector per listed score (32 (s + m) per cube) against the 4 C of a row.
2. ``kernel_f64``: cc_rank_cuts_f64 on 4096 graph-score rows (``GraphRecommender.scores(zero_diag=True)``, M of the
   20 000 training cubes) and on one shared popularity row (ld = 0).
3. ``end_to_end``: ``evaluate_cuts`` for the ML model (tf32, untrained), the graph and popularity on 16 384 held-out
   cubes, in cubes/s, against ``evaluate_recommendations`` on the same cubes.

Kernel times: CUDA events around single launches (the route: around its three steps), L2 overwritten (256 MB) before
each, median of ``REPS``.  End-to-end times: host clock around calls that end in their host read, median of 3, the
splits drawn beforehand.  Card name and power limit are read in the same run.

    python profiles/cut_rank_bench.py > profiles/r07_cuts/cut_rank_bench.json
"""
import json
import os
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "profiles"))
from baseline_rank_bench import card, clock, timed  # noqa: E402
from cubecobrarecommender_b200 import _lib, graph as G  # noqa: E402
from cubecobrarecommender_b200.ml import generator as GEN, model as M, ranking as R, train as T  # noqa: E402
from cubecobrarecommender_b200.sparse import CubeCSR  # noqa: E402
from cubecobrarecommender_b200.synth import synth_cubes_csr  # noqa: E402

B, C = 4096, 20884
K_TRAIN, K_VAL = 20000, 16384
dev = torch.device("cuda", 0)


def kernel_f32():
    ip, ix = synth_cubes_csr(B, C, seed=71)
    cor, intr, _ = R.intruder_split(CubeCSR(ip, ix, C), 0.2, seed=3)
    cp, ci = (torch.from_numpy(a).to(dev) for a in (cor.indptr, cor.indices))
    tp, ti = (torch.from_numpy(a).to(dev) for a in (intr.indptr, intr.indices))
    g = torch.Generator(device=dev).manual_seed(1)
    z = torch.randn(B, C, device=dev, generator=g) * 2
    z[:, :300] += 3
    nl, nt = len(cor.indices), len(intr.indices)
    ranks = torch.empty(nt, dtype=torch.int32, device=dev)
    new = timed(lambda: G.rank_cuts(z, cp, ci, tp, ti, sigmoid=True, out=ranks))
    got = ranks.clone()

    n = cor.max_size
    probs = torch.empty_like(z)
    outs = (torch.empty(B, n, dtype=torch.int32, device=dev), torch.empty(B, n, dtype=torch.float32, device=dev),
            torch.empty(B, dtype=torch.int32, device=dev))
    slot = torch.arange(n, dtype=torch.int32, device=dev).expand(B, n)
    cube = torch.from_numpy(np.repeat(np.arange(B), np.diff(intr.indptr))).to(dev)
    pos = torch.empty(B, C + 1, dtype=torch.int32, device=dev)        # column C takes the -1 padding of short rows

    def sigmoid():
        _lib.call("cc_sigmoid_f32", _lib.ptr(z), _lib.ptr(probs), probs.numel(), _lib.stream_ptr())

    def select():
        G.topn_masked(probs, cp, ci, n, only_listed=True, descending=False, out=outs)

    def invert():
        ids = outs[0].long()
        pos.scatter_(1, torch.where(ids < 0, C, ids), slot)
        ranks.copy_(pos[cube, ti.long()])

    def route():
        sigmoid(); select(); invert()
    total = timed(route)
    assert torch.equal(ranks, got), "the route and cc_rank_cuts_f32 disagree"
    parts = {name: timed(fn)[0] for name, fn in (("sigmoid_us", sigmoid), ("select_us", select), ("invert_us", invert))}
    return {"listed_per_cube": nl / B, "intruders_per_cube": nt / B, "select_n": n,
            "rank_cuts_f32_sigmoid_us": new[0], "rank_cuts_f32_sigmoid_min_us": new[1],
            "gathered_sector_bytes_per_cube": 32 * nl / B, "row_bytes": 4 * C,
            "gathered_sectors_GBps": 32 * nl / new[0] / 1e3,
            "route_us": total[0], "route_min_us": total[1], "route_parts_us": parts,
            "route_over_rank_cuts": total[0] / new[0], "ranks_equal": True}


def kernel_f64(rec, pop):
    ip, ix = synth_cubes_csr(B, C, seed=72)
    cor, intr, _ = R.intruder_split(CubeCSR(ip, ix, C), 0.2, seed=4)
    scores, cp, ci = rec.scores(cor, zero_diag=True)
    tp, ti = (torch.from_numpy(a).to(dev) for a in (intr.indptr, intr.indices))
    ranks = torch.empty(len(intr.indices), dtype=torch.int32, device=dev)
    graph = timed(lambda: G.rank_cuts(scores, cp, ci, tp, ti, out=ranks))
    shared = timed(lambda: G.rank_cuts(pop.scores.expand(B, C), cp, ci, tp, ti, out=ranks))
    return {"rank_cuts_f64_graph_rows_us": graph[0], "rank_cuts_f64_graph_rows_min_us": graph[1],
            "rank_cuts_f64_ld0_us": shared[0], "rank_cuts_f64_ld0_min_us": shared[1]}


def main():
    torch.cuda.set_device(0)
    out = {"card": card(), "B": B, "C": C, "l2": "256 MB overwritten before every timed kernel launch"}
    out["kernel_f32"] = kernel_f32()
    ip, ix = synth_cubes_csr(K_TRAIN + K_VAL, C, seed=73)
    csr = CubeCSR(ip, ix, C)
    mhat = G.build_graph(csr, dev, want_m64=False, want_neg=False).mhat
    gen = GEN.DataGenerator(mhat, csr, batch_size=4096, noise=0.2, seed=1)
    train, val = gen.split(K_VAL / (K_TRAIN + K_VAL))
    g = G.build_graph(train.csr, dev, allreduce=False, want_m64=True, want_mhat=False, want_neg=False)
    rec, pop = G.GraphRecommender(g.m64), G.PopularityRecommender(train.csr, dev)
    del g
    out["kernel_f64"] = kernel_f64(rec, pop)
    model = M.CC_Recommender(C, device=dev, seed=0, precision="tf32")
    val.holdout_split(0.2)
    val.intruder_split(0.2)                                   # drawn once per generator; not timed
    e2e = {"cubes": K_VAL}
    for name, m in (("ml", model), ("graph", rec), ("popularity", pop)):
        cuts = clock(lambda: T.evaluate_cuts(m, val, at=(10, 50)))
        adds = clock(lambda: T.evaluate_recommendations(m, val, at=(10, 50)))
        e2e[name] = {"evaluate_cuts_s": cuts, "evaluate_cuts_cubes_per_s": K_VAL / cuts,
                     "evaluate_recommendations_s": adds, "evaluate_recommendations_cubes_per_s": K_VAL / adds,
                     "cut_metrics": T.evaluate_cuts(m, val, at=(10, 50))}
    out["end_to_end"] = e2e
    out["card_after"] = card()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
