"""NumPy restatement of the leave-k-out ranking evaluation (cubecobrarecommender_b200/ml/ranking.py and
cc_rank_targets_f32), for the tests: ranks from the reference's own ranking walk, metrics one cube at a time."""
import numpy as np

from oracle.dae import rank_additions


def target_ranks_np(results, in_cube, hidden):
    """0-based position of every card of ``hidden`` in the full list ``rank_additions(results, in_cube, C)`` (the
    reference's ``argsort()[::-1]`` walk that skips in-cube cards), -1 for a card not in that list."""
    full = rank_additions(results, in_cube, len(results))
    pos = {card: i for i, card in enumerate(full)}
    return np.array([pos.get(int(c), -1) for c in hidden], dtype=np.int64)


def ranking_metrics_np(ranks_per_cube, n_candidates, at=(10, 50)):
    """Means over the cubes with at least one hidden card of recall@k, NDCG@k, hit rate@k, MRR and the mean
    percentile rank, from each cube's hidden-card ranks and candidate count, plus ``cubes``."""
    rows = []
    for ranks, n in zip(ranks_per_cube, n_candidates):
        r = np.asarray(ranks, dtype=np.float64)
        h = len(r)
        if h == 0:
            continue
        row = {}
        for k in at:
            inside = r[r < k]
            row[f"recall_at_{k}"] = len(inside) / min(k, h)
            dcg = sum(1.0 / np.log2(x + 2.0) for x in inside)
            idcg = sum(1.0 / np.log2(i + 2.0) for i in range(min(k, h)))
            row[f"ndcg_at_{k}"] = dcg / idcg
            row[f"hit_rate_at_{k}"] = 1.0 if len(inside) else 0.0
        row["mrr"] = 1.0 / (1.0 + r.min())
        row["mpr"] = r.mean() / (n - 1) if n > 1 else 0.0
        rows.append(row)
    out = {key: float(np.mean([row[key] for row in rows])) for key in rows[0]} if rows else {}
    out["cubes"] = len(rows)
    return out
