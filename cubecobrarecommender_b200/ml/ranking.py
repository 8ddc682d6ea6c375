"""Leave-k-out ranking evaluation of the recommender (recall@k and NDCG@k as in Liang et al. 2018, Mult-VAE, plus MRR
and the mean percentile rank).

A held-out cube is split into visible and hidden cards (:func:`holdout_split`); the model sees the visible ones and
ranks every other card, and each hidden card's 0-based position in that list (``MLRecommender.target_ranks_device``)
is what the metrics are computed from (:func:`ranking_sums`).  ``train.evaluate_recommendations`` puts the two together.
"""
from __future__ import annotations

import numpy as np
import torch

from ..sparse import CubeCSR

# the hidden-card draw: its own seed (the generator seed mixed with this salt), fixed for the generator's lifetime
HOLDOUT_SEED_SALT = 0x4E1D0B7C

_M1, _M2 = np.uint64(0xBF58476D1CE4E5B9), np.uint64(0x94D049BB133111EB)


def mix64(x):
    """The splitmix64 finaliser, in wrapping uint64 arithmetic (element-wise)."""
    x = np.asarray(x, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = (x ^ (x >> np.uint64(30))) * _M1
        x = (x ^ (x >> np.uint64(27))) * _M2
    return x ^ (x >> np.uint64(31))


def hidden_counts(sizes, fraction):
    """Cards hidden per cube: ``min(s - 1, max(1, floor(fraction * s + 0.5)))`` for a cube of s >= 2 cards, else 0."""
    s = np.asarray(sizes, dtype=np.int64)
    h = np.minimum(s - 1, np.maximum(1, np.floor(float(fraction) * s + 0.5).astype(np.int64)))
    return np.where(s >= 2, h, 0)


def holdout_split(csr: CubeCSR, fraction: float, seed: int, cube_offset: int = 0):
    """``(visible, hidden, evaluated)``: two CSRs over the same cubes, each row a disjoint split of the cube's cards
    (row order kept), and a bool (K,) array, False for cubes of fewer than two cards (their row stays visible).  Cube
    ``b`` hides the :func:`hidden_counts` cards with the smallest ``(mix64(mix64(seed ^ (b + cube_offset)) + card),
    card)``, so the split of rows [lo, hi) with ``cube_offset = lo`` is the whole set's split restricted to them.  Rows
    must be sets."""
    if not 0.0 < float(fraction) < 1.0:
        raise ValueError(f"holdout fraction must lie in (0, 1), got {fraction}")
    ip = np.ascontiguousarray(csr.indptr, dtype=np.int64)
    card = np.ascontiguousarray(csr.indices).astype(np.int64)
    k = csr.num_cubes
    sizes = np.diff(ip)
    cube = np.repeat(np.arange(k, dtype=np.int64), sizes)
    by_card = np.lexsort((card, cube))
    sc, cc = card[by_card], cube[by_card]
    dup = (sc[1:] == sc[:-1]) & (cc[1:] == cc[:-1])
    if dup.any():
        raise ValueError(f"cube {int(cc[1:][dup][0]) + cube_offset} lists card {int(sc[1:][dup][0])} twice: rows must be sets")
    h = hidden_counts(sizes, fraction)
    key = mix64(mix64(np.uint64(int(seed) % (1 << 64)) ^ (cube + int(cube_offset)).astype(np.uint64)) + card.astype(np.uint64))
    order = np.lexsort((card, key, cube))                 # by cube, then key, then card
    pos = np.arange(len(card), dtype=np.int64) - ip[cube[order]]
    hidden = np.empty(len(card), dtype=bool)
    hidden[order] = pos < h[cube[order]]

    def part(sel):
        out_ip = np.zeros(k + 1, dtype=np.int64)
        np.cumsum(np.bincount(cube[sel], minlength=k), out=out_ip[1:])
        return CubeCSR(out_ip, np.ascontiguousarray(csr.indices[sel], dtype=np.int32), csr.num_cards)

    return part(~hidden), part(hidden), sizes >= 2


def metric_names(at):
    """Keys of :func:`ranking_sums` / ``evaluate_recommendations`` in order, without ``cubes``."""
    names = []
    for k in at:
        names += [f"recall_at_{k}", f"ndcg_at_{k}", f"hit_rate_at_{k}"]
    return names + ["mrr", "mpr"]


def ranking_sums(ranks: torch.Tensor, hidden_indptr: torch.Tensor, n_candidates: torch.Tensor, at) -> torch.Tensor:
    """float64 device vector ``[cubes, *per-cube sums in metric_names(at) order]`` over the cubes with at least one
    hidden card, without a host sync.  ``ranks``: int32 (nnz,) 0-based ranks of the hidden cards, aligned with the
    hidden CSR ``hidden_indptr`` (int64 (K + 1,)); ``n_candidates``: (K,) cards each cube's ranking ran over
    (C - visible).  Per cube, with h hidden cards of ranks r_t and n candidates:
    recall@k = #{r_t < k} / min(k, h); ndcg@k = sum_{r_t < k} 1 / log2(r_t + 2) / sum_{i < min(k, h)} 1 / log2(i + 2);
    hit_rate@k = [any r_t < k]; mrr = 1 / (1 + min r_t); mpr = mean r_t / (n - 1), 0 when n = 1."""
    dev = ranks.device
    h = (hidden_indptr[1:] - hidden_indptr[:-1]).to(torch.int64)
    kk = h.numel()
    seg = torch.repeat_interleave(torch.arange(kk, device=dev), h, output_size=ranks.numel())
    r = ranks.to(torch.float64)
    live = h > 0
    hd = h.to(torch.float64)

    def per_cube(v):
        return torch.zeros(kk, dtype=torch.float64, device=dev).index_add_(0, seg, v)

    def total(v):
        return torch.where(live, v, torch.zeros_like(v)).sum()

    disc = 1.0 / torch.log2(r + 2.0)
    kmax = max(int(k) for k in at)
    ideal = torch.cat([torch.zeros(1, dtype=torch.float64, device=dev),
                       torch.cumsum(1.0 / torch.log2(torch.arange(kmax, dtype=torch.float64, device=dev) + 2.0), 0)])
    out = [live.to(torch.float64).sum()]
    for k in at:
        k = int(k)
        inside = r < k
        hits = per_cube(inside.to(torch.float64))
        cap = torch.clamp(h, max=k)
        out.append(total(hits / cap.clamp(min=1).to(torch.float64)))
        out.append(total(per_cube(torch.where(inside, disc, torch.zeros_like(disc))) / ideal[cap].clamp(min=1e-300)))
        out.append(total((hits > 0).to(torch.float64)))
    best = torch.full((kk,), float("inf"), dtype=torch.float64, device=dev).scatter_reduce_(0, seg, r, "amin")
    out.append(total(1.0 / (1.0 + best)))
    span = n_candidates.to(torch.float64) - 1.0
    mean_r = per_cube(r) / hd.clamp(min=1.0)
    out.append(total(torch.where(span > 0, mean_r / span.clamp(min=1.0), torch.zeros_like(mean_r))))
    return torch.stack(out)
