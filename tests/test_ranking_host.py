"""Leave-k-out ranking evaluation, host side: the hidden-card split, the metric formulas (the NumPy restatement and the
torch sums, which run on CPU tensors too), the CLI flag, fit's argument check and the argument checks of
cc_rank_targets_f32 (rejected before any device work, so no GPU is needed)."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from cubecobrarecommender_b200 import _lib, build
from cubecobrarecommender_b200.ml import generator as GEN, ranking as R, train as T
from cubecobrarecommender_b200.sparse import CubeCSR
from cubecobrarecommender_b200.synth import synth_cubes_csr
from ranking_oracle import ranking_metrics_np


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def _csr(k=200, c=500, lo=1, hi=40, seed=3):
    ip, ix = synth_cubes_csr(k, c, size_lo=lo, size_hi=hi, seed=seed)
    return CubeCSR(ip, ix, c)


def _rows(csr):
    return [csr.indices[csr.indptr[b]:csr.indptr[b + 1]] for b in range(csr.num_cubes)]


def test_mix64_is_splitmix64():
    def ref(x):
        m = (1 << 64) - 1
        x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & m
        x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & m
        return x ^ (x >> 31)
    xs = [0, 1, 2, 12345, (1 << 63) + 7, (1 << 64) - 1]
    assert [int(v) for v in R.mix64(np.array(xs, dtype=np.uint64))] == [ref(x) for x in xs]


def test_split_partitions_every_row_and_hides_the_smallest_keys():
    csr = _csr()
    vis, hid, ev = R.holdout_split(csr, 0.2, seed=11)
    assert vis.num_cubes == hid.num_cubes == csr.num_cubes and vis.num_cards == hid.num_cards == csr.num_cards
    for b, (row, v, h) in enumerate(zip(_rows(csr), _rows(vis), _rows(hid))):
        assert set(v).isdisjoint(h) and sorted(np.concatenate([v, h]).tolist()) == sorted(row.tolist())
        s = len(row)
        assert len(h) == (min(s - 1, max(1, int(np.floor(0.2 * s + 0.5)))) if s >= 2 else 0)
        assert ev[b] == (s >= 2)
        # the row order is kept in both parts
        assert list(v) == [x for x in row if x in set(v)] and list(h) == [x for x in row if x in set(h)]
        # the hidden cards are the ones with the smallest (key, card)
        keys = R.mix64(R.mix64(np.uint64(11) ^ np.uint64(b)) + row.astype(np.uint64))
        order = np.lexsort((row, keys))
        assert sorted(h.tolist()) == sorted(row[order[:len(h)]].tolist())


@pytest.mark.parametrize("s,fraction,h", [(1, 0.2, 0), (2, 0.2, 1), (3, 0.2, 1), (2, 0.9, 1), (3, 0.9, 2),
                                          (2, 0.25, 1), (6, 0.25, 2), (10, 0.25, 3), (10, 0.05, 1), (10, 0.15, 2),
                                          (14, 0.25, 4), (0, 0.5, 0)])
def test_hidden_count_formula(s, fraction, h):
    """h = min(s - 1, max(1, floor(fraction * s + 0.5))); 0.25 * 2, 0.25 * 6, 0.25 * 10, 0.05 * 10, 0.15 * 10 and
    0.25 * 14 land exactly on .5 (binary fractions) and round up."""
    assert R.hidden_counts([s], fraction)[0] == h
    csr = CubeCSR.from_lists([list(range(s))], 50)
    _, hid, ev = R.holdout_split(csr, fraction, seed=1)
    assert hid.indptr[-1] == h and ev[0] == (s >= 2)


def test_split_is_deterministic_and_depends_on_the_seed():
    csr = _csr()
    a, b = R.holdout_split(csr, 0.3, seed=5), R.holdout_split(csr, 0.3, seed=5)
    for x, y in zip(a[:2], b[:2]):
        assert np.array_equal(x.indptr, y.indptr) and np.array_equal(x.indices, y.indices)
    c = R.holdout_split(csr, 0.3, seed=6)
    assert not np.array_equal(a[1].indices, c[1].indices)


def test_shard_split_equals_the_whole_split_restricted():
    csr = _csr(k=301)
    vis, hid, ev = R.holdout_split(csr, 0.2, seed=99)
    for world in (2, 3, 8):
        for rank in range(world):
            lo, hi = T.shard_range(csr.num_cubes, rank, world)
            sv, sh, sev = R.holdout_split(csr.shard(rank, world), 0.2, seed=99, cube_offset=lo)
            for whole, part in ((vis, sv), (hid, sh)):
                ref = whole.shard(rank, world)
                assert np.array_equal(ref.indptr, part.indptr) and np.array_equal(ref.indices, part.indices)
            assert np.array_equal(ev[lo:hi], sev)


def test_split_rejects_rows_with_duplicates_and_bad_fractions():
    csr = CubeCSR(np.array([0, 3, 6], dtype=np.int64), np.array([1, 2, 3, 4, 5, 4], dtype=np.int32), 10)
    with pytest.raises(ValueError, match="twice"):
        R.holdout_split(csr, 0.2, seed=0)
    for f in (0.0, 1.0, -0.5):
        with pytest.raises(ValueError):
            R.holdout_split(_csr(k=3), f, seed=0)


def test_generator_caches_the_split_and_counts_skipped_cubes(lib):
    csr = CubeCSR.from_lists([[3], [1, 2], [], [4, 5, 6, 7, 8], [9]], 64)
    rng = np.random.default_rng(0)
    adj = rng.random((64, 64))
    gen = GEN.DataGenerator(adj / adj.sum(1)[:, None], csr, batch_size=2, seed=9, device="cpu")
    state = gen.indices.copy()
    vis, hid, ev = gen.holdout_split(0.2)
    assert gen.holdout_split(0.2)[1] is hid                          # drawn once
    assert ev.tolist() == [False, True, False, True, False] and int((~ev).sum()) == 3
    assert np.array_equal(gen.indices, state)                        # the training shuffle is not touched
    seed = (9 * 0x9E3779B97F4A7C15 + R.HOLDOUT_SEED_SALT) % (1 << 64)
    ref = R.holdout_split(csr, 0.2, seed)[1]
    assert np.array_equal(hid.indices, ref.indices)
    # a subset generator (validation split) draws for its own cubes
    _, val = gen.split(0.4)
    assert val._holdout is None and val.holdout_split(0.2)[1].num_cubes == 2


def test_ranking_metrics_np_hand_computed():
    # cube 0: h = 2 < k = 3, ranks 0 and 4 of n = 11 candidates
    # cube 1: h = 4 > k = 3, ranks 1, 2, 7, 9 of n = 11
    # cube 2: no hit (rank 5, h = 1); cube 3: n = 1 (the one candidate is the hidden card, rank 0); cube 4: h = 0
    ranks = [[0, 4], [1, 2, 7, 9], [5], [0], []]
    n = [11, 11, 6, 1, 10]
    out = ranking_metrics_np(ranks, n, at=(3,))
    l2 = lambda x: 1.0 / np.log2(x + 2.0)
    per = {
        "recall_at_3": [1 / 2, 2 / 3, 0.0, 1.0],
        "ndcg_at_3": [l2(0) / (l2(0) + l2(1)), (l2(1) + l2(2)) / (l2(0) + l2(1) + l2(2)), 0.0, 1.0],
        "hit_rate_at_3": [1.0, 1.0, 0.0, 1.0],
        "mrr": [1.0, 1 / 2, 1 / 6, 1.0],
        "mpr": [2 / 10, 4.75 / 10, 5 / 5, 0.0],
    }
    assert out["cubes"] == 4
    for key, vals in per.items():
        assert out[key] == pytest.approx(np.mean(vals), rel=1e-14), key


def test_ranking_sums_equal_the_numpy_restatement():
    """ranking.ranking_sums (torch segment ops, here on CPU tensors) against ranking_metrics_np on random cubes."""
    rng = np.random.default_rng(4)
    k, at = 300, (1, 10, 50)
    h = rng.integers(0, 40, size=k)
    h[:3] = 0
    n = h + rng.integers(0, 3000, size=k)
    n[5] = 1; h[5] = 1
    ranks = [rng.choice(max(n_, 1), size=h_, replace=False) for h_, n_ in zip(h, n)]
    ip = np.zeros(k + 1, dtype=np.int64); np.cumsum(h, out=ip[1:])
    flat = torch.from_numpy(np.concatenate(ranks).astype(np.int32))
    sums = R.ranking_sums(flat, torch.from_numpy(ip), torch.from_numpy(n), at).numpy()
    ref = ranking_metrics_np(ranks, n, at)
    assert sums[0] == ref["cubes"] == k - int((h == 0).sum())
    for name, v in zip(R.metric_names(at), sums[1:]):
        assert v / sums[0] == pytest.approx(ref[name], rel=1e-12), name


def test_cli_parsing_rank_at():
    o = T.parse_args(["5", "64", "run", "0.1", "0.2", "--validation-split", "0.2", "--rank-at", "10,50"])
    assert o["rank_at"] == (10, 50) and o["validation_split"] == 0.2
    o = T.parse_args(["5", "64", "run", "0.1", "0.2", "--rank-at", "20", "--validation-split", "0.1"])
    assert o["rank_at"] == (20,)
    assert T.parse_args(["5", "64", "run", "0.1", "0.2"])["rank_at"] is None
    for bad in (["5", "64", "run", "0.1", "0.2", "--validation-split", "0.2", "--rank-at"],
                ["5", "64", "run", "0.1", "0.2", "--validation-split", "0.2", "--rank-at", "0,10"],
                ["5", "64", "run", "0.1", "0.2", "--validation-split", "0.2", "--rank-at", "ten"],
                ["5", "64", "run", "0.1", "0.2", "--rank-at", "10"]):
        with pytest.raises(SystemExit):
            T.parse_args(bad)


def test_fit_ranking_at_needs_validation_data(lib):
    ip, ix = synth_cubes_csr(10, 64, size_lo=3, size_hi=12, seed=4)
    rng = np.random.default_rng(0)
    adj = rng.random((64, 64))
    gen = GEN.DataGenerator(adj / adj.sum(1)[:, None], CubeCSR(ip, ix, 64), batch_size=4, seed=9, device="cpu")
    with pytest.raises(ValueError, match="ranking_at"):
        T.fit(None, gen, epochs=1, reg=0.1, ranking_at=(10,))
    with pytest.raises(ValueError, match="ranking_at"):
        T.fit(None, gen, epochs=1, reg=0.1, ranking_at=(0,), validation_split=0.2)


def test_rank_targets_rejects_bad_arguments(lib):
    fake = ctypes.c_void_p(256)                  # never dereferenced: every call below fails its argument checks
    good = dict(scores=fake, ld=1000, c=1000, batch=4, mp=fake, mi=fake, tp=fake, ti=fake, out=fake)

    def run(**kw):
        a = dict(good, **kw)
        return lib.cc_rank_targets_f32(a["scores"], a["ld"], a["c"], a["batch"], a["mp"], a["mi"], a["tp"], a["ti"], 1,
                                       a["out"], None)
    for name in ("scores", "mp", "mi", "tp", "ti", "out"):
        assert run(**{name: None}) == -1 and "null pointer" in _lib.last_error()
    for kw in (dict(ld=999), dict(c=0), dict(c=0, ld=0), dict(batch=-1)):
        assert run(**kw) == -1 and "bad sizes" in _lib.last_error()
    assert run(batch=0) == 0                      # nothing to rank: no launch
