"""Cut-list evaluation, host side: the intruder draw (``ranking.intruder_split`` and its generator cache), the argument
checks of cc_rank_cuts_f32 / _f64 (rejected before any device work, so no GPU is needed), the ``--rank-cuts`` flag,
``fit``'s argument check and ``ranking_sums`` against a NumPy restatement with n = s + m candidates."""
import copy
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from cubecobrarecommender_b200 import _lib, build
from cubecobrarecommender_b200.ml import generator as GEN, ranking as R, train as T
from cubecobrarecommender_b200.sparse import CubeCSR
from cubecobrarecommender_b200.synth import synth_cubes_csr
from ranking_oracle import ranking_metrics_np


def _rows(csr, b):
    return csr.indices[csr.indptr[b]:csr.indptr[b + 1]]


def _csr(k=300, c=500, lo=0, hi=60, seed=3):
    ip, ix = synth_cubes_csr(k, c, size_lo=max(lo, 1), size_hi=hi, seed=seed)
    rows = [ix[ip[b]:ip[b + 1]].tolist() for b in range(k)]
    if lo == 0:                                   # a few empty cubes and a one-card cube
        rows[3], rows[50], rows[51] = [], [], [rows[51][0]]
    return CubeCSR.from_lists(rows, c)


def _restated(csr, fraction, seed):
    """The draw one cube at a time: donor, eligible cards, key order, count."""
    k = csr.num_cubes
    out = []
    for b in range(k):
        hb = R.mix64(np.uint64(seed) ^ np.uint64(b))
        d = int((b + 1 + int(hb % np.uint64(k - 1))) % k)
        own = _rows(csr, b)
        s = len(own)
        m = max(1, int(np.floor(fraction * s + 0.5))) if s else 0
        elig = [int(x) for x in _rows(csr, d) if x not in set(own.tolist())]
        keyed = sorted(elig, key=lambda x: (int(R.mix64(hb + np.uint64(x))), x))
        out.append((d, own, keyed[:m]))
    return out


@pytest.mark.parametrize("fraction", [0.2, 0.05, 1.0])
def test_intruder_split_matches_its_definition(fraction):
    csr = _csr()
    cor, intr, ev = R.intruder_split(csr, fraction, seed=11)
    ref = _restated(csr, fraction, 11)
    assert cor.num_cubes == intr.num_cubes == csr.num_cubes and cor.num_cards == intr.num_cards == csr.num_cards
    assert cor.indices.dtype == intr.indices.dtype == np.int32
    short = 0
    for b, (d, own, want) in enumerate(ref):
        got = _rows(intr, b)
        assert d != b
        assert got.tolist() == want, b                                   # count, key order
        assert not set(got.tolist()) & set(own.tolist())                 # disjoint from the cube
        assert set(got.tolist()) <= set(_rows(csr, d).tolist())          # from the donor
        assert _rows(cor, b).tolist() == own.tolist() + want             # own cards, then intruders
        assert ev[b] == (len(own) >= 1 and len(want) >= 1)
        short += len(own) >= 1 and len(want) < max(1, int(np.floor(fraction * len(own) + 0.5)))
    assert not ev[3] and not ev[50] and ev[51]
    if fraction == 1.0:
        assert short > 0                                                  # donors with too few eligible cards


def test_intruder_split_is_deterministic_and_seeded():
    csr = _csr(seed=4)
    a = R.intruder_split(csr, 0.2, seed=5)
    b = R.intruder_split(csr, 0.2, seed=5)
    c = R.intruder_split(csr, 0.2, seed=6)
    for x, y in zip(a, b):
        assert np.array_equal(x.indices if hasattr(x, "indices") else x, y.indices if hasattr(y, "indices") else y)
    assert not np.array_equal(a[1].indices, c[1].indices)


@pytest.mark.parametrize("world", [2, 3, 8])
def test_shards_of_the_whole_split_are_its_rows(world):
    csr = _csr(seed=9)
    cor, intr, _ = R.intruder_split(csr, 0.2, seed=2)
    for r in range(world):
        lo, hi = T.shard_range(csr.num_cubes, r, world)
        for whole in (cor, intr):
            part, rows = whole.shard(r, world), whole.rows(np.arange(lo, hi))
            assert np.array_equal(part.indptr, rows.indptr) and np.array_equal(part.indices, rows.indices)


def test_intruder_split_rejects_bad_input():
    csr = _csr(k=60)
    for f in (0.0, -0.1, 1.01, 2.0):
        with pytest.raises(ValueError, match="fraction"):
            R.intruder_split(csr, f, seed=0)
    with pytest.raises(ValueError, match="twice"):
        R.intruder_split(CubeCSR(np.array([0, 3, 4]), np.array([1, 2, 1, 5], dtype=np.int32), 10), 0.2, seed=0)
    with pytest.raises(ValueError, match="2 cubes"):
        R.intruder_split(CubeCSR(np.array([0, 3]), np.array([1, 2, 3], dtype=np.int32), 10), 0.2, seed=0)


def _host_generator(csr, seed):
    g = GEN.DataGenerator.__new__(GEN.DataGenerator)     # the cached draws need no device state
    g.csr, g.seed, g.N_cubes, g.N_cards = csr, seed, csr.num_cubes, csr.num_cards
    g._intruders = None
    return g


def test_generator_caches_the_split_per_fraction():
    csr = _csr(seed=12)
    g = _host_generator(csr, seed=7)
    a = g.intruder_split(0.2)
    assert g.intruder_split(0.2) is a and g.intruder_split(0.3) is not a
    seed = (7 * 0x9E3779B97F4A7C15 + R.INTRUDER_SEED_SALT) % (1 << 64)
    ref = R.intruder_split(csr, 0.2, seed)
    assert np.array_equal(a[0].indices, ref[0].indices) and np.array_equal(a[1].indices, ref[1].indices)
    h = copy.copy(g)
    h.seed = 8
    h._intruders = None
    assert not np.array_equal(h.intruder_split(0.2)[1].indices, a[1].indices)


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


@pytest.mark.parametrize("name", ["cc_rank_cuts_f32", "cc_rank_cuts_f64"])
def test_rank_cuts_rejects_bad_arguments(lib, name):
    fake = ctypes.c_void_p(256)                  # never dereferenced: every call below fails its argument checks
    good = dict(scores=fake, ld=1000, c=1000, batch=4, lp=fake, li=fake, tp=fake, ti=fake, out=fake)
    is32 = name.endswith("f32")

    def run(**kw):
        a = dict(good, **kw)
        args = [a["scores"], a["ld"], a["c"], a["batch"], a["lp"], a["li"], a["tp"], a["ti"]]
        return getattr(lib, name)(*args, *([1] if is32 else []), a["out"], None)
    for p in ("scores", "lp", "li", "tp", "ti", "out"):
        assert run(**{p: None}) == -1 and "null pointer" in _lib.last_error() and name in _lib.last_error()
    for kw in (dict(ld=999), dict(ld=1), dict(ld=-1), dict(c=0), dict(c=0, ld=0), dict(c=-5, ld=0), dict(batch=-1)):
        assert run(**kw) == -1 and "bad sizes" in _lib.last_error(), kw
    assert run(c=2_000_000, ld=2_000_000) == -1 and "shared memory" in _lib.last_error()
    assert run(batch=0) == 0                      # nothing to rank: no launch
    if is32:                                      # the float32 entry point keeps ld >= C
        assert run(ld=0) == -1 and "bad sizes" in _lib.last_error()
    else:
        assert run(batch=0, ld=0) == 0            # one shared row (stride 0) is a valid layout


def test_rank_cuts_wrapper_type_checks(lib):
    from cubecobrarecommender_b200 import graph as G
    z = torch.zeros(2, 5, dtype=torch.float64)
    p = torch.zeros(3, dtype=torch.int64)
    i = torch.zeros(1, dtype=torch.int32)
    with pytest.raises(TypeError, match="sigmoid"):
        G.rank_cuts(z, p, i, p, i, sigmoid=True)
    for bad in (torch.zeros(2, 5, dtype=torch.float16), torch.zeros(5, dtype=torch.float64),
                torch.zeros(5, 2, dtype=torch.float64).t()):
        with pytest.raises(TypeError):
            G.rank_cuts(bad, p, i, p, i)


BASE = ["5", "64", "run", "0.1", "0.2"]


def test_cli_parsing_rank_cuts():
    o = T.parse_args(BASE + ["--validation-split", "0.2", "--rank-at", "10,50", "--rank-cuts"])
    assert o["rank_cuts"] is True and o["rank_at"] == (10, 50)
    o = T.parse_args(BASE + ["--rank-cuts", "--rank-at", "10", "--validation-split", "0.1", "--rank-baselines", "graph"])
    assert o["rank_cuts"] and o["rank_baselines"] == ("graph",) and o["epochs"] == 5
    assert T.parse_args(BASE + ["--validation-split", "0.2", "--rank-at", "10"])["rank_cuts"] is False
    assert T.parse_args(BASE)["rank_cuts"] is False
    for bad in (BASE + ["--rank-cuts"], BASE + ["--validation-split", "0.2", "--rank-cuts"]):
        with pytest.raises(SystemExit, match="--rank-at"):
            T.parse_args(bad)


def test_fit_rejects_cuts_without_ranking_at():
    with pytest.raises(ValueError, match="ranking_at"):
        T.fit(None, None, 1, 0.1, ranking_cuts=True)


def test_ranking_baselines_rejects_unknown_task():
    with pytest.raises(ValueError, match="task"):
        T.ranking_baselines(None, None, at=(10,), task="swaps")


def test_ranking_sums_equal_the_restatement_with_s_plus_m_candidates():
    csr = _csr(seed=21)
    cor, intr, ev = R.intruder_split(csr, 0.2, seed=3)
    rng = np.random.default_rng(0)
    n = np.diff(cor.indptr)
    ranks, per_cube = [], []
    for b in range(csr.num_cubes):                 # distinct ranks among the s + m corrupted cards
        m = int(intr.indptr[b + 1] - intr.indptr[b])
        r = rng.choice(n[b], size=m, replace=False) if m else np.zeros(0, dtype=np.int64)
        ranks.append(r); per_cube.append(r)
    at = (1, 10, 50)
    sums = R.ranking_sums(torch.from_numpy(np.concatenate(ranks).astype(np.int32)), torch.from_numpy(intr.indptr),
                          torch.from_numpy(n), at).numpy()
    ref = ranking_metrics_np(per_cube, n, at)
    assert sums[0] == ref["cubes"] == int(ev.sum())
    for key, v in zip(R.metric_names(at), sums[1:] / sums[0]):
        assert v == pytest.approx(ref[key], rel=1e-12, abs=1e-15), key
