"""Leave-k-out baselines, host side: the argument checks of cc_rank_targets_f64 (rejected before any device work, so no
GPU is needed), the Python wrapper's type checks, the baseline name check and the ``--rank-baselines`` CLI flag."""
import ctypes

import pytest

torch = pytest.importorskip("torch")

from cubecobrarecommender_b200 import _lib, build, graph as G
from cubecobrarecommender_b200.ml import train as T


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def test_rank_targets_f64_rejects_bad_arguments(lib):
    fake = ctypes.c_void_p(256)                  # never dereferenced: every call below fails its argument checks
    good = dict(scores=fake, ld=1000, c=1000, batch=4, mp=fake, mi=fake, tp=fake, ti=fake, out=fake)

    def run(**kw):
        a = dict(good, **kw)
        return lib.cc_rank_targets_f64(a["scores"], a["ld"], a["c"], a["batch"], a["mp"], a["mi"], a["tp"], a["ti"],
                                       a["out"], None)
    for name in ("scores", "mp", "mi", "tp", "ti", "out"):
        assert run(**{name: None}) == -1 and "null pointer" in _lib.last_error()
    for kw in (dict(ld=999), dict(ld=1), dict(ld=-1), dict(c=0), dict(c=0, ld=0), dict(c=-5, ld=0), dict(batch=-1),
               dict(batch=-1, ld=0)):
        assert run(**kw) == -1 and "bad sizes" in _lib.last_error(), kw
    assert run(batch=0) == 0                      # nothing to rank: no launch
    assert run(batch=0, ld=0) == 0                # one shared row (stride 0) is a valid layout
    # the float32 entry point keeps ld >= C
    assert lib.cc_rank_targets_f32(fake, 0, 1000, 4, fake, fake, fake, fake, 0, fake, None) == -1
    assert "bad sizes" in _lib.last_error()


def test_rank_targets_wrapper_type_checks(lib):
    z = torch.zeros(2, 5, dtype=torch.float64)
    p = torch.zeros(3, dtype=torch.int64)
    i = torch.zeros(1, dtype=torch.int32)
    with pytest.raises(TypeError, match="sigmoid"):
        G.rank_targets(z, p, i, p, i, sigmoid=True)
    for bad in (torch.zeros(2, 5, dtype=torch.float16), torch.zeros(5, dtype=torch.float64),
                torch.zeros(5, 2, dtype=torch.float64).t()):
        with pytest.raises(TypeError):
            G.rank_targets(bad, p, i, p, i)


def test_ranking_baselines_rejects_unknown_names():
    with pytest.raises(ValueError, match="knn"):
        T.ranking_baselines(None, None, names=("graph", "knn"), at=(10,), holdout=0.2)


BASE = ["5", "64", "run", "0.1", "0.2"]


def test_cli_parsing_rank_baselines():
    o = T.parse_args(BASE + ["--validation-split", "0.2", "--rank-at", "10,50", "--rank-baselines", "graph,popularity"])
    assert o["rank_baselines"] == ("graph", "popularity") and o["rank_at"] == (10, 50)
    o = T.parse_args(BASE + ["--rank-baselines", "popularity", "--rank-at", "10", "--validation-split", "0.1"])
    assert o["rank_baselines"] == ("popularity",)
    assert T.parse_args(BASE + ["--validation-split", "0.2", "--rank-at", "10"])["rank_baselines"] is None
    assert T.parse_args(BASE)["rank_baselines"] is None
    for bad in (BASE + ["--validation-split", "0.2", "--rank-at", "10", "--rank-baselines"],
                BASE + ["--validation-split", "0.2", "--rank-at", "10", "--rank-baselines", "graph,knn"],
                BASE + ["--validation-split", "0.2", "--rank-at", "10", "--rank-baselines", ","],
                BASE + ["--validation-split", "0.2", "--rank-baselines", "graph"],
                BASE + ["--rank-baselines", "graph"]):
        with pytest.raises(SystemExit):
            T.parse_args(bad)
    with pytest.raises(SystemExit, match="knn"):
        T.parse_args(BASE + ["--validation-split", "0.2", "--rank-at", "10", "--rank-baselines", "graph,knn"])
