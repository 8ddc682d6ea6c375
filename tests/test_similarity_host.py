"""Similar cards and cubes, host side: the argument checks of cc_cosine_neg_many_f32 (rejected before any device work,
so no GPU is needed), the query-block plan of ``MLRecommender.nearest`` and the ``--table`` command line."""
import ctypes

import pytest

torch = pytest.importorskip("torch")

from cubecobrarecommender_b200 import _lib, build
from cubecobrarecommender_b200.ml import inference as INF
from cubecobrarecommender_b200.scripts import similarity as SIM


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def test_cosine_neg_many_rejects_bad_arguments(lib):
    fake = ctypes.c_void_p(256)                  # 16-byte aligned, never dereferenced: every call below fails a check
    good = dict(q=fake, ldq=64, nq=10, c=fake, ldc=64, nc=100, dim=64, out=fake, ldo=100)

    def run(**kw):
        a = dict(good, **kw)
        return lib.cc_cosine_neg_many_f32(a["q"], a["ldq"], a["nq"], a["c"], a["ldc"], a["nc"], a["dim"], a["out"],
                                          a["ldo"], None)

    for p in ("q", "c", "out"):
        assert run(**{p: None}) == -1 and "null pointer" in _lib.last_error() and "cc_cosine_neg_many_f32" in _lib.last_error()
    for d in (63, 65, 32, 128, 0):
        assert run(dim=d, ldq=128, ldc=128) == -1 and "dim must be 64" in _lib.last_error(), d
    for kw in (dict(ldq=60), dict(ldc=48), dict(ldo=99), dict(nc=0), dict(nc=-3), dict(nq=-1)):
        assert run(**kw) == -1 and "bad sizes" in _lib.last_error(), kw
    for kw in (dict(ldq=66), dict(ldc=65), dict(q=ctypes.c_void_p(260)), dict(c=ctypes.c_void_p(264))):
        assert run(**kw) == -1 and "16-byte aligned" in _lib.last_error(), kw
    assert run(nq=0) == 0                        # nothing to compare: no launch
    assert run(nq=0, ldo=101, out=ctypes.c_void_p(257)) == 0      # the output takes any stride and alignment


def test_query_block_plan(lib):
    c = 20884
    rows, ldo = INF.plan_query_blocks(20884, c, 50, 1 << 30)
    assert ldo == 20884 and rows == (1 << 30) // (4 * 20884)     # 12 853 rows of distances, no workspace for n <= 2048
    assert INF.plan_query_blocks(100, c, 50, 1 << 30) == (100, 20884)            # never more than the queries
    assert INF.plan_query_blocks(7, 30001, 10, 1 << 30)[1] == 30004                # rows padded to 4 floats
    assert INF.plan_query_blocks(7, 30001, 10, 10)[0] == 1                         # one row even past the budget
    assert INF.plan_query_blocks(0, 5, 1, 1 << 20) == (1, 8)
    # n > 2048: the full-ranking select needs next_pow2(C) 8-byte keys per row on top of the row itself
    per_row = 4 * 20884 + 8 * 32768
    assert lib.cc_topn_workspace_bytes(c, 1, c, 0) == 8 * 32768
    assert INF.plan_query_blocks(20884, c, c, 1 << 30) == ((1 << 30) // per_row, 20884)
    assert INF.plan_query_blocks(20884, c, c, 3 * per_row - 1)[0] == 2


def test_table_arguments_and_positional_form():
    assert SIM.parse_args(["--table", "50", "out.npz"]) == ("table", 50, "out.npz", False)
    assert SIM.parse_args(["--table", "7", "t.npz", "--exclude-self"]) == ("table", 7, "t.npz", True)
    assert SIM.parse_args(["--table", "--exclude-self", "7", "t.npz"]) == ("table", 7, "t.npz", True)
    assert SIM.parse_args(["Lightning_Bolt", "10"]) == ("card", "Lightning Bolt", 10)
    assert SIM.parse_args(["card_17", "5"]) == ("card", "card 17", 5)
    for bad in (["--table", "5"], ["--table", "5", "a.npz", "extra"]):
        with pytest.raises(SystemExit):
            SIM.parse_args(bad)
    with pytest.raises(ValueError):
        SIM.parse_args(["--table", "five", "a.npz"])
