"""Leave-k-out baselines on the GPU: cc_rank_targets_f64 against NumPy's stable argsort and against the float64 top-N
select, the graph recommender's ranks against ``oracle.graph.simple_recs``, the popularity ranks against their NumPy
restatement, ``evaluate_recommendations`` / ``ranking_baselines`` against the metric oracle, their lack of side effects,
the graph beating popularity where co-occurrence carries the signal, the CLI flag and a two-GPU run."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from cubecobrarecommender_b200 import _lib, graph as G
from cubecobrarecommender_b200.ml import generator as GEN, ranking as R, train as T
from cubecobrarecommender_b200.sparse import CubeCSR
from cubecobrarecommender_b200.synth import synth_cubes_csr
from oracle import graph as og
from ranking_oracle import ranking_metrics_np
from test_gpu_ranking import _csr_dev, _expected, _rows_for

call, ptr, stream_ptr = _lib.call, _lib.ptr, _lib.stream_ptr
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SPECIAL = np.array([np.inf, -np.inf, 0.0, -0.0, 5e-324, -5e-324, 2.5e-310, -2.5e-310, 1.0, -1.0, 1e308, -1e308],
                   dtype=np.float64)


def _scores64(kind, b, c, rng):
    if kind == "normal":
        return rng.standard_normal((b, c)) * 3
    if kind == "ties":                                                     # a few integers: long tie runs
        return rng.integers(-2, 3, size=(b, c)).astype(np.float64)
    # +-inf, -0.0 next to +0.0, subnormals, a few ordinary values
    return rng.choice(SPECIAL, size=(b, c))


def _layout64(host, layout):
    """Device rows: ``vector`` an even ld on a 16-byte aligned base (+inf past each row, which must never be read),
    ``scalar`` an odd ld on a base 8 bytes off alignment, ``shared`` row 0 expanded to every cube (ld = 0)."""
    b, c = host.shape
    if layout == "shared":
        return torch.from_numpy(host[0].copy()).cuda().expand(b, c)
    if layout == "vector":
        ld = c + (c & 1)
        buf = torch.full((b, ld), float("inf"), dtype=torch.float64, device="cuda")
        buf[:, :c] = torch.from_numpy(host).cuda()
        return buf[:, :c]
    ld = c + 1 if (c + 1) % 2 else c + 2
    flat = torch.full((b * ld + 1,), float("inf"), dtype=torch.float64, device="cuda")
    view = flat[1:].view(b, ld)
    view[:, :c] = torch.from_numpy(host).cuda()
    return view[:, :c]


@pytest.mark.parametrize("c", [20884, 1000, 129, 3])
@pytest.mark.parametrize("layout", ["vector", "scalar", "shared"])
@pytest.mark.parametrize("kind", ["normal", "ties", "special"])
def test_rank_targets_f64_equals_stable_argsort(c, layout, kind):
    rng = np.random.default_rng(c + 11 * len(layout) + len(kind))
    rows = _rows_for(c, rng)
    host = _scores64(kind, len(rows), c, rng)
    if layout == "shared":
        host[:] = host[0]
    sc = _layout64(host, layout)
    if layout == "vector":
        assert sc.stride(0) % 2 == 0 and sc.data_ptr() % 16 == 0
    elif layout == "scalar":
        assert sc.stride(0) % 2 == 1 and sc.data_ptr() % 16 == 8
    else:
        assert sc.stride(0) == 0
    mp, mi, _ = _csr_dev([m for m, _ in rows])
    tp, ti, tip = _csr_dev([t for _, t in rows])
    got = G.rank_targets(sc, mp, mi, tp, ti).cpu().numpy()
    for b, (mask, targets) in enumerate(rows):
        assert np.array_equal(got[tip[b]:tip[b + 1]], _expected(host[b], mask, targets)), b


def test_rank_targets_f64_batch_zero_is_a_no_op():
    z = torch.zeros(1, 10, dtype=torch.float64, device="cuda")
    p = torch.zeros(2, dtype=torch.int64, device="cuda")
    i = torch.zeros(1, dtype=torch.int32, device="cuda")
    out = torch.full((1,), 123, dtype=torch.int32, device="cuda")
    call("cc_rank_targets_f64", ptr(z), 0, 10, 0, ptr(p), ptr(i), ptr(p), ptr(i), ptr(out), stream_ptr())
    assert int(out.item()) == 123


@pytest.mark.parametrize("shared", [False, True])
def test_rank_targets_f64_agrees_with_the_select(shared):
    """2048 x 20 884 float64 rows with many ties (quarter steps): every target of rank r < 50 is what
    topn_masked(float64, n=50) returns at slot r, and every returned target sits at the slot of its rank."""
    b, c, n = 2048, 20884, 50
    ip, ix = synth_cubes_csr(b, c, seed=22)
    vis, hid, _ = R.holdout_split(CubeCSR(ip, ix, c), 0.2, seed=4)
    g = torch.Generator(device="cuda").manual_seed(6)
    z = torch.round(torch.randn(1 if shared else b, c, device="cuda", dtype=torch.float64, generator=g) * 8) / 4
    z[:, :300] += 3
    z = z.expand(b, c) if shared else z
    mp, mi = (torch.from_numpy(a).cuda() for a in (vis.indptr, vis.indices))
    tp, ti = (torch.from_numpy(a).cuda() for a in (hid.indptr, hid.indices))
    ranks = G.rank_targets(z, mp, mi, tp, ti).cpu().numpy()
    ids = G.topn_masked(z.contiguous(), mp, mi, n)[0].cpu().numpy()
    assert (ranks >= 0).all()
    cube = np.repeat(np.arange(b), np.diff(hid.indptr))
    top = ranks < n
    assert top.sum() > 1000
    assert np.array_equal(ids[cube[top], ranks[top]], hid.indices[top])
    rank_of = {(int(q), int(t)): int(r) for q, t, r in zip(cube, hid.indices, ranks)}
    seen = 0
    for q in range(b):
        for slot, card in enumerate(ids[q]):
            if (q, int(card)) in rank_of:
                assert rank_of[q, int(card)] == slot
                seen += 1
    assert seen == int(top.sum())


# ------------------------------------------------------------------ the two baselines
def _graph_oracle(m_host, vis, hid):
    """Per cube: the position of each hidden card in ``simple_recs(stable=True)`` of the visible cards."""
    out = []
    for b in range(vis.num_cubes):
        cube = np.zeros(vis.num_cards)
        cube[vis.indices[vis.indptr[b]:vis.indptr[b + 1]]] = 1
        h = hid.indices[hid.indptr[b]:hid.indptr[b + 1]]
        if len(h) == 0:
            out.append(np.zeros(0, dtype=np.int64))
            continue
        pos = {card: i for i, card in enumerate(og.simple_recs(cube, m_host, stable=True))}
        out.append(np.array([pos.get(int(t), -1) for t in h], dtype=np.int64))
    return out


def _popularity_oracle(train_csr, vis, hid):
    counts = np.bincount(train_csr.indices, minlength=train_csr.num_cards).astype(np.float64)
    return [_expected(counts, vis.indices[vis.indptr[b]:vis.indptr[b + 1]], hid.indices[hid.indptr[b]:hid.indptr[b + 1]])
            for b in range(vis.num_cubes)]


def _m_oracle(csr):
    return og.adjacency_from_counts(og.cooc_counts(csr.indptr, csr.indices, csr.num_cards))


def test_graph_target_ranks_equal_simple_recs():
    """Cubes of 5-300 cards (several pairwise leaves each) scored against M of 2000 other cubes, in chunks of a few cubes
    (budget of ~6 cubes), one cube per chunk and one chunk: every hidden card sits where simple_recs lists it."""
    c = 1000
    ip, ix = synth_cubes_csr(2000, c, size_lo=10, size_hi=200, seed=41)
    train = CubeCSR(ip, ix, c)
    ip, ix = synth_cubes_csr(300, c, size_lo=5, size_hi=300, seed=42)
    vis, hid, ev = R.holdout_split(CubeCSR(ip, ix, c), 0.2, seed=7)
    m = G.build_graph(train, "cuda", want_mhat=False, want_neg=False).m64
    m_host = m.cpu().numpy()
    assert np.array_equal(m_host, _m_oracle(train))
    ref = np.concatenate(_graph_oracle(m_host, vis, hid))
    assert (ref >= 0).all() and ev.sum() == 300
    small = G.GraphRecommender(m, budget_bytes=6 * 3 * c * 8)
    assert np.array_equal(small.target_ranks_device(vis, hid).cpu().numpy(), ref)
    assert np.array_equal(G.GraphRecommender(m).target_ranks_device(vis, hid).cpu().numpy(), ref)
    sel = np.arange(20)
    one = G.GraphRecommender(m, budget_bytes=1).target_ranks_device(vis.rows(sel), hid.rows(sel)).cpu().numpy()
    assert np.array_equal(one, ref[:int(hid.indptr[20])])
    # the slot is the one GraphRecommender.recs lists the card at
    ids = small.recs(vis.rows(sel), 50)[0].cpu().numpy()
    for b in range(20):
        for t, r in zip(hid.indices[hid.indptr[b]:hid.indptr[b + 1]], ref[hid.indptr[b]:hid.indptr[b + 1]]):
            if r < 50:
                assert ids[b, r] == t


def test_popularity_target_ranks_equal_numpy():
    c = 20884
    ip, ix = synth_cubes_csr(3000, c, seed=43)
    train = CubeCSR(ip, ix, c)
    ip, ix = synth_cubes_csr(500, c, size_lo=1, size_hi=400, seed=44)
    vis, hid, _ = R.holdout_split(CubeCSR(ip, ix, c), 0.25, seed=8)
    rec = G.PopularityRecommender(train, "cuda")
    assert np.array_equal(rec.scores.cpu().numpy(), np.bincount(train.indices, minlength=c))
    got = rec.target_ranks_device(vis, hid).cpu().numpy()
    assert np.array_equal(got, np.concatenate(_popularity_oracle(train, vis, hid)))


def _generator(c, k, batch, seed, size_lo=2, size_hi=80, csr=None):
    if csr is None:
        ip, ix = synth_cubes_csr(k, c, size_lo=size_lo, size_hi=size_hi, seed=seed)
        csr = CubeCSR(ip, ix, c)
    gr = G.build_graph(csr, "cuda", want_m64=False)
    return GEN.DataGenerator(gr.mhat, csr, batch_size=batch, noise=0.2, seed=seed)


def _baseline_oracle(train, val, at, holdout):
    vis, hid, _ = val.holdout_split(holdout)
    n_cand = val.N_cards - np.diff(vis.indptr)
    return {"graph": ranking_metrics_np(_graph_oracle(_m_oracle(train.csr), vis, hid), n_cand, at),
            "popularity": ranking_metrics_np(_popularity_oracle(train.csr, vis, hid), n_cand, at)}


def test_ranking_baselines_equal_the_oracle():
    """evaluate_recommendations over both baselines (built from the training cubes only) equals the metric oracle on
    the oracle ranks; a cube of one card is skipped like in the ML evaluation."""
    c, at, holdout = 1000, (1, 10, 50), 0.25
    ip, ix = synth_cubes_csr(495, c, size_lo=2, size_hi=160, seed=45)
    rows = [ix[ip[b]:ip[b + 1]].tolist() for b in range(495)] + [[7 * i] for i in range(5)]   # 5 one-card cubes
    gen = _generator(c, 0, 64, seed=45, csr=CubeCSR.from_lists(rows, c))
    train, val = gen.split(0.3)
    res = T.ranking_baselines(train, val, at=at, holdout=holdout)
    assert list(res) == ["graph", "popularity"]
    ref = _baseline_oracle(train, val, at, holdout)
    for name in res:
        assert res[name]["cubes"] == ref[name]["cubes"] and res[name]["skipped"] == val.N_cubes - ref[name]["cubes"] > 0
        for key in R.metric_names(at):
            assert res[name][key] == pytest.approx(ref[name][key], rel=1e-12, abs=1e-15), (name, key)
    # evaluate_recommendations takes the recommenders directly, too
    direct = T.evaluate_recommendations(G.PopularityRecommender(train.csr, "cuda"), val, at=at, holdout=holdout)
    assert direct == res["popularity"]
    assert T.ranking_baselines(train, val, names=("popularity",), at=at, holdout=holdout) == {"popularity": direct}


def test_baselines_have_no_side_effects():
    c = 512
    gen = _generator(c, 300, 32, seed=46)
    train, val = gen.split(0.25)
    split = val.holdout_split(0.2)
    m = G.build_graph(train.csr, "cuda", want_mhat=False, want_neg=False).m64
    graph_rec, pop = G.GraphRecommender(m, budget_bytes=1 << 20), G.PopularityRecommender(train.csr, "cuda")
    m0, p0 = m.clone(), pop.scores.clone()
    r1 = {n: T.evaluate_recommendations(r, val, at=(10, 50)) for n, r in (("graph", graph_rec), ("popularity", pop))}
    r2 = {n: T.evaluate_recommendations(r, val, at=(10, 50)) for n, r in (("graph", graph_rec), ("popularity", pop))}
    torch.cuda.synchronize()
    assert torch.equal(m, m0) and torch.equal(pop.scores, p0)
    assert val.holdout_split(0.2) is split and all(a is b for a, b in zip(val.holdout_split(0.2), split))
    assert r1 == r2
    # ranking_baselines frees its graph: no (C, C) matrix stays allocated
    del graph_rec, m, m0
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    out = T.ranking_baselines(train, val, at=(10, 50), holdout=0.2)
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() - before < c * c * 4
    assert out["graph"] == r1["graph"] and out["popularity"] == r1["popularity"]


def _pool_cubes(k, pools, per_pool, rng):
    """Cubes drawn from one of ``pools`` disjoint card pools each, with a skewed popularity inside the pool."""
    w = 1.0 / (np.arange(per_pool) + 5.0)
    w /= w.sum()
    rows = []
    for _ in range(k):
        p = rng.integers(pools)
        s = rng.integers(20, 50)
        rows.append(np.sort(p * per_pool + rng.choice(per_pool, size=s, replace=False, p=w)))
    return CubeCSR.from_lists([r.tolist() for r in rows], pools * per_pool)


def test_graph_beats_popularity_on_disjoint_pools():
    rng = np.random.default_rng(47)
    csr = _pool_cubes(1200, 4, 150, rng)
    gen = _generator(csr.num_cards, 0, 64, seed=47, csr=csr)
    train, val = gen.split(0.25)
    res = T.ranking_baselines(train, val, at=(10,), holdout=0.2)
    print(json.dumps(res))
    assert res["graph"]["recall_at_10"] > res["popularity"]["recall_at_10"] + 0.1
    assert res["graph"]["mpr"] < 0.5 and res["popularity"]["mpr"] < 0.5
    assert res["graph"]["mpr"] < res["popularity"]["mpr"]


def test_cli_prints_baselines(tmp_path, capsys, monkeypatch):
    from cubecobrarecommender_b200.non_ml import create_mtx
    k, c = 60, 96
    ip, ix = synth_cubes_csr(k, c, size_lo=5, size_hi=30, seed=5)
    names = {f"card {i}": [f"id{i}a", f"id{i}b"] for i in range(c)}
    os.makedirs(tmp_path / "data/maps"); os.makedirs(tmp_path / "data/cube")
    json.dump(names, open(tmp_path / "data/maps/nameToId.json", "w"))
    cubes = [{"_id": f"c{r}", "cards": [{"cardID": f"id{j}{'ab'[j % 2]}"} for j in ix[ip[r]:ip[r + 1]]]} for r in range(k)]
    json.dump(cubes, open(tmp_path / "data/cube/a.json", "w"))
    create_mtx.main(str(tmp_path))
    monkeypatch.chdir(tmp_path)
    monkeypatch.setenv("PYTHONHASHSEED", "0")       # (the CLI's seed argument sets it)
    T.main(["2", "16", "run", "0.1", "0.2", "3", "--validation-split", "0.25", "--rank-at", "10,50",
            "--rank-baselines", "graph,popularity"])
    lines = capsys.readouterr().out.splitlines()
    keys = ["recall_at_10", "ndcg_at_10", "hit_rate_at_10", "recall_at_50", "ndcg_at_50", "hit_rate_at_50", "mrr", "mpr"]
    first_epoch = lines.index("Epoch 1/2")
    for name in ("graph", "popularity"):
        found = [i for i, line in enumerate(lines) if line.startswith(f"baseline {name} - ")]
        assert len(found) == 1 and found[0] < first_epoch
        assert all(f" - {key}: " in lines[found[0]] for key in keys)
    epoch_lines = [line for line in lines if line.startswith("2/2 - ")]
    assert len(epoch_lines) == 2 and all(" - val_recall_at_10: " in line for line in epoch_lines)
    assert os.path.exists(tmp_path / "ml_files/run/cc_recommender.npz")


# ------------------------------------------------------------------ data parallel
def _multi_problem():
    gen = _generator(700, 400, 64, seed=48, size_lo=2, size_hi=150)
    return gen.split(0.4)


def _worker():
    import torch.distributed as dist
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl")
    train, val = _multi_problem()
    res = T.ranking_baselines(train, val, at=(1, 10, 50), holdout=0.2)
    if dist.get_rank() == 0:
        print(json.dumps({"world": dist.get_world_size(), "res": res}))
    dist.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_two_gpu_baselines_equal_one_gpu():
    train, val = _multi_problem()
    ref = T.ranking_baselines(train, val, at=(1, 10, 50), holdout=0.2)
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    env = dict(os.environ, PYTHONPATH=REPO + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)], cwd=REPO, env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip(), r.stderr[-3000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["world"] == 2
    for name, metrics in ref.items():
        for key, v in metrics.items():
            assert out["res"][name][key] == pytest.approx(v, rel=1e-12, abs=1e-15), (name, key)


if __name__ == "__main__":
    _worker()
