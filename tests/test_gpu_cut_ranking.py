"""Cut-list evaluation on the GPU: cc_rank_cuts_f32 / _f64 against NumPy's stable argsort over the listed cards and
against the ascending only-listed select, the cut ranks of the autoencoder, the graph (``oracle.graph.simple_cuts``)
and popularity against NumPy, ``evaluate_cuts`` / ``ranking_baselines(task="cuts")`` against the metric oracle, their
lack of side effects, what they measure on cubes from disjoint card pools, the CLI flag and a two-GPU run."""
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
from cubecobrarecommender_b200.ml import engine as E, model as M, ranking as R, train as T
from cubecobrarecommender_b200.ml.inference import MLRecommender
from cubecobrarecommender_b200.sparse import CubeCSR
from cubecobrarecommender_b200.synth import synth_cubes_csr
from oracle import graph as og
from ranking_oracle import ranking_metrics_np
from test_gpu_ranking import _csr_dev, _layout, _params, _scores
from test_gpu_ranking_baselines import _generator, _layout64, _m_oracle, _pool_cubes, _scores64

call, ptr, stream_ptr = _lib.call, _lib.ptr, _lib.stream_ptr
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _expected_cuts(vals, lst, targets):
    """NumPy oracle: position of each target in argsort(kind='stable') over the distinct listed cards (ascending score,
    ties to the smaller index), -1 for a target that is not listed or out of range."""
    c = len(vals)
    cand = np.unique(np.asarray([x for x in lst if 0 <= x < c], dtype=np.int64))
    order = cand[np.argsort(vals[cand], kind="stable")]
    pos = np.full(c, -1, dtype=np.int64)
    pos[order] = np.arange(len(order))
    return np.array([pos[t] if 0 <= t < c else -1 for t in targets], dtype=np.int64)


def _cut_rows(c, rng):
    """(list, targets) per cube: an empty list; the row's ends with duplicate and out-of-range list entries and
    unlisted, out-of-range and duplicate targets; a random cube with some of its cards and some others as targets; no
    targets; every listed card a target; and (C >= 20 000) 6000 listed cards with 1500 targets."""
    rows = []
    perm = rng.permutation(c)
    nl = max(1, c // 10)
    rows.append(([], list(perm[:max(1, c // 5)])))
    ends = [0, c - 1]
    rows.append((ends + [c // 2, c // 2, 0, -1, c, c + 7], ends + [c // 2, c // 2, -1, c, c + 7, 1 % c] + ends))
    lst = list(perm[:nl])
    rows.append((lst, list(rng.choice(lst, size=max(1, nl // 3), replace=False)) + list(perm[nl:nl + 3])))
    rows.append((lst, []))
    rows.append((lst, list(perm[:nl])[::-1]))
    if c >= 20000:
        big = list(perm[:6000])
        rows.append((big, list(rng.choice(big, size=1500, replace=False)) + list(perm[6000:6010])))
    return rows


def _same(a, b):
    """Two metric dicts equal up to summation order (ranking_sums adds with float atomics, in no fixed order)."""
    return a.keys() == b.keys() and all(a[k] == pytest.approx(b[k], rel=1e-12, abs=1e-15) for k in a)


def _check(got, tip, host, rows):
    for b, (lst, targets) in enumerate(rows):
        assert np.array_equal(got[tip[b]:tip[b + 1]], _expected_cuts(host[b], lst, targets)), b


@pytest.mark.parametrize("c", [100000, 20884, 1000, 129, 3])
@pytest.mark.parametrize("padded", [True, False])
@pytest.mark.parametrize("kind", ["normal", "ties", "saturated"])
def test_rank_cuts_f32_equals_stable_argsort(c, padded, kind):
    rng = np.random.default_rng(c + 5 * padded + len(kind))
    rows = _cut_rows(c, rng)
    logits = _layout(_scores(kind, len(rows), c, rng), padded)
    lp, li, _ = _csr_dev([x for x, _ in rows])
    tp, ti, tip = _csr_dev([t for _, t in rows])
    probs = torch.empty_like(logits.contiguous())
    call("cc_sigmoid_f32", ptr(logits.contiguous()), ptr(probs), probs.numel(), stream_ptr())
    got_raw = G.rank_cuts(logits, lp, li, tp, ti).cpu().numpy()
    got_sig = G.rank_cuts(logits, lp, li, tp, ti, sigmoid=True).cpu().numpy()
    got_prob = G.rank_cuts(_layout(probs.cpu().numpy(), padded), lp, li, tp, ti).cpu().numpy()
    assert np.array_equal(got_sig, got_prob)
    _check(got_raw, tip, logits.cpu().numpy(), rows)
    _check(got_sig, tip, probs.cpu().numpy(), rows)
    assert (got_raw == -1).sum() > 0 and (got_raw >= 0).sum() > 0


@pytest.mark.parametrize("c", [100000, 20884, 1000, 129, 3])
@pytest.mark.parametrize("layout", ["vector", "scalar", "shared"])
@pytest.mark.parametrize("kind", ["normal", "ties", "special"])
def test_rank_cuts_f64_equals_stable_argsort(c, layout, kind):
    rng = np.random.default_rng(c + 13 * len(layout) + len(kind))
    rows = _cut_rows(c, rng)
    host = _scores64(kind, len(rows), c, rng)
    if layout == "shared":
        host[:] = host[0]
    sc = _layout64(host, layout)
    assert (sc.stride(0) == 0) == (layout == "shared")
    lp, li, _ = _csr_dev([x for x, _ in rows])
    tp, ti, tip = _csr_dev([t for _, t in rows])
    _check(G.rank_cuts(sc, lp, li, tp, ti).cpu().numpy(), tip, host, rows)


@pytest.mark.parametrize("name", ["cc_rank_cuts_f32", "cc_rank_cuts_f64"])
def test_rank_cuts_batch_zero_is_a_no_op(name):
    is32 = name.endswith("f32")
    z = torch.zeros(1, 10, dtype=torch.float32 if is32 else torch.float64, device="cuda")
    p = torch.zeros(2, dtype=torch.int64, device="cuda")
    i = torch.zeros(1, dtype=torch.int32, device="cuda")
    out = torch.full((1,), 123, dtype=torch.int32, device="cuda")
    call(name, ptr(z), 10, 10, 0, ptr(p), ptr(i), ptr(p), ptr(i), *([1] if is32 else []), ptr(out), stream_ptr())
    torch.cuda.synchronize()
    assert int(out.item()) == 123


@pytest.mark.parametrize("mode", ["sigmoid", "f32", "f64"])
def test_rank_cuts_agrees_with_the_ascending_select(mode):
    """4096 corrupted cubes of 20 884 cards with tied scores: every intruder of rank r < 50 is what
    topn_masked(only_listed=True, descending=False, n=50) returns at slot r, and every returned intruder sits at the
    slot of its rank."""
    b, c, n = 4096, 20884, 50
    ip, ix = synth_cubes_csr(b, c, seed=23)
    cor, intr, _ = R.intruder_split(CubeCSR(ip, ix, c), 0.2, seed=9)
    g = torch.Generator(device="cuda").manual_seed(7)
    z = torch.randn(b, (c + 3) // 4 * 4, device="cuda", generator=g)[:, :c]
    if mode == "f64":
        z = (torch.round(z.double() * 8) / 4).contiguous()
    elif mode == "f32":
        z = torch.round(z * 8) / 4
    else:
        z = z * 6                                         # saturated probabilities tie
    cp, ci = (torch.from_numpy(a).cuda() for a in (cor.indptr, cor.indices))
    tp, ti = (torch.from_numpy(a).cuda() for a in (intr.indptr, intr.indices))
    sig = mode == "sigmoid"
    ranks = G.rank_cuts(z, cp, ci, tp, ti, sigmoid=sig).cpu().numpy()
    ids = G.topn_masked(z, cp, ci, n, only_listed=True, descending=False, sigmoid=sig)[0].cpu().numpy()
    assert (ranks >= 0).all()
    cube = np.repeat(np.arange(b), np.diff(intr.indptr))
    top = ranks < n
    assert top.sum() > 1000
    assert np.array_equal(ids[cube[top], ranks[top]], intr.indices[top])
    rank_of = {(int(q), int(t)): int(r) for q, t, r in zip(cube, intr.indices, ranks)}
    seen = 0
    for q in range(b):
        for slot, card in enumerate(ids[q]):
            if (q, int(card)) in rank_of:
                assert rank_of[q, int(card)] == slot
                seen += 1
    assert seen == int(top.sum())


# ------------------------------------------------------------------ the three recommenders
def _ml_oracle(model, cor, intr):
    """Per cube: NumPy cut ranks of probabilities from a forward pass over the same cubes (same batch shape)."""
    probs = MLRecommender(model).probabilities(cor).cpu().numpy()
    return [_expected_cuts(probs[b], cor.indices[cor.indptr[b]:cor.indptr[b + 1]],
                           intr.indices[intr.indptr[b]:intr.indptr[b + 1]]) for b in range(cor.num_cubes)]


@pytest.mark.parametrize("c,k,size_lo,size_hi", [(1000, 700, 1, 80), (20884, 400, 360, 720)])
def test_ml_cut_ranks_equal_numpy(c, k, size_lo, size_hi):
    ip, ix = synth_cubes_csr(k, c, size_lo=size_lo, size_hi=size_hi, seed=c + 1)
    cor, intr, ev = R.intruder_split(CubeCSR(ip, ix, c), 0.2, seed=1)
    model = M.CC_Recommender(c, device="cuda", precision="tf32")
    model.set_weights_dict(_params(c, seed=4))
    ref = np.concatenate(_ml_oracle(model, cor, intr))
    assert (ref >= 0).all() and ev.sum() > 0.9 * k
    got = MLRecommender(model).cut_ranks_device(cor, intr).cpu().numpy()
    assert np.array_equal(got, ref)
    got300 = MLRecommender(model, chunk=300).cut_ranks_device(cor, intr).cpu().numpy()
    sel = [np.arange(lo, min(lo + 300, k)) for lo in range(0, k, 300)]
    ref300 = np.concatenate([np.concatenate(_ml_oracle(model, cor.rows(s_), intr.rows(s_))) for s_ in sel])
    assert np.array_equal(got300, ref300)


def _graph_cut_oracle(m_host, cor, intr):
    out = []
    for b in range(cor.num_cubes):
        cube = np.zeros(cor.num_cards)
        cube[cor.indices[cor.indptr[b]:cor.indptr[b + 1]]] = 1
        h = intr.indices[intr.indptr[b]:intr.indptr[b + 1]]
        pos = {card: i for i, card in enumerate(og.simple_cuts(cube, m_host.copy(), stable=True))} if len(h) else {}
        out.append(np.array([pos.get(int(t), -1) for t in h], dtype=np.int64))
    return out


def _popularity_cut_oracle(train_csr, cor, intr):
    counts = np.bincount(train_csr.indices, minlength=train_csr.num_cards).astype(np.float64)
    return [_expected_cuts(counts, cor.indices[cor.indptr[b]:cor.indptr[b + 1]],
                           intr.indices[intr.indptr[b]:intr.indptr[b + 1]]) for b in range(cor.num_cubes)]


def test_graph_cut_ranks_equal_simple_cuts():
    """Cubes of 5-300 cards scored against M of 2000 other cubes, in chunks of a few cubes, one cube per chunk and one
    chunk: every intruder sits where simple_cuts lists it, and where GraphRecommender.cuts returns it."""
    c = 1000
    ip, ix = synth_cubes_csr(2000, c, size_lo=10, size_hi=200, seed=51)
    train = CubeCSR(ip, ix, c)
    ip, ix = synth_cubes_csr(300, c, size_lo=5, size_hi=300, seed=52)
    cor, intr, ev = R.intruder_split(CubeCSR(ip, ix, c), 0.2, seed=7)
    m = G.build_graph(train, "cuda", want_mhat=False, want_neg=False).m64
    m_host = m.cpu().numpy()
    ref = np.concatenate(_graph_cut_oracle(m_host, cor, intr))
    assert (ref >= 0).all() and ev.sum() == 300
    small = G.GraphRecommender(m, budget_bytes=6 * 3 * c * 8)
    assert np.array_equal(small.cut_ranks_device(cor, intr).cpu().numpy(), ref)
    assert np.array_equal(G.GraphRecommender(m).cut_ranks_device(cor, intr).cpu().numpy(), ref)
    sel = np.arange(20)
    one = G.GraphRecommender(m, budget_bytes=1).cut_ranks_device(cor.rows(sel), intr.rows(sel)).cpu().numpy()
    assert np.array_equal(one, ref[:int(intr.indptr[20])])
    ids = small.cuts(cor.rows(sel), 50)[0].cpu().numpy()
    for b in range(20):
        for t, r in zip(intr.indices[intr.indptr[b]:intr.indptr[b + 1]], ref[intr.indptr[b]:intr.indptr[b + 1]]):
            if r < 50:
                assert ids[b, r] == t


def test_popularity_cut_ranks_equal_numpy():
    c = 20884
    ip, ix = synth_cubes_csr(3000, c, seed=53)
    train = CubeCSR(ip, ix, c)
    ip, ix = synth_cubes_csr(500, c, size_lo=1, size_hi=400, seed=54)
    cor, intr, _ = R.intruder_split(CubeCSR(ip, ix, c), 0.25, seed=8)
    got = G.PopularityRecommender(train, "cuda").cut_ranks_device(cor, intr).cpu().numpy()
    assert np.array_equal(got, np.concatenate(_popularity_cut_oracle(train, cor, intr)))


# ------------------------------------------------------------------ metrics
def _with_empty_cubes(c, k, seed, size_lo=2, size_hi=80):
    ip, ix = synth_cubes_csr(k, c, size_lo=size_lo, size_hi=size_hi, seed=seed)
    rows = [ix[ip[b]:ip[b + 1]].tolist() for b in range(k)]
    rows[10] = rows[450] = []                     # no cards: skipped (one of them in a 0.4 validation split)
    return _generator(c, 0, 64, seed=seed, csr=CubeCSR.from_lists(rows, c))


def test_evaluate_cuts_equals_the_oracle_and_shards_add_up():
    c, at = 1000, (1, 10, 50)
    gen = _with_empty_cubes(c, 500, seed=61)
    model = M.CC_Recommender(c, device="cuda", precision="tf32")
    model.set_weights_dict(_params(c, seed=5))
    res = T.evaluate_cuts(model, gen, at=at, inject=0.25)
    cor, intr, ev = gen.intruder_split(0.25)
    ref = ranking_metrics_np(_ml_oracle(model, cor, intr), np.diff(cor.indptr), at)
    assert res["cubes"] == ref["cubes"] == int(ev.sum()) and res["skipped"] == 500 - int(ev.sum()) >= 2
    for key in R.metric_names(at):
        assert res[key] == pytest.approx(ref[key], rel=1e-12, abs=1e-15), key
    assert 0.0 < res["mpr"] < 1.0
    rec = MLRecommender(model, chunk=250)

    def sums(v, h):
        hp = torch.from_numpy(h.indptr).cuda()
        nc = torch.from_numpy(np.diff(v.indptr)).cuda()
        return R.ranking_sums(rec.cut_ranks_device(v, h), hp, nc, at).cpu().numpy()
    whole = sums(cor, intr)
    parts = sum(sums(cor.shard(r, 2), intr.shard(r, 2)) for r in range(2))
    assert np.allclose(parts, whole, rtol=1e-12, atol=0) and whole[0] == res["cubes"]
    # any object with cut_ranks_device
    assert _same(T.evaluate_cuts(MLRecommender(model), gen, at=at, inject=0.25), res)


def test_cut_baselines_equal_the_oracle():
    c, at, inject = 1000, (1, 10, 50), 0.25
    gen = _with_empty_cubes(c, 500, seed=62, size_hi=160)
    train, val = gen.split(0.4)
    res = T.ranking_baselines(train, val, at=at, task="cuts", inject=inject)
    assert list(res) == ["graph", "popularity"]
    cor, intr, ev = val.intruder_split(inject)
    n = np.diff(cor.indptr)
    ref = {"graph": ranking_metrics_np(_graph_cut_oracle(_m_oracle(train.csr), cor, intr), n, at),
           "popularity": ranking_metrics_np(_popularity_cut_oracle(train.csr, cor, intr), n, at)}
    for name in res:
        assert res[name]["cubes"] == ref[name]["cubes"] == int(ev.sum())
        assert res[name]["skipped"] == val.N_cubes - int(ev.sum()) >= 1
        for key in R.metric_names(at):
            assert res[name][key] == pytest.approx(ref[name][key], rel=1e-12, abs=1e-15), (name, key)
    direct = T.evaluate_cuts(G.PopularityRecommender(train.csr, "cuda"), val, at=at, inject=inject)
    assert _same(direct, res["popularity"])
    # the adds task is still the default
    assert _same(T.ranking_baselines(train, val, names=("popularity",), at=at)["popularity"],
                 T.evaluate_recommendations(G.PopularityRecommender(train.csr, "cuda"), val, at=at))


def test_evaluate_cuts_has_no_side_effects():
    c, batch = 384, 32
    gen = _generator(c, 150, batch, seed=63, size_lo=10, size_hi=60)
    train, val = gen.split(0.3)
    model = M.CC_Recommender(c, device="cuda", seed=1, precision="tf32")
    eng = E.DAEEngine(model, gen.mhat_device(), batch=batch, reg_rows=batch, reg=0.1,
                      max_cube_size=max(train.csr.max_size, val.csr.max_size))
    for b_ in range(2):                                          # live gradients, Adam slots, counters
        eng.sample_batch(train.indptr, train.indices_dev, train.batch_ids(b_), train.alias_prob, train.alias_idx, seed=3)
        eng.train_step()
    s = model.store
    snap = lambda: [t.clone() for t in (s.params, s.grads, s.adam_m, s.adam_v, s.step, eng.noise_step, train._step,
                                        val._step) + ((s.shadow,) if s.shadow is not None else ())]
    before = snap()
    order = train.indices.copy()
    split = val.intruder_split(0.2)
    r1 = T.evaluate_cuts(model, val, at=(10, 50))
    b1 = T.ranking_baselines(train, val, at=(10, 50), task="cuts")
    r2 = T.evaluate_cuts(model, val, at=(10, 50))
    b2 = T.ranking_baselines(train, val, at=(10, 50), task="cuts")
    torch.cuda.synchronize()
    for a, b_ in zip(before, snap()):
        assert torch.equal(a, b_)
    assert np.array_equal(order, train.indices)
    assert val.intruder_split(0.2) is split
    assert _same(r1, r2) and all(_same(b1[n], b2[n]) for n in b1)


def test_fit_with_cut_ranking_adds_the_keys_and_changes_nothing_else():
    """Same fit with and without ranking_cuts: the same training, val_* loss and ranking history (exact-fp32 mode; only
    the float atomics of the train step separate two runs), plus the cut keys."""
    c, k, b = 256, 128, 32
    hist, lines = {}, []
    for cuts in (False, True):
        gen = _generator(c, k, b, seed=8, size_lo=10, size_hi=60)
        model = M.CC_Recommender(c, device="cuda", seed=0, precision="fp32")
        hist[cuts] = T.fit(model, gen, epochs=3, reg=0.1, log=lines.append if cuts else (lambda *_: None),
                           validation_split=0.2, max_cube_size=64, ranking_at=(10, 50), ranking_cuts=cuts)
    new = ["val_cut_recall_at_10", "val_cut_ndcg_at_10", "val_cut_hit_rate_at_10", "val_cut_recall_at_50",
           "val_cut_ndcg_at_50", "val_cut_hit_rate_at_50", "val_cut_mrr", "val_cut_mpr"]
    for h0, h1 in zip(hist[False], hist[True]):
        assert set(h1) == set(h0) | set(new) and not set(new) & set(h0)
        for key, v in h0.items():
            assert abs(h1[key] - v) <= 1e-5 * abs(v), key
        assert 0.0 <= h1["val_cut_recall_at_50"] <= 1.0 and 0.0 < h1["val_cut_mpr"] < 1.0
    assert all(" - val_cut_recall_at_10: " in line and " - val_cut_mpr: " in line for line in lines
               if line.startswith("3/3"))


def test_cuts_measure_co_occurrence_and_learning():
    """Cubes from four disjoint card pools: most intruders come from another pool, so the graph, which never saw them
    beside the cube's cards, cuts them first and beats popularity; and a trained model cuts them better than an
    untrained one.  (With a single popularity law the graph ranks like popularity: there is no pool to tell apart.)"""
    rng = np.random.default_rng(64)
    csr = _pool_cubes(3200, 4, 150, rng)
    gen = _generator(csr.num_cards, 0, 128, seed=64, csr=csr)
    train, val = gen.split(0.25)
    base = T.ranking_baselines(train, val, at=(10,), task="cuts")
    model = M.CC_Recommender(csr.num_cards, device="cuda", seed=0, precision="tf32")
    before = T.evaluate_cuts(model, val, at=(10,))
    T.fit(model, train, epochs=8, reg=0.1, log=lambda *_: None)
    after = T.evaluate_cuts(model, val, at=(10,))
    print(json.dumps({"baselines": base, "untrained": before, "trained": after}))
    assert base["graph"]["recall_at_10"] > base["popularity"]["recall_at_10"] + 0.1
    assert base["graph"]["mpr"] < base["popularity"]["mpr"]
    assert after["recall_at_10"] > before["recall_at_10"] + 0.1 and after["mpr"] < before["mpr"]


def test_cli_prints_cut_metrics_and_baselines(tmp_path, capsys, monkeypatch):
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
    T.main(["2", "16", "run", "0.1", "0.2", "3", "--validation-split", "0.25", "--rank-at", "10,50", "--rank-cuts",
            "--rank-baselines", "graph,popularity"])
    lines = capsys.readouterr().out.splitlines()
    keys = ["recall_at_10", "ndcg_at_10", "hit_rate_at_10", "recall_at_50", "ndcg_at_50", "hit_rate_at_50", "mrr", "mpr"]
    first_epoch = lines.index("Epoch 1/2")
    for name in ("graph", "popularity"):
        for prefix in (f"baseline {name} - ", f"baseline {name} cuts - "):
            found = [i for i, line in enumerate(lines) if line.startswith(prefix)]
            assert len(found) == 1 and found[0] < first_epoch, prefix
            assert all(f" - {key}: " in lines[found[0]] for key in keys)
    epoch_lines = [line for line in lines if line.startswith("2/2 - ")]
    assert len(epoch_lines) == 2
    assert all(f" - val_{key}: " in line and f" - val_cut_{key}: " in line for line in epoch_lines for key in keys)


# ------------------------------------------------------------------ data parallel
def _multi_problem():
    gen = _generator(700, 400, 64, seed=65, size_lo=2, size_hi=150)
    train, val = gen.split(0.4)
    model = M.CC_Recommender(700, device="cuda", precision="tf32")
    model.set_weights_dict(_params(700, seed=6))
    return train, val, model


def _multi_run(train, val, model, chunk):
    at = (1, 10, 50)
    out = T.ranking_baselines(train, val, at=at, task="cuts")
    out["model"] = T.evaluate_cuts(MLRecommender(model, chunk=chunk), val, at=at)
    return out


def _worker():
    import torch.distributed as dist
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl")
    train, val, model = _multi_problem()
    res = _multi_run(train, val, model, chunk=8192)
    if dist.get_rank() == 0:
        print(json.dumps({"world": dist.get_world_size(), "res": res}))
    dist.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_two_gpu_cuts_equal_one_gpu():
    train, val, model = _multi_problem()
    assert val.N_cubes % 2 == 0
    ref = _multi_run(train, val, model, chunk=val.N_cubes // 2)        # the shards' forward shapes
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
