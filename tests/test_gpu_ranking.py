"""Leave-k-out ranking evaluation on the GPU: cc_rank_targets_f32 against NumPy's stable argsort and against the top-N
select, ``target_ranks_device`` and ``evaluate_recommendations`` against the NumPy oracle, their lack of side effects,
a trained model scoring above an untrained one, and the CLI flag."""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from cubecobrarecommender_b200 import _lib, graph as G
from cubecobrarecommender_b200.ml import engine as E, generator as GEN, model as M, ranking as R, train as T
from cubecobrarecommender_b200.ml.inference import MLRecommender
from cubecobrarecommender_b200.sparse import CubeCSR
from cubecobrarecommender_b200.synth import synth_cubes_csr
from oracle import dae as od
from ranking_oracle import ranking_metrics_np, target_ranks_np

call, ptr, stream_ptr = _lib.call, _lib.ptr, _lib.stream_ptr


def _csr_dev(lists):
    ip = np.zeros(len(lists) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in lists], out=ip[1:])
    ix = np.concatenate([np.asarray(x, dtype=np.int32) for x in lists]) if ip[-1] else np.zeros(1, np.int32)
    return torch.from_numpy(ip).cuda(), torch.from_numpy(ix.astype(np.int32)).cuda(), ip


def _expected(vals, mask, targets):
    """NumPy oracle: position of each target in argsort(kind='stable')[::-1] over the row's candidates."""
    c = len(vals)
    masked = np.zeros(c, dtype=bool)
    masked[[m for m in mask if 0 <= m < c]] = True
    order = np.argsort(vals, kind="stable")[::-1]
    order = order[~masked[order]]
    pos = np.full(c, -1, dtype=np.int64)
    pos[order] = np.arange(len(order))
    return np.array([pos[t] if 0 <= t < c else -1 for t in targets], dtype=np.int64)


def _rows_for(c, rng):
    """(mask, targets) per cube: empty mask; the row's ends plus masked, out-of-range and duplicate targets; a random
    cube; no targets; only masked targets; and (at C = 20 884) 10 000 targets, more than one shared-memory chunk."""
    rows = []
    t = rng.choice(c, size=max(1, c // 5), replace=False)
    rows.append(([], list(t)))
    ends = [0, c - 1]
    rows.append((ends, ends + [c // 2, c // 2, -1, c, c + 7] + list(rng.integers(0, c, size=5)) * 2))
    perm = rng.permutation(c)
    nm = max(1, c // 10)
    rows.append((list(perm[:nm]), list(perm[nm:nm + max(1, c // 5)])))
    rows.append((list(perm[:nm]), []))
    rows.append((list(perm[:nm]), list(perm[:nm])))
    if c >= 20000:
        rows.append((list(perm[:500]), list(perm[500:10500])))
    else:
        rows.append((list(perm[:nm]), list(perm[nm:])))                  # every candidate is a target
    return rows


def _scores(kind, b, c, rng):
    if kind == "normal":
        return (rng.standard_normal((b, c)) * 3).astype(np.float32)
    if kind == "ties":                                                     # a few distinct values: long tie runs
        return rng.integers(-2, 3, size=(b, c)).astype(np.float32)
    # saturated logits: +20 (float32 sigmoid exactly 1.0, ties), -100 (denormal / 0), a few ordinary values
    return rng.choice(np.array([20.0, 25.0, -100.0, -104.0, 0.5, -0.5], dtype=np.float32), size=(b, c))


def _layout(host, padded):
    """Device rows: ld padded to a multiple of 4 with a 16-byte aligned base, or ld % 4 != 0 on a misaligned base."""
    b, c = host.shape
    if padded:
        ld = (c + 3) // 4 * 4
        buf = torch.full((b, ld), float("nan"), device="cuda")
        buf[:, :c] = torch.from_numpy(host).cuda()
        return buf[:, :c]
    ld = c + 1 if (c + 1) % 4 else c + 2
    flat = torch.full((b * ld + 1,), float("nan"), device="cuda")
    view = flat[1:].view(b, ld)
    view[:, :c] = torch.from_numpy(host).cuda()
    return view[:, :c]


@pytest.mark.parametrize("c", [20884, 1000, 129, 3])
@pytest.mark.parametrize("padded", [True, False])
@pytest.mark.parametrize("kind", ["normal", "ties", "saturated"])
def test_rank_targets_equals_stable_argsort(c, padded, kind):
    rng = np.random.default_rng(c + 7 * padded + len(kind))
    rows = _rows_for(c, rng)
    logits = _layout(_scores(kind, len(rows), c, rng), padded)
    assert (logits.stride(0) % 4 != 0) == (not padded) and (logits.data_ptr() % 16 != 0) == (not padded)
    mp, mi, _ = _csr_dev([m for m, _ in rows])
    tp, ti, tip = _csr_dev([t for _, t in rows])
    # device probabilities, ranked by NumPy (its float32 exp is not CUDA's expf)
    probs = torch.empty_like(logits.contiguous())
    call("cc_sigmoid_f32", ptr(logits.contiguous()), ptr(probs), probs.numel(), stream_ptr())
    probs_l = _layout(probs.cpu().numpy(), padded)
    got_raw = G.rank_targets(logits, mp, mi, tp, ti).cpu().numpy()
    got_sig = G.rank_targets(logits, mp, mi, tp, ti, sigmoid=True).cpu().numpy()
    got_prob = G.rank_targets(probs_l, mp, mi, tp, ti).cpu().numpy()
    assert np.array_equal(got_sig, got_prob)
    lh, ph = logits.cpu().numpy(), probs.cpu().numpy()
    for b, (mask, targets) in enumerate(rows):
        sl = slice(tip[b], tip[b + 1])
        assert np.array_equal(got_raw[sl], _expected(lh[b], mask, targets)), (b, "raw")
        assert np.array_equal(got_sig[sl], _expected(ph[b], mask, targets)), (b, "sigmoid")


def test_rank_targets_batch_zero_is_a_no_op():
    z = torch.zeros(1, 10, device="cuda")
    p = torch.zeros(2, dtype=torch.int64, device="cuda")
    i = torch.zeros(1, dtype=torch.int32, device="cuda")
    out = torch.full((1,), 123, dtype=torch.int32, device="cuda")
    call("cc_rank_targets_f32", ptr(z), 10, 10, 0, ptr(p), ptr(i), ptr(p), ptr(i), 1, ptr(out), stream_ptr())
    assert int(out.item()) == 123


def test_rank_targets_agrees_with_the_select():
    """4096 x 20 884 logits: every target of rank r < 50 is what topn_masked(sigmoid=True, n=50) returns at slot r, and
    every returned target sits at the slot of its rank."""
    b, c, n = 4096, 20884, 50
    ip, ix = synth_cubes_csr(b, c, seed=21)
    csr = CubeCSR(ip, ix, c)
    vis, hid, _ = R.holdout_split(csr, 0.2, seed=3)
    g = torch.Generator(device="cuda").manual_seed(5)
    z = torch.randn(b, (c + 3) // 4 * 4, device="cuda", generator=g)[:, :c] * 2
    z[:, :300] += 3                                                        # popular cards, as a trained model ranks them
    mp, mi = (torch.from_numpy(a).cuda() for a in (vis.indptr, vis.indices))
    tp, ti = (torch.from_numpy(a).cuda() for a in (hid.indptr, hid.indices))
    ranks = G.rank_targets(z, mp, mi, tp, ti, sigmoid=True).cpu().numpy()
    ids = G.topn_masked(z, mp, mi, n, sigmoid=True)[0].cpu().numpy()
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


def _params(c, seed=0):
    params = od.init_params(c, seed=seed)
    rng = np.random.default_rng(seed + 1)
    for kname in params:          # non-zero biases, livelier logits
        if kname.endswith("bias"):
            params[kname] = (rng.standard_normal(params[kname].shape) * 0.1).astype(np.float32)
    return params


def _oracle_ranks(model, vis, hid):
    probs = MLRecommender(model).probabilities(vis).cpu().numpy()
    out, per_cube = [], []
    for b in range(vis.num_cubes):
        in_cube = np.zeros(vis.num_cards)
        in_cube[vis.indices[vis.indptr[b]:vis.indptr[b + 1]]] = 1
        r = target_ranks_np(probs[b], in_cube, hid.indices[hid.indptr[b]:hid.indptr[b + 1]])
        out.append(r); per_cube.append(r)
    return np.concatenate(out), per_cube


@pytest.mark.parametrize("c,k,size_lo,size_hi", [(1000, 700, 2, 80), (20884, 400, 360, 720)])
def test_target_ranks_device_equals_the_oracle(c, k, size_lo, size_hi):
    """Chunk 8192 (one chunk) against the oracle on ``probabilities`` of the whole set; chunk 300 against the oracle on
    ``probabilities`` of each 300-cube slice -- the same GEMM shapes, so the same logits bit for bit (a forward of
    another batch size may round differently, see test_gpu_zz_late_additions.py)."""
    ip, ix = synth_cubes_csr(k, c, size_lo=size_lo, size_hi=size_hi, seed=c)
    vis, hid, _ = R.holdout_split(CubeCSR(ip, ix, c), 0.2, seed=1)
    model = M.CC_Recommender(c, device="cuda", precision="tf32")
    model.set_weights_dict(_params(c, seed=2))
    ref, _ = _oracle_ranks(model, vis, hid)
    got = MLRecommender(model, chunk=8192).target_ranks_device(vis, hid).cpu().numpy()
    assert np.array_equal(got, ref)
    got300 = MLRecommender(model, chunk=300).target_ranks_device(vis, hid).cpu().numpy()
    sel = [np.arange(lo, min(lo + 300, k)) for lo in range(0, k, 300)]
    ref300 = np.concatenate([_oracle_ranks(model, vis.rows(s_), hid.rows(s_))[0] for s_ in sel])
    assert np.array_equal(got300, ref300)
    # ranks that differ between the two chunkings come from logits a rounding apart
    assert (got300 != got).mean() < 1e-3


def _generator(c, k, batch, seed=5, size_lo=10, size_hi=60):
    ip, ix = synth_cubes_csr(k, c, size_lo=size_lo, size_hi=size_hi, seed=seed)
    csr = CubeCSR(ip, ix, c)
    gr = G.build_graph(csr, "cuda", want_m64=False)
    return GEN.DataGenerator(gr.mhat, csr, batch_size=batch, noise=0.2, seed=seed), csr


def test_evaluate_recommendations_equals_the_oracle_and_shards_add_up():
    c, k = 1000, 500
    gen, _ = _generator(c, k, 64, seed=6, size_lo=1, size_hi=80)
    model = M.CC_Recommender(c, device="cuda", precision="tf32")
    model.set_weights_dict(_params(c, seed=3))
    at = (1, 10, 50)
    res = T.evaluate_recommendations(model, gen, at=at, holdout=0.25)
    vis, hid, ev = gen.holdout_split(0.25)
    _, per_cube = _oracle_ranks(model, vis, hid)
    ref = ranking_metrics_np(per_cube, c - np.diff(vis.indptr), at)
    assert res["cubes"] == ref["cubes"] == int(ev.sum()) and res["skipped"] == k - int(ev.sum()) > 0
    for key in R.metric_names(at):
        assert res[key] == pytest.approx(ref[key], rel=1e-12, abs=1e-15), key
    # two ranks' shards (shard_range at world 2, one GPU): their sums add up to the whole set's (chunks of 250 cubes
    # give the whole set the forward shapes of the shards)
    rec = MLRecommender(model, chunk=250)

    def sums(v, h):
        hp = torch.from_numpy(h.indptr).cuda()
        nc = torch.from_numpy(c - np.diff(v.indptr)).cuda()
        return R.ranking_sums(rec.target_ranks_device(v, h), hp, nc, at).cpu().numpy()
    whole = sums(vis, hid)
    parts = sum(sums(vis.shard(r, 2), hid.shard(r, 2)) for r in range(2))
    assert np.allclose(parts, whole, rtol=1e-12, atol=0)
    assert whole[0] == res["cubes"]
    for key, v in zip(R.metric_names(at), whole[1:] / whole[0]):
        assert abs(v - res[key]) <= 1e-3, key


def test_evaluate_recommendations_has_no_side_effects():
    c, batch = 384, 32
    gen, _ = _generator(c, 150, batch, seed=9)
    train, val = gen.split(0.3)
    model = M.CC_Recommender(c, device="cuda", seed=1, precision="tf32")
    eng = E.DAEEngine(model, gen.mhat_device(), batch=batch, reg_rows=batch, reg=0.1,
                      max_cube_size=max(train.csr.max_size, val.csr.max_size))
    for b_ in range(2):                                          # live gradients, Adam slots, counters
        eng.sample_batch(train.indptr, train.indices_dev, train.batch_ids(b_), train.alias_prob, train.alias_idx, seed=3)
        eng.train_step()
    s = model.store
    snap = lambda: [t.clone() for t in (s.params, s.grads, s.adam_m, s.adam_v, s.step, eng.noise_step, train._step)
                    + ((s.shadow,) if s.shadow is not None else ())]
    before = snap()
    order = train.indices.copy()
    r1 = T.evaluate_recommendations(model, val, at=(10, 50))
    r2 = T.evaluate_recommendations(model, val, at=(10, 50))
    torch.cuda.synchronize()
    for a, b_ in zip(before, snap()):
        assert torch.equal(a, b_)
    assert np.array_equal(order, train.indices)
    assert r1.keys() == r2.keys() and all(r1[key] == pytest.approx(r2[key], rel=1e-12) for key in r1)


def test_fit_with_ranking_adds_the_keys_and_changes_nothing_else():
    """Same fit with and without ranking_at: the same training and val_* loss history (exact-fp32 mode; only the
    float atomics of the train step separate two runs, as in test_gpu_validation.py), plus the ranking keys."""
    c, k, b = 256, 128, 32
    quiet = lambda *_: None
    hist = {}
    for at in (None, (10, 50)):
        gen, _ = _generator(c, k, b, seed=8)
        model = M.CC_Recommender(c, device="cuda", seed=0, precision="fp32")
        lines = []
        hist[at] = T.fit(model, gen, epochs=3, reg=0.1, log=lines.append if at else quiet, validation_split=0.2,
                         max_cube_size=64, ranking_at=at)
    new = ["val_recall_at_10", "val_ndcg_at_10", "val_hit_rate_at_10", "val_recall_at_50", "val_ndcg_at_50",
           "val_hit_rate_at_50", "val_mrr", "val_mpr"]
    for h0, h1 in zip(hist[None], hist[(10, 50)]):
        assert set(h1) == set(h0) | set(new) and not set(new) & set(h0)
        for key, v in h0.items():
            assert abs(h1[key] - v) <= 1e-5 * abs(v), key
        assert 0.0 <= h1["val_recall_at_50"] <= 1.0 and 0.0 < h1["val_mpr"] < 1.0
    assert all(" - val_recall_at_10: " in line and " - val_mpr: " in line for line in lines if line.startswith("3/3"))


def test_ranking_measures_learning():
    """Zipf cubes at C = 1000: after training, recall@50 on held-out cubes beats the untrained model's and the
    uniform expectation 50 / n by a wide margin (the model learns at least the popularity of the cards)."""
    c, k, b = 1000, 4096, 128
    gen, _ = _generator(c, k, b, seed=31, size_lo=40, size_hi=120)
    train, val = gen.split(0.25)
    model = M.CC_Recommender(c, device="cuda", seed=0, precision="tf32")
    before = T.evaluate_recommendations(model, val, at=(50,))
    T.fit(model, train, epochs=8, reg=0.1, log=lambda *_: None)
    after = T.evaluate_recommendations(model, val, at=(50,))
    vis, _, _ = val.holdout_split(0.2)
    uniform = float(np.mean(50.0 / (c - np.diff(vis.indptr))))
    print(json.dumps({"untrained": before, "trained": after, "uniform_recall_at_50": uniform}))
    assert after["recall_at_50"] > 2 * uniform and after["recall_at_50"] > before["recall_at_50"] + 0.1
    assert after["mpr"] < before["mpr"]


def test_cli_prints_ranking_metrics(tmp_path, capsys, monkeypatch):
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
    T.main(["2", "16", "run", "0.1", "0.2", "3", "--validation-split", "0.25", "--rank-at", "10,50"])
    out = capsys.readouterr().out
    epoch_lines = [line for line in out.splitlines() if line.startswith("2/2 - ")]
    keys = ["val_loss", "val_recall_at_10", "val_ndcg_at_10", "val_hit_rate_at_10", "val_recall_at_50",
            "val_ndcg_at_50", "val_hit_rate_at_50", "val_mrr", "val_mpr"]
    assert len(epoch_lines) == 2 and all(f" - {key}: " in line for line in epoch_lines for key in keys)
