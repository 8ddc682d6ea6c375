"""Similar cards and cubes on the GPU: cc_cosine_neg_many_f32 bit for bit against cc_cosine_neg_f32 and against the
float64 restatement of Keras' CosineSimilarity loss; the similar-cards table, ``similar`` and the query blocks of
``nearest`` bit for bit against the one-card route (cc_cosine_neg_f32 + a batch-1 select); ``cube_embeddings`` against
the oracle encoder; ``similar_cubes`` against NumPy's stable argsort of the kernel's own distances, with the corpus as
a CSR or as embeddings, past the row select's 26 000-candidate limit and for a tf32 model; no side effects; the
``--table`` command line."""
import json

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from cubecobrarecommender_b200 import _lib, graph as G
from cubecobrarecommender_b200.ml import model as M
from cubecobrarecommender_b200.ml.inference import MLRecommender
from cubecobrarecommender_b200.sparse import CubeCSR
from cubecobrarecommender_b200.synth import synth_cubes_csr
from oracle import dae as od

call, ptr, stream_ptr = _lib.call, _lib.ptr, _lib.stream_ptr
NAN_BITS = 0x7FC01234                     # sentinel in the output's padding columns


def _emb(n, seed, ld=64):
    """(n, 64) float32 rows in an (n, ld) buffer: ReLU-like rows (many exact zeros) with magnitudes over several decades;
    among the first 16 rows (which kinds land where depends on the seed) an all-zero row, a row below the 1e-12 clamp, a
    row near 1e16, rows with disjoint supports (an exact +0 dot product), a signed row and an exact duplicate; past 16
    rows, every 97th row repeats row 10 (exact ties)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.relu(torch.randn(n, 64, device="cuda", generator=g) - 0.3)
    x *= torch.exp(2 * torch.randn(n, 1, device="cuda", generator=g))
    for r in range(min(n, 16)):
        k = (r + seed) % 16
        if k == 0:
            x[r] = 0
        elif k == 1:
            x[r] *= 1e-7 / max(float(x[r].abs().max()), 1e-30)
        elif k == 2:
            x[r] *= 1e16 / max(float(x[r].abs().max()), 1e-30)
        elif k == 3:
            x[r, 32:] = 0
        elif k == 4:
            x[r, :32] = 0
        elif k == 5:
            x[r] = torch.randn(64, device="cuda", generator=g)
        elif k == 6 and r > 0:
            x[r] = x[r - 1]
    if n > 16:
        x[50::97] = x[10]
    buf = torch.full((n, ld), float("nan"), device="cuda")
    buf[:, :64] = x
    return buf[:, :64]


def _bits_equal(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _many(q, c, ldo=None):
    """cc_cosine_neg_many_f32 into an (nq, ldo) buffer whose padding holds a NaN sentinel; returns (values, padding)."""
    nq, nc = q.shape[0], c.shape[0]
    ldo = ldo or nc
    out = torch.full((nq, ldo), 0, dtype=torch.int32, device="cuda").fill_(NAN_BITS).view(torch.float32)
    call("cc_cosine_neg_many_f32", ptr(q), q.stride(0), nq, ptr(c), c.stride(0), nc, 64, ptr(out), ldo, stream_ptr())
    return out[:, :nc], out[:, nc:]


def _one_card(allm, rows, ref):
    """cc_cosine_neg_f32 for every row index in ``rows`` of ``allm`` (one launch each) into the rows of ``ref``."""
    for i, r in enumerate(rows):
        call("cc_cosine_neg_f32", ptr(allm), allm.stride(0), allm.shape[0], 64, int(r), ptr(ref[i]), stream_ptr())
    return ref


SHAPES = [(1, 30001), (7, 20884), (129, 4099), (4099, 129), (20884, 7), (30001, 1), (129, 30001), (4099, 20884)]


@pytest.mark.parametrize("nq,nc", SHAPES)
def test_kernel_bit_equal_to_the_one_card_kernel(nq, nc):
    q, c = _emb(nq, 1, ld=72), _emb(nc, 2, ld=68)                  # ld > 64 on both sides
    allm = torch.cat([c, q]).contiguous()                         # candidates first: row j of the output is cand j
    ref = torch.empty((nq, nc + nq), device="cuda")
    _one_card(allm, range(nc, nc + nq), ref)
    ref = ref[:, :nc]
    pad4 = (nc + 3) // 4 * 4
    for ldo in (nc, pad4 + 4, nc + (1 if (nc + 1) % 4 else 2)):  # tight, padded float4 rows, padded unaligned rows
        got, pad = _many(q, c, ldo)
        assert _bits_equal(got, ref), ldo
        assert (pad.view(torch.int32) == NAN_BITS).all(), "wrote past num_cands"
    got, _ = _many(q.contiguous(), c.contiguous())
    assert _bits_equal(got, ref)


def test_kernel_zero_queries_is_a_no_op():
    q, c = _emb(4, 3), _emb(9, 4)
    out = torch.full((4, 9), 7.0, device="cuda")
    call("cc_cosine_neg_many_f32", ptr(q), 64, 0, ptr(c), 64, 9, 64, ptr(out), 9, stream_ptr())
    torch.cuda.synchronize()
    assert (out == 7.0).all()


def test_kernel_against_the_float64_formula():
    q, c = _emb(129, 5), _emb(4099, 6)
    got, _ = _many(q, c)
    qn, cn = (x.double().cpu().numpy() for x in (q, c))
    qn = qn / np.sqrt(np.maximum((qn * qn).sum(1, keepdims=True), 1e-12))
    cn = cn / np.sqrt(np.maximum((cn * cn).sum(1, keepdims=True), 1e-12))
    ref = -(qn @ cn.T)
    assert np.abs(got.cpu().numpy() - ref).max() < 1e-6
    # the restatement the single-card tests use, on one row
    allm = torch.cat([q, c]).double().cpu().numpy()
    assert np.abs(got[3].cpu().numpy() - od.similarity_np(allm, 3)[129:]).max() < 1e-6


# ---------------------------------------------------------------- the table against the one-card route
def _parent_similar(emb, c, q, n):
    """``MLRecommender.similar`` as it was: one cc_cosine_neg_f32 row, a batch-1 ascending select; device results."""
    dists = torch.empty((1, c), dtype=torch.float32, device="cuda")
    call("cc_cosine_neg_f32", ptr(emb), emb.stride(0), c, emb.shape[1], int(q), ptr(dists), stream_ptr())
    n = max(1, min(int(n), c))
    none_ptr = torch.zeros(2, dtype=torch.int64, device="cuda")
    none_idx = torch.zeros(1, dtype=torch.int32, device="cuda")
    ids, vals, _ = G.topn_masked(dists, none_ptr, none_idx, n, only_listed=False, descending=False)
    return ids[0], vals[0]


def _parent_table(emb, c, n, rows=None):
    rows = range(c) if rows is None else rows
    got = [_parent_similar(emb, c, q, n) for q in rows]
    return torch.stack([g[0] for g in got]), torch.stack([g[1] for g in got])


@pytest.fixture(scope="module", params=[4001, 20884], ids=["C4001", "C20884"])
def card_model(request):
    c = request.param
    model = M.CC_Recommender(c, device="cuda", seed=11, precision="fp32")
    rec = MLRecommender(model)
    return c, model, rec, rec.card_embeddings()


def test_table_equals_the_one_card_route(card_model):
    c, model, rec, emb = card_model
    ns = (1, 50, 128, 129, c) if c < 10000 else (50, 129)
    for n in ns:
        ids, dists = rec.similar_cards(None, n)
        pid, pd = _parent_table(emb, c, n)
        assert ids.shape == (c, min(n, c)) and torch.equal(ids, pid), n
        assert _bits_equal(dists, pd), n


def test_exclude_self_removes_exactly_the_query(card_model):
    c, model, rec, emb = card_model
    n = 50
    ids, dists = rec.similar_cards(None, n, exclude_self=True)
    pid, pd = (x.cpu().numpy() for x in _parent_table(emb, c, n + 1))
    ids, dists = ids.cpu().numpy(), dists.cpu().numpy()
    for q in range(c):
        keep = pid[q] != q
        assert np.array_equal(ids[q], pid[q][keep][:n]), q
        assert np.array_equal(dists[q].view(np.int32), pd[q][keep][:n].view(np.int32)), q
    sel = [5, 0, c - 1, 5]                                   # a list of ids, duplicates allowed
    lid, ld = rec.similar_cards(sel, n, exclude_self=True)
    assert np.array_equal(lid.cpu().numpy(), ids[sel]) and np.array_equal(ld.cpu().numpy(), dists[sel])


def test_similar_returns_the_one_card_route(card_model):
    c, model, rec, emb = card_model
    for q, n in ((0, 25), (17, 1), (c - 1, 129), (c // 2, c + 5), (3, 0)):
        ids, dists = rec.similar(q, n)
        pid, pd = _parent_similar(emb, c, q, n)
        assert np.array_equal(ids, pid.cpu().numpy()) and np.array_equal(dists.view(np.int32), pd.cpu().numpy().view(np.int32))
    ids, dists = rec.similar(9, 40, embeddings=emb)
    pid, pd = _parent_similar(emb, c, 9, 40)
    assert np.array_equal(ids, pid.cpu().numpy()) and np.array_equal(dists.view(np.int32), pd.cpu().numpy().view(np.int32))


def test_query_blocks_give_the_same_bits(card_model):
    c, model, rec, emb = card_model
    for n, self_offset in ((50, None), (50, 0), (c, None), (3000, 0)):
        one = rec.nearest(emb, emb, n, self_offset=self_offset)
        small = (4 * ((c + 3) // 4) + _lib.load().cc_topn_workspace_bytes(c, 1, n, 0)) * 37 + 5    # 37 rows a block
        many = rec.nearest(emb, emb, n, self_offset=self_offset, budget_bytes=small)
        assert torch.equal(one[0], many[0]) and _bits_equal(one[1], many[1]), (n, self_offset)
        assert one[0].shape == (c, min(n, c - (self_offset is not None)))
    # a query block that is a window of the corpus: self_offset names the window's first row
    sub = emb[100:400]
    a = rec.nearest(sub, emb, 20, self_offset=100)
    b = rec.similar_cards(list(range(100, 400)), 20, exclude_self=True)
    assert torch.equal(a[0], b[0]) and _bits_equal(a[1], b[1])
    with pytest.raises(ValueError):
        rec.nearest(sub, emb, 20, self_offset=c - 10)
    with pytest.raises(ValueError):
        rec.nearest(emb[:, :32], emb, 5)


# ---------------------------------------------------------------- cubes
def _expected(dist_rows, n, exclude=None):
    """NumPy's stable argsort of each distance row, with row i's excluded id dropped: (ids, values) of the first n."""
    ids, vals = [], []
    for i, row in enumerate(dist_rows):
        order = np.argsort(row, kind="stable")
        if exclude is not None:
            order = order[order != exclude[i]]
        ids.append(order[:n]); vals.append(row[order[:n]])
    return np.array(ids), np.array(vals)


@pytest.fixture(scope="module")
def cube_model():
    c = 1001                                                 # C % 4 != 0
    params = od.init_params(c, seed=4)
    model = M.CC_Recommender(c, device="cuda", precision="fp32")
    model.set_weights_dict(params)
    return c, params, model


def test_cube_embeddings_match_the_oracle_encoder(cube_model):
    c, params, model = cube_model
    ip, ix = synth_cubes_csr(300, c, size_lo=1, size_hi=120, seed=8)
    lists = [ix[ip[b]:ip[b + 1]].tolist() for b in range(300)]
    lists[7] = []                                            # an empty cube: the encoder of the zero vector
    csr = CubeCSR.from_lists(lists, c)
    rec = MLRecommender(model, chunk=64)                     # five chunks, the last one short
    got = rec.cube_embeddings(csr).cpu().numpy()
    _, _, cache = od.forward_np(params, csr.to_dense(), [0], onehot_rows_as_gather=True)
    ref = cache["main"][1][4]                                # the bottleneck's activations
    assert got.shape == (300, 64) and np.abs(got - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max())
    one = MLRecommender(model, chunk=8192).cube_embeddings(csr).cpu().numpy()          # one chunk
    assert np.abs(one - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max())
    with pytest.raises(ValueError):
        rec.cube_embeddings(CubeCSR.from_lists([[0]], c + 1))


def test_similar_cubes_ranks_the_kernels_distances(cube_model):
    c, params, model = cube_model
    ip, ix = synth_cubes_csr(700, c, size_lo=5, size_hi=90, seed=9)
    lists = [ix[ip[b]:ip[b + 1]].tolist() for b in range(700)]
    lists[30] = list(lists[12])                              # an identical cube: a tie at the top of row 12
    csr = CubeCSR.from_lists(lists, c)
    rec = MLRecommender(model, chunk=256)
    e = rec.cube_embeddings(csr)
    d, _ = _many(e, e)
    d = d.cpu().numpy()
    for n in (1, 50, 700):
        ids, dists = rec.similar_cubes(csr, n)
        want, wv = _expected(d, n, exclude=np.arange(700))
        assert np.array_equal(ids.cpu().numpy(), want) and np.array_equal(dists.cpu().numpy(), wv), n
    # an outside corpus, as a CSR or as its embeddings: nothing excluded
    q = csr.rows(np.arange(40))
    ip2, ix2 = synth_cubes_csr(500, c, size_lo=5, size_hi=90, seed=10)
    corpus = CubeCSR(ip2, ix2, c)
    ce = rec.cube_embeddings(corpus)
    a = rec.similar_cubes(q, 25, corpus=corpus)
    b = rec.similar_cubes(q, 25, corpus=ce)
    assert torch.equal(a[0], b[0]) and _bits_equal(a[1], b[1])
    dq, _ = _many(rec.cube_embeddings(q), ce)
    want, wv = _expected(dq.cpu().numpy(), 25)
    assert np.array_equal(a[0].cpu().numpy(), want) and np.array_equal(a[1].cpu().numpy(), wv)
    with pytest.raises(ValueError):
        rec.similar_cubes(CubeCSR.from_lists([[0]], c + 3), 5)
    with pytest.raises(ValueError):
        rec.similar_cubes(q, 5, corpus=CubeCSR.from_lists([[0]], c - 1))


def test_similar_cubes_past_the_row_select(cube_model):
    """27 500 corpus cubes: rows too long for the shared-memory row select (two rows of up to ~26 900 floats), so the
    streaming select ranks them."""
    c, params, model = cube_model
    k = 27500
    ip, ix = synth_cubes_csr(k, c, size_lo=5, size_hi=60, seed=12)
    corpus = CubeCSR(ip, ix, c)
    rec = MLRecommender(model)
    e = rec.cube_embeddings(corpus)
    q = corpus.rows(np.arange(0, k, 550))
    ids, dists = rec.similar_cubes(q, 50, corpus=e)
    dq, _ = _many(rec.cube_embeddings(q), e)
    want, wv = _expected(dq.cpu().numpy(), 50)
    assert np.array_equal(ids.cpu().numpy(), want) and np.array_equal(dists.cpu().numpy(), wv)
    ids, dists = rec.similar_cubes(corpus, 50)              # against each other, self excluded
    sample = np.arange(7, k, 611)
    ds, _ = _many(e[torch.from_numpy(sample).cuda()], e)
    want, wv = _expected(ds.cpu().numpy(), 50, exclude=sample)
    assert np.array_equal(ids.cpu().numpy()[sample], want) and np.array_equal(dists.cpu().numpy()[sample], wv)


def test_tf32_model_ranks_its_own_embeddings():
    c = 2003
    model = M.CC_Recommender(c, device="cuda", seed=5, precision="tf32")
    rec = MLRecommender(model, chunk=128)
    ip, ix = synth_cubes_csr(400, c, size_lo=5, size_hi=90, seed=13)
    csr = CubeCSR(ip, ix, c)
    e = rec.cube_embeddings(csr)
    d, _ = _many(e, e)
    ids, dists = rec.similar_cubes(csr, 30)
    want, wv = _expected(d.cpu().numpy(), 30, exclude=np.arange(400))
    assert np.array_equal(ids.cpu().numpy(), want) and np.array_equal(dists.cpu().numpy(), wv)
    emb = rec.card_embeddings()
    tid, td = rec.similar_cards(None, 40)
    pid, pd = _parent_table(emb, c, 40)
    assert torch.equal(tid, pid) and _bits_equal(td, pd)


# ---------------------------------------------------------------- side effects and the command line
def test_no_side_effects_and_the_table_cli(tmp_path, capsys):
    from cubecobrarecommender_b200.scripts import similarity as SIM
    c = 300
    params = od.init_params(c, seed=3)
    model = M.CC_Recommender(c, device="cuda", precision="fp32")
    model.set_weights_dict(params)
    model.save(str(tmp_path / "model"))
    before = {k: v.copy() for k, v in model.get_weights_dict().items()}
    rec = MLRecommender(model, chunk=32)
    ip, ix = synth_cubes_csr(90, c, size_lo=5, size_hi=40, seed=14)
    csr = CubeCSR(ip, ix, c)
    emb = rec.card_embeddings()
    emb_before = emb.clone()
    rec.similar_cards(None, 10, exclude_self=True, embeddings=emb)
    rec.similar(4, 10, embeddings=emb)
    rec.similar_cubes(csr, 10)
    rec.similar_cubes(csr.rows(np.arange(5)), 10, corpus=rec.cube_embeddings(csr))
    rec.nearest(emb[:50], emb, 7, self_offset=0)
    after = model.get_weights_dict()
    assert all(np.array_equal(before[k], after[k]) for k in before)
    assert _bits_equal(emb, emb_before)
    for exclude in (False, True):
        path = str(tmp_path / f"table_{int(exclude)}.npz")
        SIM.main(["--table", "12", path] + (["--exclude-self"] if exclude else []), model_dir=str(tmp_path / "model"))
        line = capsys.readouterr().out.strip().splitlines()
        assert len(line) == 1 and line[0].startswith(f"similar-cards table: {c} cards x 12 neighbours")
        z = np.load(path)
        ids, dists = rec.similar_cards(None, 12, exclude_self=exclude)
        assert z["ids"].dtype == np.int32 and z["dists"].dtype == np.float32 and z["ids"].shape == (c, 12)
        assert np.array_equal(z["ids"], ids.cpu().numpy())
        assert np.array_equal(z["dists"].view(np.int32), dists.cpu().numpy().view(np.int32))
        assert not exclude or (z["ids"] != np.arange(c)[:, None]).all()
    # the reference form is unchanged
    json.dump({str(i): f"card {i}" for i in range(c)}, open(tmp_path / "id_map.json", "w"))
    out = SIM.main(["card_17", "5"], model_dir=str(tmp_path / "model"), id_map=str(tmp_path / "id_map.json"))
    assert len(out) == 5 and out[0][0] == "card 17"
