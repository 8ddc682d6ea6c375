"""Rows wider than 22 528 cards: every card-count boundary at which the softmax-KL kernels, the top-N selects and the
engine change their code path, from both sides, against float64 / NumPy references.

Which code each boundary selects (loss.cu cc_softmax_kl_fwd_bwd_metrics / cc_softmax_kl_fuses_dbias, topn.cu
select_small_n / rowselect_eligible, engine.py DAEEngine._forward); the parametrisation ids name the kernel a case
reaches:

    cards C                  softmax-KL with dbias          softmax-KL without dbias     top-N, n <= 128, whole row
    <= 21 504, C % 4 == 0    softmax_kl_regs_kernel 768x7   softmax_kl_rows_fast_kernel  REGS row select
    21 508 - 22 528          softmax_kl_regs_kernel 512x11  softmax_kl_rows_fast_kernel  REGS row select
    22 532 - 25 600          persistent, 1024 threads       softmax_kl_rows_fast_kernel  row select in shared memory
    25 604 - 26 968          (none: rows kernel + colsum)   softmax_kl_rows_kernel<0>    row select in shared memory
    > 26 968                 (none)                         softmax_kl_rows_kernel<0>    warp-per-cube streaming select
    C % 4 != 0 (<= 25 600)   (none)                         softmax_kl_rows_kernel<1>    row select if ld % 4 == 0

The engine cases build a cooccurrence graph of up to 30 000 cards (M-hat alone is 3.6 GB) once per card count; the
module-scoped fixture frees it before the next one is built."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from cubecobrarecommender_b200 import _lib, graph as G
from cubecobrarecommender_b200.ml import engine as E, generator as GEN, inference as INF, model as M, train as T
from cubecobrarecommender_b200.sparse import CubeCSR
from oracle import dae as od, graph as og
from test_gpu_baseline_shapes import BIG_GRADS, GRAD_TOL, GRAD_TOL_FIRST_LAYER, LOSS_TOL
from test_gpu_validation import _readback

EPS = 1e-7          # Keras' clip of both softmax-KL operands


def _cpad(c):
    return (c + 127) // 128 * 128


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ------------------------------------------------------------------ softmax-KL kernels
def _kl_problem(c, rows, nt, seed):
    """Logits (rows, cpad) and target rows (nt, cpad) in float32 with NaN in columns [c, cpad), which no kernel may read;
    target row 0 has its maximum in column 11, row 1 in column c - 3.  Rows 2 and 3 hold their maximal logit twice, in
    columns 11 and c - 3: row 2 (target row 0) is a hit under the first-index rule, row 3 (target row 1) a miss.  Row 1
    has one huge logit (most of its q fall below the 1e-7 clip); every other even row from 4 on has its maximal logit at
    its target row's argmax.  Target rows repeat (nt < rows)."""
    cpad = _cpad(c)
    rng = np.random.default_rng(seed)
    t = rng.random((nt, c))
    t[t < 0.7] = 0
    t[0, 11] = t[1, c - 3] = 2.0
    t /= t.sum(1, keepdims=True)
    t32 = np.full((nt, cpad), np.nan, dtype=np.float32)
    t32[:, :c] = t
    tr = rng.integers(0, nt, size=rows).astype(np.int32)
    tr[2], tr[3] = 0, 1
    am = np.argmax(t32[:, :c], axis=1)
    z = np.full((rows, cpad), np.nan, dtype=np.float32)
    z[:, :c] = rng.standard_normal((rows, c)).astype(np.float32) * 3
    for i in (2, 3):
        z[i, 11] = z[i, c - 3] = z[i, :c].max() + 1
    z[1, 5] = 45.0
    for i in range(4, rows, 2):
        z[i, am[tr[i]]] = z[i, :c].max() + 0.5
    # no q within 1% of the 1e-7 clip: a q that float rounding may put on either side also moves S, the sum of t' over
    # the unclipped cards, and with it every dlogit of its row (one such flip measured 5.5e-5 of max |dz| at 22 532
    # cards against the 2e-5 bar)
    q = od.softmax_np(z[:, :c].astype(np.float64))
    z[:, :c][np.abs(q - EPS) < 1e-2 * EPS] += np.float32(0.03)
    return z, t32, tr


def _kl_oracle(z, t32, tr, c, scale):
    zz = z[:, :c].astype(np.float64)
    tt = t32[tr, :c].astype(np.float64)
    q = od.softmax_np(zz)
    tcl = np.clip(tt, EPS, 1.0)
    rows_ref = (tcl * np.log(tcl / np.clip(q, EPS, 1.0))).sum(1)
    un = (q >= EPS) & (q <= 1)
    dz_ref = scale * (q * (tcl * un).sum(1, keepdims=True) - tcl * un)
    hits_ref = (np.argmax(tt, axis=1) == np.argmax(zz, axis=1)).astype(np.int32)
    return rows_ref, dz_ref, np.abs(q - EPS) < 1e-10, hits_ref


def _check_kl(rl, dz, c, fast, rows_ref, dz_ref, edge, what):
    """The bars of test_gpu_dae.py::test_softmax_kl_persistent_kernels_vs_oracle."""
    got_rows = rl.cpu().numpy()
    err = np.abs(got_rows - rows_ref).max() / np.abs(rows_ref).max()
    assert err < (2e-5 if fast else 5e-6), (what, err)
    got = dz[:, :c].double().cpu().numpy()
    err = np.abs(got - dz_ref)[~edge].max() / np.abs(dz_ref).max()
    assert err < (2e-3 if fast else 2e-5), (what, err)            # fast: MUFU exp + tf32-rounded dlogits
    assert (dz[:, c:] == 0).all(), what


# (C, kernel with dbias, kernel without dbias)
KL_CASES = [(21504, "regs768x7", "rows_fast"), (21508, "regs512x11", "rows_fast"), (22528, "regs512x11", "rows_fast"),
            (22532, "persistent1024", "rows_fast"), (25600, "persistent1024", "rows_fast"),
            (25604, None, "rows_nocache"), (30000, None, "rows_nocache"), (24001, None, "rows_cache")]


@pytest.mark.parametrize("fast", [0, 1])
@pytest.mark.parametrize("c,with_dbias,without_dbias", KL_CASES, ids=[f"{c}-{a or 'unfused'}-{b}" for c, a, b in KL_CASES])
def test_softmax_kl_kernels_vs_oracle(c, with_dbias, without_dbias, fast):
    """Row loss, dlogits, bias gradient and categorical hits of every softmax-KL kernel against float64: 320 rows (more
    than two per CTA of the persistent kernels), NaN in the padding of logits and target rows, clipped q, a maximal
    logit that appears twice."""
    lib = _lib.load()
    rows, nt = 320, 64
    cpad = _cpad(c)
    scale = 0.1 / rows
    z_h, t_h, tr_h = _kl_problem(c, rows, nt, seed=c)
    z, t, tr = _dev(z_h), _dev(t_h), _dev(tr_h)
    rows_ref, dz_ref, edge, hits_ref = _kl_oracle(z_h, t_h, tr_h, c, scale)
    assert hits_ref[2] == 1 and hits_ref[3] == 0 and 0.4 < hits_ref.mean() < 0.6
    st = E.stream_ptr()
    fused = lib.cc_softmax_kl_fuses_dbias(c, cpad, cpad, cpad, cpad)
    assert bool(fused) == (with_dbias is not None)

    # without dbias: rows_fast (aligned rows, C <= 25 600), else the 1024-thread rows kernel with or without the
    # shared-memory row cache
    dz = torch.full((rows, cpad), 9.0, device="cuda")
    rl = torch.zeros(rows, dtype=torch.float64, device="cuda")
    E.call("cc_softmax_kl_fwd_bwd_metrics", E.ptr(z), cpad, E.ptr(t), cpad, E.ptr(tr), rows, c, cpad, scale, E.ptr(dz),
           cpad, E.ptr(rl), fast, None, None, 0, None, None, None, st)
    _check_kl(rl, dz, c, fast, rows_ref, dz_ref, edge, without_dbias)
    if not fused:
        return
    # with dbias: the persistent kernels, with and without the t' log t' table, counting categorical hits
    table = torch.zeros(nt, dtype=torch.float64, device="cuda")
    E.call("cc_kl_target_table", E.ptr(t), cpad, nt, c, E.ptr(table), st)
    am = torch.zeros(nt, dtype=torch.int32, device="cuda")
    E.call("cc_kl_target_argmax", E.ptr(t), cpad, nt, c, E.ptr(am), st)
    assert np.array_equal(am.cpu().numpy(), np.argmax(t_h[:, :c], axis=1))
    for use_table in (False, True):
        dz = torch.full((rows, cpad), 9.0, device="cuda")
        rl = torch.zeros(rows, dtype=torch.float64, device="cuda")
        db = torch.full((c,), 3.0, device="cuda")
        hit = torch.full((rows,), -1, dtype=torch.int32, device="cuda")
        E.call("cc_softmax_kl_fwd_bwd_metrics", E.ptr(z), cpad, E.ptr(t), cpad, E.ptr(tr), rows, c, cpad, scale, E.ptr(dz),
               cpad, E.ptr(rl), fast, E.ptr(db), None, 0, E.ptr(table) if use_table else None, E.ptr(am), E.ptr(hit), st)
        _check_kl(rl, dz, c, fast, rows_ref, dz_ref, edge, (with_dbias, use_table))
        ref_db = dz[:, :c].double().sum(0)
        assert (db.double() - ref_db).abs().max().item() < 2e-6 * ref_db.abs().max().item() + 1e-12
        got_hits = hit.cpu().numpy()
        assert np.array_equal(got_hits, hits_ref), np.nonzero(got_hits != hits_ref)
        assert got_hits.mean() == od.categorical_accuracy_np(z_h[:, :c], t_h[tr_h, :c])
    # the loss-only kernel: the training kernel's row losses and hits, bit for bit, up to 22 528 cards and no further
    rl_e = torch.zeros(rows, dtype=torch.float64, device="cuda")
    hit_e = torch.full((rows,), -1, dtype=torch.int32, device="cuda")
    args = (E.ptr(z), cpad, E.ptr(t), cpad, E.ptr(tr), rows, c, cpad, E.ptr(table), E.ptr(am), E.ptr(rl_e), E.ptr(hit_e),
            fast, st)
    if c <= E.KL_LOSS_MAX_CARDS:
        E.call("cc_softmax_kl_loss", *args)
        assert torch.equal(rl_e, rl) and torch.equal(hit_e, hit)
    else:
        with pytest.raises(_lib.CubeCobraError, match="cc_softmax_kl_loss"):
            E.call("cc_softmax_kl_loss", *args)


@pytest.mark.parametrize("c", [20884, 22532])
def test_categorical_hits_helper_equals_the_kernel_count(c):
    """engine.categorical_hits (the count where no persistent kernel runs) gives exactly the persistent kernel's row_hit
    on the same logits: every row holds its maximal logit twice, one copy at the target row's argmax, the other before or
    after it, so the first-index rule decides every row."""
    rows, nt = 320, 64
    cpad = _cpad(c)
    z_h, t_h, tr_h = _kl_problem(c, rows, nt, seed=c + 1)
    am_h = np.argmax(t_h[:, :c], axis=1)
    for i in range(rows):
        a = am_h[tr_h[i]]
        other = (a + (1 + i % 7) * (1 if i % 2 == 0 else -1)) % c       # after the target's argmax, or before it
        z_h[i, a] = z_h[i, other] = np.nanmax(z_h[i]) + 1
    ref = (np.argmax(z_h[:, :c], axis=1) == am_h[tr_h]).astype(np.int32)
    assert 0.2 < ref.mean() < 0.8
    z, t, tr = _dev(z_h), _dev(t_h), _dev(tr_h)
    st = E.stream_ptr()
    am = torch.zeros(nt, dtype=torch.int32, device="cuda")
    E.call("cc_kl_target_argmax", E.ptr(t), cpad, nt, c, E.ptr(am), st)
    dz = torch.empty((rows, cpad), device="cuda")
    rl = torch.zeros(rows, dtype=torch.float64, device="cuda")
    db = torch.zeros(c, device="cuda")
    hit_k = torch.full((rows,), -1, dtype=torch.int32, device="cuda")
    E.call("cc_softmax_kl_fwd_bwd_metrics", E.ptr(z), cpad, E.ptr(t), cpad, E.ptr(tr), rows, c, cpad, 0.1 / rows,
           E.ptr(dz), cpad, E.ptr(rl), 1, E.ptr(db), None, 0, None, E.ptr(am), E.ptr(hit_k), st)
    hit_h = torch.full((rows + 5,), -1, dtype=torch.int32, device="cuda")
    E.categorical_hits(z, rows, c, tr, am, hit_h)
    assert np.array_equal(hit_k.cpu().numpy(), ref)
    assert torch.equal(hit_h[:rows], hit_k) and (hit_h[rows:] == -1).all()


# ------------------------------------------------------------------ top-N and target ranks
def _algo(a):
    _lib.call("cc_topn_set_algo", a)


def _radix(on):
    _lib.call("cc_topn_set_force_radix", on)


def _wide_values(c, batch, rng):
    vals = (rng.standard_normal((batch, c)) * 2).astype(np.float32)
    vals[0] = np.sort(vals[0])                                                  # ascending
    vals[1] = np.sort(vals[1])[::-1]                                            # descending
    vals[2] = rng.integers(0, 30, size=c).astype(np.float32) / 4 - 3           # long tie runs
    vals[3][rng.random(c) < 0.7] = -np.inf
    vals[4][rng.random(c) < 0.3] = np.inf
    vals[5] = np.where(rng.random(c) < 0.5, np.float32(-0.0), np.float32(0.0))  # -0.0 ties with +0.0
    vals[5][rng.random(c) < 0.01] = 1.0
    return vals


def _mask_lists(c, batch, rng):
    lists = [np.sort(rng.choice(c, size=rng.integers(0, 700), replace=False)) for _ in range(batch)]
    lists[2] = np.zeros(0, np.int64)
    lists[-1] = np.arange(3, c)                                                 # 3 candidates left (only-listed: c - 3)
    lists[-2] = np.sort(rng.choice(c, size=40, replace=False))                  # only-listed: fewer than n
    return lists


def _expected_select(v, listed, only_listed, desc, n):
    order = v.argsort(kind="stable")
    if desc:
        order = order[::-1]                       # descending score, ties -> larger index first
    inm = np.zeros(len(v), bool)
    inm[listed] = True
    return order[inm[order] == bool(only_listed)][:n]


# (C, automatic path with ld = C, with ld padded past C)
TOPN_CASES = [(22528, "regs", "regs"), (22529, "streaming", "smem"), (22532, "smem", "smem"), (26968, "smem", "smem"),
              (26969, "streaming", "streaming"), (30000, "streaming", "streaming")]


@pytest.mark.parametrize("padded", [False, True], ids=["ld=C", "ld>C"])
@pytest.mark.parametrize("c,path_unpadded,path_padded", TOPN_CASES, ids=[f"{c}-{a}-{b}" for c, a, b in TOPN_CASES])
def test_topn_wide_rows_vs_numpy(c, path_unpadded, path_padded, padded):
    """The automatic float32 select (both the scores and the fused-sigmoid form) against NumPy's stable argsort in all
    four mask / direction modes, and against the streaming select and the radix select: ties, +-inf, -0.0 beside +0.0,
    sorted rows, masks that leave fewer than n candidates, padding of +inf that must not be read."""
    batch, n = 8, 100
    ld = (c // 128 + 1) * 128 if padded else c
    rng = np.random.default_rng(c + ld)
    vals = _wide_values(c, batch, rng)
    lists = _mask_lists(c, batch, rng)
    csr = CubeCSR.from_lists(lists, c)
    mp, mi = _dev(csr.indptr.astype(np.int64)), _dev(csr.indices.astype(np.int32))
    full = torch.full((batch, ld), np.inf, dtype=torch.float32, device="cuda")
    full[:, :c] = _dev(vals)
    probs_full = torch.empty_like(full)
    E.call("cc_sigmoid_f32", E.ptr(full), E.ptr(probs_full), full.numel(), E.stream_ptr())
    probs = probs_full[:, :c].cpu().numpy()         # the float32 sigmoid the fused select ranks (CUDA's expf, not NumPy's)
    scores = full[:, :c]
    assert scores.stride(0) == ld
    try:
        for sigmoid in (False, True):
            ranked = probs if sigmoid else vals
            for only_listed, desc in ((False, True), (True, False), (False, False), (True, True)):
                kw = dict(only_listed=only_listed, descending=desc, sigmoid=sigmoid)
                auto = G.topn_masked(scores, mp, mi, n, **kw)
                _algo(1)
                stream = G.topn_masked(scores, mp, mi, n, **kw)
                _algo(0)
                for x, y in zip(auto, stream):
                    assert torch.equal(x, y), (sigmoid, only_listed, desc)
                if not sigmoid:
                    _radix(1)
                    radix = G.topn_masked(scores, mp, mi, n, **kw)
                    _radix(0)
                    for x, y in zip(auto, radix):
                        assert torch.equal(x, y), (only_listed, desc)
                ids, v, cnt = (a.cpu().numpy() for a in auto)
                for r in range(batch):
                    expect = _expected_select(ranked[r], lists[r], only_listed, desc, n)
                    assert cnt[r] == len(expect) and np.array_equal(ids[r][:cnt[r]], expect), (sigmoid, only_listed, desc, r)
                    assert np.array_equal(v[r][:cnt[r]], ranked[r][expect])
                    assert (ids[r][cnt[r]:] == -1).all()
        if c == 22529 and padded:               # the rows qualify for the row select, but not for its register form
            _algo(4)
            with pytest.raises(_lib.CubeCobraError, match="REGS"):
                G.topn_masked(scores, mp, mi, n)
    finally:
        _algo(0)
        _radix(0)


@pytest.mark.parametrize("padded", [False, True], ids=["ld=C", "ld>C"])
def test_rank_targets_sigmoid_wide_rows_vs_numpy(padded):
    """cc_rank_targets_f32 with the fused sigmoid at 30 000 cards: a row with 3000 targets (three sweeps of 1024),
    masked and duplicate targets, ties and saturated logits, against NumPy's stable argsort of the device probabilities."""
    c, batch = 30000, 6
    ld = _cpad(c) if padded else c
    rng = np.random.default_rng(7 + padded)
    vals = _wide_values(c, batch, rng)
    vals[4] = rng.choice(np.array([20.0, 25.0, -100.0, 0.5, -0.5], dtype=np.float32), size=c)   # sigmoid 1.0 / 0: ties
    lists = _mask_lists(c, batch, rng)
    lists[-1] = np.sort(rng.choice(c, size=5000, replace=False))
    targets = []
    for b in range(batch):
        k = 3000 if b == 0 else int(rng.integers(1, 500))
        tg = rng.choice(c, size=k, replace=False)
        if len(lists[b]):
            tg[:3] = lists[b][:3]                                   # masked targets: -1
        targets.append(np.concatenate([tg, tg[-2:]]))               # duplicates: the same rank
    csr = CubeCSR.from_lists(lists, c)
    mp, mi = _dev(csr.indptr.astype(np.int64)), _dev(csr.indices.astype(np.int32))
    tp = np.zeros(batch + 1, np.int64)
    tp[1:] = np.cumsum([len(x) for x in targets])
    ti = np.concatenate(targets).astype(np.int32)
    full = torch.full((batch, ld), np.inf, dtype=torch.float32, device="cuda")
    full[:, :c] = _dev(vals)
    probs_full = torch.empty_like(full)
    E.call("cc_sigmoid_f32", E.ptr(full), E.ptr(probs_full), full.numel(), E.stream_ptr())
    probs = probs_full[:, :c].cpu().numpy()
    got = G.rank_targets(full[:, :c], mp, mi, _dev(tp), _dev(ti), sigmoid=True).cpu().numpy()
    for b in range(batch):
        cand = _expected_select(probs[b], lists[b], False, True, c)
        pos = np.full(c, -1, np.int64)
        pos[cand] = np.arange(len(cand))
        assert np.array_equal(got[tp[b]:tp[b + 1]], pos[targets[b]]), b


# ------------------------------------------------------------------ the engine end to end
REG = 0.1
K_CUBES, B = 384, 256
# accuracy bands of test_gpu_dae.py::test_keras_accuracy_metrics_vs_oracle: cells / rows whose logits are within the
# mode's rounding of the decision may flip
BAND = {"fp32": 1e-5, "tf32": 5e-3, "bf16": 3e-2}


def _params(c, seed=0):
    params = od.init_params(c, seed=seed)
    rng = np.random.default_rng(seed + 1)
    for kname in params:                    # non-zero biases: every bias gradient matters, livelier logits
        if kname.endswith("bias"):
            params[kname] = (rng.standard_normal(params[kname].shape) * 0.1).astype(np.float32)
    params["reg_reconstruction/bias"][0] = 5.0      # the reg tower's first maximal logit is card 0 (see _two_pool_cubes)
    return params


def _two_pool_cubes(k, c, seed):
    """Even cubes draw from cards [1, c/2) and all hold card 0; odd cubes draw from [c/2, c).  So M-hat's first maximal
    column is card 0 for every card of the first pool and another card for the second: with the reg tower's logits
    peaked at card 0, about half of the reg rows are categorical hits, and a hit depends on which M-hat row the reg row
    uses, not on its position in the batch."""
    rng = np.random.default_rng(seed)
    lists = []
    for i in range(k):
        size = int(rng.integers(200, 400))
        if i % 2 == 0:
            lists.append(np.concatenate([[0], np.sort(rng.choice(np.arange(1, c // 2), size, replace=False))]))
        else:
            lists.append(np.sort(rng.choice(np.arange(c // 2, c), size, replace=False)))
    return CubeCSR.from_lists(lists, c)


@pytest.fixture(scope="module", params=[24000, 30000, 24001], ids=["24000-persistent", "30000-rows_nocache",
                                                                      "24001-rows_cache"])
def wide(request):
    """Cubes, graph, one noise draw of the CUDA noise kernel read back, and the float64 oracle's loss, gradients and
    accuracies on exactly that (x, y, r), following test_gpu_baseline_shapes.headline_step at B = R = 256."""
    c = request.param
    csr = _two_pool_cubes(K_CUBES, c, seed=c % 1009)
    gr = G.build_graph(csr, "cuda", want_m64=False, want_mhat=True, want_neg=True)
    prob, alias = E.alias_table(gr.neg_sampler.cpu().numpy(), "cuda")
    params = _params(c)
    model = M.CC_Recommender(c, device="cuda", precision="fp32")
    eng = E.DAEEngine(model, gr.mhat, batch=B, reg_rows=B, reg=REG, max_cube_size=csr.max_size)
    indptr, indices = G.upload_csr(csr, "cuda")
    eng.sample_batch(indptr, indices, torch.arange(B, dtype=torch.int32, device="cuda"), prob, alias, 0.2, 0.1, seed=99)
    eng.check_overflow()
    xl, xi = eng.x_len.cpu().numpy(), eng.x_idx.cpu().numpy()
    x = np.zeros((B, c))
    for i in range(B):
        x[i, xi[i, :xl[i]]] = 1
    bits = eng.y_bits.cpu().numpy().view(np.uint32)
    y = ((bits[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(B, -1)[:, :c].astype(np.float64)
    rows = eng.reg_rows[:B].cpu().numpy().astype(np.int64)
    fixed = dict(x_idx=eng.x_idx.clone(), x_len=eng.x_len.clone(), y_bits=eng.y_bits.clone(), reg_rows=eng.reg_rows.clone())
    t_rows = og.m_hat_rows(csr.indptr, csr.indices, c, rows)
    got_rows = gr.mhat[torch.from_numpy(rows).cuda(), :c].cpu().numpy().astype(np.float64)
    nz = t_rows > 0
    assert (np.abs(got_rows[nz] - t_rows[nz]) / t_rows[nz]).max() < 1e-6 and (got_rows[~nz] == 0).all()
    t32 = t_rows.astype(np.float32).astype(np.float64)
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    (tot, bce, kl), grads = od.loss_and_grads_np(p64, x, y, rows, t32, REG, onehot_rows_as_gather=True)
    z1, z2, _ = od.forward_np(p64, x, rows, onehot_rows_as_gather=True)
    acc = (od.binary_accuracy_np(z1, y), od.categorical_accuracy_np(z2, t32.astype(np.float32)))
    assert 0.2 < acc[1] < 0.8, acc
    top2 = np.sort(z2, axis=1)[:, -2:]
    near = {p: (float(np.mean(np.abs(z1) < band * np.abs(z1).max())),
                float(np.mean((top2[:, 1] - top2[:, 0]) < band * np.abs(z2).max()))) for p, band in BAND.items()}
    keep = {k: grads[k] for k in BIG_GRADS}
    del eng, model, x, y, z1, z2, grads
    torch.cuda.empty_cache()
    yield dict(c=c, csr=csr, mhat=gr.mhat, params=params, fixed=fixed, loss=(tot, bce, kl), grads=keep, acc=acc, near=near)
    del gr
    torch.cuda.empty_cache()


STEP_MODES = {24000: ("fp32", "tf32", "bf16"), 30000: ("fp32", "tf32"), 24001: ("fp32",)}


def _engine(w, precision, batch=B, metrics=True):
    model = M.CC_Recommender(w["c"], device="cuda", precision=precision)
    model.set_weights_dict(w["params"])
    eng = E.DAEEngine(model, w["mhat"], batch=batch, reg_rows=batch, reg=REG, max_cube_size=w["csr"].max_size,
                      metrics=metrics)
    return model, eng


def test_train_step_vs_oracle(wide):
    """One train step with metrics on, in every mode the card count allows, against the float64 loss, the five big
    gradients and both Keras accuracies; the modes it does not allow fail with their errors."""
    w = wide
    c = w["c"]
    f = w["fixed"]
    tot, bce, kl = w["loss"]
    for precision in STEP_MODES[c]:
        model, eng = _engine(w, precision)
        eng.x_idx.copy_(f["x_idx"]); eng.x_len.copy_(f["x_len"])
        eng.set_batch(M.SparseBatch(eng.x_idx.view(-1), eng.x_start, eng.x_len), f["y_bits"], f["reg_rows"][:B])
        eng.forward_backward()
        got = eng.loss3.cpu().numpy()
        tol = LOSS_TOL[precision]
        for g, ref in zip(got, (bce, kl, tot)):
            assert abs(g - ref) / ref < tol, (precision, got, w["loss"])
        for kname, gref in w["grads"].items():
            g = model.store.g(kname).cpu().numpy().astype(np.float64)
            scale = np.abs(gref).max()
            assert scale > 0
            tol_g = (GRAD_TOL_FIRST_LAYER if kname == "encoder_e1/kernel" else GRAD_TOL)[precision]
            assert np.abs(g - gref).max() / scale < tol_g, (precision, kname, np.abs(g - gref).max() / scale)
        acc = eng.metrics2.cpu().numpy()
        near = w["near"][precision]
        for i in range(2):
            assert abs(acc[i] - w["acc"][i]) <= near[i] + 1e-12, (precision, i, acc, w["acc"], near)
        del eng, model
    if c == 30000:
        model, eng = _engine(w, "bf16")
        eng.x_idx.copy_(f["x_idx"]); eng.x_len.copy_(f["x_len"])
        eng.set_batch(M.SparseBatch(eng.x_idx.view(-1), eng.x_start, eng.x_len), f["y_bits"], f["reg_rows"][:B])
        with pytest.raises(RuntimeError, match="bf16 mode needs the persistent softmax-KL kernel"):
            eng.forward_backward()
        torch.cuda.synchronize()
    if c % 4:
        for precision in ("tf32", "bf16"):
            with pytest.raises(ValueError, match="tensor-core precision modes need num_cards % 4 == 0"):
                _engine(w, precision)


EVAL_MODES = {24000: ("tf32", "bf16"), 30000: ("fp32", "tf32"), 24001: ("fp32",)}


@pytest.mark.parametrize("metrics", [True, False])
def test_evaluate_vs_oracle(wide, metrics):
    """train.evaluate over 192 held-out cubes in batches of 64 against the float64 loss and both accuracies of the same
    noise draws and reg rows (read back), in the modes the card count allows."""
    w = wide
    c = w["c"]
    gen = GEN.DataGenerator(w["mhat"], w["csr"], batch_size=64, noise=0.2, seed=5)
    _, val = gen.split(0.5)
    for precision in EVAL_MODES[c]:
        model = M.CC_Recommender(c, device="cuda", precision=precision)
        model.set_weights_dict(w["params"])
        res = T.evaluate(model, val, REG, metrics=metrics)
        assert set(res) == {"loss", "output_1_loss", "output_2_loss"} | (
            {"output_1_accuracy", "output_2_accuracy"} if metrics else set())
        x, y, rows = _readback(val, model)
        p64 = {k: v.astype(np.float64) for k, v in w["params"].items()}
        z1, z2, _ = od.forward_np(p64, x, rows, onehot_rows_as_gather=True)
        t = w["mhat"][torch.from_numpy(rows).cuda(), :c].double().cpu().numpy()
        bce, kl = od.bce_from_logits_np(z1, y), od.kld_np(t, od.softmax_np(z2))
        tol = LOSS_TOL[precision]
        assert abs(res["output_1_loss"] - bce) / bce < tol, (precision, res, bce)
        assert abs(res["output_2_loss"] - kl) / kl < tol, (precision, res, kl)
        assert abs(res["loss"] - (bce + REG * kl)) / (bce + REG * kl) < tol
        if metrics:
            band = BAND[precision]
            near1 = float(np.mean(np.abs(z1) < band * np.abs(z1).max()))
            top2 = np.sort(z2, axis=1)[:, -2:]
            near2 = float(np.mean((top2[:, 1] - top2[:, 0]) < band * np.abs(z2).max()))
            ref1, ref2 = od.binary_accuracy_np(z1, y), od.categorical_accuracy_np(z2, t.astype(np.float32))
            assert abs(res["output_1_accuracy"] - ref1) <= near1 + 1e-12, (precision, res, ref1, near1)
            assert abs(res["output_2_accuracy"] - ref2) <= near2 + 1e-12, (precision, res, ref2, near2)
            assert 0.0 < ref2 < 1.0


def test_recommend_and_target_ranks_vs_numpy(wide):
    """recommend_device (fused-sigmoid top-50) and target_ranks_device against the reference's ranking walk on the
    float32 probabilities of a forward pass over the same 128 cubes (one chunk: the same batch shape, so the same
    logits bit for bit)."""
    w = wide
    c = w["c"]
    model = M.CC_Recommender(c, device="cuda", precision="fp32" if c % 4 else "tf32")
    model.set_weights_dict(w["params"])
    rec = INF.MLRecommender(model)
    cubes = w["csr"].rows(np.arange(128))
    n = 50
    ids, vals, cnt = (a.cpu().numpy() for a in rec.recommend_device(cubes, n))
    probs = rec.probabilities(cubes).cpu().numpy()
    for j in range(cubes.num_cubes):
        in_cube = np.zeros(c, dtype=np.int8)
        in_cube[cubes.indices[cubes.indptr[j]:cubes.indptr[j + 1]]] = 1
        expect = od.rank_additions(probs[j], in_cube, n)
        assert cnt[j] == n and ids[j].tolist() == expect, j
        assert np.array_equal(vals[j], probs[j][expect])
    lists = [cubes.indices[cubes.indptr[j]:cubes.indptr[j + 1]] for j in range(cubes.num_cubes)]
    visible = CubeCSR.from_lists([x[x % 5 != 0] for x in lists], c)
    hidden = CubeCSR.from_lists([x[x % 5 == 0] for x in lists], c)
    ranks = rec.target_ranks_device(visible, hidden).cpu().numpy()
    pv = rec.probabilities(visible).cpu().numpy()
    for j in range(visible.num_cubes):
        vis = visible.indices[visible.indptr[j]:visible.indptr[j + 1]]
        cand = _expected_select(pv[j], vis, False, True, c)
        pos = np.full(c, -1, np.int64)
        pos[cand] = np.arange(len(cand))
        assert np.array_equal(ranks[hidden.indptr[j]:hidden.indptr[j + 1]],
                              pos[hidden.indices[hidden.indptr[j]:hidden.indptr[j + 1]]]), j


def test_fit_with_metrics_and_validation(wide):
    """fit with the default metrics=True and a validation split trains at every card count, including those where no
    persistent softmax-KL kernel counts the categorical accuracy."""
    w = wide
    c = w["c"]
    gen = GEN.DataGenerator(w["mhat"], w["csr"], batch_size=64, noise=0.2, seed=3)
    model = M.CC_Recommender(c, device="cuda", seed=0, precision="fp32" if c % 4 else "tf32")
    hist = T.fit(model, gen, epochs=2, reg=REG, log=lambda *_: None, validation_split=0.25,
                 max_cube_size=w["csr"].max_size)
    assert len(hist) == 2
    for h in hist:
        assert {"output_1_accuracy", "output_2_accuracy", "val_loss", "val_output_1_accuracy",
                "val_output_2_accuracy"} <= set(h)
        for key, v in h.items():
            assert np.isfinite(v), (key, h)
            if key.endswith("accuracy"):
                assert 0.0 <= v <= 1.0, (key, h)
