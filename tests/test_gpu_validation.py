"""Held-out validation on the GPU: the loss-only kernels against the training kernels bit for bit, ``evaluate`` against
the float64 oracle and against the training step's loss, its lack of side effects, its reproducibility across batch
sizes and ranks, and ``fit`` / the CLI with validation."""
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
from cubecobrarecommender_b200.ml import engine as E, generator as GEN, model as M, tensorcore as TC, train as T
from cubecobrarecommender_b200.sparse import CubeCSR
from cubecobrarecommender_b200.synth import synth_cubes_csr
from oracle import dae as od

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
call, ptr, stream_ptr = _lib.call, _lib.ptr, _lib.stream_ptr


@pytest.fixture
def pair_mode():
    yield lambda mode: call("cc_gemm_tc_set_pair_mode", mode)
    call("cc_gemm_tc_set_pair_mode", -1)


# ------------------------------------------------------------------ kernels, bit for bit
@pytest.mark.parametrize("precision", ["tf32", "bf16"])
@pytest.mark.parametrize("pair", [0, -1])
@pytest.mark.parametrize("m", [4096, 1000, 293])
@pytest.mark.parametrize("n", [20884, 1000])
def test_loss_only_bce_gemm_equals_dlogit_writing_gemm(precision, pair, m, n, pair_mode):
    pair_mode(pair)
    k, cpad = 512, (n + 127) // 128 * 128
    g = torch.Generator(device="cuda").manual_seed(m + n)
    dt = torch.bfloat16 if precision == "bf16" else torch.float32
    a = torch.randn(m, k, device="cuda", generator=g).to(dt)
    w_pad = (torch.randn(k, cpad, device="cuda", generator=g) * 0.05).to(dt)   # rows padded to 16 bytes, as the engine keeps them
    if precision == "tf32":
        call("cc_round_tf32", ptr(a), ptr(a), a.numel(), stream_ptr())
        call("cc_round_tf32", ptr(w_pad), ptr(w_pad), w_pad.numel(), stream_ptr())
    w = w_pad[:, :n]
    bias = torch.randn(n, device="cuda", generator=g) * 0.5
    yb = torch.randint(-2 ** 31, 2 ** 31 - 1, (m, cpad // 32), dtype=torch.int32, device="cuda", generator=g)
    count = TC.bce_partial_count(m, cpad)
    dz = torch.zeros(m, cpad, dtype=dt, device="cuda")
    out = {}
    for name, dz_, dbias in (("train", dz, torch.zeros(n, device="cuda")), ("eval", None, None)):
        for acc in (False, True):
            part = torch.full((count,), -1.0, dtype=torch.float64, device="cuda")
            accp = torch.full((count,), -1.0, dtype=torch.float64, device="cuda") if acc else None
            TC.gemm_bce(a, w, bias, yb, float(m * n), dz_, part, precision=precision, dbias=dbias, acc_partial=accp,
                        lddz=cpad)
            out[name, acc] = (part, accp)
    torch.cuda.synchronize()
    for acc in (False, True):
        assert torch.equal(out["train", acc][0], out["eval", acc][0])
        if acc:
            assert torch.equal(out["train", acc][1], out["eval", acc][1])
    assert (out["eval", True][0] != -1.0).any()


def _kl_problem(c, rows, seed=3):
    g = torch.Generator(device="cuda").manual_seed(seed)
    cpad = (c + 127) // 128 * 128
    z = torch.zeros(rows, cpad, device="cuda")
    z[:, :c] = torch.randn(rows, c, device="cuda", generator=g) * 3
    t = torch.rand(c, c, device="cuda", generator=g) ** 8
    t /= t.sum(1, keepdim=True)
    trow = torch.randint(0, c, (rows,), dtype=torch.int32, device="cuda", generator=g)
    tlogt = torch.zeros(c, dtype=torch.float64, device="cuda")
    argmax = torch.zeros(c, dtype=torch.int32, device="cuda")
    call("cc_kl_target_table", ptr(t), t.stride(0), c, c, ptr(tlogt), stream_ptr())
    call("cc_kl_target_argmax", ptr(t), t.stride(0), c, c, ptr(argmax), stream_ptr())
    return z, cpad, t, trow, tlogt, argmax


@pytest.mark.parametrize("fast", [1, 0])
@pytest.mark.parametrize("c", [20884, 22000])          # 768 x 7 and 512 x 11 launch shapes
def test_loss_only_softmax_kl_equals_training_kernel(c, fast):
    rows = 300
    z, cpad, t, trow, tlogt, argmax = _kl_problem(c, rows)
    z0 = z.clone()
    loss_t = torch.zeros(rows, dtype=torch.float64, device="cuda"); hit_t = torch.zeros(rows, dtype=torch.int32, device="cuda")
    loss_e = torch.full((rows,), -1.0, dtype=torch.float64, device="cuda"); hit_e = torch.full((rows,), -1, dtype=torch.int32, device="cuda")
    dz = torch.empty_like(z); dbias = torch.zeros(c, device="cuda")
    call("cc_softmax_kl_fwd_bwd_metrics", ptr(z), z.stride(0), ptr(t), t.stride(0), ptr(trow), rows, c, cpad, 1e-3,
         ptr(dz), dz.stride(0), ptr(loss_t), fast, ptr(dbias), None, 0, ptr(tlogt), ptr(argmax), ptr(hit_t), stream_ptr())
    call("cc_softmax_kl_loss", ptr(z), z.stride(0), ptr(t), t.stride(0), ptr(trow), rows, c, cpad, ptr(tlogt), ptr(argmax),
         ptr(loss_e), ptr(hit_e), fast, stream_ptr())
    loss_n = torch.full((rows,), -1.0, dtype=torch.float64, device="cuda")          # without the accuracy pair
    call("cc_softmax_kl_loss", ptr(z), z.stride(0), ptr(t), t.stride(0), ptr(trow), rows, c, cpad, ptr(tlogt), None,
         ptr(loss_n), None, fast, stream_ptr())
    torch.cuda.synchronize()
    assert torch.equal(loss_t, loss_e) and torch.equal(hit_t, hit_e) and torch.equal(loss_t, loss_n)
    assert torch.equal(z, z0)                       # z is only read


# ------------------------------------------------------------------ engine and API
def _generator(c, k, batch, seed=5, size_lo=10, size_hi=60):
    ip, ix = synth_cubes_csr(k, c, size_lo=size_lo, size_hi=size_hi, seed=seed)
    csr = CubeCSR(ip, ix, c)
    gr = G.build_graph(csr, "cuda", want_m64=False)
    return GEN.DataGenerator(gr.mhat, csr, batch_size=batch, noise=0.2, seed=seed), csr


def _params(c, seed=0):
    params = od.init_params(c, seed=seed)
    rng = np.random.default_rng(seed + 1)
    for kname in params:          # non-zero biases, livelier logits
        if kname.endswith("bias"):
            params[kname] = (rng.standard_normal(params[kname].shape) * 0.1).astype(np.float32)
    return params


def _readback(gen, model):
    """The validation x / y / reg rows exactly as evaluate draws them, read back from an engine holding the whole set."""
    k, c = gen.N_cubes, gen.N_cards
    eng = E.DAEEngine(model, gen.mhat_device(), batch=k, reg_rows=k, reg=0.1, max_cube_size=gen.csr.max_size)
    seed, counter, rows = gen.validation_draws()
    eng.sample_eval_batch(gen.indptr, gen.indices_dev, torch.arange(k, dtype=torch.int32, device="cuda"), gen.alias_prob,
                          gen.alias_idx, gen.noise, gen.noise_std, seed, counter)
    eng.check_overflow()
    xl, xi = eng.x_len.cpu().numpy(), eng.x_idx.cpu().numpy()
    bits = eng.y_bits.cpu().numpy().view(np.uint32)
    y = ((bits[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(k, -1)[:, :c].astype(np.float64)
    x = np.zeros((k, c))
    for i in range(k):
        x[i, xi[i, :xl[i]]] = 1
    del eng
    return x, y, rows[:k].cpu().numpy().astype(np.int64)


def _oracle(params, x, y, rows, mhat, chunk=500):
    """Loss part of oracle/dae.py on the read-back set (in row chunks): bce sum, kl sum, binary / categorical hits."""
    p64 = {k_: v.astype(np.float64) for k_, v in params.items()}
    c = x.shape[1]
    out = np.zeros(4); near = np.zeros(2)
    for lo in range(0, x.shape[0], chunk):
        sl = slice(lo, lo + chunk)
        n = len(x[sl])
        z1, z2, _ = od.forward_np(p64, x[sl], rows[sl])
        t = mhat[torch.from_numpy(rows[sl]).to(mhat.device), :c].double().cpu().numpy()
        out[0] += od.bce_from_logits_np(z1, y[sl]) * n * c
        out[1] += od.kld_np(t, od.softmax_np(z2)) * n
        out[2] += od.binary_accuracy_np(z1, y[sl]) * n * c
        out[3] += od.categorical_accuracy_np(z2, t.astype(np.float32)) * n
        near[0] += float(np.sum(np.abs(z1) < 3e-2 * np.abs(z1).max()))
        top2 = np.sort(z2, axis=1)[:, -2:]
        near[1] += float(np.sum((top2[:, 1] - top2[:, 0]) < 3e-2 * np.abs(z2).max()))
    return out, near


TOL = {"fp32": 1e-5, "tf32": 1e-3, "bf16": 2e-3}


def _check_against_oracle(res, params, gen, model, reg):
    x, y, rows = _readback(gen, model)
    ref, near = _oracle(params, x, y, rows, gen.mhat_device())
    k, c = x.shape
    tol = TOL[model.precision]
    bce, kl = ref[0] / (k * c), ref[1] / k
    assert abs(res["output_1_loss"] - bce) / bce < tol, (res, bce)
    assert abs(res["output_2_loss"] - kl) / kl < tol, (res, kl)
    assert abs(res["loss"] - (bce + reg * kl)) / (bce + reg * kl) < tol
    # cells / rows whose logits sit within the mode's rounding of the decision may flip
    assert abs(res["output_1_accuracy"] - ref[2] / (k * c)) <= near[0] / (k * c) + 1e-12
    assert abs(res["output_2_accuracy"] - ref[3] / k) <= near[1] / k + 1e-12


@pytest.mark.parametrize("precision", ["fp32", "tf32", "bf16"])
def test_evaluate_matches_oracle(precision):
    c, batch = 384, 32
    gen, _ = _generator(c, 80, batch)                  # 80 cubes: two full batches and a partial one
    params = _params(c)
    model = M.CC_Recommender(c, device="cuda", precision=precision)
    model.set_weights_dict(params)
    res = T.evaluate(model, gen, 0.1)
    assert set(res) == {"loss", "output_1_loss", "output_2_loss", "output_1_accuracy", "output_2_accuracy"}
    _check_against_oracle(res, params, gen, model, 0.1)


def test_evaluate_matches_oracle_full_width_and_batch_size_does_not_matter():
    """tf32 at C = 20 884 with 4096 + 904 validation cubes: one full and one partial batch of 4096; an engine of batch
    1024 (five batches) gives the same numbers up to summation order."""
    c, k = 20884, 4096 + 904
    gen, _ = _generator(c, k, 4096, seed=2, size_lo=300, size_hi=540)
    params = _params(c, seed=4)
    model = M.CC_Recommender(c, device="cuda", precision="tf32")
    model.set_weights_dict(params)
    res = T.evaluate(model, gen, 0.1)
    gen.batch_size = 1024
    res_1024 = T.evaluate(model, gen, 0.1)
    for key in res:
        assert abs(res[key] - res_1024[key]) <= 1e-6 * abs(res[key]), (key, res[key], res_1024[key])
    _check_against_oracle(res, params, gen, model, 0.1)


def _bits_from_dense(y):
    b, c = y.shape
    w = (c + 127) // 128 * 128 // 32
    out = np.zeros((b, w), dtype=np.uint32)
    rr, cc = np.nonzero(y == 1)
    np.bitwise_or.at(out, (rr, cc // 32), (np.uint32(1) << (cc % 32).astype(np.uint32)))
    return out.view(np.int32)


@pytest.mark.parametrize("precision", ["fp32", "tf32", "bf16"])
def test_evaluate_batch_matches_the_training_loss(precision):
    """Same batch, same weights: the loss-only pass and the training step's loss3 agree to 1e-6 (a forward GEMM's
    stream-K reduce-add order may differ between the two launches, so not bit for bit)."""
    c, b = 384, 64
    gen, csr = _generator(c, b, b, seed=7)
    model = M.CC_Recommender(c, device="cuda", precision=precision)
    model.set_weights_dict(_params(c, seed=2))
    eng = E.DAEEngine(model, gen.mhat_device(), batch=b, reg_rows=b, reg=0.1, max_cube_size=gen.csr.max_size)
    rng = np.random.default_rng(1)
    x = csr.to_dense(); y = x.copy()
    flip = rng.random(x.shape) < 0.02
    x[flip] = 1 - x[flip]
    rows = torch.tensor(rng.integers(0, c, size=b), dtype=torch.int32, device="cuda")
    eng.set_batch(M.SparseBatch.from_csr(CubeCSR.from_dense(x), "cuda"), torch.tensor(_bits_from_dense(y)).cuda(), rows)
    sums = torch.zeros(4, dtype=torch.float64, device="cuda")
    eng.evaluate_batch(b, rows, sums)
    eng.forward_backward()
    loss3 = eng.loss3.cpu().numpy()
    s = sums.cpu().numpy()
    assert abs(s[0] / (b * c) - loss3[0]) <= 1e-6 * loss3[0], (s, loss3)
    assert abs(s[1] / b - loss3[1]) <= 1e-6 * loss3[1], (s, loss3)


@pytest.mark.parametrize("precision", ["fp32", "tf32", "bf16"])
def test_evaluate_has_no_side_effects_and_is_reproducible(precision):
    c, batch = 384, 32
    gen, _ = _generator(c, 150, batch, seed=9)
    train, val = gen.split(0.3)
    model = M.CC_Recommender(c, device="cuda", seed=1, precision=precision)
    eng = E.DAEEngine(model, gen.mhat_device(), batch=batch, reg_rows=batch, reg=0.1,
                      max_cube_size=max(train.csr.max_size, val.csr.max_size))
    for b_ in range(2):                                          # live gradients, Adam slots, counters
        eng.sample_batch(train.indptr, train.indices_dev, train.batch_ids(b_), train.alias_prob, train.alias_idx, seed=3)
        eng.train_step()
    s = model.store
    snap = lambda: [t.clone() for t in (s.params, s.grads, s.adam_m, s.adam_v, s.step, eng.noise_step)
                    + ((s.shadow,) if s.shadow is not None else ())]
    before = snap()
    r1 = T.evaluate(model, val, 0.1, engine=eng)
    r2 = T.evaluate(model, val, 0.1, engine=eng)
    torch.cuda.synchronize()
    for a, b_ in zip(before, snap()):
        assert torch.equal(a, b_)
    for key in r1:
        assert abs(r1[key] - r2[key]) <= 1e-7 * abs(r1[key]), key
    # a pending prefetched batch is never overwritten
    nb = dict(indptr=train.indptr, indices=train.indices_dev, batch_ids=train.batch_ids(2), alias_prob=train.alias_prob,
              alias_idx=train.alias_idx, seed=3)
    eng.train_step(next_batch=nb)
    with pytest.raises(RuntimeError, match="prefetched"):
        T.evaluate(model, val, 0.1, engine=eng)


def test_fit_with_validation_split():
    c, k, b = 256, 128, 32
    gen, csr = _generator(c, k, b, seed=8)
    quiet = lambda *_: None
    lines = []
    m_val = M.CC_Recommender(c, device="cuda", seed=0, precision="fp32")
    h_val = T.fit(m_val, gen, epochs=4, reg=0.1, log=lines.append, validation_split=0.25, validation_freq=2,
                  max_cube_size=64)
    keys = ["val_loss", "val_output_1_loss", "val_output_2_loss", "val_output_1_accuracy", "val_output_2_accuracy"]
    for e, h in enumerate(h_val):
        assert all((key in h) == (e in (1, 3)) for key in keys), (e, h)
    for h in (h_val[1], h_val[3]):
        assert abs(h["val_loss"] - (h["val_output_1_loss"] + 0.1 * h["val_output_2_loss"])) <= 1e-9
    assert sum("val_loss: " in line for line in lines) == 2
    # the same training as fit on the first 96 cubes without validation
    gen_train = GEN.DataGenerator(gen.mhat_device(), csr.rows(np.arange(96)), batch_size=b, noise=0.2, seed=8)
    m_ref = M.CC_Recommender(c, device="cuda", seed=0, precision="fp32")
    h_ref = T.fit(m_ref, gen_train, epochs=4, reg=0.1, log=quiet, max_cube_size=64)
    assert int(m_val.store.step.item()) == int(m_ref.store.step.item()) == 4 * (96 // b)
    split_train, _ = gen.split(0.25)
    for e in range(4):
        split_train.reset_indices(e); gen_train.reset_indices(e)
        assert np.array_equal(split_train.indices, gen_train.indices)
    # exact-fp32 mode: only float atomics separate the two runs (an accuracy may move by a cell or two)
    for a, r in zip(h_val, h_ref):
        for key in ("loss", "output_1_loss", "output_2_loss"):
            assert abs(a[key] - r[key]) <= 1e-5 * abs(r[key]), key
        for key in ("output_1_accuracy", "output_2_accuracy"):
            assert abs(a[key] - r[key]) <= 1e-3, key
    wa, wb = m_val.get_weights_dict(), m_ref.get_weights_dict()
    assert max(np.abs(wa[n] - wb[n]).max() for n in wa) < 2e-4


def test_cli_prints_val_loss(tmp_path, capsys, monkeypatch):
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
    T.main(["2", "16", "run", "0.1", "0.2", "3", "--validation-split", "0.25"])
    out = capsys.readouterr().out
    epoch_lines = [line for line in out.splitlines() if line.startswith("2/2 - ")]
    assert len(epoch_lines) == 2 and all(" - val_loss: " in line and " - val_output_1_loss: " in line for line in epoch_lines)
    assert os.path.exists(tmp_path / "ml_files/run/cc_recommender.npz")


# ------------------------------------------------------------------ data parallel
def _multi_problem():
    c, k = 512, 300
    gen, _ = _generator(c, k, 64, seed=12)
    return c, gen


def _worker():
    import torch.distributed as dist
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl")
    c, gen = _multi_problem()
    model = M.CC_Recommender(c, device="cuda", precision="tf32")
    model.set_weights_dict(_params(c, seed=6))
    res = T.evaluate(model, gen, 0.1)
    if dist.get_rank() == 0:
        print(json.dumps({"world": dist.get_world_size(), "res": res}))
    dist.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_two_gpu_evaluate_equals_one_gpu():
    c, gen = _multi_problem()
    model = M.CC_Recommender(c, device="cuda", precision="tf32")
    model.set_weights_dict(_params(c, seed=6))
    ref = T.evaluate(model, gen, 0.1)
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    env = dict(os.environ, PYTHONPATH=REPO + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)], cwd=REPO, env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip(), r.stderr[-3000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["world"] == 2
    for key, v in ref.items():
        assert abs(out["res"][key] - v) <= 1e-6 * abs(v), (key, out["res"][key], v)


if __name__ == "__main__":
    _worker()
