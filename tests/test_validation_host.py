"""Held-out validation, host side: the split arithmetic, the per-rank shards, the progress line, the CLI flags and the
argument checks of the two loss-only entry points (rejected before any device work, so no GPU is needed)."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from cubecobrarecommender_b200 import _lib, build
from cubecobrarecommender_b200.ml import generator as GEN, train as T
from cubecobrarecommender_b200.sparse import CubeCSR
from cubecobrarecommender_b200.synth import synth_cubes_csr


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def _gen(k=10, c=64):
    ip, ix = synth_cubes_csr(k, c, size_lo=3, size_hi=12, seed=4)
    csr = CubeCSR(ip, ix, c)
    rng = np.random.default_rng(0)
    adj = rng.random((c, c))
    return GEN.DataGenerator(adj / adj.sum(1)[:, None], csr, batch_size=4, seed=9, device="cpu"), csr


@pytest.mark.parametrize("k,split,k_val", [(10, 0.25, 2), (10, 0.3, 3), (37, 0.1, 4), (4096 + 904, 0.5, 2500)])
def test_split_takes_the_last_cubes_and_shares_device_state(lib, k, split, k_val):
    gen, csr = _gen(k)
    train, val = gen.split(split)
    assert val.N_cubes == k_val == int(round(k * split)) and train.N_cubes == k - k_val
    for part, lo, hi in ((train, 0, k - k_val), (val, k - k_val, k)):
        ref = csr.rows(np.arange(lo, hi))
        assert np.array_equal(part.csr.indptr, ref.indptr) and np.array_equal(part.csr.indices, ref.indices)
        assert np.array_equal(part.indptr.numpy(), ref.indptr) and np.array_equal(part.indices_dev.numpy(), ref.indices)
        # one M-hat, one negative sampler, one alias table for both halves
        assert part.mhat_dev is gen.mhat_dev and part.alias_prob is gen.alias_prob and part.alias_idx is gen.alias_idx
        assert part.neg_sampler is gen.neg_sampler
        assert sorted(part.indices.tolist()) == list(range(hi - lo))
    assert gen.N_cubes == k                      # the source generator is left as it was


@pytest.mark.parametrize("split", [0.0, 1.0, -0.1, 0.01])
def test_split_rejects_an_empty_side(lib, split):
    gen, _ = _gen(10)
    with pytest.raises(ValueError):
        gen.split(split)


def test_validation_shards_partition_the_set():
    for k in (1, 7, 80, 5000):
        for world in (1, 2, 3, 8):
            ranges = [T.shard_range(k, r, world) for r in range(world)]
            assert ranges[0][0] == 0 and ranges[-1][1] == k
            assert all(a[1] == b[0] for a, b in zip(ranges, ranges[1:]))
            sizes = [hi - lo for lo, hi in ranges]
            assert max(sizes) - min(sizes) <= 1


def test_progress_line_keeps_the_keras_format():
    logs = {"loss": 0.5, "output_1_loss": 0.25, "output_2_loss": 2.5, "output_1_accuracy": 0.9, "output_2_accuracy": 0.125}
    # what fit printed before validation existed
    old = "12/12 - 3s - loss: 0.5000 - output_1_loss: 0.2500 - output_2_loss: 2.5000 - output_1_accuracy: 0.9000 - output_2_accuracy: 0.1250"
    assert T.progress_line(12, 3.2, logs) == old
    logs.update({"val_loss": 0.75, "val_output_1_loss": 0.5})
    assert T.progress_line(12, 3.2, logs) == old + " - val_loss: 0.7500 - val_output_1_loss: 0.5000"


def test_cli_parsing():
    o = T.parse_args(["5", "64", "run", "0.1", "0.2"])
    assert (o["epochs"], o["batch_size"], o["name"], o["reg"], o["noise"], o["seed"]) == (5, 64, "run", 0.1, 0.2, 0)
    assert not o["seed_given"] and not o["resume"] and o["save_every"] is None and o["validation_split"] == 0.0
    o = T.parse_args(["5", "64", "run", "0.1", "0.2", "7", "--validation-split", "0.2", "--save-every", "2", "--resume"])
    assert o["seed"] == 7 and o["seed_given"] and o["resume"] and o["save_every"] == 2 and o["validation_split"] == 0.2
    o = T.parse_args(["--validation-split", "0.1", "5", "64", "run", "0.1", "0.2"])
    assert o["validation_split"] == 0.1 and o["epochs"] == 5
    for bad in (["5", "64", "run", "0.1"], ["5", "64", "run", "0.1", "0.2", "--validation-split"],
                ["5", "64", "run", "0.1", "0.2", "--validation-split", "1.5"]):
        with pytest.raises(SystemExit):
            T.parse_args(bad)


def test_loss_only_entry_points_reject_bad_arguments(lib):
    fake = ctypes.c_void_p(256)                  # never dereferenced: every call below fails its argument checks
    # loss-only BCE GEMM (dz = NULL) with a bias-gradient output or bf16 dlogits
    for dbias, dz16 in ((fake, 0), (None, 1)):
        rc = lib.cc_gemm_bce_tc_ex(2, 256, 1000, 512, fake, 512, fake, 1024, fake, fake, 32, 256000.0, None, 1024, fake,
                                   dbias, 0, dz16, None, None)
        assert rc == -1 and "loss only" in _lib.last_error()
    # loss-only softmax-KL outside the register kernel's shapes, and half of the accuracy pair
    for c, hit, argmax in ((22532, None, None), (22530, None, None), (20884, fake, None), (20884, None, fake)):
        cpad = (c + 127) // 128 * 128
        rc = lib.cc_softmax_kl_loss(fake, cpad, fake, c + 4 - c % 4, None, 100, c, cpad, None, argmax, fake, hit, 1, None)
        assert rc == -1 and "cc_softmax_kl_loss" in _lib.last_error()
