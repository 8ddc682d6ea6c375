"""The card-count boundaries that tests/test_gpu_wide_rows.py aims its cases at, pinned on the host: if a boundary moves,
these fail before the GPU cases silently stop reaching the kernel they were written for.  cc_softmax_kl_fuses_dbias
only evaluates a predicate on its arguments, so no GPU is needed."""
import pytest

from cubecobrarecommender_b200 import _lib, build
from cubecobrarecommender_b200.ml import engine as E


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def _cpad(c):
    return (c + 127) // 128 * 128


# (cards, ld of M-hat, persistent kernel with the fused bias gradient?)  ld as the engine sees it: M-hat rows padded to 4
@pytest.mark.parametrize("c,ldt,fused", [(20884, 20884, 1), (22528, 22528, 1), (22532, 22532, 1), (24000, 24000, 1),
                                         (25600, 25600, 1), (25604, 25604, 0), (30000, 30000, 0), (24001, 24004, 0),
                                         (333, 336, 0)])
def test_persistent_softmax_kl_boundaries(lib, c, ldt, fused):
    cpad = _cpad(c)
    assert lib.cc_softmax_kl_fuses_dbias(c, cpad, cpad, ldt, cpad) == fused


def test_persistent_softmax_kl_needs_aligned_strides(lib):
    c = 22532
    assert lib.cc_softmax_kl_fuses_dbias(c, _cpad(c), _cpad(c), c, _cpad(c))
    for ldz, ldt, lddz in ((c + 2, c, c + 4), (c + 4, c + 2, c + 4), (c + 4, c, c + 6)):
        assert not lib.cc_softmax_kl_fuses_dbias(c, c + 4, ldz, ldt, lddz), (ldz, ldt, lddz)


def test_loss_only_kernel_limit_matches_the_engine():
    # the widest rows the register kernel (512 threads x 11 float4 slots) holds; evaluation of wider rows runs the
    # training kernel into scratch
    assert E.KL_LOSS_MAX_CARDS == 4 * 512 * 11 == 22528
