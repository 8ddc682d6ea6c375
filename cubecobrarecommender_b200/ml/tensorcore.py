"""tcgen05 tensor-core GEMM wrappers (precision modes "tf32" and "bf16"); see csrc/gemm_tc.cu."""
from __future__ import annotations

import numpy as np
import torch

from .. import _lib
from .._lib import call, ptr, stream_ptr

PRECISION_CODE = {"tf32": 1, "bf16": 2}
_SMS = None


def _sms():
    global _SMS
    if _SMS is None:
        _SMS = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    return _SMS


def gemm(a, b, c, *, transa=False, transb=False, bias=None, relu=False, mask=None, accumulate=False,
         precision="tf32", split_k=0, tile_n=0, round_out=False):
    """split_k = 0 / tile_n = 0: the library picks the tile width (128 | 256) and the K split from a
    wave-quantisation model (csrc/gemm_tc.cu plan_eff).  ``round_out``: round the fp32 output to tf32 (it feeds a
    kind::tf32 GEMM), whatever the operand kind of this GEMM."""
    m, n = c.shape
    k = a.shape[0] if transa else a.shape[1]
    want = torch.float32 if precision == "tf32" else torch.bfloat16
    if a.dtype != want or b.dtype != want:
        raise TypeError(f"precision {precision} needs {want} operands, got {a.dtype} / {b.dtype}")
    call("cc_gemm_tc", PRECISION_CODE[precision], int(transa), int(transb), m, n, k, ptr(a), a.stride(0), ptr(b),
         b.stride(0), ptr(c), c.stride(0), ptr(bias), int(relu), ptr(mask), mask.stride(0) if mask is not None else 0,
         int(accumulate), int(split_k or 0), int(tile_n), int(round_out), stream_ptr())
    return c


def gemm_bce(a, w, bias, ybits, count, dz, loss_partial, precision="tf32", round_out=True, dbias=None, acc_partial=None,
             lddz=None):
    """Fused  z = a @ w + bias -> BCE loss partials + dlogits  (z never stored); ``dbias`` (optional, float [n])
    receives the column sums of dlogits = the gradient of ``bias``; ``acc_partial`` (optional, float64 like
    ``loss_partial``) the counts of correctly rounded cells (Keras binary_accuracy).  ``dz`` None: loss (and accuracy)
    partials only, laid out for a dlogit matrix of row stride ``lddz``."""
    m, k = a.shape
    n = w.shape[1]
    dz16 = dz is not None and dz.dtype == torch.bfloat16        # bf16 dlogits for the bf16 dW / dX GEMMs ("bf16" mode)
    if dz16 and precision != "bf16":
        raise TypeError("bf16 dlogits come with bf16 operands")
    call("cc_gemm_bce_tc_ex", PRECISION_CODE[precision], m, n, k, ptr(a), a.stride(0), ptr(w), w.stride(0), ptr(bias),
         ptr(ybits), ybits.stride(0), float(count), ptr(dz), dz.stride(0) if dz is not None else int(lddz),
         ptr(loss_partial), ptr(dbias),
         int(round_out and precision == "tf32"), int(dz16), ptr(acc_partial), stream_ptr())


def bce_partial_count(m, lddz):
    return _lib.load().cc_gemm_bce_partial_count(m, lddz)


def chain(a, layers, *, relu=True, round_out=True):
    """Up to three consecutive small Dense layers in one launch (cc_chain_tc): ``layers`` = [(w, w_is_kn, bias, mask,
    out[, bits_out]), ...]; layer l computes ``out = epi(in @ (w if w_is_kn else w.T))`` with ``in`` = ``a`` for the first
    layer and the previous ``out`` afterwards.  ``bias`` / ``mask`` may be None; ``mask`` is either a float matrix (keep
    where > 0) or an int32 (m, n / 32) bit matrix as written through ``bits_out`` (one bit per positive output).  The
    host-side pointer arrays are built per call (the C side reads them before it returns)."""
    n = len(layers)
    widths = np.zeros(n + 1, dtype=np.int32)
    widths[0] = a.shape[1]
    addr = lambda t: 0 if t is None else t.data_ptr()
    w_p, b_p, m_p, mb_p, bo_p, o_p = (np.zeros(n, dtype=np.uint64) for _ in range(6))
    ldw, ldm, ldo = (np.zeros(n, dtype=np.int64) for _ in range(3))
    kn = np.zeros(n, dtype=np.int32)
    for l, layer in enumerate(layers):
        w, w_is_kn, bias, mask, out = layer[:5]
        bits_out = layer[5] if len(layer) > 5 else None
        widths[l + 1] = out.shape[1]
        k_in, n_out = int(widths[l]), out.shape[1]
        if (tuple(w.shape) != ((k_in, n_out) if w_is_kn else (n_out, k_in)) or out.shape[0] != a.shape[0]
                or w.dtype != torch.float32 or out.dtype != torch.float32):
            raise ValueError(f"chain layer {l}: shapes {tuple(w.shape)} / {tuple(out.shape)} do not follow {k_in} inputs")
        for bits in (bits_out, mask if (mask is not None and mask.dtype == torch.int32) else None):
            if bits is not None and (bits.dtype != torch.int32 or tuple(bits.shape) != (a.shape[0], n_out // 32)
                                     or not bits.is_contiguous()):
                raise ValueError(f"chain layer {l}: a bit matrix must be contiguous int32 ({a.shape[0]}, {n_out // 32})")
        w_p[l], b_p[l], o_p[l], bo_p[l] = addr(w), addr(bias), addr(out), addr(bits_out)
        if mask is not None and mask.dtype == torch.int32:
            mb_p[l] = addr(mask)
        elif mask is not None:
            m_p[l], ldm[l] = addr(mask), mask.stride(0)
        ldw[l], ldo[l], kn[l] = w.stride(0), out.stride(0), int(bool(w_is_kn))
    np_ptr = lambda x: x.ctypes.data
    call("cc_chain_tc", a.shape[0], n, np_ptr(widths), ptr(a), a.stride(0), np_ptr(w_p), np_ptr(ldw), np_ptr(kn),
         np_ptr(b_p), np_ptr(m_p), np_ptr(ldm), np_ptr(mb_p), np_ptr(bo_p), int(relu), np_ptr(o_p), np_ptr(ldo),
         int(round_out), stream_ptr())
