"""One training step of the regularised DAE on one GPU (and its data-parallel form).

Reference: ``autoencoder.fit(generator)`` -- per step ``DataGenerator.__getitem__``
(``src/ml/generator.py:38-61``) followed by the Keras train step compiled at
``src/ml/train.py:83-88``:

    loss = 1.0 * BCE(y, D1(E(x))) + reg * KLD(M-hat[r], D2(E(I[r])))       Adam(lr=1e-3)

Everything stays in HBM: cubes as CSR, x as index lists, y as bit rows, I[r] as the row
ids r, M-hat as a float32 (C, ld) matrix whose rows r are read in place.

Data parallel (one process per GPU): each rank takes B/G cubes and R/G regulariser rows,
scales its losses by the GLOBAL B*C and R, and one all_reduce(SUM) over the flat gradient
buffer makes every rank apply the same Adam update.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from .. import _lib
from .._lib import call, ptr, stream_ptr
from .model import (CC_Recommender, ENC_NAMES, HIDDEN, SparseBatch, bag_bwd, bag_fwd, colsum, dec_names, gemm)

KERAS_ADAM = dict(lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-7)
# which CC_FIRST_LAYER values select the tensor-core first layer.  "auto" is in: measured on the B200 at B = 4096,
# C = 20 884 (profiles/r02/ab_first_layer.txt): x W1 as a kind::tf32 GEMM 144 us against 225 us for the gather (bf16: 79 us)
FIRST_LAYER_TENSOR_WHEN = ("tensor", "auto")
# widest rows the loss-only softmax-KL kernel takes (cc_softmax_kl_loss: the register kernel's 512 x 11 shape); evaluation
# of wider rows runs the training kernel into scratch
KL_LOSS_MAX_CARDS = 22528


def alias_table(p: np.ndarray, device):
    """Vose alias table of a probability vector (neg_sampler, reference generator.py:30)."""
    p = np.ascontiguousarray(p, dtype=np.float64)
    prob = np.empty(len(p), dtype=np.float32)
    alias = np.empty(len(p), dtype=np.int32)
    call("cc_alias_build_host", ptr(p), len(p), ptr(prob), ptr(alias))
    return torch.from_numpy(prob).to(device), torch.from_numpy(alias).to(device)


def _to_bf16(src, dst):
    """fp32 (rows, cols) view -> bf16 matrix, on the current stream."""
    call("cc_convert_f32_bf16", ptr(src), src.stride(0), ptr(dst), dst.stride(0), src.shape[0], src.shape[1], stream_ptr())


def categorical_hits(z, rows, num_cards, target_rows, target_argmax, row_hit):
    """Keras' categorical_accuracy of the softmax tower for row shapes the persistent softmax-KL kernel does not take
    (num_cards % 4 != 0 or more than 25 600 cards): ``row_hit[i] = 1`` where the first maximal logit of ``z[i, :num_cards]``
    sits in column ``target_argmax[target_rows[i]]``, for i < ``rows``.  The logits' argmax is cc_kl_target_argmax, the
    same first-maximum rule the persistent kernels count with.  Device work only, no host sync; ``z`` must still hold
    the logits (call it before the softmax-KL kernel turns them into dlogits)."""
    am = torch.empty(rows, dtype=torch.int32, device=z.device)
    call("cc_kl_target_argmax", ptr(z), z.stride(0), rows, num_cards, ptr(am), stream_ptr())
    row_hit[:rows].copy_(am == target_argmax[target_rows[:rows].long()])


def full_identity_shard(num_cards: int, rank: int = 0, world: int = 1):
    """Rows of I (cards) that rank ``rank`` of ``world`` regularises in full-I mode: an exact partition of
    ``[0, C)`` (shard sizes differ by at most one; each rank builds its engine with its own shard size)."""
    return (num_cards * rank) // world, (num_cards * (rank + 1)) // world


class DAEEngine:
    def __init__(self, model: CC_Recommender, mhat: torch.Tensor, *, batch: int, reg_rows: int | None = None,
                 reg: float = 0.1, max_cube_size: int = 720, global_batch: int | None = None,
                 global_reg_rows: int | None = None, group=None, adam=None, data_parallel: bool = True,
                 metrics: bool = False):
        self.model = model
        self.store = model.store
        self.dev = model.device
        self.C = model.N
        self.cpad = (self.C + 127) // 128 * 128
        self.B = int(batch)
        self.R = int(reg_rows if reg_rows is not None else batch)
        self.reg = float(reg)
        self.global_B = int(global_batch or self.B)
        self.global_R = int(global_reg_rows or self.R)
        self.group = group
        self.data_parallel = bool(data_parallel)   # False: never exchange, even under torchrun (single-GPU reference runs)
        # Keras metrics=['accuracy'] (reference train.py:87): binary accuracy of the sigmoid tower and categorical
        # accuracy of the softmax tower, counted inside the loss kernels; off by default (bench, parity tests)
        self.want_metrics = bool(metrics)
        self.adam = dict(KERAS_ADAM, **(adam or {}))
        self.mhat = mhat
        assert mhat.dtype == torch.float32 and mhat.shape[0] == self.C and mhat.shape[1] >= self.C
        self.precision = model.precision
        self.max_cube_size = int(max_cube_size)
        self.x_stride = (int(max_cube_size * 1.8) + 8 + 3) // 4 * 4
        self.yw = self.cpad // 32
        self.launches = 0          # kernels launched by the last step (for bench's gpu_launches)
        self.prof = None
        # data parallel (one process per GPU), CC_DP_MODE =
        #   "auto" (default) p2p_overlap for local batches of >= 3072 cubes in the fp32 / tf32 modes, else p2p
        #   "p2p"  Adam fused with the gradient exchange over NVLink peer memory: every rank owns 1/world of
        #          the parameters, reduces that slice of all ranks' gradients with peer loads, updates it and stores
        #          the result into every rank's parameters (cc_adam_step_p2p; symmetric memory)
        #   "p2p_overlap"    the same kernel per gradient bucket (main decoder, reg decoder, encoder) on a side stream,
        #          started as soon as backward has finished the bucket, between two symmetric-memory barriers: the two
        #          decoders' exchange (2/3 of the bytes) runs under the rest of backward
        #   "nccl_overlap"   bucketed asynchronous NCCL all_reduce overlapped with backward (dist.GradBuckets)
        #   "nccl"           one blocking all_reduce of the whole flat gradient buffer after backward
        import os
        from ..dist import GradBuckets
        self.buckets = GradBuckets(self.store.layout, self.store.total)
        self.dp_mode = os.environ.get("CC_DP_MODE", "auto")
        if self.dp_mode == "auto":
            # [B200] weak scaling at 4096 cubes per GPU: p2p_overlap 2.118 vs 2.178 ms at 2 GPUs, 2.226 vs 2.376 ms at 8
            # (92.6% vs 86.8% efficiency); strong scaling at 2048 cubes per GPU (2 GPUs): 1.967 vs 1.794 ms -- with half
            # the backward to hide under, the three bucket exchanges and their six barriers cost more than they save
            # (profiles/r02/overlap_n2_*.json, profiles/r02/n8_*.json).  bf16 mode at 8 GPUs: 2.124 ms overlapped against
            # 1.910 ms plain -- its backward is a third shorter, and the exchange kernels slow the bf16 GEMMs they run beside
            # (profiles/r02/final_n8/bench_weak_bf16_overlap.json): p2p there
            self.dp_mode = "p2p_overlap" if (self.B >= 3072 and self.precision != "bf16") else "p2p"
        if os.environ.get("CC_DP_OVERLAP") is not None:          # older switch: 1 = overlapped buckets, 0 = blocking
            self.dp_mode = "nccl_overlap" if os.environ["CC_DP_OVERLAP"] != "0" else "nccl"
        if self.dp_mode not in ("p2p", "p2p_overlap", "nccl_overlap", "nccl"):
            raise ValueError(f"CC_DP_MODE={self.dp_mode!r}: expected auto, p2p, p2p_overlap, nccl_overlap or nccl")
        self.overlap = self.dp_mode == "nccl_overlap"
        self.p2p_buckets = self.dp_mode == "p2p_overlap"
        if self.p2p_buckets:
            self.dp_mode = "p2p"                 # same memory layout and kernel; only the schedule and the slicing differ
        self._xchg = None
        self._dp_ready = False
        self._fixed_reg_rows = False
        self._dynamic_tiles = None
        # the small layers' weight-gradient GEMMs ([x | 1]^T dY, a few microseconds each, <= 64 CTAs) run on a side
        # stream, off the dY -> dX -> dY chain that backward is serialised on (CC_SIDE_STREAM=0 keeps one stream)
        self.use_side = os.environ.get("CC_SIDE_STREAM", "1") != "0" and self.dp_mode != "nccl_overlap"
        # the three small layers either side of the bottleneck (and their input gradients) as ONE launch each, the
        # intermediate activations kept in tensor memory (cc_chain_tc): 5 launches instead of 15 on the step's critical
        # path.  Bit-identical to the separate GEMMs; CC_SMALL_CHAIN=0 restores them (A/B measurements)
        self.small_chain = self.precision != "fp32" and os.environ.get("CC_SMALL_CHAIN", "1") != "0"
        # first layer of the main rows: "gather" = warp-per-cube embedding bag over W1 (exact fp32 sums), "tensor" = dense
        # 0/1 rows x W1 on the tensor cores (tensor-core precision modes only).  CC_FIRST_LAYER overrides; see DESIGN.md
        fl = os.environ.get("CC_FIRST_LAYER", "auto")
        if fl not in ("auto", "gather", "tensor"):
            raise ValueError(f"CC_FIRST_LAYER={fl!r}: expected auto, gather or tensor")
        self.first_layer_tc = model.precision != "fp32" and fl in FIRST_LAYER_TENSOR_WHEN
        self._side = None
        self._side_events = []
        self._noise_stream = None
        self._prefetch_ready = None
        self.noise_step = self.store.step.clone()      # batches drawn so far (see _launch_noise)
        self._alloc()

    # -- buffers --------------------------------------------------------------------
    def _alloc(self):
        d, f32 = self.dev, torch.float32
        B, R, T = self.B, self.R, self.B + self.R
        e = lambda *s: torch.empty(s, dtype=f32, device=d)
        self.x_idx = torch.zeros((B, self.x_stride), dtype=torch.int32, device=d)
        self.x_len = torch.zeros(B, dtype=torch.int32, device=d)
        self.x_start = torch.arange(B, dtype=torch.int64, device=d) * self.x_stride
        self.y_bits = torch.zeros((B, self.yw), dtype=torch.int32, device=d)
        self.reg_rows = torch.zeros(max(R, 1), dtype=torch.int32, device=d)
        self.reg_start = torch.arange(max(R, 1), dtype=torch.int64, device=d)
        self.reg_len = torch.ones(max(R, 1), dtype=torch.int32, device=d)
        self.overflow = torch.zeros(1, dtype=torch.int32, device=d)
        self.flips = torch.zeros(B, dtype=torch.int32, device=d)
        # activations (encoder runs main rows then reg rows in one matrix).  Every activation buffer carries a
        # column of ones right after its last feature (row stride = width + 4): the weight-gradient GEMM then runs
        # on [x | 1]^T dY, whose extra last row IS the bias gradient -- no separate column-sum kernels.
        def act(rows, w):
            buf = torch.zeros((rows, w + 4), dtype=f32, device=d)
            buf[:, w] = 1.0
            return buf
        self.a_buf = [act(T, w) for w in HIDDEN]                    # a1..a4 with their ones column
        self.md_buf = [act(B, w) for w in (128, 256, 512)]
        self.rd_buf = [act(max(R, 1), w) for w in (128, 256, 512)]
        self.a = [b_[:, :w] for b_, w in zip(self.a_buf, HIDDEN)]
        self.md = [b_[:, :w] for b_, w in zip(self.md_buf, (128, 256, 512))]
        self.rd = [b_[:, :w] for b_, w in zip(self.rd_buf, (128, 256, 512))]
        # the same activations widened by their column of ones: A operands of the [x | 1]^T dY gradient GEMMs
        self.a_1 = [b_[:, :w + 1] for b_, w in zip(self.a_buf, HIDDEN)]
        self.md_1 = [b_[:, :w + 1] for b_, w in zip(self.md_buf, (128, 256, 512))]
        self.rd_1 = [b_[:, :w + 1] for b_, w in zip(self.rd_buf, (128, 256, 512))]
        self.z1 = e(B if self.precision != "bf16" else 1, self.cpad)   # logits -> dlogits in place (bf16 mode: dz1_16)
        self.z2 = e(max(R, 1), self.cpad)
        # ReLU masks of the activations the small-layer chains produce, one bit per element (cc_chain_tc bits_out /
        # mask_bits): backward reads 4 bytes per row and 32 columns instead of 128
        bits = lambda rows, w: torch.zeros((rows, w // 32), dtype=torch.int32, device=d)
        self.a_bits = [None] + [bits(T, w) for w in HIDDEN[1:]]                 # a2..a4 (a1 comes from the first layer)
        self.md_bits = [bits(B, w) for w in (128, 256, 512)]
        self.rd_bits = [bits(max(R, 1), w) for w in (128, 256, 512)]
        self.ga = [e(T, w) for w in HIDDEN]
        self.gmd = [e(B, w) for w in (128, 256, 512)]
        self.grd = [e(max(R, 1), w) for w in (128, 256, 512)]
        self.row_bce = torch.zeros(B, dtype=torch.float64, device=d)
        self.row_kl = torch.zeros(max(R, 1), dtype=torch.float64, device=d)
        self.loss3 = torch.zeros(3, dtype=torch.float64, device=d)
        self.metrics2 = torch.zeros(2, dtype=torch.float64, device=d)     # [output_1_accuracy, output_2_accuracy]
        self.acc_partial = None
        self.row_hit = torch.zeros(max(R, 1), dtype=torch.int32, device=d) if self.want_metrics else None
        self.row_correct = torch.zeros(B, dtype=torch.float64, device=d) if self.want_metrics else None
        self.bce_partial = None
        self.x_dense = None               # dense 0/1 rows of x: operand of the tensor-core dW1 = x^T g1 GEMM
        self.big16 = self.precision == "bf16"     # the seven 512 <-> C passes on bf16 operands (kind::f16)
        if self.big16:
            bf = torch.bfloat16
            zb = lambda *s_: torch.zeros(s_, dtype=bf, device=d)
            self.md2_16, self.rd2_16, self.g1_16 = zb(B, 512), zb(max(R, 1), 512), zb(B, 512)
            self.dz1_16, self.dz2_16 = zb(B, self.cpad), zb(max(R, 1), self.cpad)      # dlogits only ever exist as bf16
            self.w4_16 = {"main": zb(512, self.cpad), "reg": zb(512, self.cpad)}         # bf16 copies of the two 512 x C kernels
            if self.first_layer_tc:
                self.w1_16 = zb(self.C, 512)                                             # and of the C x 512 first-layer kernel
        if self.precision != "fp32":
            self.x_dense = torch.zeros((B, self.cpad), dtype=torch.bfloat16 if self.big16 else f32, device=d)
            if self.C % 4:
                raise ValueError("tensor-core precision modes need num_cards % 4 == 0 (16-byte TMA rows)")
            from . import tensorcore
            self.bce_partial = torch.zeros(tensorcore.bce_partial_count(B, self.cpad), dtype=torch.float64, device=d)
            if self.want_metrics:
                self.acc_partial = torch.zeros_like(self.bce_partial)
        lib = _lib.load()
        ws = max(lib.cc_colsum_workspace_bytes(T, max(self.cpad, max(HIDDEN))), 1024)
        self.cs_ws = torch.empty(ws // 4, dtype=f32, device=d)

    def kl_argmax(self):
        """First maximal column of every row of M-hat (int32 (C,)): the target side of Keras' categorical_accuracy."""
        if getattr(self, "_kl_argmax", None) is None:
            self._kl_argmax = torch.empty(self.C, dtype=torch.int32, device=self.dev)
            call("cc_kl_target_argmax", ptr(self.mhat), self.mhat.stride(0), self.C, self.C, ptr(self._kl_argmax), stream_ptr())
        return self._kl_argmax

    def kl_table(self):
        """sum_c t' log t' of every row of M-hat (float64 (C,)): the model-independent half of the KLD, built on first
        use (one pass over M-hat) and kept with the engine -- the per-step kernel then needs no logarithm per element."""
        if getattr(self, "_kl_table", None) is None:
            self._kl_table = torch.empty(self.C, dtype=torch.float64, device=self.dev)
            call("cc_kl_target_table", ptr(self.mhat), self.mhat.stride(0), self.C, self.C, ptr(self._kl_table), stream_ptr())
        return self._kl_table

    # -- per-kernel CUDA-event timing (bench.py's roofline leg) ------------------------
    def enable_kernel_timing(self, on=True):
        self.prof = {} if on else None

    def _timed(self, name):
        eng = self

        class _Ctx:
            def __enter__(self_c):
                if eng.prof is not None:
                    self_c.a = torch.cuda.Event(enable_timing=True); self_c.b = torch.cuda.Event(enable_timing=True)
                    self_c.a.record()
                return self_c

            def __exit__(self_c, *exc):
                if eng.prof is not None:
                    self_c.b.record()
                    eng.prof.setdefault(name, []).append((self_c.a, self_c.b))
                return False
        return _Ctx()

    def kernel_times_ms(self):
        """{name: (launches, total ms)} of the timed kernels since enable_kernel_timing()."""
        torch.cuda.synchronize()
        return {k: (len(v), sum(a.elapsed_time(b) for a, b in v)) for k, v in (self.prof or {}).items()}

    # -- inputs ---------------------------------------------------------------------
    def set_batch(self, x: SparseBatch, y_bits: torch.Tensor, reg_rows: torch.Tensor):
        """Inject a fixed (x, y, r) batch (parity tests hold the noise output fixed)."""
        assert x.batch == self.B
        self._x = x
        if self.x_dense is not None:
            rows = torch.repeat_interleave(torch.arange(self.B, device=self.dev), x.row_len.long())
            pos = torch.arange(rows.numel(), device=self.dev) - torch.repeat_interleave(
                torch.cumsum(x.row_len.long(), 0) - x.row_len.long(), x.row_len.long())
            cols = x.idx[(torch.repeat_interleave(x.row_start, x.row_len.long()) + pos)].long()
            self.x_dense.zero_()
            self.x_dense[rows, cols] = 1.0
        self.y_bits.zero_()
        self.y_bits[:, :y_bits.shape[1]].copy_(y_bits)
        if self.R:
            self.reg_rows[:self.R].copy_(reg_rows.to(torch.int32))

    def _launch_noise(self, indptr, indices, batch_ids, alias_prob, alias_idx, noise, noise_std, seed):
        """The noise kernel + reg-row draw + counter increment on the CURRENT stream.  The draws are keyed by
        (seed, cube position, batch counter); the counter is the engine's own (``noise_step``, started from the model's
        Adam step, so a resumed run continues the sequence) because a prefetched batch is drawn before the Adam step
        of the batch in flight has advanced the model's counter."""
        st = stream_ptr()
        with self._timed("noise"):
            call("cc_noise_ex", ptr(indptr), ptr(indices), ptr(batch_ids), self.B, self.C, ptr(alias_prob),
                 ptr(alias_idx), float(noise), float(noise_std), int(seed), ptr(self.noise_step), self.max_cube_size,
                 self.x_stride, ptr(self.x_idx), ptr(self.x_len), ptr(self.y_bits), self.yw, ptr(self.flips),
                 ptr(self.overflow), ptr(self.x_dense), self.cpad if self.x_dense is not None else 0,
                 int(self.big16), st)
        if self.R and not self._fixed_reg_rows:
            call("cc_sample_reg_rows", ptr(alias_prob), ptr(alias_idx), self.C, self.R, int(seed) ^ 0x5DEECE66D,
                 ptr(self.noise_step), ptr(self.reg_rows), st)
        call("cc_step_increment", ptr(self.noise_step), st)
        self._x = SparseBatch(self.x_idx, self.x_start, self.x_len)
        self.launches += 3

    def sample_batch(self, indptr, indices, batch_ids, alias_prob, alias_idx, noise=0.2, noise_std=0.1, seed=0):
        """Noise function F + reg-row draw on the device (reference generator.py:38-103), on the current stream."""
        self._join_prefetch()               # (a prefetched batch is simply replaced)
        self._launch_noise(indptr, indices, batch_ids, alias_prob, alias_idx, noise, noise_std, seed)

    # -- batch prefetch: the NEXT batch's noise kernel under this step's gradient exchange / Adam ------------------
    def has_prefetched_batch(self):
        return self._prefetch_ready is not None

    def _join_prefetch(self):
        if self._prefetch_ready is not None:
            torch.cuda.current_stream(self.dev).wait_event(self._prefetch_ready)
            self._prefetch_ready = None

    def _prefetch_batch(self, nb):
        """``nb``: dict(indptr, indices, batch_ids, alias_prob, alias_idx, noise, noise_std, seed[, wait_event, done_event]).
        Called between backward and the optimiser: backward was the last reader of x / y / the dense rows, the
        optimiser touches none of them, so the latency-bound noise kernel (0.09 ms) runs on a side stream under the
        HBM-bound Adam pass instead of in front of the next forward."""
        main = torch.cuda.current_stream(self.dev)
        if self._noise_stream is None:
            self._noise_stream = torch.cuda.Stream(device=self.dev)
            self._noise_fork, self._noise_join = torch.cuda.Event(), torch.cuda.Event()
        self._noise_fork.record(main)
        with torch.cuda.stream(self._noise_stream):
            self._noise_stream.wait_event(self._noise_fork)
            if nb.get("wait_event") is not None:
                self._noise_stream.wait_event(nb["wait_event"])
            self._launch_noise(nb["indptr"], nb["indices"], nb.get("batch_ids"), nb["alias_prob"], nb["alias_idx"],
                               nb.get("noise", 0.2), nb.get("noise_std", 0.1), nb.get("seed", 0))
            if nb.get("done_event") is not None:
                nb["done_event"].record(self._noise_stream)
            self._noise_join.record(self._noise_stream)
        self._prefetch_ready = self._noise_join

    def set_full_identity_rows(self, rank: int = 0, world: int = 1):
        """"Full-I" regulariser (README formula KL(M-hat, D2(E(I))) over ALL rows of I, the reference code samples
        B of them per step, generator.py:47-51): this rank takes the contiguous shard ``[rank*C/world, (rank+1)*C/world)``
        of the rows, every step, instead of drawing rows.  The engine must have been built with ``reg_rows`` equal to
        the shard size (``full_identity_shard``) and ``global_reg_rows = C``."""
        lo, hi = full_identity_shard(self.C, rank, world)
        if hi - lo != self.R:
            raise ValueError(f"engine has {self.R} reg rows, the full-I shard of rank {rank}/{world} has {hi - lo}")
        self.reg_rows[:self.R].copy_(torch.arange(lo, hi, dtype=torch.int32, device=self.dev))
        self._fixed_reg_rows = True

    # -- the step -------------------------------------------------------------------
    def _forward(self, rows=None, reg_rows=None, sums=None, metrics=False):
        """The forward half of the step: layers, fused losses, accuracy counts.  Training (``rows`` None): logits become
        dlogits and the output biases' gradients are written, as ``forward_backward`` needs them.  Evaluation: the first
        ``rows`` cubes of the loaded batch against reg rows ``reg_rows[:rows]``, loss-only kernels (no dlogits, no
        gradient), and [bce_sum, kl_sum, binary_hits, categorical_hits] added into the device float64 vector ``sums``.
        Returns (launches, BCE partials, their count, reg_dbias_fused) for the training path."""
        s, B, R, T = self.store, self.B, self.R, self.B + self.R
        ev = rows is not None
        Bm = rows if ev else B              # main rows and reg rows this pass computes
        Rm = min(rows, R) if ev else R
        rr = reg_rows if ev else self.reg_rows
        big16 = self.big16
        pr = "tf32" if big16 else self.precision     # every layer but the 512 <-> C passes of the "bf16" mode
        tc = pr != "fp32"               # tensor-core modes: operands rounded to tf32 where produced

        to_bf16 = _to_bf16
        x = self._x
        P, G, W = s.p, s.g, s.w         # master params, grads, the copy of the kernels the GEMMs read
        n_launch = 0
        st = stream_ptr()
        # ---------------- forward ----------------
        if big16:                       # bf16 copies of the two 512 x C kernels, from the fp32 masters
            for prefix in ("main", "reg") if R else ("main",):
                to_bf16(P(dec_names(prefix)[3] + "/kernel"), self.w4_16[prefix])
                n_launch += 1
        a1 = self.a[0]
        if self.first_layer_tc:
            # first layer of the main rows on the tensor cores: x W1 over the dense 0/1 rows the noise kernel already
            # writes for the dW1 GEMM (x is exact in tf32 / bf16; W1 from the tf32 shadow, or a bf16 copy).  The gather
            # moves s * 2 KB = 1.1 MB per cube out of L2 and sits on the L2 -> SM cap; this is one more 2*B*512*C pass
            if big16:
                to_bf16(P("encoder_e1/kernel"), self.w1_16)
                n_launch += 1
            with self._timed("fw1_gemm"):
                if big16:
                    gemm(self.x_dense[:Bm, :self.C], self.w1_16, a1[:Bm], bias=P("encoder_e1/bias"), relu=True,
                         precision="bf16", round_out=True)
                else:
                    gemm(self.x_dense[:Bm, :self.C], W("encoder_e1/kernel"), a1[:Bm], bias=P("encoder_e1/bias"), relu=True,
                         precision=pr, round_out=True)
        else:
            with self._timed("bag_fwd"):
                bag_fwd(P("encoder_e1/kernel"), x.idx, x.row_start[:Bm], x.row_len[:Bm], P("encoder_e1/bias"), a1[:Bm],
                        round_tf32=tc)
        n_launch += 1
        if R:
            bag_fwd(P("encoder_e1/kernel"), rr, self.reg_start[:Rm], self.reg_len[:Rm], P("encoder_e1/bias"), a1[B:B + Rm],
                    round_tf32=tc)
            n_launch += 1
        if self.small_chain:
            from . import tensorcore
            tensorcore.chain(self.a[0], [(W(name + "/kernel"), True, P(name + "/bias"), None, self.a[i + 1], self.a_bits[i + 1])
                                         for i, name in enumerate(ENC_NAMES[1:])], relu=True, round_out=tc)
            n_launch += 1
        else:
            for i, name in enumerate(ENC_NAMES[1:]):
                gemm(self.a[i], W(name + "/kernel"), self.a[i + 1], bias=P(name + "/bias"), relu=True, precision=pr,
                     round_out=tc)
                n_launch += 1

        def dec_small_fwd(names_, h_, acts_, bits_):
            """The decoder's three small layers 64 -> 128 -> 256 -> 512 (one chain launch, or three GEMMs)."""
            if self.small_chain:
                from . import tensorcore
                tensorcore.chain(h_, [(W(names_[i] + "/kernel"), True, P(names_[i] + "/bias"), None, acts_[i], bits_[i])
                                      for i in range(3)], relu=True, round_out=tc)
                return 1
            for i in range(3):
                gemm(h_, W(names_[i] + "/kernel"), acts_[i], bias=P(names_[i] + "/bias"), relu=True, precision=pr,
                     round_out=tc)
                h_ = acts_[i]
            return 3
        rows_of = lambda bufs, n: [b_[:n] for b_ in bufs]
        md, rd = rows_of(self.md, Bm), rows_of(self.rd, Rm)
        md_bits, rd_bits = rows_of(self.md_bits, Bm), rows_of(self.rd_bits, Rm)
        towers = [("main", self.a[3][:Bm], md, self.z1, Bm)]
        if R:
            towers.append(("reg", self.a[3][B:B + Rm], rd, self.z2, Rm))
        bce_rows, bce_n = self.row_bce, B
        main_stream = torch.cuda.current_stream(self.dev)
        if self.use_side and self._side is None:
            self._side = torch.cuda.Stream(device=self.dev)
            self._side_events = [torch.cuda.Event() for _ in range(16)]
        reg_small_on_side = self.use_side and R > 0
        if reg_small_on_side:
            # the reg tower's three small decoder layers run on the side stream, under the main tower's layers and
            # its big fused-BCE GEMM; the main stream picks them up before the reg tower's 512 -> C GEMM
            fork, join = self._side_events[12], self._side_events[13]
            fork.record(main_stream)                       # the shared encoder's output is complete
            with torch.cuda.stream(self._side):
                self._side.wait_event(fork)
                n_launch += dec_small_fwd(dec_names("reg"), self.a[3][B:B + Rm], rd, rd_bits)
                join.record(self._side)
        if ev:
            eb = self._eval_buffers()
            if tc:
                eb["part"].zero_()          # a partial batch covers fewer (tile, warp) slots than the last one
                if metrics:
                    eb["acc"].zero_()
        for prefix, h, acts, z, nrows in towers:
            names = dec_names(prefix)
            if prefix == "reg" and reg_small_on_side:
                main_stream.wait_event(join)
                h = acts[2]
            else:
                n_launch += dec_small_fwd(names, h, acts, md_bits if prefix == "main" else rd_bits)
                h = acts[2]
            if big16:                   # the 512-wide activation as a bf16 operand
                h16 = (self.md2_16 if prefix == "main" else self.rd2_16)[:nrows]
                to_bf16(h, h16)
                n_launch += 1
            if tc and prefix == "main":
                # fused 512 -> C layer + sigmoid-BCE: logits stay in TMEM, only dlogits are written (evaluation: nothing
                # but the loss / accuracy partials)
                from . import tensorcore
                with self._timed("big_gemm"):       # the epilogue also reduces dlogits' columns into the bias gradient
                    if ev:
                        tensorcore.gemm_bce(h16 if big16 else h, self.w4_16["main"][:, :self.C] if big16 else W(names[3] + "/kernel"),
                                            P(names[3] + "/bias"), self.y_bits[:Bm], float(Bm) * float(self.C), None,
                                            eb["part"], precision="bf16" if big16 else pr, lddz=self.cpad,
                                            acc_partial=eb["acc"] if metrics else None)
                    elif big16:
                        tensorcore.gemm_bce(h16, self.w4_16["main"][:, :self.C], P(names[3] + "/bias"), self.y_bits,
                                            float(self.global_B) * float(self.C), self.dz1_16, self.bce_partial,
                                            precision="bf16", dbias=G(names[3] + "/bias"), acc_partial=self.acc_partial)
                    else:
                        tensorcore.gemm_bce(h, W(names[3] + "/kernel"), P(names[3] + "/bias"), self.y_bits,
                                            float(self.global_B) * float(self.C), self.z1, self.bce_partial, precision=pr,
                                            dbias=G(names[3] + "/bias"), acc_partial=self.acc_partial)
                bce_rows, bce_n = self.bce_partial, self.bce_partial.numel()
            else:
                with self._timed("big_gemm"):
                    if big16:
                        gemm(h16, self.w4_16[prefix][:, :self.C], z[:nrows, :self.C], bias=P(names[3] + "/bias"),
                             precision="bf16")
                    else:
                        gemm(h, W(names[3] + "/kernel"), z[:nrows, :self.C], bias=P(names[3] + "/bias"), precision=pr)
            n_launch += 1
        # ---------------- losses (training: logits -> dlogits in place) ----------------
        if not tc:
            if ev:
                if metrics:
                    call("cc_binary_accuracy_rows", ptr(self.z1), self.z1.stride(0), ptr(self.y_bits), self.yw, Bm, self.C,
                         ptr(eb["correct"]), st)
                call("cc_bce_logits_fwd_bwd", ptr(self.z1), self.z1.stride(0), ptr(self.y_bits), self.yw, Bm, self.C,
                     self.cpad, float(Bm) * float(self.C), None, 0, ptr(eb["bce"]), st)
            else:
                if self.want_metrics:       # the exact-fp32 mode keeps its logits in memory: count before they become dlogits
                    call("cc_binary_accuracy_rows", ptr(self.z1), self.z1.stride(0), ptr(self.y_bits), self.yw, B, self.C,
                         ptr(self.row_correct), st)
                    n_launch += 1
                with self._timed("bce"):
                    call("cc_bce_logits_fwd_bwd", ptr(self.z1), self.z1.stride(0), ptr(self.y_bits), self.yw, B, self.C,
                         self.cpad, float(self.global_B) * float(self.C), ptr(self.z1), self.z1.stride(0),
                         ptr(self.row_bce), st)
                n_launch += 1
        reg_dbias_fused = False
        if R:
            # the persistent softmax-KL kernel also reduces dlogits' columns into the reg tower's output bias gradient
            reg_dbias_fused = bool(_lib.load().cc_softmax_kl_fuses_dbias(self.C, self.cpad, self.z2.stride(0),
                                                                         self.mhat.stride(0), self.z2.stride(0)))
            want_hit = metrics if ev else self.want_metrics
            row_kl, row_hit = (eb["kl"], eb["hit"]) if ev else (self.row_kl, self.row_hit)
            with self._timed("softmax_kl"):
                if ev and self.C % 4 == 0 and self.C <= KL_LOSS_MAX_CARDS and self.mhat.stride(0) % 4 == 0:
                    call("cc_softmax_kl_loss", ptr(self.z2), self.z2.stride(0), ptr(self.mhat), self.mhat.stride(0), ptr(rr),
                         Rm, self.C, self.cpad, ptr(self.kl_table()), ptr(self.kl_argmax()) if want_hit else None,
                         ptr(row_kl), ptr(row_hit) if want_hit else None, int(tc), st)
                else:
                    # training; and evaluation of rows wider than the loss-only kernel takes: the training kernel with
                    # its dlogits written over the (scratch) logits and its bias gradient into a scratch vector
                    dbias = eb["dbias"] if ev else G(dec_names("reg")[3] + "/bias")
                    if big16:
                        if not reg_dbias_fused:
                            raise RuntimeError("bf16 mode needs the persistent softmax-KL kernel (num_cards % 4 == 0, C <= 25600)")
                        call("cc_softmax_kl_fwd_bwd_metrics", ptr(self.z2), self.z2.stride(0), ptr(self.mhat), self.mhat.stride(0),
                             ptr(rr), Rm, self.C, self.cpad, self.reg / float(self.global_R), None, 0,
                             ptr(row_kl), 1, ptr(dbias), ptr(self.dz2_16),
                             self.dz2_16.stride(0), ptr(self.kl_table()), ptr(self.kl_argmax()) if want_hit else None,
                             ptr(row_hit) if want_hit else None, st)
                    else:
                        hit_in_kernel = want_hit and reg_dbias_fused
                        if want_hit and not reg_dbias_fused:      # only the persistent kernels count hits
                            categorical_hits(self.z2, Rm, self.C, rr, self.kl_argmax(), row_hit)
                            n_launch += 1
                        call("cc_softmax_kl_fwd_bwd_metrics", ptr(self.z2), self.z2.stride(0), ptr(self.mhat), self.mhat.stride(0),
                             ptr(rr), Rm, self.C, self.cpad, self.reg / float(self.global_R), ptr(self.z2),
                             self.z2.stride(0), ptr(row_kl), int(tc),
                             ptr(dbias) if reg_dbias_fused else None, None, 0,
                             ptr(self.kl_table()) if reg_dbias_fused else None,
                             ptr(self.kl_argmax()) if hit_in_kernel else None,
                             ptr(row_hit) if hit_in_kernel else None, st)
            n_launch += 1
        if ev:
            sums[0] += (eb["part"] if tc else eb["bce"][:Bm]).sum()
            if R:
                sums[1] += eb["kl"][:Rm].sum()
            if metrics:
                sums[2] += (eb["acc"] if tc else eb["correct"][:Bm]).sum()
                if R:
                    sums[3] += eb["hit"][:Rm].sum()
        return n_launch, bce_rows, bce_n, reg_dbias_fused

    def _eval_buffers(self):
        """Scratch of the evaluation pass (allocated on first use): BCE / accuracy partials of the loss-only GEMM,
        per-row sums, and a bias-gradient sink for rows too wide for the loss-only KL kernel."""
        if getattr(self, "_eval_bufs", None) is None:
            d, f64 = self.dev, torch.float64
            n_part = self.bce_partial.numel() if self.bce_partial is not None else 1
            self._eval_bufs = dict(part=torch.zeros(n_part, dtype=f64, device=d), acc=torch.zeros(n_part, dtype=f64, device=d),
                                   bce=torch.zeros(self.B, dtype=f64, device=d), correct=torch.zeros(self.B, dtype=f64, device=d),
                                   kl=torch.zeros(max(self.R, 1), dtype=f64, device=d),
                                   hit=torch.zeros(max(self.R, 1), dtype=torch.int32, device=d),
                                   dbias=torch.zeros(self.C, dtype=torch.float32, device=d))
        return self._eval_bufs

    def sample_eval_batch(self, indptr, indices, batch_ids, alias_prob, alias_idx, noise, noise_std, seed, counter):
        """Noise function F for ``len(batch_ids)`` (<= B) validation cubes, keyed by (seed, cube id, ``*counter``): the
        caller holds the counter constant, so a cube gets the same corruption whenever it is evaluated.  Draws no reg
        rows and advances no counter; overwrites the batch loaded by sample_batch / set_batch."""
        self._check_no_prefetch()
        n = int(batch_ids.numel())
        if not 0 < n <= self.B:
            raise ValueError(f"{n} validation cubes in a batch of an engine built for {self.B}")
        call("cc_noise_ex", ptr(indptr), ptr(indices), ptr(batch_ids), n, self.C, ptr(alias_prob), ptr(alias_idx),
             float(noise), float(noise_std), int(seed), ptr(counter), self.max_cube_size, self.x_stride, ptr(self.x_idx),
             ptr(self.x_len), ptr(self.y_bits), self.yw, ptr(self.flips), ptr(self.overflow), ptr(self.x_dense),
             self.cpad if self.x_dense is not None else 0, int(self.big16), stream_ptr())
        self._x = SparseBatch(self.x_idx, self.x_start, self.x_len)

    def evaluate_batch(self, rows, reg_rows, sums, metrics=True):
        """Loss-only forward of the first ``rows`` cubes of the loaded batch, cube i paired with reg row ``reg_rows[i]``;
        adds [bce_sum, kl_sum, binary_hits, categorical_hits] into ``sums`` (device float64 (4,)), no host sync.  Leaves
        the parameters, gradients, tf32 shadow, Adam slots and both step counters untouched."""
        self._check_no_prefetch()
        rows = int(rows)
        if not 0 < rows <= (min(self.B, self.R) if self.R else self.B):
            raise ValueError(f"evaluate_batch: rows={rows} outside (0, {min(self.B, self.R) if self.R else self.B}]")
        if self.R and reg_rows.numel() < rows:
            raise ValueError("evaluate_batch: fewer reg rows than cubes")
        self._forward(rows, reg_rows, sums, bool(metrics))

    def _check_no_prefetch(self):
        if self._prefetch_ready is not None:
            raise RuntimeError("a batch prefetched by train_step(next_batch=...) is pending: evaluating now would overwrite it")

    def forward_backward(self):
        s, B, R = self.store, self.B, self.R
        big16 = self.big16
        pr = "tf32" if big16 else self.precision
        tc = pr != "fp32"

        to_bf16 = _to_bf16
        x = self._x
        P, G, W = s.p, s.g, s.w
        main_stream = torch.cuda.current_stream(self.dev)
        n_launch, bce_rows, bce_n, reg_dbias_fused = self._forward()
        side_used = [0]

        def on_side(fn):
            """Run ``fn`` (kernel launches that nothing on the backward chain waits for) on the side stream, behind
            everything enqueued so far on the main stream; the streams join before the gradient exchange."""
            if not self.use_side:
                fn()
                return
            ev = self._side_events[side_used[0]]; side_used[0] += 1
            ev.record(main_stream)
            with torch.cuda.stream(self._side):
                self._side.wait_event(ev)
                fn()
        # (a single CTA that sums ~25 000 partials: 15 us that backward does not have to wait for)
        on_side(lambda: call("cc_loss_finalize", ptr(bce_rows), bce_n, float(self.global_B) * float(self.C), ptr(self.row_kl),
                             R, float(self.global_R), self.reg, ptr(self.loss3), stream_ptr()))
        n_launch += 1
        if self.want_metrics:       # this rank's share of the two accuracies (summed over the ranks with the losses)
            hits1 = (self.acc_partial if tc else self.row_correct).sum()
            self.metrics2[0] = hits1 / (float(self.global_B) * float(self.C))
            self.metrics2[1] = (self.row_hit[:R].sum().double() / float(self.global_R)) if R else 0.0
        # ---------------- backward: decoders ----------------
        ga4 = self.ga[3]
        GKB = s.g_kernel_and_bias           # (in + 1, out) view: kernel gradient rows + the bias gradient row

        def small_dw(a_1, gy, out):
            """Weight (+ bias) gradient of a small layer; on the side stream it overlaps the dX chain (gy and the
            activations are complete at this point of the main stream)."""
            on_side(lambda: gemm(a_1, gy, out, transa=True, precision=pr))
        gtowers = [("main", self.a[3][:B], self.a_1[3][:B], self.md, self.md_1, self.gmd, self.z1, ga4[:B])]
        if R:
            gtowers.append(("reg", self.a[3][B:], self.a_1[3][B:], self.rd, self.rd_1, self.grd, self.z2, ga4[B:]))
        for prefix, h_in, h_in_1, acts, acts_1, gacts, dz, g_in in gtowers:
            names = dec_names(prefix)
            if big16:                   # bf16 dlogits, bf16 activation copy, bf16 kernel copy
                dzc = (self.dz1_16 if prefix == "main" else self.dz2_16)[:, :self.C]
                a16 = self.md2_16 if prefix == "main" else self.rd2_16
                with self._timed("big_gemm"):
                    gemm(a16, dzc, G(names[3] + "/kernel"), transa=True, precision="bf16")
                with self._timed("big_gemm"):
                    gemm(dzc, self.w4_16[prefix][:, :self.C], gacts[2], transb=True, mask=acts[2], precision="bf16",
                         round_out=True)
                n_launch += 2
            else:
                dzc = dz[:, :self.C]
                with self._timed("big_gemm"):
                    gemm(acts[2], dzc, G(names[3] + "/kernel"), transa=True, precision=pr)
                n_launch += 1
            # (the fused BCE epilogue / the persistent softmax-KL kernel already produced this bias gradient)
            if not big16 and not ((tc and prefix == "main") or (prefix == "reg" and reg_dbias_fused)):
                with self._timed("colsum_big"):
                    colsum(dzc, G(names[3] + "/bias"), self.cs_ws)
                n_launch += 2
            if not big16:
                with self._timed("big_gemm"):
                    gemm(dzc, W(names[3] + "/kernel"), gacts[2], transb=True, mask=acts[2], precision=pr, round_out=tc)
                n_launch += 1
            if self.small_chain:
                # dX chain 512 -> 256 -> 128 -> 64 in one launch; the three weight-gradient GEMMs around it on the side stream
                from . import tensorcore
                small_dw(acts_1[1], gacts[2], GKB(names[2]))
                abits = self.md_bits if prefix == "main" else self.rd_bits
                hbits = self.a_bits[3][:B] if prefix == "main" else self.a_bits[3][B:]       # (row slices stay contiguous)
                tensorcore.chain(gacts[2], [(W(names[2] + "/kernel"), False, None, abits[1], gacts[1]),
                                            (W(names[1] + "/kernel"), False, None, abits[0], gacts[0]),
                                            (W(names[0] + "/kernel"), False, None, hbits, g_in)], round_out=tc)
                small_dw(acts_1[0], gacts[1], GKB(names[1]))
                small_dw(h_in_1, gacts[0], GKB(names[0]))
                n_launch += 4
            else:
                for i in (2, 1):
                    small_dw(acts_1[i - 1], gacts[i], GKB(names[i]))
                    gemm(gacts[i], W(names[i] + "/kernel"), gacts[i - 1], transb=True, mask=acts[i - 1], precision=pr,
                         round_out=tc)
                    n_launch += 2
                small_dw(h_in_1, gacts[0], GKB(names[0]))
                gemm(gacts[0], W(names[0] + "/kernel"), g_in, transb=True, mask=h_in, precision=pr, round_out=tc)
                n_launch += 2
            self._grads_ready(prefix)
        if not R:
            for n_ in dec_names("reg"):
                G(n_ + "/kernel").zero_(); G(n_ + "/bias").zero_()
            self._grads_ready("reg")
        # ---------------- backward: shared encoder (main + reg rows together) ----------------
        if self.small_chain:
            from . import tensorcore
            small_dw(self.a_1[2], self.ga[3], GKB(ENC_NAMES[3]))
            # (a1, the first layer's output, has no bit mask: its float activations are the mask of the last layer)
            tensorcore.chain(self.ga[3], [(W(ENC_NAMES[i] + "/kernel"), False, None,
                                           self.a_bits[i - 1] if i > 1 else self.a[0], self.ga[i - 1])
                                          for i in (3, 2, 1)], round_out=tc)
            small_dw(self.a_1[1], self.ga[2], GKB(ENC_NAMES[2]))
            small_dw(self.a_1[0], self.ga[1], GKB(ENC_NAMES[1]))
            n_launch += 4
        else:
            for i in (3, 2, 1):
                name = ENC_NAMES[i]
                small_dw(self.a_1[i - 1], self.ga[i], GKB(name))
                gemm(self.ga[i], W(name + "/kernel"), self.ga[i - 1], transb=True, mask=self.a[i - 1], precision=pr,
                     round_out=tc)
                n_launch += 2
        g1 = self.ga[0]
        on_side(lambda: colsum(g1, G("encoder_e1/bias"), self.cs_ws)); n_launch += 2     # beside the dW1 GEMM
        gw1 = G("encoder_e1/kernel")
        if big16:
            to_bf16(g1[:B], self.g1_16)
            with self._timed("dw1_gemm"):
                gemm(self.x_dense[:, :self.C], self.g1_16, gw1, transa=True, precision="bf16")
            n_launch += 1
        elif tc:
            # dW1 = x^T g1 on the tensor cores (x dense 0/1 is exact in tf32); beats 1.1e9 L2 atomics
            with self._timed("dw1_gemm"):
                gemm(self.x_dense[:, :self.C], g1[:B], gw1, transa=True, precision=pr)
        else:
            gw1.zero_()
            with self._timed("bag_bwd"):
                bag_bwd(g1[:B], x.idx, x.row_start, x.row_len, gw1)
        n_launch += 1
        if R:
            bag_bwd(g1[B:], self.reg_rows, self.reg_start, self.reg_len, gw1); n_launch += 1
        if side_used[0]:                                   # every gradient is complete before the exchange / Adam
            done = self._side_events[-1]
            done.record(self._side)
            main_stream.wait_event(done)
        self._grads_ready("enc")
        self.launches += n_launch

    # -- data-parallel exchange ---------------------------------------------------------
    def _distributed(self):
        import torch.distributed as dist
        return (self.data_parallel and dist.is_available() and dist.is_initialized()
                and dist.get_world_size(self.group) > 1)

    def _grads_ready(self, bucket):
        """Backward has finished every gradient of `bucket`: start its all_reduce (NCCL's own stream; it first
        waits for the kernels enqueued so far) while the compute stream carries on with the next bucket."""
        if self.overlap and self._distributed():
            self.buckets.launch(self.store.grads, bucket, self.group)
        if self.p2p_buckets and self._distributed():
            self._xchg_bucket(bucket)

    def _p2p_slice(self, bucket=None, rank=None):
        """[lo, hi) of the flat buffer whose Adam state rank ``rank`` (default: this one) owns -- of the whole buffer in the
        plain p2p mode, of every bucket in the overlapped one."""
        from ..dist import bucket_owner_slice, owner_slice
        s = self.store
        rank = s.dp_rank if rank is None else rank
        if bucket is None:
            return owner_slice(s.total, rank, s.dp_world)
        lo, hi = self.buckets.ranges[bucket]
        return bucket_owner_slice(lo, hi, rank, s.dp_world)

    def _xchg_bucket(self, bucket):
        """p2p_overlap: exchange + Adam of one gradient bucket on the exchange stream, behind everything enqueued so far on
        the compute stream and the weight-gradient side stream.  Barrier 1: every rank has finished this bucket's gradients
        AND its last read of this bucket's parameters (a peer's all-gather stores land in them); barrier 2: every rank's
        slice has landed; then the local tf32 shadow of the bucket."""
        s, a = self.store, self.adam
        main = torch.cuda.current_stream(self.dev)
        if self._xchg is None:
            self._xchg = torch.cuda.Stream(device=self.dev)
            self._xchg_ev = [torch.cuda.Event() for _ in range(8)]
            self._xchg_n = 0
        ev = self._xchg_ev[self._xchg_n % 8]; self._xchg_n += 1
        ev.record(main)
        evs = None
        if self._side is not None:
            evs = self._xchg_ev[self._xchg_n % 8]; self._xchg_n += 1
            evs.record(self._side)
        lo, hi = self._p2p_slice(bucket)
        blo, bhi = self.buckets.ranges[bucket]
        with torch.cuda.stream(self._xchg):
            self._xchg.wait_event(ev)
            if evs is not None:
                self._xchg.wait_event(evs)
            st = stream_ptr()
            s._g_hdl.barrier(channel=0)
            with self._timed("adam"):
                call("cc_adam_step_p2p", ptr(s.peer_grads), ptr(s.peer_params), s.dp_world, s.dp_rank, ptr(s.adam_m),
                     ptr(s.adam_v), lo, hi, ptr(s.step), a["lr"], a["beta1"], a["beta2"], a["eps"],
                     ctypes.c_void_p(s.mc_grads) if self._multicast else None,
                     ctypes.c_void_p(s.mc_params) if self._multicast else None, st)
            s._g_hdl.barrier(channel=0)
            if s.shadow is not None:
                off = blo
                if bucket == "enc" and not (self.first_layer_tc and not self.big16):
                    off = s.layout["encoder_e1/bias"][0]     # the first-layer kernel's shadow is never read then
                call("cc_round_tf32", ptr(s.params[off:bhi]), ptr(s.shadow[off:bhi]), bhi - off, st)
                self.launches += 1
            self.launches += 3
            if bucket == "enc":                              # the last bucket of a step
                call("cc_step_increment", ptr(s.step), st)
                self.launches += 1
                self._xchg_done = self._xchg_ev[self._xchg_n % 8]; self._xchg_n += 1
                self._xchg_done.record(self._xchg)

    def _dp_setup(self):
        """First distributed step: move params/grads to symmetric memory for the p2p mode (collective).  There is no
        silent downgrade: if the peer-memory rendezvous is impossible on this system every rank raises, and the NCCL
        all_reduce path has to be asked for explicitly (CC_DP_MODE=nccl)."""
        import torch.distributed as dist
        self._dp_ready = True
        if not self._distributed() or self.dp_mode != "p2p":
            return
        ok = torch.ones(1, dtype=torch.int32, device=self.dev)
        err = None
        try:
            self.store.make_symmetric(self.group)
        except Exception as e:                      # no peer access / no symmetric-memory support
            err = e
            ok.zero_()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)      # every rank fails together, nobody hangs
        if int(ok.item()) == 0:
            raise RuntimeError("CC_DP_MODE=p2p: symmetric-memory rendezvous failed on at least one rank"
                               + (f" (here: {err!r})" if err is not None else "")
                               + "; set CC_DP_MODE=nccl to use the NCCL all_reduce exchange instead")
        self._sync_flag = torch.zeros(1, dtype=torch.float32, device=self.dev)
        # in-switch reduction / broadcast (multimem.ld_reduce / multimem.st) when the fabric offers multicast
        import os
        want = os.environ.get("CC_P2P_MULTICAST")
        have = self.dp_mode == "p2p" and bool(getattr(self.store, "mc_params", 0)) and bool(getattr(self.store, "mc_grads", 0))
        # measured: 2 GPUs unicast 0.19 ms vs multicast 0.34 ms; 8 GPUs unicast 0.36 ms vs multicast 0.30 ms
        self._multicast = have and (want == "1" or (want is None and self.store.dp_world >= 4))
        # (cross-rank barriers around the fused kernel: the loss all_reduce before, a one-element all_reduce after;
        # symmetric memory's signal-pad barrier was measured no faster: 2.661 vs 2.645 ms per step at 2 GPUs)
        if want == "1" and not have:
            raise RuntimeError("CC_P2P_MULTICAST=1 but the symmetric-memory handles expose no multicast pointer")

    def allreduce_grads(self):
        """NCCL modes: the blocking all_reduce of the whole flat gradient buffer (mode "nccl"), and the loss scalars."""
        import torch.distributed as dist
        if self._distributed():
            if self.dp_mode == "nccl":
                dist.all_reduce(self.store.grads, op=dist.ReduceOp.SUM, group=self.group)
            dist.all_reduce(self.loss3, op=dist.ReduceOp.SUM, group=self.group)
            if self.want_metrics:
                dist.all_reduce(self.metrics2, op=dist.ReduceOp.SUM, group=self.group)

    def _adam_p2p(self):
        """Reduce-scatter + Adam + all-gather in one kernel over NVLink peer memory (cc_adam_step_p2p).  The loss
        all_reduce issued just before is the barrier "every rank's gradients are complete"; the one-element
        all_reduce after it is the barrier "every rank's slice has landed in my parameters"."""
        import torch.distributed as dist
        s, a = self.store, self.adam
        st = stream_ptr()
        lo, hi = s.dp_slice
        with self._timed("adam"):
            call("cc_adam_step_p2p", ptr(s.peer_grads), ptr(s.peer_params), s.dp_world, s.dp_rank, ptr(s.adam_m),
                 ptr(s.adam_v), lo, hi, ptr(s.step), a["lr"], a["beta1"], a["beta2"], a["eps"],
                 ctypes.c_void_p(s.mc_grads) if self._multicast else None,
                 ctypes.c_void_p(s.mc_params) if self._multicast else None, st)
        dist.all_reduce(self._sync_flag, op=dist.ReduceOp.SUM, group=self.group)
        if s.shadow is not None:
            # tf32 copy of the parameters for the tensor-core GEMMs.  The first-layer kernel (a third of all
            # parameters) is skipped: it is only ever read by the embedding-bag gather, which takes the master copy.
            off = 0 if (self.first_layer_tc and not self.big16) else s.layout["encoder_e1/bias"][0]
            call("cc_round_tf32", ptr(s.params[off:]), ptr(s.shadow[off:]), s.total - off, st)
            self.launches += 1
        call("cc_step_increment", ptr(s.step), st)
        self.launches += 2

    def gather_adam_state(self):
        """p2p mode: every rank keeps Adam's m and v only for the slice of the parameters it owns (the fused exchange
        kernel updates nothing else).  Before a checkpoint is written the slices are exchanged so that every rank --
        rank 0 writes the file -- holds the complete, current m and v.  Collective; a no-op in every other mode."""
        import torch.distributed as dist
        if not (self._distributed() and self.dp_mode == "p2p" and self._dp_ready):
            return
        s = self.store
        world = dist.get_world_size(self.group)
        for bucket in (self.buckets.ORDER if self.p2p_buckets else (None,)):
            for r in range(world):
                lo, hi = self._p2p_slice(bucket, r)
                src = dist.get_global_rank(self.group, r) if self.group is not None else r
                for buf in (s.adam_m, s.adam_v):
                    if hi > lo:
                        dist.broadcast(buf[lo:hi], src=src, group=self.group)

    def apply_adam(self):
        """TF-style Adam over all parameters, then the step counter advances."""
        self._adam_range(None)
        call("cc_step_increment", ptr(self.store.step), stream_ptr())
        self.launches += 1

    def _adam_range(self, bucket=None):
        """Adam over the whole flat buffer, or over one gradient bucket of it (the step counter is untouched)."""
        s, a = self.store, self.adam
        st = stream_ptr()
        lo, hi = (0, s.total) if bucket is None else self.buckets.ranges[bucket]
        sl = lambda t: t[lo:hi] if t is not None else None
        with self._timed("adam"):
            call("cc_adam_step", ptr(sl(s.params)), ptr(sl(s.grads)), ptr(sl(s.adam_m)), ptr(sl(s.adam_v)), hi - lo,
                 ptr(s.step), a["lr"], a["beta1"], a["beta2"], a["eps"], ptr(sl(s.shadow)), st)
        self.launches += 1

    def train_step(self, next_batch=None):
        """forward + backward + (all_reduce) + Adam on the batch set by set_batch/sample_batch (or prefetched by the
        previous call).  ``next_batch`` (see _prefetch_batch): draw the NEXT step's batch under this step's optimiser.
        Returns the device tensor loss3 = [bce, kl, bce + reg*kl] (no synchronisation)."""
        if self._dynamic_tiles is None:
            # overlapped all_reduces take SMs away from the persistent GEMMs at unpredictable moments: hand tiles
            # out dynamically then (CC_DYNAMIC_TILES=0/1 overrides)
            import os
            want = os.environ.get("CC_DYNAMIC_TILES")
            self._dynamic_tiles = (self.dp_mode == "nccl_overlap" and self._distributed()) if want is None else want == "1"
            if self.precision != "fp32":
                call("cc_gemm_tc_set_dynamic_tiles", int(self._dynamic_tiles))
        if not self._dp_ready:
            self._dp_setup()
        self._join_prefetch()
        self.forward_backward()
        if next_batch is not None:
            self._prefetch_batch(next_batch)
        self.allreduce_grads()
        if self.p2p_buckets and self._distributed():
            torch.cuda.current_stream(self.dev).wait_event(self._xchg_done)    # all three buckets exchanged and applied
        elif self.dp_mode == "p2p" and self._distributed():
            self._adam_p2p()
        elif self.overlap and self._distributed():
            for bucket in self.buckets.ORDER:          # Adam follows the reductions bucket by bucket
                self.buckets.wait(bucket)
                self._adam_range(bucket)
            call("cc_step_increment", ptr(self.store.step), stream_ptr())
            self.launches += 1
        else:
            self.apply_adam()
        return self.loss3

    def check_overflow(self):
        v = int(self.overflow.item())
        if v:
            raise RuntimeError("noise kernel overflow: " + ("cube larger than max_cube_size" if v == 1
                                                            else "x list longer than x_stride"))


class HostBatchStream:
    """Feeds an engine from HOST-resident cubes: every step's batch (CSR rows) is copied from pinned host memory
    into one of two device slots on a copy stream while the previous step computes, and the step's loss is read
    back into pinned memory asynchronously (the host looks at the loss of step i after it has queued step i+1).
    Per step: one H2D copy of the batch's CSR, one D2H copy of the 3 loss scalars, no host-side stall.

        feed = HostBatchStream(engine, batches)      # batches: list of CubeCSR (one per step, reused cyclically)
        for i in range(steps):
            loss = feed.step(i, alias_prob, alias_idx, noise, noise_std, seed)   # loss of step i-1 (None at i = 0)
        last = feed.drain()
    """

    def __init__(self, engine: DAEEngine, batches):
        self.eng = engine
        dev = engine.dev
        self.host = []
        for b in batches:
            assert b.num_cubes == engine.B
            self.host.append((torch.from_numpy(np.ascontiguousarray(b.indptr, dtype=np.int64)).pin_memory(),
                              torch.from_numpy(np.ascontiguousarray(b.indices, dtype=np.int32)).pin_memory()))
        max_nnz = max(max(h[1].numel() for h in self.host), 1)
        self.slots = [(torch.zeros(engine.B + 1, dtype=torch.int64, device=dev),
                       torch.zeros(max_nnz, dtype=torch.int32, device=dev)) for _ in range(2)]
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.copied = [torch.cuda.Event() for _ in range(2)]       # slot filled (copy stream)
        self.consumed = [torch.cuda.Event() for _ in range(2)]     # slot read by the noise kernel (compute stream)
        self.loss_host = [torch.zeros(3, dtype=torch.float64).pin_memory() for _ in range(2)]
        self.ovf_host = [torch.zeros(1, dtype=torch.int32).pin_memory() for _ in range(2)]   # the noise kernel's overflow flag
        self.loss_done = [torch.cuda.Event() for _ in range(2)]
        self.h2d_bytes = int(np.mean([h[0].numel() * 8 + h[1].numel() * 4 for h in self.host]))
        self._next_prefetched = -1
        self._pending = None

    def _prefetch(self, i):
        slot = i % 2
        hp, hi = self.host[i % len(self.host)]
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.consumed[slot])       # the step that last used this slot has read it
            self.slots[slot][0].copy_(hp, non_blocking=True)
            self.slots[slot][1][:hi.numel()].copy_(hi, non_blocking=True)
            self.copied[slot].record(self.copy_stream)
        self._next_prefetched = i

    def step(self, i, alias_prob, alias_idx, noise=0.2, noise_std=0.1, seed=0):
        slot, nslot = i % 2, (i + 1) % 2
        cur = torch.cuda.current_stream()
        if not self.eng.has_prefetched_batch():                    # first step (or after a gap): draw this batch now
            if self._next_prefetched < i:
                self._prefetch(i)
            cur.wait_event(self.copied[slot])
            self.eng.sample_batch(self.slots[slot][0], self.slots[slot][1], None, alias_prob, alias_idx, noise, noise_std,
                                  seed=seed)
            self.consumed[slot].record(cur)
        if self._next_prefetched < i + 1:
            self._prefetch(i + 1)                                  # H2D of the next batch: overlaps this step's compute
        # the next batch's noise kernel runs under this step's optimiser, as soon as its CSR has landed
        nxt = dict(indptr=self.slots[nslot][0], indices=self.slots[nslot][1], batch_ids=None, alias_prob=alias_prob,
                   alias_idx=alias_idx, noise=noise, noise_std=noise_std, seed=seed, wait_event=self.copied[nslot],
                   done_event=self.consumed[nslot])
        l3 = self.eng.train_step(next_batch=nxt)
        self.loss_host[slot].copy_(l3, non_blocking=True)
        self.ovf_host[slot].copy_(self.eng.overflow, non_blocking=True)       # rides along with the loss: no extra sync
        self.loss_done[slot].record(cur)
        prev = self._pending
        self._pending = slot
        if prev is None:
            return None
        self.loss_done[prev].synchronize()                         # finished long ago: step i was queued meanwhile
        self._raise_on_overflow(prev)
        return self.loss_host[prev].clone().numpy()

    def _raise_on_overflow(self, slot):
        v = int(self.ovf_host[slot][0])
        if v:
            raise RuntimeError("noise kernel overflow: " + ("cube larger than max_cube_size" if v == 1
                                                            else "x list longer than x_stride"))

    def drain(self):
        if self._pending is None:
            return None
        self.loss_done[self._pending].synchronize()
        self._raise_on_overflow(self._pending)
        out = self.loss_host[self._pending].clone().numpy()
        self._pending = None
        return out
