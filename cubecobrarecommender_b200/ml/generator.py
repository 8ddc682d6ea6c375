"""Drop-in mirror of reference ``src/ml/generator.py`` (``DataGenerator``), backed by the CUDA noise kernel.

Same constructor arguments and attributes (``indices``, ``neg_sampler``, ``N_cubes``, ``N_cards``),
``__len__``, ``__getitem__``, ``on_epoch_end``, ``reset_indices``, ``generate_data``.

* ``__getitem__(b)`` keeps the reference contract -- ``([x, I[r]], [y, M-hat[r]])`` as dense float64
  arrays -- for callers that want Keras-shaped batches; it materialises 4 x (B, C) arrays, so it is the
  compatibility path, not the fast one.
* ``device_batch(b, engine)`` is what the trainer uses: the noise function F and the reg-row draw run on
  the GPU and leave x as index lists, y as bit rows and r as row ids inside ``engine``'s buffers.

The draws come from Philox streams seeded by ``seed`` and the step counter, not from NumPy's global
MT19937 state.  The epoch shuffle (reference generator.py:63-72) runs ON THE DEVICE: a permutation drawn from a
generator seeded by ``(seed, epoch)``, so (a) every data-parallel rank holds the same permutation whether or not a
CLI seed was given, (b) a resumed run continues with the permutation the interrupted one would have used, and (c) a
step's batch ids are a slice of a device tensor -- no host array, no H2D copy per step.  ``indices`` stays available
as the NumPy array the reference exposes (one small D2H per epoch).
"""
from __future__ import annotations

import copy

import numpy as np
import torch

from ..sparse import CubeCSR

# validation noise: its own seed (the generator seed mixed with this salt) and a counter held at this value
VALIDATION_SEED_SALT = 0x7A11DA7E
VALIDATION_COUNTER = 0


class DataGenerator:
    def __init__(self, adj_mtx, cubes, batch_size=64, shuffle=True, to_fit=True, noise=0.2, noise_std=0.1,
                 device="cuda", seed=0):
        from .engine import alias_table
        self.noise_std = noise_std
        self.batch_size = batch_size
        self.shuffle = shuffle
        self.to_fit = to_fit
        self.noise = noise
        self.device = torch.device(device)
        self.seed = int(seed)
        self.y_reg = adj_mtx                       # M-hat: numpy float64 (C, C) or torch float32 on the device
        self.csr = cubes if isinstance(cubes, CubeCSR) else CubeCSR.from_dense(np.asarray(cubes))
        self.N_cubes = self.csr.num_cubes
        self.N_cards = self.csr.num_cards
        self.epoch = 0
        self.reset_indices()
        if isinstance(adj_mtx, torch.Tensor):
            col = adj_mtx[:, :self.N_cards].double().sum(0)
            self.neg_sampler = (col / col.sum()).cpu().numpy()
            self.mhat_dev = adj_mtx
        else:
            adj = np.asarray(adj_mtx)
            self.neg_sampler = adj.sum(0) / adj.sum()                      # generator.py:30
            self.mhat_dev = None
        self.alias_prob, self.alias_idx = alias_table(self.neg_sampler, self.device)
        self.indptr = torch.from_numpy(np.ascontiguousarray(self.csr.indptr)).to(self.device)
        self.indices_dev = torch.from_numpy(np.ascontiguousarray(self.csr.indices)).to(self.device)
        self._step = torch.zeros(1, dtype=torch.int64, device=self.device)
        self._validation = None
        self._holdout = None

    def split(self, validation_split: float):
        """``(train, val)`` generators: Keras' ``validation_split`` -- the validation cubes are the last
        ``round(N_cubes * validation_split)`` cubes in CSR order, taken before any shuffling.  Both share this generator's
        device M-hat, ``neg_sampler`` and alias table; each gets its own (small) device copy of its cubes."""
        if not 0.0 < float(validation_split) < 1.0:
            raise ValueError(f"validation_split must lie in (0, 1), got {validation_split}")
        k_val = int(round(self.N_cubes * float(validation_split)))
        if not 0 < k_val < self.N_cubes:
            raise ValueError(f"validation_split {validation_split} of {self.N_cubes} cubes leaves an empty side")
        self.mhat_device()                  # built once here, shared by both halves
        cut = self.N_cubes - k_val
        return self._subset(0, cut), self._subset(cut, self.N_cubes)

    def _subset(self, lo, hi):
        g = copy.copy(self)
        g.csr = self.csr.rows(np.arange(lo, hi))
        g.N_cubes = g.csr.num_cubes
        g.indptr = torch.from_numpy(np.ascontiguousarray(g.csr.indptr)).to(self.device)
        g.indices_dev = torch.from_numpy(np.ascontiguousarray(g.csr.indices)).to(self.device)
        g._step = torch.zeros(1, dtype=torch.int64, device=self.device)
        g._validation = None
        g._holdout = None
        g.reset_indices()
        return g

    def validation_draws(self):
        """``(seed, counter, reg_rows)`` of this generator used as a validation set.  The noise kernel keys its draws by
        (seed, cube id, counter): validation uses a seed of its own and a counter that never moves, so every cube gets
        the same corruption in every epoch, whatever the batch size or the number of ranks -- epochs are comparable
        (training redraws its noise every step).  ``reg_rows`` (device int32, one per cube) pairs validation cube v with
        M-hat row ``reg_rows[v]``; drawn once."""
        if getattr(self, "_validation", None) is None:
            from .._lib import call, ptr, stream_ptr
            seed = (self.seed * 0x9E3779B97F4A7C15 + VALIDATION_SEED_SALT) % (1 << 64)
            counter = torch.full((1,), VALIDATION_COUNTER, dtype=torch.int64, device=self.device)
            rows = torch.empty(max(self.N_cubes, 1), dtype=torch.int32, device=self.device)
            call("cc_sample_reg_rows", ptr(self.alias_prob), ptr(self.alias_idx), self.N_cards, self.N_cubes,
                 seed ^ 0x5DEECE66D, ptr(counter), ptr(rows), stream_ptr())
            self._validation = (seed, counter, rows)
        return self._validation

    def holdout_split(self, fraction: float):
        """``(visible, hidden, evaluated)`` of ``ranking.holdout_split`` over this generator's cubes, with a seed of its
        own (the generator seed mixed with ``ranking.HOLDOUT_SEED_SALT``): computed once per fraction on the host, so
        every epoch hides the same cards, and no random stream of the generator is drawn from."""
        from .ranking import HOLDOUT_SEED_SALT, holdout_split
        if self._holdout is None:
            self._holdout = {}
        fraction = float(fraction)
        if fraction not in self._holdout:
            seed = (self.seed * 0x9E3779B97F4A7C15 + HOLDOUT_SEED_SALT) % (1 << 64)
            self._holdout[fraction] = holdout_split(self.csr, fraction, seed)
        return self._holdout[fraction]

    def mhat_device(self, ld=None) -> torch.Tensor:
        """float32 M-hat on the device (what Keras would see after its float32 cast)."""
        if self.mhat_dev is None:
            self.mhat_dev = torch.from_numpy(np.asarray(self.y_reg, dtype=np.float32)).to(self.device)
        return self.mhat_dev

    def __len__(self):
        return self.N_cubes // self.batch_size                               # generator.py:36

    def reset_indices(self, epoch: int | None = None):
        """The epoch's cube order (reference generator.py:63-66), drawn on the device from ``(seed, epoch)``."""
        if epoch is not None:
            self.epoch = int(epoch)
        if self.shuffle == True:  # noqa: E712
            if self.device.type == "cuda":
                g = torch.Generator(device=self.device)
                g.manual_seed((self.seed * 1_000_003 + self.epoch * 7919 + 12345) & 0x7FFFFFFFFFFFFFFF)
                self.indices_dev_order = torch.randperm(self.N_cubes, generator=g, device=self.device).to(torch.int32)
            else:   # host-only use of the mirror (no kernels can run there anyway)
                rng = np.random.default_rng([self.seed, self.epoch])
                self.indices_dev_order = torch.from_numpy(rng.permutation(self.N_cubes).astype(np.int32))
        else:
            self.indices_dev_order = torch.arange(self.N_cubes, dtype=torch.int32, device=self.device)
        self.indices = self.indices_dev_order.cpu().numpy().astype(np.int64)

    def on_epoch_end(self):
        self.epoch += 1
        self.reset_indices()

    def batch_ids(self, batch_number, rank: int = 0, world: int = 1) -> torch.Tensor:
        """Device int32 ids of batch ``batch_number`` (of rank ``rank``'s share of it): a view of the epoch's permutation."""
        ids = self.indices_dev_order[batch_number * self.batch_size:(batch_number + 1) * self.batch_size]
        if world > 1:
            per = self.batch_size // world
            ids = ids[rank * per:(rank + 1) * per]
        return ids

    def device_batch(self, batch_number, engine):
        """Noise + reg rows for batch ``batch_number`` straight into ``engine`` (no host round trip)."""
        engine.sample_batch(self.indptr, self.indices_dev, self.batch_ids(batch_number), self.alias_prob,
                            self.alias_idx, self.noise, self.noise_std, seed=self.seed)

    # ---- reference-shaped (dense) batches ------------------------------------------------
    def _run_noise(self, main_indices):
        from .._lib import call, ptr, stream_ptr
        b = len(main_indices)
        c = self.N_cards
        max_size = max(self.csr.max_size, 1)
        x_stride = (int(max_size * 1.8) + 8 + 3) // 4 * 4
        yw = (c + 127) // 128 * 4
        dev = self.device
        ids = torch.from_numpy(np.ascontiguousarray(main_indices, dtype=np.int32)).to(dev)
        x_idx = torch.zeros((b, x_stride), dtype=torch.int32, device=dev)
        x_len = torch.zeros(b, dtype=torch.int32, device=dev)
        yb = torch.zeros((b, yw), dtype=torch.int32, device=dev)
        ovf = torch.zeros(1, dtype=torch.int32, device=dev)
        call("cc_noise", ptr(self.indptr), ptr(self.indices_dev), ptr(ids), b, c, ptr(self.alias_prob),
             ptr(self.alias_idx), float(self.noise), float(self.noise_std), self.seed, ptr(self._step), max_size,
             x_stride, ptr(x_idx), ptr(x_len), ptr(yb), yw, None, ptr(ovf), None, 0, stream_ptr())
        call("cc_step_increment", ptr(self._step), stream_ptr())
        if int(ovf.item()):
            raise RuntimeError("noise kernel overflow")
        xi, xl = x_idx.cpu().numpy(), x_len.cpu().numpy()
        x = np.zeros((b, c))
        for r in range(b):
            x[r, xi[r, :xl[r]]] = 1
        bits = yb.cpu().numpy().view(np.uint32)
        y = ((bits[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(b, -1)[:, :c].astype(np.float64)
        return x, y

    def generate_data(self, main_indices, reg_indices):
        """Reference generator.py:74-103 -> [(x_cubes, x_reg), (y_cubes, y_reg)], dense float64."""
        x, y = self._run_noise(main_indices)
        reg_indices = np.asarray(reg_indices)
        x_reg = np.zeros((len(reg_indices), self.N_cards))
        x_reg[np.arange(len(reg_indices)), reg_indices] = 1
        y_src = self.y_reg.cpu().numpy()[:, :self.N_cards] if isinstance(self.y_reg, torch.Tensor) else np.asarray(self.y_reg)
        return [(x, x_reg), (y, np.asarray(y_src[reg_indices], dtype=np.float64))]

    def __getitem__(self, batch_number):
        from .._lib import call, ptr, stream_ptr
        main_indices = self.indices[batch_number * self.batch_size:(batch_number + 1) * self.batch_size]
        rows = torch.zeros(len(main_indices), dtype=torch.int32, device=self.device)
        call("cc_sample_reg_rows", ptr(self.alias_prob), ptr(self.alias_idx), self.N_cards, len(main_indices),
             self.seed ^ 0x5DEECE66D, ptr(self._step), ptr(rows), stream_ptr())
        X, y = self.generate_data(main_indices, rows.cpu().numpy())
        if self.to_fit:
            return [X[0], X[1]], [y[0], y[1]]
        return [X[0], X[1]]
