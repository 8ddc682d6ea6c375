"""Device-side co-occurrence graph and graph recommender (host logic above the C ABI).

Mirrors, on CSR cubes resident in HBM:
  * ``utils.create_adjacency_matrix``   reference ``src/non_ml/utils.py:75-92``
  * ``y_mtx`` / ``neg_sampler``         reference ``src/ml/train.py:69-71``, ``src/ml/generator.py:30``
  * ``simple_recs`` / ``simple_cuts``   reference ``src/scripts/recommend.py:7-18``, ``cut_cards.py:7-18``

plus the leave-k-out and cut ranks of the graph recommender and of a popularity ranking (the baselines the
autoencoder's ranking metrics are read against, ``train.ranking_baselines``).

Multi-GPU: cubes are sharded across ranks; each rank counts its own shard into a private
int32 ``(C, C)`` and one NCCL ``all_reduce(SUM)`` combines them (exact, order independent).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from ._lib import call, ptr, stream_ptr
from .sparse import CubeCSR


@dataclass
class CoocGraph:
    num_cards: int
    counts: torch.Tensor                 # int32 (C, C)
    m64: torch.Tensor | None = None      # float64 (C, C)   M   (utils.py:85-89)
    mhat: torch.Tensor | None = None     # float32 (C, ld)  M-hat (train.py:69-71)
    rowsum: torch.Tensor | None = None   # float64 (C,)
    neg_sampler: torch.Tensor | None = None   # float64 (C,)  (generator.py:30)


def upload_csr(csr: CubeCSR, device):
    indptr = torch.from_numpy(np.ascontiguousarray(csr.indptr, dtype=np.int64)).to(device)
    indices = torch.from_numpy(np.ascontiguousarray(csr.indices, dtype=np.int32)).to(device)
    return indptr, indices


def count_cooccurrence(indptr: torch.Tensor, indices: torch.Tensor, num_cubes: int, num_cards: int,
                       counts: torch.Tensor | None = None, accumulate: bool = False,
                       bits: torch.Tensor | None = None, method: str = "auto",
                       workspace: torch.Tensor | None = None) -> torch.Tensor:
    """int32 counts of the cubes in (indptr, indices), ``cnt = X^T X`` (reference utils.py:82-84).

    method "tensor": byte-expanded X^T contracted with tcgen05.mma kind::i8 (exact int32);
    method "popcount": bit-packed cubes, AND + POPC tiles;
    "auto" takes the tensor-core path whenever the counts buffer meets TMA's 16-byte rules."""
    lib = _lib.load()
    dev = indptr.device
    bad = torch.zeros(1, dtype=torch.int32, device=dev)
    if counts is None:
        ld = (num_cards + 3) // 4 * 4           # TMA rows are multiples of 16 bytes
        counts = torch.zeros((num_cards, ld), dtype=torch.int32, device=dev)[:, :num_cards] if ld != num_cards \
            else torch.empty((num_cards, num_cards), dtype=torch.int32, device=dev)
        accumulate = False
    st = stream_ptr()
    tensor_ok = counts.stride(0) % 4 == 0 and counts.data_ptr() % 16 == 0 and counts.stride(1) == 1
    if method == "auto":
        method = "tensor" if tensor_ok else "popcount"
    if method == "tensor":
        if not tensor_ok:
            raise ValueError("tensor-core count path needs a 16-byte aligned counts buffer with stride % 4 == 0")
        wsb = lib.cc_cooc_tc_workspace_bytes(num_cubes, num_cards)
        if workspace is None or workspace.numel() * workspace.element_size() < wsb:
            workspace = torch.empty(wsb, dtype=torch.uint8, device=dev)
        call("cc_cooc_count_tc", ptr(indptr), ptr(indices), num_cubes, num_cards, ptr(workspace),
             workspace.numel() * workspace.element_size(), ptr(counts), counts.stride(0), int(accumulate), ptr(bad), st)
    elif method == "popcount":
        kw, cpad = lib.cc_bits_words(num_cubes), lib.cc_bits_cpad(num_cards)
        if bits is None:
            bits = torch.empty((max(kw, 1), cpad), dtype=torch.int32, device=dev)
        call("cc_bitpack_cubes", ptr(indptr), ptr(indices), num_cubes, num_cards, ptr(bits), ptr(bad), st)
        call("cc_cooc_count", ptr(bits), num_cubes, num_cards, ptr(counts), counts.stride(0), int(accumulate), st)
    else:
        raise ValueError(f"unknown count method {method!r}")
    if int(bad.item()):
        raise ValueError(f"card index out of range [0, {num_cards})")
    return counts


def normalise(counts: torch.Tensor, *, want_m64=True, want_mhat=True, want_neg=True, force_diag=None,
              mhat_ld: int | None = None, mhat: torch.Tensor | None = None) -> CoocGraph:
    """M (float64), M-hat (float32) and the negative-sampling distribution from int32 counts in one pass.
    ``mhat``: caller-owned float32 (C, >= C) output (at C = 100 000 the 40 GB allocation costs as much as the pass)."""
    c = counts.shape[0]
    dev = counts.device
    m64 = torch.empty((c, c), dtype=torch.float64, device=dev) if want_m64 else None
    if mhat is not None:
        if mhat.dtype != torch.float32 or mhat.shape[0] != c or mhat.shape[1] < c or mhat.stride(1) != 1:
            raise ValueError("mhat must be float32 (C, >= C) with unit column stride")
    elif want_mhat:
        ld = mhat_ld or c
        mhat = torch.zeros((c, ld), dtype=torch.float32, device=dev) if ld != c else \
            torch.empty((c, c), dtype=torch.float32, device=dev)
    rowsum = torch.empty(c, dtype=torch.float64, device=dev)
    st = stream_ptr()
    call("cc_row_normalise", ptr(counts), counts.stride(0), c, ptr(m64), c, ptr(mhat),
         mhat.stride(0) if mhat is not None else 0, ptr(rowsum), int(force_diag is not None),
         float(force_diag or 0.0), st)
    neg = None
    if want_neg:
        ws = torch.empty(_lib.load().cc_col_mass_workspace_bytes(c) // 8, dtype=torch.float64, device=dev)
        neg = torch.empty(c, dtype=torch.float64, device=dev)
        call("cc_col_mass", ptr(counts), counts.stride(0), c, ptr(rowsum), ptr(ws), ptr(neg), st)
    return CoocGraph(c, counts, m64, mhat, rowsum, neg)


def normalise_rows(counts_rows: torch.Tensor, row0: int, num_cards: int, *, want_m64=False, want_mhat=True,
                   mhat: torch.Tensor | None = None, group=None) -> CoocGraph:
    """Row block ``[row0, row0 + nrows)`` of M / M-hat from the matching block of the (summed) int32 counts, plus the
    FULL negative-sampling distribution (the blocks' column masses are all_reduced: C doubles).  The sharded form of
    :func:`normalise` for a build whose counts were reduce-scattered by row block (SURVEY.md 8e)."""
    import torch.distributed as dist
    nrows = counts_rows.shape[0]
    dev = counts_rows.device
    m64 = torch.empty((nrows, num_cards), dtype=torch.float64, device=dev) if want_m64 else None
    if mhat is None and want_mhat:
        mhat = torch.empty((nrows, num_cards), dtype=torch.float32, device=dev)
    rowsum = torch.empty(max(nrows, 1), dtype=torch.float64, device=dev)
    st = stream_ptr()
    call("cc_row_normalise_rows", ptr(counts_rows), counts_rows.stride(0), int(row0), nrows, num_cards, ptr(m64),
         num_cards, ptr(mhat), mhat.stride(0) if mhat is not None else 0, ptr(rowsum), 0, 0.0, st)
    ws = torch.empty(_lib.load().cc_col_mass_workspace_bytes(num_cards) // 8, dtype=torch.float64, device=dev)
    neg = torch.empty(num_cards, dtype=torch.float64, device=dev)
    call("cc_col_mass_rows", ptr(counts_rows), counts_rows.stride(0), int(row0), nrows, num_cards, ptr(rowsum), ptr(ws),
         ptr(neg), st)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(neg, op=dist.ReduceOp.SUM, group=group)
    call("cc_col_mass_scale", ptr(neg), num_cards, st)
    return CoocGraph(num_cards, counts_rows, m64, mhat, rowsum[:nrows], neg)


def reduce_scatter_counts(counts: torch.Tensor, rank: int, world: int, group=None):
    """Sum the ranks' private (C, ld) int32 counts and leave rank r with the row block ``[r*blk, min((r+1)*blk, C))``,
    ``blk = ceil(C / world)``, of the sum -- IN PLACE in its own buffer (returned as a view, with the block's first
    row): half the NVLink traffic of an all_reduce and no replicated (C, C) result.  Exact (integer sum).  The
    collective runs on ``world`` equal blocks; rows >= C of the last one are zero padding (``alloc_counts``)."""
    import torch.distributed as dist
    c, ld = counts.shape[0], counts.stride(0)
    if world == 1:
        return counts, 0
    blk = -(-c // world)
    flat = counts._base if counts._base is not None else counts
    flat = flat.view(-1)
    need = blk * world * ld
    if flat.numel() < need:
        raise ValueError(f"reduce_scatter_counts: the counts buffer needs {blk * world} rows of storage (has {flat.numel() // ld}); "
                         f"allocate it with graph.alloc_counts(num_cards, world)")
    # equal blocks of `blk` rows: block r = rows [r*blk, (r+1)*blk) (rows >= C are zero padding)
    out = flat[rank * blk * ld:(rank + 1) * blk * ld]
    dist.reduce_scatter_tensor(out, flat[:need], op=dist.ReduceOp.SUM, group=group)
    r0 = rank * blk
    nrows = max(0, min(blk, c - r0))
    return out.view(blk, ld)[:nrows, :c], r0


def alloc_counts(num_cards: int, world: int, device="cuda") -> torch.Tensor:
    """int32 (C, ld) counts whose storage is padded to ``world`` equal row blocks (see reduce_scatter_counts)."""
    ld = (num_cards + 3) // 4 * 4
    blk = -(-num_cards // world)
    buf = torch.zeros((blk * world, ld), dtype=torch.int32, device=device)
    return buf[:num_cards, :num_cards] if ld != num_cards else buf[:num_cards]


def build_graph(csr: CubeCSR, device="cuda", *, allreduce=True, group=None, method="auto", **kw) -> CoocGraph:
    """Counts of this rank's cubes (+ all_reduce when torch.distributed is initialised with
    more than one rank, i.e. the cubes are sharded) and the normalised matrices."""
    import torch.distributed as dist
    indptr, indices = upload_csr(csr, device)
    counts = count_cooccurrence(indptr, indices, csr.num_cubes, csr.num_cards, method=method)
    if allreduce and dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        buf = counts if counts.is_contiguous() else counts._base      # padded rows: reduce the whole buffer
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    return normalise(counts, **kw)


def create_adjacency_matrix_host(csr: CubeCSR, force_diag=None, return_counts=False):
    """Host in / host out through the single C-ABI call a reference binding would make."""
    c = csr.num_cards
    m = np.empty((c, c), dtype=np.float64)
    counts = np.empty((c, c), dtype=np.int32) if return_counts else None
    indptr = np.ascontiguousarray(csr.indptr, dtype=np.int64)
    indices = np.ascontiguousarray(csr.indices, dtype=np.int32)
    call("cc_create_adjacency_matrix_host", ptr(indptr), ptr(indices), csr.num_cubes, c,
         int(force_diag is not None), float(force_diag or 0.0), ptr(m), ptr(counts))
    return (m, counts) if return_counts else m


# --------------------------------------------------------------------------- top-N
def topn_masked(scores: torch.Tensor, mask_ptr: torch.Tensor, mask_idx: torch.Tensor, n: int, *,
                only_listed=False, descending=True, want_vals=True, sigmoid=False, out=None):
    """Rank each row of ``scores`` (float32 or float64, (batch, >=C)); see cc_topn_masked_*.

    ``sigmoid=True`` (float32, n <= 128): ``scores`` are logits, the ranking and the returned values are
    their float32 sigmoid probabilities, computed on the fly (cc_topn_masked_sigmoid_f32).
    ``out=(ids, vals, cnt)``: write into caller-owned (batch, n) / (batch,) tensors instead of allocating."""
    lib = _lib.load()
    batch = scores.shape[0]
    c = int(scores.shape[1])
    dev = scores.device
    is64 = scores.dtype == torch.float64
    if scores.dtype not in (torch.float32, torch.float64):
        raise TypeError("scores must be float32 or float64")
    if out is not None:
        ids, vals, cnt = out
    else:
        ids = torch.empty((batch, n), dtype=torch.int32, device=dev)
        vals = torch.empty((batch, n), dtype=scores.dtype, device=dev) if want_vals else None
        cnt = torch.empty(batch, dtype=torch.int32, device=dev)
    if sigmoid:
        if is64:
            raise TypeError("the fused sigmoid select ranks float32 logits")
        call("cc_topn_masked_sigmoid_f32", ptr(scores), scores.stride(0), c, batch, ptr(mask_ptr), ptr(mask_idx),
             int(only_listed), int(descending), n, ptr(ids), ptr(vals), ptr(cnt), stream_ptr())
        return ids, vals, cnt
    wsb = lib.cc_topn_workspace_bytes(c, batch, n, int(is64))
    ws = torch.empty(max(wsb, 16), dtype=torch.uint8, device=dev)
    call("cc_topn_masked_f64" if is64 else "cc_topn_masked_f32", ptr(scores), scores.stride(0), c, batch,
         ptr(mask_ptr), ptr(mask_idx), int(only_listed), int(descending), n, ptr(ws), wsb, ptr(ids), ptr(vals),
         ptr(cnt), stream_ptr())
    return ids, vals, cnt


def rank_targets(scores: torch.Tensor, mask_ptr: torch.Tensor, mask_idx: torch.Tensor, target_ptr: torch.Tensor,
                 target_idx: torch.Tensor, *, sigmoid=False, out=None) -> torch.Tensor:
    """int32 rank of every target entry (cc_rank_targets_f32 / _f64): the 0-based slot at which the descending
    :func:`topn_masked` select over the cards not listed in the mask row would return it, or -1 for a target that is
    masked or out of range.  ``scores`` float32 or float64 (batch, >= C) with unit column stride, C =
    ``scores.shape[1]``; float64 rows may also have stride 0 (``row.expand(batch, C)``: one row ranked for every cube).
    ``sigmoid=True`` (float32 only): ``scores`` are logits, ranked by their float32 sigmoid.  ``out``: int32, one entry
    per ``target_idx`` entry (default: allocated)."""
    if scores.dtype not in (torch.float32, torch.float64) or scores.dim() != 2 or scores.stride(1) != 1:
        raise TypeError("scores must be a float32 or float64 (batch, C) tensor with unit column stride")
    if out is None:
        out = torch.empty(target_idx.numel(), dtype=torch.int32, device=scores.device)
    if scores.dtype == torch.float64:
        if sigmoid:
            raise TypeError("the fused sigmoid ranks float32 logits")
        call("cc_rank_targets_f64", ptr(scores), scores.stride(0), int(scores.shape[1]), int(scores.shape[0]),
             ptr(mask_ptr), ptr(mask_idx), ptr(target_ptr), ptr(target_idx), ptr(out), stream_ptr())
        return out
    call("cc_rank_targets_f32", ptr(scores), scores.stride(0), int(scores.shape[1]), int(scores.shape[0]),
         ptr(mask_ptr), ptr(mask_idx), ptr(target_ptr), ptr(target_idx), int(sigmoid), ptr(out), stream_ptr())
    return out


def rank_cuts(scores: torch.Tensor, list_ptr: torch.Tensor, list_idx: torch.Tensor, target_ptr: torch.Tensor,
              target_idx: torch.Tensor, *, sigmoid=False, out=None) -> torch.Tensor:
    """int32 cut rank of every target entry (cc_rank_cuts_f32 / _f64): the 0-based slot at which the ascending
    :func:`topn_masked` select over the cards listed in the row (``only_listed=True, descending=False``, the cut list)
    would return it, or -1 for a target that is not listed or out of range.  Scores, strides, ``sigmoid`` and ``out`` as
    in :func:`rank_targets`."""
    if scores.dtype not in (torch.float32, torch.float64) or scores.dim() != 2 or scores.stride(1) != 1:
        raise TypeError("scores must be a float32 or float64 (batch, C) tensor with unit column stride")
    if out is None:
        out = torch.empty(target_idx.numel(), dtype=torch.int32, device=scores.device)
    if scores.dtype == torch.float64:
        if sigmoid:
            raise TypeError("the fused sigmoid ranks float32 logits")
        call("cc_rank_cuts_f64", ptr(scores), scores.stride(0), int(scores.shape[1]), int(scores.shape[0]),
             ptr(list_ptr), ptr(list_idx), ptr(target_ptr), ptr(target_idx), ptr(out), stream_ptr())
        return out
    call("cc_rank_cuts_f32", ptr(scores), scores.stride(0), int(scores.shape[1]), int(scores.shape[0]),
         ptr(list_ptr), ptr(list_idx), ptr(target_ptr), ptr(target_idx), int(sigmoid), ptr(out), stream_ptr())
    return out


def _check_holdout_pair(visible: CubeCSR, hidden: CubeCSR, num_cards: int, names=("visible", "hidden")):
    if hidden.num_cubes != visible.num_cubes or hidden.num_cards != visible.num_cards:
        raise ValueError(f"{names[0]} and {names[1]} must hold the same cubes over the same cards")
    if visible.num_cards != num_cards:
        raise ValueError(f"the cubes span {visible.num_cards} cards, the recommender {num_cards}")


class GraphRecommender:
    """M resident in HBM (float64); batched ``simple_recs`` / ``simple_cuts``.  ``budget_bytes``: device memory one
    chunk of :meth:`target_ranks_device` may take for its leaf partials and score rows."""

    def __init__(self, m64: torch.Tensor, budget_bytes: int = 1 << 30):
        assert m64.dtype == torch.float64 and m64.dim() == 2
        self.m = m64.contiguous()
        self.num_cards = m64.shape[0]
        self.device = self.m.device
        self.budget_bytes = int(budget_bytes)

    def scores(self, csr: CubeCSR, zero_diag=False) -> torch.Tensor:
        lib = _lib.load()
        dev = self.m.device
        batch = csr.num_cubes
        row_ptr_h = np.ascontiguousarray(csr.indptr, dtype=np.int64)
        total_leaves = int(sum(lib.cc_pairwise_leaf_count(int(n)) for n in np.diff(row_ptr_h) if n > 0))
        plan_h = np.zeros((max(total_leaves, 1), 4), dtype=np.int32)
        leaf_ptr_h = np.zeros(batch + 1, dtype=np.int32)
        call("cc_pairwise_plan_host", ptr(row_ptr_h), batch, ptr(plan_h), ptr(leaf_ptr_h))
        rows = torch.from_numpy(np.ascontiguousarray(csr.indices, dtype=np.int32)).to(dev)
        row_ptr = torch.from_numpy(row_ptr_h).to(dev)
        plan = torch.from_numpy(plan_h).to(dev)
        leaf_ptr = torch.from_numpy(leaf_ptr_h).to(dev)
        partial = torch.empty((max(total_leaves, 1), self.num_cards), dtype=torch.float64, device=dev)
        scores = torch.empty((batch, self.num_cards), dtype=torch.float64, device=dev)
        call("cc_score_gather_f64", ptr(self.m), self.m.stride(0), self.num_cards, ptr(rows), ptr(row_ptr), batch,
             ptr(plan), ptr(leaf_ptr), total_leaves, int(zero_diag), ptr(partial), ptr(scores), scores.stride(0),
             stream_ptr())
        return scores, row_ptr, rows

    def recs(self, csr: CubeCSR, n: int):
        """Top-``n`` missing cards per cube, descending score (recommend.py:7-18)."""
        scores, row_ptr, rows = self.scores(csr, zero_diag=False)
        return topn_masked(scores, row_ptr, rows, n, only_listed=False, descending=True)

    def cuts(self, csr: CubeCSR, n: int):
        """``n`` lowest-scored in-cube cards per cube, ascending (cut_cards.py:7-18)."""
        scores, row_ptr, rows = self.scores(csr, zero_diag=True)
        return topn_masked(scores, row_ptr, rows, n, only_listed=True, descending=False)

    def target_ranks_device(self, visible: CubeCSR, hidden: CubeCSR) -> torch.Tensor:
        """Leave-k-out ranks, int32 aligned with ``hidden.indices``, on the device: each hidden card of cube b gets the
        0-based slot at which :meth:`recs` (and so ``simple_recs``) would list it for the cube's ``visible`` cards, or
        -1 if it is also visible.  The cubes are scored in chunks (the float64 sums of :meth:`scores`, NumPy's pairwise
        order) whose leaf partials and score rows fit ``budget_bytes``, then ranked by cc_rank_targets_f64.  Chunk
        i+1's plan is built on the host and its rows are uploaded on a copy stream while chunk i computes; nothing
        synchronises with the host."""
        _check_holdout_pair(visible, hidden, self.num_cards)
        return self._chunked_ranks(visible, hidden, 0, rank_targets)

    def cut_ranks_device(self, corrupted: CubeCSR, intruders: CubeCSR) -> torch.Tensor:
        """Cut ranks, int32 aligned with ``intruders.indices``, on the device: each intruder of cube b gets the 0-based
        slot at which :meth:`cuts` (and so ``simple_cuts``) would list it among the cube's ``corrupted`` cards, or -1
        if it is not one of them.  The chunks of :meth:`target_ranks_device`, scored with M's diagonal zeroed (the
        scores of :meth:`cuts`) and ranked by cc_rank_cuts_f64; nothing synchronises with the host."""
        _check_holdout_pair(corrupted, intruders, self.num_cards, ("corrupted", "intruders"))
        return self._chunked_ranks(corrupted, intruders, 1, rank_cuts)

    def _chunked_ranks(self, inputs: CubeCSR, targets: CubeCSR, zero_diag: int, rank) -> torch.Tensor:
        """``rank(scores, row_ptr, rows, target_ptr, target_idx, out=...)`` of every chunk of cubes, the scores being
        those of :meth:`scores` over the ``inputs`` rows: int32 ranks aligned with ``targets.indices``."""
        lib = _lib.load()
        dev, c, k = self.device, self.num_cards, inputs.num_cubes
        vp = np.ascontiguousarray(inputs.indptr, dtype=np.int64)
        vi = np.ascontiguousarray(inputs.indices, dtype=np.int32)
        hp = np.ascontiguousarray(targets.indptr, dtype=np.int64)
        hi_ = np.ascontiguousarray(targets.indices, dtype=np.int32)
        ranks = torch.empty(max(int(hp[-1]), 1), dtype=torch.int32, device=dev)
        if k == 0:
            return ranks[:0]
        sizes = np.diff(vp)
        uniq, inv = np.unique(sizes, return_inverse=True)
        leaves = np.array([lib.cc_pairwise_leaf_count(int(n)) if n > 0 else 0 for n in uniq], dtype=np.int64)[inv]
        # a cube costs its leaf partials plus its score row; every chunk takes at least one cube
        cum = np.concatenate([[0], np.cumsum((leaves + 1) * c * 8)])
        bounds = [0]
        while bounds[-1] < k:
            lo = bounds[-1]
            bounds.append(max(lo + 1, int(np.searchsorted(cum, cum[lo] + self.budget_bytes, side="right")) - 1))
        spans = list(zip(bounds[:-1], bounds[1:]))
        max_leaves = max(int(leaves[lo:hi].sum()) for lo, hi in spans)
        max_cubes = max(hi - lo for lo, hi in spans)
        partial = torch.empty((max(max_leaves, 1), c), dtype=torch.float64, device=dev)
        scores = torch.empty((max_cubes, c), dtype=torch.float64, device=dev)
        compute = torch.cuda.current_stream(dev)
        copier = self._copy_stream = getattr(self, "_copy_stream", None) or torch.cuda.Stream(device=dev)

        def upload(lo, hi):
            nl = int(leaves[lo:hi].sum())
            row_ptr_h = vp[lo:hi + 1] - vp[lo]
            plan_h = np.zeros((max(nl, 1), 4), dtype=np.int32)
            leaf_ptr_h = np.zeros(hi - lo + 1, dtype=np.int32)
            call("cc_pairwise_plan_host", ptr(row_ptr_h), hi - lo, ptr(plan_h), ptr(leaf_ptr_h))
            arrays = (vi[vp[lo]:vp[hi]], row_ptr_h, plan_h, leaf_ptr_h, hi_[hp[lo]:hp[hi]], hp[lo:hi + 1] - hp[lo])
            with torch.cuda.stream(copier):
                parts = [torch.from_numpy(a if len(a) else np.zeros(1, a.dtype)).to(dev, non_blocking=True)
                         for a in arrays]
                ev = torch.cuda.Event()
                ev.record(copier)
            for t in parts:
                t.record_stream(compute)           # allocated on the copy stream, consumed on the compute stream
            return lo, hi, nl, parts, ev

        nxt = upload(*spans[0])
        for i in range(len(spans)):
            lo, hi, nl, (rows, row_ptr, plan, leaf_ptr, t_idx, t_ptr), ev = nxt
            nxt = upload(*spans[i + 1]) if i + 1 < len(spans) else None       # overlaps this chunk's kernels
            compute.wait_event(ev)
            sc = scores[:hi - lo]
            call("cc_score_gather_f64", ptr(self.m), self.m.stride(0), c, ptr(rows), ptr(row_ptr), hi - lo, ptr(plan),
                 ptr(leaf_ptr), nl, zero_diag, ptr(partial), ptr(sc), sc.stride(0), stream_ptr())
            if hp[hi] > hp[lo]:
                rank(sc, row_ptr, rows, t_ptr, t_idx, out=ranks[int(hp[lo]):int(hp[hi])])
        return ranks[:int(hp[-1])]


class PopularityRecommender:
    """The popularity floor: every cube gets the same ranking, the cards listed by the most training cubes first (ties
    to the larger index, the order of every select), minus the cube's own cards.  ``scores`` is one float64 row, the
    number of cubes of ``csr`` that list each card (rows are sets)."""

    def __init__(self, csr: CubeCSR, device="cuda"):
        counts = np.bincount(np.asarray(csr.indices, dtype=np.int64), minlength=csr.num_cards)
        self.num_cards = csr.num_cards
        self.device = torch.device(device)
        self.scores = torch.from_numpy(counts.astype(np.float64)).to(self.device)

    def target_ranks_device(self, visible: CubeCSR, hidden: CubeCSR) -> torch.Tensor:
        """Leave-k-out ranks, int32 aligned with ``hidden.indices``, on the device: each hidden card's 0-based slot in
        the popularity list without the cube's ``visible`` cards, or -1 if it is also visible.  One cc_rank_targets_f64
        launch over every cube, all reading the one score row (row stride 0)."""
        _check_holdout_pair(visible, hidden, self.num_cards)
        k = visible.num_cubes
        hp = np.ascontiguousarray(hidden.indptr, dtype=np.int64)
        ranks = torch.empty(max(int(hp[-1]), 1), dtype=torch.int32, device=self.device)
        if k == 0 or hp[-1] == 0:
            return ranks[:int(hp[-1])]
        mp, mi = upload_csr(visible, self.device)
        tp, ti = upload_csr(hidden, self.device)
        if mi.numel() == 0:                    # no visible card anywhere: a valid (never read) mask pointer
            mi = mi.new_zeros(1)
        rank_targets(self.scores.expand(k, self.num_cards), mp, mi, tp, ti, out=ranks)
        return ranks

    def cut_ranks_device(self, corrupted: CubeCSR, intruders: CubeCSR) -> torch.Tensor:
        """Cut ranks, int32 aligned with ``intruders.indices``, on the device: each intruder's 0-based slot among the
        cube's ``corrupted`` cards ordered least listed first (ties to the smaller index, the ascending select's
        order), or -1 if it is not one of them.  One cc_rank_cuts_f64 launch over every cube (row stride 0)."""
        _check_holdout_pair(corrupted, intruders, self.num_cards, ("corrupted", "intruders"))
        k = corrupted.num_cubes
        tp_h = np.ascontiguousarray(intruders.indptr, dtype=np.int64)
        ranks = torch.empty(max(int(tp_h[-1]), 1), dtype=torch.int32, device=self.device)
        if k == 0 or tp_h[-1] == 0:
            return ranks[:int(tp_h[-1])]
        cp, ci = upload_csr(corrupted, self.device)
        tp, ti = upload_csr(intruders, self.device)
        if ci.numel() == 0:                    # no listed card anywhere: a valid (never read) list pointer
            ci = ci.new_zeros(1)
        rank_cuts(self.scores.expand(k, self.num_cards), cp, ci, tp, ti, out=ranks)
        return ranks
