"""Batched ML recommendation: D1(E(cube)) -> masked top-N (BASELINE.json configs[3]).

Mirrors the ranking walk of reference ``src/scripts/ml_recommend.py:78-116`` /
``web/ml_recommend_web.py:39-64`` for many cubes at once with the model resident in HBM (the
reference reloads a 390 MB SavedModel per request, web/ml_recommend_web.py:37):

    results   = decoder(encoder(cube))            float32 sigmoid probabilities (C,)
    additions = first `amount` of argsort(results)[::-1] with cube[rec] != 1
    cuts      = results[idx] for every in-cube idx

Ranking is done on the float32 probabilities (not the logits) so that saturated scores tie exactly as
they do in the reference; ties are ordered larger-index-first (``argsort(kind='stable')[::-1]``).
"""
from __future__ import annotations

import numpy as np
import torch

from .._lib import call, ptr, stream_ptr
from ..graph import rank_targets, topn_masked
from ..sparse import CubeCSR
from .model import CC_Recommender, SparseBatch


class MLRecommender:
    def __init__(self, model: CC_Recommender, chunk: int = 8192):
        # cubes per pass through the model.  [B200] 100 000 cubes, top-50: 4.9 M recs/s at 2048 (the host cannot enqueue
        # 49 x 14 launches as fast as the GPU runs them), 6.8 M at 4096, 7.2-7.7 M at 8192 (0.68 GB of logits per pass);
        # profiles/r02/ml_recommend_profile.jsonl
        self.model = model
        self.chunk = int(chunk)

    def probabilities(self, csr: CubeCSR) -> torch.Tensor:
        """(batch, C) float32 sigmoid outputs of ``decoder(encoder(x))``."""
        m = self.model
        sb = SparseBatch.from_csr(csr, m.device)
        z = m._decode(m._encode(sb), "main")
        # sigmoid in place over the whole (padded) buffer the logits view lives in
        full = z._base if z._base is not None else z
        call("cc_sigmoid_f32", ptr(full), ptr(full), full.numel(), stream_ptr())
        return z

    FUSED_MAX_N = 128        # cc_topn_masked_sigmoid_f32's limit (warp-per-cube streaming select)

    def _forward_chunks(self, csr: CubeCSR, *others: CubeCSR):
        """The chunked forward of ``recommend_device`` and ``target_ranks_device``: yields ``(lo, hi, idx, ptr_, z,
        rest)`` per chunk of ``self.chunk`` cubes, where ``idx`` / ``ptr_`` are rows [lo, hi) of ``csr`` on the device,
        ``z`` the (hi - lo, C) logits of ``decoder(encoder(rows))`` and ``rest`` one ``(idx, ptr)`` device pair of rows
        [lo, hi) per CSR in ``others``.  Chunk i+1's rows are uploaded on a copy stream while chunk i computes; nothing
        synchronises with the host."""
        m = self.model
        dev = m.device
        k = csr.num_cubes
        host = [(np.ascontiguousarray(c.indptr, dtype=np.int64), np.ascontiguousarray(c.indices, dtype=np.int32))
                for c in (csr,) + others]
        compute = torch.cuda.current_stream(dev)
        copier = self._copy_stream = getattr(self, "_copy_stream", None) or torch.cuda.Stream(device=dev)

        def upload(lo):
            hi = min(lo + self.chunk, k)
            parts = []
            with torch.cuda.stream(copier):
                for ip, ix in host:
                    rows_h = ix[ip[lo]:ip[hi]]
                    idx = torch.from_numpy(rows_h if len(rows_h) else np.zeros(1, np.int32)).to(dev, non_blocking=True)
                    ptr_ = torch.from_numpy(ip[lo:hi + 1] - ip[lo]).to(dev, non_blocking=True)
                    parts.append((idx, ptr_))
                ev = torch.cuda.Event()
                ev.record(copier)
            for pair in parts:
                for t in pair:
                    t.record_stream(compute)       # allocated on the copy stream, consumed on the compute stream
            return lo, hi, parts, ev

        nxt = upload(0) if k else None
        while nxt is not None:
            lo, hi, parts, ev = nxt
            nxt = upload(hi) if hi < k else None   # overlaps this chunk's kernels
            compute.wait_event(ev)
            idx, ptr_ = parts[0]
            row_len = (ptr_[1:] - ptr_[:-1]).to(torch.int32)
            sb = SparseBatch(idx, ptr_[:-1], row_len)
            z = m._decode(m._encode(sb), "main")
            yield lo, hi, idx, ptr_, z, parts[1:]

    def recommend_device(self, csr: CubeCSR, amount: int, want_cuts: bool = False):
        """The cubes run through encoder, decoder and the masked select in chunks of ``self.chunk`` with NO host
        synchronisation in between; chunk i+1's CSR rows are uploaded on a copy stream while chunk i computes, and
        the results stay on the device: (add_ids int32 (K, n), add_scores float32 (K, n), counts int32 (K,)).
        ``want_cuts``: also return the probability of every in-cube card, float32 (nnz,) aligned with ``csr.indices``
        (the reference's ``cuts`` dict, ml_recommend.py:105-108, for the whole batch) as a fourth element."""
        m = self.model
        dev = m.device
        k = csr.num_cubes
        n = max(1, min(int(amount), csr.num_cards))
        ip = np.ascontiguousarray(csr.indptr, dtype=np.int64)
        ids = torch.empty((k, n), dtype=torch.int32, device=dev)
        vals = torch.empty((k, n), dtype=torch.float32, device=dev)
        cnts = torch.empty(k, dtype=torch.int32, device=dev)
        cuts = torch.empty(max(int(ip[-1]), 1), dtype=torch.float32, device=dev) if want_cuts else None
        fused = n <= self.FUSED_MAX_N
        for lo, hi, idx, ptr_, z, _ in self._forward_chunks(csr):
            out = (ids[lo:hi], vals[lo:hi], cnts[lo:hi])
            if fused:    # sigmoid applied inside the select: the probability rows are never written
                topn_masked(z, ptr_, idx, n, sigmoid=True, out=out)
            else:
                full = z._base if z._base is not None else z
                call("cc_sigmoid_f32", ptr(full), ptr(full), full.numel(), stream_ptr())
                topn_masked(z, ptr_, idx, n, out=out)
            if want_cuts and ip[hi] > ip[lo]:      # z holds logits (fused) or probabilities (sigmoid pass above)
                call("cc_cuts_gather_f32", ptr(z), z.stride(0), m.N, hi - lo, ptr(ptr_), ptr(idx), int(fused),
                     ptr(cuts[int(ip[lo]):int(ip[hi])]), stream_ptr())
        if want_cuts:
            return ids, vals, cnts, cuts[:int(ip[-1])]
        return ids, vals, cnts

    def target_ranks_device(self, visible: CubeCSR, hidden: CubeCSR) -> torch.Tensor:
        """Leave-k-out ranks, int32 aligned with ``hidden.indices``, on the device.  Cube b's ``visible`` cards are the
        model input and the mask; each of its ``hidden`` cards gets the 0-based slot at which ``recommend_device``
        would list it (for any ``amount``), or -1 if it is also visible.  Same chunked pipeline as ``recommend_device``
        with no host synchronisation; the ranks come from cc_rank_targets_f32 on the logits with the sigmoid fused
        in, so no probability row is written."""
        if hidden.num_cubes != visible.num_cubes or hidden.num_cards != visible.num_cards:
            raise ValueError("visible and hidden must hold the same cubes over the same cards")
        if visible.num_cards != self.model.N:
            raise ValueError(f"the cubes span {visible.num_cards} cards, the model {self.model.N}")
        hp = np.ascontiguousarray(hidden.indptr, dtype=np.int64)
        ranks = torch.empty(max(int(hp[-1]), 1), dtype=torch.int32, device=self.model.device)
        for lo, hi, idx, ptr_, z, ((t_idx, t_ptr),) in self._forward_chunks(visible, hidden):
            if hp[hi] > hp[lo]:
                rank_targets(z, ptr_, idx, t_ptr, t_idx, sigmoid=True, out=ranks[int(hp[lo]):int(hp[hi])])
        return ranks[:int(hp[-1])]

    def recommend(self, csr: CubeCSR, amount: int, copy: bool = True, want_cuts: bool = False):
        """Returns (add_ids int32 (K, n), add_scores float32 (K, n), counts int32 (K,)) on the host.  Pass a
        ``csr.pin_memory()`` batch to make the chunk uploads asynchronous.  ``want_cuts``: a fourth array, float32 (nnz,),
        the probability of every in-cube card in ``csr.indices`` order (the reference's ``cuts`` scores)."""
        if want_cuts:
            ids, vals, cnts, cuts = self.recommend_device(csr, amount, want_cuts=True)
            return ids.cpu().numpy(), vals.cpu().numpy(), cnts.cpu().numpy(), cuts.cpu().numpy()
        ids, vals, cnts = self.recommend_device(csr, amount)
        if not copy:
            # results land in page-locked buffers owned by this recommender (asynchronous DMA, no page faults on
            # fresh host memory): the returned arrays are views, valid until the next call
            k, n = ids.shape
            buf = getattr(self, "_host_out", None)
            if buf is None or buf[0].shape[0] < k or buf[0].shape[1] != n:
                buf = self._host_out = (torch.empty((k, n), dtype=torch.int32).pin_memory(),
                                        torch.empty((k, n), dtype=torch.float32).pin_memory(),
                                        torch.empty(k, dtype=torch.int32).pin_memory())
            for dst, src in zip(buf, (ids, vals, cnts)):
                dst[:k].copy_(src, non_blocking=True)
            torch.cuda.current_stream(self.model.device).synchronize()
            return buf[0][:k].numpy(), buf[1][:k].numpy(), buf[2][:k].numpy()
        return ids.cpu().numpy(), vals.cpu().numpy(), cnts.cpu().numpy()

    # -- card similarity (reference src/scripts/similarity.py) -------------------------------------------
    def card_embeddings(self) -> torch.Tensor:
        """``model.encoder(I)``: the 64-d embedding of every card, (C, 64) float32 on the device.  The one-hot rows
        are never built: row r of I is the index list [r] for the embedding-bag first layer."""
        m = self.model
        rows = torch.arange(m.N, dtype=torch.int32, device=m.device)
        return m._encode(SparseBatch.from_rows(rows))

    def similar(self, card_idx: int, n: int, embeddings: torch.Tensor | None = None):
        """The ``n`` cards most similar to ``card_idx``: ``(ids, dists)`` ranked like the reference's
        ``dists.argsort()`` (similarity.py:31), dists = Keras CosineSimilarity loss = -cosine (the card itself
        comes first with -1).  Ties: smaller index first (stable argsort)."""
        m = self.model
        emb = self.card_embeddings() if embeddings is None else embeddings
        dists = torch.empty((1, m.N), dtype=torch.float32, device=m.device)
        call("cc_cosine_neg_f32", ptr(emb), emb.stride(0), m.N, emb.shape[1], int(card_idx), ptr(dists), stream_ptr())
        n = max(1, min(int(n), m.N))
        none_ptr = torch.zeros(2, dtype=torch.int64, device=m.device)          # empty mask: every card is a candidate
        none_idx = torch.zeros(1, dtype=torch.int32, device=m.device)
        ids, vals, cnt = topn_masked(dists, none_ptr, none_idx, n, only_listed=False, descending=False)
        return ids[0].cpu().numpy(), vals[0].cpu().numpy()

    def recommend_one(self, cube_indices, amount, int_to_card):
        """The ``{"additions": {...}, "cuts": {...}}`` dict of reference web/ml_recommend_web.py:48-67."""
        num_cards = self.model.N
        csr = CubeCSR.from_lists([cube_indices], num_cards)
        probs = self.probabilities(csr)
        dev = self.model.device
        mp = torch.from_numpy(csr.indptr).to(dev)
        mi = torch.from_numpy(csr.indices if len(csr.indices) else np.zeros(1, np.int32)).to(dev)
        n = max(1, min(int(amount), num_cards))
        ids, vals, cnt = topn_masked(probs, mp, mi, n, only_listed=False, descending=True)
        c = int(cnt[0])
        ids = ids[0, :c].cpu().numpy(); vals = vals[0, :c].cpu().numpy()
        results = probs[0].cpu().numpy()
        output = {"additions": dict(), "cuts": dict()}
        for rec, score in zip(ids, vals):
            output["additions"][int_to_card[int(rec)]] = float(score)
        for idx in cube_indices:                       # cubelist order, duplicates overwrite (dict)
            output["cuts"][int_to_card[idx]] = float(results[idx])
        return output
