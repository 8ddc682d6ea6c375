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

from .. import _lib
from .._lib import call, ptr, stream_ptr
from ..graph import rank_cuts, rank_targets, topn_masked
from ..sparse import CubeCSR
from .model import CC_Recommender, SparseBatch

EMBED_DIM = 64           # the encoder's bottleneck width, the only one cc_cosine_neg_many_f32 takes


def plan_query_blocks(num_queries: int, num_cands: int, n: int, budget_bytes: int):
    """``(rows, ldo)`` of ``MLRecommender.nearest``'s query blocks: each block's distance rows (ldo = num_cands rounded
    up to 4 floats) plus the select's workspace for them (cc_topn_workspace_bytes, none for n <= 2048) fit
    ``budget_bytes``; a block holds at least one row and at most ``num_queries``."""
    ldo = (int(num_cands) + 3) // 4 * 4
    per_row = 4 * ldo + int(_lib.load().cc_topn_workspace_bytes(int(num_cands), 1, int(n), 0))
    return max(1, min(int(num_queries), int(budget_bytes) // per_row)), ldo


def _embedding_rows(x: torch.Tensor, device, what: str) -> torch.Tensor:
    """``x`` as float32 (rows, 64) on ``device`` with the 16-byte aligned rows cc_cosine_neg_many_f32 reads as float4
    (copied only when the layout does not already qualify)."""
    if not isinstance(x, torch.Tensor) or x.dim() != 2 or x.shape[1] != EMBED_DIM or x.dtype != torch.float32:
        raise ValueError(f"{what} must be a float32 (rows, {EMBED_DIM}) tensor")
    dev = torch.device(device)
    if x.device.type != dev.type or (dev.index is not None and x.device.index != dev.index):
        raise ValueError(f"{what} live on {x.device}, the model on {dev}")
    if x.stride(1) == 1 and x.stride(0) % 4 == 0 and x.data_ptr() % 16 == 0:
        return x
    return torch.empty(x.shape, dtype=x.dtype, device=x.device).copy_(x)


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

    def _forward_chunks(self, csr: CubeCSR, *others: CubeCSR, decode: bool = True):
        """The chunked forward of ``recommend_device``, ``target_ranks_device`` and ``cut_ranks_device``: yields ``(lo, hi, idx, ptr_, z,
        rest)`` per chunk of ``self.chunk`` cubes, where ``idx`` / ``ptr_`` are rows [lo, hi) of ``csr`` on the device,
        ``z`` the (hi - lo, C) logits of ``decoder(encoder(rows))`` and ``rest`` one ``(idx, ptr)`` device pair of rows
        [lo, hi) per CSR in ``others``.  Chunk i+1's rows are uploaded on a copy stream while chunk i computes; nothing
        synchronises with the host.  ``decode=False`` (``cube_embeddings``): ``z`` is the (hi - lo, 64) encoder output."""
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
            z = m._encode(sb)
            if decode:
                z = m._decode(z, "main")
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
        return self._ranks(visible, hidden, rank_targets, ("visible", "hidden"))

    def cut_ranks_device(self, corrupted: CubeCSR, intruders: CubeCSR) -> torch.Tensor:
        """Cut ranks, int32 aligned with ``intruders.indices``, on the device.  Cube b's ``corrupted`` cards (its own
        plus its intruders) are the model input and the candidates; each of its ``intruders`` gets the 0-based slot at
        which the cube's cut list -- its cards by ascending probability, ties to the smaller index, the order of
        ``GraphRecommender.cuts`` and ``ml_recommend.py``'s lowest-scored lines -- would list it, or -1 if it is not one
        of the corrupted cards.  Same chunked pipeline as ``recommend_device`` with no host synchronisation; the ranks
        come from cc_rank_cuts_f32 on the logits with the sigmoid fused in."""
        return self._ranks(corrupted, intruders, rank_cuts, ("corrupted", "intruders"))

    def _ranks(self, inputs: CubeCSR, targets: CubeCSR, rank, names) -> torch.Tensor:
        if targets.num_cubes != inputs.num_cubes or targets.num_cards != inputs.num_cards:
            raise ValueError(f"{names[0]} and {names[1]} must hold the same cubes over the same cards")
        if inputs.num_cards != self.model.N:
            raise ValueError(f"the cubes span {inputs.num_cards} cards, the model {self.model.N}")
        hp = np.ascontiguousarray(targets.indptr, dtype=np.int64)
        ranks = torch.empty(max(int(hp[-1]), 1), dtype=torch.int32, device=self.model.device)
        for lo, hi, idx, ptr_, z, ((t_idx, t_ptr),) in self._forward_chunks(inputs, targets):
            if hp[hi] > hp[lo]:
                rank(z, ptr_, idx, t_ptr, t_idx, sigmoid=True, out=ranks[int(hp[lo]):int(hp[hi])])
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
        comes first with -1).  Ties: smaller index first (stable argsort).  Row 0 of ``similar_cards([card_idx], n)``:
        the same bits as one cc_cosine_neg_f32 row ranked by cc_topn_masked_f32."""
        ids, dists = self.similar_cards([int(card_idx)], max(1, int(n)), embeddings=embeddings)
        return ids[0].cpu().numpy(), dists[0].cpu().numpy()

    def similar_cards(self, card_ids, n: int, *, exclude_self: bool = False, embeddings: torch.Tensor | None = None):
        """``similar`` for many cards at once: ``(ids int32 (Q, n'), dists float32 (Q, n'))`` on the device, row i the
        cards nearest to ``card_ids[i]`` by -cosine of their encoder embeddings, ascending, ties to the smaller index.
        ``card_ids=None``: every card, in id order (the similar-cards table).  ``exclude_self``: each card is left out of
        its own row.  n' = min(n, candidates per row).  ``embeddings``: ``card_embeddings()`` computed beforehand."""
        m = self.model
        emb = _embedding_rows(self.card_embeddings() if embeddings is None else embeddings, m.device, "embeddings")
        if emb.shape[0] != m.N:
            raise ValueError(f"embeddings hold {emb.shape[0]} cards, the model {m.N}")
        if card_ids is None:
            queries = emb
            exclude = torch.arange(m.N, dtype=torch.int32, device=m.device) if exclude_self else None
        else:
            ids = np.asarray(card_ids, dtype=np.int64).reshape(-1)
            if len(ids) and (ids.min() < 0 or ids.max() >= m.N):
                raise ValueError(f"card ids must lie in [0, {m.N})")
            if len(ids) and (np.diff(ids) == 1).all():    # a run of ids (one card: ``similar``): rows of emb, no gather
                lo = int(ids[0])
                queries = emb[lo:lo + len(ids)]
                exclude = (torch.arange(lo, lo + len(ids), dtype=torch.int32, device=m.device)
                           if exclude_self else None)
            else:
                rows = torch.from_numpy(ids).to(m.device)
                queries = emb.index_select(0, rows)
                exclude = rows.to(torch.int32) if exclude_self else None
        return self._nearest(queries, emb, n, exclude)

    def nearest(self, queries: torch.Tensor, corpus: torch.Tensor, n: int, *, self_offset: int | None = None,
                budget_bytes: int = 1 << 30):
        """The ``n`` rows of ``corpus`` nearest to each query by -cosine (Keras' CosineSimilarity loss), for float32
        ``(Q, 64)`` queries and ``(K, 64)`` corpus embeddings on the device: ``(ids int32 (Q, n'), dists float32
        (Q, n'))`` on the device, each row ascending with ties to the smaller index, n' = min(n, candidates per row).
        ``self_offset=o``: query i is corpus row o + i and is left out of its own row.

        The queries go in blocks whose (rows, ldo) distance matrix -- ldo = K rounded up to 4 floats, so the row
        select takes it -- plus any select workspace fits ``budget_bytes`` (at least one row per block).  Per block
        cc_cosine_neg_many_f32 writes the distances (bit for bit cc_cosine_neg_f32's) and the masked select ranks
        them into the caller-sized outputs; nothing synchronises with the host."""
        queries = _embedding_rows(queries, self.model.device, "queries")
        corpus = _embedding_rows(corpus, self.model.device, "corpus")
        exclude = None
        if self_offset is not None:
            o = int(self_offset)
            if o < 0 or o + queries.shape[0] > corpus.shape[0]:
                raise ValueError(f"self_offset {o} puts queries past the {corpus.shape[0]} corpus rows")
            exclude = torch.arange(o, o + queries.shape[0], dtype=torch.int32, device=self.model.device)
        return self._nearest(queries, corpus, n, exclude, budget_bytes)

    def _nearest(self, queries, corpus, n, exclude, budget_bytes=1 << 30):
        """``nearest`` on validated rows; ``exclude``: None or int32 (Q,), the one corpus row left out of row i."""
        dev = self.model.device
        nq, nc = queries.shape[0], corpus.shape[0]
        if int(n) < 1:
            raise ValueError("n must be >= 1")
        n = min(int(n), nc - (exclude is not None))
        ids = torch.empty((nq, max(n, 0)), dtype=torch.int32, device=dev)
        dists = torch.empty((nq, max(n, 0)), dtype=torch.float32, device=dev)
        if nq == 0 or n <= 0:
            return ids, dists
        rows, ldo = plan_query_blocks(nq, nc, n, budget_bytes)
        buf = torch.empty((rows, ldo), dtype=torch.float32, device=dev)
        cnt = torch.empty(nq, dtype=torch.int32, device=dev)
        if exclude is None:                          # an empty mask: every corpus row is a candidate
            mask_ptr = torch.zeros(rows + 1, dtype=torch.int64, device=dev)
            mask_idx = torch.zeros(1, dtype=torch.int32, device=dev)
        else:                                        # one masked id per row
            mask_ptr = torch.arange(rows + 1, dtype=torch.int64, device=dev)
        for lo in range(0, nq, rows):
            hi = min(lo + rows, nq)
            d = buf[:hi - lo]
            call("cc_cosine_neg_many_f32", ptr(queries[lo:hi]), queries.stride(0), hi - lo, ptr(corpus),
                 corpus.stride(0), nc, EMBED_DIM, ptr(d), ldo, stream_ptr())
            topn_masked(d[:, :nc], mask_ptr[:hi - lo + 1], mask_idx if exclude is None else exclude[lo:hi], n,
                        only_listed=False, descending=False, out=(ids[lo:hi], dists[lo:hi], cnt[lo:hi]))
        return ids, dists

    def cube_embeddings(self, csr: CubeCSR) -> torch.Tensor:
        """``model.encoder(cubes)``: the 64-d embedding of every cube, (K, 64) float32 on the device, encoded in chunks
        of ``self.chunk`` cubes with the upload pipeline of ``recommend_device``."""
        m = self.model
        if csr.num_cards != m.N:
            raise ValueError(f"the cubes span {csr.num_cards} cards, the model {m.N}")
        out = torch.empty((csr.num_cubes, EMBED_DIM), dtype=torch.float32, device=m.device)
        for lo, hi, _, _, e, _ in self._forward_chunks(csr, decode=False):
            out[lo:hi].copy_(e)
        return out

    def similar_cubes(self, queries: CubeCSR, n: int, corpus=None):
        """Cubes like each of ``queries``: ``(ids int32 (Q, n'), dists float32 (Q, n'))`` on the device, the ``n``
        corpus cubes nearest by -cosine of their encoder embeddings, ascending, ties to the smaller index.
        ``corpus=None``: the query cubes ranked against each other, each cube left out of its own row (cubes with the
        same card list have the same embedding, so they still rank first, at -1 up to rounding).  ``corpus``: a
        ``CubeCSR``, or the ``(K, 64)`` ``cube_embeddings`` of one (a server embeds its corpus once); nothing is left
        out then."""
        q = self.cube_embeddings(queries)
        if corpus is None:
            return self._nearest(q, q, n, torch.arange(q.shape[0], dtype=torch.int32, device=q.device))
        if isinstance(corpus, CubeCSR):
            corpus = self.cube_embeddings(corpus)
        else:
            corpus = _embedding_rows(corpus, self.model.device, "corpus")
        return self._nearest(q, corpus, n, None)

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
