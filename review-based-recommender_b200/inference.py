"""Inference scoring (BASELINE.json configs[4]), the per-entity feature cache (SURVEY §8f-2) and full-catalogue top-k.

The reference has no predict entry point: scoring is `valid_one_epoch` (trainer/train_deepconn_pp.py:191-212) — `model.eval()`,
`torch.no_grad()`, the same forward — and every example carries its own two padded documents (:274), so the encoder runs
twice per (user, item) pair although a user's document is the same in every pair the user appears in.

`PairScorer.score_pairs` is that data flow on the fused kernels.  `PairScorer.build_cache` encodes each entity's side ONCE
and `score_cached` then scores pairs from the cached features only: 10 M pairs over U + I = 32 k documents is ≈ 600x less
encoder work.  In eval mode every model puts an entity's side through that entity's inputs alone, so all three cache:
  DeepCoNN  the entity's document (K2) → [U, H] / [I, H]; pairs score through K1 gather + K4 head, bit-identical;
  NARRE     the entity's reviews (K2) + LinearAttention over the ids of the counterparts they review → [U, H] / [I, H];
            pairs score through K1 + K4 as for DeepCoNN;
  D-ATT     fc(encode(document)) per side → [U, 50] / [I, 50]; a pair's score is the dot product of its two rows.

`PairScorer.recommend` answers "the k best items for these users out of the whole catalogue" with K10 (ops.factor_topk),
which never materialises the users x items score matrix; `rank_items` / `evaluate` give the exact full-catalogue rank of
held-out items and HR@k / Recall@k / NDCG@k / MRR / AUC from it with K11 (ops.factor_rank), on the same scores.  The FM head factorises exactly:
  relu(u*i) = relu(u)*relu(i) + relu(-u)*relu(-i)   ⇒   score(u,i) = A[u] . B[i] + row_bias[u] + col_bias[i]
with A = [h*relu(u_lat), h*relu(-u_lat)], B = [relu(i_lat), relu(-i_lat)], row_bias = ub + g, col_bias = ib (fm_factors);
D-ATT's score is already a dot product of the two FC outputs.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from . import ops
from .deepconn import DeepCoNNpp
from .dual_att import DualAtt
from .layers import fused_head
from .narre import NARRE


def fm_factors(u_lat: torch.Tensor, i_lat: torch.Tensor, h: torch.Tensor, user_bias: torch.Tensor, item_bias: torch.Tensor,
               g_bias: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """FM head (models/deepconn/layers.py:200-207) as a factor product: score(u, i) = A[u] . B[i] + row_bias[u] + col_bias[i]
    for latents u_lat [U, K], i_lat [I, K] (LastFeat outputs of entity rows u / i), h [K, 1], user_bias [U, 1],
    item_bias [I, 1], g_bias [1].  Returns (A [U, 2K], row_bias [U], B [I, 2K], col_bias [I]) in the inputs' dtype."""
    hv = h.reshape(1, -1)
    A = torch.cat([hv * torch.relu(u_lat), hv * torch.relu(-u_lat)], dim=1)
    B = torch.cat([torch.relu(i_lat), torch.relu(-i_lat)], dim=1)
    return A, user_bias.reshape(-1) + g_bias.reshape(()), B, item_bias.reshape(-1)


def _is_narre(model) -> bool:
    return isinstance(model, NARRE)


def _is_datt(model) -> bool:
    return isinstance(model, DualAtt)


class PairScorer:
    def __init__(self, model):
        if not isinstance(model, (DeepCoNNpp, NARRE, DualAtt)):
            raise TypeError("PairScorer serves DeepCoNNpp, NARRE and DualAtt")
        self.model = model.eval()
        self.user_feat: Optional[torch.Tensor] = None
        self.item_feat: Optional[torch.Tensor] = None
        self._factors = None         # (key, (A, row_bias, B, col_bias)) derived from the current head parameters
        self._explain = None         # per-side tensors kept by build_cache(explain=True)

    @torch.no_grad()
    def score_pairs(self, *inputs) -> torch.Tensor:
        """The reference's per-pair data flow: both sides encoded for every pair (the model's own eval forward)."""
        out = self.model(*inputs)
        return out[0] if isinstance(out, tuple) else out

    @torch.no_grad()
    def build_cache(self, user_docs: torch.Tensor, item_docs: torch.Tensor, user_masks: Optional[torch.Tensor] = None,
                    item_masks: Optional[torch.Tensor] = None, chunk: int = 4096, *, user_rev_ids: Optional[torch.Tensor] = None,
                    item_rev_ids: Optional[torch.Tensor] = None, explain: bool = False) -> None:
        """Row e of every argument belongs to entity id e (row 0 = the padding entity).
        DeepCoNN: user_docs [U, L], item_docs [I, L]; masks default to ids != 0 (utils.py:30-42).
        NARRE: user_docs [U, R, T], item_docs [I, R, T] (the entity's reviews), optional masks of the same shapes, and
          user_rev_ids [U, R] / item_rev_ids [I, R]: the ids of the items a user reviewed / the users who reviewed an item —
          what NARRE's dataset supplies as reuid / reiid for a pair with that entity.
        D-ATT: user_docs [U, L], item_docs [I, L] (no masks).
        explain=True also keeps what `explain` needs per entity (references to the documents and masks; for DeepCoNN and
        NARRE the conv arg-max and the tap contributions of every pooled window (K12a), for NARRE the per-review features
        and attention weights; for D-ATT the two K5 gates, the conv arg-max, the FC hidden ReLU mask and the per-entity
        terms of gradient x input, rbr_datt_explain_contrib).  The cached features are the same either way."""
        m = self.model
        self.model.eval()
        self._factors = None
        self._explain = None
        if explain and not _is_datt(m) and m.ngram.arch != "CNN":
            raise NotImplementedError("PairScorer.explain covers the CNN encoder; arch='HierPooling' pools averages, "
                                      "which have no per-window tap contributions")
        if _is_datt(m):
            if user_masks is not None or item_masks is not None:
                raise ValueError("DualAtt takes no masks")

            if explain:
                self._build_datt_explain_cache(user_docs, item_docs, chunk)
                return

            def side(docs, s):
                return torch.cat([m.fc(m.encode([docs[lo:lo + chunk]], [s])[0]) for lo in range(0, docs.shape[0], chunk)], 0)
            self.user_feat, self.item_feat = side(user_docs, "u"), side(item_docs, "i")
            return
        if explain:
            self._build_explain_cache(user_docs, item_docs, user_masks, item_masks, chunk, user_rev_ids, item_rev_ids)
            return
        if _is_narre(m):
            if user_rev_ids is None or item_rev_ids is None:
                raise ValueError("NARRE's build_cache needs user_rev_ids [U, R] and item_rev_ids [I, R]")
            R, T = m.doc_num, m.doc_len
            ent_chunk = max(1, chunk // R)

            def side(docs, masks, rev_ids, att):
                if docs.shape[1:] != (R, T) or rev_ids.shape != docs.shape[:2]:
                    raise ValueError(f"NARRE was built for [*, {R}, {T}] reviews with [*, {R}] review ids, got "
                                     f"{tuple(docs.shape)} / {tuple(rev_ids.shape)}")
                outs = []
                for lo in range(0, docs.shape[0], ent_chunk):
                    d = docs[lo:lo + ent_chunk]
                    mk = None if masks is None else masks[lo:lo + ent_chunk].reshape(-1, T)
                    (f,) = m.ngram.encode(m.word_embeddings, [d.reshape(-1, T)], [mk])
                    outs.append(att(f.view(d.shape[0], R, -1), rev_ids[lo:lo + ent_chunk])[0])
                return torch.cat(outs, 0)
            self.user_feat = side(user_docs, user_masks, user_rev_ids, m.user_att)
            self.item_feat = side(item_docs, item_masks, item_rev_ids, m.item_att)
            return

        def encode(docs, masks):
            outs = []
            for lo in range(0, docs.shape[0], chunk):
                mk = None if masks is None else masks[lo:lo + chunk]
                (f,) = m.ngram.encode(m.word_embeddings, [docs[lo:lo + chunk]], [mk])
                outs.append(f)
            return torch.cat(outs, dim=0)
        self.user_feat = encode(user_docs, user_masks)
        self.item_feat = encode(item_docs, item_masks)

    def _datt_side_prm(self, s: str):
        m = self.model
        return [p.detach() for p in m._side_params(getattr(m, f"{s}_local_atten"), getattr(m, f"{s}_global_atten"))]

    def _build_datt_explain_cache(self, user_docs, item_docs, chunk):
        """D-ATT with explain=True: the encoder once per chunk (ops.datt_encode_side, the kernels DualAtt.encode runs), the FC
        stack layer by layer (the same modules in the same order as m.fc, so the cached features are bit-identical to
        build_cache(explain=False)) to keep its hidden ReLU mask, then K12's per-entity terms (ops.datt_explain_contrib)."""
        m = self.model
        table = m.word_embeddings.embedding.weight.detach()
        shadow = m.word_embeddings.bf16_shadow() if m.precision == "bf16" else None
        lin0, relu, drop, lin1 = m.fc
        sides, outs = {}, {}
        for name, s, docs in (("user", "u", user_docs), ("item", "i", item_docs)):
            if docs.shape[-1] != m.doc_len:
                raise ValueError(f"DualAtt was built for doc_len={m.doc_len}, got {docs.shape[-1]}")
            prm = self._datt_side_prm(s)
            packed = ops.datt_side_packs(prm)
            keep = {k: [] for k in ("gate_l", "gate_g", "argmax", "contrib", "gate_coef", "gate_vec", "hid_mask")}
            out = []
            for lo in range(0, docs.shape[0], chunk):
                d = docs[lo:lo + chunk]
                feat, amax, _, gl, gg = ops.datt_encode_side(table, d, prm, m.precision, shadow, packed)
                z = lin0(feat)
                out.append(lin1(drop(relu(z))))
                contrib, coef, vec = ops.datt_explain_contrib(table, d, prm, gl, gg, feat, amax, packed)
                for k, v in (("gate_l", gl), ("gate_g", gg), ("argmax", amax), ("contrib", contrib), ("gate_coef", coef),
                             ("gate_vec", vec), ("hid_mask", z > 0)):
                    keep[k].append(v)
            sides[name] = {"docs": docs, **{k: torch.cat(v) for k, v in keep.items()}}
            outs[name] = torch.cat(out, 0)
        self.user_feat, self.item_feat = outs["user"], outs["item"]
        self._explain = sides

    def _conv_specs(self):
        conv = self.model.ngram.conv
        return [(c.weight.shape[0], k, (k - 1) // 2) for c, k in zip(conv.list_of_conv1d, conv.kernel_sizes)]

    def _encode_explain(self, docs: torch.Tensor, masks: Optional[torch.Tensor], chunk: int):
        """docs [N, L] (masks None: ids != 0) → (feat [N, H], argmax int32 [N, H], contrib [N, sum_c H_c * k_c]): the encoder's
        own features and first arg-max (EncodeDocsFn), then the tap contributions of every pooled window (K12a)."""
        m = self.model
        conv = m.ngram.conv
        table = m.word_embeddings.embedding.weight.detach()
        specs = self._conv_specs()
        taps = sum(h * k for h, k, _ in specs)
        feats, amaxes = [], []
        contrib = torch.empty(docs.shape[0], taps, dtype=torch.float32, device=table.device)
        for lo in range(0, docs.shape[0], chunk):
            d = docs[lo:lo + chunk]
            mk = None if masks is None else masks[lo:lo + chunk]
            f, a = m.ngram.encode(m.word_embeddings, [d], [mk], return_argmax=True)
            col = tcol = 0
            for i, (h, k, pad) in enumerate(specs):
                ops.conv_window_contrib(table, d, mk, conv.list_of_conv1d[i].weight.detach(), pad, a[:, col:col + h],
                                        packed=conv.packed(i), mask_from_ids=True, out=contrib[lo:lo + chunk, tcol:tcol + h * k])
                col += h
                tcol += h * k
            feats.append(f)
            amaxes.append(a)
        return torch.cat(feats), torch.cat(amaxes), contrib

    def _build_explain_cache(self, user_docs, item_docs, user_masks, item_masks, chunk, user_rev_ids, item_rev_ids):
        m = self.model
        if not _is_narre(m):
            sides = {}
            for name, docs, masks in (("user", user_docs, user_masks), ("item", item_docs, item_masks)):
                feat, amax, contrib = self._encode_explain(docs, masks, chunk)
                sides[name] = {"docs": docs, "masks": masks, "feat": feat, "argmax": amax, "contrib": contrib}
            self.user_feat, self.item_feat = sides["user"]["feat"], sides["item"]["feat"]
            self._explain = sides
            return
        if user_rev_ids is None or item_rev_ids is None:
            raise ValueError("NARRE's build_cache needs user_rev_ids [U, R] and item_rev_ids [I, R]")
        R, T = m.doc_num, m.doc_len
        ent_chunk = max(1, chunk // R)
        sides = {}
        for name, docs, masks, rev_ids, att in (("user", user_docs, user_masks, user_rev_ids, m.user_att),
                                                ("item", item_docs, item_masks, item_rev_ids, m.item_att)):
            if docs.shape[1:] != (R, T) or rev_ids.shape != docs.shape[:2]:
                raise ValueError(f"NARRE was built for [*, {R}, {T}] reviews with [*, {R}] review ids, got "
                                 f"{tuple(docs.shape)} / {tuple(rev_ids.shape)}")
            n = docs.shape[0]
            feat, amax, contrib = self._encode_explain(docs.reshape(n * R, T), None if masks is None else masks.reshape(n * R, T),
                                                       ent_chunk * R)
            outs, scores = [], []
            for lo in range(0, n, ent_chunk):
                o, s = att(feat[lo * R:(lo + ent_chunk) * R].view(-1, R, feat.shape[1]), rev_ids[lo:lo + ent_chunk])
                outs.append(o)
                scores.append(s.view(-1, R))
            sides[name] = {"docs": docs, "masks": masks, "rev_ids": rev_ids, "feat": feat, "argmax": amax, "contrib": contrib,
                           "att": torch.cat(scores), "out": torch.cat(outs)}
        self.user_feat, self.item_feat = sides["user"].pop("out"), sides["item"].pop("out")
        self._explain = sides
    @torch.no_grad()
    def score_cached(self, u_ids: torch.Tensor, i_ids: torch.Tensor) -> torch.Tensor:
        """preds for pairs (u_ids[b], i_ids[b]) from the cached features, no encoder: K1 row gather + K4 head (DeepCoNN,
        NARRE) or K1 + dot product (D-ATT, dual_att.py:59-61)."""
        if self.user_feat is None:
            raise RuntimeError("PairScorer.build_cache(...) first")
        m = self.model
        u_text = ops.gather_rows(self.user_feat, u_ids)
        i_text = ops.gather_rows(self.item_feat, i_ids)
        if _is_datt(m):
            return torch.sum(torch.mul(u_text, i_text), 1).view(-1)
        return fused_head(m.user_feat, m.item_feat, m.fm, u_text, i_text, u_ids, i_ids, False, None).view(-1)

    def _head_params(self):
        m = self.model
        if _is_datt(m):
            return []
        return [m.user_feat.W, m.user_feat.b, m.user_feat.ebd.weight, m.item_feat.W, m.item_feat.b, m.item_feat.ebd.weight,
                m.fm.h, m.fm.user_bias.weight, m.fm.item_bias.weight, m.fm.g_bias]

    def factors(self) -> Tuple[torch.Tensor, Optional[torch.Tensor], torch.Tensor, Optional[torch.Tensor]]:
        """(A [U, D], row_bias [U] or None, B [I, D], col_bias [I] or None) with score(u, i) = A[u] . B[i] + biases for the
        cached entities under the CURRENT head parameters.  Re-derived when a parameter changed (optimizer steps bump
        its version counter) or the cache was rebuilt."""
        if self.user_feat is None:
            raise RuntimeError("PairScorer.build_cache(...) first")
        params = self._head_params()
        key = tuple((p._version, p.data_ptr()) for p in params) + ((self.user_feat.data_ptr(), self.item_feat.data_ptr()),)
        if self._factors is None or self._factors[0] != key:
            if _is_datt(self.model):
                f = (self.user_feat, None, self.item_feat, None)
            else:
                with torch.no_grad():
                    # LastFeat (models/deepconn/layers.py:163) in float64: exact fp32 latents whatever the TF32 setting
                    d = [p.detach().double() for p in params]
                    Wu, bu, eu, Wi, bi, ei, h, ub, ib, g = d
                    n_u, n_i = self.user_feat.shape[0], self.item_feat.shape[0]
                    u_lat = self.user_feat.double() @ Wu + bu + eu[:n_u]
                    i_lat = self.item_feat.double() @ Wi + bi + ei[:n_i]
                    f = tuple(t.float().contiguous() for t in fm_factors(u_lat, i_lat, h, ub[:n_u], ib[:n_i], g))
            self._factors = (key, f)
        return self._factors[1]

    @torch.no_grad()
    def recommend(self, u_ids: torch.Tensor, k: int, exclude: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
                  exclude_padding: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
        """The k best cached items for each user u_ids[r], by score descending then item id ascending (K10: one fused
        score GEMM + per-row top-k, the [len(u_ids), I] score matrix is never materialised).
        exclude = (indptr [len(u_ids) + 1], indices) int64 CUDA CSR: items to leave out per row (e.g. those already rated).
        exclude_padding drops the item padding row (fm.item_padding_idx; 0 for D-ATT).
        Returns (scores [len(u_ids), k] fp32, items [len(u_ids), k] int64); rows with fewer than k eligible items end in
        (-inf, -1).  Scores agree with score_cached on the same pairs to fp32 rounding."""
        A_rows, rb_rows, B, cb, _ = self._user_rows(u_ids, exclude_padding)
        return ops.factor_topk(A_rows, rb_rows, B, cb, k, exclude=exclude)

    def _user_rows(self, u_ids: torch.Tensor, exclude_padding: bool):
        """(A rows, row_bias rows, B, col_bias, padding item or None) for users u_ids under the current head parameters;
        with exclude_padding the padding item's column bias is -inf, so it never enters a top-k nor counts in a rank."""
        self.model.eval()
        A, rb, B, cb = self.factors()
        u_ids = u_ids.to(device=A.device, dtype=torch.int64).reshape(-1)
        if u_ids.numel() and (int(u_ids.min()) < 0 or int(u_ids.max()) >= A.shape[0]):
            raise ValueError(f"user ids must lie in [0, {A.shape[0]})")
        A_rows = A.index_select(0, u_ids)
        rb_rows = None if rb is None else rb.index_select(0, u_ids)
        pad = None
        if exclude_padding:
            pad = 0 if _is_datt(self.model) else self.model.fm.item_padding_idx
            if pad is not None and 0 <= pad < B.shape[0]:
                # a -inf column bias: the padding item's score never beats a threshold, so it is never returned
                cb = torch.zeros(B.shape[0], dtype=torch.float32, device=B.device) if cb is None else cb.clone()
                cb[pad] = float("-inf")
            else:
                pad = None
        return A_rows, rb_rows, B, cb, pad

    @torch.no_grad()
    def rank_items(self, u_ids: torch.Tensor, targets: Tuple[torch.Tensor, torch.Tensor],
                   exclude: Optional[Tuple[torch.Tensor, torch.Tensor]] = None, exclude_padding: bool = True
                   ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """The exact full-catalogue rank of each target item for user u_ids[r] (K11, ops.factor_rank): 1 + the number of
        eligible items ahead of it by (score desc, item id asc), i.e. its 1-based position in recommend(k = inf).
        targets = (indptr [len(u_ids) + 1], indices) int64 CUDA CSR, e.g. each user's held-out items; exclude as for
        recommend, e.g. the items the user rated in training.  exclude_padding leaves the item padding row out of every
        count (a target that is the padding item then raises ValueError).
        Returns (ranks int64 [nnz], scores fp32 [nnz], both in the order of `indices` — rank -1 for a NaN / -inf score —,
        n_candidates int64 [len(u_ids)]: the eligible items per row, the padding item not counted).  A target with
        rank <= k is in recommend(u_ids, k) at position rank - 1 with the identical score."""
        A_rows, rb_rows, B, cb, pad = self._user_rows(u_ids, exclude_padding)
        if pad is not None:
            t_idx = targets[1]
            if bool((t_idx == pad).any()):
                raise ValueError(f"target item {pad} is the padding item, which exclude_padding=True leaves out")
        ranks, scores, n_cand = ops.factor_rank(A_rows, rb_rows, B, cb, targets, exclude=exclude)
        if pad is not None:
            pad_listed = torch.zeros(A_rows.shape[0], dtype=torch.bool, device=A_rows.device)
            if exclude is not None:
                e_ptr, e_idx = exclude
                rows = torch.repeat_interleave(torch.arange(A_rows.shape[0], device=e_ptr.device), e_ptr[1:] - e_ptr[:-1])
                pad_listed[rows[e_idx == pad]] = True
            n_cand = n_cand - (~pad_listed).long()
        return ranks, scores, n_cand

    @torch.no_grad()
    def evaluate(self, u_ids: torch.Tensor, targets: Tuple[torch.Tensor, torch.Tensor], ks=(10,),
                 exclude: Optional[Tuple[torch.Tensor, torch.Tensor]] = None, exclude_padding: bool = True) -> dict:
        """Full-catalogue ranking metrics of the held-out `targets` (rank_items, then ranking_metrics): hr@k, recall@k and
        ndcg@k for each k in ks, mrr, auc and n_rows, averaged over the rows that have at least one target."""
        ranks, _, n_cand = self.rank_items(u_ids, targets, exclude=exclude, exclude_padding=exclude_padding)
        return ranking_metrics(ranks, targets[0], n_cand, ks)

    @torch.no_grad()
    def explain(self, u_ids: torch.Tensor, i_ids: torch.Tensor, m: int = 5, width: Optional[int] = None,
                return_maps: bool = False, chunk: int = 16384, *, attribution: bool = False) -> "Explanation":
        """Why the model predicts what score_cached(u_ids, i_ids) returns, from the cache of build_cache(explain=True).

        DeepCoNN / NARRE: gradient x input on the embedded tokens of each side's document(s), at the model's own arg-max and
        ReLU decisions (K12, DESIGN.md): attr[t] = sum over pooled features h whose window covers t (feat > 0) of
        g[h] * c[h, j], g = d pred / d feat from K4's backward (NARRE: further through K3's backward to each review's
        feature), c = the cached tap contribution.  Per side: text_total (= the map's sum), the top-m / bottom-m windows of
        `width` positions (default: the largest kernel size; greedy without overlap, ties to the lower start, never across a
        review) and, with return_maps, the map itself ([B, L], NARRE [B, R, T]; 4 bytes per position and pair, so it is
        only written when asked for).  NARRE also gives review_weight (the entity's attention weights) and review_attr
        (per-review sums of the map).  D-ATT: the local gate per token and the global gate per document (K5); by default
        also the m positions with the largest local gate.  With attribution=True (D-ATT only; DeepCoNN and NARRE always
        attribute) D-ATT's top / bottom windows, text_total and map are gradient x input as for DeepCoNN, through both
        gates and the FC stack at the model's own arg-max and ReLU decisions: g = d pred / d feat from the cached FC outputs
        and hidden ReLU masks (ops.datt_fc_grads), then K12b over the cached per-entity terms with the global gate as a
        dense term; the default width is the local window size.  Positions are flat (NARRE: r * T + t); `tokens_at` turns
        them into ids.  Pairs run in chunks of `chunk`, so scratch memory does not grow with B."""
        if self._explain is None or self.user_feat is None:
            raise RuntimeError("PairScorer.build_cache(..., explain=True) first")
        mdl = self.model
        mdl.eval()
        dev = self.user_feat.device
        u_ids = u_ids.to(device=dev, dtype=torch.int64).reshape(-1)
        i_ids = i_ids.to(device=dev, dtype=torch.int64).reshape(-1)
        if u_ids.numel() != i_ids.numel():
            raise ValueError("u_ids and i_ids must hold one id per pair")
        n_u, n_i = self.user_feat.shape[0], self.item_feat.shape[0]
        if u_ids.numel():
            lo_u, hi_u, lo_i, hi_i = torch.stack([u_ids.min(), u_ids.max(), i_ids.min(), i_ids.max()]).tolist()
            if lo_u < 0 or hi_u >= n_u or lo_i < 0 or hi_i >= n_i:
                raise ValueError(f"user ids must lie in [0, {n_u}) and item ids in [0, {n_i})")
        m = int(m)
        pred = self.score_cached(u_ids, i_ids)
        if _is_datt(mdl) and attribution:
            return self._explain_datt(u_ids, i_ids, pred, m, width, return_maps, chunk)
        if _is_datt(mdl):
            L = self._explain["user"]["gate_l"].shape[1]
            if not 1 <= m <= L:
                raise ValueError(f"m must lie in [1, {L}]")
            sides = []
            for name, ids in (("user", u_ids), ("item", i_ids)):
                c = self._explain[name]
                gl = c["gate_l"].index_select(0, ids)
                # stable sort: equal gates keep the lower position first
                order = torch.sort(gl, dim=1, descending=True, stable=True).indices[:, :m]
                sides.append(SideExplanation(local_att=gl, global_att=c["gate_g"].index_select(0, ids), top_pos=order,
                                             top_attr=gl.gather(1, order)))
            return Explanation(pred, *sides)
        specs = self._conv_specs()
        R, T = (mdl.doc_num, mdl.doc_len) if _is_narre(mdl) else (1, self._explain["user"]["docs"].shape[1])
        width = max(k for _, k, _ in specs) if width is None else int(width)
        if not ops.explain_supported(R * T, m, width, len(specs)):
            raise ValueError(f"explain takes 1 <= m <= {ops.EXPLAIN_MAX_M}, 1 <= width <= {ops.EXPLAIN_MAX_WIDTH} and at most "
                             f"{ops.EXPLAIN_MAX_POSITIONS} positions per entity (got m={m}, width={width}, {R} x {T})")
        head = self._head_params()
        pads = (mdl.user_feat.padding_idx, mdl.item_feat.padding_idx, mdl.fm.padding_idx, mdl.fm.item_padding_idx)
        head_scratch = [torch.empty_like(p) for p in head]
        if _is_narre(mdl):
            att_prm = [[a.W_rv, a.W_id, a.h, a.b_1, a.b_2, a.ebd_vals.weight] for a in (mdl.user_att, mdl.item_att)]
            att_scratch = [[torch.empty_like(p) for p in sp] for sp in att_prm]
            att_pads = (mdl.user_att.padding_idx, mdl.item_att.padding_idx)
        parts = {"user": [], "item": []}
        for lo in range(0, u_ids.numel(), chunk):
            u, i = u_ids[lo:lo + chunk], i_ids[lo:lo + chunk]
            g_u, g_i = ops.head_text_grads(ops.gather_rows(self.user_feat, u), ops.gather_rows(self.item_feat, i), u, i, head,
                                           pads, head_scratch)
            if _is_narre(mdl):
                cu, ci = self._explain["user"], self._explain["item"]
                H = cu["feat"].shape[1]
                g_u, g_i = ops.narre_feat_grads(
                    [cu["feat"].view(-1, R, H).index_select(0, u), ci["feat"].view(-1, R, H).index_select(0, i)],
                    [cu["rev_ids"].index_select(0, u), ci["rev_ids"].index_select(0, i)],
                    [cu["att"].index_select(0, u), ci["att"].index_select(0, i)], [g_u, g_i], att_prm, att_pads, att_scratch)
            for name, ids, g in (("user", u, g_u), ("item", i, g_i)):
                c = self._explain[name]
                parts[name].append(ops.explain_attrib(ids * R, g.view(ids.numel(), R, -1), c["feat"], c["argmax"], c["contrib"],
                                                      specs, R, T, m, width, return_map=return_maps,
                                                      return_review_attr=_is_narre(mdl)))
        sides = []
        for name, ids in (("user", u_ids), ("item", i_ids)):
            p = parts[name]
            cat = {k: torch.cat([x[k] for x in p]) if p else None for k in (p[0] if p else {})}
            if not p:                                   # no pairs: empty results of the right shapes
                cat = ops.explain_attrib(ids, torch.empty(0, R, sum(h for h, _, _ in specs), device=dev),
                                         self._explain[name]["feat"], self._explain[name]["argmax"],
                                         self._explain[name]["contrib"], specs, R, T, m, width, return_maps, _is_narre(mdl))
            mp = cat.get("map")
            sides.append(SideExplanation(
                text_total=cat["text_total"], top_pos=cat["top_pos"], top_attr=cat["top_attr"], bottom_pos=cat["bottom_pos"],
                bottom_attr=cat["bottom_attr"], map=None if mp is None else (mp.view(-1, R, T) if _is_narre(mdl) else mp),
                review_weight=self._explain[name]["att"].index_select(0, ids) if _is_narre(mdl) else None,
                review_attr=cat.get("review_attr")))
        return Explanation(pred, *sides)

    def _explain_datt(self, u_ids, i_ids, pred, m, width, return_maps, chunk) -> "Explanation":
        mdl = self.model
        L = mdl.doc_len
        specs = ops.datt_explain_convs(self._datt_side_prm("u"))
        width = specs[0][1] if width is None else int(width)
        if not ops.explain_supported(L, m, width, len(specs)):
            raise ValueError(f"explain takes 1 <= m <= {ops.EXPLAIN_MAX_M}, 1 <= width <= {ops.EXPLAIN_MAX_WIDTH} and at most "
                             f"{ops.EXPLAIN_MAX_POSITIONS} positions per entity (got m={m}, width={width}, L={L})")
        cu, ci = self._explain["user"], self._explain["item"]
        w0, w3 = mdl.fc[0].weight.detach(), mdl.fc[3].weight.detach()
        parts = {"user": [], "item": []}
        for lo in range(0, u_ids.numel(), chunk):
            u, i = u_ids[lo:lo + chunk], i_ids[lo:lo + chunk]
            g_u, g_i = ops.datt_fc_grads(u, i, self.user_feat, self.item_feat, cu["hid_mask"], ci["hid_mask"], w0, w3)
            for name, ids, g in (("user", u, g_u), ("item", i, g_i)):
                c = self._explain[name]
                parts[name].append(ops.explain_attrib(ids, g.view(ids.numel(), 1, -1), None, c["argmax"], c["contrib"], specs, 1,
                                                      L, m, width, return_map=return_maps, dense_coef=c["gate_coef"],
                                                      dense_vec=c["gate_vec"]))
        sides = []
        for name, ids in (("user", u_ids), ("item", i_ids)):
            c = self._explain[name]
            p = parts[name]
            if p:
                cat = {k: torch.cat([x[k] for x in p]) for k in p[0]}
            else:                                       # no pairs: empty results of the right shapes
                cat = ops.explain_attrib(ids, torch.empty(0, 1, c["argmax"].shape[1], device=ids.device), None, c["argmax"],
                                         c["contrib"], specs, 1, L, m, width, return_maps, dense_coef=c["gate_coef"],
                                         dense_vec=c["gate_vec"])
            sides.append(SideExplanation(
                text_total=cat["text_total"], top_pos=cat["top_pos"], top_attr=cat["top_attr"], bottom_pos=cat["bottom_pos"],
                bottom_attr=cat["bottom_attr"], map=cat.get("map"), local_att=c["gate_l"].index_select(0, ids),
                global_att=c["gate_g"].index_select(0, ids)))
        return Explanation(pred, *sides)

    def tokens_at(self, side: str, ent_ids: torch.Tensor, pos: torch.Tensor) -> torch.Tensor:
        """Token ids at flat positions pos [B, m] (explain's top_pos / bottom_pos) of the kept documents of entities
        ent_ids [B] on `side` ("user" / "item"); -1 where pos is -1."""
        if self._explain is None:
            raise RuntimeError("PairScorer.build_cache(..., explain=True) first")
        docs = self._explain[side]["docs"]
        flat = docs.reshape(docs.shape[0], -1).index_select(0, ent_ids.to(device=docs.device, dtype=torch.int64).reshape(-1))
        pos = pos.to(device=docs.device, dtype=torch.int64)
        tok = flat.to(torch.int64).gather(1, pos.clamp_min(0))
        return torch.where(pos >= 0, tok, torch.full_like(tok, -1))


@dataclass
class SideExplanation:
    """One side (user or item) of PairScorer.explain, one row per pair; fields a model does not have are None."""
    text_total: Optional[torch.Tensor] = None       # [B] sum of the attribution map
    top_pos: Optional[torch.Tensor] = None          # [B, m] int64 window starts (D-ATT without attribution: positions by
                                                    # local gate), -1 = none
    top_attr: Optional[torch.Tensor] = None         # [B, m] window sums (D-ATT without attribution: the local gate), NaN
                                                    # where top_pos is -1
    bottom_pos: Optional[torch.Tensor] = None       # [B, m] most negative windows
    bottom_attr: Optional[torch.Tensor] = None
    map: Optional[torch.Tensor] = None              # [B, L] (NARRE [B, R, T]) with return_maps
    review_weight: Optional[torch.Tensor] = None    # NARRE [B, R]: the entity's review attention weights
    review_attr: Optional[torch.Tensor] = None      # NARRE [B, R]: per-review sums of the map
    local_att: Optional[torch.Tensor] = None        # D-ATT [B, L]: local attention gate per token
    global_att: Optional[torch.Tensor] = None       # D-ATT [B]: global attention gate of the document


@dataclass
class Explanation:
    pred: torch.Tensor                              # [B], bit-identical to score_cached
    user: SideExplanation
    item: SideExplanation


def ranking_metrics(ranks: torch.Tensor, indptr: torch.Tensor, n_candidates: torch.Tensor, ks=(10,)) -> dict:
    """Binary-relevance ranking metrics from full-catalogue ranks (any device, no GPU needed).

    ranks [nnz]: the 1-based rank of each target among its row's n_candidates eligible items, -1 for a target that cannot
    be ranked (NaN / -inf score); row r's targets are ranks[indptr[r] : indptr[r+1]], m = their number.  Per row:
      hr@k      1 if the row's best rank <= k, else 0
      recall@k  hits@k / m
      ndcg@k    sum over hits of 1 / log2(rank + 1), divided by sum_{j=1..min(m, k)} 1 / log2(j + 1)
      mrr       1 / best rank (0 when no target has a rank)
      auc       mean over the row's targets of 1 - (negatives above t) / (n_candidates - m), where negatives above t =
                rank(t) - 1 - (other targets above t); a rank -1 target is below every negative (its term is 0)
    Each metric is the mean over rows with m >= 1 (n_rows of them); auc leaves out rows with n_candidates == m."""
    ranks = ranks.reshape(-1).to(torch.int64)
    dev = ranks.device
    indptr = indptr.to(device=dev, dtype=torch.int64)
    n_cand = n_candidates.to(device=dev, dtype=torch.int64).reshape(-1)
    n = indptr.numel() - 1
    m = indptr[1:] - indptr[:-1]
    rows = torch.repeat_interleave(torch.arange(n, device=dev), m)
    has = m > 0
    n_rows = int(has.sum())
    out = {}
    valid = ranks > 0
    r = ranks.double()

    def row_sum(x):
        return torch.zeros(n, dtype=torch.float64, device=dev).index_add_(0, rows, x.double())

    def mean(x, sel):
        return float(x[sel].mean()) if bool(sel.any()) else 0.0

    inf = float("inf")
    best = torch.full((n,), inf, dtype=torch.float64, device=dev).scatter_reduce(
        0, rows, torch.where(valid, r, torch.full_like(r, inf)), "amin")
    max_m = int(m.max()) if n else 0
    for k in ks:
        hit = valid & (ranks <= k)
        disc = 1.0 / torch.log2(torch.arange(2, max(min(max_m, k), 1) + 2, dtype=torch.float64, device=dev))
        idcg = torch.cumsum(disc, 0)[(torch.clamp(m, max=k) - 1).clamp_min(0)]
        out[f"hr@{k}"] = mean((best <= k).double(), has)
        out[f"recall@{k}"] = mean(row_sum(hit) / m.clamp_min(1), has)
        out[f"ndcg@{k}"] = mean(row_sum(torch.where(hit, 1.0 / torch.log2(r + 1), torch.zeros_like(r))) / idcg, has)
    out["mrr"] = mean(1.0 / best, has)                                  # 1 / inf = 0 for rows without a ranked target
    # other targets of the row above t: its position among the row's ranked targets (ranks within a row are distinct)
    vrow = rows[valid]
    order = torch.argsort(vrow * (int(ranks.max()) + 1) + ranks[valid]) if vrow.numel() else vrow
    vcount = torch.bincount(vrow, minlength=n)
    vstart = torch.cumsum(vcount, 0) - vcount
    above = torch.empty_like(vrow)
    above[order] = torch.arange(vrow.numel(), device=dev) - vstart[vrow[order]]
    neg = (n_cand - m).double()
    term = torch.zeros_like(r)
    term[valid] = 1.0 - (r[valid] - 1 - above.double()) / neg[vrow].clamp_min(1)
    out["auc"] = mean(row_sum(term) / m.clamp_min(1), has & (n_cand > m))
    out["n_rows"] = n_rows
    return out
