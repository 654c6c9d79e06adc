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
  SimpleSiamese  the entity's reviews, masked average pooling (K9), the optional latent transform and the review attention
            (SimpleSiamese.encode_side) → [U, F] / [I, F]; pairs score through the model's own head (K4 where it is fused).

`PairScorer.recommend` answers "the k best items for these users out of the whole catalogue" with K10 (ops.factor_topk),
which never materialises the users x items score matrix; `rank_items` / `evaluate` give the exact full-catalogue rank of
held-out items and HR@k / Recall@k / NDCG@k / MRR / AUC from it with K11 (ops.factor_rank), on the same scores;
`recommend_diverse` re-ranks recommend's top-P by maximal marginal relevance over item-vector similarity with K14
(ops.mmr_select), and `list_metrics` gives the lists' intra-list diversity and catalogue coverage.  `add` / `update` grow
the cache by new entities (served under the side's padding id through a row -> model-id map) and re-encode changed ones in
place, encoding and re-deriving only those rows (DESIGN.md §5).  The FM head factorises
exactly:
  relu(u*i) = relu(u)*relu(i) + relu(-u)*relu(-i)   ⇒   score(u,i) = A[u] . B[i] + row_bias[u] + col_bias[i]
with A = [h*relu(u_lat), h*relu(-u_lat)], B = [relu(i_lat), relu(-i_lat)], row_bias = ub + g, col_bias = ib (fm_factors);
D-ATT's score is already a dot product of the two FC outputs.
"""
from __future__ import annotations

import functools
from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from . import ops
from .deepconn import DeepCoNNpp
from .dual_att import DualAtt
from .layers import FM, fused_head, head_params
from .narre import NARRE
from .simple_siamese import SimpleSiamese


def fm_factors(u_lat: torch.Tensor, i_lat: torch.Tensor, h: torch.Tensor, user_bias: torch.Tensor, item_bias: torch.Tensor,
               g_bias: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """FM head (models/deepconn/layers.py:200-207) as a factor product: score(u, i) = A[u] . B[i] + row_bias[u] + col_bias[i]
    for latents u_lat [U, K], i_lat [I, K] (LastFeat outputs of entity rows u / i), h [K, 1], user_bias [U, 1],
    item_bias [I, 1], g_bias [1].  Returns (A [U, 2K], row_bias [U], B [I, 2K], col_bias [I]) in the inputs' dtype."""
    hv = h.reshape(1, -1)
    A = torch.cat([hv * torch.relu(u_lat), hv * torch.relu(-u_lat)], dim=1)
    B = torch.cat([torch.relu(i_lat), torch.relu(-i_lat)], dim=1)
    return A, user_bias.reshape(-1) + g_bias.reshape(()), B, item_bias.reshape(-1)


SIDES = ("user", "item")
_CHUNK = 4096                   # entities per encoder launch in add / update (build_cache's default chunk)


def _reserve(buf: torch.Tensor, used: int, need: int) -> torch.Tensor:
    """buf if it has `need` rows, else a new buffer of max(need, 2 x its rows) rows holding its first `used` rows: a run of
    appends copies O(total) rows."""
    if buf.shape[0] >= need:
        return buf
    out = buf.new_empty((max(need, 2 * buf.shape[0]),) + tuple(buf.shape[1:]))
    out[:used] = buf[:used]
    return out


class _Side:
    """One side of the feature cache.  Every per-entity tensor lives in a buffer with spare rows (`bufs`; "cached" = the
    cached features, "model_ids" = the row -> model-id map, the rest build_cache(explain=True)'s tensors, `per[key]` rows of
    it per entity); the first n entities are in use.  `log` holds (generation, rows) of every add / update since the
    derived caches (factors, unit item vectors) last took them in.  `shape` is the documents' shape past the entity axis
    (None when the features were assigned, not built from documents)."""

    def __init__(self, feat: torch.Tensor, kept: Optional[dict] = None, shape: Optional[tuple] = None):
        n = feat.shape[0]
        self.n = self.n_built = n
        self.shape = None if shape is None else tuple(shape)
        self.bufs = {"cached": feat, "model_ids": torch.arange(n, device=feat.device), **(kept or {})}
        self.kept = None if kept is None else list(kept)
        self.per = {k: 1 if t is None or not n else t.shape[0] // n for k, t in self.bufs.items()}
        self.caller_owned = {"docs", "masks"}      # build_cache keeps references to the caller's documents and masks
        self.gen, self.log = 0, []

    def view(self, key: str) -> Optional[torch.Tensor]:
        t = self.bufs[key]
        return None if t is None else t[:self.n * self.per[key]]

    def write(self, rows: Optional[torch.Tensor], new: dict) -> None:
        """Entity rows `rows` (None: append) <- new {key: rows of that buffer}; a caller's tensor is copied on the first
        write, never written."""
        need = self.n + (new["cached"].shape[0] if rows is None else 0)
        for k, v in new.items():
            buf, p = self.bufs[k], self.per[k]
            if k in self.caller_owned:
                buf = buf[:self.n * p].clone(memory_format=torch.contiguous_format)
                self.caller_owned.discard(k)
            buf = _reserve(buf, self.n * p, need * p)
            if rows is None:
                buf[self.n * p:need * p] = v
            else:
                at = rows if p == 1 else (rows.view(-1, 1) * p + torch.arange(p, device=rows.device)).view(-1)
                buf.index_copy_(0, at, v.to(buf.dtype))
            self.bufs[k] = buf
        if rows is None:
            rows = torch.arange(self.n, need, device=new["cached"].device)
        self.n = need
        self.gen += 1
        self.log.append((self.gen, rows))

    def changed(self, since: int) -> Optional[torch.Tensor]:
        """The rows added or updated after generation `since`, ascending; None if there are none."""
        rows = [r for g, r in self.log if g > since]
        return torch.unique(torch.cat(rows)) if rows else None


class PairScorer:
    def __init__(self, model):
        if not isinstance(model, (DeepCoNNpp, NARRE, DualAtt, SimpleSiamese)):
            raise TypeError("PairScorer serves DeepCoNNpp, NARRE, DualAtt and SimpleSiamese")
        self.model = model.eval()
        self._sides = dict.fromkeys(SIDES)   # name -> _Side
        self._factors = None         # dict: head-parameter key, per side the generation and rows taken in, factor buffers
        self._unit_items = None      # dict: source key (None: the cached item features), unit-normalised item vectors

    def _get_feat(self, name):
        s = self._sides[name]
        return None if s is None else s.view("cached")

    def _set_feat(self, name, feat):
        self._sides[name] = None if feat is None else _Side(feat)
        self._factors = self._unit_items = None

    user_feat = property(lambda self: self._get_feat("user"), lambda self, t: self._set_feat("user", t),
                         doc="The cached user features [U, D] (row e = cache row e)")
    item_feat = property(lambda self: self._get_feat("item"), lambda self, t: self._set_feat("item", t),
                         doc="The cached item features [I, D]")

    @property
    def _explain(self) -> Optional[dict]:
        """Per side, the per-entity tensors build_cache(explain=True) keeps (views of the rows in use), or None."""
        if any(s is None or s.kept is None for s in self._sides.values()):
            return None
        return {name: {k: s.view(k) for k in s.kept} for name, s in self._sides.items()}

    @torch.no_grad()
    def score_pairs(self, *inputs) -> torch.Tensor:
        """The reference's per-pair data flow: both sides encoded for every pair (the model's own eval forward)."""
        out = self.model(*inputs)
        return out[0] if isinstance(out, tuple) else out

    @torch.no_grad()
    def build_cache(self, user_docs: torch.Tensor, item_docs: torch.Tensor, user_masks: Optional[torch.Tensor] = None,
                    item_masks: Optional[torch.Tensor] = None, chunk: int = 4096, *, user_rev_ids: Optional[torch.Tensor] = None,
                    item_rev_ids: Optional[torch.Tensor] = None, user_rev_masks: Optional[torch.Tensor] = None,
                    item_rev_masks: Optional[torch.Tensor] = None, explain: bool = False) -> None:
        """Row e of every argument belongs to entity id e (row 0 = the padding entity).
        DeepCoNN: user_docs [U, L], item_docs [I, L]; masks default to ids != 0 (utils.py:30-42).
        NARRE: user_docs [U, R, T], item_docs [I, R, T] (the entity's reviews), optional masks of the same shapes, and
          user_rev_ids [U, R] / item_rev_ids [I, R]: the ids of the items a user reviewed / the users who reviewed an item —
          what NARRE's dataset supplies as reuid / reiid for a pair with that entity.
        D-ATT: user_docs [U, L], item_docs [I, L] (no masks).
        SimpleSiamese: user_docs [U, R_u, T], item_docs [I, R_i, T] (the entity's reviews; R_u and R_i may differ), optional
          word masks of the same shapes (default ids != 0) and user_rev_masks [U, R_u] / item_rev_masks [I, R_i] (default:
          the review has a masked-in word, models/simple_siamese/utils.py get_rev_mask).
        Each side is encoded in chunks of `chunk` documents (review models: chunk // R entities of R reviews).
        explain=True also keeps what `explain` needs per entity (references to the documents and masks; for DeepCoNN and
        NARRE the conv arg-max and the tap contributions of every pooled window (K12a), for NARRE the per-review features
        and attention weights; for D-ATT the two K5 gates, the conv arg-max, the FC hidden ReLU mask and the per-entity
        terms of gradient x input, rbr_datt_explain_contrib; for SimpleSiamese the attention's inputs v, weights s and
        logit gradients a (K13), and the LastFeat outputs where the head is not fused).  The cached features are the same
        either way."""
        m = self.model
        m.eval()
        # per side: (documents, masks, the model's per-review input: NARRE's review ids, SimpleSiamese's review masks)
        sides = {"user": (user_docs, user_masks, None), "item": (item_docs, item_masks, None)}
        if isinstance(m, SimpleSiamese):
            sides = {"user": (user_docs, user_masks, user_rev_masks), "item": (item_docs, item_masks, item_rev_masks)}
            for name, (docs, wm, rm) in sides.items():
                if (docs.dim() != 3 or (wm is not None and tuple(wm.shape) != tuple(docs.shape))
                        or (rm is not None and tuple(rm.shape) != tuple(docs.shape[:2]))):
                    raise ValueError(f"SimpleSiamese takes {name}_docs [n, R, T] with word masks [n, R, T] and review masks "
                                     f"[n, R], got {tuple(docs.shape)} / {None if wm is None else tuple(wm.shape)} / "
                                     f"{None if rm is None else tuple(rm.shape)}")
        elif isinstance(m, DualAtt):
            if user_masks is not None or item_masks is not None:
                raise ValueError("DualAtt takes no masks")
            for docs in (user_docs, item_docs):
                if docs.shape[-1] != m.doc_len:
                    raise ValueError(f"DualAtt was built for doc_len={m.doc_len}, got {docs.shape[-1]} "
                                     "(the global attention kernel spans the whole document)")
        elif explain and m.ngram.arch != "CNN":
            raise NotImplementedError("PairScorer.explain covers the CNN encoder; arch='HierPooling' pools averages, "
                                      "which have no per-window tap contributions")
        elif isinstance(m, NARRE):
            if user_rev_ids is None or item_rev_ids is None:
                raise ValueError("NARRE's build_cache needs user_rev_ids [U, R] and item_rev_ids [I, R]")
            sides = {"user": (user_docs, user_masks, user_rev_ids), "item": (item_docs, item_masks, item_rev_ids)}
            for docs, _, rev_ids in sides.values():
                if docs.shape[1:] != (m.doc_num, m.doc_len) or rev_ids.shape != docs.shape[:2]:
                    raise ValueError(f"NARRE was built for [*, {m.doc_num}, {m.doc_len}] reviews with [*, {m.doc_num}] review "
                                     f"ids, got {tuple(docs.shape)} / {tuple(rev_ids.shape)}")
        encode = self._encoder(explain)
        feats, kept = {}, {}
        for name, (docs, masks, rev) in sides.items():
            feats[name], kept[name] = self._encode_rows(encode, name, explain, docs, masks, rev, chunk)
        if explain and isinstance(m, SimpleSiamese) and not ops.head_supported(feats["user"].shape[1], m.fm.h.shape[0]):
            for name in SIDES:
                kept[name]["lat"] = self._latent64(name, feats[name]).float()
        for name in SIDES:
            self._sides[name] = _Side(feats[name], kept[name], sides[name][0].shape[1:])
        self._factors = self._unit_items = None

    def _encoder(self, explain: bool):
        """The model's chunk encoder (below)."""
        m = self.model
        if isinstance(m, SimpleSiamese):
            return functools.partial(self._encode_siamese, att64=self._siamese_att64() if explain else None)
        if isinstance(m, DualAtt):
            return self._encode_datt
        return self._encode_narre if isinstance(m, NARRE) else self._encode_deepconn

    @staticmethod
    def _encode_rows(encode, name, explain, docs, masks, rev, chunk):
        """One side's entities through `encode` in chunks of `chunk` documents (review models: chunk // R entities) →
        (cached features, None or with explain the per-entity explain tensors with the documents and masks)."""
        step = max(1, chunk // docs.shape[1]) if docs.dim() == 3 else chunk
        parts = [encode(name, explain, *(None if t is None else t[lo:lo + step] for t in (docs, masks, rev)))
                 for lo in range(0, docs.shape[0], step)]
        feat = torch.cat([f for f, _ in parts])
        if not explain:
            return feat, None
        return feat, {"docs": docs, "masks": masks, **{k: torch.cat([x[k] for _, x in parts]) for k in parts[0][1]}}

    @torch.no_grad()
    def add(self, side: str, docs: torch.Tensor, masks: Optional[torch.Tensor] = None, *,
            rev_ids: Optional[torch.Tensor] = None, rev_masks: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Encode new entities on `side` ("user" / "item") from their documents and append them to the cache; returns their
        cache rows (int64, from the current row count up), which every serving method takes as ids from then on.
        docs, masks, rev_ids / rev_masks: what build_cache takes for that side and model, for the new entities only.  A new
        entity has no row in the model's ID tables: it is served under the side's padding id (DeepCoNN / NARRE:
        fm.padding_idx / fm.item_padding_idx, SimpleSiamese 0; D-ATT has no ids), i.e. exactly as the model's eval forward
        scores the same documents under that id.  NARRE's rev_ids are MODEL ids of the counterparts, as K3 gathers them from
        ebd_vals: a review by a counterpart the model has no id for is given as the padding id.  With an explain cache the
        new rows' explain tensors are appended too.  Nothing is written when a check fails."""
        s = self._check_rows(side, None, docs, masks, rev_ids, rev_masks)
        n = docs.shape[0]
        if not n:
            return torch.empty(0, dtype=torch.int64, device=s.bufs["cached"].device)
        pad = 0 if isinstance(self.model, (DualAtt, SimpleSiamese)) else (
            self.model.fm.padding_idx if side == "user" else self.model.fm.item_padding_idx)
        mids = torch.full((n,), pad, dtype=torch.int64, device=s.bufs["cached"].device)
        new = self._encode_new(side, s, docs, masks, rev_ids, rev_masks, mids)
        new["model_ids"] = mids
        first = s.n
        s.write(None, new)
        self._trim(side)
        return torch.arange(first, s.n, device=mids.device)

    @torch.no_grad()
    def update(self, side: str, ids: torch.Tensor, docs: torch.Tensor, masks: Optional[torch.Tensor] = None, *,
               rev_ids: Optional[torch.Tensor] = None, rev_masks: Optional[torch.Tensor] = None) -> None:
        """Re-encode the cached entities `ids` (distinct cache rows) on `side` from new documents, in place: e.g. after a
        user posted a review, or to refresh an entity cached with stale text.  Their model ids are kept.  Inputs as for
        `add`, one entity per id.  Only these rows are encoded, and factors() / recommend_diverse's item vectors then
        re-derive only these rows.  The caller's tensors that build_cache(explain=True) kept are copied, never written."""
        s = self._check_rows(side, ids, docs, masks, rev_ids, rev_masks)
        ids = ids.to(device=s.bufs["cached"].device, dtype=torch.int64).reshape(-1)
        if not ids.numel():
            return
        s.write(ids, self._encode_new(side, s, docs, masks, rev_ids, rev_masks, s.view("model_ids").index_select(0, ids)))
        self._trim(side)

    def _check_rows(self, side, ids, docs, masks, rev_ids, rev_masks) -> _Side:
        """add / update's checks of the caller's input (ValueError before anything is launched) → the side."""
        m = self.model
        if side not in SIDES:
            raise ValueError(f"side must be 'user' or 'item', got {side!r}")
        s = self._sides[side]
        if s is None or s.shape is None:
            raise ValueError("PairScorer.build_cache(...) first: add / update extend a cache built from documents")
        dev = s.bufs["cached"].device
        if (not isinstance(docs, torch.Tensor) or docs.device != dev or docs.dim() != len(s.shape) + 1
                or tuple(docs.shape[1:]) != s.shape or docs.is_floating_point()):
            raise ValueError(f"{side} documents must be a [n, {', '.join(map(str, s.shape))}] tensor on {dev} (the cached "
                             f"side's shape), got {tuple(docs.shape) if isinstance(docs, torch.Tensor) else type(docs).__name__}")
        n = docs.shape[0]
        if masks is not None and (isinstance(m, DualAtt) or not isinstance(masks, torch.Tensor)
                                  or masks.device != dev or masks.shape != docs.shape):
            raise ValueError(f"masks must be None or of the documents' shape {tuple(docs.shape)} on {dev}"
                             + (" (DualAtt takes no masks)" if isinstance(m, DualAtt) else ""))
        for name, t, ok in (("rev_ids", rev_ids, isinstance(m, NARRE)), ("rev_masks", rev_masks, isinstance(m, SimpleSiamese))):
            if t is None and not (ok and name == "rev_ids"):
                continue
            if not ok:
                raise ValueError(f"{type(m).__name__} takes no {name}")
            if not isinstance(t, torch.Tensor) or t.device != dev or tuple(t.shape) != tuple(docs.shape[:2]):
                raise ValueError(f"{name} must be a [{n}, {s.shape[0]}] tensor on {dev}, got "
                                 f"{tuple(t.shape) if isinstance(t, torch.Tensor) else type(t).__name__}")
        if isinstance(m, NARRE) and rev_ids.numel():
            n_other = (m.user_att if side == "user" else m.item_att).ebd_vals.weight.shape[0]
            lo, hi = torch.stack([rev_ids.min(), rev_ids.max()]).tolist()
            if lo < 0 or hi >= n_other:
                raise ValueError(f"rev_ids are model ids of the counterparts and must lie in [0, {n_other}) (a counterpart "
                                 f"the model has no id for is given as the padding id), got [{lo}, {hi}]")
        if not isinstance(m, DualAtt):
            n_ids = self._last_feats()[side == "item"].ebd.weight.shape[0]
            if s.n_built > n_ids:
                raise ValueError(f"the {side} cache was built with {s.n_built} rows, more than the model's {n_ids} ids")
        if ids is not None:
            if not isinstance(ids, torch.Tensor) or ids.dim() != 1 or ids.numel() != n or ids.is_floating_point():
                raise ValueError(f"ids must be a 1-D integer tensor with one id per document ({n}), got "
                                 f"{tuple(ids.shape) if isinstance(ids, torch.Tensor) else type(ids).__name__}")
            if n:
                lo, hi = torch.stack([ids.min(), ids.max()]).tolist()
                if lo < 0 or hi >= s.n:
                    raise ValueError(f"ids must lie in [0, {s.n}) (the cached {side} rows), got [{lo}, {hi}]")
                if torch.unique(ids).numel() != n:
                    raise ValueError("ids must be distinct")
        return s

    def _encode_new(self, side, s, docs, masks, rev_ids, rev_masks, mids) -> dict:
        """The chunk encoder on new documents of entities with model ids `mids` → {buffer key: new rows} for _Side.write."""
        m = self.model
        m.eval()
        explain = s.kept is not None
        rev = rev_ids if isinstance(m, NARRE) else rev_masks
        feat, kept = self._encode_rows(self._encoder(explain), side, explain, docs, masks, rev, _CHUNK)
        new = {"cached": feat}
        if explain:
            if kept["masks"] is None and s.bufs["masks"] is not None:
                kept["masks"] = docs != 0                               # the default mask, as the encoder took it
            elif kept["masks"] is not None and s.bufs["masks"] is None:
                s.bufs["masks"] = s.view("docs") != 0                   # the cached rows' default masks, materialised
                s.per["masks"], s.caller_owned = s.per["docs"], s.caller_owned - {"masks"}
            if kept["masks"] is None:
                del kept["masks"]
            if "lat" in s.kept:
                kept["lat"] = self._latent64(side, feat, mids).float()
            new.update(kept)
        return new

    def _trim(self, name):
        """Drop the change-log entries that every derived cache has taken in."""
        s = self._sides[name]
        gens = [] if self._factors is None else [self._factors["gen"][name]]
        if name == "item" and self._unit_items is not None and self._unit_items["key"] is None:
            gens.append(self._unit_items["gen"])
        lo = min(gens, default=s.gen)
        s.log = [(g, r) for g, r in s.log if g > lo]

    # build_cache's chunk encoders, one per model: (side, explain, documents, masks, per-review input) of a chunk of entities
    # → (the entities' cached features, None or with explain a dict of their per-entity explain tensors)

    def _encode_deepconn(self, side, explain, docs, masks, _):
        m = self.model
        out = m.ngram.encode(m.word_embeddings, [docs], [masks], return_argmax=explain)      # (HierPooling: no arg-max)
        if not explain:
            return out[0], None
        feat, amax = out
        return feat, {"feat": feat, "argmax": amax, "contrib": self._window_contrib(docs, masks, amax)}

    def _encode_narre(self, side, explain, docs, masks, rev_ids):
        m = self.model
        n, R, T = docs.shape
        docs = docs.reshape(-1, T)
        masks = None if masks is None else masks.reshape(-1, T)
        out = m.ngram.encode(m.word_embeddings, [docs], [masks], return_argmax=explain)
        feat, att = (m.user_att if side == "user" else m.item_att)(out[0].view(n, R, -1), rev_ids)
        if not explain:
            return feat, None
        return feat, {"rev_ids": rev_ids, "feat": out[0], "argmax": out[1], "att": att.view(-1, R),
                      "contrib": self._window_contrib(docs, masks, out[1])}

    def _encode_datt(self, side, explain, docs, masks, _):
        """The encoder (ops.datt_encode_side, the kernels DualAtt.encode runs), then the FC stack layer by layer (the modules
        of m.fc in its order) to keep its hidden ReLU mask; with explain K12's per-entity terms (ops.datt_explain_contrib)."""
        m = self.model
        table = m.word_embeddings.embedding.weight.detach()
        shadow = m.word_embeddings.bf16_shadow() if m.precision == "bf16" else None
        prm = m.side_params("u" if side == "user" else "i")
        packed = ops.datt_side_packs(prm)
        feat, amax, _, gl, gg = ops.datt_encode_side(table, docs, prm, m.precision, shadow, packed, conv_flags=m.conv_flags)
        lin0, relu, drop, lin1 = m.fc
        hid = lin0(feat)
        out = lin1(drop(relu(hid)))
        if not explain:
            return out, None
        contrib, coef, vec = ops.datt_explain_contrib(table, docs, prm, gl, gg, feat, amax, packed)
        return out, {"gate_l": gl, "gate_g": gg, "argmax": amax, "contrib": contrib, "gate_coef": coef, "gate_vec": vec,
                     "hid_mask": hid > 0}

    def _encode_siamese(self, side, explain, docs, masks, rev_masks, att64):
        """SimpleSiamese.encode_side; explain also keeps per entity the attention's inputs v [R, F] and weights s [R], and
        a = P^T (w * (1 - tanh^2(P v + c))) [R, F] (zero for a masked review; in float64, then fp32)."""
        rm = ((docs != 0) if masks is None else masks).any(-1) if rev_masks is None else rev_masks
        feat, s, v = self.model.encode_side(docs, masks, rm)
        if not explain:
            return feat, None
        P, c, w = att64
        th = torch.tanh(v.double() @ P.t() + c)
        return feat, {"v": v.contiguous(), "att": s.reshape(-1, docs.shape[1]),
                      "a": (((w * (1 - th * th)) @ P) * rm.unsqueeze(-1)).float()}

    def _siamese_att64(self):
        """(P, c, w) of SimpleSiamese's review attention in float64."""
        att = self.model.review_att_layer
        proj = att.proj_layer[0]
        return proj.weight.detach().double(), proj.bias.detach().double(), att.inner_product.weight.detach().double().view(-1)

    def _conv_specs(self):
        conv = self.model.ngram.conv
        return [(c.weight.shape[0], k, (k - 1) // 2) for c, k in zip(conv.list_of_conv1d, conv.kernel_sizes)]

    def _window_contrib(self, docs: torch.Tensor, masks: Optional[torch.Tensor], argmax: torch.Tensor) -> torch.Tensor:
        """K12a: the tap contributions [N, sum_c H_c * k_c] of every pooled window of docs [N, L] at the arg-max."""
        m = self.model
        conv = m.ngram.conv
        table = m.word_embeddings.embedding.weight.detach()
        specs = self._conv_specs()
        contrib = torch.empty(docs.shape[0], sum(h * k for h, k, _ in specs), dtype=torch.float32, device=table.device)
        col = tcol = 0
        for i, (h, k, pad) in enumerate(specs):
            ops.conv_window_contrib(table, docs, masks, conv.list_of_conv1d[i].weight.detach(), pad, argmax[:, col:col + h],
                                    packed=conv.packed(i), mask_from_ids=True, out=contrib[:, tcol:tcol + h * k])
            col += h
            tcol += h * k
        return contrib

    def _siamese_fused_g(self) -> bool:
        """Whether g = d pred / d feat comes from K4's backward (ops.head_text_grads) rather than from K13 itself."""
        return ops.head_supported(self.user_feat.shape[1], self.model.fm.h.shape[0])

    @torch.no_grad()
    def score_cached(self, u_ids: torch.Tensor, i_ids: torch.Tensor) -> torch.Tensor:
        """preds for pairs (u_ids[b], i_ids[b]) from the cached features, no encoder: K1 row gather + K4 head (DeepCoNN,
        NARRE) or K1 + dot product (D-ATT, dual_att.py:59-61)."""
        if self.user_feat is None:
            raise RuntimeError("PairScorer.build_cache(...) first")
        m = self.model
        u_text = ops.gather_rows(self.user_feat, u_ids)
        i_text = ops.gather_rows(self.item_feat, i_ids)
        if not u_text.shape[0]:                 # no pairs (K4 takes batches of at least one)
            return u_text.new_empty(0)
        if isinstance(m, DualAtt):
            return torch.sum(torch.mul(u_text, i_text), 1).view(-1)
        u_ids, i_ids = self._model_ids("user", u_ids), self._model_ids("item", i_ids)
        if isinstance(m, SimpleSiamese):
            return m.head(u_text, i_text, u_ids, i_ids).view(-1)
        return fused_head(m.user_feat, m.item_feat, m.fm, u_text, i_text, u_ids, i_ids, False, None).view(-1)

    def _model_ids(self, name: str, rows: torch.Tensor) -> torch.Tensor:
        """The model ids of cache rows `rows` (the row -> model-id map); a row outside the cache passes unchanged (K1 reads
        it as a zero row, K4 as an id outside its tables, as without the map)."""
        s = self._sides[name]
        if s.n == s.n_built:                     # rows build_cache wrote map to themselves
            return rows
        inside = (rows >= 0) & (rows < s.n)
        return torch.where(inside, s.view("model_ids").index_select(0, rows.clamp(0, s.n - 1)), rows)

    def _last_feats(self):
        m = self.model
        return (m.user_last_feat_layer, m.item_last_feat_layer) if isinstance(m, SimpleSiamese) else (m.user_feat, m.item_feat)

    def _head_params(self):
        """K4's parameters for the model's head in layers.head_params' order (D-ATT: none)."""
        m = self.model
        return [] if isinstance(m, DualAtt) else head_params(*self._last_feats(), m.fm)[0]

    def _latent64(self, name: str, feat: torch.Tensor, mids: Optional[torch.Tensor] = None) -> torch.Tensor:
        """LastFeat (models/deepconn/layers.py:163) in float64 of `name`-side features feat [n, H] of entities with model ids
        `mids` (None: rows 0..n-1) → [n, K]: exact fp32 latents whatever the TF32 setting."""
        lf = self._last_feats()[name == "item"]
        ebd = lf.ebd.weight.detach().double()
        return (feat.double() @ lf.W.detach().double() + lf.b.detach().double()
                + (ebd[:feat.shape[0]] if mids is None else ebd.index_select(0, mids)))

    def factors(self) -> Tuple[torch.Tensor, Optional[torch.Tensor], torch.Tensor, Optional[torch.Tensor]]:
        """(A [U, D], row_bias [U] or None, B [I, D], col_bias [I] or None) with score(u, i) = A[u] . B[i] + biases for the
        cached entities under the CURRENT head parameters, each row from its entity's model id (the row -> model-id map).
        Re-derived when a parameter changed (optimizer steps bump its version counter) or the cache was rebuilt; after
        add / update only the added and updated rows are derived (the same float64 expression, row by row)."""
        if self.user_feat is None:
            raise RuntimeError("PairScorer.build_cache(...) first")
        m = self.model
        if isinstance(m, DualAtt):
            return self.user_feat, None, self.item_feat, None
        key = tuple((p._version, p.data_ptr()) for p in self._head_params() if p is not None)
        f = self._factors
        full = f is None or f["key"] != key
        rows = dict.fromkeys(SIDES) if full else {name: self._sides[name].changed(f["gen"][name]) for name in SIDES}
        if full or any(r is not None for r in rows.values()):
            with torch.no_grad():
                lat, bias = {}, {}
                fm = m.fm
                for name, tab in zip(SIDES, (getattr(fm, "user_bias", None), getattr(fm, "item_bias", None))):
                    s, r = self._sides[name], rows[name]
                    mids = None if s.n == s.n_built else s.view("model_ids")
                    feat = s.view("cached")
                    if not full:
                        r = r if r is not None else torch.empty(0, dtype=torch.int64, device=feat.device)
                        feat, mids = feat.index_select(0, r), (r if mids is None else mids.index_select(0, r))
                    lat[name] = self._latent64(name, feat, mids)
                    if isinstance(fm, FM):                   # FMWithoutUIBias: row_bias = g_bias, no column bias
                        w = tab.weight.detach().double()
                        bias[name] = w[:feat.shape[0]] if mids is None else w.index_select(0, mids)
                    else:
                        bias[name] = lat[name].new_zeros(feat.shape[0], 1)
                new = [t.float().contiguous() for t in fm_factors(lat["user"], lat["item"], fm.h.detach().double(), bias["user"],
                                                                  bias["item"], fm.g_bias.detach().double())]
                if not isinstance(fm, FM):
                    new[3] = None
            if full:
                f = {"key": key, "user": new[:2], "item": new[2:]}
            else:
                for name, vals in (("user", new[:2]), ("item", new[2:])):
                    if rows[name] is None:
                        continue
                    n = self._sides[name].n
                    for j, v in enumerate(vals):
                        if v is not None:
                            f[name][j] = _reserve(f[name][j], f["n"][name], n)
                            f[name][j].index_copy_(0, rows[name], v)
            f["n"] = {name: self._sides[name].n for name in SIDES}
            f["gen"] = {name: self._sides[name].gen for name in SIDES}
            self._factors = f
            for name in SIDES:
                self._trim(name)
        f = self._factors
        n_u, n_i = f["n"]["user"], f["n"]["item"]
        return tuple(None if t is None else t[:n] for t, n in zip(f["user"] + f["item"], (n_u, n_u, n_i, n_i)))

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

    @torch.no_grad()
    def recommend_diverse(self, u_ids: torch.Tensor, k: int, lam: float = 0.5, pool: Optional[int] = None,
                          exclude: Optional[Tuple[torch.Tensor, torch.Tensor]] = None, exclude_padding: bool = True,
                          item_vecs: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """k items per user u_ids[r], relevant and not redundant: maximal marginal relevance (K14, ops.mmr_select) over the
        pool recommend(u_ids, pool, exclude, exclude_padding) (K10; default pool = min(256, 4 k)).  Step 0 takes the pool's
        best item; each later step the eligible unpicked item with the largest lam * rel - (1 - lam) * max sim to the items
        picked so far, rel = the score min-max scaled over the row's pool, sim = the cosine of the items' vectors: item_vecs
        [I, D] (default: the cached item features; e.g. factors()[2]), rows unit-normalised once (a zero row has sim 0 to
        everything).  Returns (scores [len(u_ids), k] fp32, items [len(u_ids), k] int64) in selection order; the scores are
        recommend's, bit for bit, and rows with fewer than k eligible items end in (-inf, -1).  lam = 1 is recommend(u_ids,
        k); pool = k gives a permutation of it.  Results do not depend on the other rows of the call."""
        k = int(k)
        pool = min(ops.MMR_MAX_POOL, 4 * k) if pool is None else int(pool)
        lam = float(lam)
        vecs = self._unit_item_vecs(item_vecs)
        if not 0.0 <= lam <= 1.0:
            raise ValueError(f"lam must lie in [0, 1], got {lam}")
        if not ops.mmr_supported(pool, vecs.shape[1], k):
            raise ValueError(f"recommend_diverse takes 1 <= k <= pool <= {ops.MMR_MAX_POOL} and item vectors of at most "
                             f"{ops.MMR_MAX_DIM} columns (got k={k}, pool={pool}, dim={vecs.shape[1]})")
        A_rows, rb_rows, B, cb, _ = self._user_rows(u_ids, exclude_padding)
        pool_scores, pool_items = ops.factor_topk(A_rows, rb_rows, B, cb, pool, exclude=exclude)
        return ops.mmr_select(pool_scores, pool_items, vecs, k, lam)

    def _unit_item_vecs(self, item_vecs: Optional[torch.Tensor]) -> torch.Tensor:
        """ops.unit_rows of item_vecs (default: the cached item features), kept until the source changes.  The default
        source follows the item side's change log, so add / update normalise only their rows; a caller's tensor is keyed
        by its data pointer, layout and version counter, and referenced so that the pointer cannot be reused."""
        if self.item_feat is None:
            raise RuntimeError("PairScorer.build_cache(...) first")
        if item_vecs is None:
            s, u = self._sides["item"], self._unit_items
            if u is None or u["key"] is not None:
                u = {"key": None, "vecs": ops.unit_rows(self.item_feat).contiguous()}
            else:
                rows = s.changed(u["gen"])
                if rows is not None:
                    u["vecs"] = _reserve(u["vecs"], u["n"], s.n)
                    u["vecs"].index_copy_(0, rows, ops.unit_rows(self.item_feat.index_select(0, rows)))
            u["n"], u["gen"] = s.n, s.gen
            self._unit_items = u
            self._trim("item")
            return u["vecs"][:u["n"]]
        src = item_vecs
        if not isinstance(src, torch.Tensor) or src.dim() != 2 or src.shape[0] != self.item_feat.shape[0]:
            raise ValueError(f"item_vecs must be [{self.item_feat.shape[0]}, D] (one row per cached item), got "
                             f"{tuple(src.shape) if isinstance(src, torch.Tensor) else type(src).__name__}")
        if src.device != self.item_feat.device:
            raise ValueError(f"item_vecs is on {src.device}, the cache on {self.item_feat.device}")
        key = (src.data_ptr(), tuple(src.shape), src.stride(), src.dtype, src._version)
        if self._unit_items is None or self._unit_items["key"] != key:
            self._unit_items = {"key": key, "src": src, "vecs": ops.unit_rows(src).contiguous()}
        return self._unit_items["vecs"]

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
            pad = 0 if isinstance(self.model, (DualAtt, SimpleSiamese)) else self.model.fm.item_padding_idx
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
        dense term; the default width is the local window size.  SimpleSiamese: gradient x input through the masked average
        pooling, the latent transform and the review attention (K13, DESIGN.md), g from K4's backward where the head is
        fused, else from the cached LastFeat outputs at the FM's ReLU decision; the outputs are NARRE's (map [B, R, T],
        review_weight, review_attr) and the default width is 1, the token (the model is a bag of words per review).
        Positions are flat (NARRE, SimpleSiamese: r * T + t); `tokens_at` turns them into ids.  Pairs run in chunks of
        `chunk`, so scratch memory does not grow with B."""
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
        cache = self._explain
        if isinstance(mdl, DualAtt) and not attribution:
            L = mdl.doc_len
            if not 1 <= m <= L:
                raise ValueError(f"m must lie in [1, {L}]")
            sides = []
            for name, ids in (("user", u_ids), ("item", i_ids)):
                gl = cache[name]["gate_l"].index_select(0, ids)
                # stable sort: equal gates keep the lower position first
                order = torch.sort(gl, dim=1, descending=True, stable=True).indices[:, :m]
                sides.append(SideExplanation(local_att=gl, global_att=cache[name]["gate_g"].index_select(0, ids), top_pos=order,
                                             top_attr=gl.gather(1, order)))
            return Explanation(pred, *sides)

        # per model: the default width, whether the kernels take (m, width), g_u, g_i = grads(u, i) for a chunk of pairs, g0 =
        # an empty g, and attrib(side, ids, other side's ids, g) → explain_attrib's dict
        if isinstance(mdl, SimpleSiamese):
            table = mdl.word_embedding.embedding.weight.detach()
            lt_w = mdl.latent_transform_layer[0].weight.detach() if mdl.latent_transform else None
            last = dict(zip(("user", "item"), self._last_feats()))
            feats = {"user": self.user_feat, "item": self.item_feat}
            width = 1 if width is None else int(width)
            ok = all(ops.explain_avgpool_supported(R * T, R, table.shape[1], self.user_feat.shape[1], m, width)
                     for R, T in (c["docs"].shape[1:] for c in cache.values()))
            fused = self._siamese_fused_g()
            grads = self._head_grads() if fused else lambda u, i: (None, None)      # None: K13 forms g from the latents
            g0 = torch.empty(0, self.user_feat.shape[1], device=dev) if fused else None

            def attrib(name, ids, other, g):
                c, o = cache[name], cache["item" if name == "user" else "user"]
                return ops.explain_avgpool_attrib(table, c["docs"], c["masks"], ids, c["v"], c["a"], c["att"], feats[name], m,
                                                  width, g=g, other=other, lat=c.get("lat"), lat_other=o.get("lat"),
                                                  w_side=last[name].W, fm_h=mdl.fm.h, lt_w=lt_w, return_map=return_maps)
        else:
            docs = cache["user"]["docs"]
            R, T = docs.shape[1:] if docs.dim() == 3 else (1, docs.shape[1])
            if isinstance(mdl, DualAtt):
                specs = ops.datt_explain_convs(mdl.side_params("u"))
                width = specs[0][1] if width is None else int(width)              # the local window
                w0, w3 = mdl.fc[0].weight, mdl.fc[3].weight

                def grads(u, i):
                    return ops.datt_fc_grads(u, i, self.user_feat, self.item_feat, cache["user"]["hid_mask"],
                                             cache["item"]["hid_mask"], w0, w3)
            else:
                specs = self._conv_specs()
                width = max(k for _, k, _ in specs) if width is None else int(width)
                grads = self._head_grads()
                if isinstance(mdl, NARRE):
                    grads = self._narre_grads(grads)
            h_tot = sum(h for h, _, _ in specs)
            ok = ops.explain_supported(R * T, m, width, len(specs))
            g0 = torch.empty(0, R, h_tot, device=dev)

            def attrib(name, ids, other, g):
                c = cache[name]
                return ops.explain_attrib(ids * R, g.view(ids.numel(), R, h_tot), c.get("feat"), c["argmax"], c["contrib"],
                                          specs, R, T, m, width, return_map=return_maps, return_review_attr="att" in c,
                                          dense_coef=c.get("gate_coef"), dense_vec=c.get("gate_vec"))
        if not ok:
            raise ValueError(f"explain takes 1 <= m <= {ops.EXPLAIN_MAX_M}, 1 <= width <= {ops.EXPLAIN_MAX_WIDTH} and at most "
                             f"{ops.EXPLAIN_MAX_POSITIONS} positions per entity within the kernel's shared memory (got m={m}, "
                             f"width={width}, documents {tuple(c['docs'].shape[1:] for c in cache.values())})")
        parts = {"user": [], "item": []}
        for lo in range(0, u_ids.numel(), chunk):
            u, i = u_ids[lo:lo + chunk], i_ids[lo:lo + chunk]
            g_u, g_i = grads(u, i)
            parts["user"].append(attrib("user", u, i, g_u))
            parts["item"].append(attrib("item", i, u, g_i))
        sides = []
        for name, ids in (("user", u_ids), ("item", i_ids)):
            c = cache[name]
            # no pairs: K4 takes at least one, so only the attribution runs, on an empty g (empty results of the right shapes)
            p = parts[name] or [attrib(name, ids, ids, g0)]
            cat = {k: torch.cat([x[k] for x in p]) for k in p[0]}
            mp = cat.get("map")
            sides.append(SideExplanation(
                text_total=cat["text_total"], top_pos=cat["top_pos"], top_attr=cat["top_attr"], bottom_pos=cat["bottom_pos"],
                bottom_attr=cat["bottom_attr"], map=None if mp is None else mp.view(-1, *c["docs"].shape[1:]),
                review_weight=c["att"].index_select(0, ids) if "att" in c else None, review_attr=cat.get("review_attr"),
                local_att=c["gate_l"].index_select(0, ids) if "gate_l" in c else None,
                global_att=c["gate_g"].index_select(0, ids) if "gate_g" in c else None))
        return Explanation(pred, *sides)

    def _head_grads(self):
        """grads(u, i) → (g_u, g_i) = d pred / d feat of both sides for pairs (u, i) from K4's backward on the cached
        features."""
        mdl = self.model
        head, pads = head_params(*self._last_feats(), mdl.fm, zero_bias=True)
        scratch = [torch.empty_like(p) for p in head]

        def grads(u, i):
            u_text, i_text = ops.gather_rows(self.user_feat, u), ops.gather_rows(self.item_feat, i)
            return ops.head_text_grads(u_text, i_text, self._model_ids("user", u), self._model_ids("item", i), head, pads,
                                       scratch)
        return grads

    def _narre_grads(self, head_grads):
        """grads(u, i) → (g_u, g_i) = d pred / d feat [P, R, H] of each review's features: head_grads(u, i) through K3's
        backward, with the cached attention weights."""
        mdl = self.model
        cu, ci = self._explain["user"], self._explain["item"]
        R, H = mdl.doc_num, cu["feat"].shape[1]
        atts = (mdl.user_att, mdl.item_att)
        att_prm = [a.kernel_params() for a in atts]
        att_scratch = [[torch.empty_like(p) for p in sp] for sp in att_prm]

        def grads(u, i):
            return ops.narre_feat_grads(
                [cu["feat"].view(-1, R, H).index_select(0, u), ci["feat"].view(-1, R, H).index_select(0, i)],
                [cu["rev_ids"].index_select(0, u), ci["rev_ids"].index_select(0, i)],
                [cu["att"].index_select(0, u), ci["att"].index_select(0, i)], head_grads(u, i), att_prm,
                [a.padding_idx for a in atts], att_scratch)
        return grads

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
    map: Optional[torch.Tensor] = None              # [B, L] (NARRE, SimpleSiamese [B, R, T]) with return_maps
    review_weight: Optional[torch.Tensor] = None    # NARRE, SimpleSiamese [B, R]: the entity's review attention weights
    review_attr: Optional[torch.Tensor] = None      # NARRE, SimpleSiamese [B, R]: per-review sums of the map
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


def list_metrics(items: torch.Tensor, item_vecs: torch.Tensor, n_items: int, chunk: int = 1024) -> dict:
    """List-level metrics of recommendation lists (any device, no GPU needed), e.g. to compare recommend with
    recommend_diverse.

    items [n, k] int64: each row's list, -1 for an empty slot (recommend's tail); item_vecs [I, D]: the item vectors the
    similarity is taken on, unit-normalised as recommend_diverse does (ops.unit_rows: float64, then fp32; a zero row has
    sim 0 to everything); n_items: the number of items a list could hold (e.g. I - 1 without the padding item).
      ild       intra-list diversity: per row, the mean over pairs of its valid items of 1 - sim(a, b) (in float64), then
                the mean over the rows with at least two valid items (n_rows of them); 0.0 when there is none
      coverage  the number of distinct valid items over all lists / n_items"""
    items = items.to(torch.int64)
    if items.dim() != 2:
        raise ValueError(f"items must be [n, k], got {tuple(items.shape)}")
    vecs = ops.unit_rows(item_vecs).to(items.device).double()
    valid = items >= 0
    if bool((items >= vecs.shape[0]).any()):
        raise ValueError(f"item ids must lie in [-1, {vecs.shape[0]})")
    total, n_rows = 0.0, 0
    for lo in range(0, items.shape[0], chunk):
        it, ok = items[lo:lo + chunk], valid[lo:lo + chunk]
        v = vecs[it.clamp_min(0)] * ok.unsqueeze(-1)
        dist = 1.0 - v @ v.transpose(1, 2)
        pair = ok.unsqueeze(2) & ok.unsqueeze(1)
        pair &= torch.triu(torch.ones_like(pair[0]), diagonal=1)
        n_pairs = pair.sum((1, 2))
        has = n_pairs > 0
        total += float(((dist * pair).sum((1, 2))[has] / n_pairs[has]).sum())
        n_rows += int(has.sum())
    coverage = torch.unique(items[valid]).numel() / max(int(n_items), 1)
    return {"ild": total / n_rows if n_rows else 0.0, "coverage": coverage, "n_rows": n_rows}
