"""SimpleSiamese — drop-in for the reference's models/simple_siamese/simple_siamese.py:8-88 (same constructor, forward
signature, parameter names and state_dict keys); SURVEY §8f-4: the alternate encoder that reuses the hot path's kernels.

The encoder — word embedding gather → per-review masked average pooling (layers.py:90-110) — is one fused kernel (K9,
ops.MaskedAvgPoolFn: the [bz·R, T, E] embeddings are never materialised); LastFeat ×2 + FM is the fused head (K4).  The small
additive review attention (layers.py:171-197) and the optional latent transform are library ops.  The reference's
VariationalDropout (one mask per (review, embedding channel), shared by the time steps) commutes with the masked mean and is
applied to the pooled rows."""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops
from .layers import FM, HotPathModule, LastFeat, WordEmbedding, fused_head


class NodeDropout(nn.Dropout):
    """Drops whole reviews: one mask per (sample, review) (layers.py:7-22)."""

    def forward(self, x):
        ones = x.new_ones(x.shape[0], x.shape[1])
        return F.dropout(ones, self.p, self.training).unsqueeze(2) * x


class VariationalDropout(nn.Dropout):
    """One mask per (row, channel) shared by all time steps (layers.py:24-51); here applied to the POOLED rows [N, E]."""

    def forward(self, x):
        return F.dropout(x.new_ones(x.shape), self.p, self.training) * x


class MaskedAvgPooling1d(nn.Module):
    def forward(self, inputs, input_masks):
        raise RuntimeError("rbr_b200.MaskedAvgPooling1d is fused with the embedding gather (ops.MaskedAvgPoolFn)")


class AddictiveAttention(nn.Module):
    """(sic) layers.py:171-197: softmax over the reviews of tanh(Linear(x)) · w, masked reviews at -1e8."""

    def __init__(self, hidden_dim, latent_dim):
        super().__init__()
        self.proj_layer = nn.Sequential(nn.Linear(hidden_dim, latent_dim), nn.Tanh())
        self.inner_product = nn.Linear(latent_dim, 1, bias=False)

    def forward(self, inputs, input_masks):
        logits = self.inner_product(self.proj_layer(inputs))
        scores = F.softmax(torch.masked_fill(logits, ~input_masks.unsqueeze(2), -1e8), dim=1)
        return torch.sum(scores * inputs, dim=1), scores


class FMWithoutUIBias(nn.Module):
    def __init__(self, user_size, item_size, latent_dim, dropout, user_padding_idx, item_padding_idx):
        super().__init__()
        self.dropout = nn.Dropout(dropout)
        self.h = nn.Parameter(torch.empty(latent_dim, 1).uniform_(-0.1, 0.1))
        self.g_bias = nn.Parameter(torch.full((1,), 4.0))

    def forward(self, u_feat, i_feat):
        return self.dropout(F.relu(u_feat * i_feat)) @ self.h + self.g_bias


class SimpleSiamese(HotPathModule):
    staging_spec = dict(tokens=(0, 1), masks=(2, 3))

    def __init__(self, embedding_dim, latent_dim, vocab_size, user_size, item_size, pretrained_embeddings, freeze_embeddings,
                 dropout, word_dropout, review_dropout, use_ui_bias, latent_transform):
        super().__init__()
        self.use_ui_bias = use_ui_bias
        self.embedding_dim = embedding_dim
        self.latent_transform = latent_transform
        self.word_embedding = WordEmbedding(vocab_size, embedding_dim, pretrained_embeddings=pretrained_embeddings,
                                            freeze_embeddings=freeze_embeddings, padding_idx=0)
        self.var_dropout = VariationalDropout(p=word_dropout)
        self.review_dropout = NodeDropout(p=review_dropout)
        self.masked_pooling_1d = MaskedAvgPooling1d()
        feat = latent_dim if latent_transform else embedding_dim
        if latent_transform:
            self.latent_transform_layer = nn.Sequential(nn.Linear(embedding_dim, latent_dim), nn.Tanh())
        self.user_last_feat_layer = LastFeat(user_size, feat, latent_dim, padding_idx=0)
        self.item_last_feat_layer = LastFeat(item_size, feat, latent_dim, padding_idx=0)
        self.review_att_layer = AddictiveAttention(feat, latent_dim)
        if use_ui_bias:
            self.fm = FM(user_size, item_size, latent_dim, dropout, user_padding_idx=0, item_padding_idx=0)
            nn.init.constant_(self.fm.g_bias, 4.0)                       # simple_siamese/layers.py:318
        else:
            self.fm = FMWithoutUIBias(user_size, item_size, latent_dim, dropout, user_padding_idx=0, item_padding_idx=0)
        self.last_arena = None

    def forward(self, u_revs, i_revs, u_rev_word_masks, i_rev_word_masks, u_rev_masks, i_rev_masks, u_ids, i_ids):
        """u_revs/i_revs [bz, R, T] int64 (or int32), word masks [bz, R, T] bool (None: ids != 0), review masks [bz, R] bool,
        ids [bz] → (out_logits [bz], None, None)."""
        arena = ops.GradArena.for_module(self)
        self.last_arena = arena
        bz, ur, T = u_revs.shape
        ir = i_revs.shape[1]
        um = None if u_rev_word_masks is None else u_rev_word_masks.reshape(-1, T)
        im = None if i_rev_word_masks is None else i_rev_word_masks.reshape(-1, T)
        u_pool, i_pool = ops.MaskedAvgPoolFn.apply(self.word_embedding.embedding.weight, self._pool_cfg(arena), u_revs.reshape(-1, T),
                                                   um, i_revs.reshape(-1, T), im)
        (u_feat, _, _), (i_feat, _, _) = self._attend([u_pool.view(bz, ur, -1), i_pool.view(bz, ir, -1)],
                                                      [u_rev_masks, i_rev_masks])
        out = self.head(u_feat, i_feat, u_ids, i_ids, arena)
        self._after_forward()
        return out.view(bz), None, None

    def _pool_cfg(self, arena):
        pad = self.word_embedding.padding_idx
        return {"padding_idx": 0 if pad is None else pad, "arena": arena, "table_param": self.word_embedding.embedding.weight,
                "mask_from_ids": True}

    def _attend(self, pooled, rev_masks):
        """Pooled reviews [bz, R, E] of each side → per side (feat [bz, feat], the attention's inputs v [bz, R, feat], its
        weights [bz, R, 1]); stage by stage across the sides, so training draws its dropout masks in the reference's order."""
        xs = [self.var_dropout(p) for p in pooled]                                         # simple_siamese.py:59-64
        if self.latent_transform:
            xs = [self.latent_transform_layer(x) for x in xs]
        xs = [self.review_dropout(x) for x in xs]
        return [(*self.review_att_layer(x, m), x) for x, m in zip(xs, rev_masks)]

    def encode_side(self, revs, word_masks, rev_masks):
        """One side's text feature as forward computes it — revs [bz, R, T], word_masks [bz, R, T] bool or None (ids != 0),
        rev_masks [bz, R] bool → (feat [bz, feat], the review attention's weights [bz, R, 1] and inputs v [bz, R, feat])."""
        bz, R, T = revs.shape
        wm = None if word_masks is None else word_masks.reshape(-1, T)
        (pool,) = ops.MaskedAvgPoolFn.apply(self.word_embedding.embedding.weight, self._pool_cfg(None), revs.reshape(-1, T), wm)
        ((feat, scores, v),) = self._attend([pool.view(bz, R, -1)], [rev_masks])
        return feat, scores, v

    def head(self, u_feat, i_feat, u_ids, i_ids, arena=None):
        """LastFeat x2 + FM(WithoutUIBias) on the two text features → [bz, 1]."""
        if self.use_ui_bias and ops.head_supported(u_feat.shape[1], self.fm.h.shape[0]):
            return fused_head(self.user_last_feat_layer, self.item_last_feat_layer, self.fm, u_feat.contiguous(),
                              i_feat.contiguous(), u_ids, i_ids, self.training, arena)
        if self.use_ui_bias:                     # feature width beyond the fused head's shared-memory budget: the layers' own forwards
            return self.fm(self.user_last_feat_layer(u_feat, u_ids), self.item_last_feat_layer(i_feat, i_ids), u_ids, i_ids)
        return self.fm(self.user_last_feat_layer(u_feat, u_ids), self.item_last_feat_layer(i_feat, i_ids))
