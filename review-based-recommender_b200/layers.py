"""Host-side mirror of the reference's layer classes (same names, constructor arguments, parameter names
and state_dict keys) with forwards that call the rbr_b200 CUDA kernels.

Reference classes mirrored (paths under the reference root):
  WordEmbedding    models/deepconn/layers.py:9-24   (= narre/narre.py:9-24, dual_att/layers.py:8-23)
  MyConv1d         models/deepconn/layers.py:26-60  (= narre/layers.py:119-153)
  NgramFeat        models/deepconn/layers.py:100-136 (= narre/layers.py:365-401)
  LastFeat         models/deepconn/layers.py:138-165 (= narre/narre.py:66-93)
  FM               models/deepconn/layers.py:167-209 (= narre/narre.py:95-137)
  LinearAttention  models/narre/narre.py:26-64

The model classes (deepconn.py / narre.py) do not chain these forwards the way the reference does: they
fuse gather+mask+conv+pool (EncodeDocsFn) and LastFeat x2 + FM (HeadFn).  The standalone forwards below keep
every layer usable — and testable against the reference — on its own.
"""
from __future__ import annotations

import os
from typing import List, Optional, Sequence

import torch
import torch.nn as nn

from . import ops


def default_precision() -> str:
    """Conv precision: "bf16" (tcgen05 tensor cores, 1e-2) unless RBR_PRECISION=fp32 (CUDA cores, 1e-5)."""
    p = os.environ.get("RBR_PRECISION", "bf16").lower()
    if p not in ("bf16", "fp32"):
        raise ValueError(f"RBR_PRECISION must be bf16 or fp32, got {p}")
    return p


class HotPathModule(nn.Module):
    """Base of the three model classes: out-of-range id detection at mode switches.

    The kernels read an id outside its table as a padding (zero) row and count it instead of faulting; the reference raises
    IndexError (CPU) or trips a device assert (CUDA).  Reading the counter synchronises the stream, so it is polled where
    the trainers switch mode — `model.train()` at the start of an epoch, `model.eval()` before validation
    (trainer/train_deepconn_pp.py:149,196) — never inside a step or a CUDA-graph capture; RBR_CHECK_IDS=1 polls after every
    forward (debugging)."""

    def check_ids(self) -> None:
        prm = next(self.parameters(), None)
        if prm is None or not prm.is_cuda or torch.cuda.is_current_stream_capturing():
            return
        from ._lib import lib
        with torch.cuda.device(prm.device):
            n = lib.rbr_consume_oob_count(ops._stream(True))
        if n < 0:
            lib.check(n, "rbr_consume_oob_count")
        if n > 0:
            raise IndexError(f"rbr_b200: {n} token / id values outside their embedding tables since the last check "
                             "(they were read as padding rows); check vocab_size / user_size / item_size against the data")

    def train(self, mode: bool = True):
        super().train(mode)
        self.check_ids()
        return self

    def _after_forward(self):
        if _CHECK_IDS_EVERY_FORWARD:
            self.check_ids()


_CHECK_IDS_EVERY_FORWARD = os.environ.get("RBR_CHECK_IDS", "0") == "1"


class WordEmbedding(nn.Module):
    def __init__(self, vocab_size, embedding_dim, pretrained_embeddings=None, padding_idx=0, freeze_embeddings=False):
        super().__init__()
        self.freeze_embeddings = freeze_embeddings
        self.padding_idx = padding_idx
        self.embedding = nn.Embedding(vocab_size, embedding_dim, padding_idx=padding_idx)   # parameter holder
        self.embedding.weight.requires_grad = not self.freeze_embeddings
        if pretrained_embeddings is not None:
            self.embedding.load_state_dict({"weight": torch.as_tensor(pretrained_embeddings)})
        self._shadow = None          # (table version, bf16 shadow) cache
        self._arena = None

    def forward(self, inputs):
        """[...] int64 ids → [..., E] fp32, bit-exact with nn.Embedding (K1); backward = K1b."""
        return ops.EmbeddingFn.apply(self.embedding.weight, inputs, self.padding_idx, self._arena)

    def bf16_shadow(self) -> torch.Tensor:
        """bf16 copy of the table for the tensor-core conv, re-cast only when the table changed
        (optimizer steps bump the tensor's version counter)."""
        w = self.embedding.weight
        key = (w._version, w.data_ptr())
        if self._shadow is None or self._shadow[0] != key:
            self._shadow = (key, ops.table_to_bf16(w.detach()))
        return self._shadow[1]

    def invalidate_operand_cache(self):
        """Drop the bf16 shadow (as an optimizer step would, by bumping the table's version)."""
        self._shadow = None

    def refresh_operand_cache(self):
        """Re-cast the table into the EXISTING shadow buffer (same address: a captured CUDA graph keeps reading it) and mark
        it current — after parameters were changed outside a graph whose optimizer keeps the shadow up to date itself."""
        if self._shadow is None:
            return
        w = self.embedding.weight
        self._shadow[1].copy_(ops.table_to_bf16(w.detach()))
        self._shadow = ((w._version, w.data_ptr()), self._shadow[1])


class MyConv1d(nn.Module):
    """Holder of one nn.Conv1d per kernel size; the arithmetic runs inside NgramFeat's fused kernel."""

    def __init__(self, kernel_sizes, in_features, out_features):
        super().__init__()
        if type(kernel_sizes) is str:
            kernel_sizes = [int(x) for x in kernel_sizes.split(",")]      # "3,4,5" form, layers.py:34-36
        assert out_features % len(kernel_sizes) == 0
        assert all([kz % 2 == 1 for kz in kernel_sizes])
        self.kernel_sizes = list(kernel_sizes)
        self.out_features_per_kz = out_features // len(kernel_sizes)
        self.list_of_conv1d = nn.ModuleList([
            nn.Conv1d(in_features, self.out_features_per_kz, kz, padding=(kz - 1) // 2) for kz in kernel_sizes
        ])
        self._packed = {}

    def packed(self, i: int) -> torch.Tensor:
        w = self.list_of_conv1d[i].weight
        key = (w._version, w.data_ptr())
        hit = self._packed.get(i)
        if hit is None or hit[0] != key:
            hit = (key, ops.conv_pack(w.detach()))
            self._packed[i] = hit
        return hit[1]

    def invalidate_operand_cache(self):
        self._packed.clear()

    def forward(self, inputs):
        raise RuntimeError("rbr_b200.MyConv1d is a parameter holder: the [N,H,L] conv output is never materialised; "
                           "call NgramFeat (conv + ReLU + max-over-time fused)")


class HierPooling(nn.Module):
    """Holder of the optional projection of the reference's HierPooling (models/deepconn/layers.py:62-98): avg-pool with the
    given kernel (stride 1) then max-pool over time run in K8 (ops.HierPoolFn) fused with the embedding gather; the
    Linear(in → out), present only when the sizes differ, is a library GEMM."""

    def __init__(self, in_features, out_features, kernel_size):
        super().__init__()
        self.kernel_size = kernel_size
        self.proj_layer = nn.Linear(in_features, out_features) if in_features != out_features else None

    def forward(self, inputs):
        raise RuntimeError("rbr_b200.HierPooling is a parameter holder: call NgramFeat (gather + avg-pool + max-pool fused)")


class NgramFeat(nn.Module):
    def __init__(self, kernel_sizes, in_features, out_features, seq_len, dropout=0., arch="CNN", precision=None):
        super().__init__()
        self.arch = arch
        if arch == "CNN":
            self.feature_layer = nn.Sequential(MyConv1d(kernel_sizes, in_features, out_features), nn.ReLU(),
                                               nn.MaxPool1d(seq_len))
        elif arch == "HierPooling":
            if type(kernel_sizes) is str:
                kernel_sizes = [int(x) for x in kernel_sizes.split(",")]
            assert len(kernel_sizes) == 1                           # layers.py:112
            self.feature_layer = nn.Sequential(HierPooling(in_features, out_features, kernel_sizes[0]), nn.ReLU())
        else:
            raise ValueError(f"{arch} is not predefined.")
        self.seq_len = seq_len
        self.out_features = out_features
        self.dropout = nn.Dropout(p=dropout) if dropout else None       # created but never applied, as in the reference
        self.precision = precision or default_precision()
        self._arena = None
        self.table_grad_hook = None     # called with the word-table gradient buffer once it is complete (parallel.py)
        self.conv_flags = 0             # ops.CONV_* kernel-selection flags passed with every call (tests, A/B timing)

    @property
    def conv(self):
        return self.feature_layer[0]

    def _hier(self, table, sides, masks, padding_idx, mask_from_ids):
        hp = self.feature_layer[0]
        cfg = {"ksize": hp.kernel_size, "padding_idx": padding_idx, "arena": self._arena, "table_param": table,
               "mask_from_ids": mask_from_ids}
        flat = []
        for ids, m in zip(sides, masks):
            flat += [ids, m]
        outs = []
        for pooled in ops.HierPoolFn.apply(table, cfg, *flat):
            if hp.proj_layer is not None:
                pooled = hp.proj_layer(pooled)
            outs.append(torch.relu(pooled))
        return outs

    def encode(self, word_embeddings: WordEmbedding, sides: Sequence[torch.Tensor],
               masks: Sequence[Optional[torch.Tensor]], return_argmax: bool = False) -> List[torch.Tensor]:
        """Fused path used by the models: token ids → pooled features, [n_docs, H] per side (with return_argmax: followed by
        the int32 [n_docs, H] first-arg-max positions per side)."""
        if self.arch == "HierPooling":
            table = word_embeddings.embedding.weight
            pidx = -1 if word_embeddings.padding_idx is None else word_embeddings.padding_idx
            return self._hier(table, sides, masks, pidx, True)
        conv = self.conv
        convs = list(conv.list_of_conv1d)
        table = word_embeddings.embedding.weight
        cfg = {
            "n_conv": len(convs),
            "precision": self.precision,
            "act": ops.ACT_RELU,
            "pads": [(k - 1) // 2 for k in conv.kernel_sizes],
            "shadow_fn": word_embeddings.bf16_shadow,
            "pack_fn": conv.packed,
            "arena": self._arena,
            "table_param": table,
            "weight_params": [c.weight for c in convs],
            "bias_params": [c.bias for c in convs],
            "padding_idx": -1 if word_embeddings.padding_idx is None else word_embeddings.padding_idx,
            "table_ready": self.table_grad_hook,
            "flags": self.conv_flags,
            "mask_from_ids": True,      # a side passed without a mask: mask = (ids != 0), what collate_fn computes (utils.py:30-42)
        }
        # one bf16 conv whose dense tensor-core backward (K2c) writes EVERY element of the table gradient: the arena need not
        # zero-fill that 60 MB slot and the GEMM epilogue stores without reading
        if (self._arena is not None and len(convs) == 1 and self.precision == "bf16" and table.requires_grad
                and not (self.conv_flags & ops.CONV_BWD_SPARSE) and torch.is_grad_enabled()
                and ops.lib.rbr_conv_bwd_cmat_supported(table.shape[0], table.shape[1], convs[0].weight.shape[0], conv.kernel_sizes[0])):
            cfg["table_overwrite"] = True
            self._arena.no_zero.add(id(table))
        flat = []
        for ids, m in zip(sides, masks):
            flat += [ids, m]
        outs = list(ops.EncodeDocsFn.apply(table, cfg, *[c.weight for c in convs], *[c.bias for c in convs], *flat))
        return outs if return_argmax else outs[:len(sides)]

    def forward(self, inputs, input_masks):
        """Reference signature (layers.py:123-136): inputs [bz, seq_len, E] fp32, masks [bz, seq_len] → [bz, H, 1].

        The dense activations are treated as a bz*seq_len-row table indexed by arange, so the same fused
        kernel (and its backward, which yields d inputs) serves the standalone layer."""
        bz, seq_len, emb = inputs.shape
        x = inputs.contiguous().view(bz * seq_len, emb)
        ids = torch.arange(bz * seq_len, device=inputs.device, dtype=torch.int64).view(bz, seq_len)
        if self.arch == "HierPooling":
            return self._hier(x, [ids], [input_masks], -1, False)[0]     # [bz, out_features], as the reference returns it
        conv = self.conv
        convs = list(conv.list_of_conv1d)
        cfg = {
            "n_conv": len(convs), "precision": self.precision, "act": ops.ACT_RELU,
            "pads": [(k - 1) // 2 for k in conv.kernel_sizes],
            "shadow_fn": lambda: ops.table_to_bf16(x.detach()), "pack_fn": conv.packed, "arena": self._arena,
            "table_param": x, "weight_params": [c.weight for c in convs], "bias_params": [c.bias for c in convs],
            "padding_idx": -1, "flags": self.conv_flags,
            "dense_bwd": False,          # the "table" is this call's activations: no persistent coefficient-matrix workspace for it
        }
        feat, _ = ops.EncodeDocsFn.apply(x, cfg, *[c.weight for c in convs], *[c.bias for c in convs], ids, input_masks)
        return feat.view(bz, self.out_features, 1)


class LastFeat(nn.Module):
    def __init__(self, vocab_size, feat_size, latent_dim, padding_idx):
        super().__init__()
        self.W = nn.Parameter(torch.Tensor(feat_size, latent_dim))
        self.b = nn.Parameter(torch.Tensor(latent_dim))
        self.ebd = nn.Embedding(vocab_size, latent_dim, padding_idx=padding_idx)
        self.padding_idx = padding_idx
        self.reset_parameters()

    def reset_parameters(self):
        bound = 0.1
        nn.init.uniform_(self.W, -bound, bound)
        nn.init.constant_(self.b, bound)
        nn.init.uniform_(self.ebd.weight, -bound, bound)

    def forward(self, text_feat, my_id):
        """Standalone convenience (not on the fused path, which runs K4): text_feat @ W + b + ebd(my_id)."""
        return text_feat @ self.W + self.b + ops.EmbeddingFn.apply(self.ebd.weight, my_id, self.padding_idx, None)


class FM(nn.Module):
    def __init__(self, user_size, item_size, latent_dim, dropout, user_padding_idx, item_padding_idx):
        super().__init__()
        self.dropout = nn.Dropout(dropout)
        self.h = nn.Parameter(torch.Tensor(latent_dim, 1))
        self.user_bias = nn.Embedding(user_size, 1, padding_idx=user_padding_idx)
        self.item_bias = nn.Embedding(item_size, 1, padding_idx=item_padding_idx)
        self.g_bias = nn.Parameter(torch.Tensor(1))
        self.padding_idx = user_padding_idx
        self.item_padding_idx = item_padding_idx
        self.reset_parameters()

    def reset_parameters(self):
        bound = 0.1
        nn.init.uniform_(self.h, -bound, bound)
        nn.init.uniform_(self.user_bias.weight, -bound, bound)
        nn.init.uniform_(self.item_bias.weight, -bound, bound)
        nn.init.constant_(self.g_bias, bound)

    def forward(self, u_feat, i_feat, u_id, i_id):
        """Standalone convenience (the models run the fused K4 instead)."""
        fm = self.dropout(torch.relu(u_feat * i_feat))
        ub = ops.EmbeddingFn.apply(self.user_bias.weight, u_id, self.padding_idx, None)
        ib = ops.EmbeddingFn.apply(self.item_bias.weight, i_id, self.item_padding_idx, None)
        return fm @ self.h + ub + ib + self.g_bias


def head_params(user_feat: LastFeat, item_feat: LastFeat, fm: nn.Module, zero_bias: bool = False):
    """K4's parameters (Wu, bu, ebd_u, Wi, bi, ebd_i, fm_h, user_bias, item_bias, g_bias) and padding indices (user, item,
    FM user, FM item) for LastFeat(user) + LastFeat(item) + `fm`.  An FM without user / item bias tables (SimpleSiamese's
    FMWithoutUIBias) has None in their two slots and padding index 0 for them, or with zero_bias zero tables of the LastFeat
    embeddings' heights, which K4 can read (the biases do not enter d pred / d text)."""
    if isinstance(fm, FM):
        bias, fm_pads = [fm.user_bias.weight, fm.item_bias.weight], (fm.padding_idx, fm.item_padding_idx)
    else:
        bias, fm_pads = [None, None], (0, 0)
        if zero_bias:
            bias = [torch.zeros(f.ebd.weight.shape[0], 1, device=f.ebd.weight.device) for f in (user_feat, item_feat)]
    params = [user_feat.W, user_feat.b, user_feat.ebd.weight, item_feat.W, item_feat.b, item_feat.ebd.weight, fm.h, *bias,
              fm.g_bias]
    return params, (user_feat.padding_idx, item_feat.padding_idx, *fm_pads)


def fused_head(user_feat: LastFeat, item_feat: LastFeat, fm: FM, u_text, i_text, u_id, i_id, training: bool, arena,
               ratings: Optional[torch.Tensor] = None):
    """K4: LastFeat(user) + LastFeat(item) + FM in one kernel (reference deepconn.py:48-51).  With `ratings` the same launch
    also evaluates nn.MSELoss (trainer/train_deepconn_pp.py:140,164) and returns (loss, pred)."""
    p = fm.dropout.p if training else 0.0
    # dropout mask seed: a fresh host value per call, or — inside graphs.GraphedTrainStep's body (warm-up and capture) — a fixed
    # base plus a step counter that lives on the device and is bumped at the start of every replay
    seed_dev = fm.__dict__.get("_rbr_seed_dev") if p > 0 else None
    seed = 0 if p <= 0 else (0x5EED if seed_dev is not None else int(torch.randint(0, 2 ** 62, (1,)).item()))
    params, pads = head_params(user_feat, item_feat, fm)
    fm.__dict__["_rbr_last_drop"] = (p, seed, seed_dev)          # for tests: ops.head_dropout_mask(B, K, *this)
    if ratings is not None:
        return ops.HeadLossFn.apply(u_text, i_text, u_id, i_id, ratings, *params, p, seed, pads, arena, params, seed_dev)
    return ops.HeadFn.apply(u_text, i_text, u_id, i_id, *params, p, seed, pads, arena, params, seed_dev)


class LinearAttention(nn.Module):
    def __init__(self, vocab_size, feat_size, hidden_dim, dropout, padding_idx=0):
        super().__init__()
        self.W_rv = nn.Parameter(torch.empty(feat_size, hidden_dim).uniform_(-0.1, 0.1))
        self.W_id = nn.Parameter(torch.empty(hidden_dim, hidden_dim).uniform_(-0.1, 0.1))
        self.h = nn.Parameter(torch.empty(hidden_dim, 1).uniform_(-0.1, 0.1))
        self.b_1 = nn.Parameter(torch.empty(hidden_dim).fill_(0.1))
        self.b_2 = nn.Parameter(torch.empty(1).fill_(0.1))
        self.ebd_vals = nn.Embedding(vocab_size, hidden_dim, padding_idx=padding_idx)
        self.padding_idx = padding_idx
        self.dropout = nn.Dropout(p=dropout)
        self._arena = None

    def kernel_params(self) -> List[torch.Tensor]:
        """The six parameters in K3's order: (W_rv, W_id, h, b_1, b_2, ebd_vals)."""
        return [self.W_rv, self.W_id, self.h, self.b_1, self.b_2, self.ebd_vals.weight]

    def forward(self, feat, other_id):
        """feat [bz, dnum, H], other_id [bz, dnum] → (out [bz, H], att_scores [bz, dnum, 1])  (narre.py:40-64)."""
        params = self.kernel_params()
        out, scores = ops.NarreAttnFn.apply(feat, other_id, *params, self.padding_idx, self._arena, params)
        return self.dropout(out), scores
