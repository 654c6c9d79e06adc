"""DualAtt (D-ATT) — drop-in for the reference's models/dual_att/dual_att.py:19-61 and models/dual_att/layers.py
(same constructor, forward signature, parameter names and state_dict keys), running on the rbr_b200 CUDA kernels.

The embedding gather, both attention gates, the four gated tanh convolutions and their max-over-time (layers.py:43-53,
81-89) are one fused encoder per side (ops.DattEncodeFn: K5 gates + gated K2 convs).  The shared two-layer FC stack and
the final dot product (dual_att.py:31-35, 51, 57-61) are plain library GEMMs / elementwise ops left to PyTorch."""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .layers import HotPathModule, WordEmbedding, default_precision


class LocalAttention(nn.Module):
    """Parameter holder mirroring models/dual_att/layers.py:25-41."""

    def __init__(self, doc_len, window_size, out_size, emb_size=100):
        super().__init__()
        self.window_size, self.doc_len, self.out_size, self.emb_size = window_size, doc_len, out_size, emb_size
        self.padding_size = (window_size - 1) // 2
        self.attn = nn.Sequential(nn.Conv1d(emb_size, 1, kernel_size=window_size, padding=self.padding_size), nn.Sigmoid())
        self.conv = nn.Sequential(nn.Conv1d(emb_size, out_size, kernel_size=1), nn.Tanh(), nn.MaxPool1d(doc_len))

    def forward(self, x):
        raise RuntimeError("rbr_b200.LocalAttention is a parameter holder: DualAtt runs the fused gated encoder")


class GlobalAttention(nn.Module):
    """Parameter holder mirroring models/dual_att/layers.py:55-79 (window sizes 2, 3, 4 are hard-coded there)."""

    def __init__(self, doc_len, out_size, emb_size=100):
        super().__init__()
        self.doc_len, self.out_size, self.emb_size = doc_len, out_size, emb_size
        self.attn = nn.Sequential(nn.Conv1d(emb_size, 1, kernel_size=doc_len), nn.Sigmoid())
        self.conv1 = nn.Sequential(nn.Conv1d(emb_size, out_size, kernel_size=2), nn.Tanh(), nn.MaxPool1d(doc_len - 1))
        self.conv2 = nn.Sequential(nn.Conv1d(emb_size, out_size, kernel_size=3), nn.Tanh(), nn.MaxPool1d(doc_len - 2))
        self.conv3 = nn.Sequential(nn.Conv1d(emb_size, out_size, kernel_size=4), nn.Tanh(), nn.MaxPool1d(doc_len - 3))

    def forward(self, x):
        raise RuntimeError("rbr_b200.GlobalAttention is a parameter holder: DualAtt runs the fused gated encoder")


class DualAtt(HotPathModule):
    staging_spec = dict(tokens=(0, 1), masks=())      # which forward() inputs are token-id tensors / their masks (staging.StagedInputs)

    def __init__(self, vocab_size, doc_len, l_window_size=5, l_out_size=200, g_out_size=100, emb_size=100,
                 hidden_size_1=500, hidden_size_2=50, dropout=0.5, pretrained_embeddings=None, precision=None):
        super().__init__()
        self.fc_input = l_out_size + 3 * g_out_size
        self.doc_len = doc_len
        self.word_embeddings = WordEmbedding(vocab_size, emb_size, pretrained_embeddings=pretrained_embeddings)
        self.u_local_atten = LocalAttention(doc_len, l_window_size, l_out_size, emb_size)
        self.u_global_atten = GlobalAttention(doc_len, g_out_size, emb_size)
        self.i_local_atten = LocalAttention(doc_len, l_window_size, l_out_size, emb_size)
        self.i_global_atten = GlobalAttention(doc_len, g_out_size, emb_size)
        self.fc = nn.Sequential(nn.Linear(self.fc_input, hidden_size_1), nn.ReLU(), nn.Dropout(dropout),
                                nn.Linear(hidden_size_1, hidden_size_2))
        self.precision = precision or default_precision()
        self.last_arena = None
        self.conv_flags = 0             # ops.CONV_TC_* kernel-selection flags passed with every gated conv (tests, A/B timing)

    def invalidate_operand_cache(self):
        self.word_embeddings.invalidate_operand_cache()

    @staticmethod
    def _side_params(local: LocalAttention, glob: GlobalAttention):
        return [local.attn[0].weight, local.attn[0].bias, local.conv[0].weight, local.conv[0].bias,
                glob.attn[0].weight, glob.attn[0].bias, glob.conv1[0].weight, glob.conv1[0].bias,
                glob.conv2[0].weight, glob.conv2[0].bias, glob.conv3[0].weight, glob.conv3[0].bias]

    def encode(self, docs, sides, arena=None):
        """Fused encoder: docs = list of [bz, doc_len] id tensors, sides = matching list of "u" / "i" → list of
        [bz, l_out + 3*g_out] features (dual_att.py:45-50, 53-56 without the FC)."""
        mods = {"u": (self.u_local_atten, self.u_global_atten), "i": (self.i_local_atten, self.i_global_atten)}
        params, args = [], []
        for ids, s in zip(docs, sides):
            if ids.shape[-1] != self.doc_len:
                raise ValueError(f"DualAtt was built for doc_len={self.doc_len}, got {ids.shape[-1]} "
                                 "(the global attention kernel spans the whole document)")
            prm = self._side_params(*mods[s])
            params.append(prm)
            args += [ids, *prm]
        table = self.word_embeddings.embedding.weight
        pidx = self.word_embeddings.padding_idx
        cfg = {"precision": self.precision, "shadow_fn": self.word_embeddings.bf16_shadow, "arena": arena,
               "table_param": table, "params": params, "padding_idx": -1 if pidx is None else pidx, "flags": self.conv_flags}
        return list(ops.DattEncodeFn.apply(table, cfg, *args))

    def forward(self, u_docs, i_docs):
        """u_docs, i_docs: [bz, doc_len] int64 → ratings [bz]."""
        arena = ops.GradArena.for_module(self)
        self.last_arena = arena
        u_cat, i_cat = self.encode([u_docs, i_docs], ["u", "i"], arena)
        u_feat = self.fc(u_cat)                                                                   # dual_att.py:49-51
        i_feat = self.fc(i_cat)                                                                   # dual_att.py:55-57
        self._after_forward()
        return torch.sum(torch.mul(u_feat, i_feat), 1).view(-1)                                   # dual_att.py:59-61
