"""Host-side operators: torch.autograd.Functions whose forward/backward call the C-ABI kernels.

PyTorch provides device memory, the current CUDA stream and autograd bookkeeping; every arithmetic step
of the hot path runs in librbr_b200.so.  Tensors handed to the library must be CUDA, contiguous, fp32 /
int64 / bool — anything else raises (there is no CPU path).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import torch

from ._lib import lib

PREC_FP32, PREC_BF16 = 0, 1
ACT_RELU, ACT_TANH = 0, 1
_PREC = {"fp32": PREC_FP32, "bf16": PREC_BF16}
# per-call `flags` of the conv entry points (include/rbr_b200.h)
CONV_TC_SINGLE_CTA, CONV_TC_PAIR_ONLY, CONV_BWD_DENSE_TC, CONV_BWD_SPARSE, IDS_I32, MASK_FROM_IDS, IDS_U16 = 1, 2, 4, 8, 16, 32, 64


_STREAM_CACHE = [0, None]


def _stream(refresh: bool = False) -> int:
    """Raw handle of torch's current CUDA stream.  torch.cuda.current_stream() costs ~10 us; autograd Functions refresh it
    once on entry (refresh=True) and the launches inside reuse the handle."""
    if refresh or _STREAM_CACHE[1] is None:
        try:
            _STREAM_CACHE[0] = torch.cuda.current_stream().cuda_stream
        except Exception as e:      # no driver / no device
            raise RuntimeError(f"rbr_b200: a CUDA device is required (the hot path has no CPU implementation): {e}") from None
        _STREAM_CACHE[1] = True
    return _STREAM_CACHE[0]


_SIDE_STREAMS: Dict[str, list] = {}


def _side_streams(device, n: int) -> list:
    """n persistent auxiliary streams on `device` (created once)."""
    pool = _SIDE_STREAMS.setdefault(str(device), [])
    while len(pool) < n:
        pool.append(torch.cuda.Stream(device=device))
    return pool[:n]


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _req(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"rbr_b200: `{name}` must be a CUDA tensor (the hot path has no CPU implementation)")
    if t.dtype != dtype:
        raise TypeError(f"rbr_b200: `{name}` must be {dtype}, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


def _ids(t: torch.Tensor, name: str) -> torch.Tensor:
    """Token ids: int64 (torch.LongTensor, what the reference's collate_fn yields), or int32 / uint16 (staged input pipeline)."""
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"rbr_b200: `{name}` must be a CUDA tensor (the hot path has no CPU implementation)")
    if t.dtype not in (torch.int64, torch.int32, torch.uint16):
        raise TypeError(f"rbr_b200: `{name}` must be int64, int32 or uint16, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


def _id_width_flag(ids: torch.Tensor) -> int:
    return IDS_I32 if ids.dtype == torch.int32 else (IDS_U16 if ids.dtype == torch.uint16 else 0)


def _id_flags(ids: torch.Tensor, mask: Optional[torch.Tensor], mask_from_ids: bool) -> int:
    return _id_width_flag(ids) | (MASK_FROM_IDS if (mask is None and mask_from_ids) else 0)


def _mask_u8(mask: Optional[torch.Tensor], name: str) -> Optional[torch.Tensor]:
    if mask is None:
        return None
    if not mask.is_cuda:
        raise RuntimeError(f"rbr_b200: `{name}` must be a CUDA tensor")
    if mask.dtype == torch.bool:
        return mask.contiguous().view(torch.uint8)
    if mask.dtype == torch.uint8:
        return mask.contiguous()
    raise TypeError(f"rbr_b200: `{name}` must be bool, got {mask.dtype}")


# ---------------------------------------------------------------------------------------------------
# Step context: one flat fp32 gradient buffer per backward pass, with a view per parameter.
# ---------------------------------------------------------------------------------------------------
class GradArena:
    """Allocates ONE zero-filled flat buffer holding the gradient of every trainable parameter of a model
    (allocated at the first backward call of a step) and hands out per-parameter views.  The kernels
    accumulate straight into these views, autograd installs them as `.grad`, and data-parallel training
    all-reduces the flat buffer with a single NCCL call (parallel.py)."""

    def __init__(self, named_params: Sequence[Tuple[str, torch.nn.Parameter]], layout: Optional["GradArena"] = None):
        if layout is not None:                  # same model, next step: reuse the slot layout, fresh buffer
            self.slots, self.total, self.signature = layout.slots, layout.total, layout.signature
        else:
            self.slots: Dict[int, Tuple[int, torch.Size]] = {}
            off = 0
            for _, prm in named_params:
                if prm.requires_grad and id(prm) not in self.slots:
                    self.slots[id(prm)] = (off, prm.shape)
                    off += (prm.numel() + 63) // 64 * 64            # 256-byte aligned slots (float4 atomics)
            self.total = off
            self.signature = GradArena.signature_of(named_params)
        self.flat: Optional[torch.Tensor] = None
        self.device = None
        self.external: Optional[torch.Tensor] = None
        self.params = named_params
        self.no_zero: set = set()       # id(param) of slots whose producer OVERWRITES every element (dense table gradient, K2c)

    @staticmethod
    def signature_of(named_params) -> tuple:
        return tuple((id(p), p.requires_grad) for _, p in named_params)

    @staticmethod
    def for_module(module: torch.nn.Module) -> Optional["GradArena"]:
        """A fresh arena for this step (None under no_grad); the slot layout is computed once per module and reused while
        the parameter objects and their requires_grad flags are unchanged (building it walks named_parameters(): ~0.15 ms
        of host time per step).  Parameters registered after the first forward are not picked up."""
        if not torch.is_grad_enabled():
            return None
        params = module.__dict__.get("_rbr_param_list")
        if params is None:
            params = list(module.named_parameters())
            module.__dict__["_rbr_param_list"] = params
            module.__dict__["_rbr_arena_layout"] = None
        layout = module.__dict__.get("_rbr_arena_layout")
        if layout is None or layout.signature != GradArena.signature_of(params):
            layout = GradArena(params)
            module.__dict__["_rbr_arena_layout"] = layout
        arena = GradArena(params, layout=layout)
        arena.external = module.__dict__.get("_rbr_arena_buffer")
        return arena

    def _ensure(self, device):
        if self.flat is None:
            ext = self.external
            if ext is not None:          # persistent buffer (symmetric memory for the NVLS all-reduce): re-zeroed, not re-allocated
                lo, hi = ext.data_ptr(), ext.data_ptr() + ext.numel() * 4
                for name, prm in self.params:
                    g = prm.grad
                    if g is not None and lo <= g.data_ptr() < hi:
                        raise RuntimeError(
                            f"rbr_b200: `{name}.grad` still aliases the persistent (NVLS symmetric-memory) gradient arena, which "
                            "is re-zeroed by every backward: call zero_grad(set_to_none=True) before each step — gradient "
                            "accumulation over micro-batches is not supported with enable_nvls_allreduce")
                self.flat = ext[:self.total]
            else:
                self.flat = torch.empty(self.total, dtype=torch.float32, device=device)
            # zero-fill, except the slots a kernel is going to overwrite completely (the 60 MB word-table gradient)
            # (only the slot's own elements are skipped: the alignment gap behind it is zeroed like everything else, so the flat
            # buffer can be summed / all-reduced / fed to the fused optimizer as it is)
            skip = sorted((self.slots[i][0], self.slots[i][0] + self.slots[i][1].numel()) for i in self.no_zero if i in self.slots)
            pos = 0
            for lo, hi in skip + [(self.total, self.total)]:
                if lo > pos:
                    self.flat[pos:lo].zero_()
                pos = max(pos, hi)

    def view(self, prm: torch.Tensor) -> Optional[torch.Tensor]:
        slot = self.slots.get(id(prm))
        if slot is None:
            return None
        self._ensure(prm.device)
        off, shape = slot
        return self.flat[off:off + shape.numel()].view(shape)


def _grad_buf(arena: Optional[GradArena], prm: torch.Tensor, needs: bool) -> Optional[torch.Tensor]:
    if not needs:
        return None
    if arena is not None:
        v = arena.view(prm)
        if v is not None:
            return v
    return torch.zeros_like(prm)


# ---------------------------------------------------------------------------------------------------
# K1 / K1b: embedding gather
# ---------------------------------------------------------------------------------------------------
def gather_rows(table: torch.Tensor, ids: torch.Tensor) -> torch.Tensor:
    table = _req(table, torch.float32, "table")
    ids = _req(ids, torch.int64, "ids")
    out = torch.empty(*ids.shape, table.shape[1], dtype=torch.float32, device=table.device)
    lib.check(lib.rbr_gather_fwd(_p(table), table.shape[0], table.shape[1], _p(ids), ids.numel(), _p(out), _stream(True)),
              "rbr_gather_fwd")
    return out


def embedding_dense_grad(ids: torch.Tensor, grad_rows: torch.Tensor, vocab: int, padding_idx: Optional[int],
                         out: Optional[torch.Tensor] = None) -> torch.Tensor:
    ids = _req(ids, torch.int64, "ids")
    grad_rows = _req(grad_rows, torch.float32, "grad_rows")
    emb = grad_rows.shape[-1]
    if out is None:
        out = torch.zeros(vocab, emb, dtype=torch.float32, device=grad_rows.device)
    n = ids.numel()
    ws_bytes = lib.rbr_embgrad_workspace_bytes(n, vocab)
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=grad_rows.device)
    lib.check(lib.rbr_embgrad_scatter_add(_p(ids), _p(grad_rows), n, emb, vocab, -1 if padding_idx is None else padding_idx,
                                          _p(out), _p(ws), ws_bytes, _stream(True)), "rbr_embgrad_scatter_add")
    return out


class EmbeddingFn(torch.autograd.Function):
    """nn.Embedding forward/backward (reference models/deepconn/layers.py:15,23)."""

    @staticmethod
    def forward(ctx, table, ids, padding_idx, arena):
        _stream(refresh=True)
        ctx.save_for_backward(ids)
        ctx.vocab, ctx.padding_idx, ctx.arena, ctx.table = table.shape[0], padding_idx, arena, table
        return gather_rows(table, ids)

    @staticmethod
    def backward(ctx, grad_out):
        _stream(refresh=True)
        (ids,) = ctx.saved_tensors
        buf = _grad_buf(ctx.arena, ctx.table, True)
        embedding_dense_grad(ids, grad_out.contiguous(), ctx.vocab, ctx.padding_idx, out=buf)
        return buf, None, None, None


# ---------------------------------------------------------------------------------------------------
# K0 staging: bf16 shadow table + packed conv weights
# ---------------------------------------------------------------------------------------------------
def table_to_bf16(table: torch.Tensor) -> torch.Tensor:
    table = _req(table, torch.float32, "table")
    emb_pad = lib.rbr_emb_pad(table.shape[1])
    shadow = torch.empty(table.shape[0], emb_pad, dtype=torch.bfloat16, device=table.device)
    lib.check(lib.rbr_table_to_bf16(_p(table), table.shape[0], table.shape[1], _p(shadow), _stream(True)), "rbr_table_to_bf16")
    return shadow


def conv_pack(weight: torch.Tensor) -> torch.Tensor:
    weight = _req(weight, torch.float32, "conv weight")
    h, e, k = weight.shape
    nbytes = lib.rbr_conv_pack_bytes(e, h, k)
    packed = torch.empty(nbytes, dtype=torch.uint8, device=weight.device)
    lib.check(lib.rbr_conv_pack(_p(weight), e, h, k, _p(packed), _stream(True)), "rbr_conv_pack")
    return packed


# ---------------------------------------------------------------------------------------------------
# K2 / K2b: fused gather → mask → conv → activation → max-over-time, for one or several token tensors
# ("sides": DeepCoNN's user and item documents share the table and the conv, deepconn.py:43-47)
# ---------------------------------------------------------------------------------------------------
class EncodeDocsFn(torch.autograd.Function):
    """feats[s] = max_t act(conv(mask(table[ids[s]])))  for every side s; all sides share table/weights.

    Replaces WordEmbedding.forward + NgramFeat.forward (reference models/deepconn/layers.py:22-24, 123-136).
    Inputs after the fixed ones: n_conv conv weights, n_conv conv biases, then per side (ids, mask-or-None).
    """

    @staticmethod
    def forward(ctx, table, cfg, *rest):
        _stream(refresh=True)
        n_conv = cfg["n_conv"]
        weights, biases = rest[:n_conv], rest[n_conv:2 * n_conv]
        sides = rest[2 * n_conv:]
        ids_l = [_ids(t, "token ids") for t in sides[0::2]]
        mask_l = [_mask_u8(m, "token mask") for m in sides[1::2]]
        table = _req(table, torch.float32, "embedding table")
        prec = _PREC[cfg["precision"]]
        mfi = bool(cfg.get("mask_from_ids", False))
        flags_l = [cfg.get("flags", 0) | _id_flags(i, m, mfi) for i, m in zip(ids_l, mask_l)]
        act, pads = cfg["act"], cfg["pads"]
        vocab, emb = table.shape
        shadow = cfg["shadow_fn"]() if prec == PREC_BF16 else None
        packed = [cfg["pack_fn"](i) for i in range(n_conv)]
        h_total = sum(w.shape[0] for w in weights)
        feats, argmaxes, scratch = [], [], []
        for ids, mask in zip(ids_l, mask_l):             # every buffer is allocated on the calling stream, before the fork
            doc_len = ids.shape[-1]
            n_docs = ids.numel() // doc_len
            if mask is not None and mask.numel() != ids.numel():
                raise ValueError("rbr_b200: mask shape does not match token ids")
            feats.append(torch.empty(n_docs, h_total, dtype=torch.float32, device=table.device))
            argmaxes.append(torch.empty(n_docs, h_total, dtype=torch.int32, device=table.device))
            ws_bytes = (max(lib.rbr_conv_fwd_workspace_bytes2(n_docs, doc_len, w.shape[2], pad) for w, pad in zip(weights, pads))
                        if prec == PREC_BF16 else 0)
            scratch.append((torch.empty(ws_bytes, dtype=torch.uint8, device=table.device) if ws_bytes else None, ws_bytes))
        # The sides are independent: side s > 0 runs on its own stream, so its pre-pass kernels (document selection, row-index
        # table: a few small launches) overlap the previous side's tensor-core kernel, which leaves room for them on every SM.
        main = torch.cuda.current_stream()
        side_streams = _side_streams(table.device, max(0, len(ids_l) - 1))
        ev_fork = main.record_event() if len(ids_l) > 1 else None
        for s, (ids, mask, fl) in enumerate(zip(ids_l, mask_l, flags_l)):
            doc_len = ids.shape[-1]
            n_docs = ids.numel() // doc_len
            feat, amax, (ws, ws_bytes) = feats[s], argmaxes[s], scratch[s]
            stream_s = main if s == 0 else side_streams[s - 1]
            if s > 0:
                stream_s.wait_event(ev_fork)
            with torch.cuda.stream(stream_s):
                sh = _stream(refresh=True)
                col = 0
                for w, b, pk, pad in zip(weights, biases, packed, pads):
                    h, _, k = w.shape
                    lib.check(lib.rbr_conv_act_maxpool_fwd(
                        prec, act, _p(table), _p(shadow), vocab, emb, _p(ids), _p(mask), None, 0, n_docs, doc_len, _p(pk),
                        _p(_req(b, torch.float32, "conv bias")), h, k, pad, feat.data_ptr() + 4 * col, amax.data_ptr() + 4 * col,
                        None, h_total, _p(ws), ws_bytes, fl, sh), "rbr_conv_act_maxpool_fwd")
                    col += h
        for s in range(1, len(ids_l)):
            main.wait_event(side_streams[s - 1].record_event())
        _stream(refresh=True)
        del scratch
        ctx.cfg, ctx.n_conv, ctx.n_sides = cfg, n_conv, len(ids_l)
        ctx.table, ctx.weights, ctx.biases = table, weights, biases
        ctx.shadow, ctx.packed = shadow, packed
        ctx.save_for_backward(*ids_l, *[m for m in mask_l if m is not None], *feats, *argmaxes)
        ctx.mask_present = [m is not None for m in mask_l]
        ctx.flags_l = flags_l
        ctx.mark_non_differentiable(*argmaxes)
        ctx.set_materialize_grads(False)              # a side the loss does not use arrives as None and is skipped, not scattered as zeros
        return tuple(feats) + tuple(argmaxes)          # [n_docs, H] features per side, then the int32 arg-max positions

    @staticmethod
    def backward(ctx, *out_grads):
        _stream(refresh=True)
        cfg, n_conv, ns = ctx.cfg, ctx.n_conv, ctx.n_sides
        feat_grads = out_grads[:ns]
        saved = list(ctx.saved_tensors)
        ids_l = saved[:ns]
        n_masks = sum(ctx.mask_present)
        masks_present = saved[ns:ns + n_masks]
        feats = saved[ns + n_masks:ns + n_masks + ns]
        argmaxes = saved[ns + n_masks + ns:]
        mask_l, mi = [], 0
        for present in ctx.mask_present:
            mask_l.append(masks_present[mi] if present else None)
            mi += int(present)
        table = ctx.table
        arena: Optional[GradArena] = cfg.get("arena")
        prec = _PREC[cfg["precision"]]
        vocab, emb = table.shape
        need_table = ctx.needs_input_grad[0]
        g_table = _grad_buf(arena, cfg["table_param"], need_table)
        g_w = [_grad_buf(arena, cfg["weight_params"][i], True) for i in range(n_conv)]
        g_b = [_grad_buf(arena, cfg["bias_params"][i], True) for i in range(n_conv)]
        h_total = feats[0].shape[1]
        shapes = [tuple(w.shape) for w in ctx.weights]                   # (H, E, k) per conv
        cols = [sum(sh[0] for sh in shapes[:i]) for i in range(n_conv)]
        flags0 = cfg.get("flags", 0)
        # Formulation per conv: bf16 → the dense tensor-core backward over the coefficient matrix (K2c) when the shape allows,
        # else (fp32 precision, CONV_BWD_SPARSE, unsupported shapes) the arg-max-sparse CUDA-core kernels (K2b).
        dense = [prec == PREC_BF16 and not (flags0 & CONV_BWD_SPARSE) and ctx.shadow is not None and cfg.get("dense_bwd", True)
                 and bool(lib.rbr_conv_bwd_cmat_supported(vocab, emb, sh[0], sh[2])) for sh in shapes]
        if flags0 & CONV_BWD_DENSE_TC and not all(dense):
            raise RuntimeError("rbr_b200: CONV_BWD_DENSE_TC requested but the dense tensor-core backward does not take this shape / precision")
        cm_ws = {i: _cmat_workspace(table, i, vocab, emb, shapes[i][0], shapes[i][2]) for i in range(n_conv) if dense[i]}
        # The table gradient of every side is finished first (it is by far the largest gradient: data-parallel training starts
        # its all-reduce from the `table_ready` hook while the weight-gradient kernels still run), then the weight part.
        hook = cfg.get("table_ready") if need_table else None
        # The document sides are independent (they only meet in += accumulations, all atomic): side s > 0 runs on its own
        # stream, so the small kernels of one side overlap the other side's work.
        main = torch.cuda.current_stream()
        live = [s for s in range(ns) if feat_grads[s] is not None]
        side_streams = _side_streams(table.device, max(0, len(live) - 1))
        fgs = {s: feat_grads[s].contiguous() for s in live}

        def per_side(fn):
            ev_fork = main.record_event() if len(live) > 1 else None
            for rank_s, s in enumerate(live):
                stream_s = main if rank_s == 0 else side_streams[rank_s - 1]
                if rank_s > 0:
                    stream_s.wait_event(ev_fork)
                with torch.cuda.stream(stream_s):
                    fn(s, _stream(refresh=True))
            for rank_s in range(1, len(live)):
                main.wait_event(side_streams[rank_s - 1].record_event())
            _stream(refresh=True)

        def sparse_part(do_table, do_weight):
            def run(s, sh):
                ids, mask = ids_l[s], mask_l[s]
                doc_len = ids.shape[-1]
                n_docs = ids.numel() // doc_len
                for i in range(n_conv):
                    if dense[i]:
                        continue
                    h, _, k = shapes[i]
                    gt = g_table if do_table else None
                    if gt is None and not do_weight:
                        continue
                    ws_bytes = lib.rbr_conv_bwd_workspace_bytes(n_docs, h, k, emb, vocab)
                    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=table.device)
                    lib.check(lib.rbr_conv_act_maxpool_bwd(
                        prec, cfg["act"], _p(table), _p(ctx.shadow), vocab, emb, _p(ids), _p(mask), None, 0, n_docs, doc_len,
                        _p(ctx.packed[i]), h, k, cfg["pads"][i], feats[s].data_ptr() + 4 * cols[i],
                        argmaxes[s].data_ptr() + 4 * cols[i], fgs[s].data_ptr() + 4 * cols[i], None, h_total, cfg["padding_idx"],
                        _p(g_w[i]) if do_weight else None, _p(g_b[i]) if do_weight else None, _p(gt), None, _p(ws),
                        ws_bytes, ctx.flags_l[s], sh), "rbr_conv_act_maxpool_bwd")
            return run

        def dense_scatter_chunk(i, c):
            """Block c of conv i's coefficient matrix, one document side (run per side, possibly on two streams)."""
            ws = cm_ws[i]
            h, _, k = shapes[i]

            def run(s, sh):
                ids, mask = ids_l[s], mask_l[s]
                doc_len = ids.shape[-1]
                n_docs = ids.numel() // doc_len
                lib.check(lib.rbr_conv_bwd_cmat_scatter(
                    _p(ids), _p(mask), n_docs, doc_len, vocab, emb, h, k, cfg["pads"][i], cfg["act"],
                    feats[s].data_ptr() + 4 * cols[i], argmaxes[s].data_ptr() + 4 * cols[i], fgs[s].data_ptr() + 4 * cols[i],
                    h_total, _p(g_b[i]), c, _p(ws), ws.numel(), ctx.flags_l[s], sh), "rbr_conv_bwd_cmat_scatter")
            return run

        def dense_accumulate():
            """Per conv and filter block: zero-fill the block (it then sits in L2), scatter every side into it, split it into the
            bf16 hi|lo operand while it is still there."""
            for i, ws in cm_ws.items():
                h, _, k = shapes[i]
                for c in range(lib.rbr_conv_bwd_cmat_chunks(vocab, emb, h, k)):
                    lib.check(lib.rbr_conv_bwd_cmat_begin(c, vocab, emb, h, k, _p(ws), ws.numel(), _stream()), "rbr_conv_bwd_cmat_begin")
                    per_side(dense_scatter_chunk(i, c))
                    lib.check(lib.rbr_conv_bwd_cmat_finish(1, c, None, _p(ctx.packed[i]), vocab, emb, h, k, cfg["padding_idx"], None, None,
                                                           _p(ws), ws.numel(), _stream()), "rbr_conv_bwd_cmat_finish")

        # the arena left the table slot un-zeroed because this backward writes every element of it (NgramFeat.encode decided)
        overwrite = bool(cfg.get("table_overwrite")) and need_table and arena is not None and id(cfg["table_param"]) in arena.no_zero
        if overwrite and not (all(dense) and n_conv == 1 and live):
            g_table.zero_()                 # nothing will overwrite it after all
            overwrite = False

        def dense_finish(what):
            if overwrite and (what & 2):
                what |= 8
            for i, ws in cm_ws.items():
                h, _, k = shapes[i]
                lib.check(lib.rbr_conv_bwd_cmat_finish(what, -1, _p(ctx.shadow), _p(ctx.packed[i]), vocab, emb, h, k,
                                                       cfg["padding_idx"], _p(g_table), _p(g_w[i]), _p(ws), ws.numel(), _stream()),
                          "rbr_conv_bwd_cmat_finish")

        any_sparse = not all(dense)
        if live:
            two_pass = hook is not None
            if any_sparse:
                per_side(sparse_part(True, not two_pass) if need_table else sparse_part(False, True))
            if cm_ws:
                dense_accumulate()
            if cm_ws and need_table:
                dense_finish(2)
            if hook is not None:
                hook(g_table)
            if any_sparse and two_pass:
                per_side(sparse_part(False, True))
            if cm_ws:
                dense_finish(4)
        return (g_table, None, *g_w, *g_b, *([None] * (2 * ns)))


_CMAT_WS: Dict[tuple, torch.Tensor] = {}


def _cmat_workspace(table: torch.Tensor, conv_index: int, vocab: int, emb: int, filters: int, ksize: int) -> torch.Tensor:
    """Persistent workspace of the dense tensor-core backward (K2c) for one (table, conv), allocated once per shape.  Only the
    weight scratch is self-cleaning (the unpack kernel re-zeroes what it reads); each filter block of the coefficient matrix C32 is
    zero-filled by rbr_conv_bwd_cmat_begin right before its scatter, while the block is about to be hot in L2."""
    key = (table.device.index, table.data_ptr(), conv_index, vocab, emb, filters, ksize)
    ws = _CMAT_WS.get(key)
    if ws is None:
        for k in [k for k in _CMAT_WS if k[:2] == key[:2] and k[2] == conv_index]:
            del _CMAT_WS[k]                        # same table storage, new shape: the old buffer is dead
        nbytes = lib.rbr_conv_bwd_cmat_workspace_bytes(vocab, emb, filters, ksize)
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("rbr_b200: run one eager step before capturing a CUDA graph (the dense backward's workspace is "
                               "allocated and zero-filled on first use)")
        while len(_CMAT_WS) >= 8:                  # a handful of (model, conv) pairs per process; drop the oldest beyond that
            del _CMAT_WS[next(iter(_CMAT_WS))]
        ws = torch.zeros(nbytes, dtype=torch.uint8, device=table.device)
        _CMAT_WS[key] = ws
    return ws


class HierPoolFn(torch.autograd.Function):
    """pooled[s] = max_t mean_{j<k} mask(table[ids[s]])[t+j]  per document and embedding channel, for every side s —
    HierPooling.forward (reference models/deepconn/layers.py:81-98) on the masked embeddings (layers.py:131-133).
    All sides go through ONE autograd node: they share the table, whose gradient buffer is accumulated into by every side and
    handed to autograd once.  Inputs after (table, cfg): per side (ids, mask-or-None).  → [n_docs, E] per side."""

    @staticmethod
    def forward(ctx, table, cfg, *flat):
        _stream(refresh=True)
        table = _req(table, torch.float32, "embedding table")
        vocab, emb = table.shape
        ids_l = [_ids(t, "token ids") for t in flat[0::2]]
        mask_l = [_mask_u8(m, "token mask") for m in flat[1::2]]
        flags_l = [_id_flags(i, m, bool(cfg.get("mask_from_ids", False))) for i, m in zip(ids_l, mask_l)]
        outs, amaxes = [], []
        for ids, mask, fl in zip(ids_l, mask_l, flags_l):
            doc_len = ids.shape[-1]
            n_docs = ids.numel() // doc_len
            pooled = torch.empty(n_docs, emb, dtype=torch.float32, device=table.device)
            amax = torch.empty(n_docs, emb, dtype=torch.int32, device=table.device)
            lib.check(lib.rbr_hier_pool_fwd(_p(table), vocab, emb, _p(ids), _p(mask), n_docs, doc_len, cfg["ksize"], _p(pooled), _p(amax),
                                            fl, _stream()), "rbr_hier_pool_fwd")
            outs.append(pooled)
            amaxes.append(amax)
        ctx.save_for_backward(*ids_l, *amaxes, *[m for m in mask_l if m is not None])
        ctx.cfg, ctx.flags_l, ctx.mask_present, ctx.shape = cfg, flags_l, [m is not None for m in mask_l], (vocab, emb)
        return tuple(outs)

    @staticmethod
    def backward(ctx, *grads):
        _stream(refresh=True)
        cfg = ctx.cfg
        ns = len(ctx.flags_l)
        vocab, emb = ctx.shape
        if not ctx.needs_input_grad[0]:
            return (None,) * (2 + 2 * ns)
        saved = ctx.saved_tensors
        ids_l, amaxes, masks = saved[:ns], saved[ns:2 * ns], list(saved[2 * ns:])
        g_table = _grad_buf(cfg.get("arena"), cfg["table_param"], True)
        for s in range(ns):
            mask = masks.pop(0) if ctx.mask_present[s] else None
            if grads[s] is None:
                continue
            ids = ids_l[s]
            doc_len = ids.shape[-1]
            lib.check(lib.rbr_hier_pool_bwd(_p(ids), _p(mask), ids.numel() // doc_len, doc_len, vocab, emb, cfg["ksize"], cfg["padding_idx"],
                                            _p(amaxes[s]), _p(grads[s].contiguous()), _p(g_table), ctx.flags_l[s], _stream()),
                      "rbr_hier_pool_bwd")
        return (g_table, None, *([None] * (2 * ns)))


class MaskedAvgPoolFn(torch.autograd.Function):
    """out[s][n, :] = sum_t mask * table[ids[s][n, t]] / (sum_t mask + 1e-8) for every side s (K9) — the SimpleSiamese encoder
    (reference models/simple_siamese/layers.py:90-110 on the gathered embeddings).  One autograd node for all sides (shared
    table gradient).  Inputs after (table, cfg): per side (ids [n_docs, T], mask-or-None)."""

    @staticmethod
    def forward(ctx, table, cfg, *flat):
        _stream(refresh=True)
        table = _req(table, torch.float32, "embedding table")
        vocab, emb = table.shape
        ids_l = [_ids(t, "token ids") for t in flat[0::2]]
        mask_l = [_mask_u8(m, "token mask") for m in flat[1::2]]
        flags_l = [_id_flags(i, m, bool(cfg.get("mask_from_ids", False))) for i, m in zip(ids_l, mask_l)]
        outs = []
        for ids, mask, fl in zip(ids_l, mask_l, flags_l):
            doc_len = ids.shape[-1]
            n_docs = ids.numel() // doc_len
            out = torch.empty(n_docs, emb, dtype=torch.float32, device=table.device)
            lib.check(lib.rbr_masked_avg_pool_fwd(_p(table), vocab, emb, _p(ids), _p(mask), n_docs, doc_len, _p(out), fl, _stream()),
                      "rbr_masked_avg_pool_fwd")
            outs.append(out)
        ctx.save_for_backward(*ids_l, *[m for m in mask_l if m is not None])
        ctx.cfg, ctx.flags_l, ctx.mask_present, ctx.shape = cfg, flags_l, [m is not None for m in mask_l], (vocab, emb)
        return tuple(outs)

    @staticmethod
    def backward(ctx, *grads):
        _stream(refresh=True)
        cfg = ctx.cfg
        ns = len(ctx.flags_l)
        vocab, emb = ctx.shape
        if not ctx.needs_input_grad[0]:
            return (None,) * (2 + 2 * ns)
        saved = ctx.saved_tensors
        ids_l, masks = saved[:ns], list(saved[ns:])
        g_table = _grad_buf(cfg.get("arena"), cfg["table_param"], True)
        for s in range(ns):
            mask = masks.pop(0) if ctx.mask_present[s] else None
            if grads[s] is None:
                continue
            ids = ids_l[s]
            doc_len = ids.shape[-1]
            lib.check(lib.rbr_masked_avg_pool_bwd(_p(ids), _p(mask), ids.numel() // doc_len, doc_len, vocab, emb, cfg["padding_idx"],
                                                  _p(grads[s].contiguous()), _p(g_table), ctx.flags_l[s], _stream()),
                      "rbr_masked_avg_pool_bwd")
        return (g_table, None, *([None] * (2 * ns)))


# ---------------------------------------------------------------------------------------------------
# K3: NARRE attention
# ---------------------------------------------------------------------------------------------------
class NarreAttnFn(torch.autograd.Function):
    """LinearAttention.forward without dropout (reference models/narre/narre.py:40-60)."""

    @staticmethod
    def forward(ctx, feat, other_id, W_rv, W_id, h, b_1, b_2, ebd, padding_idx, arena, params):
        _stream(refresh=True)
        feat = _req(feat, torch.float32, "feat")
        other_id = _req(other_id, torch.int64, "other_id")
        B, R, H = feat.shape
        A = W_rv.shape[1]
        out = torch.empty(B, H, dtype=torch.float32, device=feat.device)
        scores = torch.empty(B, R, dtype=torch.float32, device=feat.device)
        args = [_req(t, torch.float32, n) for t, n in ((W_rv, "W_rv"), (W_id, "W_id"), (h, "h"), (b_1, "b_1"), (b_2, "b_2"),
                                                        (ebd, "ebd_vals"))]
        lib.check(lib.rbr_narre_attn_fwd(_p(feat), _p(other_id), B, R, H, A, *[_p(a) for a in args], ebd.shape[0], _p(out),
                                         _p(scores), _stream()), "rbr_narre_attn_fwd")
        ctx.save_for_backward(feat, other_id, scores, *args)
        ctx.padding_idx, ctx.arena, ctx.params = padding_idx, arena, params
        # an output the loss does not use (usually the scores) reaches backward as None rather than a zero-filled tensor:
        # the kernels then skip the score-gradient term
        ctx.set_materialize_grads(False)
        return out, scores.view(B, R, 1)

    @staticmethod
    def backward(ctx, g_out, g_scores):
        _stream(refresh=True)
        feat, other_id, scores, W_rv, W_id, h, b_1, b_2, ebd = ctx.saved_tensors
        B, R, H = feat.shape
        A = W_rv.shape[1]
        g_out = torch.zeros(B, H, device=feat.device) if g_out is None else g_out.contiguous()
        g_scores = None if g_scores is None else g_scores.contiguous()
        g_feat = torch.empty_like(feat)
        grads = [_grad_buf(ctx.arena, p, True) for p in ctx.params]
        lib.check(lib.rbr_narre_attn_bwd(_p(feat), _p(other_id), B, R, H, A, _p(W_rv), _p(W_id), _p(h), _p(b_1), _p(b_2), _p(ebd),
                                         ebd.shape[0], -1 if ctx.padding_idx is None else ctx.padding_idx, _p(scores), _p(g_out),
                                         _p(g_scores), _p(g_feat), *[_p(g) for g in grads], _stream()), "rbr_narre_attn_bwd")
        return (g_feat, None, *grads, None, None, None)


def _ptr_array(ptrs):
    import ctypes
    return (ctypes.c_void_p * len(ptrs))(*[None if p is None else int(p) for p in ptrs])


def _i64_array(vals):
    import ctypes
    return (ctypes.c_int64 * len(vals))(*[int(v) for v in vals])


class NarreAttnPairFn(torch.autograd.Function):
    """Both LinearAttention modules of NARRE (narre.py:184-185) in ONE launch per direction on the tensor cores
    (csrc/attn_tc.cu).  Inputs: feat_u, id_u, feat_i, id_i, then the 6 parameters of each side
    (W_rv, W_id, h, b_1, b_2, ebd_vals).  Returns (out_u, scores_u [B,R,1], out_i, scores_i [B,R,1]), dropout excluded."""

    @staticmethod
    def forward(ctx, feat_u, id_u, feat_i, id_i, *rest):
        _stream(refresh=True)
        prm = [_req(t, torch.float32, "attention parameter") for t in rest[:12]]
        pads, arena, params = rest[12], rest[13], rest[14]
        feats = [_req(feat_u, torch.float32, "feat"), _req(feat_i, torch.float32, "feat")]
        ids = [_req(id_u, torch.int64, "other_id"), _req(id_i, torch.int64, "other_id")]
        B, R, H = feats[0].shape
        if feats[1].shape != feats[0].shape:
            raise ValueError("rbr_b200: the two attention sides must have the same [B, R, H] shape")
        A = prm[0].shape[1]
        outs = [torch.empty(B, H, dtype=torch.float32, device=feats[0].device) for _ in range(2)]
        scores = [torch.empty(B, R, dtype=torch.float32, device=feats[0].device) for _ in range(2)]
        side = [prm[:6], prm[6:]]
        lib.check(lib.rbr_narre_attn_pair_fwd(
            2, _ptr_array([_p(f) for f in feats]), _ptr_array([_p(i) for i in ids]), B, R, H, A,
            *[_ptr_array([_p(side[0][j]), _p(side[1][j])]) for j in range(6)],
            _i64_array([side[0][5].shape[0], side[1][5].shape[0]]), _ptr_array([_p(o) for o in outs]),
            _ptr_array([_p(s) for s in scores]), _stream()), "rbr_narre_attn_pair_fwd")
        ctx.save_for_backward(*feats, *ids, *scores, *prm)
        ctx.pads, ctx.arena, ctx.params = pads, arena, params
        return outs[0], scores[0].view(B, R, 1), outs[1], scores[1].view(B, R, 1)

    @staticmethod
    def backward(ctx, g_out_u, g_sc_u, g_out_i, g_sc_i):
        _stream(refresh=True)
        saved = ctx.saved_tensors
        feats, ids, scores, prm = saved[0:2], saved[2:4], saved[4:6], saved[6:18]
        B, R, H = feats[0].shape
        A = prm[0].shape[1]
        dev = feats[0].device
        g_outs = [torch.zeros(B, H, device=dev) if g is None else g.contiguous() for g in (g_out_u, g_out_i)]
        g_scs = [None if g is None else g.contiguous() for g in (g_sc_u, g_sc_i)]
        g_feats = [torch.empty_like(feats[0]), torch.empty_like(feats[1])]
        grads = [_grad_buf(ctx.arena, p, True) for p in ctx.params]             # 12: side u then side i
        side, gside = [prm[:6], prm[6:]], [grads[:6], grads[6:]]
        pads = [-1 if x is None else int(x) for x in ctx.pads]
        any_sc = any(g is not None for g in g_scs)
        lib.check(lib.rbr_narre_attn_pair_bwd(
            2, _ptr_array([_p(f) for f in feats]), _ptr_array([_p(i) for i in ids]), B, R, H, A,
            *[_ptr_array([_p(side[0][j]), _p(side[1][j])]) for j in range(6)],
            _i64_array([side[0][5].shape[0], side[1][5].shape[0]]), _i64_array(pads), _ptr_array([_p(s) for s in scores]),
            _ptr_array([_p(g) for g in g_outs]), _ptr_array([_p(g) for g in g_scs]) if any_sc else None,
            _ptr_array([_p(g) for g in g_feats]),
            *[_ptr_array([_p(gside[0][j]), _p(gside[1][j])]) for j in range(6)], _stream()), "rbr_narre_attn_pair_bwd")
        return (g_feats[0], None, g_feats[1], None, *grads, None, None, None)


def narre_attn_pair_supported(R: int, H: int, A: int) -> bool:
    return bool(lib.rbr_narre_attn_pair_supported(R, H, A))


# ---------------------------------------------------------------------------------------------------
# K4: LastFeat x2 + FM head
# ---------------------------------------------------------------------------------------------------
class HeadFn(torch.autograd.Function):
    """pred = FM(LastFeat_u(u_text, u_id), LastFeat_i(i_text, i_id))  (reference layers.py:156-165, 188-209)."""

    @staticmethod
    def forward(ctx, u_text, i_text, u_id, i_id, Wu, bu, ebd_u, Wi, bi, ebd_i, fm_h, user_bias, item_bias, g_bias, drop_p,
                drop_seed, padding_idx, arena, params, seed_dev=None):
        """padding_idx: one int / None for all four id tables, or a 4-tuple (LastFeat_u.ebd, LastFeat_i.ebd, FM.user_bias,
        FM.item_bias) — each nn.Embedding keeps its own padding row."""
        _stream(refresh=True)
        u_text = _req(u_text, torch.float32, "u_text")
        i_text = _req(i_text, torch.float32, "i_text")
        u_id = _req(u_id, torch.int64, "u_id")
        i_id = _req(i_id, torch.int64, "i_id")
        B, H = u_text.shape
        K = Wu.shape[1]
        fl = [_req(t, torch.float32, "head parameter") for t in (Wu, bu, ebd_u, Wi, bi, ebd_i, fm_h, user_bias, item_bias, g_bias)]
        pred = torch.empty(B, dtype=torch.float32, device=u_text.device)
        u_lat = torch.empty(B, K, dtype=torch.float32, device=u_text.device)
        i_lat = torch.empty(B, K, dtype=torch.float32, device=u_text.device)
        lib.check(lib.rbr_head_fwd(_p(u_text), _p(i_text), _p(u_id), _p(i_id), B, H, K, *[_p(t) for t in fl], ebd_u.shape[0],
                                   ebd_i.shape[0], float(drop_p), int(drop_seed), _p(seed_dev), _p(pred), _p(u_lat), _p(i_lat), None,
                                   0.0, None, None, _stream()), "rbr_head_fwd")
        ctx.save_for_backward(u_text, i_text, u_id, i_id, fl[0], fl[3], fl[6], u_lat, i_lat)
        if not isinstance(padding_idx, (tuple, list)):
            padding_idx = (padding_idx,) * 4
        padding_idx = tuple(-1 if x is None else int(x) for x in padding_idx)
        ctx.drop, ctx.padding_idx, ctx.arena, ctx.params = (float(drop_p), int(drop_seed), seed_dev), padding_idx, arena, params
        ctx.sizes = (ebd_u.shape[0], ebd_i.shape[0])
        return pred

    @staticmethod
    def backward(ctx, g_pred):
        _stream(refresh=True)
        u_text, i_text, u_id, i_id, Wu, Wi, fm_h, u_lat, i_lat = ctx.saved_tensors
        B, H = u_text.shape
        K = Wu.shape[1]
        g_pred = g_pred.contiguous()
        g_ut, g_it = torch.empty_like(u_text), torch.empty_like(i_text)
        # params order: Wu, bu, ebd_u, Wi, bi, ebd_i, fm_h, user_bias, item_bias, g_bias
        grads = [_grad_buf(ctx.arena, p, True) for p in ctx.params]
        lib.check(lib.rbr_head_bwd(_p(u_text), _p(i_text), _p(u_id), _p(i_id), B, H, K, _p(Wu), _p(Wi), _p(fm_h), _p(u_lat),
                                   _p(i_lat), ctx.drop[0], ctx.drop[1], _p(ctx.drop[2]), *ctx.padding_idx,
                                   ctx.sizes[0], ctx.sizes[1], _p(g_pred), _p(g_ut), _p(g_it), *[_p(g) for g in grads],
                                   _stream()), "rbr_head_bwd")
        return (g_ut, g_it, None, None, *grads, None, None, None, None, None, None)


class HeadLossFn(torch.autograd.Function):
    """(loss, pred) = (MSELoss(pred, ratings), pred) with pred as in HeadFn: the fused-MSE branch of rbr_head_fwd
    (reference layers.py:156-165, 188-209 + trainer/train_deepconn_pp.py:140,164: nn.MSELoss(), reduction 'mean').
    The forward launch also writes d loss / d pred = 2 (pred - rating) / B, so the backward is one rbr_head_bwd launch."""

    @staticmethod
    def forward(ctx, u_text, i_text, u_id, i_id, ratings, Wu, bu, ebd_u, Wi, bi, ebd_i, fm_h, user_bias, item_bias, g_bias,
                drop_p, drop_seed, padding_idx, arena, params, seed_dev=None):
        _stream(refresh=True)
        u_text = _req(u_text, torch.float32, "u_text")
        i_text = _req(i_text, torch.float32, "i_text")
        u_id = _req(u_id, torch.int64, "u_id")
        i_id = _req(i_id, torch.int64, "i_id")
        ratings = _req(ratings, torch.float32, "ratings").view(-1)
        B, H = u_text.shape
        if ratings.numel() != B:
            raise ValueError("rbr_b200: ratings must have one value per sample")
        K = Wu.shape[1]
        fl = [_req(t, torch.float32, "head parameter") for t in (Wu, bu, ebd_u, Wi, bi, ebd_i, fm_h, user_bias, item_bias, g_bias)]
        dev = u_text.device
        pred = torch.empty(B, dtype=torch.float32, device=dev)
        u_lat = torch.empty(B, K, dtype=torch.float32, device=dev)
        i_lat = torch.empty(B, K, dtype=torch.float32, device=dev)
        pred_grad = torch.empty(B, dtype=torch.float32, device=dev)
        loss = torch.zeros((), dtype=torch.float32, device=dev)         # the kernel accumulates sum (pred - rating)^2 / B into it
        lib.check(lib.rbr_head_fwd(_p(u_text), _p(i_text), _p(u_id), _p(i_id), B, H, K, *[_p(t) for t in fl], ebd_u.shape[0],
                                   ebd_i.shape[0], float(drop_p), int(drop_seed), _p(seed_dev), _p(pred), _p(u_lat), _p(i_lat),
                                   _p(ratings), 1.0 / B, _p(loss), _p(pred_grad), _stream()), "rbr_head_fwd")
        ctx.save_for_backward(u_text, i_text, u_id, i_id, fl[0], fl[3], fl[6], u_lat, i_lat, pred_grad)
        if not isinstance(padding_idx, (tuple, list)):
            padding_idx = (padding_idx,) * 4
        padding_idx = tuple(-1 if x is None else int(x) for x in padding_idx)
        ctx.drop, ctx.padding_idx, ctx.arena, ctx.params = (float(drop_p), int(drop_seed), seed_dev), padding_idx, arena, params
        ctx.sizes = (ebd_u.shape[0], ebd_i.shape[0])
        ctx.mark_non_differentiable(pred)
        return loss, pred

    @staticmethod
    def backward(ctx, g_loss, g_pred):
        _stream(refresh=True)
        u_text, i_text, u_id, i_id, Wu, Wi, fm_h, u_lat, i_lat, pred_grad = ctx.saved_tensors
        B, H = u_text.shape
        K = Wu.shape[1]
        pg = pred_grad * g_loss                         # upstream d / d loss (a device scalar: no host read)
        g_ut, g_it = torch.empty_like(u_text), torch.empty_like(i_text)
        grads = [_grad_buf(ctx.arena, p, True) for p in ctx.params]
        lib.check(lib.rbr_head_bwd(_p(u_text), _p(i_text), _p(u_id), _p(i_id), B, H, K, _p(Wu), _p(Wi), _p(fm_h), _p(u_lat),
                                   _p(i_lat), ctx.drop[0], ctx.drop[1], _p(ctx.drop[2]), *ctx.padding_idx,
                                   ctx.sizes[0], ctx.sizes[1], _p(pg), _p(g_ut), _p(g_it), *[_p(g) for g in grads],
                                   _stream()), "rbr_head_bwd")
        return (g_ut, g_it, None, None, None, *grads, None, None, None, None, None, None)


def head_supported(hidden: int, latent: int) -> bool:
    """Whether the fused head kernels (K4) take this shape: both LastFeat weights, their CTA-partial gradients and a 32-sample
    tile must fit shared memory (csrc/head.cu)."""
    bwd = (2 * hidden * (latent + 1) + 2 * hidden * latent + 2 * 32 * hidden + 2 * 32 * latent) * 4
    return latent <= 128 and bwd <= 200 * 1024


def head_dropout_mask(batch: int, latent: int, drop_p: float, drop_seed: int, seed_dev: Optional[torch.Tensor],
                      device=None) -> torch.Tensor:
    """The FM dropout keep-scale [B, K] (values 0 or 1/(1-p)) the head kernels apply for this (p, seed, device counter) — a
    test / debug aid: the mask is a counter hash, not torch's Philox stream, so parity at p > 0 is checked by feeding this mask
    to the oracle."""
    dev = device or (seed_dev.device if seed_dev is not None else torch.device("cuda"))
    keep = torch.empty(batch, latent, dtype=torch.float32, device=dev)
    lib.check(lib.rbr_head_dropout_mask(batch, latent, float(drop_p), int(drop_seed), _p(seed_dev), _p(keep), _stream(True)),
              "rbr_head_dropout_mask")
    return keep


# ---------------------------------------------------------------------------------------------------
# Raw (no-autograd) entry used by the kernel-level tests and by bench.py's per-kernel roofline timing
# ---------------------------------------------------------------------------------------------------
def conv_act_maxpool(table: torch.Tensor, ids: torch.Tensor, mask: Optional[torch.Tensor], weight: torch.Tensor,
                     bias: torch.Tensor, pad: int, act: int = ACT_RELU, precision: str = "bf16",
                     shadow: Optional[torch.Tensor] = None, packed: Optional[torch.Tensor] = None, flags: int = 0,
                     mask_from_ids: bool = False, select_docs: bool = True, row_index_table: bool = True,
                     gate: Optional[torch.Tensor] = None, gate_mode: int = 0, return_pool_raw: bool = False,
                     feat_ld: Optional[int] = None):
    """One K2 launch: returns (feat [n_docs, H] fp32, argmax [n_docs, H] int32).  `flags`: CONV_TC_* kernel selection.
    `select_docs=False`: no scratch at all; `row_index_table=False`: scratch for the document selection only, so the kernel's
    index warp resolves ids and masks itself (rbr_conv_fwd_workspace_bytes vs ..._bytes2).
    `gate` / `gate_mode`: D-ATT's gate, passed straight to the C-ABI (1: per token [n_docs, doc_len], k = 1; 2: per document
    [n_docs]).  `return_pool_raw`: also return pool_raw [n_docs, H], the pooled value before bias and activation.
    `feat_ld` (>= H): row stride of the outputs, which are then [n_docs, feat_ld]; columns H.. are NaN (feat, pool_raw) and
    -1 (argmax) unless the kernel wrote past its filters."""
    table = _req(table, torch.float32, "table")
    ids = _ids(ids, "ids")
    flags |= _id_flags(ids, mask, mask_from_ids)
    mask = _mask_u8(mask, "mask")
    prec = _PREC[precision]
    if prec == PREC_BF16 and shadow is None:
        shadow = table_to_bf16(table)
    if packed is None:
        packed = conv_pack(weight)
    if gate is not None:
        gate = _req(gate, torch.float32, "gate")
    h, emb, k = weight.shape
    doc_len = ids.shape[-1]
    n_docs = ids.numel() // doc_len
    ld = h if feat_ld is None else feat_ld
    dev = table.device
    if ld > h:
        feat = torch.full((n_docs, ld), float("nan"), device=dev)
        amax = torch.full((n_docs, ld), -1, dtype=torch.int32, device=dev)
    else:
        feat = torch.empty(n_docs, h, dtype=torch.float32, device=dev)
        amax = torch.empty(n_docs, h, dtype=torch.int32, device=dev)
    pool_raw = torch.full((n_docs, ld), float("nan"), device=dev) if return_pool_raw else None
    ws_bytes = 0
    if prec == PREC_BF16 and select_docs:
        ws_bytes = (lib.rbr_conv_fwd_workspace_bytes2(n_docs, doc_len, k, pad) if row_index_table
                    else lib.rbr_conv_fwd_workspace_bytes(n_docs))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=table.device) if ws_bytes else None
    lib.check(lib.rbr_conv_act_maxpool_fwd(prec, act, _p(table), _p(shadow), table.shape[0], emb, _p(ids), _p(mask), _p(gate),
                                           gate_mode, n_docs, doc_len, _p(packed), _p(_req(bias, torch.float32, "bias")), h, k, pad,
                                           _p(feat), _p(amax), _p(pool_raw), ld, _p(ws), ws_bytes, flags, _stream(True)),
              "rbr_conv_act_maxpool_fwd")
    return (feat, amax, pool_raw) if return_pool_raw else (feat, amax)


# ---------------------------------------------------------------------------------------------------
# K5 + gated K2: one side of the D-ATT encoder (local attention + global attention), ids → [N, l_out + 3*g_out]
# ---------------------------------------------------------------------------------------------------
def datt_side_packs(prm: Sequence[torch.Tensor]) -> List[torch.Tensor]:
    """conv_pack of one D-ATT side's four conv weights (local k = 1, then global k = 2, 3, 4) from its 12 parameters
    (DattEncodeFn's order)."""
    return [conv_pack(prm[i]) for i in (2, 6, 8, 10)]


def datt_encode_side(table: torch.Tensor, ids: torch.Tensor, prm: Sequence[torch.Tensor], precision: str = "bf16",
                     shadow: Optional[torch.Tensor] = None, packed: Optional[Sequence[torch.Tensor]] = None,
                     stream: Optional[int] = None, conv_flags: int = 0
                     ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """One side of the D-ATT encoder forward (models/dual_att/layers.py:43-53, 81-89): K5's two gates, then the four gated
    tanh convs with max-over-time.  ids [n_docs, doc_len] int64 / int32; prm = the side's 12 parameters in DattEncodeFn's
    order; shadow = the bf16 table (bf16 only; made here when None); packed = datt_side_packs(prm) (made here when None);
    stream = a raw stream handle (None: torch's current stream); conv_flags = CONV_TC_* kernel selection for the four convs.
    Returns (feat [n_docs, l_out + 3 g_out], argmax int32, pre-activation at the arg-max, gate_local [n_docs, doc_len],
    gate_global [n_docs]); filter columns: local conv, then the k = 2, 3, 4 global convs."""
    table = _req(table, torch.float32, "embedding table")
    ids = _ids(ids, "token ids")
    prm = [_req(t, torch.float32, "D-ATT parameter") for t in prm]
    prec = _PREC[precision]
    if prec == PREC_BF16 and shadow is None:
        shadow = table_to_bf16(table)
    if packed is None:
        packed = datt_side_packs(prm)
    vocab, emb = table.shape
    dev = table.device
    idf = _id_width_flag(ids)
    la_w, la_b, lc_w, lc_b, ga_w, ga_b = prm[:6]
    g_convs = [(prm[6 + 2 * i], prm[7 + 2 * i]) for i in range(3)]
    n_docs, doc_len = ids.shape
    win = la_w.shape[2]
    s = _stream(True) if stream is None else stream
    ws_bytes = lib.rbr_datt_gate_workspace_bytes(n_docs, doc_len, emb, win, vocab)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    gate_l = torch.empty(n_docs, doc_len, dtype=torch.float32, device=dev)
    gate_g = torch.empty(n_docs, dtype=torch.float32, device=dev)
    lib.check(lib.rbr_datt_gate_fwd(_p(table), vocab, emb, _p(ids), n_docs, doc_len, _p(la_w), _p(la_b), win, _p(ga_w),
                                    _p(ga_b), _p(gate_l), _p(gate_g), _p(ws), ws_bytes, idf, s), "rbr_datt_gate_fwd")
    convs = [(lc_w, lc_b, gate_l, 1)] + [(w, b, gate_g, 2) for w, b in g_convs]
    h_total = sum(w.shape[0] for w, _, _, _ in convs)
    feat = torch.empty(n_docs, h_total, dtype=torch.float32, device=dev)
    amax = torch.empty(n_docs, h_total, dtype=torch.int32, device=dev)
    pre = torch.empty(n_docs, h_total, dtype=torch.float32, device=dev)
    col = 0
    ws_bytes = (max(lib.rbr_conv_fwd_workspace_bytes2(n_docs, doc_len, w.shape[2], 0) for w, _, _, _ in convs)
                if prec == PREC_BF16 else 0)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev) if ws_bytes else None
    for (w, b, gate, mode), pk in zip(convs, packed):
        h, _, k = w.shape
        lib.check(lib.rbr_conv_act_maxpool_fwd(prec, ACT_TANH, _p(table), _p(shadow), vocab, emb, _p(ids), None, _p(gate),
                                               mode, n_docs, doc_len, _p(pk), _p(b), h, k, 0, feat.data_ptr() + 4 * col,
                                               amax.data_ptr() + 4 * col, pre.data_ptr() + 4 * col, h_total, _p(ws), ws_bytes,
                                               idf | conv_flags, s), "rbr_conv_act_maxpool_fwd")
        col += h
    return feat, amax, pre, gate_l, gate_g


# ---------------------------------------------------------------------------------------------------
# K5 + gated K2: one side of the D-ATT encoder (local attention + global attention), ids → [N, l_out + 3*g_out]
# ---------------------------------------------------------------------------------------------------
class DattEncodeFn(torch.autograd.Function):
    """feats[s] = cat(LocalAttention_s(x_s), *GlobalAttention_s(x_s)) for x_s = table[ids_s], s in (user, item)
    (reference models/dual_att/layers.py:43-53, 81-89 and dual_att.py:45-50, 53-56), without materialising x, its
    permuted copy or the gated copies.  Both sides go through ONE autograd node because they share the embedding table
    (dual_att.py:22): its gradient buffer is accumulated into by both and handed to autograd once.

    Inputs after (table, cfg): per side (ids, then 12 parameters: local attn w, b; local conv w, b; global attn w, b;
    conv1 w, b; conv2 w, b; conv3 w, b)."""

    N_PRM = 12

    @staticmethod
    def forward(ctx, table, cfg, *rest):
        _stream(refresh=True)
        table = _req(table, torch.float32, "embedding table")
        stride = 1 + DattEncodeFn.N_PRM
        n_sides = len(rest) // stride
        prec = _PREC[cfg["precision"]]
        shadow = cfg["shadow_fn"]() if prec == PREC_BF16 else None
        saved, feats, side_ctx = [], [], []
        for s in range(n_sides):
            ids = _ids(rest[s * stride], "token ids")
            prm = [_req(t, torch.float32, "D-ATT parameter") for t in rest[s * stride + 1:(s + 1) * stride]]
            packed = datt_side_packs(prm)
            feat, amax, pre, gate_l, gate_g = datt_encode_side(table, ids, prm, cfg["precision"], shadow, packed, _stream(),
                                                               cfg.get("flags", 0))
            saved += [ids, gate_l, gate_g, feat, amax, pre]
            feats.append(feat)
            side_ctx.append((prm, packed))
        ctx.cfg, ctx.table, ctx.shadow, ctx.side_ctx, ctx.n_sides = cfg, table, shadow, side_ctx, n_sides
        ctx.save_for_backward(*saved)
        return tuple(feats)

    @staticmethod
    def backward(ctx, *feat_grads):
        _stream(refresh=True)
        cfg, table = ctx.cfg, ctx.table
        arena: Optional[GradArena] = cfg.get("arena")
        prec = _PREC[cfg["precision"]]
        vocab, emb = table.shape
        dev = table.device
        need_table = ctx.needs_input_grad[0]
        g_table = _grad_buf(arena, cfg["table_param"], need_table)
        ret = []
        # the user and item sides only meet in the (atomic) table gradient: the second side runs on its own stream
        main = torch.cuda.current_stream()
        side_streams = _side_streams(dev, max(0, ctx.n_sides - 1))
        # every buffer the side stream accumulates into is allocated AND zero-filled on the main stream before the fork event
        # (a frozen table or arena=None materialises them here for the first time)
        all_grads = [[_grad_buf(arena, p, True) for p in cfg["params"][s]] for s in range(ctx.n_sides)]
        fgs = [None if feat_grads[s] is None else feat_grads[s].contiguous() for s in range(ctx.n_sides)]
        ev_fork = main.record_event() if ctx.n_sides > 1 else None
        for s in range(ctx.n_sides):
            ids, gate_l, gate_g, feat, amax, pre = ctx.saved_tensors[6 * s:6 * s + 6]
            prm, packed = ctx.side_ctx[s]
            grads = all_grads[s]
            ret += [None, *grads]
            if fgs[s] is None:
                continue
            n_docs, doc_len = ids.shape
            fg = fgs[s]
            stream_s = main if s == 0 else side_streams[s - 1]
            if s > 0:
                stream_s.wait_event(ev_fork)
            with torch.cuda.stream(stream_s):
                _stream(refresh=True)
                DattEncodeFn._side_backward(cfg, table, ctx.shadow, prec, arena, ids, gate_l, gate_g, feat, amax, pre, prm, packed,
                                            grads, fg, g_table, vocab, emb, dev)
        for s in range(1, ctx.n_sides):
            if fgs[s] is not None:
                main.wait_event(side_streams[s - 1].record_event())
        _stream(refresh=True)
        return (g_table, None, *ret)

    @staticmethod
    def _side_backward(cfg, table, shadow, prec, arena, ids, gate_l, gate_g, feat, amax, pre, prm, packed, grads, fg, g_table, vocab,
                       emb, dev):
        if True:
            n_docs, doc_len = ids.shape
            idf = _id_width_flag(ids)
            la_w, la_b, lc_w, lc_b, ga_w, ga_b = prm[:6]
            convs = [(lc_w, lc_b, gate_l, 1, 2, 3)] + [(prm[6 + 2 * i], prm[7 + 2 * i], gate_g, 2, 6 + 2 * i, 7 + 2 * i)
                                                       for i in range(3)]
            d_gate_l = torch.zeros_like(gate_l)
            d_gate_g = torch.zeros_like(gate_g)
            h_total = feat.shape[1]
            col = 0
            for (w, b, gate, mode, wi, bi), pk in zip(convs, packed):
                h, _, k = w.shape
                ws_bytes = lib.rbr_conv_bwd_workspace_bytes(n_docs, h, k, emb, vocab)
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
                lib.check(lib.rbr_conv_act_maxpool_bwd(
                    prec, ACT_TANH, _p(table), _p(shadow), vocab, emb, _p(ids), None, _p(gate), mode, n_docs, doc_len, _p(pk),
                    h, k, 0, feat.data_ptr() + 4 * col, amax.data_ptr() + 4 * col, fg.data_ptr() + 4 * col,
                    pre.data_ptr() + 4 * col, h_total, cfg["padding_idx"], _p(grads[wi]), _p(grads[bi]), _p(g_table),
                    _p(d_gate_l if mode == 1 else d_gate_g), _p(ws), ws_bytes, idf, _stream()), "rbr_conv_act_maxpool_bwd")
                col += h
            win = la_w.shape[2]
            ws_bytes = lib.rbr_datt_gate_workspace_bytes(n_docs, doc_len, emb, win, vocab)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            lib.check(lib.rbr_datt_gate_bwd(_p(table), vocab, emb, _p(ids), n_docs, doc_len, _p(la_w), win, _p(ga_w), _p(gate_l),
                                            _p(gate_g), _p(d_gate_l), _p(d_gate_g), cfg["padding_idx"], _p(grads[0]), _p(grads[1]),
                                            _p(grads[4]), _p(grads[5]), _p(g_table), _p(ws), ws_bytes, idf, _stream()),
                      "rbr_datt_gate_bwd")


# ---------------------------------------------------------------------------------------------------
# K10: per-row top-k of a factorised score matrix (full-catalogue recommendation)
# ---------------------------------------------------------------------------------------------------
FACTOR_TOPK_MAX_K, FACTOR_TOPK_MAX_DIM = 256, 512


def _csr_keys(indptr: torch.Tensor, indices: torch.Tensor, n_rows: int, n_items: int, what: str
              ) -> Tuple[torch.Tensor, torch.Tensor, int]:
    """Validates a CSR of item lists (what: "exclusion" / "target") → (row of each entry, row * n_items + item per entry,
    longest row).  Ids outside [0, n_items) and a malformed indptr raise ValueError."""
    if indptr.dtype != torch.int64 or indices.dtype != torch.int64:
        raise ValueError(f"rbr_b200: {what} indptr / indices must be int64")
    if indptr.dim() != 1 or indptr.numel() != n_rows + 1 or indices.dim() != 1:
        raise ValueError(f"rbr_b200: {what} indptr must be [n_rows + 1] = [{n_rows + 1}] and indices 1-D")
    counts = indptr[1:] - indptr[:-1]
    lo_hi = torch.stack([indices.min(), indices.max()]) if indices.numel() else indptr.new_zeros(2)
    longest = counts.max().view(1) if n_rows else indptr.new_zeros(1)
    # one device-to-host read for every check
    first, last, neg, lo, hi, longest = torch.cat([indptr[:1], indptr[-1:], (counts < 0).any().view(1).long(), lo_hi,
                                                   longest]).tolist()
    if first != 0 or last != indices.numel() or neg:
        raise ValueError(f"rbr_b200: {what} indptr must start at 0, be non-decreasing and end at len(indices)")
    if lo < 0 or hi >= n_items:
        raise ValueError(f"rbr_b200: {what} item ids must lie in [0, {n_items})")
    rows = torch.repeat_interleave(torch.arange(n_rows, device=indices.device), counts)
    return rows, rows * n_items + indices, int(longest)


def normalize_exclusions(indptr: torch.Tensor, indices: torch.Tensor, n_rows: int, n_items: int
                         ) -> Tuple[torch.Tensor, torch.Tensor]:
    """CSR exclusion lists (row r excludes indices[indptr[r]:indptr[r+1]], in any order, duplicates allowed) → the same
    lists sorted ascending without duplicates, as rbr_factor_topk reads them.  Ids outside [0, n_items) raise ValueError."""
    _, keys, _ = _csr_keys(indptr, indices, n_rows, n_items, "exclusion")
    keys = torch.unique(keys, sorted=True)
    new_counts = torch.bincount(torch.div(keys, n_items, rounding_mode="floor"), minlength=n_rows)
    ptr = torch.zeros(n_rows + 1, dtype=torch.int64, device=indices.device)
    torch.cumsum(new_counts, 0, out=ptr[1:])
    return ptr, keys % n_items


def _check_factors(A: torch.Tensor, row_bias: Optional[torch.Tensor], B: torch.Tensor, col_bias: Optional[torch.Tensor]
                   ) -> Tuple[int, int, int]:
    """Validates the factor operands of K10 / K11 → (n_rows, n_items, dim)."""
    for t, name in ((A, "A"), (B, "B"), (row_bias, "row_bias"), (col_bias, "col_bias")):
        if t is None:
            continue
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise RuntimeError(f"rbr_b200: `{name}` must be a CUDA tensor (the hot path has no CPU implementation)")
        if t.dtype != torch.float32:
            raise ValueError(f"rbr_b200: `{name}` must be float32, got {t.dtype}")
        if t.device != A.device:
            raise ValueError(f"rbr_b200: `{name}` is on {t.device}, A on {A.device}")
    if A.dim() != 2 or B.dim() != 2 or A.shape[1] != B.shape[1]:
        raise ValueError(f"rbr_b200: A [n_rows, dim] and B [n_items, dim] must share dim, got {tuple(A.shape)} / {tuple(B.shape)}")
    n_rows, dim = A.shape
    n_items = B.shape[0]
    if row_bias is not None and row_bias.numel() != n_rows:
        raise ValueError("rbr_b200: row_bias must hold n_rows values")
    if col_bias is not None and col_bias.numel() != n_items:
        raise ValueError("rbr_b200: col_bias must hold n_items values")
    return n_rows, n_items, dim


def _cuda_csr(csr: Tuple[torch.Tensor, torch.Tensor], what: str) -> Tuple[torch.Tensor, torch.Tensor]:
    indptr, indices = csr
    for t, name in ((indptr, f"{what} indptr"), (indices, f"{what} indices")):
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise RuntimeError(f"rbr_b200: `{name}` must be a CUDA tensor")
    return indptr.contiguous(), indices.contiguous()


def _exclusions(exclude: Optional[Tuple[torch.Tensor, torch.Tensor]], n_rows: int, n_items: int
                ) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """Normalised exclusion CSR, or (None, None) when nothing is excluded."""
    if exclude is None:
        return None, None
    ptr, idx = normalize_exclusions(*_cuda_csr(exclude, "exclude"), n_rows, n_items)
    return (None, None) if idx.numel() == 0 else (ptr, idx)


def factor_topk_workspace_bytes(n_rows: int, n_items: int, dim: int, k: int) -> int:
    n = lib.rbr_factor_topk_workspace_bytes(n_rows, n_items, dim, k)
    if n < 0:
        raise ValueError(f"rbr_b200: factor_topk does not take n_items={n_items}, dim={dim}, k={k} "
                         f"(1 <= k <= {FACTOR_TOPK_MAX_K}, 1 <= dim <= {FACTOR_TOPK_MAX_DIM}, 1 <= n_items < 2^31)")
    return int(n)


def factor_topk_slices(n_rows: int, n_items: int, dim: int, k: int) -> int:
    """How many item slices rbr_factor_topk splits each row's scan into on the current device (host-only plan query)."""
    factor_topk_workspace_bytes(n_rows, n_items, dim, k)
    return int(lib.rbr_factor_topk_slices(n_rows, n_items, dim, k))


def factor_topk(A: torch.Tensor, row_bias: Optional[torch.Tensor], B: torch.Tensor, col_bias: Optional[torch.Tensor], k: int,
                exclude: Optional[Tuple[torch.Tensor, torch.Tensor]] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """K10: for each row r, the k items i (excluding exclude = (indptr [n_rows+1], indices) CSR lists) with the largest
    score A[r] . B[i] + row_bias[r] + col_bias[i], by score descending then item id ascending; fp32-grade scores.
    Returns (scores [n_rows, k] fp32, items [n_rows, k] int64); slots past the eligible items hold (-inf, -1)."""
    n_rows, n_items, dim = _check_factors(A, row_bias, B, col_bias)
    k = int(k)
    ws_bytes = factor_topk_workspace_bytes(n_rows, n_items, dim, k)
    ptr, idx = _exclusions(exclude, n_rows, n_items)
    A, B = A.contiguous(), B.contiguous()
    rb = None if row_bias is None else row_bias.contiguous().view(-1)
    cb = None if col_bias is None else col_bias.contiguous().view(-1)
    scores = torch.empty(n_rows, k, dtype=torch.float32, device=A.device)
    items = torch.empty(n_rows, k, dtype=torch.int64, device=A.device)
    if n_rows == 0:
        return scores, items
    with torch.cuda.device(A.device):
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=A.device)
        lib.check(lib.rbr_factor_topk(_p(A), _p(rb), n_rows, _p(B), _p(cb), n_items, dim, _p(ptr), _p(idx), k, _p(scores),
                                      _p(items), _p(ws), ws_bytes, _stream(True)), "rbr_factor_topk")
    return scores, items


# ---------------------------------------------------------------------------------------------------
# K11: exact full-catalogue rank of target items under a factorised score matrix (evaluation)
# ---------------------------------------------------------------------------------------------------
FACTOR_RANK_MAX_TARGETS = 64


def factor_rank_workspace_bytes(n_rows: int, n_items: int, dim: int, n_targets: int, max_targets: int) -> int:
    n = lib.rbr_factor_rank_workspace_bytes(n_rows, n_items, dim, n_targets, max_targets)
    if n < 0:
        raise ValueError(f"rbr_b200: factor_rank does not take n_items={n_items}, dim={dim}, max_targets={max_targets} "
                         f"(1 <= dim <= {FACTOR_TOPK_MAX_DIM}, 1 <= n_items < 2^31, "
                         f"1 <= max_targets <= {FACTOR_RANK_MAX_TARGETS})")
    return int(n)


def split_target_rows(counts: torch.Tensor, cap: int = FACTOR_RANK_MAX_TARGETS) -> Tuple[torch.Tensor, torch.Tensor]:
    """Cuts rows holding `counts` targets each into pieces of at most `cap` consecutive targets; rows without targets get no
    piece.  Returns (row of each piece, piece indptr into the rows' concatenated target lists).  A piece is ranked as a row
    of its own with its row's factors and exclusions: exact, since the row's targets in other pieces are ordinary items."""
    counts = counts.to(torch.int64)
    n_pieces = torch.div(counts + cap - 1, cap, rounding_mode="floor")
    piece_row = torch.repeat_interleave(torch.arange(counts.numel(), device=counts.device), n_pieces)
    first = torch.zeros(counts.numel() + 1, dtype=torch.int64, device=counts.device)
    torch.cumsum(n_pieces, 0, out=first[1:])                   # first piece of each row
    start = torch.zeros_like(first)
    torch.cumsum(counts, 0, out=start[1:])                     # first target of each row
    k = torch.arange(piece_row.numel(), device=counts.device) - first[piece_row]
    # pieces tile the target lists in order, so each piece starts where the previous one ends
    hi = torch.minimum(start[piece_row] + (k + 1) * cap, start[piece_row + 1])
    return piece_row, torch.cat([hi.new_zeros(1), hi])


def gather_csr_rows(indptr: torch.Tensor, indices: torch.Tensor, rows: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """CSR whose row p is row rows[p] of (indptr, indices)."""
    counts = indptr[1:] - indptr[:-1]
    c = counts[rows]
    ptr = torch.zeros(rows.numel() + 1, dtype=torch.int64, device=indptr.device)
    torch.cumsum(c, 0, out=ptr[1:])
    within = torch.arange(int(ptr[-1]), device=indptr.device) - torch.repeat_interleave(ptr[:-1], c)
    return ptr, indices[torch.repeat_interleave(indptr[:-1][rows], c) + within]


def rank_inputs(t_ptr: torch.Tensor, t_idx: torch.Tensor, n_rows: int, n_items: int,
                exclude: Optional[Tuple[torch.Tensor, torch.Tensor]] = None) -> dict:
    """Host side of factor_rank (any device): validates the target CSR against the exclusions and lays it out as
    rbr_factor_rank reads it.  Raises ValueError for a target id outside [0, n_items), a target listed twice in its row
    and a target in its row's exclusion list.  Returns a dict:
      order         [nnz]: caller position of each target in the kernel's order (rows ascending, ids ascending)
      targets       [nnz]: the target ids in the kernel's order
      piece_row, piece_ptr, max_targets: rows of at most FACTOR_RANK_MAX_TARGETS targets (split_target_rows)
      excl_ptr, excl_idx: the normalised exclusions of each piece's row (None when nothing is excluded)
      n_candidates  [n_rows]: n_items minus the row's distinct excluded items"""
    _, keys, longest = _csr_keys(t_ptr, t_idx, n_rows, n_items, "target")
    dev = t_idx.device
    ptr = idx = None
    if exclude is not None:
        ptr, idx = normalize_exclusions(exclude[0], exclude[1], n_rows, n_items)
    n_excl = torch.zeros(n_rows, dtype=torch.int64, device=dev) if ptr is None else ptr[1:] - ptr[:-1]
    sorted_keys, order = torch.sort(keys)
    checks = [(sorted_keys[1:] == sorted_keys[:-1]).any()]
    if idx is not None and idx.numel() and sorted_keys.numel():
        excl_keys = torch.repeat_interleave(torch.arange(n_rows, device=dev), n_excl) * n_items + idx     # ascending
        pos = torch.searchsorted(excl_keys, sorted_keys).clamp_max(excl_keys.numel() - 1)
        checks.append((excl_keys[pos] == sorted_keys).any())
    dup, *overlap = torch.stack(checks).tolist()
    if dup:
        raise ValueError("rbr_b200: a target is listed twice in its row")
    if overlap and overlap[0]:
        raise ValueError("rbr_b200: a target is also in its row's exclusion list")
    # rows without targets are not scanned; longer rows become several pieces
    piece_row, piece_ptr = split_target_rows(t_ptr[1:] - t_ptr[:-1])
    e_ptr = e_idx = None
    if idx is not None and idx.numel():
        e_ptr, e_idx = gather_csr_rows(ptr, idx, piece_row)
        if e_idx.numel() == 0:
            e_ptr = e_idx = None
    return {"order": order, "targets": sorted_keys % n_items, "piece_row": piece_row, "piece_ptr": piece_ptr,
            "max_targets": max(1, min(longest, FACTOR_RANK_MAX_TARGETS)), "excl_ptr": e_ptr, "excl_idx": e_idx,
            "n_candidates": n_items - n_excl}


def factor_rank(A: torch.Tensor, row_bias: Optional[torch.Tensor], B: torch.Tensor, col_bias: Optional[torch.Tensor],
                targets: Tuple[torch.Tensor, torch.Tensor], exclude: Optional[Tuple[torch.Tensor, torch.Tensor]] = None
                ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """K11: the exact rank of each target item among all eligible items of its row, under factor_topk's score and order.

    targets = (indptr [n_rows+1], indices) int64 CUDA CSR: row r's targets, in any order, without duplicates, none of them
    in the row's exclusion list (exclude, as for factor_topk: any order, duplicates allowed).
    rank = #{ eligible i : (score_i, -i) >= (score_t, -t) }, 1-based: the position + 1 that t takes in factor_topk(k = inf).
    Other targets of the row count as ordinary competitors; NaN and -inf scores never count; a target whose own score is
    NaN or -inf gets rank -1.  Returns (ranks int64 [nnz], scores fp32 [nnz], both in the order of `indices`,
    n_candidates int64 [n_rows] = n_items minus the row's distinct excluded items)."""
    n_rows, n_items, dim = _check_factors(A, row_bias, B, col_bias)
    factor_rank_workspace_bytes(n_rows, n_items, dim, 0, 1)             # the shape limits, before any device work
    t_ptr, t_idx = _cuda_csr(targets, "targets")
    plan = rank_inputs(t_ptr, t_idx, n_rows, n_items, None if exclude is None else _cuda_csr(exclude, "exclude"))
    dev = A.device
    nnz = t_idx.numel()
    ranks = torch.empty(nnz, dtype=torch.int64, device=dev)
    scores = torch.empty(nnz, dtype=torch.float32, device=dev)
    if nnz == 0:
        return ranks, scores, plan["n_candidates"]
    piece_row = plan["piece_row"]
    n_pieces, mt = piece_row.numel(), plan["max_targets"]
    A_p = A.contiguous().index_select(0, piece_row)
    rb_p = None if row_bias is None else row_bias.contiguous().view(-1).index_select(0, piece_row)
    cb = None if col_bias is None else col_bias.contiguous().view(-1)
    ws_bytes = factor_rank_workspace_bytes(n_pieces, n_items, dim, nnz, mt)
    r_sorted = torch.empty(nnz, dtype=torch.int64, device=dev)
    s_sorted = torch.empty(nnz, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        lib.check(lib.rbr_factor_rank(_p(A_p), _p(rb_p), n_pieces, _p(B.contiguous()), _p(cb), n_items, dim,
                                      _p(plan["excl_ptr"]), _p(plan["excl_idx"]), _p(plan["piece_ptr"]), _p(plan["targets"]),
                                      nnz, mt, _p(r_sorted), _p(s_sorted), _p(ws), ws_bytes, _stream(True)), "rbr_factor_rank")
    ranks[plan["order"]] = r_sorted
    scores[plan["order"]] = s_sorted
    return ranks, scores, plan["n_candidates"]


# ---------------------------------------------------------------------------------------------------
# K14: diversified top-k — maximal marginal relevance over a relevance pool
# ---------------------------------------------------------------------------------------------------
MMR_MAX_POOL, MMR_MAX_DIM = 256, 512


def mmr_supported(pool: int, dim: int, k: int) -> bool:
    """Whether rbr_mmr_select takes pools of `pool` entries, `dim`-wide item vectors and k picks (host-only query)."""
    return bool(lib.rbr_mmr_supported(int(pool), int(dim), int(k)))


def unit_rows(x: torch.Tensor) -> torch.Tensor:
    """x [n, dim] with every row scaled to unit length, in float64 and then rounded to fp32; a zero row stays zero."""
    x64 = x.detach().double()
    norm = x64.norm(dim=1, keepdim=True)
    return torch.where(norm > 0, x64 / norm.clamp_min(torch.finfo(torch.float64).tiny), torch.zeros_like(x64)).float()


def mmr_select(pool_scores: torch.Tensor, pool_items: torch.Tensor, item_vecs: torch.Tensor, k: int, lam: float
               ) -> Tuple[torch.Tensor, torch.Tensor]:
    """K14: per row, k picks from the row's pool by maximal marginal relevance (include/rbr_b200.h, K14).

    pool_scores [n, P] fp32 / pool_items [n, P] int64 CUDA: the row's candidates (e.g. factor_topk's output for k = P); a
    position is eligible when its item lies in [0, n_items) and its score is finite.  item_vecs [n_items, dim] fp32 CUDA:
    unit-normalised item vectors (unit_rows), sim = fp32 dot product.  Step 0 picks the largest relevance (the score min-max
    scaled over the row's eligible positions), step t the largest lam * rel - (1 - lam) * max sim to the items picked so
    far; ties to the lower position.  Returns (scores [n, k] fp32, items [n, k] int64) in selection order, the pool's own
    scores; rows with fewer than k eligible positions end in (-inf, -1)."""
    pool_scores = _req(pool_scores, torch.float32, "pool_scores")
    pool_items = _req(pool_items, torch.int64, "pool_items")
    item_vecs = _req(item_vecs, torch.float32, "item_vecs")
    for t, name in ((pool_items, "pool_items"), (item_vecs, "item_vecs")):
        if t.device != pool_scores.device:
            raise ValueError(f"rbr_b200: `{name}` is on {t.device}, pool_scores on {pool_scores.device}")
    if pool_scores.dim() != 2 or pool_items.shape != pool_scores.shape or item_vecs.dim() != 2:
        raise ValueError(f"rbr_b200: mmr_select takes pool_scores / pool_items [n, P] and item_vecs [n_items, dim], got "
                         f"{tuple(pool_scores.shape)} / {tuple(pool_items.shape)} / {tuple(item_vecs.shape)}")
    n, P = pool_scores.shape
    n_items, dim = item_vecs.shape
    k, lam = int(k), float(lam)
    if not 0.0 <= lam <= 1.0:
        raise ValueError(f"rbr_b200: lam must lie in [0, 1], got {lam}")
    if not mmr_supported(P, dim, k):
        raise ValueError(f"rbr_b200: mmr_select does not take k={k}, pool={P}, dim={dim} "
                         f"(1 <= k <= pool <= {MMR_MAX_POOL}, 1 <= dim <= {MMR_MAX_DIM})")
    dev = pool_scores.device
    scores = torch.empty(n, k, dtype=torch.float32, device=dev)
    items = torch.empty(n, k, dtype=torch.int64, device=dev)
    if n == 0:
        return scores, items
    with torch.cuda.device(dev):
        lib.check(lib.rbr_mmr_select(_p(pool_scores), _p(pool_items), n, P, _p(item_vecs), n_items, dim, k, lam, _p(scores),
                                     _p(items), _stream(True)), "rbr_mmr_select")
    return scores, items


# ---------------------------------------------------------------------------------------------------
# K12: token attributions of a predicted rating from the per-entity feature cache
# ---------------------------------------------------------------------------------------------------
EXPLAIN_MAX_POSITIONS, EXPLAIN_MAX_M, EXPLAIN_MAX_WIDTH, EXPLAIN_MAX_CONVS = 16384, 32, 16, 8


def explain_supported(positions: int, m: int, width: int, n_conv: int = 1) -> bool:
    """Whether rbr_explain_attrib takes rows of `positions` = docs_per_entity * doc_len tokens with m windows of `width`
    positions over n_conv convs (host-only query)."""
    return bool(lib.rbr_explain_supported(int(positions), int(m), int(width), int(n_conv)))


def _check_argmax(argmax: torch.Tensor, n_docs: int, filters: int, n_pos: int, what: str) -> torch.Tensor:
    if not isinstance(argmax, torch.Tensor) or not argmax.is_cuda:
        raise RuntimeError(f"rbr_b200: `{what}` must be a CUDA tensor")
    if argmax.dtype != torch.int32 or argmax.dim() != 2 or argmax.shape[0] != n_docs or argmax.shape[1] < filters:
        raise ValueError(f"rbr_b200: `{what}` must be int32 [{n_docs}, >= {filters}], got {argmax.dtype} {tuple(argmax.shape)}")
    if argmax.stride(1) != 1:
        raise ValueError(f"rbr_b200: `{what}` must have unit column stride")
    if argmax.numel():
        lo, hi = torch.stack([argmax[:, :filters].min(), argmax[:, :filters].max()]).tolist()
        if lo < 0 or hi >= n_pos:
            raise ValueError(f"rbr_b200: `{what}` positions must lie in [0, {n_pos}) (the pooled conv outputs)")
    return argmax


def conv_window_contrib(table: torch.Tensor, ids: torch.Tensor, mask: Optional[torch.Tensor], weight: torch.Tensor, pad: int,
                        argmax: torch.Tensor, packed: Optional[torch.Tensor] = None, mask_from_ids: bool = False,
                        out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """K12a: the tap contributions c[n, h, j] = sum_e weight[h, e, j] * x[n, argmax[n, h] + j - pad, e] of every pooled
    window, in fp32 from the fp32 table (x reads as zeros outside the document, where the mask is false — mask None with
    mask_from_ids: ids != 0 — and for ids outside the table, as in the forward).  ids [n_docs, doc_len] int64 / int32 /
    uint16; weight [H, E, k] (nn.Conv1d); argmax int32 [n_docs, H] (or a column slice of a wider array, e.g. one conv's
    filters of EncodeDocsFn's arg-max).  Returns contrib [n_docs, H * k] (column h * k + j), or writes into `out`, which may
    be a column slice of a wider [n_docs, sum_c H_c * k_c] array shared by several convs."""
    table = _req(table, torch.float32, "table")
    ids = _ids(ids, "ids")
    weight = _req(weight, torch.float32, "conv weight")
    if ids.dim() < 1 or table.dim() != 2 or weight.dim() != 3 or weight.shape[1] != table.shape[1]:
        raise ValueError(f"rbr_b200: table [V, E], weight [H, E, k] and ids [..., L] do not fit: {tuple(table.shape)} / "
                         f"{tuple(weight.shape)} / {tuple(ids.shape)}")
    h, emb, k = weight.shape
    pad = int(pad)
    doc_len = ids.shape[-1]
    n_docs = ids.numel() // max(doc_len, 1)
    if pad < 0 or doc_len < 1:
        raise ValueError("rbr_b200: pad must be >= 0 and documents non-empty")
    if mask is not None and tuple(mask.shape) != tuple(ids.shape):
        raise ValueError(f"rbr_b200: mask {tuple(mask.shape)} does not match ids {tuple(ids.shape)}")
    flags = _id_flags(ids, mask, mask_from_ids)
    mask = _mask_u8(mask, "mask")
    argmax = _check_argmax(argmax, n_docs, h, doc_len + 2 * pad - k + 1, "argmax")
    if packed is None:
        packed = conv_pack(weight)
    if out is None:
        out = torch.empty(n_docs, h * k, dtype=torch.float32, device=table.device)
    elif (out.dtype != torch.float32 or out.dim() != 2 or out.shape[0] != n_docs or out.shape[1] < h * k or out.stride(1) != 1
          or out.device != table.device):
        raise ValueError(f"rbr_b200: `out` must be fp32 [{n_docs}, >= {h * k}] with unit column stride")
    if n_docs == 0:
        return out
    lib.check(lib.rbr_conv_window_contrib(_p(table), table.shape[0], emb, _p(ids), _p(mask), n_docs, doc_len, _p(packed), h, k,
                                          pad, _p(argmax), argmax.stride(0), _p(out), out.stride(0), flags, _stream(True)),
              "rbr_conv_window_contrib")
    return out


def explain_attrib(ent_row: torch.Tensor, g: torch.Tensor, feat: Optional[torch.Tensor], argmax: torch.Tensor,
                   contrib: torch.Tensor, convs: Sequence[Tuple[int, int, int]], docs_per_entity: int, doc_len: int, m: int,
                   width: int, return_map: bool = False, return_review_attr: bool = False,
                   dense_coef: Optional[torch.Tensor] = None, dense_vec: Optional[torch.Tensor] = None) -> dict:
    """K12b: per (pair, side) row p, the token attribution map of the docs_per_entity cached documents starting at row
    ent_row[p] of feat / argmax / contrib, under g [P, docs_per_entity, Htot] = d pred / d feat, and its top-m / bottom-m
    windows of `width` positions (greedy, no overlap, ties to the lower start, never across a document boundary).
    convs = [(filters, ksize, pad)] per conv, in the column order of feat / argmax (Htot = sum of filters) and contrib
    (sum of filters * ksize, conv_window_contrib's layout).
    Returns a dict of text_total [P], top_pos / bottom_pos int64 [P, m] (flat positions r * doc_len + t, -1 = no window
    left), top_attr / bottom_attr [P, m] (NaN where -1), and with return_map `map` [P, docs_per_entity * doc_len], with
    return_review_attr `review_attr` [P, docs_per_entity].
    feat None: every filter counts (D-ATT's tanh features have no liveness predicate).  dense_coef [n_docs, >= Htot] with
    dense_vec [n_docs, doc_len] add a dense term per cached document: (sum_h g * dense_coef) * dense_vec (D-ATT's global
    gate, datt_explain_contrib), reduced in a fixed order (rbr_explain_attrib_ex)."""
    R, T, m, width = int(docs_per_entity), int(doc_len), int(m), int(width)
    convs = [tuple(int(x) for x in c) for c in convs]
    if R < 1 or T < 1 or not explain_supported(R * T, m, width, len(convs)):
        raise ValueError(f"rbr_b200: explain_attrib takes 1 <= docs_per_entity * doc_len <= {EXPLAIN_MAX_POSITIONS}, "
                         f"1 <= m <= {EXPLAIN_MAX_M}, 1 <= width <= {EXPLAIN_MAX_WIDTH} and 1 to {EXPLAIN_MAX_CONVS} convs "
                         f"(got {R} x {T}, m={m}, width={width}, {len(convs)} convs)")
    if any(h < 1 or k < 1 or pad < 0 for h, k, pad in convs):
        raise ValueError(f"rbr_b200: bad conv description {convs}")
    h_tot = sum(h for h, _, _ in convs)
    taps = sum(h * k for h, k, _ in convs)
    contrib = _req(contrib, torch.float32, "contrib")
    ent_row = _req(ent_row, torch.int64, "ent_row").view(-1)
    g = _req(g, torch.float32, "g")
    argmax = _req(argmax, torch.int32, "argmax")
    feat = argmax if feat is None else _req(feat, torch.float32, "feat")       # only shapes and the device are read from it
    n_docs = feat.shape[0] if feat.dim() == 2 else -1
    if feat.dim() != 2 or feat.shape[1] < h_tot or contrib.dim() != 2 or contrib.shape[0] != n_docs or contrib.shape[1] < taps:
        raise ValueError(f"rbr_b200: feat / argmax [n_docs, >= {h_tot}] and contrib [n_docs, >= {taps}] expected, got "
                         f"{tuple(feat.shape)} / {tuple(contrib.shape)}")
    P = ent_row.numel()
    if tuple(g.shape) != (P, R, h_tot):
        raise ValueError(f"rbr_b200: g must be [{P}, {R}, {h_tot}], got {tuple(g.shape)}")
    if tuple(argmax.shape) != tuple(feat.shape):
        raise ValueError(f"rbr_b200: argmax {tuple(argmax.shape)} must match feat {tuple(feat.shape)}")
    if (dense_coef is None) != (dense_vec is None):
        raise ValueError("rbr_b200: dense_coef and dense_vec go together")
    if dense_coef is not None:
        dense_coef = _req(dense_coef, torch.float32, "dense_coef")
        dense_vec = _req(dense_vec, torch.float32, "dense_vec")
        if (dense_coef.dim() != 2 or dense_coef.shape[0] != n_docs or dense_coef.shape[1] < h_tot
                or tuple(dense_vec.shape) != (n_docs, T)):
            raise ValueError(f"rbr_b200: dense_coef [{n_docs}, >= {h_tot}] and dense_vec [{n_docs}, {T}] expected, got "
                             f"{tuple(dense_coef.shape)} / {tuple(dense_vec.shape)}")
    for t, name in ((g, "g"), (contrib, "contrib"), (argmax, "argmax"), (ent_row, "ent_row"), (dense_coef, "dense_coef"),
                    (dense_vec, "dense_vec")):
        if t is not None and t.device != feat.device:
            raise ValueError(f"rbr_b200: `{name}` is on {t.device}, feat on {feat.device}")
    if P and n_docs % R:
        raise ValueError(f"rbr_b200: {n_docs} cached documents are not whole entities of {R}")
    if P:
        lo, hi, odd = torch.stack([ent_row.min(), ent_row.max(), (ent_row % R != 0).any().long()]).tolist()
        if lo < 0 or hi > n_docs - R or odd:
            raise ValueError(f"rbr_b200: ent_row must be multiples of {R} in [0, {n_docs - R}]")
    dev = feat.device
    out = {"text_total": torch.empty(P, dtype=torch.float32, device=dev)}
    for side in ("top", "bottom"):
        out[f"{side}_pos"] = torch.empty(P, m, dtype=torch.int64, device=dev)
        out[f"{side}_attr"] = torch.empty(P, m, dtype=torch.float32, device=dev)
    if return_map:
        out["map"] = torch.empty(P, R * T, dtype=torch.float32, device=dev)
    if return_review_attr:
        out["review_attr"] = torch.empty(P, R, dtype=torch.float32, device=dev)
    if P == 0:
        return out
    if dense_coef is None and feat is not argmax:
        lib.check(lib.rbr_explain_attrib(
            _p(ent_row), P, R, T, _p(g), _p(feat), _p(argmax), feat.shape[1], _p(contrib), contrib.shape[1], n_docs, len(convs),
            _i64_array([x for c in convs for x in c]), m, width, _p(out["text_total"]), _p(out["top_pos"]), _p(out["top_attr"]),
            _p(out["bottom_pos"]), _p(out["bottom_attr"]), _p(out.get("map")), _p(out.get("review_attr")), _stream(True)),
            "rbr_explain_attrib")
        return out
    lib.check(lib.rbr_explain_attrib_ex(
        _p(ent_row), P, R, T, _p(g), None if feat is argmax else _p(feat), _p(argmax), feat.shape[1], _p(contrib),
        contrib.shape[1], n_docs, len(convs), _i64_array([x for c in convs for x in c]), _p(dense_coef),
        0 if dense_coef is None else dense_coef.shape[1], _p(dense_vec), T, m, width, _p(out["text_total"]),
        _p(out["top_pos"]), _p(out["top_attr"]), _p(out["bottom_pos"]), _p(out["bottom_attr"]), _p(out.get("map")),
        _p(out.get("review_attr")), _stream(True)), "rbr_explain_attrib_ex")
    return out


def window_select(attr: torch.Tensor, doc_len: int, m: int, width: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor,
                                                                                  torch.Tensor]:
    """The window rule of explain_attrib in plain torch (any device; a statement of the rule, not a hot path): for each row
    of attr [P, S] (S = docs * doc_len flat positions), the m windows of `width` consecutive positions with the largest
    float64 sum, chosen greedily without overlap, ties to the lower start, no window across a multiple of doc_len; then
    the same for the smallest sums.  Returns (top_pos, top_attr, bottom_pos, bottom_attr), -1 / NaN where no window is left."""
    P, S = attr.shape
    a = attr.double()
    starts = torch.arange(S, device=attr.device)
    valid = (starts % doc_len) + width <= doc_len
    ws = torch.zeros(P, S, dtype=torch.float64, device=attr.device)
    for j in range(min(width, S)):  # window sums as in-order additions (what the kernel does), not a cumsum difference
        ws[:, :S - j] += a[:, j:]
    out = []
    for top in (True, False):
        pos = torch.full((P, m), -1, dtype=torch.int64, device=attr.device)
        val = torch.full((P, m), float("nan"), dtype=torch.float32, device=attr.device)
        avail = valid.unsqueeze(0).expand(P, S).clone()
        for it in range(m):
            key = torch.where(avail, ws if top else -ws, torch.full_like(ws, float("-inf")))
            best = key.max(1).values
            hit = avail & (key == best.unsqueeze(1))
            s = torch.where(hit, starts, torch.full_like(starts, S)).min(1).values      # lowest start among the ties
            has = avail.any(1)
            pos[:, it] = torch.where(has, s, torch.full_like(s, -1))
            val[:, it] = torch.where(has, ws.gather(1, s.clamp_max(S - 1).view(-1, 1)).view(-1).float(),
                                     torch.full((P,), float("nan"), device=attr.device))
            block = (starts.view(1, -1) > (s.view(-1, 1) - width)) & (starts.view(1, -1) < (s.view(-1, 1) + width))
            avail &= ~(block & has.view(-1, 1))
        out += [pos, val]
    return tuple(out)


def datt_gates(table: torch.Tensor, ids: torch.Tensor, w_local: torch.Tensor, b_local: torch.Tensor, w_global: torch.Tensor,
               b_global: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """K5's two D-ATT gates for documents ids [n_docs, doc_len]: (local [n_docs, doc_len], global [n_docs]), the values the
    gated convs of DattEncodeFn multiply the token rows by."""
    table = _req(table, torch.float32, "table")
    ids = _ids(ids, "ids")
    n_docs, doc_len = ids.shape
    vocab, emb = table.shape
    prm = [_req(t, torch.float32, n) for t, n in ((w_local, "w_local"), (b_local, "b_local"), (w_global, "w_global"),
                                                  (b_global, "b_global"))]
    win = prm[0].shape[2]
    gate_l = torch.empty(n_docs, doc_len, dtype=torch.float32, device=table.device)
    gate_g = torch.empty(n_docs, dtype=torch.float32, device=table.device)
    ws_bytes = lib.rbr_datt_gate_workspace_bytes(n_docs, doc_len, emb, win, vocab)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=table.device)
    lib.check(lib.rbr_datt_gate_fwd(_p(table), vocab, emb, _p(ids), n_docs, doc_len, _p(prm[0]), _p(prm[1]), win, _p(prm[2]),
                                    _p(prm[3]), _p(gate_l), _p(gate_g), _p(ws), ws_bytes, _id_width_flag(ids), _stream(True)),
              "rbr_datt_gate_fwd")
    return gate_l, gate_g


def _datt_side_prm(prm: Sequence[torch.Tensor]) -> List[torch.Tensor]:
    prm = [_req(t.detach(), torch.float32, "D-ATT parameter") for t in prm]
    if len(prm) != DattEncodeFn.N_PRM:
        raise ValueError(f"rbr_b200: a D-ATT side has {DattEncodeFn.N_PRM} parameters, got {len(prm)}")
    return prm


def datt_explain_contrib(table: torch.Tensor, ids: torch.Tensor, prm: Sequence[torch.Tensor], gate_l: torch.Tensor,
                         gate_g: torch.Tensor, feat: torch.Tensor, argmax: torch.Tensor,
                         packed: Optional[Sequence[torch.Tensor]] = None) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """The per-entity terms of D-ATT's gradient x input (rbr_datt_explain_contrib) for documents ids [n_docs, L] (int64 /
    int32) of one side: prm = the side's 12 parameters (DattEncodeFn's order), gate_l [n_docs, L] / gate_g [n_docs] / feat /
    argmax [n_docs, l_out + 3 g_out] from datt_encode_side.  In fp32 from the fp32 table whatever the forward's precision.
    Returns (contrib [n_docs, l_out * window + 9 g_out], gate_coef [n_docs, l_out + 3 g_out], gate_vec [n_docs, L]): the
    contributions for explain_attrib with convs datt_explain_convs(prm) and feat None, and its dense term."""
    table = _req(table, torch.float32, "table")
    ids = _ids(ids, "ids")
    if ids.dtype == torch.uint16:
        raise TypeError("rbr_b200: D-ATT takes int64 or int32 ids")
    prm = _datt_side_prm(prm)
    if table.dim() != 2 or ids.dim() != 2:
        raise ValueError(f"rbr_b200: table [V, E] and ids [n_docs, L] expected, got {tuple(table.shape)} / {tuple(ids.shape)}")
    vocab, emb = table.shape
    n_docs, L = ids.shape
    la_w, ga_w = prm[0], prm[4]
    win = la_w.shape[-1]
    l_out, g_out = prm[2].shape[0], prm[6].shape[0]
    if (tuple(la_w.shape) != (1, emb, win) or tuple(ga_w.shape) != (1, emb, L) or tuple(prm[2].shape) != (l_out, emb, 1)
            or any(tuple(prm[6 + 2 * c].shape) != (g_out, emb, c + 2) for c in range(3))):
        raise ValueError(f"rbr_b200: D-ATT parameters do not fit emb={emb}, doc_len={L}: "
                         f"{[tuple(p.shape) for p in prm[::2]]}")
    if L < 4 or win % 2 == 0 or not 1 <= win <= EXPLAIN_MAX_WIDTH:
        raise ValueError(f"rbr_b200: datt_explain_contrib takes doc_len >= 4 and an odd window <= {EXPLAIN_MAX_WIDTH} "
                         f"(got {L}, {win})")
    htot = l_out + 3 * g_out
    gate_l = _req(gate_l, torch.float32, "gate_l")
    gate_g = _req(gate_g, torch.float32, "gate_g")
    feat = _req(feat, torch.float32, "feat")
    if tuple(gate_l.shape) != (n_docs, L) or tuple(gate_g.reshape(-1).shape) != (n_docs,) or tuple(feat.shape) != (n_docs, htot):
        raise ValueError(f"rbr_b200: gate_l [{n_docs}, {L}], gate_g [{n_docs}] and feat [{n_docs}, {htot}] expected, got "
                         f"{tuple(gate_l.shape)} / {tuple(gate_g.shape)} / {tuple(feat.shape)}")
    argmax = _req(argmax, torch.int32, "argmax")
    if tuple(argmax.shape) != (n_docs, htot):
        raise ValueError(f"rbr_b200: argmax must be int32 [{n_docs}, {htot}], got {tuple(argmax.shape)}")
    if n_docs:
        for c, (lo, hi) in enumerate(((0, l_out), (l_out, l_out + g_out), (l_out + g_out, l_out + 2 * g_out),
                                      (l_out + 2 * g_out, htot))):
            _check_argmax(argmax[:, lo:hi], n_docs, hi - lo, L - (c + 1) + 1 if c else L, "argmax")
    for t, name in ((ids, "ids"), (gate_l, "gate_l"), (gate_g, "gate_g"), (feat, "feat"), (argmax, "argmax")):
        if t.device != table.device:
            raise ValueError(f"rbr_b200: `{name}` is on {t.device}, the table on {table.device}")
    if packed is None:
        packed = datt_side_packs(prm)
    wlT = la_w.reshape(emb, win).t().contiguous()
    wgT = ga_w.reshape(emb, L).t().contiguous()
    dev = table.device
    contrib = torch.empty(n_docs, l_out * win + 9 * g_out, dtype=torch.float32, device=dev)
    gate_coef = torch.empty(n_docs, htot, dtype=torch.float32, device=dev)
    gate_vec = torch.empty(n_docs, L, dtype=torch.float32, device=dev)
    if n_docs == 0:
        return contrib, gate_coef, gate_vec
    lib.check(lib.rbr_datt_explain_contrib(
        _p(table), vocab, emb, _p(ids), n_docs, L, _p(wlT), win, _p(wgT), _p(packed[0]), l_out, _p(packed[1]), _p(packed[2]),
        _p(packed[3]), g_out, _p(gate_l), _p(gate_g), _p(feat), _p(argmax), htot, _p(contrib), contrib.shape[1], _p(gate_coef),
        htot, _p(gate_vec), L, _id_width_flag(ids), _stream(True)), "rbr_datt_explain_contrib")
    return contrib, gate_coef, gate_vec


def datt_explain_convs(prm: Sequence[torch.Tensor]) -> List[Tuple[int, int, int]]:
    """explain_attrib's conv description of datt_explain_contrib's layout: the local filters as one width-`window` conv with
    pad (window - 1) / 2, then the k = 2, 3, 4 global convs without padding."""
    win = prm[0].shape[-1]
    return [(prm[2].shape[0], win, (win - 1) // 2)] + [(prm[6 + 2 * c].shape[0], c + 2, 0) for c in range(3)]


DATT_FC_MAX_HIDDEN = 768


def datt_fc_grads(u_ids: torch.Tensor, i_ids: torch.Tensor, user_out: torch.Tensor, item_out: torch.Tensor,
                  user_mask: torch.Tensor, item_mask: torch.Tensor, w0: torch.Tensor, w3: torch.Tensor
                  ) -> Tuple[torch.Tensor, torch.Tensor]:
    """g = d pred / d cat [P, in_dim] of both D-ATT sides for pairs (u_ids[p], i_ids[p]) (rbr_datt_fc_grads): pred =
    fc(cat_u) . fc(cat_i) with the shared FC stack, so g_u = W0^T (user_mask[u] * W3^T item_out[i]) and symmetrically.
    user_out [U, out_dim] / item_out [I, out_dim]: the cached FC outputs; user_mask / item_mask [*, hidden] bool: the cached
    hidden ReLU masks; w0 = fc.0.weight [hidden, in_dim], w3 = fc.3.weight [out_dim, hidden].  3xTF32 tensor cores, one
    fixed summation order per element: bit-identical whatever the batch or the pair order."""
    u_ids = _req(u_ids, torch.int64, "u_ids").view(-1)
    i_ids = _req(i_ids, torch.int64, "i_ids").view(-1)
    user_out = _req(user_out, torch.float32, "user_out")
    item_out = _req(item_out, torch.float32, "item_out")
    user_mask = _mask_u8(user_mask, "user_mask")
    item_mask = _mask_u8(item_mask, "item_mask")
    w0 = _req(w0.detach(), torch.float32, "w0")
    w3 = _req(w3.detach(), torch.float32, "w3")
    if w0.dim() != 2 or w3.dim() != 2:
        raise ValueError("rbr_b200: w0 [hidden, in_dim] and w3 [out_dim, hidden] expected")
    hidden, in_dim = w0.shape
    out_dim = w3.shape[0]
    if not 1 <= hidden <= DATT_FC_MAX_HIDDEN:
        raise ValueError(f"rbr_b200: datt_fc_grads takes 1 <= hidden <= {DATT_FC_MAX_HIDDEN}, got {hidden}")
    if tuple(w3.shape) != (out_dim, hidden):
        raise ValueError(f"rbr_b200: w3 must be [out_dim, {hidden}], got {tuple(w3.shape)}")
    for out, mask, name in ((user_out, user_mask, "user"), (item_out, item_mask, "item")):
        if out.dim() != 2 or out.shape[1] != out_dim or mask.dim() != 2 or tuple(mask.shape) != (out.shape[0], hidden):
            raise ValueError(f"rbr_b200: {name}_out [n, {out_dim}] and {name}_mask [n, {hidden}] expected, got "
                             f"{tuple(out.shape)} / {tuple(mask.shape)}")
    P = u_ids.numel()
    if i_ids.numel() != P:
        raise ValueError("rbr_b200: u_ids and i_ids must hold one id per pair")
    for t, name in ((i_ids, "i_ids"), (user_out, "user_out"), (item_out, "item_out"), (user_mask, "user_mask"),
                    (item_mask, "item_mask"), (w0, "w0"), (w3, "w3")):
        if t.device != u_ids.device:
            raise ValueError(f"rbr_b200: `{name}` is on {t.device}, u_ids on {u_ids.device}")
    if P:
        lo_u, hi_u, lo_i, hi_i = torch.stack([u_ids.min(), u_ids.max(), i_ids.min(), i_ids.max()]).tolist()
        if lo_u < 0 or hi_u >= user_out.shape[0] or lo_i < 0 or hi_i >= item_out.shape[0]:
            raise ValueError(f"rbr_b200: user ids must lie in [0, {user_out.shape[0]}) and item ids in [0, {item_out.shape[0]})")
    g_u = torch.empty(P, in_dim, dtype=torch.float32, device=u_ids.device)
    g_i = torch.empty(P, in_dim, dtype=torch.float32, device=u_ids.device)
    if P == 0:
        return g_u, g_i
    lib.check(lib.rbr_datt_fc_grads(_p(u_ids), _p(i_ids), P, _p(user_out), user_out.shape[0], _p(item_out), item_out.shape[0],
                                    out_dim, _p(user_mask), _p(item_mask), hidden, _p(w0), in_dim, _p(w3), _p(g_u), _p(g_i),
                                    _stream(True)), "rbr_datt_fc_grads")
    return g_u, g_i


def head_text_grads(u_text: torch.Tensor, i_text: torch.Tensor, u_id: torch.Tensor, i_id: torch.Tensor,
                    params: Sequence[torch.Tensor], padding_idx: Sequence[int], scratch: Optional[List[torch.Tensor]] = None
                    ) -> Tuple[torch.Tensor, torch.Tensor]:
    """d pred / d u_text and d pred / d i_text [B, H] of K4 in eval mode (rbr_head_fwd, then rbr_head_bwd at pred_grad = 1).
    params: (Wu, bu, ebd_u, Wi, bi, ebd_i, fm_h, user_bias, item_bias, g_bias); the parameter gradients the backward
    accumulates go to `scratch` (one buffer per parameter, reused across calls and never read), not to `.grad`."""
    u_text = _req(u_text, torch.float32, "u_text")
    i_text = _req(i_text, torch.float32, "i_text")
    u_id = _req(u_id, torch.int64, "u_id")
    i_id = _req(i_id, torch.int64, "i_id")
    fl = [_req(t.detach(), torch.float32, "head parameter") for t in params]
    B, H = u_text.shape
    K = fl[0].shape[1]
    dev = u_text.device
    if scratch is None:
        scratch = [torch.empty_like(t) for t in fl]
    pred = torch.empty(B, dtype=torch.float32, device=dev)
    u_lat = torch.empty(B, K, dtype=torch.float32, device=dev)
    i_lat = torch.empty(B, K, dtype=torch.float32, device=dev)
    s = _stream(True)
    lib.check(lib.rbr_head_fwd(_p(u_text), _p(i_text), _p(u_id), _p(i_id), B, H, K, *[_p(t) for t in fl], fl[2].shape[0],
                               fl[5].shape[0], 0.0, 0, None, _p(pred), _p(u_lat), _p(i_lat), None, 0.0, None, None, s),
              "rbr_head_fwd")
    ones = torch.ones(B, dtype=torch.float32, device=dev)
    g_ut, g_it = torch.empty_like(u_text), torch.empty_like(i_text)
    pads = [-1 if x is None else int(x) for x in padding_idx]
    lib.check(lib.rbr_head_bwd(_p(u_text), _p(i_text), _p(u_id), _p(i_id), B, H, K, _p(fl[0]), _p(fl[3]), _p(fl[6]), _p(u_lat),
                               _p(i_lat), 0.0, 0, None, *pads, fl[2].shape[0], fl[5].shape[0], _p(ones), _p(g_ut), _p(g_it),
                               *[_p(t) for t in scratch], s), "rbr_head_bwd")
    return g_ut, g_it


def narre_feat_grads(feats: Sequence[torch.Tensor], other_ids: Sequence[torch.Tensor], scores: Sequence[torch.Tensor],
                     out_grads: Sequence[torch.Tensor], side_params: Sequence[Sequence[torch.Tensor]],
                     padding_idx: Sequence[int], scratch: Optional[List[List[torch.Tensor]]] = None) -> List[torch.Tensor]:
    """d pred / d feat [B, R, H] of each NARRE side from d pred / d out [B, H], through K3's backward (the tensor-core pair
    kernel when the shape allows, else one K3 launch per side) with the forward's attention scores [B, R].  side_params: per
    side (W_rv, W_id, h, b_1, b_2, ebd_vals); the parameter gradients go to `scratch`, never to `.grad`."""
    feats = [_req(f, torch.float32, "feat") for f in feats]
    ids = [_req(i, torch.int64, "other_id") for i in other_ids]
    scores = [_req(s, torch.float32, "scores") for s in scores]
    g_outs = [_req(g, torch.float32, "out_grad") for g in out_grads]
    prm = [[_req(t.detach(), torch.float32, "attention parameter") for t in sp] for sp in side_params]
    if scratch is None:
        scratch = [[torch.empty_like(t) for t in sp] for sp in prm]
    B, R, H = feats[0].shape
    A = prm[0][0].shape[1]
    pads = [-1 if x is None else int(x) for x in padding_idx]
    g_feats = [torch.empty_like(f) for f in feats]
    s = _stream(True)
    if narre_attn_pair_supported(R, H, A) and len(feats) == 2:
        lib.check(lib.rbr_narre_attn_pair_bwd(
            2, _ptr_array([_p(f) for f in feats]), _ptr_array([_p(i) for i in ids]), B, R, H, A,
            *[_ptr_array([_p(prm[0][j]), _p(prm[1][j])]) for j in range(6)],
            _i64_array([prm[0][5].shape[0], prm[1][5].shape[0]]), _i64_array(pads), _ptr_array([_p(x) for x in scores]),
            _ptr_array([_p(g) for g in g_outs]), None, _ptr_array([_p(g) for g in g_feats]),
            *[_ptr_array([_p(scratch[0][j]), _p(scratch[1][j])]) for j in range(6)], s), "rbr_narre_attn_pair_bwd")
        return g_feats
    for f, i, sc, go, p, pad, gf, scr in zip(feats, ids, scores, g_outs, prm, pads, g_feats, scratch):
        lib.check(lib.rbr_narre_attn_bwd(_p(f), _p(i), B, R, H, A, *[_p(t) for t in p], p[5].shape[0], pad, _p(sc), _p(go), None,
                                         _p(gf), *[_p(t) for t in scr], s), "rbr_narre_attn_bwd")
    return g_feats


# ---------------------------------------------------------------------------------------------------
# K13: token attributions for SimpleSiamese (masked average pooling + additive review attention)
# ---------------------------------------------------------------------------------------------------
def explain_avgpool_supported(positions: int, reviews: int, emb: int, feat: int, m: int, width: int) -> bool:
    """Whether rbr_explain_avgpool_attrib takes entities of `reviews` reviews with `positions` = reviews * doc_len tokens,
    embedding width emb, side feature width feat, m windows of `width` positions (host-only query)."""
    return bool(lib.rbr_explain_avgpool_supported(int(positions), int(reviews), int(emb), int(feat), int(m), int(width)))


def explain_avgpool_attrib(table: torch.Tensor, ids: torch.Tensor, mask: Optional[torch.Tensor], ent: torch.Tensor,
                           v: torch.Tensor, att_a: torch.Tensor, att_s: torch.Tensor, feat: torch.Tensor, m: int, width: int, *,
                           g: Optional[torch.Tensor] = None, other: Optional[torch.Tensor] = None,
                           lat: Optional[torch.Tensor] = None, lat_other: Optional[torch.Tensor] = None,
                           w_side: Optional[torch.Tensor] = None, fm_h: Optional[torch.Tensor] = None,
                           lt_w: Optional[torch.Tensor] = None, return_map: bool = False) -> dict:
    """K13: gradient x input on the embedded tokens of one SimpleSiamese side (rbr_explain_avgpool_attrib), per (pair, side)
    row p for entity ent[p]: ids [n_ent, R, T] (int64 / int32 / uint16) are the entities' reviews, mask [n_ent, R, T] bool
    their word masks (None: ids != 0); v / att_a [n_ent, R, F] and att_s [n_ent, R] the review attention's inputs, logit
    gradients and weights; feat [n_ent, F] the side features; lt_w [F, E] the latent transform's weight (None: F == E).
    g [P, F] = d pred / d feat, or None to form it in the kernel from the FM head: other [P] (the pair's other entity),
    lat [n_ent, K] / lat_other [n_other, K] (the two sides' LastFeat outputs), w_side [F, K] (this side's LastFeat.W) and
    fm_h [K].  Returns explain_attrib's dict for one document of R * T flat positions: text_total [P], top_pos /
    bottom_pos int64 [P, m] (-1 = none), top_attr / bottom_attr [P, m], review_attr [P, R] and with return_map `map`
    [P, R * T]."""
    table = _req(table, torch.float32, "table")
    ids = _ids(ids, "ids")
    if table.dim() != 2 or ids.dim() != 3:
        raise ValueError(f"rbr_b200: table [V, E] and ids [n_ent, R, T] expected, got {tuple(table.shape)} / {tuple(ids.shape)}")
    emb = table.shape[1]
    n_ent, R, T = ids.shape
    m, width = int(m), int(width)
    feat = _req(feat, torch.float32, "feat")
    F = feat.shape[1] if feat.dim() == 2 else 0
    if R < 1 or T < 1 or F < 1 or not explain_avgpool_supported(R * T, R, emb, F, m, width):
        raise ValueError(f"rbr_b200: explain_avgpool_attrib takes 1 <= R * T <= {EXPLAIN_MAX_POSITIONS}, 1 <= m <= "
                         f"{EXPLAIN_MAX_M}, 1 <= width <= {EXPLAIN_MAX_WIDTH} within 227 KB of shared memory (got {R} x {T}, "
                         f"emb={emb}, feat={F}, m={m}, width={width})")
    v, att_a = _req(v, torch.float32, "v"), _req(att_a, torch.float32, "att_a")
    att_s = _req(att_s, torch.float32, "att_s")
    if (feat.shape[0] != n_ent or tuple(v.shape) != (n_ent, R, F) or tuple(att_a.shape) != (n_ent, R, F)
            or tuple(att_s.shape) != (n_ent, R)):
        raise ValueError(f"rbr_b200: feat [{n_ent}, F], v / att_a [{n_ent}, {R}, F] and att_s [{n_ent}, {R}] expected, got "
                         f"{tuple(feat.shape)} / {tuple(v.shape)} / {tuple(att_a.shape)} / {tuple(att_s.shape)}")
    if mask is not None and tuple(mask.shape) != tuple(ids.shape):
        raise ValueError(f"rbr_b200: mask {tuple(mask.shape)} does not match ids {tuple(ids.shape)}")
    flags = _id_flags(ids, mask, True)
    mask = _mask_u8(mask, "mask")
    if lt_w is not None:
        lt_w = _req(lt_w.detach(), torch.float32, "lt_w")
        if tuple(lt_w.shape) != (F, emb):
            raise ValueError(f"rbr_b200: lt_w must be [{F}, {emb}], got {tuple(lt_w.shape)}")
    elif F != emb:
        raise ValueError(f"rbr_b200: without the latent transform the side feature width ({F}) must be emb ({emb})")
    ent = _req(ent, torch.int64, "ent").view(-1)
    P = ent.numel()
    n_other, K = 0, 0
    if g is not None:
        g = _req(g, torch.float32, "g")
        if tuple(g.shape) != (P, F):
            raise ValueError(f"rbr_b200: g must be [{P}, {F}], got {tuple(g.shape)}")
        checked = (g,)
    else:
        if any(t is None for t in (other, lat, lat_other, w_side, fm_h)):
            raise ValueError("rbr_b200: without g, other, lat, lat_other, w_side and fm_h are needed")
        other = _req(other, torch.int64, "other").view(-1)
        lat, lat_other = _req(lat, torch.float32, "lat"), _req(lat_other, torch.float32, "lat_other")
        w_side = _req(w_side.detach(), torch.float32, "w_side")
        fm_h = _req(fm_h.detach(), torch.float32, "fm_h").view(-1)
        K = fm_h.numel()
        n_other = lat_other.shape[0] if lat_other.dim() == 2 else -1
        if (other.numel() != P or tuple(lat.shape) != (n_ent, K) or lat_other.dim() != 2 or lat_other.shape[1] != K
                or tuple(w_side.shape) != (F, K) or K < 1):
            raise ValueError(f"rbr_b200: other [{P}], lat [{n_ent}, K], lat_other [n, K], w_side [{F}, K] and fm_h [K] expected, "
                             f"got {tuple(other.shape)} / {tuple(lat.shape)} / {tuple(lat_other.shape)} / "
                             f"{tuple(w_side.shape)} / {tuple(fm_h.shape)}")
        if P:
            lo, hi = torch.stack([other.min(), other.max()]).tolist()
            if lo < 0 or hi >= n_other:
                raise ValueError(f"rbr_b200: other ids must lie in [0, {n_other})")
        checked = (other, lat, lat_other, w_side, fm_h)
    for t, name in ((ids, "ids"), (mask, "mask"), (ent, "ent"), (v, "v"), (att_a, "att_a"), (att_s, "att_s"), (feat, "feat"),
                    (lt_w, "lt_w")) + tuple((t, "head input") for t in checked):
        if t is not None and t.device != table.device:
            raise ValueError(f"rbr_b200: `{name}` is on {t.device}, the table on {table.device}")
    if P:
        lo, hi = torch.stack([ent.min(), ent.max()]).tolist()
        if lo < 0 or hi >= n_ent:
            raise ValueError(f"rbr_b200: ent must lie in [0, {n_ent})")
    dev = table.device
    out = {"text_total": torch.empty(P, dtype=torch.float32, device=dev)}
    for side in ("top", "bottom"):
        out[f"{side}_pos"] = torch.empty(P, m, dtype=torch.int64, device=dev)
        out[f"{side}_attr"] = torch.empty(P, m, dtype=torch.float32, device=dev)
    if return_map:
        out["map"] = torch.empty(P, R * T, dtype=torch.float32, device=dev)
    out["review_attr"] = torch.empty(P, R, dtype=torch.float32, device=dev)
    if P == 0:
        return out
    lib.check(lib.rbr_explain_avgpool_attrib(
        _p(table), table.shape[0], emb, _p(ids), _p(mask), n_ent, R, T, _p(ent), P, _p(g), _p(other), _p(lat), _p(lat_other),
        n_other, _p(w_side), _p(fm_h), K, _p(v), _p(att_a), _p(att_s), _p(feat), F, _p(lt_w), m, width, _p(out["text_total"]),
        _p(out["top_pos"]), _p(out["top_attr"]), _p(out["bottom_pos"]), _p(out["bottom_attr"]), _p(out.get("map")),
        _p(out["review_attr"]), flags, _stream(True)), "rbr_explain_avgpool_attrib")
    return out
