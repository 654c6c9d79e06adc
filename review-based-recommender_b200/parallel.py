"""Data-parallel plumbing: one process per GPU, batch sharded across ranks, ONE all-reduce of the flat
parameter-gradient buffer per step (SURVEY.md §8e).  The reference's only parallel mode is
nn.DataParallel (trainer/train_deepconn_pp.py:129-131), which re-broadcasts every parameter each step.

The forward/backward has no collective: every rank encodes its own shard.  After `loss.backward()` the
model's GradArena holds all parameter gradients in one contiguous fp32 buffer (ops.GradArena), so the
exchange is a single NCCL all-reduce over NVLink/NVSwitch followed by a scale by 1/world_size (each rank's
MSELoss averaged over its own shard → mean over the global batch).
"""
from __future__ import annotations

import os
from typing import Iterable, Optional

import torch
import torch.distributed as dist


def init_from_env(backend: Optional[str] = None) -> tuple:
    """Initialise torch.distributed from torchrun's env (RANK / LOCAL_RANK / WORLD_SIZE / MASTER_*)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
        dist.init_process_group(backend=backend, rank=rank, world_size=world)
    return rank, local, world


def shard_range(n: int, rank: int, world: int) -> range:
    """Contiguous shard of n samples for this rank (first n % world ranks get one extra)."""
    base, extra = divmod(n, world)
    start = rank * base + min(rank, extra)
    return range(start, start + base + (1 if rank < extra else 0))


def _arena_covers(model: torch.nn.Module) -> bool:
    arena = getattr(model, "last_arena", None)
    if arena is None or arena.flat is None:
        return False
    lo = arena.flat.data_ptr()
    hi = lo + arena.flat.numel() * 4
    for p in model.parameters():
        if p.requires_grad:
            if p.grad is None or not (lo <= p.grad.data_ptr() < hi):
                return False
    return True


class _EarlyTableReduce:
    """State of the overlapped word-table all-reduce of one backward pass (see enable_overlap).

    Only the ADDRESS RANGE of the gradient is remembered, never the tensor autograd is about to receive: an extra Python
    reference to that tensor raises its use_count, AccumulateGrad then clones it instead of stealing it, and the clone —
    made on the main stream while the collective is still writing the buffer — would be a data race and would detach `.grad`
    from the arena.  The collective runs on a separate alias (own TensorImpl, same storage)."""

    def __init__(self):
        self.work = None
        self.alias: Optional[torch.Tensor] = None     # detached alias the collective reduces in place
        self.ptr = 0
        self.numel = 0

    def clear(self):
        self.work, self.alias, self.ptr, self.numel = None, None, 0, 0


def enable_overlap(model: torch.nn.Module, group=None) -> None:
    """Start the all-reduce of the word-embedding gradient (≈ 90 % of all gradient bytes) as soon as it is complete.

    The encoder's backward (ops.EncodeDocsFn) finishes the table gradient of every document side first and then calls
    this hook; the collective runs on NCCL's stream while the conv weight/bias-gradient kernels still execute, and
    allreduce_gradients() later reduces only the remaining (small) gradients and waits for it."""
    ngram = getattr(model, "ngram", None)
    if ngram is None or not hasattr(ngram, "table_grad_hook"):
        return
    state = _EarlyTableReduce()
    model._rbr_early_table = state

    def hook(g_table: torch.Tensor):
        if dist.is_initialized() and dist.get_world_size(group) > 1:
            state.ptr, state.numel = g_table.data_ptr(), g_table.numel()
            state.alias = g_table.detach().view(-1)          # new TensorImpl on the same storage: g_table's use_count is untouched
            state.work = dist.all_reduce(state.alias, op=dist.ReduceOp.AVG if dist.get_backend(group) == "nccl" else dist.ReduceOp.SUM,
                                         group=group, async_op=True)

    ngram.table_grad_hook = hook


class _NvlsState:
    def __init__(self, hdl, mc, n, rank, world, device, overlap, kind="multimem"):
        self.hdl, self.mc, self.n, self.rank, self.world = hdl, mc, n, rank, world
        # kind "p2p": plain peer loads / stores over the symmetric-memory peer mappings (rbr_p2p_allreduce_f32) — fewer link
        # bytes than the switch reduction for small worlds; "multimem": the NVLS kernel
        self.kind = kind
        self.peers = None
        if kind == "p2p":
            import ctypes
            ptrs = [int(x) for x in hdl.buffer_ptrs]
            self.peers = (ctypes.c_uint64 * len(ptrs))(*ptrs)
        self.overlap = overlap
        self.side = torch.cuda.Stream(device=device, priority=-1) if overlap else None
        self.ev_ready = torch.cuda.Event() if overlap else None
        self.ev_done = torch.cuda.Event() if overlap else None
        self.early: Optional[tuple] = None          # (lo, hi) float range already being reduced on the side stream

    def reduce(self, lo: int, cnt: int, scale: float, stream: int) -> None:
        """All-reduce floats [lo, lo + cnt) of the arena on `stream` (between the caller's two cross-GPU barriers)."""
        from ._lib import lib
        if self.kind == "p2p":
            import ctypes
            lib.check(lib.rbr_p2p_allreduce_f32(ctypes.cast(self.peers, ctypes.c_void_p), lo, cnt, self.rank, self.world, scale, 0, stream),
                      "rbr_p2p_allreduce_f32")
        else:
            lib.check(lib.rbr_multimem_allreduce_f32(self.mc + 4 * lo, cnt, self.rank, self.world, scale, 0, stream),
                      "rbr_multimem_allreduce_f32")


def enable_nvls_allreduce(model: torch.nn.Module, group=None, overlap: bool = True, kind: str = "auto") -> bool:
    """Put the model's flat gradient arena in symmetric memory (torch.distributed._symmetric_memory) and let
    allreduce_gradients() reduce it with the library's own NVLS kernel (rbr_multimem_allreduce_f32: multimem.ld_reduce /
    multimem.st through the NVSwitch, 1/world folded in) instead of ncclAllReduce.  Collective call (every rank, after
    init and before the first training step).  Returns False — and leaves the NCCL path in place — when the GPUs have
    no NVLS multicast support.

    kind: "multimem" (the switch reduces), "p2p" (plain peer loads / stores: a third of the link bytes at world 2, 0.6 at 4),
    "auto" = p2p for world 2, multimem above.  Measured on the 64.6 MB arena, barriers included (tools/allreduce_sweep.py):
    world 2: p2p 113 us, multimem 180 us, ncclAllReduce 148 us; world 4: p2p 165 us, multimem 163 us (with a quarter of the
    CTAs, which matters for the overlapped word-table slice), ncclAllReduce 185 us.

    overlap=True: the word-embedding gradient (≈ 90 % of the bytes) is reduced on a side stream from inside backward,
    as soon as the table gradients of all document sides are complete (ops.EncodeDocsFn runs them first), concurrently
    with the conv weight-gradient kernels: the reduction kernel is link-bound with 32 CTAs, so it takes few SMs."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1 or dist.get_backend(group) != "nccl":
        return False
    from .ops import GradArena
    was = torch.is_grad_enabled()
    torch.set_grad_enabled(True)
    try:
        layout = GradArena.for_module(model)
    finally:
        torch.set_grad_enabled(was)
    if layout is None or layout.total == 0:
        return False
    try:
        import torch.distributed._symmetric_memory as symm_mem
        pg = group if group is not None else dist.group.WORLD
        dev = next(model.parameters()).device
        n = (layout.total + 1023) // 1024 * 1024
        buf = symm_mem.empty(n, dtype=torch.float32, device=dev)
        hdl = symm_mem.rendezvous(buf, pg)
        mc = int(getattr(hdl, "multicast_ptr", 0) or 0)
        ok = torch.tensor([1 if mc else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
        if int(ok.item()) == 0:
            return False
    except Exception:
        return False
    ngram = getattr(model, "ngram", None)
    overlap = bool(overlap and ngram is not None and hasattr(ngram, "table_grad_hook"))
    world = dist.get_world_size(group)
    if kind == "auto":
        kind = "p2p" if world == 2 else "multimem"
    if kind == "p2p" and world not in (2, 4, 8):
        kind = "multimem"
    st = _NvlsState(hdl, mc, n, dist.get_rank(group), world, dev, overlap, kind)
    model.__dict__["_rbr_arena_buffer"] = buf
    model.__dict__["_rbr_nvls"] = st
    if overlap:
        from ._lib import lib

        def hook(g_table: torch.Tensor):
            lo = (g_table.data_ptr() - buf.data_ptr()) // 4
            cnt = g_table.numel() // 4 * 4
            if lo < 0 or lo + cnt > n or lo % 4 or cnt == 0:
                return
            main = torch.cuda.current_stream()
            st.ev_ready.record(main)
            with torch.cuda.stream(st.side):
                st.side.wait_event(st.ev_ready)
                hdl.barrier(channel=2)          # every rank's table gradient is complete
                st.reduce(lo, cnt, 1.0 / st.world, st.side.cuda_stream)
                hdl.barrier(channel=3)
                st.ev_done.record(st.side)
            st.early = (lo, lo + cnt)

        ngram.table_grad_hook = hook
    return True


def _nvls_allreduce(model: torch.nn.Module, flat: torch.Tensor, average: bool) -> bool:
    st = model.__dict__.get("_rbr_nvls")
    buf = model.__dict__.get("_rbr_arena_buffer")
    if st is None or buf is None or flat.data_ptr() != buf.data_ptr():
        return False
    from ._lib import lib
    main = torch.cuda.current_stream()
    scale = (1.0 / st.world) if average else 1.0
    ranges = [(0, st.n)]
    if st.early is not None:
        lo, hi = st.early
        ranges = [r for r in ((0, lo), (hi, st.n)) if r[1] > r[0]]
    st.hdl.barrier(channel=0)                   # every rank has finished writing its gradients (stream-ordered, device side)
    for lo, hi in ranges:
        st.reduce(lo, hi - lo, scale, main.cuda_stream)
    st.hdl.barrier(channel=1)                   # every slice has been broadcast before anyone reads the result
    if st.early is not None:
        main.wait_event(st.ev_done)             # the overlapped word-table reduction
        st.early = None
    return True


def allreduce_gradients(model: torch.nn.Module, group=None, average: bool = True, compress: Optional[str] = None) -> int:
    """Sum (and average) parameter gradients across ranks.  Returns the number of collectives issued after backward:
    1 when every `.grad` lives in the step's flat arena (the fast path), else one flattened bucket.  With
    enable_overlap(model) the word-table gradient was already started from inside backward and is excluded here."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return 0
    world = dist.get_world_size(group)
    nccl = dist.get_backend(group) == "nccl"
    op = dist.ReduceOp.AVG if (average and nccl) else dist.ReduceOp.SUM       # NCCL averages in the collective itself
    post_scale = average and not nccl
    early = getattr(model, "_rbr_early_table", None)
    if compress not in (None, "bf16"):
        raise ValueError("compress must be None or 'bf16'")
    if _arena_covers(model):
        flat = model.last_arena.flat
        if (early is None or early.work is None) and compress is None and _nvls_allreduce(model, flat, average):
            return 1
        if compress == "bf16" and nccl and (early is None or early.work is None):
            # optional gradient compression: halves the bytes on the wire; the averaged gradient is rounded to bf16
            # (relative error 2^-9 per element) — off by default, the reference's DataParallel reduces in fp32
            half = flat.to(torch.bfloat16)
            dist.all_reduce(half, op=op, group=group)
            flat.copy_(half)
            return 1
        pieces = [flat]
        if early is not None and early.work is not None:
            lo = (early.ptr - flat.data_ptr()) // 4
            hi = lo + early.numel
            if 0 <= lo and hi <= flat.numel():
                pieces = [t for t in (flat[:lo], flat[hi:]) if t.numel() > 0]
            else:                                   # the early gradient did not come from this arena: nothing to exclude
                early.work.wait()
                early.clear()
        n = 0
        for t in pieces:
            dist.all_reduce(t, op=op, group=group)
            if post_scale:
                t.mul_(1.0 / world)
            n += 1
        if early is not None and early.work is not None:
            early.work.wait()
            if average and not nccl:
                early.alias.mul_(1.0 / world)
            early.clear()
        return n
    done_ptr = None
    if early is not None and early.work is not None:          # mixed case: finish the early one; the bucket below skips it
        early.work.wait()
        if average and not nccl:
            early.alias.mul_(1.0 / world)
        done_ptr = early.ptr
        early.clear()
    grads = [p.grad for p in model.parameters() if p.requires_grad and p.grad is not None
             and not (done_ptr is not None and p.grad.data_ptr() == done_ptr)]
    if not grads:
        return 0
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, op=op, group=group)
    if post_scale:
        flat.mul_(1.0 / world)
    off = 0
    for g in grads:
        g.copy_(flat[off:off + g.numel()].view_as(g))
        off += g.numel()
    return 1


def broadcast_parameters(model: torch.nn.Module, src: int = 0, group=None) -> None:
    """Make every rank start from rank `src`'s parameters (replicated-parameter DP)."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return
    for p in model.parameters():
        dist.broadcast(p.data, src=src, group=group)
