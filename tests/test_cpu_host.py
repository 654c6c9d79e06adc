"""CPU-side tests (no GPU): the C-ABI library loads and exports every declared symbol, the host logic
(gradient arena, sharding, data-parallel all-reduce over gloo with world_size 2) and the synthetic data."""
import os
import subprocess
import sys

import pytest
import torch

import rbr_b200
from rbr_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cabi_loads_and_exports_every_declared_symbol():
    import __graft_entry__ as ge
    if not os.path.exists(os.path.join(ge.CSRC, "librbr_b200.so")):
        ge.build()
    from rbr_b200._lib import lib
    assert len(lib.protos) >= 17
    for name in lib.protos:
        assert getattr(lib, name) is not None, name
    assert lib.rbr_version() >= 100
    assert lib.rbr_emb_pad(300) == 320 and lib.rbr_emb_pad(100) == 128
    assert lib.rbr_conv_pack_bytes(300, 100, 3) > 0
    assert lib.rbr_conv_bwd_workspace_bytes(8, 100, 3, 300, 50000) > 0
    assert lib.rbr_embgrad_workspace_bytes(1000, 50000) > 0


def test_no_cpu_fallback():
    m = rbr_b200.DeepCoNNpp(9, 7, 60, [3], 12, 8, 6, 20, None, 0.0)
    ids = torch.zeros(2, 20, dtype=torch.long)
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        m(ids, ids, ids != 0, ids != 0, torch.ones(2, dtype=torch.long), torch.ones(2, dtype=torch.long))


def test_state_dict_keys_match_reference_goldens():
    from conftest import Golden
    g = Golden("deepconn_multik")
    m = g.meta
    model = rbr_b200.DeepCoNNpp(m["U"], m["I"], m["V"], "3,5", m["E"], m["H"], m["K"], m["L"], None, 0.0)
    assert set(model.state_dict()) == set(g.params)
    for k, v in model.state_dict().items():
        assert v.shape == g.params[k].shape, k
    n = Golden("narre_small")
    m = n.meta
    model = rbr_b200.NARRE(m["U"], m["I"], m["V"], [3], m["H"], m["E"], m["A"], m["K"], m["R"], m["T"], 0.5, 0, 0, 0, None, "CNN")
    assert set(model.state_dict()) == set(n.params)
    with pytest.raises(ValueError):
        rbr_b200.layers.NgramFeat([3], 8, 8, 10, arch="nope")
    h = Golden("deepconn_hier")
    m = h.meta
    model = rbr_b200.DeepCoNNpp(m["U"], m["I"], m["V"], [m["k"]], m["E"], m["H"], m["K"], m["L"], None, 0.0, arch="HierPooling")
    assert set(model.state_dict()) == set(h.params)                  # incl. ngram.feature_layer.0.proj_layer.{weight,bias}
    with pytest.raises(AssertionError):
        rbr_b200.layers.MyConv1d([2], 8, 8)              # even kernel sizes are rejected, layers.py:39


def test_grad_arena_views_are_disjoint_and_aligned():
    from rbr_b200.ops import GradArena
    ps = [("a", torch.nn.Parameter(torch.zeros(3, 5))), ("b", torch.nn.Parameter(torch.zeros(7))),
          ("c", torch.nn.Parameter(torch.zeros(2, 2), requires_grad=False))]
    arena = GradArena(ps)
    va, vb = arena.view(ps[0][1]), arena.view(ps[1][1])
    assert arena.view(ps[2][1]) is None
    assert va.shape == (3, 5) and vb.shape == (7,)
    assert va.data_ptr() % 256 == arena.flat.data_ptr() % 256 and (vb.data_ptr() - va.data_ptr()) % 256 == 0
    va.fill_(1.0)
    assert float(vb.sum()) == 0.0 and float(arena.flat.sum()) == 15.0


def test_synthetic_batches_follow_the_preprocessing_contract():
    (u, i, um, im, uid, iid), r = synth.deepconn_batch(16, 50, 1000, 30, 20, seed=3)
    assert u.dtype == torch.int64 and um.dtype == torch.bool and torch.equal(um, u != 0)
    assert int(u.max()) < 1000 and int(u[um].min()) >= 3
    assert ((u == 0).long().diff(dim=1) >= 0).all()                      # padding only at the tail
    assert set(r.tolist()) <= {1.0, 2.0, 3.0, 4.0, 5.0} and int(uid.min()) >= 1
    (ut, it, utm, itm, uid, iid, reu, rei), r = synth.narre_batch(8, 5, 12, 500, 30, 20, seed=3)
    assert ut.shape == (8, 5, 12) and reu.shape == (8, 5)
    pad_reviews = (reu == 0)
    assert (ut[pad_reviews] == 0).all()                                   # padded reviews are all-zero with id 0
    again = synth.narre_batch(8, 5, 12, 500, 30, 20, seed=3)[0][0]
    assert torch.equal(ut, again)


def test_shard_range_partitions_batch():
    from rbr_b200.parallel import shard_range
    for n, w in ((4096, 8), (10, 4), (7, 2), (3, 8)):
        seen = []
        for r in range(w):
            seen += list(shard_range(n, r, w))
        assert seen == list(range(n))


_DP_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.environ["RBR_ROOT"])
import rbr_b200
from rbr_b200 import parallel
from rbr_b200.ops import GradArena
rank, local, world = parallel.init_from_env("gloo")
torch.manual_seed(0)
model = torch.nn.Linear(6, 3)
parallel.broadcast_parameters(model)
x = torch.arange(8 * 6, dtype=torch.float32).view(8, 6) / 10
y = torch.ones(8, 3)
sh = parallel.shard_range(8, rank, world)
# gradients placed in a flat arena, as the CUDA backward does
arena = GradArena(list(model.named_parameters()))
loss = torch.nn.functional.mse_loss(model(x[sh.start:sh.stop]), y[sh.start:sh.stop])
gw, gb = torch.autograd.grad(loss, [model.weight, model.bias])
model.weight.grad = arena.view(model.weight); model.weight.grad.copy_(gw)
model.bias.grad = arena.view(model.bias); model.bias.grad.copy_(gb)
model.last_arena = arena
n = parallel.allreduce_gradients(model)
assert n == 1
ref = torch.nn.Linear(6, 3); ref.load_state_dict(model.state_dict())
torch.nn.functional.mse_loss(ref(x), y).backward()
assert torch.allclose(model.weight.grad, ref.weight.grad, atol=1e-6), (model.weight.grad, ref.weight.grad)
assert torch.allclose(model.bias.grad, ref.bias.grad, atol=1e-6)
# overlapped path: the (large) first gradient is reduced from a hook fired inside backward, the rest afterwards
import types
model.ngram = types.SimpleNamespace(table_grad_hook=None)
parallel.enable_overlap(model)
arena2 = GradArena(list(model.named_parameters()))
model.weight.grad = arena2.view(model.weight); model.weight.grad.copy_(gw)
model.bias.grad = arena2.view(model.bias); model.bias.grad.copy_(gb)
model.last_arena = arena2
model.ngram.table_grad_hook(model.weight.grad)            # what ops.EncodeDocsFn.backward does once the table gradient is complete
n = parallel.allreduce_gradients(model)
assert n == 1                                             # only the remainder is reduced after backward
assert torch.allclose(model.weight.grad, ref.weight.grad, atol=1e-6)
assert torch.allclose(model.bias.grad, ref.bias.grad, atol=1e-6)
# the same through AUTOGRAD: a backward that accumulates into an arena view, fires the hook and RETURNS that view (what
# ops.EncodeDocsFn.backward does).  The hook must not keep a reference to the returned tensor: AccumulateGrad would then
# clone it, `.grad` would leave the arena and the early reduction would be lost.
class _ArenaMatmul(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, arena, hook):
        ctx.save_for_backward(x); ctx.w, ctx.arena, ctx.hook = w, arena, hook
        return x @ w.t()
    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        buf = ctx.arena.view(ctx.w)
        buf.add_(g.t() @ x)
        ctx.hook(buf)
        return None, buf, None, None
model.zero_grad(set_to_none=True)
arena3 = GradArena(list(model.named_parameters()))
out = _ArenaMatmul.apply(x[sh.start:sh.stop], model.weight, arena3, model.ngram.table_grad_hook) + model.bias
torch.nn.functional.mse_loss(out, y[sh.start:sh.stop]).backward()
lo = arena3.flat.data_ptr(); hi = lo + arena3.flat.numel() * 4
assert lo <= model.weight.grad.data_ptr() < hi, "the weight gradient was cloned out of the arena (hook kept a reference?)"
bslot = arena3.view(model.bias); bslot.copy_(model.bias.grad); model.bias.grad = bslot
model.last_arena = arena3
n = parallel.allreduce_gradients(model)
assert n == 1
assert torch.allclose(model.weight.grad, ref.weight.grad, atol=1e-6), (model.weight.grad, ref.weight.grad)
assert torch.allclose(model.bias.grad, ref.bias.grad, atol=1e-6)
del model.ngram, model._rbr_early_table
# slow path: grads not in the arena
model.last_arena = None
model.weight.grad = gw.clone(); model.bias.grad = gb.clone()
parallel.allreduce_gradients(model)
assert torch.allclose(model.weight.grad, ref.weight.grad, atol=1e-6)
dist.barrier()
print("rank", rank, "ok")
'''


def test_data_parallel_allreduce_world2_gloo(tmp_path):
    script = tmp_path / "dp_worker.py"
    script.write_text(_DP_WORKER)
    env = dict(os.environ, RBR_ROOT=ROOT, OMP_NUM_THREADS="1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29731", str(script)],
                         env=env, capture_output=True, text=True, timeout=240)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.count("ok") == 2


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours) prints ONE JSON line with the contract's keys,
    and extra ranks of a torchrun launch exit without work."""
    import json
    env = dict(os.environ, OMP_NUM_THREADS="4")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["higher_is_better"] is True
    from oracle import ref_loader
    assert d["value"] > 0 and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["kind"] == ("reference" if ref_loader.available() else "port")
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "DeepCoNN" in d["metric"] and "workload" in d["config"]
    assert d["steps"] == 1 and d["warmup"] == 1                         # the requested counts are echoed
    assert d["narre"]["impl"] == "reference" and "NARRE" in d["narre"]["metric"] and d["narre"]["value"] > 0
    out2 = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                          env=dict(env, RANK="1", WORLD_SIZE="2"), capture_output=True, text=True, timeout=120)
    assert out2.returncode == 0 and out2.stdout.strip() == ""


def test_grad_arena_layout_is_cached_per_module_and_tracks_requires_grad():
    from rbr_b200.ops import GradArena
    m = torch.nn.Sequential(torch.nn.Linear(5, 3), torch.nn.Linear(3, 2))
    a1, a2 = GradArena.for_module(m), GradArena.for_module(m)
    assert a1 is not a2 and a1.slots is a2.slots            # fresh arena per step, shared layout
    assert a1.total == 64 * 4                                # four parameters, 256-byte (64-float) aligned slots
    v = a1.view(m[0].weight)
    assert v.shape == m[0].weight.shape and float(v.abs().sum()) == 0.0
    v.add_(1.0)
    assert float(a1.flat.sum()) == 15.0 and a2.flat is None  # lazily allocated, independent buffers
    m[1].bias.requires_grad_(False)
    a3 = GradArena.for_module(m)
    assert a3.slots is not a1.slots and a3.view(m[1].bias) is None and a3.total == 64 * 3
    with torch.no_grad():
        assert GradArena.for_module(m) is None
    # a persistent external buffer (the NVLS symmetric-memory arena) is re-zeroed, not re-allocated
    buf = torch.ones(1024)
    m.__dict__["_rbr_arena_buffer"] = buf
    a4 = GradArena.for_module(m)
    w = a4.view(m[0].weight)
    assert w.data_ptr() == buf.data_ptr() and float(buf[:a4.total].sum()) == 0.0 and float(buf[a4.total:].sum()) == 1024 - a4.total
    # ... and a `.grad` that still aliases it when the next backward starts (gradient accumulation, zero_grad(set_to_none=False))
    # is an error instead of a silent wipe
    m[0].weight.grad = w
    a5 = GradArena.for_module(m)
    with pytest.raises(RuntimeError, match="set_to_none=True"):
        a5.view(m[0].weight)
    m[0].weight.grad = None
    assert GradArena.for_module(m).view(m[0].weight) is not None


def test_conv_tc2_plan_invariants():
    """Tiling logic of the CTA-pair conv kernel (host code, no GPU): shared memory / TMEM budgets, UMMA shape rules, ring depth,
    short-document packing."""
    import ctypes
    from rbr_b200._lib import lib
    out = (ctypes.c_int64 * 16)()
    shapes = [(300, 100, 3, 500, 1), (300, 150, 3, 60, 1), (300, 100, 3, 60, 1), (100, 200, 1, 500, 0), (100, 100, 2, 500, 0),
              (100, 100, 4, 500, 0), (300, 300, 3, 200, 1), (16, 16, 1, 40, 0), (8, 1, 3, 3, 1), (72, 48, 7, 260, 3),
              (100, 200, 5, 31, 2), (40, 33, 3, 17, 1), (300, 100, 5, 500, 2), (512, 256, 3, 128, 1), (300, 100, 3, 10, 1)]
    n_ok = 0
    for E, H, K, L, pad in shapes:
        assert lib.rbr_conv_tc2_plan(E, H, K, L, pad, 1000, ctypes.cast(out, ctypes.c_void_p)) == 0
        ok, P, Nb, NL, nkb, ksteps, groups, stage_bytes, nst, w_bytes, mode_b, D, S, tpu, smem, tmem = list(out)
        if not ok:
            continue
        n_ok += 1
        Lext, Lout = L + 2 * pad, L + 2 * pad - K + 1
        assert P >= 1 and P * Nb >= H and Nb % 16 == 0 and 16 <= Nb <= 256 and NL * 2 == Nb          # UMMA N rules, M = 256
        assert nkb * 64 >= E and ksteps * 16 >= E and ksteps <= nkb * 4
        assert groups * 4 >= 128 + K - 1 and stage_bytes % 1024 == 0 and stage_bytes >= groups * 512   # swizzle-atom aligned stages
        assert nst >= 3 and smem <= 232448 and w_bytes == K * ((E + 15) // 16 * 2) * NL * 16
        assert tmem in (256, 512) and tmem >= 2 * Nb
        if mode_b:
            assert S % 32 == 0 and S >= Lext and 1 <= D <= 4 and tpu == 1
            assert (D - 1) * S + Lext <= 128 + K - 1                                                   # all documents' rows are staged
            assert (D - 1) * S + Lout <= 128                                                           # and their outputs are TMEM lanes
        else:
            assert D == 1 and tpu == (Lout + 127) // 128
    assert n_ok >= 12
    # the benchmark shapes take one pass each (A operand gathered once)
    lib.rbr_conv_tc2_plan(300, 100, 3, 500, 1, 4096, ctypes.cast(out, ctypes.c_void_p))
    assert out[0] == 1 and out[1] == 1 and out[2] == 112 and out[8] >= 6
    lib.rbr_conv_tc2_plan(300, 150, 3, 60, 1, 40960, ctypes.cast(out, ctypes.c_void_p))
    assert out[0] == 1 and out[1] == 1 and out[2] == 160 and out[10] == 1 and out[11] == 2 and out[12] == 64


def test_conv_fwd_workspace_holds_the_row_index_table():
    """rbr_conv_fwd_workspace_bytes2 = the document lists + one int32 per staged position of every document (and one all -1 row):
    a row is `tiles * 128 + 8` entries with one document per tile (a tile's 136 indices are then one contiguous, 16-byte aligned
    run for the index warp's bulk copy) or the slot stride S with several documents per tile (host code, no GPU)."""
    import ctypes
    from rbr_b200._lib import lib
    out = (ctypes.c_int64 * 16)()
    for E, H, K, L, pad, n in [(300, 100, 3, 500, 1, 4096), (300, 150, 3, 60, 1, 40960), (300, 100, 5, 1000, 2, 333), (300, 100, 1, 200, 0, 130),
                               (300, 100, 4, 129, 0, 67), (300, 100, 2, 14, 0, 999)]:
        lib.rbr_conv_tc2_plan(E, H, K, L, pad, n, ctypes.cast(out, ctypes.c_void_p))
        assert out[0] == 1
        mode_b, S, tpu = out[10], out[12], out[13]
        rs = S if mode_b else tpu * 128 + 8
        assert rs % 4 == 0 and rs >= L + 2 * pad
        base = lib.rbr_conv_fwd_workspace_bytes(n)
        assert base % 256 == 0                                                       # the table starts 16-byte aligned behind the lists
        assert lib.rbr_conv_fwd_workspace_bytes2(n, L, K, pad) == base + (n + 1) * rs * 4


def test_staged_inputs_wire_format_on_cpu():
    """staging.StagedInputs host logic (no GPU): token ids travel as uint16 when the vocabulary fits and as int32 otherwise, masks
    are not sent, everything else travels unchanged; `pack` refuses ids that would alias under the narrowing."""
    import pytest
    from rbr_b200 import synth
    from rbr_b200.staging import StagedInputs
    batch, ratings = synth.deepconn_batch(16, 40, 600, 50, 30, seed=3)
    ref_bytes = sum(t.numel() * t.element_size() for t in batch) + ratings.numel() * 4
    for vocab, dt, frac in ((600, torch.uint16, 0.30), (65536, torch.uint16, 0.30), (65537, torch.int32, 0.52), (None, torch.int32, 0.52)):
        st = StagedInputs(batch, ratings, "cpu", vocab=vocab)
        assert st.token_dtype == dt and st.batch[0].dtype == dt and st.batch[2] is None and st.batch[3] is None
        assert st.h2d_bytes % 256 == 0 and st.h2d_bytes < frac * ref_bytes + 6 * 256
        host = st.pack(batch, ratings, out=torch.empty(st.nbytes, dtype=torch.uint8))
        st.dev.copy_(host)                                   # the one H2D copy
        assert torch.equal(st.batch[0].to(torch.int64), batch[0]) and torch.equal(st.batch[1].to(torch.int64), batch[1])
        assert torch.equal(st.batch[4], batch[4]) and torch.equal(st.batch[5], batch[5]) and torch.equal(st.ratings, ratings)
    st = StagedInputs(batch, ratings, "cpu", vocab=600)
    bad = [t.clone() for t in batch]
    bad[0][0, 0] = 70000
    with pytest.raises(ValueError, match="uint16"):
        st.pack(bad, ratings, out=torch.empty(st.nbytes, dtype=torch.uint8))
    # masks that are NOT ids != 0 can still be sent
    st = StagedInputs(batch, ratings, "cpu", vocab=600, derive_masks=False)
    assert st.batch[2] is not None and st.batch[2].dtype == torch.uint8


def test_conv_bwd_cmat_filter_blocks_and_declined_shapes():
    """Filter blocks of the dense tensor-core backward's coefficient matrix (host code, no GPU): C32 = V x round_up(H k, 64) fp32 is
    cut into ceil(bytes / 80 MiB) blocks (at most 16) of round_up(ceil(H / blocks), 4) filters.  tests/test_gpu_conv_bwd_variants.py
    runs these shapes on the GPU.  Shapes the backward cannot finish get no workspace, and go to the sparse kernels."""
    from rbr_b200._lib import lib
    chunks, ws = lib.rbr_conv_bwd_cmat_chunks, lib.rbr_conv_bwd_cmat_workspace_bytes
    assert chunks(327680, 64, 16, 4) == 1 and chunks(327681, 64, 16, 4) == 2          # C32 exactly 80 MiB, and one row more
    for shape, n in {(3000, 300, 100, 3): 1, (60000, 300, 150, 3): 2, (100000, 100, 150, 3): 3, (350000, 64, 512, 4): 16,
                     (200000, 64, 9, 8): 2, (400000, 64, 9, 4): 2, (2000, 32, 1024, 4): 1, (2000, 100, 820, 3): 1}.items():
        assert chunks(*shape) == n, shape
    rup = lambda x, m: (x + m - 1) // m * m
    for V, E, H, k in ((350000, 64, 512, 4), (3000, 300, 100, 3), (1, 4, 1, 1), (1000, 448, 24, 3)):
        hjp = rup(H * k, 64)                                           # C32 fp32 + [hi | lo] bf16 + the [H k][E] weight scratch
        assert ws(V, E, H, k) == rup(V * hjp * 4, 1024) + rup(V * 2 * hjp * 2, 1024) + rup(H * k * rup(E, 4) * 4, 1024), (V, E, H, k)
    # declined: E in (448, 512] (the weight GEMM's ring would need 240 KB of shared memory), E % 4, E > 512, k > 8, H > 1024,
    # H k beyond 4096 columns, C32 over 3 GiB
    for shape in ((5000, 452, 100, 3), (5000, 480, 100, 3), (5000, 512, 100, 3), (5000, 30, 100, 3), (5000, 516, 100, 3),
                  (5000, 64, 100, 9), (5000, 64, 1025, 1), (5000, 64, 1024, 5), (2000, 100, 820, 5), (800000, 64, 1024, 1)):
        assert ws(*shape) == 0 and chunks(*shape) == 0, shape
    assert ws(5000, 448, 100, 3) > 0 and ws(5000, 444, 100, 3) > 0


def test_narre_attn_pair_plan_boundary():
    """Which NARRE attention shapes the two-sided tensor-core kernel takes (host code, no GPU).  NARRE falls back to the per-side
    kernels outside this set, and test_attention_pair_tensor_core_kernels_vs_oracle runs the edge shapes pinned here."""
    from rbr_b200._lib import lib
    sup = lambda R, H, A: bool(lib.rbr_narre_attn_pair_supported(R, H, A))
    assert sup(10, 150, 32)                                   # the benchmarked NARRE shape
    for R, h_max in ((1, 128), (10, 160), (64, 192)):        # largest hidden per review count, whatever att_dim <= 32
        for A in (1, 16, 32):
            assert sup(R, h_max, A) and not sup(R, h_max + 1, A), (R, A)
    assert sup(10, 101, 16) and sup(10, 1, 1)
    assert not sup(65, 64, 32) and not sup(0, 64, 32)        # reviews in [1, 64]
    assert not sup(10, 150, 33) and not sup(10, 150, 0)      # att_dim in [1, 32]
    assert not sup(10, 0, 32)


def test_datt_gate_entry_points_decline_unsupported_shapes_without_a_device():
    """K5 takes E <= 128 and odd windows up to 7: the gate forward and backward return RBR_EUNSUPPORTED for E = 129, window 2
    and window 9 before they look at any pointer (all NULL here) or touch a device."""
    from rbr_b200._lib import lib
    for emb, win in ((129, 5), (100, 2), (100, 9)):
        assert lib.rbr_datt_gate_fwd(None, 10, emb, None, 1, 8, None, None, win, None, None, None, None, None, 0, 0, None) == -4
        assert b"rbr_datt_gate_fwd" in lib.rbr_last_error()
        assert lib.rbr_datt_gate_bwd(None, 10, emb, None, 1, 8, None, win, None, None, None, None, None, 0, None, None, None,
                                     None, None, None, 0, 0, None) == -4
        assert b"rbr_datt_gate_bwd" in lib.rbr_last_error()
