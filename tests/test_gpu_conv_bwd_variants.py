"""Every variant of the conv backward against a float64 reference, at the shapes that select it.

`EncodeDocsFn.backward` (ops.py) picks, per conv:

  K2c  dense tensor-core backward (csrc/conv_bwd_tc.cu), bf16 precision, shapes rbr_conv_bwd_cmat_supported accepts:
         cmat_scatter_fast_kernel<k, 2, id width, mask mode>   k in {1, 3, 5}
         cmat_scatter_kernel<0, 2>                            any other k (the generic scatter)
         cmat_split_kernel                                    once per filter block of C32 (blocks of <= 80 MiB, at most 16)
         cmat_table_gemm_kernel / cmat_weight_gemm_kernel     the two tcgen05 GEMMs
  K2b  arg-max-sparse CUDA-core kernels (csrc/conv_bwd.cu): fp32 precision, CONV_BWD_SPARSE, and shapes K2c declines:
         conv_bwd_weight_kernel<K, nq> / conv_bwd_table_kernel<nq>   E % 4 == 0, E <= 512, K in {1, 2, 3, 4, 5, 7}
         conv_bwd_weight_scalar_kernel / conv_bwd_table_scalar_kernel  otherwise

Each case names the variant it targets and checks, under torch.profiler, that this is what ran.

Reference.  The forward is linearised at the point the kernels computed: the kernel's arg-max routes each (document, filter)
to one window, the float64 pre-activation y of that window on the forward's operands gives the activation derivative
(relu: y > 0, tanh: 1 - tanh(y)^2), and the gradients are those of sum(G * act'(y) * y) over the backward's operands — in
bf16 mode the bf16-rounded table and conv weights (K2c multiplies the bf16 shadow and the rounded weights; K2b's vector
kernels read the same), in fp32 mode (and in K2b's scalar kernels, which read the fp32 table and weights in both precisions)
the fp32 values.  Out-of-range ids read as zero rows and row `padding_idx` of the table gradient is zero (torch semantics:
the forward still reads that row, so the weight gradients include it).  Where y lies within TAU of 0, G is set to 0: a ReLU
that opens on one side of the comparison and closes on the other would move a whole gradient term.

Tolerances (max-abs error over max-abs reference): 3e-5 for the table, weight and bias gradients in both precisions.
K2c's arithmetic is fp32-grade against the rounded operands: the coefficient sums are fp32 atomics, C = hi + lo holds them to
2^-17, and both GEMMs multiply bf16-exact operands into fp32 accumulators.
"""
import collections
import json
import types

import pytest
import torch

import rbr_b200
from conftest import rel_err
from oracle import rbr_oracle as orc
from rbr_b200 import ops, synth
from rbr_b200._lib import lib

pytestmark = pytest.mark.gpu
GRAD_TOL = 3e-5
TAU = 2e-5                                    # ReLU margin on the float64 pre-activation
OBSERVED = collections.defaultdict(float)     # (precision, gradient) -> largest relative error seen


@pytest.fixture(autouse=True)
def _release_cmat_workspaces():
    """The K2c workspace cache keeps up to eight workspaces alive; the 16-block case alone takes 5.7 GB."""
    yield
    ops._CMAT_WS.clear()
    torch.cuda.empty_cache()


@pytest.fixture(scope="module", autouse=True)
def _report_observed():
    yield
    print("\nlargest relative gradient errors:", {k: f"{v:.2e}" for k, v in sorted(OBSERVED.items())})


def _note(prec, what, err):
    OBSERVED[(prec, what)] = max(OBSERVED[(prec, what)], err)
    return err


_DEFAULTS = dict(V=3000, E=64, H=40, ks=(3,), n=24, L=100, ids="i64", mask="bytes", prec="bf16", sparse=False,
                 act=ops.ACT_RELU, pidx=0, live=(0, 1), oob=False, hot=False, freeze=False,
                 scatter="fast", splits=1, k2b=None, exact=(), sparse_convs=None, repeat=False)


def C(**kw):
    """One case.  scatter: 'fast' / 'generic' / None (no K2c conv); splits: cmat_split_kernel launches (filter blocks summed over
    the K2c convs); k2b: (weight kernel, table kernel) name prefixes of the K2b conv, or None; exact: indices of convs whose
    backward multiplies the fp32 operands in bf16 mode (K2b's scalar kernels); sparse_convs: indices of the convs K2b runs when
    some run K2c (default: all or none, from `scatter`); repeat: a second step on the same workspace (each
    coefficient block is zero-filled before its scatter) must agree with the first within 1e-6 (fp32 atomics: not bitwise)."""
    d = dict(_DEFAULTS)
    d.update(kw)
    return types.SimpleNamespace(**d)


def _k2b(K, E, bf16=False):
    """Name prefixes of the K2b kernels a (K, E) conv runs."""
    if E % 4 == 0 and E <= 512 and K in (1, 2, 3, 4, 5, 7):
        nq = (E // 4 + 31) // 32
        return (f"conv_bwd_weight_kernel<{7 if K not in (1, 2, 3, 4, 5) else K},{nq},", f"conv_bwd_table_kernel<{nq},")
    return ("conv_bwd_weight_scalar_kernel", "conv_bwd_table_scalar_kernel")


CASES = {
    # ---- K2c: filter blocks
    "k2c_1blk_fast_deepconn_dims": C(V=3000, E=300, H=100, n=24, L=500),
    "k2c_2blk_76+74_narre_dims_i32_maskids": C(V=60000, E=300, H=150, n=600, L=60, ids="i32", mask="ids", splits=2,
                                                  repeat=True),
    "k2c_3blk_52/52/46_last_holds_62_zero_cols_nomask": C(V=100000, E=100, H=150, n=64, L=100, mask="none", pidx=None, splits=3,
                                                              repeat=True),
    "k2c_16blk_cap_hjp2048_generic_k4": C(V=350000, E=64, H=512, ks=(4,), n=64, L=200, scatter="generic", splits=16),
    # (the forward takes k in {1, 2, 3, 4, 5, 7} only: k = 4 stands in for k = 8, H k = 36 -> 64 columns as with k = 8's 72 -> 128)
    "k2c_2blk_8+1_filters_generic_k4": C(V=400000, E=64, H=9, ks=(4,), n=64, L=100, scatter="generic", splits=2),
    "k2c_hjp4096_splitk2_generic_k4": C(V=2000, E=32, H=1024, ks=(4,), n=16, L=60, scatter="generic"),
    # ---- K2c: generic scatter at every k it takes that the forward also takes
    **{f"k2c_generic_k{k}": C(V=500, E=32, H=24, ks=(k,), n=20, L=50, scatter="generic", oob=True) for k in (2, 4, 7)},
    # ---- K2c: activation, padding rows, table-GEMM edges (vocabulary not a multiple of 128, N tiles of 16..160 columns)
    "k2c_tanh": C(E=100, act=ops.ACT_TANH),
    **{f"k2c_padding_idx_{p}": C(V=500, pidx=p) for p in (None, 0, 7, 499)},
    **{f"k2c_table_gemm_V{V}_E{E}": C(V=V, E=E, H=24, n=8, L=40, mask="none" if V == 1 else "bytes", pidx=None if V == 1 else 0)
       for V, E in ((1, 4), (127, 16), (128, 100), (129, 128), (1000, 132), (1000, 164), (129, 300), (1000, 448), (5000, 4))},
    # ---- several convs: both dense; dense + sparse in one call (H = 820: k = 3 gives 2496 coefficient columns, k = 5 would
    # need 4160 > 4096, so K2c declines the second conv)
    "k2c_two_dense_convs_3_5": C(V=2000, E=100, H=32, ks=(3, 5), splits=2),
    "k2c+k2b_mixed_3_5_H820": C(V=2000, E=100, H=820, ks=(3, 5), n=8, L=60, k2b=_k2b(5, 100), sparse_convs=(1,)),
    # ---- frozen table over two blocks; a side the loss does not use
    "k2c_2blk_frozen_table": C(V=60000, E=300, H=150, n=100, L=60, freeze=True, splits=2),
    "k2c_2blk_one_live_side": C(V=60000, E=300, H=150, n=100, L=60, live=(1,), splits=2),
    # ---- bf16 shapes K2c declines (the weight GEMM's ring would need 240 KB of shared memory): K2b in bf16
    "k2b_bf16_E452": C(V=2000, E=452, H=64, scatter=None, splits=0, k2b=_k2b(3, 452)),
    "k2b_bf16_E512": C(V=2000, E=512, H=64, scatter=None, splits=0, k2b=_k2b(3, 512)),
    # ---- K2b, fp32: the weight kernel per K, the table kernel per nq, the scalar kernels, a hot token over a large vocabulary
    **{f"k2b_fp32_K{k}": C(ks=(k,), prec="fp32", scatter=None, splits=0, k2b=_k2b(k, 64), oob=True) for k in (1, 2, 3, 4, 5, 7)},
    **{f"k2b_fp32_E{E}": C(E=E, prec="fp32", scatter=None, splits=0, k2b=_k2b(3, E)) for E in (4, 128, 132, 260, 388, 512)},
    # (the scalar kernels' other trigger, k not in {1, 2, 3, 4, 5, 7}, is a shape the forward rejects)
    **{f"k2b_fp32_scalar_E{E}": C(E=E, prec="fp32", scatter=None, splits=0, k2b=_k2b(3, E), oob=E == 30) for E in (30, 301, 520)},
    "k2b_fp32_hot_token_V350000": C(V=350000, n=64, L=200, prec="fp32", hot=True, scatter=None, splits=0, k2b=_k2b(3, 64)),
    # ---- K2b in bf16 (CONV_BWD_SPARSE)
    **{f"k2b_bf16_sparse_K{k}": C(ks=(k,), sparse=True, scatter=None, splits=0, k2b=_k2b(k, 64)) for k in (1, 2, 5, 7)},
    **{f"k2b_bf16_sparse_E{E}": C(E=E, sparse=True, scatter=None, splits=0, k2b=_k2b(3, E)) for E in (132, 388)},
    "k2b_bf16_sparse_scalar_E30": C(E=30, sparse=True, scatter=None, splits=0, k2b=_k2b(3, 30), exact=(0,)),
    "k2b_bf16_sparse_hot_token_V350000": C(V=350000, n=64, L=200, sparse=True, hot=True, scatter=None, splits=0, k2b=_k2b(3, 64)),
}
# the fast scatter, every instance: k x id width x mask mode (out-of-range ids in every width: negative and >= V, or >= V for uint16)
FAST = {f"k2c_fast_k{k}_{i}_{m}": C(V=3000, E=64, H=40, ks=(k,), n=30, L=80, ids=i, mask=m, oob=True, pidx=0 if m != "none" else None)
        for k in (1, 3, 5) for i in ("i64", "i32", "u16") for m in ("bytes", "ids", "none")}
_WIDTH = {"i64": 0, "i32": 1, "u16": 2}
_MM = {"none": 0, "bytes": 1, "ids": 2}


def _sparse_convs(c):
    """Indices of the convs K2b runs."""
    if c.sparse_convs is not None:
        return c.sparse_convs
    return tuple(range(len(c.ks))) if c.scatter is None else ()


def _round(t):
    return t.to(torch.bfloat16).to(torch.float32)


def _inputs(c, seed):
    gen = torch.Generator().manual_seed(seed)
    table = torch.randn(c.V, c.E, generator=gen) * 0.5          # the padding row is NOT zero: it must still come out 0
    ws = [(torch.rand(c.H, c.E, k, generator=gen) * 2 - 1) / (c.E * k) ** 0.5 for k in c.ks]
    bs = [(torch.rand(c.H, generator=gen) * 2 - 1) * 0.1 for _ in c.ks]
    sides = []
    for s in range(2):
        ids = torch.randint(0 if c.mask == "none" else min(1, c.V - 1), c.V, (c.n, c.L), generator=gen)
        if c.hot:
            ids[torch.rand(c.n, c.L, generator=gen) < 0.5] = 1 + s
        if c.pidx not in (None, 0):
            ids[torch.rand(c.n, c.L, generator=gen) < 0.05] = c.pidx    # padding tokens the forward reads
        mask = None
        if c.mask != "none":
            lens = torch.randint(0, c.L + 1, (c.n,), generator=gen)
            lens[0] = c.L
            valid = torch.arange(c.L).unsqueeze(0) < lens.unsqueeze(1)
            ids = ids * valid                                               # id 0 in the tail
            if c.mask == "bytes":
                mask = valid & (torch.rand(c.n, c.L, generator=gen) > 0.05)  # holes: a mask that is not ids != 0
        if c.oob:
            # negative (not for uint16) and in [V, 2V + 40): a scatter that let such an id through would add into rows past the
            # coefficient block, which in the fast-scatter shapes are the workspace's bf16 operand and weight scratch, so the
            # weight gradient shows it
            pos = torch.rand(c.n, c.L, generator=gen) < 0.04
            big = torch.randint(c.V, 2 * c.V + 40, (c.n, c.L), generator=gen)
            neg = torch.randint(-100, 0, (c.n, c.L), generator=gen)
            use_neg = (torch.rand(c.n, c.L, generator=gen) < 0.5) & (c.ids != "u16")
            ids = torch.where(pos, torch.where(use_neg, neg, big), ids)
        sides.append((ids, mask))
    G = [torch.randn(c.n, c.H * len(c.ks), generator=gen) for _ in range(2)]
    return table, ws, bs, sides, G


def _dev_ids(ids, width):
    return {"i64": ids, "i32": ids.int(), "u16": ids.to(torch.uint16)}[width].cuda()


def _x(tab, ids, mask):
    """Embedded documents: out-of-range ids read as zero rows, masked positions are zero."""
    V = tab.shape[0]
    ok = (ids >= 0) & (ids < V)
    if mask is not None:
        ok = ok & mask
    return tab[ids.clamp(0, V - 1)] * ok.unsqueeze(-1).to(tab.dtype)


def _act(act, y):
    return torch.relu(y) if act == ops.ACT_RELU else torch.tanh(y)


def _forward_point(c, table, ws, bs, sides, feats, ams):
    """Per side: (keep, act') [n, H_total] at the kernel's arg-max, from the float64 pre-activation on the operands the forward
    multiplied.  Checks the routing (the kernel's arg-max attains the oracle's max) and the pooled values on the way.  In bf16
    mode the forward ran on the tensor cores (rounded operands) unless the shape is outside them (then the fp32 kernel ran)."""
    variants = [("r", _round)] if c.prec == "bf16" else []
    variants.append(("f", lambda t: t))
    out = []
    for s, (ids, mask) in enumerate(sides):
        keep_s, d_s, col = [], [], 0
        for i, (w, b) in enumerate(zip(ws, bs)):
            k, h = w.shape[2], w.shape[0]
            am = ams[s][:, col:col + h].long()
            fk = feats[s][:, col:col + h].double()
            best = None
            for tag, rnd in variants:
                x = _x(rnd(table).cuda().double(), ids, mask)
                y = orc.conv1d_valid(x, rnd(w).cuda().double(), b.cuda().double(), (k - 1) // 2)
                pre = torch.gather(y, 1, am.unsqueeze(1)).squeeze(1)
                err = rel_err(fk, _act(c.act, pre))
                if best is None or err < best[0]:
                    best = (err, y, pre)
            err, y, pre = best
            assert err < 1e-5, ("pooled values", i, err)
            ya = _act(c.act, y)
            top, got = ya.max(dim=1).values, _act(c.act, pre)
            assert float(((top - got).abs() / top.abs().clamp_min(1e-3)).max()) < 1e-5, ("routing", i)
            if c.act == ops.ACT_RELU:
                keep_s.append((pre.abs() >= TAU).double())
                d_s.append((pre > 0).double())
            else:
                keep_s.append(torch.ones_like(pre))
                d_s.append(1 - torch.tanh(pre) ** 2)
            col += h
        out.append((torch.cat(keep_s, 1), torch.cat(d_s, 1)))
    return out


def _reference_grads(c, table, ws, bs, sides, ams, point, G):
    """float64 gradients of sum_s sum(G_s * act'(y) * y at the arg-max) over the backward's operands."""
    bf16 = c.prec == "bf16"
    tabs = {"r": _round(table).cuda().double().requires_grad_(), "f": table.cuda().double().requires_grad_()}
    w64 = [(_round(w) if bf16 and i not in c.exact else w).cuda().double().requires_grad_() for i, w in enumerate(ws)]
    b64 = [b.cuda().double().requires_grad_() for b in bs]
    loss = 0
    for s in c.live:
        ids, mask = sides[s]
        keep, d = point[s]
        col = 0
        for i, (w, b) in enumerate(zip(w64, b64)):
            k, h = w.shape[2], w.shape[0]
            tab = tabs["r" if bf16 and i not in c.exact else "f"]
            y = orc.conv1d_valid(_x(tab, ids, mask), w, b, (k - 1) // 2)
            pre = torch.gather(y, 1, ams[s][:, col:col + h].long().unsqueeze(1)).squeeze(1)
            loss = loss + (G[s].cuda().double()[:, col:col + h] * keep[:, col:col + h] * d[:, col:col + h] * pre).sum()
            col += h
    loss.backward()
    gt = sum(t.grad for t in tabs.values() if t.grad is not None)
    if c.pidx is not None:
        gt[c.pidx] = 0
    return gt, [w.grad for w in w64], [b.grad for b in b64]


def _launches(fn, tmp_path):
    """[(kernel name without spaces, grid x)] of every CUDA kernel `fn` launches, from a torch.profiler trace."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    events = json.loads(path.read_text())["traceEvents"]
    return [(e["name"].replace(" ", ""), e["args"]["grid"][0]) for e in events if e.get("cat") == "kernel"]


def _cfg(c, tab, wl, bl, shadow, packed, hook=None):
    """What NgramFeat.encode passes, with the case's activation, id / mask handling and padding row."""
    return {"n_conv": len(c.ks), "precision": c.prec, "act": c.act, "pads": [(k - 1) // 2 for k in c.ks],
            "shadow_fn": lambda: shadow, "pack_fn": lambda i: packed[i], "arena": None, "table_param": tab,
            "weight_params": wl, "bias_params": bl, "padding_idx": -1 if c.pidx is None else c.pidx, "table_ready": hook,
            "flags": ops.CONV_BWD_SPARSE if c.sparse else 0, "mask_from_ids": c.mask == "ids"}


def _check_case(c, seed, tmp_path):
    table, ws, bs, sides, G = _inputs(c, seed)
    sides_dev = [(ids.cuda(), None if m is None else m.cuda()) for ids, m in sides]
    ref_sides = [(ids, (ids != 0) if c.mask == "ids" else m) for ids, m in sides_dev]
    tab = table.cuda().requires_grad_(not c.freeze)
    wl = [w.cuda().requires_grad_() for w in ws]
    bl = [b.cuda().requires_grad_() for b in bs]
    shadow = ops.table_to_bf16(tab.detach()) if c.prec == "bf16" else None
    packed = [ops.conv_pack(w.detach()) for w in wl]
    flat = []
    for ids, m in sides_dev:
        flat += [_dev_ids(ids, c.ids), None if m is None else m]
    state = {}

    def step():
        outs = ops.EncodeDocsFn.apply(tab, _cfg(c, tab, wl, bl, shadow, packed), *wl, *bl, *flat)
        feats, ams = outs[:2], outs[2:]
        lib.rbr_consume_oob_count(None)                   # out-of-range ids were counted: leave the counter clean
        point = _forward_point(c, table, ws, bs, ref_sides, feats, ams)
        Gk = [(G[s].cuda().double() * point[s][0]).float() for s in range(2)]
        sum((feats[s] * Gk[s]).sum() for s in c.live).backward()
        state.update(ams=ams, point=point, G=Gk)

    launched = _launches(step, tmp_path)
    # ---- routing
    live = len(c.live)
    dense_ks = [k for i, k in enumerate(c.ks) if i not in _sparse_convs(c)]
    if c.scatter == "fast":
        for k in set(dense_ks):
            name = f"cmat_scatter_fast_kernel<{k},2,{_WIDTH[c.ids]},{_MM[c.mask]}>"
            per_conv = c.splits // len(dense_ks)
            assert sum(name in n for n, _ in launched) == per_conv * dense_ks.count(k) * live, (name, launched)
    fast = sum("cmat_scatter_fast_kernel<" in n for n, _ in launched)
    generic = sum("cmat_scatter_kernel<" in n for n, _ in launched)
    assert (fast, generic) == ((c.splits * live, 0) if c.scatter == "fast" else
                               (0, c.splits * live) if c.scatter == "generic" else (0, 0)), (fast, generic)
    assert sum("cmat_split_kernel" in n for n, _ in launched) == c.splits
    gemm = [g for n, g in launched if "cmat_table_gemm_kernel" in n]
    assert gemm == ([] if c.freeze or not c.splits else [(c.V + 127) // 128] * len(dense_ks)), gemm
    if c.k2b:
        wk, tk = c.k2b
        assert sum(wk in n for n, _ in launched) == live, (wk, launched)
        assert sum(tk in n for n, _ in launched) == (0 if c.freeze else live), (tk, launched)
    else:
        assert not any("conv_bwd_" in n for n, _ in launched), launched
    # ---- gradients
    gt, gw, gb = _reference_grads(c, table, ws, bs, ref_sides, state["ams"], state["point"], state["G"])
    if c.freeze:
        assert tab.grad is None
    else:
        assert _note(c.prec, "table", rel_err(tab.grad, gt)) < GRAD_TOL
        if c.pidx is not None:
            assert float(tab.grad[c.pidx].abs().max()) == 0.0
    for i in range(len(c.ks)):
        assert _note(c.prec, "weight", rel_err(wl[i].grad, gw[i])) < GRAD_TOL, i
        assert _note(c.prec, "bias", rel_err(bl[i].grad, gb[i])) < GRAD_TOL, i
    if c.repeat:
        first = [t.grad.clone() for t in [tab] + wl + bl]
        for t in [tab] + wl + bl:
            t.grad = None
        step()
        for a, b in zip([tab] + wl + bl, first):
            assert rel_err(a.grad, b, 1e-9) < 1e-6


@pytest.mark.parametrize("name", list(CASES))
def test_conv_backward_variant_vs_float64(name, tmp_path):
    _check_case(CASES[name], seed=sum(map(ord, name)), tmp_path=tmp_path)


@pytest.mark.parametrize("name", list(FAST))
def test_fast_scatter_instance_vs_float64(name, tmp_path):
    _check_case(FAST[name], seed=sum(map(ord, name)), tmp_path=tmp_path)


def test_wide_embedding_bf16_model_trains():
    """E in (448, 512]: K2c declines these shapes (its weight GEMM would need more shared memory than a CTA may have), so a bf16
    DeepCoNN step runs K2b and does not leave the table slot of the gradient arena unwritten."""
    for E in (452, 512):
        model = rbr_b200.DeepCoNNpp(7, 6, 2000, [3], E, 64, 8, 50, None, 0.0, precision="bf16").cuda().train()
        batch, ratings = synth.deepconn_batch(8, 50, 2000, 7, 6, seed=E)
        torch.nn.MSELoss()(model(*[t.cuda() for t in batch]), ratings.cuda()).backward()
        g = model.word_embeddings.embedding.weight.grad
        assert bool(torch.isfinite(g).all()) and float(g.abs().max()) > 0 and float(g[0].abs().max()) == 0.0
        assert lib.rbr_conv_bwd_cmat_supported(2000, E, 64, 3) == 0


# ----------------------------------------------------------------------------------------------------------------------
# the gradient arena: overwrite mode (the table slot is not zero-filled), a repeated step
# ----------------------------------------------------------------------------------------------------------------------
ARENA_CASES = {"overwrite": (3,), "two_convs_zero_filled": (3, 5)}


@pytest.mark.parametrize("name", list(ARENA_CASES))
def test_arena_table_gradient(name, tmp_path):
    """DeepCoNN bf16 with a persistent arena buffer filled with NaN before each step.  With one conv the table slot is not
    zero-filled (K2c overwrites every element), with two it is.  The table-gradient hook sees the whole gradient once per step.
    A second step on the same model (the coefficient blocks re-zeroed before their atomics) gives the same gradients."""
    ks = ARENA_CASES[name]
    V, E, H, L, n = 5000, 100, 40, 80, 16
    params = synth.deepconn_params(7, 6, V, E, H, 8, ks, seed=3)
    batch, ratings = synth.deepconn_batch(n, L, V, 7, 6, seed=4)
    model = rbr_b200.DeepCoNNpp(7, 6, V, list(ks), E, H, 8, L, None, 0.0, precision="bf16")
    model.load_state_dict(params)
    model.cuda().train()
    layout = ops.GradArena.for_module(model)
    buf = torch.empty(layout.total + 1024, device="cuda")
    model.__dict__["_rbr_arena_buffer"] = buf
    convs = list(model.ngram.conv.list_of_conv1d)
    c = C(V=V, E=E, H=H, ks=ks, n=n, L=L)
    table = model.word_embeddings.embedding.weight
    ws, bs = [cv.weight.detach().cpu() for cv in convs], [cv.bias.detach().cpu() for cv in convs]
    ref_sides = [(batch[0].cuda(), batch[2].cuda()), (batch[1].cuda(), batch[3].cuda())]
    cap = {}
    encode = model.ngram.encode

    def encode_capturing(we, sides, masks, return_argmax=False):
        outs = encode(we, sides, masks, return_argmax=True)
        feats, ams = outs[:2], outs[2:]
        point = _forward_point(c, table.detach().cpu(), ws, bs, ref_sides, feats, ams)
        cap.update(ams=ams, point=point, G=[None, None])
        for s, f in enumerate(feats):
            def keep(g, s=s):
                g = g * point[s][0].float()                       # the ReLU margin, applied to what the backward receives
                cap["G"][s] = g.detach().clone()
                return g
            f.register_hook(keep)
        return list(outs) if return_argmax else list(feats)

    model.ngram.encode = encode_capturing
    hooked = []

    def hook(g):
        hooked.append(g.detach().clone())

    model.ngram.table_grad_hook = hook
    results = []
    for rep in range(2):
        buf.fill_(float("nan"))
        hooked.clear()
        model.zero_grad(set_to_none=True)

        def step():
            torch.nn.MSELoss()(model(*[t.cuda() for t in batch]), ratings.cuda()).backward()

        launched = _launches(step, tmp_path)
        g = table.grad
        assert bool(torch.isfinite(g).all()) and float(g[0].abs().max()) == 0.0
        gemm = [gx for nm, gx in launched if "cmat_table_gemm_kernel" in nm]
        assert gemm == [(V + 127) // 128] * len(ks), gemm
        gt, gw, gb = _reference_grads(c, table.detach().cpu(), ws, bs, ref_sides, cap["ams"], cap["point"], cap["G"])
        assert _note("bf16", "table", rel_err(g, gt)) < GRAD_TOL
        for i, cv in enumerate(convs):
            assert _note("bf16", "weight", rel_err(cv.weight.grad, gw[i])) < GRAD_TOL, i
            assert _note("bf16", "bias", rel_err(cv.bias.grad, gb[i])) < GRAD_TOL, i
        assert len(hooked) == 1
        results.append({k: p.grad.detach().clone() for k, p in model.named_parameters()})
    for k in results[0]:
        assert rel_err(results[1][k], results[0][k], 1e-9) < 1e-6, k
