"""D-ATT's gate kernels (K5, csrc/datt.cu) and its gated encoder, every variant against float64, at the shapes that select it.

K5 has three templated kernels, each with 8 instances (window WIN in {1, 3, 5, 7} x V4 = E % 4 == 0):
  datt_gate_fwd_kernel<V4, WIN>     both gates, one CTA per document
  datt_gate_wgrad_kernel<WIN, V4>   the two attention-weight gradients, one CTA per position, 256 documents per iteration
  datt_gate_table_kernel<WIN, V4>   the table gradient, warp-segmented over token-sorted positions
plus datt_gate_dz_kernel, whose grid is capped at 1184 blocks: its grid-stride loop runs past 303 104 tokens.

The K5 tests call ops.datt_gates and rbr_datt_gate_bwd directly and compare with float64 autograd of sigmoid(conv) for both
gates: gates to 1e-5 absolute, gradients to 3e-5 relative (max-abs error over max-abs reference).  The gradient buffers are
pre-filled: the call adds into them.

The encoder tests run DattEncodeFn forward and backward (K5 + the four gated convs of K2 + K2b's gated backward) for both sides,
against float64 gradients linearised at the kernel's arg-max, as test_gpu_conv_bwd_variants.py does.  The conv's operands are
the ones each kernel multiplies: in bf16 the rounded table and weights (the forward on the tensor cores; K2b's vector kernels
read the bf16 shadow and the rounded weights), in fp32 and in K2b's scalar kernels (E % 4 != 0) the fp32 ones.  The gates are
the kernel's fp32 values, with float64 gradients of sigmoid(conv) on the fp32 table flowing through them.  Where a column's
maximum is an exact tie in float64 (a gate of exactly 0 makes every candidate 0), the reference is linearised at torch's
first arg-max instead: the tensor-core kernels may report another position there (DESIGN §3), and the gradients must not
depend on it.
"""
import json

import pytest
import torch

from conftest import rel_err
from oracle import rbr_oracle as orc
from rbr_b200 import ops
from rbr_b200._lib import lib

pytestmark = pytest.mark.gpu
GATE_TOL = 1e-5
GRAD_TOL = 3e-5                                     # FP32_GRAD_TOL


def _kernels_launched(fn, tmp_path):
    """[kernel name without spaces] of every CUDA kernel `fn` launches, from a torch.profiler trace."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    events = json.loads(path.read_text())["traceEvents"]
    return out, [e["name"].replace(" ", "") for e in events if e.get("cat") == "kernel"]


def _round(t):
    return t.to(torch.bfloat16).to(torch.float32)


def _dev_ids(ids, width):
    return {"i64": ids, "i32": ids.int(), "u16": ids.to(torch.uint16)}[width].cuda()


def _x(tab, ids):
    """Embedded documents: out-of-range ids read as zero rows (the gates read every other token, padding included)."""
    V = tab.shape[0]
    ok = (ids >= 0) & (ids < V)
    return tab[ids.clamp(0, V - 1)] * ok.unsqueeze(-1).to(tab.dtype)


def _gates64(table64, ids, la_w, la_b, ga_w, ga_b):
    """float64 sigmoid(conv) of both gates: local [n, L], global [n]."""
    x = _x(table64, ids)
    win = la_w.shape[2]
    zl = orc.conv1d_valid(x, la_w, la_b, (win - 1) // 2)[..., 0]
    zg = torch.einsum("nle,el->n", x, ga_w[0]) + ga_b
    return torch.sigmoid(zl), torch.sigmoid(zg)


# ----------------------------------------------------------------------------------------------------------------------
# K5 forward and backward, called directly
# ----------------------------------------------------------------------------------------------------------------------
def _k5_case(win, E, L, n, ids_w="i64", pidx=0, oob=False, hot=False, V=300, seed=0):
    return dict(win=win, E=E, L=L, n=n, ids_w=ids_w, pidx=pidx, oob=oob, hot=hot, V=V, seed=seed)


_IDW = ("i64", "i32", "u16")
K5 = {}
for i, (win, E) in enumerate([(w, e) for w in (1, 3, 5, 7) for e in (3, 4, 30, 100, 126, 128)]):
    L, n = ((7, 31), (60, 257), (1, 31), (33, 1))[i % 4]
    K5[f"win{win}_E{E}_L{L}_n{n}"] = _k5_case(win, E, L, n, ids_w=_IDW[i % 3], pidx=(None, 0, 7)[i % 3], oob=i % 2 == 0,
                                              hot=i % 5 == 0, seed=i)
K5.update({
    "win5_E100_L500_n700_dz_grid_stride": _k5_case(5, 100, 500, 700, ids_w="i32", pidx=0, oob=True, V=3000),
    "win7_E128_L7185_smem_limit": _k5_case(7, 128, 7185, 2, pidx=7, V=500),
    "win3_E30_L500_n257_hot": _k5_case(3, 30, 500, 257, ids_w="u16", pidx=7, oob=True, hot=True),
    "win1_E100_L500_n31_hot": _k5_case(1, 100, 500, 31, pidx=None, hot=True),
})


def _k5_inputs(c):
    g = torch.Generator().manual_seed(1000 + c["seed"])
    V, E, L, n, win = c["V"], c["E"], c["L"], c["n"], c["win"]
    table = torch.randn(V, E, generator=g)
    la_w = (torch.rand(1, E, win, generator=g) * 2 - 1) / (E * win) ** 0.5 * 3
    la_b = torch.rand(1, generator=g) - 0.5
    ga_w = (torch.rand(1, E, L, generator=g) * 2 - 1) / (E * L) ** 0.5 * 3
    ga_b = torch.rand(1, generator=g) - 0.5
    ids = torch.randint(0, V, (n, L), generator=g)
    if c["hot"]:
        ids[torch.rand(n, L, generator=g) < 0.6] = 1                # segments far past a warp's 32 entries
    if c["pidx"] not in (None, 0):
        ids[torch.rand(n, L, generator=g) < 0.05] = c["pidx"]
    oob = torch.zeros(n, L, dtype=torch.bool)
    if c["oob"]:
        oob = torch.rand(n, L, generator=g) < 0.04
        big = torch.randint(V, 2 * V + 40, (n, L), generator=g)
        neg = torch.randint(-100, 0, (n, L), generator=g)
        use_neg = (torch.rand(n, L, generator=g) < 0.5) & (c["ids_w"] != "u16")
        ids = torch.where(oob, torch.where(use_neg, neg, big), ids)
    gl_grad = torch.randn(n, L, generator=g)
    gg_grad = torch.randn(n, generator=g)
    return table, la_w, la_b, ga_w, ga_b, ids, int(oob.sum()), gl_grad, gg_grad


def _k5_reference(c, table, la_w, la_b, ga_w, ga_b, ids, gl_grad, gg_grad):
    leaves = [t.cuda().double().requires_grad_() for t in (table, la_w, la_b, ga_w, ga_b)]
    gl, gg = _gates64(leaves[0], ids.cuda(), *leaves[1:])
    ((gl * gl_grad.cuda().double()).sum() + (gg * gg_grad.cuda().double()).sum()).backward()
    grads = [t.grad for t in leaves]
    if c["pidx"] is not None:
        grads[0][c["pidx"]] = 0
    return gl.detach(), gg.detach(), grads


def _k5_backward(c, table, ids_dev, la_w, ga_w, gl, gg, gl_grad, gg_grad, out):
    """rbr_datt_gate_bwd into the pre-filled buffers out = [table, la_w, la_b, ga_w, ga_b] gradients."""
    V, E = table.shape
    n, L = ids_dev.shape
    win = la_w.shape[2]
    ws_bytes = lib.rbr_datt_gate_workspace_bytes(n, L, E, win, V)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    pidx = -1 if c["pidx"] is None else c["pidx"]
    p = ops._p
    lib.check(lib.rbr_datt_gate_bwd(p(table), V, E, p(ids_dev), n, L, p(la_w), win, p(ga_w), p(gl), p(gg), p(gl_grad),
                                    p(gg_grad), pidx, p(out[1]), p(out[2]), p(out[3]), p(out[4]), p(out[0]), p(ws), ws_bytes,
                                    ops._id_width_flag(ids_dev), ops._stream(True)), "rbr_datt_gate_bwd")


def k5_instances(win, E):
    v4 = "true" if E % 4 == 0 else "false"
    return (f"datt_gate_fwd_kernel<{v4},{win}>(", f"datt_gate_wgrad_kernel<{win},{v4}>(",
            f"datt_gate_table_kernel<{win},{v4}>(")


@pytest.mark.parametrize("name", list(K5))
def test_k5_gates_and_gradients_vs_float64(name, tmp_path):
    c = K5[name]
    table, la_w, la_b, ga_w, ga_b, ids, n_oob, gl_grad, gg_grad = _k5_inputs(c)
    ref_gl, ref_gg, ref = _k5_reference(c, table, la_w, la_b, ga_w, ga_b, ids, gl_grad, gg_grad)
    dev = [t.cuda() for t in (table, la_w, la_b, ga_w, ga_b)]
    ids_dev = _dev_ids(ids, c["ids_w"])
    gen = torch.Generator(device="cuda").manual_seed(5)
    # the table gradient already holds the gated convs' part: the call must add to every buffer, not overwrite it
    pre = [torch.randn(r.shape, device="cuda", generator=gen, dtype=torch.float32) * float(r.abs().max()) for r in ref]
    out = [t.clone() for t in pre]
    lib.rbr_consume_oob_count(None)

    def both():
        gl, gg = ops.datt_gates(dev[0], ids_dev, *dev[1:])
        _k5_backward(c, dev[0], ids_dev, dev[1], dev[3], gl, gg, gl_grad.cuda(), gg_grad.cuda(), out)
        return gl, gg

    (gl, gg), names = _kernels_launched(both, tmp_path)
    for inst in k5_instances(c["win"], c["E"]):
        assert sum(inst in nm for nm in names) == 1, (inst, names)
    if c["n"] * c["L"] > 303104:
        assert any("datt_gate_dz_kernel" in nm for nm in names)
    counted = lib.rbr_consume_oob_count(None)
    assert counted >= n_oob and (counted > 0) == (n_oob > 0), (counted, n_oob)
    assert float((gl.double() - ref_gl).abs().max()) < GATE_TOL
    assert float((gg.double() - ref_gg).abs().max()) < GATE_TOL
    for what, got, p, r in zip(("table", "w_local", "b_local", "w_global", "b_global"), out, pre, ref):
        assert rel_err(got.double() - p.double(), r) < GRAD_TOL, (what, rel_err(got.double() - p.double(), r))
    if c["pidx"] is not None:
        assert torch.equal(out[0][c["pidx"]], pre[0][c["pidx"]])


def test_k5_declines_cleanly(tmp_path):
    """doc_len one past the gate forward's shared-memory limit (window 7, E = 128: 7186 positions) raises, and enqueues
    nothing: the workspace and the outputs are untouched."""
    V, E, win = 50, 128, 7
    for L, ok in ((7185, True), (7186, False)):
        table = torch.randn(V, E, device="cuda")
        la_w, la_b = torch.randn(1, E, win, device="cuda"), torch.zeros(1, device="cuda")
        ga_w, ga_b = torch.randn(1, E, L, device="cuda") * 0.01, torch.zeros(1, device="cuda")
        ids = torch.randint(0, V, (2, L), device="cuda")
        ws_bytes = lib.rbr_datt_gate_workspace_bytes(2, L, E, win, V)
        ws = torch.full((ws_bytes,), 0xAB, dtype=torch.uint8, device="cuda")
        gl = torch.full((2, L), -1.0, device="cuda")
        gg = torch.full((2,), -1.0, device="cuda")
        p = ops._p

        def call():
            return lib.rbr_datt_gate_fwd(p(table), V, E, p(ids), 2, L, p(la_w), p(la_b), win, p(ga_w), p(ga_b), p(gl), p(gg),
                                         p(ws), ws_bytes, 0, ops._stream(True))

        rc, names = _kernels_launched(call, tmp_path)
        if ok:
            assert rc == 0 and any("datt_gate_fwd_kernel<true,7>" in nm for nm in names)
        else:
            assert rc == -4 and b"shared memory" in lib.rbr_last_error()
            assert names == [], names
            assert bool((ws == 0xAB).all()) and bool((gl == -1).all()) and bool((gg == -1).all())


def test_routing_every_k5_instance_launched(tmp_path):
    def calls():
        for win in (1, 3, 5, 7):
            for E in (30, 100):
                c = _k5_case(win, E, 20, 3)
                table, la_w, la_b, ga_w, ga_b, ids, _, gl_grad, gg_grad = _k5_inputs(c)
                dev = [t.cuda() for t in (table, la_w, la_b, ga_w, ga_b)]
                gl, gg = ops.datt_gates(dev[0], ids.cuda(), *dev[1:])
                out = [torch.zeros_like(t) for t in dev]
                _k5_backward(c, dev[0], ids.cuda(), dev[1], dev[3], gl, gg, gl_grad.cuda(), gg_grad.cuda(), out)

    _, names = _kernels_launched(calls, tmp_path)
    for win in (1, 3, 5, 7):
        for E in (30, 100):
            for inst in k5_instances(win, E):
                assert any(inst in nm for nm in names), (inst, sorted(set(names)))


# ----------------------------------------------------------------------------------------------------------------------
# the whole encoder: DattEncodeFn forward + backward, both sides, gated K2 + K2b + K5
# ----------------------------------------------------------------------------------------------------------------------
def _enc(**kw):
    d = dict(V=600, E=100, lw=5, lo=40, go=24, L=500, n=6, prec="bf16", flags=0, sat=None, pidx=0, seed=0)
    d.update(kw)
    return d


ENC = {}
for prec in ("fp32", "bf16"):
    ENC.update({
        f"{prec}_defaults_E100_lw5_L500": _enc(prec=prec),
        f"{prec}_L60_packed": _enc(prec=prec, L=60, n=70),
        f"{prec}_win1": _enc(prec=prec, lw=1, L=120),
        f"{prec}_win7": _enc(prec=prec, lw=7, L=120),
        f"{prec}_E30": _enc(prec=prec, E=30, L=120),
        f"{prec}_E128": _enc(prec=prec, E=128, L=120),
        f"{prec}_n300_docs": _enc(prec=prec, L=40, n=300, pidx=7),
        f"{prec}_global_gate_0": _enc(prec=prec, L=60, n=12, sat="global"),
        f"{prec}_local_gates_0_win1": _enc(prec=prec, lw=1, L=60, n=12, sat="local"),
    })
ENC.update({
    "bf16_single_cta_L60": _enc(L=60, n=70, flags=ops.CONV_TC_SINGLE_CTA),
    "bf16_pair_only_L60": _enc(L=60, n=70, flags=ops.CONV_TC_PAIR_ONLY),
    "bf16_single_cta_L500": _enc(flags=ops.CONV_TC_SINGLE_CTA),
    "bf16_pair_only_global_gate_0": _enc(L=60, n=12, sat="global", flags=ops.CONV_TC_PAIR_ONLY),
    "bf16_single_cta_local_gates_0": _enc(lw=1, L=60, n=12, sat="local", flags=ops.CONV_TC_SINGLE_CTA),
})


def _enc_inputs(c):
    g = torch.Generator().manual_seed(77 + c["seed"] + c["L"] + c["E"])
    V, E, L, lw, lo, go, n = c["V"], c["E"], c["L"], c["lw"], c["lo"], c["go"], c["n"]

    def conv(h, k, scale=1.0):
        bound = 1.0 / (E * k) ** 0.5
        return (torch.rand(h, E, k, generator=g) * 2 - 1) * bound * scale, (torch.rand(h, generator=g) * 2 - 1) * bound

    table = torch.randn(V, E, generator=g) * 0.5
    sides, ids_all = [], []
    for s in range(2):
        la_w, la_b = conv(1, lw, 4.0)
        lc_w, lc_b = conv(lo, 1)
        ga_w, ga_b = conv(1, L, 4.0)
        if c["sat"] == "global":
            ga_b = ga_b - 200.0                                     # sigmoid(z) == 0 exactly in fp32: every position ties
        prm = [la_w, la_b, lc_w, lc_b, ga_w, ga_b]
        for k in (2, 3, 4):
            prm += list(conv(go, k))
        ids = torch.randint(0, V, (n, L), generator=g)
        if c["pidx"] not in (None, 0):
            ids[torch.rand(n, L, generator=g) < 0.05] = c["pidx"]
        sides.append(prm)
        ids_all.append(ids)
    if c["sat"] == "local":
        sides[1][0] = sides[0][0].clone()                           # one local gate weight: the rows below saturate both sides
        # tokens 1 and 2: rows with <w_local, row> = -150 (local gate exactly 0), and components orthogonal to the gate's
        # weight that give their local conv either sign; documents 0 and 1 alternate them, so every position is a +0 or -0
        for s in range(2):
            w0 = sides[s][0][0, :, 0]
            for tok, sign in ((1, 1.0), (2, -1.0)):
                v = torch.randn(E, generator=g)
                v -= (v @ w0) / (w0 @ w0) * w0
                table[tok] = -150.0 * w0 / (w0 @ w0) + sign * 0.5 * v
            ids_all[s][2:][ids_all[s][2:] <= 2] = 3                 # the other documents stay clear of them
            ids_all[s][0] = torch.tensor([1, 2] * (L // 2) + [1] * (L % 2))
            ids_all[s][1] = torch.tensor([2, 1] * (L // 2) + [2] * (L % 2))
    G = [torch.randn(n, lo + 3 * go, generator=g) for _ in range(2)]
    return table, sides, ids_all, G


def _vector_k2b(E):
    return E % 4 == 0 and E <= 512


def _exact_ties(raw):
    """[n, H] bool: the column's float64 maximum is attained at two or more positions."""
    top = raw.max(dim=1, keepdim=True).values
    return (raw == top).sum(dim=1) > 1


def _first_argmax(raw):
    T = raw.shape[1]
    pos = torch.arange(T, device=raw.device).view(1, T, 1).expand_as(raw)
    top = raw.max(dim=1, keepdim=True).values
    return torch.where(raw == top, pos, torch.full_like(pos, T)).min(dim=1).values


def _enc_reference(c, table, sides, ids_all, G, kernel_out):
    """float64 gradients [table, per side 12 parameters] of sum_s sum(G_s * feat_s) linearised at the kernel's arg-max (or
    torch's first arg-max on exact float64 ties); checks the forward on the way."""
    bf16 = c["prec"] == "bf16"
    fwd_r = _round if bf16 else (lambda t: t)
    bwd_r = _round if bf16 and _vector_k2b(c["E"]) else (lambda t: t)
    tab_f = table.cuda().double().requires_grad_()
    tab_b = bwd_r(table).cuda().double().requires_grad_()
    tab_fwd = fwd_r(table).cuda().double()
    prm64 = [[t.cuda().double().requires_grad_() for t in prm] for prm in sides]
    loss = 0
    for s in range(2):
        ids = ids_all[s].cuda()
        feat_k, amax_k, pre_k, gl_k, gg_k = kernel_out[s]
        p = prm64[s]
        gl64, gg64 = _gates64(tab_f, ids, p[0], p[1], p[4], p[5])
        assert float((gl_k.double() - gl64.detach()).abs().max()) < GATE_TOL and float((gg_k.double() - gg64.detach()).abs().max()) < GATE_TOL
        gl = gl64 + (gl_k.double() - gl64).detach()                 # the kernel's gate values, float64 gradients
        gg = gg64 + (gg_k.double() - gg64).detach()
        convs = [(p[2], p[3], gl.unsqueeze(-1))] + [(p[6 + 2 * i], p[7 + 2 * i], gg.view(-1, 1, 1)) for i in range(3)]
        col = 0
        for w, b, gate in convs:
            h, _, k = w.shape
            zero = torch.zeros(h, dtype=torch.float64, device="cuda")
            conv_f = orc.conv1d_valid(_x(tab_fwd, ids), fwd_r(w.detach().float()).double(), zero, 0)
            w_b = bwd_r(w.detach().float()).double() + (w - w.detach())   # the backward's weights, gradient to w
            conv_b = orc.conv1d_valid(_x(tab_b, ids), w_b, zero, 0)
            raw = gate.detach() * conv_f
            am_k = amax_k[:, col:col + h].long()
            ties = _exact_ties(raw)
            am = torch.where(ties, _first_argmax(raw), am_k)
            top = raw.max(dim=1).values
            got = torch.gather(raw, 1, am_k.unsqueeze(1)).squeeze(1)
            noise = 2e-5 * float(raw.abs().max().clamp_min(1e-30))
            assert float(torch.where(ties, torch.zeros_like(top), (top - got).abs()).max()) <= noise, ("routing", col)
            pre = torch.gather(raw, 1, am.unsqueeze(1)).squeeze(1)
            assert rel_err(feat_k[:, col:col + h], torch.tanh(pre + b.detach())) < 2e-5, ("feat", col)
            assert rel_err(pre_k[:, col:col + h], pre) < 2e-5, ("pool_raw", col)
            dact = 1 - torch.tanh(pre + b.detach()) ** 2
            lin = gate.detach() * conv_b + gate * conv_f                # d/d(x, W) through conv_b, d/d gate through conv_f
            lin_am = torch.gather(lin, 1, am.unsqueeze(1)).squeeze(1) + b
            loss = loss + (G[s].cuda().double()[:, col:col + h] * dact * lin_am).sum()
            col += h
    loss.backward()
    gt = tab_f.grad + tab_b.grad
    if c["pidx"] is not None:
        gt[c["pidx"]] = 0
    return gt, [[t.grad for t in p] for p in prm64]


_PRM_NAMES = ["la_w", "la_b", "lc_w", "lc_b", "ga_w", "ga_b", "c1_w", "c1_b", "c2_w", "c2_b", "c3_w", "c3_b"]


@pytest.mark.parametrize("name", list(ENC))
def test_datt_encoder_vs_float64(name, tmp_path):
    c = ENC[name]
    table, sides, ids_all, G = _enc_inputs(c)
    tab = table.cuda().requires_grad_()
    prm = [[t.cuda().requires_grad_() for t in p] for p in sides]
    shadow = ops.table_to_bf16(tab.detach()) if c["prec"] == "bf16" else None
    ids_dev = [i.cuda() for i in ids_all]
    cfg = {"precision": c["prec"], "shadow_fn": lambda: shadow, "arena": None, "table_param": tab, "params": prm,
           "padding_idx": -1 if c["pidx"] is None else c["pidx"], "flags": c["flags"]}
    args = []
    for s in range(2):
        args += [ids_dev[s], *prm[s]]

    def step():
        feats = ops.DattEncodeFn.apply(tab, cfg, *args)
        sum((f * G[s].cuda()).sum() for s, f in enumerate(feats)).backward()
        return feats

    feats, names = _kernels_launched(step, tmp_path)
    if c["flags"] == ops.CONV_TC_SINGLE_CTA:
        assert any("conv_tc_kernel<" in nm for nm in names) and not any("conv_tc2_kernel<" in nm for nm in names)
    if c["flags"] == ops.CONV_TC_PAIR_ONLY:
        assert any("conv_tc2_kernel<" in nm for nm in names) and not any("conv_tc_kernel<" in nm for nm in names)
    conv_fwd = [nm for nm in names if "conv_fp32_kernel<" in nm or "conv_tc_kernel<" in nm or "conv_tc2_kernel<" in nm]
    assert len(conv_fwd) == 8
    assert all(("fp32" in nm) == (c["prec"] == "fp32") for nm in conv_fwd), conv_fwd
    wk = "conv_bwd_weight_kernel<" if _vector_k2b(c["E"]) else "conv_bwd_weight_scalar_kernel"
    assert sum(wk in nm for nm in names) == 8, names
    # the kernel's arg-max, pool_raw and gates: the same calls again (the forward is deterministic)
    kernel_out = []
    for s in range(2):
        out = ops.datt_encode_side(tab.detach(), ids_dev[s], [t.detach() for t in prm[s]], c["prec"], shadow,
                                   conv_flags=c["flags"])
        assert torch.equal(out[0], feats[s].detach())
        kernel_out.append(out)
    if c["sat"] == "global":
        assert all(bool((o[4] == 0).all()) for o in kernel_out)
    if c["sat"] == "local":
        assert all(bool((o[3][:2] == 0).all()) for o in kernel_out)
        assert all(bool((o[3][2:] > 0).any()) for o in kernel_out)
    gt, gp = _enc_reference(c, table, sides, ids_all, G, kernel_out)
    assert rel_err(tab.grad, gt) < GRAD_TOL, ("table", rel_err(tab.grad, gt))
    for s in range(2):
        for i, nm in enumerate(_PRM_NAMES):
            assert rel_err(prm[s][i].grad, gp[s][i]) < GRAD_TOL, (s, nm, rel_err(prm[s][i].grad, gp[s][i]))
    if c["pidx"] is not None:
        assert float(tab.grad[c["pidx"]].abs().max()) == 0.0


def test_dual_att_conv_flags_pin_each_tensor_core_kernel(tmp_path):
    """DualAtt.conv_flags reaches every gated conv: CONV_TC_SINGLE_CTA runs only conv_tc, CONV_TC_PAIR_ONLY only conv_tc2,
    with the same features."""
    import rbr_b200
    from rbr_b200 import synth
    V, L = 400, 60
    params = synth.dual_att_params(V, L, 5, 40, 24, 100, 50, 10, seed=2)
    batch, _ = synth.dual_att_batch(8, L, V, seed=3)
    feats = {}
    for flags, want, other in ((ops.CONV_TC_SINGLE_CTA, "conv_tc_kernel<", "conv_tc2_kernel<"),
                               (ops.CONV_TC_PAIR_ONLY, "conv_tc2_kernel<", "conv_tc_kernel<")):
        model = rbr_b200.DualAtt(V, L, 5, 40, 24, 100, 50, 10, 0.0, None, precision="bf16")
        model.load_state_dict(params)
        model.cuda()
        model.conv_flags = flags
        with torch.no_grad():
            out, names = _kernels_launched(lambda: model.encode([batch[0].cuda()], ["u"])[0], tmp_path)
        assert sum(want in nm for nm in names) == 4 and not any(other in nm for nm in names), names
        feats[flags] = out
    assert rel_err(feats[ops.CONV_TC_SINGLE_CTA], feats[ops.CONV_TC_PAIR_ONLY]) < 1e-5
