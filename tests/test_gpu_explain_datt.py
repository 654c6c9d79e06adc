"""D-ATT token attributions on the GPU (ops.datt_explain_contrib, ops.datt_fc_grads, ops.explain_attrib's dense term and
PairScorer.explain(attribution=True)): the per-entity terms against a float64 statement of them, maps against float64
autograd gradient x input through both attention gates and the FC stack, g against float64, completeness, the window rule,
determinism, and the default mode left as it was."""
import ctypes

import pytest
import torch

import rbr_b200
from oracle import rbr_oracle as orc
from rbr_b200 import ops, synth
from rbr_b200.inference import PairScorer

pytestmark = pytest.mark.gpu

DEV = "cuda"
U, I, V = 300, 257, 500
LO, GO, WIN, E, H1, H2 = 200, 100, 5, 100, 500, 50


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _docs(n, L, seed):
    g = _gen(seed)
    d = torch.randint(1, V, (n, L), generator=g)
    d[:, L // 2 + seed % 7:] = 0                                          # padding tails: row 0 of the table, as stored
    return d.to(DEV)


def _model(prec, L):
    m = rbr_b200.DualAtt(V, L, WIN, LO, GO, E, H1, H2, 0.0, None, precision=prec)
    m.load_state_dict(synth.dual_att_params(V, L, WIN, LO, GO, E, H1, H2, seed=0))
    return m.cuda()


def _scorer(prec, L=120, explain=True):
    sc = PairScorer(_model(prec, L))
    ud, idd = _docs(U, L, 6), _docs(I, L, 7)
    sc.build_cache(ud, idd, explain=explain)
    return sc, (ud, idd)


def _pairs(n, seed):
    g = _gen(seed)
    return torch.randint(1, U, (n,), generator=g).to(DEV), torch.randint(1, I, (n,), generator=g).to(DEV)


def _p64(model):
    return {k: v.detach().double() for k, v in model.state_dict().items()}


def _side_prm(model, s):
    return [p.detach() for p in model._side_params(getattr(model, f"{s}_local_atten"), getattr(model, f"{s}_global_atten"))]


# ---------------------------------------------------------------------------------------------------------------------
# the per-entity terms
# ---------------------------------------------------------------------------------------------------------------------
def _ref_contrib(table, ids, p, s, gl, gg, feat, amax):
    """float64 statement of (contrib, gate_coef, gate_vec) at the kernels' gates, features and arg-max; x rows are zero for
    ids outside the table."""
    t64 = table.double()
    ok = (ids >= 0) & (ids < t64.shape[0])
    x = torch.where(ok.unsqueeze(-1), t64[ids.clamp(0, t64.shape[0] - 1)], torch.zeros((), dtype=torch.float64, device=DEV))
    N, L, Ed = x.shape
    wl = p[f"{s}_local_atten.attn.0.weight"][0]                           # [E, WIN]
    W = wl.shape[1]
    pad = (W - 1) // 2
    wg = p[f"{s}_global_atten.attn.0.weight"][0]                          # [E, L]
    lc = p[f"{s}_local_atten.conv.0.weight"][:, :, 0]                     # [LO, E]
    xp = torch.zeros(N, L + 2 * W, Ed, dtype=torch.float64, device=DEV)
    xp[:, W:W + L] = x

    def rows(t):                                                          # x at positions t [N, H] (zero outside) → [N, H, E]
        return xp.gather(1, (t + W).unsqueeze(-1).expand(-1, -1, Ed))

    d = 1.0 - feat.double() ** 2
    a = amax.long()
    gl64, gg64 = gl.double(), gg.double().view(-1, 1)
    nl = lc.shape[0]
    ts = a[:, :nl]
    q = (rows(ts) * lc).sum(-1)
    glt = gl64.gather(1, ts)
    loc = torch.empty(N, nl, W, dtype=torch.float64, device=DEV)
    for j in range(W):
        tap = (rows(ts + j - pad) * wl[:, j]).sum(-1)
        loc[:, :, j] = d[:, :nl] * q * glt * (1 - glt) * tap + (d[:, :nl] * glt * q if j == pad else 0.0)
    cols, coef, col = [loc.view(N, -1)], [torch.zeros(N, nl, dtype=torch.float64, device=DEV)], nl
    for c in (1, 2, 3):
        w = p[f"{s}_global_atten.conv{c}.0.weight"]
        G, _, k = w.shape
        tg = a[:, col:col + G]
        cj = torch.stack([(rows(tg + j) * w[:, :, j]).sum(-1) for j in range(k)], -1)
        dd = d[:, col:col + G]
        cols.append((dd.unsqueeze(-1) * gg64.unsqueeze(-1) * cj).reshape(N, -1))
        coef.append(dd * cj.sum(-1))
        col += G
    vec = gg64 * (1 - gg64) * (x * wg.t().unsqueeze(0)).sum(-1)
    return torch.cat(cols, 1), torch.cat(coef, 1), vec


def _rel(got, ref):
    return float((got.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("id_dtype", [torch.int64, torch.int32])
def test_datt_explain_contrib(prec, id_dtype):
    L, N = 120, 96
    m = _model(prec, L)
    p = _p64(m)
    table = m.word_embeddings.embedding.weight.detach()
    ids = _docs(N, L, 11)
    ids[3, 7] = V + 5                                                     # outside the table: a zero row everywhere
    ids[5, 0] = V
    ids[8, L - 1] = V + 100
    ids = ids.to(id_dtype)
    for s in ("u", "i"):
        prm = _side_prm(m, s)
        feat, amax, _, gl, gg = ops.datt_encode_side(table, ids, prm, prec)
        contrib, coef, vec = ops.datt_explain_contrib(table, ids, prm, gl, gg, feat, amax)
        assert contrib.shape == (N, LO * WIN + GO * 9) and coef.shape == (N, LO + 3 * GO) and vec.shape == (N, L)
        r_contrib, r_coef, r_vec = _ref_contrib(table, ids.long(), p, s, gl, gg, feat, amax)
        assert _rel(contrib, r_contrib) <= 1e-6, _rel(contrib, r_contrib)
        assert _rel(coef, r_coef) <= 1e-6, _rel(coef, r_coef)
        assert _rel(vec, r_vec) <= 1e-6, _rel(vec, r_vec)
        assert bool((coef[:, :LO] == 0).all())
    assert ops.lib.rbr_consume_oob_count(None) > 0                        # the ids outside the table were seen (and reset)


# ---------------------------------------------------------------------------------------------------------------------
# g through the FC stack
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("P,n_u,n_i,hidden,out_dim,in_dim", [(1000, 37, 53, 500, 50, 500), (70, 5, 9, 37, 3, 13),
                                                             (130, 300, 2, 768, 64, 17)])
def test_datt_fc_grads(P, n_u, n_i, hidden, out_dim, in_dim):
    g = _gen(P + hidden)
    u = torch.randint(0, n_u, (P,), generator=g).to(DEV)
    i = torch.randint(0, n_i, (P,), generator=g).to(DEV)
    uo, io = torch.randn(n_u, out_dim, generator=g).to(DEV), torch.randn(n_i, out_dim, generator=g).to(DEV)
    um, im = (torch.rand(n_u, hidden, generator=g) > 0.4).to(DEV), (torch.rand(n_i, hidden, generator=g) > 0.4).to(DEV)
    w0 = (torch.randn(hidden, in_dim, generator=g) / hidden ** 0.5).to(DEV)
    w3 = (torch.randn(out_dim, hidden, generator=g) / out_dim ** 0.5).to(DEV)
    g_u, g_i = ops.datt_fc_grads(u, i, uo, io, um, im, w0, w3)
    W0, W3 = w0.double(), w3.double()
    ref_u = (um[u].double() * (io[i].double() @ W3)) @ W0
    ref_i = (im[i].double() * (uo[u].double() @ W3)) @ W0
    assert _rel(g_u, ref_u) <= 1e-5 and _rel(g_i, ref_i) <= 1e-5, (_rel(g_u, ref_u), _rel(g_i, ref_i))
    # bit-identical whatever the batch or the order
    perm = torch.randperm(P, generator=_gen(1)).to(DEV)
    pu, pi = ops.datt_fc_grads(u[perm], i[perm], uo, io, um, im, w0, w3)
    assert torch.equal(pu, g_u[perm]) and torch.equal(pi, g_i[perm])
    parts = [ops.datt_fc_grads(u[lo:lo + 29], i[lo:lo + 29], uo, io, um, im, w0, w3) for lo in range(0, P, 29)]
    assert torch.equal(torch.cat([x[0] for x in parts]), g_u) and torch.equal(torch.cat([x[1] for x in parts]), g_i)


# ---------------------------------------------------------------------------------------------------------------------
# maps against float64 autograd
# ---------------------------------------------------------------------------------------------------------------------
def _ref_maps(sc, inputs, u, i):
    """float64 autograd gradient x input on the embedded tokens of both sides (oracle's D-ATT formulation, pooled at the
    cache's arg-max) → (user map, item map, user hidden pre-activations, item hidden pre-activations)."""
    p = _p64(sc.model)
    table = p["word_embeddings.embedding.weight"]
    c = sc._explain
    ud, idd = inputs

    def side(docs, s, amax):
        x = orc.embedding_gather(table, docs).requires_grad_()
        aw, ab = p[f"{s}_local_atten.attn.0.weight"], p[f"{s}_local_atten.attn.0.bias"]
        gate = torch.sigmoid(orc.conv1d_valid(x, aw, ab, pad=(aw.shape[2] - 1) // 2))
        a = amax.long()
        y = torch.tanh(orc.conv1d_valid(gate * x, p[f"{s}_local_atten.conv.0.weight"], p[f"{s}_local_atten.conv.0.bias"]))
        feats, col = [y.gather(1, a[:, :LO].unsqueeze(1)).squeeze(1)], LO
        gg = torch.sigmoid(orc.conv1d_valid(x, p[f"{s}_global_atten.attn.0.weight"], p[f"{s}_global_atten.attn.0.bias"]))
        for k in (1, 2, 3):
            w, b = p[f"{s}_global_atten.conv{k}.0.weight"], p[f"{s}_global_atten.conv{k}.0.bias"]
            y = torch.tanh(orc.conv1d_valid(gg * x, w, b))
            feats.append(y.gather(1, a[:, col:col + GO].unsqueeze(1)).squeeze(1))
            col += GO
        return x, torch.cat(feats, 1)

    def fc(f):
        z = f @ p["fc.0.weight"].t() + p["fc.0.bias"]
        return torch.relu(z) @ p["fc.3.weight"].t() + p["fc.3.bias"], z

    ux, uf = side(ud[u], "u", c["user"]["argmax"][u])
    ix, itf = side(idd[i], "i", c["item"]["argmax"][i])
    uo, uz = fc(uf)
    io, iz = fc(itf)
    (uo * io).sum().backward()
    return (ux * ux.grad).sum(-1).detach(), (ix * ix.grad).sum(-1).detach(), uz.detach(), iz.detach()


def _check_maps(got, ref, tol):
    scale = ref.abs().amax(1).clamp_min(1e-12)
    err = (got.double() - ref).abs().amax(1) / scale
    assert float(err.max()) <= tol, float(err.max())


@pytest.mark.parametrize("prec,L,n", [("fp32", 120, 300), ("bf16", 120, 300), ("fp32", 500, 64)])
def test_datt_maps(prec, L, n):
    sc, inputs = _scorer(prec, L)
    u, i = _pairs(n, 1)
    ref_u, ref_i, uz, iz = _ref_maps(sc, inputs, u, i)
    c = sc._explain
    # pairs where every FC ReLU is clearly decided and the cache decided it the same way
    keep = ((uz.abs() >= 2e-5).all(1) & (iz.abs() >= 2e-5).all(1) & ((uz > 0) == c["user"]["hid_mask"][u]).all(1)
            & ((iz > 0) == c["item"]["hid_mask"][i]).all(1))
    assert int(keep.sum()) >= (n // 10), int(keep.sum())
    e = sc.explain(u[keep], i[keep], m=5, return_maps=True, attribution=True)
    tol = 1e-5 if prec == "fp32" else 1e-2
    assert e.user.map.shape == (int(keep.sum()), L)
    _check_maps(e.user.map, ref_u[keep], tol)
    _check_maps(e.item.map, ref_i[keep], tol)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_datt_completeness_and_windows(prec):
    sc, _ = _scorer(prec)
    u, i = _pairs(500, 2)
    e = sc.explain(u, i, m=6, return_maps=True, attribution=True)
    e2 = sc.explain(u, i, m=6, return_maps=False, attribution=True)
    for side, ids in (("user", u), ("item", i)):
        s, s2 = getattr(e, side), getattr(e2, side)
        mp = s.map.double()
        scale = mp.abs().sum(1).clamp_min(1e-12)
        assert float(((s.text_total.double() - mp.sum(1)).abs() / scale).max()) <= 1e-6
        tp, ta, bp, ba = ops.window_select(s.map, 120, 6, WIN)                # the default width is the local window
        assert torch.equal(tp, s.top_pos) and torch.equal(bp, s.bottom_pos)
        assert torch.equal(ta, s.top_attr) and torch.equal(ba, s.bottom_attr)
        for f in ("text_total", "top_pos", "top_attr", "bottom_pos", "bottom_attr", "local_att", "global_att"):
            assert torch.equal(getattr(s, f), getattr(s2, f)), f
        assert s2.map is None
        tok = sc.tokens_at(side, ids, s.top_pos)
        docs = sc._explain[side]["docs"][ids]
        assert torch.equal(tok, torch.where(s.top_pos >= 0, docs.gather(1, s.top_pos.clamp_min(0)), torch.full_like(tok, -1)))
    w3 = sc.explain(u, i, m=4, width=3, attribution=True)
    assert torch.equal(w3.user.top_pos, ops.window_select(e.user.map, 120, 4, 3)[0])


def test_datt_consistency():
    sc, _ = _scorer("bf16")
    u, i = _pairs(1000, 6)
    e1 = sc.explain(u, i, m=5, return_maps=True, attribution=True)
    e2 = sc.explain(u, i, m=5, return_maps=True, attribution=True)
    e3 = sc.explain(u, i, m=5, return_maps=True, attribution=True, chunk=77)
    perm = torch.randperm(u.numel(), generator=_gen(7)).to(DEV)
    ep = sc.explain(u[perm], i[perm], m=5, return_maps=True, attribution=True)
    assert torch.equal(e1.pred, sc.score_cached(u, i))
    assert torch.equal(e1.pred[perm], ep.pred)
    for side in ("user", "item"):
        for f in ("text_total", "top_pos", "top_attr", "bottom_pos", "bottom_attr", "map", "local_att", "global_att"):
            a = getattr(getattr(e1, side), f)
            assert torch.equal(a, getattr(getattr(e2, side), f)), f
            assert torch.equal(a, getattr(getattr(e3, side), f)), f
            assert torch.equal(a[perm], getattr(getattr(ep, side), f)), f
    empty = sc.explain(u[:0], i[:0], attribution=True, return_maps=True)
    assert empty.user.top_pos.shape == (0, 5) and empty.item.map.shape == (0, 120)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_datt_default_mode_unchanged(prec):
    sc, (ud, idd) = _scorer(prec)
    sc0, _ = _scorer(prec, explain=False)
    assert torch.equal(sc.user_feat, sc0.user_feat) and torch.equal(sc.item_feat, sc0.item_feat)
    m = sc.model
    table = m.word_embeddings.embedding.weight.detach()
    u, i = _pairs(200, 5)
    e = sc.explain(u, i, m=7)
    ea = sc.explain(u, i, m=7, attribution=True)
    for s, docs, side in ((e.user, ud[u], "u"), (e.item, idd[i], "i")):
        la, ga = getattr(m, f"{side}_local_atten"), getattr(m, f"{side}_global_atten")
        gl, gg = ops.datt_gates(table, docs, la.attn[0].weight, la.attn[0].bias, ga.attn[0].weight, ga.attn[0].bias)
        assert torch.equal(s.local_att, gl) and torch.equal(s.global_att, gg)
        order = torch.sort(gl, dim=1, descending=True, stable=True).indices[:, :7]
        assert torch.equal(s.top_pos, order) and torch.equal(s.top_attr, gl.gather(1, order))
        assert s.text_total is None and s.bottom_pos is None and s.map is None
    for s, sa in ((e.user, ea.user), (e.item, ea.item)):
        assert torch.equal(s.local_att, sa.local_att) and torch.equal(s.global_att, sa.global_att)
    assert torch.equal(e.pred, ea.pred) and torch.equal(e.pred, sc.score_cached(u, i))


def test_explain_attrib_ex_matches_explain_attrib_on_deepconn():
    """rbr_explain_attrib_ex with feat and no dense term is rbr_explain_attrib, bit for bit"""
    Ud, Id, Ed, H, K, L = 120, 90, 64, 100, 32, 60
    m = rbr_b200.DeepCoNNpp(Ud, Id, V, [3, 5], Ed, H, K, L, None, 0.0, precision="bf16")
    m.load_state_dict(synth.deepconn_params(Ud, Id, V, Ed, H, K, (3, 5), seed=0))
    sc = PairScorer(m.cuda())
    sc.build_cache(_docs(Ud, L, 1), _docs(Id, L, 2), explain=True)
    g = _gen(3)
    u = torch.randint(1, Ud, (300,), generator=g).to(DEV)
    c = sc._explain["user"]
    specs = sc._conv_specs()
    grad = torch.randn(300, 1, sum(h for h, _, _ in specs), generator=g).to(DEV)
    ref = ops.explain_attrib(u, grad, c["feat"], c["argmax"], c["contrib"], specs, 1, L, 5, 5, return_map=True)
    out = {k: torch.empty_like(v) for k, v in ref.items()}
    conv = (ctypes.c_int64 * 6)(*[x for sp in specs for x in sp])
    ops.lib.check(ops.lib.rbr_explain_attrib_ex(
        u.data_ptr(), 300, 1, L, grad.data_ptr(), c["feat"].data_ptr(), c["argmax"].data_ptr(), c["feat"].shape[1],
        c["contrib"].data_ptr(), c["contrib"].shape[1], c["feat"].shape[0], 2, conv, None, 0, None, 0, 5, 5,
        out["text_total"].data_ptr(), out["top_pos"].data_ptr(), out["top_attr"].data_ptr(), out["bottom_pos"].data_ptr(),
        out["bottom_attr"].data_ptr(), out["map"].data_ptr(), None, torch.cuda.current_stream().cuda_stream),
        "rbr_explain_attrib_ex")
    for k in ref:
        assert torch.equal(ref[k], out[k]), k


def test_datt_kernels_in_profiler_trace():
    from torch.profiler import ProfilerActivity, profile
    u, i = _pairs(64, 9)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sc, _ = _scorer("bf16")
        sc.explain(u, i, attribution=True)
        torch.cuda.synchronize()
    names = " ".join(evt.key for evt in prof.key_averages())
    for k in ("datt_explain_contrib_kernel", "datt_fc_grads_kernel", "explain_attrib_kernel"):
        assert k in names, k
