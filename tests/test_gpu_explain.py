"""K12 (ops.conv_window_contrib / ops.explain_attrib) and PairScorer.explain on the GPU: tap contributions against float64,
attribution maps against float64 autograd gradient x input on the embedded tokens, completeness, the window rule, NARRE's
review level, D-ATT's gates, and determinism."""
import pytest
import torch

import rbr_b200
from oracle import rbr_oracle as orc
from rbr_b200 import ops, synth
from rbr_b200.inference import PairScorer

pytestmark = pytest.mark.gpu

DEV = "cuda"
U, I, V, E, HID, K = 300, 257, 500, 64, 100, 32


def _gen(seed):
    return torch.Generator().manual_seed(seed)


# ---------------------------------------------------------------------------------------------------------------------
# contributions
# ---------------------------------------------------------------------------------------------------------------------
def _ref_contrib(table, ids, mask, weight, pad, argmax):
    """float64 c[n, h, j] with rows read as zeros outside the document, at masked positions and for ids outside the table."""
    N, L = ids.shape
    H, _, k = weight.shape
    t64, w64 = table.double(), weight.double()
    ok = (ids >= 0) & (ids < table.shape[0]) & mask
    x = torch.where(ok.unsqueeze(-1), t64[ids.clamp(0, table.shape[0] - 1)], torch.zeros((), dtype=torch.float64, device=DEV))
    xp = torch.zeros(N, L + 2 * k, table.shape[1], dtype=torch.float64, device=DEV)
    xp[:, k:k + L] = x
    out = torch.empty(N, H, k, dtype=torch.float64, device=DEV)
    for j in range(k):
        t = argmax.long() + j - pad + k                                   # index into xp
        rows = xp.gather(1, t.unsqueeze(-1).expand(N, H, table.shape[1]))  # [N, H, E]
        out[:, :, j] = (rows * w64[:, :, j].unsqueeze(0)).sum(-1)
    return out.view(N, H * k)


@pytest.mark.parametrize("emb,filters", [(30, 100), (300, 150)])
@pytest.mark.parametrize("id_dtype", [torch.int64, torch.int32, torch.uint16])
@pytest.mark.parametrize("k", [1, 3, 5, 7])
def test_conv_window_contrib(k, id_dtype, emb, filters):
    g = _gen(k * 10 + emb)
    N, L, pad = 48, 40, (k - 1) // 2
    table = torch.randn(V, emb, generator=g).to(DEV)
    weight = (torch.randn(filters, emb, k, generator=g) * 0.1).to(DEV)
    ids = torch.randint(1, V, (N, L), generator=g)
    ids[torch.arange(L).view(1, -1) >= (L - 5 - torch.arange(N) % 7).view(-1, 1)] = 0     # padding tails of different lengths
    ids[3, 4] = V + 7                                               # outside the table: reads as zeros
    ids = ids.to(DEV)
    n_pos = L + 2 * pad - k + 1
    amax = torch.randint(0, n_pos, (N, filters), generator=g, dtype=torch.int32).to(DEV)
    amax[:, 0] = 0                                                  # windows hanging over the front
    amax[:, 1] = n_pos - 1                                          # ... and over the end
    mask = torch.rand(N, L, generator=g).to(DEV) > 0.2
    mask[ids == 0] = True                                           # disagrees with ids != 0 both ways
    for msk, mfi in ((mask, False), (None, True), (None, False)):
        got = ops.conv_window_contrib(table, ids.to(id_dtype), msk, weight, pad, amax, mask_from_ids=mfi)
        eff = msk if msk is not None else ((ids != 0) if mfi else torch.ones_like(ids, dtype=torch.bool))
        ref = _ref_contrib(table, ids, eff, weight, pad, amax)
        assert float((got.double() - ref).abs().max() / ref.abs().max()) <= 1e-6


def test_conv_window_contrib_column_slices():
    """two convs writing one shared output through column offsets, as build_cache(explain=True) lays them out"""
    g = _gen(3)
    N, L, emb = 20, 30, 64
    table = torch.randn(V, emb, generator=g).to(DEV)
    ids = torch.randint(0, V, (N, L), generator=g).to(DEV)
    w3, w5 = torch.randn(50, emb, 3, generator=g).to(DEV), torch.randn(50, emb, 5, generator=g).to(DEV)
    amax = torch.randint(0, L, (N, 100), generator=g, dtype=torch.int32).to(DEV)
    out = torch.full((N, 50 * 3 + 50 * 5), float("nan"), device=DEV)
    ops.conv_window_contrib(table, ids, None, w3, 1, amax[:, :50], mask_from_ids=True, out=out[:, :150])
    ops.conv_window_contrib(table, ids, None, w5, 2, amax[:, 50:], mask_from_ids=True, out=out[:, 150:])
    assert torch.equal(out[:, :150], ops.conv_window_contrib(table, ids, None, w3, 1, amax[:, :50].contiguous(), mask_from_ids=True))
    assert torch.equal(out[:, 150:], ops.conv_window_contrib(table, ids, None, w5, 2, amax[:, 50:].contiguous(), mask_from_ids=True))


# ---------------------------------------------------------------------------------------------------------------------
# models
# ---------------------------------------------------------------------------------------------------------------------
def _docs(n, L, seed):
    g = _gen(seed)
    d = torch.randint(1, V, (n, L), generator=g)
    d[:, L // 2 + seed % 7:] = 0
    return d.to(DEV)


def _deepconn(prec, ks=(3,), L=60, explain=True):
    m = rbr_b200.DeepCoNNpp(U, I, V, list(ks), E, HID, K, L, None, 0.0, precision=prec)
    m.load_state_dict(synth.deepconn_params(U, I, V, E, HID, K, tuple(ks), seed=0))
    sc = PairScorer(m.cuda())
    ud, idd = _docs(U, L, 1), _docs(I, L, 2)
    sc.build_cache(ud, idd, explain=explain)
    return sc, (ud, idd)


def _narre(prec, R=10, T=60, explain=True):
    m = rbr_b200.NARRE(U, I, V, [3], 150, E, 32, K, R, T, 0.0, 0, 0, 0, None, "CNN", precision=prec)
    m.load_state_dict(synth.narre_params(U, I, V, E, 150, 32, K, (3,), seed=0))
    sc = PairScorer(m.cuda())
    ud, idd = _docs(U * R, T, 3).view(U, R, T), _docs(I * R, T, 4).view(I, R, T)
    g = _gen(5)
    urev, irev = torch.randint(0, I, (U, R), generator=g).to(DEV), torch.randint(0, U, (I, R), generator=g).to(DEV)
    sc.build_cache(ud, idd, user_rev_ids=urev, item_rev_ids=irev, explain=explain)
    return sc, (ud, idd, urev, irev)


def _datt(prec, L=120):
    m = rbr_b200.DualAtt(V, L, 5, 200, 100, 100, 500, 50, 0.0, None, precision=prec)
    m.load_state_dict(synth.dual_att_params(V, L, 5, 200, 100, 100, 500, 50, seed=0))
    sc = PairScorer(m.cuda())
    ud, idd = _docs(U, L, 6), _docs(I, L, 7)
    sc.build_cache(ud, idd, explain=True)
    return sc, (ud, idd)


def _pairs(n, seed):
    g = _gen(seed)
    return torch.randint(1, U, (n,), generator=g).to(DEV), torch.randint(1, I, (n,), generator=g).to(DEV)


def _p64(model):
    return {k: v.detach().double() for k, v in model.state_dict().items()}


def _conv64(p):
    return orc._conv_params(p, "ngram.feature_layer.0.list_of_conv1d")


def _clean_pairs(sc, inputs, u, i, name, tau=2e-5):
    """The pairs whose every ReLU is at least tau from 0 in float64 (orc.relu_margins) and whose conv ReLU decisions at the
    cache's arg-max agree with the cache's features (bf16 features are ~1e-3 off): there every implementation takes the same
    branches, so maps compare at the stated tolerance."""
    p = _p64(sc.model)
    table = p["word_embeddings.embedding.weight"]
    ws, bs = _conv64(p)
    c = sc._explain
    with torch.no_grad():
        if name == "deepconn":
            ud, idd = inputs
            batch = [ud[u], idd[i], ud[u] != 0, idd[i] != 0, u, i]
            sides = [(ud[u], c["user"]["argmax"][u], c["user"]["feat"][u]), (idd[i], c["item"]["argmax"][i], c["item"]["feat"][i])]
        else:
            ud, idd, urev, irev = inputs
            batch = [ud[u], idd[i], ud[u] != 0, idd[i] != 0, u, i, urev[u], irev[i]]
            R, T = ud.shape[1:]
            H = c["user"]["feat"].shape[1]
            sides = [(ud[u].reshape(-1, T), c["user"]["argmax"].view(-1, R, H)[u].reshape(-1, H),
                      c["user"]["feat"].view(-1, R, H)[u].reshape(-1, H)),
                     (idd[i].reshape(-1, T), c["item"]["argmax"].view(-1, R, H)[i].reshape(-1, H),
                      c["item"]["feat"].view(-1, R, H)[i].reshape(-1, H))]
        keep = orc.relu_margins(name, p, batch) >= tau
        texts = []
        for ids, amax, feat in sides:
            x = orc.embedding_gather(table, ids)
            f64 = orc.ngram_feat(x, ids != 0, ws, bs, argmax_override=amax)
            keep &= ((f64 > 0) == (feat > 0)).view(u.numel(), -1).all(1)
            texts.append((f64, feat.double()))
        if name == "deepconn":
            # the FM ReLU decisions under the cached features equal those under the float64 ones
            def fm_sign(ut, it):
                ul = orc.last_feat(ut, u, p["user_feat.W"], p["user_feat.b"], p["user_feat.ebd.weight"])
                il = orc.last_feat(it, i, p["item_feat.W"], p["item_feat.b"], p["item_feat.ebd.weight"])
                return ul * il > 0
            keep &= (fm_sign(texts[0][0], texts[1][0]) == fm_sign(texts[0][1], texts[1][1])).all(1)
    return u[keep], i[keep]


def _ref_maps(sc, inputs, u, i, name):
    """float64 autograd gradient x input on the embedded tokens of each pair's documents, routed through the cache's
    arg-max (orc.ngram_feat's argmax_override) → (user map, item map): [B, L] or [B, R, T]."""
    p = _p64(sc.model)
    table = p["word_embeddings.embedding.weight"]
    ws, bs = _conv64(p)
    c = sc._explain
    if name == "deepconn":
        ud, idd = inputs
        ux = orc.embedding_gather(table, ud[u]).requires_grad_()
        ix = orc.embedding_gather(table, idd[i]).requires_grad_()
        uf = orc.ngram_feat(ux, ud[u] != 0, ws, bs, argmax_override=c["user"]["argmax"][u])
        itf = orc.ngram_feat(ix, idd[i] != 0, ws, bs, argmax_override=c["item"]["argmax"][i])
    else:
        ud, idd, urev, irev = inputs
        b, R, T = ud[u].shape
        H = c["user"]["feat"].shape[1]
        ux = orc.embedding_gather(table, ud[u]).requires_grad_()
        ix = orc.embedding_gather(table, idd[i]).requires_grad_()
        u_rf = orc.ngram_feat(ux.view(b * R, T, -1), (ud[u] != 0).view(b * R, T), ws, bs,
                              argmax_override=c["user"]["argmax"].view(-1, R, H)[u].reshape(-1, H)).view(b, R, H)
        i_rf = orc.ngram_feat(ix.view(b * R, T, -1), (idd[i] != 0).view(b * R, T), ws, bs,
                              argmax_override=c["item"]["argmax"].view(-1, R, H)[i].reshape(-1, H)).view(b, R, H)
        att = {s: {k: p[f"{s}_att.{k}"] for k in ("W_rv", "W_id", "h", "b_1", "b_2")} for s in ("user", "item")}
        uf, _ = orc.linear_attention(u_rf, urev[u], ebd_vals=p["user_att.ebd_vals.weight"], **att["user"])
        itf, _ = orc.linear_attention(i_rf, irev[i], ebd_vals=p["item_att.ebd_vals.weight"], **att["item"])
    u_f = orc.last_feat(uf, u, p["user_feat.W"], p["user_feat.b"], p["user_feat.ebd.weight"])
    i_f = orc.last_feat(itf, i, p["item_feat.W"], p["item_feat.b"], p["item_feat.ebd.weight"])
    pred = orc.fm_head(u_f, i_f, u, i, p["fm.h"], p["fm.g_bias"], p["fm.user_bias.weight"], p["fm.item_bias.weight"])
    pred.sum().backward()
    return (ux * ux.grad).sum(-1).detach(), (ix * ix.grad).sum(-1).detach()


def _check_maps(got, ref, tol):
    scale = ref.flatten(1).abs().amax(1).clamp_min(1e-12)
    err = (got.double() - ref).flatten(1).abs().amax(1) / scale
    assert float(err.max()) <= tol, float(err.max())


@pytest.mark.parametrize("prec,ks", [("fp32", (3,)), ("bf16", (3,)), ("fp32", (3, 5))])
def test_deepconn_maps(prec, ks):
    sc, inputs = _deepconn(prec, ks)
    u, i = _pairs(400, 1)
    u, i = _clean_pairs(sc, inputs, u, i, "deepconn")
    assert u.numel() >= 100
    e = sc.explain(u, i, m=5, return_maps=True)
    ref_u, ref_i = _ref_maps(sc, inputs, u, i, "deepconn")
    tol = 1e-5 if prec == "fp32" else 1e-2
    _check_maps(e.user.map, ref_u, tol)
    _check_maps(e.item.map, ref_i, tol)
    assert e.user.map.shape == (u.numel(), 60)


@pytest.mark.parametrize("prec,ks", [("fp32", (3,)), ("bf16", (3,)), ("fp32", (3, 5))])
def test_completeness_and_windows(prec, ks):
    sc, inputs = _deepconn(prec, ks)
    u, i = _pairs(500, 2)
    e = sc.explain(u, i, m=6, return_maps=True)
    e2 = sc.explain(u, i, m=6, return_maps=False)
    m = sc.model
    head = sc._head_params()
    pads = (m.user_feat.padding_idx, m.item_feat.padding_idx, m.fm.padding_idx, m.fm.item_padding_idx)
    g_u, g_i = ops.head_text_grads(sc.user_feat[u], sc.item_feat[i], u, i, head, pads)
    conv = m.ngram.conv
    specs = [(c.weight.shape[0], k) for c, k in zip(conv.list_of_conv1d, conv.kernel_sizes)]
    bias = torch.cat([c.bias.detach() for c in conv.list_of_conv1d]).double()
    width = max(ks)
    for side, ids, g in (("user", u, g_u), ("item", i, g_i)):
        s, s2 = getattr(e, side), getattr(e2, side)
        c = sc._explain[side]
        mp = s.map.double()
        scale = mp.abs().sum(1).clamp_min(1e-12)
        assert float(((s.text_total.double() - mp.sum(1)).abs() / scale).max()) <= 1e-6
        # sum_h g * sum_j c over live features
        live = c["feat"][ids] > 0
        contrib = c["contrib"][ids].double()
        csum, col = [], 0
        for h, k in specs:
            csum.append(contrib[:, col:col + h * k].view(-1, h, k).sum(-1))
            col += h * k
        rhs_terms = torch.where(live, g.double() * torch.cat(csum, 1), torch.zeros((), dtype=torch.float64, device=DEV))
        rscale = rhs_terms.abs().sum(1).clamp_min(1e-12)
        assert float(((s.text_total.double() - rhs_terms.sum(1)).abs() / rscale).max()) <= 1e-6
        if prec == "fp32":
            fb = torch.where(live, g.double() * (c["feat"][ids].double() - bias), torch.zeros((), dtype=torch.float64, device=DEV))
            assert float(((s.text_total.double() - fb.sum(1)).abs() / rscale).max()) <= 1e-5
        # the windows are the rule applied to the returned map, and do not depend on return_maps
        tp, ta, bp, ba = ops.window_select(s.map, 60, 6, width)
        assert torch.equal(tp, s.top_pos) and torch.equal(bp, s.bottom_pos)
        assert torch.equal(ta, s.top_attr) and torch.equal(ba, s.bottom_attr)
        for f in ("text_total", "top_pos", "top_attr", "bottom_pos", "bottom_attr"):
            assert torch.equal(getattr(s, f), getattr(s2, f)), f
        assert s2.map is None
        # the tokens helper reads the kept documents
        tok = sc.tokens_at(side, ids, s.top_pos)
        docs = c["docs"][ids]
        assert torch.equal(tok, torch.where(s.top_pos >= 0, docs.gather(1, s.top_pos.clamp_min(0)), torch.full_like(tok, -1)))


def test_narre_maps_and_review_level():
    sc, inputs = _narre("fp32")
    u, i = _pairs(300, 3)
    u, i = _clean_pairs(sc, inputs, u, i, "narre")
    assert u.numel() >= 50
    e = sc.explain(u, i, m=5, return_maps=True)
    ref_u, ref_i = _ref_maps(sc, inputs, u, i, "narre")
    assert e.user.map.shape == (u.numel(), 10, 60)
    _check_maps(e.user.map, ref_u, 1e-5)
    _check_maps(e.item.map, ref_i, 1e-5)
    ud, idd, urev, irev = inputs
    with torch.no_grad():
        _, u_sc, i_sc = sc.model(ud[u], idd[i], None, None, u, i, urev[u], irev[i])
    for s, ref_sc in ((e.user, u_sc), (e.item, i_sc)):
        assert float((s.review_weight - ref_sc.view(-1, 10)).abs().max()) <= 1e-5
        mp = s.map.double()
        scale = mp.abs().flatten(1).sum(1, keepdim=True).clamp_min(1e-12)
        assert float(((s.review_attr.double() - mp.sum(-1)).abs() / scale).max()) <= 1e-6
        assert float(((s.text_total.double() - mp.flatten(1).sum(1)).abs() / scale.view(-1)).max()) <= 1e-6
        tp, ta, bp, ba = ops.window_select(s.map.flatten(1), 60, 5, 3)
        assert torch.equal(tp, s.top_pos) and torch.equal(bp, s.bottom_pos)
        # windows never cross a review boundary
        ok = s.top_pos < 0
        assert bool(((s.top_pos % 60 + 3 <= 60) | ok).all())


def test_narre_bf16_runs_and_is_complete():
    sc, _ = _narre("bf16")
    u, i = _pairs(200, 4)
    e = sc.explain(u, i, return_maps=True)
    for s in (e.user, e.item):
        mp = s.map.double().flatten(1)
        assert bool(torch.isfinite(mp).all())
        scale = mp.abs().sum(1).clamp_min(1e-12)
        assert float(((s.text_total.double() - mp.sum(1)).abs() / scale).max()) <= 1e-6


def test_datt_gates():
    sc, (ud, idd) = _datt("fp32")
    m = sc.model
    p = _p64(m)
    table = p["word_embeddings.embedding.weight"]
    u, i = _pairs(200, 5)
    e = sc.explain(u, i, m=7)
    for s, docs, side in ((e.user, ud[u], "u"), (e.item, idd[i], "i")):
        x = orc.embedding_gather(table, docs)
        lw, lb = p[f"{side}_local_atten.attn.0.weight"], p[f"{side}_local_atten.attn.0.bias"]
        gw, gb = p[f"{side}_global_atten.attn.0.weight"], p[f"{side}_global_atten.attn.0.bias"]
        ref_l = torch.sigmoid(orc.conv1d_valid(x, lw, lb, pad=(lw.shape[2] - 1) // 2)).squeeze(-1)
        ref_g = torch.sigmoid(orc.conv1d_valid(x, gw, gb)).view(-1)
        assert float((s.local_att.double() - ref_l).abs().max()) <= 1e-5
        assert float((s.global_att.double() - ref_g).abs().max()) <= 1e-5
        order = torch.sort(s.local_att, dim=1, descending=True, stable=True).indices[:, :7]
        assert torch.equal(s.top_pos, order)
        assert torch.equal(s.top_attr, s.local_att.gather(1, order))
    assert torch.equal(e.pred, sc.score_cached(u, i))


@pytest.mark.parametrize("name", ["deepconn", "narre"])
def test_consistency(name):
    sc, _ = (_deepconn if name == "deepconn" else _narre)("bf16")
    u, i = _pairs(1000, 6)
    e1 = sc.explain(u, i, m=5, return_maps=True)
    e2 = sc.explain(u, i, m=5, return_maps=True)
    e3 = sc.explain(u, i, m=5, return_maps=True, chunk=77)                # other batch compositions
    assert torch.equal(e1.pred, sc.score_cached(u, i))
    perm = torch.randperm(u.numel(), generator=_gen(7)).to(DEV)
    ep = sc.explain(u[perm], i[perm], m=5, return_maps=True)
    fields = ["text_total", "top_pos", "top_attr", "bottom_pos", "bottom_attr", "map"] + (
        ["review_weight", "review_attr"] if name == "narre" else [])
    for side in ("user", "item"):
        for f in fields:
            a = getattr(getattr(e1, side), f)
            assert torch.equal(a, getattr(getattr(e2, side), f)), f
            assert torch.equal(a, getattr(getattr(e3, side), f)), f
            assert torch.equal(a[perm], getattr(getattr(ep, side), f)), f
    assert torch.equal(e1.pred[perm], ep.pred)


def test_explain_needs_the_explain_cache():
    sc, _ = _deepconn("fp32", explain=False)
    u, i = _pairs(10, 8)
    with pytest.raises(RuntimeError):
        sc.explain(u, i)
    assert sc._explain is None
    sc2, _ = _deepconn("fp32", explain=True)
    assert torch.equal(sc.user_feat, sc2.user_feat) and torch.equal(sc.item_feat, sc2.item_feat)
    with pytest.raises(ValueError):
        sc2.explain(u, i, m=33)
    with pytest.raises(ValueError):
        sc2.explain(u, i, width=17)
    with pytest.raises(ValueError):
        sc2.explain(torch.tensor([U], device=DEV), torch.tensor([1], device=DEV))
    hier = rbr_b200.DeepCoNNpp(U, I, V, [3], E, E, K, 60, None, 0.0, arch="HierPooling").cuda()
    with pytest.raises(NotImplementedError):
        PairScorer(hier).build_cache(_docs(U, 60, 1), _docs(I, 60, 2), explain=True)


def test_narre_cache_unchanged_by_explain():
    sc0, _ = _narre("bf16", explain=False)
    sc1, _ = _narre("bf16", explain=True)
    assert torch.equal(sc0.user_feat, sc1.user_feat) and torch.equal(sc0.item_feat, sc1.item_feat)


def test_kernels_in_profiler_trace():
    from torch.profiler import ProfilerActivity, profile
    u, i = _pairs(64, 9)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sc, _ = _deepconn("bf16")
        sc.explain(u, i)
        torch.cuda.synchronize()
    names = " ".join(evt.key for evt in prof.key_averages())
    assert "conv_window_contrib_kernel" in names
    assert "explain_attrib_kernel" in names
