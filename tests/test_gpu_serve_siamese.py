"""PairScorer for SimpleSiamese on the GPU, for every use_ui_bias x latent_transform: cached features against the float64
oracle, cached scores against the model's own forward, recommend / rank_items / evaluate against a brute-force float64 score
matrix, and K13's token attributions against float64 autograd gradient x input, with completeness, exact zeros, the window
rule, determinism, boundaries and the kernel's name in a profiler trace."""
import pytest
import torch

import rbr_b200
from oracle import rbr_oracle as orc
from rbr_b200 import ops, synth
from rbr_b200.inference import PairScorer, ranking_metrics

pytestmark = pytest.mark.gpu

DEV = "cuda"
V = 500
# "full": R = 10, T = 60, E = 300 (without the latent transform F = 300 is past the fused head, so K13 forms g itself);
# "small": every variant takes the fused head's g
SHAPES = {"full": dict(U=40, I=33, E=300, K=32, Ru=10, Ri=10, T=60),
          "small": dict(U=30, I=25, E=24, K=8, Ru=3, Ri=5, T=7)}
VARIANTS = [(ub, lt) for ub in (True, False) for lt in (False, True)]
VID = [f"{'bias' if ub else 'nobias'}-{'lt' if lt else 'nolt'}" for ub, lt in VARIANTS]


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _docs(n, R, T, seed):
    """Reviews with padding tails of every length, empty reviews, the padding entity 0 and an entity (1) with no reviews."""
    g = _gen(seed)
    d = torch.randint(1, V, (n, R, T), generator=g)
    lens = torch.randint(0, T + 1, (n, R), generator=g)
    d[torch.arange(T).view(1, 1, -1) >= lens.unsqueeze(-1)] = 0
    d[0] = 0
    d[1] = 0
    return d.to(DEV)


_CACHE = {}


def _setup(shape, ub, lt):
    key = (shape, ub, lt)
    if key not in _CACHE:
        s = SHAPES[shape]
        m = rbr_b200.SimpleSiamese(s["E"], s["K"], V, s["U"], s["I"], None, False, 0.0, 0.0, 0.0, ub, lt)
        m.load_state_dict(synth.simple_siamese_params(s["U"], s["I"], V, s["E"], s["K"], ub, lt, seed=0))
        sc = PairScorer(m.cuda())
        ud, idd = _docs(s["U"], s["Ru"], s["T"], 1), _docs(s["I"], s["Ri"], s["T"], 2)
        sc.build_cache(ud, idd, explain=True)
        _CACHE[key] = (sc, ud, idd)
    return _CACHE[key]


def _pairs(shape, n, seed):
    s = SHAPES[shape]
    g = _gen(seed)
    u, i = torch.randint(1, s["U"], (n,), generator=g), torch.randint(1, s["I"], (n,), generator=g)
    u[:3] = torch.tensor([1, 0, 2])                              # no reviews, the padding entity
    return u.to(DEV), i.to(DEV)


def _p64(model):
    return {k: v.detach().double() for k, v in model.state_dict().items()}


def _side64(p, x, wm):
    """float64 side feature from embedded tokens x [B, R, T, E] (oracle.simple_siamese_forward's side, rev mask = any word)"""
    B, R, T, E = x.shape
    pooled = orc.masked_avg_pool(x.reshape(-1, T, E), wm.reshape(-1, T)).view(B, R, E)
    if "latent_transform_layer.0.weight" in p:
        pooled = torch.tanh(pooled @ p["latent_transform_layer.0.weight"].t() + p["latent_transform_layer.0.bias"])
    hid = torch.tanh(pooled @ p["review_att_layer.proj_layer.0.weight"].t() + p["review_att_layer.proj_layer.0.bias"])
    logits = hid @ p["review_att_layer.inner_product.weight"].t()
    logits = torch.where(wm.any(-1).unsqueeze(2), logits, torch.full((), -1e8, dtype=logits.dtype, device=logits.device))
    return (torch.softmax(logits, dim=1) * pooled).sum(dim=1)


def _lat64(p, feat, ids, side):
    return orc.last_feat(feat, ids, p[f"{side}_last_feat_layer.W"], p[f"{side}_last_feat_layer.b"],
                         p[f"{side}_last_feat_layer.ebd.weight"])


def _head64(p, u_lat, i_lat, u, i):
    if "fm.user_bias.weight" in p:
        return orc.fm_head(u_lat, i_lat, u, i, p["fm.h"], p["fm.g_bias"], p["fm.user_bias.weight"], p["fm.item_bias.weight"]).view(-1)
    return (torch.relu(u_lat * i_lat) @ p["fm.h"] + p["fm.g_bias"]).view(-1)


def _ref_attr(sc, ud, idd, u, i):
    """float64 autograd: (pred, attr_u [B, R_u, T], attr_i [B, R_i, T], min |u_lat * i_lat| per pair)"""
    p = _p64(sc.model)
    table = p["word_embedding.embedding.weight"]
    xu = orc.embedding_gather(table, ud[u]).requires_grad_(True)
    xi = orc.embedding_gather(table, idd[i]).requires_grad_(True)
    u_lat, i_lat = _lat64(p, _side64(p, xu, ud[u] != 0), u, "user"), _lat64(p, _side64(p, xi, idd[i] != 0), i, "item")
    pred = _head64(p, u_lat, i_lat, u, i)
    pred.sum().backward()
    ref = orc.simple_siamese_forward(p, ud[u], idd[i], ud[u] != 0, idd[i] != 0, (ud[u] != 0).any(-1), (idd[i] != 0).any(-1), u, i)
    assert float((pred - ref).abs().max()) <= 1e-12                  # this restatement is the oracle's forward
    return (pred.detach(), (xu.grad * xu).sum(-1).detach(), (xi.grad * xi).sum(-1).detach(),
            (u_lat * i_lat).abs().min(1).values.detach())


# ---------------------------------------------------------------------------------------------------------------------
# cache, scores, top-k, ranks
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", ["full", "small"])
@pytest.mark.parametrize("ub,lt", VARIANTS, ids=VID)
def test_cached_features_and_scores(shape, ub, lt):
    sc, ud, idd = _setup(shape, ub, lt)
    p = _p64(sc.model)
    table = p["word_embedding.embedding.weight"]
    with torch.no_grad():
        for feat, docs in ((sc.user_feat, ud), (sc.item_feat, idd)):
            ref = _side64(p, orc.embedding_gather(table, docs), docs != 0)
            assert float((feat.double() - ref).abs().max()) <= 1e-5
    # explain=False keeps nothing extra and caches the same features
    plain = PairScorer(sc.model)
    plain.build_cache(ud, idd)
    assert plain._explain is None
    assert torch.equal(plain.user_feat, sc.user_feat) and torch.equal(plain.item_feat, sc.item_feat)
    # against the model's own eval forward on per-pair batches built from the entities' reviews
    u, i = _pairs(shape, 300, 3)
    got = sc.score_cached(u, i)
    with torch.no_grad():
        want = sc.model(ud[u], idd[i], None, None, (ud[u] != 0).any(-1), (idd[i] != 0).any(-1), u, i)[0]
    assert float((got.double() - want.double()).abs().max() / want.double().abs().max()) <= 2e-6


def _brute(sc):
    """float64 score matrix over all users x items from the cached features, padding item at -inf"""
    p = _p64(sc.model)
    U, I = sc.user_feat.shape[0], sc.item_feat.shape[0]
    uu = torch.arange(U, device=DEV).repeat_interleave(I)
    ii = torch.arange(I, device=DEV).repeat(U)
    S = _head64(p, _lat64(p, sc.user_feat.double()[uu], uu, "user"), _lat64(p, sc.item_feat.double()[ii], ii, "item"), uu, ii)
    S = S.view(U, I)
    S[:, 0] = float("-inf")
    return S


@pytest.mark.parametrize("ub,lt", VARIANTS, ids=VID)
def test_recommend_rank_evaluate(ub, lt):
    sc, _, _ = _setup("full", ub, lt)
    U, I = sc.user_feat.shape[0], sc.item_feat.shape[0]
    S = _brute(sc)
    users = torch.arange(1, U, device=DEV)
    k = 10
    scores, items = sc.recommend(users, k)
    assert not bool((items == 0).any())
    # position j holds the float64 j-th best score (ties to fp32 rounding aside), and exactly the float64 order (score desc,
    # id asc) on the rows whose top k + 1 scores are all apart
    S_cpu = S.cpu()
    sorted_ids = torch.stack([torch.tensor(sorted(range(I), key=lambda j: (-float(S_cpu[u, j]), j))) for u in users.tolist()]).to(DEV)
    srt = S[users.view(-1, 1), sorted_ids]
    scale = srt[:, :k + 1].abs().amax(1, keepdim=True)
    assert float(((S[users.view(-1, 1), items] - srt[:, :k]).abs() / scale).max()) <= 2e-6
    assert float(((scores.double() - S[users.view(-1, 1), items]).abs() / scale).max()) <= 2e-6
    clean = (srt[:, :k] - srt[:, 1:k + 1]).amin(1) > 2e-6 * scale.view(-1)
    assert bool(clean.any())
    assert torch.equal(items[clean], sorted_ids[clean, :k])
    # ranks of 4 targets per user; rank <= k <=> position rank - 1 of recommend with the same score bits
    g = _gen(4)
    tgt = torch.stack([torch.randperm(I - 1, generator=g)[:4] + 1 for _ in range(U - 1)]).to(DEV)
    ptr = torch.arange(0, 4 * (U - 1) + 1, 4, device=DEV)
    ranks, rscores, n_cand = sc.rank_items(users, (ptr, tgt.view(-1)))
    assert torch.equal(n_cand, torch.full((U - 1,), I - 1, device=DEV))
    s_all, i_all = sc.recommend(users, 64)
    rows = torch.arange(U - 1, device=DEV).repeat_interleave(4)
    for r, t, rk, s in zip(rows.tolist(), tgt.view(-1).tolist(), ranks.tolist(), rscores.tolist()):
        if rk <= 64:
            assert int(i_all[r, rk - 1]) == t and float(s_all[r, rk - 1]) == s
        else:
            assert t not in i_all[r].tolist()
    st = S[users[rows], tgt.view(-1)]
    pos = (S[users[rows]] - st.view(-1, 1))
    ref_rank = 1 + (pos > 0).sum(1) + ((pos == 0) & (torch.arange(I, device=DEV).view(1, -1) < tgt.view(-1, 1))).sum(1)
    near = ((pos.abs() <= 2e-6 * S[users[rows], 1:].abs().amax(1, keepdim=True)).sum(1) > 1)
    assert float(near.float().mean()) < 0.5
    assert torch.equal(ranks[~near], ref_rank[~near])
    # evaluate = ranking_metrics of the brute-force ranks, on the users whose targets are all clear of near-ties
    ok_row = ~near.view(U - 1, 4).any(1)
    sel = torch.nonzero(ok_row).view(-1)
    assert sel.numel() > 0
    t_c = (torch.arange(0, 4 * sel.numel() + 1, 4, device=DEV), tgt[sel].reshape(-1))
    got = sc.evaluate(users[sel], t_c, ks=(1, 5, 10))
    want = ranking_metrics(ref_rank.view(U - 1, 4)[sel].reshape(-1), t_c[0], n_cand[sel], ks=(1, 5, 10))
    for key in want:
        assert got[key] == pytest.approx(want[key], rel=1e-12, abs=1e-12), key


def test_factors_without_ui_bias():
    sc, _, _ = _setup("full", False, True)
    A, rb, B, cb = sc.factors()
    assert cb is None
    assert torch.equal(rb, torch.full_like(rb, float(sc.model.fm.g_bias.detach())))


# ---------------------------------------------------------------------------------------------------------------------
# token attributions
# ---------------------------------------------------------------------------------------------------------------------
def _nan_equal(a, b):
    if a is None or b is None:
        return a is None and b is None
    if not a.is_floating_point():
        return torch.equal(a, b)
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(a[~na], b[~nb])


FIELDS = ["text_total", "top_pos", "top_attr", "bottom_pos", "bottom_attr", "map", "review_weight", "review_attr"]


@pytest.mark.parametrize("shape", ["full", "small"])
@pytest.mark.parametrize("ub,lt", VARIANTS, ids=VID)
def test_maps_against_float64_autograd(shape, ub, lt):
    sc, ud, idd = _setup(shape, ub, lt)
    s = SHAPES[shape]
    u, i = _pairs(shape, 64, 5)
    ex = sc.explain(u, i, m=5, return_maps=True)
    assert torch.equal(ex.pred, sc.score_cached(u, i))
    pred, ref_u, ref_i, margin = _ref_attr(sc, ud, idd, u, i)
    clean = margin > 1e-6                                            # every FM ReLU decision is clear of 0
    assert float(clean.float().mean()) > 0.9
    for side, ref, docs, ids, R in ((ex.user, ref_u, ud, u, s["Ru"]), (ex.item, ref_i, idd, i, s["Ri"])):
        mp = side.map
        assert tuple(mp.shape) == (u.numel(), R, s["T"])
        scale = ref.flatten(1).abs().amax(1).clamp_min(1e-30)
        err = (mp.double() - ref).flatten(1).abs().amax(1) / scale
        assert float(err[clean].max()) <= 1e-5, float(err[clean].max())
        # exact zeros: masked tokens (padding ids), empty reviews, the entity without reviews, the padding entity
        assert bool((mp[docs[ids] == 0] == 0).all())
        assert bool((mp[ids <= 1] == 0).all())
        # completeness on the fixed-point grid, review sums, the window rule (width 1) on the returned map
        m64 = mp.double().flatten(1)
        tol = m64.abs().sum(1).clamp_min(1e-30)
        assert float(((side.text_total.double() - m64.sum(1)).abs() / tol).max()) <= 1e-6
        assert float(((side.review_attr.double() - mp.double().sum(-1)).abs() / tol.view(-1, 1)).max()) <= 1e-6
        tp, ta, bp, ba = ops.window_select(mp.flatten(1), s["T"], 5, 1)
        assert torch.equal(tp, side.top_pos) and torch.equal(bp, side.bottom_pos)
        assert _nan_equal(ta, side.top_attr) and _nan_equal(ba, side.bottom_attr)
        c = sc._explain["user" if side is ex.user else "item"]
        assert torch.equal(side.review_weight, c["att"][ids])
    assert float((ex.pred.double() - pred).abs().max() / pred.abs().max()) <= 1e-5


@pytest.mark.parametrize("ub,lt", VARIANTS, ids=VID)
def test_determinism(ub, lt):
    sc, _, _ = _setup("full", ub, lt)
    u, i = _pairs("full", 200, 6)
    e1 = sc.explain(u, i, m=6, width=3, return_maps=True)
    e2 = sc.explain(u, i, m=6, width=3, return_maps=True)
    e3 = sc.explain(u, i, m=6, width=3, return_maps=True, chunk=17)
    perm = torch.randperm(u.numel(), generator=_gen(7)).to(DEV)
    ep = sc.explain(u[perm], i[perm], m=6, width=3, return_maps=True)
    for name in ("user", "item"):
        for f in FIELDS:
            a = getattr(getattr(e1, name), f)
            for b in (getattr(getattr(e2, name), f), getattr(getattr(e3, name), f)):
                assert _nan_equal(a, b), (name, f)
            assert _nan_equal(a[perm], getattr(getattr(ep, name), f)), (name, f)
    # without maps: the same windows and totals
    e4 = sc.explain(u, i, m=6, width=3)
    assert e4.user.map is None
    for f in ("text_total", "top_pos", "top_attr", "review_attr"):
        assert _nan_equal(getattr(e1.user, f), getattr(e4.user, f)), f
    tok = sc.tokens_at("user", u, e1.user.top_pos)
    assert bool((tok[e1.user.top_pos >= 0] >= 0).all())
    # no pairs, with g from K4's backward or from K13
    e0 = sc.explain(u[:0], i[:0], return_maps=True)
    assert e0.user.top_pos.shape == (0, 5) and e0.item.map.shape[0] == 0


def test_ids_outside_the_table_read_as_zero_rows():
    sc, ud, _ = _setup("small", True, True)
    c = sc._explain["user"]
    table = sc.model.word_embedding.embedding.weight.detach()
    docs = ud.clone()
    docs[5, 0, 0] = V + 3
    u = torch.tensor([5, 6], device=DEV)
    g = torch.randn(2, sc.user_feat.shape[1], device=DEV)
    kw = dict(g=g, lt_w=sc.model.latent_transform_layer[0].weight.detach(), return_map=True)
    a = ops.explain_avgpool_attrib(table, docs, None, u, c["v"], c["a"], c["att"], sc.user_feat, 5, 1, **kw)
    docs[5, 0, 0] = V                                                # the appended zero row
    b = ops.explain_avgpool_attrib(torch.cat([table, torch.zeros_like(table[:1])]), docs, None, u, c["v"], c["a"], c["att"],
                                   sc.user_feat, 5, 1, **kw)
    for k in a:
        assert _nan_equal(a[k], b[k]), k
    for dt in (torch.int32, torch.uint16):                           # narrower ids: the same results
        e = ops.explain_avgpool_attrib(table, ud.to(dt), None, u, c["v"], c["a"], c["att"], sc.user_feat, 5, 1, **kw)
        f = ops.explain_avgpool_attrib(table, ud, None, u, c["v"], c["a"], c["att"], sc.user_feat, 5, 1, **kw)
        for k in e:
            assert _nan_equal(e[k], f[k]), (dt, k)


def test_boundaries():
    sc, _, _ = _setup("small", False, False)
    u, i = _pairs("small", 8, 8)
    for kw in (dict(m=0), dict(m=33), dict(width=0), dict(width=17)):
        with pytest.raises(ValueError):
            sc.explain(u, i, **kw)
    with pytest.raises(ValueError):
        sc.explain(u + 100, i)
    with pytest.raises(ValueError):
        sc.explain(u, i - 100)
    sc.explain(u, i, m=32, width=16)                                 # the limits themselves
    with pytest.raises(ValueError):
        PairScorer(sc.model).build_cache(torch.zeros(5, 7, dtype=torch.int64, device=DEV),
                                         torch.zeros(5, 3, 7, dtype=torch.int64, device=DEV))


@pytest.mark.parametrize("ub,lt", [(True, False), (True, True)], ids=["in-kernel-g", "fused-g"])
def test_kernel_in_profiler_trace(ub, lt):
    from torch.profiler import ProfilerActivity, profile
    sc, _, _ = _setup("full", ub, lt)
    u, i = _pairs("full", 64, 9)
    sc.explain(u, i)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sc.explain(u, i)
        torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    assert any("explain_avgpool_attrib_kernel" in n for n in names), sorted(names)
