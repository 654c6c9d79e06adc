"""PairScorer.add / update on the GPU, for DeepCoNN (CNN bf16 / fp32, HierPooling), NARRE, D-ATT and SimpleSiamese (K4's g
and K13's in-kernel g): new entities score as the model's eval forward under the padding id, an update serves what a rebuild
on the changed documents serves, added items are served everywhere while the padding row stays apart, derived state never
goes stale, the work follows the change, and bad input is refused before any encoder runs."""
import pytest
import torch

import rbr_b200
import test_gpu_explain as X
import test_gpu_serve_siamese as S
from rbr_b200 import ops, synth
from rbr_b200.inference import PairScorer, fm_factors

pytestmark = pytest.mark.gpu

DEV = "cuda"
V = 500
CASES = ["cnn_fp32", "cnn_bf16", "hier", "narre", "datt", "siamese_fused_g", "siamese_kernel_g"]
EXACT = {"cnn_fp32", "cnn_bf16", "narre"}   # batch-invariant encoders; elsewhere an nn.Linear changes bits with batch size


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _hier():
    m = rbr_b200.DeepCoNNpp(X.U, X.I, V, [3], 64, 64, 32, 60, None, 0.0, arch="HierPooling")
    m.load_state_dict(synth.deepconn_hier_params(X.U, X.I, V, 64, 64, 32, seed=0))
    sc = PairScorer(m.cuda())
    ud, idd = X._docs(X.U, 60, 1), X._docs(X.I, 60, 2)
    sc.build_cache(ud, idd)
    return sc, (ud, idd)


def _case(name):
    """(scorer, {side: [documents, per-review input]}) on a fresh scorer (and, but for SimpleSiamese, a fresh model)"""
    if name.startswith("siamese"):
        base, ud, idd = S._setup("full", True, name == "siamese_fused_g")
        sc = PairScorer(base.model)                           # _setup's scorer is shared with other tests: never changed
        sc.build_cache(ud, idd, explain=True)
        inputs = (ud, idd)
    elif name == "hier":
        sc, inputs = _hier()
    else:
        make = {"cnn": X._deepconn, "narre": X._narre, "datt": X._datt}[name.split("_")[0]]
        sc, inputs = make(name.split("_")[1] if "_" in name else "fp32")
    rev = inputs[2:] if name == "narre" else (None, None)
    return sc, {"user": [inputs[0], rev[0]], "item": [inputs[1], rev[1]]}


def _kw(sc, side, rev):
    if isinstance(sc.model, rbr_b200.NARRE):
        return {"rev_ids": rev}
    return {}


def _rebuild(sc, data, added=None):
    """a fresh scorer on the same model: build_cache on data's documents, then one add per side of `added`"""
    fresh = PairScorer(sc.model)
    kw = {}
    if isinstance(sc.model, rbr_b200.NARRE):
        kw = {"user_rev_ids": data["user"][1], "item_rev_ids": data["item"][1]}
    fresh.build_cache(data["user"][0], data["item"][0], explain=sc._explain is not None, **kw)
    for side, (docs, rev) in (added or {}).items():
        fresh.add(side, docs, **_kw(sc, side, rev))
    return fresh


def _new_docs(sc, data, side, n, seed):
    """n seeded documents of the side's shape, and for NARRE review ids of counterparts (model ids, the padding id among)"""
    shape = data[side][0].shape[1:]
    g = _gen(seed)
    d = torch.randint(1, V, (n, *shape), generator=g)
    d[..., shape[-1] // 2 + seed % 5:] = 0
    rev = None
    if isinstance(sc.model, rbr_b200.NARRE):
        n_other = X.I if side == "user" else X.U
        rev = torch.randint(0, n_other, (n, shape[0]), generator=g).to(DEV)
    return d.to(DEV), rev


def _forward(sc, data, u_docs, i_docs, u_rev, i_rev, u_mid, i_mid):
    """the model's own eval forward on per-pair batches (PairScorer.score_pairs)"""
    m = sc.model
    if isinstance(m, rbr_b200.NARRE):
        return sc.score_pairs(u_docs, i_docs, None, None, u_mid, i_mid, u_rev, i_rev)
    if isinstance(m, rbr_b200.DualAtt):
        return sc.score_pairs(u_docs, i_docs)
    if isinstance(m, rbr_b200.SimpleSiamese):
        return sc.score_pairs(u_docs, i_docs, None, None, (u_docs != 0).any(-1), (i_docs != 0).any(-1), u_mid, i_mid)
    return sc.score_pairs(u_docs, i_docs, None, None, u_mid, i_mid)


def _close(a, b, exact, tol=2e-5):
    if a is None or b is None:
        assert a is None and b is None
        return
    if exact or not (a.is_floating_point()):
        assert a.shape == b.shape and torch.equal(torch.nan_to_num(a, nan=7.5), torch.nan_to_num(b, nan=7.5))
        return
    a, b = (torch.nan_to_num(t.double(), nan=7.5, posinf=float("inf"), neginf=float("-inf")) for t in (a, b))
    fin = torch.isfinite(b)
    assert torch.equal(fin, torch.isfinite(a)) and torch.equal(a[~fin], b[~fin])
    scale = b[fin].abs().max().clamp_min(1e-12) if fin.any() else 1.0
    assert float((a[fin] - b[fin]).abs().max() / scale) <= tol if fin.any() else True


def _topk_close(got, ref, exact):
    """(scores, items) of a top-k: equal, or (through an nn.Linear) the same items on nearly every row"""
    if exact:
        _close(got[0], ref[0], True)
        _close(got[1], ref[1], True)
        return
    same = (got[1] == ref[1]).all(1)
    assert float(same.double().mean()) >= 0.97
    _close(got[0][same], ref[0][same], False)


def _csr(rows_lists):
    ptr = torch.tensor([0] + [len(r) for r in rows_lists]).cumsum(0)
    return ptr.to(DEV), torch.tensor([x for r in rows_lists for x in r], dtype=torch.int64).to(DEV)


def _serving(sc, n_users, n_items, seed):
    """every serving output on seeded users / pairs that span all rows: {name: tensor(s)}"""
    g = _gen(seed)
    u = torch.randint(0, n_users, (200,), generator=g).to(DEV)
    i = torch.randint(0, n_items, (200,), generator=g).to(DEV)
    users = torch.arange(1, n_users, device=DEV)
    targets = _csr([(torch.randperm(n_items - 1, generator=g)[:3] + 1).tolist() for _ in range(n_users - 1)])
    out = {"feat_u": sc.user_feat, "feat_i": sc.item_feat, "score": sc.score_cached(u, i), "factors": sc.factors(),
           "recommend": sc.recommend(users, 10), "rank": sc.rank_items(users, targets),
           "evaluate": sc.evaluate(users, targets, ks=(5, 10)), "diverse": sc.recommend_diverse(users, 5)}
    if sc._explain is not None:
        explain = [sc.explain(u, i, m=4, return_maps=True)]
        if isinstance(sc.model, rbr_b200.DualAtt):
            explain.append(sc.explain(u, i, m=4, return_maps=True, attribution=True))
        out["explain"] = explain
        e = explain[-1]
        out["tokens"] = (sc.tokens_at("user", u, e.user.top_pos), sc.tokens_at("item", i, e.item.top_pos))
    return out


def _same_serving(a, b, exact):
    for key in ("feat_u", "feat_i", "score"):
        _close(a[key], b[key], exact)
    for x, y in zip(a["factors"], b["factors"]):
        _close(x, y, exact)
    _topk_close(a["recommend"], b["recommend"], exact)
    _topk_close(a["diverse"], b["diverse"], exact)
    if exact:
        for x, y in zip(a["rank"], b["rank"]):
            _close(x, y, True)
        assert a["evaluate"] == b["evaluate"]
    else:
        assert float((a["rank"][0] != b["rank"][0]).double().mean()) <= 0.02
        assert torch.equal(a["rank"][2], b["rank"][2])
        for k, v in a["evaluate"].items():
            assert abs(v - b["evaluate"][k]) <= 0.02 * max(1.0, abs(v)), k
    if "explain" in a:
        for ea, eb in zip(a["explain"], b["explain"]):
            _close(ea.pred, eb.pred, exact)
            for side in ("user", "item"):
                sa, sb = getattr(ea, side), getattr(eb, side)
                for f in ("text_total", "top_pos", "top_attr", "bottom_pos", "bottom_attr", "map", "review_weight",
                          "review_attr", "local_att", "global_att"):
                    x, y = getattr(sa, f), getattr(sb, f)
                    if exact or x is None or f in ("local_att", "global_att"):
                        _close(x, y, True)
                    elif not x.is_floating_point():
                        assert float((x != y).double().mean()) <= 0.05, f
                    else:
                        _close(x, y, False, tol=1e-3)
        if exact:
            for x, y in zip(a["tokens"], b["tokens"]):
                _close(x, y, True)


# ---------------------------------------------------------------------------------------------------------------------
# 1. cold start
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", CASES)
def test_cold_start_scores_equal_the_model(name):
    sc, data = _case(name)
    n_u, n_i = sc.user_feat.shape[0], sc.item_feat.shape[0]
    nu_docs, nu_rev = _new_docs(sc, data, "user", 5, 11)
    ni_docs, ni_rev = _new_docs(sc, data, "item", 4, 12)
    new_u = sc.add("user", nu_docs, **_kw(sc, "user", nu_rev))
    new_i = sc.add("item", ni_docs, **_kw(sc, "item", ni_rev))
    assert new_u.dtype == torch.int64 and new_u.tolist() == list(range(n_u, n_u + 5)) and new_u.is_contiguous()
    assert new_i.tolist() == list(range(n_i, n_i + 4))
    assert sc.user_feat.shape[0] == n_u + 5 and sc.item_feat.shape[0] == n_i + 4
    m = sc.model
    pad_u, pad_i = (0, 0) if isinstance(m, (rbr_b200.DualAtt, rbr_b200.SimpleSiamese)) else (m.fm.padding_idx,
                                                                                           m.fm.item_padding_idx)
    g = _gen(13)
    old_u, old_i = torch.randint(1, n_u, (6,), generator=g).to(DEV), torch.randint(1, n_i, (6,), generator=g).to(DEV)
    u = torch.cat([new_u.repeat_interleave(6)[:24], old_u.repeat(4), new_u[:4]])
    i = torch.cat([old_i.repeat(4), new_i.repeat_interleave(6), new_i])
    ud_all = torch.cat([data["user"][0], nu_docs])
    id_all = torch.cat([data["item"][0], ni_docs])
    u_mid = torch.where(u >= n_u, torch.full_like(u, pad_u), u)
    i_mid = torch.where(i >= n_i, torch.full_like(i, pad_i), i)
    u_rev = i_rev = None
    if name == "narre":
        u_rev, i_rev = torch.cat([data["user"][1], nu_rev])[u], torch.cat([data["item"][1], ni_rev])[i]
    ref = _forward(sc, data, ud_all[u], id_all[i], u_rev, i_rev, u_mid, i_mid)
    got = sc.score_cached(u, i)
    if name.startswith("cnn"):
        assert torch.equal(got, ref)
    else:
        assert float((got.double() - ref.double()).abs().max() / ref.double().abs().max()) <= 1e-5


# ---------------------------------------------------------------------------------------------------------------------
# 2. update = rebuild
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", CASES)
def test_update_equals_rebuild(name):
    sc, data = _case(name)
    n_u, n_i = sc.user_feat.shape[0], sc.item_feat.shape[0]
    before = {side: [None if t is None else t.clone() for t in data[side]] for side in data}
    g = _gen(21)
    for side, n, cnt in (("user", n_u, 9), ("item", n_i, 6)):
        ids = torch.randperm(n, generator=g)[:cnt].to(DEV)
        docs, rev = _new_docs(sc, data, side, cnt, 22 + cnt)
        sc.update(side, ids, docs, **_kw(sc, side, rev))
        # the caller's tensors are unchanged; the test's own copies take the change
        assert all(t is None or torch.equal(t, b) for t, b in zip(data[side], before[side]))
        data[side] = [t.clone() if t is not None else None for t in data[side]]
        data[side][0][ids] = docs.to(data[side][0].dtype)
        if rev is not None:
            data[side][1][ids] = rev
    fresh = _rebuild(sc, data)
    _same_serving(_serving(sc, n_u, n_i, 23), _serving(fresh, n_u, n_i, 23), name in EXACT)


# ---------------------------------------------------------------------------------------------------------------------
# 3. added items are served everywhere; the padding row stays apart
# ---------------------------------------------------------------------------------------------------------------------
def _factors64(sc, n_built):
    """(A, row_bias, B, col_bias) derived here in float64 from the cached features under the map: row r -> r for the built
    rows, the padding id for added ones"""
    m = sc.model
    p = X._p64(m)
    out = []
    for side, feat, n0 in (("user", sc.user_feat, n_built[0]), ("item", sc.item_feat, n_built[1])):
        pad = m.fm.padding_idx if side == "user" else m.fm.item_padding_idx
        rows = torch.arange(feat.shape[0], device=DEV)
        mid = torch.where(rows < n0, rows, torch.full_like(rows, pad))
        lat = feat.double() @ p[f"{side}_feat.W"] + p[f"{side}_feat.b"] + p[f"{side}_feat.ebd.weight"][mid]
        out += [lat, p[f"fm.{side}_bias.weight"][mid]]
    A, rb, B, cb = fm_factors(out[0], out[2], p["fm.h"], out[1], out[3], p["fm.g_bias"])
    return A.float(), rb.float(), B.float(), cb.float()


@pytest.mark.parametrize("name", ["cnn_fp32", "narre"])
def test_added_items_served_and_padding_apart(name):
    sc, data = _case(name)
    n_u, n_i = sc.user_feat.shape[0], sc.item_feat.shape[0]
    docs, rev = _new_docs(sc, data, "item", 8, 31)
    new_i = sc.add("item", docs, **_kw(sc, "item", rev))
    pad = sc.model.fm.item_padding_idx
    with torch.no_grad():                     # the padding id's bias lifts the added items, and cache row `pad`, to the top
        sc.model.fm.item_bias.weight[pad] += 50.0
    A, rb, B, cb = _factors64(sc, (n_u, n_i))
    users = torch.arange(1, n_u, device=DEV)
    cbp = cb.clone()
    cbp[pad] = float("-inf")
    k = 100
    got = sc.recommend(users, k)
    ref = ops.factor_topk(A[users], rb[users], B, cbp, k)
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    assert bool(torch.isin(got[1][:, :8], new_i).all())                # added items earn their places
    assert not bool((got[1] == pad).any())                             # only cache row `pad` is dropped
    every = sc.recommend(users, 256, exclude_padding=False)
    ref = ops.factor_topk(A[users], rb[users], B, cb, 256)
    assert torch.equal(every[0], ref[0]) and torch.equal(every[1], ref[1]) and bool((every[1] == pad).any())
    # ranks count the added items, and rank them
    targets = _csr([[int(new_i[r % 8]), 1 + r % (n_i - 1)] for r in range(users.numel())])
    ranks, scores, n_cand = sc.rank_items(users, targets)
    r_ref, s_ref, c_ref = ops.factor_rank(A[users], rb[users], B, cbp, targets)
    assert torch.equal(ranks, r_ref) and torch.equal(scores, s_ref)
    assert bool((n_cand == n_i + 8 - 1).all())
    assert bool((ranks[0::2] <= 8).all()) and bool((ranks[1::2] > 1).all())
    ev = sc.evaluate(users, targets, ks=(10,))
    assert ev["n_rows"] == users.numel()
    # diversified lists can pick them
    div = sc.recommend_diverse(users, 10, lam=0.7)
    assert bool(torch.isin(div[1][:, 0], new_i).all()) and not bool((div[1] == pad).any())
    with pytest.raises(ValueError):
        sc.rank_items(users[:1], _csr([[pad]]))


# ---------------------------------------------------------------------------------------------------------------------
# 4. no stale state
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["cnn_fp32", "narre", "datt"])
def test_interleaved_changes_leave_nothing_stale(name):
    sc, data = _case(name)
    n_u, n_i = sc.user_feat.shape[0], sc.item_feat.shape[0]
    added = {"user": [], "item": []}
    exact = name in EXACT
    m = sc.model

    def check(seed):
        adds = {side: (torch.cat([d for d, _ in lst]), None if lst[0][1] is None else torch.cat([r for _, r in lst]))
                for side, lst in added.items() if lst}
        fresh = _rebuild(sc, data, adds)
        nu, ni = sc.user_feat.shape[0], sc.item_feat.shape[0]
        assert (nu, ni) == (fresh.user_feat.shape[0], fresh.item_feat.shape[0])
        _same_serving(_serving(sc, nu, ni, seed), _serving(fresh, nu, ni, seed), exact)

    def add(side, n, seed):
        docs, rev = _new_docs(sc, data, side, n, seed)
        sc.add(side, docs, **_kw(sc, side, rev))
        added[side].append((docs, rev))

    def update(side, seed):
        g = _gen(seed)
        rows = torch.randperm(n_u if side == "user" else n_i, generator=g)[:5].to(DEV)
        docs, rev = _new_docs(sc, data, side, 5, seed)
        sc.update(side, rows, docs, **_kw(sc, side, rev))
        data[side] = [None if t is None else t.clone() for t in data[side]]
        data[side][0][rows] = docs.to(data[side][0].dtype)
        if rev is not None:
            data[side][1][rows] = rev

    check(40)
    add("user", 6, 41)
    check(42)
    update("item", 43)
    add("item", 5, 44)
    check(45)
    if name != "datt":                              # D-ATT has no head: its FC stack belongs to the encoder
        params = [m.item_feat.W, m.fm.h, m.fm.item_bias.weight]
        opt = torch.optim.SGD(params, lr=0.1)
        for p in params:
            p.grad = torch.randn_like(p) * 0.1
        opt.step()
        check(46)
    update("user", 47)
    add("user", 3, 48)
    check(49)


# ---------------------------------------------------------------------------------------------------------------------
# 5. the work follows the change
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["deepconn", "narre"])
def test_cost_follows_the_change(name, monkeypatch):
    U, I, L, R, T = 20000, 300, 60, 4, 30
    if name == "deepconn":
        m = rbr_b200.DeepCoNNpp(U, I, V, [3], 64, 100, 32, L, None, 0.0)
        m.load_state_dict(synth.deepconn_params(U, I, V, 64, 100, 32, (3,), seed=0))
        ud, idd = X._docs(U, L, 1), X._docs(I, L, 2)
        kw, per = {}, 1
    else:
        m = rbr_b200.NARRE(U, I, V, [3], 150, 64, 32, 32, R, T, 0.0, 0, 0, 0, None, "CNN")
        m.load_state_dict(synth.narre_params(U, I, V, 64, 150, 32, 32, (3,), seed=0))
        ud, idd = X._docs(U * R, T, 3).view(U, R, T), X._docs(I * R, T, 4).view(I, R, T)
        g = _gen(5)
        kw = {"user_rev_ids": torch.randint(0, I, (U, R), generator=g).to(DEV),
              "item_rev_ids": torch.randint(0, U, (I, R), generator=g).to(DEV)}
        per = R
    sc = PairScorer(m.cuda())
    sc.build_cache(ud, idd, **kw)
    sc.factors()
    docs_seen, rows_seen = [], []
    real_encode, real_lat = m.ngram.encode, sc._latent64
    monkeypatch.setattr(m.ngram, "encode", lambda emb, sides, *a, **k: docs_seen.append(sides[0].shape[0])
                        or real_encode(emb, sides, *a, **k))
    monkeypatch.setattr(sc, "_latent64", lambda name, feat, mids=None: rows_seen.append((name, feat.shape[0]))
                        or real_lat(name, feat, mids))
    new = ud[:8].flip(-1)
    rev = {"rev_ids": kw["user_rev_ids"][:8]} if kw else {}
    sc.update("user", torch.arange(100, 108, device=DEV), new, **rev)
    assert docs_seen == [8 * per]
    sc.factors()
    assert rows_seen == [("user", 8), ("item", 0)]
    docs_seen.clear()
    rows_seen.clear()
    sc.add("user", new, **rev)
    assert docs_seen == [8 * per]
    top = sc.recommend(torch.arange(U, U + 8, device=DEV), 10)
    assert rows_seen == [("user", 8), ("item", 0)] and top[1].shape == (8, 10)


# ---------------------------------------------------------------------------------------------------------------------
# 6. errors
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["cnn_fp32", "narre", "siamese_fused_g"])
def test_bad_input_is_refused_before_any_encoding(name, monkeypatch):
    sc, data = _case(name)
    called = []
    for fn in ("gather_rows", "datt_encode_side", "conv_window_contrib", "narre_feat_grads"):
        real = getattr(ops, fn)
        monkeypatch.setattr(ops, fn, lambda *a, _r=real, _f=fn, **k: called.append(_f) or _r(*a, **k))
    monkeypatch.setattr(ops.EncodeDocsFn, "apply", lambda *a, **k: called.append("encode"))
    monkeypatch.setattr(ops.MaskedAvgPoolFn, "apply", lambda *a, **k: called.append("pool"))
    n_u, n_i = sc.user_feat.shape[0], sc.item_feat.shape[0]
    docs, rev = _new_docs(sc, data, "user", 3, 51)
    kw = _kw(sc, "user", rev)
    bad = [lambda: sc.add("users", docs, **kw),
           lambda: sc.add("user", docs[:, :-1], **kw),
           lambda: sc.add("user", docs.cpu(), **kw),
           lambda: sc.update("user", torch.tensor([1, 1, 2], device=DEV), docs, **kw),
           lambda: sc.update("user", torch.tensor([1, 2, n_u], device=DEV), docs, **kw),
           lambda: PairScorer(sc.model).add("user", docs, **kw)]
    if name == "narre":
        bad += [lambda: sc.add("user", docs, rev_ids=torch.full_like(rev, X.I)),
                lambda: sc.add("user", docs, rev_ids=rev[:, :-1]),
                lambda: sc.add("user", docs)]
    for call in bad:
        with pytest.raises(ValueError):
            call()
    assert called == []
    assert (sc.user_feat.shape[0], sc.item_feat.shape[0]) == (n_u, n_i)
    empty = sc.add("item", docs[:0], **({"rev_ids": rev[:0]} if rev is not None else {}))
    assert empty.shape == (0,) and empty.dtype == torch.int64 and called == []
