"""K10 (ops.factor_topk) and PairScorer.recommend on the GPU: per-row top-k over a factorised score matrix against a
float64 reference, and the NARRE / D-ATT feature caches against the models' own eval forward."""
import pytest
import torch

import rbr_b200
from rbr_b200 import ops, synth
from rbr_b200.inference import PairScorer

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _ref_scores(A, rb, B, cb, excl=None):
    """float64 scores [n, I] with excluded items at -inf (excl: list of per-row iterables)."""
    S = A.double() @ B.double().T
    if rb is not None:
        S += rb.double().view(-1, 1)
    if cb is not None:
        S += cb.double().view(1, -1)
    if excl is not None:
        for r, ex in enumerate(excl):
            if len(ex):
                S[r, torch.as_tensor(sorted(set(ex)), device=S.device)] = float("-inf")
    return S


def check_topk(scores, items, S, k, exact_rows=True):
    """(a)-(e) of the reference comparison; S = float64 scores with ineligible items at -inf (NaN rows count as ineligible)."""
    n, I = S.shape
    S = torch.where(torch.isnan(S), torch.full_like(S, float("-inf")), S)
    fin = torch.isfinite(S)
    scale = torch.where(fin, S.abs(), torch.zeros_like(S)).amax(1).clamp_min(1e-30)
    n_elig = fin.sum(1)
    assert scores.shape == (n, k) and items.shape == (n, k)
    valid = items >= 0
    # the -1 / -inf tail is exactly the slots past the eligible count
    assert torch.equal(valid.sum(1), torch.clamp(n_elig, max=k))
    assert bool((valid[:, :-1] | ~valid[:, 1:]).all())
    assert bool(torch.isneginf(scores[~valid]).all())
    it = items.clamp_min(0)
    # (a) in range, eligible, distinct
    assert bool((items[valid] < I).all())
    got64 = S.gather(1, it)
    assert bool(torch.isfinite(got64[valid]).all()), "returned an excluded / ineligible item"
    srt = torch.sort(torch.where(valid, items, torch.full_like(items, -1 - I)), 1).values
    assert bool(((srt[:, 1:] != srt[:, :-1]) | (srt[:, 1:] < 0)).all()), "duplicate items"
    # (b) score accuracy
    err = ((scores.double() - got64).abs() / scale.view(-1, 1))[valid]
    assert float(err.max()) < 1e-5 if err.numel() else True
    # (c) order: non-increasing, exact ties by ascending id
    s0, s1 = scores[:, :-1], scores[:, 1:]
    both = valid[:, :-1] & valid[:, 1:]
    assert bool((s0 >= s1)[both].all())
    tie = both & (s0 == s1)
    assert bool((items[:, :-1] < items[:, 1:])[tie].all())
    # (d) nothing left out beats the k-th returned item by more than 2e-5 relative
    last = valid.sum(1) - 1
    has = last >= 0
    kth = torch.where(has, got64.gather(1, last.clamp_min(0).view(-1, 1)).view(-1), torch.full_like(scale, float("inf")))
    rest = S.clone()
    rest.scatter_(1, it, float("-inf"))
    full = n_elig >= k
    over = (rest.amax(1) - kth) / scale
    assert float(over[full & has].max()) <= 2e-5 if bool((full & has).any()) else True
    # (e) rows whose float64 gaps around the top k+1 are > 1e-4 relative: exact items, in order
    if exact_rows:
        ref_s, ref_i = torch.sort(S, dim=1, descending=True, stable=True)
        kk = min(k + 1, I)
        top = ref_s[:, :kk]
        gaps = (top[:, :-1] - top[:, 1:]) / scale.view(-1, 1)
        gaps = torch.where(torch.isfinite(gaps), gaps, torch.full_like(gaps, float("inf")))
        clean = (gaps.amin(1) > 1e-4) if kk > 1 else torch.ones(n, dtype=torch.bool, device=S.device)
        m = min(k, I)
        ref_items = torch.where(torch.isfinite(ref_s[:, :m]), ref_i[:, :m], torch.full_like(ref_i[:, :m], -1))
        assert torch.equal(items[clean][:, :m], ref_items[clean])
        return int(clean.sum())
    return 0


def _rand(n, d, seed, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(n, d, generator=g, dtype=torch.float64) * scale).float().to(DEV)


@pytest.mark.parametrize("n_rows,n_items,dim,k", [
    (1, 1, 1, 1), (127, 255, 50, 10), (128, 256, 64, 100), (129, 257, 65, 256), (1, 12001, 512, 10),
    (300, 12001, 256, 100), (129, 255, 1, 256), (20000, 12001, 64, 10), (1000, 12001, 64, 256),
])
def test_factor_topk_shapes(n_rows, n_items, dim, k):
    A, B = _rand(n_rows, dim, 1), _rand(n_items, dim, 2)
    rb, cb = _rand(n_rows, 1, 3).view(-1), _rand(n_items, 1, 4).view(-1)
    scores, items = ops.factor_topk(A, rb, B, cb, k)
    S = _ref_scores(A, rb, B, cb)
    for lo in range(0, n_rows, 4096):
        check_topk(scores[lo:lo + 4096], items[lo:lo + 4096], S[lo:lo + 4096], k)
    slices = ops.factor_topk_slices(n_rows, n_items, dim, k)
    assert slices >= 1
    if (n_rows, n_items) == (20000, 12001):
        assert slices > 1                    # 157 row tiles: the items are split across CTAs
    if n_items <= 256:
        assert slices == 1


def test_factor_topk_ties_across_slices_and_determinism():
    n_items, dim, k = 12001, 64, 10
    A, B = _rand(200, dim, 5).abs(), _rand(n_items, dim, 6, 0.1)
    best = torch.full((1, dim), 3.0, device=DEV)       # a row every (positive) query scores far above the rest
    for j in (3, 300, n_items - 2):
        B[j] = best
    assert ops.factor_topk_slices(200, n_items, dim, k) > 1 or ops.factor_topk_slices(20000, n_items, dim, k) > 1
    for rows in (200, 20000):
        Ar = A.repeat((rows + 199) // 200, 1)[:rows].contiguous()
        s1, i1 = ops.factor_topk(Ar, None, B, None, k)
        s2, i2 = ops.factor_topk(Ar, None, B, None, k)
        assert torch.equal(s1, s2) and torch.equal(i1, i2)
        assert bool(((s1[:, 0] == s1[:, 1]) & (s1[:, 1] == s1[:, 2])).all())
        assert bool((i1[:, :3] == torch.tensor([3, 300, n_items - 2], device=DEV)).all())
        check_topk(s1[:2000], i1[:2000], _ref_scores(Ar[:2000], None, B, None), k, exact_rows=False)


def test_factor_topk_exclusions():
    n_rows, n_items, dim, k = 300, 2000, 64, 10
    A, B = _rand(n_rows, dim, 7), _rand(n_items, dim, 8)
    g = torch.Generator().manual_seed(9)
    lists = []
    for r in range(n_rows):
        if r % 3 == 0:
            lists.append([])
        elif r == 1:
            keep = {5, 700, 1999}
            lists.append([i for i in range(n_items) if i not in keep][::-1])
        else:
            ex = torch.randint(0, n_items, (int(torch.randint(1, 80, (1,), generator=g)),), generator=g).tolist()
            lists.append(ex + ex[:3])                  # unsorted, with duplicates
    ptr = torch.tensor([0] + torch.cumsum(torch.tensor([len(x) for x in lists]), 0).tolist(), device=DEV)
    idx = torch.tensor([i for x in lists for i in x], dtype=torch.int64, device=DEV)
    scores, items = ops.factor_topk(A, None, B, None, k, exclude=(ptr, idx))
    check_topk(scores, items, _ref_scores(A, None, B, None, lists), k)
    assert sorted(items[1, :3].tolist()) == [5, 700, 1999] and items[1, 3:].eq(-1).all()
    empty = (torch.zeros(n_rows + 1, dtype=torch.int64, device=DEV), torch.zeros(0, dtype=torch.int64, device=DEV))
    s0, i0 = ops.factor_topk(A, None, B, None, k)
    s1, i1 = ops.factor_topk(A, None, B, None, k, exclude=empty)
    assert torch.equal(s0, s1) and torch.equal(i0, i1)


def test_factor_topk_biases_and_nan():
    n_rows, n_items, dim, k = 129, 3000, 50, 100
    A, B = _rand(n_rows, dim, 10), _rand(n_items, dim, 11)
    rb, cb = _rand(n_rows, 1, 12).view(-1), _rand(n_items, 1, 13).view(-1)
    for r_, c_ in ((None, None), (rb, None), (None, cb), (rb, cb)):
        s, i = ops.factor_topk(A, r_, B, c_, k)
        check_topk(s, i, _ref_scores(A, r_, B, c_), k)
    Bn = B.clone()
    Bn[17] = float("nan")
    Bn[18] = 100.0                                    # would top every row with positive sum
    s, i = ops.factor_topk(A, rb, Bn, cb, k)
    assert not bool((i == 17).any())
    check_topk(s, i, _ref_scores(A, rb, Bn, cb), k)


def test_factor_topk_memory():
    n_rows, n_items, dim, k = 20000, 12000, 64, 100
    A, B = _rand(n_rows, dim, 14), _rand(n_items, dim, 15)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    s, i = ops.factor_topk(A, None, B, None, k)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak < n_rows * n_items * 4 / 4, peak
    check_topk(s[:1000], i[:1000], _ref_scores(A[:1000], None, B, None), k)


def test_factor_topk_errors():
    A, B = _rand(4, 8, 1), _rand(10, 8, 2)
    with pytest.raises(RuntimeError):
        ops.factor_topk(A.cpu(), None, B, None, 3)
    with pytest.raises(ValueError):
        ops.factor_topk(A.double(), None, B, None, 3)
    for k in (0, 257):
        with pytest.raises(ValueError):
            ops.factor_topk(A, None, B, None, k)
    with pytest.raises(ValueError):
        ops.factor_topk(_rand(4, 513, 1), None, _rand(10, 513, 2), None, 3)
    with pytest.raises(ValueError):
        ops.factor_topk(A, None, B, None, 3, exclude=(torch.tensor([0, 1, 1, 1, 1], device=DEV),
                                                      torch.tensor([10], device=DEV)))


# ---------------------------------------------------------------------------------------------------------------------
# through the models
# ---------------------------------------------------------------------------------------------------------------------
U, I, V, E, HID, K = 300, 257, 500, 64, 100, 32


def _docs(n, L, seed):
    g = torch.Generator().manual_seed(seed)
    d = torch.randint(1, V, (n, L), generator=g)
    d[:, L // 2 + seed % 7:] = 0
    return d.to(DEV)


def _deepconn(prec):
    m = rbr_b200.DeepCoNNpp(U, I, V, [3], E, HID, K, 60, None, 0.0, precision=prec)
    m.load_state_dict(synth.deepconn_params(U, I, V, E, HID, K, (3,), seed=0))
    sc = PairScorer(m.cuda())
    ud, idd = _docs(U, 60, 1), _docs(I, 60, 2)
    sc.build_cache(ud, idd)
    return sc, (ud, idd)


def _narre(prec, R=10, T=60):
    m = rbr_b200.NARRE(U, I, V, [3], 150, E, 32, K, R, T, 0.0, 0, 0, 0, None, "CNN", precision=prec)
    m.load_state_dict(synth.narre_params(U, I, V, E, 150, 32, K, (3,), seed=0))
    sc = PairScorer(m.cuda())
    ud, idd = _docs(U * R, T, 3).view(U, R, T), _docs(I * R, T, 4).view(I, R, T)
    g = torch.Generator().manual_seed(5)
    urev, irev = torch.randint(0, I, (U, R), generator=g).to(DEV), torch.randint(0, U, (I, R), generator=g).to(DEV)
    sc.build_cache(ud, idd, user_rev_ids=urev, item_rev_ids=irev)
    return sc, (ud, idd, urev, irev)


def _datt(prec, L=120):
    m = rbr_b200.DualAtt(V, L, 5, 200, 100, 100, 500, 50, 0.0, None, precision=prec)
    m.load_state_dict(synth.dual_att_params(V, L, 5, 200, 100, 100, 500, 50, seed=0))
    sc = PairScorer(m.cuda())
    ud, idd = _docs(U, L, 6), _docs(I, L, 7)
    sc.build_cache(ud, idd)
    return sc, (ud, idd)


def _forward(sc, inputs, u, i):
    """the model's own eval forward on the pairs' full inputs"""
    m = sc.model
    with torch.no_grad():
        if isinstance(m, rbr_b200.NARRE):
            ud, idd, urev, irev = inputs
            return m(ud[u], idd[i], None, None, u, i, urev[u], irev[i])[0]
        if isinstance(m, rbr_b200.DualAtt):
            return m(inputs[0][u], inputs[1][i])
        return m(inputs[0][u], inputs[1][i], None, None, u, i)


def _pairs(n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, U, (n,), generator=g).to(DEV), torch.randint(0, I, (n,), generator=g).to(DEV)


MODELS = {"deepconn": _deepconn, "narre": _narre, "dual_att": _datt}


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("name", ["narre", "dual_att"])
def test_score_cached_matches_forward(name, prec):
    sc, inputs = MODELS[name](prec)
    u, i = _pairs(512, 1)
    ref = _forward(sc, inputs, u, i)
    got = sc.score_cached(u, i)
    assert float((got.double() - ref.double()).abs().max() / ref.double().abs().max()) < 1e-5


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("name", ["deepconn", "narre", "dual_att"])
def test_recommend(name, prec):
    sc, inputs = MODELS[name](prec)
    k = 10
    u_ids = torch.arange(1, U, device=DEV)
    scores, items = sc.recommend(u_ids, k)
    A, rb, B, cb = sc.factors()
    cbp = torch.zeros(I, device=DEV) if cb is None else cb.clone()
    cbp[0] = float("-inf")
    S = _ref_scores(A[u_ids], None if rb is None else rb[u_ids], B, cbp)
    check_topk(scores, items, S, k)
    assert not bool((items == 0).any())
    # the scores are the model's: score_cached and the eval forward on the returned pairs
    uu = u_ids.view(-1, 1).expand(-1, k).reshape(-1)
    ii = items.reshape(-1)
    sc_c = sc.score_cached(uu, ii)
    scale = sc_c.double().abs().max()
    assert float((scores.reshape(-1).double() - sc_c.double()).abs().max() / scale) < 1e-5
    sel = torch.arange(0, uu.numel(), 37, device=DEV)
    fwd = _forward(sc, inputs, uu[sel], ii[sel])
    assert float((scores.reshape(-1)[sel].double() - fwd.double()).abs().max() / scale) < 1e-5
    # the padding item comes back when allowed: 256 of the 257 items
    s2, i2 = sc.recommend(u_ids, 256)
    s3, i3 = sc.recommend(u_ids, 256, exclude_padding=False)
    assert bool((i2 >= 1).all())
    assert bool((i3 == 0).any())


@pytest.mark.parametrize("name", ["deepconn", "narre"])
def test_recommend_follows_head_parameters(name):
    sc, _ = MODELS[name]("fp32")
    u_ids = torch.arange(1, 100, device=DEV)
    s0, i0 = sc.recommend(u_ids, 10)
    m = sc.model
    opt = torch.optim.SGD([m.item_feat.W, m.fm.h, m.fm.item_bias.weight], lr=0.5)
    for p in opt.param_groups[0]["params"]:
        p.grad = torch.randn_like(p)
    opt.step()
    s1, i1 = sc.recommend(u_ids, 10)
    assert not torch.equal(s0, s1)
    uu = u_ids.view(-1, 1).expand(-1, 10).reshape(-1)
    sc_c = sc.score_cached(uu, i1.reshape(-1))
    assert float((s1.reshape(-1).double() - sc_c.double()).abs().max() / sc_c.double().abs().max()) < 1e-5
