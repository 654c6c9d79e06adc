"""K14 (ops.mmr_select) and PairScorer.recommend_diverse on the GPU: the greedy MMR re-rank against a float64 restatement on
small seeded caches of every served model, bit-exact invariants (lam = 1 is recommend, pool = k permutes it, rows are
independent of the batch, repeated calls agree), a bit-exact fp32 restatement where every similarity is exact, the edges, and
the launches in a profiler trace."""
import pytest
import torch

import rbr_b200
from rbr_b200 import ops, synth
from rbr_b200.inference import PairScorer, list_metrics

pytestmark = pytest.mark.gpu

DEV = "cuda"
U, I, V = 300, 257, 500


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _docs(n, L, seed):
    d = torch.randint(1, V, (n, L), generator=_gen(seed))
    d[:, L // 2 + seed % 7:] = 0
    return d.to(DEV)


def _deepconn(arch="CNN"):
    if arch == "CNN":
        m = rbr_b200.DeepCoNNpp(U, I, V, [3], 64, 100, 32, 60, None, 0.0)
        m.load_state_dict(synth.deepconn_params(U, I, V, 64, 100, 32, (3,), seed=0))
    else:
        m = rbr_b200.DeepCoNNpp(U, I, V, [3], 64, 64, 32, 60, None, 0.0, arch="HierPooling")
        m.load_state_dict(synth.deepconn_hier_params(U, I, V, 64, 64, 32, seed=0))
    sc = PairScorer(m.cuda())
    sc.build_cache(_docs(U, 60, 1), _docs(I, 60, 2))
    return sc


def _narre(R=4, T=30):
    m = rbr_b200.NARRE(U, I, V, [3], 150, 64, 32, 32, R, T, 0.0, 0, 0, 0, None, "CNN")
    m.load_state_dict(synth.narre_params(U, I, V, 64, 150, 32, 32, (3,), seed=0))
    sc = PairScorer(m.cuda())
    g = _gen(5)
    urev, irev = torch.randint(0, I, (U, R), generator=g).to(DEV), torch.randint(0, U, (I, R), generator=g).to(DEV)
    sc.build_cache(_docs(U * R, T, 3).view(U, R, T), _docs(I * R, T, 4).view(I, R, T), user_rev_ids=urev, item_rev_ids=irev)
    return sc


def _datt(L=64):
    m = rbr_b200.DualAtt(V, L, 5, 200, 100, 100, 500, 50, 0.0, None)
    m.load_state_dict(synth.dual_att_params(V, L, 5, 200, 100, 100, 500, 50, seed=0))
    sc = PairScorer(m.cuda())
    sc.build_cache(_docs(U, L, 6), _docs(I, L, 7))
    return sc


def _siamese(ub, R=3, T=7, E=24, K=8):
    m = rbr_b200.SimpleSiamese(E, K, V, U, I, None, False, 0.0, 0.0, 0.0, ub, False)
    m.load_state_dict(synth.simple_siamese_params(U, I, V, E, K, ub, False, seed=0))
    sc = PairScorer(m.cuda())
    sc.build_cache(_docs(U * R, T, 8).view(U, R, T), _docs(I * R, T, 9).view(I, R, T))
    return sc


MODELS = {"deepconn": _deepconn, "deepconn_hier": lambda: _deepconn("HierPooling"), "narre": _narre, "dual_att": _datt,
          "siamese": lambda: _siamese(True), "siamese_nobias": lambda: _siamese(False)}
_CACHE = {}


def _scorer(name):
    if name not in _CACHE:
        _CACHE[name] = MODELS[name]()
    return _CACHE[name]


# ---------------------------------------------------------------------------------------------------------------------
# restatements of the greedy step
# ---------------------------------------------------------------------------------------------------------------------
def _elig(ps, pi, n_items):
    return (pi >= 0) & (pi < n_items) & torch.isfinite(ps)


def greedy(ps, pi, vecs, k, lam, n_items, dtype):
    """MMR on pools ps / pi [n, P] in `dtype`: float64 (the reference) or float32 (each operation rounded as the kernel's;
    the sims are torch's, so they match the kernel's bits only where every product and sum is exact).
    Returns (items [n, k] with -1 tails, positions [n, k], per-step objectives [k, n, P] with -inf where not live)."""
    n, P = ps.shape
    inf = float("inf")
    elig = _elig(ps, pi, n_items)
    s = ps.to(dtype)
    lo = torch.where(elig, s, inf).amin(1, keepdim=True)
    hi = torch.where(elig, s, -inf).amax(1, keepdim=True)
    rel = torch.where(hi == lo, torch.ones_like(s), (s - lo) / (hi - lo))
    lam_t = torch.tensor(lam, dtype=torch.float32).to(dtype)
    oml = 1 - torch.tensor(lam, dtype=torch.float32).to(dtype)
    Vr = vecs.to(dtype)[pi.clamp(0, vecs.shape[0] - 1)]
    live = elig.clone()
    maxsim = torch.full_like(s, -inf)
    pos = torch.arange(P, device=ps.device).expand(n, P)
    rows = torch.arange(n, device=ps.device)
    items = torch.full((n, k), -1, dtype=torch.int64, device=ps.device)
    picks = torch.full((n, k), -1, dtype=torch.int64, device=ps.device)
    objs = []
    for t in range(k):
        obj = rel if t == 0 else lam_t * rel - oml * maxsim
        obj = torch.where(live, torch.where(obj == 0, torch.zeros_like(obj), obj), torch.full_like(obj, -inf))
        objs.append(obj)
        best = obj.amax(1, keepdim=True)
        cand = live & (obj == best)
        has = cand.any(1)
        p = torch.where(cand, pos, P).amin(1).clamp_max(P - 1)
        items[:, t] = torch.where(has, pi[rows, p], -1)
        picks[:, t] = torch.where(has, p, -1)
        live[rows[has], p[has]] = False
        sim = (Vr * Vr[rows, p].unsqueeze(1)).sum(-1)
        maxsim = torch.maximum(maxsim, sim)
    return items, picks, torch.stack(objs)


def check_against_reference(scores, items, ps, pi, vecs, k, lam, n_items, tol=1e-5):
    """Lists equal the float64 reference's up to the first step whose best and second-best objectives lie within tol; at
    that step the pick's objective is within tol of the best; >= 99 % of rows equal end to end.  Scores are the pool's."""
    ref_items, _, objs = greedy(ps, pi, vecs, k, lam, n_items, torch.float64)
    n = ps.shape[0]
    top2 = objs.topk(2, dim=2).values if ps.shape[1] > 1 else torch.cat([objs, torch.full_like(objs, -float("inf"))], 2)
    near = (top2[..., 0] - top2[..., 1] <= tol) & torch.isfinite(top2[..., 1])          # [k, n]
    first = torch.where(near.any(0), near.float().argmax(0), torch.full((n,), k, device=ps.device))
    steps = torch.arange(k, device=ps.device).view(1, -1)
    before = steps < first.view(-1, 1)
    assert torch.equal(torch.where(before, items, 0), torch.where(before, ref_items, 0))
    amb = first < k
    if bool(amb.any()):
        r = torch.nonzero(amb).view(-1)
        t = first[r]
        it = items[r, t]
        p = (pi[r] == it.view(-1, 1)).float().argmax(1)
        got = objs[t, r, p]
        assert bool((got >= top2[t, r, 0] - tol).all())
    same = (items == ref_items).all(1).float().mean()
    assert float(same) >= 0.99, float(same)
    # the scores are the pool's scores of the picked items
    pos = torch.where(items >= 0, (pi.unsqueeze(1) == items.unsqueeze(2)).float().argmax(2), 0)
    want = torch.where(items >= 0, ps.gather(1, pos), torch.full_like(scores, -float("inf")))
    assert torch.equal(scores, want)
    return float(same)


# ---------------------------------------------------------------------------------------------------------------------
# through the models
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(MODELS))
def test_against_float64_reference(name):
    sc = _scorer(name)
    u_ids = torch.arange(U, device=DEV)
    vecs = ops.unit_rows(sc.item_feat)
    for k, pool, lam in ((10, None, 0.5), (20, 256, 0.3), (5, 64, 0.9), (8, 32, 0.0)):
        s, i = sc.recommend_diverse(u_ids, k, lam=lam, pool=pool)
        ps, pi = sc.recommend(u_ids, pool or 4 * k)
        check_against_reference(s, i, ps, pi, vecs, k, lam, I)
        assert not bool((i == 0).any())


@pytest.mark.parametrize("name", list(MODELS))
def test_bit_exact_invariants(name):
    sc = _scorer(name)
    u_ids = torch.randint(0, U, (U,), generator=_gen(11)).to(DEV)
    for k in (1, 10, 64):
        rs, ri = sc.recommend(u_ids, k)
        s1, i1 = sc.recommend_diverse(u_ids, k, lam=1.0)
        assert torch.equal(s1, rs) and torch.equal(i1, ri)
        s2, i2 = sc.recommend_diverse(u_ids, k, lam=0.2, pool=k)
        order = torch.sort(i2, dim=1).indices
        assert torch.equal(torch.sort(i2, dim=1).values, torch.sort(ri, dim=1).values)
        assert torch.equal(s2.gather(1, order), rs.gather(1, torch.sort(ri, dim=1).indices))
    s, i = sc.recommend_diverse(u_ids, 10, lam=0.5)
    s_again, i_again = sc.recommend_diverse(u_ids, 10, lam=0.5)
    assert torch.equal(s, s_again) and torch.equal(i, i_again)
    perm = torch.randperm(U, generator=_gen(12)).to(DEV)
    sp, ip = sc.recommend_diverse(u_ids[perm], 10, lam=0.5)
    assert torch.equal(sp, s[perm]) and torch.equal(ip, i[perm])
    for chunk in (1, 7, 128):
        parts = [sc.recommend_diverse(u_ids[lo:lo + chunk], 10, lam=0.5) for lo in range(0, U, chunk)]
        assert torch.equal(torch.cat([p[0] for p in parts]), s) and torch.equal(torch.cat([p[1] for p in parts]), i)


def test_exclusions_short_rows_and_padding():
    sc = _scorer("deepconn")
    n, k = 60, 10
    u_ids = torch.arange(1, n + 1, device=DEV)
    g = _gen(13)
    lists = []
    for r in range(n):
        if r % 5 == 0:                               # all but 6 items excluded: a (-inf, -1) tail
            keep = set(torch.randperm(I - 1, generator=g)[:6].add(1).tolist())
            lists.append([j for j in range(I) if j not in keep])
        else:
            lists.append(torch.randint(0, I, (int(torch.randint(0, 60, (1,), generator=g)),), generator=g).tolist())
    ptr = torch.tensor([0] + torch.cumsum(torch.tensor([len(x) for x in lists]), 0).tolist(), device=DEV)
    idx = torch.tensor([j for x in lists for j in x], dtype=torch.int64, device=DEV)
    s, i = sc.recommend_diverse(u_ids, k, lam=0.5, exclude=(ptr, idx))
    ps, pi = sc.recommend(u_ids, 4 * k, exclude=(ptr, idx))
    s_ref, i_ref = ops.mmr_select(ps, pi, ops.unit_rows(sc.item_feat), k, 0.5)
    assert torch.equal(s, s_ref) and torch.equal(i, i_ref)
    check_against_reference(s, i, ps, pi, ops.unit_rows(sc.item_feat), k, 0.5, I)
    for r in range(n):
        got = [j for j in i[r].tolist() if j >= 0]
        assert not set(got) & set(lists[r])
        if r % 5 == 0:
            assert len(got) == 6 and i[r, 6:].eq(-1).all() and torch.isneginf(s[r, 6:]).all()
    # the padding item: left out by default, a candidate with exclude_padding=False
    s0, i0 = sc.recommend_diverse(torch.arange(U, device=DEV), 256, lam=0.5, pool=256)
    s1, i1 = sc.recommend_diverse(torch.arange(U, device=DEV), 256, lam=0.5, pool=256, exclude_padding=False)
    assert bool((i0 >= 1).all()) and bool((i1 == 0).any())                 # 256 slots, 256 eligible items
    ps, pi = sc.recommend(torch.arange(U, device=DEV), 256, exclude_padding=False)
    check_against_reference(s1, i1, ps, pi, ops.unit_rows(sc.item_feat), 256, 0.5, I)


def test_item_vecs_zero_rows_and_factors():
    sc = _scorer("dual_att")
    u_ids = torch.arange(U, device=DEV)
    k = 10
    ps, pi = sc.recommend(u_ids, 40)
    # an all-zero vector for the most recommended item: sim 0 to everything
    top = torch.mode(pi[:, 0]).values
    vecs = sc.item_feat.clone()
    vecs[top] = 0
    s, i = sc.recommend_diverse(u_ids, k, item_vecs=vecs)
    unit = ops.unit_rows(vecs)
    assert bool((unit[top] == 0).all())
    check_against_reference(s, i, ps, pi, unit, k, 0.5, I)
    # the cache follows in-place changes of the passed tensor
    vecs[top] = 1.0
    s2, i2 = sc.recommend_diverse(u_ids, k, item_vecs=vecs)
    check_against_reference(s2, i2, ps, pi, ops.unit_rows(vecs), k, 0.5, I)
    # the factor matrix B of another model
    sc2 = _scorer("narre")
    B = sc2.factors()[2]
    s3, i3 = sc2.recommend_diverse(u_ids, k, item_vecs=B)
    ps3, pi3 = sc2.recommend(u_ids, 40)
    check_against_reference(s3, i3, ps3, pi3, ops.unit_rows(B), k, 0.5, I)
    d = list_metrics(i3, B, I - 1)
    r = list_metrics(pi3[:, :k], B, I - 1)
    assert d["ild"] >= r["ild"] and d["n_rows"] == r["n_rows"] == U


def test_zero_users_and_errors():
    sc = _scorer("deepconn")
    s, i = sc.recommend_diverse(torch.zeros(0, dtype=torch.int64, device=DEV), 10)
    assert s.shape == (0, 10) and i.shape == (0, 10) and i.dtype == torch.int64
    u = torch.arange(5, device=DEV)
    for kw in (dict(k=0), dict(k=257), dict(k=10, pool=9), dict(k=10, pool=257), dict(k=10, lam=1.5), dict(k=10, lam=-0.1),
               dict(k=10, item_vecs=torch.zeros(I - 1, 4, device=DEV)), dict(k=10, item_vecs=torch.zeros(I, 513, device=DEV))):
        with pytest.raises(ValueError):
            sc.recommend_diverse(u, **kw)
    ps, pi = sc.recommend(u, 20)
    vecs = ops.unit_rows(sc.item_feat)
    with pytest.raises(TypeError):
        ops.mmr_select(ps.double(), pi, vecs, 10, 0.5)
    with pytest.raises(ValueError):
        ops.mmr_select(ps, pi[:, :10], vecs, 10, 0.5)
    with pytest.raises(RuntimeError):
        ops.mmr_select(ps, pi, vecs.cpu(), 10, 0.5)


# ---------------------------------------------------------------------------------------------------------------------
# ops.mmr_select on synthetic pools: bit-exact against the fp32 restatement where every similarity is exact
# ---------------------------------------------------------------------------------------------------------------------
def _exact_pools(n, P, n_items, dim, seed):
    """Vectors with entries in {-1, -7/8, ..., 1} (every product and partial sum exact in fp32, so torch's sims are the
    kernel's bits), duplicated vectors and tied scores, and ineligible slots: -1, ids >= n_items, -inf and NaN scores."""
    g = _gen(seed)
    vecs = torch.randint(-8, 9, (n_items + 5, dim), generator=g).float() / 8
    vecs[3] = vecs[4]
    vecs[7] = 0
    pi = torch.stack([torch.randperm(n_items + 5, generator=g)[:P] for _ in range(n)])
    ps = torch.randint(-20, 20, (n, P), generator=g).float() / 4              # many exact ties
    ps = torch.sort(ps, dim=1, descending=True).values
    ps[1] = 2.0                                                             # one row of equal scores: rel = 1
    pi[2, P // 2:] = -1
    ps[2, P // 2:] = -float("inf")
    ps[3, 0] = float("nan")
    ps[4, -1] = -float("inf")
    return ps.to(DEV), pi.to(DEV), vecs[:n_items].to(DEV)


@pytest.mark.parametrize("dim", [1, 3, 16, 300, 512])
@pytest.mark.parametrize("P,k", [(256, 256), (256, 10), (10, 10), (40, 10), (1, 1)])
def test_bit_exact_fp32_restatement(dim, P, k):
    n, n_items = 64, 300
    ps, pi, vecs = _exact_pools(n, P, n_items, dim, seed=dim * 1000 + P + k)
    for lam in (0.0, 0.3, 0.5, 1.0):
        s, i = ops.mmr_select(ps, pi, vecs, k, lam)
        ref_i, ref_p, _ = greedy(ps, pi, vecs, k, lam, n_items, torch.float32)
        assert torch.equal(i, ref_i), (lam, torch.nonzero((i != ref_i).any(1)).view(-1)[:5])
        want = torch.where(ref_p >= 0, ps.gather(1, ref_p.clamp_min(0)), torch.full_like(s, -float("inf")))
        assert torch.equal(s, want)


def test_ids_outside_the_table_are_ineligible():
    ps = torch.tensor([[3.0, 2.0, 1.0, 0.0]], device=DEV)
    pi = torch.tensor([[5, 1, -3, 0]], device=DEV)
    vecs = torch.eye(4, device=DEV)
    s, i = ops.mmr_select(ps, pi, vecs, 4, 0.5)
    assert i.tolist() == [[1, 0, -1, -1]] and s[0, :2].tolist() == [2.0, 0.0] and torch.isneginf(s[0, 2:]).all()


def test_launches_in_profiler_trace():
    from torch.profiler import ProfilerActivity, profile
    sc = _scorer("deepconn")
    u_ids = torch.arange(U, device=DEV)
    sc.recommend_diverse(u_ids, 50, lam=0.5)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sc.recommend_diverse(u_ids, 50, lam=0.5)
        torch.cuda.synchronize()
    kernels = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
               and not e.name.startswith(("Memcpy", "Memset"))]
    assert sum("mmr_select_kernel" in n for n in kernels) == 1, kernels
    assert any("factor_topk_kernel" in n for n in kernels), kernels
    assert any("factor_topk_merge_kernel" in n for n in kernels), kernels
    assert len(kernels) < 20, kernels            # no per-step loop: 50 steps would launch hundreds
