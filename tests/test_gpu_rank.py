"""K11 (ops.factor_rank) and PairScorer.rank_items / evaluate on the GPU: exact full-catalogue ranks of target items against
a float64 reference, bit-consistency with K10 (factor_topk / recommend), special values, and the three models."""
import pytest
import torch

from rbr_b200 import ops
from rbr_b200.inference import ranking_metrics
from test_gpu_recommend import MODELS, U, I, _ref_scores, _rand

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _csr(lists):
    ptr = torch.tensor([0] + torch.cumsum(torch.tensor([len(x) for x in lists], dtype=torch.int64), 0).tolist(), device=DEV)
    return ptr, torch.tensor([i for x in lists for i in x], dtype=torch.int64, device=DEV)


def _lists(n_rows, n_items, per_row, seed, excl=None):
    """per_row distinct targets per row (fewer when the row has fewer eligible items), in random order."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for r in range(n_rows):
        perm = torch.randperm(n_items, generator=g)
        if excl is not None and len(excl[r]):
            ex = torch.zeros(n_items, dtype=torch.bool)
            ex[torch.tensor(excl[r])] = True
            perm = perm[~ex[perm]]
        out.append(perm[:per_row].tolist())
    return out


def _excl_lists(n_rows, n_items, seed):
    g = torch.Generator().manual_seed(seed)
    out = []
    for r in range(n_rows):
        if r % 3 == 0:
            out.append([])
            continue
        ex = torch.randint(0, n_items, (int(torch.randint(1, 60, (1,), generator=g)),), generator=g).tolist()
        out.append(ex + ex[:3])                          # unsorted, with duplicates
    return out


def check_ranks(S, t_ptr, t_idx, ranks, scores, tol=1e-5):
    """Each rank lies between the float64 counts with a tol-relative margin on either side (so it is exact where no other
    eligible item is within the margin); scores within tol of the row's largest |score|.  S: float64 scores with excluded
    items at -inf.  Returns the fraction of targets whose bounds are tight."""
    S = torch.where(torch.isnan(S), torch.full_like(S, float("-inf")), S)
    fin = torch.isfinite(S)
    scale = torch.where(fin, S.abs(), torch.zeros_like(S)).amax(1).clamp_min(1e-30)
    rows = torch.repeat_interleave(torch.arange(S.shape[0], device=DEV), t_ptr[1:] - t_ptr[:-1])
    st = S[rows, t_idx]
    ok = torch.isfinite(st)
    assert torch.equal(ranks[~ok], torch.full_like(ranks[~ok], -1)), "a NaN / -inf target must have rank -1"
    tight = 0
    for lo in range(0, rows.numel(), 4096):
        r, s, rk, sc = rows[lo:lo + 4096], st[lo:lo + 4096], ranks[lo:lo + 4096], scores[lo:lo + 4096]
        v = torch.isfinite(s)
        r, s, rk, sc = r[v], s[v], rk[v], sc[v]
        Sr, m = S[r], (tol * scale[r]).view(-1, 1)
        hi = (Sr >= s.view(-1, 1) - m).sum(1)
        low = (Sr > s.view(-1, 1) + m).sum(1) + 1
        assert bool(((rk >= low) & (rk <= hi)).all()), "rank outside the float64 bounds"
        if s.numel():
            assert float(((sc.double() - s).abs() / scale[r]).max()) <= tol
        tight += int((low == hi).sum())
    return tight / max(1, int(ok.sum()))


def check_against_topk(t_ptr, t_idx, ranks, scores, top_s, top_i):
    """No tolerance: a target of rank <= k sits at items[r, rank-1] with the bit-identical score; none of rank > k (or -1)
    appears in the top-k."""
    k = top_i.shape[1]
    rows = torch.repeat_interleave(torch.arange(top_i.shape[0], device=DEV), t_ptr[1:] - t_ptr[:-1])
    inside = (ranks >= 1) & (ranks <= k)
    pos = (ranks - 1).clamp(0, k - 1)
    assert torch.equal(top_i[rows[inside], pos[inside]], t_idx[inside])
    assert torch.equal(top_s[rows[inside], pos[inside]].view(torch.int32), scores[inside].view(torch.int32))
    present = (top_i[rows] == t_idx.view(-1, 1)).any(1)
    assert not bool(present[~inside].any()), "a target of rank > k is in the top-k"
    return int(inside.sum())


SHAPES = [(1, 1, 1), (127, 255, 64), (129, 257, 65), (1, 12001, 512), (129, 255, 1), (20000, 12001, 64)]


@pytest.mark.parametrize("n_rows,n_items,dim", SHAPES)
@pytest.mark.parametrize("per_row", [0, 1, 5, 64, 65, 300])
def test_factor_rank_shapes(n_rows, n_items, dim, per_row):
    big = n_rows >= 20000
    if big and per_row in (0, 64, 300):
        pytest.skip("the multi-slice shape runs 1, 5 and 65 targets per row")
    A, B = _rand(n_rows, dim, 1), _rand(n_items, dim, 2)
    rb, cb = _rand(n_rows, 1, 3).view(-1), _rand(n_items, 1, 4).view(-1)
    use_excl = per_row in (1, 65) or (per_row == 5 and not big)
    n_ref = min(n_rows, 300)                            # the float64 check reads the first 300 rows
    e_lists = _excl_lists(n_rows, n_items, 5) if use_excl else None
    t_lists = _lists(n_rows, n_items, per_row, 6, e_lists)
    targets = _csr(t_lists)
    exclude = _csr(e_lists) if use_excl else None
    ranks, scores, n_cand = ops.factor_rank(A, rb, B, cb, targets, exclude=exclude)
    nnz = targets[1].numel()
    assert ranks.shape == (nnz,) and scores.shape == (nnz,) and n_cand.shape == (n_rows,)
    n_excl = torch.tensor([len(set(x)) for x in e_lists], device=DEV) if use_excl else 0
    assert torch.equal(n_cand, n_items - n_excl + torch.zeros(n_rows, dtype=torch.int64, device=DEV))
    # 1. against float64
    S = _ref_scores(A[:n_ref], rb[:n_ref], B, cb, None if e_lists is None else e_lists[:n_ref])
    rp, ri = targets[0][:n_ref + 1], targets[1][:int(targets[0][n_ref])]
    tight = check_ranks(S, rp, ri, ranks[:ri.numel()], scores[:ri.numel()])
    if ri.numel() >= 100:
        assert tight > 0.3                               # the bounds pin most ranks exactly
    # 2. against K10, exactly
    k = min(256, n_items)
    top_s, top_i = ops.factor_topk(A, rb, B, cb, k, exclude=exclude)
    check_against_topk(targets[0], targets[1], ranks, scores, top_s, top_i)
    # 3. determinism
    r2, s2, _ = ops.factor_rank(A, rb, B, cb, targets, exclude=exclude)
    assert torch.equal(ranks, r2) and torch.equal(scores.view(torch.int32), s2.view(torch.int32))


def test_factor_rank_ties_and_slice_count():
    n_items, dim = 12001, 64
    A, B = _rand(200, dim, 5).abs(), _rand(n_items, dim, 6, 0.1)
    best = torch.full((1, dim), 3.0, device=DEV)        # a row every (positive) query scores far above the rest
    tied = [3, 300, 5000, n_items - 2]
    for j in tied:
        B[j] = best
    t_lists = [[5000, 3, n_items - 2, 17] for _ in range(200)]
    ranks, scores, _ = ops.factor_rank(A, None, B, None, _csr(t_lists))
    r = ranks.view(200, 4)
    assert bool((r[:, 1] == 1).all() & (r[:, 0] == 3).all() & (r[:, 2] == 4).all() & (r[:, 3] > 4).all())
    s = scores.view(200, 4)
    assert torch.equal(s[:, 0], s[:, 1]) and torch.equal(s[:, 1], s[:, 2])
    top_s, top_i = ops.factor_topk(A, None, B, None, 256)
    targets = _csr(t_lists)
    check_against_topk(*targets, ranks, scores, top_s, top_i)
    # rows replicated to 20 000: a different slice count, the same ranks
    rows = 20000
    Ar = A.repeat(rows // 200, 1).contiguous()
    big = _csr(t_lists * (rows // 200))
    rb, sb, _ = ops.factor_rank(Ar, None, B, None, big)
    assert torch.equal(rb.view(-1, 800), ranks.view(1, 800).expand(rows // 200, -1))
    assert torch.equal(sb.view(-1, 800).view(torch.int32), scores.view(1, 800).expand(rows // 200, -1).view(torch.int32))


def test_factor_rank_special_values():
    n_rows, n_items, dim = 129, 3000, 50
    A, B = _rand(n_rows, dim, 10), _rand(n_items, dim, 11)
    rb, cb = _rand(n_rows, 1, 12).view(-1), _rand(n_items, 1, 13).view(-1)
    B[17] = float("nan")                                # a NaN item: never counts, rank -1 as a target
    B[18] = 100.0
    cb[19] = float("-inf")                              # a -inf item: never counts, rank -1 as a target
    rb[7] = float("-inf")                               # a -inf row: every target -1
    t_lists = [[17, 19, 18, 5, 2999] if r % 2 else [5, 18] for r in range(n_rows)]
    t_lists[4] = []
    targets = _csr(t_lists)
    ranks, scores, _ = ops.factor_rank(A, rb, B, cb, targets)
    S = _ref_scores(A, rb, B, cb)
    check_ranks(S, *targets, ranks, scores)
    rows = torch.repeat_interleave(torch.arange(n_rows, device=DEV), targets[0][1:] - targets[0][:-1])
    assert bool((ranks[(targets[1] == 17) | (targets[1] == 19) | (rows == 7)] == -1).all())
    assert bool(torch.isnan(scores[targets[1] == 17]).all()) and bool(torch.isneginf(scores[targets[1] == 19]).all())
    # the NaN and -inf items are no competitors: the largest rank is the number of items with a finite score
    assert int(ranks.max()) <= n_items - 2
    top_s, top_i = ops.factor_topk(A, rb, B, cb, 256)
    check_against_topk(*targets, ranks, scores, top_s, top_i)
    # no rows, and rows without targets
    z = ops.factor_rank(A[:0], None, B, None, (torch.zeros(1, dtype=torch.int64, device=DEV),
                                                torch.zeros(0, dtype=torch.int64, device=DEV)))
    assert z[0].numel() == 0 and z[1].numel() == 0 and z[2].numel() == 0
    e = ops.factor_rank(A, None, B, None, _csr([[] for _ in range(n_rows)]))
    assert e[0].numel() == 0 and torch.equal(e[2], torch.full((n_rows,), n_items, device=DEV))


def test_factor_rank_errors():
    A, B = _rand(4, 8, 1), _rand(10, 8, 2)
    t = _csr([[1], [2], [], [3]])
    with pytest.raises(RuntimeError):
        ops.factor_rank(A.cpu(), None, B, None, t)
    with pytest.raises(ValueError):
        ops.factor_rank(A.double(), None, B, None, t)
    with pytest.raises(ValueError):
        ops.factor_rank(_rand(4, 513, 1), None, _rand(10, 513, 2), None, t)
    with pytest.raises(ValueError):
        ops.factor_rank(A, None, B, None, _csr([[1], [10], [], [3]]))
    with pytest.raises(ValueError):
        ops.factor_rank(A, None, B, None, _csr([[1, 1], [2], [], [3]]))
    with pytest.raises(ValueError):
        ops.factor_rank(A, None, B, None, t, exclude=_csr([[], [0, 2], [], []]))


def test_kernel_names_in_trace():
    A, B = _rand(300, 64, 1), _rand(3000, 64, 2)
    targets = _csr(_lists(300, 3000, 3, 1))
    ops.factor_rank(A, None, B, None, targets)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        ops.factor_rank(A, None, B, None, targets)
        torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    for k in ("factor_split_kernel", "factor_rank_capture_kernel", "factor_rank_count_kernel", "factor_rank_finish_kernel"):
        assert any(k in n for n in names), (k, sorted(names))


# ---------------------------------------------------------------------------------------------------------------------
# through the models
# ---------------------------------------------------------------------------------------------------------------------
def _model_targets(seed, per_row=5, with_pad=False):
    g = torch.Generator().manual_seed(seed)
    lists = [(torch.randperm(I - 1, generator=g)[:per_row] + 1).tolist() for _ in range(U - 1)]
    if with_pad:
        lists[3].append(0)
    return _csr(lists)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("name", ["deepconn", "narre", "dual_att"])
def test_rank_items(name, prec):
    sc, _ = MODELS[name](prec)
    u_ids = torch.arange(1, U, device=DEV)
    targets = _model_targets(1)
    ranks, scores, n_cand = sc.rank_items(u_ids, targets)
    assert torch.equal(n_cand, torch.full((U - 1,), I - 1, device=DEV))       # the padding item is not a candidate
    s256, i256 = sc.recommend(u_ids, 256)                                      # every eligible item
    assert check_against_topk(*targets, ranks, scores, s256, i256) == targets[1].numel()
    uu = torch.repeat_interleave(u_ids, targets[0][1:] - targets[0][:-1])
    ref = sc.score_cached(uu, targets[1])
    assert float((scores.double() - ref.double()).abs().max() / ref.double().abs().max()) < 1e-5
    with pytest.raises(ValueError):
        sc.rank_items(u_ids, _model_targets(1, with_pad=True))
    r2, _, n2 = sc.rank_items(u_ids, _model_targets(1, with_pad=True), exclude_padding=False)
    assert torch.equal(n2, torch.full((U - 1,), I, device=DEV))


@pytest.mark.parametrize("name", ["deepconn", "narre"])
def test_rank_items_follows_head_parameters(name):
    sc, _ = MODELS[name]("fp32")
    u_ids = torch.arange(1, 100, device=DEV)
    targets = _model_targets(2)
    targets = (targets[0][:100], targets[1][:int(targets[0][99])])
    r0, s0, _ = sc.rank_items(u_ids, targets)
    m = sc.model
    opt = torch.optim.SGD([m.item_feat.W, m.fm.h, m.fm.item_bias.weight], lr=0.5)
    for p in opt.param_groups[0]["params"]:
        p.grad = torch.randn_like(p)
    opt.step()
    r1, s1, _ = sc.rank_items(u_ids, targets)
    assert not torch.equal(s0, s1)
    s256, i256 = sc.recommend(u_ids, 256)
    check_against_topk(*targets, r1, s1, s256, i256)


def test_evaluate():
    sc, _ = MODELS["deepconn"]("fp32")
    u_ids = torch.arange(1, U, device=DEV)
    n = U - 1
    g = torch.Generator().manual_seed(3)
    seen = [(torch.randperm(I - 1, generator=g)[:int(torch.randint(0, 30, (1,), generator=g))] + 1).tolist() for _ in range(n)]
    t_lists = _lists(n, I, 4, 4, seen)
    t_lists = [[t for t in x if t != 0] for x in t_lists]
    t_lists[5] = []
    targets, exclude = _csr(t_lists), _csr(seen)
    ks = (1, 5, 10)
    res = sc.evaluate(u_ids, targets, ks=ks, exclude=exclude)
    # the float64 reference ranks, on rows whose targets are clear of near-ties
    A, rb, B, cb = sc.factors()
    cbp = cb.clone()
    cbp[0] = float("-inf")
    S = _ref_scores(A[u_ids], rb[u_ids], B, cbp, seen)
    S = torch.where(torch.isnan(S), torch.full_like(S, float("-inf")), S)
    rows = torch.repeat_interleave(torch.arange(n, device=DEV), targets[0][1:] - targets[0][:-1])
    st = S[rows, targets[1]]
    ref_rank = (S[rows] >= st.view(-1, 1)).sum(1)
    scale = S.where(torch.isfinite(S), torch.zeros_like(S)).abs().amax(1)
    near = ((S[rows] - st.view(-1, 1)).abs() <= 1e-5 * scale[rows].view(-1, 1)).sum(1) > 1
    clean_row = torch.ones(n, dtype=torch.bool, device=DEV).index_put_((rows[near],), torch.tensor(False, device=DEV))
    assert float(clean_row.float().mean()) > 0.5
    n_cand = I - 1 - torch.tensor([len(set(x)) for x in seen], device=DEV)
    keep = clean_row[rows]
    cnt = (targets[0][1:] - targets[0][:-1])[clean_row]
    ptr_c = torch.cat([torch.zeros(1, dtype=torch.int64, device=DEV), torch.cumsum(cnt, 0)])
    ref = ranking_metrics(ref_rank[keep], ptr_c, n_cand[clean_row], ks)
    sel = torch.nonzero(clean_row).view(-1)
    t_c = (ptr_c, targets[1][keep])
    e_c = _csr([seen[i] for i in sel.tolist()])
    got = sc.evaluate(u_ids[sel], t_c, ks=ks, exclude=e_c)
    for k in ref:
        assert got[k] == pytest.approx(ref[k], rel=1e-12, abs=1e-12), k
    # hr@k is exactly the fraction of rows (with a target) whose recommend(k) holds one of them
    for k in ks:
        _, items = sc.recommend(u_ids, k, exclude=exclude)
        found = (items[rows] == targets[1].view(-1, 1)).any(1).double()
        hit = torch.zeros(n, dtype=torch.float64, device=DEV).index_add_(0, rows, found) > 0
        has = (targets[0][1:] - targets[0][:-1]) > 0
        assert res[f"hr@{k}"] == float(hit[has].double().mean())
    assert res["n_rows"] == n - 1
