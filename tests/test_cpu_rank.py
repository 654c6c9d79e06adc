"""Host side of full-catalogue ranking (no GPU): K11's limits and workspace query, target validation, the row-splitting
helper and the ranking metrics against a brute-force computation."""
import math

import numpy as np
import pytest
import torch

from rbr_b200 import ops
from rbr_b200.inference import ranking_metrics


@pytest.mark.parametrize("n_items,dim,max_targets", [(1000, 0, 1), (1000, 513, 1), (0, 64, 1), (1000, 64, 0), (1000, 64, 65),
                                                     (2 ** 31, 64, 1)])
def test_factor_rank_limits_refused(n_items, dim, max_targets):
    with pytest.raises(ValueError):
        ops.factor_rank_workspace_bytes(100, n_items, dim, 10, max_targets)
    assert ops.lib.rbr_factor_rank_workspace_bytes(100, n_items, dim, 10, max_targets) == -4          # RBR_EUNSUPPORTED
    # refused before anything is launched: no stream, no workspace, no data needed
    assert ops.lib.rbr_factor_rank(None, None, 100, None, None, n_items, dim, None, None, None, None, 10, max_targets, None,
                                   None, None, 0, None) == -4


def test_factor_rank_workspace_query():
    for n, i, d, t, mt in [(1, 1, 1, 1, 1), (20000, 12000, 64, 200000, 10), (129, 257, 65, 300, 64)]:
        ws = ops.factor_rank_workspace_bytes(n, i, d, t, mt)
        assert ws >= t * 12 + n * 6 * 32 * 2 + i * 6 * 32 * 2      # keys + counters + the split operands
    assert ops.factor_rank_workspace_bytes(20000, 12000, 64, 200000, 10) < 20000 * 12000 * 4 / 4
    # a call without rows or targets needs nothing else
    assert ops.lib.rbr_factor_rank(None, None, 0, None, None, 100, 8, None, None, None, None, 0, 1, None, None, None, 0,
                                   None) == 0
    # a workspace that is too small is refused before any launch
    assert ops.lib.rbr_factor_rank(1, None, 10, 1, None, 100, 8, None, None, 1, 1, 5, 1, 1, 1, 1, 16, None) == -3     # RBR_EWORKSPACE


def _csr(lists):
    ptr = torch.tensor([0] + np.cumsum([len(x) for x in lists]).tolist(), dtype=torch.int64)
    return ptr, torch.tensor([i for x in lists for i in x], dtype=torch.int64)


def test_rank_inputs_validation():
    tp, ti = _csr([[9, 3], [], [4, 1, 0]])
    ex = _csr([[2, 2, 7], [5], []])
    plan = ops.rank_inputs(tp, ti, 3, 10, ex)
    assert plan["targets"].tolist() == [3, 9, 0, 1, 4]
    assert ti[plan["order"]].tolist() == plan["targets"].tolist()
    assert plan["piece_row"].tolist() == [0, 2] and plan["piece_ptr"].tolist() == [0, 2, 5]
    assert plan["excl_ptr"].tolist() == [0, 2, 2] and plan["excl_idx"].tolist() == [2, 7]
    assert plan["n_candidates"].tolist() == [8, 9, 10] and plan["max_targets"] == 3
    with pytest.raises(ValueError, match="lie in"):
        ops.rank_inputs(*_csr([[9, 10], [], [1]]), 3, 10)
    with pytest.raises(ValueError, match="lie in"):
        ops.rank_inputs(*_csr([[9, -1], [], [1]]), 3, 10)
    with pytest.raises(ValueError, match="twice"):
        ops.rank_inputs(*_csr([[9, 3, 9], [], [1]]), 3, 10)
    with pytest.raises(ValueError, match="exclusion"):
        ops.rank_inputs(*_csr([[9, 3], [], [1]]), 3, 10, _csr([[0], [3], [5, 1]]))
    with pytest.raises(ValueError):
        ops.rank_inputs(torch.tensor([0, 2, 1, 3]), torch.tensor([1, 2, 3]), 3, 10)
    # the same id in different rows, or excluded in another row, is fine
    ops.rank_inputs(*_csr([[3], [3], [1]]), 3, 10, _csr([[1], [], [3]]))


def test_split_target_rows():
    counts = torch.tensor([0, 3, 130, 0, 64, 65, 1])
    rows, ptr = ops.split_target_rows(counts, 64)
    assert rows.tolist() == [1, 2, 2, 2, 4, 5, 5, 6]
    assert ptr.tolist() == [0, 3, 67, 131, 133, 197, 261, 262, 263]
    for cap in (1, 2, 5, 64):
        c = torch.randint(0, 12, (40,), generator=torch.Generator().manual_seed(cap))
        rows, ptr = ops.split_target_rows(c, cap)
        lens = (ptr[1:] - ptr[:-1])
        assert int(lens.max()) <= cap and bool((lens > 0).all())
        assert torch.equal(torch.bincount(rows, weights=lens.double(), minlength=40).long(), c)
    rows, ptr = ops.split_target_rows(torch.zeros(3, dtype=torch.int64))
    assert rows.numel() == 0 and ptr.tolist() == [0]
    p, x = ops.gather_csr_rows(torch.tensor([0, 2, 2, 5]), torch.tensor([1, 2, 7, 8, 9]), torch.tensor([2, 0, 0, 1]))
    assert p.tolist() == [0, 3, 5, 7, 7] and x.tolist() == [7, 8, 9, 1, 2, 1, 2]


def brute_metrics(rank_lists, n_cand, ks):
    """The definitions of ranking_metrics' docstring, row by row."""
    out = {f"{n}@{k}": [] for k in ks for n in ("hr", "recall", "ndcg")}
    out.update(mrr=[], auc=[])
    for ranks, nc in zip(rank_lists, n_cand):
        m = len(ranks)
        if m == 0:
            continue
        valid = sorted(r for r in ranks if r > 0)
        best = valid[0] if valid else None
        for k in ks:
            hits = [r for r in valid if r <= k]
            out[f"hr@{k}"].append(1.0 if hits else 0.0)
            out[f"recall@{k}"].append(len(hits) / m)
            idcg = sum(1 / math.log2(j + 1) for j in range(1, min(m, k) + 1))
            out[f"ndcg@{k}"].append(sum(1 / math.log2(r + 1) for r in hits) / idcg)
        out["mrr"].append(1 / best if best else 0.0)
        if nc > m:
            terms = []
            for r in ranks:
                if r < 0:
                    terms.append(0.0)
                else:
                    others = sum(1 for q in valid if q < r)
                    terms.append(1 - (r - 1 - others) / (nc - m))
            out["auc"].append(sum(terms) / m)
    res = {k: (float(np.mean(v)) if v else 0.0) for k, v in out.items()}
    res["n_rows"] = sum(1 for r in rank_lists if len(r))
    return res


def _random_ranks(n_rows, seed):
    rng = np.random.default_rng(seed)
    lists, n_cand = [], []
    for r in range(n_rows):
        nc = int(rng.integers(1, 300))
        m = int(rng.integers(0, min(nc, 40) + 1)) if r % 7 else 0
        ranks = sorted(rng.choice(np.arange(1, nc + 1), size=m, replace=False).tolist())
        ranks = [x if rng.random() > 0.1 else -1 for x in ranks]          # some targets without a rank
        if r % 11 == 5:
            nc = m                                                       # no negatives: left out of AUC
        rng.shuffle(ranks)
        lists.append(ranks)
        n_cand.append(nc)
    return lists, n_cand


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_ranking_metrics_against_brute_force(seed):
    lists, n_cand = _random_ranks(200, seed)
    lists[3] = [-1, -1]                                                  # every target unranked
    lists[4] = [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12]                   # m > k
    n_cand[4] = 12 if seed == 0 else 500
    ks = (1, 5, 10, 20)
    ptr, ranks = _csr(lists)
    got = ranking_metrics(ranks, ptr, torch.tensor(n_cand), ks)
    ref = brute_metrics(lists, n_cand, ks)
    assert set(got) == set(ref)
    for k in ref:
        assert got[k] == pytest.approx(ref[k], rel=1e-12, abs=1e-12), k


def test_ranking_metrics_edge_cases():
    empty = ranking_metrics(torch.zeros(0, dtype=torch.int64), torch.zeros(4, dtype=torch.int64), torch.full((3,), 10),
                            (10,))
    assert empty["n_rows"] == 0 and empty["hr@10"] == 0.0 and empty["auc"] == 0.0
    one = ranking_metrics(torch.tensor([1]), torch.tensor([0, 1]), torch.tensor([100]), (1, 10))
    assert one["hr@1"] == one["ndcg@1"] == one["mrr"] == one["auc"] == 1.0
    last = ranking_metrics(torch.tensor([100]), torch.tensor([0, 1]), torch.tensor([100]), (10,))
    assert last["hr@10"] == 0.0 and last["auc"] == 0.0 and last["mrr"] == pytest.approx(0.01)
