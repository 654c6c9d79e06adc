"""Host side of diversified top-k (no GPU): list_metrics on hand-computed lists, K14's limits through the C-ABI, the header
prototypes, and the unit normalisation of item vectors."""
import math

import pytest
import torch

from rbr_b200 import ops
from rbr_b200._lib import parse_header
from rbr_b200.inference import list_metrics


def test_list_metrics_hand_computed():
    # unit vectors: 1 = e0, 2 = e1, 3 = (e0 + e1) / sqrt 2 (given unnormalised), 4 = zero, 0 = e0 again
    vecs = torch.tensor([[1.0, 0.0], [2.0, 0.0], [0.0, 3.0], [1.0, 1.0], [0.0, 0.0]])
    items = torch.tensor([[1, 2, 3],          # pairs: (1,2) 1 - 0, (1,3) 1 - 1/sqrt2, (2,3) 1 - 1/sqrt2
                          [1, 4, -1],         # one pair with the zero vector: 1 - 0
                          [2, -1, -1],        # one valid item: no pair, not counted
                          [-1, -1, -1]])
    out = list_metrics(items, vecs, n_items=4)
    r0 = (1.0 + 2 * (1 - 1 / math.sqrt(2))) / 3
    assert out["n_rows"] == 2
    assert abs(out["ild"] - (r0 + 1.0) / 2) < 1e-7
    assert out["coverage"] == 4 / 4                     # {1, 2, 3, 4}
    same = list_metrics(torch.tensor([[1, 0], [0, 1]]), vecs, n_items=4)    # two copies of e0: 1 - 1 = 0
    assert abs(same["ild"]) < 1e-7 and same["coverage"] == 2 / 4
    empty = list_metrics(torch.full((3, 2), -1, dtype=torch.int64), vecs, n_items=4)
    assert empty == {"ild": 0.0, "coverage": 0.0, "n_rows": 0}
    with pytest.raises(ValueError):
        list_metrics(torch.tensor([[5, 1]]), vecs, n_items=4)


def test_unit_rows():
    x = torch.tensor([[3.0, 4.0], [0.0, 0.0], [1e-30, 0.0]])
    u = ops.unit_rows(x)
    assert u.dtype == torch.float32
    assert torch.equal(u, torch.tensor([[0.6, 0.8], [0.0, 0.0], [1.0, 0.0]]))


@pytest.mark.parametrize("k,pool,dim", [(0, 10, 8), (11, 10, 8), (10, 257, 8), (10, 20, 0), (10, 20, 513)])
def test_mmr_limits_refused(k, pool, dim):
    assert ops.lib.rbr_mmr_supported(pool, dim, k) == 0
    assert not ops.mmr_supported(pool, dim, k)
    # refused before anything is launched: no stream, no data needed
    assert ops.lib.rbr_mmr_select(None, None, 100, pool, None, 1000, dim, k, 0.5, None, None, None) == -4   # RBR_EUNSUPPORTED


def test_mmr_limits_accepted_and_bad_lam():
    for k, pool, dim in [(1, 1, 1), (256, 256, 512), (10, 40, 300)]:
        assert ops.lib.rbr_mmr_supported(pool, dim, k) == 1
        # zero rows: nothing to do, nothing launched
        assert ops.lib.rbr_mmr_select(None, None, 0, pool, None, 1000, dim, k, 0.5, None, None, None) == 0
    for lam in (-0.1, 1.5, float("nan")):
        assert ops.lib.rbr_mmr_select(None, None, 0, 40, None, 1000, 8, 10, lam, None, None, None) == -1   # RBR_EINVAL


def test_header_prototypes():
    protos = parse_header()
    assert protos["rbr_mmr_supported"][2] == ["pool", "dim", "k"]
    assert protos["rbr_mmr_select"][2] == ["pool_scores", "pool_items", "n_rows", "pool", "item_vecs", "n_items", "dim", "k",
                                           "lam", "out_scores", "out_items", "stream"]


def test_mmr_select_argument_checks_before_the_device():
    s = torch.zeros(2, 4)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.mmr_select(s, torch.zeros(2, 4, dtype=torch.int64), torch.zeros(10, 3), 2, 0.5)
