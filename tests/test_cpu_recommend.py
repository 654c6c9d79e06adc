"""Host side of full-catalogue top-k (no GPU): the FM head as a factor product, K10's limits and workspace query, and the
normalisation of exclusion lists."""
import pytest
import torch

from oracle import rbr_oracle as orc
from rbr_b200 import ops
from rbr_b200.inference import fm_factors


def test_fm_factors_reproduce_fm_head():
    g = torch.Generator().manual_seed(0)
    U, I, K = 7, 11, 32
    u_lat = torch.randn(U, K, generator=g, dtype=torch.float64)
    i_lat = torch.randn(I, K, generator=g, dtype=torch.float64)
    u_lat[0, :5] = 0.0
    i_lat[:, 7] = 0.0
    i_lat[3] = -i_lat[3].abs()
    u_lat[2] = u_lat[2].abs()
    h = torch.randn(K, 1, generator=g, dtype=torch.float64)
    ub, ib = torch.randn(U, 1, generator=g, dtype=torch.float64), torch.randn(I, 1, generator=g, dtype=torch.float64)
    gb = torch.randn(1, generator=g, dtype=torch.float64)
    A, rb, B, cb = fm_factors(u_lat, i_lat, h, ub, ib, gb)
    got = A @ B.T + rb.view(-1, 1) + cb.view(1, -1)
    uu = torch.arange(U).repeat_interleave(I)
    ii = torch.arange(I).repeat(U)
    ref = orc.fm_head(u_lat[uu], i_lat[ii], uu, ii, h, gb, ub, ib).view(U, I)
    assert float((got - ref).abs().max()) < 1e-12


@pytest.mark.parametrize("k,dim", [(0, 64), (257, 64), (10, 0), (10, 513)])
def test_factor_topk_limits_refused(k, dim):
    with pytest.raises(ValueError):
        ops.factor_topk_workspace_bytes(100, 1000, dim, k)
    assert ops.lib.rbr_factor_topk_workspace_bytes(100, 1000, dim, k) == -4          # RBR_EUNSUPPORTED
    # refused before anything is launched: no stream, no workspace, no data needed
    assert ops.lib.rbr_factor_topk(None, None, 100, None, None, 1000, dim, None, None, k, None, None, None, 0, None) == -4


def test_factor_topk_workspace_query():
    for n, i, d, k in [(1, 1, 1, 1), (20000, 12000, 64, 100), (129, 257, 65, 256)]:
        ws = ops.factor_topk_workspace_bytes(n, i, d, k)
        s = ops.factor_topk_slices(n, i, d, k)
        assert 1 <= s <= 16
        assert ws >= n * s * k * 8 + n * 6 * 64 * 2           # partial lists + the split operands
    assert ops.factor_topk_workspace_bytes(20000, 12000, 64, 100) < 20000 * 12000 * 4 / 4


def test_normalize_exclusions():
    ptr = torch.tensor([0, 4, 4, 7])
    idx = torch.tensor([9, 2, 9, 0, 5, 5, 5])
    p, x = ops.normalize_exclusions(ptr, idx, 3, 10)
    assert p.tolist() == [0, 3, 3, 4] and x.tolist() == [0, 2, 9, 5]
    with pytest.raises(ValueError):
        ops.normalize_exclusions(ptr, torch.tensor([9, 2, 10, 0, 5, 5, 5]), 3, 10)
    with pytest.raises(ValueError):
        ops.normalize_exclusions(ptr, torch.tensor([9, 2, -1, 0, 5, 5, 5]), 3, 10)
    with pytest.raises(ValueError):
        ops.normalize_exclusions(torch.tensor([0, 4, 3, 7]), idx, 3, 10)
