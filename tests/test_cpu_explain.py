"""Host side of PairScorer.explain (no GPU): K12's symbols and limits, input validation of ops.conv_window_contrib /
ops.explain_attrib, and the window rule (ops.window_select) against a brute-force statement of it."""
import ctypes
import itertools
import math
import os

import pytest
import torch

from rbr_b200 import ops
from rbr_b200._lib import HEADER, LIB_PATH, parse_header

SYMBOLS = ("rbr_explain_supported", "rbr_conv_window_contrib", "rbr_explain_attrib")


def test_symbols_declared_and_bound():
    protos = parse_header(HEADER)
    for name in SYMBOLS:
        assert name in protos, name
    if not os.path.exists(LIB_PATH):
        pytest.skip("native library not built")
    for name in SYMBOLS:
        assert callable(getattr(ops.lib, name))


def test_explain_supported_limits():
    sup = ops.lib.rbr_explain_supported
    assert sup(16384, 32, 16, 8) == 1
    assert sup(1, 1, 1, 1) == 1
    for args in [(16385, 5, 3, 1), (0, 5, 3, 1), (500, 33, 3, 1), (500, 0, 3, 1), (500, 5, 17, 1), (500, 5, 0, 1),
                 (500, 5, 3, 9), (500, 5, 3, 0)]:
        assert sup(*args) == 0, args
    assert (ops.EXPLAIN_MAX_POSITIONS, ops.EXPLAIN_MAX_M, ops.EXPLAIN_MAX_WIDTH, ops.EXPLAIN_MAX_CONVS) == (16384, 32, 16, 8)
    # refused before anything is launched: no stream and no data needed
    conv = (ctypes.c_int64 * 3)(100, 3, 1)
    rc = ops.lib.rbr_explain_attrib(None, 10, 1, 500, None, None, None, 100, None, 300, 10, 1, conv, 33, 3, None, None, None,
                                    None, None, None, None, None)
    assert rc == -4                                                              # RBR_EUNSUPPORTED


class _FakeCuda(torch.Tensor):
    """Stand-in that passes the is_cuda checks so that validation is reached without a device; the shape / range checks
    run before any launch."""

    @property
    def is_cuda(self):
        return True


def _cuda(t):
    return t.as_subclass(_FakeCuda)


def _explain_inputs(P=3, R=1, T=20, H=4, k=3, n_ent=5):
    feat = _cuda(torch.rand(n_ent * R, H))
    amax = _cuda(torch.randint(0, T, (n_ent * R, H), dtype=torch.int32))
    contrib = _cuda(torch.randn(n_ent * R, H * k))
    g = _cuda(torch.randn(P, R, H))
    ent = _cuda(torch.arange(P, dtype=torch.int64) * R)
    return ent, g, feat, amax, contrib, [(H, k, (k - 1) // 2)]


@pytest.mark.parametrize("change", ["m0", "m33", "w0", "w17", "positions", "ent_hi", "ent_neg", "g_shape", "contrib_cols",
                                    "argmax_shape", "convs0", "bad_conv"])
def test_explain_attrib_validation(change):
    ent, g, feat, amax, contrib, convs = _explain_inputs()
    kw = dict(docs_per_entity=1, doc_len=20, m=5, width=3)
    if change == "m0":
        kw["m"] = 0
    elif change == "m33":
        kw["m"] = 33
    elif change == "w0":
        kw["width"] = 0
    elif change == "w17":
        kw["width"] = 17
    elif change == "positions":
        kw["doc_len"] = 16385
    elif change == "ent_hi":
        ent = _cuda(torch.tensor([0, 1, 5]))
    elif change == "ent_neg":
        ent = _cuda(torch.tensor([0, -1, 2]))
    elif change == "g_shape":
        g = _cuda(torch.randn(3, 1, 5))
    elif change == "contrib_cols":
        contrib = _cuda(torch.randn(5, 11))
    elif change == "argmax_shape":
        amax = _cuda(torch.zeros(4, 4, dtype=torch.int32))
    elif change == "convs0":
        convs = []
    elif change == "bad_conv":
        convs = [(4, 0, 1)]
    with pytest.raises(ValueError):
        ops.explain_attrib(ent, g, feat, amax, contrib, convs, **kw)


def test_explain_attrib_narre_entities_are_whole():
    ent, g, feat, amax, contrib, convs = _explain_inputs(P=2, R=3, n_ent=4)
    with pytest.raises(ValueError):                     # row 1 does not start an entity's block of 3 reviews
        ops.explain_attrib(_cuda(torch.tensor([0, 4])), g, feat, amax, contrib, convs, 3, 20, 5, 3)


@pytest.mark.parametrize("change", ["argmax_hi", "argmax_neg", "mask_shape", "pad", "weight_emb", "out_shape"])
def test_conv_window_contrib_validation(change):
    V, E, H, k, N, L = 50, 8, 4, 3, 6, 20
    table = _cuda(torch.randn(V, E))
    ids = _cuda(torch.randint(0, V, (N, L)))
    w = _cuda(torch.randn(H, E, k))
    amax = _cuda(torch.randint(0, L, (N, H), dtype=torch.int32))
    mask, pad, out = None, 1, None
    if change == "argmax_hi":
        amax = _cuda(torch.full((N, H), L, dtype=torch.int32))           # positions are [0, L + 2 pad - k + 1) = [0, L)
    elif change == "argmax_neg":
        amax = _cuda(torch.full((N, H), -1, dtype=torch.int32))
    elif change == "mask_shape":
        mask = _cuda(torch.ones(N, L + 1, dtype=torch.bool))
    elif change == "pad":
        pad = -1
    elif change == "weight_emb":
        w = _cuda(torch.randn(H, E + 1, k))
    elif change == "out_shape":
        out = _cuda(torch.empty(N, H * k - 1))
    with pytest.raises(ValueError):
        ops.conv_window_contrib(table, ids, mask, w, pad, amax, packed=_cuda(torch.zeros(1, dtype=torch.uint8)), out=out)


# ---------------------------------------------------------------------------------------------------------------------
# the window rule
# ---------------------------------------------------------------------------------------------------------------------
def brute_windows(row, doc_len, m, width, top):
    """Greedy selection written out: candidate windows inside one document, best sum first (top) or lowest first, the lower
    start on ties, skipping any window that shares a position with one already chosen."""
    S = len(row)
    cands = [(sum(row[s:s + width]), s) for s in range(S) if s % doc_len + width <= doc_len]
    chosen = []
    while len(chosen) < m:
        free = [(v, s) for v, s in cands if all(s + width <= c or c + width <= s for _, c in chosen)]
        if not free:
            break
        best = max(free, key=lambda vs: (vs[0] if top else -vs[0], -vs[1]))
        chosen.append(best)
    pos = [s for _, s in chosen] + [-1] * (m - len(chosen))
    val = [v for v, _ in chosen] + [math.nan] * (m - len(chosen))
    return pos, val


def _compare(attr, doc_len, m, width):
    tp, ta, bp, ba = ops.window_select(attr, doc_len, m, width)
    for r in range(attr.shape[0]):
        row = attr[r].double().tolist()
        for pos, val, top in ((tp, ta, True), (bp, ba, False)):
            bpos, bval = brute_windows(row, doc_len, m, width, top)
            assert pos[r].tolist() == bpos, (r, top, pos[r].tolist(), bpos)
            got = val[r].tolist()
            for a, b in zip(got, bval):
                assert (math.isnan(a) and math.isnan(b)) or abs(a - b) <= 1e-6 * max(1.0, abs(b))


@pytest.mark.parametrize("doc_len,reviews,m,width", [(20, 1, 5, 3), (7, 4, 6, 3), (5, 3, 8, 5), (4, 2, 3, 5), (30, 1, 32, 1),
                                                     (12, 1, 4, 16)])
def test_window_select_matches_brute_force(doc_len, reviews, m, width):
    g = torch.Generator().manual_seed(doc_len * 100 + m)
    # small integers: many exact ties, negative and positive windows, runs of zeros
    attr = torch.randint(-3, 4, (6, reviews * doc_len), generator=g).float()
    attr[0] = 0.0
    attr[1] = -1.0
    _compare(attr, doc_len, m, width)
    _compare(torch.randn(4, reviews * doc_len, generator=g), doc_len, m, width)


def test_window_select_cases():
    # greedy non-overlap: the best window wins and the overlapping second-best is skipped
    a = torch.tensor([[0., 1, 2, -1, 5, 0, 0, 3, 1, 1, 1, 1]])
    tp, ta, bp, ba = ops.window_select(a, 12, 4, 2)
    assert tp.tolist() == [[4, 7, 1, 9]] and ta.tolist() == [[5., 4., 3., 2.]]
    assert bp.tolist() == [[5, 0, 2, 8]]
    # review boundaries at multiples of 6: starts 5 and 11 cross one and are never chosen
    tp, _, bp, _ = ops.window_select(a, 6, 4, 2)
    assert bp.tolist() == [[0, 2, 8, 10]]
    assert not any(s % 6 == 5 for s in tp.view(-1).tolist() + bp.view(-1).tolist())
    # running out: a 5-position document holds two non-overlapping windows of 2
    tp, ta, bp, ba = ops.window_select(torch.ones(1, 5), 5, 4, 2)
    assert tp.tolist() == [[0, 2, -1, -1]] and math.isnan(ta[0, 2]) and math.isnan(ba[0, 3])
    # no window fits at all
    tp, ta, _, _ = ops.window_select(torch.ones(2, 6), 3, 2, 4)
    assert tp.eq(-1).all() and ta.isnan().all()
    # exhaustive check of every 0/1 pattern of a short document
    for bits in itertools.product([0.0, 1.0, -1.0], repeat=6):
        _compare(torch.tensor([bits]), 6, 3, 2)
