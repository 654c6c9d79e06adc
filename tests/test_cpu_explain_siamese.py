"""Host side of SimpleSiamese's explanations (no GPU): K13's symbols and limits, input validation of
ops.explain_avgpool_attrib, and the window rule at width 1 (the token windows K13 picks by default) against brute force."""
import ctypes
import os

import pytest
import torch

from rbr_b200 import ops
from rbr_b200._lib import HEADER, LIB_PATH, parse_header

from test_cpu_explain import _compare, _cuda

SYMBOLS = ("rbr_explain_avgpool_supported", "rbr_explain_avgpool_attrib")


def test_symbols_declared_and_bound():
    protos = parse_header(HEADER)
    for name in SYMBOLS:
        assert name in protos, name
    if not os.path.exists(LIB_PATH):
        pytest.skip("native library not built")
    for name in SYMBOLS:
        assert callable(getattr(ops.lib, name))


def test_explain_avgpool_supported_limits():
    sup = ops.lib.rbr_explain_avgpool_supported
    assert sup(600, 10, 300, 300, 5, 1) == 1                   # 10 reviews x 60 tokens, E = 300, no latent transform
    assert sup(600, 10, 300, 32, 32, 16) == 1
    assert sup(16384, 1, 300, 300, 5, 1) == 1
    assert sup(1, 1, 1, 1, 1, 1) == 1
    for args in [(16385, 1, 300, 300, 5, 1), (0, 1, 300, 300, 5, 1), (600, 0, 300, 300, 5, 1), (600, 7, 300, 300, 5, 1),
                 (600, 10, 300, 300, 0, 1), (600, 10, 300, 300, 33, 1), (600, 10, 300, 300, 5, 0), (600, 10, 300, 300, 5, 17),
                 (600, 10, 0, 300, 5, 1), (600, 10, 300, 0, 5, 1),
                 (1000, 100, 300, 300, 5, 1)]:                 # 100 reviews x (300 + 300) floats: past 227 KB of shared memory
        assert sup(*args) == 0, args
    assert ops.explain_avgpool_supported(600, 10, 300, 300, 5, 1)
    assert not ops.explain_avgpool_supported(600, 10, 300, 300, 33, 1)
    # refused before anything is launched: no stream and no data needed
    rc = ops.lib.rbr_explain_avgpool_attrib(None, 100, 300, None, None, 5, 10, 60, None, 4, None, None, None, None, 0, None, None,
                                            32, None, None, None, None, 300, None, 33, 1, None, None, None, None, None, None,
                                            None, 0, None)
    assert rc == -4                                                              # RBR_EUNSUPPORTED


def _inputs(P=3, n_ent=5, R=4, T=6, E=8, F=8, K=4, V=50):
    return dict(table=_cuda(torch.randn(V, E)), ids=_cuda(torch.randint(0, V, (n_ent, R, T))), mask=None,
                ent=_cuda(torch.arange(P, dtype=torch.int64)), v=_cuda(torch.randn(n_ent, R, F)),
                att_a=_cuda(torch.randn(n_ent, R, F)), att_s=_cuda(torch.rand(n_ent, R)), feat=_cuda(torch.randn(n_ent, F)),
                m=3, width=1, g=_cuda(torch.randn(P, F)))


def _head(P=3, n_ent=5, F=8, K=4, n_other=7):
    return dict(g=None, other=_cuda(torch.arange(P, dtype=torch.int64)), lat=_cuda(torch.randn(n_ent, K)),
                lat_other=_cuda(torch.randn(n_other, K)), w_side=_cuda(torch.randn(F, K)), fm_h=_cuda(torch.randn(K, 1)))


@pytest.mark.parametrize("change", ["m0", "m33", "w0", "w17", "positions", "ent_hi", "ent_neg", "g_shape", "v_shape", "a_shape",
                                    "s_shape", "feat_rows", "mask_shape", "ids_2d", "emb_no_lt", "lt_shape", "no_head",
                                    "other_hi", "other_neg", "lat_shape", "w_side_shape", "lat_other_k"])
def test_explain_avgpool_attrib_validation(change):
    kw = _inputs()
    if change == "m0":
        kw["m"] = 0
    elif change == "m33":
        kw["m"] = 33
    elif change == "w0":
        kw["width"] = 0
    elif change == "w17":
        kw["width"] = 17
    elif change == "positions":
        kw["ids"] = _cuda(torch.zeros(5, 4, 4097, dtype=torch.int64))
    elif change == "ent_hi":
        kw["ent"] = _cuda(torch.tensor([0, 1, 5]))
    elif change == "ent_neg":
        kw["ent"] = _cuda(torch.tensor([0, -1, 2]))
    elif change == "g_shape":
        kw["g"] = _cuda(torch.randn(3, 7))
    elif change == "v_shape":
        kw["v"] = _cuda(torch.randn(5, 3, 8))
    elif change == "a_shape":
        kw["att_a"] = _cuda(torch.randn(5, 4, 7))
    elif change == "s_shape":
        kw["att_s"] = _cuda(torch.rand(5, 4, 1))
    elif change == "feat_rows":
        kw["feat"] = _cuda(torch.randn(4, 8))
    elif change == "mask_shape":
        kw["mask"] = _cuda(torch.ones(5, 4, 7, dtype=torch.bool))
    elif change == "ids_2d":
        kw["ids"] = _cuda(torch.zeros(5, 24, dtype=torch.int64))
    elif change == "emb_no_lt":                                   # without the latent transform F must be E
        kw["table"] = _cuda(torch.randn(50, 9))
    elif change == "lt_shape":
        kw["lt_w"] = _cuda(torch.randn(8, 7))
    elif change == "no_head":                                     # neither g nor the head's inputs
        kw["g"] = None
    else:
        kw.update(_head())
        if change == "other_hi":
            kw["other"] = _cuda(torch.tensor([0, 1, 7]))
        elif change == "other_neg":
            kw["other"] = _cuda(torch.tensor([0, -1, 1]))
        elif change == "lat_shape":
            kw["lat"] = _cuda(torch.randn(4, 4))
        elif change == "w_side_shape":
            kw["w_side"] = _cuda(torch.randn(8, 5))
        elif change == "lat_other_k":
            kw["lat_other"] = _cuda(torch.randn(7, 5))
    with pytest.raises(ValueError):
        ops.explain_avgpool_attrib(**kw)


@pytest.mark.parametrize("doc_len,reviews,m", [(60, 10, 5), (7, 3, 32), (1, 4, 6), (5, 1, 8)])
def test_window_select_width1_matches_brute_force(doc_len, reviews, m):
    g = torch.Generator().manual_seed(doc_len * 10 + reviews)
    attr = torch.randint(-3, 4, (6, reviews * doc_len), generator=g).float()     # many exact ties
    attr[0] = 0.0
    attr[1, ::2] = 0.0                                                           # masked positions read as 0
    _compare(attr, doc_len, m, 1)
    _compare(torch.randn(4, reviews * doc_len, generator=g), doc_len, m, 1)
