"""Host side of D-ATT's token attributions (no GPU): the symbols of rbr_datt_explain_contrib / rbr_explain_attrib_ex /
rbr_datt_fc_grads, their limits (refused before any launch), and the input validation of ops.datt_explain_contrib,
ops.datt_fc_grads and the new arguments of ops.explain_attrib."""
import ctypes
import os

import pytest
import torch

from rbr_b200 import ops
from rbr_b200._lib import HEADER, LIB_PATH, parse_header

SYMBOLS = ("rbr_datt_explain_contrib", "rbr_explain_attrib_ex", "rbr_datt_fc_grads")


def test_symbols_declared_and_bound():
    protos = parse_header(HEADER)
    for name in SYMBOLS:
        assert name in protos, name
    if not os.path.exists(LIB_PATH):
        pytest.skip("native library not built")
    for name in SYMBOLS:
        assert callable(getattr(ops.lib, name))


def test_limits_refused_before_launch():
    """no stream and no data: the limits are checked first (RBR_EUNSUPPORTED = -4)"""
    lib = ops.lib
    for window, doc_len in ((2, 500), (17, 500), (0, 500), (5, 3)):
        rc = lib.rbr_datt_explain_contrib(None, 50, 100, None, 10, doc_len, None, window, None, None, 200, None, None, None, 100,
                                          None, None, None, None, 500, None, 1900, None, 500, None, doc_len, 0, None)
        assert rc == -4, (window, doc_len)
    for hidden in (0, 769):
        assert lib.rbr_datt_fc_grads(None, None, 10, None, 5, None, 5, 50, None, None, hidden, None, 500, None, None, None,
                                     None) == -4, hidden
    conv = (ctypes.c_int64 * 3)(100, 3, 1)
    for m, width, doc_len in ((33, 3, 500), (5, 17, 500), (5, 3, 16385)):
        rc = lib.rbr_explain_attrib_ex(None, 10, 1, doc_len, None, None, None, 100, None, 300, 10, 1, conv, None, 100, None,
                                       doc_len, m, width, None, None, None, None, None, None, None, None)
        assert rc == -4, (m, width, doc_len)
    # a dense term needs 8 more bytes of shared memory per document: 8192 one-token documents no longer fit
    rc = lib.rbr_explain_attrib_ex(None, 10, 16384, 1, None, None, None, 100, None, 300, 16384, 1, conv, ctypes.c_void_p(8),
                                   100, ctypes.c_void_p(8), 1, 5, 1, None, None, None, None, None, None, None, None)
    assert rc == -4


class _FakeCuda(torch.Tensor):
    """Stand-in that passes the is_cuda checks so that validation is reached without a device; the shape / range checks
    run before any launch."""

    @property
    def is_cuda(self):
        return True


def _cuda(t):
    return t.as_subclass(_FakeCuda)


V, E, L, W, LO, GO, N = 50, 8, 20, 5, 6, 4, 7


def _side_prm(E=E, L=L, W=W):
    g = torch.Generator().manual_seed(0)
    shapes = [(1, E, W), (1,), (LO, E, 1), (LO,), (1, E, L), (1,), (GO, E, 2), (GO,), (GO, E, 3), (GO,), (GO, E, 4), (GO,)]
    return [_cuda(torch.randn(*s, generator=g)) for s in shapes]


def _contrib_inputs():
    htot = LO + 3 * GO
    amax = torch.zeros(N, htot, dtype=torch.int32)
    return dict(table=_cuda(torch.randn(V, E)), ids=_cuda(torch.randint(0, V, (N, L))), prm=_side_prm(),
                gate_l=_cuda(torch.rand(N, L)), gate_g=_cuda(torch.rand(N)), feat=_cuda(torch.rand(N, htot)),
                argmax=_cuda(amax), packed=[_cuda(torch.zeros(1, dtype=torch.uint8))] * 4)


@pytest.mark.parametrize("change", ["ids_u16", "ids_1d", "prm_count", "emb", "global_len", "even_window", "short_doc",
                                    "gate_l", "gate_g", "feat", "argmax_dtype", "argmax_shape", "argmax_local_hi",
                                    "argmax_k4_hi", "argmax_neg"])
def test_datt_explain_contrib_validation(change):
    kw = _contrib_inputs()
    htot = LO + 3 * GO
    if change == "ids_u16":
        kw["ids"] = _cuda(torch.randint(0, V, (N, L)).to(torch.uint16))
    elif change == "ids_1d":
        kw["ids"] = _cuda(torch.randint(0, V, (N * L,)))
    elif change == "prm_count":
        kw["prm"] = kw["prm"][:10]
    elif change == "emb":
        kw["table"] = _cuda(torch.randn(V, E + 1))
    elif change == "global_len":
        kw["prm"][4] = _cuda(torch.randn(1, E, L - 1))
    elif change == "even_window":
        kw["prm"][0] = _cuda(torch.randn(1, E, 4))
    elif change == "short_doc":
        kw["ids"] = _cuda(torch.randint(0, V, (N, 3)))
        kw["prm"] = _side_prm(L=3, W=3)
        kw["gate_l"] = _cuda(torch.rand(N, 3))
    elif change == "gate_l":
        kw["gate_l"] = _cuda(torch.rand(N, L + 1))
    elif change == "gate_g":
        kw["gate_g"] = _cuda(torch.rand(N + 1))
    elif change == "feat":
        kw["feat"] = _cuda(torch.rand(N, htot - 1))
    elif change == "argmax_dtype":
        kw["argmax"] = _cuda(torch.zeros(N, htot, dtype=torch.int64))
    elif change == "argmax_shape":
        kw["argmax"] = _cuda(torch.zeros(N, htot + 1, dtype=torch.int32))
    elif change == "argmax_local_hi":
        a = torch.zeros(N, htot, dtype=torch.int32)
        a[2, 0] = L                                                      # the k = 1 conv pools over [0, L)
        kw["argmax"] = _cuda(a)
    elif change == "argmax_k4_hi":
        a = torch.zeros(N, htot, dtype=torch.int32)
        a[:, LO + 2 * GO:] = L - 3                                       # the k = 4 conv pools over [0, L - 3)
        kw["argmax"] = _cuda(a)
    elif change == "argmax_neg":
        a = torch.zeros(N, htot, dtype=torch.int32)
        a[0, LO] = -1
        kw["argmax"] = _cuda(a)
    with pytest.raises((ValueError, TypeError)):
        ops.datt_explain_contrib(**kw)


def test_datt_explain_convs():
    assert ops.datt_explain_convs(_side_prm()) == [(LO, W, 2), (GO, 2, 0), (GO, 3, 0), (GO, 4, 0)]


def _fc_inputs(P=5, U=6, I=4, H1=12, H2=3, D=10):
    return dict(u_ids=_cuda(torch.arange(P) % U), i_ids=_cuda(torch.arange(P) % I), user_out=_cuda(torch.randn(U, H2)),
                item_out=_cuda(torch.randn(I, H2)), user_mask=_cuda(torch.rand(U, H1) > 0.5),
                item_mask=_cuda(torch.rand(I, H1) > 0.5), w0=_cuda(torch.randn(H1, D)), w3=_cuda(torch.randn(H2, H1)))


@pytest.mark.parametrize("change", ["u_hi", "i_neg", "pairs", "w3_shape", "mask_shape", "out_dim", "hidden_cap", "mask_dtype",
                                    "ids_dtype"])
def test_datt_fc_grads_validation(change):
    kw = _fc_inputs()
    if change == "u_hi":
        kw["u_ids"] = _cuda(torch.tensor([0, 1, 6, 2, 3]))
    elif change == "i_neg":
        kw["i_ids"] = _cuda(torch.tensor([0, 1, -1, 2, 3]))
    elif change == "pairs":
        kw["i_ids"] = _cuda(torch.tensor([0, 1]))
    elif change == "w3_shape":
        kw["w3"] = _cuda(torch.randn(3, 11))
    elif change == "mask_shape":
        kw["item_mask"] = _cuda(torch.rand(4, 11) > 0.5)
    elif change == "out_dim":
        kw["user_out"] = _cuda(torch.randn(6, 4))
    elif change == "hidden_cap":
        kw.update(w0=_cuda(torch.randn(769, 10)), w3=_cuda(torch.randn(3, 769)), user_mask=_cuda(torch.rand(6, 769) > 0.5),
                  item_mask=_cuda(torch.rand(4, 769) > 0.5))
    elif change == "mask_dtype":
        kw["user_mask"] = _cuda(torch.rand(6, 12))
    elif change == "ids_dtype":
        kw["u_ids"] = _cuda(torch.arange(5, dtype=torch.int32))
    with pytest.raises((ValueError, TypeError)):
        ops.datt_fc_grads(**kw)


def _attrib_inputs(P=3, T=20, H=4, k=3, n_ent=5):
    amax = _cuda(torch.randint(0, T, (n_ent, H), dtype=torch.int32))
    contrib = _cuda(torch.randn(n_ent, H * k))
    g = _cuda(torch.randn(P, 1, H))
    ent = _cuda(torch.arange(P, dtype=torch.int64))
    coef, vec = _cuda(torch.randn(n_ent, H)), _cuda(torch.randn(n_ent, T))
    return ent, g, amax, contrib, [(H, k, (k - 1) // 2)], coef, vec


@pytest.mark.parametrize("change", ["coef_only", "vec_only", "coef_rows", "coef_cols", "vec_len", "argmax_cols", "ent_hi"])
def test_explain_attrib_dense_validation(change):
    ent, g, amax, contrib, convs, coef, vec = _attrib_inputs()
    if change == "coef_only":
        vec = None
    elif change == "vec_only":
        coef = None
    elif change == "coef_rows":
        coef = _cuda(torch.randn(4, 4))
    elif change == "coef_cols":
        coef = _cuda(torch.randn(5, 3))
    elif change == "vec_len":
        vec = _cuda(torch.randn(5, 21))
    elif change == "argmax_cols":
        amax = _cuda(torch.zeros(5, 3, dtype=torch.int32))
    elif change == "ent_hi":
        ent = _cuda(torch.tensor([0, 1, 5]))
    with pytest.raises(ValueError):
        ops.explain_attrib(ent, g, None, amax, contrib, convs, 1, 20, 5, 3, dense_coef=coef, dense_vec=vec)
