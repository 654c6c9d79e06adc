"""Host side of PairScorer.add / update (no GPU): the input checks, the spare-capacity buffers, the row -> model-id map, and
the incremental factors and unit item vectors, on caches installed from CPU tensors (what build_cache leaves behind, without
its encoder)."""
import pytest
import torch

import rbr_b200
from rbr_b200 import ops
from rbr_b200.inference import SIDES, PairScorer, _reserve, _Side, fm_factors

U, I, V, L, H, K = 30, 20, 50, 12, 24, 8


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _installed(model, shapes, seed=0, kept=None):
    """A scorer whose cache holds seeded features [U, H] / [I, H] as if build_cache had encoded documents of `shapes`."""
    g = _gen(seed)
    sc = PairScorer(model)
    for name, n, shape in zip(SIDES, (U, I), shapes):
        sc._sides[name] = _Side(torch.rand(n, H, generator=g) - 0.3, None if kept is None else kept[name], shape)
    return sc


def _deepconn():
    return rbr_b200.DeepCoNNpp(U, I, V, [3], 16, H, K, L, None, 0.0)


def _factors64(sc):
    """fm_factors in float64 on the LastFeat of every cached row under its model id, rounded to fp32"""
    m = sc.model
    lat, bias = [], []
    for name, lf, tab in zip(SIDES, (m.user_feat, m.item_feat), (m.fm.user_bias, m.fm.item_bias)):
        s = sc._sides[name]
        mids = s.view("model_ids")
        lat.append(s.view("cached").double() @ lf.W.detach().double() + lf.b.detach().double()
                   + lf.ebd.weight.detach().double()[mids])
        bias.append(tab.weight.detach().double()[mids])
    return [t.float() for t in fm_factors(lat[0], lat[1], m.fm.h.detach().double(), bias[0], bias[1],
                                          m.fm.g_bias.detach().double())]


def test_reserve_grows_geometrically_and_keeps_rows():
    buf = torch.arange(3.0).view(3, 1)
    allocs, used = 0, 3
    for step in range(1000):
        new = _reserve(buf, used, used + 1)
        allocs += new is not buf
        assert torch.equal(new[:used].view(-1), torch.arange(float(used)))
        buf = new
        buf[used] = used
        used += 1
    assert allocs <= 10                              # 3 -> 6 -> 12 -> ... -> 1536
    assert _reserve(buf, used, 5) is buf


def test_checks_raise_before_anything_changes():
    sc = PairScorer(_deepconn())
    docs = torch.randint(1, V, (4, L))
    with pytest.raises(ValueError):
        sc.add("user", docs)                           # no cache
    sc.user_feat, sc.item_feat = torch.rand(U, H), torch.rand(I, H)
    with pytest.raises(ValueError):
        sc.add("user", docs)                           # features assigned, not built from documents
    sc = _installed(_deepconn(), ((L,), (L,)))
    before = {name: (s.n, s.gen, {k: None if t is None else t.clone() for k, t in s.bufs.items()})
              for name, s in sc._sides.items()}
    ids = torch.tensor([1, 2, 3, 4])
    bad = [
        lambda: sc.add("users", docs),
        lambda: sc.add("user", torch.randint(1, V, (4, L + 1))),
        lambda: sc.add("user", docs.view(4, 1, L)),
        lambda: sc.add("user", docs.float()),
        lambda: sc.add("user", docs, torch.ones(4, L - 1, dtype=torch.bool)),
        lambda: sc.add("user", docs, rev_ids=torch.zeros(4, 1, dtype=torch.int64)),
        lambda: sc.add("user", docs, rev_masks=torch.ones(4, 1, dtype=torch.bool)),
        lambda: sc.update("item", torch.tensor([1, 2, 2, 4]), docs),
        lambda: sc.update("item", torch.tensor([1, 2, 3, I]), docs),
        lambda: sc.update("item", torch.tensor([-1, 2, 3, 4]), docs),
        lambda: sc.update("item", ids[:3], docs),
        lambda: sc.update("item", ids.view(2, 2), docs),
        lambda: sc.update("item", ids.float(), docs),
        lambda: sc.update("side", ids, docs),
    ]
    for call in bad:
        with pytest.raises(ValueError):
            call()
    for name, s in sc._sides.items():
        n, gen, bufs = before[name]
        assert (s.n, s.gen, s.log) == (n, gen, [])
        assert all(torch.equal(bufs[k], t) for k, t in s.bufs.items() if t is not None)


def test_datt_takes_no_masks_and_narre_rev_ids_are_checked():
    datt = _installed(rbr_b200.DualAtt(V, L, 5, 20, 10, 10, 50, 5, 0.0, None), ((L,), (L,)))
    with pytest.raises(ValueError):
        datt.add("user", torch.randint(1, V, (2, L)), torch.ones(2, L, dtype=torch.bool))
    R, T = 3, 10
    narre = _installed(rbr_b200.NARRE(U, I, V, [3], H, 16, 8, K, R, T, 0.0, 0, 0, 0, None, "CNN"), ((R, T), (R, T)))
    docs = torch.randint(1, V, (2, R, T))
    for rev in (None, torch.zeros(2, R + 1, dtype=torch.int64), torch.full((2, R), I), torch.full((2, R), -1)):
        with pytest.raises(ValueError):
            narre.add("user", docs, rev_ids=rev)       # user reviews name items: model ids in [0, I)
    with pytest.raises(ValueError):
        narre.update("item", torch.tensor([3, 4]), docs, rev_ids=torch.full((2, R), U))
    assert narre._sides["user"].n == U and narre._sides["item"].gen == 0


def test_zero_rows_change_nothing():
    sc = _installed(_deepconn(), ((L,), (L,)))
    A0 = [None if t is None else t.clone() for t in sc.factors()]
    out = sc.add("item", torch.empty(0, L, dtype=torch.int64))
    assert out.dtype == torch.int64 and out.shape == (0,)
    sc.update("user", torch.empty(0, dtype=torch.int64), torch.empty(0, L, dtype=torch.int64))
    assert sc._sides["item"].n == I and sc._sides["item"].gen == 0 and sc._sides["user"].gen == 0
    assert all(torch.equal(a, b) for a, b in zip(A0, sc.factors()))


def test_model_ids_map_added_rows_to_padding():
    sc = _installed(_deepconn(), ((L,), (L,)))
    s = sc._sides["item"]
    rows = torch.tensor([0, 5, I - 1, I, -1])
    assert sc._model_ids("item", rows) is rows                  # the identity while no row was added
    s.write(None, {"cached": torch.rand(3, H), "model_ids": torch.full((3,), 0, dtype=torch.int64)})
    got = sc._model_ids("item", torch.tensor([0, 5, I - 1, I, I + 2, I + 3, -1]))
    assert got.tolist() == [0, 5, I - 1, 0, 0, I + 3, -1]      # rows outside the cache pass unchanged


def test_factors_derive_only_changed_rows_and_follow_the_head():
    sc = _installed(_deepconn(), ((L,), (L,)))
    counted = []
    real = sc._latent64

    def counting(name, feat, mids=None):
        counted.append((name, feat.shape[0]))
        return real(name, feat, mids)
    sc._latent64 = counting
    g = _gen(1)
    assert all(torch.equal(a, b) for a, b in zip(sc.factors(), _factors64(sc)))
    assert counted == [("user", U), ("item", I)]

    def step(kind):
        counted.clear()
        s = sc._sides["user" if kind != "add_item" else "item"]
        if kind == "update":
            rows = torch.tensor([3, 7, 11])
            s.write(rows, {"cached": torch.rand(3, H, generator=g)})
        else:
            s.write(None, {"cached": torch.rand(4, H, generator=g), "model_ids": torch.zeros(4, dtype=torch.int64)})
        got = sc.factors()
        assert all(torch.equal(a, b) for a, b in zip(got, _factors64(sc)))
        return got

    step("update")
    assert counted == [("user", 3), ("item", 0)]
    step("add_item")
    assert counted == [("user", 0), ("item", 4)]
    for _ in range(3):
        step("add_user")
    assert sc._sides["user"].n == U + 12 and sc._sides["user"].log == []
    # two changes between calls: the union of their rows
    s = sc._sides["user"]
    s.write(torch.tensor([1, 2]), {"cached": torch.rand(2, H, generator=g)})
    s.write(torch.tensor([2, 9]), {"cached": torch.rand(2, H, generator=g)})
    counted.clear()
    assert all(torch.equal(a, b) for a, b in zip(sc.factors(), _factors64(sc)))
    assert counted == [("user", 3), ("item", 0)]
    # a head parameter change re-derives every row
    with torch.no_grad():
        sc.model.fm.h.add_(0.01)
    counted.clear()
    assert all(torch.equal(a, b) for a, b in zip(sc.factors(), _factors64(sc)))
    assert counted == [("user", U + 12), ("item", I + 4)]
    counted.clear()
    sc.factors()
    assert counted == []


def test_unit_item_vectors_follow_the_item_rows(monkeypatch):
    sc = _installed(_deepconn(), ((L,), (L,)))
    seen = []
    real = ops.unit_rows
    monkeypatch.setattr(ops, "unit_rows", lambda x: seen.append(x.shape[0]) or real(x))
    g = _gen(2)
    assert torch.equal(sc._unit_item_vecs(None), real(sc.item_feat))
    s = sc._sides["item"]
    s.write(torch.tensor([2, 4]), {"cached": torch.rand(2, H, generator=g)})
    s.write(None, {"cached": torch.rand(5, H, generator=g), "model_ids": torch.zeros(5, dtype=torch.int64)})
    seen.clear()
    assert torch.equal(sc._unit_item_vecs(None), real(sc.item_feat))
    assert seen == [7]
    seen.clear()
    sc._unit_item_vecs(None)
    assert seen == [] and s.log == []
    with pytest.raises(ValueError):
        sc._unit_item_vecs(torch.rand(I, 3))                     # one row per current item row: I + 5


def test_caller_tensors_are_copied_on_first_write():
    docs = {name: torch.randint(1, V, (n, L)) for name, n in zip(SIDES, (U, I))}
    kept = {name: {"docs": docs[name], "masks": None} for name in SIDES}
    sc = _installed(_deepconn(), ((L,), (L,)), kept=kept)
    before = docs["user"].clone()
    s = sc._sides["user"]
    new = torch.randint(1, V, (2, L), dtype=torch.int32)
    s.write(torch.tensor([0, 5]), {"cached": torch.rand(2, H), "docs": new})
    assert torch.equal(docs["user"], before)
    cur = sc._explain["user"]["docs"]
    assert cur.dtype == before.dtype and torch.equal(cur[[0, 5]], new.long())
    keep = torch.ones(U, dtype=torch.bool)
    keep[[0, 5]] = False
    assert torch.equal(cur[keep], before[keep])
    assert sc._explain["item"]["docs"] is not None and sc._explain["item"]["masks"] is None
