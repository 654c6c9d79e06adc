"""Every variant of the conv forward (K2) against a float64 reference, at the shapes that select it, gated ones included.

`rbr_conv_act_maxpool_fwd` (csrc/api.cu) runs:

  conv_fp32_kernel<TM, K>   fp32 precision, and bf16 shapes both tensor-core kernels decline (csrc/conv_fp32.cu):
                            TM = 64 when Lout <= 96, else 128; K in {1, 2, 3, 4, 5, 7}; a 256-filter block per grid.y
  conv_tc_kernel<K, kps>    bf16, the single-CTA cp.async kernel (CONV_TC_SINGLE_CTA pins it; csrc/conv_tc.cu)
  conv_tc2_kernel<K, ...>   bf16, the CTA-pair TMA kernel (CONV_TC_PAIR_ONLY pins it; csrc/conv_tc2.cu)

D-ATT multiplies the token rows by a gate: gate mode 1 is one gate per token (k = 1), mode 2 one per document.  The fp32
kernel applies it to every position before the max; the tensor-core kernels scale the accumulator rows (mode 1) or the pooled
maximum (mode 2).  With short documents several share a tile, and each row must read its own document's gate.

Reference.  The float64 conv (oracle.conv1d_valid, on the GPU) of the operands the kernel multiplies: the fp32 table and
weights for conv_fp32, the bf16-rounded ones for the tensor-core kernels; the gate stays fp32.  Then gate, bias, activation
and the first arg-max.  Tolerances (max-abs error over max-abs reference) are 1e-5 for fp32 and 2e-5 for bf16: a product of
two bf16 values is exact in fp32, so only the accumulation rounds.  The kernel's arg-max must attain the reference maximum
within that noise; on constructed ties (integer-valued operands, repeated tokens) it must equal torch's first arg-max.

One deliberate difference (DESIGN §3): where every candidate of a column is an exact zero because its gate is exactly 0 (a
gate-mode-2 document gate of 0, or per-token gates of 0), the tensor-core kernels keep the ungated arg-max (mode 2) or the
first +0 (mode 1), where torch takes position 0.  Every consumer multiplies by that gate at the arg-max, so no value or
gradient moves; test_gpu_datt_variants.py checks the gradients for it.
"""
import json
import types

import pytest
import torch

from conftest import rel_err
from oracle import rbr_oracle as orc
from rbr_b200 import ops
from rbr_b200._lib import lib

pytestmark = pytest.mark.gpu
FP32_TOL, BF16_TOL = 1e-5, 2e-5
RELU, TANH = ops.ACT_RELU, ops.ACT_TANH
SINGLE, PAIR = ops.CONV_TC_SINGLE_CTA, ops.CONV_TC_PAIR_ONLY


def _kernels_launched(fn, tmp_path):
    """[(kernel name without spaces, grid x, block x)] of every CUDA kernel `fn` launches, from a torch.profiler trace."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    events = json.loads(path.read_text())["traceEvents"]
    launched = [(e["name"].replace(" ", ""), e["args"]["grid"][0], e["args"]["block"][0])
                for e in events if e.get("cat") == "kernel"]
    return out, launched


def _names(launched):
    return [n for n, _, _ in launched]


def fp32_instance(K, Lout):
    return f"conv_fp32_kernel<{128 if Lout > 96 else 64},{K}>("


_DEF = dict(V=400, E=64, H=40, K=3, pad=None, n=12, L=100, ids="i64", mask="bytes", act=RELU, prec="fp32", flags=0,
            gate=0, oob=False, all_pad=True, feat_ld=None, ri=True, lout=None, target=None)


def C(**kw):
    d = dict(_DEF)
    d.update(kw)
    if d["pad"] is None:
        d["pad"] = (d["K"] - 1) // 2
    if d["lout"] is not None:                                  # choose L for the wanted output length
        d["L"] = d["lout"] - 2 * d["pad"] + d["K"] - 1
    return types.SimpleNamespace(**d)


def _round(t):
    return t.to(torch.bfloat16).to(torch.float32)


def _dev_ids(ids, width):
    return {"i64": ids, "i32": ids.int(), "u16": ids.to(torch.uint16)}[width].cuda()


def _inputs(c, seed):
    """Table, weights, bias, ids [n, L], mask (None / bool), gate (None / fp32) on the CPU, and the count of ids the kernel
    reads and must report as out of range."""
    g = torch.Generator().manual_seed(seed)
    table = torch.randn(c.V, c.E, generator=g)
    w = (torch.rand(c.H, c.E, c.K, generator=g) * 2 - 1) / (c.E * c.K) ** 0.5
    b = (torch.rand(c.H, generator=g) * 2 - 1) * 0.1
    ids = torch.randint(1, c.V, (c.n, c.L), generator=g)
    lens = torch.randint(1, c.L + 1, (c.n,), generator=g)
    lens[-1] = c.L
    valid = torch.arange(c.L).unsqueeze(0) < lens.unsqueeze(1)
    if c.all_pad:
        valid[0] = False                                          # an all-padding document
    mask = None
    if c.mask in ("bytes", "ids"):
        ids = ids * valid
        if c.mask == "bytes":
            mask = valid & (torch.rand(c.n, c.L, generator=g) > 0.05)
    oob_read = 0
    if c.oob:
        pos = torch.rand(c.n, c.L, generator=g) < 0.05
        pos[0] = False                                            # (document 0 stays all padding)
        big = torch.randint(c.V, 2 * c.V + 40, (c.n, c.L), generator=g)
        neg = torch.randint(-100, 0, (c.n, c.L), generator=g)
        use_neg = (torch.rand(c.n, c.L, generator=g) < 0.5) & (c.ids != "u16")
        ids = torch.where(pos, torch.where(use_neg, neg, big), ids)
        read = pos.clone()
        if c.mask == "bytes":
            read &= mask
        if c.mask == "ids":
            read &= ids != 0
        oob_read = int(read.sum())
    gate = None
    if c.gate == 1:
        gate = torch.rand(c.n, c.L, generator=g)
        gate[torch.rand(c.n, c.L, generator=g) < 0.05] = 1.0
        gate[torch.rand(c.n, c.L, generator=g) < 0.05] = 0.0
    elif c.gate == 2:
        gate = torch.rand(c.n, generator=g) * 0.9 + 0.05
        gate[1 % c.n] = 1.0
        gate[2 % c.n] = 0.0
    return table, w, b, ids, mask, gate, oob_read


def _x(tab, ids, mask):
    """Embedded documents [n, L, E]: out-of-range ids and masked positions read as zero rows."""
    V = tab.shape[0]
    ok = (ids >= 0) & (ids < V)
    if mask is not None:
        ok = ok & mask
    return tab[ids.clamp(0, V - 1)] * ok.unsqueeze(-1).to(tab.dtype)


def _act(act, y):
    return torch.relu(y) if act == RELU else torch.tanh(y)


def first_argmax(y):
    """torch's rule over dim 1 of [n, T, H]: the first position attaining the max, -0 == +0; a NaN wins, first NaN first."""
    T = y.shape[1]
    pos = torch.arange(T, device=y.device).view(1, T, 1).expand_as(y)
    nan = torch.isnan(y)
    top = torch.where(nan, torch.full_like(y, -float("inf")), y).max(dim=1, keepdim=True).values
    hit = torch.where(nan.any(dim=1, keepdim=True), nan, y == top)
    return torch.where(hit, pos, torch.full_like(pos, T)).min(dim=1).values


def reference(c, table, w, b, ids, mask, gate, rnd):
    """float64 (raw [n, Lout, H] = gate * conv_nobias, pooled raw [n, H] = its max, first arg-max [n, H]) on the GPU."""
    x = _x(rnd(table).cuda().double(), ids, mask)
    raw = orc.conv1d_valid(x, rnd(w).cuda().double(), torch.zeros(c.H, dtype=torch.float64, device="cuda"), c.pad)
    if c.gate == 1:
        raw = raw * gate.cuda().double().unsqueeze(-1)
    elif c.gate == 2:
        raw = raw * gate.cuda().double().view(-1, 1, 1)
    am = first_argmax(raw)
    return raw, torch.gather(raw, 1, am.unsqueeze(1)).squeeze(1), am


def run(c, table, w, b, ids, mask, gate, tmp_path):
    mask_dev = None if mask is None else mask.cuda()

    def call():
        return ops.conv_act_maxpool(table.cuda(), _dev_ids(ids, c.ids), mask_dev, w.cuda(), b.cuda(), c.pad, act=c.act,
                                    precision=c.prec, flags=c.flags, mask_from_ids=c.mask == "ids", row_index_table=c.ri,
                                    gate=None if gate is None else gate.cuda(), gate_mode=c.gate, return_pool_raw=True,
                                    feat_ld=c.feat_ld)
    return _kernels_launched(call, tmp_path)


def check_against_reference(c, feat, amax, pool_raw, raw, top, tol, tie_exempt=None):
    """Values, pool_raw and the routing of one conv.  tie_exempt [n, H] bool: columns whose documented tensor-core arg-max
    differs from torch's (every candidate an exact zero because of a zero gate); their arg-max is checked by the caller."""
    b = c.b_dev
    ref_feat = _act(c.act, top + b)
    assert rel_err(feat, ref_feat) < tol, ("feat", rel_err(feat, ref_feat))
    assert rel_err(pool_raw, top) < tol, ("pool_raw", rel_err(pool_raw, top))
    Lout = raw.shape[1]
    assert int(amax.min()) >= 0 and int(amax.max()) < Lout
    got = torch.gather(raw, 1, amax.long().unsqueeze(1)).squeeze(1)
    noise = tol * float(raw.abs().max().clamp_min(1e-30))
    gap = (top - got).abs()
    if tie_exempt is not None:
        gap = torch.where(tie_exempt, torch.zeros_like(gap), gap)
    assert float(gap.max()) <= noise, ("routing", float(gap.max()), noise)


def _check_case(name, c, tmp_path):
    table, w, b, ids, mask, gate, oob_read = _inputs(c, seed=sum(map(ord, name)))
    lib.rbr_consume_oob_count(None)
    (feat, amax, pool_raw), launched = run(c, table, w, b, ids, mask, gate, tmp_path)
    assert lib.rbr_consume_oob_count(None) >= oob_read
    if c.oob:
        assert oob_read > 0
    if c.target:
        assert sum(c.target in n for n in _names(launched)) == 1, (c.target, _names(launched))
    conv_kernels = [n for n in _names(launched) if "conv_fp32_kernel<" in n or "conv_tc_kernel<" in n or "conv_tc2_kernel<" in n]
    assert len(conv_kernels) == 1, conv_kernels
    if c.feat_ld is not None:
        assert bool(torch.isnan(feat[:, c.H:]).all()) and bool(torch.isnan(pool_raw[:, c.H:]).all())
        assert bool((amax[:, c.H:] == -1).all())
        feat, amax, pool_raw = feat[:, :c.H], amax[:, :c.H], pool_raw[:, :c.H]
    tc = c.prec == "bf16" and "conv_fp32_kernel" not in conv_kernels[0]
    ref_mask = (ids != 0) if c.mask == "ids" else mask
    raw, top, am = reference(c, table, w, b, ids.cuda(), None if ref_mask is None else ref_mask.cuda(), gate,
                             _round if tc else (lambda t: t))
    c.b_dev = b.cuda().double()
    exempt = None
    if tc and c.gate:
        # every candidate of the column an exact zero: the documented tensor-core difference
        exempt = (raw == 0).all(dim=1)
    check_against_reference(c, feat, amax, pool_raw, raw, top, BF16_TOL if tc else FP32_TOL, exempt)
    if exempt is not None and c.gate == 2 and bool(exempt.any()):
        # a document gate of 0: the tensor-core kernels keep the ungated arg-max, which attains the ungated maximum
        z = gate == 0
        c0 = types.SimpleNamespace(**{**vars(c), "gate": 0})
        raw0, top0, _ = reference(c0, table, w, b, ids.cuda(), None if ref_mask is None else ref_mask.cuda(), None, _round)
        got = torch.gather(raw0[z.cuda()], 1, amax[z.cuda()].long().unsqueeze(1)).squeeze(1)
        assert float((top0[z.cuda()] - got).abs().max()) <= BF16_TOL * float(raw0.abs().max())
    if c.all_pad and c.mask != "none":
        # an all-padding document reads zero rows everywhere: act(bias) at position 0
        assert rel_err(feat[0], _act(c.act, c.b_dev)) < 1e-6 and int(amax[0].abs().max()) == 0
    return launched


# ----------------------------------------------------------------------------------------------------------------------
# conv_fp32_kernel: every <TM, K> at the TM boundary, filter blocks, embedding widths, ids / masks, gates, strided output
# ----------------------------------------------------------------------------------------------------------------------
_IDW = ("i64", "i32", "u16")
_MASKS = ("bytes", "ids", "none")
FP32_CASES = {}
for i, (K, lout) in enumerate([(K, lo) for K in (1, 2, 3, 4, 5, 7) for lo in (96, 97)]):
    pad = (K - 1) // 2 if i % 2 else 0
    FP32_CASES[f"fp32_K{K}_Lout{lout}_pad{pad}"] = C(K=K, lout=lout, pad=pad, act=(RELU, TANH)[i % 2], ids=_IDW[i % 3],
                                                     mask=_MASKS[i % 3], target=fp32_instance(K, lout))
for i, H in enumerate((1, 7, 256, 257, 300, 513)):
    FP32_CASES[f"fp32_H{H}"] = C(H=H, n=6, ids=_IDW[i % 3], act=(RELU, TANH)[i % 2], target=fp32_instance(3, 100))
for i, E in enumerate((4, 16, 17, 30, 300, 301, 520)):
    FP32_CASES[f"fp32_E{E}"] = C(E=E, K=(7, 5, 3)[i % 3], n=8, mask=_MASKS[i % 3], ids=_IDW[i % 3],
                                 target=fp32_instance((7, 5, 3)[i % 3], 100))
FP32_CASES.update({
    "fp32_E520_K7_H300": C(E=520, K=7, H=300, n=4, lout=140, target=fp32_instance(7, 140)),
    **{f"fp32_oob_{w}_{m}": C(oob=True, ids=w, mask=m, target=fp32_instance(3, 100)) for w in _IDW for m in _MASKS},
    "fp32_feat_ld": C(H=37, feat_ld=45, target=fp32_instance(3, 100)),
    "fp32_feat_ld_2blocks": C(H=260, feat_ld=300, n=4, target=fp32_instance(3, 100)),
    "fp32_gate1_k1": C(K=1, gate=1, act=TANH, mask="none", all_pad=False, target=fp32_instance(1, 100)),
    "fp32_gate1_k1_short": C(K=1, L=37, gate=1, act=TANH, mask="none", all_pad=False, target=fp32_instance(1, 37)),
    **{f"fp32_gate2_k{K}": C(K=K, pad=0, gate=2, act=TANH, mask="none", all_pad=False, target=fp32_instance(K, 100 - K + 1))
       for K in (2, 3, 4)},
    "fp32_gate2_H300_L500": C(K=3, pad=0, H=300, L=500, n=5, gate=2, act=TANH, mask="none", all_pad=False,
                              target=fp32_instance(3, 498)),
})


@pytest.mark.parametrize("name", list(FP32_CASES))
def test_conv_fp32_instance_vs_float64(name, tmp_path):
    _check_case(name, FP32_CASES[name], tmp_path)


def test_bf16_fallback_to_fp32_kernel(tmp_path):
    """E = 2048, k = 7: both tensor-core kernels decline (their resident weight tile would not fit shared memory), so bf16
    precision runs conv_fp32_kernel on the fp32 operands.  Pinning either tensor-core kernel raises instead."""
    c = C(V=300, E=2048, H=64, K=7, n=4, L=120, prec="bf16", target=fp32_instance(7, 120))
    plan = (torch.zeros(16, dtype=torch.int64))
    import ctypes
    assert lib.rbr_conv_tc2_plan(c.E, c.H, c.K, c.L, c.pad, c.n, ctypes.cast(plan.data_ptr(), ctypes.c_void_p)) == 0
    assert int(plan[0]) == 0
    _check_case("bf16_fallback", c, tmp_path)
    table, w, b, ids, mask, _, _ = _inputs(c, 1)
    for flags in (SINGLE, PAIR):
        with pytest.raises(RuntimeError, match="outside"):
            ops.conv_act_maxpool(table.cuda(), ids.cuda(), mask.cuda(), w.cuda(), b.cuda(), c.pad, precision="bf16", flags=flags)


# ----------------------------------------------------------------------------------------------------------------------
# gated tensor-core forward: both kernels, long and packed short documents, gates per document, exactly 0 and 1
# ----------------------------------------------------------------------------------------------------------------------
TC_GATED = {}
for flags, kname in ((SINGLE, "conv_tc_kernel<"), (PAIR, "conv_tc2_kernel<")):
    for L in (500, 20, 37, 60):
        for K in (1, 2, 3, 4):
            for ri in ((True, False) if K in (1, 3) else (True,)):
                tag = f"{'single' if flags == SINGLE else 'pair'}_L{L}_k{K}_gate{1 if K == 1 else 2}{'' if ri else '_noidx'}"
                TC_GATED[tag] = C(V=600, E=100, H=200 if K == 1 else 100, K=K, pad=0, L=L, n=70 if L < 100 else 9,
                                  gate=1 if K == 1 else 2, act=TANH, prec="bf16", flags=flags, ri=ri, mask="bytes",
                                  all_pad=False, target=f"{kname}{K},")


@pytest.mark.parametrize("name", list(TC_GATED))
def test_gated_tensor_core_vs_float64(name, tmp_path):
    """With a byte mask and n_docs >= 64 an ungated call would run the document selection; gated calls must not (it would
    give skipped documents act(bias) without their gate)."""
    c = TC_GATED[name]
    launched = _check_case(name, c, tmp_path)
    assert not any("conv_doc_select_kernel" in n or "conv_doc_tiles" in n for n in _names(launched)), _names(launched)


def test_gated_packed_tiles_read_their_own_gate(tmp_path):
    """Short documents packed 2 to 4 per tile, gates that differ only by document: a gate read from another slot of the
    tile changes the pooled value of every filter."""
    for flags in (SINGLE, PAIR):
        for L in (20, 37, 60):
            for K, mode in ((1, 1), (3, 2)):
                c = C(V=50, E=32, H=32, K=K, pad=0, L=L, n=8, gate=mode, act=TANH, prec="bf16", flags=flags, mask="none",
                      all_pad=False)
                g = torch.Generator().manual_seed(L + K)
                table = torch.rand(c.V, c.E, generator=g) + 0.5                     # positive rows, positive weights:
                w = torch.rand(c.H, c.E, c.K, generator=g) / (c.E * c.K)           # the conv is positive everywhere
                b = torch.zeros(c.H)
                ids = torch.randint(0, c.V, (c.n, c.L), generator=g)
                per_doc = torch.tensor([0.1 * (d + 1) for d in range(c.n)])
                gate = per_doc.unsqueeze(1).expand(c.n, c.L).contiguous() if mode == 1 else per_doc
                (feat, amax, pool_raw), _ = run(c, table, w, b, ids, None, gate, tmp_path)
                raw, top, _ = reference(c, table, w, b, ids.cuda(), None, gate, _round)
                assert rel_err(pool_raw, top) < BF16_TOL, (flags, L, K)


# ----------------------------------------------------------------------------------------------------------------------
# ties and NaN on all three kernels
# ----------------------------------------------------------------------------------------------------------------------
KERNELS = {"fp32": ("fp32", 0), "single": ("bf16", SINGLE), "pair": ("bf16", PAIR)}


def _tie_inputs(K, L, n, H, E, seed):
    """Integer-valued table and weights (every product and sum exact in fp32 and bf16) and ids from a 6-token vocabulary, so
    that many windows repeat exactly."""
    g = torch.Generator().manual_seed(seed)
    table = torch.randint(-2, 3, (6, E), generator=g).float()
    w = torch.randint(-1, 2, (H, E, K), generator=g).float()
    b = torch.randint(-2, 3, (H,), generator=g).float() * 0.25
    ids = torch.randint(0, 6, (n, L), generator=g)
    return table, w, b, ids


@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("K,L", [(1, 40), (3, 130), (3, 20), (4, 60)])
def test_exact_ties_first_argmax(kernel, K, L, tmp_path):
    prec, flags = KERNELS[kernel]
    c = C(V=6, E=32, H=48, K=K, pad=(K - 1) // 2, L=L, n=66, act=RELU, prec=prec, flags=flags, mask="none", all_pad=False)
    table, w, b, ids = _tie_inputs(K, L, c.n, c.H, c.E, seed=K * 1000 + L)
    (feat, amax, pool_raw), _ = run(c, table, w, b, ids, None, None, tmp_path)
    raw, top, am = reference(c, table, w, b, ids.cuda(), None, None, lambda t: t)
    ties = int(((raw == top.unsqueeze(1)).sum(dim=1) > 1).sum())
    assert ties >= c.n * c.H // 10, ties                                  # the case really is about ties
    assert torch.equal(pool_raw.double(), top) and torch.equal(amax.long(), am)


@pytest.mark.parametrize("kernel", list(KERNELS))
def test_signed_zero_ties_under_a_zero_gate(kernel, tmp_path):
    """Per-token gate (mode 1) exactly 0 on a run of tokens whose conv is negative then positive: those positions hold -0 and
    +0.  With every other position negative the max is 0.  torch (and the fp32 kernel) take the first zero; the tensor-core
    kernels compare raw bits and take the first +0 (DESIGN §3).  Values agree exactly either way."""
    prec, flags = KERNELS[kernel]
    E, H, L, n = 16, 16, 40, 4
    c = C(V=3, E=E, H=H, K=1, pad=0, L=L, n=n, act=TANH, prec=prec, flags=flags, mask="none", all_pad=False, gate=1)
    table = torch.stack([torch.full((E,), -1.0), torch.full((E,), 1.0), torch.full((E,), -2.0)])
    w = torch.ones(H, E, 1)
    b = torch.zeros(H)
    ids = torch.full((n, L), 2)                                   # conv -32 everywhere ...
    ids[:, 5], ids[:, 9] = 0, 1                                   # ... -16 at 5 and +16 at 9
    gate = torch.full((n, L), 0.5)
    gate[:, 5], gate[:, 9] = 0.0, 0.0                             # -0 at 5, +0 at 9; -16 elsewhere
    (feat, amax, pool_raw), _ = run(c, table, w, b, ids, None, gate, tmp_path)
    assert bool((pool_raw == 0).all()) and bool((feat == 0).all())
    expected = 5 if prec == "fp32" else 9
    assert bool((amax == expected).all()), (kernel, amax[0].tolist())


@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("sign", [1.0, -1.0])
def test_nan_row_propagates_first_nan(kernel, sign, tmp_path):
    """A NaN table row (either sign) read at some positions: the pooled value is NaN and the arg-max the first window that
    reads it, as torch's max_pool1d gives."""
    prec, flags = KERNELS[kernel]
    E, H, L, n, K = 32, 32, 60, 66, 3
    c = C(V=20, E=E, H=H, K=K, pad=1, L=L, n=n, act=RELU, prec=prec, flags=flags, mask="none", all_pad=False)
    g = torch.Generator().manual_seed(7)
    table = torch.randn(c.V, E, generator=g)
    table[3] = torch.tensor(float("nan")).copysign(torch.tensor(sign))
    w = torch.randn(H, E, K, generator=g) / (E * K) ** 0.5
    b = torch.zeros(H)
    ids = torch.randint(4, c.V, (n, L), generator=g)
    for d in range(0, n, 3):
        ids[d, (d * 7) % (L - 2) + 1] = 3                         # one NaN token in every third document
    (feat, amax, pool_raw), _ = run(c, table, w, b, ids, None, None, tmp_path)
    raw, top, am = reference(c, table, w, b, ids.cuda(), None, None, _round if prec == "bf16" else (lambda t: t))
    has_nan = torch.isnan(top)
    assert bool(has_nan[::3].all()) and not bool(has_nan[1::3].any())
    assert bool(torch.isnan(feat[has_nan]).all()) and bool(torch.isnan(pool_raw[has_nan]).all())
    assert torch.equal(amax.long()[has_nan], am[has_nan]), (kernel, sign)
    c.b_dev = b.cuda().double()
    keep = ~has_nan.any(dim=1)
    check_against_reference(c, feat[keep], amax[keep], pool_raw[keep], raw[keep], top[keep],
                            BF16_TOL if prec == "bf16" else FP32_TOL)


# ----------------------------------------------------------------------------------------------------------------------
# routing: every instance named above is launched
# ----------------------------------------------------------------------------------------------------------------------
def test_routing_every_forward_instance_launched(tmp_path):
    want = [fp32_instance(K, lo) for K in (1, 2, 3, 4, 5, 7) for lo in (96, 97)]

    def calls():
        for K in (1, 2, 3, 4, 5, 7):
            for lo in (96, 97):
                c = C(K=K, lout=lo, n=2, H=16)
                table, w, b, ids, mask, _, _ = _inputs(c, K)
                ops.conv_act_maxpool(table.cuda(), ids.cuda(), mask.cuda(), w.cuda(), b.cuda(), c.pad, precision="fp32")
        for flags in (SINGLE, PAIR):
            for K, mode in ((1, 1), (3, 2)):
                c = C(E=100, H=32, K=K, pad=0, L=60, n=4, gate=mode, prec="bf16", mask="none", all_pad=False)
                table, w, b, ids, _, gate, _ = _inputs(c, K)
                ops.conv_act_maxpool(table.cuda(), ids.cuda(), None, w.cuda(), b.cuda(), 0, act=TANH, precision="bf16",
                                     flags=flags, gate=gate.cuda(), gate_mode=mode, return_pool_raw=True)

    _, launched = _kernels_launched(calls, tmp_path)
    names = _names(launched)
    for k in want + ["conv_tc_kernel<1,", "conv_tc_kernel<3,", "conv_tc2_kernel<1,", "conv_tc2_kernel<3,"]:
        assert any(k in n for n in names), (k, sorted(set(names)))
