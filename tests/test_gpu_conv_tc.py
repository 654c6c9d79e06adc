"""GPU parity of the tcgen05 (bf16) conv kernel.  Two references:
 (1) the CPU oracle evaluated on bf16-ROUNDED table and weights — isolates the kernel logic (tiling, tap shifts,
     document packing, masks, arg-max) from the quantisation, so the tolerance can be tight (1e-3);
 (2) the fp32 oracle / reference goldens at BASELINE.json's bf16 tolerance (1e-2 relative)."""
import pytest
import torch

import rbr_b200
from conftest import Golden, grad_floor, rel_err
from oracle import rbr_oracle as orc
from rbr_b200 import ops, synth
from test_gpu_parity import DEEPCONN_CASES, NARRE_CASES, build_model, run_step

pytestmark = pytest.mark.gpu


@pytest.fixture(params=[ops.CONV_TC_SINGLE_CTA, ops.CONV_TC_PAIR_ONLY], ids=["cta1-cpasync", "pair-tma"])
def tc_flags(request):
    """Tests taking this fixture run on BOTH tensor-core kernels: conv_tc.cu (single CTA, cp.async operands) and
    conv_tc2.cu (CTA pair, cta_group::2, TMA gather4 operands), selected per call through the C-ABI's `flags` argument
    (either flag errors out instead of falling back)."""
    return request.param


def _bf16_round(t):
    return t.to(torch.bfloat16).to(torch.float32)


# (n_docs, L, V, E, H, k)  — covers: one K-step / many, one tile / many (long docs), several docs per tile (short docs),
# filter passes (H=150), ragged tail tiles, k=1 (no tap shift) / 3 / 5
SHAPES = [
    (5, 40, 50, 16, 16, 1),
    (5, 40, 50, 16, 16, 3),
    (7, 128, 80, 32, 24, 3),
    (3, 129, 80, 48, 40, 3),
    (9, 500, 300, 300, 100, 3),
    (33, 60, 300, 300, 150, 3),
    (40, 10, 60, 24, 20, 3),
    (6, 300, 200, 100, 200, 5),
    (300, 500, 2000, 300, 100, 3),
    # edge shapes: one document, documents shorter than the kernel's tile and than a warp, one filter, filters split into
    # passes (H=300), tiny / odd embedding widths, k=7 halo, odd number of documents for the CTA pair
    (1, 500, 300, 300, 100, 3),
    (1, 3, 20, 8, 1, 3),
    (3, 1, 20, 8, 5, 1),
    (65, 17, 90, 40, 33, 3),
    (11, 200, 400, 300, 300, 3),
    (9, 260, 300, 72, 48, 7),
    (130, 31, 500, 100, 200, 5),
]


@pytest.mark.parametrize("shape", SHAPES)
def test_conv_tc_vs_bf16_rounded_oracle(shape, tc_flags):
    n, L, V, E, H, k = shape
    gen = torch.Generator().manual_seed(n * 1000 + L)
    table = torch.randn(V, E, generator=gen)
    table[0] = 0
    w = (torch.rand(H, E, k, generator=gen) * 2 - 1) / (E * k) ** 0.5
    b = (torch.rand(H, generator=gen) * 2 - 1) * 0.1
    ids, mask = synth.doc_batch(n, L, V, seed=L + 5)
    mask = mask.clone()
    mask[0, min(3, L - 1)] = False                      # a real token masked out by the caller
    if n > 2:
        ids[2] = 0
        mask[2] = False                                  # fully padded document → relu(bias)
    feat, amax = ops.conv_act_maxpool(table.cuda(), ids.cuda(), mask.cuda(), w.cuda(), b.cuda(), (k - 1) // 2,
                                      precision="bf16", flags=tc_flags)
    x = orc.mask_rows(orc.embedding_gather(_bf16_round(table), ids), mask)
    y = orc.conv1d_same(x, _bf16_round(w), b)
    ref, ref_arg = orc.first_argmax_pool(torch.relu(y))
    assert rel_err(feat.cpu(), ref) < 1e-3
    # arg-max: the position the kernel reports attains the oracle's max up to fp32 summation-order noise
    pre = y.max(dim=1).values
    got = torch.gather(y, 1, amax.cpu().long().unsqueeze(1)).squeeze(1)
    assert float(((pre - got).abs() / pre.abs().clamp_min(1e-3)).max()) < 1e-5
    if n > 2:
        assert torch.allclose(feat[2].cpu(), torch.relu(b), atol=1e-6)


def test_conv_tc_tanh_and_no_mask(tc_flags):
    gen = torch.Generator().manual_seed(4)
    V, E, H, k, n, L = 100, 64, 32, 3, 6, 200
    table = torch.randn(V, E, generator=gen)
    w = (torch.rand(H, E, k, generator=gen) * 2 - 1) / (E * k) ** 0.5
    b = (torch.rand(H, generator=gen) * 2 - 1) * 0.1
    ids = torch.randint(0, V, (n, L), generator=gen)
    feat, _ = ops.conv_act_maxpool(table.cuda(), ids.cuda(), None, w.cuda(), b.cuda(), 1, act=ops.ACT_TANH, precision="bf16",
                                   flags=tc_flags)
    y = orc.conv1d_same(orc.embedding_gather(_bf16_round(table), ids), _bf16_round(w), b)
    assert rel_err(feat.cpu(), torch.tanh(y).max(dim=1).values) < 1e-3


def _rounded_params(params):
    """What the tensor-core kernel actually multiplies: bf16-rounded embedding table and conv weights."""
    out = dict(params)
    for k in params:
        if k == "word_embeddings.embedding.weight" or (k.startswith("ngram.") and k.endswith(".weight")):
            out[k] = _bf16_round(params[k])
    return out


def _fro_err(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-12))


@pytest.mark.parametrize("case", DEEPCONN_CASES + NARRE_CASES)
def test_golden_bf16(case, tc_flags):
    """End-to-end bf16 step.  Outputs against the reference's own numbers at the 1e-2 tolerance.  Gradients:
    (a) within 1e-2 of the oracle run on the bf16-rounded operands (same arg-max routing as the kernel);
    (b) against the fp32 reference on the Frobenius norm — bf16 rounding can move an arg-max to a near-tied
        position, which moves a whole gradient row (SURVEY.md §7), so max-abs is not a stable metric there."""
    g = Golden(case)
    model = build_model(g, "bf16")
    model.ngram.conv_flags = tc_flags
    out, loss, grads = run_step(model, g.batch, g.ratings)
    pred = out[0] if isinstance(out, tuple) else out
    assert rel_err(pred.detach().cpu(), g.out["pred"]) < 1e-2
    assert rel_err(loss, g.out["loss"]) < 1e-2
    rp, rl, rg = orc.loss_and_grads(g.model, _rounded_params(g.params), g.batch, g.ratings)
    assert rel_err(pred.detach().cpu(), rp) < 2e-3
    for k, ref in g.grads.items():
        assert rel_err(grads[k], rg[k], max(grad_floor(k), 1e-6)) < 1e-2, k
        if ref.abs().max() > 1e-6:
            assert _fro_err(grads[k], ref) < 1e-1, k


def test_seeded_midsize_bf16_vs_oracle(tc_flags):
    B, L, V, U, I, E, H, K = 24, 500, 3000, 50, 40, 300, 100, 32
    params = synth.deepconn_params(U, I, V, E, H, K, (3,), seed=1)
    batch, ratings = synth.deepconn_batch(B, L, V, U, I, seed=123)
    model = rbr_b200.DeepCoNNpp(U, I, V, [3], E, H, K, L, None, 0.0, precision="bf16")
    model.load_state_dict(params)
    model.cuda()
    model.ngram.conv_flags = tc_flags
    out, loss, grads = run_step(model, batch, ratings)
    rp, rl, rg = orc.loss_and_grads("deepconn", params, batch, ratings)
    assert rel_err(out.detach().cpu(), rp) < 1e-2
    assert rel_err(loss, rl) < 1e-2
    for k in rg:
        assert _fro_err(grads[k], rg[k]) < 1.5e-1, k      # arg-max flips under bf16 rounding move whole rows
    _, _, rgr = orc.loss_and_grads("deepconn", _rounded_params(params), batch, ratings)
    for k in rgr:
        assert rel_err(grads[k], rgr[k], 1e-7) < 1e-2, k


def test_bf16_full_batch_properties(tc_flags):
    """B=4096-sized run of the tensor-core path: deterministic, mask-invariant, permutation-equivariant, and
    equal (within bf16 tolerance) to the fp32 CUDA-core variant on the same inputs."""
    B, L, V, U, I, E, H, K = 1024, 500, 50000, 2000, 1200, 300, 100, 32
    params = synth.deepconn_params(U, I, V, E, H, K, (3,), seed=2)
    batch, _ = synth.deepconn_batch(B, L, V, U, I, seed=77)
    b = [t.cuda() for t in batch]
    preds = {}
    for prec in ("bf16", "fp32"):
        model = rbr_b200.DeepCoNNpp(U, I, V, [3], E, H, K, L, None, 0.5, precision=prec)
        model.load_state_dict(params)
        model.cuda().eval()
        model.ngram.conv_flags = tc_flags if prec == "bf16" else 0
        with torch.no_grad():
            preds[prec] = model(*b)
            if prec == "bf16":
                assert torch.equal(model(*b), preds[prec])
                scr = b[0].clone()
                scr[~b[2]] = 17
                assert torch.equal(model(scr, b[1], b[2], b[3], b[4], b[5]), preds[prec])
                perm = torch.randperm(B, device="cuda")
                assert torch.equal(model(*[t[perm] for t in b]), preds[prec][perm])
    assert rel_err(preds["bf16"].cpu(), preds["fp32"].cpu()) < 1e-2


def test_variants_agree_bitwise_on_values():
    """The two kernels issue the same K-step / tap order into fp32 TMEM accumulators: identical pooled values."""
    gen = torch.Generator().manual_seed(12)
    V, E, H, k, n, L = 4000, 300, 100, 3, 300, 500
    table = torch.randn(V, E, generator=gen)
    w = (torch.rand(H, E, k, generator=gen) * 2 - 1) / (E * k) ** 0.5
    b = (torch.rand(H, generator=gen) * 2 - 1) * 0.1
    ids, mask = synth.doc_batch(n, L, V, seed=99)
    outs = []
    for fl in (ops.CONV_TC_SINGLE_CTA, ops.CONV_TC_PAIR_ONLY):
        outs.append(ops.conv_act_maxpool(table.cuda(), ids.cuda(), mask.cuda(), w.cuda(), b.cuda(), 1, precision="bf16", flags=fl))
    assert torch.equal(outs[0][0], outs[1][0])
    assert torch.equal(outs[0][1], outs[1][1])


@pytest.mark.parametrize("L,k", [(500, 3), (1000, 5), (257, 3)])
def test_padding_tail_tiles_skipped_bitwise(L, k):
    """Long documents: the CTA-pair kernel runs only the 128-position tiles up to one position past each document's last
    token (conv_doc_tiles_* pre-pass, documents sorted by tile count).  Values AND arg-max must equal the single-CTA
    kernel's, which visits every tile — lengths sit on the tile boundaries, include empty and full documents, and one
    document has a masked-out hole followed by a late token."""
    gen = torch.Generator().manual_seed(L)
    V, E, H, n = 3000, 300, 100, 333
    table = torch.randn(V, E, generator=gen)
    w = (torch.rand(H, E, k, generator=gen) * 2 - 1) / (E * k) ** 0.5
    b = (torch.rand(H, generator=gen) * 2 - 1) * 0.1
    b[:H // 2] -= 1.0                                              # many units whose max is the padding value relu(bias) = 0
    table[:, :] = table.abs()
    w[:10] = -w[:10].abs()                                         # filters 0..9 answer < 0 on every window that holds a token: their
    #                                                                max is the 0 of the FIRST all-padding position, len + pad
    lens = torch.randint(0, L + 1, (n,), generator=gen)
    edge = [0, 1, 2, 125, 126, 127, 128, 129, 130, 254, 255, 256, 257, L - 2, L - 1, L]
    lens[:len(edge)] = torch.tensor([min(e, L) for e in edge])
    ids = torch.randint(1, V, (n, L), generator=gen)
    mask = torch.arange(L).unsqueeze(0) < lens.unsqueeze(1)
    mask[20, :] = False
    mask[20, min(L - 1, 200)] = True                               # a lone late token
    ids = ids * mask
    outs = []
    for fl in (ops.CONV_TC_SINGLE_CTA, ops.CONV_TC_PAIR_ONLY):
        outs.append(ops.conv_act_maxpool(table.cuda(), ids.cuda(), mask.cuda(), w.cuda(), b.cuda(), (k - 1) // 2, precision="bf16",
                                         flags=fl))
    assert torch.equal(outs[0][0], outs[1][0])
    assert torch.equal(outs[0][1], outs[1][1])
    pad = (k - 1) // 2
    short = (lens > 0) & (lens + pad < L + 2 * pad - k + 1)
    short[20] = False
    assert torch.equal(outs[1][1][short.cuda()][:, :10].cpu().long(), (lens[short] + pad).unsqueeze(1).expand(-1, 10))
    # and with the mask derived from the ids (id != 0), the int32 staging path
    f3, a3 = ops.conv_act_maxpool(table.cuda(), ids.int().cuda(), None, w.cuda(), b.cuda(), (k - 1) // 2, precision="bf16",
                                  flags=ops.CONV_TC_PAIR_ONLY, mask_from_ids=True)
    assert torch.equal(f3, outs[0][0]) and torch.equal(a3, outs[0][1])
    x = orc.mask_rows(orc.embedding_gather(_bf16_round(table), ids), mask)
    ref, _ = orc.first_argmax_pool(torch.relu(orc.conv1d_same(x, _bf16_round(w), b)))
    assert rel_err(outs[1][0].cpu(), ref) < 1e-3


# ----------------------------------------------------------------------------------------------------------------------
# K2c: dense tensor-core backward (coefficient matrix + two tcgen05 GEMMs, conv_bwd_tc.cu) against the arg-max-sparse
# CUDA-core kernels (K2b) and the oracle.  (n_docs per side, L, V, E, H, k)
# ----------------------------------------------------------------------------------------------------------------------
BWD_SHAPES = [
    (5, 40, 50, 16, 16, 3),          # one M tile, one N chunk, one token block
    (9, 129, 300, 64, 40, 3),
    (33, 60, 700, 300, 150, 3),      # NARRE dims: HJ = 450 → 512 columns, 5 N chunks (two MMA groups)
    (24, 500, 3000, 300, 100, 3),    # DeepCoNN dims: HJ = 300 → 320
    (40, 10, 90, 24, 20, 5),
    (12, 200, 5000, 100, 200, 1),    # k = 1, two N chunks, vocabulary spanning many token blocks and split-K slices
    (7, 64, 130, 128, 8, 7),
    (3, 33, 20000, 300, 100, 3),     # most of the vocabulary untouched: zero rows
]


def _encode_step(shape, flags, seed, freeze_table=False):
    n, L, V, E, H, k = shape
    U, I, K = 7, 6, 8
    params = synth.deepconn_params(U, I, V, E, H, K, (k,), seed=seed)
    batch, ratings = synth.deepconn_batch(n, L, V, U, I, seed=seed + 1)
    model = rbr_b200.DeepCoNNpp(U, I, V, [k], E, H, K, L, None, 0.0, precision="bf16")
    model.load_state_dict(params)
    model.cuda().train()
    model.ngram.conv_flags = flags
    if freeze_table:
        model.word_embeddings.embedding.weight.requires_grad_(False)
    out, loss, grads = None, None, None
    model.zero_grad(set_to_none=True)
    pred = model(*[t.cuda() for t in batch])
    loss = torch.nn.MSELoss()(pred, ratings.cuda())
    loss.backward()
    grads = {kk: p.grad.detach().cpu() for kk, p in model.named_parameters() if p.grad is not None}
    return params, batch, ratings, pred.detach().cpu(), grads, model


@pytest.mark.parametrize("shape", BWD_SHAPES)
def test_dense_tc_backward_matches_sparse_kernels_and_oracle(shape):
    params, batch, ratings, pred_d, g_dense, model = _encode_step(shape, ops.CONV_BWD_DENSE_TC, seed=shape[0] + shape[1])
    _, _, _, pred_s, g_sparse, _ = _encode_step(shape, ops.CONV_BWD_SPARSE, seed=shape[0] + shape[1])
    assert torch.equal(pred_d, pred_s)
    for kk in g_sparse:
        # same operands (bf16 shadow rows, bf16-rounded weights), same routing: only the summation order and the 2^-17 split differ
        assert rel_err(g_dense[kk], g_sparse[kk], 1e-9) < 2e-4, kk
    _, _, rg = orc.loss_and_grads("deepconn", _rounded_params(params), batch, ratings)
    for kk in rg:
        assert rel_err(g_dense[kk], rg[kk], 1e-7) < 1e-2, kk
    assert float(g_dense["word_embeddings.embedding.weight"][0].abs().max()) == 0.0                  # padding row
    # a second step on the same model reuses the workspace (C32 re-zeroed per block, weight scratch left zeroed): same gradients
    model.zero_grad(set_to_none=True)
    loss = torch.nn.MSELoss()(model(*[t.cuda() for t in batch]), ratings.cuda())
    loss.backward()
    for kk, p in model.named_parameters():
        assert rel_err(p.grad.cpu(), g_dense[kk], 1e-9) < 1e-5, kk


def test_dense_tc_backward_with_frozen_table_and_table_hook():
    shape = (9, 129, 300, 64, 40, 3)
    _, _, _, _, g_ref, _ = _encode_step(shape, ops.CONV_BWD_SPARSE, seed=5)
    _, _, _, _, g_frozen, _ = _encode_step(shape, ops.CONV_BWD_DENSE_TC, seed=5, freeze_table=True)
    assert "word_embeddings.embedding.weight" not in g_frozen
    for kk in g_frozen:
        assert rel_err(g_frozen[kk], g_ref[kk], 1e-9) < 2e-4, kk
    # data-parallel split: table part, hook, then weight part
    n, L, V, E, H, k = shape
    params = synth.deepconn_params(7, 6, V, E, H, 8, (k,), seed=5)
    batch, ratings = synth.deepconn_batch(n, L, V, 7, 6, seed=6)
    model = rbr_b200.DeepCoNNpp(7, 6, V, [k], E, H, 8, L, None, 0.0, precision="bf16")
    model.load_state_dict(params)
    model.cuda().train()
    seen = {}
    model.ngram.table_grad_hook = lambda t: seen.setdefault("table", t.detach().clone())
    torch.nn.MSELoss()(model(*[t.cuda() for t in batch]), ratings.cuda()).backward()
    assert rel_err(seen["table"].cpu(), g_ref["word_embeddings.embedding.weight"], 1e-9) < 2e-4
    for kk, p in model.named_parameters():
        assert rel_err(p.grad.cpu(), g_ref[kk], 1e-9) < 2e-4, kk


@pytest.mark.parametrize("L,k,pad,n,H", [(500, 3, 1, 300, 100), (30, 3, 1, 4001, 150), (60, 5, 2, 777, 100), (200, 1, 0, 130, 64),
                                         (129, 4, 0, 67, 100), (1000, 7, 3, 70, 50), (14, 2, 0, 999, 100)])
@pytest.mark.parametrize("width", [64, 32, 16])
def test_row_index_table_equals_index_warp(L, k, pad, n, H, width):
    """The CTA-pair kernel gets its tile row indices either from the row-index table (conv_rowidx_kernel + bulk copies into
    the index buffers) or from its index warp resolving ids / masks itself, and with no scratch at all (no document selection):
    all three must agree bit for bit, and with the single-CTA kernel.  Short documents (several per tile, all-padding documents
    dropped), long ones (tile skipping), k = 1 (no halo rows), explicit masks and masks derived from int32 / uint16 ids."""
    gen = torch.Generator().manual_seed(L * 31 + k)
    V, E = 2000, 300 if L < 600 else 64
    table = torch.randn(V, E, generator=gen)
    w = (torch.rand(H, E, k, generator=gen) * 2 - 1) / (E * k) ** 0.5
    b = (torch.rand(H, generator=gen) * 2 - 1) * 0.1
    lens = torch.randint(0, L + 1, (n,), generator=gen)
    lens[::7] = 0                                                  # all-padding documents
    lens[1::11] = L
    ids = torch.randint(1, V, (n, L), generator=gen)
    mask = torch.arange(L).unsqueeze(0) < lens.unsqueeze(1)
    i32 = width != 64
    if not i32:
        mask = mask & (torch.rand(n, L, generator=gen) > 0.05)    # holes: an explicit mask that disagrees with ids != 0
    else:
        ids = ids * mask
    args = dict(precision="bf16")
    if i32:
        narrow = ids.int().cuda() if width == 32 else ids.to(torch.uint16).cuda()
        call = lambda **kw: ops.conv_act_maxpool(table.cuda(), narrow, None, w.cuda(), b.cuda(), pad, mask_from_ids=True, **args, **kw)
    else:
        call = lambda **kw: ops.conv_act_maxpool(table.cuda(), ids.cuda(), mask.cuda(), w.cuda(), b.cuda(), pad, **args, **kw)
    ref = call(flags=ops.CONV_TC_SINGLE_CTA)
    for kw in (dict(), dict(row_index_table=False), dict(select_docs=False)):
        out = call(flags=ops.CONV_TC_PAIR_ONLY, **kw)
        assert torch.equal(out[0], ref[0]), kw
        assert torch.equal(out[1], ref[1]), kw
