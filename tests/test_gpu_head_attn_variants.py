"""Every kernel variant of the rating head (K4, csrc/head.cu) and of the per-side NARRE attention (K3, csrc/attn.cu) against the
float64 oracle, at the shapes that select it.

Both entry points pick a kernel by shape, batch size and pointer alignment:

  head forward    head_fwd2_kernel<4>   latent % 4 == 0, batch <= 9472 (16-sample CTAs, at most 592: never loops)
                  head_fwd2_kernel<8>   latent % 4 == 0, batch > 9472 (32-sample CTAs; they loop once batch > 18944)
                  head_fwd_kernel       otherwise (8 samples per CTA, at most 296 CTAs: loops once batch > 2368)
  head backward   head_bwd2_kernel<8>   latent % 4 == 0 (32-sample tiles, at most 592 CTAs: loops once batch > 18944)
                  head_bwd_kernel       otherwise (32-sample tiles, at most 296 CTAs: loops once batch > 9472)
  attention       narre_attn2_*         att_dim <= 32, hidden <= 160 and the per-warp staging fits shared memory (the
                                        backward needs more, so large R can run attn2 forward with the generic backward)
                  narre_attn_*          att_dim up to 128 with 8/4/2/1 warps per CTA, as many as fit (at most 296 CTAs)

Each case names the kernels it targets; test_routing_runs_the_targeted_kernels checks under torch.profiler that they, and
only they, ran, and that the cases together run every kernel with a single round of CTAs and with CTAs that loop.

Tolerances are BASELINE's: 1e-5 on outputs, 3e-5 on batch-summed gradients.  Inputs are screened so that no ReLU input lies
within 2e-5 of zero in float64 (fp32 summation-order noise is ~1e-7 here): a ReLU that opens on one side of the comparison
and closes on the other would move a whole gradient term.
"""
import collections
import json

import pytest
import torch

from conftest import grad_floor, rel_err
from oracle import rbr_oracle as orc
from rbr_b200 import layers, ops
from rbr_b200._lib import lib

pytestmark = pytest.mark.gpu
FP32_TOL, FP32_GRAD_TOL = 1e-5, 3e-5
TAU = 2e-5                       # ReLU screening margin (float64 pre-activation)

# ----------------------------------------------------------------------------------------------------------------------
# rating head: LastFeat x2 + FM (+ fused MSE)
# ----------------------------------------------------------------------------------------------------------------------
# padding rows of LastFeat_u.ebd, LastFeat_i.ebd, FM.user_bias, FM.item_bias: distinct, so a mixed-up index shows
HEAD_PADS = (1, 2, 3, 4)
HeadCase = collections.namedtuple("HeadCase", "B H K loss drop hot offset fwd bwd")
# loss: the fused-MSE form (HeadLossFn) instead of pred.backward(g) (HeadFn); hot: 6 users / 7 items, so every id repeats
# thousands of times (the embedding-gradient atomics); offset: text features at storage offset 1 (not 16-byte aligned: the
# scalar staging path, vec = 0)
HEAD_CASES = {
    "fwd2<4>+bwd2_one_tile_K32": HeadCase(64, 100, 32, False, 0.0, False, False, "head_fwd2_kernel<4>", "head_bwd2_kernel<8>"),
    "fwd2<4>_last_batch_9472_K36_drop": HeadCase(9472, 52, 36, True, 0.5, True, False, "head_fwd2_kernel<4>", "head_bwd2_kernel<8>"),
    "fwd2<8>_first_batch_9473_K64_offset": HeadCase(9473, 64, 64, False, 0.0, False, True, "head_fwd2_kernel<8>", "head_bwd2_kernel<8>"),
    "fwd2<8>+bwd2_loop_18945_K128": HeadCase(18945, 100, 128, True, 0.0, False, False, "head_fwd2_kernel<8>", "head_bwd2_kernel<8>"),
    "fwd2<8>+bwd2_loop_K100_H150_drop": HeadCase(24000, 150, 100, False, 0.5, False, False, "head_fwd2_kernel<8>", "head_bwd2_kernel<8>"),
    "fwd2<4>+bwd2_H7_K64_offset": HeadCase(777, 7, 64, True, 0.0, True, True, "head_fwd2_kernel<4>", "head_bwd2_kernel<8>"),
    "fwd2<4>+bwd2_K128_H128_offset": HeadCase(100, 128, 128, False, 0.0, False, True, "head_fwd2_kernel<4>", "head_bwd2_kernel<8>"),
    "scalar_K1_partial_tile": HeadCase(5, 12, 1, False, 0.0, False, False, "head_fwd_kernel", "head_bwd_kernel"),
    "scalar_fwd_one_round_2368_K5_drop": HeadCase(2368, 40, 5, True, 0.5, False, False, "head_fwd_kernel", "head_bwd_kernel"),
    "scalar_fwd_loop_2369_K31": HeadCase(2369, 100, 31, False, 0.0, True, False, "head_fwd_kernel", "head_bwd_kernel"),
    "scalar_bwd_one_round_9472_K33_drop": HeadCase(9472, 64, 33, False, 0.5, False, False, "head_fwd_kernel", "head_bwd_kernel"),
    "scalar_bwd_loop_9473_K33_H150": HeadCase(9473, 150, 33, True, 0.0, False, False, "head_fwd_kernel", "head_bwd_kernel"),
    "scalar_loop_20000_K5_hot_offset": HeadCase(20000, 30, 5, True, 0.0, True, True, "head_fwd_kernel", "head_bwd_kernel"),
}
# samples one CTA covers per round, and the grid cap (csrc/head.cu rbr_head_fwd / rbr_head_bwd)
HEAD_CTA = {"head_fwd2_kernel<4>": (16, 592), "head_fwd2_kernel<8>": (32, 592), "head_bwd2_kernel<8>": (32, 592),
            "head_fwd_kernel": (8, 296), "head_bwd_kernel": (32, 296)}


def _uniform(gen, shape, lo, hi):
    return torch.rand(*shape, generator=gen) * (hi - lo) + lo


def _head_build(c: HeadCase, seed: int, screen: bool = True):
    """Modules with seeded parameters, text features (fp32, on the device, possibly at storage offset 1), ids, ratings and the
    upstream gradient of pred."""
    gen = torch.Generator().manual_seed(seed)
    U, I = (6, 7) if c.hot else (5000, 3000)
    uf = layers.LastFeat(U, c.H, c.K, padding_idx=HEAD_PADS[0])
    itf = layers.LastFeat(I, c.H, c.K, padding_idx=HEAD_PADS[1])
    fm = layers.FM(U, I, c.K, c.drop, user_padding_idx=HEAD_PADS[2], item_padding_idx=HEAD_PADS[3])
    with torch.no_grad():
        for lf in (uf, itf):
            lf.W.copy_(_uniform(gen, lf.W.shape, -0.1, 0.1))
            lf.b.copy_(_uniform(gen, lf.b.shape, -0.1, 0.1))
            lf.ebd.weight.copy_(_uniform(gen, lf.ebd.weight.shape, -0.3, 0.3))      # padding rows too: the forward reads them
        fm.h.copy_(_uniform(gen, fm.h.shape, -0.5, 0.5))
        fm.user_bias.weight.copy_(_uniform(gen, fm.user_bias.weight.shape, -0.1, 0.1))
        fm.item_bias.weight.copy_(_uniform(gen, fm.item_bias.weight.shape, -0.1, 0.1))
        fm.g_bias.fill_(0.1)
    uf, itf, fm = uf.cuda(), itf.cuda(), fm.cuda()
    uid = torch.randint(0, U, (c.B,), generator=gen)
    iid = torch.randint(0, I, (c.B,), generator=gen)
    uid[0::7], uid[3::7] = HEAD_PADS[0], HEAD_PADS[2]                  # every padding row is hit
    iid[1::7], iid[5::7] = HEAD_PADS[1], HEAD_PADS[3]
    uid, iid = uid.cuda(), iid.cuda()
    ut = torch.randn(c.B, c.H, generator=gen).cuda() * 0.5
    it = torch.randn(c.B, c.H, generator=gen).cuda() * 0.5
    if screen:
        # resample the text rows of samples with an FM ReLU input u_lat * i_lat within TAU of 0 (float64)
        W = [p.detach().double() for p in (uf.W, uf.b, uf.ebd.weight, itf.W, itf.b, itf.ebd.weight)]
        for _ in range(50):
            ul = orc.last_feat(ut.double(), uid, *W[:3])
            il = orc.last_feat(it.double(), iid, *W[3:])
            bad = ((ul * il).abs() < TAU).any(dim=1).nonzero().flatten()
            if bad.numel() == 0:
                break
            ut[bad] = torch.randn(bad.numel(), c.H, generator=gen).cuda() * 0.5
            it[bad] = torch.randn(bad.numel(), c.H, generator=gen).cuda() * 0.5
        assert bad.numel() == 0
    if c.offset:
        texts = []
        for t in (ut, it):
            buf = torch.empty(c.B * c.H + 1, device=t.device)
            v = buf[1:].view(c.B, c.H)
            v.copy_(t)
            assert v.is_contiguous() and v.data_ptr() % 16 != 0
            texts.append(v)
        ut, it = texts
    ratings = torch.randint(1, 6, (c.B,), generator=gen).float().cuda()
    g_pred = torch.randn(c.B, generator=gen).cuda()
    return uf, itf, fm, ut.requires_grad_(True), it.requires_grad_(True), uid, iid, ratings, g_pred


def _head_params(uf, itf, fm):
    """(name, parameter, padding row or None) in the order of the oracle's arguments."""
    return [("user_feat.W", uf.W, None), ("user_feat.b", uf.b, None), ("user_feat.ebd", uf.ebd.weight, HEAD_PADS[0]),
            ("item_feat.W", itf.W, None), ("item_feat.b", itf.b, None), ("item_feat.ebd", itf.ebd.weight, HEAD_PADS[1]),
            ("fm.h", fm.h, None), ("fm.user_bias", fm.user_bias.weight, HEAD_PADS[2]),
            ("fm.item_bias", fm.item_bias.weight, HEAD_PADS[3]), ("fm.g_bias", fm.g_bias, None)]


def _head_run(c: HeadCase, uf, itf, fm, ut, it, uid, iid, ratings, g_pred):
    if c.loss:
        loss, pred = layers.fused_head(uf, itf, fm, ut, it, uid, iid, True, None, ratings=ratings)
        loss.backward()
        return pred, loss
    pred = layers.fused_head(uf, itf, fm, ut, it, uid, iid, True, None)
    pred.backward(g_pred)
    return pred, None


@pytest.mark.parametrize("name", list(HEAD_CASES))
def test_head_variant_vs_float64_oracle(name):
    """pred, loss, every parameter gradient and both text-feature gradients; padding rows get exactly zero gradient."""
    c = HEAD_CASES[name]
    uf, itf, fm, ut, it, uid, iid, ratings, g_pred = _head_build(c, seed=c.B + c.H + c.K)
    pred, loss = _head_run(c, uf, itf, fm, ut, it, uid, iid, ratings, g_pred)
    p, seed, _ = fm.__dict__["_rbr_last_drop"]
    assert p == c.drop
    keep = ops.head_dropout_mask(c.B, c.K, p, seed, None).double() if p > 0 else None
    prm = _head_params(uf, itf, fm)
    leaves = [q.detach().double().requires_grad_(True) for _, q, _ in prm]
    ut64, it64 = ut.detach().double().requires_grad_(True), it.detach().double().requires_grad_(True)
    ul = orc.last_feat(ut64, uid, *leaves[0:3])
    il = orc.last_feat(it64, iid, *leaves[3:6])
    pred64 = orc.fm_head(ul, il, uid, iid, leaves[6], leaves[9], leaves[7], leaves[8], drop_mask=keep).view(-1)
    assert rel_err(pred.detach(), pred64.detach()) < FP32_TOL
    if c.loss:
        loss64 = orc.mse_loss(pred64, ratings.double())
        assert rel_err(loss.detach(), loss64.detach()) < FP32_TOL
        loss64.backward()
    else:
        pred64.backward(g_pred.double())
    assert rel_err(ut.grad, ut64.grad) < FP32_GRAD_TOL
    assert rel_err(it.grad, it64.grad) < FP32_GRAD_TOL
    for (key, q, pad), ref in zip(prm, leaves):
        g = ref.grad.clone()
        if pad is not None:
            g[pad] = 0                                   # nn.Embedding(padding_idx=pad)
            assert float(q.grad[pad].abs().max()) == 0.0, key
        assert rel_err(q.grad, g) < FP32_GRAD_TOL, key


def test_head_outside_shared_memory_raises():
    """A head shape neither kernel takes raises the library's RuntimeError; it does not return numbers."""
    # latent 128, hidden 140: the forward fits (fwd2) but no backward kernel does
    c = HeadCase(64, 140, 128, False, 0.0, False, False, None, None)
    uf, itf, fm, ut, it, uid, iid, ratings, g_pred = _head_build(c, seed=1, screen=False)
    pred = layers.fused_head(uf, itf, fm, ut, it, uid, iid, True, None)
    with pytest.raises(RuntimeError, match="rbr_head_bwd"):
        pred.backward(g_pred)
    # hidden 200: not even the forward fits
    c = HeadCase(64, 200, 128, True, 0.0, False, False, None, None)
    uf, itf, fm, ut, it, uid, iid, ratings, g_pred = _head_build(c, seed=2, screen=False)
    with pytest.raises(RuntimeError, match="rbr_head_fwd"):
        layers.fused_head(uf, itf, fm, ut, it, uid, iid, True, None, ratings=ratings)
    # latent 129: past the four lanes per latent column
    c = HeadCase(8, 16, 129, False, 0.0, False, False, None, None)
    uf, itf, fm, ut, it, uid, iid, ratings, g_pred = _head_build(c, seed=3, screen=False)
    with pytest.raises(RuntimeError, match="latent_dim"):
        layers.fused_head(uf, itf, fm, ut, it, uid, iid, True, None)


def test_score_cached_2pow20_pairs_vs_float64_oracle():
    """PairScorer.score_cached at 2^20 + 3 pairs (head_fwd2_kernel<8>, CTAs looping: what bench.py --pairs scores) against
    the oracle's encoder and head in float64, fp32 model."""
    import rbr_b200
    from rbr_b200 import synth
    from rbr_b200.inference import PairScorer
    U, I, V, E, H, K, L, N = 300, 200, 5000, 64, 100, 32, 120, (1 << 20) + 3
    params = synth.deepconn_params(U, I, V, E, H, K, (3,), seed=6)
    model = rbr_b200.DeepCoNNpp(U, I, V, [3], E, H, K, L, None, 0.5, precision="fp32")
    model.load_state_dict(params)
    scorer = PairScorer(model.cuda())
    user_docs, _ = synth.doc_batch(U, L, V, seed=3)
    item_docs, _ = synth.doc_batch(I, L, V, seed=4)
    user_docs[0] = 0
    item_docs[0] = 0
    user_docs, item_docs = user_docs.cuda(), item_docs.cuda()
    scorer.build_cache(user_docs, item_docs, chunk=128)
    gen = torch.Generator().manual_seed(5)
    u_ids = torch.randint(0, U, (N,), generator=gen).cuda()
    i_ids = torch.randint(0, I, (N,), generator=gen).cuda()
    cached = scorer.score_cached(u_ids, i_ids)
    p64 = {k: v.cuda().double() for k, v in params.items()}
    w = [p64["ngram.feature_layer.0.list_of_conv1d.0.weight"]]
    b = [p64["ngram.feature_layer.0.list_of_conv1d.0.bias"]]
    table = p64["word_embeddings.embedding.weight"]
    u_feat = orc.ngram_feat(orc.embedding_gather(table, user_docs), user_docs != 0, w, b)     # one document per entity
    i_feat = orc.ngram_feat(orc.embedding_gather(table, item_docs), item_docs != 0, w, b)
    assert rel_err(scorer.user_feat, u_feat) < FP32_TOL and rel_err(scorer.item_feat, i_feat) < FP32_TOL
    ul = orc.last_feat(u_feat[u_ids], u_ids, p64["user_feat.W"], p64["user_feat.b"], p64["user_feat.ebd.weight"])
    il = orc.last_feat(i_feat[i_ids], i_ids, p64["item_feat.W"], p64["item_feat.b"], p64["item_feat.ebd.weight"])
    ref = orc.fm_head(ul, il, u_ids, i_ids, p64["fm.h"], p64["fm.g_bias"], p64["fm.user_bias.weight"],
                      p64["fm.item_bias.weight"]).view(-1)
    assert cached.shape == (N,)
    assert rel_err(cached, ref) < FP32_TOL


# ----------------------------------------------------------------------------------------------------------------------
# per-side NARRE attention: layers.LinearAttention (ops.NarreAttnFn)
# ----------------------------------------------------------------------------------------------------------------------
ATTN_PAD = 3
AttnCase = collections.namedtuple("AttnCase", "B R H A scores oob fwd bwd")
# scores: the loss also reads the attention scores (else the score gradient is None); oob: some review ids lie outside the
# id table (read as zero rows and counted).  fwd / bwd: targeted kernel and its warps per CTA
A2F, A2B, GF, GB = "narre_attn2_fwd_kernel", "narre_attn2_bwd_kernel", "narre_attn_fwd_kernel", "narre_attn_bwd_kernel"
ATTN_CASES = {
    "attn2_R1": AttnCase(37, 1, 150, 32, False, False, (A2F, 8), (A2B, 8)),
    "attn2_R5_loop": AttnCase(3000, 5, 8, 5, True, True, (A2F, 8), (A2B, 8)),
    "attn2_R6_A17": AttnCase(64, 6, 100, 17, True, False, (A2F, 8), (A2B, 8)),
    "attn2_R11_H160_loop": AttnCase(2369, 11, 160, 32, False, True, (A2F, 8), (A2B, 8)),
    "attn2_R11_H157": AttnCase(50, 11, 157, 32, True, False, (A2F, 8), (A2B, 8)),
    "attn2_fwd_generic4_bwd_R26": AttnCase(40, 26, 160, 32, True, False, (A2F, 8), (GB, 4)),
    "attn2_fwd_generic8_bwd_R32_A1_loop": AttnCase(2400, 32, 4, 1, False, True, (A2F, 8), (GB, 8)),
    "generic8_A33": AttnCase(300, 10, 150, 33, True, True, (GF, 8), (GB, 8)),
    "generic8_4_A64_bwd_loop": AttnCase(1200, 10, 150, 64, False, False, (GF, 8), (GB, 4)),
    "generic8_4_A100": AttnCase(200, 4, 100, 100, True, True, (GF, 8), (GB, 4)),
    "generic8_1_A128_bwd_loop": AttnCase(300, 3, 64, 128, True, False, (GF, 8), (GB, 1)),
    "generic4_2_R40_loop": AttnCase(1200, 40, 100, 64, True, True, (GF, 4), (GB, 2)),
    "generic2_1_R60_loop": AttnCase(700, 60, 150, 64, False, False, (GF, 2), (GB, 1)),
    "generic1_1_R60_H300_loop": AttnCase(300, 60, 300, 32, True, True, (GF, 1), (GB, 1)),
    "generic8_4_H300_loop": AttnCase(2400, 10, 300, 32, False, True, (GF, 8), (GB, 4)),
}
ATTN_CTA_CAP = 296                # at most 2 CTAs per SM; a CTA covers one sample per warp per round


def _attn_build(c: AttnCase, seed: int, screen: bool = True):
    gen = torch.Generator().manual_seed(seed)
    n_ids = 40
    att = layers.LinearAttention(n_ids, c.H, c.A, 0.0, padding_idx=ATTN_PAD)
    with torch.no_grad():
        att.W_rv.copy_(_uniform(gen, (c.H, c.A), -0.1, 0.1))
        att.W_id.copy_(_uniform(gen, (c.A, c.A), -0.1, 0.1))
        att.h.copy_(_uniform(gen, (c.A, 1), -0.3, 0.3))
        att.b_1.copy_(_uniform(gen, (c.A,), -0.1, 0.1))
        att.b_2.fill_(0.1)
        att.ebd_vals.weight.copy_(torch.randn(n_ids, c.A, generator=gen) * 0.5)
    att = att.cuda()
    feat = (torch.randn(c.B, c.R, c.H, generator=gen).abs() * 0.5).cuda()           # pooled ReLU features are non-negative
    oid = torch.randint(0, n_ids, (c.B, c.R), generator=gen)
    oid[:, -1] = ATTN_PAD                                                            # a padded review per sample
    if c.oob:
        oid[1::9, 0], oid[2::9, 0], oid[4::9, 0] = -1, n_ids, n_ids + 1000
    oid = oid.cuda()
    if screen:
        # resample the features of samples with an attention hidden unit whose input is within TAU of 0 (float64)
        valid = (oid >= 0) & (oid < n_ids)
        e = torch.where(valid.unsqueeze(-1), att.ebd_vals.weight.detach().double()[oid.clamp(0, n_ids - 1)], 0.0)
        eW = e @ att.W_id.detach().double() + att.b_1.detach().double()
        for _ in range(50):
            pre = feat.double() @ att.W_rv.detach().double() + eW
            bad = (pre.abs() < TAU).flatten(1).any(dim=1).nonzero().flatten()
            if bad.numel() == 0:
                break
            feat[bad] = (torch.randn(bad.numel(), c.R, c.H, generator=gen).abs() * 0.5).cuda()
        assert bad.numel() == 0
    g_out = torch.randn(c.B, c.H, generator=gen).cuda()
    g_sc = (torch.randn(c.B, c.R, 1, generator=gen) * 0.1).cuda()
    return att, feat, oid, g_out, g_sc


def _attn_run(c: AttnCase, att, feat, oid, g_out, g_sc):
    fg = feat.clone().requires_grad_(True)
    out, sc = att(fg, oid)
    loss = (out * g_out).sum()
    if c.scores:
        loss = loss + (sc * g_sc).sum()
    loss.backward()
    return fg, out, sc


@pytest.mark.parametrize("name", list(ATTN_CASES))
def test_attention_variant_vs_float64_oracle(name):
    """out, scores, the feature gradient and the gradients of all six parameters; the padding row gets no gradient, and
    out-of-range ids are read as zero rows and counted once per review."""
    c = ATTN_CASES[name]
    att, feat, oid, g_out, g_sc = _attn_build(c, seed=c.B + c.R + c.H + c.A)
    n_ids = att.ebd_vals.weight.shape[0]
    lib.rbr_consume_oob_count(None)                                   # start from a clean counter
    fg, out, sc = _attn_run(c, att, feat, oid, g_out, g_sc)
    n_oob = int(((oid < 0) | (oid >= n_ids)).sum())
    assert lib.rbr_consume_oob_count(None) == n_oob and (n_oob > 0) == c.oob
    # oracle: out-of-range ids index an appended zero row that is not a parameter
    prm = [att.W_rv, att.W_id, att.h, att.b_1, att.b_2, att.ebd_vals.weight]
    leaves = [p.detach().double().requires_grad_(True) for p in prm]
    f64 = feat.double().requires_grad_(True)
    ebd_ext = torch.cat([leaves[5], leaves[5].new_zeros(1, c.A)])
    oid_ext = torch.where((oid >= 0) & (oid < n_ids), oid, n_ids)
    ro, rs = orc.linear_attention(f64, oid_ext, *leaves[:5], ebd_ext)
    assert rel_err(out.detach(), ro.detach()) < FP32_TOL
    assert rel_err(sc.detach(), rs.detach()) < FP32_TOL
    loss64 = (ro * g_out.double()).sum()
    if c.scores:
        loss64 = loss64 + (rs * g_sc.double()).sum()
    loss64.backward()
    assert rel_err(fg.grad, f64.grad) < FP32_GRAD_TOL
    for name_p, p, ref in zip(("W_rv", "W_id", "h", "b_1", "b_2", "ebd_vals"), prm, leaves):
        g = ref.grad.clone()
        if name_p == "ebd_vals":
            g[ATTN_PAD] = 0                                            # nn.Embedding(padding_idx=ATTN_PAD)
            assert float(p.grad[ATTN_PAD].abs().max()) == 0.0
        # d loss / d b_2 is ~0 by the softmax's shift invariance: what any implementation stores there is the rounding noise of a
        # sum of B*R terms of size |d logit| (as in test_attention_pair_tensor_core_kernels_vs_oracle)
        floor = float(c.B * c.R) ** 0.5 * 0.1 if name_p == "b_2" else 1e-6
        if c.R == 1:
            # one review: the score is 1 / (1 + 1e-8) and every logit gradient is ~1e-8 of the upstream gradient, below fp32's
            # resolution of the score (the kernel's is exactly 0).  The parameters only see those logit gradients (~1e-7 here),
            # so they are compared on an absolute scale (3e-6) instead of relative to themselves.
            floor = max(floor, 0.1)
        assert rel_err(p.grad, g, floor) < FP32_GRAD_TOL, name_p


def test_attention_outside_shared_memory_raises():
    """att_dim 128 at hidden 150: the generic forward fits, no backward does — the backward raises the library's RuntimeError.
    att_dim 129 is refused by the forward."""
    c = AttnCase(8, 4, 150, 128, False, False, None, None)
    att, feat, oid, g_out, g_sc = _attn_build(c, seed=1, screen=False)
    fg = feat.clone().requires_grad_(True)
    out, sc = att(fg, oid)
    assert torch.isfinite(out).all()
    with pytest.raises(RuntimeError, match="rbr_narre_attn_bwd"):
        (out * g_out).sum().backward()
    c = AttnCase(8, 4, 16, 129, False, False, None, None)
    att, feat, oid, g_out, g_sc = _attn_build(c, seed=2, screen=False)
    with pytest.raises(RuntimeError, match="rbr_narre_attn_fwd"):
        att(feat, oid)


# ----------------------------------------------------------------------------------------------------------------------
# NARRE on the per-side attention path (narre.py _encode_attend: item side on an auxiliary stream)
# ----------------------------------------------------------------------------------------------------------------------
def _narre(att_dim, seed, B=24):
    import rbr_b200
    from rbr_b200 import synth
    U, I, V, E, H, K, R, T = 50, 40, 3000, 100, 100, 32, 10, 40
    params = synth.narre_params(U, I, V, E, H, att_dim, K, (3,), seed=seed)
    model = rbr_b200.NARRE(U, I, V, [3], H, E, att_dim, K, R, T, 0.0, 0, 0, 0, None, "CNN", precision="fp32")
    model.load_state_dict(params)
    model.cuda().train()
    batches = []
    for s in range(3):
        b, r = synth.narre_batch(B, R, T, V, U, I, seed=seed + 1 + s)
        batches.append(([t.cuda() for t in b], r.cuda()))
    return model, params, batches


@pytest.mark.parametrize("att_dim, fused", [(64, True), (32, False)])
def test_narre_per_side_attention_step_vs_oracle(att_dim, fused, tmp_path):
    """One fp32 NARRE step where the two-sided tensor-core attention is not used — att_dim 64, which it declines, or
    fused_attention = False — against the oracle: pred, scores, loss and every parameter gradient."""
    from test_gpu_benchcfg import _clear_relu_margins
    model, params, batches = _narre(att_dim, seed=11)
    model.fused_attention = fused
    R, H = model.doc_num, model.hiddem_dim
    assert ops.narre_attn_pair_supported(R, H, att_dim) == (att_dim <= 32)
    batch, ratings = batches[0]
    p64 = {k: v.cuda().double() for k, v in params.items()}
    _clear_relu_margins("narre", p64, batch)
    T = batch[0].shape[-1]
    with torch.no_grad():
        _, _, ua, ia = model.ngram.encode(model.word_embeddings, [batch[0].view(-1, T), batch[1].view(-1, T)],
                                          [batch[2].view(-1, T), batch[3].view(-1, T)], return_argmax=True)
    res = {}

    def step():
        model.zero_grad(set_to_none=True)
        res["out"] = model(*batch)
        res["loss"] = torch.nn.MSELoss()(res["out"][0], ratings)
        res["loss"].backward()
    launched = _kernels_launched(step, tmp_path)
    names = "".join(n for n, _, _ in launched)
    assert "narre_attn_tc" not in names and names.count("narre_attn") == 4          # two sides, forward and backward
    pred, u_sc, i_sc = res["out"]
    _, ru_sc, ri_sc = orc.narre_forward(p64, *batch, argmax_override=(ua, ia))
    rp, rl, rg = orc.loss_and_grads("narre", p64, batch, ratings.double(), argmax_override=(ua, ia))
    assert rel_err(pred.detach(), rp) < FP32_TOL
    assert rel_err(u_sc.detach(), ru_sc) < FP32_TOL and rel_err(i_sc.detach(), ri_sc) < FP32_TOL
    assert rel_err(res["loss"].detach(), rl) < FP32_TOL
    for k, p in model.named_parameters():
        assert rel_err(p.grad, rg[k], grad_floor(k)) < FP32_GRAD_TOL, k


def test_graphed_step_narre_per_side_attention_matches_eager():
    """GraphedTrainStep of the att_dim 64 NARRE (the item-side attention forks onto an auxiliary stream inside the capture)
    against eager steps on the same batches, every batch twice."""
    from rbr_b200.graphs import GraphedTrainStep
    model, _, batches = _narre(64, seed=21)

    def eager(b, r):       # the eager graph must be gone before the capture (its AccumulateGrad nodes live on this stream)
        model.zero_grad(set_to_none=True)
        loss = torch.nn.MSELoss()(model(*b)[0], r)
        loss.backward()
        return float(loss), {k: p.grad.detach().clone() for k, p in model.named_parameters()}
    ref = [eager(b, r) for b, r in batches]
    step = GraphedTrainStep(model, torch.nn.MSELoss(), *batches[0])
    for _ in range(2):
        for (b, r), (ref_loss, ref_grads) in zip(batches, ref):
            loss = step(b, r)
            torch.cuda.synchronize()
            assert abs(float(loss) - ref_loss) <= 2e-6 * max(1.0, abs(ref_loss))
            for k, p in model.named_parameters():                # replay vs eager: the fp32 atomics land in a different order
                assert rel_err(p.grad, ref_grads[k], 1e-9) < 1e-5, k


# ----------------------------------------------------------------------------------------------------------------------
# routing: each case runs the kernels it names
# ----------------------------------------------------------------------------------------------------------------------
def _kernels_launched(fn, tmp_path):
    """[(kernel name, grid x, block x)] of every CUDA kernel `fn` launches, from a torch.profiler trace."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    events = json.loads(path.read_text())["traceEvents"]
    out = []
    for e in events:
        if e.get("cat") == "kernel":
            args = e.get("args", {})
            out.append((e["name"], args["grid"][0], args["block"][0]))
    return out


def _pick(launched, kernel):
    """The one launch of `kernel` (matched on the name up to its argument list: head_fwd_kernel is not head_fwd2_kernel)."""
    hits = [(g, b) for n, g, b in launched if kernel + "(" in n.replace(" ", "")]
    assert len(hits) == 1, (kernel, launched)
    return hits[0]


def test_routing_runs_the_targeted_kernels(tmp_path):
    """Every case above runs exactly the kernels it names (and, for the generic attention kernels, the warps per CTA it names);
    together the cases run every kernel both with a single round of CTAs and with CTAs that loop (head_fwd2_kernel<4> never
    loops: its grid cap covers 9472 samples)."""
    head_family = list(HEAD_CTA) + ["head_bwd2_kernel<4>"]
    attn_family = [A2F, A2B, GF, GB, "narre_attn_tc_fwd_kernel", "narre_attn_tc_bwd_kernel"]
    rounds = collections.defaultdict(set)                # kernel (+ warps) → {single round, looped}
    for name, c in HEAD_CASES.items():
        built = _head_build(c, seed=7, screen=False)
        launched = _kernels_launched(lambda: _head_run(c, *built), tmp_path)
        ran = {k for k in head_family if any(k + "(" in n.replace(" ", "") for n, _, _ in launched)}
        assert ran == {c.fwd, c.bwd}, (name, ran)
        for k in (c.fwd, c.bwd):
            grid, block = _pick(launched, k)
            per_cta, cap = HEAD_CTA[k]
            assert grid == min((c.B + per_cta - 1) // per_cta, cap), (name, k, grid)
            rounds[k].add(c.B > grid * per_cta)
    for name, c in ATTN_CASES.items():
        built = _attn_build(c, seed=7, screen=False)
        launched = _kernels_launched(lambda: _attn_run(c, *built), tmp_path)
        lib.rbr_consume_oob_count(None)                  # out-of-range ids were counted: leave the counter clean
        ran = {k for k in attn_family if any(k + "(" in n.replace(" ", "") for n, _, _ in launched)}
        assert ran == {c.fwd[0], c.bwd[0]}, (name, ran)
        for k, warps in (c.fwd, c.bwd):
            grid, block = _pick(launched, k)
            assert block == 32 * warps, (name, k, block)
            assert grid == min((c.B + warps - 1) // warps, ATTN_CTA_CAP), (name, k, grid)
            rounds[(k, warps) if k in (GF, GB) else k].add(c.B > grid * warps)
    for k in list(HEAD_CTA) + [A2F, A2B, GF, GB]:
        seen = set().union(*[v for key, v in rounds.items() if key == k or (isinstance(key, tuple) and key[0] == k)])
        assert seen == ({False} if k == "head_fwd2_kernel<4>" else {False, True}), (k, seen)
    for k in (GF, GB):
        assert {key[1] for key in rounds if isinstance(key, tuple) and key[0] == k} == {8, 4, 2, 1}, k
