"""Parity AT THE BENCHMARKED CONFIGURATIONS and IN THE BENCHMARKED MODE (bench.py's shapes; dropout 0.5; fused MSE).

Every number in BENCH / SCALE rests on these shapes: DeepCoNN B=4096 (configs[1]), NARRE H=150 (configs[2]), D-ATT
(configs[3]) and the vocab-200k inference (configs[4]).  The checker is the oracle (oracle/rbr_oracle.py, a device-agnostic
functional restatement pinned against the reference's goldens) evaluated ON THE GPU IN FLOAT64 — the exact value both the
reference's fp32 path and ours approximate — so that the comparison finishes in seconds at full size.

Tolerances (BASELINE.json): fp32 kernels 1e-5 on outputs, 3e-5 on batch-summed gradients; bf16 kernels 1e-2 against the
oracle run on the bf16-ROUNDED table / conv weights (what the tensor cores multiply).  Arg-max routing: at 8e5 pooled maxima
per step two positions can tie to within rounding; the forward check proves that every position the kernel reports attains
the oracle's max up to summation-order noise, and gradients are then compared under the kernel's routing
(`argmax_override`), so a near-tie does not move a whole gradient row between the two sides of the comparison.
"""
import pytest
import torch

import rbr_b200
from conftest import grad_floor, rel_err
from oracle import rbr_oracle as orc
from rbr_b200 import ops, synth

pytestmark = pytest.mark.gpu
FP32_TOL, FP32_GRAD_TOL, BF16_TOL = 1e-5, 3e-5, 1e-2


def _cuda(ts):
    return [t.cuda() for t in ts]


def _f64(params, round_bf16=False):
    out = {}
    for k, v in params.items():
        if round_bf16 and (k == "word_embeddings.embedding.weight" or (k.startswith("ngram.") and k.endswith(".weight"))
                           or (("_atten.conv" in k) and k.endswith(".weight"))):
            v = v.to(torch.bfloat16).to(torch.float32)
        out[k] = v.cuda().double()
    return out


def _check_routing(y_max, y_at_kernel_argmax, tol):
    """every position the kernel pooled at attains the oracle's max within summation-order noise"""
    err = ((y_max - y_at_kernel_argmax).abs() / y_max.abs().clamp_min(1e-2)).max()
    assert float(err) < tol, float(err)


def _encoder_oracle_pre(table64, w64, b64, ids, mask):
    x = orc.embedding_gather(table64, ids)
    if mask is not None:
        x = orc.mask_rows(x, mask)
    return torch.relu(orc.conv1d_same(x, w64, b64))           # [N, L, H]


def _clear_relu_margins(model_name, p64, batch, tau=2e-5):
    """Replace (in place) the samples that own a ReLU whose input is within `tau` of 0 in the float64 oracle by copies of
    samples that do not (orc.relu_margins): fp32 summation-order noise is ~1e-6 on these O(0.1-1) pre-activations, so on
    the remaining batch every implementation opens and closes the same ReLUs.  Returns how many samples were replaced."""
    margins = orc.relu_margins(model_name, p64, batch)
    bad = (margins < tau).nonzero().flatten()
    good = (margins >= 10 * tau).nonzero().flatten()
    assert bad.numel() <= batch[0].shape[0] // 4 and good.numel() >= bad.numel()
    for t in batch:
        t[bad] = t[good[:bad.numel()]]
    assert float(orc.relu_margins(model_name, p64, batch).min()) >= tau
    return int(bad.numel())


def _step(model, batch, ratings, fused_loss=False):
    model.zero_grad(set_to_none=True)
    if fused_loss:
        loss, out = model.forward_loss(*batch, ratings)
    else:
        out = model(*batch)
        loss = torch.nn.MSELoss()(out[0] if isinstance(out, tuple) else out, ratings)
    loss.backward()
    pred = out[0] if isinstance(out, tuple) else out
    return pred.detach(), loss.detach(), {k: p.grad.detach() for k, p in model.named_parameters()}


# ----------------------------------------------------------------------------------------------------------------------
# configs[1]: DeepCoNN, B=4096, doc 500, vocab 50k, emb 300, 100 filters k=3
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_deepconn_full_config_vs_oracle(precision):
    c = dict(B=4096, L=500, V=50000, E=300, H=100, K=32, U=20000, I=12000)
    params = synth.deepconn_params(c["U"], c["I"], c["V"], c["E"], c["H"], c["K"], (3,), seed=0)
    batch, ratings = synth.deepconn_batch(c["B"], c["L"], c["V"], c["U"], c["I"], seed=synth.SEED_BASE)
    batch, ratings = _cuda(batch), ratings.cuda()
    model = rbr_b200.DeepCoNNpp(c["U"], c["I"], c["V"], [3], c["E"], c["H"], c["K"], c["L"], None, 0.0, precision=precision)
    model.load_state_dict(params)
    model.cuda().train()
    bf = precision == "bf16"
    p64 = _f64(params, round_bf16=bf)
    tol, gtol = (BF16_TOL, BF16_TOL) if bf else (FP32_TOL, FP32_GRAD_TOL)
    n_replaced = _clear_relu_margins("deepconn", p64, batch)
    assert n_replaced < 200
    # forward routing: kernel arg-max positions attain the oracle's max
    with torch.no_grad():
        u_feat, i_feat, u_arg, i_arg = model.ngram.encode(model.word_embeddings, batch[:2], batch[2:4], return_argmax=True)
    w64, b64 = p64["ngram.feature_layer.0.list_of_conv1d.0.weight"], p64["ngram.feature_layer.0.list_of_conv1d.0.bias"]
    for ids, mask, feat, arg in ((batch[0], batch[2], u_feat, u_arg), (batch[1], batch[3], i_feat, i_arg)):
        for lo in range(0, c["B"], 1024):                          # chunks: [1024, 500, 100] float64 at a time
            y = _encoder_oracle_pre(p64["word_embeddings.embedding.weight"], w64, b64, ids[lo:lo + 1024], mask[lo:lo + 1024])
            ymax = y.max(dim=1).values
            _check_routing(ymax, torch.gather(y, 1, arg[lo:lo + 1024].long().unsqueeze(1)).squeeze(1), 1e-5)
            assert rel_err(feat[lo:lo + 1024].cpu(), ymax.cpu()) < (1e-3 if bf else FP32_TOL)
            del y
    # whole step under the kernel's routing
    pred, loss, grads = _step(model, batch, ratings)
    rp, rl, rg = orc.loss_and_grads("deepconn", p64, batch, ratings.double(), argmax_override=(u_arg, i_arg))
    assert rel_err(pred.cpu(), rp.cpu()) < tol
    assert rel_err(loss.cpu(), rl.cpu()) < tol
    for k in rg:
        assert rel_err(grads[k].cpu(), rg[k].cpu(), grad_floor(k)) < gtol, k
    assert float(grads["word_embeddings.embedding.weight"][0].abs().max()) == 0.0


# ----------------------------------------------------------------------------------------------------------------------
# configs[2]: NARRE, 10 reviews x 60 tokens, H=150 (trainer/train_narre.py:125), B=512
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_narre_full_config_vs_oracle(precision):
    c = dict(B=512, R=10, T=60, V=50000, E=300, H=150, A=32, K=32, U=20000, I=12000)
    params = synth.narre_params(c["U"], c["I"], c["V"], c["E"], c["H"], c["A"], c["K"], (3,), seed=0)
    batch, ratings = synth.narre_batch(c["B"], c["R"], c["T"], c["V"], c["U"], c["I"], seed=synth.SEED_BASE)
    batch, ratings = _cuda(batch), ratings.cuda()
    model = rbr_b200.NARRE(c["U"], c["I"], c["V"], [3], c["H"], c["E"], c["A"], c["K"], c["R"], c["T"], 0.0, 0, 0, 0, None, "CNN",
                           precision=precision)
    model.load_state_dict(params)
    model.cuda().train()
    bf = precision == "bf16"
    p64 = _f64(params, round_bf16=bf)
    tol, gtol = (BF16_TOL, BF16_TOL) if bf else (FP32_TOL, FP32_GRAD_TOL)
    _clear_relu_margins("narre", p64, batch)
    docs = [batch[0].view(-1, c["T"]), batch[1].view(-1, c["T"])]
    masks = [batch[2].view(-1, c["T"]), batch[3].view(-1, c["T"])]
    with torch.no_grad():
        u_feat, i_feat, u_arg, i_arg = model.ngram.encode(model.word_embeddings, docs, masks, return_argmax=True)
    w64, b64 = p64["ngram.feature_layer.0.list_of_conv1d.0.weight"], p64["ngram.feature_layer.0.list_of_conv1d.0.bias"]
    for ids, mask, feat, arg in ((docs[0], masks[0], u_feat, u_arg), (docs[1], masks[1], i_feat, i_arg)):
        y = _encoder_oracle_pre(p64["word_embeddings.embedding.weight"], w64, b64, ids, mask)
        ymax = y.max(dim=1).values
        _check_routing(ymax, torch.gather(y, 1, arg.long().unsqueeze(1)).squeeze(1), 1e-5)
        assert rel_err(feat.cpu(), ymax.cpu()) < (1e-3 if bf else FP32_TOL)
    out = model(*batch)
    model.zero_grad(set_to_none=True)
    loss = torch.nn.MSELoss()(out[0], ratings)
    loss.backward()
    grads = {k: p.grad.detach() for k, p in model.named_parameters()}
    leaves_pred, u_sc, i_sc = orc.narre_forward(p64, *batch, argmax_override=(u_arg, i_arg))
    rp, rl, rg = orc.loss_and_grads("narre", p64, batch, ratings.double(), argmax_override=(u_arg, i_arg))
    assert rel_err(out[0].detach().cpu(), rp.cpu()) < tol
    assert rel_err(out[1].detach().cpu(), u_sc.cpu()) < tol and rel_err(out[2].detach().cpu(), i_sc.cpu()) < tol
    assert rel_err(loss.detach().cpu(), rl.cpu()) < tol
    for k in rg:
        assert rel_err(grads[k].cpu(), rg[k].cpu(), grad_floor(k)) < gtol, k


# ----------------------------------------------------------------------------------------------------------------------
# configs[3]: D-ATT, doc 500, emb 100, B=256
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_dual_att_full_config_vs_oracle(precision):
    c = dict(B=256, L=500, V=50000, E=100, lw=5, lo=200, go=100, h1=500, h2=50)
    params = synth.dual_att_params(c["V"], c["L"], c["lw"], c["lo"], c["go"], c["E"], c["h1"], c["h2"], seed=0)
    batch, ratings = synth.dual_att_batch(c["B"], c["L"], c["V"], seed=synth.SEED_BASE)
    batch, ratings = _cuda(batch), ratings.cuda()
    model = rbr_b200.DualAtt(c["V"], c["L"], c["lw"], c["lo"], c["go"], c["E"], c["h1"], c["h2"], 0.0, None, precision=precision)
    model.load_state_dict(params)
    model.cuda().train()
    pred, loss, grads = _step(model, batch, ratings)
    p64 = _f64(params)
    rp, rl, rg = orc.loss_and_grads("dual_att", p64, batch, ratings.double())
    if precision == "fp32":
        assert rel_err(pred.cpu(), rp.cpu()) < FP32_TOL
        assert rel_err(loss.cpu(), rl.cpu()) < FP32_TOL
        for k in rg:
            # tanh pooling has no exact ties at these sizes; the routing is the oracle's own
            assert rel_err(grads[k].cpu(), rg[k].cpu()) < FP32_GRAD_TOL, k
    else:
        # the gates are computed in fp32, the four gated convs on bf16 operands: 1e-2 on the outputs; gradients on the
        # Frobenius norm (a bf16-induced arg-max move relocates a whole row, SURVEY §7)
        assert rel_err(pred.cpu(), rp.cpu()) < BF16_TOL
        assert rel_err(loss.cpu(), rl.cpu()) < BF16_TOL
        for k in rg:
            num = (grads[k].double() - rg[k]).norm()
            assert float(num / rg[k].norm().clamp_min(1e-12)) < 0.1, k


# ----------------------------------------------------------------------------------------------------------------------
# configs[4]: inference scoring at vocab 200k (the fp32 table does not fit L2)
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_deepconn_infer_vocab200k_vs_oracle(precision):
    c = dict(B=1024, L=500, V=200000, E=300, H=100, K=32, U=20000, I=12000)
    params = synth.deepconn_params(c["U"], c["I"], c["V"], c["E"], c["H"], c["K"], (3,), seed=0)
    batch, _ = synth.deepconn_batch(c["B"], c["L"], c["V"], c["U"], c["I"], seed=synth.SEED_BASE + 5)
    batch = _cuda(batch)
    model = rbr_b200.DeepCoNNpp(c["U"], c["I"], c["V"], [3], c["E"], c["H"], c["K"], c["L"], None, 0.5, precision=precision)
    model.load_state_dict(params)
    model.cuda().eval()
    with torch.no_grad():
        pred = model(*batch)
        rp = orc.deepconn_forward(_f64(params, round_bf16=(precision == "bf16")), *batch)
        rp32 = orc.deepconn_forward(_f64(params), *batch)
    assert rel_err(pred.cpu(), rp.cpu()) < (2e-3 if precision == "bf16" else FP32_TOL)
    assert rel_err(pred.cpu(), rp32.cpu()) < (BF16_TOL if precision == "bf16" else FP32_TOL)
    # int32 token ids and device-derived masks (the staged input pipeline) score identically
    with torch.no_grad():
        p2 = model(batch[0].int(), batch[1].int(), None, None, batch[4], batch[5])
    assert torch.equal(p2, pred)


# ----------------------------------------------------------------------------------------------------------------------
# the benchmarked MODE: FM dropout 0.5 (a counter-hash keep mask, exported by rbr_head_dropout_mask) and the fused MSE
# ----------------------------------------------------------------------------------------------------------------------
def _midsize_deepconn(dropout, precision="fp32", B=512):
    c = dict(B=B, L=200, V=5000, E=300, H=100, K=32, U=300, I=200)
    params = synth.deepconn_params(c["U"], c["I"], c["V"], c["E"], c["H"], c["K"], (3,), seed=4)
    batch, ratings = synth.deepconn_batch(c["B"], c["L"], c["V"], c["U"], c["I"], seed=99)
    model = rbr_b200.DeepCoNNpp(c["U"], c["I"], c["V"], [3], c["E"], c["H"], c["K"], c["L"], None, dropout, precision=precision)
    model.load_state_dict(params)
    return c, params, _cuda(batch), ratings.cuda(), model.cuda().train()


@pytest.mark.parametrize("fused_loss", [False, True])
def test_dropout_half_matches_oracle_given_the_exported_mask(fused_loss):
    c, params, batch, ratings, model = _midsize_deepconn(0.5)
    with torch.no_grad():
        _, _, u_arg, i_arg = model.ngram.encode(model.word_embeddings, batch[:2], batch[2:4], return_argmax=True)
    pred, loss, grads = _step(model, batch, ratings, fused_loss=fused_loss)
    p, seed, seed_dev = model.fm.__dict__["_rbr_last_drop"]
    assert p == 0.5 and seed_dev is None
    keep = ops.head_dropout_mask(c["B"], c["K"], p, seed, None, device=pred.device)
    # values are exactly 0 or 1/(1-p); keep fraction 0.5 within 4 sigma of a fair coin over B*K draws
    vals = set(keep.unique().tolist())
    assert vals == {0.0, 2.0}
    n = c["B"] * c["K"]
    assert abs(float((keep > 0).float().mean()) - 0.5) < 4 * 0.5 / n ** 0.5
    # columns and rows are not degenerate (the hash mixes sample and latent index)
    assert float((keep > 0).float().mean(dim=0).min()) > 0.35 and float((keep > 0).float().mean(dim=1).min()) > 0.05
    rp, rl, rg = orc.loss_and_grads("deepconn", _f64(params), batch, ratings.double(), fm_drop_mask=keep.double(),
                                    argmax_override=(u_arg, i_arg))
    assert rel_err(pred.cpu(), rp.cpu()) < FP32_TOL
    assert rel_err(loss.cpu(), rl.cpu()) < FP32_TOL
    for k in rg:                                                   # backward regenerated the SAME mask
        assert rel_err(grads[k].cpu(), rg[k].cpu()) < FP32_GRAD_TOL, k
    # a second call draws a different mask
    model(*batch)
    assert model.fm.__dict__["_rbr_last_drop"][1] != seed


def test_dropout_mask_under_graph_replay_is_shared_by_forward_and_backward():
    """GraphedTrainStep: the seed is a device-resident counter bumped inside the graph; forward and backward of one replay
    read the same value, consecutive replays different ones."""
    from rbr_b200.graphs import GraphedTrainStep
    c, params, batch, ratings, model = _midsize_deepconn(0.5, B=256)
    with torch.no_grad():
        _, _, u_arg, i_arg = model.ngram.encode(model.word_embeddings, batch[:2], batch[2:4], return_argmax=True)
    step = GraphedTrainStep(model, torch.nn.MSELoss(), batch, ratings)
    assert step.fused_loss
    seen = []
    for _ in range(3):
        loss = step.replay()
        torch.cuda.synchronize()
        keep = ops.head_dropout_mask(c["B"], c["K"], 0.5, 0x5EED, step._seed_dev)
        seen.append(keep.clone())
        rp, rl, rg = orc.loss_and_grads("deepconn", _f64(params), batch, ratings.double(), fm_drop_mask=keep.double(),
                                        argmax_override=(u_arg, i_arg))
        assert rel_err(loss.detach().cpu(), rl.cpu()) < FP32_TOL
        for k, prm in model.named_parameters():
            assert rel_err(prm.grad.cpu(), rg[k].cpu()) < FP32_GRAD_TOL, k
    assert not torch.equal(seen[0], seen[1]) and not torch.equal(seen[1], seen[2])
    # eager calls after the graph was built draw fresh host seeds again (the device counter is attached only inside the body)
    assert "_rbr_seed_dev" not in model.fm.__dict__
    model(*batch)
    s1 = model.fm.__dict__["_rbr_last_drop"]
    model(*batch)
    s2 = model.fm.__dict__["_rbr_last_drop"]
    assert s1[2] is None and s1[1] != s2[1]


@pytest.mark.parametrize("model_name", ["deepconn", "narre"])
def test_fused_mse_head_matches_unfused_and_oracle(model_name):
    """a9: the fused-MSE branch of rbr_head_fwd (model.forward_loss) against nn.MSELoss on the same model and the oracle."""
    if model_name == "deepconn":
        c, params, batch, ratings, model = _midsize_deepconn(0.0, B=200)
    else:
        c = dict(B=96, R=10, T=60, V=3000, E=300, H=150, A=32, K=32, U=50, I=40)
        params = synth.narre_params(c["U"], c["I"], c["V"], c["E"], c["H"], c["A"], c["K"], (3,), seed=1)
        b, r = synth.narre_batch(c["B"], c["R"], c["T"], c["V"], c["U"], c["I"], seed=5)
        model = rbr_b200.NARRE(c["U"], c["I"], c["V"], [3], c["H"], c["E"], c["A"], c["K"], c["R"], c["T"], 0.0, 0, 0, 0, None, "CNN",
                               precision="fp32")
        model.load_state_dict(params)
        batch, ratings, model = _cuda(b), r.cuda(), model.cuda().train()
    p64 = _f64(params)
    _clear_relu_margins(model_name, p64, batch)
    p0, l0, g0 = _step(model, batch, ratings, fused_loss=False)
    p1, l1, g1 = _step(model, batch, ratings, fused_loss=True)
    assert torch.equal(p0, p1)
    assert rel_err(l1.cpu(), l0.cpu()) < 1e-6
    for k in g0:
        assert rel_err(g1[k].cpu(), g0[k].cpu(), grad_floor(k)) < 5e-6, k          # two runs: fp32 atomics in a different order
    if model_name == "deepconn":
        with torch.no_grad():
            _, _, ua, ia = model.ngram.encode(model.word_embeddings, batch[:2], batch[2:4], return_argmax=True)
    else:
        T = batch[0].shape[-1]
        with torch.no_grad():
            _, _, ua, ia = model.ngram.encode(model.word_embeddings, [batch[0].view(-1, T), batch[1].view(-1, T)],
                                              [batch[2].view(-1, T), batch[3].view(-1, T)], return_argmax=True)
    rp, rl, rg = orc.loss_and_grads(model_name, p64, batch, ratings.double(), argmax_override=(ua, ia))
    assert rel_err(l1.cpu(), orc.mse_loss(rp, ratings.double()).cpu()) < FP32_TOL
    for k in rg:
        assert rel_err(g1[k].cpu(), rg[k].cpu(), grad_floor(k)) < FP32_GRAD_TOL, k
    # the loss scales through: backward of 3*loss gives 3x the gradients (upstream d/d loss is applied on the device)
    model.zero_grad(set_to_none=True)
    loss, _ = model.forward_loss(*batch, ratings)
    (3.0 * loss).backward()
    for k, prm in model.named_parameters():
        assert rel_err(prm.grad.cpu(), 3.0 * g1[k].cpu(), grad_floor(k)) < 1e-5, k


def test_separate_padding_rows_per_id_table():
    """Each of the four id tables of the head keeps its own padding row (ADVICE r1): user padding 0, item padding 3."""
    U, I, H, K, B = 9, 8, 12, 6, 64
    gen = torch.Generator().manual_seed(3)
    uf = rbr_b200.layers.LastFeat(U, H, K, padding_idx=0).cuda()
    itf = rbr_b200.layers.LastFeat(I, H, K, padding_idx=3).cuda()
    fm = rbr_b200.layers.FM(U, I, K, 0.0, user_padding_idx=0, item_padding_idx=3).cuda()
    ut, it = torch.randn(B, H, generator=gen).cuda(), torch.randn(B, H, generator=gen).cuda()
    uid, iid = torch.randint(0, U, (B,), generator=gen).cuda(), torch.randint(0, I, (B,), generator=gen).cuda()
    pred = rbr_b200.layers.fused_head(uf, itf, fm, ut, it, uid, iid, True, None)
    pred.sum().backward()
    assert float(uf.ebd.weight.grad[0].abs().max()) == 0.0 and float(fm.user_bias.weight.grad[0].abs().max()) == 0.0
    assert float(itf.ebd.weight.grad[3].abs().max()) == 0.0 and float(fm.item_bias.weight.grad[3].abs().max()) == 0.0
    assert float(itf.ebd.weight.grad[0].abs().max()) > 0.0 and float(fm.item_bias.weight.grad[0].abs().max()) > 0.0
    assert float(uf.ebd.weight.grad[3].abs().max()) > 0.0


def test_out_of_range_ids_raise_at_the_mode_switch():
    from rbr_b200._lib import lib
    c, params, batch, ratings, model = _midsize_deepconn(0.0, B=8)
    lib.rbr_consume_oob_count(None)                                 # start from a clean counter
    model.eval()
    bad = batch[0].clone()
    bad[0, 0] = c["V"] + 7
    with torch.no_grad():
        model(bad, *batch[1:])
    with pytest.raises(IndexError, match="outside their embedding tables"):
        model.train()
    model.train()                                                   # counter was consumed: clean again


def test_saturated_gate_gives_finite_gate_gradient():
    """D-ATT: a global gate that saturates to exactly 0 must not produce inf/NaN (VERDICT r1 #22)."""
    V, L, E = 60, 24, 16
    params = synth.dual_att_params(V, L, 5, 12, 8, E, 20, 5, seed=2)
    params["u_global_atten.attn.0.bias"] = torch.full((1,), -200.0)         # sigmoid(-200) == 0 in fp32
    batch, ratings = synth.dual_att_batch(5, L, V, seed=3)
    model = rbr_b200.DualAtt(V, L, 5, 12, 8, E, 20, 5, 0.0, None, precision="fp32")
    model.load_state_dict(params)
    model.cuda().train()
    pred, loss, grads = _step(model, _cuda(batch), ratings.cuda())
    assert all(bool(torch.isfinite(g).all()) for g in grads.values())
    rp, rl, rg = orc.loss_and_grads("dual_att", params, batch, ratings)
    assert rel_err(pred.cpu(), rp) < FP32_TOL
    for k in rg:
        assert rel_err(grads[k].cpu(), rg[k], 1e-9) < FP32_GRAD_TOL, k


def test_feature_cache_scores_are_bit_identical_to_per_pair_scoring():
    """SURVEY §8f-2: encode each entity's document once, score pairs with K1 gather + K4 head: same bits as the reference's
    per-pair data flow (both documents encoded for every pair)."""
    from rbr_b200.inference import PairScorer
    U, I, V, E, H, K, L = 300, 200, 5000, 300, 100, 32, 500
    params = synth.deepconn_params(U, I, V, E, H, K, (3,), seed=4)
    model = rbr_b200.DeepCoNNpp(U, I, V, [3], E, H, K, L, None, 0.5, precision="bf16")
    model.load_state_dict(params)
    scorer = PairScorer(model.cuda())
    user_docs, _ = synth.doc_batch(U, L, V, seed=1)
    item_docs, _ = synth.doc_batch(I, L, V, seed=2)
    user_docs[0] = 0
    item_docs[0] = 0                                                   # the padding entities
    user_docs, item_docs = user_docs.cuda(), item_docs.cuda()
    scorer.build_cache(user_docs, item_docs, chunk=128)
    gen = torch.Generator().manual_seed(3)
    u_ids = torch.randint(0, U, (4096,), generator=gen).cuda()
    i_ids = torch.randint(0, I, (4096,), generator=gen).cuda()
    cached = scorer.score_cached(u_ids, i_ids)
    ud, idd = user_docs[u_ids], item_docs[i_ids]
    direct = scorer.score_pairs(ud, idd, ud != 0, idd != 0, u_ids, i_ids)
    assert torch.equal(cached, direct)
    rp = orc.deepconn_forward(_f64(params, round_bf16=True), ud, idd, ud != 0, idd != 0, u_ids, i_ids)
    assert rel_err(cached.cpu(), rp.cpu()) < 2e-3


@pytest.mark.parametrize("H", [100, 300], ids=["proj", "noproj"])
def test_feature_cache_scores_hier_pooling(H):
    """arch="HierPooling" (K8, then the Linear projection when E != H): the feature cache's scores against per-pair scoring."""
    from rbr_b200.inference import PairScorer
    U, I, V, E, K, L = 300, 200, 5000, 300, 32, 500
    model = rbr_b200.DeepCoNNpp(U, I, V, [3], E, H, K, L, None, 0.5, arch="HierPooling")
    model.load_state_dict(synth.deepconn_hier_params(U, I, V, E, H, K, seed=4))
    scorer = PairScorer(model.cuda())
    user_docs, _ = synth.doc_batch(U, L, V, seed=1)
    item_docs, _ = synth.doc_batch(I, L, V, seed=2)
    user_docs[0] = 0
    item_docs[0] = 0
    user_docs, item_docs = user_docs.cuda(), item_docs.cuda()
    scorer.build_cache(user_docs, item_docs, chunk=128)
    gen = torch.Generator().manual_seed(3)
    u_ids = torch.randint(0, U, (4096,), generator=gen).cuda()
    i_ids = torch.randint(0, I, (4096,), generator=gen).cuda()
    cached = scorer.score_cached(u_ids, i_ids)
    ud, idd = user_docs[u_ids], item_docs[i_ids]
    direct = scorer.score_pairs(ud, idd, ud != 0, idd != 0, u_ids, i_ids)
    if H == E:
        assert torch.equal(cached, direct)
    else:                       # the projection is a library GEMM, whose bits may depend on the batch (128 entities vs 4096 pairs)
        assert rel_err(cached, direct) < FP32_TOL
