"""GPU parity tests: the CUDA path (through the C-ABI library) against the committed reference golden
fixtures and against the CPU oracle on seeded inputs.  Tolerances are BASELINE.json's: bit-exact gathers,
1e-5 relative in fp32, 1e-2 relative in bf16."""
import os

import pytest
import torch

import rbr_b200
from conftest import Golden, grad_floor, rel_err
from oracle import rbr_oracle as orc
from rbr_b200 import ops, synth

pytestmark = pytest.mark.gpu
FP32_TOL = 1e-5
FP32_GRAD_TOL = 3e-5      # sums over the batch in a different association order than the CPU oracle
BF16_TOL = 1e-2

DEEPCONN_CASES = ["deepconn_small", "deepconn_edge", "deepconn_multik", "deepconn_odd"]
NARRE_CASES = ["narre_small", "narre_h150ish"]


def dev(t):
    return t.cuda() if isinstance(t, torch.Tensor) else t


def build_model(g: Golden, precision="fp32"):
    m = g.meta
    if g.model == "deepconn":
        model = rbr_b200.DeepCoNNpp(m["U"], m["I"], m["V"], m["ks"], m["E"], m["H"], m["K"], m["L"], None, 0.0,
                                    precision=precision)
    else:
        model = rbr_b200.NARRE(m["U"], m["I"], m["V"], [3], m["H"], m["E"], m["A"], m["K"], m["R"], m["T"], 0.0, 0, 0, 0,
                               None, "CNN", precision=precision)
    assert set(model.state_dict()) == set(g.params)
    model.load_state_dict(g.params)
    return model.cuda()


def run_step(model, batch, ratings):
    model.train()
    model.zero_grad()
    out = model(*[dev(t) for t in batch])
    pred = out[0] if isinstance(out, tuple) else out
    loss = torch.nn.MSELoss()(pred, dev(ratings))
    loss.backward()
    grads = {k: p.grad.detach().cpu() for k, p in model.named_parameters()}
    return out, loss.detach().cpu(), grads


# ------------------------------------------------------------------------------------------------
def test_gather_bit_exact_and_dense_grad():
    g = Golden("deepconn_odd")
    table = g.params["word_embeddings.embedding.weight"].cuda()
    ids = g.batch[0].cuda()
    out = ops.gather_rows(table, ids)
    assert torch.equal(out.cpu(), orc.embedding_gather(table.cpu(), ids.cpu()))
    gr = torch.randn(*ids.shape, table.shape[1], generator=torch.Generator().manual_seed(1))
    dense = ops.embedding_dense_grad(ids, gr.cuda(), table.shape[0], 0).cpu()
    ref = orc.embedding_dense_grad(ids.cpu(), gr, table.shape[0], 0)
    assert rel_err(dense, ref) < 1e-6
    assert float(dense[0].abs().max()) == 0.0


def test_gather_large_bit_exact():
    gen = torch.Generator().manual_seed(3)
    table = torch.randn(5000, 300, generator=gen)
    ids, _ = synth.doc_batch(64, 500, 5000, seed=11)
    out = ops.gather_rows(table.cuda(), ids.cuda()).cpu()
    assert torch.equal(out, table[ids])
    # scalar path (emb % 4 != 0) and empty input
    t2 = torch.randn(50, 7, generator=gen)
    i2 = torch.randint(0, 50, (3, 5), generator=gen)
    assert torch.equal(ops.gather_rows(t2.cuda(), i2.cuda()).cpu(), t2[i2])
    assert ops.gather_rows(t2.cuda(), i2[:0].cuda()).shape == (0, 5, 7)


def test_dense_grad_hot_rows_and_scalar_path():
    gen = torch.Generator().manual_seed(5)
    ids = synth.skewed_tokens(gen, (4096 * 4,), 300)          # heavy duplicates → long segments
    ids[::7] = 0
    gr = torch.randn(ids.numel(), 64, generator=gen)
    dense = ops.embedding_dense_grad(ids.cuda(), gr.cuda(), 300, 0).cpu()
    assert rel_err(dense, orc.embedding_dense_grad(ids, gr, 300, 0)) < 1e-5
    gr7 = torch.randn(ids.numel(), 7, generator=gen)
    dense7 = ops.embedding_dense_grad(ids.cuda(), gr7.cuda(), 300, 0).cpu()
    assert rel_err(dense7, orc.embedding_dense_grad(ids, gr7, 300, 0)) < 1e-5


@pytest.mark.parametrize("case", DEEPCONN_CASES + NARRE_CASES)
def test_golden_fp32(case):
    """Forward outputs, loss and EVERY parameter gradient against the reference's own numbers."""
    g = Golden(case)
    model = build_model(g, "fp32")
    out, loss, grads = run_step(model, g.batch, g.ratings)
    pred = out[0] if isinstance(out, tuple) else out
    assert rel_err(pred.detach().cpu(), g.out["pred"]) < FP32_TOL
    assert rel_err(loss, g.out["loss"]) < FP32_TOL
    if isinstance(out, tuple):
        assert out[1].shape == g.out["u_att_scores"].shape
        assert rel_err(out[1].detach().cpu(), g.out["u_att_scores"]) < FP32_TOL
        assert rel_err(out[2].detach().cpu(), g.out["i_att_scores"]) < FP32_TOL
    assert set(grads) == set(g.grads)
    for k, ref in g.grads.items():
        assert grads[k].shape == ref.shape, k
        assert rel_err(grads[k], ref, grad_floor(k)) < FP32_GRAD_TOL, k
    assert float(grads["word_embeddings.embedding.weight"][0].abs().max()) == 0.0      # padding row


def test_edge_semantics_fp32():
    """all-pad doc pools to relu(bias); masks are honoured even where ids != 0; eval == train at dropout 0."""
    g = Golden("deepconn_edge")
    model = build_model(g, "fp32")
    u_feat, i_feat = model.ngram.encode(model.word_embeddings, [g.batch[0].cuda(), g.batch[1].cuda()],
                                        [g.batch[2].cuda(), g.batch[3].cuda()])
    assert rel_err(u_feat.detach().cpu(), g.out["u_rev_feats"]) < FP32_TOL
    assert rel_err(i_feat.detach().cpu(), g.out["i_rev_feats"]) < FP32_TOL
    bias = g.params["ngram.feature_layer.0.list_of_conv1d.0.bias"]
    assert torch.allclose(u_feat[0].detach().cpu(), torch.relu(bias), atol=1e-7)
    model.eval()
    with torch.no_grad():
        p = model(*[t.cuda() for t in g.batch])
    assert rel_err(p.cpu(), g.out["pred"]) < FP32_TOL


def test_ngramfeat_standalone_matches_oracle():
    """Reference-signature NgramFeat.forward(inputs [bz,L,E], masks) incl. gradient w.r.t. the dense inputs."""
    gen = torch.Generator().manual_seed(9)
    bz, L, E, H = 6, 33, 20, 12
    x = torch.randn(bz, L, E, generator=gen)
    mask = torch.rand(bz, L, generator=gen) > 0.2
    layer = rbr_b200.layers.NgramFeat([3], E, H, L, precision="fp32").cuda()
    w = layer.conv.list_of_conv1d[0].weight.detach().cpu()
    b = layer.conv.list_of_conv1d[0].bias.detach().cpu()
    xg = x.cuda().requires_grad_(True)
    out = layer(xg, mask.cuda())
    assert out.shape == (bz, H, 1)
    xo = x.clone().requires_grad_(True)
    ref = orc.ngram_feat(xo, mask, [w], [b])
    assert rel_err(out.detach().cpu().view(bz, H), ref.detach()) < FP32_TOL
    gout = torch.randn(bz, H, generator=gen)
    out.view(bz, H).backward(gout.cuda())
    ref.backward(gout)
    assert rel_err(xg.grad.cpu(), xo.grad) < FP32_GRAD_TOL


def test_linear_attention_standalone_and_padding_quirk():
    """Padded reviews are NOT masked out of the softmax (narre.py:58): they keep non-zero weight."""
    g = Golden("narre_small")
    m = g.meta
    att = rbr_b200.layers.LinearAttention(m["I"], m["H"], m["A"], 0.0).cuda()
    sd = {k[len("user_att."):]: v for k, v in g.params.items() if k.startswith("user_att.")}
    att.load_state_dict(sd)
    gen = torch.Generator().manual_seed(2)
    feat = torch.randn(m["B"], m["R"], m["H"], generator=gen)
    out, sc = att(feat.cuda(), g.batch[6].cuda())
    ro, rs = orc.linear_attention(feat, g.batch[6], sd["W_rv"], sd["W_id"], sd["h"], sd["b_1"], sd["b_2"], sd["ebd_vals.weight"])
    assert rel_err(out.detach().cpu(), ro) < FP32_TOL and rel_err(sc.detach().cpu(), rs) < FP32_TOL
    assert torch.allclose(sc.sum(dim=1).cpu(), torch.ones(m["B"], 1), atol=1e-6)
    assert float(sc.min()) > 0.0


@pytest.mark.parametrize("model_name", ["deepconn", "narre"])
def test_seeded_midsize_vs_oracle_fp32(model_name):
    """Realistic dims (E=300, k=3, H=100/150) at a batch the CPU oracle finishes in seconds."""
    if model_name == "deepconn":
        B, L, V, U, I, E, H, K = 24, 500, 3000, 50, 40, 300, 100, 32
        params = synth.deepconn_params(U, I, V, E, H, K, (3,), seed=1)
        batch, ratings = synth.deepconn_batch(B, L, V, U, I, seed=123)
        model = rbr_b200.DeepCoNNpp(U, I, V, [3], E, H, K, L, None, 0.0, precision="fp32")
    else:
        B, R, T, V, U, I, E, H, A, K = 12, 10, 60, 3000, 50, 40, 300, 150, 32, 32
        params = synth.narre_params(U, I, V, E, H, A, K, (3,), seed=1)
        batch, ratings = synth.narre_batch(B, R, T, V, U, I, seed=123)
        model = rbr_b200.NARRE(U, I, V, [3], H, E, A, K, R, T, 0.0, 0, 0, 0, None, "CNN", precision="fp32")
    model.load_state_dict(params)
    model.cuda()
    out, loss, grads = run_step(model, batch, ratings)
    pred = out[0] if isinstance(out, tuple) else out
    rp, rl, rg = orc.loss_and_grads(model_name, params, batch, ratings)
    assert rel_err(pred.detach().cpu(), rp) < FP32_TOL
    assert rel_err(loss, rl) < FP32_TOL
    for k in rg:
        assert rel_err(grads[k], rg[k], grad_floor(k)) < FP32_GRAD_TOL, k


def test_properties_full_size_fp32_forward():
    """Size-independent properties at a larger batch: changing tokens under a false mask changes nothing;
    permuting the batch permutes the predictions; eval forward is deterministic."""
    B, L, V, U, I, E, H, K = 256, 500, 50000, 200, 120, 300, 100, 32
    params = synth.deepconn_params(U, I, V, E, H, K, (3,), seed=2)
    batch, _ = synth.deepconn_batch(B, L, V, U, I, seed=77)
    model = rbr_b200.DeepCoNNpp(U, I, V, [3], E, H, K, L, None, 0.5, precision="fp32")
    model.load_state_dict(params)
    model.cuda().eval()
    b = [t.cuda() for t in batch]
    with torch.no_grad():
        p0 = model(*b)
        p1 = model(*b)
        assert torch.equal(p0, p1)
        scr = b[0].clone()
        scr[~b[2]] = 17                                     # garbage under the mask
        assert torch.equal(model(scr, b[1], b[2], b[3], b[4], b[5]), p0)
        perm = torch.randperm(B, device="cuda")
        pp = model(*[t[perm] for t in b])
        assert torch.equal(pp, p0[perm])


def test_oob_ids_are_counted_not_fatal():
    from rbr_b200._lib import lib
    lib.rbr_consume_oob_count(None)
    table = torch.randn(10, 8).cuda()
    ids = torch.tensor([[1, 2, 99, -4]]).cuda()
    out = ops.gather_rows(table, ids)
    assert float(out[0, 2].abs().max()) == 0.0 and float(out[0, 3].abs().max()) == 0.0
    assert lib.rbr_consume_oob_count(None) == 2


def test_two_pass_backward_with_table_hook_matches_single_pass():
    """Data-parallel overlap splits the encoder backward (table gradients of all sides first, hook, then weight
    gradients): same gradients as the single pass, and the hook sees the complete table gradient."""
    g = Golden("deepconn_small")
    seen = {}
    grads = []
    for use_hook in (False, True):
        model = build_model(g, "fp32")
        if use_hook:
            model.ngram.table_grad_hook = lambda t: seen.setdefault("table", t.detach().clone())
        _, _, gr = run_step(model, g.batch, g.ratings)
        grads.append(gr)
    for k in grads[0]:
        assert rel_err(grads[1][k], grads[0][k]) < 1e-6, k
    assert rel_err(seen["table"].cpu(), g.grads["word_embeddings.embedding.weight"]) < FP32_GRAD_TOL


@pytest.mark.parametrize("shape", [(33, 10, 150, 32), (7, 4, 8, 5), (5, 5, 15, 6), (100, 6, 100, 16), (3, 2, 40, 8), (70, 17, 64, 32),
                                   (4096, 10, 150, 32),
                                   # plan edges: one review; 64 reviews (one sample per tile); att_dim 1; the largest hidden
                                   # accepted at 10 and at 64 reviews (pinned in test_cpu_host); hidden not a multiple of 8
                                   (50, 1, 128, 32), (40, 64, 192, 32), (33, 10, 150, 1), (100, 10, 160, 32), (150, 10, 101, 16)])
def test_attention_pair_tensor_core_kernels_vs_oracle(shape):
    """K3 on tensor cores (csrc/attn_tc.cu, 3xTF32 mma.sync, both sides in one launch): outputs, scores and every gradient
    against the oracle's LinearAttention at the fp32 tolerance; padded reviews (id 0) keep softmax mass and give the padding
    row no gradient."""
    B, R, H, A = shape
    assert ops.narre_attn_pair_supported(R, H, A)
    gen = torch.Generator().manual_seed(B + R + H)
    n_ids = (23, 31)
    sides = []
    for s in range(2):
        feat = torch.randn(B, R, H, generator=gen).abs() * 0.5                   # pooled ReLU features are non-negative
        oid = torch.randint(0, n_ids[s], (B, R), generator=gen)
        oid[:, -1] = 0                                                           # a padded review per sample
        prm = [(torch.rand(H, A, generator=gen) * 2 - 1) * 0.1, (torch.rand(A, A, generator=gen) * 2 - 1) * 0.1,
               (torch.rand(A, 1, generator=gen) * 2 - 1) * 0.1, torch.full((A,), 0.1), torch.full((1,), 0.1),
               torch.randn(n_ids[s], A, generator=gen)]
        prm[5][0] = 0
        sides.append((feat, oid, prm))
    g_out = [torch.randn(B, H, generator=gen) for _ in range(2)]
    g_sc = [torch.randn(B, R, 1, generator=gen) * 0.1 for _ in range(2)]
    # oracle (float64)
    ref = []
    for (feat, oid, prm), go, gs in zip(sides, g_out, g_sc):
        f64 = feat.double().requires_grad_(True)
        p64 = [p.double().requires_grad_(True) for p in prm]
        out, sc = orc.linear_attention(f64, oid, *p64)
        ((out * go.double()).sum() + (sc * gs.double()).sum()).backward()
        ge = p64[5].grad.clone()
        ge[0] = 0                                                                # nn.Embedding(padding_idx=0)
        ref.append((out.detach(), sc.detach(), f64.grad, [p.grad for p in p64[:5]] + [ge]))
    cu = [(f.cuda().requires_grad_(True), o.cuda(), [p.cuda().requires_grad_(True) for p in prm]) for f, o, prm in sides]
    params = cu[0][2] + cu[1][2]
    out_u, sc_u, out_i, sc_i = ops.NarreAttnPairFn.apply(cu[0][0], cu[0][1], cu[1][0], cu[1][1], *params, (0, 0), None, params)
    loss = (out_u * g_out[0].cuda()).sum() + (sc_u * g_sc[0].cuda()).sum() + (out_i * g_out[1].cuda()).sum() + (sc_i * g_sc[1].cuda()).sum()
    loss.backward()
    for s, (o, sc) in enumerate(((out_u, sc_u), (out_i, sc_i))):
        assert rel_err(o.detach().cpu(), ref[s][0]) < FP32_TOL
        assert rel_err(sc.detach().cpu(), ref[s][1]) < FP32_TOL
        assert rel_err(cu[s][0].grad.cpu(), ref[s][2]) < FP32_GRAD_TOL
        for j, name in enumerate(("W_rv", "W_id", "h", "b_1", "b_2", "ebd_vals")):
            # d loss / d b_2 is ~0 by the softmax's shift invariance: what any implementation stores there is the rounding
            # noise of a sum of B*R terms of size |d logit| — compare it on that scale
            floor = float(B * R) ** 0.5 * 0.1 if name == "b_2" else 1e-6
            if R == 1:
                # one review: the score is 1 / (1 + 1e-8) and every logit gradient is ~1e-8 of the upstream gradient, below fp32's
                # resolution of the score.  The parameters only see those logit gradients (~1e-7 here): compare them on an
                # absolute scale (3e-6)
                floor = max(floor, 0.1)
            assert rel_err(cu[s][2][j].grad.cpu(), ref[s][3][j], floor) < FP32_GRAD_TOL, (s, name)
        assert float(cu[s][2][5].grad[0].abs().max()) == 0.0


@pytest.mark.parametrize("case", ["deepconn_hier", "deepconn_hier_noproj"])
def test_golden_hier_pooling_fp32(case):
    """SURVEY §8f-4: DeepCoNNpp(arch="HierPooling") — K8 (gather + avg-pool + max-pool fused) against the reference's numbers."""
    g = Golden(case)
    m = g.meta
    model = rbr_b200.DeepCoNNpp(m["U"], m["I"], m["V"], [m["k"]], m["E"], m["H"], m["K"], m["L"], None, 0.0, arch="HierPooling")
    assert set(model.state_dict()) == set(g.params)
    model.load_state_dict(g.params)
    model.cuda()
    out, loss, grads = run_step(model, g.batch, g.ratings)
    assert rel_err(out.detach().cpu(), g.out["pred"]) < FP32_TOL
    assert rel_err(loss, g.out["loss"]) < FP32_TOL
    for k, ref in g.grads.items():
        assert rel_err(grads[k], ref) < FP32_GRAD_TOL, k
    assert float(grads["word_embeddings.embedding.weight"][0].abs().max()) == 0.0


def test_hier_pooling_midsize_and_standalone_vs_oracle():
    B, L, V, U, I, E, H, K, k = 16, 500, 3000, 50, 40, 300, 100, 32, 3
    params = synth.deepconn_hier_params(U, I, V, E, H, K, seed=1)
    batch, ratings = synth.deepconn_batch(B, L, V, U, I, seed=123)
    model = rbr_b200.DeepCoNNpp(U, I, V, [k], E, H, K, L, None, 0.0, arch="HierPooling")
    model.load_state_dict(params)
    model.cuda()
    out, loss, grads = run_step(model, batch, ratings)
    rp, rl, rg = orc.loss_and_grads("deepconn", params, batch, ratings, hier_kernel=k)
    assert rel_err(out.detach().cpu(), rp) < FP32_TOL and rel_err(loss, rl) < FP32_TOL
    for kk in rg:
        assert rel_err(grads[kk], rg[kk]) < FP32_GRAD_TOL, kk
    # int32 ids + derived masks give the same bits
    with torch.no_grad():
        b = [t.cuda() for t in batch]
        assert torch.equal(model(b[0].int(), b[1].int(), None, None, b[4], b[5]), model(*b))
    # reference-signature NgramFeat.forward on dense inputs (odd width → scalar kernel path), gradient w.r.t. the inputs
    gen = torch.Generator().manual_seed(4)
    x = torch.randn(5, 21, 10, generator=gen)
    mask = torch.rand(5, 21, generator=gen) > 0.2
    layer = rbr_b200.layers.NgramFeat([5], 10, 10, 21, arch="HierPooling").cuda()
    xg = x.cuda().requires_grad_(True)
    y = layer(xg, mask.cuda())
    xo = x.clone().requires_grad_(True)
    ref = orc.hier_pooling(xo, mask, 5)
    assert y.shape == (5, 10) and rel_err(y.detach().cpu(), ref.detach()) < FP32_TOL
    go = torch.randn(5, 10, generator=gen)
    y.backward(go.cuda())
    ref.backward(go)
    assert rel_err(xg.grad.cpu(), xo.grad) < FP32_GRAD_TOL


@pytest.mark.parametrize("case", ["simple_siamese_small", "simple_siamese_lt"])
def test_golden_simple_siamese(case):
    """SURVEY §8f-4: the SimpleSiamese drop-in (K9 masked average pooling fused with the gather + the fused head) against the
    reference's own numbers: pred, loss and every parameter gradient."""
    g = Golden(case)
    m = g.meta
    model = rbr_b200.SimpleSiamese(m["E"], m["K"], m["V"], m["U"], m["I"], None, False, 0.0, 0.0, 0.0, bool(m["ui"]), bool(m["lt"]))
    assert set(model.state_dict()) == set(g.params)
    model.load_state_dict(g.params)
    model.cuda()
    out, loss, grads = run_step(model, g.batch, g.ratings)
    assert rel_err(out[0].detach().cpu(), g.out["pred"]) < FP32_TOL
    assert rel_err(loss, g.out["loss"]) < FP32_TOL
    for k, ref in g.grads.items():
        assert rel_err(grads[k], ref, 1e-9) < FP32_GRAD_TOL, k
    assert float(grads["word_embedding.embedding.weight"][0].abs().max()) == 0.0


def test_simple_siamese_midsize_vs_oracle():
    B, R, T, V, U, I, E, K = 48, 10, 60, 3000, 50, 40, 300, 32
    params = synth.simple_siamese_params(U, I, V, E, K, True, False, seed=1)
    batch, ratings = synth.simple_siamese_batch(B, R, T, V, U, I, seed=123)
    model = rbr_b200.SimpleSiamese(E, K, V, U, I, None, False, 0.0, 0.0, 0.0, True, False)
    model.load_state_dict(params)
    model.cuda()
    out, loss, grads = run_step(model, batch, ratings)
    rp, rl, rg = orc.loss_and_grads("simple_siamese", params, batch, ratings)
    assert rel_err(out[0].detach().cpu(), rp) < FP32_TOL and rel_err(loss, rl) < FP32_TOL
    for k in rg:
        assert rel_err(grads[k], rg[k], 1e-9) < FP32_GRAD_TOL, k
    with torch.no_grad():                                    # int32 ids + derived word masks: same bits
        b = [t.cuda() for t in batch]
        assert torch.equal(model(b[0].int(), b[1].int(), None, None, *b[4:])[0], model(*b)[0])
