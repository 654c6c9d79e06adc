"""Pins the CPU oracle (oracle/rbr_oracle.py) to outputs of the unmodified reference modules
(tests/golden/*.npz, written by tests/golden/make_golden.py in the build container)."""
import pytest
import torch

from conftest import Golden, grad_floor, rel_err
from oracle import rbr_oracle as orc

TOL = 1e-5   # fp32 tolerance stated by BASELINE.json north_star


def test_oracle_matches_reference(golden: Golden):
    pred, loss, grads = orc.loss_and_grads(golden.model, golden.params, golden.batch, golden.ratings)
    assert rel_err(pred, golden.out["pred"]) < TOL
    assert rel_err(loss, golden.out["loss"]) < TOL
    assert set(grads) == set(golden.grads)
    for k, g in golden.grads.items():
        assert grads[k].shape == g.shape, k
        assert rel_err(grads[k], g, grad_floor(k)) < 2e-5, k


def test_oracle_aux_outputs():
    g = Golden("deepconn_edge")
    pred, aux = orc.deepconn_forward(g.params, *g.batch, return_aux=True)
    assert rel_err(aux["u_rev_feats"], g.out["u_rev_feats"]) < TOL
    assert rel_err(aux["i_rev_feats"], g.out["i_rev_feats"]) < TOL
    # all-pad doc pools to relu(bias)  (SURVEY.md §8c)
    bias = g.params["ngram.feature_layer.0.list_of_conv1d.0.bias"]
    assert torch.allclose(aux["u_rev_feats"][0], torch.relu(bias), atol=1e-7)
    n = Golden("narre_small")
    p, us, is_ = orc.narre_forward(n.params, *n.batch)
    assert rel_err(us, n.out["u_att_scores"]) < TOL and rel_err(is_, n.out["i_att_scores"]) < TOL
    assert torch.allclose(us.sum(dim=1), torch.ones(us.shape[0], 1), atol=1e-6)


def test_padding_row_gets_zero_grad(golden: Golden):
    _, _, grads = orc.loss_and_grads(golden.model, golden.params, golden.batch, golden.ratings)
    assert float(grads["word_embeddings.embedding.weight"][0].abs().max()) == 0.0


def test_gather_is_bit_exact():
    g = Golden("deepconn_small")
    table = g.params["word_embeddings.embedding.weight"]
    ids = g.batch[0]
    out = orc.embedding_gather(table, ids)
    assert torch.equal(out, torch.nn.functional.embedding(ids, table))
    gr = torch.randn(*ids.shape, table.shape[1])
    dense = orc.embedding_dense_grad(ids, gr, table.shape[0])
    ref = torch.zeros_like(table).index_add_(0, ids.reshape(-1), gr.reshape(-1, table.shape[1]))
    ref[0] = 0
    assert rel_err(dense, ref) < 1e-6
    assert torch.equal(orc.get_mask(ids), ids != 0)


def test_first_argmax_tie_rule():
    y = torch.tensor([[[1.0], [3.0], [3.0], [2.0]]])
    vals, idx = orc.first_argmax_pool(y)
    assert vals.item() == 3.0 and idx.item() == 1


def test_vendored_reference_is_byte_identical_and_agrees_with_the_oracle():
    """oracle/_ref (built by oracle/Makefile from /root/reference, git-ignored) is what bench.py's CPU arm times: its files
    match the recorded SHA-256 sums and, on a seeded batch, the unmodified modules give the oracle's numbers."""
    import hashlib
    import os
    import pytest
    from oracle import ref_loader
    from rbr_b200 import synth
    if not ref_loader.available():
        pytest.skip("oracle/_ref not built (make -C oracle where /root/reference exists)")
    sums = open(os.path.join(ref_loader.REF_DIR, "SHA256SUMS")).read().split("\n")
    n = 0
    for line in sums:
        if not line.strip():
            continue
        digest, rel = line.split()
        assert hashlib.sha256(open(os.path.join(ref_loader.REF_DIR, rel), "rb").read()).hexdigest() == digest, rel
        n += 1
    assert n >= 15
    cfg = dict(U=9, I=7, V=60, E=12, H=8, K=6, L=20, ks=(3,))
    params = synth.deepconn_params(cfg["U"], cfg["I"], cfg["V"], cfg["E"], cfg["H"], cfg["K"], cfg["ks"], seed=1)
    batch, ratings = synth.deepconn_batch(5, cfg["L"], cfg["V"], cfg["U"], cfg["I"], seed=3)
    ref = ref_loader.build_reference("deepconn", cfg, params, dropout=0.0).train()
    pred = ref(*batch)
    loss = torch.nn.MSELoss()(pred, ratings)
    loss.backward()
    rp, rl, rg = orc.loss_and_grads("deepconn", params, batch, ratings)
    assert rel_err(pred.detach(), rp) < 1e-6 and rel_err(loss.detach(), rl) < 1e-6
    for k, p in ref.named_parameters():
        assert rel_err(p.grad, rg[k]) < 1e-5, k


@pytest.mark.parametrize("kind", ["deepconn", "narre", "dual_att"])
def test_restated_trainer_loop_reproduces_reference_trainer_goldens(kind):
    """trainer_harness.run_loop (the loop body of the reference's train_one_epoch restated: zero_grad → forward → MSELoss →
    backward → clip_grad_norm_(5.0) → Adam(lr 0.002).step) driving the oracle gives the losses and final parameters the
    unmodified trainer wrote to tests/golden/trainer_*_3steps.npz, so the GPU test may use it where oracle/_ref is absent."""
    import trainer_harness as th
    params = {k: v.clone().requires_grad_(True) for k, v in th.initial_params(kind).items()}
    for k in orc._PADDED_TABLES:               # nn.Embedding(padding_idx=0): row 0 gets no gradient
        if k in params:
            params[k].register_hook(lambda g: g.index_fill(0, torch.zeros(1, dtype=torch.long), 0.0))
    forward = {"deepconn": orc.deepconn_forward, "narre": orc.narre_forward, "dual_att": orc.dual_att_forward}[kind]
    losses, final = th.run_loop(kind, params, lambda *batch: forward(params, *batch))
    th.assert_matches_golden(kind, losses, final, tol=1e-5)


@pytest.mark.parametrize("case", ["deepconn_hier", "deepconn_hier_noproj"])
def test_oracle_hier_pooling_matches_reference_golden(case):
    """arch="HierPooling" (models/deepconn/layers.py:62-98, 110-114): the oracle's avg-pool → max-pool → [Linear] → ReLU
    against the numbers the unmodified reference produced (with and without the projection)."""
    g = Golden(case)
    rp, rl, rg = orc.loss_and_grads("deepconn", g.params, g.batch, g.ratings, hier_kernel=g.meta["k"])
    assert rel_err(rp, g.out["pred"]) < 1e-5 and rel_err(rl, g.out["loss"]) < 1e-5
    assert set(rg) == set(g.grads)
    for k, ref in g.grads.items():
        assert rel_err(rg[k], ref) < 1e-5, k


@pytest.mark.parametrize("case", ["simple_siamese_small", "simple_siamese_lt"])
def test_oracle_simple_siamese_matches_reference_golden(case):
    """SimpleSiamese (models/simple_siamese/simple_siamese.py:55-88): masked average pooling + additive review attention +
    LastFeat + FM, with and without user/item biases and the latent transform."""
    g = Golden(case)
    rp, rl, rg = orc.loss_and_grads("simple_siamese", g.params, g.batch, g.ratings)
    assert rel_err(rp, g.out["pred"]) < 1e-5 and rel_err(rl, g.out["loss"]) < 1e-5
    assert set(rg) == set(g.grads)
    for k, ref in g.grads.items():
        assert rel_err(rg[k], ref, 1e-9) < 1e-5, k
