"""Drive the reference's UNMODIFIED trainer loop (`*Experiment.train_one_epoch`, trainer/train_deepconn_pp.py:143-189,
trainer/train_narre.py:142-190, trainer/train_dual_att.py:137-180) over a stub dataset — with the reference's own model
(golden generation, tests/golden/make_golden.py) or with this package's drop-in model aliased into the trainer's import
(`sys.modules["models.deepconn.deepconn"] = rbr_b200.deepconn`, INTEGRATION.md).  Test infrastructure only.

Nothing of the trainer is edited or re-implemented: the Experiment class is constructed as its __main__ does (args from
the reference's default_*.json with the sizes shrunk, dropout 0, logging off), parameters are loaded from a seeded set,
`loss_func` is wrapped by a recorder, and `train_one_epoch(0)` runs zero_grad → forward → MSELoss → backward →
clip_grad_norm_ → Adam.step over the stub loader's batches.

The trainer needs the reference's sources (oracle/_ref).  Without them, `run_loop` runs the same loop body restated here;
tests/test_oracle_golden.py pins that restatement, driving the CPU oracle, to the goldens the unmodified trainer wrote.
"""
from __future__ import annotations

import importlib
import os
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import ref_loader  # noqa: E402
from rbr_b200 import synth  # noqa: E402

TRAINER = {
    "deepconn": ("trainer.train_deepconn_pp", "DeepCoNNExperiment", "models.deepconn.deepconn", "models/deepconn/default_deepconn_pp.json"),
    "narre": ("trainer.train_narre", "NarreExperiment", "models.narre.narre", "models/narre/default_narre.json"),
    "dual_att": ("trainer.train_dual_att", "DualAttExperiment", "models.dual_att.dual_att", "models/dual_att/default_dual_att.json"),
}

# small shapes (the NARRE trainer hard-codes hidden_dim=150, trainer/train_narre.py:125)
SHAPES = {
    "deepconn": dict(B=6, L=40, V=200, U=30, I=20, E=32, H=16, K=8, ks=(3,)),
    "narre": dict(B=4, R=4, T=12, V=150, U=20, I=15, E=24, H=150, A=8, K=8, ks=(3,)),
    "dual_att": dict(B=4, L=30, V=120, E=20, lw=5, lo=24, go=12, h1=30, h2=7),
}
N_STEPS = 3
LR, MAX_GRAD_NORM = 0.002, 5.0          # lr and max_grad_norm of the reference's default_*.json
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class _StubDataset:
    """The attributes the trainers' build_model reads off `train_dataloader.dataset`."""

    def __init__(self, kind, c):
        self.word_vocab = range(c["V"])
        if kind != "dual_att":
            self.user_num, self.item_num = c["U"], c["I"]
        if kind == "narre":
            self.rv_num, self.rv_len = c["R"], c["T"]
        else:
            self.doc_len = c["L"]


class _StubLoader(list):
    """A list of collated batches with the `.dataset` attribute the trainer expects of a DataLoader."""


def batches(kind):
    c = SHAPES[kind]
    out = []
    for s in range(N_STEPS):
        seed = 4242 + s
        if kind == "deepconn":
            b, r = synth.deepconn_batch(c["B"], c["L"], c["V"], c["U"], c["I"], seed=seed)
            out.append((*b, r))                                       # collate order, train_deepconn_pp.py:281-292
        elif kind == "narre":
            b, r = synth.narre_batch(c["B"], c["R"], c["T"], c["V"], c["U"], c["I"], seed=seed)
            out.append((*b, r))                                       # train_narre.py:318-331
        else:
            b, r = synth.dual_att_batch(c["B"], c["L"], c["V"], seed=seed)
            out.append((*b, r))
    return out


def initial_params(kind):
    c = SHAPES[kind]
    if kind == "deepconn":
        return synth.deepconn_params(c["U"], c["I"], c["V"], c["E"], c["H"], c["K"], c["ks"], seed=11)
    if kind == "narre":
        return synth.narre_params(c["U"], c["I"], c["V"], c["E"], c["H"], c["A"], c["K"], c["ks"], seed=12)
    return synth.dual_att_params(c["V"], c["L"], c["lw"], c["lo"], c["go"], c["E"], c["h1"], c["h2"], seed=13)


class _LossRecorder:
    def __init__(self, fn):
        self.fn, self.values = fn, []

    def __call__(self, pred, target):
        loss = self.fn(pred, target)
        self.values.append(float(loss.detach().cpu()))
        return loss


def run_trainer_epoch(kind: str, model_module=None):
    """Run `train_one_epoch(0)` of the reference trainer for `kind`.  model_module: None = the reference's own model class;
    otherwise a module object to alias as the trainer's `models.<kind>.<kind>` import (this package's drop-in).
    Returns (losses per step, final state_dict on the CPU, model)."""
    ref_loader.activate()
    mod_name, exp_name, model_mod_name, cfg_rel = TRAINER[kind]
    saved = sys.modules.get(model_mod_name)
    if model_module is not None:
        sys.modules[model_mod_name] = model_module
    else:
        sys.modules.pop(model_mod_name, None)
        importlib.import_module(model_mod_name)
    try:
        tm = importlib.reload(sys.modules[mod_name]) if mod_name in sys.modules else importlib.import_module(mod_name)
        c = SHAPES[kind]
        args = tm.parse_args(os.path.join(ref_loader.REF_DIR, cfg_rel))
        args.dropout = 0.0
        args.log, args.verbose, args.stats, args.parallel, args.use_pretrain = False, False, False, False, False
        args.log_idx = 10 ** 9
        if kind != "dual_att":
            args.embedding_dim, args.latent_dim, args.hidden_dim = c["E"], c["K"], c["H"]
        if kind == "narre":
            args.att_dim = c["A"]
        if kind == "dual_att":
            args.l_window_size, args.l_out_size, args.g_out_size, args.emb_size = c["lw"], c["lo"], c["go"], c["E"]
            args.hidden_size_1, args.hidden_size_2 = c["h1"], c["h2"]
        cwd = os.getcwd()
        with tempfile.TemporaryDirectory() as tmp:
            os.chdir(tmp)                       # Experiment.setup() creates ./<log_dir>/<dataset>/<model>/<uid>
            try:
                loader = _StubLoader(batches(kind))
                loader.dataset = _StubDataset(kind, c)
                exp = getattr(tm, exp_name)(args, {"train": loader, "valid": None, "test": None})
                exp.model.load_state_dict(initial_params(kind))
                rec = _LossRecorder(exp.loss_func)
                exp.loss_func = rec
                exp.train_one_epoch(0)
            finally:
                os.chdir(cwd)
        if exp.device.type == "cuda":
            torch.cuda.synchronize()
        final = {k: v.detach().cpu().clone() for k, v in exp.model.state_dict().items()}
        return rec.values, final, exp.model
    finally:
        if saved is not None:
            sys.modules[model_mod_name] = saved
        else:
            sys.modules.pop(model_mod_name, None)


def build_model(kind: str):
    """This package's drop-in model at SHAPES[kind] (dropout 0), constructed with the arguments the trainer's build_model passes,
    initial_params(kind) loaded."""
    import rbr_b200
    c = SHAPES[kind]
    if kind == "deepconn":
        model = rbr_b200.DeepCoNNpp(c["U"], c["I"], c["V"], list(c["ks"]), c["E"], c["H"], c["K"], c["L"], None, 0.0)
    elif kind == "narre":
        model = rbr_b200.NARRE(c["U"], c["I"], c["V"], list(c["ks"]), c["H"], c["E"], c["A"], c["K"], c["R"], c["T"], 0.0,
                               0, 0, 0, None, "CNN")
    else:
        model = rbr_b200.DualAtt(c["V"], c["L"], c["lw"], c["lo"], c["go"], c["E"], c["h1"], c["h2"], 0.0, None)
    model.load_state_dict(initial_params(kind))
    return model


def run_loop(kind: str, params: dict, forward):
    """The body of `train_one_epoch` restated over batches(kind): optimizer.zero_grad() → forward → nn.MSELoss → backward →
    clip_grad_norm_(5.0) → Adam(lr 0.002).step → loss.item(), with Adam and the clip over `params` in the order given.
    params: {state_dict name: leaf tensor}; forward(*batch) returns pred, or a tuple led by pred, on the params' device.
    Returns (losses per step, final params on the CPU)."""
    dev = next(iter(params.values())).device
    opt = torch.optim.Adam(list(params.values()), lr=LR)
    loss_fn = torch.nn.MSELoss()
    losses = []
    for *batch, ratings in batches(kind):
        opt.zero_grad()
        out = forward(*[t.to(dev) for t in batch])
        pred = out[0] if isinstance(out, tuple) else out
        loss = loss_fn(pred, ratings.to(dev))
        loss.backward()
        torch.nn.utils.clip_grad_norm_(list(params.values()), MAX_GRAD_NORM)
        opt.step()
        losses.append(loss.item())
    return losses, {k: v.detach().cpu().clone() for k, v in params.items()}


def assert_matches_golden(kind: str, losses, final, tol: float, check_params: bool = True) -> None:
    """Per-step losses within `tol` (relative) of tests/golden/trainer_<kind>_3steps.npz and, with check_params, the final
    parameters: Adam's first updates are lr·sign(g), so an entry whose gradient is rounding noise can differ by a fraction of
    one lr step between any two summation orders — bounded as a fraction of outliers (|diff| > 1e-5 on at most 0.2 % of the
    entries) and the worst entry (< half an lr step); rows no batch touched must not have moved at all."""
    import numpy as np
    z = np.load(os.path.join(GOLDEN, f"trainer_{kind}_{N_STEPS}steps.npz"))
    ref_losses = z["losses"]
    assert len(losses) == N_STEPS
    for a, b in zip(losses, ref_losses):
        assert abs(a - b) <= tol * abs(b), (losses, ref_losses.tolist())
    if not check_params:
        return
    init = initial_params(kind)
    n_bad = n_all = 0
    worst = 0.0
    for k, v in final.items():
        ref = torch.from_numpy(z["final/" + k])
        d = (v - ref).abs()
        n_bad += int((d > 1e-5).sum())
        n_all += d.numel()
        worst = max(worst, float(d.max()))
        # rows no batch touched did not move at all (dense gradients with exact zeros, Adam leaves them in place)
        untouched = (ref == init[k])
        assert torch.equal(v[untouched], init[k][untouched]), k
    assert n_bad <= 2e-3 * n_all, (n_bad, n_all)
    assert worst < 1e-3, worst
