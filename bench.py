#!/usr/bin/env python
"""bench.py — fwd+bwd samples/s of the review-encoder hot path on N B200s (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--model all|deepconn|narre|dual_att] [--mode train|infer]
                    [--impl ours|reference] [--dump-outputs DIR]

One "step" = optimizer.zero_grad() + forward + nn.MSELoss + backward (+ the gradient all-reduce when N > 1), i.e.
trainer/train_deepconn_pp.py:161-165 of the reference.  BASELINE.json's metric names DeepCoNN AND NARRE, so the default run
times both: the top-level keys are DeepCoNN on configs[1] (B=4096 per GPU, doc 500 tokens, vocab 50k, emb 300, 100 filters
k=3, bf16 conv) and the `narre` key holds the same measurements for configs[2] (10 reviews x 60 tokens, H=150 as
trainer/train_narre.py:125 builds it).  N > 1 is launched by torchrun (RANK/LOCAL_RANK/WORLD_SIZE/MASTER_* from the env);
the headline is weak scaling (per-GPU batch fixed), the `strong` key reports the §8e partitioning (global B=4096 split over
the ranks) beside it; the only collective is the parameter-gradient all-reduce.

Rank 0 prints ONE JSON line: value = device-timed whole-job samples/s with inputs resident in HBM; e2e = the same step
driven from pinned HOST buffers through the public API (H2D of every input and a D2H read of the loss inside the timed
region); roofline = the dominant kernel (tcgen05 conv) against the measured bf16 peak; cpu_baseline = the reference's own
modules (oracle/_ref, unmodified) timed on this box's host cores; library_gpu_baseline = the reference's formulation on
ATen/cuBLAS kernels on the same GPU.  `--impl reference` times the CPU path alone, as the reference arm.

--dump-outputs DIR writes what the last timed step returned to its caller as DIR/<workload>.<name>.npy (float32): the loss
and every parameter gradient of a training step, the predictions of an inference step, the scores of `--pairs`.  Inputs,
parameters and dropout masks depend on the arguments only, so two builds run with the same arguments can be compared
array by array.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

DUMP_BYTES = 64 * 10 ** 6          # --dump-outputs writes at most this much in all

CFG = {
    "deepconn": dict(B=4096, L=500, V=50000, E=300, H=100, K=32, U=20000, I=12000, ks=(3,)),
    "narre": dict(B=4096, R=10, T=60, V=50000, E=300, H=150, A=32, K=32, U=20000, I=12000, ks=(3,)),
    # BASELINE.json configs[3]; dims from default_dual_att.json:17 and dual_att.py:20-21
    "dual_att": dict(B=4096, L=500, V=50000, E=100, lw=5, lo=200, go=100, h1=500, h2=50),
    # BASELINE.json configs[4]: inference scoring, vocab 200k (the fp32 table, 240 MB, does not fit L2), pairs sharded over ranks
    "deepconn_infer": dict(B=4096, L=500, V=200000, E=300, H=100, K=32, U=20000, I=12000, ks=(3,)),
}
METRIC = {"deepconn": "DeepCoNN fwd+bwd samples/sec", "narre": "NARRE fwd+bwd samples/sec",
          "dual_att": "D-ATT fwd+bwd samples/sec", "deepconn_infer": "DeepCoNN inference pairs/sec"}
PARITY_NOTE = ("bf16 conv: outputs within 1e-2 of the fp32 reference; gradients within 1e-2 of the oracle evaluated on the "
               "bf16-rounded table/conv weights under the kernel's arg-max routing (tests/test_gpu_benchcfg.py at these shapes); "
               "against the fp32 reference the gradient bound is Frobenius 0.1-0.15 because bf16 rounding can move a max-pool "
               "arg-max to a near-tied position, which moves a whole gradient row (SURVEY.md §7)")


def workload_name(model):
    c = CFG[model]
    if model == "dual_att":
        return (f"D-ATT train step B={c['B']}/GPU doc={c['L']} vocab={c['V']} emb={c['E']} local {c['lo']}@k1 (window {c['lw']}) "
                f"global 3x{c['go']}@k2,3,4 fc {c['h1']}-{c['h2']} (BASELINE.json configs[3])")
    if model == "deepconn_infer":
        return (f"DeepCoNN eval forward B={c['B']} pairs/step/GPU doc={c['L']} vocab={c['V']} emb={c['E']} filters={c['H']} k=3 "
                f"(BASELINE.json configs[4]; pairs sharded over GPUs, no collective)")
    if model == "deepconn":
        return (f"DeepCoNN train step B={c['B']}/GPU doc={c['L']} vocab={c['V']} emb={c['E']} filters={c['H']} k=3 "
                f"latent={c['K']} (BASELINE.json configs[1])")
    return (f"NARRE train step B={c['B']}/GPU reviews={c['R']}x{c['T']} vocab={c['V']} emb={c['E']} filters={c['H']} k=3 "
            f"att={c['A']} latent={c['K']} (BASELINE.json configs[2])")


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], tf=p["bf16_tflops"], tf_sus=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf=1590.0, tf_sus=1400.0, src="fallback (B200_PROFILING.md)")


def synth_params(model):
    from rbr_b200 import synth
    c = CFG[model]
    if model in ("deepconn", "deepconn_infer"):
        return synth.deepconn_params(c["U"], c["I"], c["V"], c["E"], c["H"], c["K"], c["ks"], seed=0)
    if model == "dual_att":
        return synth.dual_att_params(c["V"], c["L"], c["lw"], c["lo"], c["go"], c["E"], c["h1"], c["h2"], seed=0)
    return synth.narre_params(c["U"], c["I"], c["V"], c["E"], c["H"], c["A"], c["K"], c["ks"], seed=0)


def synth_batch(model, b, seed):
    from rbr_b200 import synth
    c = CFG[model]
    if model in ("deepconn", "deepconn_infer"):
        return synth.deepconn_batch(b, c["L"], c["V"], c["U"], c["I"], seed=seed)
    if model == "dual_att":
        return synth.dual_att_batch(b, c["L"], c["V"], seed=seed)
    return synth.narre_batch(b, c["R"], c["T"], c["V"], c["U"], c["I"], seed=seed)


# ----------------------------------------------------------------------------------------------------
# CPU arm: the reference's own modules (oracle/_ref, unmodified) on the host cores; the oracle port when _ref is absent
# ----------------------------------------------------------------------------------------------------
def cpu_arm(model, sample_b, steps, warmup, budget_s=150.0):
    """Seconds per step of zero_grad + forward + nn.MSELoss + backward (no clip, no optimizer: the same step as the GPU arm)
    on `sample_b` samples of the workload; eval forward for the inference workload.  BASELINE.md §5."""
    from oracle import ref_loader
    from rbr_b200 import synth
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    params = synth_params(model)
    batch, ratings = synth_batch(model, sample_b, synth.SEED_BASE)
    kind = "reference" if ref_loader.available() else "port"
    infer = model == "deepconn_infer"
    if kind == "reference":
        ref = ref_loader.build_reference("deepconn" if infer else model, CFG[model], params, dropout=0.5)
        ref.eval() if infer else ref.train()
        loss_fn = torch.nn.MSELoss()

        def one():
            if infer:
                with torch.no_grad():
                    return ref(*batch)
            ref.zero_grad()
            out = ref(*batch)
            loss = loss_fn(out[0] if isinstance(out, tuple) else out, ratings)
            loss.backward()
            return loss
        what = "oracle/_ref: the reference's unmodified nn.Modules"
    else:
        from oracle import rbr_oracle as orc

        def one():
            if infer:
                with torch.no_grad():
                    return orc.deepconn_forward(params, *batch)
            return orc.loss_and_grads(model, params, batch, ratings)
        what = "oracle/rbr_oracle.py (port; oracle/_ref not built)"
    t0 = time.perf_counter()
    one()
    first = time.perf_counter() - t0
    # keep the whole arm inside the budget: fewer timed steps when one step is slow (never fewer than 1)
    steps_eff = max(1, min(steps, int(budget_s / max(first, 1e-3)) - warmup))
    warm_eff = max(0, min(warmup - 1, int(0.25 * budget_s / max(first, 1e-3))))
    for _ in range(warm_eff):
        one()
    t0 = time.perf_counter()
    for _ in range(steps_eff):
        one()
    sec = (time.perf_counter() - t0) / steps_eff
    nthreads = torch.get_num_threads()
    return dict(value=sample_b / sec, unit="samples/s", cores=nthreads, kind=kind,
                sample=f"{sample_b} samples of the same workload per step, {steps_eff} timed steps after {warm_eff + 1} warm-up "
                       f"({what}, torch CPU, {nthreads} threads of {os.cpu_count()} cores)"), sec, steps_eff, warm_eff + 1


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    models = ["deepconn_infer"] if args.mode == "infer" else (["deepconn", "narre"] if args.model == "all" else [args.model])
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    line = None
    for mi, m in enumerate(models):
        sample_b = 128
        cb, sec, k_eff, w_eff = cpu_arm(m, sample_b, args.steps, args.warmup, budget_s=100.0 if len(models) > 1 else 150.0)
        d = {
            "impl": "reference", "metric": METRIC[m], "value": cb["value"], "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "steps_effective": k_eff, "warmup_effective": w_eff,
            "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(m), "global_batch": world * CFG[m]["B"], "parallelism": f"dp{world}"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        if mi == 0:
            line = d
        else:
            line[m] = d
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------
# clocks sampler (NVML in a background thread, ~50 ms period; samples kept from the timed regions only)
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        if self.nv is not None and not os.environ.get("RBR_BENCH_NO_NVML") and self._thr is None:
            self._stop.clear()
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def mark(self):
        """Forget what was sampled so far (the thread keeps running: its first NVML calls are slow and contend with kernel
        launches for the driver lock, so it is started before the warm-up and only marked at the start of a timed region)."""
        self.samples, self.reasons = [], set()

    def take(self):
        s, r = list(self.samples), set(self.reasons)
        self.mark()
        return s, r

    def stop(self):
        if self._thr is not None:
            self._stop.set()
            self._thr.join()
            self._thr = None

    def summarise(self, samples, reasons):
        return {"sm_mhz": statistics.median(samples) if samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(reasons), "samples": len(samples)}


# ----------------------------------------------------------------------------------------------------
def build(model_name, dev, precision):
    import rbr_b200
    c = CFG[model_name]
    params = synth_params(model_name)
    if model_name in ("deepconn", "deepconn_infer"):
        model = rbr_b200.DeepCoNNpp(c["U"], c["I"], c["V"], list(c["ks"]), c["E"], c["H"], c["K"], c["L"], None, 0.5,
                                    precision=precision)
    elif model_name == "dual_att":
        model = rbr_b200.DualAtt(c["V"], c["L"], c["lw"], c["lo"], c["go"], c["E"], c["h1"], c["h2"], 0.5, None, precision=precision)
    else:
        model = rbr_b200.NARRE(c["U"], c["I"], c["V"], list(c["ks"]), c["H"], c["E"], c["A"], c["K"], c["R"], c["T"], 0.5,
                               0, 0, 0, None, "CNN", precision=precision)
    model.load_state_dict(params)
    model = model.to(dev)
    return model.eval() if model_name == "deepconn_infer" else model.train()


def make_batches(model_name, n, rank, b=None):
    from rbr_b200 import synth
    return [synth_batch(model_name, b or CFG[model_name]["B"], synth.SEED_BASE + rank * 1000 + i) for i in range(n)]


def eager_step(model, batch, ratings, loss_fn, post=None, keep=None):
    if not model.training:                # inference scoring (configs[4]): eval forward under no_grad, no collective
        with torch.no_grad():
            pred = model(*batch)
        if keep is not None:
            keep["pred"] = pred
        return pred.sum()
    model.zero_grad(set_to_none=True)
    model.invalidate_operand_cache()      # as after an optimizer step: re-stage the bf16 table shadow + packed weights
    out = model(*batch)
    pred = out[0] if isinstance(out, tuple) else out
    loss = loss_fn(pred, ratings)
    loss.backward()
    if post is not None:
        post()
    return loss


class Ctx:
    pass


def time_graph_loop(ctx, steps_objs, K):
    """K replays over the rotating step objects, CUDA events on the current stream, max over ranks → (total ms, last loss)."""
    import torch.distributed as dist
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.sync_all()
    ctx.sampler.mark()
    e0.record()
    loss = None
    for i in range(K):
        loss = steps_objs[i % len(steps_objs)]()
    e1.record()
    ctx.sync_all()
    ms = torch.tensor([e0.elapsed_time(e1)], device=ctx.dev)
    if ctx.world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()), loss


def measure(ctx, name, args):
    """All measurements of one workload → (dict, {name: output of the last timed step} with --dump-outputs) on rank 0,
    (None, None) elsewhere."""
    import torch.distributed as dist
    from rbr_b200 import ops, parallel, synth
    from rbr_b200._lib import lib
    from rbr_b200.graphs import GraphedTrainStep
    rank, world, dev, peaks, sampler = ctx.rank, ctx.world, ctx.dev, ctx.peaks, ctx.sampler
    c = CFG[name]
    K, W = args.steps, max(args.warmup, 3)
    train = name != "deepconn_infer"
    loss_fn = torch.nn.MSELoss()
    model = build(name, dev, args.precision)
    parallel.broadcast_parameters(model)
    ar_kind = None
    if world > 1 and train:
        ar_kind = "nccl"
        if args.allreduce != "nccl" and args.grad_allreduce == "fp32":
            kind = {"nvls": "auto", "multimem": "multimem", "p2p": "p2p"}[args.allreduce]
            if parallel.enable_nvls_allreduce(model, overlap=True, kind=kind):
                k = model.__dict__["_rbr_nvls"].kind
                ar_kind = (("own kernel over the symmetric-memory arena: peer loads / stores (rbr_p2p_allreduce_f32)" if k == "p2p" else
                            "nvls-multimem (own kernel)") + ", word-table slice overlapped with the weight-gradient kernels")
            else:
                ar_kind = "nccl (no NVLS multicast)"
    compress = "bf16" if args.grad_allreduce == "bf16" else None
    post = (lambda: parallel.allreduce_gradients(model, compress=compress)) if (world > 1 and train) else None
    NB = 4   # distinct input batches rotated through: 4 x 37 MB of ids+masks > L2 together with table/grad traffic
    host_batches = make_batches(name, NB, rank)
    dev_batches = [([t.to(dev) for t in b], r.to(dev)) for b, r in host_batches]

    # ------------------------------ gradient-exchange self-check (N > 1): own NVLS kernel vs ncclAllReduce ------------------------------
    allreduce_check = None
    if post is not None:
        # local gradients with the early-reduction hook detached (with it, backward already starts averaging the word-table slice
        # on a side stream), averaged by NCCL; then the same step again through the real path (hook + own NVLS kernel)
        ngram_ = getattr(model, "ngram", None)
        hook_ = getattr(ngram_, "table_grad_hook", None)
        if ngram_ is not None:
            ngram_.table_grad_hook = None
        torch.manual_seed(4321 + rank)                 # both steps draw the same dropout masks
        eager_step(model, *dev_batches[0], loss_fn, None)
        if ngram_ is not None:
            ngram_.table_grad_hook = hook_
        expect = model.last_arena.flat.detach().clone()
        dist.all_reduce(expect, op=dist.ReduceOp.AVG)
        torch.manual_seed(4321 + rank)
        eager_step(model, *dev_batches[0], loss_fn, None)
        flat = model.last_arena.flat
        parallel.allreduce_gradients(model, compress=compress)
        torch.cuda.synchronize()
        err = ((flat.double() - expect.double()).abs().max() / expect.double().abs().max().clamp_min(1e-30)).reshape(1)
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
        allreduce_check = {"max_rel": float(err.item()),
                           "against": "ncclAllReduce(AVG) of the local gradients of the same batch (a separate backward: fp32 atomics order differs), max over ranks",
                           "elements": int(flat.numel())}
        del expect

    # ------------------------------ warm-up: at least W steps and ~0.4 s (clock ramp), count agreed between ranks ------------------------------
    sampler.start()
    for i in range(W):
        eager_step(model, *dev_batches[i % NB], loss_fn, post)
    ctx.sync_all()
    t_w = time.perf_counter()
    for i in range(3):
        eager_step(model, *dev_batches[i % NB], loss_fn, post)
    torch.cuda.synchronize()
    t_step = max((time.perf_counter() - t_w) / 3, 1e-5)
    n_extra = torch.tensor([min(2000, int(0.4 / t_step))], device=dev)
    if world > 1:
        dist.all_reduce(n_extra, op=dist.ReduceOp.MAX)
    n_extra = int(n_extra.item())
    for i in range(n_extra):
        eager_step(model, *dev_batches[i % NB], loss_fn, post)
    n_warm = W + 3 + n_extra
    ctx.sync_all()

    # ------------------------------ device-resident timing (value): CUDA-graph replays of the whole step ------------------------------
    graphs, graph_note, per_step, pool = None, "eager nn.Module calls", None, None
    graph_grads = []                      # --dump-outputs: the .grad tensors each captured graph writes
    if args.graphs == "auto" and train:
        try:
            graphs = []
            for i in range(NB):
                c0 = lib.rbr_launch_count()
                gs = GraphedTrainStep(model, loss_fn, *dev_batches[i], warmup=1, pool=pool, post_backward=post)
                per_step = (lib.rbr_launch_count() - c0) // 2          # one warm-up + one captured execution
                pool = gs.pool
                graphs.append(gs)
                if args.dump_outputs:
                    graph_grads.append({n: p.grad for n, p in model.named_parameters()})
            for gs in graphs:
                gs.replay()
            torch.cuda.synchronize()
            graph_note = (f"CUDA-graph replay of the step (rbr_b200.graphs.GraphedTrainStep, {NB} graphs, one per rotating batch; "
                          f"nn.MSELoss evaluated in the head kernel's launch: {graphs[0].fused_loss})")
        except Exception as e:
            if world > 1:
                raise                                # ranks must not diverge (one eager, one graphed) inside collectives
            graphs, graph_note = None, f"eager (graph capture failed: {type(e).__name__}: {str(e)[:100]})"
            torch.cuda.synchronize()
    l0 = lib.rbr_launch_count()
    keep = {}
    if graphs is not None:
        objs = [g.replay for g in graphs]
    else:
        objs = [(lambda j=j: eager_step(model, *dev_batches[j], loss_fn, post, keep)) for j in range(NB)]
    # the warm-up above ran a timing-dependent number of steps: reseed so that the dropout masks of the timed steps (and what
    # --dump-outputs writes) depend on the arguments only
    torch.manual_seed(synth.SEED_BASE + rank)
    total_ms, loss = time_graph_loop(ctx, objs, K)
    value_clocks = sampler.take()
    launches = (per_step * K) if graphs is not None else (lib.rbr_launch_count() - l0)
    value = world * c["B"] * K / (total_ms * 1e-3)
    final_loss = float(loss.item())
    outputs = None
    if args.dump_outputs and rank == 0:
        outputs = {"loss": loss}
        if train:
            grads = graph_grads[(K - 1) % NB] if graphs is not None else {n: p.grad for n, p in model.named_parameters()}
            outputs.update({"grad." + n: g for n, g in grads.items() if g is not None})
        else:
            outputs["pred"] = keep["pred"]
        outputs = {f"{name}.{k}": v.detach().float().cpu() for k, v in outputs.items()}
    graph_grads = keep = None

    # exposed collective time per step (N > 1): the same graphed step WITHOUT the gradient exchange
    exposed = None
    if post is not None and graphs is not None:
        ngram = getattr(model, "ngram", None)
        saved_hook = getattr(ngram, "table_grad_hook", None)
        if ngram is not None:
            ngram.table_grad_hook = None               # no early (in-backward) reduction either: nothing would join its stream
        g_local = GraphedTrainStep(model, loss_fn, *dev_batches[0], warmup=1, pool=pool, post_backward=None)
        if ngram is not None:
            ngram.table_grad_hook = saved_hook
        ms_local, _ = time_graph_loop(ctx, [g_local.replay], K)
        exposed = {"ms_per_step_without_exchange": ms_local / K, "exposed_collective_ms_per_step": (total_ms - ms_local) / K}
        del g_local

    # ------------------------------ end-to-end timing from pinned host buffers (e2e) ------------------------------
    pinned = [([t.pin_memory() for t in b], r.pin_memory()) for b, r in host_batches]
    h2d_bytes = sum(t.numel() * t.element_size() for t in pinned[0][0]) + pinned[0][1].numel() * 4
    h2d_ref = h2d_bytes          # what the reference's loop moves per step: int64 ids + bool masks, one copy per tensor
    copy_stream = torch.cuda.Stream(device=dev)
    loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()

    def upload(i):
        with torch.cuda.stream(copy_stream):
            b, r = pinned[i % NB]
            d = [t.to(dev, non_blocking=True) for t in b], r.to(dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return d, ev

    def e2e_loop_eager(n):
        nxt = upload(0)
        last = None
        for i in range(n):
            (b, r), ev = nxt
            if i + 1 < n:
                nxt = upload(i + 1)                      # H2D of step i+1 overlaps the compute of step i
            torch.cuda.current_stream().wait_event(ev)
            for t in b + [r]:
                t.record_stream(torch.cuda.current_stream())
            loss = eager_step(model, b, r, loss_fn, post)
            loss_host[i & 1].copy_(loss.detach(), non_blocking=True)     # D2H read of the step's result
            done = torch.cuda.Event()
            done.record()
            if last is not None:
                last.synchronize()                       # the host consumes step i-1's loss while step i runs
            last = done
        if last is not None:
            last.synchronize()

    # graphed public API (rbr_b200.graphs.GraphedTrainStep, staged=True): two step objects ping-pong, so that the H2D of step
    # i+1 overlaps the replay of step i.  Staged input pipeline (rbr_b200.staging, SURVEY §8f-3): each step's inputs are ONE
    # pinned host arena in wire format (token ids int32, masks derived on the device as ids != 0, the rest unchanged) uploaded
    # by ONE cudaMemcpyAsync into the device arena whose typed views are the graph's static inputs.  Packing a batch into its
    # arena is collate work (the DataLoader's pin thread) and is done before the timed region, like pin_memory().
    e2e_steps, e2e_note, packed = None, "nn.Module forward/backward (eager), one H2D copy per input tensor (int64 ids + bool masks)", None
    if graphs is not None:
        e2e_steps = [GraphedTrainStep(model, loss_fn, *dev_batches[j], warmup=1, pool=pool, post_backward=post, staged=True,
                                      host_loss=True) for j in range(2)]
        packed = [e2e_steps[0].staged.pack(b, r) for b, r in host_batches]
        h2d_bytes = e2e_steps[0].staged.h2d_bytes
        e2e_note = ("rbr_b200.graphs.GraphedTrainStep(staged=True): CUDA-graph replay; one cudaMemcpyAsync per step from a pinned arena "
                    f"({str(e2e_steps[0].staged.token_dtype).replace('torch.', '')} token ids — the narrowest type the vocabulary of "
                    f"{c['V']} allows —, masks derived on the device) straight into the graph's static inputs")
    def e2e_loop_graphed(n):
        # Two step objects ping-pong.  The main stream carries NOTHING but graph launches: the loss read-back is the last node
        # of each graph (host_loss=True), and instead of a device-side event wait in front of a launch the HOST waits for the
        # upload of step i+1 (0.15 ms, while step i runs 0.8 ms) before it launches graph i+1 — an event wait or a copy between
        # two launches keeps the next graph from being staged during the current one (tools/e2e_probe.py: +30..70 us per step).
        def load(i):
            e2e_steps[i & 1].load_packed(packed[i % NB], stream=copy_stream)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
            return ev
        done = [None, None]
        seen = 0.0
        load(0).synchronize()
        for i in range(n):
            o = e2e_steps[i & 1]
            o.replay()                                   # inputs of step i are in place (host-verified)
            d = torch.cuda.Event()
            d.record()
            done[i & 1] = d
            if i + 1 < n:
                if done[(i + 1) & 1] is not None:
                    done[(i + 1) & 1].synchronize()      # step i-1 finished: its loss is on the host, its input arena is free
                    seen += float(e2e_steps[(i + 1) & 1].loss_host[0])
                load(i + 1).synchronize()                # upload of step i+1 overlaps the replay of step i
        for j in range(2):
            if done[j] is not None:
                done[j].synchronize()
        loss_host[0] = float(e2e_steps[(n - 1) & 1].loss_host[0])
        return seen

    e2e_loop = e2e_loop_graphed if e2e_steps is not None else e2e_loop_eager
    e2e_loop(W)
    ctx.sync_all()
    sampler.mark()
    t0 = time.perf_counter()
    e2e_loop(K)
    ctx.sync_all()
    t1 = time.perf_counter()
    e2e_clocks = sampler.take()
    et = torch.tensor([t1 - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(et, op=dist.ReduceOp.MAX)
    e2e_value = world * c["B"] * K / float(et.item())
    del e2e_steps

    # ------------------------------ strong scaling beside the weak headline (N > 1): global B split over the ranks (§8e) ------------------------------
    strong = None
    if post is not None and graphs is not None and c["B"] % world == 0:
        bs = c["B"] // world
        sb = [([t.to(dev) for t in b], r.to(dev)) for b, r in make_batches(name, 2, rank, b=bs)]
        sg = [GraphedTrainStep(model, loss_fn, *sb[j], warmup=2, pool=None, post_backward=post) for j in range(2)]
        ngram = getattr(model, "ngram", None)
        saved_hook = getattr(ngram, "table_grad_hook", None)
        if ngram is not None:
            ngram.table_grad_hook = None
        sl = GraphedTrainStep(model, loss_fn, *sb[0], warmup=1, pool=sg[0].pool, post_backward=None)
        if ngram is not None:
            ngram.table_grad_hook = saved_hook
        for _ in range(20):
            sg[0].replay(); sg[1].replay()
        ms_s, _ = time_graph_loop(ctx, [g.replay for g in sg], K)
        ms_sl, _ = time_graph_loop(ctx, [sl.replay], K)
        strong = {"scaling": "strong", "global_batch": c["B"], "per_gpu_batch": bs, "value": c["B"] * K / (ms_s * 1e-3),
                  "unit": "samples/s", "ms_per_step": ms_s / K, "ms_per_step_without_exchange": ms_sl / K,
                  "exposed_collective_ms_per_step": (ms_s - ms_sl) / K}
        del sg, sl, sb
    graphs = None

    # ------------------------------ dominant kernel: tcgen05 conv forward, timed alone (rank 0) ------------------------------
    roofline, extras = None, {}
    if rank == 0:
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def time_kernel(fn, reps=20, warm=3):
            """Device time of one `fn(i)`: `reps` calls (rotating inputs) are captured into ONE CUDA graph and the replay is timed with
            CUDA events on the replay stream, so the host's launch overhead between the calls (tens of microseconds for an eager
            autograd.Function call — more than the small kernels themselves) is not part of the figure.  Falls back to eager calls
            on torch's current stream (the stream the library launches on) if the capture fails."""
            for i in range(warm):
                fn(i)
            torch.cuda.synchronize()
            try:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    for i in range(reps):
                        fn(i)
                g.replay()
                torch.cuda.synchronize()
                k0.record()
                g.replay()
                k1.record()
                torch.cuda.synchronize()
                ms = k0.elapsed_time(k1) / reps
                del g
                return ms
            except Exception:
                torch.cuda.synchronize()
            k0.record()
            for i in range(reps):
                fn(i)
            k1.record()
            torch.cuda.synchronize()
            return k0.elapsed_time(k1) / reps

        we = model.word_embeddings
        table = we.embedding.weight.detach()
        shadow = we.bf16_shadow() if args.precision == "bf16" else None
        if name == "dual_att":
            conv_mod = model.u_local_atten.conv[0]                  # the largest conv of the encoder: E -> 200, k = 1, gated, tanh
            w0, b0 = conv_mod.weight.detach(), conv_mod.bias.detach()
            packed = ops.conv_pack(w0)
            sides = [(dev_batches[i][0][0], None) for i in range(NB)]
            kname, act, ksz, pad, n_per_step = "local-attention conv E->200 k=1 (gated tanh)", ops.ACT_TANH, 1, 0, 2
        else:
            conv = model.ngram.conv
            packed = conv.packed(0)
            w0, b0 = conv.list_of_conv1d[0].weight.detach(), conv.list_of_conv1d[0].bias.detach()
            kname, act, ksz, pad, n_per_step = "gather+conv+bias+ReLU+max-over-time", ops.ACT_RELU, 3, 1, 2
            if name == "narre":
                sides = [(dev_batches[i][0][0].view(-1, c["T"]), dev_batches[i][0][2].view(-1, c["T"])) for i in range(NB)]
            else:
                sides = [(dev_batches[i][0][0], dev_batches[i][0][2]) for i in range(NB)]
        n_tok = sides[0][0].numel()
        hh = w0.shape[0]
        # algorithmic FLOPs: 2 * positions * H * E * k over the positions the result depends on.  A position past a document's
        # last token + 1 sees only zero rows and yields the bias again, so max-over-time does not need it: per document the needed
        # positions are min(L, len + 2) (0 for a document without tokens — NARRE pads every user / item to R reviews and ~45 % of
        # the review slots are all padding).  The kernel skips the all-padding documents (short documents) and the all-padding
        # 128-position tiles (long documents); counting the dense L positions per document, as the reference computes them, would
        # credit skipped work (a fraction above 1 is possible that way) — that figure is reported beside as "dense_equiv".
        live_frac, need_frac = 1.0, 1.0
        if sides[0][1] is not None:
            m0_ = sides[0][1].view(-1, sides[0][1].shape[-1])
            Ld = m0_.shape[1]
            pos = torch.arange(1, Ld + 1, device=m0_.device).unsqueeze(0)
            lens = (m0_.to(torch.int64) * pos).max(dim=1).values
            live_frac = float((lens > 0).float().mean().item())
            need = torch.where(lens > 0, (lens + 2).clamp(max=Ld), torch.zeros_like(lens))
            need_frac = float(need.double().sum().item() / m0_.numel())
        flops_dense = 2.0 * n_tok * hh * c["E"] * ksz
        flops = flops_dense * need_frac
        kms = time_kernel(lambda i: ops.conv_act_maxpool(table, *sides[i % NB], w0, b0, pad, act=act, precision=args.precision,
                                                         shadow=shadow, packed=packed))
        achieved = flops / (kms * 1e-3) / 1e12
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "conv_tc_traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            traffic = tj.get(name)
            traffic_src = tj.get("source", "profiles/conv_tc_traffic.json") + " (ncu --set full capture of this kernel at this shape; not re-measured in this run)"
        roofline = {"kernel": f"conv_tc2_kernel ({kname}; tcgen05 cta_group::2, TMA gather4 operands)" if args.precision == "bf16"
                    else "conv_fp32_kernel", "bound": "tensor", "achieved": achieved, "peak": peaks["tf"], "unit": "TFLOP/s",
                    "frac": achieved / peaks["tf"], "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peaks["src"] + ", burst (kernel timed alone)",
                    "ms_per_launch": kms, "timed": "CUDA events around one CUDA-graph replay of 20 back-to-back calls on rotating inputs "
                                                    "(includes the kernel's own pre-pass launches; no host launch gaps)",
                    "algorithmic_flops_per_launch": flops, "launches_per_step": n_per_step,
                    "documents_with_tokens_frac": live_frac, "positions_needed_frac": need_frac,
                    "dense_equiv": {"flops_per_launch": flops_dense, "achieved": flops_dense / (kms * 1e-3) / 1e12,
                                    "frac": flops_dense / (kms * 1e-3) / 1e12 / peaks["tf"],
                                    "note": "all L positions of every document counted, as the reference's Conv1d computes them"}}
        if not args.no_extras:
            def hbm(bytes_, ms):
                gbs = bytes_ / (ms * 1e-3) / 1e9
                return {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs / peaks["hbm"],
                        "ms_per_launch": ms, "algorithmic_bytes_per_launch": bytes_}
            # K1 standalone fp32 gather: tokens * (8 + 2*E*4) bytes (SURVEY §8d)
            outs = [None]
            gms = time_kernel(lambda i: outs.__setitem__(0, ops.gather_rows(table, sides[i % NB][0])), reps=5, warm=2)
            outs[0] = None
            extras["gather_fp32"] = hbm(n_tok * (8 + 2 * c["E"] * 4), gms)
            extras["gather_fp32"]["note"] = ("algorithmic bytes over time can exceed the HBM copy peak: the table is L2-resident "
                                             "(60 MB at vocab 50k), only the output stream reaches HBM; profiles/ holds the ncu dram__bytes")
            # K0 operand staging: fp32 table -> bf16 shadow (V*E*4 read + V*emb_pad*2 written)
            if args.precision == "bf16":
                sms = time_kernel(lambda i: ops.table_to_bf16(table), reps=10, warm=2)
                extras["table_to_bf16"] = hbm(table.numel() * 4 + shadow.numel() * 2, sms)
            if name in ("deepconn", "deepconn_infer", "narre"):
                from rbr_b200.layers import fused_head
                Bn, Hh, Kk = c["B"], c["H"], c["K"]
                ut, it = torch.randn(Bn, Hh, device=dev), torch.randn(Bn, Hh, device=dev)
                uid, iid = dev_batches[0][0][4], dev_batches[0][0][5]
                with torch.no_grad():
                    hms = time_kernel(lambda i: fused_head(model.user_feat, model.item_feat, model.fm, ut, it, uid, iid, False, None))
                # K4 head: (2H + 2K + 4)*4 + 16 bytes per sample (SURVEY §8d)
                extras["head_fwd"] = hbm(Bn * ((2 * Hh + 2 * Kk + 4) * 4 + 16), hms)
            if name == "narre":
                Bn, R, Hh, A = c["B"], c["R"], c["H"], c["A"]
                feat = torch.randn(Bn, R, Hh, device=dev)
                rid = dev_batches[0][0][6]
                att = model.user_att
                with torch.no_grad():
                    ams = time_kernel(lambda i: att(feat, rid))
                # K3 attention, one side: (R*H + R*A + H + R)*4 + R*8 bytes per sample (SURVEY §8d)
                extras["narre_attention_fwd"] = hbm(Bn * ((R * Hh + R * A + Hh + R) * 4 + R * 8), ams)

    # ------------------------------ CPU baseline on this box's host cores (rank 0, N=1 only) ------------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline, _, _, _ = cpu_arm(name, 128, 4, 1, budget_s=25.0)
        if train:
            cb32, _, _, _ = cpu_arm(name, 32, 4, 1, budget_s=8.0)
            cpu_baseline["config1_B32"] = {"value": cb32["value"], "sample": cb32["sample"]}

    # ------------------------------ the reference's formulation on library kernels, same GPU (rank 0, N=1 only) ------------------------------
    library = None
    if rank == 0 and world == 1 and train and not args.no_library_baseline:
        # checker code timed as a baseline (never on the product path): the oracle's functional PyTorch forward + autograd
        from oracle import rbr_oracle as orc
        prm = {k: v.to(dev) for k, v in synth_params(name).items()}
        b0_, r0_ = dev_batches[0]
        mname = name
        library = {}
        for tag, actx in (("fp32", torch.autocast("cuda", enabled=False)), ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16))):
            try:
                with actx:
                    for _ in range(2):
                        orc.loss_and_grads(mname, prm, b0_, r0_)
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for _ in range(3):
                        orc.loss_and_grads(mname, prm, b0_, r0_)
                    torch.cuda.synchronize()
                    sec = (time.perf_counter() - t0) / 3
                library[tag] = {"value": c["B"] / sec, "unit": "samples/s", "ms_per_step": sec * 1e3}
            except Exception as e:          # e.g. out of memory on the materialised [B,L,E] / [B,H,L] tensors
                library[tag] = {"error": f"{type(e).__name__}: {str(e)[:120]}"}
            torch.cuda.empty_cache()
        library["what"] = ("the reference's formulation (nn.Embedding gather, masked_fill, conv as shifted matmuls, max-pool, autograd "
                           "backward: oracle/rbr_oracle.py) executed with ATen/cuBLAS kernels on the same GPU and batch — the "
                           "'existing kernels' of SURVEY §2.1")
        del prm

    # ------------------------------ full trainer step: + global-norm clip + Adam in the same graph (SURVEY §8f-1) ------------------------------
    # (last: the fused optimizer re-homes the parameters into one flat buffer, which invalidates the graphs captured above)
    full_step = None
    if train and args.graphs == "auto" and not args.no_full_step:
        from rbr_b200.optim import FusedClipAdam
        opt = FusedClipAdam(model, lr=0.002, max_grad_norm=5.0)                # the reference's lr / max_grad_norm (default_*.json)
        fg, fpool = [], None
        for j in range(NB):
            g_ = GraphedTrainStep(model, loss_fn, *dev_batches[j], warmup=1, pool=fpool, post_backward=post, optimizer=opt,
                                  max_grad_norm=5.0)
            fpool = g_.pool
            fg.append(g_)
        for _ in range(8):
            for g_ in fg:
                g_.replay()
        ms_f, loss_f = time_graph_loop(ctx, [g_.replay for g_ in fg], K)
        full_step = {"value": world * c["B"] * K / (ms_f * 1e-3), "unit": "samples/s", "ms_per_step": ms_f / K,
                     "final_loss": float(loss_f.item()),
                     "what": "zero_grad + forward + MSELoss + backward" + (" + gradient all-reduce" if world > 1 else "") +
                             " + clip_grad_norm_(5.0) + Adam(lr 0.002) as ONE CUDA-graph replay (rbr_b200.optim.FusedClipAdam: Σg² + "
                             "clip·Adam over flat arenas, bf16 shadow of the word table rewritten by the update)"}
        del fg

    out = None
    if rank == 0:
        samples, reasons = value_clocks[0] + e2e_clocks[0], value_clocks[1] | e2e_clocks[1]
        out = {
            "metric": METRIC[name], "value": value, "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.precision, "data": "synthetic",
            "config": {"workload": workload_name(name), "global_batch": world * c["B"], "parallelism": f"dp{world}"},
            "run": {"warmup_requested": args.warmup, "warmup_effective": n_warm,
                    "warmup_note": "at least --warmup steps, extended to ~0.4 s so the clocks reach their boost state before the timed region",
                    "grad_allreduce": (f"{args.grad_allreduce} {ar_kind}") if ar_kind else None,
                    "l2": f"inputs rotate over {NB} distinct batches ({NB * h2d_bytes / 1e6:.0f} MB of ids+masks) on top of "
                          f"the {c['V'] * c['E'] * 4 / 1e6:.0f} MB table, its bf16 shadow and the dense gradient buffer touched every "
                          f"step: larger than the 126 MB L2",
                    "timed_loop": graph_note,
                    "step": ("eval forward under no_grad (scores only)" if not train else
                             "zero_grad + forward + MSELoss + backward" + (" + gradient all-reduce" if world > 1 else "")),
                    "parity_note": PARITY_NOTE},
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                    "how": "pinned host buffers → H2D on a copy stream (prefetch depth 1) → " + e2e_note + " → "
                           "loss copied to pinned host memory every step by the graph's last node (the host consumes step i-1's loss "
                           "while step i runs, and waits for the upload of step i+1 before launching its graph, so the compute stream "
                           "carries graph launches only); wall clock, max over ranks",
                    "h2d_bytes_per_step_reference_loop": h2d_ref},
            "gpu_launches": int(launches), "gpu_launches_per_step": launches / K,
            "clocks": sampler.summarise(samples, reasons), "roofline": roofline, "cpu_baseline": cpu_baseline,
            "final_loss": final_loss, "roofline_other": extras,
        }
        if allreduce_check is not None:
            out["allreduce_check"] = allreduce_check
        if exposed is not None:
            out["collective"] = exposed
        if strong is not None:
            out["strong"] = strong
        if library is not None:
            out["library_gpu_baseline"] = library
        if full_step is not None:
            out["full_trainer_step"] = full_step
    del model, dev_batches, pinned
    torch.cuda.empty_cache()
    return out, outputs


def measure_infer_pairs(ctx, args):
    """BASELINE.json configs[4] as written: --pairs (user, item) pairs in total, vocab 200k, each pair carrying its own two
    500-token documents (the reference's data flow, trainer/train_deepconn_pp.py:274), sharded contiguously over the ranks,
    NO collective; every rank writes its slice of the score vector.  Ids are generated on the device chunk by chunk (10 M pairs
    = 80 GB of int64 ids: never materialised).  Also reported: the same pairs scored from the per-entity feature cache
    (rbr_b200.inference.PairScorer, SURVEY §8f-2)."""
    import torch.distributed as dist
    from rbr_b200 import parallel, synth
    from rbr_b200._lib import lib
    from rbr_b200.inference import PairScorer
    name = "deepconn_infer"
    c = CFG[name]
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    model = build(name, dev, args.precision)
    parallel.broadcast_parameters(model)
    scorer = PairScorer(model)
    sh = parallel.shard_range(args.pairs, rank, world)
    n_mine = len(sh)
    scores = torch.empty(n_mine, dtype=torch.float32, device=dev)
    Bc = c["B"]
    gen = torch.Generator(device=dev)
    gen.manual_seed(synth.SEED_BASE + rank)
    NBUF = 4                                              # chunk buffers in flight: generation of chunk i+1 queues behind scoring of i

    def make_chunk(n):
        u = synth.doc_batch_device(n, c["L"], c["V"], gen, dev, dtype=torch.int32)
        i = synth.doc_batch_device(n, c["L"], c["V"], gen, dev, dtype=torch.int32)
        uid = torch.randint(1, c["U"], (n,), device=dev, generator=gen)
        iid = torch.randint(1, c["I"], (n,), device=dev, generator=gen)
        return u, i, uid, iid
    # warm-up (clock ramp) on throw-away chunks
    ctx.sampler.start()
    for _ in range(max(args.warmup, 3) + 40):
        u, i, uid, iid = make_chunk(Bc)
        scorer.score_pairs(u, i, None, None, uid, iid)
    ctx.sync_all()
    l0 = lib.rbr_launch_count()
    ev_score = []
    ctx.sampler.mark()
    t0 = time.perf_counter()
    done = 0
    while done < n_mine:
        n = min(Bc, n_mine - done)
        u, i, uid, iid = make_chunk(n)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        scores[done:done + n] = scorer.score_pairs(u, i, None, None, uid, iid)
        e1.record()
        ev_score.append((e0, e1))
        done += n
    ctx.sync_all()
    wall = time.perf_counter() - t0
    clocks = ctx.sampler.take()
    launches = lib.rbr_launch_count() - l0
    score_ms = sum(a.elapsed_time(b) for a, b in ev_score)
    outputs = {f"{name}.scores": scores.cpu()} if args.dump_outputs and rank == 0 else None   # rank 0's slice
    t = torch.tensor([wall, score_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    wall, score_ms = float(t[0]), float(t[1])
    checksum = scores.double().sum().reshape(1)
    if world > 1:
        dist.all_reduce(checksum)
    # the same number of pairs from the per-entity feature cache: U + I documents encoded once, then K1 gather + K4 head
    user_docs = synth.doc_batch_device(c["U"], c["L"], c["V"], gen, dev, dtype=torch.int32)
    item_docs = synth.doc_batch_device(c["I"], c["L"], c["V"], gen, dev, dtype=torch.int32)
    torch.cuda.synchronize()
    tb = time.perf_counter()
    scorer.build_cache(user_docs, item_docs)
    torch.cuda.synchronize()
    build_s = time.perf_counter() - tb
    big = 1 << 20
    tc0 = time.perf_counter()
    done = 0
    while done < n_mine:
        n = min(big, n_mine - done)
        uid = torch.randint(1, c["U"], (n,), device=dev, generator=gen)
        iid = torch.randint(1, c["I"], (n,), device=dev, generator=gen)
        scores[done:done + n] = scorer.score_cached(uid, iid)
        done += n
    ctx.sync_all()
    cached_s = time.perf_counter() - tc0
    tt = torch.tensor([build_s, cached_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    if rank != 0:
        return None, None
    return {
        "metric": METRIC[name], "value": args.pairs / (score_ms * 1e-3), "unit": "pairs/s", "n_gpus": world,
        "steps": len(ev_score), "warmup": args.warmup, "ms_per_step": score_ms / max(len(ev_score), 1), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
        "config": {"workload": workload_name(name), "total_pairs": args.pairs, "pairs_per_gpu": n_mine, "parallelism": f"dp{world} (no collective)"},
        "run": {"value_is": "total pairs / summed CUDA-event time of the scoring calls (max over ranks)",
                "total_wall_s": wall, "total_wall_includes": "on-device generation of the ids (80 GB of int64-equivalent for 10 M pairs, produced "
                "per 4096-pair chunk as int32) + scoring + writing each rank's slice of the score vector",
                "pairs_per_s_wall": args.pairs / wall, "score_checksum": float(checksum.item())},
        "e2e": {"value": args.pairs / wall, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "how": "ids are synthesised on the device (config 5 has no host data set); wall clock of the whole job, max over ranks"},
        "feature_cache": {"build_s": float(tt[0]), "entities": c["U"] + c["I"], "score_s": float(tt[1]),
                          "pairs_per_s": args.pairs / float(tt[1]), "pairs_per_s_incl_build": args.pairs / float(tt[0] + tt[1]),
                          "what": "rbr_b200.inference.PairScorer: each entity's document encoded once, pairs scored with K1 gather + K4 head "
                                  "(bit-identical scores, tests/test_gpu_benchcfg.py)"},
        "gpu_launches": int(launches), "gpu_launches_per_step": launches / max(len(ev_score), 1),
        "clocks": ctx.sampler.summarise(*clocks),
    }, outputs


def dump_outputs(outputs, out_dir):
    """Write each CPU tensor of `outputs` as out_dir/<name>.npy in float32, DUMP_BYTES in all.  Smaller arrays are written
    whole; an array over its share of what is left is cut to that many of its elements, flattened, at indices drawn by a
    fixed seed (the same for the same arguments, so two builds write the same sample)."""
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(outputs.items(), key=lambda kv: (kv[1].numel(), kv[0]))
    left = (DUMP_BYTES - 256 * len(items)) // 4          # float32 elements, after a 256-byte allowance per .npy header
    for j, (name, t) in enumerate(items):
        share = left // (len(items) - j)
        if t.numel() > share:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:share].sort().values
            t = t.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), t.to(torch.float32).numpy())
        left -= t.numel()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--model", default="all", choices=["all", "deepconn", "narre", "dual_att"],
                    help="all (default) = DeepCoNN at the top level + NARRE under the `narre` key: BASELINE.json's metric names both")
    ap.add_argument("--mode", default="train", choices=["train", "infer"],
                    help="infer = DeepCoNN eval forward at vocab 200k (BASELINE.json configs[4])")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--grad-allreduce", default="fp32", choices=["fp32", "bf16"],
                    help="wire dtype of the data-parallel gradient all-reduce (bf16 = optional compression, rounds the averaged gradient)")
    ap.add_argument("--allreduce", default="nvls", choices=["nvls", "multimem", "p2p", "nccl"],
                    help="nvls = the library's own kernels on a symmetric-memory gradient arena: peer loads / stores on 2 GPUs, the "
                         "multimem kernel through the NVSwitch above (falls back to nccl when multicast is unavailable); multimem / "
                         "p2p force one of the two; nccl = one ncclAllReduce of the arena")
    ap.add_argument("--graphs", default="auto", choices=["auto", "off"],
                    help="auto: the timed loops replay CUDA graphs of the step (rbr_b200.graphs.GraphedTrainStep, one per rotating "
                         "batch; at N>1 the gradient exchange is captured with it), so host scheduling jitter cannot make them "
                         "CPU-bound; off: eager nn.Module calls")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true",
                    help="skip timing the reference's formulation on ATen/cuBLAS kernels on this GPU (library_gpu_baseline)")
    ap.add_argument("--no-extras", action="store_true", help="skip the per-kernel extras (roofline_other)")
    ap.add_argument("--no-full-step", action="store_true", help="skip the full trainer step (clip + Adam captured with the step)")
    ap.add_argument("--pairs", type=int, default=0,
                    help="--mode infer: score this many synthetic (user, item) pairs in total (BASELINE.json configs[4]: 10000000), "
                         "sharded over the ranks with no collective, ids generated on the device chunk by chunk")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<workload>.<name>.npy (float32, at most "
                         "64 MB in all: larger arrays are cut to a fixed, seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of --impl ours")
        return run_reference_arm(args)

    import torch.distributed as dist
    from rbr_b200 import parallel
    try:
        torch.autograd.graph.set_warn_on_accumulate_grad_stream_mismatch(False)      # side-stream backward is intentional
    except Exception:
        pass

    ctx = Ctx()
    ctx.rank, ctx.local, ctx.world = parallel.init_from_env("nccl")
    if ctx.world != args.gpus and ctx.rank == 0 and ctx.world > 1:
        print(f"[bench] note: --gpus {args.gpus} but WORLD_SIZE={ctx.world}", file=sys.stderr)
    torch.cuda.set_device(ctx.local)
    ctx.dev = torch.device("cuda", ctx.local)
    ctx.peaks = load_peaks()
    ctx.sampler = ClockSampler(ctx.local)

    def sync_all():
        torch.cuda.synchronize()
        if ctx.world > 1:
            dist.barrier()
            torch.cuda.synchronize()
    ctx.sync_all = sync_all

    if args.mode == "infer" and args.pairs > 0:
        line, outputs = measure_infer_pairs(ctx, args)
        ctx.sampler.stop()
        if ctx.rank == 0:
            if args.dump_outputs:
                dump_outputs(outputs, args.dump_outputs)
            print(json.dumps(line), flush=True)
        if ctx.world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    if args.mode == "infer":
        models = ["deepconn_infer"]
    elif args.model == "all":
        models = ["deepconn", "narre"]
    else:
        models = [args.model]
    line, outputs = None, {}
    for mi, m in enumerate(models):
        d, o = measure(ctx, m, args)
        if ctx.rank == 0:
            if mi == 0:
                line = d
            else:
                line[m] = d
            outputs.update(o or {})
    ctx.sampler.stop()
    if ctx.rank == 0:
        if args.dump_outputs:
            dump_outputs(outputs, args.dump_outputs)
        print(json.dumps(line), flush=True)
    if ctx.world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
