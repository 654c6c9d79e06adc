"""Full-catalogue top-k: PairScorer.recommend (K10) against the dense baseline (chunked fp32 scores with TF32 off, then
torch.topk), on the synthetic sizes of SURVEY §8d: U = 20 000 users (all of them as rows), I = 12 000 items, k = 10 / 100.

The entity caches are filled with seeded random features of the shape build_cache produces ([U, H] / [I, H]; D-ATT: the FC
outputs [U, 50] / [I, 50]); recommend's cost does not depend on how they were computed.  The factors (a few MB) sit in
L2, so K10 is compute / issue bound, not HBM bound.  Both results are compared in the same run: per row, the k returned
scores must agree within 1e-5 of the row's largest |score| (items may differ only where scores tie to that tolerance).

    python tools/bench_recommend.py --out DIR [--reps 20]      → DIR/bench_recommend.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import rbr_b200  # noqa: E402
from rbr_b200 import synth  # noqa: E402
from rbr_b200.inference import PairScorer  # noqa: E402

U, I = 20000, 12000
BF16_PEAK = 2.25e15          # dense bf16 FLOP/s of one B200 (data sheet, 1000 W)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, pl, sm, smax = [x.strip() for x in q[torch.cuda.current_device()].split(",")]
    return {"device": name, "power_limit": pl, "sm_clock": sm, "sm_clock_max": smax}


def scorer(model: str):
    g = torch.Generator().manual_seed(0)
    if model == "dual_att":
        m = rbr_b200.DualAtt(1000, 64, 5, 200, 100, 100, 500, 50, 0.0, None)
        m.load_state_dict(synth.dual_att_params(1000, 64, 5, 200, 100, 100, 500, 50, seed=0))
        H = 50
    elif model == "narre":
        m = rbr_b200.NARRE(U, I, 1000, [3], 150, 64, 32, 32, 10, 60, 0.0, 0, 0, 0, None, "CNN")
        m.load_state_dict(synth.narre_params(U, I, 1000, 64, 150, 32, 32, (3,), seed=0))
        H = 150
    else:
        m = rbr_b200.DeepCoNNpp(U, I, 1000, [3], 64, 100, 32, 500, None, 0.0)
        m.load_state_dict(synth.deepconn_params(U, I, 1000, 64, 100, 32, (3,), seed=0))
        H = 100
    sc = PairScorer(m.cuda())
    # pooled ReLU / attention outputs are >= 0 (ReLU) or in (-1, 1) (D-ATT FC: any sign)
    feats = [torch.rand(n, H, generator=g) * 0.5 for n in (U, I)]
    if model == "dual_att":
        feats = [f * 4 - 1 for f in feats]
    sc.user_feat, sc.item_feat = feats[0].cuda(), feats[1].cuda()
    return sc


def dense(sc, u_ids, k, excl, chunk=4096):
    A, rb, B, cb = sc.factors()
    cbp = torch.zeros(B.shape[0], device=B.device) if cb is None else cb.clone()
    cbp[0] = float("-inf")                                      # the padding item, as recommend(exclude_padding=True)
    ss, ii = [], []
    for lo in range(0, u_ids.numel(), chunk):
        u = u_ids[lo:lo + chunk]
        S = A[u] @ B.T + cbp.view(1, -1)
        if rb is not None:
            S += rb[u].view(-1, 1)
        if excl is not None:
            ptr, idx = excl
            rows = torch.repeat_interleave(torch.arange(u.numel(), device=S.device), ptr[lo + 1:lo + u.numel() + 1] - ptr[lo:lo + u.numel()])
            S[rows, idx[ptr[lo]:ptr[lo + u.numel()]]] = float("-inf")
        s, i = torch.topk(S, k, dim=1)
        ss.append(s)
        ii.append(i)
    return torch.cat(ss), torch.cat(ii)


def timed(fn, reps):
    for _ in range(3):
        out = fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_recommend needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()
    u_ids = torch.arange(U, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(1)
    excl_idx = torch.randint(1, I, (U * 50,), device="cuda", generator=g)
    excl = (torch.arange(0, U * 50 + 1, 50, device="cuda"), excl_idx)
    runs = []
    for model, ex in (("deepconn", None), ("narre", None), ("dual_att", None), ("deepconn", excl)):
        sc = scorer(model)
        A, _, B, _ = sc.factors()
        for k in (10, 100):
            t_rec, (s_rec, i_rec) = timed(lambda: sc.recommend(u_ids, k, exclude=ex), args.reps)
            t_den, (s_den, i_den) = timed(lambda: dense(sc, u_ids, k, ex), args.reps)
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            sc.recommend(u_ids, k, exclude=ex)
            torch.cuda.synchronize()
            peak = torch.cuda.max_memory_allocated() - base
            scale = torch.maximum(s_den.abs().amax(1), s_rec.abs().amax(1)).clamp_min(1e-30)
            dev = float(((s_rec.double() - s_den.double()).abs() / scale.view(-1, 1).double()).max())
            same_items = float((i_rec == i_den).double().mean())
            dim = A.shape[1]
            dimp = (dim + 31) // 32 * 32
            flops = 2.0 * ((U + 127) // 128 * 128) * ((I + 255) // 256 * 256) * 6 * dimp
            runs.append({
                "model": model, "k": k, "dim": dim, "excluded_per_user": 0 if ex is None else 50,
                "recommend_ms": round(t_rec, 4), "dense_fp32_topk_ms": round(t_den, 4), "speedup": round(t_den / t_rec, 2),
                "scores_per_s": U * I / (t_rec * 1e-3),
                "split_gemm_gflop": round(flops / 1e9, 1), "split_gemm_share_of_bf16_peak": round(flops / (t_rec * 1e-3) / BF16_PEAK, 4),
                "recommend_peak_mb": round(peak / 2 ** 20, 1), "dense_score_matrix_mb": round(U * I * 4 / 2 ** 20, 1),
                "max_rel_score_dev": dev, "fraction_same_items": round(same_items, 5), "ok": dev <= 1e-5,
            })
            print(json.dumps(runs[-1]), flush=True)
    res = {**info, "U": U, "I": I, "reps": args.reps,
           "bound": "compute / issue: the split factors are a few MB and stay in L2; no U x I matrix is written",
           "runs": runs, "all_ok": all(r["ok"] for r in runs),
           "all_faster": all(r["speedup"] > 1 for r in runs)}
    with open(os.path.join(args.out, "bench_recommend.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "runs"}))


if __name__ == "__main__":
    main()
