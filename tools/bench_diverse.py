"""Diversified top-k: PairScorer.recommend_diverse (K10 pool + K14 MMR re-rank) against the same greedy loop written in
batched torch fp32 on the GPU after recommend(u, P), on the synthetic sizes of tools/bench_recommend.py: U = 20 000 users
(all of them as rows), I = 12 000 items with seeded cache features, DeepCoNN (item vectors H = 100) and D-ATT (D = 50),
(P, k) in {(40, 10), (256, 10), (256, 100)}, lam = 0.5.

Per run: recommend_diverse ms (CUDA events, after warm-up), K14's own ms on the same pools and its share, peak MB of the
call, the baseline's ms, intra-list diversity and catalogue coverage (inference.list_metrics) of the kernel's, the
baseline's and plain recommend(u, k)'s lists, and the fraction of rows where kernel and baseline pick the same list (the
baseline's sims come from a torch bmm, whose summation order differs from K14's, so near-ties may resolve differently).
The item features (≤ 4.8 MB) stay in L2 between passes.

    python tools/bench_diverse.py --out DIR [--reps 10]      → DIR/bench_diverse.json
"""
import argparse
import json
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

from bench_recommend import I, U, gpu_info, scorer, timed  # noqa: E402
from rbr_b200 import ops  # noqa: E402
from rbr_b200.inference import list_metrics  # noqa: E402

FP32_FMA_PEAK = 148 * 128 * 1.965e9        # fp32 FMA/s of one B200 at its 1965 MHz boost clock (148 SMs x 128 lanes)


def torch_mmr(ps, pi, vecs, k, lam, chunk=2048):
    """The greedy step of K14 in batched torch fp32: per chunk of rows k dependent steps, each an objective, an argmax, a
    gather of the picked vectors and a [rows, P, D] x [rows, D] similarity product."""
    n, P = ps.shape
    outs, outi = [], []
    lam_t = torch.tensor(lam, dtype=torch.float32, device=ps.device)
    oml = 1 - lam_t
    for lo in range(0, n, chunk):
        s, it = ps[lo:lo + chunk], pi[lo:lo + chunk]
        c = s.shape[0]
        rows = torch.arange(c, device=s.device)
        live = (it >= 0) & torch.isfinite(s)
        lo_s = torch.where(live, s, float("inf")).amin(1, keepdim=True)
        hi_s = torch.where(live, s, -float("inf")).amax(1, keepdim=True)
        rel = torch.where(hi_s == lo_s, torch.ones_like(s), (s - lo_s) / (hi_s - lo_s))
        V = vecs[it.clamp_min(0)]
        maxsim = torch.zeros_like(s)
        o_s = torch.full((c, k), -float("inf"), device=s.device)
        o_i = torch.full((c, k), -1, dtype=torch.int64, device=s.device)
        for t in range(k):
            obj = rel if t == 0 else lam_t * rel - oml * maxsim
            obj = torch.where(live, obj, -float("inf"))
            p = obj.argmax(1)
            has = live[rows, p]
            o_s[:, t] = torch.where(has, s[rows, p], -float("inf"))
            o_i[:, t] = torch.where(has, it[rows, p], -1)
            live[rows, p] = False
            sim = torch.bmm(V, V[rows, p].unsqueeze(2)).squeeze(2)
            maxsim = sim if t == 0 else torch.maximum(maxsim, sim)
        outs.append(o_s)
        outi.append(o_i)
    return torch.cat(outs), torch.cat(outi)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_diverse needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()                          # the SM clock at the start
    u_ids = torch.arange(U, device="cuda")
    lam = 0.5
    runs = []
    for model in ("deepconn", "dual_att"):
        sc = scorer(model)
        vecs = ops.unit_rows(sc.item_feat)
        D = vecs.shape[1]
        for P, k in ((40, 10), (256, 10), (256, 100)):
            t_div, (s_div, i_div) = timed(lambda: sc.recommend_diverse(u_ids, k, lam=lam, pool=P), args.reps)
            ps, pi = sc.recommend(u_ids, P)
            t_k14, _ = timed(lambda: ops.mmr_select(ps, pi, vecs, k, lam), args.reps)
            t_base, (s_b, i_b) = timed(lambda: torch_mmr(*sc.recommend(u_ids, P), vecs, k, lam), max(1, args.reps // 5))
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            sc.recommend_diverse(u_ids, k, lam=lam, pool=P)
            torch.cuda.synchronize()
            peak = torch.cuda.max_memory_allocated() - base
            m_div = list_metrics(i_div, sc.item_feat, I - 1)
            m_base = list_metrics(i_b, sc.item_feat, I - 1)
            m_rel = list_metrics(pi[:, :k], sc.item_feat, I - 1)
            fma = U * k * P * D                  # one dot per candidate and step: an upper bound (picked ones skip)
            runs.append({
                "model": model, "dim": D, "pool": P, "k": k, "lam": lam,
                "recommend_diverse_ms": round(t_div, 3), "k14_ms": round(t_k14, 3), "k14_share": round(t_k14 / t_div, 3),
                "k14_gfma": round(fma / 1e9, 2), "k14_fma_per_s": fma / (t_k14 * 1e-3),
                "k14_share_of_fp32_fma_peak": round(fma / (t_k14 * 1e-3) / FP32_FMA_PEAK, 4),
                "recommend_diverse_peak_mb": round(peak / 2 ** 20, 1), "torch_baseline_ms": round(t_base, 3),
                "speedup": round(t_base / t_div, 2),
                "ild": round(m_div["ild"], 5), "coverage": round(m_div["coverage"], 5),
                "baseline_ild": round(m_base["ild"], 5), "baseline_coverage": round(m_base["coverage"], 5),
                "relevance_only_ild": round(m_rel["ild"], 5), "relevance_only_coverage": round(m_rel["coverage"], 5),
                "fraction_same_list": round(float((i_div == i_b).all(1).double().mean()), 5),
            })
            print(json.dumps(runs[-1]), flush=True)
    res = {**info, "U": U, "I": I, "reps": args.reps, "runs": runs}
    with open(os.path.join(args.out, "bench_diverse.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "runs"}))


if __name__ == "__main__":
    main()
