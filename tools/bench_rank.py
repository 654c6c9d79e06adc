"""Full-catalogue ranking of held-out items: PairScorer.rank_items (K11) against a dense baseline (chunked fp32 scores with TF32
off, then per-target comparison counts with the same tie rule), at bench_recommend's sizes: U = 20 000 users (all of them as
rows) x I = 12 000 items, seeded features for DeepCoNN, NARRE and D-ATT (bench_recommend.scorer).

Four workloads per model: 1 target per user (leave-one-out) and 10 targets per user, each without and with 50 excluded
items per user; targets and exclusions are distinct random items other than the padding item.  Both results are compared in
the same run: ranks must be equal except where another eligible item's score lies within 1e-5 of the row's largest |score|
of the target's score (there fp32 rounding may order them either way), and scores must agree to that tolerance.

    python tools/bench_rank.py --out DIR [--reps 10]      → DIR/bench_rank.json
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_recommend import I, U, gpu_info, scorer, timed  # noqa: E402


def dense(sc, u_ids, targets, excl, chunk=2048):
    """From the materialised fp32 score matrix, chunk rows at a time, per target: rank, score, the number of other eligible
    items within 1e-5 of the row's largest |score| of its score, and that largest |score|."""
    A, rb, B, cb = sc.factors()
    cbp = torch.zeros(B.shape[0], device=B.device) if cb is None else cb.clone()
    cbp[0] = float("-inf")                                      # the padding item, as rank_items(exclude_padding=True)
    t_ptr, t_idx = targets
    ids = torch.arange(B.shape[0], device=B.device)
    ranks, scores, near, scales = [], [], [], []
    for lo in range(0, u_ids.numel(), chunk):
        n = min(chunk, u_ids.numel() - lo)
        u = u_ids[lo:lo + n]
        S = A[u] @ B.T + cbp.view(1, -1)
        if rb is not None:
            S += rb[u].view(-1, 1)
        if excl is not None:
            ptr, idx = excl
            rows = torch.repeat_interleave(torch.arange(n, device=S.device), ptr[lo + 1:lo + n + 1] - ptr[lo:lo + n])
            S[rows, idx[ptr[lo]:ptr[lo + n]]] = float("-inf")
        S = torch.where(torch.isnan(S), torch.full_like(S, float("-inf")), S)
        rows = torch.repeat_interleave(torch.arange(n, device=S.device), t_ptr[lo + 1:lo + n + 1] - t_ptr[lo:lo + n])
        t = t_idx[t_ptr[lo]:t_ptr[lo + n]]
        Sr = S[rows]
        st = Sr.gather(1, t.view(-1, 1))
        beats = (Sr > st) | ((Sr == st) & (ids.view(1, -1) <= t.view(-1, 1)))
        r = (beats & (Sr > float("-inf"))).sum(1)
        ranks.append(torch.where(st.view(-1) > float("-inf"), r, torch.full_like(r, -1)))
        scores.append(st.view(-1))
        scale = torch.where(torch.isfinite(S), S.abs(), torch.zeros_like(S)).amax(1)[rows].view(-1, 1)
        near.append(((Sr - st).abs() <= 1e-5 * scale).sum(1) - 1)
        scales.append(scale.view(-1))
    return torch.cat(ranks), torch.cat(scores), torch.cat(near), torch.cat(scales)


def workload(n_tgt, n_excl, seed):
    """n_tgt targets and n_excl exclusions per user: distinct items in [1, I), the two sets disjoint"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    picks = torch.rand(U, I - 1, device="cuda", generator=g).topk(n_tgt + n_excl, dim=1).indices + 1
    t_idx = picks[:, :n_tgt].reshape(-1).contiguous()
    targets = (torch.arange(0, U * n_tgt + 1, n_tgt, device="cuda"), t_idx)
    excl = None
    if n_excl:
        excl = (torch.arange(0, U * n_excl + 1, n_excl, device="cuda"), picks[:, n_tgt:].reshape(-1).contiguous())
    return targets, excl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rank needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()
    u_ids = torch.arange(U, device="cuda")
    loads = {(t, e): workload(t, e, 1 + t + e) for t in (1, 10) for e in (0, 50)}
    runs = []
    for model in ("deepconn", "narre", "dual_att"):
        sc = scorer(model)
        A, _, _, _ = sc.factors()
        for (n_tgt, n_excl), (targets, excl) in loads.items():
            t_rank, (r_k, s_k, _) = timed(lambda: sc.rank_items(u_ids, targets, exclude=excl), args.reps)
            t_den, (r_d, s_d, near, scale) = timed(lambda: dense(sc, u_ids, targets, excl), args.reps)
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            sc.rank_items(u_ids, targets, exclude=excl)
            torch.cuda.synchronize()
            peak = torch.cuda.max_memory_allocated() - base
            diff = (r_k - r_d).abs()
            score_dev = float(((s_k.double() - s_d.double()).abs() / scale.double().clamp_min(1e-30)).max())
            ranks_ok = bool((diff <= near).all())
            runs.append({
                "model": model, "dim": A.shape[1], "targets_per_user": n_tgt, "excluded_per_user": n_excl,
                "rank_items_ms": round(t_rank, 4), "dense_fp32_count_ms": round(t_den, 4), "speedup": round(t_den / t_rank, 2),
                "rank_items_peak_mb": round(peak / 2 ** 20, 1), "dense_score_matrix_mb": round(U * I * 4 / 2 ** 20, 1),
                "fraction_equal_ranks": round(float((diff == 0).double().mean()), 6), "max_rank_diff": int(diff.max()),
                "max_rel_score_dev": score_dev, "ok": ranks_ok and score_dev <= 1e-5,
            })
            print(json.dumps(runs[-1]), flush=True)
    res = {**info, "U": U, "I": I, "reps": args.reps, "runs": runs, "all_ok": all(r["ok"] for r in runs)}
    with open(os.path.join(args.out, "bench_rank.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "runs"}))
    if not res["all_ok"]:
        raise SystemExit("bench_rank: K11 and the dense baseline disagree")


if __name__ == "__main__":
    main()
