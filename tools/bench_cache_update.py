"""Incremental feature-cache changes: PairScorer.update / add against a full PairScorer.build_cache.

Set-up: tools/bench_explain.py's models and seeded documents at U = 20 000 users x I = 12 000 items (DeepCoNN: E = 300,
L = 500, H = 100; NARRE: E = 300, 10 reviews of 60 tokens, H = 150; D-ATT: E = 100, L = 500, FC 500 -> 500 -> 50).

Reported per model, for the plain cache and the explain=True cache: build_cache time; update of n in {1, 64, 4096} users
(new documents: other users' documents) alone and followed by factors() (the refresh a serving call then does); add of 64
new users followed by recommend(k = 10) for them.  Times are CUDA events over --reps calls after warm-up calls of the same
shapes; the card's name, power limit and SM clocks are read in the same run.

    python tools/bench_cache_update.py --out DIR [--model deepconn|narre|datt|all] [--reps 5]  → DIR/bench_cache_update.json
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_explain import build, once_ms  # noqa: E402
from bench_recommend import I, U, gpu_info, timed  # noqa: E402


def side_inputs(model, inputs, kw, rows):
    """the user-side inputs of `rows` as add / update take them"""
    docs = inputs[0][rows]
    return docs, ({"rev_ids": kw["user_rev_ids"][rows]} if model == "narre" else {})


def run(model, explain, reps):
    sc, inputs, kw = build(model, "bf16")
    sc.build_cache(*inputs, **kw, explain=explain)                        # warm-up
    t_build, _ = once_ms(lambda: sc.build_cache(*inputs, **kw, explain=explain))
    sc.factors()
    out = {"model": model, "explain": explain, "build_cache_ms": round(t_build, 3)}
    g = torch.Generator().manual_seed(1)
    for n in (1, 64, 4096):
        ids = torch.randperm(U, generator=g)[:n].cuda()
        docs, rkw = side_inputs(model, inputs, kw, torch.randperm(U, generator=g)[:n].cuda())
        t_upd, _ = timed(lambda: sc.update("user", ids, docs, **rkw), reps)
        t_upd_f, _ = timed(lambda: (sc.update("user", ids, docs, **rkw), sc.factors()), reps)
        out[f"update_{n}_ms"] = round(t_upd, 3)
        out[f"update_{n}_then_factors_ms"] = round(t_upd_f, 3)
        out[f"update_{n}_vs_build"] = round(t_upd / t_build, 5)
    docs, rkw = side_inputs(model, inputs, kw, torch.arange(64, device="cuda"))

    def add_recommend():
        new = sc.add("user", docs, **rkw)
        return sc.recommend(new, 10)
    t_add, _ = timed(add_recommend, reps)
    out["add_64_then_recommend_10_ms"] = round(t_add, 3)
    out["rows_after"] = int(sc.user_feat.shape[0])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--model", default="all", choices=["deepconn", "narre", "datt", "all"])
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    res = {"gpu": gpu_info(), "U": U, "I": I, "reps": args.reps, "runs": []}
    for model in (["deepconn", "narre", "datt"] if args.model == "all" else [args.model]):
        for explain in (False, True):
            r = run(model, explain, args.reps)
            print(json.dumps(r), flush=True)
            res["runs"].append(r)
            torch.cuda.empty_cache()
    res["gpu_after"] = gpu_info()
    with open(os.path.join(args.out, "bench_cache_update.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
