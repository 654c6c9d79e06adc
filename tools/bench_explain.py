"""Explanations of served recommendations: PairScorer.explain (K12) for every user's top-10 from recommend, against gradient x
input by autograd on the oracle formulation (fp32 on the GPU, TF32 off, in chunks, with the embedded tokens materialised).

Set-up: U = 20 000 users x I = 12 000 items, vocabulary 50 000, seeded parameters and documents:
  DeepCoNN  E = 300, documents of L = 500 tokens (lengths 200..500), H = 100 filters of width 3;
  NARRE     E = 300, 10 reviews of 60 tokens per entity (lengths 20..60, trailing all-padding reviews), H = 150, attention 32;
  D-ATT     E = 100, documents of L = 500 tokens (lengths 200..500), local window 5, 200 local and 3 x 100 global filters,
            FC 500 → 500 → 50; explain(attribution=True).
Pairs: each user's top-10 from recommend = 200 000 pairs.

Reported per model: build_cache() and build_cache(explain=True) times and the bytes the explain cache adds; explain time
(CUDA events over --reps calls after warm-up) and peak memory on the 200 000 pairs with and without maps, and on the first
--baseline-pairs pairs; the baseline's time and peak memory on those same pairs, and the largest map difference between the
two relative to each pair's largest |attribution| (the baseline routes through the cache's arg-max, so both compute the same
quantity).

    python tools/bench_explain.py --out DIR [--model deepconn|narre|datt|all] [--precision bf16|fp32] [--reps 3]
        [--baseline-pairs 4096]   → DIR/bench_explain_<precision>.json (--model all, the default: DeepCoNN and NARRE),
                                    DIR/bench_explain_<model>_<precision>.json otherwise
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import rbr_b200  # noqa: E402
from bench_recommend import I, U, gpu_info, timed  # noqa: E402
from oracle import rbr_oracle as orc  # noqa: E402
from rbr_b200 import synth  # noqa: E402
from rbr_b200.inference import PairScorer  # noqa: E402

VOCAB, EMB = 50000, 300
DATT_EMB, DATT_L = 100, 500


def docs(n, L, seed, min_len):
    g = torch.Generator(device="cuda").manual_seed(seed)
    d = torch.randint(1, VOCAB, (n, L), device="cuda", generator=g)
    lens = torch.randint(min_len, L + 1, (n, 1), device="cuda", generator=g)
    return torch.where(torch.arange(L, device="cuda").view(1, -1) < lens, d, torch.zeros_like(d))


def build(model, precision):
    if model == "datt":
        m = rbr_b200.DualAtt(VOCAB, DATT_L, 5, 200, 100, DATT_EMB, 500, 50, 0.0, None, precision=precision)
        m.load_state_dict(synth.dual_att_params(VOCAB, DATT_L, 5, 200, 100, DATT_EMB, 500, 50, seed=0))
        return PairScorer(m.cuda()), (docs(U, DATT_L, 1, 200), docs(I, DATT_L, 2, 200)), {}
    if model == "narre":
        R, T = 10, 60
        m = rbr_b200.NARRE(U, I, VOCAB, [3], 150, EMB, 32, 32, R, T, 0.0, 0, 0, 0, None, "CNN", precision=precision)
        m.load_state_dict(synth.narre_params(U, I, VOCAB, EMB, 150, 32, 32, (3,), seed=0))
        ud, idd = docs(U * R, T, 1, 20).view(U, R, T), docs(I * R, T, 2, 20).view(I, R, T)
        nrev_u = torch.randint(1, R + 1, (U, 1), device="cuda")              # trailing reviews are all padding
        nrev_i = torch.randint(1, R + 1, (I, 1), device="cuda")
        ud = torch.where((torch.arange(R, device="cuda").view(1, -1) < nrev_u).unsqueeze(-1), ud, torch.zeros_like(ud))
        idd = torch.where((torch.arange(R, device="cuda").view(1, -1) < nrev_i).unsqueeze(-1), idd, torch.zeros_like(idd))
        kw = {"user_rev_ids": torch.randint(1, I, (U, R), device="cuda"), "item_rev_ids": torch.randint(1, U, (I, R), device="cuda")}
    else:
        m = rbr_b200.DeepCoNNpp(U, I, VOCAB, [3], EMB, 100, 32, 500, None, 0.0, precision=precision)
        m.load_state_dict(synth.deepconn_params(U, I, VOCAB, EMB, 100, 32, (3,), seed=0))
        ud, idd = docs(U, 500, 1, 200), docs(I, 500, 2, 200)
        kw = {}
    return PairScorer(m.cuda()), (ud, idd), kw


def once_ms(fn):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def peak_mb(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return round((torch.cuda.max_memory_allocated() - base) / 2 ** 20, 1)


def datt_side(p, x, s, amax):
    """D-ATT's pooled features of one side on the oracle formulation (orc.local_attention / global_attention), pooled at
    the cache's arg-max amax [N, 200 + 3 * 100]"""
    aw, ab = p[f"{s}_local_atten.attn.0.weight"], p[f"{s}_local_atten.attn.0.bias"]
    gate = torch.sigmoid(orc.conv1d_valid(x, aw, ab, pad=(aw.shape[2] - 1) // 2))
    a = amax.long()
    lo = p[f"{s}_local_atten.conv.0.weight"].shape[0]
    y = torch.tanh(orc.conv1d_valid(gate * x, p[f"{s}_local_atten.conv.0.weight"], p[f"{s}_local_atten.conv.0.bias"]))
    feats, col = [y.gather(1, a[:, :lo].unsqueeze(1)).squeeze(1)], lo
    gg = torch.sigmoid(orc.conv1d_valid(x, p[f"{s}_global_atten.attn.0.weight"], p[f"{s}_global_atten.attn.0.bias"]))
    for c in (1, 2, 3):
        w, b = p[f"{s}_global_atten.conv{c}.0.weight"], p[f"{s}_global_atten.conv{c}.0.bias"]
        y = torch.tanh(orc.conv1d_valid(gg * x, w, b))
        feats.append(y.gather(1, a[:, col:col + w.shape[0]].unsqueeze(1)).squeeze(1))
        col += w.shape[0]
    return torch.cat(feats, 1)


def baseline(sc, inputs, kw, u_all, i_all, chunk):
    """fp32 autograd gradient x input on the oracle formulation, chunk pairs at a time → (user maps, item maps)"""
    p = {k: v.detach().float() for k, v in sc.model.state_dict().items()}
    table = p["word_embeddings.embedding.weight"]
    if isinstance(sc.model, rbr_b200.DualAtt):
        c = sc._explain
        ud, idd = inputs
        maps_u, maps_i = [], []
        for lo in range(0, u_all.numel(), chunk):
            u, i = u_all[lo:lo + chunk], i_all[lo:lo + chunk]
            ux = orc.embedding_gather(table, ud[u]).requires_grad_()
            ix = orc.embedding_gather(table, idd[i]).requires_grad_()
            outs = []
            for x, s, amax in ((ux, "u", c["user"]["argmax"][u]), (ix, "i", c["item"]["argmax"][i])):
                f = datt_side(p, x, s, amax)
                outs.append(torch.relu(f @ p["fc.0.weight"].t() + p["fc.0.bias"]) @ p["fc.3.weight"].t() + p["fc.3.bias"])
            (outs[0] * outs[1]).sum().backward()
            maps_u.append((ux * ux.grad).sum(-1).detach())
            maps_i.append((ix * ix.grad).sum(-1).detach())
        return torch.cat(maps_u), torch.cat(maps_i)
    ws, bs = orc._conv_params(p, "ngram.feature_layer.0.list_of_conv1d")
    c = sc._explain
    ud, idd = inputs
    narre = isinstance(sc.model, rbr_b200.NARRE)
    maps_u, maps_i = [], []
    for lo in range(0, u_all.numel(), chunk):
        u, i = u_all[lo:lo + chunk], i_all[lo:lo + chunk]
        ux = orc.embedding_gather(table, ud[u]).requires_grad_()
        ix = orc.embedding_gather(table, idd[i]).requires_grad_()
        if narre:
            b, R, T = ud[u].shape
            H = c["user"]["feat"].shape[1]
            feats = []
            for x, d, ids, side, rev in ((ux, ud[u], u, "user", kw["user_rev_ids"]), (ix, idd[i], i, "item", kw["item_rev_ids"])):
                rf = orc.ngram_feat(x.view(b * R, T, -1), (d != 0).view(b * R, T), ws, bs,
                                    argmax_override=c[side]["argmax"].view(-1, R, H)[ids].reshape(-1, H)).view(b, R, H)
                att = {k: p[f"{side}_att.{k}"] for k in ("W_rv", "W_id", "h", "b_1", "b_2")}
                feats.append(orc.linear_attention(rf, rev[ids], ebd_vals=p[f"{side}_att.ebd_vals.weight"], **att)[0])
            uf, itf = feats
        else:
            uf = orc.ngram_feat(ux, ud[u] != 0, ws, bs, argmax_override=c["user"]["argmax"][u])
            itf = orc.ngram_feat(ix, idd[i] != 0, ws, bs, argmax_override=c["item"]["argmax"][i])
        u_f = orc.last_feat(uf, u, p["user_feat.W"], p["user_feat.b"], p["user_feat.ebd.weight"])
        i_f = orc.last_feat(itf, i, p["item_feat.W"], p["item_feat.b"], p["item_feat.ebd.weight"])
        pred = orc.fm_head(u_f, i_f, u, i, p["fm.h"], p["fm.g_bias"], p["fm.user_bias.weight"], p["fm.item_bias.weight"])
        pred.sum().backward()
        maps_u.append((ux * ux.grad).sum(-1).detach())
        maps_i.append((ix * ix.grad).sum(-1).detach())
    return torch.cat(maps_u), torch.cat(maps_i)


def rel_per_pair(a, b):
    """per pair: the largest |difference| over its positions relative to the pair's largest |attribution|"""
    a, b = a.flatten(1).double(), b.flatten(1).double()
    return (a - b).abs().amax(1) / b.abs().amax(1).clamp_min(1e-30)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--baseline-pairs", type=int, default=4096)
    ap.add_argument("--baseline-chunk", type=int, default=256)
    ap.add_argument("--precision", choices=("bf16", "fp32"), default="bf16", help="the conv forward's precision")
    ap.add_argument("--model", choices=("all", "deepconn", "narre", "datt"), default="all",
                    help="all: DeepCoNN and NARRE; datt: D-ATT's gradient x input (explain(attribution=True))")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_explain needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()
    runs = []
    models = ("deepconn", "narre") if args.model == "all" else (args.model,)
    for model in models:
        sc, inputs, kw = build(model, args.precision)
        datt = model == "datt"
        xkw = {"attribution": True} if datt else {}
        sc.build_cache(*inputs, **kw)                                         # warm-up (module loads, operand staging)
        t_plain, _ = once_ms(lambda: sc.build_cache(*inputs, **kw))
        sc.build_cache(*inputs, **kw, explain=True)
        t_expl, _ = once_ms(lambda: sc.build_cache(*inputs, **kw, explain=True))
        keys = ("argmax", "contrib", "gate_coef", "gate_vec", "hid_mask") if datt else ("feat", "argmax", "contrib")
        cache_mb = {k: round(sum(v[k].numel() * v[k].element_size() for v in sc._explain.values()) / 2 ** 20, 1)
                    for k in keys}
        cache_bytes_per_entity = round(sum(v[k].numel() * v[k].element_size() for v in sc._explain.values() for k in keys)
                                       / (U + I))
        u_ids = torch.arange(U, device="cuda")
        _, items = sc.recommend(u_ids, 10)
        uu = u_ids.view(-1, 1).expand(-1, 10).reshape(-1)
        ii = items.reshape(-1)
        t_nomap, e = timed(lambda: sc.explain(uu, ii, **xkw), args.reps)
        t_map, _ = timed(lambda: sc.explain(uu, ii, return_maps=True, **xkw), args.reps)
        mem_nomap = peak_mb(lambda: sc.explain(uu, ii, **xkw))
        mem_map = peak_mb(lambda: sc.explain(uu, ii, return_maps=True, **xkw))
        nb = args.baseline_pairs
        ub, ib = uu[:nb], ii[:nb]
        t_sub, es = timed(lambda: sc.explain(ub, ib, return_maps=True, **xkw), args.reps)
        t_base, (bu, bi) = timed(lambda: baseline(sc, inputs, kw, ub, ib, args.baseline_chunk), 1)
        mem_base = peak_mb(lambda: baseline(sc, inputs, kw, ub, ib, args.baseline_chunk))
        diff = torch.cat([rel_per_pair(es.user.map, bu), rel_per_pair(es.item.map, bi)])
        runs.append({
            "model": model, "precision": sc.model.precision if datt else sc.model.ngram.precision, "pairs": uu.numel(),
            "build_cache_ms": round(t_plain, 2), "build_cache_explain_ms": round(t_expl, 2), "explain_cache_mb": cache_mb,
            "explain_cache_bytes_per_entity": cache_bytes_per_entity,
            "explain_ms": round(t_nomap, 3), "explain_maps_ms": round(t_map, 3),
            "explain_peak_mb": mem_nomap, "explain_maps_peak_mb": mem_map,
            "baseline_pairs": nb, "explain_baseline_pairs_ms": round(t_sub, 3),
            "autograd_baseline_ms": round(t_base, 2), "autograd_baseline_peak_mb": mem_base,
            "speedup_on_baseline_pairs": round(t_base / t_sub, 1),
            "map_diff_rel_to_pair_max": {"max": float(diff.max()), "p99": float(diff.quantile(0.99)),
                                         "median": float(diff.median()),
                                         "fraction_below_1e-2": float((diff <= 1e-2).double().mean()),
                                         "fraction_below_1e-5": float((diff <= 1e-5).double().mean())},
            "nan_windows": int(e.user.top_pos.lt(0).sum() + e.item.top_pos.lt(0).sum()),
        })
        print(json.dumps(runs[-1]), flush=True)
        del sc, e, es
        torch.cuda.empty_cache()
    res = {**info, "U": U, "I": I, "vocab": VOCAB, "emb": DATT_EMB if args.model == "datt" else EMB,
           "precision": args.precision, "reps": args.reps, "runs": runs}
    name = "bench_explain" if args.model == "all" else f"bench_explain_{args.model}"
    with open(os.path.join(args.out, f"{name}_{args.precision}.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "runs"}))


if __name__ == "__main__":
    main()
