"""Timing harness for the K2c coefficient scatter on synthetic NARRE / DeepCoNN shaped inputs (L2 flushed between launches).
    [UB_I64=1] [UB_FLUSH=write|read|none] python tools/ubench_scatter.py narre|deepconn
(The numbers in profiles/r02_ub_scatter.txt with "dbg=1" were taken with a since-removed switch that disabled the atomics.)"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from rbr_b200 import ops
from rbr_b200._lib import lib

name = sys.argv[1] if len(sys.argv) > 1 else "narre"
V, E = 50000, 300
n_docs, L, H, k = (40960, 60, 150, 3) if name == "narre" else (4096, 500, 100, 3)
dev = torch.device("cuda:0")
g = torch.Generator(device=dev).manual_seed(1)
ids = torch.randint(1, V, (n_docs, L), device=dev, generator=g, dtype=torch.int32)
if name == "narre":
    ids[torch.rand(n_docs, device=dev, generator=g) < 0.45] = 0
feat = torch.rand(n_docs, H, device=dev, generator=g) + 0.1
grad = torch.randn(n_docs, H, device=dev, generator=g)
amax = torch.randint(0, L, (n_docs, H), device=dev, generator=g, dtype=torch.int32)
bias_g = torch.zeros(H, device=dev)
ws = torch.zeros(lib.rbr_conv_bwd_cmat_workspace_bytes(V, E, H, k), dtype=torch.uint8, device=dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
p = lambda t: t.data_ptr()
st = torch.cuda.current_stream().cuda_stream
I64 = os.environ.get("UB_I64") == "1"
ids_k = ids.long() if I64 else ids
mask_k = (ids != 0).to(torch.uint8) if I64 else None
fl = 0 if I64 else (ops.IDS_I32 | ops.MASK_FROM_IDS)
nch = lib.rbr_conv_bwd_cmat_chunks(V, E, H, k)
def run(chunk=-1, bias=True, begin=True):
    if begin:
        lib.check(lib.rbr_conv_bwd_cmat_begin(chunk, V, E, H, k, p(ws), ws.numel(), st), "begin")
    lib.check(lib.rbr_conv_bwd_cmat_scatter(p(ids_k), p(mask_k) if mask_k is not None else None, n_docs, L, V, E, H, k, 1, ops.ACT_RELU,
                                            p(feat), p(amax), p(grad), H, p(bias_g) if bias else None, chunk, p(ws), ws.numel(), fl, st),
              "scatter")
FLUSH = os.environ.get("UB_FLUSH", "write")
def timeit(fn, reps=5):
    ts = []
    for _ in range(reps):
        if FLUSH == "write":
            flush.zero_()
        elif FLUSH == "read":
            flush.sum()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return min(ts[1:])
print(f"flush={FLUSH} i64={I64} {name} chunks={nch}: all blocks (zero-fill + scatter) {timeit(run):.1f} us | "
      f"without the zero-fill {timeit(lambda: run(begin=False)):.1f} us | block 0 only: with fill {timeit(lambda: run(0)):.1f} us, without {timeit(lambda: run(0, begin=False)):.1f} us")
