"""bench_gat.py — graph attention on the GPU (not a pytest file).

Kernels, on R-MAT (default scale 22) at (H, K) = (64, 1), (64, 8), (128, 4), (256, 1), CUDA-event timed with the L2
overwritten between launches, beside SUM at the same H: scores (roc_gat_scores), forward (softmax statistics +
weighted aggregate, roc_gat_forward), c (roc_gat_bwd_c), backward gather (roc_gat_backward) and finish
(roc_gat_bwd_finish), and a torch fp32 composition of the same forward + backward (index_select, scatter_reduce,
exp, index_add, autograd) where its E x H intermediates fit.  Algorithmic bytes (A = round_up4(2K) floats per att /
bst row, N own rows, E edges):
    scores  N(4H + 4A)                     forward  E(4 + 4K) + N(4A + 4A)  +  E(4H + 4 + 4K) + N(4H + 8A)
    c       N(8H + 4A)                     gather   E(8H + 4 + 8A) + N(12H + 16A)
    finish  N(12H + 8A)
Then the training-step time of build_gat 602-64(8x8)-41 on the configs[1] graph and 100-256(4x64)-256-47 on the
products-shaped configs[2] graph, beside GCN and SAGE-mean steps from the same run.  One JSON line per case; the
first line names the GPU and its power limit.
    python tests/bench_gat.py [--scale 22] [--iters 10] [--steps 5] [--no-step] [--no-kernels]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from bench_aggr import gpu_info, timeit  # noqa: E402
from roc_b200 import datasets  # noqa: E402
from roc_b200 import kernels as K  # noqa: E402

SHAPES = [(64, 1), (64, 8), (128, 4), (256, 1)]


def torch_gat(x, a, dst, src, n, k, slope=0.2):
    h = x.shape[1]
    f = h // k
    xs = x.view(n, k, f)
    s_src = (xs * a[0].view(k, f)).sum(-1)
    s_dst = (xs * a[1].view(k, f)).sum(-1)
    e = torch.nn.functional.leaky_relu(s_src[src] + s_dst[dst], slope)
    m = torch.full((n, k), -float("inf"), device=x.device).scatter_reduce(0, dst[:, None].expand(-1, k), e.detach(),
                                                                         "amax")
    ex = torch.exp(e - m[dst])
    z = torch.zeros((n, k), device=x.device).index_add(0, dst, ex)
    alpha = ex / z[dst]
    return torch.zeros((n, k, f), device=x.device).index_add(0, dst, alpha[:, :, None] * xs[src]).view(n, h)


def kernels(a, flush):
    dev = "cuda"
    re, col = datasets.rmat_graph(a.scale, 1 << (a.scale + 3), seed=1, device=dev)
    n, e = re.shape[0], col.shape[0]
    plan = K.SgPlan(0, n - 1, 0, re, col)
    print(json.dumps({"graph": "R-MAT scale-%d" % a.scale, "N": n, "E": e, "plan": plan.info()}), flush=True)
    dst = torch.repeat_interleave(torch.arange(n, device=dev), torch.diff(re, prepend=torch.zeros(1, dtype=re.dtype,
                                                                                                 device=dev)))
    src = col.long()
    for h, k in SHAPES:
        A = (2 * k + 3) // 4 * 4
        x = K.padded(n, h, dev, fill=torch.rand((n, h), device=dev) - 0.5)
        gy = K.padded(n, h, dev, fill=torch.rand((n, h), device=dev) - 0.5)
        aw = (torch.rand((2, h), device=dev) - 0.5) / (h // k) ** 0.5
        out, dx, sumo = K.padded(n, h, dev), K.padded(n, h, dev), K.padded(n, h, dev)
        plan.reserve(h)
        plan.gat_reserve(h, k)
        att = K.gat_scores(x, aw, k)
        bst = K.padded(n, 2 * k, dev)
        ds = K.padded(n, 2 * k, dev)
        plan.gat_forward(x, att, k, out=out, bst=bst)
        K.gat_c(gy, out, bst, k)
        ws = torch.empty(int(K.lib.roc_gat_finish_workspace_bytes(h)) // 4, device=dev)
        da = torch.empty((2, h), device=dev)

        def finish():
            K.check(K.lib.roc_gat_bwd_finish(n, h, k, K._ptr(x), K._ld(x), K._ptr(aw), K._ptr(ds), K._ld(ds),
                                             K._ptr(dx), K._ld(dx), K._ptr(da), K._ptr(ws), ws.numel() * 4,
                                             K._stream()))
        rows = [("sum", lambda: plan.forward(x, out=sumo), e * (4 * h + 4) + n * (4 * h + 8)),
                ("scores", lambda: K.gat_scores(x, aw, k), n * (4 * h + 4 * A)),
                ("fwd", lambda: plan.gat_forward(x, att, k, out=out, bst=bst),
                 e * (4 + 4 * k) + n * 8 * A + e * (4 * h + 4 + 4 * k) + n * (4 * h + 8 * A)),
                ("c", lambda: K.gat_c(gy, out, bst, k), n * (8 * h + 4 * A)),
                ("bwd_gather", lambda: plan.gat_backward(x, att, bst, gy, k, dx=dx, ds=ds),
                 e * (8 * h + 4 + 8 * A) + n * (12 * h + 16 * A)),
                ("finish", finish, n * (12 * h + 8 * A))]
        res = {"H": h, "K": k}
        for name, fn, b in rows:
            ms = timeit(fn, a.iters, flush)
            res[name + "_ms"] = round(ms, 4)
            res[name + "_GBps"] = round(b / ms / 1e6, 1)
        res["gat_fwd_total_ms"] = round(res["scores_ms"] + res["fwd_ms"], 4)
        res["gat_bwd_total_ms"] = round(res["c_ms"] + res["bwd_gather_ms"] + res["finish_ms"], 4)
        free = torch.cuda.mem_get_info()[0]
        if e * h * 4 * 6 < free:
            xt = x.contiguous().requires_grad_(True)
            at = aw.clone().requires_grad_(True)
            gyc = gy.contiguous()

            def tb():
                o = torch_gat(xt, at, dst, src, n, k)
                o.backward(gyc)
                xt.grad = None
                at.grad = None
            ms = timeit(tb, max(2, a.iters // 2), flush)
            res["torch_fwd_bwd_ms"] = round(ms, 4)
            res["speedup_vs_torch"] = round(ms / (res["gat_fwd_total_ms"] + res["gat_bwd_total_ms"]), 1)
            del xt, at
            torch.cuda.empty_cache()
        else:
            res["torch"] = "E x H intermediates do not fit"
        print(json.dumps(res), flush=True)
        del x, gy, out, dx, sumo, att, bst, ds, ws
        torch.cuda.empty_cache()
    del plan


def steps(a):
    from roc_b200.model import Host, Model, build_gat, build_gcn, build_sage
    re, col = datasets.rmat_graph(22, 1 << 25, seed=1, device="cuda")
    cfg1 = (re.cpu().numpy().astype(np.uint64), col.cpu().numpy().astype(np.uint32))
    del re, col
    re, col = datasets.powerlaw_graph(2449029, 30_000_000, alpha=1.6, seed=1, device="cuda")
    cfg2 = (re.cpu().numpy().astype(np.uint64), col.cpu().numpy().astype(np.uint32))
    del re, col
    cases = [("configs[1]", cfg1, [602, 64, 41], [("gat_8x8", lambda m, l: build_gat(m, l, 8, 0.5)),
                                                    ("gcn", lambda m, l: build_gcn(m, l, 0.5)),
                                                    ("sage_mean", lambda m, l: build_sage(m, l, 0.5, aggr="mean"))]),
             ("configs[2]", cfg2, [100, 256, 256, 47], [("gat_4x64", lambda m, l: build_gat(m, l, 4, 0.5)),
                                                         ("gcn", lambda m, l: build_gcn(m, l, 0.5)),
                                                         ("sage_mean", lambda m, l: build_sage(m, l, 0.5, aggr="mean"))])]
    for gname, (row_end, colh), layers, builders in cases:
        n = row_end.shape[0]
        feats, labels, mask = datasets.node_data(n, layers[0], layers[-1], seed=1)
        print(json.dumps({"graph": gname, "N": n, "E": int(row_end[-1]), "layers": layers}), flush=True)
        for rep in range(2):                      # alternate the models: run-to-run spread is visible
            for name, build in builders:
                host = Host(0, 0, 1)
                host.graph_from_arrays(row_end, colh)
                m = Model(host, seed=1)
                h = build(m, list(layers))
                m.set_tensor(h["input"], feats.numpy())
                m.set_labels(h["label"], labels.numpy())
                m.set_tensor(h["mask"], mask.numpy().astype(np.int32))
                for _ in range(2):
                    m.train_epoch()
                host.synchronize()
                t0 = time.perf_counter()
                for _ in range(a.steps):
                    m.train_epoch()
                host.synchronize()
                ms = (time.perf_counter() - t0) / a.steps * 1e3
                print(json.dumps({"graph": gname, "model": name, "rep": rep, "step_ms": round(ms, 3)}), flush=True)
                host.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=int, default=22)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--no-step", action="store_true")
    ap.add_argument("--no-kernels", action="store_true")
    a = ap.parse_args()
    print(json.dumps(gpu_info()), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")     # 256 MB > 126 MB L2
    if not a.no_kernels:
        kernels(a, flush)
    torch.cuda.empty_cache()
    if not a.no_step:
        steps(a)


if __name__ == "__main__":
    main()
