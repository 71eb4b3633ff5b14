"""bench_aggr.py — the native aggregators on the GPU (not a pytest file).

Kernels, on R-MAT (default scale 22) at H = 64 / 128 / 256, CUDA-event timed with the L2 overwritten between
launches: SUM, AVG (the MEAN epilogue), MAX forward (with winner ids), MAX backward (roc_sg_arg_backward) and a
torch baseline (index_select + scatter_reduce_ "amax" / "mean", include_self=False) where its E x H
intermediate fits.  Algorithmic bytes: SUM / AVG E(4H+4) + N(4H+8); MAX forward E(4H+4) + N(8H+8); MAX backward
E(8H+4) + N(4H+8).  Then the training-step time of build_sage(mean), build_sage(max) and the composed
build_sage_mean on the products-shaped graph of BASELINE configs[2] (100-256-256-47).  One JSON line per case;
the first line names the GPU and its power limit.
    python tests/bench_aggr.py [--scale 22] [--hs 64,128,256] [--iters 10] [--steps 5] [--no-step]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from roc_b200 import datasets  # noqa: E402
from roc_b200 import kernels as K  # noqa: E402


def timeit(fn, iters, flush):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / iters


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # noqa: BLE001
        q = "nvidia-smi unavailable: %s" % e
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q}


def kernels(a, flush):
    dev = "cuda"
    re, col = datasets.rmat_graph(a.scale, 1 << (a.scale + 3), seed=1, device=dev)
    n, e = re.shape[0], col.shape[0]
    plan = K.SgPlan(0, n - 1, 0, re, col)
    print(json.dumps({"graph": "R-MAT scale-%d" % a.scale, "N": n, "E": e, "plan": plan.info()}), flush=True)
    dst = torch.repeat_interleave(torch.arange(n, device=dev), torch.diff(re, prepend=torch.zeros(1, dtype=re.dtype,
                                                                                                 device=dev)))
    col64 = col.long()
    for h in [int(v) for v in a.hs.split(",")]:
        x = K.padded(n, h, dev)
        x.copy_(torch.rand((n, h), device=dev) - 0.5)
        gy = K.padded(n, h, dev)
        gy.copy_(torch.rand((n, h), device=dev) - 0.5)
        out = K.padded(n, h, dev)
        arg = K.padded(n, h, dev, dtype=torch.int32)
        gin = K.padded(n, h, dev)
        plan.reserve(h)
        plan.reserve_arg(h)
        sum_b = e * (4 * h + 4) + n * (4 * h + 8)
        rows = [("sum", lambda: plan.forward(x, out=out), sum_b),
                ("avg", lambda: plan.forward(x, out=out, epilogue=4), sum_b),
                ("max_fwd", lambda: plan.aggr_forward(x, "max", out=out, arg=arg), e * (4 * h + 4) + n * (8 * h + 8)),
                ("max_bwd", lambda: plan.arg_backward(gy, arg, out=gin), e * (8 * h + 4) + n * (4 * h + 8))]
        res = {"H": h}
        for name, fn, b in rows:
            ms = timeit(fn, a.iters, flush)
            res[name + "_ms"] = round(ms, 4)
            res[name + "_GBps"] = round(b / ms / 1e6, 1)
        free = torch.cuda.mem_get_info()[0]
        if e * h * 4 * 2.5 < free:
            xd = x.contiguous()
            for red in ("amax", "mean"):
                def tb():
                    g = xd.index_select(0, col64)
                    o = torch.zeros((n, h), device=dev)
                    o.scatter_reduce_(0, dst[:, None].expand(-1, h), g, red, include_self=False)
                    return o
                ms = timeit(tb, max(2, a.iters // 2), flush)
                res["torch_%s_ms" % red] = round(ms, 4)
            torch.cuda.empty_cache()
        else:
            res["torch"] = "E x H intermediate does not fit"
        print(json.dumps(res), flush=True)
    del plan


def steps(a):
    from roc_b200.model import Host, Model, build_sage, build_sage_mean
    layers = [100, 256, 256, 47]
    re, col = datasets.powerlaw_graph(2449029, 30_000_000, alpha=1.6, seed=1, device="cuda")
    row_end, colh = re.cpu().numpy().astype(np.uint64), col.cpu().numpy().astype(np.uint32)
    del re, col
    n = row_end.shape[0]
    feats, labels, mask = datasets.node_data(n, layers[0], layers[-1], seed=1)
    print(json.dumps({"graph": "products-shaped", "N": n, "E": int(row_end[-1]), "layers": layers}), flush=True)
    builders = [("sage_native_mean", lambda m: build_sage(m, layers, 0.5, aggr="mean")),
                ("sage_native_max", lambda m: build_sage(m, layers, 0.5, aggr="max")),
                ("sage_composed_mean", lambda m: build_sage_mean(m, layers, 0.5))]
    for rep in range(2):                      # alternate the models: run-to-run spread is visible
        for name, build in builders:
            host = Host(0, 0, 1)
            host.graph_from_arrays(row_end, colh)
            m = Model(host, seed=1)
            h = build(m)
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
            print(json.dumps({"model": name, "rep": rep, "step_ms": round(ms, 3)}), flush=True)
            host.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=int, default=22)
    ap.add_argument("--hs", default="64,128,256")
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
