#!/usr/bin/env python
"""bench.py — GCN training edges/sec on synthetic graphs (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1..5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workloads (BASELINE.json `configs`, --config; the default, 2, is the one the metric is quoted on):
  1  2-layer GCN 16-16-5 on a 1K-vertex / 10K-edge uniform graph (launch-bound)
  2  2-layer GCN 602-64-41 on R-MAT scale 22 (+log2 N: weak scaling, 2^25 pairs per GPU)
  3  3-layer GraphSAGE-mean 100-256-256-47 on a products-shaped graph (2.45M vertices / ~62M edges; strong scaling)
  4  2-layer GCN 602-128-41 on R-MAT scale 22 + log2 N (the N = 8 point is the scale-25 graph; weak scaling)
  5  4-layer GCN with the residual branch 602-256-256-256-41 on a Reddit-shaped graph (233K vertices / ~115M
     edges; strong scaling)
Graphs are symmetrised, given self loops and vertex-range partitioned by the reference's own partitioner.

A "step" is one training epoch: zero_gradients + forward + backward + update (gnn.cc:103-106), everything
resident in HBM.  `value` = total edges * steps / max-over-ranks device time (CUDA events on the engine's
stream).  `e2e` = the same metric through the public API with HOST buffers: every step re-uploads the
features / labels / mask from pinned host memory (H2D inside the timed region) and reads the loss metrics back
(D2H).  `roofline` is the ScatterGather launch at the hidden width, timed live with CUDA events inside the timed
steps; `frac` is algorithmic bytes / time / peak (can exceed 1: hub rows are served by L2), `frac_dram` uses the
DRAM traffic ncu measured for that (config, N) when profiles/sg_traffic.json has it.  `cpu_baseline` /
`--impl reference` time the CPU oracle (OpenMP, all host cores, thread count set explicitly) on a bounded sample
of the same workload — ROC ships no CPU kernels (SURVEY §8c/d).  For N > 1 a `parity_check` (outside the timed
region) trains a bounded graph on the N-rank engine and on a 1-rank engine and compares logits / loss / dW.

`--dump-outputs DIR` writes, after the timed steps, what the last timed step handed back (see dump_outputs) as
DIR/<name>.npy.  Graph, features, labels, mask and initial weights all come from fixed seeds, so two builds run
with the same arguments can be compared output for output.
"""
import argparse
import importlib.util
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DROPOUT = 0.5
LR, WD = 0.01, 0.0001          # example_run.sh: -lr 0.01 -decay 0.0001
BASE_SCALE = 22
BASE_PAIRS = 1 << 25
CPU_SAMPLE_SCALE = 19          # cpu_baseline / reference arm: same generator, 1/8 of the vertices
DUMP_ROWS = 1 << 16            # --dump-outputs: logits rows written (at most 47 classes: 12 MB)

CONFIGS = {
    1: dict(kind="gcn", layers=[16, 16, 5], graph="uniform", scaling="strong",
            desc="2-layer GCN 16-16-5, uniform 1K vertices / 10K edges"),
    2: dict(kind="gcn", layers=[602, 64, 41], graph="rmat", scaling="weak",
            desc="2-layer GCN 602-64-41, R-MAT"),
    3: dict(kind="sage", layers=[100, 256, 256, 47], graph="products", scaling="strong",
            desc="3-layer GraphSAGE-mean 100-256-256-47, products-shaped power-law graph"),
    4: dict(kind="gcn", layers=[602, 128, 41], graph="rmat", scaling="weak",
            desc="2-layer GCN 602-128-41, R-MAT"),
    5: dict(kind="gcn", layers=[602, 256, 256, 256, 41], graph="reddit", scaling="strong",
            desc="4-layer GCN + residual branch 602-256-256-256-41, Reddit-shaped power-law graph"),
}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def datasets_module():
    """roc_b200/datasets.py loaded as a plain file: the generators need only numpy + torch, and the reference
    arm must not import the product package (its .so would show up in that arm's loaded libraries)."""
    spec = importlib.util.spec_from_file_location("roc_synth_datasets", os.path.join(ROOT, "roc_b200", "datasets.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_graph(ds, cfg, world, device, scale_override=0):
    """(row_end u64, col u32, label) of config `cfg` at `world` GPUs."""
    import torch
    t0 = time.time()
    g = CONFIGS[cfg]["graph"]
    shrink = (1 << (BASE_SCALE - scale_override)) if scale_override else 1     # --scale also shrinks the fixed-size graphs (debug)
    if g == "uniform":
        row_end, col = ds.uniform_graph(1000, 4500, seed=1, device=device)
        label = "uniform 1K/10K"
    elif g == "rmat":
        scale = BASE_SCALE + int(round(math.log2(world)))
        pairs = BASE_PAIRS * world
        if scale_override:
            scale, pairs = scale_override, 1 << (scale_override + 3)
        row_end, col = ds.rmat_graph(scale, pairs, seed=1, device=device)
        label = "R-MAT scale-%d" % scale
    elif g == "products":      # configs[2]: 2.45M vertices, ~62M edges
        row_end, col = ds.powerlaw_graph(2449029 // shrink, 30_000_000 // shrink, alpha=1.6, seed=1, device=device)
        label = "products-shaped" + (" / %d" % shrink if shrink > 1 else "")
    elif g == "reddit":        # configs[4]: 233K vertices, ~115M edges (mean degree ~490)
        row_end, col = ds.powerlaw_graph(232965 // shrink, 57_500_000 // shrink, alpha=1.3, seed=1, device=device)
        label = "Reddit-shaped" + (" / %d" % shrink if shrink > 1 else "")
    else:
        raise KeyError(g)
    if device != "cpu":
        torch.cuda.synchronize()
    re_h = row_end.cpu().numpy().astype(np.uint64)
    col_h = col.cpu().numpy().astype(np.uint32)
    del row_end, col
    if device != "cpu":
        torch.cuda.empty_cache()
    log("[bench] %s: N=%d E=%d (%.1fs)" % (label, re_h.shape[0], col_h.shape[0], time.time() - t0))
    return re_h, col_h, label


def sg_bytes(n, e, h):
    """Algorithmic bytes of one ScatterGather launch (SURVEY §8d): E*(4H+4) + N*(4H+8)."""
    return e * (4 * h + 4) + n * (4 * h + 8)


def sg_compulsory_bytes(n, e, h):
    """Lower bound with perfect reuse of gathered rows (SURVEY §8d): E*4 + N*(8 + 8H)."""
    return e * 4 + n * (8 + 8 * h)


# --------------------------------------------------------------------- CPU arm ---
def cpu_epoch_rate(steps, warmup, layers):
    """Oracle GCN epoch (fp32, OpenMP on every host core) on the bounded sample.
    Returns (median edges/s, best edges/s, median ms/step, info)."""
    cores = os.cpu_count() or 1
    # torchrun exports OMP_NUM_THREADS=1; libgomp reads the environment when the oracle library is loaded
    os.environ["OMP_NUM_THREADS"] = str(cores)
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    from oracle import oracle
    ds = datasets_module()
    oracle.set_num_threads(cores)          # and set the team size explicitly as well
    pairs = BASE_PAIRS >> (BASE_SCALE - CPU_SAMPLE_SCALE)
    re_t, col_t = ds.rmat_graph(CPU_SAMPLE_SCALE, pairs, seed=1, device="cpu")
    re_h, col_h = re_t.numpy().astype(np.uint64), col_t.numpy().astype(np.uint32)
    n, e = re_h.shape[0], col_h.shape[0]
    feats, labels, mask = ds.node_data(n, layers[0], layers[-1], seed=1)
    rng = np.random.RandomState(1)
    dims = list(zip(layers[:-1], layers[1:]))
    if len(layers) > 3:                     # residual branch: a second weight per layer (gnn.cc:86-90)
        dims = [d for d in dims for _ in (0, 1)]
    ws = [((rng.rand(o, i).astype(np.float32) * 2 - 1) * np.float32(math.sqrt(6.0 / (i + o)))) for (i, o) in dims]
    m = oracle.GcnOracle(re_h, col_h, layers, ws, lr=LR, weight_decay=WD, dropout=DROPOUT, acc64=False)
    oh = ds.onehot(labels.numpy(), layers[-1])
    f, mk = feats.numpy(), mask.numpy()
    for _ in range(warmup):
        m.train_epoch(f, oh, mk)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        m.train_epoch(f, oh, mk)
        times.append(time.perf_counter() - t0)
    med, best = float(np.median(times)), float(np.min(times))
    info = {"cores": oracle.num_threads(), "kind": "port",
            "sample": "oracle GCN %s epoch (fp32, OpenMP) on R-MAT scale-%d (N=%d, E=%d), %d steps after %d warm-up; "
                      "value = median, best_value = fastest step" %
                      ("-".join(map(str, layers)), CPU_SAMPLE_SCALE, n, e, steps, warmup)}
    return e / med, e / best, 1e3 * med, info


def run_reference(args, rank, world):
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    layers = cfg["layers"] if cfg["kind"] == "gcn" else CONFIGS[2]["layers"]
    steps = args.steps
    warm = max(1, min(args.warmup, 2))
    rate, best, ms, info = cpu_epoch_rate(steps, warm, layers)
    info["value"] = rate
    info["best_value"] = best
    info["unit"] = "edges/s"
    line = {"impl": "reference", "metric": "gcn_training_edges_per_sec", "value": rate, "unit": "edges/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True,
            "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "%s (bounded CPU sample: R-MAT scale %d; the GPU arm runs the full-size graph — "
                                   "a rate metric)" % (cfg["desc"], CPU_SAMPLE_SCALE),
                       "note": "ROC ships CUDA-only kernels and cannot be built here (Legion absent); the reference "
                               "arm is the CPU restatement of its algorithm (oracle/) on all host cores"},
            "cpu_baseline": info,
            "e2e": {"value": rate, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------- GPU arm ---
def build_model(m, cfg):
    from roc_b200.model import build_gcn, build_sage_mean
    c = CONFIGS[cfg]
    if c["kind"] == "gcn":
        return build_gcn(m, c["layers"], DROPOUT, lr=LR, weight_decay=WD)
    return build_sage_mean(m, c["layers"], DROPOUT, lr=LR, weight_decay=WD)


def dump_outputs(outdir, m, hnd, perf, row_left):
    """--dump-outputs: the logits of the last timed forward pass (rank 0's rows; a fixed, seeded sample of
    DUMP_ROWS of them when there are more, with their global ids in logits_rows), its loss metrics (PerfMetrics
    order), and every weight and weight gradient after its update — fp32 / fp64, about 20 MB at most."""
    from roc_b200._lib import PerfMetrics
    os.makedirs(outdir, exist_ok=True)
    logits = m.get_tensor(hnd["logits"])
    rows = np.arange(logits.shape[0])
    if rows.shape[0] > DUMP_ROWS:
        rows = np.sort(np.random.RandomState(0).choice(rows.shape[0], DUMP_ROWS, replace=False))
    out = {"logits": logits[rows], "logits_rows": (row_left + rows).astype(np.float64),
           "metrics": np.array([perf[k] for k, _ in PerfMetrics._fields_], dtype=np.float64)}
    for p in range(m.num_parameters()):
        out["weight%d" % p] = m.get_parameter(p)
        out["weight%d_grad" % p] = m.get_parameter(p, "grad")
    for name, a in out.items():
        np.save(os.path.join(outdir, name + ".npy"), a)
    log("[bench] wrote %d arrays (%.1f MB) to %s" % (len(out), sum(a.nbytes for a in out.values()) / 1e6, outdir))


def parity_check(rank, local_rank, world, dist, dev):
    """N-rank engine vs 1-rank engine on a bounded graph (R-MAT scale 16, GCN 64-32-16-8 incl. the residual
    branch, dropout 0.5): stitched logits, loss and all-reduced dW of the first step at 1e-4 relative
    (+1e-5 * max|x| for cancellation).  Runs outside every timed region; every rank takes part."""
    import torch
    from roc_b200 import datasets
    from roc_b200.model import Host, Model, build_gcn
    layers = [64, 32, 16, 8]
    re_t, col_t = datasets.rmat_graph(16, 1 << 19, seed=7, device=dev)
    re_h, col_h = re_t.cpu().numpy().astype(np.uint64), col_t.cpu().numpy().astype(np.uint32)
    n = re_h.shape[0]
    feats, labels, mask = datasets.node_data(n, layers[0], layers[-1], seed=3)
    feats, labels, mask = feats.numpy(), labels.numpy(), mask.numpy().astype(np.int32)

    def run(host):
        host.graph_from_arrays(re_h, col_h)
        info = host.graph_info()
        rl, rr = info["rowLeft"], info["rowRight"]
        m = Model(host, seed=1)
        h = build_gcn(m, layers, 0.5, lr=LR, weight_decay=WD)
        m.set_tensor(h["input"], feats[rl:rr + 1])
        m.set_labels(h["label"], labels[rl:rr + 1])
        m.set_tensor(h["mask"], mask[rl:rr + 1])
        m.train_mode(); m.zero_gradients(); m.forward()
        logits = m.get_tensor(h["logits"])
        m.backward()
        perf = m.metrics()
        m.update()
        dw = [m.get_parameter(p, "grad") for p in range(m.num_parameters())]
        host.close()
        return rl, rr, logits, perf, dw

    host = Host(local_rank, rank, world)
    uid = [Host.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    host.nccl_init(uid[0])
    rl, rr, logits, perf, dw = run(host)
    gathered = [None] * world
    dist.all_gather_object(gathered, (rl, rr, logits, perf["trainLoss"], perf["trainAll"]))
    if rank != 0:
        return None
    _, _, logits1, perf1, dw1 = run(Host(local_rank, 0, 1))
    stitched = np.concatenate([g[2] for g in sorted(gathered, key=lambda g: g[0])])

    def rel_err(a, b):
        """max |a-b| / (|b| + 0.1 * max|b|): at most 1e-4 when a matches b to 1e-4 relative + 1e-5 * max|b| absolute."""
        a, b = a.astype(np.float64), b.astype(np.float64)
        return float((np.abs(a - b) / (np.abs(b) + 0.1 * np.abs(b).max() + 1e-30)).max())
    errs = {"logits": rel_err(stitched, logits1),
            "loss": abs(sum(g[3] for g in gathered) - perf1["trainLoss"]) / abs(perf1["trainLoss"]),
            "dW": max(rel_err(a, b) for a, b in zip(dw, dw1))}
    ok = (errs["logits"] <= 1e-4 and errs["loss"] <= 1e-4 and errs["dW"] <= 1e-4 and
          sum(g[4] for g in gathered) == perf1["trainAll"] and stitched.shape == logits1.shape)
    return {"ranks": world, "graph": "R-MAT scale-16 (N=%d, E=%d)" % (n, col_h.shape[0]), "model": "GCN 64-32-16-8 + residual, dropout 0.5",
            "max_rel_err": max(errs.values()), "errs": errs, "tolerance": 1e-4, "ok": bool(ok)}


def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from roc_b200 import _lib, datasets
    from roc_b200.model import Host, Model

    _lib.require_device()
    torch.cuda.set_device(local_rank)
    dev = "cuda:%d" % local_rank
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    cfg = CONFIGS[args.config]
    layers = cfg["layers"]

    parity = None
    if world > 1 and not args.no_parity:
        parity = parity_check(rank, local_rank, world, dist, dev)
        if rank == 0:
            log("[bench] parity_check: %s" % json.dumps(parity))

    re_h, col_h, glabel = make_graph(datasets, args.config, world, dev, args.scale)
    n, e = re_h.shape[0], col_h.shape[0]

    host = Host(local_rank, rank, world)
    if world > 1:
        uid = [Host.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        host.nccl_init(uid[0])
    host.graph_from_arrays(re_h, col_h)
    info = host.graph_info()
    rl, rr = info["rowLeft"], info["rowRight"]
    nloc = rr - rl + 1
    m = Model(host, seed=1)
    hnd = build_model(m, args.config)

    # synthetic node data: pinned host copies (e2e uploads them every step) of this rank's rows
    g = torch.Generator(device="cpu"); g.manual_seed(1000 + rank)
    feats = torch.empty((nloc, layers[0]), dtype=torch.float32, pin_memory=True)
    chunk = 1 << 18
    dg = torch.Generator(device=dev); dg.manual_seed(1000 + rank)
    for a in range(0, nloc, chunk):
        b = min(nloc, a + chunk)
        feats[a:b].copy_(torch.rand((b - a, layers[0]), device=dev, generator=dg) * 2 - 1)
    labels = torch.randint(0, layers[-1], (nloc,), generator=g, dtype=torch.int32).pin_memory()
    u = torch.rand(nloc, generator=g)
    mask = torch.full((nloc,), 2, dtype=torch.int32)
    mask[u < 0.76] = 1
    mask[u < 0.66] = 0
    mask = mask.pin_memory()
    torch.cuda.synchronize()

    def upload():
        m.set_tensor_from_host_ptr(hnd["input"], feats.data_ptr())
        m.set_labels(hnd["label"], labels.numpy())
        m.set_tensor_from_host_ptr(hnd["mask"], mask.data_ptr())
    upload()
    log("[bench] model built, inputs uploaded")
    h2d = feats.numel() * 4 + labels.numel() * 4 + mask.numel() * 4
    d2h = 28   # sizeof(PerfMetrics)

    stream = torch.cuda.ExternalStream(host.stream, device=dev)
    # configs whose working set fits in the 126 MB L2 (config 1) get an L2 flush between timed steps
    small = (nloc * (layers[0] + 2 * max(layers[1:])) * 4 + e * 4) < (256 << 20)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if small else None

    def barrier():
        host.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """K steps between one pair of events (the contract's number) and, separately, per-step events for
        median / best.  With an L2 flush between steps only the per-step events are meaningful."""
        barrier()
        per = []
        with torch.cuda.stream(stream):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            marks = [torch.cuda.Event(enable_timing=True) for _ in range(2 * steps)]
            e0.record(stream)
            for i in range(steps):
                if flush is not None:
                    flush.zero_()
                marks[2 * i].record(stream)
                fn()
                marks[2 * i + 1].record(stream)
            e1.record(stream)
        barrier()
        per = [marks[2 * i].elapsed_time(marks[2 * i + 1]) for i in range(steps)]
        ms = sum(per) if flush is not None else e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms] + per, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, per = float(t[0]), [float(v) for v in t[1:]]
        return ms, per

    # ---- resident-in-HBM arm
    for _ in range(max(args.warmup, 3)):
        m.train_epoch()
    host.synchronize()
    log("[bench] warm-up done")
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    m.profile_sg(True)
    l0 = _lib.lib.roc_launch_count()
    ms_total, per_step = timed(m.train_epoch, args.steps)
    launches = _lib.lib.roc_launch_count() - l0
    sg_times = m.profile_sg_read()
    m.profile_sg(False)
    clocks = sampler.stop() if rank == 0 else None
    perf = m.metrics()
    value = e * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:    # before the end-to-end arm trains further
        dump_outputs(args.dump_outputs, m, hnd, perf, rl)

    # ---- end-to-end arm: host buffers in, metrics out, every step
    def e2e_step():
        upload()
        m.train_epoch()
        m.metrics()
    e2e_steps = max(1, min(args.steps, 3))
    if args.no_e2e:
        ms_e2e, e2e_value = float("nan"), None
    else:
        e2e_step()
        ms_e2e, _ = timed(e2e_step, e2e_steps)
        e2e_value = e * e2e_steps / (ms_e2e * 1e-3)

    # ---- roofline of the dominant kernel: ScatterGather at the hidden width on this rank's partition
    eloc = info["colRight"] - info["colLeft"] + 1
    hsg = layers[1]
    sgh = [t for (h, t) in sg_times if h == hsg]   # (exchange entries carry negative widths)
    peak, peak_src = peaks()
    roof = None
    if sgh:
        t_avg = sum(sgh) / len(sgh)
        ach = sg_bytes(nloc, eloc, hsg) / (t_avg * 1e-3) / 1e9
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "sg_traffic.json")
        if os.path.exists(tp):
            try:
                tab = json.load(open(tp)).get("per_config", {})
                ent = tab.get("cfg%d_n%d" % (args.config, world))
                if ent:
                    traffic, traffic_src = ent["dram_bytes_per_launch"], ent.get("source")
            except Exception:
                traffic = None
        roof = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                "traffic_source": traffic_src,
                "kernel": "ScatterGather main kernel (+fix-up) H=%d" % hsg, "launch_ms": t_avg,
                "launch_ms_best": min(sgh), "launches_timed": len(sgh), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": sg_bytes(nloc, eloc, hsg),
                "compulsory_bytes_per_launch": sg_compulsory_bytes(nloc, eloc, hsg),
                "frac_compulsory": sg_compulsory_bytes(nloc, eloc, hsg) / (t_avg * 1e-3) / 1e9 / peak,
                # the algorithmic bytes are mostly neighbour-row gathers and most of those sectors hit in L2
                # (hub rows), so `frac` can exceed 1; this one uses the ncu DRAM traffic of this (config, N)
                "frac_dram": (traffic / (t_avg * 1e-3) / 1e9 / peak) if traffic else None}
    # negative widths are the part of the halo exchange the compute stream had to wait for (N > 1)
    exch_times = [(-h, t) for (h, t) in sg_times if h < 0]
    sg_times = [(h, t) for (h, t) in sg_times if h > 0]
    sg_share = sum(t for _, t in sg_times) / ms_total if sg_times else None
    exch_ms = sum(t for _, t in exch_times) / args.steps if exch_times else None

    # ---- side columns (rank 0, N = 1 only): CPU oracle + the reference's own kernel on this GPU
    cpu = None
    refk = None
    if rank == 0 and world == 1 and not args.no_cpu:
        if cfg["kind"] == "gcn":
            try:
                rate, best, _, cinfo = cpu_epoch_rate(3, 1, layers)
                cinfo["value"] = rate
                cinfo["best_value"] = best
                cinfo["unit"] = "edges/s"
                cpu = cinfo
            except Exception as ex:   # the oracle is a checker; its absence must not hide the GPU number
                cpu = {"error": repr(ex)}
        if hsg <= 512 and n * hsg < (1 << 31):
            try:
                refk = reference_kernel_column(re_h, col_h, dev, h=hsg)
            except Exception as ex:
                refk = {"error": repr(ex)}

    if rank == 0:
        per_sorted = sorted(per_step)
        line = {"metric": "gcn_training_edges_per_sec", "value": value, "unit": "edges/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps,
                "ms_per_step_median": per_sorted[len(per_sorted) // 2], "ms_per_step_best": per_sorted[0],
                "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": "%s, %s (N=%d, E=%d incl. self loops), dropout %.1f, Adam"
                                       % (cfg["desc"], glabel, n, e, DROPOUT),
                           "baseline_config": args.config,
                           "parallelism": "vertex-range dp%d" % world,
                           "l2": ("L2 flushed (256 MB write) before every timed step" if flush is not None else
                                  "inputs larger than L2 (features %.1f GB/GPU, graph %.2f GB)" %
                                  (nloc * round_up4(layers[0]) * 4 / 1e9, (e * 4 + n * 8) / 1e9))},
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "edges/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": ms_e2e / e2e_steps, "steps": e2e_steps},
                "gpu_launches": int(launches),
                "roofline": roof, "cpu_baseline": cpu,
                "sg_share_of_step": sg_share, "exposed_exchange_ms_per_step": exch_ms, "reference_kernel": refk,
                "train_loss": perf["trainLoss"], "plan": host.plan_info(), "parity_check": parity}
        print(json.dumps(line), flush=True)
    host.close()
    if world > 1:
        dist.destroy_process_group()


def round_up4(x):
    return (x + 3) // 4 * 4


def reference_kernel_column(row_end_h, col_h, dev, h=64, iters=5):
    """The reference's own aggre_coop_kernel (cut from scattergather_kernel.cu:20-76 into oracle/_ref) on
    the same graph and GPU, HBM-resident buffers, the reference's grid.  It omits the reference's
    per-call PCIe staging (types.cu:28, scattergather_kernel.cu:145-157): an upper bound for ROC."""
    import torch
    from oracle import ref
    if not ref.available():
        return {"unavailable": "oracle/_ref/libroc_ref.so not built"}
    n, e = row_end_h.shape[0], col_h.shape[0]
    d_re = torch.from_numpy(row_end_h.astype(np.int64)).to(dev)
    d_col = torch.from_numpy(col_h.astype(np.int32)).to(dev)
    rp, es = ref.edge_structs(d_col, d_re, 0, 0)
    x = torch.rand((n, h), device=dev) - 0.5
    out = torch.empty((n, h), device=dev)
    for _ in range(2):
        ref.scatter_gather(0, n - 1, 0, rp, es, x, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        ref.scatter_gather(0, n - 1, 0, rp, es, x, out=out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    return {"kernel": "aggre_coop_kernel (reference, sm_100a build)", "H": h, "launch_ms": ms,
            "algorithmic_GBps": sg_bytes(n, e, h) / (ms * 1e-3) / 1e9, "edges_per_s": e / (ms * 1e-3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json configs[n-1]")
    ap.add_argument("--scale", type=int, default=0, help="override the R-MAT scale (debug)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (profiling runs)")
    ap.add_argument("--no-parity", action="store_true", help="skip the N-rank vs 1-rank parity check (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus:
        log("[bench] WORLD_SIZE=%d but --gpus %d: launch with torch.distributed.run --nproc-per-node %d"
            % (world, args.gpus, args.gpus))
        if world == 1 and args.gpus > 1:
            sys.exit(2)
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
