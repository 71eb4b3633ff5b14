"""GPU suite, part 2: the host (Model / op-builder API over the C-ABI kernels)
against the oracle's GCN on the same graph, features, labels, masks and weights —
forward logits, every dW, and the weights after several Adam steps.  Covers
BASELINE.json configs[0] (1K-node / 10K-edge, 16 -> 16), the residual variant
(more than 3 layer dims), dropout with the shared Philox mask, fused vs unfused
schedules, the dataset file loaders and the stand-alone driver."""
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_close
from witness import torch_witness
from oracle import oracle
from roc_b200 import _lib, datasets
from roc_b200.model import Host, Model, build_gcn, build_sage_mean

pytestmark = pytest.mark.gpu


def make_case(n=1000, pairs=4500, layers=(16, 16, 5), seed=1):
    re_t, col_t = datasets.uniform_graph(n, pairs, seed=seed)
    row_end, col = re_t.numpy().astype(np.uint64), col_t.numpy().astype(np.uint32)
    feats, labels, mask = datasets.node_data(n, layers[0], layers[-1], seed=seed)
    return row_end, col, feats.numpy(), labels.numpy(), mask.numpy()


def run_product(row_end, col, feats, labels, mask, layers, dropout, epochs, fuse, lr=0.01, wd=0.05):
    host = Host(0, 0, 1)
    host.graph_from_arrays(row_end, col)
    m = Model(host, seed=1)
    m.set_fusion(fuse)
    h = build_gcn(m, list(layers), dropout, lr=lr, weight_decay=wd)
    m.set_tensor(h["input"], feats)
    m.set_labels(h["label"], labels)
    m.set_tensor(h["mask"], mask.astype(np.int32))
    w0 = [m.get_parameter(p) for p in range(m.num_parameters())]
    out = {"w0": w0, "perf": [], "logits": None, "dW": None, "relu_masks": []}
    for ep in range(epochs):
        m.train_mode()
        m.zero_gradients()
        m.forward()
        out["relu_masks"].append([m.get_tensor(t) > 0 for t in h["relu_outs"]])
        if ep == 0:
            out["logits"] = m.get_tensor(h["logits"])
        m.backward()
        if ep == 0:
            out["dW"] = [m.get_parameter(p, "grad") for p in range(m.num_parameters())]
        out["perf"].append(m.metrics())
        m.update()
    out["w"] = [m.get_parameter(p) for p in range(m.num_parameters())]
    m.infer_mode()
    m.forward()
    out["infer_perf"] = m.metrics()
    host.close()
    return out


def sync_relu_masks(o, masks):
    """ReLU at a pre-activation within rounding of 0 is ill-conditioned: the product (fp32 / 3xTF32 sums)
    and the oracle (fp64 sums) may legitimately disagree on its sign, which changes a whole dW row.  Masks
    may differ ONLY there (|pre| <= 1e-4 * max|pre|, the parity tolerance); where they do, the oracle's
    backward uses the product's mask so the gradients stay comparable."""
    recs = [r for r in o.saved if r["relu"]]
    assert len(recs) == len(masks)
    for rec, pm in zip(recs, masks):
        om = rec["a"] > 0
        diff = pm != om
        if diff.any():
            pre = rec["pre"]
            assert np.abs(pre[diff]).max() <= 1e-4 * np.abs(pre).max(), "relu masks differ away from zero"
            rec["a_override"] = pm.astype(np.float32)
    return int(sum((pm != (r["a"] > 0)).sum() for r, pm in zip(recs, masks)))


def run_oracle(row_end, col, feats, labels, mask, layers, dropout, epochs, w0, lr=0.01, wd=0.05, relu_masks=None):
    o = oracle.GcnOracle(row_end, col, layers, w0, lr=lr, weight_decay=wd, dropout=dropout)
    oh = datasets.onehot(labels, layers[-1])
    res = {"perf": [], "flips": 0}
    for ep in range(epochs):
        o.forward(feats, train=True)
        if relu_masks is not None:
            res["flips"] += sync_relu_masks(o, relu_masks[ep])
        if ep == 0:
            res["logits"] = o.logits.copy()
        o.backward(oh, mask)
        if ep == 0:
            res["dW"] = [d.copy() for d in o.dW]
        res["perf"].append(o.perf)
        o.update()
    res["w"] = o.W
    o.forward(feats, train=False)
    _, res["infer_perf"] = oracle.softmax_xent_bwd(o.logits, oh, mask)
    return res


@pytest.mark.parametrize("layers,dropout", [((16, 16, 5), 0.0), ((16, 16, 5), 0.5), ((24, 32, 16, 7), 0.0),
                                            ((24, 32, 16, 7), 0.3), ((602, 64, 41), 0.5)])
@pytest.mark.parametrize("fuse", [True, False])
def test_gcn_training_matches_oracle(layers, dropout, fuse):
    case = make_case(layers=layers)
    epochs = 4
    got = run_product(*case, layers, dropout, epochs, fuse)
    want = run_oracle(*case, layers, dropout, epochs, got["w0"], relu_masks=got["relu_masks"])
    assert want["flips"] <= 4, "too many relu sign disagreements: %d" % want["flips"]
    rel_close(got["logits"], want["logits"], what="logits epoch 0")
    for p, (a, b) in enumerate(zip(got["dW"], want["dW"])):
        rel_close(a, b, rtol=2e-4, what="dW[%d] epoch 0" % p)
    for ep in range(epochs):
        gp, wp = got["perf"][ep], want["perf"][ep]
        assert gp["trainAll"] == wp["trainAll"]
        assert abs(gp["trainLoss"] - wp["trainLoss"]) <= 2e-4 * abs(wp["trainLoss"]), (ep, gp, wp)
    for p, (a, b) in enumerate(zip(got["w"], want["w"])):
        # Adam's first steps are ~sign(g)*lr, so weights track within the gradient's tolerance
        rel_close(a, b, rtol=1e-3, atol_scale=1e-4, what="W[%d] after %d epochs" % (p, epochs))
    assert got["infer_perf"]["trainAll"] == want["infer_perf"]["trainAll"]
    assert got["infer_perf"]["testAll"] == want["infer_perf"]["testAll"]


def test_fused_and_unfused_schedules_agree_bitwise():
    case = make_case(layers=(16, 16, 5))
    a = run_product(*case, (16, 16, 5), 0.5, 3, True)
    b = run_product(*case, (16, 16, 5), 0.5, 3, False)
    assert np.array_equal(a["logits"], b["logits"])
    for x, y in zip(a["w"], b["w"]):
        assert np.array_equal(x, y)


def test_glorot_weights_match_reference_curand(golden):
    """std::srand(1) then one std::rand() per linear -> cuRAND XORWOW seeds 1804289383, 846930886
    (initializer.cc:38, initializer_kernel.cu:40-48); weights must match the reference's bit for bit."""
    case = make_case(layers=(16, 16, 5))
    got = run_product(*case, (16, 16, 5), 0.0, 1, True)
    assert np.array_equal(got["w0"][0], golden["glorot_1804289383_16x16"])
    assert np.array_equal(got["w0"][1], golden["glorot_846930886_16x5"])
    big = make_case(n=64, pairs=100, layers=(602, 64, 3))
    got = run_product(*big, (602, 64, 3), 0.0, 1, True)
    assert np.array_equal(got["w0"][0][golden["glorot_602x64_rows"]], golden["glorot_1804289383_602x64"])


def test_file_loaders_and_driver(tmp_path):
    layers = (16, 16, 5)
    row_end, col, feats, labels, mask = make_case(layers=layers)
    prefix = str(tmp_path / "tiny")
    datasets.write_dataset(prefix, row_end, col, feats, labels, mask)
    host = Host(0, 0, 1)
    host.graph_from_lux(prefix)
    info = host.graph_info()
    assert info["numNodes"] == 1000 and info["numEdges"] == col.shape[0] and info["rowRight"] == 999
    m = Model(host, seed=1)
    h = build_gcn(m, list(layers), 0.0)
    m.load_features(h["input"], prefix)
    m.load_labels(h["label"], prefix)
    m.load_train_mask(h["mask"], prefix)
    assert np.array_equal(m.get_tensor(h["input"]), feats)
    assert np.array_equal(m.get_tensor(h["mask"], dtype=np.int32)[:, 0], mask)
    m.train_epoch()
    perf_files = m.metrics()
    host.close()
    got = run_product(row_end, col, feats, labels, mask, layers, 0.0, 1, True)
    ref_perf = got["perf"][0]
    for k in perf_files:     # the loss is summed with float atomics across CTAs: equal up to rounding
        if k == "trainLoss":
            assert abs(perf_files[k] - ref_perf[k]) <= 1e-5 * abs(ref_perf[k])
        else:
            assert perf_files[k] == ref_perf[k]
    # CSV path: parse, then the .feats.bin cache must appear (load_task.cu:63-65)
    prefix2 = str(tmp_path / "csv")
    datasets.write_lux(prefix2, row_end, col)
    datasets.write_feats_csv(prefix2, feats)
    datasets.write_labels(prefix2, labels)
    datasets.write_mask(prefix2, mask)
    exe = os.path.join(ROOT, "roc_b200", "bin", "roc_gnn")
    p = subprocess.run([exe, "-ll:gpu", "1", "-file", prefix2, "-layers", "16-16-5", "-e", "6", "-lr", "0.01",
                        "-decay", "0.0001", "-dropout", "0.5"], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    assert os.path.exists(prefix2 + ".feats.bin")
    assert np.array_equal(np.fromfile(prefix2 + ".feats.bin", dtype=np.float32).reshape(feats.shape), feats)
    lines = [l for l in p.stderr.splitlines() if "[INFER]" in l]
    assert len(lines) == 2 and "train_accuracy" in lines[0]      # epochs 0 and 5 (gnn.cc:107-110)


def test_cfg5_shape_residual_wide_hidden_dense_graph():
    """BASELINE.json configs[4] at a reduced size: 4 layers + the residual branch (5 dims), hidden 256 (the TMA
    ring ScatterGather variant), dropout, on a graph whose every row is cut at chunk boundaries (mean degree
    ~150: carries + fix-up on every row)."""
    layers = (40, 256, 256, 256, 9)
    re_t, col_t = datasets.powerlaw_graph(600, 60000, seed=4)
    row_end, col = re_t.numpy().astype(np.uint64), col_t.numpy().astype(np.uint32)
    feats, labels, mask = datasets.node_data(600, layers[0], layers[-1], seed=2)
    case = (row_end, col, feats.numpy(), labels.numpy(), mask.numpy())
    epochs = 2
    got = run_product(*case, layers, 0.5, epochs, True)
    want = run_oracle(*case, layers, 0.5, epochs, got["w0"], relu_masks=got["relu_masks"])
    assert want["flips"] <= 8
    rel_close(got["logits"], want["logits"], what="logits epoch 0")
    for p, (a, b) in enumerate(zip(got["dW"], want["dW"])):
        rel_close(a, b, rtol=2e-4, what="dW[%d] epoch 0" % p)
    for ep in range(epochs):
        assert got["perf"][ep]["trainAll"] == want["perf"][ep]["trainAll"]
        assert abs(got["perf"][ep]["trainLoss"] - want["perf"][ep]["trainLoss"]) <= 2e-4 * abs(want["perf"][ep]["trainLoss"])


@pytest.mark.parametrize("kind,layers", [("gcn", (12, 16, 5)), ("gcn", (12, 24, 16, 5)), ("sage", (12, 24, 16, 5))])
def test_torch_autograd_fp64_witness(kind, layers):
    re_t, col_t = datasets.rmat_graph(8, 1500, seed=31)
    row_end, col = re_t.numpy().astype(np.uint64), col_t.numpy().astype(np.uint32)
    n = row_end.shape[0]
    feats, labels, mask = datasets.node_data(n, layers[0], layers[-1], seed=9)
    feats, labels, mask = feats.numpy(), labels.numpy(), mask.numpy()
    host = Host(0, 0, 1)
    host.graph_from_arrays(row_end, col)
    m = Model(host, seed=1)
    h = (build_gcn if kind == "gcn" else build_sage_mean)(m, list(layers), 0.0)
    m.set_tensor(h["input"], feats)
    m.set_labels(h["label"], labels)
    m.set_tensor(h["mask"], mask.astype(np.int32))
    w0 = [m.get_parameter(p) for p in range(m.num_parameters())]
    m.train_mode(); m.zero_gradients(); m.forward()
    logits = m.get_tensor(h["logits"])
    m.backward()
    dw = [m.get_parameter(p, "grad") for p in range(m.num_parameters())]
    host.close()
    wl, wdw = torch_witness(kind, row_end, col, feats, labels, mask, layers, w0)
    rel_close(logits, wl, what="%s logits vs torch fp64" % kind)
    for p, (a, b) in enumerate(zip(dw, wdw)):
        rel_close(a, b, rtol=2e-4, atol_scale=2e-5, what="%s dW[%d] vs torch autograd" % (kind, p))
    if kind == "gcn":   # and the oracle's hand-derived backward against the same witness
        o = oracle.GcnOracle(row_end, col, layers, w0, dropout=0.0)
        o.forward(feats, train=True)
        o.backward(datasets.onehot(labels, layers[-1]), mask)
        rel_close(o.logits, wl, what="oracle logits vs torch fp64")
        for p, (a, b) in enumerate(zip(o.dW, wdw)):
            rel_close(a, b, rtol=1e-4, atol_scale=2e-5, what="oracle dW[%d] vs torch autograd" % p)


def test_oracle_comparison_at_scale_20():
    """One oracle comparison at a realistic size: R-MAT scale 20 (1 M vertices, ~17 M edges, hub rows of degree
    > 40 000 that span hundreds of chunks) — ScatterGather with the fused epilogue, then one full training step of a
    GCN 64-32-16 (forward logits, every dW, loss) against the oracle's fp64-accumulating epoch on the host cores."""
    import torch
    from roc_b200 import kernels as K
    re_t, col_t = datasets.rmat_graph(20, 1 << 23, seed=1, device="cuda")
    row_end = re_t.cpu().numpy().astype(np.uint64)
    col = col_t.cpu().numpy().astype(np.uint32)
    n = row_end.shape[0]
    # --- the hot kernel
    x = np.random.RandomState(20).rand(n, 64).astype(np.float32) - 0.5
    plan = K.SgPlan(0, n - 1, 0, re_t, col_t)
    got = plan.forward(torch.from_numpy(x).cuda()).cpu().numpy()
    want = oracle.scatter_gather(0, n - 1, 0, row_end, col, x)
    rel_close(got, want, what="SG at scale 20")
    del plan
    # --- one training step through the Model API
    layers = (64, 32, 16)
    feats, labels, mask = datasets.node_data(n, layers[0], layers[-1], seed=4)
    case = (row_end, col, feats.numpy(), labels.numpy(), mask.numpy())
    got = run_product(*case, layers, 0.5, 1, True)
    want = run_oracle(*case, layers, 0.5, 1, got["w0"], relu_masks=got["relu_masks"])
    rel_close(got["logits"], want["logits"], what="logits at scale 20")
    for p, (a, b) in enumerate(zip(got["dW"], want["dW"])):
        rel_close(a, b, rtol=2e-4, what="dW[%d] at scale 20" % p)
    assert got["perf"][0]["trainAll"] == want["perf"][0]["trainAll"]
    assert abs(got["perf"][0]["trainLoss"] - want["perf"][0]["trainLoss"]) <= 2e-4 * abs(want["perf"][0]["trainLoss"])
