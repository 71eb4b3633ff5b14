"""make_golden.py — mint golden vectors from the REFERENCE's own kernels.

The reference (jiazhihao/ROC) has no tests and no golden vectors (SURVEY §4), and
its full binary cannot be built (Legion absent).  Its CUDA kernels can: oracle/
Makefile cuts them out of the reference sources into oracle/_ref/libroc_ref.so.  This
script runs those kernels (plus the cuBLAS / cuDNN / cuRAND calls the reference
makes, same arguments) on a B200 over small seeded inputs and stores the graphs and
the outputs in tests/golden/ref_golden.npz.  The CPU oracle and the product kernels
are then both checked against this file.

The inputs are not stored: inputs() draws them from fixed seeds and the tests'
`golden` fixture regenerates them.  Outputs of more than a few thousand values are
stored at a fixed sample of rows (`<case>_rows`: the highest-degree rows plus a
seeded uniform draw), which keeps the file small.

Run on a GPU box (needs the prebuilt oracle/_ref/libroc_ref.so):
    python tests/golden/make_golden.py [outdir]       # default: tests/golden
"""
import os
import sys
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref  # noqa: E402
from roc_b200 import datasets  # noqa: E402

SEED = 20260921
N_A, N_B = 1000, 1 << 10          # uniform_graph(1000, ...), rmat_graph(10, ...)
SIDE_BY_SIDE_H = (16, 64, 128, 256)


def inputs():
    """Every seeded input of the cases below, drawn in one fixed order from one generator."""
    rng = np.random.RandomState(SEED)
    G = {}
    for H in (16, 41, 64):
        G["A_sg_in_%d" % H] = rng.rand(N_A, H).astype(np.float32) * 2 - 1
    G["B_sg_in_32"] = rng.rand(N_B, 32).astype(np.float32) * 2 - 1
    G["lin_X"] = rng.rand(200, 33).astype(np.float32) * 2 - 1
    G["lin_W"] = rng.rand(9, 33).astype(np.float32) * 2 - 1     # W_mem[o*in + i]
    G["lin_dY"] = rng.rand(200, 9).astype(np.float32) * 2 - 1
    G["act_x"] = rng.randn(64, 24).astype(np.float32)
    G["act_dy"] = rng.randn(64, 24).astype(np.float32)
    G["sm_logits"] = rng.randn(500, 7).astype(np.float32) * 2
    G["sm_labels"] = rng.randint(0, 7, size=500).astype(np.int32)
    G["sm_mask"] = rng.randint(0, 4, size=500).astype(np.int32)
    G["adam_w"] = rng.randn(1000).astype(np.float32)
    G["adam_g"] = rng.randn(3, 1000).astype(np.float32)
    G["adam_m"] = rng.randn(1000).astype(np.float32) * 0.1
    G["adam_v"] = np.abs(rng.randn(1000).astype(np.float32) * 0.1)
    return G


def side_by_side_graph():
    """R-MAT scale 14 with hub rows spanning many chunks: the graph of the side-by-side ScatterGather case."""
    re_t, col_t = datasets.rmat_graph(14, 150000, seed=8)
    return re_t.numpy().astype(np.uint64), col_t.numpy().astype(np.uint32)


def side_by_side_input(n, h):
    return np.random.RandomState(h).rand(n, h).astype(np.float32) - 0.5


def col_checksum(col):
    """crc32 of the edge sources: pins the generated graph the stored outputs belong to."""
    return zlib.crc32(np.ascontiguousarray(col, dtype=np.uint32).tobytes())


def degrees(row_end, first=0):
    return np.diff(row_end.astype(np.int64), prepend=np.int64(first))


def sample_rows(deg, k, seed):
    """k sorted row ids: the k // 4 rows of highest degree, the rest drawn uniformly with a fixed seed."""
    hubs = np.argsort(-deg, kind="stable")[:k // 4]
    rest = np.setdiff1d(np.arange(deg.shape[0]), hubs)
    pick = np.random.RandomState(seed).choice(rest, k - hubs.shape[0], replace=False)
    return np.sort(np.concatenate([hubs, pick])).astype(np.int64)


def main():
    outdir = sys.argv[1] if len(sys.argv) > 1 else os.path.dirname(os.path.abspath(__file__))
    os.makedirs(outdir, exist_ok=True)
    dev = "cuda"
    I = inputs()
    G = {}

    # ---- graph A: cfg-1 shaped (1 000 vertices, ~10 K edges), whole graph = one partition
    re_t, col_t = datasets.uniform_graph(N_A, 4500, seed=1)
    row_end = re_t.numpy().astype(np.uint64)
    col = col_t.numpy().astype(np.uint32)
    N = row_end.shape[0]
    G["A_row_end"], G["A_col"] = row_end, col
    d_rows = torch.from_numpy(row_end.astype(np.int64)).to(dev)
    d_cols = torch.from_numpy(col.astype(np.int32)).to(dev)
    rp, es = ref.edge_structs(d_cols, d_rows, 0, 0)
    G["A_rowptrs"] = rp.cpu().numpy().astype(np.uint64)
    G["A_edgestructs"] = es.cpu().numpy().astype(np.uint32)
    rows = G["A_rows"] = sample_rows(degrees(row_end), 200, 1)
    for H in (16, 41, 64):
        dx = torch.from_numpy(I["A_sg_in_%d" % H]).to(dev)
        G["A_sg_out_%d" % H] = ref.scatter_gather(0, N - 1, 0, rp, es, dx).cpu().numpy()[rows]
        G["A_norm_out_%d" % H] = ref.indegree_norm(0, N - 1, 0, rp, dx).cpu().numpy()[rows]

    # ---- graph A split in two partitions: pins rowLeft / colLeft conventions
    from oracle import oracle
    k, vb, eb = oracle.partition(row_end, 2)
    assert k == 2
    G["A_vb2"], G["A_eb2"] = vb, eb
    dx = torch.from_numpy(I["A_sg_in_16"]).to(dev)
    for c in range(2):
        rl, rr, cl, cr = int(vb[c, 0]), int(vb[c, 1]), int(eb[c, 0]), int(eb[c, 1])
        rows_c = d_rows[rl:rr + 1].contiguous()
        cols_c = d_cols[cl:cr + 1].contiguous()
        rp_c, es_c = ref.edge_structs(cols_c, rows_c, rl, cl)
        G["A_p%d_edgestructs" % c] = es_c.cpu().numpy().astype(np.uint32)
        prow = G["A_p%d_rows" % c] = sample_rows(degrees(row_end[rl:rr + 1], cl), 100, 2 + c)
        y = ref.scatter_gather(rl, rr, cl, rp_c, es_c, dx)
        G["A_p%d_sg_out_16" % c] = y.cpu().numpy()[prow]
        z = ref.indegree_norm(rl, rr, cl, rp_c, dx[rl:rr + 1].contiguous())
        G["A_p%d_norm_out_16" % c] = z.cpu().numpy()[prow]

    # ---- graph B: skewed (R-MAT scale 10) with hub rows
    re_t, col_t = datasets.rmat_graph(10, 8192, seed=3)
    row_end = re_t.numpy().astype(np.uint64)
    col = col_t.numpy().astype(np.uint32)
    N = row_end.shape[0]
    assert N == N_B
    G["B_row_end"], G["B_col"] = row_end, col
    d_rows = torch.from_numpy(row_end.astype(np.int64)).to(dev)
    d_cols = torch.from_numpy(col.astype(np.int32)).to(dev)
    rp, es = ref.edge_structs(d_cols, d_rows, 0, 0)
    rows = G["B_rows"] = sample_rows(degrees(row_end), 200, 4)
    y = ref.scatter_gather(0, N - 1, 0, rp, es, torch.from_numpy(I["B_sg_in_32"]).to(dev))
    G["B_sg_out_32"] = y.cpu().numpy()[rows]

    # ---- graph C: R-MAT scale 14 at the hidden widths of the product's ScatterGather variants
    row_end, col = side_by_side_graph()
    N = row_end.shape[0]
    G["C_col_crc32"] = np.array([col_checksum(col)], dtype=np.uint64)
    d_rows = torch.from_numpy(row_end.astype(np.int64)).to(dev)
    d_cols = torch.from_numpy(col.astype(np.int32)).to(dev)
    rp, es = ref.edge_structs(d_cols, d_rows, 0, 0)
    rows = G["C_rows"] = sample_rows(degrees(row_end), 64, 5)
    for H in SIDE_BY_SIDE_H:
        y = ref.scatter_gather(0, N - 1, 0, rp, es, torch.from_numpy(side_by_side_input(N, H)).to(dev))
        G["C_sg_out_%d" % H] = y.cpu().numpy()[rows]

    # ---- linear (cuBLAS sgemm with the reference's arguments)
    X, W, dY = I["lin_X"], I["lin_W"], I["lin_dY"]
    dX, dW_, dYt = torch.from_numpy(X).to(dev), torch.from_numpy(W).to(dev), torch.from_numpy(dY).to(dev)
    for relu in (0, 1):
        Y = ref.linear_fwd(dX, dW_, relu=bool(relu))
        G["lin_Y_relu%d" % relu] = Y.cpu().numpy()
        gw = torch.zeros_like(dW_)
        gx = torch.zeros_like(dX)
        gy = dYt.clone()
        ref.linear_bwd(dX, dW_, Y, gy, gw, gx, relu=bool(relu))
        torch.cuda.synchronize()
        G["lin_dW_relu%d" % relu], G["lin_dX_relu%d" % relu] = gw.cpu().numpy(), gx.cpu().numpy()
        G["lin_dY_after_relu%d" % relu] = gy.cpu().numpy()

    # ---- activations (cuDNN)
    a, gy = I["act_x"], I["act_dy"]
    da = torch.from_numpy(a).to(dev)
    for mode, nm in ((1, "relu"), (2, "sigmoid")):
        y = ref.activation_fwd(da, mode)
        G["act_%s_y" % nm] = y.cpu().numpy()
        dx0 = torch.full_like(da, 0.25)   # beta = 1: accumulates onto what is there
        ref.activation_bwd(da, y, torch.from_numpy(gy).to(dev), dx0, mode)
        torch.cuda.synchronize()
        G["act_%s_dx_acc" % nm] = dx0.cpu().numpy()

    # ---- softmax cross entropy backward + metrics
    logits, lab, mask = I["sm_logits"], I["sm_labels"], I["sm_mask"]
    oh = datasets.onehot(lab, logits.shape[1])
    g, perf = ref.softmax_xent_bwd(torch.from_numpy(logits).to(dev), torch.from_numpy(oh).to(dev),
                                   torch.from_numpy(mask).to(dev))
    G["sm_grad"] = g.cpu().numpy()
    G["sm_perf"] = np.array([perf["trainLoss"], perf["trainAll"], perf["testAll"], perf["valAll"],
                             perf["trainCorrect"], perf["testCorrect"], perf["valCorrect"]], dtype=np.float64)

    # ---- adam with 3 gradient replicas
    dw, dg, dm, dv = (torch.from_numpy(I[k].copy()).to(dev) for k in ("adam_w", "adam_g", "adam_m", "adam_v"))
    ref.adam_update(dw, dg, dm, dv, 0.01, 0.9, 0.999, 0.05, 1e-8)
    torch.cuda.synchronize()
    G["adam_w_out"], G["adam_m_out"], G["adam_v_out"] = dw.cpu().numpy(), dm.cpu().numpy(), dv.cpu().numpy()
    G["adam_gsum"] = dg[0].cpu().numpy()

    # ---- element add
    G["add_out"] = ref.add_fwd(torch.from_numpy(a).to(dev), torch.from_numpy(gy).to(dev)).cpu().numpy()

    # ---- Glorot init (cuRAND XORWOW seeded like initializer_kernel.cu:40-48)
    # glibc: srand(1); rand() -> 1804289383, 846930886 (gnn.cc:56 + initializer.cc:38)
    for seed, (i_dim, o_dim) in ((1804289383, (16, 16)), (846930886, (16, 5))):
        G["glorot_%d_%dx%d" % (seed, i_dim, o_dim)] = ref.glorot(i_dim, o_dim, seed).cpu().numpy()
    rows = G["glorot_602x64_rows"] = sample_rows(np.zeros(64), 16, 6)
    G["glorot_1804289383_602x64"] = ref.glorot(602, 64, 1804289383).cpu().numpy()[rows]

    path = os.path.join(outdir, "ref_golden.npz")
    np.savez_compressed(path, **G)
    print("wrote", path, "with", len(G), "arrays,", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
