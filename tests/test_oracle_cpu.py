"""CPU suite, part 1: the oracle itself — against an independent dense numpy
restatement, against the golden vectors minted from the reference's own kernels,
and on the edge cases (empty rows, single vertex, skewed partitions)."""
import numpy as np
import pytest
import torch

from conftest import rel_close
from oracle import oracle
from roc_b200 import datasets


def dense_adj(row_end, col):
    n = row_end.shape[0]
    a = np.zeros((n, n), dtype=np.float64)
    s = 0
    for v in range(n):
        for e in range(s, int(row_end[v])):
            a[v, col[e]] += 1.0
        s = int(row_end[v])
    return a


@pytest.fixture(scope="module")
def small():
    re, col = datasets.uniform_graph(300, 1200, seed=5)
    return re.numpy().astype(np.uint64), col.numpy().astype(np.uint32)


def test_generated_graph_is_symmetric_with_self_loops(small):
    re, col = small
    a = dense_adj(re, col)
    assert (a == a.T).all() and (np.diag(a) == 1).all() and a.max() == 1
    assert int(re[-1]) == col.shape[0]
    # sorted by (dst, src)
    s = 0
    for v in range(re.shape[0]):
        seg = col[s:int(re[v])]
        assert (np.diff(seg.astype(np.int64)) > 0).all()
        s = int(re[v])


@pytest.mark.parametrize("h", [1, 16, 41])
def test_sg_matches_dense(small, h):
    re, col = small
    x = np.random.RandomState(0).randn(re.shape[0], h).astype(np.float32)
    want = dense_adj(re, col) @ x.astype(np.float64)
    rel_close(oracle.scatter_gather(0, re.shape[0] - 1, 0, re, col, x, acc64=True), want, what="sg64")
    rel_close(oracle.scatter_gather(0, re.shape[0] - 1, 0, re, col, x, acc64=False), want, what="sg32")


def test_sg_partition_slices_concatenate(small):
    re, col = small
    x = np.random.RandomState(1).randn(re.shape[0], 8).astype(np.float32)
    full = oracle.scatter_gather(0, re.shape[0] - 1, 0, re, col, x)
    for parts in (2, 3, 5):
        k, vb, eb = oracle.partition(re, parts)
        assert k == parts
        outs = []
        for c in range(parts):
            rl, rr, cl, cr = int(vb[c, 0]), int(vb[c, 1]), int(eb[c, 0]), int(eb[c, 1])
            outs.append(oracle.scatter_gather(rl, rr, cl, re[rl:rr + 1], col[cl:cr + 1], x))
        assert np.array_equal(np.concatenate(outs), full)


def test_partition_properties(small):
    re, _ = small
    n, e = re.shape[0], int(re[-1])
    for parts in (1, 2, 4, 7):
        k, vb, eb = oracle.partition(re, parts)
        assert k == parts
        assert vb[0, 0] == 0 and vb[-1, 1] == n - 1
        assert (vb[1:, 0] == vb[:-1, 1] + 1).all()          # contiguous, disjoint, complete
        assert eb[0, 0] == 0 and eb[-1, 1] == e - 1
        assert (eb[1:, 0] == eb[:-1, 1] + 1).all()
        cap = (e + parts - 1) // parts
        deg = np.diff(np.concatenate([[0], re.astype(np.int64)]))
        for c in range(parts - 1):      # every closed range holds > cap edges, but not without its last vertex
            cnt = deg[vb[c, 0]:vb[c, 1] + 1].sum()
            assert cnt > cap and cnt - deg[vb[c, 1]] <= cap


def test_partition_can_produce_fewer_ranges_than_parts():
    # quirk Q16: strict '>' + greedy can leave fewer than P ranges (the reference then asserts)
    re = np.cumsum(np.array([10, 1, 1, 1], dtype=np.uint64))
    k, vb, _ = oracle.partition(re, 4)
    assert k < 4


def test_empty_rows_and_norm():
    # vertex 1 and 3 have no in-edges: SG gives 0, norm divides by sqrt(0) -> inf/nan like the reference (Q5)
    re = np.array([2, 2, 3, 3], dtype=np.uint64)
    col = np.array([0, 2, 1], dtype=np.uint32)
    x = np.arange(8, dtype=np.float32).reshape(4, 2) + 1
    y = oracle.scatter_gather(0, 3, 0, re, col, x)
    assert np.array_equal(y, np.array([[1 + 5, 2 + 6], [0, 0], [3, 4], [0, 0]], dtype=np.float32))
    with np.errstate(divide="ignore", invalid="ignore"):
        z = oracle.indegree_norm(0, 3, 0, re, x)
    assert np.isinf(z[1]).all() and np.allclose(z[0], x[0] / np.sqrt(np.float32(2)))


def test_linear_and_grads_match_numpy():
    r = np.random.RandomState(2)
    x, w, dy = r.randn(50, 13).astype(np.float32), r.randn(5, 13).astype(np.float32), r.randn(50, 5).astype(np.float32)
    y = oracle.linear_fwd(x, w)
    rel_close(y, x.astype(np.float64) @ w.T.astype(np.float64), what="fwd")
    dw = np.ones_like(w)
    dx = oracle.linear_bwd(x, w, None, dy.copy(), dw)
    rel_close(dw, 1.0 + dy.T.astype(np.float64) @ x, what="dW accumulates")
    rel_close(dx, dy.astype(np.float64) @ w, what="dX")
    yr = oracle.linear_fwd(x, w, relu=True)
    assert (yr >= 0).all() and np.array_equal(yr > 0, y > 0)


def test_philox_known_answers():
    """Philox4x32-10 against Random123's kat_vectors (Salmon et al., SC'11) — pins the dropout generator."""
    kat = [([0, 0, 0, 0], [0, 0], "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
           ([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
           ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0],
            "d16cfe09 94fdcceb 5001e420 24126ea1")]
    for ctr, key, want in kat:
        assert " ".join("%08x" % v for v in oracle.philox4x32_10(ctr, key)) == want


def test_dropout_mask_is_a_pure_function_of_row_and_column():
    a = oracle.dropout_mask(0, 512, 41, 0.5, 7, 3)
    b = oracle.dropout_mask(100, 12, 41, 0.5, 7, 3)
    assert np.array_equal(a[100:112], b)                       # depends on the global row only
    wide = oracle.dropout_mask(0, 512, 64, 0.5, 7, 3)
    assert np.array_equal(wide[:, :41], a)                     # ... and on the column, not on the width
    assert 0.45 < a.mean() < 0.55
    assert oracle.dropout_mask(0, 8, 8, 0.0, 1, 1).all()
    assert not np.array_equal(a, oracle.dropout_mask(0, 512, 41, 0.5, 7, 4))
    # the definition, spelled out: lane (c & 7) of block (row, c >> 3), 16 bits, >= round(rate * 65536)
    r, c, rate, seed, step = 77, 29, 0.3, (9 << 32) | 5, 11
    o = oracle.philox4x32_10([r, 0, c >> 3, step], [seed & 0xFFFFFFFF, seed >> 32])
    lane = c & 7
    u16 = (int(o[lane >> 1]) >> (16 * (lane & 1))) & 0xFFFF
    assert oracle.dropout_mask(r, 1, 64, rate, seed, step)[0, c] == (u16 >= int(rate * 65536 + 0.5))


def test_softmax_metrics_hand_case():
    logits = np.array([[0.0, 0.0, 0.0], [5.0, 1.0, 0.0], [0.0, 1.0, 5.0], [1.0, 9.0, 1.0]], dtype=np.float32)
    lab = np.array([1, 0, 0, 1])
    mask = np.array([0, 0, 2, 1], dtype=np.int32)
    g, perf = oracle.softmax_xent_bwd(logits, datasets.onehot(lab, 3), mask)
    # row 0: all equal -> first index wins the argmax (softmax_kernel.cu:51-57) -> wrong (true = 1)
    assert perf["trainAll"] == 2 and perf["trainCorrect"] == 1
    assert perf["testAll"] == 1 and perf["testCorrect"] == 0 and perf["valAll"] == 1 and perf["valCorrect"] == 1
    p = np.exp(logits - logits.max(1, keepdims=True)); p /= p.sum(1, keepdims=True)
    assert abs(perf["trainLoss"] - ((1 - p[0, 1]) + (1 - p[1, 0]))) < 1e-6
    assert np.allclose(g[0], p[0] - [0, 1, 0], atol=1e-6) and (g[2] == 0).all() and (g[3] == 0).all()


def test_lux_roundtrip(tmp_path, small):
    re, col = small
    prefix = str(tmp_path / "g")
    datasets.write_lux(prefix, re, col)
    n, e, rows, cols = oracle.lux_read(prefix + ".add_self_edge.lux")
    assert n == re.shape[0] and e == col.shape[0] and np.array_equal(rows, re) and np.array_equal(cols, col)
    n2, e2, r2, c2 = datasets.read_lux(prefix)
    assert np.array_equal(r2, re) and np.array_equal(c2, col)


def test_gcn_oracle_loss_decreases(small):
    re, col = small
    n = re.shape[0]
    feats, labels, mask = datasets.node_data(n, 12, 4, seed=3)
    r = np.random.RandomState(4)
    layers = [12, 8, 4]
    ws = [(r.rand(layers[i + 1], layers[i]).astype(np.float32) * 2 - 1) * np.sqrt(6.0 / (layers[i] + layers[i + 1]))
          for i in range(2)]
    m = oracle.GcnOracle(re, col, layers, ws, lr=0.01, weight_decay=0.0, dropout=0.0)
    oh = datasets.onehot(labels.numpy(), 4)
    losses = [m.train_epoch(feats.numpy(), oh, mask.numpy())["trainLoss"] for _ in range(30)]
    assert losses[-1] < losses[0]


# ------------------------------------------------ golden vectors (reference kernels) ---
def test_oracle_vs_reference_kernels(golden):
    g = golden
    re, col = g["A_row_end"], g["A_col"]
    n = re.shape[0]
    rows = g["A_rows"]
    for h in (16, 41, 64):
        rel_close(oracle.scatter_gather(0, n - 1, 0, re, col, g["A_sg_in_%d" % h])[rows], g["A_sg_out_%d" % h],
                  what="aggre_coop_kernel H=%d" % h)
        got = oracle.indegree_norm(0, n - 1, 0, re, g["A_sg_in_%d" % h])[rows]
        assert np.array_equal(got, g["A_norm_out_%d" % h]), "norm_coop_kernel must match bit for bit"
    rp, es = oracle.build_csr(0, n - 1, 0, re, col)
    assert np.array_equal(rp, g["A_rowptrs"]) and np.array_equal(es, g["A_edgestructs"])
    k, vb, eb = oracle.partition(re, 2)
    assert np.array_equal(vb, g["A_vb2"]) and np.array_equal(eb, g["A_eb2"])
    for c in range(2):
        rl, rr, cl, cr = int(vb[c, 0]), int(vb[c, 1]), int(eb[c, 0]), int(eb[c, 1])
        prow = g["A_p%d_rows" % c]
        rel_close(oracle.scatter_gather(rl, rr, cl, re[rl:rr + 1], col[cl:cr + 1], g["A_sg_in_16"])[prow],
                  g["A_p%d_sg_out_16" % c], what="partition %d sg" % c)
        _, es_c = oracle.build_csr(rl, rr, cl, re[rl:rr + 1], col[cl:cr + 1])
        assert np.array_equal(es_c, g["A_p%d_edgestructs" % c])
        assert np.array_equal(oracle.indegree_norm(rl, rr, cl, re[rl:rr + 1], g["A_sg_in_16"][rl:rr + 1])[prow],
                              g["A_p%d_norm_out_16" % c])
    re, col = g["B_row_end"], g["B_col"]
    rel_close(oracle.scatter_gather(0, re.shape[0] - 1, 0, re, col, g["B_sg_in_32"])[g["B_rows"]], g["B_sg_out_32"],
              what="rmat sg")


def test_oracle_vs_reference_library_ops(golden):
    g = golden
    x, w, dy = g["lin_X"], g["lin_W"], g["lin_dY"]
    for relu in (0, 1):
        y = oracle.linear_fwd(x, w, relu=bool(relu))
        rel_close(y, g["lin_Y_relu%d" % relu], what="sgemm fwd")
        dw = np.zeros_like(w)
        gy = dy.copy()
        dx = oracle.linear_bwd(x, w, g["lin_Y_relu%d" % relu], gy, dw, relu=bool(relu))
        rel_close(dw, g["lin_dW_relu%d" % relu], what="sgemm dW")
        rel_close(dx, g["lin_dX_relu%d" % relu], what="sgemm dX")
        assert np.array_equal(gy, g["lin_dY_after_relu%d" % relu])
    for mode, nm in ((1, "relu"), (2, "sigmoid")):
        y = oracle.activation_fwd(g["act_x"], mode)
        rel_close(y, g["act_%s_y" % nm], rtol=1e-5, what=nm)
        dx = np.full_like(y, 0.25)
        oracle.activation_bwd(g["act_%s_y" % nm], g["act_dy"], mode, dx=dx)
        rel_close(dx, g["act_%s_dx_acc" % nm], what=nm + " bwd")
    grad, perf = oracle.softmax_xent_bwd(g["sm_logits"], datasets.onehot(g["sm_labels"], 7), g["sm_mask"])
    rel_close(grad, g["sm_grad"], what="softmax grad")
    ref = g["sm_perf"]
    assert abs(perf["trainLoss"] - ref[0]) <= 1e-4 * abs(ref[0])
    assert [perf[k] for k in ("trainAll", "testAll", "valAll", "trainCorrect", "testCorrect", "valCorrect")] == \
        [int(v) for v in ref[1:]]
    wv, m, v = g["adam_w"].copy(), g["adam_m"].copy(), g["adam_v"].copy()
    gr = g["adam_g"].copy()
    gs = gr[0] + gr[1]
    gs = gs + gr[2]                 # g0 += g1; g0 += g2 (optimizer_kernel.cu:90-94)
    assert np.array_equal(gs, g["adam_gsum"])
    oracle.adam_update(wv, gs, m, v, np.float32(0.01), np.float32(0.9), np.float32(0.999), np.float32(0.05),
                       np.float32(1e-8))
    rel_close(wv, g["adam_w_out"], rtol=1e-5, what="adam w")
    rel_close(m, g["adam_m_out"], rtol=1e-5, what="adam m")
    rel_close(v, g["adam_v_out"], rtol=1e-5, what="adam v")
    assert np.array_equal(g["act_x"] + g["act_dy"], g["add_out"])


@pytest.mark.parametrize("layers", [(12, 16, 5), (12, 24, 16, 5)])
def test_gcn_oracle_backward_against_torch_autograd(layers):
    """GcnOracle's forward and its hand-derived backward (oracle.py, mirroring Model::backward's op order and the
    first-writer rule) against torch fp64 autograd of the same composition — the goldens pin kernels, this pins
    the wiring (with and without the residual branch)."""
    import torch  # noqa: F401
    from witness import torch_witness
    from roc_b200 import datasets
    re_t, col_t = datasets.rmat_graph(8, 1500, seed=31)
    row_end, col = re_t.numpy().astype(np.uint64), col_t.numpy().astype(np.uint32)
    n = row_end.shape[0]
    feats, labels, mask = datasets.node_data(n, layers[0], layers[-1], seed=9)
    feats, labels, mask = feats.numpy(), labels.numpy(), mask.numpy()
    r = np.random.RandomState(3)
    dims = list(zip(layers[:-1], layers[1:]))
    if len(layers) > 3:
        dims = [d for d in dims for _ in (0, 1)]
    w0 = [(r.rand(o, i).astype(np.float32) * 2 - 1) * np.float32(np.sqrt(6.0 / (i + o))) for (i, o) in dims]
    o = oracle.GcnOracle(row_end, col, layers, w0, dropout=0.0)
    o.forward(feats, train=True)
    o.backward(datasets.onehot(labels, layers[-1]), mask)
    wl, wdw = torch_witness("gcn", row_end, col, feats, labels, mask, layers, w0)
    assert np.allclose(o.logits, wl, rtol=1e-4, atol=1e-5 * np.abs(wl).max())
    for a, b in zip(o.dW, wdw):
        assert np.allclose(a, b, rtol=1e-4, atol=2e-5 * np.abs(b).max())


@pytest.mark.parametrize("n,i,o", [(1000, 602, 64), (1000, 64, 41)])
def test_oracle_linear_against_reference_cublas_at_headline_shapes(n, i, o):
    """The oracle's Linear restatement against outputs of the reference's own cublasSgemm calls
    (linear_kernel.cu:76-80, 220-231) at BASELINE.json configs[1]'s two shapes — minted on a B200 by
    tests/golden/make_golden_linear.py (the small 200 x 33 . 9 case lives in ref_golden.npz)."""
    import os
    from conftest import golden_module
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_golden_linear.npz"))
    X, W, dY = golden_module("make_golden_linear").inputs(n, i, o)
    k = "%dx%dx%d" % (n, i, o)
    rows, wrows = g["rows_" + k], g["wrows_" + k]
    rel_close(oracle.linear_fwd(X, W)[rows], g["Y_" + k], what="oracle Y vs reference cublasSgemm")
    dw = np.zeros_like(W)
    dx = oracle.linear_bwd(X, W, None, dY.copy(), dw, need_dx=True)
    rel_close(dw[wrows], g["dW_" + k], what="oracle dW vs reference cublasSgemm")
    rel_close(dx[rows], g["dX_" + k], what="oracle dX vs reference cublasSgemm")
