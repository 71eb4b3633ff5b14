"""GPU suite: graph attention.  Kernels (scores, softmax statistics, weighted aggregate, backward gather, backward
finish) through the C ABI against the fp64 reference of test_gat_cpu.py in the kernels' own formulation, on graphs
with heavy rows and hubs (both fix-up kernels), zero-degree rows and a partition slice with remapped sources, at
every supported head count and widths up to 256 with padded and unpadded rows; two runs bitwise equal; unsupported
shapes refused.  Model: build_gat's logits and every dW against a torch fp64 autograd witness, fusion on / off
bitwise equal over Adam steps, inference mode."""
import numpy as np
import pytest
import torch

from conftest import rel_close
from roc_b200 import _lib, datasets
from roc_b200 import kernels as K
from roc_b200.model import Host, Model, build_gat
from test_gat_cpu import ref_backward_gather, ref_c, ref_finish, ref_forward, ref_scores
from test_aggr_gpu import graph, to_dev

pytestmark = pytest.mark.gpu
DEV = "cuda"
SHAPES = [(4, 1), (16, 1), (16, 2), (16, 4), (41, 1), (47, 1), (64, 1), (64, 2), (64, 4), (64, 8),
          (128, 1), (128, 2), (128, 4), (128, 8), (256, 1), (256, 2), (256, 4), (256, 8)]


def inputs(n, h, heads, seed):
    rng = np.random.RandomState(seed)
    x = rng.randn(n, h).astype(np.float32)
    att_w = (rng.randn(2, h) / np.sqrt(h // heads)).astype(np.float32)
    gy = rng.randn(n, h).astype(np.float32)
    return x, att_w, gy


def dev(a, pad):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return K.padded(a.shape[0], a.shape[1], DEV, fill=t) if pad else t


def run_layer(plan, nloc, x, att_w, gy, heads, slope, pad, bst_halo=None):
    """Every kernel once: returns dict of numpy results.  x / gy hold the plan's own rows first; bst_halo (lse | c of
    rows nloc..) stands in for what other partitions would send."""
    xd, gd = dev(x, pad), dev(gy, pad)
    aw = torch.from_numpy(att_w).to(DEV)
    att = K.gat_scores(xd, aw, heads)
    bst = K.padded(x.shape[0], 2 * heads, DEV)
    out, bst = plan.gat_forward(xd, att, heads, slope, bst=bst)
    K.gat_c(gd[:nloc], out, bst, heads)
    if bst_halo is not None:
        bst[nloc:].copy_(torch.from_numpy(bst_halo).to(DEV))
    dx, ds = plan.gat_backward(xd, att, bst, gd, heads, slope)
    dh_agg = dx.clone()
    da = K.gat_finish(xd[:nloc], aw, ds, dx, heads)
    torch.cuda.synchronize()
    return {"att": att.cpu().numpy(), "out": out.cpu().numpy(), "lse": bst[:nloc, :heads].cpu().numpy(),
            "c": bst[:nloc, heads:2 * heads].cpu().numpy(), "dh_agg": dh_agg.cpu().numpy(),
            "ds": ds[:, :2 * heads].cpu().numpy(), "dh": dx.cpu().numpy(), "da": da.cpu().numpy()}


def check_layer(got, row_end, col, x, att_w, gy, heads, slope, what, col_left=0, halo=None):
    nloc = got["out"].shape[0]
    s_src, s_dst = ref_scores(x, att_w, heads)
    rel_close(got["att"][:, :heads], s_src, what=what + " s_src")
    rel_close(got["att"][:, heads:2 * heads], s_dst, what=what + " s_dst")
    out, lse = ref_forward(row_end, col, x, s_src, s_dst, slope, col_left=col_left)
    rel_close(got["out"], out, what=what + " out")
    rel_close(got["lse"], lse, what=what + " lse")
    c = ref_c(gy[:nloc], out, heads)
    rel_close(got["c"], c, what=what + " c")
    lse_all, c_all = lse, c
    if halo is not None:
        lse_all, c_all = np.concatenate([lse, halo[0]]), np.concatenate([c, halo[1]])
    dh_agg, ds_src, ds_dst = ref_backward_gather(row_end, col, x, s_src, s_dst, lse_all, c_all, gy, slope,
                                                 col_left=col_left)
    rel_close(got["dh_agg"], dh_agg, what=what + " dh_agg")
    # one bar for both halves: at slope 1 the softmax cancels s_dst, and ds_dst is rounding noise around 0
    rel_close(got["ds"], np.concatenate([ds_src, ds_dst], axis=1), what=what + " ds")
    dh, da = ref_finish(x[:nloc], att_w, dh_agg, ds_src, ds_dst)
    rel_close(got["dh"], dh, what=what + " dh")
    rel_close(got["da"], da, rtol=2e-4, atol_scale=2e-5, what=what + " da")


@pytest.mark.parametrize("kind", ["uniform", "rmat14", "zerodeg"])
@pytest.mark.parametrize("h,heads", SHAPES)
def test_gat_kernels_match_reference(kind, h, heads):
    row_end, col = graph(kind)
    n = row_end.shape[0]
    d_re, d_col = to_dev(row_end, col)
    plan = K.SgPlan(0, n - 1, 0, d_re, d_col)
    x, att_w, gy = inputs(n, h, heads, h + heads)
    for pad in (True, False):
        got = run_layer(plan, n, x, att_w, gy, heads, 0.2, pad)
        check_layer(got, row_end, col, x, att_w, gy, heads, 0.2, "%s H=%d K=%d pad=%s" % (kind, h, heads, pad))
        if pad and kind == "rmat14":
            again = run_layer(plan, n, x, att_w, gy, heads, 0.2, pad)
            for k in got:
                assert np.array_equal(got[k].view(np.uint32), again[k].view(np.uint32)), "%s not bitwise repeatable" % k


@pytest.mark.parametrize("h,heads", [(41, 1), (64, 8), (128, 4)])
def test_gat_slice_with_remapped_sources(h, heads):
    """A partition's slice (rowLeft > 0, colLeft > 0) whose tensors are [own rows | halo rows], as in the multi-GPU
    engine; lse and c of the halo rows come from the whole-graph reference."""
    row_end, col = graph("rmat14")
    n = row_end.shape[0]
    x, att_w, gy = inputs(n, h, heads, 3)
    s_src, s_dst = ref_scores(x, att_w, heads)
    out_full, lse_full = ref_forward(row_end, col, x, s_src, s_dst, 0.2)
    c_full = ref_c(gy, out_full, heads)
    rl, rr = n // 3, 2 * n // 3
    cl, ce = int(row_end[rl - 1]), int(row_end[rr])
    sl_re, sl_col = row_end[rl:rr + 1], col[cl:ce].astype(np.int64)
    own = np.arange(rl, rr + 1)
    halo_ids = np.setdiff1d(np.unique(sl_col), own)
    ids = np.concatenate([own, halo_ids])
    remap = np.full(n, -1, dtype=np.int64)
    remap[ids] = np.arange(ids.shape[0])
    local = remap[sl_col]
    nloc = own.shape[0]
    bst_halo = np.zeros((halo_ids.shape[0], 2 * heads), dtype=np.float32)
    bst_halo[:, :heads] = lse_full[halo_ids]
    bst_halo[:, heads:2 * heads] = c_full[halo_ids]
    d_re = torch.from_numpy(sl_re.astype(np.int64)).to(DEV)
    d_loc = torch.from_numpy(local.astype(np.int32)).to(DEV)
    plan = K.SgPlan(rl, rr, cl, d_re, d_loc)
    xl, gl = np.ascontiguousarray(x[ids]), np.ascontiguousarray(gy[ids])
    got = run_layer(plan, nloc, xl, att_w, gl, heads, 0.2, True, bst_halo=bst_halo)
    check_layer(got, sl_re, local, xl, att_w, gl, heads, 0.2, "slice H=%d K=%d" % (h, heads), col_left=cl,
                halo=(bst_halo[:, :heads].astype(np.float64), bst_halo[:, heads:2 * heads].astype(np.float64)))
    rel_close(got["out"], out_full[rl:rr + 1], what="slice out vs whole graph")


@pytest.mark.parametrize("slope", [0.0, 1.0])
def test_gat_kernels_other_slopes(slope):
    row_end, col = graph("uniform")
    n = row_end.shape[0]
    d_re, d_col = to_dev(row_end, col)
    plan = K.SgPlan(0, n - 1, 0, d_re, d_col)
    x, att_w, gy = inputs(n, 64, 4, 1)
    got = run_layer(plan, n, x, att_w, gy, 4, slope, True)
    check_layer(got, row_end, col, x, att_w, gy, 4, slope, "slope=%g" % slope)


@pytest.mark.parametrize("h,heads", [(300, 1), (24, 8), (8, 4), (48, 3), (0, 1)])
def test_gat_unsupported_shapes_rejected(h, heads):
    assert _lib.lib.roc_gat_supported(h, heads) == _lib.ROC_ERR_UNSUPPORTED
    if h == 0:
        return
    row_end, col = graph("uniform")
    n = row_end.shape[0]
    d_re, d_col = to_dev(row_end, col)
    plan = K.SgPlan(0, n - 1, 0, d_re, d_col)
    x = K.padded(n, h, DEV)
    att = K.padded(n, 2 * heads, DEV)
    with pytest.raises(_lib.RocError):
        plan.gat_forward(x, att, heads)
    with pytest.raises(_lib.RocError):
        K.gat_scores(x, torch.zeros((2, h), device=DEV), heads)


# ------------------------------------------------------------------------------------------ model level ---
def gat_case(layers):
    re_t, col_t = datasets.rmat_graph(8, 1500, seed=31)
    row_end, col = re_t.numpy().astype(np.uint64), col_t.numpy().astype(np.uint32)
    feats, labels, mask = datasets.node_data(row_end.shape[0], layers[0], layers[-1], seed=9)
    return row_end, col, feats.numpy(), labels.numpy(), mask.numpy()


def gat_witness(row_end, col, feats, labels, mask, layers, heads, weights, slope=0.2):
    """build_gat's model in torch fp64 + autograd: logits and dL/dW for every parameter (W_1, att_1, W_2, ...)."""
    n = row_end.shape[0]
    deg = np.diff(np.concatenate([[0], row_end.astype(np.int64)]))
    dst = torch.from_numpy(np.repeat(np.arange(n), deg))
    src = torch.from_numpy(col.astype(np.int64))
    ws = [torch.from_numpy(w.astype(np.float64)).requires_grad_(True) for w in weights]
    t = torch.from_numpy(feats.astype(np.float64))
    L = len(layers) - 1
    for i in range(1, L + 1):
        k = heads if i != L else 1
        z = t @ ws[2 * i - 2].T
        a = ws[2 * i - 1]
        H = z.shape[1]
        F = H // k
        zs = z.view(n, k, F)
        s_src = (zs * a[0].view(k, F)).sum(-1)
        s_dst = (zs * a[1].view(k, F)).sum(-1)
        e = torch.nn.functional.leaky_relu(s_src[src] + s_dst[dst], slope)
        m = torch.full((n, k), -np.inf, dtype=torch.float64).scatter_reduce(0, dst[:, None].expand(-1, k),
                                                                            e.detach(), "amax")
        ex = torch.exp(e - m[dst])
        zz = torch.zeros((n, k), dtype=torch.float64).index_add(0, dst, ex)
        alpha = ex / zz[dst]
        out = torch.zeros((n, k, F), dtype=torch.float64).index_add(0, dst, alpha[:, :, None] * zs[src]).view(n, H)
        t = torch.relu(out) if i != L else out
    logits = t
    train = torch.from_numpy(mask == 0)
    loss = torch.nn.functional.cross_entropy(logits[train], torch.from_numpy(labels.astype(np.int64))[train],
                                             reduction="sum")
    loss.backward()
    return logits.detach().numpy(), [w.grad.numpy() for w in ws]


def run_gat(case, layers, heads, fuse=True, epochs=1, dropout=0.0):
    row_end, col, feats, labels, mask = case
    host = Host(0, 0, 1)
    host.graph_from_arrays(row_end, col)
    m = Model(host, seed=1)
    m.set_fusion(fuse)
    h = build_gat(m, list(layers), heads, dropout)
    m.set_tensor(h["input"], feats)
    m.set_labels(h["label"], labels)
    m.set_tensor(h["mask"], mask.astype(np.int32))
    out = {"w0": [m.get_parameter(p) for p in range(m.num_parameters())], "logits": [], "att_params": h["att_params"]}
    for ep in range(epochs):
        m.train_mode(); m.zero_gradients(); m.forward()
        out["logits"].append(m.get_tensor(h["logits"]))
        if ep == 0:
            out["lse"] = [m.gat_lse(t) for t in h["gat_outs"]]
        m.backward()
        if ep == 0:
            out["dW"] = [m.get_parameter(p, "grad") for p in range(m.num_parameters())]
        m.update()
    out["w"] = [m.get_parameter(p) for p in range(m.num_parameters())]
    m.infer_mode(); m.forward()
    out["infer_logits"] = m.get_tensor(h["logits"])
    out["infer_perf"] = m.metrics()
    host.close()
    return out


@pytest.mark.parametrize("layers,heads", [((12, 32, 5), 4), ((12, 64, 32, 5), 8), ((12, 41, 5), 1)])
def test_gat_matches_fp64_witness(layers, heads):
    case = gat_case(layers)
    got = run_gat(case, layers, heads)
    assert got["att_params"] == [2 * i + 1 for i in range(len(layers) - 1)]
    for p in got["att_params"]:
        assert got["w0"][p].shape == (2, got["w0"][p - 1].shape[0])
    wl, wdw = gat_witness(*case, layers, heads, got["w0"])
    rel_close(got["logits"][0], wl, what="gat logits vs torch fp64")
    for p, (a, b) in enumerate(zip(got["dW"], wdw)):
        rel_close(a, b, rtol=2e-4, atol_scale=2e-5, what="gat dW[%d] vs torch fp64" % p)
    assert all(np.isfinite(l).all() for l in got["lse"])


def test_gat_adam_steps_and_fusion_bitwise():
    """Three Adam steps with dropout on: set_fusion(False) gives bit-identical logits and weights, and the weights
    (the attention weights included) move."""
    layers, heads = (12, 32, 16, 5), 4
    case = gat_case(layers)
    a = run_gat(case, layers, heads, fuse=True, epochs=3, dropout=0.3)
    b = run_gat(case, layers, heads, fuse=False, epochs=3, dropout=0.3)
    for x, y in zip(a["logits"], b["logits"]):
        assert np.array_equal(x, y)
    for x, y in zip(a["w"], b["w"]):
        assert np.array_equal(x, y)
    for x, y in zip(a["w0"], a["w"]):
        assert not np.array_equal(x, y)


def test_gat_infer_mode():
    layers, heads = (12, 32, 5), 4
    case = gat_case(layers)
    got = run_gat(case, layers, heads)
    assert np.isfinite(got["infer_logits"]).all()
    assert got["infer_perf"]["trainAll"] > 0 and got["infer_perf"]["testAll"] > 0
