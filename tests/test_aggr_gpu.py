"""GPU suite: the mean, max and min aggregators.  Kernels: MAX / MIN forward bit-identical (values and winner
ids) to the exact reference on graphs with heavy rows and hubs (both fix-up kernels), zero-degree rows, row
slices and remapped sources, at widths from 1 to 1100 floats with padded and unpadded rows; the MEAN epilogue
bit-identical to SUM followed by IEEE division in every ScatterGather variant; the arg backward against an fp64
scatter-add through the winners.  Model: GraphSAGE with each native aggregator against a torch fp64 witness."""
import numpy as np
import pytest
import torch

from conftest import rel_close
from roc_b200 import _lib, datasets
from roc_b200 import kernels as K
from roc_b200.model import Host, Model, build_sage, build_sage_mean
from test_aggr_cpu import NO_ARG, assert_args_differ_only_at_near_ties, ref_aggr, ref_arg_backward, sage_witness

pytestmark = pytest.mark.gpu
DEV = "cuda"
WIDTHS = [1, 3, 16, 41, 64, 128, 256, 602, 1100]


def graph(kind):
    if kind == "uniform":
        re, col = datasets.uniform_graph(1000, 4500, seed=1)
    elif kind == "rmat14":
        re, col = datasets.rmat_graph(14, 150000, seed=7)       # hubs spanning ~40 chunks: both fix-up kernels
    elif kind == "zerodeg":
        deg = np.zeros(500, dtype=np.int64)
        deg[5] = 3000; deg[10:300:7] = 1; deg[310:320] = 64; deg[320] = 65; deg[400:420] = 5
        re = torch.from_numpy(np.cumsum(deg))
        col = torch.from_numpy(np.random.RandomState(9).randint(0, 500, size=int(deg.sum())).astype(np.int32))
    else:
        raise KeyError(kind)
    return re.numpy().astype(np.uint64), col.numpy().astype(np.uint32)


def to_dev(row_end, col):
    return (torch.from_numpy(np.asarray(row_end).astype(np.int64)).to(DEV),
            torch.from_numpy(np.asarray(col).astype(np.int32)).to(DEV))


def tie_input(n, h, seed):
    """Exact ties (relu'd small integers), ordinary values, +-inf and NaN."""
    rng = np.random.RandomState(seed)
    x = np.maximum(rng.randint(-3, 4, size=(n, h)), 0).astype(np.float32)
    x[:, 1::2] = rng.randn(n, (h + 0) // 2).astype(np.float32)
    x[rng.rand(n, h) < 0.01] = np.inf
    x[rng.rand(n, h) < 0.01] = -np.inf
    x[rng.rand(n, h) < 0.01] = np.nan
    return x


def bits(t):
    a = t.cpu().numpy() if isinstance(t, torch.Tensor) else t
    return np.ascontiguousarray(a).view(np.uint32)


def check_aggr(plan, x, row_end, col, h, what, col_left=0, col_global=None, gids=None):
    for aggr in ("max", "min"):
        want, want_arg = ref_aggr(row_end, col, x, aggr, col_left=col_left, col_global=gids)
        xd = torch.from_numpy(x).to(DEV)
        cg = None if col_global is None else col_global
        xp = K.padded(x.shape[0], h, DEV, fill=xd)
        got, arg = plan.aggr_forward(xp, aggr, col_global=cg)                     # ld = round_up(h, 4)
        assert np.array_equal(bits(got), bits(want)), "%s %s padded values" % (what, aggr)
        assert np.array_equal(bits(arg), want_arg), "%s %s padded winners" % (what, aggr)
        nloc = want.shape[0]
        got2, arg2 = plan.aggr_forward(xd, aggr, col_global=cg, out=torch.empty((nloc, h), device=DEV),
                                       arg=torch.empty((nloc, h), device=DEV, dtype=torch.int32))   # ld = h
        assert np.array_equal(bits(got2), bits(want)), "%s %s dense values" % (what, aggr)
        assert np.array_equal(bits(arg2), want_arg), "%s %s dense winners" % (what, aggr)
        got3, none = plan.aggr_forward(xp, aggr, col_global=cg, want_arg=False)     # no winners stored
        assert none is None and np.array_equal(bits(got3), bits(want))


@pytest.mark.parametrize("kind", ["uniform", "rmat14", "zerodeg"])
@pytest.mark.parametrize("h", WIDTHS)
def test_max_min_forward_bit_exact(kind, h):
    row_end, col = graph(kind)
    n = row_end.shape[0]
    d_re, d_col = to_dev(row_end, col)
    plan = K.SgPlan(0, n - 1, 0, d_re, d_col)
    check_aggr(plan, tie_input(n, h, h), row_end, col, h, "%s H=%d" % (kind, h))


def test_rmat14_exercises_both_fixups():
    row_end, col = graph("rmat14")
    deg = np.diff(np.concatenate([[0], row_end.astype(np.int64)]))
    assert deg.max() > 33 * 64, "the largest row must span more than 32 chunks (the CTA-per-row fix-up)"
    assert ((deg > 64) & (deg < 30 * 64)).any(), "and some heavy rows for the per-worker fix-up"
    d_re, d_col = to_dev(row_end, col)
    assert K.SgPlan(0, row_end.shape[0] - 1, 0, d_re, d_col).info()["heavy_rows"] > 0


@pytest.mark.parametrize("h", [3, 64, 602])
def test_max_min_row_slice_with_remapped_sources(h):
    """A partition's slice (rowLeft > 0, colLeft > 0) whose plan indexes a compacted input ([own | halo] rows
    in the multi-GPU engine), with the canonical global ids passed as colGlobal."""
    row_end, col = graph("rmat14")
    n = row_end.shape[0]
    rl, rr = n // 3, 2 * n // 3
    cl, ce = int(row_end[rl - 1]), int(row_end[rr])
    sl_re, sl_col = row_end[rl:rr + 1], col[cl:ce]
    x = tie_input(n, h, 5)
    uniq, local = np.unique(sl_col, return_inverse=True)
    d_re = torch.from_numpy(sl_re.astype(np.int64)).to(DEV)
    d_loc = torch.from_numpy(local.astype(np.int32)).to(DEV)
    d_glob = torch.from_numpy(sl_col.astype(np.int32)).to(DEV)
    plan = K.SgPlan(rl, rr, cl, d_re, d_loc)
    check_aggr(plan, np.ascontiguousarray(x[uniq]), sl_re, local, h, "slice H=%d" % h, col_left=cl,
               col_global=d_glob, gids=sl_col)
    # the global-id plan on the whole input agrees
    plan2 = K.SgPlan(rl, rr, cl, d_re, d_glob)
    check_aggr(plan2, x, sl_re, sl_col, h, "slice global H=%d" % h, col_left=cl)


@pytest.mark.parametrize("kind", ["uniform", "rmat14", "zerodeg"])
@pytest.mark.parametrize("h", [4, 16, 41, 64, 128, 256, 602])
def test_mean_epilogue_is_sum_then_ieee_division(kind, h, monkeypatch):
    row_end, col = graph(kind)
    n = row_end.shape[0]
    d_re, d_col = to_dev(row_end, col)
    plan = K.SgPlan(0, n - 1, 0, d_re, d_col)
    x = np.random.RandomState(h).randn(n, h).astype(np.float32)
    xp = K.padded(n, h, DEV, fill=torch.from_numpy(x).to(DEV))
    deg = torch.from_numpy(np.diff(np.concatenate([[0], row_end.astype(np.int64)])).astype(np.float32)).to(DEV)
    monkeypatch.delenv("ROC_SG_VARIANT", raising=False)
    s = plan.forward(xp)
    want = torch.where(deg[:, None] > 0, s / deg[:, None], torch.zeros_like(s))
    got = plan.forward(xp, epilogue=_lib.SG_EPI_MEAN)
    assert np.array_equal(bits(got), bits(want))
    got_r = plan.forward(xp, epilogue=_lib.SG_EPI_MEAN | _lib.SG_EPI_RELU)
    assert torch.equal(got_r, torch.clamp_min(want, 0.0))
    for variant in ("a", "c", "t", "u", "r"):
        monkeypatch.setenv("ROC_SG_VARIANT", variant)
        for epi in (_lib.SG_EPI_MEAN, _lib.SG_EPI_MEAN | _lib.SG_EPI_RELU):
            g = plan.forward(xp, epilogue=epi)
            assert np.array_equal(bits(g), bits(got if epi == _lib.SG_EPI_MEAN else got_r)), (variant, epi)
    monkeypatch.delenv("ROC_SG_VARIANT", raising=False)
    with pytest.raises(_lib.RocError):
        plan.forward(xp, epilogue=_lib.SG_EPI_MEAN | _lib.SG_EPI_NORM)


@pytest.mark.parametrize("h", [1, 4, 41, 64, 602])
def test_indegree_div_is_ieee_division(h):
    row_end, col = graph("zerodeg")
    n = row_end.shape[0]
    rng = np.random.RandomState(h)
    x = (rng.randn(n, h) * np.exp2(rng.randint(-80, 80, size=(n, h)))).astype(np.float32)
    x[rng.rand(n, h) < 0.1] = 0.0
    x[rng.rand(n, h) < 0.05] = -0.0
    d_re, _ = to_dev(row_end, col)
    deg = torch.from_numpy(np.diff(np.concatenate([[0], row_end.astype(np.int64)])).astype(np.float32)).to(DEV)
    for xd in (torch.from_numpy(x).to(DEV), K.padded(n, h, DEV, fill=torch.from_numpy(x).to(DEV))):
        got = K.indegree_div(0, n - 1, 0, d_re, xd)
        want = torch.where(deg[:, None] > 0, xd / deg[:, None], torch.zeros_like(xd))
        assert np.array_equal(bits(got), bits(want))


@pytest.mark.parametrize("kind", ["uniform", "rmat14"])
@pytest.mark.parametrize("h", [1, 16, 41, 128, 602, 1100])
def test_arg_backward(kind, h):
    row_end, col = graph(kind)              # symmetric, duplicate-free CSRs (datasets._csr_from_pairs)
    n = row_end.shape[0]
    d_re, d_col = to_dev(row_end, col)
    plan = K.SgPlan(0, n - 1, 0, d_re, d_col)
    x = tie_input(n, h, 3)
    gy = np.random.RandomState(4).randn(n, h).astype(np.float32)
    for dense in (False, True):
        xd = torch.from_numpy(x).to(DEV)
        gd = torch.from_numpy(gy).to(DEV)
        if not dense:
            xd, gd = K.padded(n, h, DEV, fill=xd), K.padded(n, h, DEV, fill=gd)
            _, arg = plan.aggr_forward(xd, "max")
        else:
            _, arg = plan.aggr_forward(xd, "max", out=torch.empty((n, h), device=DEV),
                                       arg=torch.empty((n, h), device=DEV, dtype=torch.int32))
        got = plan.arg_backward(gd, arg)
        want = ref_arg_backward(row_end, col, gy, bits(arg))
        rel_close(got.cpu().numpy(), want, what="arg backward %s H=%d dense=%s" % (kind, h, dense))
        assert torch.equal(plan.arg_backward(gd, arg), got)          # deterministic
    # AVG backward: A (D^-1 dOut)
    deg = np.diff(np.concatenate([[0], row_end.astype(np.int64)])).astype(np.float64)
    gd = K.padded(n, h, DEV, fill=torch.from_numpy(gy).to(DEV))
    got = plan.forward(K.indegree_div(0, n - 1, 0, d_re, gd))
    scaled = gy.astype(np.float64) / deg[:, None]
    dst = np.repeat(np.arange(n), deg.astype(np.int64))
    want = np.zeros((n, h))
    np.add.at(want, dst, scaled[col.astype(np.int64)])
    rel_close(got.cpu().numpy(), want, what="mean backward %s H=%d" % (kind, h))


# ------------------------------------------------------------------------------------------ model level ---
def sage_case(layers):
    re_t, col_t = datasets.rmat_graph(8, 1500, seed=31)
    row_end, col = re_t.numpy().astype(np.uint64), col_t.numpy().astype(np.uint32)
    feats, labels, mask = datasets.node_data(row_end.shape[0], layers[0], layers[-1], seed=9)
    return row_end, col, feats.numpy(), labels.numpy(), mask.numpy()


def run_sage(case, layers, aggr, fuse=True, epochs=1, builder=None):
    row_end, col, feats, labels, mask = case
    host = Host(0, 0, 1)
    host.graph_from_arrays(row_end, col)
    m = Model(host, seed=1)
    m.set_fusion(fuse)
    h = builder(m, list(layers), 0.0) if builder else build_sage(m, list(layers), 0.0, aggr=aggr)
    m.set_tensor(h["input"], feats)
    m.set_labels(h["label"], labels)
    m.set_tensor(h["mask"], mask.astype(np.int32))
    out = {"w0": [m.get_parameter(p) for p in range(m.num_parameters())], "logits": [], "args": []}
    for ep in range(epochs):
        m.train_mode(); m.zero_gradients(); m.forward()
        out["logits"].append(m.get_tensor(h["logits"]))
        if aggr in ("max", "min") and not builder:
            out["args"].append([m.sg_arg(t) for t in h["sage_outs"]])
        m.backward()
        if ep == 0:
            out["dW"] = [m.get_parameter(p, "grad") for p in range(m.num_parameters())]
        m.update()
    out["w"] = [m.get_parameter(p) for p in range(m.num_parameters())]
    host.close()
    return out


@pytest.mark.parametrize("aggr", ["mean", "max", "min"])
def test_sage_matches_fp64_witness(aggr):
    layers = (12, 24, 16, 5)
    case = sage_case(layers)
    got = run_sage(case, layers, aggr)
    args = got["args"][0] if got["args"] else None
    if args is not None:
        _, _, own, pre = sage_witness(*case, layers, got["w0"], aggr)
        for g, o, p in zip(args, own, pre):
            assert_args_differ_only_at_near_ties(g, o, p)
    wl, wdw, _, _ = sage_witness(*case, layers, got["w0"], aggr, args=args)
    rel_close(got["logits"][0], wl, what="sage-%s logits vs torch fp64" % aggr)
    for p, (a, b) in enumerate(zip(got["dW"], wdw)):
        rel_close(a, b, rtol=2e-4, atol_scale=2e-5, what="sage-%s dW[%d] vs torch fp64" % (aggr, p))


@pytest.mark.parametrize("aggr", ["mean", "max"])
def test_fusion_leaves_native_aggregators_bitwise_unchanged(aggr):
    layers = (12, 24, 16, 5)
    case = sage_case(layers)
    a = run_sage(case, layers, aggr, fuse=True, epochs=3)
    b = run_sage(case, layers, aggr, fuse=False, epochs=3)
    for x, y in zip(a["logits"], b["logits"]):
        assert np.array_equal(x, y)
    for x, y in zip(a["w"], b["w"]):
        assert np.array_equal(x, y)


def test_native_mean_matches_composed_mean():
    layers = (12, 24, 16, 5)
    case = sage_case(layers)
    native = run_sage(case, layers, "mean")
    composed = run_sage(case, layers, "mean", builder=build_sage_mean)
    for a, b in zip(native["w0"], composed["w0"]):
        assert np.array_equal(a, b)                      # same Glorot draws: the linears are created in one order
    rel_close(native["logits"][0], composed["logits"][0], what="native vs composed mean")
