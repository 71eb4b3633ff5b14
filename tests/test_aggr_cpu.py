"""CPU suite: the fp64 / exact references of the mean, max and min aggregators that the GPU suite
(test_aggr_gpu.py, test_aggr_multigpu.py) holds the kernels to, checked here against per-row brute-force loops
(forward values and winner ids, with ties, NaN, +-inf and degree-0 rows) and against central finite differences
(the max / min backward on a tie-free graph)."""
import numpy as np
import pytest
import torch

NO_ARG = 0xFFFFFFFF


def ref_aggr(row_end, col, x, aggr, col_left=0, col_global=None):
    """MAX / MIN over each row's in-edges, exact: the first edge in CSR order wins among equal values, the first
    NaN wins over numbers, +-inf are ordinary.  Returns (values [rows][H] in x's dtype, winner ids [rows][H] uint32;
    degree-0 rows 0 / NO_ARG).  row_end: the rows' global END offsets, the first row starts at col_left; col: the
    sources (row indices of x); col_global: the ids recorded as winners (default col)."""
    row_end = np.asarray(row_end, dtype=np.int64)
    col = np.asarray(col, dtype=np.int64)
    gid = col if col_global is None else np.asarray(col_global, dtype=np.int64)
    n, h = row_end.shape[0], x.shape[1]
    out = np.zeros((n, h), dtype=x.dtype)
    arg = np.full((n, h), NO_ARG, dtype=np.uint32)
    s = col_left
    for r in range(n):
        t = int(row_end[r])
        if t > s:
            seg = x[col[s - col_left:t - col_left]]
            nan = np.isnan(seg)
            fill = -np.inf if aggr == "max" else np.inf
            vals = np.where(nan, fill, seg)
            k = np.argmax(vals, axis=0) if aggr == "max" else np.argmin(vals, axis=0)   # first occurrence
            k = np.where(nan.any(axis=0), np.argmax(nan, axis=0), k)
            out[r] = seg[k, np.arange(h)]
            arg[r] = gid[s - col_left + k]
        s = t
    return out, arg


def ref_arg_backward(row_end, col, gy, arg, row_left=0, col_left=0):
    """fp64: dIn[u][h] = sum over the edges (u <- v) of gy[v][h] where arg[v][h] == row_left + u."""
    row_end = np.asarray(row_end, dtype=np.int64)
    col = np.asarray(col, dtype=np.int64)
    n = row_end.shape[0]
    deg = np.diff(np.concatenate([[col_left], row_end]))
    dst = np.repeat(np.arange(n), deg)
    hit = arg[col].astype(np.int64) == (row_left + dst)[:, None]
    out = np.zeros((n, gy.shape[1]), dtype=np.float64)
    np.add.at(out, dst, np.where(hit, gy[col].astype(np.float64), 0.0))
    return out


def brute_aggr(row_end, col, x, aggr):
    """The rule written out one element at a time, in edge order."""
    n, h = len(row_end), x.shape[1]
    out = np.zeros((n, h), dtype=np.float32)
    arg = np.full((n, h), NO_ARG, dtype=np.uint32)
    s = 0
    for r in range(n):
        t = int(row_end[r])
        for j in range(h):
            best, win = None, NO_ARG
            for e in range(s, t):
                c = x[col[e], j]
                if best is None or (c > best if aggr == "max" else c < best) or (np.isnan(c) and not np.isnan(best)):
                    best, win = c, col[e]
            if best is not None:
                out[r, j], arg[r, j] = best, win
        s = t
    return out, arg


def awkward_case(seed):
    """Rows of degree 0, 1 and many; values from a small integer set (exact ties), relu'd (ties at 0), some
    +-inf and NaN."""
    rng = np.random.RandomState(seed)
    deg = rng.choice([0, 0, 1, 2, 5, 9, 70], size=60)
    row_end = np.cumsum(deg)
    col = rng.randint(0, 60, size=int(row_end[-1]))
    x = np.maximum(rng.randint(-3, 4, size=(60, 7)), 0).astype(np.float32)
    x[rng.rand(60, 7) < 0.05] = np.inf
    x[rng.rand(60, 7) < 0.05] = -np.inf
    x[rng.rand(60, 7) < 0.05] = np.nan
    return row_end, col, x


@pytest.mark.parametrize("aggr", ["max", "min"])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_reference_matches_brute_force(aggr, seed):
    row_end, col, x = awkward_case(seed)
    want, want_arg = brute_aggr(row_end, col, x, aggr)
    got, got_arg = ref_aggr(row_end, col, x, aggr)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert np.array_equal(got_arg, want_arg)
    assert (got_arg[np.diff(np.concatenate([[0], row_end])) == 0] == NO_ARG).all()


def test_reference_rows_slice_and_global_ids():
    row_end, col, x = awkward_case(4)
    full, full_arg = ref_aggr(row_end, col, x, "max")
    a, b = 10, 40                                    # rows [a, b) with their own edge slice
    cl = int(row_end[a - 1])
    part, part_arg = ref_aggr(row_end[a:b], col[cl:int(row_end[b - 1])], x, "max", col_left=cl,
                              col_global=col[cl:int(row_end[b - 1])] + 0)
    assert np.array_equal(part.view(np.uint32), full[a:b].view(np.uint32))
    assert np.array_equal(part_arg, full_arg[a:b])


@pytest.mark.parametrize("aggr", ["max", "min"])
def test_arg_backward_is_the_gradient(aggr):
    """On a symmetric, duplicate-free graph without ties, sum_v <dOut[v], aggr(x)[v]> has gradient
    ref_arg_backward(dOut, arg): central differences agree."""
    from roc_b200 import datasets
    re_t, col_t = datasets.uniform_graph(40, 120, seed=5)
    row_end, col = re_t.numpy(), col_t.numpy()
    rng = np.random.RandomState(6)
    x = rng.permutation(40 * 3).reshape(40, 3).astype(np.float64) / 7.0    # distinct values: no ties
    gy = rng.randn(40, 3)
    _, arg = ref_aggr(row_end, col, x, aggr)
    grad = ref_arg_backward(row_end, col, gy, arg)

    def f(z):
        v, _ = ref_aggr(row_end, col, z, aggr)
        return float((v.astype(np.float64) * gy).sum())
    eps = 1e-3
    num = np.zeros_like(x)
    for i in range(x.shape[0]):
        for j in range(x.shape[1]):
            zp, zm = x.copy(), x.copy()
            zp[i, j] += eps
            zm[i, j] -= eps
            num[i, j] = (f(zp) - f(zm)) / (2 * eps)
    np.testing.assert_allclose(grad, num, rtol=1e-4, atol=1e-4)


def sage_witness(row_end, col, feats, labels, mask, layers, weights, aggr, args=None):
    """GraphSAGE (build_sage's wiring) in torch fp64 + autograd: logits, dL/dW and, for max / min, the witness's
    own fp64 winner ids per layer.  `args` (one [N][H] uint32 array per layer) routes max / min through an explicit
    gather at those winners, so the gradient goes where the product sends it (torch's amax would split ties)."""
    n = row_end.shape[0]
    deg = np.diff(np.concatenate([[0], row_end.astype(np.int64)]))
    dst = torch.from_numpy(np.repeat(np.arange(n), deg))
    src = torch.from_numpy(col.astype(np.int64))
    ws = [torch.from_numpy(w.astype(np.float64)).requires_grad_(True) for w in weights]
    t = torch.from_numpy(feats.astype(np.float64))
    L = len(layers) - 1
    own_args, pre = [], []
    for i in range(1, L + 1):
        hw = t @ ws[2 * i - 2].T
        if aggr == "mean":
            s = torch.zeros_like(hw).index_add(0, dst, hw[src])
            nb = s / torch.from_numpy(np.maximum(deg, 1).astype(np.float64)).unsqueeze(1)
        else:
            hv = hw.detach().numpy()
            _, own = ref_aggr(row_end, col, hv, aggr)
            own_args.append(own)
            pre.append(hv)
            a = own if args is None else args[i - 1]
            valid = torch.from_numpy(a != NO_ARG)
            idx = torch.from_numpy(np.where(a == NO_ARG, 0, a).astype(np.int64))
            nb = torch.where(valid, torch.gather(hw, 0, idx), torch.zeros_like(hw))
        z = nb + t @ ws[2 * i - 1].T
        t = torch.relu(z) if i != L else z
    logits = t
    train = torch.from_numpy(mask == 0)
    loss = torch.nn.functional.cross_entropy(logits[train], torch.from_numpy(labels.astype(np.int64))[train],
                                             reduction="sum")
    loss.backward()
    return logits.detach().numpy(), [w.grad.numpy() for w in ws], own_args, pre


def assert_args_differ_only_at_near_ties(got_arg, own_arg, pre, tol=1e-4):
    """Where the product's winner differs from the fp64 witness's, the two candidates' fp64 values must be within
    rounding of each other (DESIGN §4's policy for ill-conditioned choices, as for the ReLU mask)."""
    diff = got_arg != own_arg
    if not diff.any():
        return 0
    r, c = np.nonzero(diff)
    assert (got_arg[diff] != NO_ARG).all() and (own_arg[diff] != NO_ARG).all()
    a = pre[got_arg[diff].astype(np.int64), c]
    b = pre[own_arg[diff].astype(np.int64), c]
    assert np.abs(a - b).max() <= tol * np.abs(pre).max(), "winners differ away from a tie"
    return int(diff.sum())


def test_sage_witness_mean_matches_composed_normalisation():
    """The mean witness equals the D^-1/2 D^-1/2 A composition of tests/witness.py's GraphSAGE-mean."""
    from roc_b200 import datasets
    from witness import torch_witness
    layers = (6, 8, 3)
    re_t, col_t = datasets.rmat_graph(6, 300, seed=3)
    row_end, col = re_t.numpy().astype(np.uint64), col_t.numpy().astype(np.uint32)
    n = row_end.shape[0]
    feats, labels, mask = (a.numpy() for a in datasets.node_data(n, layers[0], layers[-1], seed=2))
    rng = np.random.RandomState(1)
    w = [rng.randn(8, 6).astype(np.float32), rng.randn(8, 6).astype(np.float32),
         rng.randn(3, 8).astype(np.float32), rng.randn(3, 8).astype(np.float32)]
    l1, d1, _, _ = sage_witness(row_end, col, feats, labels, mask, layers, w, "mean")
    l2, d2 = torch_witness("sage", row_end, col, feats, labels, mask, layers, w)
    np.testing.assert_allclose(l1, l2, rtol=1e-10, atol=1e-10)
    for a, b in zip(d1, d2):
        np.testing.assert_allclose(a, b, rtol=1e-9, atol=1e-9)
