"""CPU suite: the fp64 reference of graph attention that the GPU suite (test_gat_gpu.py, test_gat_multigpu.py) holds
the kernels to, written in the kernels' own formulation — lse in a pass of its own, alpha recomputed from
(s_src, s_dst, lse), c = <dOut, out>, and the backward of row u gathered over u's own in-edges (which, on a
symmetric CSR, are the rows u feeds) — checked against torch fp64 autograd and against central finite differences."""
import numpy as np
import pytest
import torch


def leaky(z, slope):
    return np.where(z > 0, z, z * slope)


def dleaky(z, slope):
    return np.where(z > 0, 1.0, slope)


def csr_edges(row_end, col, col_left=0):
    """(dst, src): the local row and the source id of every edge, in CSR order."""
    row_end = np.asarray(row_end, dtype=np.int64)
    deg = np.diff(np.concatenate([[col_left], row_end]))
    return np.repeat(np.arange(row_end.shape[0]), deg), np.asarray(col, dtype=np.int64), deg


def ref_scores(h, att_w, heads):
    """s_src, s_dst [rows][K] in fp64; att_w: the [2][H] parameter."""
    h = np.asarray(h, dtype=np.float64)
    n, H = h.shape
    F = H // heads
    a = np.asarray(att_w, dtype=np.float64).reshape(2, heads, F)
    hs = h.reshape(n, heads, F)
    return (hs * a[0]).sum(-1), (hs * a[1]).sum(-1)


def ref_forward(row_end, col, h, s_src, s_dst, slope, col_left=0):
    """fp64: (out [nloc][H], lse [nloc][K]).  h, s_src, s_dst are indexed by col ids, their rows 0..nloc-1 being the
    own rows.  lse = max e + log sum exp(e - max e) per row and head; a degree-0 row has out = 0, lse = 0."""
    dst, src, deg = csr_edges(row_end, col, col_left)
    n, K = deg.shape[0], s_src.shape[1]
    h = np.asarray(h, dtype=np.float64)
    F = h.shape[1] // K
    e = leaky(s_src[src] + s_dst[dst], slope)
    m = np.full((n, K), -np.inf)
    np.maximum.at(m, dst, e)
    z = np.zeros((n, K))
    np.add.at(z, dst, np.exp(e - m[dst]))
    lse = np.where(deg[:, None] > 0, m + np.log(np.where(z > 0, z, 1.0)), 0.0)
    alpha = np.exp(e - lse[dst])
    out = np.zeros((n, K, F))
    np.add.at(out, dst, alpha[:, :, None] * h[src].reshape(-1, K, F))
    return out.reshape(n, K * F), lse


def ref_c(gy, out, heads):
    n, H = out.shape
    F = H // heads
    return (np.asarray(gy, np.float64).reshape(n, heads, F) * np.asarray(out, np.float64).reshape(n, heads, F)).sum(-1)


def ref_backward_gather(row_end, col, h, s_src, s_dst, lse, c, gy, slope, col_left=0):
    """The backward gather in the kernels' formulation: row u walks its in-edges v.  h, s_*, lse, c, gy are indexed
    by col ids (own rows first).  Returns (dh_agg [nloc][H], ds_src [nloc][K], ds_dst [nloc][K])."""
    u, v, deg = csr_edges(row_end, col, col_left)
    n, K = deg.shape[0], s_src.shape[1]
    h = np.asarray(h, np.float64)
    gy = np.asarray(gy, np.float64)
    F = h.shape[1] // K
    hh = h.reshape(-1, K, F)
    gg = gy.reshape(-1, K, F)
    z1 = s_src[u] + s_dst[v]
    a1 = np.exp(leaky(z1, slope) - lse[v])
    dz1 = a1 * ((gg[v] * hh[u]).sum(-1) - c[v]) * dleaky(z1, slope)
    z2 = s_src[v] + s_dst[u]
    a2 = np.exp(leaky(z2, slope) - lse[u])
    dz2 = a2 * ((gg[u] * hh[v]).sum(-1) - c[u]) * dleaky(z2, slope)
    dh = np.zeros((n, K, F))
    np.add.at(dh, u, a1[:, :, None] * gg[v])
    ds_src = np.zeros((n, K))
    np.add.at(ds_src, u, dz1)
    ds_dst = np.zeros((n, K))
    np.add.at(ds_dst, u, dz2)
    return dh.reshape(n, K * F), ds_src, ds_dst


def ref_finish(h_own, att_w, dh_agg, ds_src, ds_dst):
    """(dh, da [2][H]) from the gather's results on the own rows."""
    n, H = dh_agg.shape
    K = ds_src.shape[1]
    F = H // K
    a = np.asarray(att_w, np.float64).reshape(2, K, F)
    hh = np.asarray(h_own, np.float64).reshape(n, K, F)
    dh = dh_agg.reshape(n, K, F) + ds_src[:, :, None] * a[0] + ds_dst[:, :, None] * a[1]
    da = np.stack([(ds_src[:, :, None] * hh).sum(0).reshape(H), (ds_dst[:, :, None] * hh).sum(0).reshape(H)])
    return dh.reshape(n, H), da


def ref_gat(row_end, col, h, att_w, heads, slope, gy):
    """The whole layer on one partition: (out, lse, dh, da)."""
    s_src, s_dst = ref_scores(h, att_w, heads)
    out, lse = ref_forward(row_end, col, h, s_src, s_dst, slope)
    c = ref_c(gy, out, heads)
    dh_agg, ds_src, ds_dst = ref_backward_gather(row_end, col, h, s_src, s_dst, lse, c, gy, slope)
    dh, da = ref_finish(h, att_w, dh_agg, ds_src, ds_dst)
    return out, lse, dh, da


def torch_gat(row_end, col, h, att_w, heads, slope, gy):
    """torch fp64 autograd of the same layer (an independent derivation): (out, dh, da)."""
    dst, src, deg = csr_edges(row_end, col)
    n, H = h.shape
    K, F = heads, H // heads
    ht = torch.tensor(np.asarray(h, np.float64), requires_grad=True)
    at = torch.tensor(np.asarray(att_w, np.float64), requires_grad=True)
    dt, stt = torch.from_numpy(dst), torch.from_numpy(src)
    hs = ht.view(n, K, F)
    s_src = (hs * at[0].view(K, F)).sum(-1)
    s_dst = (hs * at[1].view(K, F)).sum(-1)
    e = torch.nn.functional.leaky_relu(s_src[stt] + s_dst[dt], slope)
    m = torch.full((n, K), -np.inf, dtype=torch.float64).scatter_reduce(0, dt[:, None].expand(-1, K), e.detach(),
                                                                        "amax")
    ex = torch.exp(e - m[dt])
    z = torch.zeros((n, K), dtype=torch.float64).index_add(0, dt, ex)
    alpha = ex / z[dt]
    out = torch.zeros((n, K, F), dtype=torch.float64).index_add(0, dt, alpha[:, :, None] * hs[stt]).view(n, H)
    (out * torch.from_numpy(np.asarray(gy, np.float64))).sum().backward()
    return out.detach().numpy(), ht.grad.numpy(), at.grad.numpy()


def symmetric_graph(n, m, seed, hub=True, isolated=(0,)):
    """Symmetric duplicate-free CSR with self-loops on every row but the isolated ones (degree 0) and, optionally,
    a hub (row 1) linked to most rows."""
    rng = np.random.RandomState(seed)
    pairs = set()
    keep = [r for r in range(n) if r not in isolated]
    for _ in range(m):
        a, b = rng.choice(keep, 2)
        pairs.add((a, b)); pairs.add((b, a))
    if hub:
        for r in keep[::2]:
            pairs.add((1, r)); pairs.add((r, 1))
    for r in keep:
        pairs.add((r, r))
    pairs = sorted(pairs)
    dst = np.array([p[0] for p in pairs], dtype=np.int64)
    src = np.array([p[1] for p in pairs], dtype=np.int64)
    row_end = np.cumsum(np.bincount(dst, minlength=n)).astype(np.uint64)
    return row_end, src.astype(np.uint32)


@pytest.mark.parametrize("heads", [1, 2, 4, 8])
@pytest.mark.parametrize("slope", [0.2, 0.0, 1.0])
@pytest.mark.parametrize("scale", [1.0, 1e3])
def test_reference_matches_torch_autograd(heads, slope, scale):
    row_end, col = symmetric_graph(60, 150, seed=heads)
    rng = np.random.RandomState(7)
    H = 5 if heads == 1 else 4 * heads
    h = rng.randn(60, H)
    att_w = rng.randn(2, H)
    s_src, s_dst = ref_scores(h, att_w, heads)
    att_w = att_w * (scale / max(np.abs(s_src).max(), np.abs(s_dst).max()))   # |e| up to ~scale
    gy = rng.randn(60, H)
    out, lse, dh, da = ref_gat(row_end, col, h, att_w, heads, slope, gy)
    assert np.isfinite(out).all() and np.isfinite(lse).all() and np.isfinite(dh).all() and np.isfinite(da).all()
    deg = np.diff(np.concatenate([[0], row_end.astype(np.int64)]))
    assert (out[deg == 0] == 0).all() and (lse[deg == 0] == 0).all()
    tout, tdh, tda = torch_gat(row_end, col, h, att_w, heads, slope, gy)
    np.testing.assert_allclose(out, tout, rtol=1e-9, atol=1e-9 * np.abs(tout).max())
    np.testing.assert_allclose(dh, tdh, rtol=1e-7, atol=1e-9 * np.abs(tdh).max())
    np.testing.assert_allclose(da, tda, rtol=1e-7, atol=1e-9 * np.abs(tda).max())


def test_lse_is_the_log_partition_function():
    row_end, col = symmetric_graph(30, 60, seed=3)
    rng = np.random.RandomState(2)
    h, att_w = rng.randn(30, 8), rng.randn(2, 8)
    s_src, s_dst = ref_scores(h, att_w, 2)
    _, lse = ref_forward(row_end, col, h, s_src, s_dst, 0.2)
    dst, src, deg = csr_edges(row_end, col)
    for v in range(30):
        if deg[v]:
            e = leaky(s_src[src[dst == v]] + s_dst[v], 0.2)
            np.testing.assert_allclose(lse[v], np.log(np.exp(e).sum(0)), rtol=1e-12)


@pytest.mark.parametrize("heads", [1, 2])
def test_backward_matches_finite_differences(heads):
    row_end, col = symmetric_graph(9, 14, seed=11, hub=False)
    rng = np.random.RandomState(12)
    H = 3 if heads == 1 else 8
    h = rng.randn(9, H)
    att_w = rng.randn(2, H)
    gy = rng.randn(9, H)
    _, _, dh, da = ref_gat(row_end, col, h, att_w, heads, 0.2, gy)

    def f(hh, aa):
        s_src, s_dst = ref_scores(hh, aa, heads)
        out, _ = ref_forward(row_end, col, hh, s_src, s_dst, 0.2)
        return float((out * gy).sum())
    eps = 1e-6
    num_h = np.zeros_like(h)
    for i in range(h.shape[0]):
        for j in range(H):
            p, m = h.copy(), h.copy()
            p[i, j] += eps
            m[i, j] -= eps
            num_h[i, j] = (f(p, att_w) - f(m, att_w)) / (2 * eps)
    num_a = np.zeros_like(att_w)
    for i in range(2):
        for j in range(H):
            p, m = att_w.copy(), att_w.copy()
            p[i, j] += eps
            m[i, j] -= eps
            num_a[i, j] = (f(h, p) - f(h, m)) / (2 * eps)
    np.testing.assert_allclose(dh, num_h, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(da[0], num_a[0], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(da[1], num_a[1], rtol=1e-5, atol=1e-6)
