"""GPU suite, part 1: every C-ABI kernel against the oracle on the same seeded
inputs, against the golden vectors minted from the reference's kernels, and (when
oracle/_ref is present) against the reference kernels run side by side.
Bit-exact for indices / masks / partition bounds; 1e-4 relative for fp32 tensors."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from conftest import golden_module, rel_close
from oracle import oracle, ref
from roc_b200 import _lib, datasets
from roc_b200 import kernels as K

pytestmark = pytest.mark.gpu
DEV = "cuda"


def to_dev(row_end, col):
    return (torch.from_numpy(np.asarray(row_end).astype(np.int64)).to(DEV),
            torch.from_numpy(np.asarray(col).astype(np.int32)).to(DEV))


def graph(kind):
    if kind == "uniform":
        re, col = datasets.uniform_graph(1000, 4500, seed=1)
    elif kind == "rmat":
        re, col = datasets.rmat_graph(12, 40000, seed=3)           # hubs with degree >> 64
    elif kind == "dense":
        re, col = datasets.powerlaw_graph(600, 60000, seed=4)      # mean degree ~150: every row heavy
    elif kind == "ragged":
        # empty rows, a 1-edge graph tail, one 5000-edge row
        deg = np.zeros(400, dtype=np.int64)
        deg[3] = 5000; deg[10:200:7] = 1; deg[250] = 63; deg[251] = 64; deg[252] = 65; deg[399] = 2
        re = torch.from_numpy(np.cumsum(deg))
        col = torch.from_numpy(np.random.RandomState(9).randint(0, 400, size=int(deg.sum())).astype(np.int32))
    elif kind == "single":
        re, col = torch.tensor([1]), torch.tensor([0], dtype=torch.int32)
    else:
        raise KeyError(kind)
    return re.numpy().astype(np.uint64), col.numpy().astype(np.uint32)


@pytest.mark.parametrize("kind", ["uniform", "rmat", "dense", "ragged", "single"])
@pytest.mark.parametrize("h", [1, 4, 16, 41, 64, 100, 128, 256, 602])
def test_sg_planned_vs_oracle(kind, h):
    row_end, col = graph(kind)
    n = row_end.shape[0]
    x = np.random.RandomState(h).randn(n, h).astype(np.float32)
    want = oracle.scatter_gather(0, n - 1, 0, row_end, col, x)
    d_re, d_col = to_dev(row_end, col)
    plan = K.SgPlan(0, n - 1, 0, d_re, d_col)
    xp = K.padded(n, h, DEV, fill=torch.from_numpy(x).to(DEV))     # ld = round_up(h, 4): vector path
    got = plan.forward(xp)
    torch.cuda.synchronize()
    rel_close(got.cpu().numpy(), want, what="%s H=%d padded" % (kind, h))
    xd = torch.from_numpy(x).to(DEV)                              # dense ld = h: scalar path when h % 4
    got2 = plan.forward(xd, out=torch.empty((n, h), device=DEV))
    rel_close(got2.cpu().numpy(), want, what="%s H=%d dense" % (kind, h))
    # determinism: same plan, same input -> identical bits
    assert torch.equal(plan.forward(xp), got)


@pytest.mark.parametrize("kind", ["uniform", "rmat", "dense", "ragged", "single"])
@pytest.mark.parametrize("h", [4, 16, 41, 64, 100, 128, 200, 256, 602])
def test_sg_variants_are_bitwise_identical(kind, h, monkeypatch):
    """The register (A), cp.async (C), TMA gather4 / bulk-copy (T) and producer/consumer ring (R) kernels share
    the chunk plan and the per-row summation order, so they must agree bit for bit — with every ring shape of
    variant T, every CTA-range split of variant R and with the fused epilogue — and the TMA paths must meet
    the oracle exactly like the others."""
    row_end, col = graph(kind)
    n = row_end.shape[0]
    x = np.random.RandomState(h).randn(n, h).astype(np.float32)
    d_re, d_col = to_dev(row_end, col)
    plan = K.SgPlan(0, n - 1, 0, d_re, d_col)
    xp = K.padded(n, h, DEV, fill=torch.from_numpy(x).to(DEV))
    monkeypatch.setenv("ROC_SG_VARIANT", "a")
    base = plan.forward(xp).clone()
    base_e = plan.forward(xp, epilogue=_lib.SG_EPI_NORM | _lib.SG_EPI_RELU).clone()
    rel_close(base.cpu().numpy(), oracle.scatter_gather(0, n - 1, 0, row_end, col, x), what="A %s H=%d" % (kind, h))
    for variant, cfgs in (("c", [None]), ("r", [None, 1, 4]), ("t", [None, 1, 2, 3, 4, 5, 6]), ("u", [None, 1, 2, 3]),
                          ("b", [None, 1, 3])):
        monkeypatch.setenv("ROC_SG_VARIANT", variant)
        for cfg in cfgs:
            if cfg is None:
                monkeypatch.delenv("ROC_SG_TCFG", raising=False)
            else:
                monkeypatch.setenv("ROC_SG_TCFG", str(cfg))
            got = plan.forward(xp)
            got_e = plan.forward(xp, epilogue=_lib.SG_EPI_NORM | _lib.SG_EPI_RELU)
            torch.cuda.synchronize()
            assert torch.equal(got, base), "variant %s cfg %s differs from A (%s, H=%d)" % (variant, cfg, kind, h)
            # as bit patterns: rows of degree 0 are 0 / sqrt(0) = NaN under the norm epilogue (quirk Q5)
            assert torch.equal(got_e.contiguous().view(torch.int32), base_e.contiguous().view(torch.int32)), \
                "variant %s cfg %s epilogue differs (%s, H=%d)" % (variant, cfg, kind, h)
    monkeypatch.delenv("ROC_SG_TCFG", raising=False)
    monkeypatch.delenv("ROC_SG_VARIANT", raising=False)


@pytest.mark.parametrize("kind", ["uniform", "rmat", "dense"])
def test_sg_epilogues(kind):
    row_end, col = graph(kind)
    n, h = row_end.shape[0], 64
    x = np.random.RandomState(1).randn(n, h).astype(np.float32)
    d_re, d_col = to_dev(row_end, col)
    plan = K.SgPlan(0, n - 1, 0, d_re, d_col)
    xd = torch.from_numpy(x).to(DEV)
    raw = plan.forward(xd).cpu().numpy()
    normed = oracle.indegree_norm(0, n - 1, 0, row_end, raw)
    got = plan.forward(xd, epilogue=_lib.SG_EPI_NORM).cpu().numpy()
    assert np.array_equal(got, normed), "fused norm must equal norm applied to the kernel's own sum"
    got = plan.forward(xd, epilogue=_lib.SG_EPI_NORM | _lib.SG_EPI_RELU).cpu().numpy()
    assert np.array_equal(got, np.maximum(normed, 0))


def test_sg_partition_slices_and_planless_abi():
    row_end, col = graph("rmat")
    n, h = row_end.shape[0], 16
    x = np.random.RandomState(2).randn(n, h).astype(np.float32)
    xd = torch.from_numpy(x).to(DEV)
    for parts in (2, 4):
        k, vb, eb = oracle.partition(row_end, parts)
        assert k == parts
        for c in range(parts):
            rl, rr, cl, cr = int(vb[c, 0]), int(vb[c, 1]), int(eb[c, 0]), int(eb[c, 1])
            d_re, d_col = to_dev(row_end[rl:rr + 1], col[cl:cr + 1])
            want = oracle.scatter_gather(rl, rr, cl, row_end[rl:rr + 1], col[cl:cr + 1], x)
            got = K.sg_forward(rl, rr, cl, d_re, d_col, xd)
            rel_close(got.cpu().numpy(), want, what="planless part %d/%d" % (c, parts))
            got_b = K.sg_backward(rl, rr, cl, d_re, d_col, xd)
            assert torch.equal(got, got_b)          # forward and backward are the same op (Q1)


def test_sg_plan_info_counts():
    row_end, col = graph("ragged")
    d_re, d_col = to_dev(row_end, col)
    plan = K.SgPlan(0, row_end.shape[0] - 1, 0, d_re, d_col)
    info = plan.info()
    e = int(row_end[-1])
    assert info["chunks"] == e // 64 + 1
    deg = np.diff(np.concatenate([[0], row_end.astype(np.int64)]))
    assert info["heavy_rows"] == int((deg > 64).sum())


def test_sg_invalid_arguments():
    row_end, col = graph("uniform")
    d_re, d_col = to_dev(row_end, col)
    plan = K.SgPlan(0, row_end.shape[0] - 1, 0, d_re, d_col)
    x = torch.zeros((1000, 8), device=DEV)
    assert _lib.lib.roc_sg_forward_planned(plan.handle, 0, x.data_ptr(), 8, x.data_ptr(), 8, 0, None) == _lib.ROC_ERR_INVALID
    assert _lib.lib.roc_sg_forward_planned(plan.handle, 8, None, 8, x.data_ptr(), 8, 0, None) == _lib.ROC_ERR_INVALID
    assert _lib.lib.roc_sg_forward_planned(plan.handle, 8, x.data_ptr(), 4, x.data_ptr(), 8, 0, None) == _lib.ROC_ERR_INVALID


def test_sg_round_trip_properties_large():
    """Size-independent properties at a size the oracle would take too long on:
    linearity, A(1) = degree, and agreement with torch's own sparse matmul."""
    re, col = datasets.rmat_graph(18, 2_000_000, seed=5, device=DEV)
    n = re.shape[0]
    plan = K.SgPlan(0, n - 1, 0, re, col)
    h = 64
    g = torch.Generator(device=DEV); g.manual_seed(1)
    x = torch.rand((n, h), device=DEV, generator=g) - 0.5
    y = torch.rand((n, h), device=DEV, generator=g) - 0.5
    ax, ay, axy = plan.forward(x), plan.forward(y), plan.forward(x + 2 * y)
    assert torch.allclose(axy, ax + 2 * ay, rtol=1e-4, atol=1e-4)
    deg = torch.diff(re, prepend=torch.zeros(1, dtype=re.dtype, device=DEV)).to(torch.float32)
    ones = plan.forward(torch.ones((n, 4), device=DEV))
    assert torch.equal(ones[:, 0], deg)
    crow = torch.cat([torch.zeros(1, dtype=torch.int64, device=DEV), re])
    a = torch.sparse_csr_tensor(crow, col.to(torch.int64), torch.ones(col.shape[0], device=DEV), size=(n, n))
    want = a @ x
    assert torch.allclose(ax, want, rtol=1e-4, atol=1e-4)


class _DevArr:
    """int32 view of library-owned device memory through __cuda_array_interface__."""
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (int(ptr), False), "version": 2}


def _dev_view(ptr, n):
    if n == 0:
        return torch.zeros(0, dtype=torch.int32, device=DEV)
    return torch.as_tensor(_DevArr(ptr, n), device=DEV).clone()


def test_halo_structures_bit_exact():
    """roc_halo_*: sorted distinct remote sources, remapped col, row packing — against numpy."""
    row_end, col = graph("rmat")
    n = row_end.shape[0]
    k, vb, eb = oracle.partition(row_end, 4)
    x = np.random.RandomState(3).randn(n, 12).astype(np.float32)
    for c in range(4):
        rl, rr, cl, cr = int(vb[c, 0]), int(vb[c, 1]), int(eb[c, 0]), int(eb[c, 1])
        cs = col[cl:cr + 1]
        d_col = torch.from_numpy(cs.astype(np.int32)).to(DEV)
        h = C.c_void_p()
        assert _lib.lib.roc_halo_create(rl, rr, cs.shape[0], d_col.data_ptr(), None, C.byref(h)) == 0
        nh = _lib.lib.roc_halo_size(h)
        remote = np.unique(cs[(cs < rl) | (cs > rr)])
        assert nh == remote.shape[0]
        torch.cuda.synchronize()
        got_ids = _dev_view(_lib.lib.roc_halo_ids(h), nh)
        got_col = _dev_view(_lib.lib.roc_halo_col_local(h), cs.shape[0])
        assert np.array_equal(got_ids.cpu().numpy().astype(np.uint32), remote)
        nloc = rr - rl + 1
        want_col = np.where((cs >= rl) & (cs <= rr), cs.astype(np.int64) - rl, nloc + np.searchsorted(remote, cs))
        assert np.array_equal(got_col.cpu().numpy().astype(np.int64), want_col)
        # SpMM over [own rows | halo rows] with the remapped col == SpMM over the whole matrix with global ids
        buf = np.concatenate([x[rl:rr + 1], x[remote]])
        d_re = torch.from_numpy(row_end[rl:rr + 1].astype(np.int64)).to(DEV)
        plan = K.SgPlan(rl, rr, cl, d_re, got_col)
        got = plan.forward(torch.from_numpy(buf).to(DEV), out=torch.empty((nloc, 12), device=DEV))
        want = oracle.scatter_gather(rl, rr, cl, row_end[rl:rr + 1], cs, x)
        rel_close(got.cpu().numpy(), want, what="halo-indexed SG part %d" % c)
        # row packing
        rows = torch.from_numpy(np.random.RandomState(c).randint(0, nloc, size=777).astype(np.int32)).to(DEV)
        src = K.padded(nloc, 12, DEV, fill=torch.from_numpy(x[rl:rr + 1]).to(DEV))
        dst = K.padded(777, 12, DEV)
        assert _lib.lib.roc_pack_rows(777, 12, rows.data_ptr(), src.data_ptr(), src.stride(0), dst.data_ptr(),
                                      dst.stride(0), None) == 0
        assert np.array_equal(dst.cpu().numpy(), x[rl:rr + 1][rows.cpu().numpy()])
        _lib.lib.roc_halo_destroy(h)


def test_build_csr_bit_exact():
    row_end, col = graph("rmat")
    k, vb, eb = oracle.partition(row_end, 3)
    for c in range(3):
        rl, rr, cl, cr = int(vb[c, 0]), int(vb[c, 1]), int(eb[c, 0]), int(eb[c, 1])
        d_re, d_col = to_dev(row_end[rl:rr + 1], col[cl:cr + 1])
        rp, es, cs = K.build_csr(rl, rr, cl, d_re, d_col)
        wrp, wes = oracle.build_csr(rl, rr, cl, row_end[rl:rr + 1], col[cl:cr + 1])
        assert np.array_equal(rp.cpu().numpy().astype(np.uint64), wrp)
        assert np.array_equal(es.cpu().numpy().astype(np.uint32), wes)
        assert np.array_equal(cs.cpu().numpy().astype(np.uint32), col[cl:cr + 1])


@pytest.mark.parametrize("h", [1, 16, 41, 64])
def test_indegree_norm_bit_exact(h):
    row_end, col = graph("rmat")
    n = row_end.shape[0]
    x = np.random.RandomState(h).randn(n, h).astype(np.float32)
    k, vb, eb = oracle.partition(row_end, 2)
    for c in range(2):
        rl, rr, cl = int(vb[c, 0]), int(vb[c, 1]), int(eb[c, 0])
        d_re, _ = to_dev(row_end[rl:rr + 1], col[:1])
        want = oracle.indegree_norm(rl, rr, cl, row_end[rl:rr + 1], x[rl:rr + 1])
        for xin in (torch.from_numpy(x[rl:rr + 1]).to(DEV), K.padded(rr - rl + 1, h, DEV, fill=torch.from_numpy(x[rl:rr + 1]).to(DEV))):
            got = K.indegree_norm(rl, rr, cl, d_re, xin)
            assert np.array_equal(got.cpu().numpy(), want)
    # fused relu-mask backward
    y = np.random.RandomState(7).randn(n, h).astype(np.float32)
    d_re, _ = to_dev(row_end, col[:1])
    got = K.indegree_norm(0, n - 1, 0, d_re, torch.from_numpy(x).to(DEV), relu_mask_of=torch.from_numpy(y).to(DEV))
    want = oracle.indegree_norm(0, n - 1, 0, row_end, np.where(y > 0, x, 0).astype(np.float32))
    assert np.array_equal(got.cpu().numpy(), want)


def test_row_uniform_division_is_ieee():
    """The fused norm epilogues use a shared-reciprocal + FMA division; it must equal `x / sqrtf(deg)`
    for EVERY fp32 bit pattern x (all 2^32, incl. zeros, denormals, inf, nan) — checked for a spread of
    degrees (incl. ones whose sqrt has an all-ones mantissa neighbourhood) and a few raw divisors."""
    degs = [1, 2, 3, 5, 7, 16, 17, 63, 64, 65, 492, 1000, 4095, 4096, 97569, 16777215, 2 ** 31 - 1]
    divisors = [float(np.sqrt(np.float32(d))) for d in degs] + [0.0, 1e-30, 3e38, float("inf")]
    bad = torch.zeros(1, dtype=torch.int64, device=DEV)
    for d in divisors:
        rc = _lib.lib.roc_selftest_rowdiv(d, 0, 1 << 32, bad.data_ptr(), None)
        assert rc == 0
    torch.cuda.synchronize()
    assert int(bad[0]) == 0, "%d of %d quotients differ from div.rn" % (int(bad[0]), len(divisors) << 32)


def test_activation_add():
    r = np.random.RandomState(3)
    x, dy = r.randn(333, 41).astype(np.float32), r.randn(333, 41).astype(np.float32)
    for mode in (1, 2):
        y = K.activation_fwd(torch.from_numpy(x).to(DEV), mode)
        wy = oracle.activation_fwd(x, mode)
        rel_close(y.cpu().numpy(), wy, rtol=1e-6, what="act fwd")
        dx = K.activation_bwd(y, torch.from_numpy(dy).to(DEV), mode)
        rel_close(dx.cpu().numpy(), oracle.activation_bwd(y.cpu().numpy(), dy, mode), rtol=1e-6, what="act bwd")
        acc = torch.full_like(y, 0.5)
        K.activation_bwd(y, torch.from_numpy(dy).to(DEV), mode, dx=acc)
        rel_close(acc.cpu().numpy(), 0.5 + dx.cpu().numpy(), rtol=1e-6, what="act bwd accumulate")
    s = K.add_fwd(torch.from_numpy(x).to(DEV), torch.from_numpy(dy).to(DEV))
    assert np.array_equal(s.cpu().numpy(), x + dy)
    da, db = torch.zeros_like(s), torch.ones_like(s)
    K.add_bwd(s, da, False, db, True)
    assert torch.equal(da, s) and torch.equal(db, s + 1)


@pytest.mark.parametrize("h,rate", [(602, 0.5), (64, 0.5), (41, 0.1), (16, 0.0)])
def test_dropout_mask_bit_exact(h, rate):
    rows, first = 257, 1000
    x = np.random.RandomState(1).randn(rows, h).astype(np.float32)
    keep = oracle.dropout_mask(first, rows, h, rate, (5 << 32) | 3, 9)
    want = oracle.dropout_apply(x, keep, rate)
    for xin in (torch.from_numpy(x).to(DEV), K.padded(rows, h, DEV, fill=torch.from_numpy(x).to(DEV))):
        got = K.dropout_fwd(xin, first, rate, (5 << 32) | 3, 9)
        assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.parametrize("h,rate", [(602, 0.5), (64, 0.5), (41, 0.1), (33, 0.9), (128, 0.5)])
def test_dropout_packed_mask_bit_exact(h, rate):
    rows, first = 300, 12345
    keep = oracle.dropout_mask(first, rows, h, rate, (7 << 32) | 1, 4)
    m = K.dropout_mask(rows, h, first, rate, (7 << 32) | 1, 4, DEV).cpu().numpy().view(np.uint32)
    assert m.shape[1] % 4 == 0 and m.shape[1] * 32 >= h
    bits = ((m[:, :, None] >> np.arange(32, dtype=np.uint32)[None, None, :]) & 1).reshape(rows, -1)
    assert np.array_equal(bits[:, :h].astype(bool), keep.astype(bool))
    assert not bits[:, h:].any()          # pad bits / words are zero


@pytest.mark.parametrize("n,i,o", [(1000, 602, 64), (777, 64, 41), (4099, 200, 16), (129, 16, 16), (5, 3, 2)])
@pytest.mark.parametrize("rate", [0.5, 0.0])
def test_linear_with_fused_dropout_matches_unfused_bitwise(n, i, o, rate):
    """dropout applied inside the GEMM operand load == dropout kernel followed by the plain GEMM."""
    r = np.random.RandomState(n + i)
    first, seed, step = 77, (3 << 32) | 2, 6
    x = K.padded(n, i, DEV, fill=torch.from_numpy(r.randn(n, i).astype(np.float32)).to(DEV))
    w = torch.from_numpy((r.randn(o, i) * 0.1).astype(np.float32)).to(DEV)
    dy = torch.from_numpy(r.randn(n, o).astype(np.float32)).to(DEV)
    mask = K.dropout_mask(n, i, first, rate, seed, step, DEV) if rate > 0 else None
    for act in (0, 1):
        # unfused
        xd = K.dropout_fwd(x, first, rate, seed, step)
        y0 = K.linear_fwd(xd, w, activation=act)
        g0 = K.padded(n, o, DEV, fill=dy)
        dw0, dxd = torch.zeros_like(w), K.padded(n, i, DEV)
        K.linear_bwd(xd, w, y0, g0, dw0, dxd, activation=act)
        dx0 = K.dropout_fwd(dxd, first, rate, seed, step)      # dropout backward is the same map
        # fused
        y1 = K.linear_fwd_dropout(x, w, mask, rate, activation=act)
        g1 = K.padded(n, o, DEV, fill=dy)
        dw1, dx1 = torch.zeros_like(w), K.padded(n, i, DEV)
        K.linear_bwd_dropout(x, w, y1, g1, dw1, mask, rate, dx=dx1, activation=act)
        assert torch.equal(y0, y1), "fwd"
        assert torch.equal(dw0, dw1), "dW"
        assert torch.equal(dx0, dx1), "dX"


@pytest.mark.parametrize("n,i,o", [(1000, 64, 41), (4099, 200, 16), (300, 16, 16), (50, 5, 3)])
@pytest.mark.parametrize("rate", [0.5, 0.0])
def test_linear_bwd_fused_epilogue_matches_separate_kernels_bitwise(n, i, o, rate):
    """dX epilogue (dropout backward -> relu mask -> / sqrt(deg)) == the three separate kernels."""
    r = np.random.RandomState(n + o)
    row_end = np.cumsum(r.randint(1, 9, size=n)).astype(np.uint64)
    d_re = torch.from_numpy(row_end.view(np.int64)).to(DEV)
    first, seed, step = 0, (1 << 32) | 7, 3
    x = K.padded(n, i, DEV, fill=torch.from_numpy(np.maximum(r.randn(n, i), 0).astype(np.float32)).to(DEV))  # a relu output
    w = torch.from_numpy((r.randn(o, i) * 0.1).astype(np.float32)).to(DEV)
    dy_np = r.randn(n, o).astype(np.float32)
    dy_np[r.rand(n) < 0.6] = 0.0          # rows outside the training mask carry no gradient (zero-row fast path)
    dy = torch.from_numpy(dy_np).to(DEV)
    mask = K.dropout_mask(n, i, first, rate, seed, step, DEV) if rate > 0 else None
    # separate: linear bwd (+dropout bwd) -> indegree_norm with relu mask
    g0 = K.padded(n, o, DEV, fill=dy)
    dw0, dxa = torch.zeros_like(w), K.padded(n, i, DEV)
    K.linear_bwd_dropout(x, w, None, g0, dw0, mask, rate, dx=dxa)
    dx0 = K.indegree_norm(0, n - 1, 0, d_re, dxa, relu_mask_of=x)
    # fused
    g1 = K.padded(n, o, DEV, fill=dy)
    dw1, dx1 = torch.zeros_like(w), K.padded(n, i, DEV)
    K.linear_bwd_fused(x, w, None, g1, dw1, dx1, mask=mask, rate=rate, relu_of=x, norm_row_end=d_re, col_left=0)
    assert torch.equal(dw0, dw1), "dW"
    assert torch.equal(dx0, dx1), "dX"


def test_softmax_with_fused_norm_backward_bitwise():
    r = np.random.RandomState(14)
    for n, c in ((3000, 41), (500, 7), (257, 100), (64, 300)):
        row_end = np.cumsum(r.randint(1, 20, size=n)).astype(np.uint64)
        d_re = torch.from_numpy(row_end.view(np.int64)).to(DEV)
        logits = K.padded(n, c, DEV, fill=torch.from_numpy((r.randn(n, c) * 2).astype(np.float32)).to(DEV))
        lab = torch.from_numpy(r.randint(0, c, size=n).astype(np.int32)).to(DEV)
        mask = torch.from_numpy(r.randint(0, 4, size=n).astype(np.int32)).to(DEV)
        g, _ = K.softmax_xent_bwd(logits, lab, mask, compact=True)
        want = K.indegree_norm(0, n - 1, 0, d_re, g)
        got = K.softmax_xent_bwd_norm(logits, lab, mask, d_re, 0, compact=True)
        assert torch.equal(got, want)
        oh = torch.from_numpy(datasets.onehot(lab.cpu().numpy(), c)).to(DEV)
        got2 = K.softmax_xent_bwd_norm(logits, oh, mask, d_re, 0, compact=False)
        assert torch.equal(got2, want)


def test_softmax_xent_both_label_forms():
    r = np.random.RandomState(4)
    for n, c in ((500, 7), (1000, 41), (64, 47), (10, 1)):
        logits = (r.randn(n, c) * 2).astype(np.float32)
        lab = r.randint(0, c, size=n).astype(np.int32)
        mask = r.randint(0, 4, size=n).astype(np.int32)
        oh = datasets.onehot(lab, c)
        wg, wp = oracle.softmax_xent_bwd(logits, oh, mask)
        for compact in (False, True):
            labels = torch.from_numpy(lab).to(DEV) if compact else torch.from_numpy(oh).to(DEV)
            g, p = K.softmax_xent_bwd(K.padded(n, c, DEV, fill=torch.from_numpy(logits).to(DEV)), labels,
                                      torch.from_numpy(mask).to(DEV), compact=compact)
            rel_close(g.cpu().numpy(), wg, what="softmax grad")
            assert abs(p["trainLoss"] - wp["trainLoss"]) <= 1e-4 * max(abs(wp["trainLoss"]), 1.0)
            for k in ("trainAll", "testAll", "valAll", "trainCorrect", "testCorrect", "valCorrect"):
                assert p[k] == wp[k], (k, p, wp)


@pytest.mark.parametrize("n,i,o", [(200, 33, 9), (1000, 602, 64), (777, 64, 41), (129, 16, 16), (5, 3, 2)])
def test_linear_fwd_bwd(n, i, o):
    r = np.random.RandomState(n)
    x, w, dy = r.randn(n, i).astype(np.float32), (r.randn(o, i) * 0.1).astype(np.float32), r.randn(n, o).astype(np.float32)
    xp = K.padded(n, i, DEV, fill=torch.from_numpy(x).to(DEV))
    wd = torch.from_numpy(w).to(DEV)
    for act in (0, 1):
        y = K.linear_fwd(xp, wd, activation=act)
        wy = oracle.linear_fwd(x, w, relu=bool(act))
        rel_close(y.cpu().numpy(), wy, what="linear fwd")
        gy = K.padded(n, o, DEV, fill=torch.from_numpy(dy).to(DEV))
        dw = torch.ones_like(wd)
        dx = K.padded(n, i, DEV)
        K.linear_bwd(xp, wd, y, gy, dw, dx, activation=act)
        wdw = np.ones_like(w)
        wgy = dy.copy()
        wdx = oracle.linear_bwd(x, w, wy, wgy, wdw, relu=bool(act))
        rel_close(dw.cpu().numpy(), wdw, what="dW")
        rel_close(dx.cpu().numpy(), wdx, what="dX")
        assert np.array_equal(gy.cpu().numpy(), wgy)      # relu mask applied in place
        K.linear_bwd(xp, wd, y, gy, dw, dx, activation=0, accumulate_dx=True)
        rel_close(dx.cpu().numpy(), 2 * wdx, what="dX accumulate")


def test_linear_norm_epilogue():
    row_end, col = graph("uniform")
    n = row_end.shape[0]
    r = np.random.RandomState(8)
    x, w = r.randn(n, 24).astype(np.float32), r.randn(16, 24).astype(np.float32)
    d_re, _ = to_dev(row_end, col[:1])
    y = K.linear_fwd(torch.from_numpy(x).to(DEV), torch.from_numpy(w).to(DEV))
    yn = K.linear_fwd(torch.from_numpy(x).to(DEV), torch.from_numpy(w).to(DEV), norm_row_end=d_re, col_left=0)
    want = oracle.indegree_norm(0, n - 1, 0, row_end, np.ascontiguousarray(y.cpu().numpy()))
    assert np.array_equal(yn.cpu().numpy(), want)


def test_adam():
    r = np.random.RandomState(6)
    w, g = r.randn(38528).astype(np.float32), r.randn(38528).astype(np.float32)
    m, v = (r.randn(38528) * 0.1).astype(np.float32), np.abs(r.randn(38528) * 0.1).astype(np.float32)
    ww, wm, wv = w.copy(), m.copy(), v.copy()
    oracle.adam_update(ww, g, wm, wv, np.float32(0.003), np.float32(0.9), np.float32(0.999), np.float32(0.05), np.float32(1e-8))
    dw, dg, dm, dv = (torch.from_numpy(t.copy()).to(DEV) for t in (w, g, m, v))
    K.adam_update(dw, dg, dm, dv, 0.003, 0.9, 0.999, 0.05, 1e-8)
    rel_close(dw.cpu().numpy(), ww, rtol=1e-6, what="adam w")
    rel_close(dm.cpu().numpy(), wm, rtol=1e-6, what="adam m")
    rel_close(dv.cpu().numpy(), wv, rtol=1e-6, what="adam v")


# ---------------------------------------------- golden vectors from the reference ---
def test_kernels_vs_reference_golden(golden):
    g = golden
    re, col = g["A_row_end"], g["A_col"]
    n = re.shape[0]
    d_re, d_col = to_dev(re, col)
    plan = K.SgPlan(0, n - 1, 0, d_re, d_col)
    rows = g["A_rows"]
    for h in (16, 41, 64):
        x = torch.from_numpy(g["A_sg_in_%d" % h]).to(DEV)
        rel_close(plan.forward(x, out=torch.empty((n, h), device=DEV)).cpu().numpy()[rows], g["A_sg_out_%d" % h],
                  what="vs aggre_coop_kernel H=%d" % h)
        assert np.array_equal(K.indegree_norm(0, n - 1, 0, d_re, x).cpu().numpy()[rows], g["A_norm_out_%d" % h])
    rp, es, _ = K.build_csr(0, n - 1, 0, d_re, d_col)
    assert np.array_equal(es.cpu().numpy().astype(np.uint32), g["A_edgestructs"])
    x, w, dy = (torch.from_numpy(g[k]).to(DEV) for k in ("lin_X", "lin_W", "lin_dY"))
    for relu in (0, 1):
        y = K.linear_fwd(x, w, activation=relu, out=torch.empty((x.shape[0], w.shape[0]), device=DEV))
        rel_close(y.cpu().numpy(), g["lin_Y_relu%d" % relu], what="vs cublasSgemm fwd")
        dw, dx, gy = torch.zeros_like(w), torch.zeros_like(x), dy.clone()
        K.linear_bwd(x, w, y, gy, dw, dx, activation=relu)
        rel_close(dw.cpu().numpy(), g["lin_dW_relu%d" % relu], what="vs cublasSgemm dW")
        rel_close(dx.cpu().numpy(), g["lin_dX_relu%d" % relu], what="vs cublasSgemm dX")
    grad, perf = K.softmax_xent_bwd(torch.from_numpy(g["sm_logits"]).to(DEV),
                                    torch.from_numpy(datasets.onehot(g["sm_labels"], 7)).to(DEV),
                                    torch.from_numpy(g["sm_mask"]).to(DEV))
    rel_close(grad.cpu().numpy(), g["sm_grad"], what="vs cudnnSoftmax+softmax_backward")
    assert [perf[k] for k in ("trainAll", "testAll", "valAll", "trainCorrect", "testCorrect", "valCorrect")] == \
        [int(v) for v in g["sm_perf"][1:]]
    dw, dg, dm, dv = (torch.from_numpy(g[k].copy()).to(DEV) for k in ("adam_w", "adam_gsum", "adam_m", "adam_v"))
    K.adam_update(dw, dg, dm, dv, 0.01, 0.9, 0.999, 0.05, 1e-8)
    rel_close(dw.cpu().numpy(), g["adam_w_out"], rtol=1e-6, what="vs adam_update")


def test_side_by_side_with_reference_kernel(golden):
    """The planned kernel on an R-MAT scale-14 graph with hub rows, at every hidden width of the variants, against
    the reference's aggre_coop_kernel: its outputs minted on a B200 (tests/golden/make_golden.py, graph C), and
    live on the whole output when oracle/_ref is there."""
    mg = golden_module("make_golden")
    row_end, col = mg.side_by_side_graph()
    assert mg.col_checksum(col) == int(golden["C_col_crc32"][0]), "the R-MAT generator no longer makes graph C"
    n = row_end.shape[0]
    d_re, d_col = to_dev(row_end, col)
    plan = K.SgPlan(0, n - 1, 0, d_re, d_col)
    if ref.available():
        rp, es = ref.edge_structs(d_col, d_re, 0, 0)
    for h in mg.SIDE_BY_SIDE_H:
        x = torch.from_numpy(mg.side_by_side_input(n, h)).to(DEV)
        got = plan.forward(x)
        torch.cuda.synchronize()
        rel_close(got.cpu().numpy()[golden["C_rows"]], golden["C_sg_out_%d" % h],
                  what="vs golden aggre_coop_kernel H=%d" % h)
        if ref.available():
            want = ref.scatter_gather(0, n - 1, 0, rp, es, x)
            rel_close(got.cpu().numpy(), want.cpu().numpy(), what="vs live aggre_coop_kernel H=%d" % h)


# ---------------------------------------- tcgen05 Linear vs the reference library at the headline shapes ---
LIN_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_golden_linear.npz")


@pytest.mark.parametrize("n,i,o", [(1000, 602, 64), (1000, 64, 41)])
def test_tcgen05_linear_meets_the_reference_cublas(n, i, o):
    """BASELINE.json configs[1]'s two Linear shapes, fed row-padded so the tcgen05 / TMEM kernels run (asserted
    through roc_last_gemm_path) — against outputs of the REFERENCE's cublasSgemm calls (linear_kernel.cu:76-80,
    220-231) minted on a B200 by tests/golden/make_golden_linear.py at a sample of rows, and live on the whole
    outputs against oracle/_ref when it is there."""
    X, W, dY = golden_module("make_golden_linear").inputs(n, i, o)
    xp = K.padded(n, i, DEV, fill=torch.from_numpy(X).to(DEV))
    w = torch.from_numpy(W).to(DEV)
    gyp = K.padded(n, o, DEV, fill=torch.from_numpy(dY).to(DEV))
    y = K.linear_fwd(xp, w)
    assert _lib.lib.roc_last_gemm_path(0) == 1, "forward did not take the tcgen05 path"
    dw = torch.zeros_like(w)
    dx = K.padded(n, i, DEV)
    K.linear_bwd(xp, w, None, gyp, dw, dx, activation=0)
    assert _lib.lib.roc_last_gemm_path(1) == 1 and _lib.lib.roc_last_gemm_path(2) == 1, "dW / dX not on tcgen05"
    torch.cuda.synchronize()
    k = "%dx%dx%d" % (n, i, o)
    g = np.load(LIN_GOLDEN)
    rows, wrows = g["rows_" + k], g["wrows_" + k]
    rel_close(y.cpu().numpy()[rows], g["Y_" + k], what="Y vs golden")
    rel_close(dw.cpu().numpy()[wrows], g["dW_" + k], what="dW vs golden")
    rel_close(dx.cpu().numpy()[rows], g["dX_" + k], what="dX vs golden")
    if ref.available():
        xd, gyd = torch.from_numpy(X).to(DEV), torch.from_numpy(dY).to(DEV)
        ry = ref.linear_fwd(xd, w, relu=False)
        rw, rx = torch.zeros_like(w), torch.zeros_like(xd)
        ref.linear_bwd(xd, w, ry, gyd.clone(), rw, rx, relu=False)
        torch.cuda.synchronize()
        rel_close(y.cpu().numpy(), ry.cpu().numpy(), what="Y vs live reference")
        rel_close(dw.cpu().numpy(), rw.cpu().numpy(), what="dW vs live reference")
        rel_close(dx.cpu().numpy(), rx.cpu().numpy(), what="dX vs live reference")


def test_unpadded_linear_reports_the_simt_fallback():
    x = torch.rand((200, 33), device=DEV)            # ld = 33: not 16-byte rows -> the tensor-core kernels decline
    w = torch.rand((9, 33), device=DEV)
    K.linear_fwd(x, w, out=torch.empty((200, 9), device=DEV))
    assert _lib.lib.roc_last_gemm_path(0) == 2
