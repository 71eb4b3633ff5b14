"""Kernel-level entry points (include/roc_b200.h) on torch CUDA tensors.

torch is used here only as the owner of device memory and streams: every
function passes raw device pointers + the current CUDA stream to the C ABI.
2-D tensors may be row-padded views (stride(0) = ld >= shape[1], stride(1) = 1).
"""
import ctypes as C

import torch

from . import _lib
from ._lib import check, lib


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _ld(t):
    assert t.dim() == 2 and t.stride(1) == 1, "need a row-major 2-D tensor"
    return t.stride(0)


def padded(rows, h, device="cuda", dtype=torch.float32, fill=None):
    """[rows][h] view of a [rows][round_up(h,4)] allocation (the host's node-tensor layout)."""
    ld = (h + 3) // 4 * 4
    buf = torch.zeros((rows, ld), device=device, dtype=dtype)
    v = buf[:, :h]
    if fill is not None:
        v.copy_(fill)
    return v


class SgPlan:
    """roc_sg_plan for one partition's CSR (rowEnd u64 END offsets, colSrc u32)."""

    def __init__(self, row_left, row_right, col_left, row_end, col_src):
        _lib.require_device()
        assert row_end.dtype == torch.int64 or row_end.dtype == torch.uint64
        assert col_src.dtype in (torch.int32, torch.uint32)
        self.row_left, self.row_right, self.col_left = int(row_left), int(row_right), int(col_left)
        self.row_end, self.col_src = row_end, col_src   # keep alive
        h = C.c_void_p()
        check(lib.roc_sg_plan_create(self.row_left, self.row_right, self.col_left, _ptr(row_end), _ptr(col_src),
                                     _stream(), C.byref(h)), "roc_sg_plan_create")
        self.handle = h

    def info(self):
        a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
        check(lib.roc_sg_plan_info(self.handle, C.byref(a), C.byref(b), C.byref(c)))
        return {"chunks": a.value, "carries": b.value, "heavy_rows": c.value}

    def reserve(self, max_h):
        check(lib.roc_sg_plan_reserve(self.handle, int(max_h)), "roc_sg_plan_reserve")

    def forward(self, x, out=None, epilogue=0):
        nloc = self.row_right - self.row_left + 1
        h = x.shape[1]
        if out is None:
            out = padded(nloc, h, x.device) if _ld(x) % 4 == 0 else torch.empty((nloc, h), device=x.device)
        check(lib.roc_sg_forward_planned(self.handle, h, _ptr(x), _ld(x), _ptr(out), _ld(out), int(epilogue),
                                         _stream()), "roc_sg_forward_planned")
        return out

    def reserve_arg(self, max_h):
        check(lib.roc_sg_plan_reserve_arg(self.handle, int(max_h)), "roc_sg_plan_reserve_arg")

    def aggr_forward(self, x, aggr, col_global=None, out=None, arg=None, want_arg=True):
        """MAX / MIN (aggr = "max" | "min" or _lib.AGGR_*): returns (out, arg); arg is a [nloc][H] int32 view of
        the u32 winner ids (global vertex ids; -1 = 0xFFFFFFFF for degree-0 rows), or None with want_arg=False."""
        aggr = _lib.AGGR[aggr] if isinstance(aggr, str) else int(aggr)
        nloc = self.row_right - self.row_left + 1
        h = x.shape[1]
        vec = _ld(x) % 4 == 0
        if out is None:
            out = padded(nloc, h, x.device) if vec else torch.empty((nloc, h), device=x.device)
        if arg is None and want_arg:
            arg = padded(nloc, h, x.device, dtype=torch.int32) if vec else torch.empty((nloc, h), device=x.device,
                                                                                     dtype=torch.int32)
        check(lib.roc_sg_aggr_forward(self.handle, aggr, h, _ptr(x), _ld(x), _ptr(col_global), _ptr(out), _ld(out),
                                      _ptr(arg), _ld(arg) if arg is not None else 0, _stream()),
              "roc_sg_aggr_forward")
        return out, arg

    def arg_backward(self, gy, arg, out=None):
        """dIn[u] = sum over the plan's edges (u <- v) of gy[v] where arg[v] == row_left + u."""
        nloc = self.row_right - self.row_left + 1
        h = gy.shape[1]
        if out is None:
            out = padded(nloc, h, gy.device) if _ld(gy) % 4 == 0 else torch.empty((nloc, h), device=gy.device)
        check(lib.roc_sg_arg_backward(self.handle, h, _ptr(gy), _ld(gy), _ptr(arg), _ld(arg), self.row_left,
                                      _ptr(out), _ld(out), _stream()), "roc_sg_arg_backward")
        return out

    # ---- graph attention (roc_gat_* in include/roc_b200.h).  Tensors the gathers index (h, att, bst, dOut) hold
    # the plan's own rows first: row r of them is local row r, further rows are what col ids beyond nloc name.
    def gat_reserve(self, h, heads):
        check(lib.roc_gat_plan_reserve(self.handle, int(h), int(heads)), "roc_gat_plan_reserve")

    def gat_forward(self, x, att, heads, slope=0.2, out=None, bst=None):
        """Returns (out [nloc][H], bst [rows of att][round_up4(2K)] with lse of the own rows in columns 0..K-1)."""
        nloc = self.row_right - self.row_left + 1
        h = x.shape[1]
        if out is None:
            out = padded(nloc, h, x.device) if _ld(x) % 4 == 0 else torch.empty((nloc, h), device=x.device)
        if bst is None:
            bst = padded(att.shape[0], 2 * heads, x.device)
        check(lib.roc_gat_forward(self.handle, h, heads, float(slope), _ptr(x), _ld(x), _ptr(att), _ld(att), _ptr(bst),
                                  _ld(bst), _ptr(out), _ld(out), _stream()), "roc_gat_forward")
        return out, bst

    def gat_backward(self, x, att, bst, gy, heads, slope=0.2, dx=None, ds=None):
        """The backward gather: returns (dh_agg [nloc][H], ds [nloc][round_up4(2K)] = ds_src | ds_dst)."""
        nloc = self.row_right - self.row_left + 1
        h = x.shape[1]
        if dx is None:
            dx = padded(nloc, h, x.device) if _ld(x) % 4 == 0 else torch.empty((nloc, h), device=x.device)
        if ds is None:
            ds = padded(nloc, 2 * heads, x.device)
        check(lib.roc_gat_backward(self.handle, h, heads, float(slope), _ptr(x), _ld(x), _ptr(att), _ld(att),
                                   _ptr(bst), _ld(bst), _ptr(gy), _ld(gy), _ptr(dx), _ld(dx), _ptr(ds), _ld(ds),
                                   _stream()), "roc_gat_backward")
        return dx, ds

    def close(self):
        if self.handle:
            lib.roc_sg_plan_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def sg_forward(row_left, row_right, col_left, row_end, col_src, x):
    """Plan-less form with the reference kernel's argument list; dense [N][H] in, [Nloc][H] out."""
    assert x.is_contiguous()
    out = torch.empty((row_right - row_left + 1, x.shape[1]), device=x.device, dtype=torch.float32)
    check(lib.roc_sg_forward(row_left, row_right, col_left, x.shape[1], _ptr(row_end), _ptr(col_src), _ptr(x),
                             _ptr(out), _stream()), "roc_sg_forward")
    return out


def sg_backward(row_left, row_right, col_left, row_end, col_src, gy):
    assert gy.is_contiguous()
    out = torch.empty((row_right - row_left + 1, gy.shape[1]), device=gy.device, dtype=torch.float32)
    check(lib.roc_sg_backward(row_left, row_right, col_left, gy.shape[1], _ptr(row_end), _ptr(col_src), _ptr(gy),
                              _ptr(out), _stream()), "roc_sg_backward")
    return out


def build_csr(row_left, row_right, col_left, raw_rows, raw_cols, want_edge_structs=True):
    nloc = row_right - row_left + 1
    eloc = raw_cols.shape[0]
    rp = torch.empty(nloc, dtype=torch.int64, device=raw_rows.device)
    es = torch.empty((max(eloc, 1), 2), dtype=torch.int32, device=raw_rows.device) if want_edge_structs else None
    cs = torch.empty(max(eloc, 1), dtype=torch.int32, device=raw_rows.device)
    check(lib.roc_build_csr(row_left, row_right, col_left, _ptr(raw_rows), _ptr(raw_cols), _ptr(rp), _ptr(es),
                            _ptr(cs), _stream()), "roc_build_csr")
    return rp, (es[:eloc] if es is not None else None), cs[:eloc]


def indegree_norm(row_left, row_right, col_left, row_end, x, out=None, relu_mask_of=None):
    if out is None:
        out = torch.empty_like(x) if x.is_contiguous() else padded(x.shape[0], x.shape[1], x.device)
    check(lib.roc_indegree_norm(row_left, row_right, col_left, x.shape[1], _ptr(row_end), _ptr(x), _ld(x), _ptr(out),
                                _ld(out), _ptr(relu_mask_of), _stream()), "roc_indegree_norm")
    return out


def indegree_div(row_left, row_right, col_left, row_end, x, out=None):
    """out = x / (float)deg per row (IEEE division; degree-0 rows give 0)."""
    if out is None:
        out = torch.empty_like(x) if x.is_contiguous() else padded(x.shape[0], x.shape[1], x.device)
    check(lib.roc_indegree_div(row_left, row_right, col_left, x.shape[1], _ptr(row_end), _ptr(x), _ld(x), _ptr(out),
                               _ld(out), _stream()), "roc_indegree_div")
    return out


def activation_fwd(x, mode):
    y = torch.empty_like(x)
    check(lib.roc_activation_fwd(x.shape[0], x.shape[1], mode, _ptr(x), _ld(x), _ptr(y), _ld(y), _stream()))
    return y


def activation_bwd(y, dy, mode, dx=None):
    acc = dx is not None
    if dx is None:
        dx = torch.empty_like(y)
    check(lib.roc_activation_bwd(y.shape[0], y.shape[1], mode, _ptr(y), _ld(y), _ptr(dy), _ld(dy), _ptr(dx), _ld(dx),
                                 int(acc), _stream()))
    return dx


def add_fwd(a, b):
    y = torch.empty_like(a)
    check(lib.roc_add_fwd(a.shape[0], a.shape[1], _ptr(a), _ld(a), _ptr(b), _ld(b), _ptr(y), _ld(y), _stream()))
    return y


def add_bwd(dy, da, acc_a, db, acc_b):
    check(lib.roc_add_bwd(dy.shape[0], dy.shape[1], _ptr(dy), _ld(dy), _ptr(da), _ld(da) if da is not None else 0,
                          int(acc_a), _ptr(db), _ld(db) if db is not None else 0, int(acc_b), _stream()))


def dropout_fwd(x, first_row, rate, seed, step, out=None):
    if out is None:
        out = torch.empty_like(x) if x.is_contiguous() else padded(x.shape[0], x.shape[1], x.device)
    check(lib.roc_dropout_fwd(x.shape[0], x.shape[1], first_row, rate, seed, step, _ptr(x), _ld(x), _ptr(out),
                              _ld(out), _stream()), "roc_dropout_fwd")
    return out


def dropout_mask(rows, h, first_row, rate, seed, step, device="cuda"):
    """Packed keep-mask [rows][round_up(ceil(h/32), 4)] uint32 (as int32 storage) of roc_dropout_fwd's mask."""
    ldm = ((h + 31) // 32 + 3) // 4 * 4
    m = torch.empty((rows, ldm), dtype=torch.int32, device=device)
    check(lib.roc_dropout_mask(rows, h, first_row, rate, seed, step, _ptr(m), ldm, _stream()), "roc_dropout_mask")
    return m


def softmax_xent_bwd(logits, labels, mask, compact=False):
    """labels: one-hot fp32 [N][C] (reference format) or, with compact=True, int32 class ids [N]."""
    g = torch.empty_like(logits)
    perf = torch.zeros(7, dtype=torch.int32, device=logits.device)
    if compact:
        check(lib.roc_softmax_xent_bwd_idx(logits.shape[0], logits.shape[1], _ptr(logits), _ld(logits), _ptr(labels),
                                           _ptr(mask), _ptr(g), _ld(g), _ptr(perf), _stream()))
    else:
        check(lib.roc_softmax_xent_bwd(logits.shape[0], logits.shape[1], _ptr(logits), _ld(logits), _ptr(labels),
                                       _ld(labels), _ptr(mask), _ptr(g), _ld(g), _ptr(perf), _stream()))
    p = perf.cpu()
    d = {"trainLoss": float(p[:1].view(torch.float32)[0]), "trainAll": int(p[1]), "testAll": int(p[2]),
         "valAll": int(p[3]), "trainCorrect": int(p[4]), "testCorrect": int(p[5]), "valCorrect": int(p[6])}
    return g, d


def linear_fwd(x, w, activation=0, norm_row_end=None, col_left=0, out=None):
    """x [N][in] (ld-padded ok), w [out][in] contiguous (= W_mem[o*in + i]) -> [N][out]."""
    assert w.is_contiguous()
    if out is None:
        out = padded(x.shape[0], w.shape[0], x.device)
    flags = _lib.LINEAR_NORM_EPILOGUE if norm_row_end is not None else 0
    check(lib.roc_linear_fwd(x.shape[0], x.shape[1], w.shape[0], _ptr(x), _ld(x), _ptr(w), _ptr(out), _ld(out),
                             activation, flags, _ptr(norm_row_end), col_left, _stream()), "roc_linear_fwd")
    return out


def linear_fwd_dropout(x, w, mask, rate, activation=0, norm_row_end=None, col_left=0, out=None):
    """linear_fwd(dropout(x)) with the dropout applied while loading x (mask from dropout_mask)."""
    assert w.is_contiguous()
    if out is None:
        out = padded(x.shape[0], w.shape[0], x.device)
    flags = _lib.LINEAR_NORM_EPILOGUE if norm_row_end is not None else 0
    check(lib.roc_linear_fwd_dropout(x.shape[0], x.shape[1], w.shape[0], _ptr(x), _ld(x), _ptr(w), _ptr(out),
                                     _ld(out), activation, flags, _ptr(norm_row_end), col_left, _ptr(mask),
                                     mask.stride(0) if mask is not None else 0, rate, _stream()),
          "roc_linear_fwd_dropout")
    return out


def linear_bwd_dropout(x, w, y, dy, dw, mask, rate, dx=None, activation=0, accumulate_dx=False):
    """linear_bwd where the forward input was dropout(x); dx is the gradient of x (pre-dropout)."""
    ws_bytes = lib.roc_linear_bwd_workspace_bytes(x.shape[0], x.shape[1], w.shape[0])
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=x.device)
    check(lib.roc_linear_bwd_dropout(x.shape[0], x.shape[1], w.shape[0], _ptr(x), _ld(x), _ptr(w), _ptr(y),
                                     _ld(y) if y is not None else 0, _ptr(dy), _ld(dy), _ptr(dw), _ptr(dx),
                                     _ld(dx) if dx is not None else 0, activation, int(accumulate_dx), _ptr(ws),
                                     ws_bytes, _ptr(mask), mask.stride(0) if mask is not None else 0, rate,
                                     _stream()), "roc_linear_bwd_dropout")
    return dw, dx


def linear_bwd_fused(x, w, y, dy, dw, dx, activation=0, mask=None, rate=0.0, relu_of=None, norm_row_end=None,
                     col_left=0):
    """roc_linear_bwd_fused: dX epilogue = dropout backward -> relu mask (relu_of > 0) -> / sqrt(deg)."""
    ws_bytes = lib.roc_linear_bwd_workspace_bytes(x.shape[0], x.shape[1], w.shape[0])
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=x.device)
    a = _lib.LinearBwdArgs()
    a.rows, a.inDim, a.outDim = x.shape[0], x.shape[1], w.shape[0]
    a.X, a.ldX, a.W = x.data_ptr(), _ld(x), w.data_ptr()
    a.Y, a.ldY = (y.data_ptr(), _ld(y)) if y is not None else (None, 0)
    a.dY, a.ldDY, a.dW = dy.data_ptr(), _ld(dy), dw.data_ptr()
    a.dX, a.ldDX = dx.data_ptr(), _ld(dx)
    a.activation, a.accumulate_dX = activation, 0
    a.workspace, a.workspaceBytes = ws.data_ptr(), ws_bytes
    if mask is not None:
        a.dropMask, a.ldMask = mask.data_ptr(), mask.stride(0)
    a.dropRate = rate
    if relu_of is not None:
        a.dxReluOf, a.ldReluOf = relu_of.data_ptr(), _ld(relu_of)
    if norm_row_end is not None:
        a.dxNormRowEnd, a.colLeft = norm_row_end.data_ptr(), col_left
    check(lib.roc_linear_bwd_fused(C.byref(a), _stream()), "roc_linear_bwd_fused")
    return dw, dx


def softmax_xent_bwd_norm(logits, labels, mask, row_end, col_left=0, compact=False):
    """softmax_xent_bwd with the logits' InDegreeNorm backward fused: grad rows divided by sqrt(deg)."""
    g = torch.empty_like(logits)
    perf = torch.zeros(7, dtype=torch.int32, device=logits.device)
    check(lib.roc_softmax_xent_bwd_norm(logits.shape[0], logits.shape[1], _ptr(logits), _ld(logits),
                                        None if compact else _ptr(labels), 0 if compact else _ld(labels),
                                        _ptr(labels) if compact else None, _ptr(mask), _ptr(g), _ld(g),
                                        _ptr(row_end), col_left, _ptr(perf), _stream()), "roc_softmax_xent_bwd_norm")
    return g


def linear_bwd(x, w, y, dy, dw, dx=None, activation=0, accumulate_dx=False):
    ws_bytes = lib.roc_linear_bwd_workspace_bytes(x.shape[0], x.shape[1], w.shape[0])
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=x.device)
    check(lib.roc_linear_bwd(x.shape[0], x.shape[1], w.shape[0], _ptr(x), _ld(x), _ptr(w), _ptr(y),
                             _ld(y) if y is not None else 0, _ptr(dy), _ld(dy), _ptr(dw), _ptr(dx),
                             _ld(dx) if dx is not None else 0, activation, int(accumulate_dx), _ptr(ws), ws_bytes,
                             _stream()), "roc_linear_bwd")
    return dw, dx


def adam_update(w, g, m, v, alpha_t, beta1, beta2, wd, eps):
    check(lib.roc_adam_update(w.numel(), alpha_t, beta1, beta2, wd, eps, _ptr(g), _ptr(m), _ptr(v), _ptr(w),
                              _stream()))


def launch_count():
    return lib.roc_launch_count()


# ---- graph attention, per-node kernels
def gat_scores(x, att_w, heads, rows=None):
    """att[r] = (s_src[r][0..K) | s_dst[r][0..K)) for rows 0 .. rows-1 (default: all of x), [x rows][round_up4(2K)];
    att_w: the [2][H] parameter (row 0 a_src, row 1 a_dst)."""
    rows = x.shape[0] if rows is None else rows
    att = padded(x.shape[0], 2 * heads, x.device)
    check(lib.roc_gat_scores(rows, x.shape[1], heads, _ptr(x), _ld(x), _ptr(att_w), _ptr(att), _ld(att), _stream()),
          "roc_gat_scores")
    return att


def gat_c(gy, out, bst, heads):
    """c = <gy, out> per row and head into bst's columns K..2K-1 (rows of gy)."""
    check(lib.roc_gat_bwd_c(gy.shape[0], gy.shape[1], heads, _ptr(gy), _ld(gy), _ptr(out), _ld(out), _ptr(bst),
                            _ld(bst), _stream()), "roc_gat_bwd_c")
    return bst


def gat_finish(x, att_w, ds, dx, heads):
    """dx[r] += ds_src[r] a_src + ds_dst[r] a_dst per head, in place, for the rows of dx; returns da [2][H]."""
    h = x.shape[1]
    da = torch.empty((2, h), device=x.device)
    nbytes = lib.roc_gat_finish_workspace_bytes(h)
    ws = torch.empty(nbytes // 4, device=x.device)
    check(lib.roc_gat_bwd_finish(dx.shape[0], h, heads, _ptr(x), _ld(x), _ptr(att_w), _ptr(ds), _ld(ds), _ptr(dx),
                                 _ld(dx), _ptr(da), _ptr(ws), nbytes, _stream()), "roc_gat_bwd_finish")
    return da
