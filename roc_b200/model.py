"""Python mirror of the reference's Model / op-builder API (gnn.h:162-203) over the
C++ host (include/roc_host.h).  Same method names and call order as the model
script in gnn.cc:65-111:

    host = Host(device, rank, world)            # Runtime (one per process / GPU)
    host.graph_from_arrays(row_end, col_src)    # Graph(ctx, runtime, config)
    m = Model(host)
    x = m.create_node_tensor(602); y = m.create_node_tensor(41); mk = m.create_node_tensor(1, is_int=True)
    t = m.dropout(x, 0.5); t = m.linear(t, 64); t = m.indegree_norm(t); t = m.scatter_gather(t) ...
    m.softmax_cross_entropy(t, y, mk)
    m.adam(lr, weight_decay); m.init()
    m.train_mode(); m.zero_gradients(); m.forward(); m.backward(); m.update()
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import PerfMetrics, check, lib


class Host:
    """Runtime + Graph of one process: owns the GPU, the stream, the partition's CSR."""

    def __init__(self, device=0, my_part=0, num_parts=1):
        _lib.require_device()
        self.device, self.my_part, self.num_parts = device, my_part, num_parts
        self.h = C.c_void_p(lib.roc_host_create(device, my_part, num_parts))
        self._keep = []

    # --- NCCL bootstrap: rank 0 makes the id, the launcher (torch.distributed) broadcasts it
    @staticmethod
    def nccl_unique_id():
        buf = (C.c_ubyte * 128)()
        check(lib.roc_host_nccl_unique_id(buf), "roc_host_nccl_unique_id")
        return bytes(buf)

    def nccl_init(self, uid):
        buf = (C.c_ubyte * 128).from_buffer_copy(uid)
        check(lib.roc_host_nccl_init(self.h, buf), "roc_host_nccl_init")

    def graph_from_lux(self, prefix):
        check(lib.roc_host_graph_from_lux(self.h, prefix.encode()))

    def graph_from_arrays(self, row_end, col_src):
        row_end = np.ascontiguousarray(row_end, dtype=np.uint64)
        col_src = np.ascontiguousarray(col_src, dtype=np.uint32)
        check(lib.roc_host_graph_from_arrays(self.h, row_end.shape[0], int(row_end[-1]), row_end.ctypes.data,
                                             col_src.ctypes.data))

    def graph_info(self):
        out = (C.c_uint64 * 6)()
        check(lib.roc_host_graph_info(self.h, out))
        k = ["numNodes", "numEdges", "rowLeft", "rowRight", "colLeft", "colRight"]
        return dict(zip(k, [int(v) for v in out]))

    def plan_info(self):
        a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
        check(lib.roc_sg_plan_info(lib.roc_host_graph_plan(self.h), C.byref(a), C.byref(b), C.byref(c)))
        return {"chunks": a.value, "carries": b.value, "heavy_rows": c.value}

    def synchronize(self):
        check(lib.roc_host_synchronize(self.h))

    @property
    def stream(self):
        return lib.roc_host_stream(self.h)

    def close(self):
        if self.h:
            lib.roc_host_destroy(self.h)
            self.h = None


class Model:
    def __init__(self, host, seed=None):
        self.host = host
        self.h = host.h
        self._gat_heads = {}
        if seed is not None:
            lib.roc_host_srand(seed)     # std::srand(config.seed), gnn.cc:56

    # ---- builders (gnn.h:165-179)
    def create_node_tensor(self, hidden, is_int=False):
        return lib.roc_host_create_node_tensor(self.h, hidden, int(is_int))

    def dropout(self, t, rate, seed=0):
        return lib.roc_host_dropout(self.h, t, rate, seed)

    def linear(self, t, out_dim, activation=_lib.AC_MODE_NONE):
        return lib.roc_host_linear(self.h, t, out_dim, activation)

    def indegree_norm(self, t):
        return lib.roc_host_indegree_norm(self.h, t)

    def scatter_gather(self, t, aggr="sum"):
        """aggr: "sum" (the reference's ScatterGather), "mean", "max" or "min"."""
        if aggr == "sum":
            return lib.roc_host_scatter_gather(self.h, t)
        return lib.roc_host_scatter_gather_aggr(self.h, t, _lib.AGGR[aggr])

    def sg_arg(self, t):
        """Winner ids (u32, global vertex ids) of the max / min scatter_gather whose output is `t`, own rows."""
        rows, hidden, _ = self.tensor_shape(t)
        out = np.empty((rows, hidden), dtype=np.uint32)
        check(lib.roc_host_sg_arg(self.h, t, out.ctypes.data), "roc_host_sg_arg")
        return out

    def graph_attention(self, t, heads=1, negative_slope=0.2):
        """GAT over tensor t (width H = heads * F, heads concatenated); owns a [2][H] parameter (a_src, a_dst)."""
        out = lib.roc_host_graph_attention(self.h, t, int(heads), float(negative_slope))
        self._gat_heads[out] = int(heads)
        return out

    def gat_lse(self, t):
        """lse [rows][heads] of the graph_attention whose output is `t`, own rows, as the latest forward left it."""
        rows, _, _ = self.tensor_shape(t)
        out = np.empty((rows, self._gat_heads[t]), dtype=np.float32)
        check(lib.roc_host_gat_lse(self.h, t, out.ctypes.data), "roc_host_gat_lse")
        return out

    def gat_param(self, t):
        """Parameter index of the [2][H] attention weight (row 0 a_src, row 1 a_dst) of the graph_attention whose
        output is `t`."""
        p = lib.roc_host_gat_param(self.h, t)
        if p < 0:
            raise _lib.RocError("tensor %d is not the output of a graph_attention" % t)
        return p

    def relu(self, t):
        return lib.roc_host_relu(self.h, t)

    def sigmoid(self, t):
        return lib.roc_host_sigmoid(self.h, t)

    def add(self, a, b):
        return lib.roc_host_add(self.h, a, b)

    def softmax_cross_entropy(self, logits, labels, mask):
        check(lib.roc_host_softmax_cross_entropy(self.h, logits, labels, mask))

    def adam(self, lr=0.01, weight_decay=0.05):
        check(lib.roc_host_adam(self.h, lr, weight_decay))

    @property
    def lr(self):
        return lib.roc_host_get_lr(self.h)

    @lr.setter
    def lr(self, v):
        check(lib.roc_host_set_lr(self.h, v))

    def set_fusion(self, on):
        check(lib.roc_host_set_fusion(self.h, int(on)))

    def init(self):
        check(lib.roc_host_init(self.h))

    # ---- data
    def load_features(self, t, prefix):
        check(lib.roc_host_load_features(self.h, t, prefix.encode()))

    def load_labels(self, t, prefix):
        check(lib.roc_host_load_labels(self.h, t, prefix.encode()))

    def load_train_mask(self, t, prefix):
        check(lib.roc_host_load_train_mask(self.h, t, prefix.encode()))

    def tensor_shape(self, t):
        out = (C.c_int64 * 3)()
        check(lib.roc_host_tensor_shape(self.h, t, out))
        return int(out[0]), int(out[1]), int(out[2])

    def tensor_ptr(self, t, grad=False):
        return lib.roc_host_tensor_ptr(self.h, t, int(grad))

    def set_tensor(self, t, arr, grad=False):
        rows, hidden, _ = self.tensor_shape(t)
        arr = np.ascontiguousarray(arr)
        assert arr.itemsize == 4 and arr.size == rows * hidden, (arr.shape, rows, hidden)
        check(lib.roc_host_set_tensor(self.h, t, arr.ctypes.data, int(grad)))

    def set_tensor_from_host_ptr(self, t, ptr, grad=False):
        """ptr: address of a dense [rows][hidden] 4-byte host buffer (e.g. pinned torch memory)."""
        check(lib.roc_host_set_tensor(self.h, t, C.c_void_p(ptr), int(grad)))

    def get_tensor(self, t, grad=False, dtype=np.float32):
        rows, hidden, _ = self.tensor_shape(t)
        out = np.empty((rows, hidden), dtype=dtype)
        check(lib.roc_host_get_tensor(self.h, t, out.ctypes.data, int(grad)))
        return out

    def set_labels(self, t, class_idx):
        a = np.ascontiguousarray(class_idx, dtype=np.int32)
        check(lib.roc_host_set_labels(self.h, t, a.ctypes.data))

    def num_parameters(self):
        return lib.roc_host_num_parameters(self.h)

    def parameter_shape(self, p):
        out = (C.c_int64 * 2)()
        check(lib.roc_host_parameter_shape(self.h, p, out))
        return int(out[0]), int(out[1])   # inDim, outDim

    def get_parameter(self, p, which="w"):
        i, o = self.parameter_shape(p)
        out = np.empty((o, i), dtype=np.float32)   # W_mem[o*inDim + i]
        check(lib.roc_host_get_parameter(self.h, p, out.ctypes.data, {"w": 0, "grad": 1, "m": 2, "v": 3}[which]))
        return out

    def set_parameter(self, p, w):
        i, o = self.parameter_shape(p)
        w = np.ascontiguousarray(w, dtype=np.float32)
        assert w.shape == (o, i)
        check(lib.roc_host_set_parameter(self.h, p, w.ctypes.data))

    # ---- train loop (gnn.cc:99-111)
    def train_mode(self):
        check(lib.roc_host_train_mode(self.h))

    def infer_mode(self):
        check(lib.roc_host_infer_mode(self.h))

    def zero_gradients(self):
        check(lib.roc_host_zero_gradients(self.h))

    def forward(self):
        check(lib.roc_host_forward(self.h))

    def backward(self):
        check(lib.roc_host_backward(self.h))

    def update(self):
        check(lib.roc_host_update(self.h))

    def train_epoch(self):
        check(lib.roc_host_train_epoch(self.h))

    def profile_sg(self, on=True):
        check(lib.roc_host_profile_sg(self.h, int(on)))

    def profile_sg_read(self, max_entries=4096):
        hs = (C.c_int * max_entries)()
        ms = (C.c_float * max_entries)()
        n = lib.roc_host_profile_sg_read(self.h, max_entries, hs, ms)
        return [(int(hs[i]), float(ms[i])) for i in range(n)]

    def metrics(self):
        pm = PerfMetrics()
        check(lib.roc_host_metrics(self.h, C.byref(pm)))
        return pm.as_dict()


def build_gcn(model, layers, dropout_rate, lr=0.01, weight_decay=0.05):
    """The model script of gnn.cc:65-98 for `-layers a-b-...-c`.  Returns the handles."""
    L = len(layers)
    x = model.create_node_tensor(layers[0])
    label = model.create_node_tensor(layers[-1])
    mask = model.create_node_tensor(1, is_int=True)
    t = x
    relu_outs = []
    for i in range(1, L):
        t = model.dropout(t, dropout_rate)
        skip = t
        t = model.linear(t, layers[i], _lib.AC_MODE_NONE)
        t = model.indegree_norm(t)
        t = model.scatter_gather(t)
        t = model.indegree_norm(t)
        if i != L - 1:
            t = model.relu(t)
            relu_outs.append(t)
        if L > 3:   # residual branch, gnn.cc:86-90
            skip = model.linear(skip, layers[i], _lib.AC_MODE_NONE)
            t = model.add(t, skip)
    model.softmax_cross_entropy(t, label, mask)
    model.adam(lr, weight_decay)
    model.init()
    return {"input": x, "label": label, "mask": mask, "logits": t, "relu_outs": relu_outs}


def build_sage_mean(model, layers, dropout_rate, lr=0.01, weight_decay=0.05):
    """GraphSAGE with the mean aggregator (BASELINE.json configs[2]) composed from the reference's own ops
    (gnn.h:165-179; AGGR_AVG is declared at gnn.h:75-80 but the reference's ScatterGather only sums):

        D    = dropout(t)
        nb   = indegree_norm(indegree_norm(scatter_gather(linear(D, d_i))))    # D^-1 A (D W_nb): the mean over
                                                                               # N(v) + v (self loops are in A)
        t    = add(nb, linear(D, d_i))                                         # + the root / self weight
        t    = relu(t)                                                         # all but the last layer

    x / sqrt(deg) / sqrt(deg) is the mean to within one fp32 rounding.  Same wiring as the reference's residual
    GCN layer (gnn.cc:79-90) with both norms after the aggregation."""
    L = len(layers)
    x = model.create_node_tensor(layers[0])
    label = model.create_node_tensor(layers[-1])
    mask = model.create_node_tensor(1, is_int=True)
    t = x
    relu_outs = []
    for i in range(1, L):
        d = model.dropout(t, dropout_rate)
        nb = model.linear(d, layers[i], _lib.AC_MODE_NONE)
        nb = model.scatter_gather(nb)
        nb = model.indegree_norm(nb)
        nb = model.indegree_norm(nb)
        root = model.linear(d, layers[i], _lib.AC_MODE_NONE)
        t = model.add(nb, root)
        if i != L - 1:
            t = model.relu(t)
            relu_outs.append(t)
    model.softmax_cross_entropy(t, label, mask)
    model.adam(lr, weight_decay)
    model.init()
    return {"input": x, "label": label, "mask": mask, "logits": t, "relu_outs": relu_outs}


def build_sage(model, layers, dropout_rate, aggr="mean", lr=0.01, weight_decay=0.05):
    """GraphSAGE with a native aggregator ("mean", "max", "min" or "sum"): build_sage_mean's wiring

        D  = dropout(t)
        t  = add(scatter_gather(linear(D, d_i), aggr), linear(D, d_i))     # neighbours + the root / self weight
        t  = relu(t)                                                          # all but the last layer

    with the aggregation done by one ScatterGather (mean: one IEEE division of the sum by the in-degree).
    "sage_outs" are the aggregation outputs (for max / min: where Model.sg_arg reads the winner ids)."""
    L = len(layers)
    x = model.create_node_tensor(layers[0])
    label = model.create_node_tensor(layers[-1])
    mask = model.create_node_tensor(1, is_int=True)
    t = x
    relu_outs, sage_outs = [], []
    for i in range(1, L):
        d = model.dropout(t, dropout_rate)
        nb = model.linear(d, layers[i], _lib.AC_MODE_NONE)
        nb = model.scatter_gather(nb, aggr)
        sage_outs.append(nb)
        root = model.linear(d, layers[i], _lib.AC_MODE_NONE)
        t = model.add(nb, root)
        if i != L - 1:
            t = model.relu(t)
            relu_outs.append(t)
    model.softmax_cross_entropy(t, label, mask)
    model.adam(lr, weight_decay)
    model.init()
    return {"input": x, "label": label, "mask": mask, "logits": t, "relu_outs": relu_outs, "sage_outs": sage_outs}


def build_gat(model, layers, heads, dropout_rate, negative_slope=0.2, lr=0.01, weight_decay=0.05):
    """Graph attention network (Velickovic et al. 2018) for `layers` = [in, h_1, ..., out]:

        t  = graph_attention(linear(dropout(t), layers[i]), K_i)     # K_i = heads, 1 in the last layer
        t  = relu(t)                                                  # all but the last layer

    Each hidden width layers[i] is K_i heads of layers[i] / K_i features, concatenated.  "gat_outs" are the
    attention outputs (Model.gat_lse / gat_param take them), "att_params" the parameter indices of their [2][H]
    attention weights."""
    L = len(layers)
    x = model.create_node_tensor(layers[0])
    label = model.create_node_tensor(layers[-1])
    mask = model.create_node_tensor(1, is_int=True)
    t = x
    relu_outs, gat_outs = [], []
    for i in range(1, L):
        d = model.dropout(t, dropout_rate)
        t = model.linear(d, layers[i], _lib.AC_MODE_NONE)
        t = model.graph_attention(t, heads if i != L - 1 else 1, negative_slope)
        gat_outs.append(t)
        if i != L - 1:
            t = model.relu(t)
            relu_outs.append(t)
    model.softmax_cross_entropy(t, label, mask)
    model.adam(lr, weight_decay)
    model.init()
    return {"input": x, "label": label, "mask": mask, "logits": t, "relu_outs": relu_outs, "gat_outs": gat_outs,
            "att_params": [model.gat_param(g) for g in gat_outs]}
