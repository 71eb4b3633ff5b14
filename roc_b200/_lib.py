"""ctypes binding of roc_b200/lib/libroc_b200.so (include/roc_b200.h + include/roc_host.h).

The product has no CPU fallback: if the library is missing this module raises at
import, and on a machine without a CUDA device every compute entry point returns
ROC_ERR_NO_DEVICE (-4) / aborts instead of silently running somewhere else.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libroc_b200.so")

ROC_OK = 0
ROC_ERR_INVALID, ROC_ERR_UNSUPPORTED, ROC_ERR_NOMEM, ROC_ERR_NO_DEVICE, ROC_ERR_IO = -1, -2, -3, -4, -5
AC_MODE_NONE, AC_MODE_RELU, AC_MODE_SIGMOID = 0, 1, 2
MASK_TRAIN, MASK_VAL, MASK_TEST, MASK_NONE = 0, 1, 2, 3
SG_EPI_NONE, SG_EPI_NORM, SG_EPI_RELU, SG_EPI_MEAN = 0, 1, 2, 4
AGGR_AVG, AGGR_MAX, AGGR_MIN, AGGR_SUM = 0, 1, 2, 3
AGGR = {"mean": AGGR_AVG, "avg": AGGR_AVG, "max": AGGR_MAX, "min": AGGR_MIN, "sum": AGGR_SUM}
SG_NO_ARG = 0xFFFFFFFF
LINEAR_NORM_EPILOGUE = 1


class LinearBwdArgs(C.Structure):
    """roc_linear_bwd_args (include/roc_b200.h)."""
    _fields_ = [("rows", C.c_int64), ("inDim", C.c_int), ("outDim", C.c_int),
                ("X", C.c_void_p), ("ldX", C.c_int64), ("W", C.c_void_p),
                ("Y", C.c_void_p), ("ldY", C.c_int64), ("dY", C.c_void_p), ("ldDY", C.c_int64),
                ("dW", C.c_void_p), ("dX", C.c_void_p), ("ldDX", C.c_int64),
                ("activation", C.c_int), ("accumulate_dX", C.c_int),
                ("workspace", C.c_void_p), ("workspaceBytes", C.c_size_t),
                ("dropMask", C.c_void_p), ("ldMask", C.c_int64), ("dropRate", C.c_float),
                ("dxReluOf", C.c_void_p), ("ldReluOf", C.c_int64),
                ("dxNormRowEnd", C.c_void_p), ("colLeft", C.c_uint64), ("parts", C.c_int)]


class PerfMetrics(C.Structure):
    """PerfMetrics, softmax_kernel.cu:35-39."""
    _fields_ = [("trainLoss", C.c_float), ("trainAll", C.c_int), ("testAll", C.c_int), ("valAll", C.c_int),
                ("trainCorrect", C.c_int), ("testCorrect", C.c_int), ("valCorrect", C.c_int)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class RocError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "roc_b200: %s is missing - build it with `make` (or __graft_entry__.build()); "
            "there is no Python/CPU fallback for the kernels" % LIB_PATH)
    return C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)


lib = _load()

vp, i32, i64, u32, u64, f32, f64, sz = (C.c_void_p, C.c_int, C.c_int64, C.c_uint32, C.c_uint64, C.c_float,
                                        C.c_double, C.c_size_t)

# name -> (restype, argtypes); every symbol include/roc_b200.h and include/roc_host.h declare
PROTOTYPES = {
    # ---- roc_b200.h
    "roc_version": (C.c_char_p, []),
    "roc_device_count": (i32, []),
    "roc_launch_count": (u64, []),
    "roc_set_sm_reserve": (i32, [i32]),
    "roc_partition": (i32, [u32, u64, i32, vp, vp, vp, vp]),
    "roc_build_csr": (i32, [u32, u32, u64, vp, vp, vp, vp, vp, vp]),
    "roc_sg_plan_create": (i32, [u32, u32, u64, vp, vp, vp, C.POINTER(vp)]),
    "roc_sg_plan_reserve": (i32, [vp, i32]),
    "roc_sg_plan_destroy": (None, [vp]),
    "roc_sg_plan_info": (i32, [vp, C.POINTER(u64), C.POINTER(u64), C.POINTER(u64)]),
    "roc_sg_forward_planned": (i32, [vp, i32, vp, i64, vp, i64, i32, vp]),
    "roc_sg_forward": (i32, [u32, u32, u64, i32, vp, vp, vp, vp, vp]),
    "roc_sg_backward": (i32, [u32, u32, u64, i32, vp, vp, vp, vp, vp]),
    "roc_sg_aggr_forward": (i32, [vp, i32, i32, vp, i64, vp, vp, i64, vp, i64, vp]),
    "roc_sg_arg_backward": (i32, [vp, i32, vp, i64, vp, i64, u32, vp, i64, vp]),
    "roc_sg_plan_reserve_arg": (i32, [vp, i32]),
    "roc_gat_supported": (i32, [i32, i32]),
    "roc_gat_plan_reserve": (i32, [vp, i32, i32]),
    "roc_gat_scores": (i32, [i64, i32, i32, vp, i64, vp, vp, i64, vp]),
    "roc_gat_forward": (i32, [vp, i32, i32, f32, vp, i64, vp, i64, vp, i64, vp, i64, vp]),
    "roc_gat_bwd_c": (i32, [i64, i32, i32, vp, i64, vp, i64, vp, i64, vp]),
    "roc_gat_backward": (i32, [vp, i32, i32, f32, vp, i64, vp, i64, vp, i64, vp, i64, vp, i64, vp, i64, vp]),
    "roc_gat_finish_workspace_bytes": (sz, [i32]),
    "roc_gat_bwd_finish": (i32, [i64, i32, i32, vp, i64, vp, vp, i64, vp, i64, vp, vp, sz, vp]),
    "roc_halo_create": (i32, [u32, u32, u64, vp, vp, C.POINTER(vp)]),
    "roc_halo_destroy": (None, [vp]),
    "roc_halo_size": (u32, [vp]),
    "roc_halo_ids": (vp, [vp]),
    "roc_halo_col_local": (vp, [vp]),
    "roc_halo_recv_layout": (i32, [u32, vp, i32, i32, vp, vp, vp]),
    "roc_halo_send_layout": (i32, [i32, i32, vp, vp, vp, vp]),
    "roc_pack_rows": (i32, [i64, i32, vp, vp, i64, vp, i64, vp]),
    "roc_pack_rows_at": (i32, [i64, i32, vp, vp, vp, i64, vp, i64, vp]),
    "roc_push_rows": (i32, [i64, i32, vp, vp, vp, vp, i64, vp, i32, i64, i32, vp]),
    "roc_indegree_norm": (i32, [u32, u32, u64, i32, vp, vp, i64, vp, i64, vp, vp]),
    "roc_indegree_div": (i32, [u32, u32, u64, i32, vp, vp, i64, vp, i64, vp]),
    "roc_activation_fwd": (i32, [i64, i32, i32, vp, i64, vp, i64, vp]),
    "roc_activation_bwd": (i32, [i64, i32, i32, vp, i64, vp, i64, vp, i64, i32, vp]),
    "roc_add_fwd": (i32, [i64, i32, vp, i64, vp, i64, vp, i64, vp]),
    "roc_add_bwd": (i32, [i64, i32, vp, i64, vp, i64, i32, vp, i64, i32, vp]),
    "roc_dropout_fwd": (i32, [i64, i32, i64, f32, u64, u32, vp, i64, vp, i64, vp]),
    "roc_dropout_bwd": (i32, [i64, i32, i64, f32, u64, u32, vp, i64, vp, i64, vp]),
    "roc_dropout_mask": (i32, [i64, i32, i64, f32, u64, u32, vp, i64, vp]),
    "roc_softmax_xent_bwd": (i32, [i64, i32, vp, i64, vp, i64, vp, vp, i64, vp, vp]),
    "roc_softmax_xent_bwd_idx": (i32, [i64, i32, vp, i64, vp, vp, vp, i64, vp, vp]),
    "roc_softmax_xent_bwd_norm": (i32, [i64, i32, vp, i64, vp, i64, vp, vp, vp, i64, vp, u64, vp, vp]),
    "roc_linear_bwd_fused": (i32, [vp, vp]),
    "roc_linear_fwd": (i32, [i64, i32, i32, vp, i64, vp, vp, i64, i32, i32, vp, u64, vp]),
    "roc_linear_bwd_workspace_bytes": (sz, [i64, i32, i32]),
    "roc_linear_bwd": (i32, [i64, i32, i32, vp, i64, vp, vp, i64, vp, i64, vp, vp, i64, i32, i32, vp, sz, vp]),
    "roc_linear_fwd_dropout": (i32, [i64, i32, i32, vp, i64, vp, vp, i64, i32, i32, vp, u64, vp, i64, f32, vp]),
    "roc_linear_bwd_dropout": (i32, [i64, i32, i32, vp, i64, vp, vp, i64, vp, i64, vp, vp, i64, i32, i32, vp, sz,
                                     vp, i64, f32, vp]),
    "roc_last_gemm_path": (i32, [i32]),
    "roc_adam_update": (i32, [i64, f32, f32, f32, f32, f32, vp, vp, vp, vp, vp]),
    "roc_scale": (i32, [i64, f32, f32, vp, vp]),
    "roc_fill": (i32, [i64, i32, f32, vp, i64, vp]),
    "roc_copy2d": (i32, [i64, i32, vp, i64, vp, i64, vp]),
    "roc_selftest_rowdiv": (i32, [f32, u64, u64, vp, vp]),
    # ---- roc_host.h
    "roc_host_create": (vp, [i32, i32, i32]),
    "roc_host_destroy": (None, [vp]),
    "roc_host_nccl_unique_id": (i32, [vp]),
    "roc_host_nccl_init": (i32, [vp, vp]),
    "roc_host_synchronize": (i32, [vp]),
    "roc_host_stream": (vp, [vp]),
    "roc_host_graph_from_lux": (i32, [vp, C.c_char_p]),
    "roc_host_graph_from_arrays": (i32, [vp, u32, u64, vp, vp]),
    "roc_host_graph_info": (i32, [vp, vp]),
    "roc_host_graph_plan": (vp, [vp]),
    "roc_host_create_node_tensor": (i32, [vp, i32, i32]),
    "roc_host_dropout": (i32, [vp, i32, f32, i32]),
    "roc_host_linear": (i32, [vp, i32, i32, i32]),
    "roc_host_indegree_norm": (i32, [vp, i32]),
    "roc_host_scatter_gather": (i32, [vp, i32]),
    "roc_host_scatter_gather_aggr": (i32, [vp, i32, i32]),
    "roc_host_graph_attention": (i32, [vp, i32, i32, f32]),
    "roc_host_relu": (i32, [vp, i32]),
    "roc_host_sigmoid": (i32, [vp, i32]),
    "roc_host_add": (i32, [vp, i32, i32]),
    "roc_host_softmax_cross_entropy": (i32, [vp, i32, i32, i32]),
    "roc_host_adam": (i32, [vp, f64, f64]),
    "roc_host_set_lr": (i32, [vp, f64]),
    "roc_host_get_lr": (f64, [vp]),
    "roc_host_srand": (None, [C.c_uint]),
    "roc_host_set_fusion": (i32, [vp, i32]),
    "roc_host_init": (i32, [vp]),
    "roc_host_load_features": (i32, [vp, i32, C.c_char_p]),
    "roc_host_load_labels": (i32, [vp, i32, C.c_char_p]),
    "roc_host_load_train_mask": (i32, [vp, i32, C.c_char_p]),
    "roc_host_set_tensor": (i32, [vp, i32, vp, i32]),
    "roc_host_get_tensor": (i32, [vp, i32, vp, i32]),
    "roc_host_set_labels": (i32, [vp, i32, vp]),
    "roc_host_tensor_shape": (i32, [vp, i32, vp]),
    "roc_host_tensor_ptr": (vp, [vp, i32, i32]),
    "roc_host_num_parameters": (i32, [vp]),
    "roc_host_parameter_shape": (i32, [vp, i32, vp]),
    "roc_host_get_parameter": (i32, [vp, i32, vp, i32]),
    "roc_host_set_parameter": (i32, [vp, i32, vp]),
    "roc_host_train_mode": (i32, [vp]),
    "roc_host_infer_mode": (i32, [vp]),
    "roc_host_zero_gradients": (i32, [vp]),
    "roc_host_forward": (i32, [vp]),
    "roc_host_backward": (i32, [vp]),
    "roc_host_update": (i32, [vp]),
    "roc_host_train_epoch": (i32, [vp]),
    "roc_host_metrics": (i32, [vp, vp]),
    "roc_host_profile_sg": (i32, [vp, i32]),
    "roc_host_profile_sg_read": (i32, [vp, i32, vp, vp]),
    "roc_host_sg_arg": (i32, [vp, i32, vp]),
    "roc_host_gat_lse": (i32, [vp, i32, vp]),
    "roc_host_gat_param": (i32, [vp, i32]),
}

for _name, (_res, _args) in PROTOTYPES.items():
    _f = getattr(lib, _name)   # AttributeError here = the library does not export a declared symbol
    _f.restype = _res
    _f.argtypes = _args


def check(rc, what=""):
    if rc != 0:
        names = {-1: "ROC_ERR_INVALID", -2: "ROC_ERR_UNSUPPORTED", -3: "ROC_ERR_NOMEM", -4: "ROC_ERR_NO_DEVICE",
                 -5: "ROC_ERR_IO"}
        raise RocError("%s failed: %s" % (what or "roc call", names.get(rc, "cudaError %d" % rc)))


def device_count():
    return lib.roc_device_count()


def require_device():
    if device_count() <= 0:
        raise RocError("roc_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
