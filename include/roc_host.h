/*
 * roc_host.h — C ABI over the C++ host (roc_gnn.h) so non-C++ callers (the
 * Python mirror in roc_b200/, bench.py, tests) can build and train a model.
 * One roc_host per process / GPU.  Mirrors the public surface of Model
 * (gnn.h:162-203): same op-builder calls, same train-loop calls.  Tensors are
 * referred to by small integer handles.  Unless stated, return 0 on success;
 * host-side precondition failures abort the process like the reference's
 * asserts do (cuda_helper.h:6-12).
 */
#ifndef ROC_HOST_H_
#define ROC_HOST_H_
#include <stdint.h>
#include "roc_b200.h"
#ifdef __cplusplus
extern "C" {
#endif

typedef struct roc_host roc_host;

/* device: CUDA ordinal; myPart/numParts: this process's vertex-range partition. */
roc_host* roc_host_create(int device, int myPart, int numParts);
void roc_host_destroy(roc_host* h);
int roc_host_nccl_unique_id(unsigned char id[128]);
int roc_host_nccl_init(roc_host* h, const unsigned char id[128]);
int roc_host_synchronize(roc_host* h);
/* the host's CUDA stream (a cudaStream_t), so callers can record events on it */
void* roc_host_stream(roc_host* h);

/* Graph (gnn.cc:751-872): from <prefix>.add_self_edge.lux, or from host arrays. */
int roc_host_graph_from_lux(roc_host* h, const char* prefix);
int roc_host_graph_from_arrays(roc_host* h, uint32_t numNodes, uint64_t numEdges,
                               const uint64_t* host_rowEnd, const uint32_t* host_colSrc);
/* out[0..5] = numNodes, numEdges(lo), rowLeft, rowRight, colLeft, colRight as u64 */
int roc_host_graph_info(roc_host* h, uint64_t out[6]);
const roc_sg_plan* roc_host_graph_plan(roc_host* h);

/* Model builder — returns a tensor handle (>= 0). */
int roc_host_create_node_tensor(roc_host* h, int hidden, int is_int);
int roc_host_dropout(roc_host* h, int t, float rate, int seed);
int roc_host_linear(roc_host* h, int t, int outDim, int activation);
int roc_host_indegree_norm(roc_host* h, int t);
int roc_host_scatter_gather(roc_host* h, int t);
/* Model::scatter_gather(t, aggr) with aggr = ROC_AGGR_AVG | _MAX | _MIN | _SUM (roc_b200.h). */
int roc_host_scatter_gather_aggr(roc_host* h, int t, int aggr);
/* Model::graph_attention(t, heads, slope): GAT with `heads` heads over tensor t (roc_b200.h's roc_gat_*). */
int roc_host_graph_attention(roc_host* h, int t, int heads, float slope);
int roc_host_relu(roc_host* h, int t);
int roc_host_sigmoid(roc_host* h, int t);
int roc_host_add(roc_host* h, int a, int b);
int roc_host_softmax_cross_entropy(roc_host* h, int logits, int labels, int mask);
/* AdamOptimizer(&model, lr) + set_weight_decay; call after all linear() calls. */
int roc_host_adam(roc_host* h, double lr, double weight_decay);
int roc_host_set_lr(roc_host* h, double lr);
double roc_host_get_lr(roc_host* h);
void roc_host_srand(unsigned seed);               /* std::srand(config.seed), gnn.cc:56 */
int roc_host_set_fusion(roc_host* h, int on);
int roc_host_init(roc_host* h);

/* data: dense host buffers of this partition's rows ([rows][hidden]) */
int roc_host_load_features(roc_host* h, int t, const char* prefix);
int roc_host_load_labels(roc_host* h, int t, const char* prefix);
int roc_host_load_train_mask(roc_host* h, int t, const char* prefix);
int roc_host_set_tensor(roc_host* h, int t, const void* host, int grad);
int roc_host_get_tensor(roc_host* h, int t, void* host, int grad);
int roc_host_set_labels(roc_host* h, int t, const int32_t* host_class_idx);
int roc_host_tensor_shape(roc_host* h, int t, int64_t out[3]);   /* rows, hidden, ld */
void* roc_host_tensor_ptr(roc_host* h, int t, int grad);          /* device pointer */
int roc_host_num_parameters(roc_host* h);
int roc_host_parameter_shape(roc_host* h, int p, int64_t out[2]); /* inDim, outDim */
int roc_host_get_parameter(roc_host* h, int p, float* host, int which); /* 0 W, 1 dW, 2 m, 3 v */
int roc_host_set_parameter(roc_host* h, int p, const float* host);

/* train loop (gnn.cc:99-111) */
int roc_host_train_mode(roc_host* h);
int roc_host_infer_mode(roc_host* h);
int roc_host_zero_gradients(roc_host* h);
int roc_host_forward(roc_host* h);
int roc_host_backward(roc_host* h);
int roc_host_update(roc_host* h);
/* one full training epoch: zero_gradients; forward; backward; update */
int roc_host_train_epoch(roc_host* h);
int roc_host_metrics(roc_host* h, roc_perf_metrics* out);
/* Per-launch device time of the ScatterGather kernels (CUDA events on the host's
 * stream around each roc_sg_forward_planned): enable, run steps, read {H, ms}. */
int roc_host_profile_sg(roc_host* h, int on);
int roc_host_profile_sg_read(roc_host* h, int maxEntries, int* H, float* ms);
/* Test hook: the winner ids ([rows][hidden] u32, global vertex ids, 0xFFFFFFFF for degree-0 rows) of the
 * MAX / MIN scatter_gather whose output is tensor `outTensor`, for this partition's own rows, as the latest
 * training-mode forward left them.  -1 if that tensor is not the output of such an op. */
int roc_host_sg_arg(roc_host* h, int outTensor, uint32_t* host);
/* Test hooks of the graph_attention whose output is tensor `outTensor` (-1 if there is none): its lse
 * ([rows][heads], own rows, as the latest forward left them), and the parameter index of its [2][H] att weight. */
int roc_host_gat_lse(roc_host* h, int outTensor, float* host);
int roc_host_gat_param(roc_host* h, int outTensor);

#ifdef __cplusplus
}
#endif
#endif
