// capi.cc — roc_host_* : C ABI over the C++ host for Python / bench / tests.
#include <cstring>

#include "host_internal.h"
#include "roc_host.h"

using namespace roc::host;

struct roc_host {
  Runtime* rt = nullptr;
  Graph* graph = nullptr;
  Model* model = nullptr;
  AdamOptimizer* adam = nullptr;
  std::vector<Tensor> tensors;
  Config config;
  int push(const Tensor& t) { tensors.push_back(t); return (int)tensors.size() - 1; }
  const Tensor& at(int i) const {
    if (i < 0 || i >= (int)tensors.size()) ROC_FATAL("roc_host: bad tensor handle");
    return tensors[(size_t)i];
  }
  Model& m() {
    if (!model) {
      if (!graph) ROC_FATAL("roc_host: graph not set");
      model = new Model(*graph, rt->context(), rt);
      model->printMetrics = false;
    }
    return *model;
  }
};

extern "C" {

roc_host* roc_host_create(int device, int myPart, int numParts) {
  roc_host* h = new roc_host();
  h->rt = new Runtime(device, myPart, numParts);
  return h;
}

void roc_host_destroy(roc_host* h) {
  if (!h) return;
  if (h->rt) h->rt->synchronize();
  if (h->graph && h->graph->plan) roc_sg_plan_destroy(h->graph->plan);
  if (h->graph && h->graph->halo) roc_halo_destroy(h->graph->halo);
  if (h->model) { for (GnnOp* op : h->model->layers) delete op; }
  delete h->adam;
  delete h->model;
  delete h->graph;
  delete h->rt;
  delete h;
}

int roc_host_nccl_unique_id(unsigned char id[128]) { return Runtime::nccl_unique_id(id) ? 0 : -1; }
int roc_host_nccl_init(roc_host* h, const unsigned char id[128]) { return h->rt->init_nccl(id) ? 0 : -1; }
int roc_host_synchronize(roc_host* h) { h->rt->synchronize(); return 0; }
void* roc_host_stream(roc_host* h) { return (void*)h->rt->impl->stream; }

int roc_host_graph_from_lux(roc_host* h, const char* prefix) {
  Config c;
  c.filename = prefix;
  c.totalGPUs = h->rt->impl->numParts;
  h->config = c;
  h->graph = new Graph(h->rt->context(), h->rt, c);
  return 0;
}

int roc_host_graph_from_arrays(roc_host* h, uint32_t numNodes, uint64_t numEdges, const uint64_t* host_rowEnd,
                               const uint32_t* host_colSrc) {
  h->graph = new Graph(h->rt->context(), h->rt, numNodes, numEdges, host_rowEnd, host_colSrc);
  return 0;
}

int roc_host_graph_info(roc_host* h, uint64_t out[6]) {
  if (!h->graph) return -1;
  out[0] = h->graph->numNodes; out[1] = h->graph->numEdges; out[2] = h->graph->rowLeft;
  out[3] = h->graph->rowRight; out[4] = h->graph->colLeft; out[5] = h->graph->colRight;
  return 0;
}

const roc_sg_plan* roc_host_graph_plan(roc_host* h) { return h->graph ? h->graph->plan : nullptr; }

int roc_host_create_node_tensor(roc_host* h, int hidden, int is_int) {
  return h->push(is_int ? h->m().create_node_tensor<int>(hidden) : h->m().create_node_tensor<DATATYPE>(hidden));
}
int roc_host_dropout(roc_host* h, int t, float rate, int seed) { return h->push(h->m().dropout(h->at(t), rate, seed)); }
int roc_host_linear(roc_host* h, int t, int outDim, int activation) {
  return h->push(h->m().linear(h->at(t), outDim, (ActiMode)activation));
}
int roc_host_indegree_norm(roc_host* h, int t) { return h->push(h->m().indegree_norm(h->at(t))); }
int roc_host_scatter_gather(roc_host* h, int t) { return h->push(h->m().scatter_gather(h->at(t))); }
int roc_host_scatter_gather_aggr(roc_host* h, int t, int aggr) {
  if (aggr != ROC_AGGR_AVG && aggr != ROC_AGGR_MAX && aggr != ROC_AGGR_MIN && aggr != ROC_AGGR_SUM)
    ROC_FATAL("roc_host_scatter_gather_aggr: unknown aggregator");
  return h->push(h->m().scatter_gather(h->at(t), (AggrType)aggr));
}
int roc_host_graph_attention(roc_host* h, int t, int heads, float slope) {
  return h->push(h->m().graph_attention(h->at(t), heads, slope));
}
int roc_host_relu(roc_host* h, int t) { return h->push(h->m().relu(h->at(t))); }
int roc_host_sigmoid(roc_host* h, int t) { return h->push(h->m().sigmoid(h->at(t))); }
int roc_host_add(roc_host* h, int a, int b) { return h->push(h->m().add(h->at(a), h->at(b))); }
int roc_host_softmax_cross_entropy(roc_host* h, int logits, int labels, int mask) {
  h->m().softmax_cross_entropy(h->at(logits), h->at(labels), h->at(mask));
  return 0;
}

int roc_host_adam(roc_host* h, double lr, double weight_decay) {
  h->adam = new AdamOptimizer(&h->m(), lr);
  h->adam->set_weight_decay(weight_decay);
  h->m().optimizer = h->adam;
  return 0;
}
int roc_host_set_lr(roc_host* h, double lr) { if (!h->adam) return -1; h->adam->alpha = lr; return 0; }
double roc_host_get_lr(roc_host* h) { return h->adam ? h->adam->alpha : 0.0; }
void roc_host_srand(unsigned seed) { std::srand(seed); }
int roc_host_set_fusion(roc_host* h, int on) { h->m().set_fusion(on != 0); return 0; }
int roc_host_init(roc_host* h) { return h->m().init(h->config) ? 0 : -1; }

int roc_host_load_features(roc_host* h, int t, const char* prefix) { h->m().load_features(h->at(t), prefix); return 0; }
int roc_host_load_labels(roc_host* h, int t, const char* prefix) { h->m().load_labels(h->at(t), prefix); return 0; }
int roc_host_load_train_mask(roc_host* h, int t, const char* prefix) { h->m().load_train_mask(h->at(t), prefix); return 0; }
int roc_host_set_tensor(roc_host* h, int t, const void* host, int grad) { h->m().set_tensor(h->at(t), host, grad != 0); return 0; }
int roc_host_get_tensor(roc_host* h, int t, void* host, int grad) { h->m().get_tensor(h->at(t), host, grad != 0); return 0; }
int roc_host_set_labels(roc_host* h, int t, const int32_t* cls) { h->m().set_labels(h->at(t), cls); return 0; }

int roc_host_tensor_shape(roc_host* h, int t, int64_t out[3]) {
  TensorImpl& x = h->rt->impl->t(h->at(t).region);
  out[0] = x.rows; out[1] = x.H; out[2] = x.ld;
  return 0;
}
void* roc_host_tensor_ptr(roc_host* h, int t, int grad) {
  return grad ? (void*)h->rt->impl->grad(h->at(t).region) : (void*)h->rt->impl->data(h->at(t).region);
}

int roc_host_num_parameters(roc_host* h) { return (int)h->m().parameters.size(); }
int roc_host_parameter_shape(roc_host* h, int p, int64_t out[2]) {
  const Tensor& w = h->m().parameters[(size_t)p];
  out[0] = (int64_t)w.dims[0]; out[1] = (int64_t)w.dims[1];
  return 0;
}
int roc_host_get_parameter(roc_host* h, int p, float* host, int which) {
  RuntimeImpl* rt = h->rt->impl;
  const Tensor& w = h->m().parameters[(size_t)p];
  size_t n = (size_t)w.dims[0] * w.dims[1];
  const float* src = nullptr;
  if (which == 0) src = rt->data(w.region);
  else if (which == 1) src = rt->grad(w.region);
  else {
    if (!h->adam) return -1;
    src = rt->data(which == 2 ? h->adam->m_regions[w.region] : h->adam->v_regions[w.region]);
  }
  ROC_CHECK(cudaMemcpyAsync(host, src, n * sizeof(float), cudaMemcpyDeviceToHost, rt->stream));
  ROC_CHECK(cudaStreamSynchronize(rt->stream));
  return 0;
}
int roc_host_set_parameter(roc_host* h, int p, const float* host) {
  RuntimeImpl* rt = h->rt->impl;
  const Tensor& w = h->m().parameters[(size_t)p];
  size_t n = (size_t)w.dims[0] * w.dims[1];
  ROC_CHECK(cudaMemcpyAsync(rt->data(w.region), host, n * sizeof(float), cudaMemcpyHostToDevice, rt->stream));
  ROC_CHECK(cudaStreamSynchronize(rt->stream));
  return 0;
}

int roc_host_train_mode(roc_host* h) { h->m().train_mode(); return 0; }
int roc_host_infer_mode(roc_host* h) { h->m().infer_mode(); return 0; }
int roc_host_zero_gradients(roc_host* h) { h->m().zero_gradients(); return 0; }
int roc_host_forward(roc_host* h) { h->m().forward(); return 0; }
int roc_host_backward(roc_host* h) { h->m().backward(); return 0; }
int roc_host_update(roc_host* h) { h->m().update(); return 0; }
int roc_host_train_epoch(roc_host* h) {
  Model& m = h->m();
  m.train_mode();
  m.zero_gradients();
  m.forward();
  m.backward();
  m.update();
  return 0;
}
int roc_host_profile_sg(roc_host* h, int on) {
  RuntimeImpl* rt = h->rt->impl;
  ROC_CHECK(cudaStreamSynchronize(rt->stream));
  for (auto& t : rt->sgTimings) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
  rt->sgTimings.clear();
  rt->profileSg = on != 0;
  return 0;
}
int roc_host_profile_sg_read(roc_host* h, int maxEntries, int* H, float* ms) {
  RuntimeImpl* rt = h->rt->impl;
  ROC_CHECK(cudaStreamSynchronize(rt->stream));
  int n = 0;
  for (auto& t : rt->sgTimings) {
    if (n >= maxEntries) break;
    float e = 0.f;
    ROC_CHECK(cudaEventElapsedTime(&e, t.a, t.b));
    H[n] = t.H; ms[n] = e; n++;
  }
  return n;
}
int roc_host_sg_arg(roc_host* h, int outTensor, uint32_t* host) {
  const int region = h->at(outTensor).region;
  for (GnnOp* op : h->m().layers) {
    const ScatterGather* sg = dynamic_cast<const ScatterGather*>(op);
    if (!sg || sg->argRegion < 0 || sg->outputs[0].region != region) continue;
    RuntimeImpl* rt = h->rt->impl;
    const TensorImpl& a = rt->t(sg->argRegion);
    ROC_CHECK(cudaMemcpy2DAsync(host, (size_t)a.H * 4, rt->data(sg->argRegion), (size_t)a.ld * 4, (size_t)a.H * 4,
                                (size_t)a.rows, cudaMemcpyDeviceToHost, rt->stream));
    ROC_CHECK(cudaStreamSynchronize(rt->stream));
    return 0;
  }
  return -1;
}
static const GraphAttention* gat_of(roc_host* h, int outTensor) {
  const int region = h->at(outTensor).region;
  for (GnnOp* op : h->m().layers) {
    const GraphAttention* ga = dynamic_cast<const GraphAttention*>(op);
    if (ga && ga->outputs[0].region == region) return ga;
  }
  return nullptr;
}
int roc_host_gat_lse(roc_host* h, int outTensor, float* host) {
  const GraphAttention* ga = gat_of(h, outTensor);
  if (!ga) return -1;
  RuntimeImpl* rt = h->rt->impl;
  const TensorImpl& b = rt->t(ga->bstRegion);
  ROC_CHECK(cudaMemcpy2DAsync(host, (size_t)ga->heads * 4, rt->data(ga->bstRegion), (size_t)b.ld * 4,
                              (size_t)ga->heads * 4, (size_t)b.rows, cudaMemcpyDeviceToHost, rt->stream));
  ROC_CHECK(cudaStreamSynchronize(rt->stream));
  return 0;
}
int roc_host_gat_param(roc_host* h, int outTensor) {
  const GraphAttention* ga = gat_of(h, outTensor);
  if (!ga) return -1;
  const std::vector<Tensor>& ps = h->m().parameters;
  for (size_t p = 0; p < ps.size(); p++)
    if (ps[p].region == ga->weight.region) return (int)p;
  return -1;
}
int roc_host_metrics(roc_host* h, roc_perf_metrics* out) { *out = h->m().last_metrics(); return 0; }

}  // extern "C"
