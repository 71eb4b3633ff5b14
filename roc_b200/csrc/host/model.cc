// model.cc — Model, the op classes, AdamOptimizer, initializers, dataset loaders.
// Mirrors gnn.cc:433-749 and the per-op .cc files of the reference; each op's
// forward/backward enqueues C-ABI kernels (roc_b200.h) on the Runtime's stream
// instead of launching a Legion index task.
#include <curand.h>
#include <algorithm>
#include <cmath>
#include <cstring>
#include <fstream>
#include <set>
#include <sstream>

#include "host_internal.h"

using namespace roc::host;

// roc_softmax_xent_bwd_idx is declared in roc_b200.h

// ------------------------------------------------------------------ GnnOp ---
// gnn.cc:433-465
GnnOp::GnnOp(const Tensor& _input) : numInputs(1), numOutputs(0), fusedInto(-1) {
  inputs[0] = _input;
  trainableInputs[0] = true;
  resetInputGrads[0] = true;
}
GnnOp::GnnOp(const Tensor& _input1, const Tensor& _input2) : numInputs(2), numOutputs(0), fusedInto(-1) {
  inputs[0] = _input1; inputs[1] = _input2;
  for (int i = 0; i < 2; i++) { trainableInputs[i] = true; resetInputGrads[i] = true; }
}
GnnOp::GnnOp(const Tensor& _input1, const Tensor& _input2, const Tensor& _input3)
    : numInputs(3), numOutputs(0), fusedInto(-1) {
  inputs[0] = _input1; inputs[1] = _input2; inputs[2] = _input3;
  for (int i = 0; i < 3; i++) { trainableInputs[i] = true; resetInputGrads[i] = true; }
}

// ------------------------------------------------------------------ Model ---
Model::Model(const Graph& _graph, Context _ctx, Runtime* _runtime)
    : mode(MD_MODE_TRAIN), myGraph(_graph), ctx(_ctx), runtime(_runtime), optimizer(NULL), epoch_num(0),
      fuse(true), printMetrics(true) {}

// gnn.cc:475-532: node tensor = [numNodes][H]; this process holds its vertex range.
template <>
Tensor Model::create_node_tensor<DATATYPE>(int _numHidden) const {
  Tensor t(Tensor::NODE_TENSOR);
  t.numDim = 2;
  t.dims[0] = _numHidden;
  t.dims[1] = myGraph.numNodes;
  t.region = ctx->new_tensor(local_rows(), _numHidden, round_up4(_numHidden), false, false);
  return t;
}
template <>
Tensor Model::create_node_tensor<int>(int _numHidden) const {
  Tensor t(Tensor::NODE_TENSOR);
  t.numDim = 2;
  t.dims[0] = _numHidden;
  t.dims[1] = myGraph.numNodes;
  t.region = ctx->new_tensor(local_rows(), _numHidden, _numHidden, true, false);
  return t;
}

// gnn.cc:591-623: weight [inDim][outDim] (dim0 = inDim fastest => W_mem[o*inDim + i]).
// The reference keeps one dW replica per GPU inside one region; here each process
// owns its replica and replicas are summed by one NCCL all-reduce (Model::update).
Tensor Model::create_weight_tensor(int _inDim, int _outDim, Initializer* initializer) const {
  Tensor w(Tensor::WEIGHT_TENSOR);
  w.numDim = 2;
  w.dims[0] = _inDim;
  w.dims[1] = _outDim;
  w.region = ctx->new_tensor(_outDim, _inDim, _inDim, false, true);
  ctx->t(w.region).requiresGrad = true;
  if (initializer == NULL) {
    GlorotUniform glorot;   // default initializer, gnn.cc:614-618
    glorot.init(this, &w);
  } else {
    initializer->init(this, &w);
  }
  return w;
}

Tensor Model::add(const Tensor& a, const Tensor& b) {
  GnnOp* op = new Element(*this, a, b, EW_TYPE_ADD);
  layers.push_back(op);
  return op->outputs[0];
}
Tensor Model::dropout(const Tensor& _input, float rate, int seed) {
  Dropout* op = new Dropout(*this, _input, rate, seed);
  op->opIndex = (int)layers.size();
  layers.push_back(op);
  return op->outputs[0];
}
Tensor Model::scatter_gather(const Tensor& _input, AggrType aggr) {
  GnnOp* op = new ScatterGather(*this, _input, aggr);
  layers.push_back(op);
  return op->outputs[0];
}
Tensor Model::graph_attention(const Tensor& _input, int heads, float negativeSlope) {
  GraphAttention* op = new GraphAttention(*this, _input, heads, negativeSlope);
  layers.push_back(op);
  parameters.push_back(op->weight);
  return op->outputs[0];
}
void Model::softmax_cross_entropy(const Tensor& logits, const Tensor& labels, const Tensor& mask) {
  layers.push_back(new SoftmaxCrossEntropy(*this, logits, labels, mask));
}
Tensor Model::indegree_norm(const Tensor& _input) {
  GnnOp* op = new InDegreeNorm(*this, _input);
  layers.push_back(op);
  return op->outputs[0];
}
Tensor Model::linear(const Tensor& _input, int outDim, ActiMode activation, Initializer* initializer) {
  Linear* op = new Linear(*this, _input, outDim, activation, initializer);
  layers.push_back(op);
  parameters.push_back(op->weight);   // linear.cc:30
  return op->outputs[0];
}
Tensor Model::relu(const Tensor& _input) {
  GnnOp* op = new Activation(*this, _input, AC_MODE_RELU);
  layers.push_back(op);
  return op->outputs[0];
}
Tensor Model::sigmoid(const Tensor& _input) {
  GnnOp* op = new Activation(*this, _input, AC_MODE_SIGMOID);
  layers.push_back(op);
  return op->outputs[0];
}

void Model::train_mode(void) { mode = MD_MODE_TRAIN; }
void Model::infer_mode(void) { mode = MD_MODE_INFER; }

namespace {
struct Wiring {
  std::map<int, int> producer;    // region -> layer index
  std::map<int, int> consumers;   // region -> number of consuming op inputs
  std::map<int, int> consumerOp;  // region -> a consuming layer index
};
Wiring wire(const std::vector<GnnOp*>& layers) {
  Wiring w;
  for (size_t l = 0; l < layers.size(); l++) {
    for (int j = 0; j < layers[l]->numOutputs; j++) w.producer[layers[l]->outputs[j].region] = (int)l;
    for (int j = 0; j < layers[l]->numInputs; j++) {
      int r = layers[l]->inputs[j].region;
      if (r < 0) continue;
      w.consumers[r] += 1;
      w.consumerOp[r] = (int)l;
    }
  }
  return w;
}
template <typename T>
T* as(GnnOp* op) { return dynamic_cast<T*>(op); }

// The tensors an op's gathers read at halo rows (multi-GPU): region, data or grad twin.  Backward reads are listed
// only when the op's backward runs.
struct HaloRead { int region; bool grad; };
std::vector<HaloRead> halo_reads(RuntimeImpl* rt, GnnOp* op) {
  std::vector<HaloRead> r;
  if (const ScatterGather* sg = as<ScatterGather>(op)) {
    r.push_back({sg->inputs[0].region, false});
    if (rt->t(sg->inputs[0].region).requiresGrad) {
      // the backward gathers dOut (SUM, MAX, MIN) or D^-1 dOut (AVG); MAX / MIN also the winner ids
      if (sg->scratch >= 0) r.push_back({sg->scratch, false});
      else r.push_back({sg->outputs[0].region, true});
      if (sg->argRegion >= 0) r.push_back({sg->argRegion, false});
    }
  } else if (const GraphAttention* ga = as<GraphAttention>(op)) {
    // forward: h and s_src / s_dst; backward (always: the op has a parameter): dOut and lse / c.  The backward also
    // reads h at halo rows, but those rows still hold this step's values: only the forward's exchange writes them.
    r.push_back({ga->inputs[0].region, false});
    r.push_back({ga->attRegion, false});
    r.push_back({ga->outputs[0].region, true});
    r.push_back({ga->bstRegion, false});
  }
  return r;
}
}  // namespace

// gnn.cc:625-673.  No graph loading / ResourceManager creation left to do here
// (Graph's constructor already built the device CSR); what remains is sizing the
// shared scratch, deciding which tensors need gradients, laying the dW replicas
// out in one flat buffer and fusing the GCN aggregate block.
bool Model::init(const Config& config) {
  (void)config;
  RuntimeImpl* rt = ctx;
  myGraph.maxHidden = 0;
  for (size_t i = 0; i < layers.size(); i++) {
    for (int j = 0; j < layers[i]->numOutputs; j++)
      myGraph.maxHidden = std::max(myGraph.maxHidden, (int)layers[i]->outputs[j].dims[0]);
    for (int j = 0; j < layers[i]->numInputs; j++)
      if (layers[i]->inputs[j].numDim == 2)
        myGraph.maxHidden = std::max(myGraph.maxHidden, (int)layers[i]->inputs[j].dims[0]);
  }
  // which tensors carry gradients: anything downstream of a parameter
  for (size_t l = 0; l < layers.size(); l++) {
    GnnOp* op = layers[l];
    bool any = false;
    for (int j = 0; j < op->numInputs; j++)
      if (op->inputs[j].region >= 0) any = any || rt->t(op->inputs[j].region).requiresGrad;
    if (as<Linear>(op) || as<GraphAttention>(op)) any = true;   // ops with a parameter
    for (int j = 0; j < op->numOutputs; j++) {
      rt->t(op->outputs[j].region).requiresGrad = any;
      rt->t(op->outputs[j].region).produced = true;
    }
  }
  // flat dW buffer (one all-reduce per step instead of the reference's serial
  // replica sum, optimizer_kernel.cu:88-94)
  size_t total = 0;
  for (size_t p = 0; p < parameters.size(); p++) total += (size_t)parameters[p].dims[0] * parameters[p].dims[1];
  rt->flatGradCount = total;
  rt->flatGrad = (float*)rt->dmalloc((total ? total : 4) * sizeof(float));
  ROC_CHECK(cudaMemsetAsync(rt->flatGrad, 0, (total ? total : 4) * sizeof(float), rt->stream));
  size_t off = 0;
  for (size_t p = 0; p < parameters.size(); p++) {
    rt->t(parameters[p].region).grad = rt->flatGrad + off;
    off += (size_t)parameters[p].dims[0] * parameters[p].dims[1];
  }
  // scratch: Linear split-K workspace, SG carry slots, the gathered feature matrix
  size_t ws = 0;
  int maxSg = 0, maxArg = 0;
  for (size_t l = 0; l < layers.size(); l++) {
    if (Linear* lin = as<Linear>(layers[l]))
      ws = std::max(ws, roc_linear_bwd_workspace_bytes(local_rows(), (int)lin->weight.dims[0], (int)lin->weight.dims[1]));
    if (ScatterGather* sg = as<ScatterGather>(layers[l])) {
      maxSg = std::max(maxSg, (int)sg->inputs[0].dims[0]);
      if (sg->argRegion >= 0) {
        maxArg = std::max(maxArg, (int)sg->inputs[0].dims[0]);
        // the backward reads two tensors at halo rows; the whole-matrix all-gather has one shared buffer
        if (rt->numParts > 1 && !myGraph.halo)
          ROC_FATAL("scatter_gather(AGGR_MAX / AGGR_MIN) needs the halo exchange (unset ROC_B200_HALO=0)");
      }
    }
    if (GraphAttention* ga = as<GraphAttention>(layers[l])) {
      const int H = (int)ga->inputs[0].dims[0];
      maxSg = std::max(maxSg, H);
      ROC_CHECK(roc_gat_plan_reserve(myGraph.plan, H, ga->heads));
      // the gathers read four tensors at halo rows; the whole-matrix all-gather has one shared buffer
      if (rt->numParts > 1 && !myGraph.halo)
        ROC_FATAL("graph_attention needs the halo exchange (unset ROC_B200_HALO=0)");
    }
  }
  rt->ensure_lin_ws(ws);
  if (maxSg > 0) {
    ROC_CHECK(roc_sg_plan_reserve(myGraph.plan, maxSg));
    if (maxArg > 0) ROC_CHECK(roc_sg_plan_reserve_arg(myGraph.plan, maxArg));
    if (rt->numParts > 1 && !myGraph.halo) rt->ensure_gather((size_t)myGraph.numNodes * (size_t)round_up4(maxSg));
    if (myGraph.halo) {
      // the tensors a gather reads get the halo slab appended to their own rows.  Usually the buffer does not exist
      // yet (lazy allocation).  A tensor the script already filled — e.g. an SGC-style scatter_gather(input) after
      // load_features / set_tensor, which the reference's script order (gnn.cc:72-74) allows — is re-homed with the
      // halo rows behind its own.
      rt->ensure_sendbuf((myGraph.numSendRows ? myGraph.numSendRows : 1) * (size_t)round_up4(maxSg));
      for (size_t l = 0; l < layers.size(); l++)
        for (const HaloRead& r : halo_reads(rt, layers[l])) rt->grow_halo(rt->t(r.region), r.grad, myGraph.numHalo);
      // Exchange by peer writes (roc_push_rows): the slabs exist now and every partition maps the others' copies.
      // ROC_B200_HALO=nccl keeps the staged-rows + NCCL all-to-all-v exchange (cross-check; also the fallback when
      // CUDA IPC is not available between the devices).
      const char* he = getenv("ROC_B200_HALO");
      rt->p2p = !(he && he[0] == 'n') && rt->numParts <= ROC_MAX_PEERS;
      // Two ways to fill the peers' slabs, chosen by measurement (r2 runs m5-m8, ms/step at 2 / 4 / 8 GPUs):
      // pack + one DMA copy per peer 20.8 / - / 33.1 (the copy engines do not keep 7 peer copies busy), the SM
      // kernel roc_push_rows 21.2 / 24.8 / 29.0, staged rows + NCCL 21.8 / 26.0 / 30.7.
      // ROC_B200_HALO=push | ce forces one.
      rt->p2pCopyEngines = (he && he[0] == 'c') ? true : (he && he[0] == 'p') ? false : rt->numParts == 2;
      for (size_t l = 0; l < layers.size() && rt->p2p; l++) {
        for (const HaloRead& r : halo_reads(rt, layers[l])) {
          if (r.grad) rt->grad(r.region); else rt->data(r.region);
          if (!rt->open_peers(rt->t(r.region), r.grad)) { rt->p2p = false; break; }
        }
      }
      if (rt->myPart == 0)
        fprintf(stderr, "[roc_b200] halo exchange: %s\n",
                !rt->p2p ? "staged rows + NCCL all-to-all-v"
                : rt->p2pCopyEngines ? "pack + copy-engine writes into the peers' slabs (CUDA IPC over NVLink), pipelined with the producer"
                                     : "roc_push_rows peer writes (CUDA IPC over NVLink), pipelined with the producer");
    }
  }
  // ---- fusion of  linear -> indegree_norm -> scatter_gather -> indegree_norm -> relu  (gnn.cc:81-85)
  if (fuse) {
    Wiring w = wire(layers);
    for (size_t l = 0; l < layers.size(); l++) {
      ScatterGather* sg = as<ScatterGather>(layers[l]);
      if (!sg || sg->aggr != AGGR_SUM) continue;   // nothing fuses into or across another aggregator
      // upstream: Linear(NONE) -> InDegreeNorm -> SG, each feeding only the next
      int rin = sg->inputs[0].region;
      if (w.producer.count(rin) && w.consumers[rin] == 1) {
        InDegreeNorm* n1 = as<InDegreeNorm>(layers[w.producer[rin]]);
        if (n1 && n1->fusedInto < 0) {
          int rl = n1->inputs[0].region;
          if (w.producer.count(rl) && w.consumers[rl] == 1) {
            Linear* lin = as<Linear>(layers[w.producer[rl]]);
            if (lin && lin->activation == AC_MODE_NONE && lin->fwdOut < 0) {
              lin->flags |= ROC_LINEAR_NORM_EPILOGUE;
              lin->fwdOut = n1->outputs[0].region;       // linear writes the normalised rows
              n1->fusedInto = w.producer[rl];
              sg->bwdEpilogue = ROC_SG_EPI_NORM;          // SG backward writes d(linear out)
              sg->bwdOut = lin->outputs[0].region;
            }
          }
        }
      }
      // downstream: SG -> InDegreeNorm -> [relu]
      int rout = sg->outputs[0].region;
      if (w.consumers[rout] == 1) {
        InDegreeNorm* n2 = as<InDegreeNorm>(layers[w.consumerOp[rout]]);
        if (n2 && n2->fusedInto < 0) {
          sg->epilogue = ROC_SG_EPI_NORM;
          sg->fwdOut = n2->outputs[0].region;
          n2->fusedInto = (int)l;   // forward only; its backward kernel still runs
          int rn = n2->outputs[0].region;
          if (w.consumers[rn] == 1) {
            Activation* act = as<Activation>(layers[w.consumerOp[rn]]);
            if (act && act->actiMode == AC_MODE_RELU && act->fusedInto < 0) {
              sg->epilogue |= ROC_SG_EPI_RELU;
              sg->fwdOut = act->outputs[0].region;
              act->fusedInto = (int)l;
              n2->reluMaskOf = act->outputs[0].region;   // backward: relu mask + norm in one pass
              n2->bwdIn = act->outputs[0].region;
            }
          }
        }
      }
    }
  }
  // ---- fusion of  dropout -> linear  (gnn.cc:79-81, 86-88): the dropout output feeds only the linear
  if (fuse) {
    Wiring w = wire(layers);
    for (size_t l = 0; l < layers.size(); l++) {
      Dropout* d = as<Dropout>(layers[l]);
      if (!d || d->fusedInto >= 0) continue;
      const int ro = d->outputs[0].region;
      if (w.consumers[ro] != 1) continue;
      Linear* lin = as<Linear>(layers[w.consumerOp[ro]]);
      if (!lin || lin->dropOp >= 0 || lin->inputs[0].region != ro) continue;
      lin->dropOp = (int)l;
      d->fusedInto = w.consumerOp[ro];
    }
  }
  // ---- backward-only fusions into epilogues
  if (fuse) {
    Wiring w = wire(layers);
    for (size_t l = 0; l < layers.size(); l++) {
      // (a) ... -> indegree_norm -> softmax_cross_entropy: the softmax kernel divides the logits'
      //     gradient by sqrt(deg) and writes it where the norm's input gradient lives
      if (SoftmaxCrossEntropy* sce = as<SoftmaxCrossEntropy>(layers[l])) {
        const int rz = sce->inputs[0].region;
        if (!w.producer.count(rz) || w.consumers[rz] != 1) continue;
        InDegreeNorm* n = as<InDegreeNorm>(layers[w.producer[rz]]);
        if (!n || n->bwdFused || n->reluMaskOf >= 0 || n->bwdIn >= 0) continue;
        if (n->fusedInto >= 0 && as<Linear>(layers[(size_t)n->fusedInto])) continue;   // handled by the SG epilogue
        if (!rt->t(n->inputs[0].region).requiresGrad) continue;
        sce->gradOut = n->inputs[0].region;
        n->bwdFused = true;
        continue;
      }
      // (b) indegree_norm -> relu -> [dropout ->] linear: the linear's dX epilogue applies the dropout
      //     backward, the relu mask and the norm, and writes the norm's input gradient directly
      Linear* lin = as<Linear>(layers[l]);
      if (!lin || lin->dxOut >= 0) continue;
      const int rin = lin->dropOp >= 0 ? layers[(size_t)lin->dropOp]->inputs[0].region : lin->inputs[0].region;
      if (!rt->t(rin).requiresGrad || !w.producer.count(rin) || w.consumers[rin] != 1) continue;
      Activation* act = as<Activation>(layers[w.producer[rin]]);
      if (!act || act->actiMode != AC_MODE_RELU || act->fusedInto < 0) continue;
      const int rn = act->inputs[0].region;
      if (!w.producer.count(rn)) continue;
      InDegreeNorm* n = as<InDegreeNorm>(layers[w.producer[rn]]);
      if (!n || n->bwdFused || n->reluMaskOf != rin || n->bwdIn != rin) continue;
      lin->dxReluOf = rin;
      lin->dxNorm = true;
      lin->dxOut = n->inputs[0].region;
      n->bwdFused = true;
    }
  }
  for (size_t l = 0; l < layers.size(); l++) layers[l]->init(*this);
  rt->opNames.clear();
  for (size_t l = 0; l < layers.size(); l++) {
    const char* nm = as<ScatterGather>(layers[l]) ? "scatter_gather" : as<GraphAttention>(layers[l]) ? "graph_attention" :
                     as<Linear>(layers[l]) ? "linear" :
                     as<InDegreeNorm>(layers[l]) ? "indegree_norm" : as<Activation>(layers[l]) ? "activation" :
                     as<Dropout>(layers[l]) ? "dropout" : as<Element>(layers[l]) ? "add" :
                     as<SoftmaxCrossEntropy>(layers[l]) ? "softmax_cross_entropy" : "op";
    rt->opNames.push_back(std::string(nm) + (layers[l]->fusedInto >= 0 ? " (fused)" : ""));
  }
  ROC_CHECK(cudaStreamSynchronize(rt->stream));
  return true;
}

// gnn.cc:696-700
void Model::forward(void) {
  if (mode == MD_MODE_TRAIN) ctx->trainStep += 1;
  for (size_t l = 0; l < layers.size(); l++) {
    ctx->op_begin((int)l, 0);
    layers[l]->forward(*this);
    ctx->op_end();
  }
}

// gnn.cc:702-716
void Model::backward(void) {
  std::set<int> resetedInputGrads;
  for (int l = (int)layers.size() - 1; l >= 0; l--) {
    for (int i = 0; i < layers[l]->numInputs; i++) {
      int r = layers[l]->inputs[i].region;
      if (resetedInputGrads.find(r) == resetedInputGrads.end()) {
        resetedInputGrads.insert(r);
        layers[l]->resetInputGrads[i] = true;
      } else {
        // This input's gradients has been reseted by other layers
        layers[l]->resetInputGrads[i] = false;
      }
    }
    ctx->op_begin(l, 1);
    layers[l]->backward(*this);
    ctx->op_end();
  }
}

// gnn.cc:718-724 (+ the replica sum of optimizer_kernel.cu:88-94 as one all-reduce)
void Model::update(void) {
  RuntimeImpl* rt = ctx;
  rt->op_begin(-1, 2);
  optimizer->next();
  if (rt->numParts > 1 && rt->flatGradCount) {
    ROC_ASSERT(rt->commReady);
    ROC_CHECK(rt->comm.allreduce_sum(rt->flatGrad, rt->flatGradCount, rt->stream));
  }
  for (int p = (int)parameters.size() - 1; p >= 0; p--) optimizer->update(&parameters[p]);
  rt->op_end();
}

// gnn.cc:726-739
void Model::zero_gradients(void) {
  RuntimeImpl* rt = ctx;
  if (rt->flatGradCount)
    ROC_CHECK(cudaMemsetAsync(rt->flatGrad, 0, rt->flatGradCount * sizeof(float), rt->stream));
}

void Model::set_tensor(const Tensor& t, const void* host, bool grad) {
  RuntimeImpl* rt = ctx;
  TensorImpl& x = rt->t(t.region);
  float* dst = grad ? rt->grad(t.region) : rt->data(t.region);
  if (x.ld == x.H || x.isInt) {
    ROC_CHECK(cudaMemcpyAsync(dst, host, (size_t)x.rows * x.H * 4, cudaMemcpyHostToDevice, rt->stream));
  } else {
    // Dense host rows -> padded device rows.  A strided cudaMemcpy2D of 2.4 KB rows runs at
    // ~17 GB/s; contiguous chunks into a staging buffer run at PCIe speed and the re-pitch
    // is a device copy at HBM speed (r1 run 4: 10.1 GB upload 600 ms -> ~190 ms).
    const int64_t chunkRows = std::max<int64_t>(1, (int64_t)(64u << 20) / x.H);   // ~256 MB of floats
    rt->ensure_staging((size_t)std::min<int64_t>(chunkRows, x.rows) * x.H * sizeof(float));
    const float* h = static_cast<const float*>(host);
    for (int64_t r0 = 0; r0 < x.rows; r0 += chunkRows) {
      const int64_t nr = std::min<int64_t>(chunkRows, x.rows - r0);
      ROC_CHECK(cudaMemcpyAsync(rt->staging, h + r0 * x.H, (size_t)nr * x.H * 4, cudaMemcpyHostToDevice, rt->stream));
      ROC_CHECK(roc_copy2d(nr, x.H, (const float*)rt->staging, x.H, dst + r0 * x.ld, x.ld, rt->stream));
    }
  }
  ROC_CHECK(cudaStreamSynchronize(rt->stream));
}

void Model::get_tensor(const Tensor& t, void* host, bool grad) const {
  RuntimeImpl* rt = ctx;
  TensorImpl& x = rt->t(t.region);
  const float* src = grad ? rt->grad(t.region) : rt->data(t.region);
  ROC_CHECK(cudaMemcpy2DAsync(host, (size_t)x.H * 4, src, (size_t)x.ld * 4, (size_t)x.H * 4, (size_t)x.rows,
                              cudaMemcpyDeviceToHost, rt->stream));
  ROC_CHECK(cudaStreamSynchronize(rt->stream));
}

void Model::set_labels(const Tensor& label, const int* host_class_idx) {
  RuntimeImpl* rt = ctx;
  TensorImpl& x = rt->t(label.region);
  if (!x.labelIdx) x.labelIdx = (int32_t*)rt->dmalloc((size_t)x.rows * sizeof(int32_t));
  for (int64_t v = 0; v < x.rows; v++) ROC_ASSERT(host_class_idx[v] >= 0 && host_class_idx[v] < x.H);  // load_task.cu:120
  ROC_CHECK(cudaMemcpyAsync(x.labelIdx, host_class_idx, (size_t)x.rows * sizeof(int32_t), cudaMemcpyHostToDevice, rt->stream));
  ROC_CHECK(cudaStreamSynchronize(rt->stream));
}

roc_perf_metrics Model::last_metrics(void) const {
  RuntimeImpl* rt = ctx;
  ROC_CHECK(cudaMemcpyAsync(&rt->h_perf, rt->d_perf, sizeof(roc_perf_metrics), cudaMemcpyDeviceToHost, rt->stream));
  ROC_CHECK(cudaStreamSynchronize(rt->stream));
  return rt->h_perf;
}

// ---- dataset loaders: load_task.cu:25-199 (formats in SURVEY Appendix C) ----
void Model::load_features(const Tensor& input, const std::string& prefix) {
  RuntimeImpl* rt = ctx;
  TensorImpl& x = rt->t(input.region);
  const int inDim = x.H;
  const size_t nloc = (size_t)x.rows;
  std::vector<float> buf(nloc * (size_t)inDim);
  std::string binFile = prefix + ".feats.bin", csvFile = prefix + ".feats.csv";
  FILE* binFin = fopen(binFile.c_str(), "rb");
  if (binFin == NULL) {
    // CSV: one line per vertex, inDim comma-separated values (load_task.cu:42-62); the
    // whole file is parsed so the .feats.bin cache can be written (load_task.cu:63-65)
    fprintf(stderr, "[roc_b200] Load features from CSV: %s\n", csvFile.c_str());
    std::ifstream csvFin(csvFile.c_str());
    if (!csvFin.good()) ROC_FATAL(("cannot open " + binFile + " or " + csvFile).c_str());
    std::vector<float> all((size_t)myGraph.numNodes * inDim);
    std::string line, word;
    for (V_ID v = 0; v < myGraph.numNodes; v++) {
      std::getline(csvFin, line);
      std::stringstream ss(line);
      int feat_cnt = 0;
      while (std::getline(ss, word, ',')) {
        ROC_ASSERT(feat_cnt < inDim);
        all[(size_t)v * inDim + feat_cnt] = std::stof(word);
        feat_cnt++;
      }
      ROC_ASSERT(feat_cnt == inDim);
    }
    if (rt->myPart == 0) {
      // the cache appears atomically (tmp + rename): another rank or job that finds <prefix>.feats.bin can read it whole
      const std::string tmpFile = binFile + ".tmp";
      FILE* binFout = fopen(tmpFile.c_str(), "wb");
      if (binFout) {
        const bool ok = fwrite(all.data(), sizeof(float), all.size(), binFout) == all.size();
        if (fclose(binFout) == 0 && ok) rename(tmpFile.c_str(), binFile.c_str());
        else remove(tmpFile.c_str());
      }
    }
    memcpy(buf.data(), all.data() + (size_t)myGraph.rowLeft * inDim, buf.size() * sizeof(float));
  } else {
    ROC_ASSERT(fseeko(binFin, (off_t)((size_t)myGraph.rowLeft * inDim * sizeof(float)), SEEK_SET) == 0);
    size_t ret = fread(buf.data(), sizeof(float), buf.size(), binFin);
    ROC_ASSERT(ret == buf.size());
    fclose(binFin);
  }
  set_tensor(input, buf.data());
}

void Model::load_labels(const Tensor& label, const std::string& prefix) {
  RuntimeImpl* rt = ctx;
  TensorImpl& x = rt->t(label.region);
  std::string filename = prefix + ".label";
  FILE* file = fopen(filename.c_str(), "r");
  if (!file) ROC_FATAL(("cannot open " + filename).c_str());
  int idx;
  for (V_ID v = 0; v < myGraph.rowLeft; v++) ROC_ASSERT(fscanf(file, "%d", &idx) == 1);
  std::vector<int> cls((size_t)x.rows);
  for (int64_t v = 0; v < x.rows; v++) {
    ROC_ASSERT(fscanf(file, "%d", &idx) == 1);
    cls[(size_t)v] = idx;
  }
  fclose(file);
  set_labels(label, cls.data());
}

void Model::load_train_mask(const Tensor& mask, const std::string& prefix) {
  RuntimeImpl* rt = ctx;
  TensorImpl& x = rt->t(mask.region);
  std::string filename = prefix + ".mask";
  std::ifstream fin(filename.c_str());
  if (!fin.good()) ROC_FATAL(("cannot open " + filename).c_str());
  std::string line;
  for (V_ID v = 0; v < myGraph.rowLeft; v++) std::getline(fin, line);
  std::vector<int> m((size_t)x.rows);
  for (int64_t v = 0; v < x.rows; v++) {
    std::getline(fin, line);
    if (line == "Train") m[(size_t)v] = MASK_TRAIN;
    else if (line == "Val") m[(size_t)v] = MASK_VAL;
    else if (line == "Test") m[(size_t)v] = MASK_TEST;
    else if (line == "None") m[(size_t)v] = MASK_NONE;
    else { printf("Unrecognized mask: %s\n", line.c_str()); ROC_ASSERT(false); }
  }
  set_tensor(mask, m.data());
}

namespace {
// Entries [selA, selB) of the block-ordered selection (or the whole requester-grouped list when blockK < 0) go to
// the peers: packed into the send buffer on commStream, then one DMA copy per peer on that peer's stream.
void exchange_rows(RuntimeImpl* rt, const Graph& g, float* local, int64_t ld, int H, std::vector<float*>& peers,
                   int blockK, bool last, int smLimit) {
  const size_t nb = g.pushBlockRow.size() - 1;
  const int P = rt->numParts, me = rt->myPart;
  ROC_CHECK(cudaEventRecord(rt->evProduced, rt->stream));
  ROC_CHECK(cudaStreamWaitEvent(rt->commStream, rt->evProduced, 0));
  if (!rt->p2pCopyEngines) {
    const size_t a = blockK < 0 ? 0 : g.pushBlockOff[(size_t)blockK], b = blockK < 0 ? g.numSendRows : g.pushBlockOff[(size_t)blockK + 1];
    if (b > a)
      ROC_CHECK(roc_push_rows((int64_t)(b - a), H, g.d_pushRows + a, g.d_pushPeer + a, g.d_pushDst + a, local, ld,
                              peers.data(), P, ld, smLimit, rt->commStream));
    if (last) ROC_CHECK(cudaEventRecord(rt->evPushed, rt->commStream));
    return;
  }
  const size_t uld = (size_t)ld;
  rt->ensure_sendbuf((g.numSendRows ? g.numSendRows : 1) * uld);
  if ((blockK <= 0) && rt->exchInFlight) {
    // the previous exchange's copies read the send buffer: the first pack of this one waits for them
    for (int q = 0; q < P; q++) if (q != me) ROC_CHECK(cudaStreamWaitEvent(rt->commStream, rt->peerDone[(size_t)q], 0));
  }
  if (blockK < 0) ROC_CHECK(roc_pack_rows((int64_t)g.numSendRows, H, g.d_sendRows, local, ld, rt->sendBuf, ld, rt->commStream));
  else ROC_CHECK(roc_pack_rows_at((int64_t)(g.packBlockOff[(size_t)blockK + 1] - g.packBlockOff[(size_t)blockK]), H,
                                  g.d_packSel + g.packBlockOff[(size_t)blockK], g.d_sendRows, local, ld, rt->sendBuf, ld,
                                  rt->commStream));
  ROC_CHECK(cudaEventRecord(rt->evPacked, rt->commStream));
  for (int q = 0; q < P; q++) {
    if (q == me) continue;
    const size_t j0 = blockK < 0 ? g.sendOffs[(size_t)q] : g.packPeerOff[(size_t)q * (nb + 1) + (size_t)blockK];
    const size_t j1 = blockK < 0 ? g.sendOffs[(size_t)q] + g.sendCounts[(size_t)q] : g.packPeerOff[(size_t)q * (nb + 1) + (size_t)blockK + 1];
    cudaStream_t ps = rt->peerStreams[(size_t)q];
    if (j1 > j0) {
      ROC_CHECK(cudaStreamWaitEvent(ps, rt->evPacked, 0));
      float* dst = peers[(size_t)q] + ((size_t)g.peerSlab0[(size_t)q] + (j0 - g.sendOffs[(size_t)q])) * uld;
      ROC_CHECK(cudaMemcpyAsync(dst, rt->sendBuf + j0 * uld, (j1 - j0) * uld * sizeof(float), cudaMemcpyDeviceToDevice, ps));
    }
    if (last) ROC_CHECK(cudaEventRecord(rt->peerDone[(size_t)q], ps));
  }
  if (last) rt->exchInFlight = true;
}
// the compute stream waits for this partition's outgoing rows, then crosses the barrier behind which every
// partition's rows have landed here
void exchange_wait(RuntimeImpl* rt) {
  if (!rt->p2pCopyEngines) ROC_CHECK(cudaStreamWaitEvent(rt->stream, rt->evPushed, 0));
  else
    for (int q = 0; q < rt->numParts; q++) if (q != rt->myPart) ROC_CHECK(cudaStreamWaitEvent(rt->stream, rt->peerDone[(size_t)q], 0));
  ROC_CHECK(rt->comm.barrier(rt->d_barrier, rt->stream));
}
}  // namespace

// ---- pipelined peer-write exchange: a producer computes its rows block by block and pushes block k's boundary
// rows (commStream) while it computes block k + 1 (compute stream, on SMs - pushSMs)
namespace {
struct PushPipe {
  RuntimeImpl* rt; const Graph* g; TensorImpl* x; bool isGrad; bool on; int prevReserve;
  // the tensor `region` (data or grad) is read by a ScatterGather through peer-mapped halo slabs?
  PushPipe(const Model& model, int region, bool grad) : rt(model.ctx), g(&model.myGraph), x(nullptr), isGrad(grad), on(false), prevReserve(0) {
    if (region < 0 || !rt->p2p || rt->numParts == 1) return;
    x = &rt->t(region);
    const std::vector<float*>& peers = grad ? x->peerGrad : x->peerData;
    on = !peers.empty() && g->pushBlockRow.size() >= 2;
    if (on && !rt->p2pCopyEngines) prevReserve = roc_set_sm_reserve(rt->pushSMs);   // the push KERNEL needs free SMs; DMA copies do not
  }
  size_t blocks() const { return on ? g->pushBlockRow.size() - 1 : 1; }
  int64_t row0(size_t k) const { return on ? (int64_t)g->pushBlockRow[k] : 0; }
  int64_t rows(size_t k, int64_t all) const { return on ? (int64_t)g->pushBlockRow[k + 1] - (int64_t)g->pushBlockRow[k] : all; }
  E_ID colLeft(size_t k) const { return on ? g->pushBlockColLeft[k] : g->colLeft; }
  // block k of `local` has been enqueued on the compute stream
  void pushed(size_t k, float* local, int64_t ld, int H) {
    if (!on) return;
    std::vector<float*>& peers = isGrad ? x->peerGrad : x->peerData;
    const bool last = k + 1 == blocks();
    exchange_rows(rt, *g, local, ld, H, peers, (int)k, last, rt->pushGridSMs >= 0 ? rt->pushGridSMs : rt->pushSMs);
    if (last) (isGrad ? x->freshGrad : x->freshData) = true;
  }
  // kernels enqueued after this may use the whole chip again
  void done() { if (on) { if (!rt->p2pCopyEngines) roc_set_sm_reserve(prevReserve); on = false; } }
  ~PushPipe() { done(); }
};
}  // namespace

// -------------------------------------------------------- ScatterGather -----
ScatterGather::ScatterGather(const Model& model, const Tensor& _input, AggrType _aggr)
    : GnnOp(_input), aggr(_aggr), scratch(-1), argRegion(-1), epilogue(0), bwdEpilogue(0), fwdOut(-1), bwdOut(-1) {
  // scattergather.cc:33-37
  ROC_ASSERT(inputs[0].type == Tensor::NODE_TENSOR);
  ROC_ASSERT(inputs[0].numDim == 2);
  ROC_ASSERT(inputs[0].dims[1] == model.myGraph.numNodes);
  ROC_ASSERT(aggr == AGGR_SUM || aggr == AGGR_AVG || aggr == AGGR_MAX || aggr == AGGR_MIN);
  numOutputs = 1;
  const int H = (int)inputs[0].dims[0];
  outputs[0] = model.create_node_tensor<DATATYPE>(H);
  // per-op buffers, allocated with the op (nothing is allocated inside a step); u32 ids live in a float tensor and
  // are only ever moved bitwise
  if (aggr == AGGR_AVG) scratch = model.ctx->new_tensor(model.local_rows(), H, round_up4(H), false, false);
  if (aggr == AGGR_MAX || aggr == AGGR_MIN) argRegion = model.ctx->new_tensor(model.local_rows(), H, round_up4(H), false, false);
}
void ScatterGather::init(const Model&) {}

namespace {
// The exchange step of ScatterGather (scattergather.cc:69-73 asks Legion for the
// WHOLE input region): all-gather every partition's slab into [numNodes][ld] so
// the kernel can index rows by global source id.  numParts == 1: no copy at all.
// Default for numParts > 1: the halo exchange — each partition packs the rows the others read
// (roc_pack_rows), one grouped NCCL send/recv moves them, and they land right behind the
// partition's own rows ([Nloc | halo] is what the remapped col indexes).  ROC_B200_HALO=0 keeps
// the whole-matrix all-gather (the reference's semantics) for comparison.
const float* gathered(const Model& model, float* local, int64_t ld, int H, TensorImpl* x, bool isGrad) {
  RuntimeImpl* rt = model.ctx;
  if (rt->numParts == 1) return local;
  ROC_ASSERT(rt->commReady);
  const Graph& g = model.myGraph;
  if (g.halo && rt->p2p) {
    // Peer writes: unless the producer already pushed its rows block by block (fresh), push them all now; then wait
    // for the pushes and cross the barrier after which every partition's rows are in this partition's slab.
    std::vector<float*>& peers = isGrad ? x->peerGrad : x->peerData;
    bool& fresh = isGrad ? x->freshGrad : x->freshData;
    ROC_ASSERT(!peers.empty());
    if (!fresh) exchange_rows(rt, g, local, ld, H, peers, /*blockK=*/-1, /*last=*/true, /*smLimit=*/0);
    fresh = false;
    exchange_wait(rt);
    return local;
  }
  if (g.halo) {
    const size_t uld = (size_t)ld;
    rt->ensure_sendbuf((g.numSendRows ? g.numSendRows : 1) * uld);
    ROC_CHECK(roc_pack_rows((int64_t)g.numSendRows, H, g.d_sendRows, local, ld, rt->sendBuf, ld, rt->stream));
    std::vector<size_t> sc(g.sendCounts), so(g.sendOffs), rc(g.recvCounts), ro(g.recvOffs);
    for (size_t q = 0; q < sc.size(); q++) { sc[q] *= uld; so[q] *= uld; rc[q] *= uld; ro[q] *= uld; }
    float* haloBase = local + (size_t)model.local_rows() * uld;
    ROC_CHECK(rt->comm.alltoallv(rt->sendBuf, sc, so, haloBase, rc, ro, /*isFloat=*/true, rt->stream));
    return local;
  }
  rt->ensure_gather((size_t)g.numNodes * (size_t)ld);
  std::vector<size_t> counts((size_t)rt->numParts), offs((size_t)rt->numParts);
  for (int r = 0; r < rt->numParts; r++) {
    counts[(size_t)r] = ((size_t)g.vbounds[2 * r + 1] - g.vbounds[2 * r] + 1) * (size_t)ld;
    offs[(size_t)r] = (size_t)g.vbounds[2 * r] * (size_t)ld;
  }
  ROC_CHECK(rt->comm.allgatherv(local, rt->gatherBuf, counts, offs, rt->stream));
  return rt->gatherBuf;
}
}  // namespace

void ScatterGather::forward(const Model& model) {
  RuntimeImpl* rt = model.ctx;
  const int H = (int)inputs[0].dims[0];
  const int64_t ldIn = rt->t(inputs[0].region).ld;
  const int outRegion = fwdOut >= 0 ? fwdOut : outputs[0].region;
  rt->sg_begin(-H);          // negative width = the exposed part of the halo exchange (profile mode only)
  const float* src = gathered(model, rt->data(inputs[0].region), ldIn, H, &rt->t(inputs[0].region), false);
  rt->sg_end();
  float* dst = rt->data(outRegion);
  rt->sg_begin(H);
  if (aggr == AGGR_MAX || aggr == AGGR_MIN) {
    // winner ids only when a backward follows
    const bool wantArg = rt->t(inputs[0].region).requiresGrad && model.mode == MD_MODE_TRAIN;
    TensorImpl& at = rt->t(argRegion);
    uint32_t* arg = wantArg ? reinterpret_cast<uint32_t*>(rt->data(argRegion)) : NULL;
    ROC_CHECK(roc_sg_aggr_forward(model.myGraph.plan, aggr == AGGR_MAX ? ROC_AGGR_MAX : ROC_AGGR_MIN, H, src, ldIn,
                                  model.myGraph.d_colSrc, dst, rt->t(outRegion).ld, arg, at.ld, rt->stream));
  } else {
    const int epi = epilogue | (aggr == AGGR_AVG ? ROC_SG_EPI_MEAN : 0);
    ROC_CHECK(roc_sg_forward_planned(model.myGraph.plan, H, src, ldIn, dst, rt->t(outRegion).ld, epi, rt->stream));
  }
  rt->sg_end();
}

void ScatterGather::backward(const Model& model) {
  RuntimeImpl* rt = model.ctx;
  ROC_ASSERT(resetInputGrads[0]);   // scattergather_kernel.cu:167
  if (!rt->t(inputs[0].region).requiresGrad) return;
  const int H = (int)inputs[0].dims[0];
  const int64_t ld = rt->t(outputs[0].region).ld;
  const int dstRegion = bwdOut >= 0 ? bwdOut : inputs[0].region;
  const Graph& g = model.myGraph;
  if (aggr == AGGR_AVG) {
    // dIn = A (D^-1 dOut): scale the dOut rows into the scratch tensor, exchange that, then SUM's gather
    TensorImpl& sc = rt->t(scratch);
    ROC_CHECK(roc_indegree_div(g.rowLeft, g.rowRight, g.colLeft, H, g.d_rowEnd, rt->grad(outputs[0].region), ld,
                               rt->data(scratch), sc.ld, rt->stream));
    rt->sg_begin(-H);
    const float* src = gathered(model, rt->data(scratch), sc.ld, H, &sc, false);
    rt->sg_end();
    rt->sg_begin(H);
    ROC_CHECK(roc_sg_forward_planned(g.plan, H, src, sc.ld, rt->grad(dstRegion), rt->t(dstRegion).ld, ROC_SG_EPI_NONE,
                                     rt->stream));
    rt->sg_end();
    return;
  }
  if (aggr == AGGR_MAX || aggr == AGGR_MIN) {
    // dIn[u] = sum over v in in(u) of dOut[v] where arg[v] == u: a gather of dOut and the winner ids at halo rows
    TensorImpl& at = rt->t(argRegion);
    rt->sg_begin(-H);
    const float* src = gathered(model, rt->grad(outputs[0].region), ld, H, &rt->t(outputs[0].region), true);
    const float* args = gathered(model, rt->data(argRegion), at.ld, H, &at, false);
    rt->sg_end();
    ROC_ASSERT(args != src);   // the whole-matrix all-gather's one buffer cannot hold both
    rt->sg_begin(H);
    ROC_CHECK(roc_sg_arg_backward(g.plan, H, src, ld, reinterpret_cast<const uint32_t*>(args), at.ld, g.rowLeft,
                                  rt->grad(dstRegion), rt->t(dstRegion).ld, rt->stream));
    rt->sg_end();
    return;
  }
  // Forward and backward do exactly the same thing, on gradients (scattergather_kernel.cu:168-169)
  rt->sg_begin(-H);
  const float* src = gathered(model, rt->grad(outputs[0].region), ld, H, &rt->t(outputs[0].region), true);
  rt->sg_end();
  float* dst = rt->grad(dstRegion);
  rt->sg_begin(H);
  ROC_CHECK(roc_sg_forward_planned(model.myGraph.plan, H, src, ld, dst, rt->t(dstRegion).ld, bwdEpilogue, rt->stream));
  rt->sg_end();
}

// ------------------------------------------------------- GraphAttention -----
GraphAttention::GraphAttention(const Model& model, const Tensor& _input, int _heads, float _slope)
    : GnnOp(_input), heads(_heads), slope(_slope), attRegion(-1), bstRegion(-1), dsRegion(-1), work(nullptr) {
  ROC_ASSERT(inputs[0].type == Tensor::NODE_TENSOR);
  ROC_ASSERT(inputs[0].numDim == 2);
  ROC_ASSERT(inputs[0].dims[1] == model.myGraph.numNodes);
  const int H = (int)inputs[0].dims[0];
  if (roc_gat_supported(H, heads) != ROC_OK) {
    char b[256];
    snprintf(b, sizeof(b), "graph_attention: unsupported shape H = %d, heads = %d (heads in {1, 2, 4, 8}, H <= 256, "
             "H / heads a multiple of 4 when heads > 1)", H, heads);
    ROC_FATAL(b);
  }
  numOutputs = 1;
  outputs[0] = model.create_node_tensor<DATATYPE>(H);
  weight = model.create_weight_tensor(H, 2, NULL);   // GlorotUniform; row 0 a_src, row 1 a_dst
  // per-op buffers, allocated with the op (nothing is allocated inside a step)
  const int A = 2 * heads;
  attRegion = model.ctx->new_tensor(model.local_rows(), A, round_up4(A), false, false);
  bstRegion = model.ctx->new_tensor(model.local_rows(), A, round_up4(A), false, false);
  dsRegion = model.ctx->new_tensor(model.local_rows(), A, round_up4(A), false, false);
  work = model.ctx->dmalloc(roc_gat_finish_workspace_bytes(H));
}
void GraphAttention::init(const Model&) {}

void GraphAttention::forward(const Model& model) {
  RuntimeImpl* rt = model.ctx;
  const int H = (int)inputs[0].dims[0];
  TensorImpl& x = rt->t(inputs[0].region);
  TensorImpl& at = rt->t(attRegion);
  TensorImpl& bt = rt->t(bstRegion);
  // s_src / s_dst of the own rows, then h and them at the halo rows
  ROC_CHECK(roc_gat_scores(model.local_rows(), H, heads, rt->data(inputs[0].region), x.ld, rt->data(weight.region),
                           rt->data(attRegion), at.ld, rt->stream));
  const float* h = gathered(model, rt->data(inputs[0].region), x.ld, H, &x, false);
  const float* att = gathered(model, rt->data(attRegion), at.ld, 2 * heads, &at, false);
  ROC_CHECK(roc_gat_forward(model.myGraph.plan, H, heads, slope, h, x.ld, att, at.ld, rt->data(bstRegion), bt.ld,
                            rt->data(outputs[0].region), rt->t(outputs[0].region).ld, rt->stream));
}

void GraphAttention::backward(const Model& model) {
  RuntimeImpl* rt = model.ctx;
  ROC_ASSERT(resetInputGrads[0]);   // dh is overwritten, like ScatterGather's
  const int H = (int)inputs[0].dims[0];
  TensorImpl& x = rt->t(inputs[0].region);
  TensorImpl& y = rt->t(outputs[0].region);
  TensorImpl& at = rt->t(attRegion);
  TensorImpl& bt = rt->t(bstRegion);
  TensorImpl& dt = rt->t(dsRegion);
  // c = <dOut, out> per row and head, then dOut and (lse | c) at the halo rows.  h's halo rows are the forward's:
  // nothing rewrites them between the two passes, so they need no second exchange.
  ROC_CHECK(roc_gat_bwd_c(model.local_rows(), H, heads, rt->grad(outputs[0].region), y.ld, rt->data(outputs[0].region),
                          y.ld, rt->data(bstRegion), bt.ld, rt->stream));
  const float* dOut = gathered(model, rt->grad(outputs[0].region), y.ld, H, &y, true);
  const float* bst = gathered(model, rt->data(bstRegion), bt.ld, 2 * heads, &bt, false);
  float* dh = rt->grad(inputs[0].region);
  ROC_CHECK(roc_gat_backward(model.myGraph.plan, H, heads, slope, rt->data(inputs[0].region), x.ld,
                             rt->data(attRegion), at.ld, bst, bt.ld, dOut, y.ld, dh, x.ld, rt->data(dsRegion), dt.ld,
                             rt->stream));
  ROC_CHECK(roc_gat_bwd_finish(model.local_rows(), H, heads, rt->data(inputs[0].region), x.ld, rt->data(weight.region),
                               rt->data(dsRegion), dt.ld, dh, x.ld, rt->grad(weight.region), work,
                               roc_gat_finish_workspace_bytes(H), rt->stream));
}

// --------------------------------------------------------- InDegreeNorm -----
InDegreeNorm::InDegreeNorm(const Model& model, const Tensor& _input)
    : GnnOp(_input), reluMaskOf(-1), bwdIn(-1), bwdFused(false) {
  ROC_ASSERT(inputs[0].type == Tensor::NODE_TENSOR);   // graphnorm.cc:33-35
  ROC_ASSERT(inputs[0].numDim == 2);
  ROC_ASSERT(inputs[0].dims[1] == model.myGraph.numNodes);
  numOutputs = 1;
  outputs[0] = model.create_node_tensor<DATATYPE>((int)inputs[0].dims[0]);
}
void InDegreeNorm::init(const Model&) {}

void InDegreeNorm::forward(const Model& model) {
  if (fusedInto >= 0) return;   // done in the producer's epilogue
  RuntimeImpl* rt = model.ctx;
  const Graph& g = model.myGraph;
  ROC_CHECK(roc_indegree_norm(g.rowLeft, g.rowRight, g.colLeft, (int)inputs[0].dims[0], g.d_rowEnd,
                              rt->data(inputs[0].region), rt->t(inputs[0].region).ld, rt->data(outputs[0].region),
                              rt->t(outputs[0].region).ld, NULL, rt->stream));
}

void InDegreeNorm::backward(const Model& model) {
  RuntimeImpl* rt = model.ctx;
  ROC_ASSERT(resetInputGrads[0]);   // graphnorm_kernel.cu:133
  if (!rt->t(inputs[0].region).requiresGrad) return;
  // fused into the linear's epilogue forward => the SG backward epilogue already
  // produced d(linear out); nothing to do here
  if (fusedInto >= 0 && dynamic_cast<Linear*>(model.layers[(size_t)fusedInto])) return;
  if (bwdFused) return;   // a Linear's dX epilogue / the softmax already wrote this gradient
  const Graph& g = model.myGraph;
  const int src = bwdIn >= 0 ? bwdIn : outputs[0].region;
  ROC_CHECK(roc_indegree_norm(g.rowLeft, g.rowRight, g.colLeft, (int)inputs[0].dims[0], g.d_rowEnd, rt->grad(src),
                              rt->t(src).ld, rt->grad(inputs[0].region), rt->t(inputs[0].region).ld,
                              reluMaskOf >= 0 ? rt->data(reluMaskOf) : NULL, rt->stream));
}

// ----------------------------------------------------------------- Linear ---
Linear::Linear(const Model& model, const Tensor& _input, int outDim, ActiMode _activation, Initializer* initializer)
    : GnnOp(_input), activation(_activation), flags(0), fwdOut(-1), bwdIn(-1), dropOp(-1), dropMask(nullptr), dropLd(0),
      dxReluOf(-1), dxNorm(false), dxOut(-1) {
  ROC_ASSERT(_input.numDim == 2);   // linear.cc:41-42
  ROC_ASSERT(_input.dims[1] == model.myGraph.numNodes);
  weight = model.create_weight_tensor((int)_input.dims[0], outDim, initializer);
  numOutputs = 1;
  outputs[0] = model.create_node_tensor<DATATYPE>(outDim);
}
void Linear::init(const Model& model) {
  if (dropOp < 0) return;
  RuntimeImpl* rt = model.ctx;
  dropLd = (((int64_t)weight.dims[0] + 31) / 32 + 3) / 4 * 4;
  dropMask = (uint32_t*)rt->dmalloc((size_t)std::max<int64_t>(model.local_rows(), 1) * (size_t)dropLd * sizeof(uint32_t));
}

namespace {
// the Dropout folded into a Linear: its rate in the current mode and its Philox key
struct FusedDrop { const Dropout* op; float rate; uint64_t key; int inRegion; };
FusedDrop fused_drop(const Model& model, int dropOp) {
  const Dropout* d = static_cast<const Dropout*>(model.layers[(size_t)dropOp]);
  FusedDrop f;
  f.op = d;
  f.rate = (model.mode == MD_MODE_TRAIN) ? d->rate : 0.0f;    // infer: dropout is a copy (dropout_kernel.cu:159-180)
  f.key = ((uint64_t)(uint32_t)d->seed << 32) | (uint32_t)d->opIndex;
  f.inRegion = d->inputs[0].region;
  return f;
}
}  // namespace

void Linear::forward(const Model& model) {
  RuntimeImpl* rt = model.ctx;
  const Graph& g = model.myGraph;
  const int outRegion = fwdOut >= 0 ? fwdOut : outputs[0].region;
  // If a ScatterGather on other GPUs reads this output (peer-mapped halo slabs), the rows are computed in blocks
  // and block k's boundary rows travel while block k + 1 is computed; otherwise one block = all rows.
  PushPipe pipe(model, outRegion, /*grad=*/false);
  const int inDim = (int)weight.dims[0], outDim = (int)weight.dims[1];
  float* Y = rt->data(outRegion);
  const int64_t ldY = rt->t(outRegion).ld;
  if (dropOp >= 0) {
    // dropout -> linear: the mask is generated packed (1 bit / element) and applied while the GEMM
    // loads X, so the dropped copy of X is never materialised
    const FusedDrop f = fused_drop(model, dropOp);
    if (f.rate > 0.0f)
      ROC_CHECK(roc_dropout_mask(model.local_rows(), inDim, g.rowLeft, f.rate, f.key, rt->trainStep,
                                 dropMask, dropLd, rt->stream));
    const float* X = rt->data(f.inRegion);
    const int64_t ldX = rt->t(f.inRegion).ld;
    for (size_t k = 0; k < pipe.blocks(); k++) {
      const int64_t r0 = pipe.row0(k), nr = pipe.rows(k, model.local_rows());
      ROC_CHECK(roc_linear_fwd_dropout(nr, inDim, outDim, X + r0 * ldX, ldX, rt->data(weight.region), Y + r0 * ldY, ldY,
                                       (int)activation, flags, g.d_rowEnd + r0, pipe.colLeft(k), dropMask + r0 * dropLd,
                                       dropLd, f.rate, rt->stream));
      pipe.pushed(k, Y, ldY, outDim);
    }
    return;
  }
  const float* X = rt->data(inputs[0].region);
  const int64_t ldX = rt->t(inputs[0].region).ld;
  for (size_t k = 0; k < pipe.blocks(); k++) {
    const int64_t r0 = pipe.row0(k), nr = pipe.rows(k, model.local_rows());
    ROC_CHECK(roc_linear_fwd(nr, inDim, outDim, X + r0 * ldX, ldX, rt->data(weight.region), Y + r0 * ldY, ldY,
                             (int)activation, flags, g.d_rowEnd + r0, pipe.colLeft(k), rt->stream));
    pipe.pushed(k, Y, ldY, outDim);
  }
}

void Linear::backward(const Model& model) {
  RuntimeImpl* rt = model.ctx;
  const Graph& g = model.myGraph;
  const int gy = bwdIn >= 0 ? bwdIn : outputs[0].region;
  roc_linear_bwd_args a;
  memset(&a, 0, sizeof(a));
  int xRegion = inputs[0].region;
  a.accumulate_dX = resetInputGrads[0] ? 0 : 1;
  if (dropOp >= 0) {
    // dW from the masked X; dX lands directly in the gradient of the dropout's input (the dropout
    // backward, dropout_kernel.cu:149-150, runs in the dX epilogue; it always overwrites, :119)
    const FusedDrop f = fused_drop(model, dropOp);
    ROC_ASSERT(resetInputGrads[0]);
    xRegion = f.inRegion;
    a.accumulate_dX = 0;
    a.dropMask = dropMask; a.ldMask = dropLd; a.dropRate = f.rate;
  }
  const int dxRegion = dxOut >= 0 ? dxOut : xRegion;
  a.rows = model.local_rows(); a.inDim = (int)weight.dims[0]; a.outDim = (int)weight.dims[1];
  a.X = rt->data(xRegion); a.ldX = rt->t(xRegion).ld;
  a.W = rt->data(weight.region);
  a.Y = (activation != AC_MODE_NONE) ? rt->data(outputs[0].region) : NULL; a.ldY = rt->t(outputs[0].region).ld;
  a.dY = rt->grad(gy); a.ldDY = rt->t(gy).ld;
  a.dW = rt->grad(weight.region);
  a.dX = rt->t(xRegion).requiresGrad ? rt->grad(dxRegion) : NULL;   // Q8: leaf grads skipped
  a.ldDX = rt->t(dxRegion).ld;
  a.activation = (int)activation;
  a.workspace = rt->linWs; a.workspaceBytes = rt->linWsBytes;
  if (a.dX && dxReluOf >= 0) { a.dxReluOf = rt->data(dxReluOf); a.ldReluOf = rt->t(dxReluOf).ld; }
  if (a.dX && dxNorm) { a.dxNormRowEnd = g.d_rowEnd; a.colLeft = g.colLeft; }
  // dX feeds a ScatterGather backward on other GPUs (peer-mapped slabs): dX in row blocks, each pushed while the
  // next is computed, then dW — which nothing downstream waits for — while the last rows travel.
  PushPipe pipe(model, (a.dX && activation == AC_MODE_NONE) ? dxRegion : -1, /*grad=*/true);
  if (pipe.on) {
    for (size_t k = 0; k < pipe.blocks(); k++) {
      const int64_t r0 = pipe.row0(k), nr = pipe.rows(k, model.local_rows());
      roc_linear_bwd_args b = a;
      b.parts = ROC_LINEAR_BWD_ONLY_DX;
      b.rows = nr;
      b.X = a.X + r0 * a.ldX;
      b.dY = a.dY + r0 * a.ldDY;
      b.dX = a.dX + r0 * a.ldDX;
      if (a.dropMask) b.dropMask = a.dropMask + r0 * a.ldMask;
      if (a.dxReluOf) b.dxReluOf = a.dxReluOf + r0 * a.ldReluOf;
      if (a.dxNormRowEnd) { b.dxNormRowEnd = a.dxNormRowEnd + r0; b.colLeft = pipe.colLeft(k); }
      ROC_CHECK(roc_linear_bwd_fused(&b, rt->stream));
      pipe.pushed(k, a.dX, a.ldDX, a.inDim);
    }
    a.parts = ROC_LINEAR_BWD_ONLY_DW;
    ROC_CHECK(roc_linear_bwd_fused(&a, rt->stream));
    return;
  }
  ROC_CHECK(roc_linear_bwd_fused(&a, rt->stream));
}

// ------------------------------------------------------------- Activation ---
Activation::Activation(const Model& model, const Tensor& _input, ActiMode _actiMode)
    : GnnOp(_input), actiMode(_actiMode) {
  ROC_ASSERT(_input.numDim == 2);
  numOutputs = 1;
  outputs[0] = model.create_node_tensor<DATATYPE>((int)_input.dims[0]);
}
void Activation::init(const Model&) {}
void Activation::forward(const Model& model) {
  if (fusedInto >= 0) return;
  RuntimeImpl* rt = model.ctx;
  ROC_CHECK(roc_activation_fwd(model.local_rows(), (int)inputs[0].dims[0], (int)actiMode, rt->data(inputs[0].region),
                               rt->t(inputs[0].region).ld, rt->data(outputs[0].region), rt->t(outputs[0].region).ld,
                               rt->stream));
}
void Activation::backward(const Model& model) {
  if (fusedInto >= 0) return;   // mask applied by the fused indegree_norm backward
  RuntimeImpl* rt = model.ctx;
  if (!rt->t(inputs[0].region).requiresGrad) return;
  ROC_CHECK(roc_activation_bwd(model.local_rows(), (int)inputs[0].dims[0], (int)actiMode, rt->data(outputs[0].region),
                               rt->t(outputs[0].region).ld, rt->grad(outputs[0].region), rt->t(outputs[0].region).ld,
                               rt->grad(inputs[0].region), rt->t(inputs[0].region).ld, resetInputGrads[0] ? 0 : 1,
                               rt->stream));
}

// ---------------------------------------------------------------- Element ---
Element::Element(const Model& model, const Tensor& input0, const Tensor& input1, ElementType _elementType)
    : GnnOp(input0, input1), elementType(_elementType) {
  ROC_ASSERT(input0.numDim == input1.numDim);   // element.cc:33-36
  for (int i = 0; i < input0.numDim; i++) ROC_ASSERT(input0.dims[i] == input1.dims[i]);
  numOutputs = 1;
  outputs[0] = model.create_node_tensor<DATATYPE>((int)input0.dims[0]);
}
void Element::init(const Model&) {}
void Element::forward(const Model& model) {
  RuntimeImpl* rt = model.ctx;
  ROC_ASSERT(elementType == EW_TYPE_ADD);
  ROC_CHECK(roc_add_fwd(model.local_rows(), (int)inputs[0].dims[0], rt->data(inputs[0].region),
                        rt->t(inputs[0].region).ld, rt->data(inputs[1].region), rt->t(inputs[1].region).ld,
                        rt->data(outputs[0].region), rt->t(outputs[0].region).ld, rt->stream));
}
void Element::backward(const Model& model) {
  RuntimeImpl* rt = model.ctx;
  ROC_ASSERT(elementType == EW_TYPE_ADD);   // element_kernel.cu:102-104
  float* dA = rt->t(inputs[0].region).requiresGrad ? rt->grad(inputs[0].region) : NULL;
  float* dB = rt->t(inputs[1].region).requiresGrad ? rt->grad(inputs[1].region) : NULL;
  ROC_CHECK(roc_add_bwd(model.local_rows(), (int)inputs[0].dims[0], rt->grad(outputs[0].region),
                        rt->t(outputs[0].region).ld, dA, rt->t(inputs[0].region).ld, resetInputGrads[0] ? 0 : 1, dB,
                        rt->t(inputs[1].region).ld, resetInputGrads[1] ? 0 : 1, rt->stream));
}

// ---------------------------------------------------------------- Dropout ---
Dropout::Dropout(const Model& model, const Tensor& _input, float _rate, int _seed)
    : GnnOp(_input), rate(_rate), seed(_seed), opIndex(0) {
  ROC_ASSERT(_input.numDim == 2);
  ROC_ASSERT(_input.type == Tensor::NODE_TENSOR);
  numOutputs = 1;
  outputs[0] = model.create_node_tensor<DATATYPE>((int)_input.dims[0]);
}
void Dropout::init(const Model&) {}
void Dropout::forward(const Model& model) {
  if (fusedInto >= 0) return;   // applied by the consuming Linear while it loads X
  RuntimeImpl* rt = model.ctx;
  // train: masked scale (dropout_kernel.cu:98-99); infer: plain copy (:159-180)
  const float r = (model.mode == MD_MODE_TRAIN) ? rate : 0.0f;
  const uint64_t key = ((uint64_t)(uint32_t)seed << 32) | (uint32_t)opIndex;
  ROC_CHECK(roc_dropout_fwd(model.local_rows(), (int)inputs[0].dims[0], model.myGraph.rowLeft, r, key, rt->trainStep,
                            rt->data(inputs[0].region), rt->t(inputs[0].region).ld, rt->data(outputs[0].region),
                            rt->t(outputs[0].region).ld, rt->stream));
}
void Dropout::backward(const Model& model) {
  RuntimeImpl* rt = model.ctx;
  if (!rt->t(inputs[0].region).requiresGrad) return;   // leaf input (Q8)
  ROC_ASSERT(resetInputGrads[0]);   // dropout_kernel.cu:119
  if (fusedInto >= 0) return;       // the consuming Linear's dX epilogue already wrote this gradient
  const float r = (model.mode == MD_MODE_TRAIN) ? rate : 0.0f;
  const uint64_t key = ((uint64_t)(uint32_t)seed << 32) | (uint32_t)opIndex;
  ROC_CHECK(roc_dropout_bwd(model.local_rows(), (int)inputs[0].dims[0], model.myGraph.rowLeft, r, key, rt->trainStep,
                            rt->grad(outputs[0].region), rt->t(outputs[0].region).ld, rt->grad(inputs[0].region),
                            rt->t(inputs[0].region).ld, rt->stream));
}

// ---------------------------------------------------- SoftmaxCrossEntropy ---
SoftmaxCrossEntropy::SoftmaxCrossEntropy(const Model&, const Tensor& _logit, const Tensor& _label, const Tensor& _mask)
    : GnnOp(_logit, _label, _mask), epoch_num(0), gradOut(-1) {
  ROC_ASSERT(_logit.numDim == 2);   // softmax.cc:36-39
  ROC_ASSERT(_label.numDim == 2);
  ROC_ASSERT(_label.dims[0] == _logit.dims[0]);
  ROC_ASSERT(_label.dims[1] == _logit.dims[1]);
  numOutputs = 0;
}
void SoftmaxCrossEntropy::init(const Model&) {}
void SoftmaxCrossEntropy::forward(const Model& model) {
  mode = model.mode;
  if (model.mode == MD_MODE_TRAIN) {
    // Do nothing in training forward (softmax.cc:48-49)
  } else {
    backward(model);   // softmax.cc:50-54: inference reuses the backward task for metrics
  }
}
void SoftmaxCrossEntropy::backward(const Model& model) {
  RuntimeImpl* rt = model.ctx;
  mode = model.mode;
  if (mode == MD_MODE_TRAIN) epoch_num++;
  ROC_ASSERT(inputs[2].region >= 0);   // softmax_kernel.cu:157-160: masks are required
  const int C = (int)inputs[0].dims[0];
  TensorImpl& lab = rt->t(inputs[1].region);
  ROC_CHECK(cudaMemsetAsync(rt->d_perf, 0, sizeof(roc_perf_metrics), rt->stream));
  const int32_t* mask = reinterpret_cast<const int32_t*>(rt->data(inputs[2].region));
  if (gradOut >= 0) {
    // the logits come from an InDegreeNorm: its backward (grad / sqrt(deg)) is applied here and the
    // result goes straight into the gradient the ScatterGather backward reads
    const Graph& g = model.myGraph;
    PushPipe pipe(model, mode == MD_MODE_TRAIN ? gradOut : -1, /*grad=*/true);
    const float* Z = rt->data(inputs[0].region);
    const int64_t ldZ = rt->t(inputs[0].region).ld;
    const float* L = lab.labelIdx ? NULL : rt->data(inputs[1].region);
    const int64_t ldL = lab.labelIdx ? 0 : lab.ld;
    float* G = rt->grad(gradOut);
    const int64_t ldG = rt->t(gradOut).ld;
    for (size_t k = 0; k < pipe.blocks(); k++) {
      const int64_t r0 = pipe.row0(k), nr = pipe.rows(k, model.local_rows());
      ROC_CHECK(roc_softmax_xent_bwd_norm(nr, C, Z + r0 * ldZ, ldZ, L ? L + r0 * ldL : NULL, ldL,
                                          lab.labelIdx ? lab.labelIdx + r0 : NULL, mask + r0, G + r0 * ldG, ldG,
                                          g.d_rowEnd + r0, pipe.colLeft(k), rt->d_perf, rt->stream));
      pipe.pushed(k, G, ldG, C);
    }
  } else if (lab.labelIdx) {
    ROC_CHECK(roc_softmax_xent_bwd_idx(model.local_rows(), C, rt->data(inputs[0].region), rt->t(inputs[0].region).ld,
                                       lab.labelIdx, mask, rt->grad(inputs[0].region), rt->t(inputs[0].region).ld,
                                       rt->d_perf, rt->stream));
  } else {
    ROC_CHECK(roc_softmax_xent_bwd(model.local_rows(), C, rt->data(inputs[0].region), rt->t(inputs[0].region).ld,
                                   rt->data(inputs[1].region), lab.ld, mask, rt->grad(inputs[0].region),
                                   rt->t(inputs[0].region).ld, rt->d_perf, rt->stream));
  }
  if (mode == MD_MODE_INFER && model.printMetrics) {
    roc_perf_metrics p = model.last_metrics();
    // softmax_kernel.cu:141-152 (printed once per partition, quirk Q20)
    // to stderr AND stdout, as the reference does (scripts scrape either)
    FILE* sinks[2] = {stderr, stdout};
    for (FILE* f : sinks)
      fprintf(f,
              "\t[INFER][%d] train_loss: %.4lf  train_accuracy: %.2lf%%(%d/%d)  val_accuracy: %.2lf%%(%d/%d)  "
              "test_accuracy: %.2lf%%(%d/%d)\n",
              epoch_num, p.trainLoss, p.trainCorrect * 100.0f / p.trainAll, p.trainCorrect, p.trainAll,
              p.valCorrect * 100.0f / p.valAll, p.valCorrect, p.valAll, p.testCorrect * 100.0f / p.testAll,
              p.testCorrect, p.testAll);
    fflush(stdout);
  }
}

// ----------------------------------------------------------- initializers ---
// initializer.cc:31-46 + initializer_kernel.cu:22-51: cuRAND's default XORWOW
// generator seeded with the next std::rand(), uniform (0,1] over the weight's
// linear memory order, then W = 2*s*u - s.  cuRAND is called at init only, so
// the weights match the reference bit for bit for a given -seed.
void GlorotUniform::init(const Model* model, const Tensor* p) {
  RuntimeImpl* rt = model->ctx;
  ROC_ASSERT(p->numDim == 2);
  int num = std::rand();
  const int inputDim = (int)p->dims[0], outputDim = (int)p->dims[1];
  const size_t vol = (size_t)inputDim * outputDim;
  float scale = sqrt(6.0 / (inputDim + outputDim));
  curandGenerator_t gen;
  ROC_CHECK(curandCreateGenerator(&gen, CURAND_RNG_PSEUDO_DEFAULT));
  ROC_CHECK(curandSetStream(gen, rt->stream));
  ROC_CHECK(curandSetPseudoRandomGeneratorSeed(gen, (unsigned long long)num));
  float* w = rt->data(p->region);
  ROC_CHECK(curandGenerateUniform(gen, w, vol));
  ROC_CHECK(roc_scale((int64_t)vol, -scale, scale, w, rt->stream));
  ROC_CHECK(cudaStreamSynchronize(rt->stream));
  curandDestroyGenerator(gen);
}

void ZerosInitializer::init(const Model* model, const Tensor* p) {
  RuntimeImpl* rt = model->ctx;
  ROC_ASSERT(p->numDim == 2);
  TensorImpl& x = rt->t(p->region);
  ROC_CHECK(roc_fill(x.rows, x.H, 0.0f, rt->data(p->region), x.ld, rt->stream));
}

// -------------------------------------------------------------- optimizer ---
// optimizer.cc:22-70: m and v per parameter, zero-initialised; must be built
// after every linear() call (it walks model->parameters).
AdamOptimizer::AdamOptimizer(const Model* _model, double _alpha, double _beta1, double _beta2, double _weight_decay,
                             double _epsilon)
    : Optimizer(_model), alpha(_alpha), beta1(_beta1), beta2(_beta2), weight_decay(_weight_decay),
      epsilon(_epsilon), alpha_t(_alpha), beta1_t(1.0f), beta2_t(1.0f) {
  RuntimeImpl* rt = _model->ctx;
  ZerosInitializer zeros;
  for (size_t i = 0; i < model->parameters.size(); i++) {
    const Tensor& p = model->parameters[i];
    Tensor t = p;
    t.region = rt->new_tensor((int64_t)p.dims[1], (int)p.dims[0], (int64_t)p.dims[0], false, true);
    v_regions[p.region] = t.region;
    zeros.init(_model, &t);
    t.region = rt->new_tensor((int64_t)p.dims[1], (int)p.dims[0], (int64_t)p.dims[0], false, true);
    m_regions[p.region] = t.region;
    zeros.init(_model, &t);
  }
}

void AdamOptimizer::set_weight_decay(double _weight_decay) { weight_decay = _weight_decay; }

// optimizer.cc:79-85
void AdamOptimizer::next(void) {
  beta1_t *= beta1;
  beta2_t *= beta2;
  alpha_t = alpha * sqrt(1 - beta2_t) / (1 - beta1_t);
}

// optimizer.cc:87-119 + optimizer_kernel.cu:66-103 (the gradient was already summed
// over partitions by Model::update's all-reduce)
void AdamOptimizer::update(const Tensor* p) {
  RuntimeImpl* rt = model->ctx;
  ROC_ASSERT(v_regions.find(p->region) != v_regions.end());
  ROC_ASSERT(m_regions.find(p->region) != m_regions.end());
  const int64_t count = (int64_t)p->dims[0] * (int64_t)p->dims[1];
  ROC_CHECK(roc_adam_update(count, (float)alpha_t, (float)beta1, (float)beta2, (float)weight_decay, (float)epsilon,
                            rt->grad(p->region), rt->data(m_regions[p->region]), rt->data(v_regions[p->region]),
                            rt->data(p->region), rt->stream));
}

// ------------------------------------------------------------------- CLI ----
// Same flags as gnn.cc:114-179, including "-dr" being taken by dropout before
// decay-rate can see it (quirk Q19).
void parse_input_args(char** argv, int argc, Config& config) {
  for (int i = 1; i < argc; i++) {
    const std::string a(argv[i]);
    const bool more = i + 1 < argc;
    if (a == "-seed" && more) config.seed = atoi(argv[++i]);
    else if ((a == "-ng" || a == "-ll:gpu") && more) config.numGPUs = atoi(argv[++i]);
    else if ((a == "-e" || a == "-epoch") && more) config.numEpochs = atoi(argv[++i]);
    else if (a == "-lr" && more) config.learning_rate = atof(argv[++i]);
    else if ((a == "-dropout" || a == "-dr") && more) config.dropout_rate = atof(argv[++i]);
    else if ((a == "-decay" || a == "-wd") && more) config.weight_decay = atof(argv[++i]);
    else if (a == "-decay-rate" && more) config.decay_rate = atof(argv[++i]);
    else if ((a == "-decay-step" || a == "-ds") && more) config.decay_steps = atoi(argv[++i]);
    else if (a == "-file" && more) config.filename = std::string(argv[++i]);
    else if (a == "-verbose" || a == "-v") config.verbose = true;
    else if (a == "-layers" && more) {
      std::stringstream ss((std::string(argv[++i])));
      std::string word;
      config.layers.clear();
      while (std::getline(ss, word, '-')) config.layers.push_back(std::stoi(word));
    }
  }
}
