/*
 * roc_gnn.h — the Model / op-builder surface of ROC's gnn.h (gnn.h:105-222,
 * optimizer.h:25-50, initializer.h) over a thin C++ host: one process per GPU,
 * CUDA streams, HBM-resident tensors, NCCL for the two exchange steps.  The
 * Legion runtime, GnnMapper, TensorAccessor staging and ResourceManager are
 * gone; `Context` / `Runtime` remain as plain handles so the reference's model
 * script (gnn.cc:65-111) compiles against this header unchanged:
 *
 *     Graph graph(ctx, runtime, config);
 *     Model model(graph, ctx, runtime);
 *     Tensor input = model.create_node_tensor<DATATYPE>(config.layers[0]);
 *     ... model.dropout / linear / indegree_norm / scatter_gather / relu / add ...
 *     model.softmax_cross_entropy(t, label, mask);
 *     AdamOptimizer* optimizer = new AdamOptimizer(&model, config.learning_rate);
 *     optimizer->set_weight_decay(config.weight_decay);
 *     model.optimizer = optimizer;  model.init(config);
 *     loop: optimizer->alpha *= decay;  train_mode; zero_gradients; forward; backward; update
 *
 * Names, argument meaning, enum values and error behaviour (assert / exit(1))
 * follow the reference; every class cites the reference definition it mirrors.
 * The device work is done by the C-ABI kernel layer in roc_b200.h.
 */
#ifndef ROC_GNN_H_
#define ROC_GNN_H_

#include <cstdint>
#include <map>
#include <string>
#include <vector>

#include "roc_b200.h"

typedef uint32_t V_ID;   /* types.h:5 */
typedef uint64_t E_ID;   /* types.h:6 */
typedef float DATATYPE;  /* types.h:7 */

#define MAX_FILE_LEN 64        /* gnn.h:27 (kept for parity; paths are not truncated here) */
#define MAX_NUM_PARTS 64       /* gnn.h:28 */
#define MAX_NUM_INPUTS 8       /* gnn.h:30 */
#define MAX_NUM_OUTPUTS 8      /* gnn.h:31 */
#define MAX_NUM_DIM 4          /* gnn.h:32 */
#define FILE_HEADER_SIZE (sizeof(E_ID) + sizeof(V_ID)) /* gnn.h:33 */

enum AggrType { AGGR_AVG, AGGR_MAX, AGGR_MIN, AGGR_SUM };            /* gnn.h:75-80 */
enum ActiMode { AC_MODE_NONE, AC_MODE_RELU, AC_MODE_SIGMOID };         /* gnn.h:82-86 */
enum ElementType { EW_TYPE_ADD, EW_TYPE_MUL };                         /* gnn.h:88-91 */
enum ModelMode { MD_MODE_TRAIN, MD_MODE_INFER };                       /* gnn.h:93-96 */
enum MaskType { MASK_TRAIN, MASK_VAL, MASK_TEST, MASK_NONE };          /* gnn.h:98-103 */

namespace roc { namespace host { struct RuntimeImpl; struct TensorImpl; struct Comm; } }

/* Stand-ins for Legion's handles.  A Runtime owns the process's GPU, stream,
 * device allocations and (for numParts > 1) the NCCL communicator. */
typedef roc::host::RuntimeImpl* Context;

class Runtime {
public:
  /* device: CUDA ordinal for this process; myPart / numParts: which vertex-range
   * partition this process owns (one process per GPU). */
  explicit Runtime(int device = 0, int myPart = 0, int numParts = 1);
  ~Runtime();
  Context context() const { return impl; }
  /* NCCL bootstrap (only place NCCL appears): rank 0 creates the id, the
   * launcher broadcasts the 128 bytes, every rank calls init_nccl. */
  static bool nccl_unique_id(unsigned char id[128]);
  bool init_nccl(const unsigned char id[128]);
  void synchronize();
  roc::host::RuntimeImpl* impl;
private:
  Runtime(const Runtime&);
  Runtime& operator=(const Runtime&);
};

struct Config {  /* gnn.h:105-113 */
  int numGPUs, numMachines, totalGPUs, numEpochs, decay_steps, seed;
  bool verbose;
  float learning_rate, weight_decay, dropout_rate;
  float decay_rate;
  std::string filename;
  std::vector<int> layers;
  Config();
};

struct Graph {  /* gnn.h:120-130; ctor = gnn.cc:751-872 (reads <file>.add_self_edge.lux) */
  Graph(Context _ctx, Runtime* _runtime, const Config& config);
  /* Same partitioning / device CSR from arrays already in host memory
   * (host_rowEnd: N global END offsets; host_colSrc: all E sources). */
  Graph(Context _ctx, Runtime* _runtime, V_ID numNodes, E_ID numEdges,
        const E_ID* host_rowEnd, const V_ID* host_colSrc);
  V_ID numNodes;
  E_ID numEdges;
  int numParts, numMachines;
  int maxHidden;
  /* this process's partition (the rects of rowPtrLP / colIdxLP for its colour) */
  int myPart;
  V_ID rowLeft, rowRight;
  E_ID colLeft, colRight;
  std::vector<V_ID> vbounds;   /* [numParts][2] */
  std::vector<E_ID> ebounds;   /* [numParts][2] */
  /* device CSR (replaces rowPtrLR / colIdxLR): END offsets + lean sources */
  E_ID* d_rowEnd;
  V_ID* d_colSrc;
  roc_sg_plan* plan;
  /* numParts > 1: halo exchange structures (derived and private; see roc_halo_* in roc_b200.h).
   * The plan is then built on the remapped col ([own rows | halo rows]); d_colSrc stays canonical. */
  roc_halo* halo;
  V_ID numHalo;
  std::vector<size_t> recvCounts, recvOffs, sendCounts, sendOffs;   /* rows, per peer partition */
  V_ID* d_sendRows;      /* local rows other partitions read, grouped by requester */
  size_t numSendRows;
  /* Peer-write exchange (roc_push_rows): the same send list sorted by source row, each entry with the partition
   * that reads it and its row in that partition's [own | halo] slab; cut into row blocks so that a producer
   * (Linear, softmax) can push block k while it computes block k + 1. */
  V_ID* d_pushRows;
  unsigned char* d_pushPeer;
  V_ID* d_pushDst;
  std::vector<V_ID> pushBlockRow;       /* [blocks + 1] first local row of each block */
  std::vector<size_t> pushBlockOff;     /* [blocks + 1] offsets into the sorted send list */
  std::vector<E_ID> pushBlockColLeft;   /* [blocks] global END offset of the row before the block */
  /* Copy-engine exchange: block k's entries of the requester-grouped send list (d_packSel[packBlockOff[k] ..]),
   * and, per requester q, where block k starts inside q's contiguous run (packPeerOff[q * (blocks + 1) + k]). */
  V_ID* d_packSel;
  std::vector<size_t> packBlockOff;
  std::vector<size_t> packPeerOff;
  std::vector<V_ID> peerSlab0;          /* [parts] first row of this partition's rows in partition q's [own | halo] slab */
private:
  void build(Context ctx, const E_ID* host_rowEnd, const V_ID* slice_colSrc);
};

struct Tensor {  /* gnn.h:132-158 */
  enum Type { NODE_TENSOR = 1, EDGE_TENSOR = 2, GRAPH_TENSOR = 3, WEIGHT_TENSOR = 4, INVALID_TENSOR = 9 };
  Tensor(void) : type(INVALID_TENSOR), numDim(0), region(-1) { dims[0] = dims[1] = dims[2] = dims[3] = 0; }
  Tensor(Type _type) : type(_type), numDim(0), region(-1) { dims[0] = dims[1] = dims[2] = dims[3] = 0; }
  Type type;
  int numDim;
  E_ID dims[MAX_NUM_DIM];   /* dims[0] = hidden width, dims[1] = numNodes (node tensors); [in][out] (weights) */
  int region;               /* handle into the Runtime's tensor table (replaces LogicalRegion) */
};

class Model;
class GnnOp;

class Initializer {  /* initializer.h */
public:
  Initializer(void) {}
  virtual ~Initializer(void) {}
  virtual void init(const Model* model, const Tensor* tensor) = 0;
};
class GlorotUniform : public Initializer {  /* initializer.cc:31-46, initializer_kernel.cu:22-51 */
public:
  void init(const Model* model, const Tensor* tensor);
};
class ZerosInitializer : public Initializer {  /* initializer.cc:54-70 */
public:
  void init(const Model* model, const Tensor* tensor);
};

class Optimizer {  /* optimizer.h:25-32 */
public:
  Optimizer(const Model* _model) : model(_model) {}
  virtual ~Optimizer() {}
  virtual void next(void) = 0;
  virtual void update(const Tensor* p) = 0;
  const Model* model;
};

class AdamOptimizer : public Optimizer {  /* optimizer.h:34-50, optimizer.cc:22-119 */
public:
  AdamOptimizer(const Model* _model, double _alpha = 0.001f, double _beta1 = 0.9f,
                double _beta2 = 0.999f, double _weight_decay = 0.0f, double _epsilon = 1e-8);
  void next(void);
  void update(const Tensor* p);
  void set_weight_decay(double _weight_decay);
  double alpha, beta1, beta2, weight_decay, epsilon;
  double alpha_t, beta1_t, beta2_t;
  std::map<int, int> v_regions, m_regions;   /* weight region -> moment buffers */
};

class Model {  /* gnn.h:162-203 */
public:
  Model(const Graph& _graph, Context _ctx, Runtime* _runtime);
  Tensor add(const Tensor& _input1, const Tensor& _input2);
  Tensor dropout(const Tensor& _input, float rate, int seed = 0);
  /* aggr: the neighbourhood reduction (gnn.h:75-80).  SUM is the reference's ScatterGather; AVG divides each
   * row's sum by its in-degree; MAX / MIN take the per-column extreme (first edge in CSR order wins ties, NaN
   * wins over numbers), with gradients routed to the recorded winner.  The backward of every aggregator assumes
   * a symmetric in-edge CSR without duplicate edges, like SUM's (quirk Q1).  Only SUM ops take part in the
   * epilogue fusions. */
  Tensor scatter_gather(const Tensor& _input, AggrType aggr = AGGR_SUM);
  /* Graph attention (GAT, Velickovic et al. 2018) with `heads` heads over the node tensor _input of width
   * H = heads * F: out[v, k-block] = sum over in-edges u of alpha[v<-u,k] _input[u, k-block], alpha the softmax over
   * v's in-edges of LeakyReLU(<h[u], a_src[k]> + <h[v], a_dst[k]>, negativeSlope) per head, heads concatenated.
   * Owns one parameter [2][H] (row 0 a_src, row 1 a_dst), Glorot-initialised and trained like a Linear weight.
   * Supported: heads in {1, 2, 4, 8}, H <= 256 and F % 4 == 0 when heads > 1.  The backward assumes a symmetric
   * in-edge CSR (quirk Q1).  Takes part in no epilogue fusion. */
  Tensor graph_attention(const Tensor& _input, int heads, float negativeSlope = 0.2f);
  void softmax_cross_entropy(const Tensor& logits, const Tensor& labels, const Tensor& mask);
  Tensor indegree_norm(const Tensor& _input);
  Tensor linear(const Tensor& _input, int outDim, ActiMode activation, Initializer* initializer = NULL);
  Tensor relu(const Tensor& _input);
  Tensor sigmoid(const Tensor& _input);
  template <typename DT> Tensor create_node_tensor(int _numHidden) const;
  Tensor create_weight_tensor(int _inDim, int _outDim, Initializer* initializer) const;
  void load_features(const Tensor& input, const std::string& filename);
  void load_labels(const Tensor& label, const std::string& filename);
  void load_train_mask(const Tensor& mask, const std::string& filename);
  bool init(const Config& config);
  void train_mode(void);
  void infer_mode(void);
  void forward(void);
  void backward(void);
  void update(void);
  void zero_gradients(void);

  /* ---- additions (not in gnn.h): host<->device access to this partition's rows ---- */
  /* Copy `rows_local x H` values between a dense host buffer and the tensor. */
  void set_tensor(const Tensor& t, const void* host, bool grad = false);
  void get_tensor(const Tensor& t, void* host, bool grad = false) const;
  /* labels as class indices (what load_labels parses, load_task.cu:118-123) */
  void set_labels(const Tensor& label, const int* host_class_idx);
  roc_perf_metrics last_metrics(void) const;   /* PerfMetrics of the latest softmax pass */
  void set_fusion(bool on) { fuse = on; }
  int64_t local_rows(void) const { return (int64_t)myGraph.rowRight - myGraph.rowLeft + 1; }

public:
  ModelMode mode;
  Graph myGraph;
  Context ctx;
  Runtime* runtime;
  Optimizer* optimizer;
  std::vector<Tensor> parameters;
  std::vector<GnnOp*> layers;
  int epoch_num;
  bool fuse;          /* fuse linear->norm and SG->norm->relu into kernel epilogues (default on) */
  bool printMetrics;  /* print the [INFER] accuracy line like softmax_kernel.cu:141-152 (default on) */
};

class GnnOp {  /* gnn.h:205-222 */
public:
  GnnOp(const Tensor& input);
  GnnOp(const Tensor& input1, const Tensor& input2);
  GnnOp(const Tensor& input1, const Tensor& input2, const Tensor& input3);
  virtual ~GnnOp() {}
  virtual void init(const Model& model) = 0;
  virtual void forward(const Model& model) = 0;
  virtual void backward(const Model& model) = 0;
public:
  int numInputs, numOutputs;
  ModelMode mode;
  Tensor inputs[MAX_NUM_INPUTS], outputs[MAX_NUM_OUTPUTS];
  bool trainableInputs[MAX_NUM_INPUTS];
  bool resetInputGrads[MAX_NUM_INPUTS];
  /* host-side scheduling state (not in gnn.h) */
  int fusedInto;    /* >= 0: this op's work is done by layers[fusedInto] */
};

class ScatterGather : public GnnOp {  /* gnn.h:225-242, scattergather.cc */
public:
  ScatterGather(const Model& model, const Tensor& input, AggrType aggr = AGGR_SUM);
  virtual void init(const Model& model);
  virtual void forward(const Model& model);
  virtual void backward(const Model& model);
  AggrType aggr;
  int scratch;       /* AVG: region of the backward's D^-1 dOut rows (+ halo rows); -1 otherwise */
  int argRegion;     /* MAX / MIN: region of the u32 winner ids [rows (+ halo)][ld] the backward reads; -1 otherwise */
  int epilogue;      /* ROC_SG_EPI_* the forward store applies (set by Model::init fusion) */
  int bwdEpilogue;   /* same for the backward launch */
  int fwdOut, bwdOut;/* region the fused forward / backward writes (-1: own output / input grad) */
};

class GraphAttention : public GnnOp {  /* not in the reference */
public:
  GraphAttention(const Model& model, const Tensor& input, int heads, float slope);
  virtual void init(const Model& model);
  virtual void forward(const Model& model);
  virtual void backward(const Model& model);
  int heads;
  float slope;
  Tensor weight;      /* [2][H]: a_src, a_dst */
  int attRegion;      /* per-node s_src | s_dst [rows (+ halo)][round_up4(2 heads)] */
  int bstRegion;      /* per-node lse | c, same shape */
  int dsRegion;       /* backward: ds_src | ds_dst of the own rows */
  void* work;         /* backward: the da partials (roc_gat_finish_workspace_bytes) */
};

class InDegreeNorm : public GnnOp {  /* gnn.h:244-261, graphnorm.cc */
public:
  InDegreeNorm(const Model& model, const Tensor& input);
  virtual void init(const Model& model);
  virtual void forward(const Model& model);
  virtual void backward(const Model& model);
  int reluMaskOf;   /* backward: also apply the relu mask of this region's values (-1: none) */
  int bwdIn;        /* region whose grad is read in backward (-1: own output) */
  bool bwdFused;    /* backward done in another op's epilogue (a Linear's dX or the softmax) */
};

class Linear : public GnnOp {  /* gnn.h:263-285, linear.cc */
public:
  Linear(const Model& model, const Tensor& input, int outDim, ActiMode _activaiton, Initializer* initializer);
  void init(const Model& model);
  void forward(const Model& model);
  void backward(const Model& model);
public:
  ActiMode activation;
  Tensor weight;
  int flags;        /* ROC_LINEAR_* (norm epilogue fused) */
  int fwdOut;       /* region the forward writes (-1: own output) */
  int bwdIn;        /* region whose grad feeds backward (-1: own output) */
  int dropOp;       /* >= 0: layers[dropOp] is the Dropout feeding this op, applied while X is loaded */
  uint32_t* dropMask;      /* packed keep-mask of that dropout, [rows][dropLd] (roc_dropout_mask) */
  int64_t dropLd;
  /* dX epilogue fusions: relu mask of region dxReluOf's values, then / sqrt(deg); dX goes to dxOut's grad */
  int dxReluOf;     /* -1: none */
  bool dxNorm;
  int dxOut;        /* -1: the input's own grad */
};

class Activation : public GnnOp {  /* gnn.h:287-302, activation.cc */
public:
  Activation(const Model& model, const Tensor& input, ActiMode _actiMode);
  void init(const Model& model);
  void forward(const Model& model);
  void backward(const Model& model);
public:
  ActiMode actiMode;
};

class Element : public GnnOp {  /* gnn.h:304-319, element.cc */
public:
  Element(const Model& model, const Tensor& input0, const Tensor& input1, ElementType _elementType);
  void init(const Model& model);
  void forward(const Model& model);
  void backward(const Model& model);
public:
  ElementType elementType;
};

class Dropout : public GnnOp {  /* gnn.h:321-344, dropout.cc */
public:
  Dropout(const Model& model, const Tensor& input, float rate, int seed);
  virtual void init(const Model& model);
  virtual void forward(const Model& model);
  virtual void backward(const Model& model);
public:
  float rate;
  int seed;
  int opIndex;      /* position in the model: distinguishes the Philox streams of the layers */
};

class SoftmaxCrossEntropy : public GnnOp {  /* gnn.h:346-363, softmax.cc */
public:
  SoftmaxCrossEntropy(const Model& model, const Tensor& logits, const Tensor& labels, const Tensor& mask);
  virtual void init(const Model& model);
  virtual void forward(const Model& model);
  virtual void backward(const Model& model);
public:
  int epoch_num;
  int gradOut;      /* >= 0: write the logits' grad / sqrt(deg) into this region's grad (fused norm backward) */
};

/* CLI of the reference driver, gnn.cc:114-179 (same flags, same `-dr` quirk). */
void parse_input_args(char** argv, int argc, Config& config);

#endif /* ROC_GNN_H_ */
