/*
 * roc_b200.h — C ABI of the B200-native kernel layer for ROC's GCN-training path.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference has no FFI: its
 * device code is reached through Legion task variants
 *   static void X::forward_task(const Task*, const std::vector<PhysicalRegion>&, Context, Runtime*)
 * (gnn.h:224-349, registered gnn.cc:241-426).  Every entry point below replaces
 * the CUDA work one of those tasks did; the comment on each cites the task /
 * kernel / library call it stands in for.  INTEGRATION.md shows the stub a ROC
 * maintainer adds inside each *_task to call it.
 *
 * Conventions
 *  - plain C, no torch / Legion types; all data pointers are DEVICE pointers
 *    unless a name says `host`; caller owns every buffer;
 *  - `roc_stream_t` is a `cudaStream_t`; calls enqueue work and return (no
 *    device sync) unless documented otherwise;
 *  - return value: 0 = ROC_OK; > 0 = a cudaError_t; < 0 = ROC_ERR_*;
 *  - node tensors are row-major [rows][ld] fp32 with `ld >= H` floats between
 *    rows (the reference's layout is ld == H, gnn.cc:480-486).  The vectorised
 *    paths need ld % 4 == 0 and 16-byte aligned bases; other shapes take a
 *    scalar path.  Pad columns H..ld-1 may be read and rewritten by the
 *    vectorised paths (whole float4s) but never influence columns < H; the host
 *    keeps them zero;
 *  - graph ids follow types.h:5-15: V_ID = uint32, E_ID = uint64;
 *    rowEnd[v-rowLeft] is the GLOBAL END offset of v's in-edge list
 *    (NodeStruct.index, load_task.cu:283-288), the first local row starts at
 *    colLeft (scattergather_kernel.cu:46-50); colSrc[e-colLeft] is the source
 *    vertex of edge e (EdgeStruct.src; the redundant .dst is dropped).
 */
#ifndef ROC_B200_H_
#define ROC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef uint32_t roc_vid_t;   /* V_ID,  types.h:5 */
typedef uint64_t roc_eid_t;   /* E_ID,  types.h:6 */
typedef void*    roc_stream_t; /* cudaStream_t */

#define ROC_OK               0
#define ROC_ERR_INVALID     (-1)  /* bad argument (NULL pointer, negative size ...) */
#define ROC_ERR_UNSUPPORTED (-2)  /* shape outside what the kernels handle */
#define ROC_ERR_NOMEM       (-3)
#define ROC_ERR_NO_DEVICE   (-4)  /* no CUDA device: the product has no CPU fallback */
#define ROC_ERR_IO          (-5)

/* ActiMode, gnn.h:82-86 */
#define ROC_AC_MODE_NONE    0
#define ROC_AC_MODE_RELU    1
#define ROC_AC_MODE_SIGMOID 2

/* MaskType, gnn.h:98-103 */
#define ROC_MASK_TRAIN 0
#define ROC_MASK_VAL   1
#define ROC_MASK_TEST  2
#define ROC_MASK_NONE  3

/* epilogue fused into the ScatterGather store (what the model applies right
 * after it, gnn.cc:83-85): NORM = the following indegree_norm, RELU = the relu
 * after that.  Applied in that order.  MEAN divides the row's sum by (float)deg
 * (one IEEE division; degree-0 rows stay 0): the AVG aggregator.  It combines with
 * RELU (MEAN first); MEAN | NORM is rejected. */
#define ROC_SG_EPI_NONE 0
#define ROC_SG_EPI_NORM 1
#define ROC_SG_EPI_RELU 2
#define ROC_SG_EPI_MEAN 4

/* AggrType of gnn.h:75-80 (the values of roc_gnn.h's enum) */
#define ROC_AGGR_AVG 0
#define ROC_AGGR_MAX 1
#define ROC_AGGR_MIN 2
#define ROC_AGGR_SUM 3

/* PerfMetrics, softmax_kernel.cu:35-39 (same field order) */
typedef struct {
  float trainLoss;
  int trainAll, testAll, valAll, trainCorrect, testCorrect, valCorrect;
} roc_perf_metrics;

const char* roc_version(void);
/* Number of usable CUDA devices (0 if none); never fails. */
int roc_device_count(void);
/* Total kernels this library has launched in this process (for bench's gpu_launches). */
uint64_t roc_launch_count(void);
/* Persistent / grid-stride kernels launched by the CALLING THREAD from now on size their grids for
 * (SMs - numSMs), leaving SMs to work running beside them on another stream (the peer-write halo exchange:
 * a tcgen05 GEMM CTA holds a whole SM, nothing co-resides with it).  0 restores full-chip grids.  Returns the
 * previous reserve. */
int roc_set_sm_reserve(int numSMs);

/* ---------------------------------------------------------------- graph --- */

/* Replaces Graph::Graph's partition loop, gnn.cc:806-829 + 852-870 (HOST code,
 * host pointers).  Greedy edge-balanced contiguous vertex ranges; a range is
 * closed when its in-edge count exceeds ceil(E/P) (strict).  vbounds[2c..2c+1] =
 * [left,right] inclusive, ebounds[2c..2c+1] = [lo,hi] inclusive.  Returns the
 * number of ranges produced in *numRanges; the reference asserts it equals
 * numParts (gnn.cc:829) — here that case returns ROC_ERR_UNSUPPORTED after
 * filling what fits. */
int roc_partition(roc_vid_t numNodes, roc_eid_t numEdges, int numParts,
                  const roc_eid_t* host_rowEnd, roc_vid_t* host_vbounds,
                  roc_eid_t* host_ebounds, int* numRanges);

/* Replaces init_graph_kernel, load_task.cu:271-294.  From the partition's raw
 * slices (rawRows = global END offsets of local rows, rawCols = sources) writes
 *   rowPtrs[n]  = rawRows[n]                          (NodeStruct, u64)     if non-NULL
 *   edgeStructs = {src = rawCols[e], dst = n+rowLeft} (EdgeStruct, 2 x u32) if non-NULL
 *   colSrc[e]   = rawCols[e]                          (lean u32 layout)     if non-NULL */
int roc_build_csr(roc_vid_t rowLeft, roc_vid_t rowRight, roc_eid_t colLeft,
                  const roc_eid_t* rawRows, const roc_vid_t* rawCols,
                  roc_eid_t* rowPtrs, roc_vid_t* edgeStructs, roc_vid_t* colSrc,
                  roc_stream_t stream);

/* -------------------------------------------------------- ScatterGather --- */

/* A plan holds the edge-balanced schedule for one partition's CSR: 64-edge
 * chunks, the first row of each chunk, carry slots for rows longer than a
 * chunk.  It is a private, derived structure; rowEnd/colSrc stay the canonical
 * CSR and must outlive the plan.  Creation synchronises the stream. */
typedef struct roc_sg_plan roc_sg_plan;

int roc_sg_plan_create(roc_vid_t rowLeft, roc_vid_t rowRight, roc_eid_t colLeft,
                       const roc_eid_t* rowEnd, const roc_vid_t* colSrc,
                       roc_stream_t stream, roc_sg_plan** plan);
/* Pre-size the carry workspace for feature widths up to maxH (otherwise it is grown on the stream of the first
 * call that needs it, with stream-ordered allocation: no device synchronisation, but the plan must then be used
 * from that one stream). */
int roc_sg_plan_reserve(roc_sg_plan* plan, int maxH);
void roc_sg_plan_destroy(roc_sg_plan* plan);
/* Introspection for tests / DESIGN.md numbers. */
int roc_sg_plan_info(const roc_sg_plan* plan, uint64_t* numChunks,
                     uint64_t* numCarries, uint64_t* numHeavyRows);

/* Replaces aggre_coop_kernel + ScatterGather::forward_task,
 * scattergather_kernel.cu:20-76, 78-158:
 *   out[v-rowLeft][h] = sum_{e in in(v)} in[colSrc[e]][h],  h < H
 * `in` is indexed by whatever ids colSrc holds (global ids over the whole
 * [N][ldIn] matrix as in scattergather.cc:69-73, or local+halo ids).
 * Deterministic: the per-row summation order is fixed by the plan — and is the same in every kernel variant the
 * library may pick for a width (registers / cp.async / TMA gather4 rings; ROC_SG_VARIANT forces one), so results
 * do not depend on the variant either. */
int roc_sg_forward_planned(const roc_sg_plan* plan, int H, const float* in,
                           int64_t ldIn, float* out, int64_t ldOut, int epilogue,
                           roc_stream_t stream);

/* Plan-less form with exactly the reference kernel's argument list
 * (scattergather_kernel.cu:21-28, EdgeStruct.dst dropped), dense ld == H.
 * Builds and frees a plan internally (synchronises); use the planned form in
 * loops. */
int roc_sg_forward(roc_vid_t rowLeft, roc_vid_t rowRight, roc_eid_t colLeft, int H,
                   const roc_eid_t* rowEnd, const roc_vid_t* colSrc,
                   const float* in, float* out, roc_stream_t stream);
/* Replaces ScatterGather::backward_task, scattergather_kernel.cu:160-170: the
 * identical computation on gradients (A, not A^T — quirk Q1). */
int roc_sg_backward(roc_vid_t rowLeft, roc_vid_t rowRight, roc_eid_t colLeft, int H,
                    const roc_eid_t* rowEnd, const roc_vid_t* colSrc,
                    const float* outGrad, float* inGrad, roc_stream_t stream);

/* MAX / MIN aggregation (aggr = ROC_AGGR_MAX | ROC_AGGR_MIN) over the plan's rows:
 *   out[v-rowLeft][h] = max / min over e in in(v) of in[col(e)][h]
 *   arg[v-rowLeft][h] = colGlobal[e] of the winning edge
 * The winner is the FIRST edge in CSR order among equal values; a NaN candidate replaces a non-NaN best (the
 * first NaN wins, like torch.amax); +-inf are ordinary values.  Degree-0 rows: out = 0, arg = 0xFFFFFFFF.
 * colGlobal (u32, parallel to the plan's colSrc) is the canonical global source id of each edge, so that arg
 * means the same on every partition; NULL = the plan's own colSrc (single partition).  arg == NULL skips the arg
 * stores (no backward follows).  Same chunk schedule as roc_sg_forward_planned, no atomics, bit-reproducible.
 * Always the register kernel (ROC_SG_VARIANT does not apply); widths past 1024 floats run in column blocks,
 * unaligned leading dimensions take a scalar path.  `arg` needs ldArg >= H u32 per row. */
int roc_sg_aggr_forward(const roc_sg_plan* plan, int aggr, int H, const float* in, int64_t ldIn,
                        const roc_vid_t* colGlobal, float* out, int64_t ldOut, uint32_t* arg,
                        int64_t ldArg, roc_stream_t stream);
/* Backward of MAX / MIN, as a gather over the same plan (no atomics, no reverse exchange):
 *   inGrad[u-rowLeft][h] = sum over e in in(u) of (arg[col(e)][h] == u ? outGrad[col(e)][h] : skipped)
 * outGrad and arg are indexed like the forward's input (col ids: global, or local + halo rows); the sum runs in
 * the plan's per-row order.  Exact only where SUM's backward is (quirk Q1): the in-edge CSR must be symmetric and
 * free of duplicate edges, so that in(u) lists every v whose in-edges contain u.  Ties send the whole gradient
 * to the recorded winner. */
int roc_sg_arg_backward(const roc_sg_plan* plan, int H, const float* outGrad, int64_t ldG, const uint32_t* arg,
                        int64_t ldArg, roc_vid_t rowLeft, float* inGrad, int64_t ldIn, roc_stream_t stream);
/* Pre-size the u32 carry slots roc_sg_aggr_forward uses for rows cut at chunk boundaries (like
 * roc_sg_plan_reserve for the float ones, which it also reserves), for widths up to maxH. */
int roc_sg_plan_reserve_arg(roc_sg_plan* plan, int maxH);

/* Graph attention (GAT, one layer, K heads) over the plan's rows.  h is [rows][H] with H = K*F, head k the columns
 * [kF, (k+1)F); attW is the op's parameter [2][H]: row 0 a_src, row 1 a_dst.  Per-node tensors (K <= 8):
 *   att [rows][ldAtt >= 2K]: s_src[r][k] = <h[r, k-block], a_src[k-block]> at column k, s_dst at column K + k
 *   bst [rows][ldB >= 2K]:   lse[r][k] at column k (the forward), c[r][k] = <dOut[r, k-block], out[r, k-block]> at
 *                            column K + k (the backward)
 * For a row v, its in-edges u (CSR order) and head k:
 *   e = LeakyReLU(s_src[u][k] + s_dst[v][k], slope);  lse[v][k] = max e + log sum exp(e - max e)
 *   alpha = expf(e - lse[v][k]);  out[v, k-block] = sum_u alpha h[u, k-block]
 * A degree-0 row has out = 0 and lse = 0.  alpha is recomputed wherever it is needed, by one device function.
 * Tensors the gathers index (h, att, bst, outGrad) are indexed by the plan's col ids, and their rows 0 .. nloc-1
 * are the plan's own rows ([own | halo] in the multi-GPU engine; the whole matrix with rowLeft = 0 otherwise).
 * Supported: K in {1, 2, 4, 8}, 1 <= H <= 256, and F % 4 == 0 when K > 1; anything else is ROC_ERR_UNSUPPORTED.
 * Pad columns (past H) enter no dot and no sum.  No atomics: every result is bit-reproducible. */
int roc_gat_supported(int H, int heads);
/* Size the plan's carry slots for the widest GAT pass at width H (init time; nothing is allocated in a step). */
int roc_gat_plan_reserve(roc_sg_plan* plan, int H, int heads);
/* att[r] = (s_src[r] | s_dst[r]) for rows 0 .. rows-1. */
int roc_gat_scores(int64_t rows, int H, int heads, const float* h, int64_t ldH, const float* attW, float* att,
                   int64_t ldAtt, roc_stream_t stream);
/* lse (into bst's first K columns of the own rows) in one pass over the edges, then out in a second. */
int roc_gat_forward(const roc_sg_plan* plan, int H, int heads, float slope, const float* h, int64_t ldH,
                    const float* att, int64_t ldAtt, float* bst, int64_t ldB, float* out, int64_t ldOut,
                    roc_stream_t stream);
/* c[r][k] = <outGrad[r, k-block], out[r, k-block]> into bst's columns K .. 2K-1, rows 0 .. rows-1. */
int roc_gat_bwd_c(int64_t rows, int H, int heads, const float* outGrad, int64_t ldG, const float* out,
                  int64_t ldOut, float* bst, int64_t ldB, roc_stream_t stream);
/* The backward gather.  Row u walks its in-edges v (which, with a symmetric in-edge CSR, are the rows u feeds;
 * quirk Q1 as for every aggregator's backward):
 *   inGrad[u]     = sum_v alpha[v<-u] outGrad[v]                                                (overwritten)
 *   ds[u][k]      = sum_v alpha[v<-u,k] (<outGrad[v], h[u]>_k - c[v][k]) LeakyReLU'(s_src[u][k] + s_dst[v][k])
 *   ds[u][K + k]  = sum_v alpha[u<-v,k] (<outGrad[u], h[v]>_k - c[u][k]) LeakyReLU'(s_src[v][k] + s_dst[u][k])
 * with LeakyReLU'(z) = 1 if z > 0 else slope.  ds is [nloc][ldDs >= 2K]. */
int roc_gat_backward(const roc_sg_plan* plan, int H, int heads, float slope, const float* h, int64_t ldH,
                     const float* att, int64_t ldAtt, const float* bst, int64_t ldB, const float* outGrad,
                     int64_t ldG, float* inGrad, int64_t ldIn, float* ds, int64_t ldDs, roc_stream_t stream);
/* inGrad[r][j] += ds[r][k(j)] a_src[j] + ds[r][K + k(j)] a_dst[j]  (rows 0 .. rows-1), and
 * attGrad[0][j] = sum_r ds[r][k(j)] h[r][j], attGrad[1][j] = sum_r ds[r][K + k(j)] h[r][j] (overwritten), as
 * fixed row blocks summed in block order.  workspace: roc_gat_finish_workspace_bytes(H). */
size_t roc_gat_finish_workspace_bytes(int H);
int roc_gat_bwd_finish(int64_t rows, int H, int heads, const float* h, int64_t ldH, const float* attW,
                       const float* ds, int64_t ldDs, float* inGrad, int64_t ldIn, float* attGrad, void* workspace,
                       size_t workspaceBytes, roc_stream_t stream);

/* ----------------------------------------------------------------- halo --- */

/* Boundary-node structures of one partition (multi-GPU).  The reference hands every
 * partition the WHOLE input region before ScatterGather (scattergather.cc:69-73); here a
 * partition receives only the distinct remote rows its edges read.  From the partition's
 * sources (global ids, device) builds
 *   ids[nHalo]      sorted distinct sources outside [rowLeft, rowRight] (grouped by owner,
 *                   since partitions are contiguous id ranges)
 *   colLocal[nEdges] = src - rowLeft (own rows) | Nloc + rank in ids (halo rows)
 * — a private, derived copy; colSrc stays the canonical CSR.  Synchronises the stream. */
typedef struct roc_halo roc_halo;
int roc_halo_create(roc_vid_t rowLeft, roc_vid_t rowRight, uint64_t nEdges, const roc_vid_t* colSrc,
                    roc_stream_t stream, roc_halo** out);
void roc_halo_destroy(roc_halo* h);
uint32_t roc_halo_size(const roc_halo* h);
const roc_vid_t* roc_halo_ids(const roc_halo* h);         /* device */
const roc_vid_t* roc_halo_col_local(const roc_halo* h);   /* device */
/* Host-side bookkeeping of the exchange (HOST pointers, no device work).  recv: the sorted halo ids are
 * grouped by owner (partitions are contiguous id ranges, host_vbounds as in roc_partition):
 * recvOffs[q] / recvCounts[q] = first halo row owned by partition q / how many; ROC_ERR_INVALID if the
 * list is not strictly increasing, leaves every range, or names one of this partition's own rows.
 * send: host_allCounts[q * P + r] = rows partition q requests from owner r (every rank's recvCounts,
 * all-gathered); this rank packs the rows q asked of it for q = 0..P-1 in order. */
int roc_halo_recv_layout(uint32_t nHalo, const roc_vid_t* host_ids, int numParts, int myPart,
                         const roc_vid_t* host_vbounds, uint64_t* recvCounts, uint64_t* recvOffs);
int roc_halo_send_layout(int numParts, int myPart, const int32_t* host_allCounts, uint64_t* sendCounts,
                         uint64_t* sendOffs, uint64_t* numSendRows);
/* roc_pack_rows for a subset: dst[sel[t]] = src[rows[sel[t]]] for t < nSel — the send-list entries of one row
 * block, written to their places in the send buffer, so that the block can travel (copy engines, peer slabs) while
 * the producer computes the next one. */
int roc_pack_rows_at(int64_t nSel, int H, const roc_vid_t* sel, const roc_vid_t* rows, const float* src,
                     int64_t ldSrc, float* dst, int64_t ldDst, roc_stream_t stream);
/* Fused pack + exchange over peer memory: row srcRows[j] of `src` is stored to
 * host_peerBase[peer[j]] + dstRow[j] * ldDst — the halo slab of the partition that reads it, in ANOTHER GPU's
 * memory (device pointers the caller mapped with cudaIpcOpenMemHandle; the stores travel over NVLink).  Replaces
 * roc_pack_rows + the NCCL all-to-all-v of the staged rows (themselves the replacement of the reference's
 * whole-region request, scattergather.cc:69-73).  srcRows / peer / dstRow are device arrays of nRows entries;
 * host_peerBase is a HOST array of numPeers <= ROC_MAX_PEERS device pointers (entries never named by peer[] may be
 * NULL).  smLimit > 0 sizes the grid for that many SMs (the ones a producer running beside it left free, see
 * roc_set_sm_reserve); 0 = whole chip.  The caller orders the consumer after every producer (a barrier across
 * the partitions). */
#define ROC_MAX_PEERS 16
int roc_push_rows(int64_t nRows, int H, const roc_vid_t* srcRows, const uint8_t* peer, const roc_vid_t* dstRow,
                  const float* src, int64_t ldSrc, float* const* host_peerBase, int numPeers, int64_t ldDst,
                  int smLimit, roc_stream_t stream);
/* dst[j][0:H] = src[rows[j]][0:H]: packs the rows another partition asked for into a send buffer. */
int roc_pack_rows(int64_t nRows, int H, const roc_vid_t* rows, const float* src, int64_t ldSrc,
                  float* dst, int64_t ldDst, roc_stream_t stream);

/* ---------------------------------------------------------- elementwise --- */

/* Replaces norm_coop_kernel, graphnorm_kernel.cu:19-57 (fwd and bwd :126-136):
 * out[n][h] = in[n][h] / sqrtf((float)deg(n)); in/out are the partition's rows.
 * If `also_relu_mask_of` is non-NULL (fused backward of relu∘norm, gnn.cc:84-85):
 * out = (also_relu_mask_of > 0 ? in : 0) / sqrtf(deg); it has `in`'s shape and
 * leading dimension (it is the relu output whose gradient `in` is). */
int roc_indegree_norm(roc_vid_t rowLeft, roc_vid_t rowRight, roc_eid_t colLeft, int H,
                      const roc_eid_t* rowEnd, const float* in, int64_t ldIn,
                      float* out, int64_t ldOut, const float* also_relu_mask_of,
                      roc_stream_t stream);
/* out[n][h] = in[n][h] / (float)deg(n), IEEE division (row-uniform reciprocal form, bit-identical to `/`);
 * degree-0 rows give 0.  The AVG aggregator's backward scaling (D^-1 dOut). */
int roc_indegree_div(roc_vid_t rowLeft, roc_vid_t rowRight, roc_eid_t colLeft, int H,
                     const roc_eid_t* rowEnd, const float* in, int64_t ldIn, float* out,
                     int64_t ldOut, roc_stream_t stream);

/* Replaces cudnnActivationForward/Backward, activation_kernel.cu:64-66, 128-132.
 * bwd: dX (+)= dY * f'(.) evaluated from the OUTPUT y; accumulate != 0 adds
 * into dX (the reference's beta = 1 on a loaded buffer, gnn.cc:704-713). */
int roc_activation_fwd(int64_t rows, int H, int mode, const float* x, int64_t ldX,
                       float* y, int64_t ldY, roc_stream_t stream);
int roc_activation_bwd(int64_t rows, int H, int mode, const float* y, int64_t ldY,
                       const float* dY, int64_t ldDY, float* dX, int64_t ldDX,
                       int accumulate, roc_stream_t stream);

/* Replaces op_kernel (EW_TYPE_ADD), element_kernel.cu:19-39, and its backward
 * add_kernel pair, :93-101. */
int roc_add_fwd(int64_t rows, int H, const float* a, int64_t ldA, const float* b,
                int64_t ldB, float* y, int64_t ldY, roc_stream_t stream);
int roc_add_bwd(int64_t rows, int H, const float* dY, int64_t ldDY, float* dA,
                int64_t ldDA, int accA, float* dB, int64_t ldDB, int accB,
                roc_stream_t stream);

/* Replaces cudnnDropoutForward/Backward, dropout_kernel.cu:98-99, 149-150.
 * y = keep ? x / (1 - rate) : 0.  cuDNN's generator is not reproducible, so the
 * mask is defined here instead: element (globalRow r, column c) keeps iff 16-bit
 * lane (c & 7) of Philox4x32-10(counter = {r lo, r hi, c >> 3, step},
 * key = {seed lo, seed hi}) >= round(rate * 65536); lanes are numbered low half
 * of word 0, high half of word 0, low half of word 1, ...  One Philox block
 * decides 8 consecutive columns of one row; the mask does not depend on the
 * tensor's width or on how rows are split across GPUs.  It is recomputed in bwd
 * (no reserve space).  `firstRow` = global index of the slab's first row (rowLeft). */
int roc_dropout_fwd(int64_t rows, int H, int64_t firstRow, float rate, uint64_t seed,
                    uint32_t step, const float* x, int64_t ldX, float* y, int64_t ldY,
                    roc_stream_t stream);
int roc_dropout_bwd(int64_t rows, int H, int64_t firstRow, float rate, uint64_t seed,
                    uint32_t step, const float* dY, int64_t ldDY, float* dX,
                    int64_t ldDX, roc_stream_t stream);

/* The same mask, packed one bit per element: bit (h & 31) of
 * mask[row * ldMask + (h >> 5)] = keep(firstRow + row, h).  ldMask (32-bit words per
 * row) must be a multiple of 4 and >= ceil(H/32); words / bits beyond H are written 0.
 * Feeds roc_linear_fwd_dropout / roc_linear_bwd_dropout, which apply dropout to the
 * Linear's input while loading it, so the dropped copy of X (dropout_kernel.cu:98's
 * output tensor) is never written to or re-read from HBM. */
int roc_dropout_mask(int64_t rows, int H, int64_t firstRow, float rate, uint64_t seed,
                     uint32_t step, uint32_t* mask, int64_t ldMask, roc_stream_t stream);

/* Replaces SoftmaxCrossEntropy::backward_task, softmax_kernel.cu:81-171:
 * cudnnSoftmaxForward(ACCURATE) -> calc_loss (:41-79) -> softmax_backward
 * (:19-33) in ONE kernel.  `labels` is the one-hot fp32 [rows][ldL] tensor the
 * reference loads (load_task.cu:118-123); `mask` is int32 per row.
 * `perf` (device, may be NULL) is ACCUMULATED into (zero it first). */
int roc_softmax_xent_bwd(int64_t rows, int C, const float* logits, int64_t ldZ,
                         const float* labels, int64_t ldL, const int32_t* mask,
                         float* grad, int64_t ldG, roc_perf_metrics* perf,
                         roc_stream_t stream);

/* Same computation with compact labels: labelIdx[v] = class index (what
 * load_task.cu:118-123 expands to one-hot); 4 B/row instead of 4C B/row. */
int roc_softmax_xent_bwd_idx(int64_t rows, int C, const float* logits, int64_t ldZ,
                             const int32_t* labelIdx, const int32_t* mask, float* grad,
                             int64_t ldG, roc_perf_metrics* perf, roc_stream_t stream);

/* roc_softmax_xent_bwd(_idx) with the backward of the InDegreeNorm that produced the logits
 * (gnn.cc:85 / graphnorm_kernel.cu:133) folded in: grad[v] = ((P - labels) or 0) / sqrtf(deg(v)).
 * Exactly one of `labels` (one-hot fp32) / `labelIdx` (class index per row) is non-NULL;
 * rowEnd is rowLeft-relative as everywhere.  Bit-identical to roc_softmax_xent_bwd followed
 * by roc_indegree_norm on the gradient. */
int roc_softmax_xent_bwd_norm(int64_t rows, int C, const float* logits, int64_t ldZ,
                              const float* labels, int64_t ldL, const int32_t* labelIdx,
                              const int32_t* mask, float* grad, int64_t ldG,
                              const roc_eid_t* rowEnd, roc_eid_t colLeft,
                              roc_perf_metrics* perf, roc_stream_t stream);

/* --------------------------------------------------------------- Linear --- */

/* Replaces cublasSgemm in Linear::forward_task, linear_kernel.cu:76-80 (+ the
 * optional in-place ReLU :83-104):  Y[v][o] = sum_i X[v][i] * W[o*inDim + i].
 * W is the reference's column-major [inDim][outDim] weight (ld = inDim, Q6).
 * flags: ROC_LINEAR_NORM_EPILOGUE divides row v by sqrtf(deg(v)) (fuses the
 * indegree_norm that follows linear in the model, gnn.cc:81-82); then needs
 * rowLeft-relative rowEnd/colLeft (else pass NULL/0). */
#define ROC_LINEAR_NORM_EPILOGUE 1
int roc_linear_fwd(int64_t rows, int inDim, int outDim, const float* X, int64_t ldX,
                   const float* W, float* Y, int64_t ldY, int activation, int flags,
                   const roc_eid_t* rowEnd, roc_eid_t colLeft, roc_stream_t stream);

/* Replaces Linear::backward_task, linear_kernel.cu:129-245:
 *   if activation == RELU: dY = (Y > 0) ? dY : 0 in place (reluBackward :120-127)
 *   dW[o*inDim+i] += sum_v X[v][i] * dY[v][o]        (sgemm beta = 1, :220-224)
 *   dX[v][i] (+)= sum_o W[o*inDim+i] * dY[v][o]       (:227-231) — skipped when
 *   dX == NULL (leaf input, quirk Q8); accumulate_dX selects += vs =.
 * `workspace` holds split-K partials of dW; size from roc_linear_bwd_workspace_bytes. */
/* roc_linear_fwd on dropout(X): Y = (keep ? X / (1 - rate) : 0) W^T with `mask` from
 * roc_dropout_mask (same rate).  Bit-identical to roc_dropout_fwd followed by
 * roc_linear_fwd.  rate == 0 ignores the mask (infer mode: dropout is a copy,
 * dropout_kernel.cu:159-180). */
int roc_linear_fwd_dropout(int64_t rows, int inDim, int outDim, const float* X, int64_t ldX,
                           const float* W, float* Y, int64_t ldY, int activation, int flags,
                           const roc_eid_t* rowEnd, roc_eid_t colLeft, const uint32_t* mask,
                           int64_t ldMask, float rate, roc_stream_t stream);

size_t roc_linear_bwd_workspace_bytes(int64_t rows, int inDim, int outDim);
int roc_linear_bwd(int64_t rows, int inDim, int outDim, const float* X, int64_t ldX,
                   const float* W, const float* Y, int64_t ldY, float* dY,
                   int64_t ldDY, float* dW, float* dX, int64_t ldDX,
                   int activation, int accumulate_dX, void* workspace,
                   size_t workspaceBytes, roc_stream_t stream);

/* roc_linear_bwd where the forward input was dropout(X) (X = the tensor BEFORE dropout):
 * dW uses the masked, scaled X; dX (if non-NULL) is the gradient of the dropout's INPUT,
 * i.e. cudnnDropoutBackward (dropout_kernel.cu:149-150) applied to the Linear's dX in
 * the same kernel.  Bit-identical to roc_linear_bwd followed by roc_dropout_bwd. */
int roc_linear_bwd_dropout(int64_t rows, int inDim, int outDim, const float* X, int64_t ldX,
                           const float* W, const float* Y, int64_t ldY, float* dY,
                           int64_t ldDY, float* dW, float* dX, int64_t ldDX, int activation,
                           int accumulate_dX, void* workspace, size_t workspaceBytes,
                           const uint32_t* mask, int64_t ldMask, float rate,
                           roc_stream_t stream);

/* roc_linear_bwd with the backward of the ops upstream of X folded into the dX epilogue,
 * so dX is written once, already as the gradient the next ScatterGather backward reads.
 * In model order (gnn.cc:81-88)  ... -> indegree_norm -> relu -> dropout -> linear:
 *   dX = dY W                                           (linear_kernel.cu:227-231)
 *   dX = keep ? dX / (1 - dropRate) : 0   if dropMask    (dropout_kernel.cu:149-150)
 *   dX = dxReluOf > 0 ? dX : 0            if dxReluOf    (Activation backward, cudnnActivationBackward
 *                                                         on the stored relu output, activation_kernel.cu)
 *   dX = dX / sqrtf(deg(row))             if dxNormRowEnd (InDegreeNorm backward, graphnorm_kernel.cu:133)
 * Zero / NULL fields switch the stage off; with all off this is roc_linear_bwd.  Each stage is
 * bit-identical to the separate kernel it replaces. */
typedef struct roc_linear_bwd_args {
  int64_t rows; int inDim, outDim;
  const float* X; int64_t ldX;
  const float* W;
  const float* Y; int64_t ldY;
  float* dY; int64_t ldDY;
  float* dW;
  float* dX; int64_t ldDX;
  int activation, accumulate_dX;
  void* workspace; size_t workspaceBytes;
  const uint32_t* dropMask; int64_t ldMask; float dropRate;
  const float* dxReluOf; int64_t ldReluOf;
  const roc_eid_t* dxNormRowEnd; roc_eid_t colLeft;
  int parts;   /* 0 = dW and dX (if non-NULL); ROC_LINEAR_BWD_ONLY_DX / _ONLY_DW compute one of them — the host
                * computes dX in row blocks (each pushed to the partitions that read it while the next is computed)
                * and dW, which nothing waits for, last.  Only with activation == NONE (no in-place relu backward). */
} roc_linear_bwd_args;
#define ROC_LINEAR_BWD_ONLY_DX 1
#define ROC_LINEAR_BWD_ONLY_DW 2
int roc_linear_bwd_fused(const roc_linear_bwd_args* args, roc_stream_t stream);

/* Test hook: which kernel family served the calling thread's last Linear GEMM — which = 0 forward, 1 dW, 2 dX;
 * returns ROC_GEMM_PATH_TCGEN05, ROC_GEMM_PATH_SIMT (the exact-fp32 fallback for shapes / alignments the tensor-core
 * kernels do not take) or 0 (none yet). */
#define ROC_GEMM_PATH_TCGEN05 1
#define ROC_GEMM_PATH_SIMT 2
int roc_last_gemm_path(int which);

/* ------------------------------------------------------------ optimizer --- */

/* Replaces adam_update, optimizer_kernel.cu:43-63 (launch :98-101).  alpha_t is
 * the bias-corrected step computed on the host in double (optimizer.cc:79-85).
 * The reference first sums per-GPU replicas g0 += g_i (:88-94); here WGrad is
 * already the all-reduced gradient. */
int roc_adam_update(int64_t count, float alpha_t, float beta1, float beta2,
                    float weight_decay, float epsilon, const float* WGrad, float* M,
                    float* V, float* W, roc_stream_t stream);

/* Replaces GlorotUniform::init_task's scale_kernel, initializer_kernel.cu:46-47 +
 * cuda_helper.cu:2-9: W = (b - a) * u + a over `count` uniforms already in W. */
int roc_scale(int64_t count, float a, float b, float* W, roc_stream_t stream);
/* Replaces assign_kernel, cuda_helper.cu:11-18 (zero_grad_task_impl,
 * ZerosInitializer): 2-D fill of the [rows][H] window of a [rows][ld] tensor. */
int roc_fill(int64_t rows, int H, float value, float* x, int64_t ld, roc_stream_t stream);
/* Test hook: the fused indegree_norm epilogues divide by a row-uniform sqrtf(deg) with a shared
 * reciprocal + FMA correction instead of one div.rn per element.  Counts, over the `count` fp32 bit
 * patterns starting at firstBits, how many results differ from `x / d` (must be 0; NaN == NaN).
 * *d_mismatches (device u64) is accumulated into. */
int roc_selftest_rowdiv(float d, uint64_t firstBits, uint64_t count, uint64_t* d_mismatches,
                        roc_stream_t stream);
/* Replaces copy_kernel, cuda_helper.cu:20-27 (dropout's infer path, staging): 2-D copy of
 * the [rows][H] window between tensors of different leading dimensions. */
int roc_copy2d(int64_t rows, int H, const float* src, int64_t ldSrc, float* dst, int64_t ldDst,
               roc_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* ROC_B200_H_ */
