// elementwise.cu — the HBM-bound pointwise ops of the GCN path for sm_100a:
// indegree_norm (+fused relu-mask backward), activation, add, dropout (Philox),
// softmax-cross-entropy backward + metrics (one kernel), Adam, scale, fill,
// device CSR build.  Each replaces a reference kernel or cuDNN call; see
// include/roc_b200.h for the file:line each one stands in for.
//
// All are grid-stride kernels over [rows][H] windows of [rows][ld] tensors,
// 16-byte vectorised when H, ld and the base pointers allow, launched with a
// grid that is a multiple of the SM count (148 on B200).
#include <initializer_list>
#include "common.cuh"

namespace roc {

std::atomic<uint64_t> g_launches{0};

// SMs a persistent / grid-stride launch sizes itself for: the device's count minus what the calling thread
// reserved with roc_set_sm_reserve (so that a peer-write exchange running on another stream finds free SMs:
// the tcgen05 GEMMs hold a whole SM's registers and shared memory per CTA, nothing can co-reside with them).
static thread_local int t_smReserve = 0;
int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, dev) != cudaSuccess) return 148;
    n = p.multiProcessorCount > 0 ? p.multiProcessorCount : 148;
  }
  const int avail = n - t_smReserve;
  return avail > 8 ? avail : 8;
}

static inline unsigned ew_grid(int64_t work_items, int threads) {
  int64_t need = (work_items + threads - 1) / threads;
  int64_t cap = (int64_t)sm_count() * 16;
  if (need < 1) need = 1;
  return (unsigned)(need < cap ? need : cap);
}

constexpr int EW_T = 256;

// ---------------------------------------------------------------- norm ------
template <int VEC>
__global__ void __launch_bounds__(EW_T)
k_norm(int64_t rows, int Wq, uint64_t colLeft, const uint64_t* __restrict__ rowEnd,
       const float* __restrict__ in, int64_t ldIn, float* __restrict__ out, int64_t ldOut,
       const float* __restrict__ reluOf, int64_t ldR) {
  const int64_t total = rows * (int64_t)Wq;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / Wq;
    int c = (int)(i - r * Wq);
    uint64_t s = (r == 0) ? colLeft : rowEnd[r - 1];
    uint32_t deg = (uint32_t)(rowEnd[r] - s);   // V_ID inDegree, graphnorm_kernel.cu:32,44
    float d = sqrtf((float)deg);
    if (VEC == 4) {
      float4 v = *reinterpret_cast<const float4*>(in + r * ldIn + 4 * c);
      if (reluOf) {
        float4 y = *reinterpret_cast<const float4*>(reluOf + r * ldR + 4 * c);
        v.x = (y.x > 0.f) ? v.x : 0.f; v.y = (y.y > 0.f) ? v.y : 0.f;
        v.z = (y.z > 0.f) ? v.z : 0.f; v.w = (y.w > 0.f) ? v.w : 0.f;
      }
      // zero numerators skip the divide (they would take div.rn's slow path; 0/d == 0 for d != 0)
      const bool dz = (d == 0.0f);
      if (v.x != 0.f || dz) v.x /= d;
      if (v.y != 0.f || dz) v.y /= d;
      if (v.z != 0.f || dz) v.z /= d;
      if (v.w != 0.f || dz) v.w /= d;
      *reinterpret_cast<float4*>(out + r * ldOut + 4 * c) = v;
    } else {
      float v = in[r * ldIn + c];
      if (reluOf) v = (reluOf[r * ldR + c] > 0.f) ? v : 0.f;
      out[r * ldOut + c] = (v != 0.f || d == 0.0f) ? v / d : v;
    }
  }
}

// out = in / (float)deg with the row-uniform IEEE divide (common.cuh); degree-0 rows give 0
template <int VEC>
__global__ void __launch_bounds__(EW_T)
k_deg_div(int64_t rows, int Wq, uint64_t colLeft, const uint64_t* __restrict__ rowEnd,
          const float* __restrict__ in, int64_t ldIn, float* __restrict__ out, int64_t ldOut) {
  const int64_t total = rows * (int64_t)Wq;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / Wq;
    const int c = (int)(i - r * Wq);
    const uint64_t s = (r == 0) ? colLeft : rowEnd[r - 1];
    const uint32_t deg = (uint32_t)(rowEnd[r] - s);
    if (VEC == 4) {
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      if (deg) {
        const float4 x = *reinterpret_cast<const float4*>(in + r * ldIn + 4 * c);
        v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w;
        rowdiv4(v, rowdiv_make((float)deg));
      }
      *reinterpret_cast<float4*>(out + r * ldOut + 4 * c) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
      out[r * ldOut + c] = deg ? rowdiv(in[r * ldIn + c], rowdiv_make((float)deg)) : 0.f;
    }
  }
}

// ---------------------------------------------------------- generic maps ----
enum { OP_RELU_F, OP_SIGM_F, OP_RELU_B, OP_SIGM_B, OP_ADD_F, OP_COPY };

template <int OP, int VEC, bool ACC>
__global__ void __launch_bounds__(EW_T)
k_map(int64_t rows, int Wq, const float* __restrict__ a, int64_t lda, const float* __restrict__ b,
      int64_t ldb, float* __restrict__ o, int64_t ldo) {
  const int64_t total = rows * (int64_t)Wq;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / Wq;
    int c = (int)(i - r * Wq) * VEC;
    float av[VEC], bv[VEC], ov[VEC];
    if (VEC == 4) {
      *reinterpret_cast<float4*>(av) = *reinterpret_cast<const float4*>(a + r * lda + c);
      if (b) *reinterpret_cast<float4*>(bv) = *reinterpret_cast<const float4*>(b + r * ldb + c);
      if (ACC) *reinterpret_cast<float4*>(ov) = *reinterpret_cast<const float4*>(o + r * ldo + c);
    } else {
      av[0] = a[r * lda + c];
      if (b) bv[0] = b[r * ldb + c];
      if (ACC) ov[0] = o[r * ldo + c];
    }
#pragma unroll
    for (int k = 0; k < VEC; k++) {
      float res;
      if (OP == OP_RELU_F) res = relu_nanprop(av[k]);
      else if (OP == OP_SIGM_F) res = 1.0f / (1.0f + expf(-av[k]));
      else if (OP == OP_RELU_B) res = (av[k] > 0.f) ? bv[k] : 0.f;           // a = y, b = dy
      else if (OP == OP_SIGM_B) res = bv[k] * av[k] * (1.0f - av[k]);
      else if (OP == OP_ADD_F) res = av[k] + bv[k];
      else res = av[k];
      ov[k] = ACC ? ov[k] + res : res;
    }
    if (VEC == 4) *reinterpret_cast<float4*>(o + r * ldo + c) = *reinterpret_cast<float4*>(ov);
    else o[r * ldo + c] = ov[0];
  }
}

// add backward: dA (+)= dY ; dB (+)= dY in one pass over dY
template <int VEC>
__global__ void __launch_bounds__(EW_T)
k_add_bwd(int64_t rows, int Wq, const float* __restrict__ dy, int64_t ldy, float* __restrict__ da,
          int64_t lda, int accA, float* __restrict__ db, int64_t ldb, int accB) {
  const int64_t total = rows * (int64_t)Wq;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / Wq;
    int c = (int)(i - r * Wq) * VEC;
#pragma unroll
    for (int k = 0; k < VEC; k++) {
      float g = dy[r * ldy + c + k];
      if (da) da[r * lda + c + k] = accA ? da[r * lda + c + k] + g : g;
      if (db) db[r * ldb + c + k] = accB ? db[r * ldb + c + k] + g : g;
    }
  }
}

// -------------------------------------------------------------- dropout -----
__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}

// keep(row, col) = 16-bit lane (col & 7) of Philox4x32-10(counter = {row lo, row hi, col >> 3, step},
// key = {seed lo, seed hi}) >= T16, lanes numbered low half of word 0, high half of word 0, low half
// of word 1, ...  T16 = round(rate * 65536): one Philox call decides 8 consecutive columns of a row.
__host__ __device__ inline uint32_t dropout_thresh16(float rate) {
  double t = (double)rate * 65536.0 + 0.5;
  return (t >= 65535.0) ? 65535u : (uint32_t)t;
}
// bit l of the result = keep of lane l (l = 0..7) of one Philox block
__device__ __forceinline__ uint32_t dropout_keep8(uint64_t row, uint32_t grp, uint32_t step, uint32_t seedLo,
                                                  uint32_t seedHi, uint32_t thresh16) {
  uint32_t c[4] = {(uint32_t)row, (uint32_t)(row >> 32), grp, step};
  philox4x32_10(c, seedLo, seedHi);
  uint32_t bits = 0u;
#pragma unroll
  for (int w = 3; w >= 0; w--) {
    bits = bits + bits + ((c[w] >> 16) >= thresh16 ? 1u : 0u);
    bits = bits + bits + ((c[w] & 0xFFFFu) >= thresh16 ? 1u : 0u);
  }
  return bits;
}

// One thread handles the 8 columns of one Philox block of UNR different (row, block) items per
// iteration, all loads issued before the Philox rounds.  VEC == 1 is the scalar fallback for
// unpadded layouts.
template <int VEC, int UNR>
__global__ void __launch_bounds__(EW_T)
k_dropout(int64_t rows, int H, int64_t firstRow, uint32_t thresh16, float scale, uint32_t seedLo,
          uint32_t seedHi, uint32_t step, const float* __restrict__ x, int64_t ldx,
          float* __restrict__ y, int64_t ldy) {
  const int Wq = (H + 7) / 8;
  const int64_t total = rows * (int64_t)Wq;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i0 < total; i0 += stride * UNR) {
    float xv[UNR][8];
    int64_t rr[UNR]; int cc[UNR];
#pragma unroll
    for (int u = 0; u < UNR; u++) {
      const int64_t i = i0 + u * stride;
      const bool ok = i < total;
      const int64_t r = ok ? i / Wq : 0;
      const int c = ok ? (int)(i - r * Wq) * 8 : 0;
      rr[u] = ok ? r : -1; cc[u] = c;
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int ch = c + 4 * h;
        if (ok && VEC == 4 && ch + 4 <= H)
          *reinterpret_cast<float4*>(&xv[u][4 * h]) = *reinterpret_cast<const float4*>(x + r * ldx + ch);
        else
#pragma unroll
          for (int j = 0; j < 4; j++) xv[u][4 * h + j] = (ok && ch + j < H) ? x[r * ldx + ch + j] : 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < UNR; u++) {
      if (rr[u] < 0) continue;
      const int64_t r = rr[u]; const int c = cc[u];
      const uint32_t keep = dropout_keep8((uint64_t)(firstRow + r), (uint32_t)(c >> 3), step, seedLo, seedHi, thresh16);
      float yv[8];
#pragma unroll
      for (int j = 0; j < 8; j++) yv[j] = ((keep >> j) & 1u) ? xv[u][j] * scale : 0.f;
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int ch = c + 4 * h;
        if (VEC == 4 && ch + 4 <= H) *reinterpret_cast<float4*>(y + r * ldy + ch) = *reinterpret_cast<float4*>(&yv[4 * h]);
        else
#pragma unroll
          for (int j = 0; j < 4; j++) if (ch + j < H) y[r * ldy + ch + j] = yv[4 * h + j];
      }
    }
  }
}

// The same mask, packed: bit b of mask[r][w] = keep(row r, column 32 w + b): four Philox blocks per
// word.  Words beyond ceil(H/32) and bits beyond H are written as zero so whole rows can be fetched
// blindly.
__global__ void __launch_bounds__(EW_T)
k_dropout_mask(int64_t rows, int H, int64_t firstRow, uint32_t thresh16, uint32_t seedLo, uint32_t seedHi,
               uint32_t step, uint32_t* __restrict__ mask, int64_t ldm) {
  const int Ww = (H + 31) / 32;
  const int64_t total = rows * ldm;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / ldm;
    const int w = (int)(i - r * ldm);
    uint32_t bits = 0u;
    if (w < Ww) {
#pragma unroll
      for (int b = 0; b < 4; b++)
        bits |= dropout_keep8((uint64_t)(firstRow + r), (uint32_t)(4 * w + b), step, seedLo, seedHi, thresh16) << (8 * b);
      const int n = H - 32 * w;
      if (n < 32) bits &= (1u << n) - 1u;
    }
    mask[i] = bits;
  }
}

// --------------------------------------------------- softmax + loss + grad ---
// One warp per row.  Lanes stride the C columns.  Metrics are reduced per block
// in shared memory and added to *perf with one atomic per field per block.
template <bool ONEHOT>
__global__ void __launch_bounds__(256)
k_softmax_xent(int64_t rows, int C, const float* __restrict__ z, int64_t ldz,
               const float* __restrict__ onehot, int64_t ldl, const int32_t* __restrict__ labelIdx,
               const int32_t* __restrict__ mask, float* __restrict__ g, int64_t ldg,
               roc_perf_metrics* perf, const uint64_t* __restrict__ rowEnd, uint64_t colLeft) {
  __shared__ float sLoss;
  __shared__ int sCnt[6];
  if (threadIdx.x == 0) sLoss = 0.f;
  if (threadIdx.x < 6) sCnt[threadIdx.x] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int warpsPerBlock = blockDim.x >> 5;
  float myLoss = 0.f;
  int cnt[6] = {0, 0, 0, 0, 0, 0};  // trainAll, testAll, valAll, trainCorrect, testCorrect, valCorrect
  for (int64_t r = blockIdx.x * (int64_t)warpsPerBlock + (threadIdx.x >> 5); r < rows;
       r += (int64_t)gridDim.x * warpsPerBlock) {
    const float* zr = z + r * ldz;
    RowDiv rd = rowdiv_make(1.0f);
    if (rowEnd) {
      const uint64_t st = (r == 0) ? colLeft : rowEnd[r - 1];
      rd = rowdiv_make(sqrtf((float)(uint32_t)(rowEnd[r] - st)));
    }
    float m = -INFINITY;
    for (int c = lane; c < C; c += 32) m = fmaxf(m, zr[c]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float sum = 0.f;
    for (int c = lane; c < C; c += 32) sum += expf(zr[c] - m);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    // argmax of p with calc_loss's rule (softmax_kernel.cu:51-57): maxVal starts at
    // 0.0f, strict '>', first index wins; true label = index with label > 0.5
    float best = 0.0f; int bestIdx = -1; int trueIdx = -1; float pTrue = 0.f;
    const int mk = mask[r];
    int tl = ONEHOT ? -1 : labelIdx[r];
    for (int c = lane; c < C; c += 32) {
      float p = expf(zr[c] - m) / sum;
      if (p > best) { best = p; bestIdx = c; }
      float lab;
      if (ONEHOT) { lab = onehot[r * ldl + c]; if (lab > 0.5f) trueIdx = c; }
      else lab = (c == tl) ? 1.0f : 0.0f;
      if (!ONEHOT && c == tl) trueIdx = c;
      if (trueIdx == c) pTrue = p;
      float gv = (mk == ROC_MASK_TRAIN) ? p - lab : 0.0f;
      if (rowEnd) gv = rowdiv(gv, rd);     // fused InDegreeNorm backward (== gv / sqrtf(deg))
      g[r * ldg + c] = gv;
    }
    // warp argmax: larger p wins, ties -> smaller index (what a serial first-max scan gives)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      float ob = __shfl_xor_sync(0xffffffffu, best, o);
      int oi = __shfl_xor_sync(0xffffffffu, bestIdx, o);
      if (ob > best || (ob == best && oi >= 0 && (bestIdx < 0 || oi < bestIdx))) { best = ob; bestIdx = oi; }
      int ot = __shfl_xor_sync(0xffffffffu, trueIdx, o);
      float op = __shfl_xor_sync(0xffffffffu, pTrue, o);
      if (ot > trueIdx) { trueIdx = ot; pTrue = op; }
    }
    if (lane == 0) {
      const bool ok = (trueIdx == bestIdx);
      if (mk == ROC_MASK_TRAIN) { myLoss += 1.0f - pTrue; cnt[0]++; if (ok) cnt[3]++; }
      else if (mk == ROC_MASK_VAL) { cnt[2]++; if (ok) cnt[5]++; }
      else if (mk == ROC_MASK_TEST) { cnt[1]++; if (ok) cnt[4]++; }
    }
  }
  if (perf) {
    if (lane == 0) {
      if (myLoss != 0.f) atomicAdd(&sLoss, myLoss);
#pragma unroll
      for (int k = 0; k < 6; k++) if (cnt[k]) atomicAdd(&sCnt[k], cnt[k]);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      if (sLoss != 0.f) atomicAdd(&perf->trainLoss, sLoss);
      if (sCnt[0]) atomicAdd(&perf->trainAll, sCnt[0]);
      if (sCnt[1]) atomicAdd(&perf->testAll, sCnt[1]);
      if (sCnt[2]) atomicAdd(&perf->valAll, sCnt[2]);
      if (sCnt[3]) atomicAdd(&perf->trainCorrect, sCnt[3]);
      if (sCnt[4]) atomicAdd(&perf->testCorrect, sCnt[4]);
      if (sCnt[5]) atomicAdd(&perf->valCorrect, sCnt[5]);
    }
  }
}

// Narrow-row version (C <= 4*LR): LR lanes per row, each lane keeps its (up to 4)
// logits in registers, so expf runs once per element and a warp handles 32/LR rows.
// Same arithmetic as k_softmax_xent (max, exp, sum, divide; first-max argmax).
template <bool ONEHOT, int LR>
__global__ void __launch_bounds__(256)
k_softmax_xent_narrow(int64_t rows, int C, const float* __restrict__ z, int64_t ldz,
                      const float* __restrict__ onehot, int64_t ldl, const int32_t* __restrict__ labelIdx,
                      const int32_t* __restrict__ mask, float* __restrict__ g, int64_t ldg,
                      roc_perf_metrics* perf, const uint64_t* __restrict__ rowEnd, uint64_t colLeft) {
  __shared__ float sLoss;
  __shared__ int sCnt[6];
  if (threadIdx.x == 0) sLoss = 0.f;
  if (threadIdx.x < 6) sCnt[threadIdx.x] = 0;
  __syncthreads();
  const int lr = threadIdx.x % LR;
  const unsigned gmask = (LR == 32) ? 0xffffffffu : (((1u << LR) - 1u) << (((threadIdx.x & 31) / LR) * LR));
  const int rowsPerBlock = blockDim.x / LR;
  float myLoss = 0.f;
  int cnt[6] = {0, 0, 0, 0, 0, 0};
  for (int64_t r = blockIdx.x * (int64_t)rowsPerBlock + threadIdx.x / LR; r < rows;
       r += (int64_t)gridDim.x * rowsPerBlock) {
    const float* zr = z + r * ldz;
    RowDiv rd = rowdiv_make(1.0f);
    if (rowEnd) {
      const uint64_t st = (r == 0) ? colLeft : rowEnd[r - 1];
      rd = rowdiv_make(sqrtf((float)(uint32_t)(rowEnd[r] - st)));
    }
    float v[4];
    float m = -INFINITY;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int c = lr + j * LR;
      v[j] = (c < C) ? zr[c] : -INFINITY;
      m = fmaxf(m, v[j]);
    }
#pragma unroll
    for (int o = LR / 2; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(gmask, m, o, LR));
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int c = lr + j * LR;
      v[j] = (c < C) ? expf(v[j] - m) : 0.f;
      sum += v[j];
    }
    // same summation tree for every row => deterministic; order differs from a serial loop (within 1e-4)
#pragma unroll
    for (int o = LR / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(gmask, sum, o, LR);
    const int mk = mask[r];
    const int tl = ONEHOT ? -1 : labelIdx[r];
    float best = 0.0f; int bestIdx = -1; int trueIdx = -1; float pTrue = 0.f;
    const RowDiv rsum = rowdiv_make(sum);      // p = v / sum, bit-identical to the IEEE divide (common.cuh)
    float pv[4] = {v[0], v[1], v[2], v[3]};    // columns beyond C hold 0 (a safe numerator)
    rowdiv4(pv, rsum);
    float gvv[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int c = lr + j * LR;
      gvv[j] = 0.f;
      if (c < C) {
        const float p = pv[j];
        if (p > best) { best = p; bestIdx = c; }
        float lab;
        if (ONEHOT) { lab = onehot[r * ldl + c]; if (lab > 0.5f) trueIdx = c; }
        else { lab = (c == tl) ? 1.0f : 0.0f; if (c == tl) trueIdx = c; }
        if (trueIdx == c) pTrue = p;
        gvv[j] = (mk == ROC_MASK_TRAIN) ? p - lab : 0.0f;
      }
    }
    if (rowEnd) rowdiv4(gvv, rd);             // fused InDegreeNorm backward (== gv / sqrtf(deg))
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int c = lr + j * LR;
      if (c < C) g[r * ldg + c] = gvv[j];
    }
    // argmax with calc_loss's rule (larger p wins, ties -> smaller index; bestIdx stays -1 when no
    // p > 0): max-reduce of the key (p bits, ~index) — p >= 0, so its bit pattern orders like the value
    unsigned long long key = (bestIdx < 0) ? 0ull
        : (((unsigned long long)__float_as_uint(best)) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)bestIdx);
#pragma unroll
    for (int o = LR / 2; o > 0; o >>= 1) {
      const unsigned long long ok = __shfl_xor_sync(gmask, key, o, LR);
      key = (ok > key) ? ok : key;
      if (ONEHOT) {
        int ot = __shfl_xor_sync(gmask, trueIdx, o, LR);
        float op = __shfl_xor_sync(gmask, pTrue, o, LR);
        if (ot > trueIdx) { trueIdx = ot; pTrue = op; }
      }
    }
    bestIdx = (key == 0ull) ? -1 : (int)(0xFFFFFFFFu - (uint32_t)key);
    if (!ONEHOT) {
      // the class index is known: its probability lives in lane (tl % LR) of this row's group
      const int owner = ((threadIdx.x & 31) / LR) * LR + ((tl >= 0 && tl < C) ? tl % LR : 0);
      const float fromOwner = __shfl_sync(gmask, pTrue, owner, 32);
      trueIdx = (tl >= 0 && tl < C) ? tl : -1;
      pTrue = (trueIdx >= 0) ? fromOwner : 0.f;
    }
    if (lr == 0) {
      const bool ok = (trueIdx == bestIdx);
      if (mk == ROC_MASK_TRAIN) { myLoss += 1.0f - pTrue; cnt[0]++; if (ok) cnt[3]++; }
      else if (mk == ROC_MASK_VAL) { cnt[2]++; if (ok) cnt[5]++; }
      else if (mk == ROC_MASK_TEST) { cnt[1]++; if (ok) cnt[4]++; }
    }
  }
  if (perf) {
    if (lr == 0) {
      if (myLoss != 0.f) atomicAdd(&sLoss, myLoss);
#pragma unroll
      for (int k = 0; k < 6; k++) if (cnt[k]) atomicAdd(&sCnt[k], cnt[k]);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      if (sLoss != 0.f) atomicAdd(&perf->trainLoss, sLoss);
      if (sCnt[0]) atomicAdd(&perf->trainAll, sCnt[0]);
      if (sCnt[1]) atomicAdd(&perf->testAll, sCnt[1]);
      if (sCnt[2]) atomicAdd(&perf->valAll, sCnt[2]);
      if (sCnt[3]) atomicAdd(&perf->trainCorrect, sCnt[3]);
      if (sCnt[4]) atomicAdd(&perf->testCorrect, sCnt[4]);
      if (sCnt[5]) atomicAdd(&perf->valCorrect, sCnt[5]);
    }
  }
}

template <bool ONEHOT>
static void launch_softmax(int64_t rows, int C, const float* logits, int64_t ldZ, const float* labels, int64_t ldL,
                           const int32_t* labelIdx, const int32_t* mask, float* grad, int64_t ldG,
                           roc_perf_metrics* perf, const uint64_t* rowEnd, uint64_t colLeft, cudaStream_t st) {
  if (C <= 32) {
    k_softmax_xent_narrow<ONEHOT, 8><<<ew_grid(rows * 8, 256), 256, 0, st>>>(rows, C, logits, ldZ, labels, ldL, labelIdx, mask, grad, ldG, perf, rowEnd, colLeft);
  } else if (C <= 64) {
    k_softmax_xent_narrow<ONEHOT, 16><<<ew_grid(rows * 16, 256), 256, 0, st>>>(rows, C, logits, ldZ, labels, ldL, labelIdx, mask, grad, ldG, perf, rowEnd, colLeft);
  } else if (C <= 128) {
    k_softmax_xent_narrow<ONEHOT, 32><<<ew_grid(rows * 32, 256), 256, 0, st>>>(rows, C, logits, ldZ, labels, ldL, labelIdx, mask, grad, ldG, perf, rowEnd, colLeft);
  } else {
    k_softmax_xent<ONEHOT><<<ew_grid(rows * 32, 256), 256, 0, st>>>(rows, C, logits, ldZ, labels, ldL, labelIdx, mask, grad, ldG, perf, rowEnd, colLeft);
  }
}

// ------------------------------------------------------------------ adam -----
__global__ void __launch_bounds__(EW_T)
k_adam(int64_t count, float alpha_t, float beta1, float beta2, float wd, float eps,
       const float* __restrict__ G, float* __restrict__ M, float* __restrict__ V, float* __restrict__ W) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count;
       i += (int64_t)gridDim.x * blockDim.x) {
    float gt = G[i] + wd * W[i];
    float mt = beta1 * M[i] + (1 - beta1) * gt;
    float vt = beta2 * V[i] + (1 - beta2) * gt * gt;
    M[i] = mt;
    V[i] = vt;
    W[i] -= alpha_t * mt / (sqrtf(vt) + eps);
  }
}

__global__ void __launch_bounds__(EW_T)
k_scale(int64_t count, float a, float b, float* __restrict__ w) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count;
       i += (int64_t)gridDim.x * blockDim.x)
    w[i] = (b - a) * w[i] + a;
}

__global__ void __launch_bounds__(EW_T)
k_fill(int64_t rows, int H, float value, float* __restrict__ x, int64_t ld) {
  const int64_t total = rows * (int64_t)H;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / H;
    x[r * ld + (i - r * H)] = value;
  }
}

// ------------------------------------------------------------- CSR build -----
// Edge-parallel (the reference loops serially over a vertex's edges,
// load_task.cu:289-292): edge e finds its row by binary search over rawRows.
__global__ void __launch_bounds__(EW_T)
k_build_csr_rows(uint32_t nloc, const uint64_t* __restrict__ rawRows, uint64_t* __restrict__ rowPtrs) {
  uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n < nloc) rowPtrs[n] = rawRows[n];
}

__global__ void __launch_bounds__(EW_T)
k_build_csr_edges(uint32_t rowLeft, uint32_t nloc, uint64_t colLeft, uint64_t nEdges,
                  const uint64_t* __restrict__ rawRows, const uint32_t* __restrict__ rawCols,
                  uint32_t* __restrict__ edgeStructs, uint32_t* __restrict__ colSrc) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < nEdges;
       i += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t src = rawCols[i];
    if (colSrc) colSrc[i] = src;
    if (edgeStructs) {
      uint64_t e = colLeft + i;          // global edge id; row = first n with rawRows[n] > e
      uint32_t lo = 0, hi = nloc;
      while (lo < hi) {
        uint32_t mid = lo + ((hi - lo) >> 1);
        if (rawRows[mid] > e) hi = mid; else lo = mid + 1;
      }
      edgeStructs[2 * i] = src;
      edgeStructs[2 * i + 1] = lo + rowLeft;
    }
  }
}

static inline bool vec_ok(int H, std::initializer_list<int64_t> lds, std::initializer_list<const void*> ptrs) {
  if (H % 4) return false;
  for (int64_t l : lds) if (l % 4) return false;
  for (const void* p : ptrs) if (p && !aligned16(p)) return false;
  return true;
}

}  // namespace roc

using namespace roc;

extern "C" const char* roc_version(void) { return "roc_b200 0.1 (sm_100a)"; }

extern "C" int roc_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

extern "C" uint64_t roc_launch_count(void) { return g_launches.load(); }
extern "C" int roc_set_sm_reserve(int numSMs) {
  const int prev = t_smReserve;
  t_smReserve = numSMs > 0 ? numSMs : 0;
  return prev;
}

extern "C" int roc_partition(roc_vid_t numNodes, roc_eid_t numEdges, int numParts,
                             const roc_eid_t* raw_rows, roc_vid_t* vb, roc_eid_t* eb, int* numRanges) {
  if (!raw_rows || !vb || !eb || numParts <= 0 || numNodes == 0) return ROC_ERR_INVALID;
  // One pass over the row ends; a range closes on the vertex that pushes its
  // edge count past the cap, and whatever is left forms the last range.
  const roc_eid_t cap = (numEdges + (roc_eid_t)numParts - 1) / (roc_eid_t)numParts;
  int n = 0;
  roc_vid_t left = 0;
  roc_eid_t have = 0, prevEnd = 0;
  for (roc_vid_t v = 0; v < numNodes; ++v) {
    have += raw_rows[v] - prevEnd;
    prevEnd = raw_rows[v];
    if (have > cap) {
      if (n < numParts) { vb[2 * n] = left; vb[2 * n + 1] = v; }
      ++n; have = 0; left = v + 1;
    }
  }
  if (have > 0) {
    if (n < numParts) { vb[2 * n] = left; vb[2 * n + 1] = numNodes - 1; }
    ++n;
  }
  roc_eid_t lo = 0;
  for (int c = 0; c < n && c < numParts; ++c) {
    roc_eid_t end = raw_rows[vb[2 * c + 1]];
    eb[2 * c] = lo; eb[2 * c + 1] = end - 1; lo = end;
  }
  if (numRanges) *numRanges = n;
  return n == numParts ? ROC_OK : ROC_ERR_UNSUPPORTED;
}

extern "C" int roc_build_csr(roc_vid_t rowLeft, roc_vid_t rowRight, roc_eid_t colLeft,
                             const roc_eid_t* rawRows, const roc_vid_t* rawCols, roc_eid_t* rowPtrs,
                             roc_vid_t* edgeStructs, roc_vid_t* colSrc, roc_stream_t stream) {
  if (!rawRows || rowRight < rowLeft) return ROC_ERR_INVALID;
  cudaStream_t st = as_stream(stream);
  uint32_t nloc = rowRight - rowLeft + 1;
  if (rowPtrs) {
    k_build_csr_rows<<<(nloc + EW_T - 1) / EW_T, EW_T, 0, st>>>(nloc, rawRows, rowPtrs);
    ROC_LAUNCH_CHECK();
  }
  if (edgeStructs || colSrc) {
    uint64_t lastEnd = 0;
    ROC_CUDA(cudaMemcpyAsync(&lastEnd, rawRows + (nloc - 1), sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    ROC_CUDA(cudaStreamSynchronize(st));
    if (lastEnd < colLeft) return ROC_ERR_INVALID;
    uint64_t nE = lastEnd - colLeft;
    if (nE) {
      if (!rawCols) return ROC_ERR_INVALID;
      k_build_csr_edges<<<ew_grid((int64_t)nE, EW_T), EW_T, 0, st>>>(rowLeft, nloc, colLeft, nE, rawRows, rawCols,
                                                                  edgeStructs, colSrc);
      ROC_LAUNCH_CHECK();
    }
  }
  return ROC_OK;
}

extern "C" int roc_indegree_norm(roc_vid_t rowLeft, roc_vid_t rowRight, roc_eid_t colLeft, int H,
                                 const roc_eid_t* rowEnd, const float* in, int64_t ldIn, float* out,
                                 int64_t ldOut, const float* reluOf, roc_stream_t stream) {
  if (!rowEnd || !in || !out || H <= 0 || rowRight < rowLeft || ldIn < H || ldOut < H) return ROC_ERR_INVALID;
  int64_t rows = (int64_t)rowRight - rowLeft + 1;
  cudaStream_t st = as_stream(stream);
  // a fused relu mask shares the output's leading dimension convention: it is the
  // forward output tensor, same shape as `in`
  int64_t ldR = ldIn;
  // padded rows (ld % 4 == 0): whole float4s, the pad columns ride along (0 / d stays 0)
  if (vec_ok(4, {ldIn, ldOut}, {in, out, reluOf})) {
    const int Wq = (H + 3) / 4;
    k_norm<4><<<ew_grid(rows * Wq, EW_T), EW_T, 0, st>>>(rows, Wq, colLeft, rowEnd, in, ldIn, out, ldOut, reluOf, ldR);
  } else {
    k_norm<1><<<ew_grid(rows * H, EW_T), EW_T, 0, st>>>(rows, H, colLeft, rowEnd, in, ldIn, out, ldOut, reluOf, ldR);
  }
  ROC_LAUNCH_CHECK();
  return ROC_OK;
}

extern "C" int roc_indegree_div(roc_vid_t rowLeft, roc_vid_t rowRight, roc_eid_t colLeft, int H,
                                const roc_eid_t* rowEnd, const float* in, int64_t ldIn, float* out, int64_t ldOut,
                                roc_stream_t stream) {
  if (!rowEnd || !in || !out || H <= 0 || rowRight < rowLeft || ldIn < H || ldOut < H) return ROC_ERR_INVALID;
  const int64_t rows = (int64_t)rowRight - rowLeft + 1;
  cudaStream_t st = as_stream(stream);
  if (vec_ok(4, {ldIn, ldOut}, {in, out})) {
    const int Wq = (H + 3) / 4;
    k_deg_div<4><<<ew_grid(rows * Wq, EW_T), EW_T, 0, st>>>(rows, Wq, colLeft, rowEnd, in, ldIn, out, ldOut);
  } else {
    k_deg_div<1><<<ew_grid(rows * H, EW_T), EW_T, 0, st>>>(rows, H, colLeft, rowEnd, in, ldIn, out, ldOut);
  }
  ROC_LAUNCH_CHECK();
  return ROC_OK;
}

template <int OP, bool ACC>
static int launch_map(int64_t rows, int H, const float* a, int64_t lda, const float* b, int64_t ldb, float* o,
                      int64_t ldo, cudaStream_t st) {
  if (vec_ok(H, {lda, b ? ldb : 4, ldo}, {a, b, o}))
    k_map<OP, 4, ACC><<<ew_grid(rows * (H / 4), EW_T), EW_T, 0, st>>>(rows, H / 4, a, lda, b, ldb, o, ldo);
  else
    k_map<OP, 1, ACC><<<ew_grid(rows * H, EW_T), EW_T, 0, st>>>(rows, H, a, lda, b, ldb, o, ldo);
  ROC_LAUNCH_CHECK();
  return ROC_OK;
}

extern "C" int roc_activation_fwd(int64_t rows, int H, int mode, const float* x, int64_t ldX, float* y,
                                  int64_t ldY, roc_stream_t stream) {
  if (!x || !y || rows < 0 || H <= 0 || ldX < H || ldY < H) return ROC_ERR_INVALID;
  if (rows == 0) return ROC_OK;
  cudaStream_t st = as_stream(stream);
  if (mode == ROC_AC_MODE_RELU) return launch_map<OP_RELU_F, false>(rows, H, x, ldX, nullptr, 0, y, ldY, st);
  if (mode == ROC_AC_MODE_SIGMOID) return launch_map<OP_SIGM_F, false>(rows, H, x, ldX, nullptr, 0, y, ldY, st);
  return ROC_ERR_UNSUPPORTED;
}

extern "C" int roc_activation_bwd(int64_t rows, int H, int mode, const float* y, int64_t ldY, const float* dY,
                                  int64_t ldDY, float* dX, int64_t ldDX, int accumulate, roc_stream_t stream) {
  if (!y || !dY || !dX || rows < 0 || H <= 0 || ldY < H || ldDY < H || ldDX < H) return ROC_ERR_INVALID;
  if (rows == 0) return ROC_OK;
  cudaStream_t st = as_stream(stream);
  if (mode == ROC_AC_MODE_RELU)
    return accumulate ? launch_map<OP_RELU_B, true>(rows, H, y, ldY, dY, ldDY, dX, ldDX, st)
                      : launch_map<OP_RELU_B, false>(rows, H, y, ldY, dY, ldDY, dX, ldDX, st);
  if (mode == ROC_AC_MODE_SIGMOID)
    return accumulate ? launch_map<OP_SIGM_B, true>(rows, H, y, ldY, dY, ldDY, dX, ldDX, st)
                      : launch_map<OP_SIGM_B, false>(rows, H, y, ldY, dY, ldDY, dX, ldDX, st);
  return ROC_ERR_UNSUPPORTED;
}

extern "C" int roc_add_fwd(int64_t rows, int H, const float* a, int64_t ldA, const float* b, int64_t ldB,
                           float* y, int64_t ldY, roc_stream_t stream) {
  if (!a || !b || !y || rows < 0 || H <= 0 || ldA < H || ldB < H || ldY < H) return ROC_ERR_INVALID;
  if (rows == 0) return ROC_OK;
  return launch_map<OP_ADD_F, false>(rows, H, a, ldA, b, ldB, y, ldY, as_stream(stream));
}

extern "C" int roc_add_bwd(int64_t rows, int H, const float* dY, int64_t ldDY, float* dA, int64_t ldDA, int accA,
                           float* dB, int64_t ldDB, int accB, roc_stream_t stream) {
  if (!dY || rows < 0 || H <= 0 || ldDY < H) return ROC_ERR_INVALID;
  if (rows == 0 || (!dA && !dB)) return ROC_OK;
  k_add_bwd<1><<<ew_grid(rows * H, EW_T), EW_T, 0, as_stream(stream)>>>(rows, H, dY, ldDY, dA, ldDA, accA, dB, ldDB, accB);
  ROC_LAUNCH_CHECK();
  return ROC_OK;
}

static int dropout_launch(int64_t rows, int H, int64_t firstRow, float rate, uint64_t seed, uint32_t step,
                          const float* x, int64_t ldX, float* y, int64_t ldY, cudaStream_t st) {
  if (!x || !y || rows < 0 || H <= 0 || ldX < H || ldY < H || rate < 0.f || rate >= 1.f) return ROC_ERR_INVALID;
  if (rows == 0) return ROC_OK;
  uint32_t thresh = dropout_thresh16(rate);
  float scale = 1.0f / (1.0f - rate);
  bool vec = (ldX % 4 == 0) && (ldY % 4 == 0) && aligned16(x) && aligned16(y);
  if (vec)
    k_dropout<4, 2><<<ew_grid((rows * ((H + 7) / 8) + 1) / 2, EW_T), EW_T, 0, st>>>(rows, H, firstRow, thresh, scale, (uint32_t)seed,
                                                                   (uint32_t)(seed >> 32), step, x, ldX, y, ldY);
  else
    k_dropout<1, 2><<<ew_grid((rows * ((H + 7) / 8) + 1) / 2, EW_T), EW_T, 0, st>>>(rows, H, firstRow, thresh, scale, (uint32_t)seed,
                                                        (uint32_t)(seed >> 32), step, x, ldX, y, ldY);
  ROC_LAUNCH_CHECK();
  return ROC_OK;
}

extern "C" int roc_dropout_fwd(int64_t rows, int H, int64_t firstRow, float rate, uint64_t seed, uint32_t step,
                               const float* x, int64_t ldX, float* y, int64_t ldY, roc_stream_t stream) {
  return dropout_launch(rows, H, firstRow, rate, seed, step, x, ldX, y, ldY, as_stream(stream));
}

extern "C" int roc_dropout_bwd(int64_t rows, int H, int64_t firstRow, float rate, uint64_t seed, uint32_t step,
                               const float* dY, int64_t ldDY, float* dX, int64_t ldDX, roc_stream_t stream) {
  // dX = dY * keep / (1 - rate): the same map as forward (dropout_kernel.cu:149-150)
  return dropout_launch(rows, H, firstRow, rate, seed, step, dY, ldDY, dX, ldDX, as_stream(stream));
}

extern "C" int roc_dropout_mask(int64_t rows, int H, int64_t firstRow, float rate, uint64_t seed, uint32_t step,
                                uint32_t* mask, int64_t ldMask, roc_stream_t stream) {
  if (!mask || rows < 0 || H <= 0 || ldMask < (H + 31) / 32 || rate < 0.f || rate >= 1.f) return ROC_ERR_INVALID;
  if (rows == 0) return ROC_OK;
  k_dropout_mask<<<ew_grid(rows * ldMask, EW_T), EW_T, 0, as_stream(stream)>>>(
      rows, H, firstRow, dropout_thresh16(rate), (uint32_t)seed, (uint32_t)(seed >> 32), step, mask, ldMask);
  ROC_LAUNCH_CHECK();
  return ROC_OK;
}

extern "C" int roc_softmax_xent_bwd(int64_t rows, int C, const float* logits, int64_t ldZ, const float* labels,
                                    int64_t ldL, const int32_t* mask, float* grad, int64_t ldG,
                                    roc_perf_metrics* perf, roc_stream_t stream) {
  if (!logits || !labels || !mask || !grad || rows < 0 || C <= 0 || ldZ < C || ldL < C || ldG < C) return ROC_ERR_INVALID;
  if (rows == 0) return ROC_OK;
  launch_softmax<true>(rows, C, logits, ldZ, labels, ldL, nullptr, mask, grad, ldG, perf, nullptr, 0, as_stream(stream));
  ROC_LAUNCH_CHECK();
  return ROC_OK;
}

// Compact-label variant used by the host (int32 class index per row instead of
// the reference's one-hot fp32 [N][C] tensor: 4 B/row instead of 4C B/row).
extern "C" int roc_softmax_xent_bwd_idx(int64_t rows, int C, const float* logits, int64_t ldZ,
                                        const int32_t* labelIdx, const int32_t* mask, float* grad, int64_t ldG,
                                        roc_perf_metrics* perf, roc_stream_t stream) {
  if (!logits || !labelIdx || !mask || !grad || rows < 0 || C <= 0 || ldZ < C || ldG < C) return ROC_ERR_INVALID;
  if (rows == 0) return ROC_OK;
  launch_softmax<false>(rows, C, logits, ldZ, nullptr, 0, labelIdx, mask, grad, ldG, perf, nullptr, 0, as_stream(stream));
  ROC_LAUNCH_CHECK();
  return ROC_OK;
}

extern "C" int roc_softmax_xent_bwd_norm(int64_t rows, int C, const float* logits, int64_t ldZ, const float* labels,
                                         int64_t ldL, const int32_t* labelIdx, const int32_t* mask, float* grad,
                                         int64_t ldG, const roc_eid_t* rowEnd, roc_eid_t colLeft,
                                         roc_perf_metrics* perf, roc_stream_t stream) {
  if (!logits || !mask || !grad || !rowEnd || rows < 0 || C <= 0 || ldZ < C || ldG < C) return ROC_ERR_INVALID;
  if ((labels != nullptr) == (labelIdx != nullptr)) return ROC_ERR_INVALID;   // exactly one label form
  if (labels && ldL < C) return ROC_ERR_INVALID;
  if (rows == 0) return ROC_OK;
  if (labels) launch_softmax<true>(rows, C, logits, ldZ, labels, ldL, nullptr, mask, grad, ldG, perf, rowEnd, colLeft, as_stream(stream));
  else launch_softmax<false>(rows, C, logits, ldZ, nullptr, 0, labelIdx, mask, grad, ldG, perf, rowEnd, colLeft, as_stream(stream));
  ROC_LAUNCH_CHECK();
  return ROC_OK;
}

extern "C" int roc_adam_update(int64_t count, float alpha_t, float beta1, float beta2, float weight_decay,
                               float epsilon, const float* WGrad, float* M, float* V, float* W, roc_stream_t stream) {
  if (!WGrad || !M || !V || !W || count < 0) return ROC_ERR_INVALID;
  if (count == 0) return ROC_OK;
  k_adam<<<ew_grid(count, EW_T), EW_T, 0, as_stream(stream)>>>(count, alpha_t, beta1, beta2, weight_decay, epsilon, WGrad, M, V, W);
  ROC_LAUNCH_CHECK();
  return ROC_OK;
}

extern "C" int roc_scale(int64_t count, float a, float b, float* W, roc_stream_t stream) {
  if (!W || count < 0) return ROC_ERR_INVALID;
  if (count == 0) return ROC_OK;
  k_scale<<<ew_grid(count, EW_T), EW_T, 0, as_stream(stream)>>>(count, a, b, W);
  ROC_LAUNCH_CHECK();
  return ROC_OK;
}

// exhaustive check of the row-uniform division against div.rn (test hook)
__global__ void __launch_bounds__(256)
k_selftest_rowdiv(float d, uint64_t firstBits, uint64_t count, unsigned long long* mismatches) {
  const roc::RowDiv rd = roc::rowdiv_make(d);
  unsigned long long bad = 0;
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
    const float a = __uint_as_float((uint32_t)(firstBits + i));
    const float want = a / d;
    const float got = roc::rowdiv(a, rd);
    if (__float_as_uint(want) != __float_as_uint(got) && !(want != want && got != got)) bad++;
  }
  if (bad) atomicAdd(mismatches, bad);
}

extern "C" int roc_selftest_rowdiv(float d, uint64_t firstBits, uint64_t count, uint64_t* d_mismatches,
                                   roc_stream_t stream) {
  if (!d_mismatches) return ROC_ERR_INVALID;
  k_selftest_rowdiv<<<sm_count() * 8, 256, 0, as_stream(stream)>>>(d, firstBits, count,
                                                                 reinterpret_cast<unsigned long long*>(d_mismatches));
  ROC_LAUNCH_CHECK();
  return ROC_OK;
}

extern "C" int roc_copy2d(int64_t rows, int H, const float* src, int64_t ldSrc, float* dst, int64_t ldDst,
                          roc_stream_t stream) {
  if (!src || !dst || rows < 0 || H <= 0 || ldSrc < H || ldDst < H) return ROC_ERR_INVALID;
  if (rows == 0) return ROC_OK;
  return launch_map<OP_COPY, false>(rows, H, src, ldSrc, nullptr, 0, dst, ldDst, as_stream(stream));
}

extern "C" int roc_fill(int64_t rows, int H, float value, float* x, int64_t ld, roc_stream_t stream) {
  if (!x || rows < 0 || H <= 0 || ld < H) return ROC_ERR_INVALID;
  if (rows == 0) return ROC_OK;
  k_fill<<<ew_grid(rows * H, EW_T), EW_T, 0, as_stream(stream)>>>(rows, H, value, x, ld);
  ROC_LAUNCH_CHECK();
  return ROC_OK;
}
