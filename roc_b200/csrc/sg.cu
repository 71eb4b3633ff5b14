// sg.cu — ScatterGather (CSR row-parallel SpMM, sum aggregation) for sm_100a.
//
// Replaces aggre_coop_kernel + ScatterGather::{forward,backward}_task
// (reference scattergather_kernel.cu:20-76, 78-170).  The reference walks one
// edge per H-thread group per iteration and accumulates with shared-memory
// float atomics; this is a different algorithm built for HBM3e:
//
//  * edge-balanced schedule ("plan"): the partition's edge array is cut into
//    CH = 64-edge chunks; one WORKER owns chunk c.  A row is owned by the chunk
//    its first edge lies in.  Rows no longer than CH are always finished by their
//    owner (so a worker does at most 2*CH-1 edges); a longer ("heavy") row is cut
//    at chunk boundaries: the owner stores its raw partial, every later chunk
//    stores its part into a carry slot and a second small kernel adds partial +
//    carries in chunk order.  No atomics anywhere => bit-reproducible sums (the
//    reference is not: smem atomicAdd, scattergather_kernel.cu:66).  The plan also
//    holds a 32-byte start record per chunk (k_chunk_desc) so a worker begins with
//    one load instead of a three-deep dependent walk.
//  * the store applies the ops the model puts right after scatter_gather
//    (indegree_norm, relu; gnn.cc:83-85) so the N x H result is written once.
//  * FIVE main kernels share that plan and the per-row summation order — they are
//    bit-identical to each other — and differ in how the neighbour rows travel:
//      A  sg_chunk_kernel      registers: L = min(32, H/4) lanes per worker, one LDG.128 per lane and row,
//                              8 rows in flight per lane (default up to 64 floats per row)
//      C  sg_chunk_kernel_c2   cp.async (LDGSTS) ring per worker (rows wider than 256 floats)
//      T  sg_chunk_kernel_t    TMA: one cp.async.bulk.tensor ... tile::gather4 per 4 edges into a shared-memory
//                              ring per worker, mbarrier completion (default for 129..256 floats)
//      U  (T, MODE 2)          the same with the source ids held by the lanes that issue them (65..128 floats)
//      b  (T, MODE 1)          one plain cp.async.bulk per row (measurement only)
//      R  sg_ring_kernel       producer / consumer ring: producer warps issue gather4s for whole chunks into a
//                              two-slot ring, two worker warps consume (the structure the measured gather ceilings
//                              ask for; not yet faster — DESIGN.md §3.1)
//    The choice per width is by measurement (pick_variant); ROC_SG_VARIANT forces one.
//
// Algorithmic bytes per launch (DESIGN.md): E*(4H+4) + Nloc*(4H+8).
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <new>
#include "common.cuh"
#include "tc_common.cuh"

namespace roc {

constexpr int SG_CH = 64;          // edges per chunk
constexpr int SG_THREADS = 256;    // threads per CTA

}  // namespace roc

struct roc_sg_plan {
  uint32_t nloc = 0, E = 0, numChunks = 0, numCarries = 0, numHeavy = 0, numBig = 0;
  uint32_t* rs = nullptr;         // [nloc+1]   local row starts (rs[r+1] = rowEnd[r]-colLeft)
  uint32_t* firstRow = nullptr;   // [numChunks+1] first row whose start >= c*CH
  uint32_t* carryIdx = nullptr;   // [numChunks+1] exclusive scan of carry-in flags
  uint32_t* heavyRows = nullptr;  // [numHeavy]  rows with degree > CH and <= 32 carries (one worker each)
  uint32_t* bigRows = nullptr;    // [numBig]    rows with more carries (one CTA each)
  const uint32_t* col = nullptr;  // caller's colSrc
  float* carry = nullptr;         // [numCarries][carryLd]
  size_t carryLd = 0;
  uint32_t* carryArg = nullptr;   // [numCarries][carryArgLd]  winner ids of the MAX / MIN carry parts
  size_t carryArgLd = 0;
  uint64_t inRows = 1;            // 1 + largest source id in col: the rows a TMA tensor map of the input spans
  uint32_t* desc = nullptr;       // [numChunks][8] per-chunk start state of the ring kernel (k_chunk_desc)
  int device = 0;
};

namespace roc {

// ------------------------------------------------------------ plan kernels ---

__global__ void k_build_rs(uint32_t nloc, uint64_t colLeft, const uint64_t* __restrict__ rowEnd,
                           uint32_t* __restrict__ rs) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) rs[0] = 0;
  if (i < nloc) rs[i + 1] = (uint32_t)(rowEnd[i] - colLeft);
}

__global__ void k_first_row(uint32_t nloc, uint32_t numChunks, const uint32_t* __restrict__ rs,
                            uint32_t* __restrict__ firstRow) {
  uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c > numChunks) return;
  if (c == numChunks) { firstRow[c] = nloc; return; }
  uint32_t target = c * (uint32_t)SG_CH;
  uint32_t lo = 0, hi = nloc;  // first r in [0,nloc) with rs[r] >= target, else nloc
  while (lo < hi) {
    uint32_t mid = lo + ((hi - lo) >> 1);
    if (rs[mid] >= target) hi = mid; else lo = mid + 1;
  }
  firstRow[c] = lo;
}

__global__ void k_carry_flag(uint32_t numChunks, const uint32_t* __restrict__ rs,
                             const uint32_t* __restrict__ firstRow, uint32_t* __restrict__ flag) {
  uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c > numChunks) return;
  uint32_t f = 0;
  if (c < numChunks) {
    uint32_t r0 = firstRow[c];
    if (r0 > 0) {
      uint32_t pe = rs[r0], ps = rs[r0 - 1];
      f = (pe > c * (uint32_t)SG_CH && pe - ps > (uint32_t)SG_CH) ? 1u : 0u;
    }
  }
  flag[c] = f;
}

__global__ void k_heavy_flag(uint32_t nloc, const uint32_t* __restrict__ rs, uint8_t* __restrict__ flag,
                             uint8_t* __restrict__ bigFlag) {
  uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= nloc) return;
  const uint32_t s = rs[r], t = rs[r + 1];
  const bool heavy = t - s > (uint32_t)SG_CH;
  const uint32_t carries = heavy ? (t - 1) / SG_CH - s / SG_CH : 0;
  flag[r] = (heavy && carries <= 32u) ? 1 : 0;      // 32 == SG_BIG
  bigFlag[r] = (carries > 32u) ? 1 : 0;
}

// Start state of the worker that owns chunk c, so that the ring kernel reads ONE 32-byte record instead
// of walking firstRow -> rs -> rs (three dependent global loads per chunk):
//   [0] eb  first edge the worker processes     [1] ee  one past its last edge
//   [2] cur first row it accumulates into        [3] curS = rs[cur]   [4] curT = rs[cur + 1]
//   [5] r1  one past its last owned row          [6] flags: 1 = carry-in (cur is a heavy row owned by an
//       earlier chunk), 2 = nothing to do        [7] carry slot of a carry-in part
__global__ void k_chunk_desc(uint32_t numChunks, uint32_t E, const uint32_t* __restrict__ rs,
                             const uint32_t* __restrict__ firstRow, const uint32_t* __restrict__ carryIdx,
                             uint32_t* __restrict__ desc) {
  const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= numChunks) return;
  constexpr uint32_t CH = SG_CH;
  const uint32_t cb = w * CH, ce = min(cb + CH, E);
  const uint32_t r0 = firstRow[w], r1 = firstRow[w + 1];
  uint32_t eb = cb, ee = cb, cur = r0, curS = 0, curT = 0, flags = 0, segEnd = cb;
  bool carryIn = false;
  if (r0 > 0) {
    const uint32_t pe = rs[r0], ps = rs[r0 - 1];
    if (pe > cb && pe - ps > CH) {
      carryIn = true; cur = r0 - 1; curS = ps; curT = pe; eb = cb; segEnd = min(pe, ce); flags = 1u;
    }
  }
  if (!carryIn) {
    if (r0 >= r1) { flags = 2u; }
    else {
      cur = r0; curS = rs[r0]; curT = rs[r0 + 1]; eb = curS;
      segEnd = (curT - curS > CH) ? min(curT, ce) : curT;
    }
  }
  if (r1 > r0) {
    const uint32_t s = rs[r1 - 1], t = rs[r1];
    ee = (t - s > CH) ? min(t, ce) : t;
  } else {
    ee = segEnd;
  }
  if (flags & 2u) { eb = cb; ee = cb; }
  uint4* d = reinterpret_cast<uint4*>(desc + (size_t)w * 8);
  d[0] = make_uint4(eb, ee, cur, curS);
  d[1] = make_uint4(curT, r1, flags, carryIdx[w]);
}

// ----------------------------------------------------------- vector helper ---

template <int VEC> struct V;
template <> struct V<4> {
  typedef float4 T;
  static __device__ __forceinline__ T zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
  static __device__ __forceinline__ T ld(const T* p) { return __ldg(p); }
  static __device__ __forceinline__ T ld_plain(const T* p) { return *p; }
  static __device__ __forceinline__ void st(T* p, const T& v) { *p = v; }
  static __device__ __forceinline__ void add(T& a, const T& b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
  // IEEE divide.  A zero numerator sends nvcc's div.rn sequence down its slow path (FCHK flags
  // zero operands) and one such lane drags the whole warp along: gradients and pad columns are
  // full of zeros (+28 % instructions in the backward launches, r1 run 12).  0/d == 0 (same
  // sign) for d != 0, so those lanes skip the divide; d == 0 (degree 0) still yields NaN/Inf.
  static __device__ __forceinline__ float div1(float a, float d) { return (a != 0.0f || d == 0.0f) ? a / d : a; }
  static __device__ __forceinline__ T div(const T& a, float d) {
    return make_float4(div1(a.x, d), div1(a.y, d), div1(a.z, d), div1(a.w, d));
  }
  static __device__ __forceinline__ T rdiv(const T& a, const RowDiv& r) {
    float v[4] = {a.x, a.y, a.z, a.w};
    rowdiv4(v, r);          // one safety test for the four quotients
    return make_float4(v[0], v[1], v[2], v[3]);
  }
  static __device__ __forceinline__ T relu(const T& a) {
    return make_float4(relu_nanprop(a.x), relu_nanprop(a.y), relu_nanprop(a.z), relu_nanprop(a.w));
  }
};
template <> struct V<1> {
  typedef float T;
  static __device__ __forceinline__ T zero() { return 0.f; }
  static __device__ __forceinline__ T ld(const T* p) { return __ldg(p); }
  static __device__ __forceinline__ T ld_plain(const T* p) { return *p; }
  static __device__ __forceinline__ void st(T* p, const T& v) { *p = v; }
  static __device__ __forceinline__ void add(T& a, const T& b) { a += b; }
  static __device__ __forceinline__ T div(const T& a, float d) { return (a != 0.0f || d == 0.0f) ? a / d : a; }
  static __device__ __forceinline__ T rdiv(const T& a, const RowDiv& r) { return rowdiv(a, r); }
  static __device__ __forceinline__ T relu(const T& a) { return relu_nanprop(a); }
};

struct SgParams {
  const uint32_t* rs;
  const uint32_t* firstRow;
  const uint32_t* carryIdx;
  const uint32_t* heavyRows;
  const uint32_t* bigRows;
  const uint32_t* col;
  const void* in;      // [*][ldIn]  (in units of T)
  void* out;           // [nloc][ldOut]
  void* carry;         // [numCarries][ldC]
  size_t ldIn, ldOut, ldC;   // in units of T (float4 or float)
  uint32_t Q;          // valid T-columns per row
  uint32_t E, numChunks, numHeavy, numBig;
  int epi;
  int dense;           // mean degree >= chunk size: nearly every row is cut at chunk boundaries
  const uint32_t* desc; // [numChunks][8] chunk start records (ring kernel)
  uint32_t nloc;        // rows of the partition (rs has nloc + 1 entries)
};

// out[v] = relu?(acc / sqrtf(deg)) — what the model applies right after
// scatter_gather (gnn.cc:84-85), IEEE sqrt and divide like graphnorm_kernel.cu:49-51.
// The divisor is uniform over the row, so the divide is the row-uniform form of common.cuh
// (one refined reciprocal, 3 FMAs per element, bit-identical to div.rn): the plain `/` here
// cost +0.7 ms (H=64) .. +1.8 ms (H=41, zero pad lanes on the slow path) per launch (r1 run 14).
// MEAN (the AVG aggregator): acc / (float)deg by the same row-uniform IEEE divide; a degree-0 row's sum is
// +0 and stays so.
template <int VEC>
__device__ __forceinline__ void epi_store(typename V<VEC>::T v, typename V<VEC>::T* dst, uint32_t deg, int epi) {
  if (epi & ROC_SG_EPI_NORM) {
    const RowDiv rd = rowdiv_make(sqrtf((float)deg));
    v = V<VEC>::rdiv(v, rd);
  }
  if ((epi & ROC_SG_EPI_MEAN) && deg) v = V<VEC>::rdiv(v, rowdiv_make((float)deg));
  if (epi & ROC_SG_EPI_RELU) v = V<VEC>::relu(v);
  V<VEC>::st(dst, v);
}

// ------------------------------------------------------------- main kernel ---
// One worker (L lanes) per chunk.  Lane `lane` owns T-columns lane + ch*L.
template <int VEC, int L, int NCH, int U, int MINB>
__global__ void __launch_bounds__(SG_THREADS, MINB)
sg_chunk_kernel(const SgParams p) {
  typedef typename V<VEC>::T T;
  constexpr int WPB = SG_THREADS / L;
  constexpr uint32_t CH = SG_CH;
  const int lane = threadIdx.x % L;
  const uint32_t w = blockIdx.x * WPB + threadIdx.x / L;
  if (w >= p.numChunks) return;
  const unsigned wmask = (L == 32) ? 0xffffffffu
                                   : (((1u << L) - 1u) << (((threadIdx.x & 31) / L) * L));

  const uint32_t* __restrict__ rs = p.rs;
  const uint32_t* __restrict__ col = p.col;
  const T* __restrict__ in = reinterpret_cast<const T*>(p.in);
  T* __restrict__ out = reinterpret_cast<T*>(p.out);

  bool act[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) act[ch] = (uint32_t)(lane + ch * L) < p.Q;

  const uint32_t cb = w * CH;
  const uint32_t ce = min(cb + CH, p.E);

  // The worker's start state comes from the plan's 32-byte chunk record (k_chunk_desc) — one load instead of
  // the dependent walk firstRow[w] -> rs[r0], rs[r0 - 1] -> ... that cost every worker three round trips
  // before its first gather (r2: ~7 % of a warp's lifetime).
  const uint4 dA = __ldg(reinterpret_cast<const uint4*>(p.desc) + 2 * (size_t)w);
  const uint4 dB = __ldg(reinterpret_cast<const uint4*>(p.desc) + 2 * (size_t)w + 1);
  if (dB.z & 2u) return;           // nothing owned, nothing carried
  uint32_t cur = dA.z;             // row id of the current segment
  uint32_t curS = dA.w, curT = dB.x;   // its [start, end) in the edge array
  uint32_t e = dA.x;               // next edge
  const uint32_t ee = dA.y;        // end of this worker's whole edge range
  const uint32_t r1 = dB.y;
  const uint32_t carrySlot = dB.w;
  int kind = (dB.z & 1u) ? 0 : ((curT - curS > CH) ? 2 : 1);   // 0 = carry-in part of a heavy row, 1 = complete row, 2 = cut heavy row
  uint32_t segEnd = (kind == 1) ? curT : min(curT, ce);        // where this worker stops accumulating into it

  T acc[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) acc[ch] = V<VEC>::zero();

  // Row store.  The epilogue (IEEE sqrt + divides) lives in ONE out-of-line copy:
  // inlining it at every edge position made the kernel 4096 SASS instructions and
  // instruction-fetch bound (ncu: stalled_no_instruction 22.9 per issue, r1 run 2).
  auto flush = [&]() {
    char* dstb = (kind == 0)
        ? reinterpret_cast<char*>(reinterpret_cast<T*>(p.carry) + lane) + (uint64_t)carrySlot * ((uint32_t)p.ldC * (uint32_t)sizeof(T))
        : reinterpret_cast<char*>(out + lane) + (uint64_t)cur * ((uint32_t)p.ldOut * (uint32_t)sizeof(T));
    T* dst = reinterpret_cast<T*>(dstb);
    const int epi = (kind == 1) ? p.epi : 0;
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
      if (act[ch]) {
        if (epi) epi_store<VEC>(acc[ch], dst + ch * L, curT - curS, epi);
        else V<VEC>::st(dst + ch * L, acc[ch]);
      }
      acc[ch] = V<VEC>::zero();
    }
  };
  auto advance = [&]() {  // move to the next owned row
    cur += 1; curS = curT; curT = rs[cur + 1];
    bool heavy = curT - curS > CH;
    segEnd = heavy ? min(curT, ce) : curT;
    kind = heavy ? 2 : 1;
  };

  // Every lane reads the source ids itself (same address across the worker: one broadcast
  // transaction from L1); sub-warp shuffles with a runtime mask cost a MATCH.ANY sequence each.
  (void)wmask;
  // Gathers are unpredicated: a group that runs past the worker's last edge re-reads that edge's
  // source (index clamped; an L1 hit) and the tail values are simply never added.  With the tail
  // predicates (16 ISETP + 20 zero-inits per group) and a 64 x 64-bit address multiply the group
  // preamble was 146 SASS instructions for 8 gathers (r1 run 39); now one VIMNMX + LDG + IMAD.WIDE
  // + LDG.128 per edge.
  // lanes beyond the row's last column gather that last column instead (same sector, no extra
  // traffic): their sums are never stored (flush tests act[]), and no load needs a predicate
  const char* inl[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++)
    inl[ch] = reinterpret_cast<const char*>(in + min((uint32_t)(lane + ch * L), p.Q - 1u));
  const uint32_t rowBytes = (uint32_t)p.ldIn * (uint32_t)sizeof(T);
  const uint32_t eLast = ee - 1u;
#pragma unroll 1
  for (uint32_t base = e; base < ee; base += U) {
    const uint32_t cnt = min((uint32_t)U, ee - base);
    uint32_t srcs[U];
    if (cnt == (uint32_t)U) {
      const uint32_t* colp = col + base;       // full group: one address, immediate offsets
#pragma unroll
      for (int u = 0; u < U; u++) srcs[u] = __ldg(colp + u);
    } else {
#pragma unroll
      for (int u = 0; u < U; u++) srcs[u] = __ldg(col + min(base + (uint32_t)u, eLast));
    }
    T v[U][NCH];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint64_t off = (uint64_t)srcs[u] * rowBytes;
#pragma unroll
      for (int ch = 0; ch < NCH; ch++) v[u][ch] = V<VEC>::ld(reinterpret_cast<const T*>(inl[ch] + off));
    }
    {
      // One rolled loop over the row segments of the group (predicated adds of the edges [pos, lim)
      // of the current segment, then ONE copy of the row store).  A separate branch-free path for
      // groups inside one row did not pay: the two 16-lane workers of a warp rarely agree, so the
      // warp ran both paths in most iterations (r1 run 45).  The
      // unrolled per-edge `while (edge == segEnd) { flush; advance; }` had 8 inlined copies of the
      // store and cost ~180 SASS instructions per row (42 % of all instructions, r1 run 39).
      uint32_t pos = 0;
      for (;;) {
        const uint32_t lim = min(cnt, segEnd - base);
#pragma unroll
        for (int u = 0; u < U; u++) {
          if ((uint32_t)u >= pos && (uint32_t)u < lim) {
#pragma unroll
            for (int ch = 0; ch < NCH; ch++) V<VEC>::add(acc[ch], v[u][ch]);
          }
        }
        pos = lim;
        if (pos >= cnt) break;
        flush();
        advance();
      }
    }
  }
  flush();
  while (cur + 1 < r1) { advance(); flush(); }  // trailing zero-degree rows
}

// ------------------------------------------------- main kernel, variant C ---
// Same schedule, same per-row summation order, but the gathered rows are staged in
// shared memory with cp.async (LDGSTS) instead of registers: every lane copies its
// own 16 bytes of each neighbour row into a per-worker ring of DEPTH = P*GROUP row
// slots and later adds exactly the bytes it copied (no cross-lane sharing, so no
// barrier — only cp.async.wait_group).  Bytes in flight per SM are bounded by the
// ring (~100 KB per CTA) rather than by the register file, and the per-edge
// instruction count drops (one LDGSTS + one LDS.128 + 4 FADD per 16-byte column).
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
               "l"(gsrc)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ------------------------------------------- main kernel, variant C (lean) ---
// Variant C with the instruction stream trimmed (r1 run 10: the first version issued
// 34 instructions per edge — generic-address arithmetic and per-edge predicates —
// and was issue-bound once the latency was hidden): 32-bit shared addresses with
// immediate slot offsets, whole-group fast paths when the group is complete and no
// row boundary falls inside it.
__device__ __forceinline__ void cp_async16_s(uint32_t saddr, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(gsrc) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr) : "memory");
  return v;
}

template <int L, int NCH, int GROUP, int P>
__global__ void __launch_bounds__(SG_THREADS, 3)
sg_chunk_kernel_c2(const SgParams p) {
  typedef float4 T;
  constexpr int WPB = SG_THREADS / L;
  constexpr uint32_t CH = SG_CH;
  constexpr uint32_t ROWB = NCH * L * 16;          // bytes per ring slot
  constexpr uint32_t GRPB = GROUP * ROWB;          // bytes per group of slots
  constexpr uint32_t RINGB = P * GRPB;             // bytes per worker ring
  extern __shared__ __align__(16) float4 sg_ring[];
  const int lane = threadIdx.x % L;
  const uint32_t w = blockIdx.x * WPB + threadIdx.x / L;
  const uint32_t ringBase = (uint32_t)__cvta_generic_to_shared(sg_ring) + (threadIdx.x / L) * RINGB + lane * 16;
  if (w >= p.numChunks) return;
  const unsigned wmask = (L == 32) ? 0xffffffffu
                                   : (((1u << L) - 1u) << (((threadIdx.x & 31) / L) * L));
  const uint32_t* __restrict__ rs = p.rs;
  const uint32_t* __restrict__ col = p.col;
  const char* inB = reinterpret_cast<const char*>(p.in) + lane * 16;
  const uint32_t strideB = (uint32_t)p.ldIn * 16u;   // bytes between input rows (ldIn is in float4 units)
  bool act[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) act[ch] = (uint32_t)(lane + ch * L) < p.Q;

  const uint32_t cb = w * CH;
  const uint32_t ce = min(cb + CH, p.E);
  const uint32_t r0 = p.firstRow[w], r1 = p.firstRow[w + 1];
  uint32_t cur, curS, curT, segEnd, e;
  int kind;
  bool carryIn = false;
  if (r0 > 0) {
    uint32_t pe = rs[r0], ps = rs[r0 - 1];
    if (pe > cb && pe - ps > CH) {
      carryIn = true;
      cur = r0 - 1; curS = ps; curT = pe; kind = 0; e = cb; segEnd = min(pe, ce);
    }
  }
  if (!carryIn) {
    if (r0 >= r1) return;
    cur = r0; curS = rs[r0]; curT = rs[r0 + 1]; e = curS;
    bool heavy = curT - curS > CH;
    segEnd = heavy ? min(curT, ce) : curT;
    kind = heavy ? 2 : 1;
  }
  uint32_t ee;
  if (r1 > r0) {
    uint32_t s = rs[r1 - 1], t = rs[r1];
    ee = (t - s > CH) ? min(t, ce) : t;
  } else {
    ee = segEnd;
  }
  const uint32_t eb = e;
  const uint32_t nE = ee - eb;
  const uint32_t nG = (nE + GROUP - 1) / GROUP;

  T acc[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) acc[ch] = make_float4(0.f, 0.f, 0.f, 0.f);

  auto flush = [&]() {
    T* dst = (kind == 0) ? reinterpret_cast<T*>(p.carry) + (size_t)p.carryIdx[w] * p.ldC
                         : reinterpret_cast<T*>(p.out) + (size_t)cur * p.ldOut;
    dst += lane;
    const int epi = (kind == 1) ? p.epi : 0;
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
      if (act[ch]) {
        if (epi) epi_store<4>(acc[ch], dst + ch * L, curT - curS, epi);
        else *(dst + ch * L) = acc[ch];
      }
      acc[ch] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto advance = [&]() {
    cur += 1; curS = curT; curT = rs[cur + 1];
    bool heavy = curT - curS > CH;
    segEnd = heavy ? min(curT, ce) : curT;
    kind = heavy ? 2 : 1;
  };

  // issue group gi into the ring slots at byte offset slotOff (= (gi % P) * GRPB).
  // Every lane of the worker reads the source id itself (same address: one broadcast
  // transaction, L1-resident): a sub-warp __shfl_sync with a runtime mask costs a
  // MATCH.ANY sequence, ~11 instructions per edge (ncu source page, r1 run 11).
  (void)wmask;
  auto issue = [&](uint32_t gi, uint32_t slotOff) {
    if (gi < nG) {
      const uint32_t off = gi * GROUP;
      const uint32_t* cp = col + eb + off;
      const uint32_t sa = ringBase + slotOff;
      if (off + GROUP <= nE) {
        uint32_t srcs[GROUP];
#pragma unroll
        for (int u = 0; u < GROUP; u++) srcs[u] = __ldg(cp + u);
#pragma unroll
        for (int u = 0; u < GROUP; u++) {
          const char* g = inB + (size_t)srcs[u] * strideB;
#pragma unroll
          for (int ch = 0; ch < NCH; ch++)
            if (act[ch]) cp_async16_s(sa + u * ROWB + ch * L * 16, g + ch * L * 16);
        }
      } else {
#pragma unroll
        for (int u = 0; u < GROUP; u++) {
          if (off + u < nE) {
            const uint32_t src = __ldg(cp + u);
            const char* g = inB + (size_t)src * strideB;
#pragma unroll
            for (int ch = 0; ch < NCH; ch++)
              if (act[ch]) cp_async16_s(sa + u * ROWB + ch * L * 16, g + ch * L * 16);
          }
        }
      }
    }
    cp_async_commit();
  };
#pragma unroll 1
  for (uint32_t g = 0; g < (uint32_t)P; g++) issue(g, g * GRPB);   // one code copy: keep the kernel in the I-cache
  uint32_t slotOff = 0;
#pragma unroll 1
  for (uint32_t g = 0; g < nG; g++) {
    cp_async_wait<P - 1>();
    const uint32_t e0 = eb + g * GROUP;
    const uint32_t sa = ringBase + slotOff;
    if (segEnd - e0 >= (uint32_t)GROUP) {
      // the whole group lies inside the current row segment: no boundary tests
#pragma unroll
      for (int u = 0; u < GROUP; u++)
#pragma unroll
        for (int ch = 0; ch < NCH; ch++)
          if (act[ch]) {
            const float4 v = lds128(sa + u * ROWB + ch * L * 16);
            acc[ch].x += v.x; acc[ch].y += v.y; acc[ch].z += v.z; acc[ch].w += v.w;
          }
    } else {
#pragma unroll
      for (int u = 0; u < GROUP; u++) {
        const uint32_t ecur = e0 + u;
        if (ecur < ee) {
          while (ecur == segEnd) { flush(); advance(); }
#pragma unroll
          for (int ch = 0; ch < NCH; ch++)
            if (act[ch]) {
              const float4 v = lds128(sa + u * ROWB + ch * L * 16);
              acc[ch].x += v.x; acc[ch].y += v.y; acc[ch].z += v.z; acc[ch].w += v.w;
            }
        }
      }
    }
    issue(g + P, slotOff);
    slotOff += GRPB;
    if (slotOff == RINGB) slotOff = 0;
  }
  flush();
  while (cur + 1 < r1) { advance(); flush(); }
}

// ------------------------------------------------- main kernel, variant T ---
// Same schedule and the same per-row summation order again, but the neighbour rows are fetched by
// the TMA unit: one `cp.async.bulk.tensor ... tile::gather4` per four edges (four row indices in
// one instruction, sm_100 only) lands 4 x rowBytes in the worker's shared-memory ring and
// completes on an mbarrier; the lanes then add with LDS.128 + FADD.  What this buys over the
// register variant A: (1) bytes in flight are bounded by the ring (P stages x S gather4s per
// worker, ~100 KB per SM) instead of by the register file — variant A holds 8 rows per lane in
// registers, issues them as a burst, waits for all of them and only then adds, so its *average*
// bytes in flight are well under half of its peak (ncu r1 run 45: latency-bound at 0.52 of the
// DRAM peak, 47 % issue utilisation, nothing saturated); the ring is refilled stage by stage,
// so it stays full.  (2) one TMA instruction per 4 edges replaces 4 x (index load + IMAD.WIDE +
// LDG.128) per lane group.  MODE 1 issues one plain `cp.async.bulk` per row instead (no tensor
// map; kept for measurement).
// The tensor map's box is L*NCH*4 floats wide (the worker's whole lane span) over a tensor
// that is Q*4 floats wide: columns past the row's end are zero-filled by the TMA unit, which
// makes the shared-memory row pitch a compile-time constant and the adds unpredicated.
__device__ __forceinline__ void mbar_init_a(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_a(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "SG_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra SG_DONE;\n\t"
      "bra SG_WAIT;\n\t"
      "SG_DONE:\n\t}"
      ::"r"(bar), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_gather4(uint32_t dst, const CUtensorMap* m, int c0, uint32_t r0, uint32_t r1,
                                            uint32_t r2, uint32_t r3, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile::gather4.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(r0), "r"(r1), "r"(r2), "r"(r3), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void bulk_row(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

template <int L, int NCH, int S, int P, int NT, int MINB, int MODE>
__global__ void __launch_bounds__(NT, MINB)
sg_chunk_kernel_t(const SgParams p, const __grid_constant__ CUtensorMap tmap) {
  typedef float4 T;
  constexpr int WPB = NT / L;
  constexpr uint32_t CH = SG_CH;
  constexpr int G = 4 * S;                       // edges per stage
  constexpr uint32_t SLOTB = NCH * L * 16;       // shared-memory bytes per gathered row
  constexpr uint32_t G4B = 4 * SLOTB;            // one gather4
  constexpr uint32_t STAGEB = S * G4B;
  constexpr uint32_t RINGB = P * STAGEB;
  extern __shared__ __align__(128) unsigned char sg_smem_t[];
  const int lane = threadIdx.x % L;
  const int wi = threadIdx.x / L;
  const uint32_t w = blockIdx.x * WPB + wi;
  if (w >= p.numChunks) return;
  const unsigned wmask = (L == 32) ? 0xffffffffu
                                   : (((1u << L) - 1u) << (((threadIdx.x & 31) / L) * L));
  const uint32_t smem0 = (uint32_t)__cvta_generic_to_shared(sg_smem_t);
  const uint32_t ring = smem0 + wi * RINGB;
  const uint32_t bars = smem0 + WPB * RINGB + wi * (P * 8);
  const uint32_t* __restrict__ rs = p.rs;
  const uint32_t* __restrict__ col = p.col;
  bool act[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) act[ch] = (uint32_t)(lane + ch * L) < p.Q;

  const uint32_t cb = w * CH;
  const uint32_t ce = min(cb + CH, p.E);
  const uint32_t r0 = p.firstRow[w], r1 = p.firstRow[w + 1];
  uint32_t cur, curS, curT, segEnd, e;
  int kind;
  bool carryIn = false;
  if (r0 > 0) {
    uint32_t pe = rs[r0], ps = rs[r0 - 1];
    if (pe > cb && pe - ps > CH) {
      carryIn = true;
      cur = r0 - 1; curS = ps; curT = pe; kind = 0; e = cb; segEnd = min(pe, ce);
    }
  }
  if (!carryIn) {
    if (r0 >= r1) return;
    cur = r0; curS = rs[r0]; curT = rs[r0 + 1]; e = curS;
    bool heavy = curT - curS > CH;
    segEnd = heavy ? min(curT, ce) : curT;
    kind = heavy ? 2 : 1;
  }
  uint32_t ee;
  if (r1 > r0) {
    uint32_t s = rs[r1 - 1], t = rs[r1];
    ee = (t - s > CH) ? min(t, ce) : t;
  } else {
    ee = segEnd;
  }
  const uint32_t eb = e;
  const uint32_t nE = ee - eb;
  const uint32_t nStages = (nE + G - 1) / G;

  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < P; s++) mbar_init_a(bars + 8 * s, 1);
    tc::fence_barrier_init();
  }
  __syncwarp(wmask);

  T acc[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) acc[ch] = make_float4(0.f, 0.f, 0.f, 0.f);

  auto flush = [&]() {
    T* dst = (kind == 0) ? reinterpret_cast<T*>(p.carry) + (size_t)p.carryIdx[w] * p.ldC
                         : reinterpret_cast<T*>(p.out) + (size_t)cur * p.ldOut;
    dst += lane;
    const int epi = (kind == 1) ? p.epi : 0;
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
      if (act[ch]) {
        if (epi) epi_store<4>(acc[ch], dst + ch * L, curT - curS, epi);
        else *(dst + ch * L) = acc[ch];
      }
      acc[ch] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto advance = [&]() {
    cur += 1; curS = curT; curT = rs[cur + 1];
    bool heavy = curT - curS > CH;
    segEnd = heavy ? min(curT, ce) : curT;
    kind = heavy ? 2 : 1;
  };

  // stage k -> ring slot `slot`: issued by the worker's first lane.  A stage that runs past the
  // worker's last edge repeats that edge's source (a duplicate row, L2-resident; never added).
  const char* inB = reinterpret_cast<const char*>(p.in);
  const uint32_t strideB = (uint32_t)p.ldIn * 16u;
  const uint32_t rowB = p.Q * 16u;
  // MODE 2: the source ids never sit in front of the issue.  Lane j of the worker loads, once and up front, the
  // ids of gather4 units j, j + L, ... of the worker's edge range (a worker has at most 127 edges = 32 units) and
  // issues those units itself when their ring slot frees (ncu on MODE 0: 21 % of the stall samples waited for the
  // id load of the stage about to be issued).
  constexpr int NU = (MODE == 2) ? (32 / L) : 1;
  uint4 ids[NU];
  if (MODE == 2 && nE) {
#pragma unroll
    for (int n = 0; n < NU; n++) {
      const uint32_t e4 = 4u * ((uint32_t)lane + (uint32_t)n * L);
      const uint32_t last = nE - 1u;
      const uint32_t* cp = col + eb;
      ids[n] = make_uint4(__ldg(cp + min(e4, last)), __ldg(cp + min(e4 + 1u, last)), __ldg(cp + min(e4 + 2u, last)),
                          __ldg(cp + min(e4 + 3u, last)));
    }
  }
  auto issue = [&](uint32_t k, uint32_t slot) {
    if (MODE == 2) {
      if (k < nStages) {
        const uint32_t off = k * G;
        const uint32_t bar = bars + slot * 8;
        const uint32_t dst = ring + slot * STAGEB;
        const uint32_t nv = min((uint32_t)G, nE - off);
        const uint32_t n4 = (nv + 3u) >> 2;
        if ((uint32_t)lane == (k * S) % (uint32_t)L) mbar_expect_tx_a(bar, n4 * G4B);
#pragma unroll
        for (int s = 0; s < S; s++) {
          const uint32_t g = k * S + (uint32_t)s;              // gather4 unit within the worker's range
          if ((uint32_t)s < n4 && (uint32_t)lane == g % (uint32_t)L) {
            uint4 id = ids[0];
#pragma unroll
            for (int n = 1; n < NU; n++) if (g / (uint32_t)L == (uint32_t)n) id = ids[n];
            tma_gather4(dst + s * G4B, &tmap, 0, id.x, id.y, id.z, id.w, bar);
          }
        }
      }
      return;
    }
    if (k < nStages && lane == 0) {
      const uint32_t off = k * G;
      const uint32_t* cp = col + eb + off;
      const uint32_t bar = bars + slot * 8;
      const uint32_t dst = ring + slot * STAGEB;
      const uint32_t nv = min((uint32_t)G, nE - off);
      if (MODE == 0) {
        const uint32_t n4 = (nv + 3u) >> 2;
        mbar_expect_tx_a(bar, n4 * G4B);
#pragma unroll
        for (int s = 0; s < S; s++) {
          if ((uint32_t)s < n4) {
            uint32_t i0, i1, i2, i3;
            if ((uint32_t)(4 * s + 4) <= nv) {
              i0 = __ldg(cp + 4 * s); i1 = __ldg(cp + 4 * s + 1); i2 = __ldg(cp + 4 * s + 2); i3 = __ldg(cp + 4 * s + 3);
            } else {
              const uint32_t last = nv - 1u;
              i0 = __ldg(cp + min((uint32_t)(4 * s), last)); i1 = __ldg(cp + min((uint32_t)(4 * s + 1), last));
              i2 = __ldg(cp + min((uint32_t)(4 * s + 2), last)); i3 = __ldg(cp + min((uint32_t)(4 * s + 3), last));
            }
            tma_gather4(dst + s * G4B, &tmap, 0, i0, i1, i2, i3, bar);
          }
        }
      } else {
        mbar_expect_tx_a(bar, nv * rowB);
#pragma unroll
        for (int u = 0; u < G; u++) {
          if ((uint32_t)u < nv) {
            const uint32_t src = __ldg(cp + u);
            bulk_row(dst + u * SLOTB, inB + (size_t)src * strideB, rowB, bar);
          }
        }
      }
    }
  };
#pragma unroll 1
  for (uint32_t k = 0; k < (uint32_t)P; k++) issue(k, k);
  uint32_t slot = 0, parity = 0;
#pragma unroll 1
  for (uint32_t k = 0; k < nStages; k++) {
    mbar_wait_a(bars + slot * 8, parity);
    const uint32_t e0 = eb + k * G;
    const uint32_t sa = ring + slot * STAGEB + lane * 16;
    if (segEnd - e0 >= (uint32_t)G) {
      // the whole stage lies inside the current row segment
#pragma unroll
      for (int u = 0; u < G; u++)
#pragma unroll
        for (int ch = 0; ch < NCH; ch++) {
          const float4 v = lds128(sa + u * SLOTB + ch * L * 16);
          acc[ch].x += v.x; acc[ch].y += v.y; acc[ch].z += v.z; acc[ch].w += v.w;
        }
    } else {
      // one rolled loop over the row segments of the stage, ONE row-store site
      const uint32_t cnt = min((uint32_t)G, ee - e0);
      uint32_t pos = 0;
      for (;;) {
        const uint32_t lim = min(cnt, segEnd - e0);
#pragma unroll
        for (int u = 0; u < G; u++) {
          if ((uint32_t)u >= pos && (uint32_t)u < lim) {
#pragma unroll
            for (int ch = 0; ch < NCH; ch++) {
              const float4 v = lds128(sa + u * SLOTB + ch * L * 16);
              acc[ch].x += v.x; acc[ch].y += v.y; acc[ch].z += v.z; acc[ch].w += v.w;
            }
          }
        }
        pos = lim;
        if (pos >= cnt) break;
        flush();
        advance();
      }
    }
    __syncwarp(wmask);          // every lane has read the slot before the TMA unit rewrites it
    issue(k + P, slot);
    slot += 1;
    if (slot == (uint32_t)P) { slot = 0; parity ^= 1u; }
  }
  flush();
  while (cur + 1 < r1) { advance(); flush(); }
}

// ------------------------------------------------- main kernel, variant R ---
// Producer / consumer ring.  What the measurements of r2 asked for (tools/gather_ceiling.cu, B200):
//  * the gather of this graph's row mix (69 % of the row fetches hit L2) is latency-bound: the pure
//    LDG.128 gather reaches 38 B/clk/SM with variant A's 8 rows x 32 warps in flight and 58 with twice
//    the warps — more requests outstanding than the register file can hold;
//  * a shared-memory ring filled by `cp.async.bulk.tensor ... tile::gather4` sustains 55-60 B/clk/SM at
//    that mix when (a) ~190 KB per SM are in flight, (b) the index loads never sit on the issue path
//    and (c) several warps per SM issue: one UTMALDG costs its warp ~68 cycles (an ELECT / R2UR loop per
//    lane), 15 B/clk per issuing warp at 1 KB per instruction.
// So: a CTA is ONE producer warp and TWO worker warps that share a two-slot ring; six CTAs per SM for rows
// of up to 256 bytes.  A slot holds one 64-edge chunk of gathered rows (64 x SLOTB bytes) and completes on
// one `full` mbarrier.  The CTA walks a contiguous range of chunk pairs; worker h owns the chunks of parity
// h and slot h holds them.  The producer's lane j (of half-warp h) holds the four source ids of gather4 #j
// of its chunk in registers — one coalesced LDG.128 per lane, loaded one pair ahead — and issues it as soon
// as the slot's `empty` barrier says both readers are done.
// Readers of a slot: the chunk's own worker, and the worker of the PREVIOUS chunk, whose last rows may run
// up to 63 edges into it (rows of degree <= 64 are finished by their owner).  Each of the two arrives on
// `empty` (count 2) after it has waited on `full` for that use, so every waiter sees every phase of the
// barriers it uses (a parity wait can only be one phase ahead).
// A worker is a whole warp: lane l owns VW consecutive floats of the row (float2 for rows of up to 64
// floats, so all 32 lanes work and an edge costs LDS.64 + 2 FADD), there is no second worker in the warp to
// diverge from, and the row ends of the chunk sit in a register batch (one coalesced load, read by shuffle)
// instead of being fetched one dependent load per row.  The per-row summation order is the chunk plan's, as
// in A / C / T: the results are bit-identical.
template <int VW> struct RV;
template <> struct RV<2> {
  typedef float2 T;
  static __device__ __forceinline__ T lds(uint32_t a) {
    T v; asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a) : "memory"); return v;
  }
  static __device__ __forceinline__ T zero() { return make_float2(0.f, 0.f); }
  static __device__ __forceinline__ void add(T& a, const T& b) { a.x += b.x; a.y += b.y; }
  static __device__ __forceinline__ void store(T* dst, T v, uint32_t deg, int epi) {
    if (epi & ROC_SG_EPI_NORM) {
      const RowDiv rd = rowdiv_make(sqrtf((float)deg));
      float t[4] = {v.x, v.y, 0.f, 0.f};
      rowdiv4(t, rd, 2);
      v = make_float2(t[0], t[1]);
    }
    if ((epi & ROC_SG_EPI_MEAN) && deg) {
      float t[4] = {v.x, v.y, 0.f, 0.f};
      rowdiv4(t, rowdiv_make((float)deg), 2);
      v = make_float2(t[0], t[1]);
    }
    if (epi & ROC_SG_EPI_RELU) v = make_float2(relu_nanprop(v.x), relu_nanprop(v.y));
    *dst = v;
  }
};
template <> struct RV<4> {
  typedef float4 T;
  static __device__ __forceinline__ T lds(uint32_t a) { return lds128(a); }
  static __device__ __forceinline__ T zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
  static __device__ __forceinline__ void add(T& a, const T& b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
  static __device__ __forceinline__ void store(T* dst, T v, uint32_t deg, int epi) {
    if (epi) epi_store<4>(v, dst, deg, epi); else *dst = v;
  }
};

template <int VW, int NCH, int NPW, int MINB>
__global__ void __launch_bounds__(32 * (NPW + 2), MINB)
sg_ring_kernel(const SgParams p, const __grid_constant__ CUtensorMap tmap, uint32_t pairsPerCta) {
  typedef typename RV<VW>::T T;
  constexpr uint32_t CH = SG_CH;
  constexpr uint32_t LANEB = VW * 4;                // bytes per lane per column block
  constexpr uint32_t SLOTB = NCH * 32 * LANEB;      // shared-memory bytes per gathered row
  constexpr uint32_t G4B = 4 * SLOTB;
  constexpr uint32_t CHUNKB = CH * SLOTB;           // one slot
  extern __shared__ __align__(128) unsigned char sg_smem_r[];
  const uint32_t ring = (uint32_t)__cvta_generic_to_shared(sg_smem_r);
  const uint32_t fullB = ring + 2 * CHUNKB, emptyB = fullB + 16;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t numPairs = (p.numChunks + 1u) >> 1;
  const uint32_t p0 = blockIdx.x * pairsPerCta;
  if (p0 >= numPairs) return;
  const uint32_t p1 = min(numPairs, p0 + pairsPerCta);
  const uint32_t nIt = p1 - p0;
  const uint32_t c0 = 2u * p0;
  const uint32_t nLoaded = (p.E + CH - 1u) / CH;           // chunks that hold at least one edge
  if (threadIdx.x == 0) {
    mbar_init_a(fullB, 1); mbar_init_a(fullB + 8, 1);
    mbar_init_a(emptyB, 2); mbar_init_a(emptyB + 8, 2);
    tc::fence_barrier_init();
  }
  __syncthreads();

  if (warp < NPW) {
    // ----------------------------------------------------------- producers ---
    // NPW warps share the 32 gather4s of a chunk pair: 32 / NPW lanes of each are active, lanes of one warp
    // always serve the same slot (so the warp sees every phase of that slot's `empty` barrier).  One UTMALDG
    // costs the issuing warp ~68 cycles (ELECT / R2UR loop), so a single warp needs ~2200 cycles per pair.
    constexpr int PERW = 32 / NPW;                        // gather4s per producer warp and pair
    const int g = warp * PERW + lane;                     // gather4 index within the pair: 0..15 slot 0, 16..31 slot 1
    const int h = g >> 4, j = g & 15;
    const bool mine = lane < PERW;
    const uint32_t* __restrict__ col = p.col;
    auto load_ids = [&](uint32_t c, uint4& v) {           // the four sources of gather4 #j of chunk c
      const uint32_t e = c * CH + 4u * (uint32_t)j;
      if (e + 4u <= p.E) {
        v = __ldg(reinterpret_cast<const uint4*>(col + e));
      } else if (e < p.E) {                                // the partial tail repeats the last edge's source
        const uint32_t last = p.E - 1u;
        v.x = __ldg(col + e); v.y = __ldg(col + min(e + 1u, last)); v.z = __ldg(col + min(e + 2u, last)); v.w = __ldg(col + min(e + 3u, last));
      } else {
        v = make_uint4(0u, 0u, 0u, 0u);
      }
    };
    if (!mine) return;
    uint4 nxt;
    load_ids(c0 + (uint32_t)h, nxt);
    // uses of slot h: it = 0 .. nIt-1, plus (h == 0 only) the chunk after the range, read by worker 1's tail
    const uint32_t uses = nIt + (h == 0 ? 1u : 0u);
#pragma unroll 1
    for (uint32_t it = 0; it < uses; it++) {
      const uint32_t c = c0 + 2u * it + (uint32_t)h;
      const uint4 ids = nxt;
      if (it + 1u < uses) load_ids(c + 2u, nxt);
      if (c < nLoaded) {
        const uint32_t nv = min(CH, p.E - c * CH);
        const uint32_t n4 = (nv + 3u) >> 2;
        mbar_wait_a(emptyB + 8u * h, (it & 1u) ^ 1u);
        if (j == 0) mbar_expect_tx_a(fullB + 8u * h, n4 * G4B);
        if ((uint32_t)j < n4) tma_gather4(ring + (uint32_t)h * CHUNKB + (uint32_t)j * G4B, &tmap, 0, ids.x, ids.y, ids.z, ids.w, fullB + 8u * h);
      }
    }
    return;
  }

  // ---------------------------------------------------------------- workers ---
  const int h = warp - NPW;                                 // worker 0 / 1
  const uint32_t* __restrict__ rs = p.rs;
  const uint32_t validLanes = (p.Q * 16u + LANEB - 1u) / LANEB;      // lanes (per column block) that hold row data
  bool act[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) act[ch] = (uint32_t)(lane + ch * 32) < validLanes;
  if (h == 1) {
    // Worker 1 first reads slot 0 at its SECOND use; it has to see the first one complete before it may wait
    // for that (parity waits).  Its arrive stands in for the previous range's last worker, which reads its
    // tail from its own CTA's copy of chunk c0.
    if (c0 < nLoaded) mbar_wait_a(fullB, 0u);
    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(emptyB) : "memory");
  }
  const uint4* __restrict__ descs = reinterpret_cast<const uint4*>(p.desc);
  uint4 d0, d1;
  {
    const uint32_t c = c0 + (uint32_t)h;
    if (c < p.numChunks) { d0 = __ldg(descs + 2 * (size_t)c); d1 = __ldg(descs + 2 * (size_t)c + 1); }
    else { d0 = make_uint4(0, 0, 0, 0); d1 = make_uint4(0, 0, 2u, 0); }
  }
  const uint32_t sa = ring + (uint32_t)lane * LANEB;
  const size_t ldOutT = p.ldOut * 4 / VW, ldCT = p.ldC * 4 / VW;     // SgParams counts rows in float4 units

#pragma unroll 1
  for (uint32_t it = 0; it < nIt; it++) {
    const uint32_t c = c0 + 2u * it + (uint32_t)h;
    // this chunk's start state; the next one's record is requested now and used next iteration
    const uint32_t eb = d0.x, ee = d0.y, r1 = d1.y, flags = d1.z, carrySlot = d1.w;
    uint32_t cur = d0.z, curS = d0.w, curT = d1.x;
    {
      const uint32_t cn = c + 2u;
      if (it + 1u < nIt && cn < p.numChunks) { d0 = __ldg(descs + 2 * (size_t)cn); d1 = __ldg(descs + 2 * (size_t)cn + 1); }
      else { d0 = make_uint4(0, 0, 0, 0); d1 = make_uint4(0, 0, 2u, 0); }
    }
    const bool idle = (flags & 2u) != 0u || c >= p.numChunks;
    const uint32_t ce = min(c * CH + CH, p.E);
    int kind = (flags & 1u) ? 0 : ((curT - curS > CH) ? 2 : 1);
    uint32_t segEnd = (kind == 1) ? curT : min(curT, ce);
    const uint32_t boundary = (c + 1u) * CH;
    // row ends of the rows after `cur`: lane i holds rs[rsBase + i] (clamped to the partition's last entry)
    uint32_t rsBase = cur + 2u;
    uint32_t rsReg = idle ? 0u : __ldg(rs + min(rsBase + (uint32_t)lane, p.nloc));

    T acc[NCH];
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) acc[ch] = RV<VW>::zero();
    auto flush = [&]() {
      T* dst = (kind == 0) ? reinterpret_cast<T*>(p.carry) + (size_t)carrySlot * ldCT
                           : reinterpret_cast<T*>(p.out) + (size_t)cur * ldOutT;
      dst += lane;
      const int epi = (kind == 1) ? p.epi : 0;
#pragma unroll
      for (int ch = 0; ch < NCH; ch++) {
        if (act[ch]) RV<VW>::store(dst + ch * 32, acc[ch], curT - curS, epi);
        acc[ch] = RV<VW>::zero();
      }
    };
    auto advance = [&]() {
      cur += 1; curS = curT;
      const uint32_t k = cur + 1u - rsBase;                // rs[cur + 1] is entry k of the batch
      if (k >= 32u) { rsBase = cur + 1u; rsReg = __ldg(rs + min(rsBase + (uint32_t)lane, p.nloc)); }
      curT = __shfl_sync(0xffffffffu, rsReg, (int)((cur + 1u - rsBase) & 31u));
      const bool heavy = curT - curS > CH;
      segEnd = heavy ? min(curT, ce) : curT;
      kind = heavy ? 2 : 1;
    };

    // phase 0: the worker's own chunk (slot h, use `it`); phase 1: its tail in the next chunk
    // (slot h^1; for worker 1 that is slot 0's NEXT use)
#pragma unroll 1
    for (int ph = 0; ph < 2; ph++) {
      const uint32_t s = (uint32_t)(h ^ ph);
      const uint32_t use = it + (uint32_t)(h & ph);
      const uint32_t cc = c + (uint32_t)ph;
      const bool loaded = cc < nLoaded;
      if (loaded) mbar_wait_a(fullB + 8u * s, use & 1u);
      const uint32_t eFrom = ph == 0 ? eb : max(eb, boundary);
      const uint32_t eTo = ph == 0 ? min(ee, boundary) : ee;
      if (!idle && eFrom < eTo) {
#pragma unroll 1
        for (uint32_t e0 = eFrom & ~3u; e0 < eTo; e0 += 4u) {
          const uint32_t lo = max(eFrom, e0) - e0;
          const uint32_t hi = min(eTo, e0 + 4u) - e0;
          const uint32_t a = sa + (e0 & 127u) * SLOTB;
          if (lo == 0u && hi == 4u && segEnd - e0 >= 4u) {
            T v[4][NCH];
#pragma unroll
            for (int u = 0; u < 4; u++)
#pragma unroll
              for (int ch = 0; ch < NCH; ch++) v[u][ch] = RV<VW>::lds(a + u * SLOTB + ch * 32 * LANEB);
#pragma unroll
            for (int u = 0; u < 4; u++)
#pragma unroll
              for (int ch = 0; ch < NCH; ch++) RV<VW>::add(acc[ch], v[u][ch]);
          } else {
            uint32_t pos = lo;
            for (;;) {
              const uint32_t lim = min(hi, segEnd - e0);
#pragma unroll
              for (int u = 0; u < 4; u++) {
                if ((uint32_t)u >= pos && (uint32_t)u < lim) {
#pragma unroll
                  for (int ch = 0; ch < NCH; ch++) RV<VW>::add(acc[ch], RV<VW>::lds(a + u * SLOTB + ch * 32 * LANEB));
                }
              }
              pos = max(pos, lim);
              if (pos >= hi) break;
              flush();
              advance();
            }
          }
        }
      }
      if (loaded) {
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(emptyB + 8u * s) : "memory");
      }
    }
    if (!idle) {
      flush();
      while (cur + 1 < r1) { advance(); flush(); }
    }
  }
}

// ----------------------------------------------------------- fix-up kernel ---
// One worker per heavy row: out[R] = epilogue(out[R] + sum_k carry[slot0 + k]), k ascending.
template <int VEC, int L, int NCH, int U>
__global__ void __launch_bounds__(SG_THREADS)
sg_fixup_kernel(const SgParams p) {
  typedef typename V<VEC>::T T;
  constexpr int WPB = SG_THREADS / L;
  constexpr uint32_t CH = SG_CH;
  const int lane = threadIdx.x % L;
  const uint32_t w = blockIdx.x * WPB + threadIdx.x / L;
  if (w >= p.numHeavy) return;
  const uint32_t R = p.heavyRows[w];
  const uint32_t s = p.rs[R], t = p.rs[R + 1];
  const uint32_t c0 = s / CH, cLast = (t - 1) / CH;
  const uint32_t n = cLast - c0;
  const uint32_t slot0 = p.carryIdx[c0 + 1];
  T* dst = reinterpret_cast<T*>(p.out) + (size_t)R * p.ldOut;
  const T* cbase = reinterpret_cast<const T*>(p.carry) + (size_t)slot0 * p.ldC;
  bool act[NCH];
  T acc[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) {
    act[ch] = (uint32_t)(lane + ch * L) < p.Q;
    acc[ch] = act[ch] ? V<VEC>::ld_plain(dst + lane + ch * L) : V<VEC>::zero();
  }
  for (uint32_t k = 0; k < n; k += U) {
    T v[U][NCH];
#pragma unroll
    for (int u = 0; u < U; u++)
#pragma unroll
      for (int ch = 0; ch < NCH; ch++)
        v[u][ch] = (k + u < n && act[ch]) ? V<VEC>::ld_plain(cbase + (size_t)(k + u) * p.ldC + lane + ch * L)
                                          : V<VEC>::zero();
#pragma unroll
    for (int u = 0; u < U; u++)
      if (k + u < n)
#pragma unroll
        for (int ch = 0; ch < NCH; ch++) V<VEC>::add(acc[ch], v[u][ch]);
  }
#pragma unroll
  for (int ch = 0; ch < NCH; ch++)
    if (act[ch]) epi_store<VEC>(acc[ch], dst + lane + ch * L, t - s, p.epi);
}

// Rows with more than SG_BIG carries (hubs: R-MAT-22's largest row spans 1 524 chunks) get a
// whole CTA: each of the 256/L lane groups sums a contiguous block of the carries, the blocks
// are combined in order through shared memory.  With one worker per row the hubs' serial
// chains set the kernel's duration (0.56 ms for 250 MB of traffic, r1 run 15).
constexpr uint32_t SG_BIG = 32;

template <int VEC, int L, int NCH, int U>
__global__ void __launch_bounds__(SG_THREADS)
sg_fixup_big_kernel(const SgParams p) {
  typedef typename V<VEC>::T T;
  constexpr int WPB = SG_THREADS / L;
  constexpr uint32_t CH = SG_CH;
  __shared__ __align__(16) float part[WPB * NCH * L * VEC];
  const int lane = threadIdx.x % L;
  const int g = threadIdx.x / L;
  const uint32_t R = p.bigRows[blockIdx.x];
  const uint32_t s = p.rs[R], t = p.rs[R + 1];
  const uint32_t c0 = s / CH, cLast = (t - 1) / CH;
  const uint32_t n = cLast - c0;
  const uint32_t slot0 = p.carryIdx[c0 + 1];
  const T* cbase = reinterpret_cast<const T*>(p.carry) + (size_t)slot0 * p.ldC;
  const uint32_t per = (n + WPB - 1) / WPB;
  const uint32_t k0 = min(n, (uint32_t)g * per), k1 = min(n, k0 + per);
  bool act[NCH];
  T acc[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) { act[ch] = (uint32_t)(lane + ch * L) < p.Q; acc[ch] = V<VEC>::zero(); }
  for (uint32_t k = k0; k < k1; k += U) {
    T v[U][NCH];
#pragma unroll
    for (int u = 0; u < U; u++)
#pragma unroll
      for (int ch = 0; ch < NCH; ch++)
        v[u][ch] = (k + u < k1 && act[ch]) ? V<VEC>::ld_plain(cbase + (size_t)(k + u) * p.ldC + lane + ch * L)
                                           : V<VEC>::zero();
#pragma unroll
    for (int u = 0; u < U; u++)
#pragma unroll
      for (int ch = 0; ch < NCH; ch++) V<VEC>::add(acc[ch], v[u][ch]);
  }
  T* sp = reinterpret_cast<T*>(part);
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) sp[(g * NCH + ch) * L + lane] = acc[ch];
  __syncthreads();
  if (g == 0) {
    T* dst = reinterpret_cast<T*>(p.out) + (size_t)R * p.ldOut;
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
      if (act[ch]) {
        T a = V<VEC>::ld_plain(dst + lane + ch * L);      // the owner chunk's raw partial
        for (int gg = 0; gg < WPB; gg++) V<VEC>::add(a, sp[(gg * NCH + ch) * L + lane]);
        epi_store<VEC>(a, dst + lane + ch * L, t - s, p.epi);
      }
    }
  }
}

// ------------------------------------------------ MAX / MIN and their backward ---
// Kernel A's structure (chunk records, per-row order, rolled segment loop, one store site) with other
// accumulators:
//   MAX / MIN  (value, winner id) per element.  The first edge of a segment is taken as is; a later one replaces
//              the best when it is strictly larger (smaller), or NaN over a non-NaN best — so among equal values
//              the first edge in CSR order wins and the first NaN wins.  Heavy rows: the owner stores its raw
//              (value, id), later chunks store theirs into the float carry slots and the u32 carryArg slots, and
//              sg_aggr_fixup(_big)_kernel merges them in chunk order with the same rule.
//   ARGBWD     sum of outGrad[src] over the edges whose arg[src] names this row; two rows gathered per edge.
//              Rows cut at chunk boundaries are plain sums: the SUM fix-up kernels finish them.
// Algorithmic bytes per launch: MAX / MIN E*(4H+4) + Nloc*(8H+8) (+ the winner ids, E*4, when colGlobal is a
// separate array); ARGBWD E*(8H+4) + Nloc*(4H+8).
enum { SG_OP_MAX = 1, SG_OP_MIN = 2, SG_OP_ARGBWD = 3 };
constexpr uint32_t SG_NO_ARG = 0xFFFFFFFFu;

struct SgAggrParams {
  SgParams p;              // schedule, in / out / carry; p.ld* and p.Q count VEC-float units
  const uint32_t* colG;    // MAX / MIN: winner id per edge (parallel to p.col)
  uint32_t* arg;           // MAX / MIN: [nloc][ldArg] winner ids out (NULL: not stored); ARGBWD: read at col ids
  uint32_t* carryArg;      // MAX / MIN: [numCarries][ldCA]
  size_t ldArg, ldCA;      // VEC-u32 units
  uint32_t rowLeft;        // ARGBWD: global id of local row 0
};

template <int VEC>
__device__ __forceinline__ void ldv(float (&a)[VEC], const float* p) {
  if constexpr (VEC == 4) {
    const float4 t = *reinterpret_cast<const float4*>(p);
    a[0] = t.x; a[1] = t.y; a[2] = t.z; a[3] = t.w;
  } else {
    a[0] = *p;
  }
}
template <int VEC>
__device__ __forceinline__ void ldv_nc(float (&a)[VEC], const float* p) {
  if constexpr (VEC == 4) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    a[0] = t.x; a[1] = t.y; a[2] = t.z; a[3] = t.w;
  } else {
    a[0] = __ldg(p);
  }
}
template <int VEC>
__device__ __forceinline__ void ldu(uint32_t (&a)[VEC], const uint32_t* p) {
  if constexpr (VEC == 4) {
    const uint4 t = *reinterpret_cast<const uint4*>(p);
    a[0] = t.x; a[1] = t.y; a[2] = t.z; a[3] = t.w;
  } else {
    a[0] = *p;
  }
}
template <int VEC>
__device__ __forceinline__ void ldu_nc(uint32_t (&a)[VEC], const uint32_t* p) {
  if constexpr (VEC == 4) {
    const uint4 t = __ldg(reinterpret_cast<const uint4*>(p));
    a[0] = t.x; a[1] = t.y; a[2] = t.z; a[3] = t.w;
  } else {
    a[0] = __ldg(p);
  }
}
template <int VEC>
__device__ __forceinline__ void stv(float* p, const float (&a)[VEC]) {
  if constexpr (VEC == 4) *reinterpret_cast<float4*>(p) = make_float4(a[0], a[1], a[2], a[3]);
  else *p = a[0];
}
template <int VEC>
__device__ __forceinline__ void stu(uint32_t* p, const uint32_t (&a)[VEC]) {
  if constexpr (VEC == 4) *reinterpret_cast<uint4*>(p) = make_uint4(a[0], a[1], a[2], a[3]);
  else *p = a[0];
}
// does candidate c replace the best b (c comes later in CSR order)?
template <int OP>
__device__ __forceinline__ bool aggr_better(float c, float b) {
  return (OP == SG_OP_MAX ? (c > b) : (c < b)) || (c != c && b == b);
}

template <int OP, int VEC, int L, int NCH, int U, int MINB>
__global__ void __launch_bounds__(SG_THREADS, MINB)
sg_aggr_kernel(const SgAggrParams a) {
  constexpr bool ARG = OP != SG_OP_ARGBWD;
  constexpr int WPB = SG_THREADS / L;
  constexpr uint32_t CH = SG_CH;
  const SgParams& p = a.p;
  const int lane = threadIdx.x % L;
  const uint32_t w = blockIdx.x * WPB + threadIdx.x / L;
  if (w >= p.numChunks) return;
  const uint32_t* __restrict__ rs = p.rs;
  const uint32_t* __restrict__ col = p.col;

  bool act[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) act[ch] = (uint32_t)(lane + ch * L) < p.Q;
  const uint32_t ce = min(w * CH + CH, p.E);
  const uint4 dA = __ldg(reinterpret_cast<const uint4*>(p.desc) + 2 * (size_t)w);
  const uint4 dB = __ldg(reinterpret_cast<const uint4*>(p.desc) + 2 * (size_t)w + 1);
  if (dB.z & 2u) return;
  uint32_t cur = dA.z, curS = dA.w, curT = dB.x;
  const uint32_t e = dA.x, ee = dA.y, r1 = dB.y, carrySlot = dB.w;
  int kind = (dB.z & 1u) ? 0 : ((curT - curS > CH) ? 2 : 1);
  uint32_t segEnd = (kind == 1) ? curT : min(curT, ce);

  float acc[NCH][VEC];
  uint32_t win[NCH][VEC];
  bool fresh = true;       // no edge of the current segment seen yet (MAX / MIN)
#pragma unroll
  for (int ch = 0; ch < NCH; ch++)
#pragma unroll
    for (int k = 0; k < VEC; k++) { acc[ch][k] = 0.f; win[ch][k] = SG_NO_ARG; }

  // one store site; a segment with no edge (degree-0 row) stores 0 / SG_NO_ARG
  auto flush = [&]() {
    float* dst = (kind == 0) ? static_cast<float*>(p.carry) + (size_t)carrySlot * p.ldC * VEC
                             : static_cast<float*>(p.out) + (size_t)cur * p.ldOut * VEC;
    uint32_t* adst = (kind == 0) ? a.carryArg + (size_t)carrySlot * a.ldCA * VEC : a.arg + (size_t)cur * a.ldArg * VEC;
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
      const int c = (lane + ch * L) * VEC;
      if (act[ch]) {
        stv<VEC>(dst + c, acc[ch]);
        if (ARG && a.arg) stu<VEC>(adst + c, win[ch]);
      }
#pragma unroll
      for (int k = 0; k < VEC; k++) { acc[ch][k] = 0.f; win[ch][k] = SG_NO_ARG; }
    }
    fresh = true;
  };
  auto advance = [&]() {
    cur += 1; curS = curT; curT = rs[cur + 1];
    bool heavy = curT - curS > CH;
    segEnd = heavy ? min(curT, ce) : curT;
    kind = heavy ? 2 : 1;
  };

  // lanes past the row's last column read that column (never stored), so no load needs a predicate
  const float* inl[NCH];
  const uint32_t* argl[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) {
    const uint32_t c = min((uint32_t)(lane + ch * L), p.Q - 1u) * VEC;
    inl[ch] = static_cast<const float*>(p.in) + c;
    argl[ch] = ARG ? nullptr : a.arg + c;
  }
  const uint64_t ldInF = (uint64_t)p.ldIn * VEC, ldArgU = (uint64_t)a.ldArg * VEC;
  const uint32_t eLast = ee - 1u;
#pragma unroll 1
  for (uint32_t base = e; base < ee; base += U) {
    const uint32_t cnt = min((uint32_t)U, ee - base);
    uint32_t srcs[U], gids[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint32_t ei = min(base + (uint32_t)u, eLast);
      srcs[u] = __ldg(col + ei);
      if (ARG) gids[u] = __ldg(a.colG + ei);
    }
    float v[U][NCH][VEC];
    uint32_t av[U][NCH][VEC];
#pragma unroll
    for (int u = 0; u < U; u++) {
#pragma unroll
      for (int ch = 0; ch < NCH; ch++) {
        ldv_nc<VEC>(v[u][ch], inl[ch] + srcs[u] * ldInF);
        if (!ARG) ldu_nc<VEC>(av[u][ch], argl[ch] + srcs[u] * ldArgU);
      }
    }
    uint32_t pos = 0;
    for (;;) {
      const uint32_t lim = min(cnt, segEnd - base);
#pragma unroll
      for (int u = 0; u < U; u++) {
        if ((uint32_t)u >= pos && (uint32_t)u < lim) {
          if constexpr (ARG) {
#pragma unroll
            for (int ch = 0; ch < NCH; ch++)
#pragma unroll
              for (int k = 0; k < VEC; k++)
                if (fresh || aggr_better<OP>(v[u][ch][k], acc[ch][k])) { acc[ch][k] = v[u][ch][k]; win[ch][k] = gids[u]; }
            fresh = false;
          } else {
            const uint32_t me = a.rowLeft + cur;
#pragma unroll
            for (int ch = 0; ch < NCH; ch++)
#pragma unroll
              for (int k = 0; k < VEC; k++)
                if (av[u][ch][k] == me) acc[ch][k] += v[u][ch][k];   // skipped, not +0: -0 sums stay -0
          }
        }
      }
      pos = lim;
      if (pos >= cnt) break;
      flush();
      advance();
    }
  }
  flush();
  while (cur + 1 < r1) { advance(); flush(); }  // trailing zero-degree rows
}

// One worker per heavy row: merge the owner's partial with the carry parts in chunk order.
template <int OP, int VEC, int L, int NCH>
__global__ void __launch_bounds__(SG_THREADS)
sg_aggr_fixup_kernel(const SgAggrParams a) {
  constexpr int WPB = SG_THREADS / L;
  constexpr uint32_t CH = SG_CH;
  const SgParams& p = a.p;
  const int lane = threadIdx.x % L;
  const uint32_t w = blockIdx.x * WPB + threadIdx.x / L;
  if (w >= p.numHeavy) return;
  const uint32_t R = p.heavyRows[w];
  const uint32_t s = p.rs[R], t = p.rs[R + 1];
  const uint32_t n = (t - 1) / CH - s / CH;
  const uint32_t slot0 = p.carryIdx[s / CH + 1];
  float* dst = static_cast<float*>(p.out) + (size_t)R * p.ldOut * VEC;
  uint32_t* adst = a.arg ? a.arg + (size_t)R * a.ldArg * VEC : nullptr;
  const float* cv = static_cast<const float*>(p.carry) + (size_t)slot0 * p.ldC * VEC;
  const uint32_t* ca = a.carryArg + (size_t)slot0 * a.ldCA * VEC;
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) {
    const int c = (lane + ch * L) * VEC;
    if ((uint32_t)(lane + ch * L) >= p.Q) continue;
    float best[VEC];
    uint32_t bw[VEC] = {};
    ldv<VEC>(best, dst + c);
    if (adst) ldu<VEC>(bw, adst + c);
#pragma unroll 4
    for (uint32_t k = 0; k < n; k++) {
      float x[VEC];
      uint32_t xw[VEC] = {};
      ldv<VEC>(x, cv + (size_t)k * p.ldC * VEC + c);
      if (adst) ldu<VEC>(xw, ca + (size_t)k * a.ldCA * VEC + c);
#pragma unroll
      for (int j = 0; j < VEC; j++)
        if (aggr_better<OP>(x[j], best[j])) { best[j] = x[j]; bw[j] = xw[j]; }
    }
    stv<VEC>(dst + c, best);
    if (adst) stu<VEC>(adst + c, bw);
  }
}

// Rows with more than SG_BIG carries: a CTA per row, the lane groups reduce contiguous blocks of the carries and
// group 0 merges owner + blocks in order (one column block at a time through shared memory).
template <int OP, int VEC, int L, int NCH>
__global__ void __launch_bounds__(SG_THREADS)
sg_aggr_fixup_big_kernel(const SgAggrParams a) {
  constexpr int WPB = SG_THREADS / L;
  constexpr uint32_t CH = SG_CH;
  __shared__ float sv[WPB][L * VEC];
  __shared__ uint32_t sw[WPB][L * VEC];
  const SgParams& p = a.p;
  const int lane = threadIdx.x % L;
  const int g = threadIdx.x / L;
  const uint32_t R = p.bigRows[blockIdx.x];
  const uint32_t s = p.rs[R], t = p.rs[R + 1];
  const uint32_t n = (t - 1) / CH - s / CH;
  const uint32_t slot0 = p.carryIdx[s / CH + 1];
  const uint32_t per = (n + WPB - 1) / WPB;
  const uint32_t k0 = min(n, (uint32_t)g * per), k1 = min(n, k0 + per);
  float* dst = static_cast<float*>(p.out) + (size_t)R * p.ldOut * VEC;
  uint32_t* adst = a.arg ? a.arg + (size_t)R * a.ldArg * VEC : nullptr;
  const float* cv = static_cast<const float*>(p.carry) + (size_t)slot0 * p.ldC * VEC;
  const uint32_t* ca = a.carryArg + (size_t)slot0 * a.ldCA * VEC;
#pragma unroll 1
  for (int ch = 0; ch < NCH; ch++) {
    const int c = (lane + ch * L) * VEC;
    const bool act = (uint32_t)(lane + ch * L) < p.Q;
    if (act && k0 < k1) {
      float best[VEC];
      uint32_t bw[VEC] = {};
      ldv<VEC>(best, cv + (size_t)k0 * p.ldC * VEC + c);
      if (adst) ldu<VEC>(bw, ca + (size_t)k0 * a.ldCA * VEC + c);
#pragma unroll 1
      for (uint32_t k = k0 + 1; k < k1; k++) {
        float x[VEC];
        uint32_t xw[VEC] = {};
        ldv<VEC>(x, cv + (size_t)k * p.ldC * VEC + c);
        if (adst) ldu<VEC>(xw, ca + (size_t)k * a.ldCA * VEC + c);
#pragma unroll
        for (int j = 0; j < VEC; j++)
          if (aggr_better<OP>(x[j], best[j])) { best[j] = x[j]; bw[j] = xw[j]; }
      }
#pragma unroll
      for (int j = 0; j < VEC; j++) { sv[g][lane * VEC + j] = best[j]; sw[g][lane * VEC + j] = bw[j]; }
    }
    __syncthreads();
    if (g == 0 && act) {
      float best[VEC];
      uint32_t bw[VEC] = {};
      ldv<VEC>(best, dst + c);                       // the owner chunk's raw partial
      if (adst) ldu<VEC>(bw, adst + c);
      for (int gg = 0; gg < WPB; gg++) {
        if ((uint32_t)gg * per >= n) break;          // this group and the later ones hold no carries
#pragma unroll
        for (int j = 0; j < VEC; j++) {
          const float x = sv[gg][lane * VEC + j];
          if (aggr_better<OP>(x, best[j])) { best[j] = x; bw[j] = sw[gg][lane * VEC + j]; }
        }
      }
      stv<VEC>(dst + c, best);
      if (adst) stu<VEC>(adst + c, bw);
    }
    __syncthreads();
  }
}

template <int OP, int VEC, int L, int NCH, int U, int MINB>
static int launch_aggr_cfg(const SgAggrParams& a, cudaStream_t st) {
  constexpr int WPB = SG_THREADS / L;
  constexpr int UU = (OP == SG_OP_ARGBWD && U > 1) ? U / 2 : U;   // two rows per edge: half the edges in flight
  // cut rows of ARGBWD are plain sums: SUM's fix-up kernels (the same instantiations SUM launches) finish them
  const SgParams& p = a.p;
  if (p.numChunks) {
    sg_aggr_kernel<OP, VEC, L, NCH, UU, MINB><<<(p.numChunks + WPB - 1) / WPB, SG_THREADS, 0, st>>>(a);
    ROC_LAUNCH_CHECK();
  }
  if (p.numHeavy) {
    const unsigned grid = (p.numHeavy + WPB - 1) / WPB;
    if constexpr (OP == SG_OP_ARGBWD) sg_fixup_kernel<VEC, L, NCH, U><<<grid, SG_THREADS, 0, st>>>(p);
    else sg_aggr_fixup_kernel<OP, VEC, L, NCH><<<grid, SG_THREADS, 0, st>>>(a);
    ROC_LAUNCH_CHECK();
  }
  if (p.numBig) {
    if constexpr (OP == SG_OP_ARGBWD) sg_fixup_big_kernel<VEC, L, NCH, U><<<p.numBig, SG_THREADS, 0, st>>>(p);
    else sg_aggr_fixup_big_kernel<OP, VEC, L, NCH><<<p.numBig, SG_THREADS, 0, st>>>(a);
    ROC_LAUNCH_CHECK();
  }
  return ROC_OK;
}

template <int OP, int VEC>
static int dispatch_aggr(const SgAggrParams& a, cudaStream_t st) {
  const uint32_t Q = a.p.Q;
  if (Q <= 4) return launch_aggr_cfg<OP, VEC, 4, 1, 4, 4>(a, st);
  if (Q <= 8) return launch_aggr_cfg<OP, VEC, 8, 1, 8, 3>(a, st);
  if (Q <= 16) return launch_aggr_cfg<OP, VEC, 16, 1, 8, 3>(a, st);
  if (Q <= 32) return launch_aggr_cfg<OP, VEC, 32, 1, 8, 3>(a, st);
  if (Q <= 64) return launch_aggr_cfg<OP, VEC, 32, 2, 4, 2>(a, st);
  if (Q <= 128) return launch_aggr_cfg<OP, VEC, 32, 4, 2, 2>(a, st);
  if (Q <= 256) return launch_aggr_cfg<OP, VEC, 32, 8, 1, 1>(a, st);
  return ROC_ERR_UNSUPPORTED;
}

// Variant A keeps the gathers in registers, variant C stages them in shared memory with
// cp.async; C wins once a row needs two or more float4 per lane at L = 32 (H > 128).
// ROC_SG_VARIANT=a|c forces one (experiments / cross-checks).
static int sg_variant_env() {   // -1 default, 0 = A, 2 = C, 3 = T (TMA gather4), 4 = T with per-row bulk copies, 5 = R (ring)
  const char* e = getenv("ROC_SG_VARIANT");   // re-read per call: the kernel bench switches it in-process
  if (!e) return -1;
  switch (e[0]) { case 'a': return 0; case 'c': return 2; case 't': return 3; case 'b': return 4; case 'r': return 5; case 'u': return 6; default: return -1; }
}
static int sg_deep_env() {   // ROC_SG_DEEP=1: variant C with a 2x deeper ring (experiments)
  const char* e = getenv("ROC_SG_DEEP");
  return (e && e[0] == '1') ? 1 : 0;
}
static int sg_tcfg_env() {   // ROC_SG_TCFG=<n>: ring shape of variant T (experiments; see launch_t_cfg)
  const char* e = getenv("ROC_SG_TCFG");
  return e ? atoi(e) : -1;
}

template <int L, int NCH, int GROUP, int P>
static cudaError_t launch_c(const SgParams& p, unsigned grid, cudaStream_t st) {
  constexpr int WPB = SG_THREADS / L;
  constexpr size_t smem = (size_t)WPB * GROUP * P * NCH * L * sizeof(float4);
  static std::atomic<uint64_t> configured{0};      // one bit per device: the attribute is per device
  cudaError_t e = once_per_device(configured, [] {
    return cudaFuncSetAttribute(sg_chunk_kernel_c2<L, NCH, GROUP, P>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  });
  if (e != cudaSuccess) return e;
  sg_chunk_kernel_c2<L, NCH, GROUP, P><<<grid, SG_THREADS, smem, st>>>(p);
  return cudaGetLastError();
}

// ---- variant T launchers: ring = P stages x S gather4s per worker, NT threads per CTA
template <int L, int NCH, int S, int P, int NT, int MINB, int MODE>
static cudaError_t launch_t(const SgParams& p, const CUtensorMap& tm, cudaStream_t st) {
  constexpr int WPB = NT / L;
  constexpr size_t smem = (size_t)WPB * P * S * 4 * NCH * L * 16 + (size_t)WPB * P * 8;
  static_assert(smem <= 227 * 1024, "ring too large");
  static std::atomic<uint64_t> configured{0};
  cudaError_t e = once_per_device(configured, [] {
    return cudaFuncSetAttribute(sg_chunk_kernel_t<L, NCH, S, P, NT, MINB, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  });
  if (e != cudaSuccess) return e;
  const unsigned grid = (p.numChunks + WPB - 1) / WPB;
  sg_chunk_kernel_t<L, NCH, S, P, NT, MINB, MODE><<<grid, NT, smem, st>>>(p, tm);
  return cudaGetLastError();
}

// ---- variant R launcher: NPW producer warps + two worker warps per CTA, MINB CTAs per SM
template <int VW, int NCH, int NPW, int MINB>
static cudaError_t launch_r(const SgParams& p, const CUtensorMap& tm, cudaStream_t st) {
  constexpr size_t smem = (size_t)2 * SG_CH * NCH * 32 * VW * 4 + 64;
  static_assert(smem * MINB <= 227 * 1024, "ring too large");
  static std::atomic<uint64_t> configured{0};
  cudaError_t e = once_per_device(configured, [] {
    return cudaFuncSetAttribute(sg_ring_kernel<VW, NCH, NPW, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  });
  if (e != cudaSuccess) return e;
  const uint32_t numPairs = (p.numChunks + 1u) >> 1;
  uint32_t grid = (uint32_t)sm_count() * MINB * 2u;        // two CTA ranges per resident slot
  if (grid > numPairs) grid = numPairs;
  const uint32_t per = (numPairs + grid - 1) / grid;
  grid = (numPairs + per - 1) / per;
  sg_ring_kernel<VW, NCH, NPW, MINB><<<grid, 32 * (NPW + 2), smem, st>>>(p, tm, per);
  return cudaGetLastError();
}
// rows of up to 256 / 512 / 1024 bytes: 32 / 64 / 128 KB of ring per CTA.  cfg = producer warps (experiments)
static cudaError_t launch_r_cfg(const SgParams& p, const CUtensorMap& tm, int cfg, cudaStream_t st) {
  if (p.Q <= 16) {
    switch (cfg) {
      case 1: return launch_r<2, 1, 1, 6>(p, tm, st);
      case 4: return launch_r<2, 1, 4, 6>(p, tm, st);
      default: return launch_r<2, 1, 2, 6>(p, tm, st);
    }
  }
  if (p.Q <= 32) {
    switch (cfg) {
      case 1: return launch_r<4, 1, 1, 3>(p, tm, st);
      case 4: return launch_r<4, 1, 4, 3>(p, tm, st);
      default: return launch_r<4, 1, 2, 3>(p, tm, st);
    }
  }
  switch (cfg) {
    case 1: return launch_r<4, 2, 1, 1>(p, tm, st);
    case 4: return launch_r<4, 2, 4, 1>(p, tm, st);
    default: return launch_r<4, 2, 2, 1>(p, tm, st);
  }
}

// Ring shapes.  cfg < 0: the default for this width (chosen by measurement, DESIGN.md §3.1).
template <int L, int NCH, int MODE>
static cudaError_t launch_t_cfg(const SgParams& p, const CUtensorMap& tm, int cfg, cudaStream_t st) {
  // bytes per row slot = NCH*L*16; per worker ring = P*S*4 slots
  if constexpr (NCH * L <= 16) {          // rows <= 256 B: 2+ workers per warp
    switch (cfg) {
      case 1: return launch_t<L, NCH, 2, 2, 128, 4, MODE>(p, tm, st);
      case 2: return launch_t<L, NCH, 1, 8, 128, 3, MODE>(p, tm, st);
      case 3: return launch_t<L, NCH, 2, 4, 128, 3, MODE>(p, tm, st);
      case 4: return launch_t<L, NCH, 1, 4, 256, 3, MODE>(p, tm, st);
      case 5: return launch_t<L, NCH, 1, 3, 128, 8, MODE>(p, tm, st);
      case 6: return launch_t<L, NCH, 1, 6, 128, 4, MODE>(p, tm, st);
      default: return launch_t<L, NCH, 1, 4, 128, 6, MODE>(p, tm, st);
    }
  } else if constexpr (NCH == 1) {        // 512 B rows, one worker per warp
    if (cfg < 0 && MODE == 2) cfg = 1;     // ids held by the lanes: two 8-edge stages (3.18 ms vs 5.45 with four 4-edge ones)
    switch (cfg) {
      case 1: return launch_t<L, NCH, 2, 2, 128, 4, MODE>(p, tm, st);
      case 2: return launch_t<L, NCH, 1, 8, 128, 3, MODE>(p, tm, st);
      case 3: return launch_t<L, NCH, 1, 3, 128, 8, MODE>(p, tm, st);
      default: return launch_t<L, NCH, 1, 4, 128, 6, MODE>(p, tm, st);
    }
  } else {                                 // 1 KB rows: two 4 KB stages per warp, 6 CTAs (7.08 ms vs 8.34 with 4 stages x 3 CTAs)
    switch (cfg) {
      case 1: return launch_t<L, NCH, 1, 4, 128, 3, MODE>(p, tm, st);
      case 2: return launch_t<L, NCH, 1, 6, 128, 2, MODE>(p, tm, st);
      case 3: return launch_t<L, NCH, 1, 3, 128, 4, MODE>(p, tm, st);
      default: return launch_t<L, NCH, 1, 2, 128, 6, MODE>(p, tm, st);
    }
  }
}

// variant C rings: DEPTH = GROUP * P row slots per worker, 64 KB per CTA (128 KB with ROC_SG_DEEP=1)
template <int L, int NCH>
static cudaError_t launch_c_cfg(const SgParams& p, unsigned grid, cudaStream_t st) {
  const bool deep = sg_deep_env() == 1;
  if constexpr (NCH == 1) return deep ? launch_c<L, NCH, 4, 8>(p, grid, st) : launch_c<L, NCH, 4, 4>(p, grid, st);
  else if constexpr (NCH == 2) return deep ? launch_c<L, NCH, 2, 8>(p, grid, st) : launch_c<L, NCH, 2, 4>(p, grid, st);
  else if constexpr (NCH == 4) return deep ? launch_c<L, NCH, 1, 8>(p, grid, st) : launch_c<L, NCH, 1, 4>(p, grid, st);
  else return deep ? launch_c<L, NCH, 1, 4>(p, grid, st) : launch_c<L, NCH, 1, 2>(p, grid, st);
}

struct SgLaunch {
  int variant;               // 0 = A, 2 = C, 3 = T (gather4), 4 = T (bulk rows)
  int tcfg;                  // ring shape of variant T (-1 = default)
  const CUtensorMap* tmap;   // variant T (gather4) only
};

template <int VEC, int L, int NCH, int U, int MINB>
static int launch_cfg(const SgParams& p, const SgLaunch& how, cudaStream_t st) {
  constexpr int WPB = SG_THREADS / L;
  if (p.numChunks) {
    unsigned grid = (p.numChunks + WPB - 1) / WPB;
    int variant = how.variant;
    bool done = false;
    if constexpr (VEC == 4 && NCH <= 2 && L >= 16) {
      if (variant == 5) {
        cudaError_t e = launch_r_cfg(p, *how.tmap, how.tcfg, st);
        if (e != cudaSuccess) return (int)e;
        count_launch();
        done = true;
      }
    }
    if constexpr (VEC == 4 && NCH <= 2 && L >= 16) {
      if (variant == 6) {
        cudaError_t e = launch_t_cfg<L, NCH, 2>(p, *how.tmap, how.tcfg, st);
        if (e != cudaSuccess) return (int)e;
        count_launch();
        done = true;
      }
    }
    if constexpr (VEC == 4 && NCH <= 2) {
      if (variant == 3 || variant == 4) {
        cudaError_t e = (variant == 3) ? launch_t_cfg<L, NCH, 0>(p, *how.tmap, how.tcfg, st)
                                       : launch_t_cfg<L, NCH, 1>(p, *how.tmap, how.tcfg, st);
        if (e != cudaSuccess) return (int)e;
        count_launch();
        done = true;
      }
    }
    if constexpr (VEC == 4) {
      if (!done && variant == 2) {
        cudaError_t e = launch_c_cfg<L, NCH>(p, grid, st);
        if (e != cudaSuccess) return (int)e;
        count_launch();
        done = true;
      }
    }
    if (!done) {
      sg_chunk_kernel<VEC, L, NCH, U, MINB><<<grid, SG_THREADS, 0, st>>>(p);
      ROC_LAUNCH_CHECK();
    }
  }
  if (p.numHeavy) {
    unsigned grid = (p.numHeavy + WPB - 1) / WPB;
    sg_fixup_kernel<VEC, L, NCH, U><<<grid, SG_THREADS, 0, st>>>(p);
    ROC_LAUNCH_CHECK();
  }
  if (p.numBig) {
    sg_fixup_big_kernel<VEC, L, NCH, U><<<p.numBig, SG_THREADS, 0, st>>>(p);
    ROC_LAUNCH_CHECK();
  }
  return ROC_OK;
}

template <int VEC>
static int dispatch(const SgParams& p, const SgLaunch& how, cudaStream_t st) {
  const uint32_t Q = p.Q;
  if (Q <= 4) return launch_cfg<VEC, 4, 1, 4, 4>(p, how, st);
  if (Q <= 8) return launch_cfg<VEC, 8, 1, 8, 4>(p, how, st);
  if (Q <= 16) return launch_cfg<VEC, 16, 1, 8, 4>(p, how, st);
  if (Q <= 32) return launch_cfg<VEC, 32, 1, 8, 4>(p, how, st);
  if (Q <= 64) return launch_cfg<VEC, 32, 2, 4, 3>(p, how, st);
  if (Q <= 128) return launch_cfg<VEC, 32, 4, 2, 3>(p, how, st);
  if (Q <= 256) return launch_cfg<VEC, 32, 8, 1, 2>(p, how, st);
  return ROC_ERR_UNSUPPORTED;
}

// The variant for a vectorised launch of Q float4 columns.  Default: chosen by measurement per width
// (DESIGN.md §3.1); ROC_SG_VARIANT=a|c|t|b forces one (experiments / cross-checks).
static int pick_variant(uint32_t Q, bool vec) {
  int v = sg_variant_env();
  if (!vec) return 0;
  // measured on R-MAT-22 (r2 runs 2 / 6 / 8 and session 5, ms at H = 64 / 128 / 256): A 1.91 / 3.55 / 7.9,
  // C 2.65 / 4.40 / 7.8, T 2.11 / 3.42 / 7.08, T with lane-held ids (U) 2.20 / 3.18 / 6.77, R 2.43 / 4.5 / 15.3
  // -> registers up to 64 floats, the TMA gather4 ring with lane-held ids for 65..128, with per-stage ids for 129..256
  if (v < 0) v = (Q > 64) ? 2 : (Q > 32 ? 3 : (Q > 16 ? 6 : 0));   // 129..256: U's 4 % over T not worth a less exercised path
  if ((v == 3 || v == 4 || v == 5 || v == 6) && Q > 64) v = 2;     // TMA boxes are at most 256 elements wide
  if ((v == 5 || v == 6) && Q <= 8) v = 0;                // these want rows of 9+ float4
  return v;
}

// Carry slots for rows cut at chunk boundaries.  roc_sg_plan_reserve sizes them up front (plain cudaMalloc, an
// init-time call).  A launch that still finds them too small grows them on its own stream with stream-ordered
// allocation: the old buffer is returned in stream order, after the launches that used it — no device
// synchronisation in the middle of a step.
template <typename W>
static int grow_carry(const roc_sg_plan* plan, W*& buf, size_t& have, size_t ld, cudaStream_t st, bool inStream) {
  if (plan->numCarries == 0 || ld <= have) return ROC_OK;
  if (buf) {
    if (inStream) ROC_CUDA(cudaFreeAsync(buf, st));
    else { ROC_CUDA(cudaDeviceSynchronize()); ROC_CUDA(cudaFree(buf)); }
    buf = nullptr; have = 0;
  }
  const size_t bytes = (size_t)plan->numCarries * ld * sizeof(W);
  cudaError_t e = inStream ? cudaMallocAsync((void**)&buf, bytes, st) : cudaMalloc((void**)&buf, bytes);
  if (e != cudaSuccess) { buf = nullptr; have = 0; return (int)e; }
  have = ld;
  return ROC_OK;
}
static int ensure_carry(roc_sg_plan* plan, size_t ldFloats, cudaStream_t st, bool inStream) {
  return grow_carry(plan, plan->carry, plan->carryLd, ldFloats, st, inStream);
}
// the u32 twins of the carry slots: winner ids of the MAX / MIN carry parts
static int ensure_carry_arg(roc_sg_plan* plan, size_t ld, cudaStream_t st, bool inStream) {
  return grow_carry(plan, plan->carryArg, plan->carryArgLd, ld, st, inStream);
}

// ------------------------------------------------------------------ graph attention (GAT) ---
// out[v, k-block] = sum over u in in(v) of alpha[v<-u,k] h[u, k-block], alpha = softmax over the row's in-edges of
// LeakyReLU(s_src[u,k] + s_dst[v,k]).  Per-node tensors: att[r] = (s_src[0..K) | s_dst[0..K)), bst[r] = (lse[0..K) |
// c[0..K)), both indexed like h ([own rows | halo rows]).  Kernels, all on the plan's chunk schedule, no atomics:
//   k_gat_rowdot        s_src / s_dst (forward) and c = <dOut, out> (backward): a warp per row, fixed-order dots
//   k_gat_stats         lse per row and head; a thread per chunk with an online (max, Z) pair; rows cut at chunk
//                       boundaries leave (max, Z) parts (owner: in its bst row, later chunks: in the carry slots)
//   k_gat_stats_fixup   merges those parts in chunk order (a warp per cut row, lanes own contiguous carry blocks)
//   sg_gat_kernel       kernel A with each gathered row scaled by alpha before the add; cut rows: SUM's fix-ups
//   sg_gat_bwd_kernel   row u gathers dOut[v], h[v], att[v], bst[v]: dh_agg[u] and ds_src / ds_dst[u]; cut rows:
//                       SUM's fix-ups over the [dh | ds] carry part
//   k_gat_finish        dh += ds_src a_src + ds_dst a_dst, and the fixed-block partials of da; k_gat_da_reduce sums
//                       the partials in block order
// alpha is never stored: gat_alpha below is the one place it is computed, by the forward and the backward alike.
constexpr int GAT_ROWDOT_WARPS = 8;
constexpr int GAT_FINISH_THREADS = 256;
constexpr uint32_t GAT_FINISH_BLOCKS = 1184;   // fixed: the da partial order depends on the row count only

__device__ __forceinline__ float gat_leaky(float z, float slope) { return z > 0.f ? z : z * slope; }
__device__ __forceinline__ float gat_dleaky(float z, float slope) { return z > 0.f ? 1.f : slope; }
__device__ __forceinline__ float gat_alpha(float sSrcU, float sDstV, float lseV, float slope) {
  return expf(gat_leaky(sSrcU + sDstV, slope) - lseV);
}
// (m, z) <- (m, z) + (m2, z2) for z = sum exp(e - m).  An empty part is (-inf, 0).
__device__ __forceinline__ void gat_lse_merge(float& m, float& z, float m2, float z2) {
  const float M = fmaxf(m, m2);
  if (M == -INFINITY) return;
  z = z * expf(m - M) + z2 * expf(m2 - M);
  m = M;
}

// dst1[r][k] = <x[r, k-block], y1[k-block]> (y1 one vector when ldY1 == 0, else a row per r); the same for y2 when
// given.  A warp per row, lanes stride the head's columns, xor-butterfly sum: fixed order.
__global__ void __launch_bounds__(32 * GAT_ROWDOT_WARPS)
k_gat_rowdot(int64_t rows, int F, int K, const float* __restrict__ x, int64_t ldX, const float* __restrict__ y1,
             int64_t ldY1, const float* __restrict__ y2, int64_t ldY2, float* __restrict__ dst1,
             float* __restrict__ dst2, int64_t ldD) {
  const int64_t r = (int64_t)blockIdx.x * GAT_ROWDOT_WARPS + threadIdx.x / 32;
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* xr = x + r * ldX;
  const float* a = y1 + r * ldY1;
  const float* b = y2 ? y2 + r * ldY2 : nullptr;
  for (int k = 0; k < K; k++) {
    float p1 = 0.f, p2 = 0.f;
    for (int j = lane; j < F; j += 32) {
      const float xv = xr[k * F + j];
      p1 = fmaf(xv, a[k * F + j], p1);
      if (b) p2 = fmaf(xv, b[k * F + j], p2);
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
      p1 += __shfl_xor_sync(0xffffffffu, p1, o);
      p2 += __shfl_xor_sync(0xffffffffu, p2, o);
    }
    if (lane == 0) {
      dst1[r * ldD + k] = p1;
      if (b) dst2[r * ldD + k] = p2;
    }
  }
}

struct GatParams {
  SgParams p;               // schedule; in / out / carry as the kernel uses them (VEC-float units)
  const float* att;         // [own | halo][ldA]  s_src | s_dst
  const float* bst;         // [own | halo][ldB]  lse | c  (written by the stats kernels, read by the others)
  float* bstOut;            // stats: the same rows, writable
  const float* dOut;        // backward: [own | halo][ldG] (VEC units)
  float* ds;                // backward: [nloc][ldDs]  ds_src | ds_dst
  size_t ldA, ldB, ldG, ldDs;
  uint32_t dsOff;           // backward: float offset of the ds part in a carry slot
  int H, F, K;              // width, floats per head, heads
  int FQ;                   // VEC-columns per head
  int hmode;                // per-head sums: 0 one head, 1 power-of-two heads narrower than the worker, 2 general
  float slope;
};

// lse per row and head: one thread per chunk walks the chunk's edges in order.
template <int K>
__global__ void __launch_bounds__(256)
k_gat_stats(const GatParams g) {
  constexpr uint32_t CH = SG_CH;
  constexpr int U = 4;
  const SgParams& p = g.p;
  const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= p.numChunks) return;
  const uint4 dA = __ldg(reinterpret_cast<const uint4*>(p.desc) + 2 * (size_t)w);
  const uint4 dB = __ldg(reinterpret_cast<const uint4*>(p.desc) + 2 * (size_t)w + 1);
  if (dB.z & 2u) return;
  const uint32_t ce = min(w * CH + CH, p.E);
  uint32_t cur = dA.z, curS = dA.w, curT = dB.x;
  const uint32_t ee = dA.y, r1 = dB.y, carrySlot = dB.w;
  int kind = (dB.z & 1u) ? 0 : ((curT - curS > CH) ? 2 : 1);
  uint32_t segEnd = (kind == 1) ? curT : min(curT, ce);
  float sd[K], m[K], z[K];
  auto rowvals = [&]() {
#pragma unroll
    for (int k = 0; k < K; k++) { sd[k] = g.att[(size_t)cur * g.ldA + K + k]; m[k] = -INFINITY; z[k] = 0.f; }
  };
  auto flush = [&]() {
    if (kind == 1) {
#pragma unroll
      for (int k = 0; k < K; k++) g.bstOut[(size_t)cur * g.ldB + k] = (curT > curS) ? m[k] + logf(z[k]) : 0.f;
    } else {
      // a raw (max, Z) part: the owner's in its own bst row (its c columns are free in the forward), later
      // chunks' in their carry slot
      float* d = (kind == 2) ? g.bstOut + (size_t)cur * g.ldB : static_cast<float*>(p.carry) + (size_t)carrySlot * p.ldC;
#pragma unroll
      for (int k = 0; k < K; k++) { d[k] = m[k]; d[K + k] = z[k]; }
    }
  };
  auto advance = [&]() {
    cur += 1; curS = curT; curT = p.rs[cur + 1];
    const bool heavy = curT - curS > CH;
    segEnd = heavy ? min(curT, ce) : curT;
    kind = heavy ? 2 : 1;
    rowvals();
  };
  rowvals();
  const uint32_t eLast = ee - 1u;
#pragma unroll 1
  for (uint32_t base = dA.x; base < ee; base += U) {
    float ss[U][K];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint32_t src = __ldg(p.col + min(base + (uint32_t)u, eLast));
#pragma unroll
      for (int k = 0; k < K; k++) ss[u][k] = __ldg(g.att + (size_t)src * g.ldA + k);
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint32_t e = base + (uint32_t)u;
      if (e < ee) {
        while (e == segEnd) { flush(); advance(); }
#pragma unroll
        for (int k = 0; k < K; k++) gat_lse_merge(m[k], z[k], gat_leaky(ss[u][k] + sd[k], g.slope), 1.f);
      }
    }
  }
  flush();
  while (cur + 1 < r1) { advance(); flush(); }   // trailing zero-degree rows
}

// Rows cut at chunk boundaries (heavy and big alike): a warp per row; lane l merges the l-th contiguous block of the
// carry parts, lane 0 then merges owner + blocks in lane order.
template <int K>
__global__ void __launch_bounds__(256)
k_gat_stats_fixup(const GatParams g) {
  constexpr uint32_t CH = SG_CH;
  const SgParams& p = g.p;
  const uint32_t wg = (blockIdx.x * blockDim.x + threadIdx.x) / 32;
  const int lane = threadIdx.x & 31;
  if (wg >= p.numHeavy + p.numBig) return;
  const uint32_t R = wg < p.numHeavy ? p.heavyRows[wg] : p.bigRows[wg - p.numHeavy];
  const uint32_t s = p.rs[R], t = p.rs[R + 1];
  const uint32_t n = (t - 1) / CH - s / CH;
  const uint32_t slot0 = p.carryIdx[s / CH + 1];
  const uint32_t per = (n + 31) / 32;
  const uint32_t k0 = min(n, (uint32_t)lane * per), k1 = min(n, k0 + per);
  const float* cv = static_cast<const float*>(p.carry);
  float m[K], z[K];
#pragma unroll
  for (int k = 0; k < K; k++) { m[k] = -INFINITY; z[k] = 0.f; }
  for (uint32_t c = k0; c < k1; c++) {
    const float* part = cv + (size_t)(slot0 + c) * p.ldC;
#pragma unroll
    for (int k = 0; k < K; k++) gat_lse_merge(m[k], z[k], part[k], part[K + k]);
  }
  float* row = g.bstOut + (size_t)R * g.ldB;
  float om[K], oz[K];
#pragma unroll
  for (int k = 0; k < K; k++) { om[k] = row[k]; oz[k] = row[K + k]; }
  for (int l = 0; l < 32; l++) {
#pragma unroll
    for (int k = 0; k < K; k++) {
      const float mm = __shfl_sync(0xffffffffu, m[k], l), zz = __shfl_sync(0xffffffffu, z[k], l);
      gat_lse_merge(om[k], oz[k], mm, zz);
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < K; k++) { row[k] = om[k] + logf(oz[k]); row[K + k] = 0.f; }
  }
}

// Per-head sums of per-lane partials p[ch] (lane's VEC-column lane + ch * L lies in head hd[ch]) over the worker's
// L lanes; every lane ends with its heads' sums, bitwise equal across the lanes (xor butterflies).
template <int L, int NCH>
__device__ __forceinline__ void gat_headsum(float (&p)[NCH], const int (&hd)[NCH], const GatParams& g, unsigned wmask) {
  if (g.hmode == 0) {
    float s = 0.f;
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) s += p[ch];
#pragma unroll
    for (int o = L / 2; o >= 1; o >>= 1) s += __shfl_xor_sync(wmask, s, o);
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) p[ch] = s;
  } else if (g.hmode == 1) {
#pragma unroll
    for (int ch = 0; ch < NCH; ch++)
      for (int o = g.FQ / 2; o >= 1; o >>= 1) p[ch] += __shfl_xor_sync(wmask, p[ch], o);
  } else {
    float q[NCH];
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) q[ch] = 0.f;
    for (int k = 0; k < g.K; k++) {
      float s = 0.f;
#pragma unroll
      for (int ch = 0; ch < NCH; ch++) s += (hd[ch] == k) ? p[ch] : 0.f;
#pragma unroll
      for (int o = L / 2; o >= 1; o >>= 1) s += __shfl_xor_sync(wmask, s, o);
#pragma unroll
      for (int ch = 0; ch < NCH; ch++) if (hd[ch] == k) q[ch] = s;
    }
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) p[ch] = q[ch];
  }
}

// Weighted aggregate: kernel A's schedule and per-row order, each gathered row scaled by its alpha (per head) before
// the add.  Rows cut at chunk boundaries store raw partial sums; SUM's fix-up kernels finish them (epi = 0).
template <int VEC, int L, int NCH, int U, int MINB>
__global__ void __launch_bounds__(SG_THREADS, MINB)
sg_gat_kernel(const GatParams g) {
  constexpr int WPB = SG_THREADS / L;
  constexpr uint32_t CH = SG_CH;
  const SgParams& p = g.p;
  const int lane = threadIdx.x % L;
  const uint32_t w = blockIdx.x * WPB + threadIdx.x / L;
  if (w >= p.numChunks) return;
  bool act[NCH];
  int hd[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) {
    act[ch] = (uint32_t)(lane + ch * L) < p.Q;
    hd[ch] = min((uint32_t)(lane + ch * L), p.Q - 1u) / (uint32_t)g.FQ;
  }
  const uint32_t ce = min(w * CH + CH, p.E);
  const uint4 dA = __ldg(reinterpret_cast<const uint4*>(p.desc) + 2 * (size_t)w);
  const uint4 dB = __ldg(reinterpret_cast<const uint4*>(p.desc) + 2 * (size_t)w + 1);
  if (dB.z & 2u) return;
  uint32_t cur = dA.z, curS = dA.w, curT = dB.x;
  const uint32_t e = dA.x, ee = dA.y, r1 = dB.y, carrySlot = dB.w;
  int kind = (dB.z & 1u) ? 0 : ((curT - curS > CH) ? 2 : 1);
  uint32_t segEnd = (kind == 1) ? curT : min(curT, ce);

  float acc[NCH][VEC], sd[NCH], ls[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++)
#pragma unroll
    for (int k = 0; k < VEC; k++) acc[ch][k] = 0.f;
  auto rowvals = [&]() {
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
      sd[ch] = g.att[(size_t)cur * g.ldA + g.K + hd[ch]];
      ls[ch] = g.bst[(size_t)cur * g.ldB + hd[ch]];
    }
  };
  auto flush = [&]() {
    float* dst = (kind == 0) ? static_cast<float*>(p.carry) + (size_t)carrySlot * p.ldC * VEC
                             : static_cast<float*>(p.out) + (size_t)cur * p.ldOut * VEC;
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
      if (act[ch]) stv<VEC>(dst + (lane + ch * L) * VEC, acc[ch]);
#pragma unroll
      for (int k = 0; k < VEC; k++) acc[ch][k] = 0.f;
    }
  };
  auto advance = [&]() {
    cur += 1; curS = curT; curT = p.rs[cur + 1];
    const bool heavy = curT - curS > CH;
    segEnd = heavy ? min(curT, ce) : curT;
    kind = heavy ? 2 : 1;
    rowvals();
  };
  rowvals();
  const float* inl[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) inl[ch] = static_cast<const float*>(p.in) + min((uint32_t)(lane + ch * L), p.Q - 1u) * VEC;
  const uint64_t ldInF = (uint64_t)p.ldIn * VEC;
  const uint32_t eLast = ee - 1u;
#pragma unroll 1
  for (uint32_t base = e; base < ee; base += U) {
    const uint32_t cnt = min((uint32_t)U, ee - base);
    uint32_t srcs[U];
#pragma unroll
    for (int u = 0; u < U; u++) srcs[u] = __ldg(p.col + min(base + (uint32_t)u, eLast));
    float v[U][NCH][VEC], ss[U][NCH];
#pragma unroll
    for (int u = 0; u < U; u++)
#pragma unroll
      for (int ch = 0; ch < NCH; ch++) {
        ldv_nc<VEC>(v[u][ch], inl[ch] + srcs[u] * ldInF);
        ss[u][ch] = __ldg(g.att + (size_t)srcs[u] * g.ldA + hd[ch]);
      }
    uint32_t pos = 0;
    for (;;) {
      const uint32_t lim = min(cnt, segEnd - base);
#pragma unroll
      for (int u = 0; u < U; u++) {
        if ((uint32_t)u >= pos && (uint32_t)u < lim) {
#pragma unroll
          for (int ch = 0; ch < NCH; ch++) {
            const float a = gat_alpha(ss[u][ch], sd[ch], ls[ch], g.slope);
#pragma unroll
            for (int k = 0; k < VEC; k++) acc[ch][k] = fmaf(a, v[u][ch][k], acc[ch][k]);
          }
        }
      }
      pos = lim;
      if (pos >= cnt) break;
      flush();
      advance();
    }
  }
  flush();
  while (cur + 1 < r1) { advance(); flush(); }
}

// Backward gather: row u (the plan's row) walks its in-edges v (by the CSR's symmetry, the v that u feeds):
//   dh_agg[u] += alpha[v<-u] dOut[v]
//   ds_src[u] += alpha[v<-u] (<dOut[v], h[u]> - c[v]) LeakyReLU'(s_src[u] + s_dst[v])
//   ds_dst[u] += alpha[u<-v] (<dOut[u], h[v]> - c[u]) LeakyReLU'(s_src[v] + s_dst[u])
// (per head).  Two rows gathered per edge.  Rows cut at chunk boundaries: the owner stores its raw parts into the
// dh and ds rows, later chunks into the carry slot ([dh | ds] at dsOff); SUM's fix-ups sum them in chunk order.
template <int VEC, int L, int NCH, int U, int MINB>
__global__ void __launch_bounds__(SG_THREADS, MINB)
sg_gat_bwd_kernel(const GatParams g) {
  constexpr int WPB = SG_THREADS / L;
  constexpr uint32_t CH = SG_CH;
  const SgParams& p = g.p;
  const int lane = threadIdx.x % L;
  const uint32_t w = blockIdx.x * WPB + threadIdx.x / L;
  if (w >= p.numChunks) return;
  const unsigned wmask = (L == 32) ? 0xffffffffu : (((1u << L) - 1u) << (((threadIdx.x & 31) / L) * L));
  bool act[NCH], first[NCH];
  int hd[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) {
    const uint32_t t = lane + ch * L;
    act[ch] = t < p.Q;
    hd[ch] = min(t, p.Q - 1u) / (uint32_t)g.FQ;
    first[ch] = act[ch] && (t % (uint32_t)g.FQ) == 0;
  }
  // a lane's real columns: pad and clamped columns enter no dot
  auto real = [&](int ch, int k) { return (int)((lane + ch * L) * VEC + k) < g.H; };
  const uint32_t ce = min(w * CH + CH, p.E);
  const uint4 dA = __ldg(reinterpret_cast<const uint4*>(p.desc) + 2 * (size_t)w);
  const uint4 dB = __ldg(reinterpret_cast<const uint4*>(p.desc) + 2 * (size_t)w + 1);
  if (dB.z & 2u) return;
  uint32_t cur = dA.z, curS = dA.w, curT = dB.x;
  const uint32_t e = dA.x, ee = dA.y, r1 = dB.y, carrySlot = dB.w;
  int kind = (dB.z & 1u) ? 0 : ((curT - curS > CH) ? 2 : 1);
  uint32_t segEnd = (kind == 1) ? curT : min(curT, ce);

  const float* hIn = static_cast<const float*>(p.in);
  const uint64_t ldHF = (uint64_t)p.ldIn * VEC, ldGF = (uint64_t)g.ldG * VEC;
  uint32_t cofs[NCH];
#pragma unroll
  for (int ch = 0; ch < NCH; ch++) cofs[ch] = min((uint32_t)(lane + ch * L), p.Q - 1u) * VEC;

  float acc[NCH][VEC], dss[NCH], dsd[NCH];
  float gu[NCH][VEC], hu[NCH][VEC], ssu[NCH], sdu[NCH], lsu[NCH], cu[NCH];
  auto zero = [&]() {
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
      dss[ch] = 0.f; dsd[ch] = 0.f;
#pragma unroll
      for (int k = 0; k < VEC; k++) acc[ch][k] = 0.f;
    }
  };
  auto rowvals = [&]() {
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
      ldv<VEC>(gu[ch], g.dOut + (uint64_t)cur * ldGF + cofs[ch]);
      ldv<VEC>(hu[ch], hIn + (uint64_t)cur * ldHF + cofs[ch]);
      ssu[ch] = g.att[(size_t)cur * g.ldA + hd[ch]];
      sdu[ch] = g.att[(size_t)cur * g.ldA + g.K + hd[ch]];
      lsu[ch] = g.bst[(size_t)cur * g.ldB + hd[ch]];
      cu[ch] = g.bst[(size_t)cur * g.ldB + g.K + hd[ch]];
    }
  };
  auto flush = [&]() {
    float* dst = (kind == 0) ? static_cast<float*>(p.carry) + (size_t)carrySlot * p.ldC * VEC
                             : static_cast<float*>(p.out) + (size_t)cur * p.ldOut * VEC;
    float* dsd_ = (kind == 0) ? static_cast<float*>(p.carry) + (size_t)carrySlot * p.ldC * VEC + g.dsOff
                              : g.ds + (size_t)cur * g.ldDs;
#pragma unroll
    for (int ch = 0; ch < NCH; ch++) {
      if (act[ch]) stv<VEC>(dst + (lane + ch * L) * VEC, acc[ch]);
      if (first[ch]) { dsd_[hd[ch]] = dss[ch]; dsd_[g.K + hd[ch]] = dsd[ch]; }
    }
    zero();
  };
  auto advance = [&]() {
    cur += 1; curS = curT; curT = p.rs[cur + 1];
    const bool heavy = curT - curS > CH;
    segEnd = heavy ? min(curT, ce) : curT;
    kind = heavy ? 2 : 1;
    rowvals();
  };
  zero();
  rowvals();
  const uint32_t eLast = ee - 1u;
#pragma unroll 1
  for (uint32_t base = e; base < ee; base += U) {
    const uint32_t cnt = min((uint32_t)U, ee - base);
    uint32_t srcs[U];
#pragma unroll
    for (int u = 0; u < U; u++) srcs[u] = __ldg(p.col + min(base + (uint32_t)u, eLast));
    float gv[U][NCH][VEC], hv[U][NCH][VEC], ssv[U][NCH], sdv[U][NCH], lsv[U][NCH], cvv[U][NCH];
#pragma unroll
    for (int u = 0; u < U; u++)
#pragma unroll
      for (int ch = 0; ch < NCH; ch++) {
        ldv_nc<VEC>(gv[u][ch], g.dOut + srcs[u] * ldGF + cofs[ch]);
        ldv_nc<VEC>(hv[u][ch], hIn + srcs[u] * ldHF + cofs[ch]);
        const float* at = g.att + (size_t)srcs[u] * g.ldA;
        const float* bt = g.bst + (size_t)srcs[u] * g.ldB;
        ssv[u][ch] = __ldg(at + hd[ch]); sdv[u][ch] = __ldg(at + g.K + hd[ch]);
        lsv[u][ch] = __ldg(bt + hd[ch]); cvv[u][ch] = __ldg(bt + g.K + hd[ch]);
      }
    uint32_t pos = 0;
    for (;;) {
      const uint32_t lim = min(cnt, segEnd - base);
#pragma unroll
      for (int u = 0; u < U; u++) {
        if ((uint32_t)u >= pos && (uint32_t)u < lim) {
          float d1[NCH], d2[NCH];
#pragma unroll
          for (int ch = 0; ch < NCH; ch++) {
            float a = 0.f, b = 0.f;
#pragma unroll
            for (int k = 0; k < VEC; k++) {
              if (real(ch, k)) {
                a = fmaf(gv[u][ch][k], hu[ch][k], a);
                b = fmaf(gu[ch][k], hv[u][ch][k], b);
              }
            }
            d1[ch] = a; d2[ch] = b;
          }
          gat_headsum<L, NCH>(d1, hd, g, wmask);
          gat_headsum<L, NCH>(d2, hd, g, wmask);
#pragma unroll
          for (int ch = 0; ch < NCH; ch++) {
            const float z1 = ssu[ch] + sdv[u][ch];
            const float a1 = gat_alpha(ssu[ch], sdv[u][ch], lsv[u][ch], g.slope);
#pragma unroll
            for (int k = 0; k < VEC; k++) acc[ch][k] = fmaf(a1, gv[u][ch][k], acc[ch][k]);
            dss[ch] = fmaf(a1 * (d1[ch] - cvv[u][ch]), gat_dleaky(z1, g.slope), dss[ch]);
            const float z2 = ssv[u][ch] + sdu[ch];
            const float a2 = gat_alpha(ssv[u][ch], sdu[ch], lsu[ch], g.slope);
            dsd[ch] = fmaf(a2 * (d2[ch] - cu[ch]), gat_dleaky(z2, g.slope), dsd[ch]);
          }
        }
      }
      pos = lim;
      if (pos >= cnt) break;
      flush();
      advance();
    }
  }
  flush();
  while (cur + 1 < r1) { advance(); flush(); }
}

// dh[r][j] += ds_src[r][hd(j)] a_src[j] + ds_dst[r][hd(j)] a_dst[j], and block b's partial of
// da_src[j] = sum_r ds_src[r][hd(j)] h[r][j] (da_dst alike) over its fixed row range, rows in order.
__global__ void __launch_bounds__(GAT_FINISH_THREADS)
k_gat_finish(int64_t rows, int H, int F, int K, const float* __restrict__ h, int64_t ldH, const float* __restrict__ a,
             const float* __restrict__ ds, int64_t ldDs, float* __restrict__ dh, int64_t ldDh, float* __restrict__ part) {
  __shared__ float red[GAT_FINISH_THREADS * 2];
  const int S = GAT_FINISH_THREADS / H;                 // row lanes per block
  const int j = threadIdx.x % H, sub = threadIdx.x / H;
  const int64_t per = (rows + gridDim.x - 1) / gridDim.x;
  const int64_t r0 = min(rows, (int64_t)blockIdx.x * per), r1 = min(rows, r0 + per);
  float s1 = 0.f, s2 = 0.f;
  if (sub < S) {
    const int k = j / F;
    const float as = a[j], ad = a[H + j];
#pragma unroll 4
    for (int64_t r = r0 + sub; r < r1; r += S) {
      const float x = h[r * ldH + j], g1 = ds[r * ldDs + k], g2 = ds[r * ldDs + K + k];
      float* d = dh + r * ldDh + j;
      *d = fmaf(g2, ad, fmaf(g1, as, *d));
      s1 = fmaf(g1, x, s1);
      s2 = fmaf(g2, x, s2);
    }
  }
  red[threadIdx.x] = s1;
  red[GAT_FINISH_THREADS + threadIdx.x] = s2;
  __syncthreads();
  if (sub == 0) {
    float t1 = 0.f, t2 = 0.f;
    for (int q = 0; q < S; q++) { t1 += red[q * H + j]; t2 += red[GAT_FINISH_THREADS + q * H + j]; }
    part[(size_t)blockIdx.x * 2 * H + j] = t1;
    part[(size_t)blockIdx.x * 2 * H + H + j] = t2;
  }
}
__global__ void k_gat_da_reduce(int H, uint32_t nb, const float* __restrict__ part, float* __restrict__ da) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * H) return;
  float s = 0.f;
  for (uint32_t b = 0; b < nb; b++) s += part[(size_t)b * 2 * H + i];
  da[i] = s;
}

enum { GAT_FWD = 0, GAT_BWD = 1 };

template <int OP, int VEC, int L, int NCH, int U, int MINB>
static int launch_gat_cfg(const GatParams& g, cudaStream_t st) {
  constexpr int WPB = SG_THREADS / L;
  constexpr int UU = (OP == GAT_BWD && U > 1) ? U / 2 : U;   // two rows per edge: half the edges in flight
  // the backward also holds its own row's dOut, h and per-node values: fewer CTAs per SM, no spills
  constexpr int MB = (OP == GAT_BWD) ? (NCH == 1 ? 2 : 1) : MINB;
  const SgParams& p = g.p;
  if (p.numChunks) {
    if constexpr (OP == GAT_FWD) sg_gat_kernel<VEC, L, NCH, UU, MINB><<<(p.numChunks + WPB - 1) / WPB, SG_THREADS, 0, st>>>(g);
    else sg_gat_bwd_kernel<VEC, L, NCH, UU, MB><<<(p.numChunks + WPB - 1) / WPB, SG_THREADS, 0, st>>>(g);
    ROC_LAUNCH_CHECK();
  }
  // cut rows are plain sums: SUM's fix-up kernels (the instantiations SUM launches) finish them
  if (p.numHeavy) {
    sg_fixup_kernel<VEC, L, NCH, U><<<(p.numHeavy + WPB - 1) / WPB, SG_THREADS, 0, st>>>(p);
    ROC_LAUNCH_CHECK();
  }
  if (p.numBig) {
    sg_fixup_big_kernel<VEC, L, NCH, U><<<p.numBig, SG_THREADS, 0, st>>>(p);
    ROC_LAUNCH_CHECK();
  }
  return ROC_OK;
}

template <int OP, int VEC>
static int dispatch_gat(const GatParams& g, cudaStream_t st) {
  const uint32_t Q = g.p.Q;
  if (Q <= 4) return launch_gat_cfg<OP, VEC, 4, 1, 4, 4>(g, st);
  if (Q <= 8) return launch_gat_cfg<OP, VEC, 8, 1, 8, 3>(g, st);
  if (Q <= 16) return launch_gat_cfg<OP, VEC, 16, 1, 8, 3>(g, st);
  if (Q <= 32) return launch_gat_cfg<OP, VEC, 32, 1, 8, 3>(g, st);
  if constexpr (VEC == 4) {
    if (Q <= 64) return launch_gat_cfg<OP, VEC, 32, 2, 4, 2>(g, st);
  } else {
    if (Q <= 64) return launch_gat_cfg<OP, VEC, 32, 2, 4, 2>(g, st);
    if (Q <= 128) return launch_gat_cfg<OP, VEC, 32, 4, 2, 2>(g, st);
    if (Q <= 256) return launch_gat_cfg<OP, VEC, 32, 8, 1, 1>(g, st);
  }
  return ROC_ERR_UNSUPPORTED;
}

// the ds rows' fix-up: SUM's per-worker / per-CTA kernels on the 2K-float ds part of the carry slots
static int gat_ds_fixup(const SgParams& p, cudaStream_t st) {
  if (p.Q <= 4) {
    if (p.numHeavy) { sg_fixup_kernel<1, 4, 1, 4><<<(p.numHeavy + 63) / 64, SG_THREADS, 0, st>>>(p); ROC_LAUNCH_CHECK(); }
    if (p.numBig) { sg_fixup_big_kernel<1, 4, 1, 4><<<p.numBig, SG_THREADS, 0, st>>>(p); ROC_LAUNCH_CHECK(); }
  } else if (p.Q <= 8) {
    if (p.numHeavy) { sg_fixup_kernel<1, 8, 1, 8><<<(p.numHeavy + 31) / 32, SG_THREADS, 0, st>>>(p); ROC_LAUNCH_CHECK(); }
    if (p.numBig) { sg_fixup_big_kernel<1, 8, 1, 8><<<p.numBig, SG_THREADS, 0, st>>>(p); ROC_LAUNCH_CHECK(); }
  } else {
    if (p.numHeavy) { sg_fixup_kernel<1, 16, 1, 8><<<(p.numHeavy + 15) / 16, SG_THREADS, 0, st>>>(p); ROC_LAUNCH_CHECK(); }
    if (p.numBig) { sg_fixup_big_kernel<1, 16, 1, 8><<<p.numBig, SG_THREADS, 0, st>>>(p); ROC_LAUNCH_CHECK(); }
  }
  return ROC_OK;
}

static bool gat_shape_ok(int H, int K) {
  if (H <= 0 || H > 256 || !(K == 1 || K == 2 || K == 4 || K == 8)) return false;
  return K == 1 || (H % K == 0 && (H / K) % 4 == 0);
}
// carry slot of the widest GAT pass: the backward's [dh | ds]
static size_t gat_carry_ld(int H, int K) { return ((size_t)H + 3) / 4 * 4 + ((size_t)2 * K + 3) / 4 * 4; }

static void gat_schedule(const roc_sg_plan* pl, SgParams& p) {
  memset(&p, 0, sizeof(p));
  p.rs = pl->rs; p.firstRow = pl->firstRow; p.carryIdx = pl->carryIdx; p.heavyRows = pl->heavyRows; p.bigRows = pl->bigRows;
  p.col = pl->col; p.carry = pl->carry; p.E = pl->E; p.numChunks = pl->numChunks; p.numHeavy = pl->numHeavy;
  p.numBig = pl->numBig; p.epi = 0; p.desc = pl->desc; p.nloc = pl->nloc;
}
// head layout of a launch: Q VEC-columns, FQ per head; hmode as gat_headsum reads it
static void gat_heads(GatParams& g, int H, int K, int VEC, int L) {
  g.H = H; g.K = K; g.F = H / K;
  g.FQ = K == 1 ? (int)g.p.Q : g.F / VEC;
  const bool pow2 = (g.FQ & (g.FQ - 1)) == 0;
  g.hmode = K == 1 ? 0 : (pow2 && g.FQ < L) ? 1 : 2;
}
static int gat_lanes(uint32_t Q) { return Q <= 4 ? 4 : Q <= 8 ? 8 : Q <= 16 ? 16 : 32; }

}  // namespace roc

using namespace roc;

extern "C" int roc_sg_plan_create(roc_vid_t rowLeft, roc_vid_t rowRight, roc_eid_t colLeft,
                                  const roc_eid_t* rowEnd, const roc_vid_t* colSrc,
                                  roc_stream_t stream, roc_sg_plan** planOut) {
  if (!planOut || !rowEnd || rowRight < rowLeft) return ROC_ERR_INVALID;
  if (roc_device_count() <= 0) return ROC_ERR_NO_DEVICE;
  cudaStream_t st = as_stream(stream);
  uint64_t nloc64 = (uint64_t)rowRight - rowLeft + 1;
  if (nloc64 >= 0xFFFFFFF0ull) return ROC_ERR_UNSUPPORTED;
  uint32_t nloc = (uint32_t)nloc64;
  uint64_t lastEnd = 0;
  ROC_CUDA(cudaMemcpyAsync(&lastEnd, rowEnd + (nloc - 1), sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
  ROC_CUDA(cudaStreamSynchronize(st));
  if (lastEnd < colLeft) return ROC_ERR_INVALID;
  uint64_t E64 = lastEnd - colLeft;
  if (E64 >= 0xFFFFFF00ull) return ROC_ERR_UNSUPPORTED;  // local edge offsets are u32
  if (E64 > 0 && !colSrc) return ROC_ERR_INVALID;

  roc_sg_plan* pl = new (std::nothrow) roc_sg_plan();
  if (!pl) return ROC_ERR_NOMEM;
  cudaGetDevice(&pl->device);
  pl->nloc = nloc; pl->E = (uint32_t)E64; pl->col = colSrc;
  pl->numChunks = pl->E / SG_CH + 1;
  uint32_t* flag = nullptr; uint8_t* hflag = nullptr; uint8_t* bflag = nullptr; void* tmp = nullptr; uint32_t* dcount = nullptr;
  int rc = ROC_OK;
  auto fail = [&](int code) { rc = code; };
#define PL_CUDA(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fail((int)e_); goto done; } } while (0)
  {
    PL_CUDA(cudaMalloc(&pl->rs, sizeof(uint32_t) * ((size_t)nloc + 1)));
    PL_CUDA(cudaMalloc(&pl->firstRow, sizeof(uint32_t) * ((size_t)pl->numChunks + 1)));
    PL_CUDA(cudaMalloc(&pl->carryIdx, sizeof(uint32_t) * ((size_t)pl->numChunks + 1)));
    PL_CUDA(cudaMalloc(&flag, sizeof(uint32_t) * ((size_t)pl->numChunks + 1)));
    PL_CUDA(cudaMalloc(&hflag, (size_t)nloc));
    PL_CUDA(cudaMalloc(&pl->heavyRows, sizeof(uint32_t) * (size_t)nloc));
    PL_CUDA(cudaMalloc(&dcount, sizeof(uint32_t)));
    const int T = 256;
    k_build_rs<<<(nloc + T) / T, T, 0, st>>>(nloc, colLeft, rowEnd, pl->rs);
    count_launch();
    k_first_row<<<(pl->numChunks + 1 + T - 1) / T, T, 0, st>>>(nloc, pl->numChunks, pl->rs, pl->firstRow);
    count_launch();
    k_carry_flag<<<(pl->numChunks + 1 + T - 1) / T, T, 0, st>>>(pl->numChunks, pl->rs, pl->firstRow, flag);
    count_launch();
    PL_CUDA(cudaMalloc(&bflag, (size_t)nloc));
    PL_CUDA(cudaMalloc(&pl->bigRows, sizeof(uint32_t) * (size_t)nloc));
    k_heavy_flag<<<(nloc + T - 1) / T, T, 0, st>>>(nloc, pl->rs, hflag, bflag);
    count_launch();
    PL_CUDA(cudaGetLastError());
    size_t tb1 = 0, tb2 = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb1, flag, pl->carryIdx, (int)(pl->numChunks + 1), st);
    thrust::counting_iterator<uint32_t> cnt(0);
    cub::DeviceSelect::Flagged(nullptr, tb2, cnt, hflag, pl->heavyRows, dcount, (int)nloc, st);
    size_t tb = tb1 > tb2 ? tb1 : tb2;
    PL_CUDA(cudaMalloc(&tmp, tb ? tb : 16));
    PL_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb1, flag, pl->carryIdx, (int)(pl->numChunks + 1), st));
    PL_CUDA(cub::DeviceSelect::Flagged(tmp, tb2, cnt, hflag, pl->heavyRows, dcount, (int)nloc, st));
    PL_CUDA(cudaMemcpyAsync(&pl->numHeavy, dcount, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    PL_CUDA(cub::DeviceSelect::Flagged(tmp, tb2, cnt, bflag, pl->bigRows, dcount, (int)nloc, st));
    count_launch(6);
    PL_CUDA(cudaMemcpyAsync(&pl->numCarries, pl->carryIdx + pl->numChunks, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    PL_CUDA(cudaMemcpyAsync(&pl->numBig, dcount, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    PL_CUDA(cudaMalloc(&pl->desc, sizeof(uint32_t) * 8 * (size_t)pl->numChunks));
    k_chunk_desc<<<(pl->numChunks + T - 1) / T, T, 0, st>>>(pl->numChunks, pl->E, pl->rs, pl->firstRow, pl->carryIdx, pl->desc);
    count_launch();
    PL_CUDA(cudaGetLastError());
    PL_CUDA(cudaStreamSynchronize(st));
    if (pl->E) {
      // rows the input matrix must have (1 + largest source id): the extent of the TMA tensor map
      size_t tb3 = 0;
      uint32_t maxSrc = 0;
      cub::DeviceReduce::Max(nullptr, tb3, colSrc, dcount, (int64_t)pl->E, st);
      if (tb3 > tb) { cudaFree(tmp); tmp = nullptr; PL_CUDA(cudaMalloc(&tmp, tb3)); }
      PL_CUDA(cub::DeviceReduce::Max(tmp, tb3, colSrc, dcount, (int64_t)pl->E, st));
      count_launch(2);
      PL_CUDA(cudaMemcpyAsync(&maxSrc, dcount, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
      PL_CUDA(cudaStreamSynchronize(st));
      pl->inRows = (uint64_t)maxSrc + 1;
    }
  }
done:
#undef PL_CUDA
  cudaFree(flag); cudaFree(hflag); cudaFree(bflag); cudaFree(tmp); cudaFree(dcount);
  if (rc != ROC_OK) { roc_sg_plan_destroy(pl); return rc; }
  *planOut = pl;
  return ROC_OK;
}

extern "C" void roc_sg_plan_destroy(roc_sg_plan* pl) {
  if (!pl) return;
  cudaFree(pl->rs); cudaFree(pl->firstRow); cudaFree(pl->carryIdx); cudaFree(pl->heavyRows); cudaFree(pl->bigRows); cudaFree(pl->carry); cudaFree(pl->desc);
  cudaFree(pl->carryArg);
  delete pl;
}

extern "C" int roc_sg_plan_reserve(roc_sg_plan* pl, int maxH) {
  if (!pl || maxH <= 0) return ROC_ERR_INVALID;
  return ensure_carry(pl, ((size_t)maxH + 3) / 4 * 4, nullptr, false);
}

extern "C" int roc_sg_plan_info(const roc_sg_plan* pl, uint64_t* numChunks, uint64_t* numCarries,
                                uint64_t* numHeavyRows) {
  if (!pl) return ROC_ERR_INVALID;
  if (numChunks) *numChunks = pl->numChunks;
  if (numCarries) *numCarries = pl->numCarries;
  if (numHeavyRows) *numHeavyRows = (uint64_t)pl->numHeavy + pl->numBig;
  return ROC_OK;
}

extern "C" int roc_sg_forward_planned(const roc_sg_plan* plc, int H, const float* in, int64_t ldIn,
                                      float* out, int64_t ldOut, int epilogue, roc_stream_t stream) {
  roc_sg_plan* pl = const_cast<roc_sg_plan*>(plc);
  if (!pl || H <= 0 || !in || !out || ldIn < H || ldOut < H) return ROC_ERR_INVALID;
  if ((epilogue & ROC_SG_EPI_MEAN) && (epilogue & ROC_SG_EPI_NORM)) return ROC_ERR_INVALID;
  cudaStream_t st = as_stream(stream);
  const bool vec = (ldIn % 4 == 0) && (ldOut % 4 == 0) && aligned16(in) && aligned16(out);
  // column blocks: the widest kernel covers 256 T-columns (1024 floats vectorised, 256 scalar);
  // the TMA variants take 64 T-columns (a tensor-map box is at most 256 elements wide)
  int variant = pick_variant(vec ? ((uint32_t)H + 3) / 4 : (uint32_t)H, vec);
  if ((variant == 3 || variant == 4 || variant == 5 || variant == 6) && H > 256 && sg_variant_env() < 0) variant = 2;
  const int blockCols = !vec ? 256 : ((variant == 3 || variant == 4 || variant == 5 || variant == 6) ? 256 : 1024);
  {
    int need = H < blockCols ? H : blockCols;
    int rc = ensure_carry(pl, ((size_t)need + 3) / 4 * 4, st, true);
    if (rc != ROC_OK) return rc;
  }
  for (int c0 = 0; c0 < H; c0 += blockCols) {
    int hb = (H - c0 < blockCols) ? H - c0 : blockCols;
    SgParams p;
    p.rs = pl->rs; p.firstRow = pl->firstRow; p.carryIdx = pl->carryIdx; p.heavyRows = pl->heavyRows; p.bigRows = pl->bigRows;
    p.col = pl->col; p.in = in + c0; p.out = out + c0; p.carry = pl->carry;
    p.E = pl->E; p.numChunks = pl->numChunks; p.numHeavy = pl->numHeavy; p.numBig = pl->numBig; p.epi = epilogue;
    p.dense = (pl->nloc > 0 && pl->E / pl->nloc >= (uint32_t)SG_CH) ? 1 : 0;
    p.desc = pl->desc; p.nloc = pl->nloc;
    SgLaunch how;
    how.variant = variant; how.tcfg = sg_tcfg_env(); how.tmap = nullptr;
    CUtensorMap tm;
    memset(&tm, 0, sizeof(tm));     // only the gather4 kernels read it
    how.tmap = &tm;
    int rc;
    if (vec) {
      p.ldIn = (size_t)ldIn / 4; p.ldOut = (size_t)ldOut / 4; p.ldC = pl->carryLd / 4;
      p.Q = ((uint32_t)hb + 3) / 4;
      if (variant == 5 && (!aligned16(pl->col) || p.Q <= 8)) how.variant = 0;   // producer reads col as uint4
      if (variant == 3 || variant == 6 || how.variant == 5) {
        // tensor map of the input: [inRows][Q*4] floats, rows ldIn floats apart; the box is the worker's
        // whole lane span (columns past Q*4 are zero-filled), one row per box — gather4 fetches four
        const uint32_t span = p.Q <= 4 ? 4u : p.Q <= 8 ? 8u : p.Q <= 16 ? 16u : p.Q <= 32 ? 32u : 64u;
        const uint64_t rowBytes = (uint64_t)p.Q * 16u;
        const CUtensorMapL2promotion promo = rowBytes >= 256 ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B
                                            : rowBytes >= 128 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B
                                                              : CU_TENSOR_MAP_L2_PROMOTION_L2_64B;
        if (!tc::make_tmap_32b_2d(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, in + c0, pl->inRows, (uint64_t)p.Q * 4u,
                                  (uint64_t)ldIn, 1u, span * 4u, CU_TENSOR_MAP_SWIZZLE_NONE, promo))
          return ROC_ERR_UNSUPPORTED;
        how.tmap = &tm;
      }
      rc = dispatch<4>(p, how, st);
    } else {
      p.ldIn = (size_t)ldIn; p.ldOut = (size_t)ldOut; p.ldC = pl->carryLd;
      p.Q = (uint32_t)hb;
      rc = dispatch<1>(p, how, st);
    }
    if (rc != ROC_OK) return rc;
  }
  return ROC_OK;
}

// MAX / MIN forward and their backward: the register kernel in column blocks of up to 1024 floats (256 on the
// scalar path)
static int aggr_run(roc_sg_plan* pl, int op, int H, const float* in, int64_t ldIn, const uint32_t* colG, float* out,
                    int64_t ldOut, uint32_t* arg, int64_t ldArg, uint32_t rowLeft, cudaStream_t st) {
  const bool vec = (ldIn % 4 == 0) && (ldOut % 4 == 0) && aligned16(in) && aligned16(out) &&
                   (!arg || ((ldArg % 4 == 0) && aligned16(arg)));
  const int blockCols = vec ? 1024 : 256;
  const size_t need = ((size_t)(H < blockCols ? H : blockCols) + 3) / 4 * 4;
  int rc = ensure_carry(pl, need, st, true);
  if (rc != ROC_OK) return rc;
  if (op != SG_OP_ARGBWD && arg) {
    rc = ensure_carry_arg(pl, need, st, true);
    if (rc != ROC_OK) return rc;
  }
  for (int c0 = 0; c0 < H; c0 += blockCols) {
    const int hb = (H - c0 < blockCols) ? H - c0 : blockCols;
    SgAggrParams a;
    SgParams& p = a.p;
    p.rs = pl->rs; p.firstRow = pl->firstRow; p.carryIdx = pl->carryIdx; p.heavyRows = pl->heavyRows; p.bigRows = pl->bigRows;
    p.col = pl->col; p.in = in + c0; p.out = out + c0; p.carry = pl->carry;
    p.E = pl->E; p.numChunks = pl->numChunks; p.numHeavy = pl->numHeavy; p.numBig = pl->numBig; p.epi = 0;
    p.dense = 0; p.desc = pl->desc; p.nloc = pl->nloc;
    a.colG = colG ? colG : pl->col;
    a.arg = arg ? arg + c0 : nullptr;
    a.carryArg = pl->carryArg;
    a.rowLeft = rowLeft;
    const size_t vw = vec ? 4 : 1;
    p.ldIn = (size_t)ldIn / vw; p.ldOut = (size_t)ldOut / vw; p.ldC = pl->carryLd / vw;
    a.ldArg = (size_t)ldArg / vw; a.ldCA = pl->carryArgLd / vw;
    p.Q = vec ? ((uint32_t)hb + 3) / 4 : (uint32_t)hb;
    if (vec) {
      rc = op == SG_OP_MAX ? dispatch_aggr<SG_OP_MAX, 4>(a, st)
         : op == SG_OP_MIN ? dispatch_aggr<SG_OP_MIN, 4>(a, st) : dispatch_aggr<SG_OP_ARGBWD, 4>(a, st);
    } else {
      rc = op == SG_OP_MAX ? dispatch_aggr<SG_OP_MAX, 1>(a, st)
         : op == SG_OP_MIN ? dispatch_aggr<SG_OP_MIN, 1>(a, st) : dispatch_aggr<SG_OP_ARGBWD, 1>(a, st);
    }
    if (rc != ROC_OK) return rc;
  }
  return ROC_OK;
}

extern "C" int roc_sg_aggr_forward(const roc_sg_plan* plc, int aggr, int H, const float* in, int64_t ldIn,
                                   const roc_vid_t* colGlobal, float* out, int64_t ldOut, uint32_t* arg,
                                   int64_t ldArg, roc_stream_t stream) {
  roc_sg_plan* pl = const_cast<roc_sg_plan*>(plc);
  if (!pl || H <= 0 || !in || !out || ldIn < H || ldOut < H || (arg && ldArg < H)) return ROC_ERR_INVALID;
  if (aggr != ROC_AGGR_MAX && aggr != ROC_AGGR_MIN) return ROC_ERR_INVALID;
  return aggr_run(pl, aggr == ROC_AGGR_MAX ? SG_OP_MAX : SG_OP_MIN, H, in, ldIn, colGlobal, out, ldOut, arg, ldArg, 0u,
                  as_stream(stream));
}

extern "C" int roc_sg_arg_backward(const roc_sg_plan* plc, int H, const float* outGrad, int64_t ldG,
                                   const uint32_t* arg, int64_t ldArg, roc_vid_t rowLeft, float* inGrad,
                                   int64_t ldIn, roc_stream_t stream) {
  roc_sg_plan* pl = const_cast<roc_sg_plan*>(plc);
  if (!pl || H <= 0 || !outGrad || !arg || !inGrad || ldG < H || ldArg < H || ldIn < H) return ROC_ERR_INVALID;
  return aggr_run(pl, SG_OP_ARGBWD, H, outGrad, ldG, nullptr, inGrad, ldIn, const_cast<uint32_t*>(arg), ldArg, rowLeft,
                  as_stream(stream));
}

extern "C" int roc_sg_plan_reserve_arg(roc_sg_plan* pl, int maxH) {
  if (!pl || maxH <= 0) return ROC_ERR_INVALID;
  const size_t ld = ((size_t)maxH + 3) / 4 * 4;
  const int rc = ensure_carry(pl, ld, nullptr, false);
  return rc != ROC_OK ? rc : ensure_carry_arg(pl, ld, nullptr, false);
}

extern "C" int roc_sg_forward(roc_vid_t rowLeft, roc_vid_t rowRight, roc_eid_t colLeft, int H,
                              const roc_eid_t* rowEnd, const roc_vid_t* colSrc, const float* in,
                              float* out, roc_stream_t stream) {
  roc_sg_plan* pl = nullptr;
  int rc = roc_sg_plan_create(rowLeft, rowRight, colLeft, rowEnd, colSrc, stream, &pl);
  if (rc != ROC_OK) return rc;
  rc = roc_sg_forward_planned(pl, H, in, H, out, H, ROC_SG_EPI_NONE, stream);
  cudaError_t e = cudaStreamSynchronize(as_stream(stream));
  roc_sg_plan_destroy(pl);
  if (rc != ROC_OK) return rc;
  return (int)e;
}

extern "C" int roc_sg_backward(roc_vid_t rowLeft, roc_vid_t rowRight, roc_eid_t colLeft, int H,
                               const roc_eid_t* rowEnd, const roc_vid_t* colSrc, const float* outGrad,
                               float* inGrad, roc_stream_t stream) {
  // Forward and backward do exactly the same thing (scattergather_kernel.cu:168-169).
  return roc_sg_forward(rowLeft, rowRight, colLeft, H, rowEnd, colSrc, outGrad, inGrad, stream);
}

// ------------------------------------------------------------------ graph attention: C ABI ---
extern "C" int roc_gat_supported(int H, int heads) { return gat_shape_ok(H, heads) ? ROC_OK : ROC_ERR_UNSUPPORTED; }

extern "C" int roc_gat_plan_reserve(roc_sg_plan* pl, int H, int heads) {
  if (!pl) return ROC_ERR_INVALID;
  if (!gat_shape_ok(H, heads)) return ROC_ERR_UNSUPPORTED;
  return ensure_carry(pl, gat_carry_ld(H, heads), nullptr, false);
}

static int gat_rowdot(int64_t rows, int H, int K, const float* x, int64_t ldX, const float* y1, int64_t ldY1,
                      const float* y2, int64_t ldY2, float* d1, float* d2, int64_t ldD, cudaStream_t st) {
  if (rows <= 0) return ROC_OK;
  const int64_t grid = (rows + GAT_ROWDOT_WARPS - 1) / GAT_ROWDOT_WARPS;
  k_gat_rowdot<<<(unsigned)grid, 32 * GAT_ROWDOT_WARPS, 0, st>>>(rows, H / K, K, x, ldX, y1, ldY1, y2, ldY2, d1, d2, ldD);
  ROC_LAUNCH_CHECK();
  return ROC_OK;
}

extern "C" int roc_gat_scores(int64_t rows, int H, int heads, const float* h, int64_t ldH, const float* attW,
                              float* att, int64_t ldAtt, roc_stream_t stream) {
  if (rows < 0 || !h || !attW || !att || ldH < H || ldAtt < 2 * heads) return ROC_ERR_INVALID;
  if (!gat_shape_ok(H, heads)) return ROC_ERR_UNSUPPORTED;
  return gat_rowdot(rows, H, heads, h, ldH, attW, 0, attW + H, 0, att, att + heads, ldAtt, as_stream(stream));
}

extern "C" int roc_gat_bwd_c(int64_t rows, int H, int heads, const float* outGrad, int64_t ldG, const float* out,
                             int64_t ldOut, float* bst, int64_t ldB, roc_stream_t stream) {
  if (rows < 0 || !outGrad || !out || !bst || ldG < H || ldOut < H || ldB < 2 * heads) return ROC_ERR_INVALID;
  if (!gat_shape_ok(H, heads)) return ROC_ERR_UNSUPPORTED;
  return gat_rowdot(rows, H, heads, outGrad, ldG, out, ldOut, nullptr, 0, bst + heads, nullptr, ldB, as_stream(stream));
}

extern "C" int roc_gat_forward(const roc_sg_plan* plc, int H, int heads, float slope, const float* h, int64_t ldH,
                               const float* att, int64_t ldAtt, float* bst, int64_t ldB, float* out, int64_t ldOut,
                               roc_stream_t stream) {
  roc_sg_plan* pl = const_cast<roc_sg_plan*>(plc);
  if (!pl || !h || !att || !bst || !out || ldH < H || ldOut < H || ldAtt < 2 * heads || ldB < 2 * heads)
    return ROC_ERR_INVALID;
  if (!gat_shape_ok(H, heads)) return ROC_ERR_UNSUPPORTED;
  cudaStream_t st = as_stream(stream);
  int rc = ensure_carry(pl, gat_carry_ld(H, heads), st, true);
  if (rc != ROC_OK) return rc;
  const bool vec = (ldH % 4 == 0) && (ldOut % 4 == 0) && aligned16(h) && aligned16(out);
  GatParams g;
  memset(&g, 0, sizeof(g));
  gat_schedule(pl, g.p);
  g.p.in = h; g.p.out = out;
  g.att = att; g.bst = bst; g.bstOut = bst; g.ldA = (size_t)ldAtt; g.ldB = (size_t)ldB; g.slope = slope;
  g.K = heads;
  // pass 1: lse (carries: raw (max, Z) parts of 2K floats)
  g.p.ldC = pl->carryLd;
  if (pl->numChunks) {
    const unsigned grid = (pl->numChunks + 255) / 256;
    switch (heads) {
      case 1: k_gat_stats<1><<<grid, 256, 0, st>>>(g); break;
      case 2: k_gat_stats<2><<<grid, 256, 0, st>>>(g); break;
      case 4: k_gat_stats<4><<<grid, 256, 0, st>>>(g); break;
      default: k_gat_stats<8><<<grid, 256, 0, st>>>(g); break;
    }
    ROC_LAUNCH_CHECK();
  }
  if (pl->numHeavy + pl->numBig) {
    const unsigned grid = (pl->numHeavy + pl->numBig + 7) / 8;
    switch (heads) {
      case 1: k_gat_stats_fixup<1><<<grid, 256, 0, st>>>(g); break;
      case 2: k_gat_stats_fixup<2><<<grid, 256, 0, st>>>(g); break;
      case 4: k_gat_stats_fixup<4><<<grid, 256, 0, st>>>(g); break;
      default: k_gat_stats_fixup<8><<<grid, 256, 0, st>>>(g); break;
    }
    ROC_LAUNCH_CHECK();
  }
  // pass 2: the weighted aggregate
  const int VEC = vec ? 4 : 1;
  g.p.ldIn = (size_t)ldH / VEC; g.p.ldOut = (size_t)ldOut / VEC; g.p.ldC = pl->carryLd / VEC;
  g.p.Q = ((uint32_t)H + VEC - 1) / VEC;
  gat_heads(g, H, heads, VEC, gat_lanes(g.p.Q));
  return vec ? dispatch_gat<GAT_FWD, 4>(g, st) : dispatch_gat<GAT_FWD, 1>(g, st);
}

extern "C" int roc_gat_backward(const roc_sg_plan* plc, int H, int heads, float slope, const float* h, int64_t ldH,
                                const float* att, int64_t ldAtt, const float* bst, int64_t ldB, const float* outGrad,
                                int64_t ldG, float* inGrad, int64_t ldIn, float* ds, int64_t ldDs,
                                roc_stream_t stream) {
  roc_sg_plan* pl = const_cast<roc_sg_plan*>(plc);
  if (!pl || !h || !att || !bst || !outGrad || !inGrad || !ds || ldH < H || ldG < H || ldIn < H ||
      ldAtt < 2 * heads || ldB < 2 * heads || ldDs < 2 * heads)
    return ROC_ERR_INVALID;
  if (!gat_shape_ok(H, heads)) return ROC_ERR_UNSUPPORTED;
  cudaStream_t st = as_stream(stream);
  int rc = ensure_carry(pl, gat_carry_ld(H, heads), st, true);
  if (rc != ROC_OK) return rc;
  const bool vec = (ldH % 4 == 0) && (ldG % 4 == 0) && (ldIn % 4 == 0) && aligned16(h) && aligned16(outGrad) &&
                   aligned16(inGrad);
  const int VEC = vec ? 4 : 1;
  GatParams g;
  memset(&g, 0, sizeof(g));
  gat_schedule(pl, g.p);
  g.p.in = h; g.p.out = inGrad;
  g.p.ldIn = (size_t)ldH / VEC; g.p.ldOut = (size_t)ldIn / VEC; g.p.ldC = pl->carryLd / VEC;
  g.p.Q = ((uint32_t)H + VEC - 1) / VEC;
  g.att = att; g.bst = bst; g.dOut = outGrad; g.ds = ds;
  g.ldA = (size_t)ldAtt; g.ldB = (size_t)ldB; g.ldG = (size_t)ldG / VEC; g.ldDs = (size_t)ldDs;
  g.dsOff = (uint32_t)(((size_t)H + 3) / 4 * 4);
  g.slope = slope;
  gat_heads(g, H, heads, VEC, gat_lanes(g.p.Q));
  rc = vec ? dispatch_gat<GAT_BWD, 4>(g, st) : dispatch_gat<GAT_BWD, 1>(g, st);
  if (rc != ROC_OK) return rc;
  // the ds rows of cut rows: owner part in ds, carry parts at dsOff of each slot
  SgParams q = g.p;
  q.out = ds; q.ldOut = (size_t)ldDs; q.carry = pl->carry ? pl->carry + g.dsOff : nullptr; q.ldC = pl->carryLd;
  q.Q = 2u * (uint32_t)heads;
  return gat_ds_fixup(q, st);
}

extern "C" size_t roc_gat_finish_workspace_bytes(int H) { return (size_t)GAT_FINISH_BLOCKS * 2 * (size_t)H * sizeof(float); }

extern "C" int roc_gat_bwd_finish(int64_t rows, int H, int heads, const float* h, int64_t ldH, const float* attW,
                                  const float* ds, int64_t ldDs, float* inGrad, int64_t ldIn, float* attGrad,
                                  void* workspace, size_t workspaceBytes, roc_stream_t stream) {
  if (rows < 0 || !h || !attW || !ds || !inGrad || !attGrad || !workspace || ldH < H || ldIn < H || ldDs < 2 * heads)
    return ROC_ERR_INVALID;
  if (!gat_shape_ok(H, heads)) return ROC_ERR_UNSUPPORTED;
  if (workspaceBytes < roc_gat_finish_workspace_bytes(H)) return ROC_ERR_INVALID;
  cudaStream_t st = as_stream(stream);
  float* part = static_cast<float*>(workspace);
  const uint32_t nb = rows > 0 ? (uint32_t)std::min<int64_t>(GAT_FINISH_BLOCKS, (rows + 63) / 64) : 1u;
  k_gat_finish<<<nb, GAT_FINISH_THREADS, 0, st>>>(rows, H, H / heads, heads, h, ldH, attW, ds, ldDs, inGrad, ldIn, part);
  ROC_LAUNCH_CHECK();
  k_gat_da_reduce<<<(2 * H + 255) / 256, 256, 0, st>>>(H, nb, part, attGrad);
  ROC_LAUNCH_CHECK();
  return ROC_OK;
}
