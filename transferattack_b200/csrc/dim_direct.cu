// dim_direct.cu — second-generation DIM kernels (input_transformation/dim.py:42-68): same arithmetic as dim.cu
// (ATen's bilinear expression with the contraction torch's CUDA build uses — bit-identical forward), different
// organisation. ncu on the four-pass kernels of dim.cu showed them instruction-issue-bound (IPC 2.6, > 100 issued
// instructions per output element, 37 % of them integer address arithmetic; profiles/ncu_tim_dim_r1.md). Here:
//
//  * every 1-D tap ((i0, i1, l1) per destination index) and every inverse range is computed ONCE on the host per call
//    (470 entries for 224 -> rnd -> 246 -> 224) and travels as a __grid_constant__ kernel parameter (8.7 / 13 KB): the
//    row loops index it with a warp-uniform counter, so row taps, row offsets and loop control live in UNIFORM registers
//    (ULDC / UIMAD on the uniform datapath) and shared-memory loads use [thread column + uniform row offset] addressing
//    with no per-thread integer arithmetic;
//  * forward = two phases instead of four passes: y1 band (direct 4-tap bilinear from the bulk-TMA-staged source rows)
//    -> shared memory (with one zero row and one zero column appended: that IS the zero padding, no predicates),
//    then out band (direct 4-tap bilinear from y1) -> coalesced global stores. hlerp/vlerp are evaluated exactly as in
//    dim.cu, so the result is bit-identical to it, to the C oracle and to torch's CUDA kernels;
//  * adjoint = the two phases transposed, each as "horizontal gather, then vertical scatter into two rotating register
//    accumulators": a thread owns one column, walks the rows of the incoming gradient once, forms the horizontal
//    inverse-range sum (<= 3 taps, weights in registers) and adds l0*h / l1*h to the two destination rows the current row
//    feeds; a destination row is complete when the (monotone) tap index moves past it and is written exactly once.
//    Deterministic (fixed ascending order), no atomics, no intermediate pass through shared memory except g1.
#include "common.cuh"
#include "dim_direct.cuh"

#include <string.h>

using namespace ta;

namespace {

constexpr int RB = kDimRB;      // destination rows per CTA
constexpr int kThreads = 256;
constexpr int kMaxW = 3;        // inverse-range weights kept in registers (bilinear at DIM's rates needs <= 3)

using Geo = DimGeo;

__device__ __forceinline__ int tap_i0(const TapE& e) { return e.i01 & 0xffff; }
__device__ __forceinline__ int tap_i1(const TapE& e) { return (int)((unsigned)e.i01 >> 16); }

// ATen: hl0*(wl0*p00 + wl1*p01) + hl1*(wl0*p10 + wl1*p11) with the FMA contraction of torch's CUDA build (dim.cu mode 1);
// MODE 0: every product and sum rounded separately; 2-4: the other contraction orders (diagnostic).
template <int MODE>
__device__ __forceinline__ float hl(float w0, float w1, float a, float b) {
  if (MODE == 0) return add_rn(mul_rn(w0, a), mul_rn(w1, b));
  if (MODE == 1 || MODE == 3) return fmaf(w0, a, mul_rn(w1, b));
  return fmaf(w1, b, mul_rn(w0, a));
}
template <int MODE>
__device__ __forceinline__ float vl(float h0, float h1, float t, float b) {
  if (MODE == 0) return add_rn(mul_rn(h0, t), mul_rn(h1, b));
  if (MODE == 1 || MODE == 4) return fmaf(h0, t, mul_rn(h1, b));
  return fmaf(h1, b, mul_rn(h0, t));
}

// ---- forward ---------------------------------------------------------------------------------------------------------
// Row descriptor of one destination row inside a band: BYTE offsets of its two source rows in the staging buffer (the
// zero row for padding) and the vertical weight. Built once per CTA by one thread per row, read back as one broadcast
// LDS.128 per row: the row loops then need 4 integer adds per element and no multiplies, compares or table decoding.
struct __align__(16) RowD { int offa, offb; float l1; int pad; };

__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_f32(uint32_t addr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}

// smem: bufA [a_rows * S] source band (offset 0: the bulk-TMA destination) | bufC [(c_rows + 1) * (rnd + 1)] y1 band,
// row nq and column rnd are zero | descA [c_rows] | descB [RB]
// table source of the forward kernel: the 8.7 KB struct itself as a kernel parameter (default: the forward reads 2 column
// taps per thread and phase, measured 34 us against 38 us with the extra upload launch) or a pointer into the workspace
struct FwdTabParam {
  DimTabF t;
  __device__ __forceinline__ const DimTabF& get() const { return t; }
  __device__ __forceinline__ Geo geo(const Geo& g) const { return g; }
  __device__ __forceinline__ Geo geow(const Geo& g) const { return g; }
  __device__ __forceinline__ bool identity() const { return false; }
};
struct FwdTabPtr {
  const DimTabF* p;
  __device__ __forceinline__ const DimTabF& get() const { return *p; }
  __device__ __forceinline__ Geo geo(const Geo& g) const { return g; }
  __device__ __forceinline__ Geo geow(const Geo& g) const { return g; }
  __device__ __forceinline__ bool identity() const { return false; }
};
// the draw comes from device memory: packs[min(*it, n - 1)] (one captured graph, a new draw per replay)
struct FwdTabDyn {
  const DimPack* packs; const int* it; int n;
  __device__ __forceinline__ const DimPack& pk() const { const int i = *it; return packs[i < n - 1 ? (i < 0 ? 0 : i) : n - 1]; }
  __device__ __forceinline__ const DimTabF& get() const { return pk().tf; }
  __device__ __forceinline__ Geo geo(const Geo&) const { return pk().gf; }
  __device__ __forceinline__ Geo geow(const Geo&) const { return pk().gw; }
  __device__ __forceinline__ bool identity() const { return pk().identity != 0; }
};

template <int MODE, bool TMA_STAGE, class TR, bool REUSE = true>
__global__ void __launch_bounds__(kThreads) dim_fwd_direct_kernel(const float* __restrict__ x, float* __restrict__ out,
                                                                  const __grid_constant__ TR tr, const Geo gm_in) {
  const DimTabF& tab = tr.get();
  const Geo gm = tr.geo(gm_in);
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t s_bar;
  if (tr.identity()) {                                   // the coin said "return x" (dim.py:47-48): this band is a copy
    const int S0 = gm.S, r0 = blockIdx.x * RB, r1 = min(r0 + RB, S0);
    const float* xp0 = x + (int64_t)blockIdx.y * S0 * S0;
    float* op0 = out + (int64_t)blockIdx.y * S0 * S0;
    for (int e = r0 * S0 + threadIdx.x; e < r1 * S0; e += kThreads) op0[e] = __ldg(xp0 + e);
    return;
  }
  const int S = gm.S, rnd = gm.rnd, top = gm.top, left = gm.left;
  const int CP = rnd + 1;
  float* bufA = reinterpret_cast<float*>(smem_raw);
  float* bufC = bufA + (size_t)gm.a_rows * S;
  RowD* descA = reinterpret_cast<RowD*>(smem_raw + (((size_t)gm.a_rows * S + (size_t)(gm.c_rows + 1) * CP) * 4 + 15 & ~(size_t)15));
  RowD* descB = descA + gm.c_rows;

  const int tid = threadIdx.x;
  const int oy0 = blockIdx.x * RB;
  const int oy1 = min(oy0 + RB, S) - 1;                 // inclusive
  const int nb = oy1 - oy0 + 1;
  const float* xp = x + (int64_t)blockIdx.y * S * S;
  float* op = out + (int64_t)blockIdx.y * S * S;

  // rows of y2 (padded), y1 and x this band depends on; the y1 range is empty when the band maps entirely into the padding
  const int pr0 = tap_i0(tab.t2[oy0]), pr1 = tap_i1(tab.t2[oy1]);
  const int q0 = max(pr0 - top, 0), q1 = min(pr1 - top, rnd - 1);
  const bool any = q0 <= q1;
  const int nq = any ? q1 - q0 + 1 : 0;
  int sr0 = 0, nsr = 0;
  if (any) { sr0 = tap_i0(tab.t1[q0]); nsr = tap_i1(tab.t1[q1]) - sr0 + 1; }

  if (TMA_STAGE) {
    if (tid == 0) {
      mbar_init(&s_bar, 1);
      mbar_fence_init();
      if (any) {
        const uint32_t bytes = (uint32_t)(nsr * S * 4);
        mbar_expect_tx(&s_bar, bytes);
        tma_bulk_g2s(bufA, xp + (int64_t)sr0 * S, bytes, &s_bar);
      }
    }
  } else if (any) {
    const float* src = xp + (int64_t)sr0 * S;
    for (int e = tid; e < nsr * S; e += kThreads) bufA[e] = __ldg(src + e);
  }
  // zero row nq and zero column rnd of the y1 band; row descriptors
  for (int e = tid; e < CP; e += kThreads) bufC[nq * CP + e] = 0.0f;
  for (int e = tid; e < nq; e += kThreads) bufC[e * CP + rnd] = 0.0f;
  for (int q = tid; q < nq; q += kThreads) {
    const TapE th = tab.t1[q0 + q];
    descA[q] = RowD{(tap_i0(th) - sr0) * S * 4, (tap_i1(th) - sr0) * S * 4, th.l1, 0};
  }
  for (int r = tid; r < nb; r += kThreads) {
    const TapE th = tab.t2[oy0 + r];
    const int ya = tap_i0(th) - top - q0, yb = tap_i1(th) - top - q0;
    descB[r] = RowD{((ya >= 0 && ya < nq) ? ya : nq) * CP * 4, ((yb >= 0 && yb < nq) ? yb : nq) * CP * 4, th.l1, 0};
  }
  __syncthreads();

  if (any) {
    if (TMA_STAGE) mbar_wait(&s_bar, 0);
    // phase A: y1[q][qx] for q in [q0, q1]; inactive lanes of the last column chunk recompute column rnd-1 (same value,
    // same address) so that the loop stays convergent. Consecutive destination rows share source rows (the tap index moves
    // by the resize scale, 0.9..1.1 rows per row): the horizontal lerp of a source row is kept in a two-entry register cache
    // keyed by the row's byte offset and reused — same value as recomputing it, half the shared-memory loads (REUSE).
    for (int c0 = 0; c0 < rnd; c0 += kThreads) {
      const int col = min(c0 + tid, rnd - 1);
      const TapE tw = tab.t1[col];
      const float wl1 = tw.l1, wl0 = sub_rn(1.0f, wl1);
      const uint32_t ca = smem_u32(bufA + tap_i0(tw)), cb = smem_u32(bufA + tap_i1(tw));
      uint32_t dst = smem_u32(bufC + col);
      const RowD* d = descA;
      int ka = -1, kb = -1;            // byte offsets of the cached rows (descriptor values are >= 0)
      float ha = 0.0f, hb = 0.0f;
#pragma unroll 2
      for (int q = 0; q < nq; ++q, ++d, dst += (uint32_t)CP * 4) {
        const int4 dd = *reinterpret_cast<const int4*>(d);
        const float hl1 = __int_as_float(dd.z), hl0 = sub_rn(1.0f, hl1);
        float t, b;
        if (REUSE && dd.x == kb) t = hb;
        else if (REUSE && dd.x == ka) t = ha;
        else t = hl<MODE>(wl0, wl1, lds_f32(ca + dd.x), lds_f32(cb + dd.x));
        if (REUSE && dd.y == dd.x) b = t;
        else if (REUSE && dd.y == kb) b = hb;
        else b = hl<MODE>(wl0, wl1, lds_f32(ca + dd.y), lds_f32(cb + dd.y));
        ka = dd.x; ha = t; kb = dd.y; hb = b;
        sts_f32(dst, vl<MODE>(hl0, hl1, t, b));
      }
    }
  }
  __syncthreads();
  // phase B: out[oy][ox] for oy in [oy0, oy1] (same two-entry row cache; the zero row of the padding is a row like any other)
  for (int c0 = 0; c0 < S; c0 += kThreads) {
    const int col = min(c0 + tid, S - 1);
    const TapE tw = tab.t2[col];
    const float wl1 = tw.l1, wl0 = sub_rn(1.0f, wl1);
    const int xa = tap_i0(tw) - left, xb = tap_i1(tw) - left;
    const uint32_t ca = smem_u32(bufC + ((xa >= 0 && xa < rnd) ? xa : rnd)), cb = smem_u32(bufC + ((xb >= 0 && xb < rnd) ? xb : rnd));
    float* o = op + (int64_t)oy0 * S + col;
    const RowD* d = descB;
    int ka = -1, kb = -1;
    float ha = 0.0f, hb = 0.0f;
#pragma unroll 2
    for (int r = 0; r < nb; ++r, ++d, o += S) {
      const int4 dd = *reinterpret_cast<const int4*>(d);
      const float hl1 = __int_as_float(dd.z), hl0 = sub_rn(1.0f, hl1);
      float t, b;
      if (REUSE && dd.x == kb) t = hb;
      else if (REUSE && dd.x == ka) t = ha;
      else t = hl<MODE>(wl0, wl1, lds_f32(ca + dd.x), lds_f32(cb + dd.x));
      if (REUSE && dd.y == dd.x) b = t;
      else if (REUSE && dd.y == kb) b = hb;
      else b = hl<MODE>(wl0, wl1, lds_f32(ca + dd.y), lds_f32(cb + dd.y));
      ka = dd.x; ha = t; kb = dd.y; hb = b;
      *o = vl<MODE>(hl0, hl1, t, b);
    }
  }
}

// ---- adjoint ---------------------------------------------------------------------------------------------------------
// weight with which tap `t` (of some destination index) reads source index `i`: l0 if i0 == i, plus l1 if i1 == i
__device__ __forceinline__ float tap_w(const TapE& t, int i) {
  float w = 0.0f;
  if (tap_i0(t) == i) w = sub_rn(1.0f, t.l1);
  if (tap_i1(t) == i) w = add_rn(w, t.l1);
  return w;
}

// One "horizontal gather + vertical scatter" sweep. The thread owns destination column `col` (weights w[], first source
// column lo, count cnt) and walks source rows r = 0..nrows-1 of the staged band at shared address `src` (pitch bytes);
// desc[r] = {i0, i1, l1} of the destination-tap that row r is (decoded once per CTA), feeding destination rows i0 / i1
// with l0 / l1. emit(row, value) is called exactly once for every destination row in [emit_lo, emit_hi], ascending.
struct __align__(16) RowT { int i0, i1; float l1; int pad; };

// Sinks: where completed destination rows go. `at(row)` positions the cursor (once), `put(v)` stores at the cursor,
// `next()` moves it one destination row down — a running address, no per-row multiply.
struct SmemSink {                                    // g1 band in shared memory
  uint32_t base, pitch, cur; int row0;
  __device__ __forceinline__ void at(int row) { cur = base + (uint32_t)(row - row0) * pitch; }
  __device__ __forceinline__ void put(float v) const { sts_f32(cur, v); }
  __device__ __forceinline__ void next() { cur += pitch; }
};
struct GlobalSink {                                  // gin rows in global memory (coalesced across the CTA's columns)
  float* base; int64_t pitch; float* cur;
  __device__ __forceinline__ void at(int row) { cur = base + (int64_t)row * pitch; }
  __device__ __forceinline__ void put(float v) const { *cur = v; }
  __device__ __forceinline__ void next() { cur += pitch; }
};

template <class Sink>
__device__ __forceinline__ void gather_scatter(uint32_t src, uint32_t pitch_bytes, int nrows, const RowT* __restrict__ desc,
                                               const TapE* __restrict__ th_tab, int lo, int cnt, int col,
                                               const float (&w)[kMaxW], int emit_lo, int emit_hi, Sink sink) {
  asm volatile("" : "+r"(pitch_bytes));                  // keep the pitch in a register (else re-read from the constant bank per row)
  const unsigned span = (unsigned)(emit_hi - emit_lo);
  int pcur = nrows > 0 ? desc[0].i0 : emit_hi + 1;
  sink.at(emit_lo);
  int p = emit_lo;
#pragma unroll 1
  for (; p < pcur && p <= emit_hi; ++p) { sink.put(0.0f); sink.next(); }     // rows before the first tap: nothing reads them
  sink.at(pcur);
  float accA = 0.0f, accB = 0.0f;
  uint32_t sp = src + (uint32_t)lo * 4;
  // software pipeline: the taps of row r + 1 and its descriptor are requested before row r is consumed
  float nx[kMaxW];
  int4 ne = make_int4(0, 0, 0, 0);
#pragma unroll
  for (int k = 0; k < kMaxW; ++k) nx[k] = (nrows > 0 && k < cnt) ? lds_f32(sp + 4 * k) : 0.0f;
  if (nrows > 0) ne = *reinterpret_cast<const int4*>(desc);
#pragma unroll 1
  for (int r = 0; r < nrows; ++r) {
    const int4 e = ne;
    float h = 0.0f;
#pragma unroll
    for (int k = 0; k < kMaxW; ++k) if (k < cnt) h = fmaf(w[k], nx[k], h);
#pragma unroll 1
    for (int k = kMaxW; k < cnt; ++k) h = fmaf(tap_w(th_tab[lo + k], col), lds_f32(sp + 4 * k), h);
    sp += pitch_bytes;
    if (r + 1 < nrows) {
#pragma unroll
      for (int k = 0; k < kMaxW; ++k) if (k < cnt) nx[k] = lds_f32(sp + 4 * k);
      ne = *reinterpret_cast<const int4*>(desc + r + 1);
    }
#pragma unroll 1
    while (pcur < e.x) {                             // rows the monotone tap index has moved past are complete
      if ((unsigned)(pcur - emit_lo) <= span) sink.put(accA);
      sink.next();
      accA = accB; accB = 0.0f; ++pcur;
    }
    const float l1 = __int_as_float(e.z), l0 = sub_rn(1.0f, l1);
    accA = fmaf(l0, h, accA);
    if (e.y == e.x) accA = fmaf(l1, h, accA); else accB = fmaf(l1, h, accB);
  }
  if (nrows > 0) {
    if ((unsigned)(pcur - emit_lo) <= span) sink.put(accA);
    sink.next();
    if ((unsigned)(pcur + 1 - emit_lo) <= span) sink.put(accB);
    p = max(pcur + 2, emit_lo);
    sink.at(p);
#pragma unroll 1
    for (; p <= emit_hi; ++p) { sink.put(0.0f); sink.next(); }
  }
}

// smem: bufU [u_rows * S] gout band (offset 0: the bulk-TMA destination) | bufG [g_rows * rnd] g1 band | descU [u_rows] |
// descQ [g_rows]
template <bool TMA_STAGE, bool DYN = false>
__global__ void __launch_bounds__(kThreads) dim_bwd_direct_kernel(const float* __restrict__ gout, float* __restrict__ gin,
                                                                  const DimTabB* __restrict__ tabp, const Geo gm_in,
                                                                  const DimPack* __restrict__ packs, const int* __restrict__ it, int n_packs) {
  const DimPack* pk = nullptr;
  if (DYN) { const int i = *it; pk = packs + (i < n_packs - 1 ? (i < 0 ? 0 : i) : n_packs - 1); }
  const DimTabB& tab = DYN ? pk->tb : *tabp;
  const Geo gm = DYN ? pk->gb : gm_in;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t s_bar;
  if (DYN && pk->identity) {                             // identity forward → identity adjoint
    const int S0 = gm.S, r0 = blockIdx.x * RB, r1 = min(r0 + RB, S0);
    const float* gp0 = gout + (int64_t)blockIdx.y * S0 * S0;
    float* ip0 = gin + (int64_t)blockIdx.y * S0 * S0;
    for (int e = r0 * S0 + threadIdx.x; e < r1 * S0; e += kThreads) ip0[e] = __ldg(gp0 + e);
    return;
  }
  const int S = gm.S, rnd = gm.rnd, top = gm.top, left = gm.left;
  float* bufU = reinterpret_cast<float*>(smem_raw);
  float* bufG = bufU + (size_t)gm.a_rows * S;
  RowT* descU = reinterpret_cast<RowT*>(smem_raw + ((((size_t)gm.a_rows * S + (size_t)gm.c_rows * rnd) * 4 + 15) & ~(size_t)15));
  RowT* descQ = descU + gm.a_rows;

  const int tid = threadIdx.x;
  const int sy0 = blockIdx.x * RB;
  const int sy1 = min(sy0 + RB, S) - 1;
  const float* gp = gout + (int64_t)blockIdx.y * S * S;
  float* ip = gin + (int64_t)blockIdx.y * S * S;

  // y1 rows feeding this band of source rows and the gout rows feeding those: scanned once on the host (band table)
  const short4 bd = tab.band[blockIdx.x];
  const int q0 = bd.x, nq = bd.y, oyA = bd.z, nu = bd.w;
  const bool any = nq > 0;
  const int q1 = q0 + nq - 1;

  if (TMA_STAGE) {
    if (tid == 0) {
      mbar_init(&s_bar, 1);
      mbar_fence_init();
      if (nu > 0) {
        const uint32_t bytes = (uint32_t)(nu * S * 4);
        mbar_expect_tx(&s_bar, bytes);
        tma_bulk_g2s(bufU, gp + (int64_t)oyA * S, bytes, &s_bar);
      }
    }
  } else {
    const float* src = gp + (int64_t)oyA * S;
    for (int e = tid; e < nu * S; e += kThreads) bufU[e] = __ldg(src + e);
  }
  for (int r = tid; r < nu; r += kThreads) { const TapE t = tab.t2[oyA + r]; descU[r] = RowT{tap_i0(t), tap_i1(t), t.l1, 0}; }
  for (int q = tid; q < nq; q += kThreads) { const TapE t = tab.t1[q0 + q]; descQ[q] = RowT{tap_i0(t), tap_i1(t), t.l1, 0}; }
  __syncthreads();
  if (TMA_STAGE && nu > 0) mbar_wait(&s_bar, 0);

  // phase B^T: g1[q][qx], q in [q0, q1]: gather over output columns, scatter over y2 rows (crop = the pad's adjoint)
  for (int col = tid; col < rnd && any; col += kThreads) {
    const int px = col + left;
    const InvE iv = tab.inv2[px];
    float w[kMaxW];
#pragma unroll
    for (int k = 0; k < kMaxW; ++k) w[k] = (k < iv.cnt) ? tap_w(tab.t2[iv.lo + k], px) : 0.0f;
    SmemSink sink{smem_u32(bufG + col), (uint32_t)rnd * 4, 0u, top + q0};
    gather_scatter(smem_u32(bufU), (uint32_t)S * 4, nu, descU, tab.t2, iv.lo, iv.cnt, px, w, q0 + top, q1 + top, sink);
  }
  __syncthreads();
  // phase A^T: gin[sy][sx], sy in [sy0, sy1]: gather over y1 columns, scatter over source rows (coalesced stores)
  for (int col = tid; col < S; col += kThreads) {
    const InvE iv = tab.inv1[col];
    float w[kMaxW];
#pragma unroll
    for (int k = 0; k < kMaxW; ++k) w[k] = (k < iv.cnt) ? tap_w(tab.t1[iv.lo + k], col) : 0.0f;
    GlobalSink sink{ip + col, (int64_t)S, nullptr};
    gather_scatter(smem_u32(bufG), (uint32_t)rnd * 4, nq, descQ, tab.t1, iv.lo, iv.cnt, col, w, sy0, sy1, sink);
  }
}

// ---- adjoint, gather form (default) -------------------------------------------------------------------------------------
// ncu on the gather/scatter form above: 43 M instructions, short_scoreboard 10.6 and mio_throttle 4.4 stall cycles per issue —
// the chain descriptor -> taps -> scatter -> retire is serial per thread. Here every destination element is an independent
// separable gather over its inverse ranges,
//   dst[r][c] = sum_{a < cy(r)} wy(r,a) * ( sum_{b < cx(c)} wx(c,b) * src[ly(r) + a][lx(c) + b] ),
// (cy, cx <= 3 at DIM's resize rates; longer ranges take a tail loop), with the row side (offset of the first source row,
// count, weights) decoded once per CTA into descriptors and the column side in registers: no carried state, no retire logic,
// rows unrollable; each source row is read by ~2 destination rows, i.e. ~2x the shared-memory loads of the scatter form but
// all of them independent. Fixed ascending summation order → deterministic.
struct __align__(16) RowG { int off; int cnt; float w0, w1; };   // + weights a >= 2 in a side array [row][wext]


// one destination value: rows [0, cnt) at byte pitch `pitch` from `addr`, 3 register column taps + tail
__device__ __forceinline__ float hsum3(uint32_t addr, int cx, const float (&wx)[3], const TapE* __restrict__ tab, int lo, int col) {
  float h = 0.0f;
  if (cx > 0) h = fmaf(wx[0], lds_f32(addr), h);
  if (cx > 1) h = fmaf(wx[1], lds_f32(addr + 4), h);
  if (cx > 2) h = fmaf(wx[2], lds_f32(addr + 8), h);
#pragma unroll 1
  for (int b = 3; b < cx; ++b) h = fmaf(tap_w(tab[lo + b], col), lds_f32(addr + 4 * b), h);
  return h;
}

__device__ __forceinline__ float gather_rows(const RowG* __restrict__ d, const float* __restrict__ wext, int wpitch, int row,
                                             uint32_t colbase, uint32_t pitch, int cx, const float (&wx)[3],
                                             const TapE* __restrict__ tab, int lo, int col) {
  const int4 dd = *reinterpret_cast<const int4*>(d + row);
  const int cy = dd.y;
  uint32_t addr = colbase + (uint32_t)dd.x;
  float acc = 0.0f;
  if (cy > 0) acc = fmaf(__int_as_float(dd.z), hsum3(addr, cx, wx, tab, lo, col), acc);
  if (cy > 1) acc = fmaf(__int_as_float(dd.w), hsum3(addr + pitch, cx, wx, tab, lo, col), acc);
  if (cy > 2) {
    addr += 2 * pitch;
#pragma unroll 1
    for (int a = 2; a < cy; ++a, addr += pitch) acc = fmaf(wext[row * wpitch + (a - 2)], hsum3(addr, cx, wx, tab, lo, col), acc);
  }
  return acc;
}

// smem: bufU [u_rows * S] | bufG [g_rows * rnd] | descQ [g_rows] | descS [RB] | wextQ [g_rows * wext] | wextS [RB * wext]
template <bool TMA_STAGE>
__global__ void __launch_bounds__(kThreads) dim_bwd_gather_kernel(const float* __restrict__ gout, float* __restrict__ gin,
                                                                  const DimTabB* __restrict__ tabp, const Geo gm, const int wext) {
  const DimTabB& tab = *tabp;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t s_bar;
  const int S = gm.S, rnd = gm.rnd, top = gm.top, left = gm.left;
  float* bufU = reinterpret_cast<float*>(smem_raw);
  float* bufG = bufU + (size_t)gm.a_rows * S;
  RowG* descQ = reinterpret_cast<RowG*>(smem_raw + ((((size_t)gm.a_rows * S + (size_t)gm.c_rows * rnd) * 4 + 15) & ~(size_t)15));
  RowG* descS = descQ + gm.c_rows;
  float* wextQ = reinterpret_cast<float*>(descS + RB);
  float* wextS = wextQ + (size_t)gm.c_rows * wext;

  const int tid = threadIdx.x;
  const int sy0 = blockIdx.x * RB;
  const int nb = min(sy0 + RB, S) - sy0;
  const float* gp = gout + (int64_t)blockIdx.y * S * S;
  float* ip = gin + (int64_t)blockIdx.y * S * S;
  const short4 bd = tab.band[blockIdx.x];
  const int q0 = bd.x, nq = bd.y, oyA = bd.z, nu = bd.w;

  if (TMA_STAGE) {
    if (tid == 0) {
      mbar_init(&s_bar, 1);
      mbar_fence_init();
      if (nu > 0) {
        const uint32_t bytes = (uint32_t)(nu * S * 4);
        mbar_expect_tx(&s_bar, bytes);
        tma_bulk_g2s(bufU, gp + (int64_t)oyA * S, bytes, &s_bar);
      }
    }
  } else {
    const float* src = gp + (int64_t)oyA * S;
    for (int e = tid; e < nu * S; e += kThreads) bufU[e] = __ldg(src + e);
  }
  // row descriptors: g1 row q gathers gout rows inv2[q0 + q + top]; gin row sy gathers g1 rows inv1[sy]
  for (int q = tid; q < nq; q += kThreads) {
    const int p = q0 + q + top;
    const InvE iv = tab.inv2[p];
    RowG d{(iv.lo - oyA) * S * 4, iv.cnt, 0.0f, 0.0f};
    if (iv.cnt > 0) d.w0 = tap_w(tab.t2[iv.lo], p);
    if (iv.cnt > 1) d.w1 = tap_w(tab.t2[iv.lo + 1], p);
    for (int a = 2; a < iv.cnt; ++a) wextQ[q * wext + (a - 2)] = tap_w(tab.t2[iv.lo + a], p);
    descQ[q] = d;
  }
  for (int r = tid; r < nb; r += kThreads) {
    const int sy = sy0 + r;
    const InvE iv = tab.inv1[sy];
    RowG d{(iv.lo - q0) * rnd * 4, iv.cnt, 0.0f, 0.0f};
    if (iv.cnt > 0) d.w0 = tap_w(tab.t1[iv.lo], sy);
    if (iv.cnt > 1) d.w1 = tap_w(tab.t1[iv.lo + 1], sy);
    for (int a = 2; a < iv.cnt; ++a) wextS[r * wext + (a - 2)] = tap_w(tab.t1[iv.lo + a], sy);
    descS[r] = d;
  }
  __syncthreads();
  if (TMA_STAGE && nu > 0) mbar_wait(&s_bar, 0);

  // phase B^T: g1[q][qx] (crop = the pad's adjoint: y2 column qx + left, y2 row q + top)
  for (int c0 = 0; c0 < rnd && nq > 0; c0 += kThreads) {
    const int col = min(c0 + tid, rnd - 1);                 // inactive lanes duplicate the last column (same value, same address)
    const int px = col + left;
    const InvE iv = tab.inv2[px];
    float wx[3];
#pragma unroll
    for (int b = 0; b < 3; ++b) wx[b] = (b < iv.cnt) ? tap_w(tab.t2[iv.lo + b], px) : 0.0f;
    const uint32_t colbase = smem_u32(bufU + iv.lo);
    uint32_t dst = smem_u32(bufG + col);
#pragma unroll 2
    for (int q = 0; q < nq; ++q, dst += (uint32_t)rnd * 4)
      sts_f32(dst, gather_rows(descQ, wextQ, wext, q, colbase, (uint32_t)S * 4, iv.cnt, wx, tab.t2, iv.lo, px));
  }
  __syncthreads();
  // phase A^T: gin[sy][sx] (coalesced stores)
  for (int c0 = 0; c0 < S; c0 += kThreads) {
    const int col = min(c0 + tid, S - 1);
    const InvE iv = tab.inv1[col];
    float wx[3];
#pragma unroll
    for (int b = 0; b < 3; ++b) wx[b] = (b < iv.cnt) ? tap_w(tab.t1[iv.lo + b], col) : 0.0f;
    const uint32_t colbase = smem_u32(bufG + iv.lo);
    float* o = ip + (int64_t)sy0 * S + col;
#pragma unroll 2
    for (int r = 0; r < nb; ++r, o += S)
      *o = nq > 0 ? gather_rows(descS, wextS, wext, r, colbase, (uint32_t)rnd * 4, iv.cnt, wx, tab.t1, iv.lo, col) : 0.0f;
  }
}

// ---- third generation: separable passes (default) ----------------------------------------------------------------------------
// ncu on the two kernels above (profiles/ncu_tim_dim_r2.md): 73 (forward) and 149 (adjoint) issued instructions per output
// element at 73 % / 86 % issue-slot utilisation — per element they decode a row descriptor, test a two-entry cache, compute
// two shared addresses and walk a pointer, all per THREAD-column. The bilinear expression is separable in VALUE, not only in
// form: hl(row) = wl0*p[row][i0] + wl1*p[row][i1] depends on (row, column) alone, and the result is vl(hl(row a), hl(row b)),
// so the band is processed as four plain passes over shared memory with nothing carried between elements:
//   h1  H[r][c]  = hl(A[r][i0(c)], A[r][i1(c)])          one thread per destination column, rows unrolled (2 LDS + 2 FP + 1 STS)
//   v1  Y1[q][c] = vl(H[ra(q)][c], H[rb(q)][c])           one thread per 4 adjacent columns (2 LDS.128 + 8 FP + 1 STS.128)
//   h2  H[q][o]  = hl(Y1[q][xa(o)], Y1[q][xb(o)])         (zero column rnd / zero row nq of Y1 are the padding)
//   v2  out[oy][o] = vl(H[ya][o], H[yb][o])               128-bit coalesced global stores
// Every value is produced by the same hl / vl expression on the same operands as in the kernels above → bit-identical.
// The adjoint is the four passes transposed, each a gather over the (<= 3 long) inverse range: vT2, hT2, vT1, hT1.
__host__ __device__ __forceinline__ int sep_pitch(int S, int R) { const int m = (R > S ? R : S) + 1; return (m + 3) & ~3; }

// The passes. SC / PC > 0: image side and row pitch are compile-time constants (the hot shape 224 -> 246: 224 / 248), so that the
// unrolled row loops address shared memory as [register + immediate] and carry no integer arithmetic; 0: run-time values.
template <int MODE, int SC, int PC>
__device__ __forceinline__ void sep_hpass(const float* __restrict__ ca, const float* __restrict__ cb, float* __restrict__ dst,
                                          float wl0, float wl1, int rows, int src_pitch_rt, int dst_pitch_rt) {
  const int sp = SC ? SC : src_pitch_rt, dp = PC ? PC : dst_pitch_rt;
  int r = 0;
  for (; r + 4 <= rows; r += 4, ca += 4 * sp, cb += 4 * sp, dst += 4 * dp) {
#pragma unroll
    for (int k = 0; k < 4; ++k) dst[k * dp] = hl<MODE>(wl0, wl1, ca[k * sp], cb[k * sp]);
  }
  for (; r < rows; ++r, ca += sp, cb += sp, dst += dp) dst[0] = hl<MODE>(wl0, wl1, ca[0], cb[0]);
}

template <int MODE>
__device__ __forceinline__ float4 vl4(float hl0, float hl1, const float4& t, const float4& b) {
  return make_float4(vl<MODE>(hl0, hl1, t.x, b.x), vl<MODE>(hl0, hl1, t.y, b.y), vl<MODE>(hl0, hl1, t.z, b.z), vl<MODE>(hl0, hl1, t.w, b.w));
}

// smem: bufA [a_rows * S] (bulk-TMA destination) | bufH [max(a_rows, c_rows + 1) * P] | bufY [(c_rows + 1) * P] | descA | descB
template <int MODE, class TR, int SC, int PC>
__global__ void __launch_bounds__(kThreads) dim_fwd_sep_kernel(const float* __restrict__ x, float* __restrict__ out,
                                                               const __grid_constant__ TR tr, const Geo gm_in) {
  const DimTabF& tab = tr.get();
  const Geo gm = tr.geo(gm_in);
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t s_bar;
  const int tid = threadIdx.x;
  if (tr.identity()) {                                   // the coin said "return x" (dim.py:47-48): this band is a copy
    const int S0 = gm.S, r0 = blockIdx.x * RB, r1 = min(r0 + RB, S0);
    const float4* xp0 = reinterpret_cast<const float4*>(x + (int64_t)blockIdx.y * S0 * S0);
    float4* op0 = reinterpret_cast<float4*>(out + (int64_t)blockIdx.y * S0 * S0);
    for (int e = (r0 * S0 >> 2) + tid; e < (r1 * S0 >> 2); e += kThreads) op0[e] = __ldg(xp0 + e);
    return;
  }
  const int S = SC ? SC : gm.S, rnd = gm.rnd, top = gm.top, left = gm.left;
  const int P = PC ? PC : sep_pitch(S, gm.R);
  const int HR = max(gm.a_rows, gm.c_rows + 1);
  float* bufA = reinterpret_cast<float*>(smem_raw);
  float* bufH = bufA + (size_t)gm.a_rows * S;
  float* bufY = bufH + (size_t)HR * P;
  RowD* descA = reinterpret_cast<RowD*>(bufY + (size_t)(gm.c_rows + 1) * P);
  RowD* descB = descA + gm.c_rows;

  const int oy0 = blockIdx.x * RB;
  const int oy1 = min(oy0 + RB, S) - 1;                 // inclusive
  const int nb = oy1 - oy0 + 1;
  const float* xp = x + (int64_t)blockIdx.y * S * S;
  float* op = out + (int64_t)blockIdx.y * S * S;

  const int pr0 = tap_i0(tab.t2[oy0]), pr1 = tap_i1(tab.t2[oy1]);
  const int q0 = max(pr0 - top, 0), q1 = min(pr1 - top, rnd - 1);
  if (q0 > q1) {                                         // the band maps entirely into the padding: vl(hl(0,0), hl(0,0)) = +0
    float4* o4 = reinterpret_cast<float4*>(op + (int64_t)oy0 * S);
    for (int e = tid; e < (nb * S >> 2); e += kThreads) o4[e] = make_float4(0.f, 0.f, 0.f, 0.f);
    return;
  }
  const int nq = q1 - q0 + 1;
  const int sr0 = tap_i0(tab.t1[q0]);
  const int nsr = tap_i1(tab.t1[q1]) - sr0 + 1;

  if (tid == 0) {
    mbar_init(&s_bar, 1);
    mbar_fence_init();
    const uint32_t bytes = (uint32_t)(nsr * S * 4);
    mbar_expect_tx(&s_bar, bytes);
    tma_bulk_g2s(bufA, xp + (int64_t)sr0 * S, bytes, &s_bar);
  }
  for (int e = tid; e < P; e += kThreads) bufY[nq * P + e] = 0.0f;                     // the zero row (padding rows of y2)
  for (int q = tid; q < nq; q += kThreads) {
    const TapE th = tab.t1[q0 + q];
    descA[q] = RowD{(tap_i0(th) - sr0) * P * 4, (tap_i1(th) - sr0) * P * 4, th.l1, 0};
  }
  for (int r = tid; r < nb; r += kThreads) {
    const TapE th = tab.t2[oy0 + r];
    const int ya = tap_i0(th) - top - q0, yb = tap_i1(th) - top - q0;
    descB[r] = RowD{((ya >= 0 && ya < nq) ? ya : nq) * P * 4, ((yb >= 0 && yb < nq) ? yb : nq) * P * 4, th.l1, 0};
  }
  __syncthreads();
  mbar_wait(&s_bar, 0);

  const int PW1 = (rnd + 1 + 3) & ~3;                   // columns of H / Y1 that are written: [rnd, PW1) = 0 (the zero column)
  // h1
  for (int c = tid; c < PW1; c += kThreads) {
    if (c < rnd) {
      const TapE tw = tab.t1[c];
      const float wl1 = tw.l1, wl0 = sub_rn(1.0f, wl1);
      sep_hpass<MODE, SC, PC>(bufA + tap_i0(tw), bufA + tap_i1(tw), bufH + c, wl0, wl1, nsr, S, P);
    } else {
      for (int r = 0; r < nsr; ++r) bufH[r * P + c] = 0.0f;
    }
  }
  __syncthreads();
  // v1
  {
    const int ncg = PW1 >> 2;
    for (int cg = (tid & 63); cg < ncg; cg += 64) {
      const unsigned char* hb = reinterpret_cast<const unsigned char*>(bufH + 4 * cg);
      float* yo = bufY + 4 * cg + (tid >> 6) * P;
#pragma unroll 2
      for (int q = tid >> 6; q < nq; q += kThreads / 64, yo += (kThreads / 64) * P) {
        const int4 dd = *reinterpret_cast<const int4*>(descA + q);
        const float hl1 = __int_as_float(dd.z), hl0 = sub_rn(1.0f, hl1);
        const float4 t = *reinterpret_cast<const float4*>(hb + dd.x), b = *reinterpret_cast<const float4*>(hb + dd.y);
        *reinterpret_cast<float4*>(yo) = vl4<MODE>(hl0, hl1, t, b);
      }
    }
  }
  __syncthreads();
  // h2 (rows 0 .. nq: the last one is the zero row)
  for (int c = tid; c < S; c += kThreads) {
    const TapE tw = tab.t2[c];
    const float wl1 = tw.l1, wl0 = sub_rn(1.0f, wl1);
    const int xa = tap_i0(tw) - left, xb = tap_i1(tw) - left;
    sep_hpass<MODE, PC, PC>(bufY + ((xa >= 0 && xa < rnd) ? xa : rnd), bufY + ((xb >= 0 && xb < rnd) ? xb : rnd), bufH + c, wl0, wl1,
                            nq + 1, P, P);
  }
  __syncthreads();
  // v2
  {
    const int ncg = S >> 2;
    for (int cg = (tid & 63); cg < ncg; cg += 64) {
      const unsigned char* hb = reinterpret_cast<const unsigned char*>(bufH + 4 * cg);
      float4* o = reinterpret_cast<float4*>(op + (int64_t)(oy0 + (tid >> 6)) * S) + cg;
#pragma unroll 2
      for (int r = tid >> 6; r < nb; r += kThreads / 64, o += (kThreads / 64) * (S >> 2)) {
        const int4 dd = *reinterpret_cast<const int4*>(descB + r);
        const float hl1 = __int_as_float(dd.z), hl0 = sub_rn(1.0f, hl1);
        const float4 t = *reinterpret_cast<const float4*>(hb + dd.x), b = *reinterpret_cast<const float4*>(hb + dd.y);
        *o = vl4<MODE>(hl0, hl1, t, b);
      }
    }
  }
}

// ---- forward, source-driven walk (default) ----------------------------------------------------------------------------------
// Same data movement as dim_fwd_direct_kernel (every horizontal lerp computed once and carried in a register to the destination
// rows that use it; the intermediate written once), but driven by the SOURCE rows: a thread owns one destination column and walks
// the band's source rows in order with static addressing (hot shape: [register + immediate]); hcur = hl(row r) costs 2 LDS + 2
// FP; a per-CTA step table says which destination rows complete at source row r (those whose second tap is r: at most two at
// DIM's resize rates — checked on the host, other geometries keep the kernel above) and with which vertical weight, so a step
// is one broadcast LDS.128, two uniform branches and, per emitted row, 1 FADD + 2 FP + 1 store. No tap decoding, row cache or
// address arithmetic per element. The intermediate band is laid out as rows / columns of the PADDED image y2 (zero-filled first),
// so the second resize addresses it with its taps directly. Same hl / vl expressions on the same operands → bit-identical.
struct __align__(16) StepF { int n; float l1a; float l0a; float l1b; };    // destination rows completing at this source row (0..2)

struct SinkS {                                     // destination rows in shared memory
  uint32_t cur, pitch;
  __device__ __forceinline__ void put(float v) { sts_f32(cur, v); cur += pitch; }
};
struct SinkG {                                     // destination rows in global memory (coalesced across the CTA's columns)
  float* cur; int pitch;
  __device__ __forceinline__ void put(float v) { *cur = v; cur += pitch; }
};

template <int MODE, class Sink>
__device__ __forceinline__ void walk_step(const int4& d, float hprev, float hcur, Sink& sink) {
  if (d.x != 0) {
    sink.put(vl<MODE>(__int_as_float(d.z), __int_as_float(d.y), hprev, hcur));
    if (d.x > 1) {
      const float l1 = __int_as_float(d.w), l0 = sub_rn(1.0f, l1);
      sink.put(vl<MODE>(l0, l1, hprev, hcur));
    }
  }
}

// tail_l1 >= 0: the band ends with the destination row whose two taps are both the LAST source row (ATen clamps i1 at the image
// edge): it completes after everything else, from hcur alone
template <int MODE, int SPC, bool GSRC, class Sink>
__device__ __forceinline__ void walk_rows(const float* __restrict__ pa, const float* __restrict__ pb, float w0, float w1, int rows,
                                          const StepF* __restrict__ prog, int src_pitch_rt, float tail_l1, Sink sink) {
  const int sp = SPC ? SPC : src_pitch_rt;
  float hprev = 0.0f, hcur = 0.0f;
  int r = 0;
  for (; r + 4 <= rows; r += 4, pa += 4 * sp, pb += 4 * sp, prog += 4) {
    float a[4], b[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { a[k] = GSRC ? __ldg(pa + k * sp) : pa[k * sp]; b[k] = GSRC ? __ldg(pb + k * sp) : pb[k * sp]; }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      hprev = hcur; hcur = hl<MODE>(w0, w1, a[k], b[k]);
      walk_step<MODE>(*reinterpret_cast<const int4*>(prog + k), hprev, hcur, sink);
    }
  }
  for (; r < rows; ++r, pa += sp, pb += sp, ++prog) {
    hprev = hcur; hcur = hl<MODE>(w0, w1, GSRC ? __ldg(pa) : pa[0], GSRC ? __ldg(pb) : pb[0]);
    walk_step<MODE>(*reinterpret_cast<const int4*>(prog), hprev, hcur, sink);
  }
  if (tail_l1 >= 0.0f) sink.put(vl<MODE>(sub_rn(1.0f, tail_l1), tail_l1, hcur, hcur));
}

// smem: bufC [c2_rows * P] y2 band | progA [a_rows] | progB [c2_rows];  c2_rows = gm.pad. The source rows are read straight from
// global memory (read-only path; a column's two taps and its neighbours' share L1 lines): staging them cost 33 KB per CTA, i.e.
// 3 instead of 5 resident CTAs per SM at 32-row bands.
// RBW: output rows per CTA (16 or 32); STAGE: the source rows are staged in shared memory by one bulk-TMA copy (else read straight
// from global memory)
template <int MODE, class TR, int SC, int PC, int RBW, bool STAGE>
__global__ void __launch_bounds__(kThreads) dim_fwd_walk_kernel(const float* __restrict__ x, float* __restrict__ out,
                                                                const __grid_constant__ TR tr, const Geo gm_in) {
  const DimTabF& tab = tr.get();
  const Geo gm = tr.geow(gm_in);
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ float s_tail[2];
  __shared__ __align__(8) uint64_t s_bar;
  const int tid = threadIdx.x;
  if (tr.identity()) {                                   // the coin said "return x" (dim.py:47-48): this band is a copy
    const int S0 = gm.S, r0 = blockIdx.x * RBW, r1 = min(r0 + RBW, S0);
    const float4* xp0 = reinterpret_cast<const float4*>(x + (int64_t)blockIdx.y * S0 * S0);
    float4* op0 = reinterpret_cast<float4*>(out + (int64_t)blockIdx.y * S0 * S0);
    for (int e = (r0 * S0 >> 2) + tid; e < (r1 * S0 >> 2); e += kThreads) op0[e] = __ldg(xp0 + e);
    return;
  }
  const int S = SC ? SC : gm.S, rnd = gm.rnd, top = gm.top, left = gm.left;
  const int P = PC ? PC : sep_pitch(S, gm.R);
  const int c2_rows = gm.pad;
  float* bufA = reinterpret_cast<float*>(smem_raw);
  float* bufC = bufA + (STAGE ? (size_t)gm.a_rows * S : 0);
  StepF* progA = reinterpret_cast<StepF*>(bufC + (size_t)c2_rows * P);
  StepF* progB = progA + gm.a_rows;

  const int oy0 = blockIdx.x * RBW;
  const int oy1 = min(oy0 + RBW, S) - 1;                 // inclusive
  const int nb = oy1 - oy0 + 1;
  const float* xp = x + (int64_t)blockIdx.y * S * S;
  float* op = out + (int64_t)blockIdx.y * S * S;

  const int pr0 = tap_i0(tab.t2[oy0]), pr1 = tap_i1(tab.t2[oy1]);
  const int nC = pr1 - pr0 + 1;                         // rows of y2 this band reads
  const int q0 = max(pr0 - top, 0), q1 = min(pr1 - top, rnd - 1);
  if (q0 > q1) {                                         // the band maps entirely into the padding: vl(hl(0,0), hl(0,0)) = +0
    float4* o4 = reinterpret_cast<float4*>(op + (int64_t)oy0 * S);
    for (int e = tid; e < (nb * S >> 2); e += kThreads) o4[e] = make_float4(0.f, 0.f, 0.f, 0.f);
    return;
  }
  const int nq = q1 - q0 + 1;
  const int sr0 = tap_i0(tab.t1[q0]);
  const int nsr = tap_i1(tab.t1[q1]) - sr0 + 1;

  if (STAGE && tid == 0) {
    mbar_init(&s_bar, 1);
    mbar_fence_init();
    const uint32_t bytes = (uint32_t)(nsr * S * 4);
    mbar_expect_tx(&s_bar, bytes);
    tma_bulk_g2s(bufA, xp + (int64_t)sr0 * S, bytes, &s_bar);
  }
  {                                                      // zero the y2 band (the padding) and the step tables
    float4* c4 = reinterpret_cast<float4*>(bufC);
    for (int e = tid; e < (nC * P >> 2); e += kThreads) c4[e] = make_float4(0.f, 0.f, 0.f, 0.f);
    int4* p4 = reinterpret_cast<int4*>(progA);
    for (int e = tid; e < gm.a_rows + c2_rows; e += kThreads) p4[e] = make_int4(0, 0, 0, 0);
    if (tid < 2) s_tail[tid] = -1.0f;
  }
  __syncthreads();
  for (int q = tid; q < nq; q += kThreads) {             // y1 row q0 + q completes at source row i1
    const TapE th = tab.t1[q0 + q];
    const int ra = tap_i0(th) - sr0, rb = tap_i1(th) - sr0;
    if (ra == rb) { s_tail[0] = th.l1; continue; }       // clamped at the image edge: the band's last row (host-checked: at most one)
    const int rank = (q > 0 && tap_i1(tab.t1[q0 + q - 1]) - sr0 == rb) ? 1 : 0;
    if (rank) progA[rb].l1b = th.l1; else { progA[rb].l1a = th.l1; progA[rb].l0a = sub_rn(1.0f, th.l1); }
    atomicAdd(&progA[rb].n, 1);
  }
  for (int r = tid; r < nb; r += kThreads) {             // output row oy0 + r completes at y2 row i1
    const TapE th = tab.t2[oy0 + r];
    const int ya = tap_i0(th) - pr0, yb = tap_i1(th) - pr0;
    if (ya == yb) { s_tail[1] = th.l1; continue; }
    const int rank = (r > 0 && tap_i1(tab.t2[oy0 + r - 1]) - pr0 == yb) ? 1 : 0;
    if (rank) progB[yb].l1b = th.l1; else { progB[yb].l1a = th.l1; progB[yb].l0a = sub_rn(1.0f, th.l1); }
    atomicAdd(&progB[yb].n, 1);
  }
  __syncthreads();
  if (STAGE) mbar_wait(&s_bar, 0);

  // phase A: y1 rows q0 .. q1 into rows (q + top - pr0), columns (left + c) of the y2 band
  for (int c = tid; c < rnd; c += kThreads) {
    const TapE tw = tab.t1[c];
    const float wl1 = tw.l1, wl0 = sub_rn(1.0f, wl1);
    SinkS sink{smem_u32(bufC + (size_t)(q0 + top - pr0) * P + left + c), (uint32_t)P * 4};
    if (STAGE) {
      walk_rows<MODE, SC, false>(bufA + tap_i0(tw), bufA + tap_i1(tw), wl0, wl1, nsr, progA, S, s_tail[0], sink);
    } else {
      const float* src = xp + (int64_t)sr0 * S;
      walk_rows<MODE, SC, true>(src + tap_i0(tw), src + tap_i1(tw), wl0, wl1, nsr, progA, S, s_tail[0], sink);
    }
  }
  __syncthreads();
  // phase B: output rows oy0 .. oy1 straight to global memory
  for (int c = tid; c < S; c += kThreads) {
    const TapE tw = tab.t2[c];
    const float wl1 = tw.l1, wl0 = sub_rn(1.0f, wl1);
    SinkG sink{op + (int64_t)oy0 * S + c, S};
    walk_rows<MODE, PC, false>(bufC + tap_i0(tw), bufC + tap_i1(tw), wl0, wl1, nC, progB, P, s_tail[1], sink);
  }
}

// 4 adjacent columns of one destination row of a transposed vertical pass: sum over the row's inverse range
__device__ __forceinline__ float4 fma4(float w, const float4& v, const float4& a) {
  return make_float4(fmaf(w, v.x, a.x), fmaf(w, v.y, a.y), fmaf(w, v.z, a.z), fmaf(w, v.w, a.w));
}
__device__ __forceinline__ float4 vgather4(const RowG* __restrict__ d, const float* __restrict__ wext, int wpitch, int row,
                                           const unsigned char* __restrict__ colbase, int pitch_bytes) {
  const int4 dd = *reinterpret_cast<const int4*>(d + row);
  const int cy = dd.y;
  const unsigned char* addr = colbase + dd.x;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (cy > 0) acc = fma4(__int_as_float(dd.z), *reinterpret_cast<const float4*>(addr), acc);
  if (cy > 1) acc = fma4(__int_as_float(dd.w), *reinterpret_cast<const float4*>(addr + pitch_bytes), acc);
  if (cy > 2) {
    addr += 2 * pitch_bytes;
#pragma unroll 1
    for (int a = 2; a < cy; ++a, addr += pitch_bytes) acc = fma4(wext[row * wpitch + (a - 2)], *reinterpret_cast<const float4*>(addr), acc);
  }
  return acc;
}
// one destination column of a transposed horizontal pass, all rows: <= 3 register weights + tail
template <int SPC, int DPC>
__device__ __forceinline__ void sep_htpass(const float* __restrict__ src, float* __restrict__ dst, int rows, int cx, const float (&wx)[3],
                                           const TapE* __restrict__ tab, int lo, int col, int src_pitch_rt, int dst_pitch_rt) {
  const int sp = SPC ? SPC : src_pitch_rt;
  const int64_t dp = DPC ? DPC : dst_pitch_rt;
  if (cx <= 3) {                                         // weights beyond the range are 0 and the extra columns exist (finite or not read)
    int r = 0;
    for (; r + 4 <= rows; r += 4, src += 4 * sp, dst += 4 * dp) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float h = 0.0f;
        if (cx > 0) h = fmaf(wx[0], src[k * sp], h);
        if (cx > 1) h = fmaf(wx[1], src[k * sp + 1], h);
        if (cx > 2) h = fmaf(wx[2], src[k * sp + 2], h);
        dst[k * dp] = h;
      }
    }
    for (; r < rows; ++r, src += sp, dst += dp) {
      float h = 0.0f;
      if (cx > 0) h = fmaf(wx[0], src[0], h);
      if (cx > 1) h = fmaf(wx[1], src[1], h);
      if (cx > 2) h = fmaf(wx[2], src[2], h);
      dst[0] = h;
    }
  } else {
    for (int r = 0; r < rows; ++r, src += sp, dst += dp) {
      float h = fmaf(wx[2], src[2], fmaf(wx[1], src[1], fmaf(wx[0], src[0], 0.0f)));
#pragma unroll 1
      for (int b = 3; b < cx; ++b) h = fmaf(tap_w(tab[lo + b], col), src[b], h);
      dst[0] = h;
    }
  }
}

__host__ __device__ __forceinline__ size_t bwd_sep_first(int S, int P, int u_rows) {     // floats: gout band, later W[RB][P]
  const size_t a = (size_t)u_rows * S, b = (size_t)RB * P;
  return a > b ? a : b;
}

// smem: bufU [max(u_rows * S, RB * P)] (bulk-TMA destination; reused as W) | bufV [g_rows * S] | bufG [g_rows * P] |
//       descQ [g_rows] | descS [RB] | wextQ [g_rows * wext] | wextS [RB * wext];   P = sep_pitch(S, R), wext = gm.pad
template <bool DYN, int SC, int PC>
__global__ void __launch_bounds__(kThreads) dim_bwd_sep_kernel(const float* __restrict__ gout, float* __restrict__ gin,
                                                               const DimTabB* __restrict__ tabp, const Geo gm_in,
                                                               const DimPack* __restrict__ packs, const int* __restrict__ it, int n_packs) {
  const DimPack* pk = nullptr;
  if (DYN) { const int i = *it; pk = packs + (i < n_packs - 1 ? (i < 0 ? 0 : i) : n_packs - 1); }
  const DimTabB& tab = DYN ? pk->tb : *tabp;
  const Geo gm = DYN ? pk->gb : gm_in;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t s_bar;
  const int tid = threadIdx.x;
  if (DYN && pk->identity) {                             // identity forward → identity adjoint
    const int S0 = gm.S, r0 = blockIdx.x * RB, r1 = min(r0 + RB, S0);
    const float4* gp0 = reinterpret_cast<const float4*>(gout + (int64_t)blockIdx.y * S0 * S0);
    float4* ip0 = reinterpret_cast<float4*>(gin + (int64_t)blockIdx.y * S0 * S0);
    for (int e = (r0 * S0 >> 2) + tid; e < (r1 * S0 >> 2); e += kThreads) ip0[e] = __ldg(gp0 + e);
    return;
  }
  const int S = SC ? SC : gm.S, rnd = gm.rnd, top = gm.top, left = gm.left, wext = gm.pad;
  const int P = PC ? PC : sep_pitch(S, gm.R);
  float* bufU = reinterpret_cast<float*>(smem_raw);
  float* bufV = bufU + bwd_sep_first(S, P, gm.a_rows);
  float* bufG = bufV + (size_t)gm.c_rows * S;
  RowG* descQ = reinterpret_cast<RowG*>(bufG + (size_t)gm.c_rows * P);
  RowG* descS = descQ + gm.c_rows;
  float* wextQ = reinterpret_cast<float*>(descS + RB);
  float* wextS = wextQ + (size_t)gm.c_rows * wext;

  const int sy0 = blockIdx.x * RB;
  const int nb = min(sy0 + RB, S) - sy0;
  const float* gp = gout + (int64_t)blockIdx.y * S * S;
  float* ip = gin + (int64_t)blockIdx.y * S * S;
  const short4 bd = tab.band[blockIdx.x];
  const int q0 = bd.x, nq = bd.y, oyA = bd.z, nu = bd.w;
  if (nq == 0) {                                         // no y1 row reads this band of source rows
    float4* o4 = reinterpret_cast<float4*>(ip + (int64_t)sy0 * S);
    for (int e = tid; e < (nb * S >> 2); e += kThreads) o4[e] = make_float4(0.f, 0.f, 0.f, 0.f);
    return;
  }
  if (tid == 0) {
    mbar_init(&s_bar, 1);
    mbar_fence_init();
    if (nu > 0) {
      const uint32_t bytes = (uint32_t)(nu * S * 4);
      mbar_expect_tx(&s_bar, bytes);
      tma_bulk_g2s(bufU, gp + (int64_t)oyA * S, bytes, &s_bar);
    }
  }
  // row descriptors: V row q gathers gout rows inv2[q0 + q + top]; W row r gathers g1 rows inv1[sy0 + r]
  for (int q = tid; q < nq; q += kThreads) {
    const int p = q0 + q + top;
    const InvE iv = tab.inv2[p];
    RowG d{(iv.lo - oyA) * S * 4, iv.cnt, 0.0f, 0.0f};
    if (iv.cnt > 0) d.w0 = tap_w(tab.t2[iv.lo], p);
    if (iv.cnt > 1) d.w1 = tap_w(tab.t2[iv.lo + 1], p);
    for (int a = 2; a < iv.cnt; ++a) wextQ[q * wext + (a - 2)] = tap_w(tab.t2[iv.lo + a], p);
    descQ[q] = d;
  }
  for (int r = tid; r < nb; r += kThreads) {
    const int sy = sy0 + r;
    const InvE iv = tab.inv1[sy];
    RowG d{(iv.lo - q0) * P * 4, iv.cnt, 0.0f, 0.0f};
    if (iv.cnt > 0) d.w0 = tap_w(tab.t1[iv.lo], sy);
    if (iv.cnt > 1) d.w1 = tap_w(tab.t1[iv.lo + 1], sy);
    for (int a = 2; a < iv.cnt; ++a) wextS[r * wext + (a - 2)] = tap_w(tab.t1[iv.lo + a], sy);
    descS[r] = d;
  }
  __syncthreads();
  if (nu > 0) mbar_wait(&s_bar, 0);

  // vT2: V[q][ox] = sum over the output rows that read y2 row q0 + q + top
  {
    const int ncg = S >> 2;
    for (int cg = (tid & 63); cg < ncg; cg += 64) {
      const unsigned char* ub = reinterpret_cast<const unsigned char*>(bufU + 4 * cg);
      float* vo = bufV + 4 * cg + (tid >> 6) * S;
#pragma unroll 2
      for (int q = tid >> 6; q < nq; q += kThreads / 64, vo += (kThreads / 64) * S)
        *reinterpret_cast<float4*>(vo) = vgather4(descQ, wextQ, wext, q, ub, S * 4);
    }
  }
  __syncthreads();
  // hT2: g1[q][qx] = sum over the output columns that read y2 column qx + left (crop = the pad's adjoint)
  for (int c = tid; c < rnd; c += kThreads) {
    const int px = c + left;
    const InvE iv = tab.inv2[px];
    float wx[3];
#pragma unroll
    for (int b = 0; b < 3; ++b) wx[b] = (b < iv.cnt) ? tap_w(tab.t2[iv.lo + b], px) : 0.0f;
    sep_htpass<SC, PC>(bufV + iv.lo, bufG + c, nq, iv.cnt, wx, tab.t2, iv.lo, px, S, P);
  }
  __syncthreads();
  // vT1: W[r][qx] = sum over the y1 rows that read source row sy0 + r   (W reuses the gout band's storage)
  float* bufW = bufU;
  {
    const int ncg = (rnd + 3) >> 2;
    for (int cg = (tid & 63); cg < ncg; cg += 64) {
      const unsigned char* gb = reinterpret_cast<const unsigned char*>(bufG + 4 * cg);
      float* wo = bufW + 4 * cg + (tid >> 6) * P;
#pragma unroll 2
      for (int r = tid >> 6; r < nb; r += kThreads / 64, wo += (kThreads / 64) * P)
        *reinterpret_cast<float4*>(wo) = vgather4(descS, wextS, wext, r, gb, P * 4);
    }
  }
  __syncthreads();
  // hT1: gin[sy][sx] = sum over the y1 columns that read source column sx (coalesced stores)
  for (int c = tid; c < S; c += kThreads) {
    const InvE iv = tab.inv1[c];
    float wx[3];
#pragma unroll
    for (int b = 0; b < 3; ++b) wx[b] = (b < iv.cnt) ? tap_w(tab.t1[iv.lo + b], c) : 0.0f;
    sep_htpass<PC, SC>(bufW + iv.lo, ip + (int64_t)sy0 * S + c, nb, iv.cnt, wx, tab.t1, iv.lo, c, P, S);
  }
}

// ---- table upload -------------------------------------------------------------------------------------------------------
// The tables are built on the host per call and must reach GLOBAL memory in stream order without a host-side staging buffer
// whose lifetime the library would have to manage: they travel as the parameter of this one-wave copy kernel (128-bit
// constant-bank reads, one per thread) into the caller's workspace. (Reading 9-13 KB of tables straight from the parameter
// space inside the main kernels was measured slow: indexed constant loads of 32 different addresses per warp serialise and
// evict the small constant cache, so that even uniform parameter reads miss — ncu: LDC consumers top the stall samples.)
template <class T>
__global__ void __launch_bounds__(256) upload_tab_kernel(const __grid_constant__ T tab, T* __restrict__ dst) {
  static_assert(sizeof(T) % 16 == 0, "table size must be a multiple of 16 bytes");
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (int)(sizeof(T) / 16)) reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(&tab)[i];
}
template <class T>
int upload_tab(const T& tab, void* ws, cudaStream_t s) {
  upload_tab_kernel<T><<<(unsigned)((sizeof(T) / 16 + 255) / 256), 256, 0, s>>>(tab, reinterpret_cast<T*>(ws));
  count_launch();
  return check_launch("ta_dim[table upload]");
}

// ---- host: tables ------------------------------------------------------------------------------------------------------
void host_taps(int in, int out, TapE* t) {           // ATen area_pixel_compute_source_index, align_corners=False
  const float scale = (float)in / (float)out;
  for (int d = 0; d < out; ++d) {
    float src = fmaf(scale, (float)d + 0.5f, -0.5f);
    if (src < 0.0f) src = 0.0f;
    const int i0 = (int)src;
    const int i1 = i0 + ((i0 < in - 1) ? 1 : 0);
    t[d].l1 = src - (float)i0;
    t[d].i01 = i0 | (i1 << 16);
  }
}
void host_inverse(const TapE* t, int out, int in, InvE* inv) {
  for (int i = 0; i < in; ++i) { inv[i].lo = 0; inv[i].cnt = 0; }
  for (int d = 0; d < out; ++d) {
    const int idx[2] = {t[d].i01 & 0xffff, (int)((unsigned)t[d].i01 >> 16)};
    for (int k = 0; k < 2; ++k) {
      InvE& e = inv[idx[k]];
      if (e.cnt == 0) { e.lo = (short)d; e.cnt = 1; }
      else e.cnt = (short)(d - e.lo + 1);             // d ascends: [lo, d] (taps are monotone: everything inside touches it)
    }
  }
}
inline int h_i0(const TapE& e) { return e.i01 & 0xffff; }
inline int h_i1(const TapE& e) { return (int)((unsigned)e.i01 >> 16); }

}  // namespace

namespace ta {

bool dim_direct_ok(int S, int rnd, int R) { return S <= kDimMaxS && R <= kDimMaxR && rnd <= kDimMaxR && S >= 1; }

size_t dim_direct_ws_bytes() { return sizeof(DimTabB) > sizeof(DimTabF) ? sizeof(DimTabB) : sizeof(DimTabF); }

// exact band maxima of one draw (rows of y1 / of the source a forward band needs; rows of g1 / of gout an adjoint band needs)
// band maxima of the walk (RBW output rows per CTA): source rows and y2 rows one band reads; false when some source row
// completes more than two destination rows (then the source-driven walk does not apply)
static bool walk_geo(const DimTabF& tab, int S, int rnd, int top, int RBW, int* a_rows_, int* c2_rows_) {
  int c2 = 1, a_rows = 1;
  for (int oy0 = 0; oy0 < S; oy0 += RBW) {
    const int oy1 = (oy0 + RBW < S ? oy0 + RBW : S) - 1;
    const int pr0 = h_i0(tab.t2[oy0]), pr1 = h_i1(tab.t2[oy1]);
    if (pr1 - pr0 + 1 > c2) c2 = pr1 - pr0 + 1;
    const int q0 = pr0 - top > 0 ? pr0 - top : 0, q1 = pr1 - top < rnd - 1 ? pr1 - top : rnd - 1;
    if (q0 > q1) continue;
    const int nsr = h_i1(tab.t1[q1]) - h_i0(tab.t1[q0]) + 1;
    if (nsr > a_rows) a_rows = nsr;
  }
  for (int stage = 0; stage < 2; ++stage) {
    const TapE* t = stage ? tab.t2 : tab.t1;
    const int n = stage ? S : rnd;
    int run = 1;
    for (int d = 1; d < n; ++d) {
      run = (h_i1(t[d]) == h_i1(t[d - 1])) ? run + 1 : 1;
      if (run > 2) return false;
    }
    for (int d = 0; d + 1 < n; ++d)
      if (h_i0(t[d]) == h_i1(t[d])) return false;           // a clamped tap (i0 == i1) anywhere but at the last destination index
  }
  *a_rows_ = a_rows; *c2_rows_ = c2;
  return true;
}
constexpr int kWalkRB = 16;          // defaults of the walk (the draw packs carry the geometry of THIS configuration)
constexpr bool kWalkStage = true;
static size_t fwd_walk_smem(int S, int R, int a_rows, int c2_rows, bool stage) {
  return sizeof(float) * ((stage ? (size_t)a_rows * S : 0) + (size_t)c2_rows * sep_pitch(S, R)) + 16 * (size_t)(a_rows + c2_rows);
}
static bool walk_enabled(int S, bool tma) { return tma && S % 4 == 0 && tune_get("dim.impl", 2) == 4; }

static void fwd_tables(int S, int rnd, int R, int top, DimTabF& tab, int* a_rows_, int* c_rows_) {
  host_taps(R, S, tab.t2);
  host_taps(S, rnd, tab.t1);
  int c_rows = 0, a_rows = 1;
  for (int oy0 = 0; oy0 < S; oy0 += RB) {
    const int oy1 = (oy0 + RB < S ? oy0 + RB : S) - 1;
    const int pr0 = h_i0(tab.t2[oy0]), pr1 = h_i1(tab.t2[oy1]);
    const int q0 = pr0 - top > 0 ? pr0 - top : 0, q1 = pr1 - top < rnd - 1 ? pr1 - top : rnd - 1;
    if (q0 > q1) continue;
    if (q1 - q0 + 1 > c_rows) c_rows = q1 - q0 + 1;
    const int nsr = h_i1(tab.t1[q1]) - h_i0(tab.t1[q0]) + 1;
    if (nsr > a_rows) a_rows = nsr;
  }
  *a_rows_ = a_rows; *c_rows_ = c_rows;
}
static void bwd_tables(int S, int rnd, int R, int top, DimTabB& tab, int* u_rows_, int* g_rows_) {
  host_taps(R, S, tab.t2);
  host_taps(S, rnd, tab.t1);
  host_inverse(tab.t2, S, R, tab.inv2);
  host_inverse(tab.t1, rnd, S, tab.inv1);
  int g_rows = 1, u_rows = 1;
  for (int sy0 = 0; sy0 < S; sy0 += RB) {
    const int sy1 = (sy0 + RB < S ? sy0 + RB : S) - 1;
    tab.band[sy0 / RB] = make_short4(0, 0, 0, 0);
    int q0 = 0x7fffffff, q1 = -1;
    for (int sy = sy0; sy <= sy1; ++sy)
      if (tab.inv1[sy].cnt > 0) {
        if (tab.inv1[sy].lo < q0) q0 = tab.inv1[sy].lo;
        if (tab.inv1[sy].lo + tab.inv1[sy].cnt - 1 > q1) q1 = tab.inv1[sy].lo + tab.inv1[sy].cnt - 1;
      }
    if (q0 > q1) continue;
    if (q1 - q0 + 1 > g_rows) g_rows = q1 - q0 + 1;
    int a = 0x7fffffff, b = -1;
    for (int q = q0; q <= q1; ++q) {
      const InvE& iv = tab.inv2[q + top];
      if (iv.cnt > 0) { if (iv.lo < a) a = iv.lo; if (iv.lo + iv.cnt - 1 > b) b = iv.lo + iv.cnt - 1; }
    }
    if (a <= b && b - a + 1 > u_rows) u_rows = b - a + 1;
    tab.band[sy0 / RB] = make_short4((short)q0, (short)(q1 - q0 + 1), (short)(a <= b ? a : 0), (short)(a <= b ? b - a + 1 : 0));
  }
  *u_rows_ = u_rows; *g_rows_ = g_rows;
}
static size_t fwd_smem(int S, int rnd, int a_rows, int c_rows) {
  return ((sizeof(float) * ((size_t)a_rows * S + (size_t)(c_rows + 1) * (rnd + 1)) + 15) & ~(size_t)15) + 16 * (size_t)(c_rows + RB);
}
static size_t bwd_smem(int S, int rnd, int u_rows, int g_rows) {
  return ((sizeof(float) * ((size_t)u_rows * S + (size_t)g_rows * rnd) + 15) & ~(size_t)15) + 16 * (size_t)(u_rows + g_rows);
}
// the separable kernels (dim_fwd_sep_kernel / dim_bwd_sep_kernel): S % 4 == 0
// dim.impl 2 (default): forward = second-generation register-carried kernel (34 us at B = 64; the separable passes need 40 us, the
// source-driven walk 32-34 us), adjoint = separable passes (48-50 us against 56 us); 3: separable passes in both directions;
// 4: source-driven walk forward + separable adjoint; 1: second generation in both directions; 0: the four-pass kernels of dim.cu
static bool sep_enabled(int S, bool tma, bool forward) {
  const int impl = tune_get("dim.impl", 2);
  return tma && S % 4 == 0 && (impl == 3 || ((impl == 2 || impl == 4) && !forward));
}
static bool sep_hot(int S, int R) { return S == 224 && sep_pitch(S, R) == 248 && tune_get("dim.sepconst", 1) != 0; }
static size_t fwd_sep_smem(int S, int R, int a_rows, int c_rows) {
  const size_t P = (size_t)sep_pitch(S, R), hr = (size_t)(a_rows > c_rows + 1 ? a_rows : c_rows + 1);
  return sizeof(float) * ((size_t)a_rows * S + hr * P + (size_t)(c_rows + 1) * P) + 16 * (size_t)(c_rows + RB);
}
static int inverse_wext(const DimTabB& tab, int S, int R) {       // weights beyond the two a row descriptor holds
  int cmax = 2;
  for (int i = 0; i < R; ++i) if (tab.inv2[i].cnt > cmax) cmax = tab.inv2[i].cnt;
  for (int i = 0; i < S; ++i) if (tab.inv1[i].cnt > cmax) cmax = tab.inv1[i].cnt;
  return cmax - 2 > 1 ? cmax - 2 : 1;
}
static size_t bwd_sep_smem(int S, int R, int u_rows, int g_rows, int wext) {
  const size_t P = (size_t)sep_pitch(S, R);
  return sizeof(float) * (bwd_sep_first(S, (int)P, u_rows) + (size_t)g_rows * S + (size_t)g_rows * P) + 16 * (size_t)(g_rows + RB) +
         sizeof(float) * (size_t)wext * (size_t)(g_rows + RB);
}

int dim_pack_build(DimPack* pack, int S, int rnd, int R, int top, int left, int identity) {
  memset(pack, 0, sizeof(DimPack));
  pack->identity = identity ? 1 : 0;
  if (identity) { pack->gf = Geo{S, S, S, 0, 0, 1, 1, 0}; pack->gb = pack->gf; pack->gw = pack->gf; return TA_OK; }
  int a = 1, c = 0, u = 1, g = 1;
  fwd_tables(S, rnd, R, top, pack->tf, &a, &c);
  bwd_tables(S, rnd, R, top, pack->tb, &u, &g);
  pack->gf = Geo{S, rnd, R, top, left, a, c, 0};
  { int aw = 1, cw = 0; const bool ok = walk_geo(pack->tf, S, rnd, top, kWalkRB, &aw, &cw); pack->gw = Geo{S, rnd, R, top, left, aw, 0, ok ? cw : 0}; }
  pack->gb = Geo{S, rnd, R, top, left, u, g, inverse_wext(pack->tb, S, R)};
  return TA_OK;
}

// shared memory that serves every draw (rnd, top) DIM can make at (S, R): scanned once per (S, R)
void dim_dyn_smem(int S, int R, size_t* fwd_bytes, size_t* bwd_bytes, size_t* fwd_sep_bytes, size_t* bwd_sep_bytes, size_t* fwd_walk_bytes) {
  static thread_local int cS = 0, cR = 0;
  static thread_local size_t cf = 0, cb = 0, cfs = 0, cbs = 0, cfw = 0;
  if (cS != S || cR != R) {
    static thread_local DimTabF tf;
    static thread_local DimTabB tb;
    size_t mf = 0, mb = 0, mfs = 0, mbs = 0, mfw = 0;
    bool walk_ok = S % 4 == 0;
    const int lo = S < R ? S : R, hi = S < R ? R : S;
    const int hi_excl = hi > lo ? hi : lo + 1;              // dim.py:54 draws rnd from [min(S,R), max(S,R)), top / left from [0, R - rnd)
    for (int rnd = lo; rnd < hi_excl; ++rnd) {
      const int ntop = R - rnd > 1 ? R - rnd : 1;
      for (int top = 0; top < ntop; ++top) {
        int a, c, u, g;
        fwd_tables(S, rnd, R, top, tf, &a, &c);
        bwd_tables(S, rnd, R, top, tb, &u, &g);
        const size_t f = fwd_smem(S, rnd, a, c), b = bwd_smem(S, rnd, u, g);
        if (f > mf) mf = f;
        if (b > mb) mb = b;
        if (S % 4 == 0) {
          const size_t fs = fwd_sep_smem(S, R, a, c), bs = bwd_sep_smem(S, R, u, g, inverse_wext(tb, S, R));
          if (fs > mfs) mfs = fs;
          if (bs > mbs) mbs = bs;
          int aw = 1, c2 = 0;
          if (!walk_geo(tf, S, rnd, top, kWalkRB, &aw, &c2)) walk_ok = false;
          else { const size_t fw = fwd_walk_smem(S, R, aw, c2, kWalkStage); if (fw > mfw) mfw = fw; }
        }
      }
    }
    cS = S; cR = R; cf = mf; cb = mb; cfs = mfs; cbs = mbs; cfw = walk_ok ? mfw : 0;   // 0: some draw does not fit the walk
  }
  *fwd_bytes = cf; *bwd_bytes = cb;
  if (fwd_sep_bytes) *fwd_sep_bytes = cfs;
  if (bwd_sep_bytes) *bwd_sep_bytes = cbs;
  if (fwd_walk_bytes) *fwd_walk_bytes = cfw;
}

int dim_fwd_dyn(const float* x, float* out, int planes, int S, int R, const DimPack* packs, int n_packs, const int* it, bool tma,
                cudaStream_t stream) {
  size_t smem, sb, smem_s, sb_s, smem_w;
  dim_dyn_smem(S, R, &smem, &sb, &smem_s, &sb_s, &smem_w);
  dim3 grid_s((unsigned)((S + RB - 1) / RB), (unsigned)planes);
  if (walk_enabled(S, tma) && smem_w > 0 && smem_w <= 200 * 1024) {
    const bool hot = sep_hot(S, R);
    auto kw = hot ? dim_fwd_walk_kernel<1, FwdTabDyn, 224, 248, kWalkRB, kWalkStage> : dim_fwd_walk_kernel<1, FwdTabDyn, 0, 0, kWalkRB, kWalkStage>;
    static SmemOptIn optin_w[2] = {};
    const int rcw = ensure_dyn_smem("ta_dim_fwd_dyn", kw, smem_w, optin_w[hot ? 0 : 1]);
    if (rcw != TA_OK) return rcw;
    dim3 grid_w((unsigned)((S + kWalkRB - 1) / kWalkRB), (unsigned)planes);
    kw<<<grid_w, kThreads, smem_w, stream>>>(x, out, FwdTabDyn{packs, it, n_packs}, Geo{});
    count_launch();
    return check_launch("ta_dim_fwd_dyn[walk]");
  }
  if (sep_enabled(S, tma, true) && aligned16(out) && smem_s <= 200 * 1024) {
    const bool hot = sep_hot(S, R);
    auto ks = hot ? dim_fwd_sep_kernel<1, FwdTabDyn, 224, 248> : dim_fwd_sep_kernel<1, FwdTabDyn, 0, 0>;
    static SmemOptIn optin_s[2] = {};
    const int rcs = ensure_dyn_smem("ta_dim_fwd_dyn", ks, smem_s, optin_s[hot ? 0 : 1]);
    if (rcs != TA_OK) return rcs;
    ks<<<grid_s, kThreads, smem_s, stream>>>(x, out, FwdTabDyn{packs, it, n_packs}, Geo{});
    count_launch();
    return check_launch("ta_dim_fwd_dyn[sep]");
  }
  TA_REQUIRE(smem <= 200 * 1024, "ta_dim_fwd_dyn: image size S=%d needs %zu B of shared memory per CTA, more than the 204800 B limit", S, smem);
  auto k = tma ? dim_fwd_direct_kernel<1, true, FwdTabDyn, true> : dim_fwd_direct_kernel<1, false, FwdTabDyn, true>;
  static SmemOptIn optin[2] = {};
  const int rc = ensure_dyn_smem("ta_dim_fwd_dyn", k, smem, optin[tma ? 0 : 1]);
  if (rc != TA_OK) return rc;
  dim3 grid((unsigned)((S + RB - 1) / RB), (unsigned)planes);
  k<<<grid, kThreads, smem, stream>>>(x, out, FwdTabDyn{packs, it, n_packs}, Geo{});
  count_launch();
  return check_launch("ta_dim_fwd_dyn");
}

int dim_bwd_dyn(const float* gout, float* gin, int planes, int S, int R, const DimPack* packs, int n_packs, const int* it, bool tma,
                cudaStream_t stream) {
  size_t sf, smem, sf_s, smem_s;
  dim_dyn_smem(S, R, &sf, &smem, &sf_s, &smem_s);
  if (sep_enabled(S, tma, false) && aligned16(gin) && smem_s <= 200 * 1024) {
    const bool hot = sep_hot(S, R);
    auto ks = hot ? dim_bwd_sep_kernel<true, 224, 248> : dim_bwd_sep_kernel<true, 0, 0>;
    static SmemOptIn optin_s[2] = {};
    const int rcs = ensure_dyn_smem("ta_dim_bwd_dyn", ks, smem_s, optin_s[hot ? 0 : 1]);
    if (rcs != TA_OK) return rcs;
    dim3 grid_s((unsigned)((S + RB - 1) / RB), (unsigned)planes);
    ks<<<grid_s, kThreads, smem_s, stream>>>(gout, gin, nullptr, Geo{}, packs, it, n_packs);
    count_launch();
    return check_launch("ta_dim_bwd_dyn[sep]");
  }
  TA_REQUIRE(smem <= 200 * 1024, "ta_dim_bwd_dyn: image size S=%d needs %zu B of shared memory per CTA, more than the 204800 B limit", S, smem);
  auto k = tma ? dim_bwd_direct_kernel<true, true> : dim_bwd_direct_kernel<false, true>;
  static SmemOptIn optin[2] = {};
  const int rc = ensure_dyn_smem("ta_dim_bwd_dyn", k, smem, optin[tma ? 0 : 1]);
  if (rc != TA_OK) return rc;
  dim3 grid((unsigned)((S + RB - 1) / RB), (unsigned)planes);
  k<<<grid, kThreads, smem, stream>>>(gout, gin, nullptr, Geo{}, packs, it, n_packs);
  count_launch();
  return check_launch("ta_dim_bwd_dyn");
}

int dim_fwd_direct(const float* x, float* out, int planes, int S, int rnd, int R, int top, int left, int blend, bool tma, void* ws,
                   cudaStream_t stream) {
  const bool reuse = tune_get("dim.reuse", 1) != 0;      // two-entry h-lerp row cache (bit-identical either way)
  static thread_local DimTabF tab;
  host_taps(R, S, tab.t2);
  host_taps(S, rnd, tab.t1);
  // exact band maxima (rows of y1 and of the source one band needs)
  int c_rows = 0, a_rows = 1;
  for (int oy0 = 0; oy0 < S; oy0 += RB) {
    const int oy1 = (oy0 + RB < S ? oy0 + RB : S) - 1;
    const int pr0 = h_i0(tab.t2[oy0]), pr1 = h_i1(tab.t2[oy1]);
    const int q0 = pr0 - top > 0 ? pr0 - top : 0, q1 = pr1 - top < rnd - 1 ? pr1 - top : rnd - 1;
    if (q0 > q1) continue;
    if (q1 - q0 + 1 > c_rows) c_rows = q1 - q0 + 1;
    const int nsr = h_i1(tab.t1[q1]) - h_i0(tab.t1[q0]) + 1;
    if (nsr > a_rows) a_rows = nsr;
  }
  Geo gm{S, rnd, R, top, left, a_rows, c_rows, 0};
  dim3 grid((unsigned)((S + RB - 1) / RB), (unsigned)planes);
  int a_w = 1, c2_rows = 0;
  const int wrb = tune_get("dim.walk_rb", kWalkRB) == 32 ? 32 : 16;
  const bool wstage = tune_get("dim.walk_stage", kWalkStage ? 1 : 0) != 0;
  if (walk_enabled(S, tma) && walk_geo(tab, S, rnd, top, wrb, &a_w, &c2_rows) && fwd_walk_smem(S, R, a_w, c2_rows, wstage) <= 200 * 1024) {
    const size_t smem_w = fwd_walk_smem(S, R, a_w, c2_rows, wstage);
    const bool hot = sep_hot(S, R);
    gm.a_rows = a_w; gm.pad = c2_rows;
    grid = dim3((unsigned)((S + wrb - 1) / wrb), (unsigned)planes);
    static SmemOptIn optin_w[80] = {};
    const int cfg = (wrb == 32 ? 2 : 0) + (wstage ? 1 : 0);
#define TA_DIM_FWD_WALK_K(MODE_, TR_, ARG_)                                                                        \
  do {                                                                                                              \
    void (*k)(const float*, float*, TR_, Geo) = nullptr;                                                            \
    if (hot) {                                                                                                      \
      k = cfg == 3 ? dim_fwd_walk_kernel<MODE_, TR_, 224, 248, 32, true> : cfg == 2 ? dim_fwd_walk_kernel<MODE_, TR_, 224, 248, 32, false> \
        : cfg == 1 ? dim_fwd_walk_kernel<MODE_, TR_, 224, 248, 16, true> : dim_fwd_walk_kernel<MODE_, TR_, 224, 248, 16, false>; \
    } else {                                                                                                        \
      k = cfg == 3 ? dim_fwd_walk_kernel<MODE_, TR_, 0, 0, 32, true> : cfg == 2 ? dim_fwd_walk_kernel<MODE_, TR_, 0, 0, 32, false> \
        : cfg == 1 ? dim_fwd_walk_kernel<MODE_, TR_, 0, 0, 16, true> : dim_fwd_walk_kernel<MODE_, TR_, 0, 0, 16, false>; \
    }                                                                                                               \
    const int rc = ensure_dyn_smem("ta_dim_fwd", k, smem_w, optin_w[(MODE_ * 2 + (ws ? 1 : 0)) * 8 + cfg * 2 + (hot ? 0 : 1)]); \
    if (rc != TA_OK) return rc;                                                                                     \
    k<<<grid, kThreads, smem_w, stream>>>(x, out, ARG_, gm);                                                        \
  } while (0)
#define TA_DIM_FWD_WALK(MODE_, SLOT_)                                                                               \
  do {                                                                                                              \
    if (ws) {                                                                                                       \
      const int ru = upload_tab(tab, ws, stream);                                                                   \
      if (ru != TA_OK) return ru;                                                                                   \
      TA_DIM_FWD_WALK_K(MODE_, FwdTabPtr, FwdTabPtr{reinterpret_cast<const DimTabF*>(ws)});                         \
    } else {                                                                                                        \
      TA_DIM_FWD_WALK_K(MODE_, FwdTabParam, *reinterpret_cast<const FwdTabParam*>(&tab));                           \
    }                                                                                                               \
  } while (0)
    switch (blend) {
      case 1: TA_DIM_FWD_WALK(1, 0); break;
      case 0: TA_DIM_FWD_WALK(0, 1); break;
      case 2: TA_DIM_FWD_WALK(2, 2); break;
      case 3: TA_DIM_FWD_WALK(3, 3); break;
      default: TA_DIM_FWD_WALK(4, 4); break;
    }
#undef TA_DIM_FWD_WALK_K
#undef TA_DIM_FWD_WALK
    count_launch();
    return check_launch("ta_dim_fwd[walk]");
  }
  if (sep_enabled(S, tma, true) && aligned16(out) && fwd_sep_smem(S, R, a_rows, c_rows) <= 200 * 1024) {
    const size_t smem_s = fwd_sep_smem(S, R, a_rows, c_rows);
    const bool hot = sep_hot(S, R);
    static SmemOptIn optin_s[20] = {};
#define TA_DIM_FWD_SEP(MODE_, SLOT_)                                                                                \
  do {                                                                                                              \
    if (ws) {                                                                                                       \
      auto k = hot ? dim_fwd_sep_kernel<MODE_, FwdTabPtr, 224, 248> : dim_fwd_sep_kernel<MODE_, FwdTabPtr, 0, 0>;   \
      const int rc = ensure_dyn_smem("ta_dim_fwd", k, smem_s, optin_s[4 * SLOT_ + (hot ? 0 : 1)]);                  \
      if (rc != TA_OK) return rc;                                                                                   \
      const int ru = upload_tab(tab, ws, stream);                                                                   \
      if (ru != TA_OK) return ru;                                                                                   \
      k<<<grid, kThreads, smem_s, stream>>>(x, out, FwdTabPtr{reinterpret_cast<const DimTabF*>(ws)}, gm);           \
    } else {                                                                                                        \
      auto k = hot ? dim_fwd_sep_kernel<MODE_, FwdTabParam, 224, 248> : dim_fwd_sep_kernel<MODE_, FwdTabParam, 0, 0>; \
      const int rc = ensure_dyn_smem("ta_dim_fwd", k, smem_s, optin_s[4 * SLOT_ + 2 + (hot ? 0 : 1)]);              \
      if (rc != TA_OK) return rc;                                                                                   \
      k<<<grid, kThreads, smem_s, stream>>>(x, out, *reinterpret_cast<const FwdTabParam*>(&tab), gm);               \
    }                                                                                                               \
  } while (0)
    switch (blend) {
      case 1: TA_DIM_FWD_SEP(1, 0); break;
      case 0: TA_DIM_FWD_SEP(0, 1); break;
      case 2: TA_DIM_FWD_SEP(2, 2); break;
      case 3: TA_DIM_FWD_SEP(3, 3); break;
      default: TA_DIM_FWD_SEP(4, 4); break;
    }
#undef TA_DIM_FWD_SEP
    count_launch();
    return check_launch("ta_dim_fwd[sep]");
  }
  const size_t smem = ((sizeof(float) * ((size_t)a_rows * S + (size_t)(c_rows + 1) * (rnd + 1)) + 15) & ~(size_t)15) + 16 * (size_t)(c_rows + RB);
  TA_REQUIRE(smem <= 200 * 1024, "ta_dim_fwd: image size S=%d needs %zu B of shared memory per CTA, more than the 204800 B limit", S, smem);
  static SmemOptIn optin[40] = {};
#define TA_DIM_FWD_LAUNCH(MODE_, SLOT_)                                                                             \
  do {                                                                                                              \
    if (ws) {                                                                                                       \
      auto k = tma ? (reuse ? dim_fwd_direct_kernel<MODE_, true, FwdTabPtr, true> : dim_fwd_direct_kernel<MODE_, true, FwdTabPtr, false>) \
                   : dim_fwd_direct_kernel<MODE_, false, FwdTabPtr, true>;                                           \
      const int rc = ensure_dyn_smem("ta_dim_fwd", k, smem, optin[4 * SLOT_ + (tma ? (reuse ? 0 : 2) : 1)]);        \
      if (rc != TA_OK) return rc;                                                                                   \
      const int ru = upload_tab(tab, ws, stream);                                                                   \
      if (ru != TA_OK) return ru;                                                                                   \
      k<<<grid, kThreads, smem, stream>>>(x, out, FwdTabPtr{reinterpret_cast<const DimTabF*>(ws)}, gm);             \
    } else {                                                                                                        \
      auto k = tma ? (reuse ? dim_fwd_direct_kernel<MODE_, true, FwdTabParam, true> : dim_fwd_direct_kernel<MODE_, true, FwdTabParam, false>) \
                   : dim_fwd_direct_kernel<MODE_, false, FwdTabParam, true>;                                         \
      const int rc = ensure_dyn_smem("ta_dim_fwd", k, smem, optin[20 + 4 * SLOT_ + (tma ? (reuse ? 0 : 2) : 1)]);   \
      if (rc != TA_OK) return rc;                                                                                   \
      k<<<grid, kThreads, smem, stream>>>(x, out, *reinterpret_cast<const FwdTabParam*>(&tab), gm);                 \
    }                                                                                                               \
  } while (0)
  switch (blend) {
    case 1: TA_DIM_FWD_LAUNCH(1, 0); break;
    case 0: TA_DIM_FWD_LAUNCH(0, 1); break;
    case 2: TA_DIM_FWD_LAUNCH(2, 2); break;
    case 3: TA_DIM_FWD_LAUNCH(3, 3); break;
    default: TA_DIM_FWD_LAUNCH(4, 4); break;
  }
#undef TA_DIM_FWD_LAUNCH
  count_launch();
  return check_launch("ta_dim_fwd[direct]");
}

int dim_bwd_direct(const float* gout, float* gin, int planes, int S, int rnd, int R, int top, int left, bool tma, bool gather,
                   void* ws, cudaStream_t stream) {
  static thread_local DimTabB tab;
  host_taps(R, S, tab.t2);
  host_taps(S, rnd, tab.t1);
  host_inverse(tab.t2, S, R, tab.inv2);
  host_inverse(tab.t1, rnd, S, tab.inv1);
  int g_rows = 1, u_rows = 1;
  for (int sy0 = 0; sy0 < S; sy0 += RB) {
    const int sy1 = (sy0 + RB < S ? sy0 + RB : S) - 1;
    tab.band[sy0 / RB] = make_short4(0, 0, 0, 0);
    int q0 = 0x7fffffff, q1 = -1;
    for (int sy = sy0; sy <= sy1; ++sy)
      if (tab.inv1[sy].cnt > 0) {
        if (tab.inv1[sy].lo < q0) q0 = tab.inv1[sy].lo;
        if (tab.inv1[sy].lo + tab.inv1[sy].cnt - 1 > q1) q1 = tab.inv1[sy].lo + tab.inv1[sy].cnt - 1;
      }
    if (q0 > q1) continue;
    if (q1 - q0 + 1 > g_rows) g_rows = q1 - q0 + 1;
    int a = 0x7fffffff, b = -1;
    for (int q = q0; q <= q1; ++q) {
      const InvE& iv = tab.inv2[q + top];
      if (iv.cnt > 0) { if (iv.lo < a) a = iv.lo; if (iv.lo + iv.cnt - 1 > b) b = iv.lo + iv.cnt - 1; }
    }
    if (a <= b && b - a + 1 > u_rows) u_rows = b - a + 1;
    tab.band[sy0 / RB] = make_short4((short)q0, (short)(q1 - q0 + 1), (short)(a <= b ? a : 0), (short)(a <= b ? b - a + 1 : 0));
  }
  Geo gm{S, rnd, R, top, left, u_rows, g_rows, 0};
  const int ru = upload_tab(tab, ws, stream);
  if (ru != TA_OK) return ru;
  const DimTabB* dtab = reinterpret_cast<const DimTabB*>(ws);
  if (sep_enabled(S, tma, false) && aligned16(gin)) {
    gm.pad = inverse_wext(tab, S, R);
    const size_t smem_s = bwd_sep_smem(S, R, u_rows, g_rows, gm.pad);
    if (smem_s <= 200 * 1024) {
      const bool hot = sep_hot(S, R);
      auto ks = hot ? dim_bwd_sep_kernel<false, 224, 248> : dim_bwd_sep_kernel<false, 0, 0>;
      static SmemOptIn optin_s[2] = {};
      const int rcs = ensure_dyn_smem("ta_dim_bwd", ks, smem_s, optin_s[hot ? 0 : 1]);
      if (rcs != TA_OK) return rcs;
      dim3 grid_s((unsigned)((S + RB - 1) / RB), (unsigned)planes);
      ks<<<grid_s, kThreads, smem_s, stream>>>(gout, gin, dtab, gm, nullptr, nullptr, 0);
      count_launch();
      return check_launch("ta_dim_bwd[sep]");
    }
    gm.pad = 0;
  }
  if (gather) {
    int cmax = 2;
    for (int i = 0; i < R; ++i) if (tab.inv2[i].cnt > cmax) cmax = tab.inv2[i].cnt;
    for (int i = 0; i < S; ++i) if (tab.inv1[i].cnt > cmax) cmax = tab.inv1[i].cnt;
    const int wext = cmax - 2 > 1 ? cmax - 2 : 1;
    const size_t smem_g = ((sizeof(float) * ((size_t)u_rows * S + (size_t)g_rows * rnd) + 15) & ~(size_t)15) +
                          16 * (size_t)(g_rows + RB) + sizeof(float) * (size_t)wext * (g_rows + RB);
    TA_REQUIRE(smem_g <= 200 * 1024, "ta_dim_bwd: image size S=%d needs %zu B of shared memory per CTA, more than the 204800 B limit", S, smem_g);
    auto kg = tma ? dim_bwd_gather_kernel<true> : dim_bwd_gather_kernel<false>;
    static SmemOptIn optin_g[2] = {};
    const int rcg = ensure_dyn_smem("ta_dim_bwd", kg, smem_g, optin_g[tma ? 0 : 1]);
    if (rcg != TA_OK) return rcg;
    dim3 grid_g((unsigned)((S + RB - 1) / RB), (unsigned)planes);
    kg<<<grid_g, kThreads, smem_g, stream>>>(gout, gin, dtab, gm, wext);
    count_launch();
    return check_launch("ta_dim_bwd[gather]");
  }
  const size_t smem = ((sizeof(float) * ((size_t)u_rows * S + (size_t)g_rows * rnd) + 15) & ~(size_t)15) + 16 * (size_t)(u_rows + g_rows);
  TA_REQUIRE(smem <= 200 * 1024, "ta_dim_bwd: image size S=%d needs %zu B of shared memory per CTA, more than the 204800 B limit", S, smem);
  auto k = tma ? dim_bwd_direct_kernel<true, false> : dim_bwd_direct_kernel<false, false>;
  static SmemOptIn optin[2] = {};
  const int rc = ensure_dyn_smem("ta_dim_bwd", k, smem, optin[tma ? 0 : 1]);
  if (rc != TA_OK) return rc;
  dim3 grid((unsigned)((S + RB - 1) / RB), (unsigned)planes);
  k<<<grid, kThreads, smem, stream>>>(gout, gin, dtab, gm, nullptr, nullptr, 0);
  count_launch();
  return check_launch("ta_dim_bwd[direct]");
}

}  // namespace ta
