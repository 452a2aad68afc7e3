// dim.cu — DIM's resize → zero-pad → resize (input_transformation/dim.py:42-68) as ONE kernel, and its exact adjoint in
// deterministic gather form (ATen's bilinear backward scatters with atomicAdd).
//
// Geometry (one (rnd, pad_top, pad_left) per batch, as in the reference):
//   y1 = bilinear(x: S x S -> rnd x rnd)     taps1[q]: source rows/cols of y1 index q
//   y2 = zero-pad(y1) to R x R at (top, left)
//   out = bilinear(y2: R x R -> S x S)       taps2[o]: y2 rows/cols of output index o
// ATen index math (align_corners=False): scale = (float)in/(float)out; src = max(0, fmaf(scale, dst+0.5f, -0.5f));
// i0 = (int)src; i1 = i0 + (i0 < in-1); l1 = src - i0; l0 = 1 - l1;
// val = hl0*(wl0*p00 + wl1*p01) + hl1*(wl0*p10 + wl1*p11).
//
// The blend is separable WITHOUT changing a single rounding: top = wl0*p00 + wl1*p01 depends only on (source row, output
// column), so it is computed once per row ("horizontal lerp") and shared by the two output rows that read that source row;
// the output is the "vertical lerp" of two such rows. Each CTA owns a band of RB output rows of one plane and runs four
// passes through shared memory: src rows (staged by one bulk-TMA copy: they are contiguous in memory) → T1 (h-lerp) → y1
// (v-lerp) → T2 (h-lerp of the zero-padded y1) → out (v-lerp, coalesced stores). Threads own columns and walk the rows, so
// column taps live in registers and row taps are warp-uniform broadcasts; no per-element integer division anywhere.
// HBM traffic: 4 B/elem in (+ halo rows re-read through L2) and 4 B/elem out.
//
// Adjoint: the four passes transposed — vertical gather from gout, horizontal gather, (crop = the pad's adjoint),
// vertical gather, horizontal gather — with inverse tap ranges built in shared memory; fixed ascending summation order.
#include "common.cuh"
#include "dim_direct.cuh"

using namespace ta;

namespace {

constexpr int RB = 16;         // output rows per CTA
constexpr int kThreads = 256;

struct Tap { int i0, i1; float l0, l1; };

__device__ __forceinline__ Tap make_tap(int in, float scale, int d) {
  float src = fmaf(scale, (float)d + 0.5f, -0.5f);      // ATen area_pixel_compute_source_index (an FMA in torch's CUDA build)
  if (src < 0.0f) src = 0.0f;
  Tap t;
  t.i0 = (int)src;
  t.i1 = t.i0 + ((t.i0 < in - 1) ? 1 : 0);
  t.l1 = sub_rn(src, (float)t.i0);
  t.l0 = sub_rn(1.0f, t.l1);
  return t;
}

// ATen's expression is  hl0*(wl0*p00 + wl1*p01) + hl1*(wl0*p10 + wl1*p11).
// mode 1 (default): inner = fma(wl0,p00, wl1*p01), outer = fma(hl0,top, hl1*bot) — the contraction nvcc applied to torch's
//   own CUDA kernel; MEASURED on B200 (tools/diag_dim_aten.py, profiles/diag_dim_r1.json): 0 differing bits against
//   F.interpolate -> F.pad -> F.interpolate for every geometry tried, so DIM's forward is bit-identical to the reference's
//   GPU path. mode 0: every product and sum rounded separately (closest to ATen's CPU kernel; used with the CPU goldens).
//   modes 2-4: the other contraction orders (kept for the diagnostic).
__device__ __forceinline__ float hlerp(int mode, float w0, float w1, float a, float b) {
  if (mode == 0) return add_rn(mul_rn(w0, a), mul_rn(w1, b));
  if (mode == 1 || mode == 3) return fmaf(w0, a, mul_rn(w1, b));
  return fmaf(w1, b, mul_rn(w0, a));
}
__device__ __forceinline__ float vlerp(int mode, float h0, float h1, float top, float bot) {
  if (mode == 0) return add_rn(mul_rn(h0, top), mul_rn(h1, bot));
  if (mode == 1 || mode == 4) return fmaf(h0, top, mul_rn(h1, bot));
  return fmaf(h1, bot, mul_rn(h0, top));
}

struct DimGeom { int S, rnd, R, top, left; int y1_rows_max, src_rows_max, t2_rows_max; int blend; };

__host__ __device__ inline size_t align16(size_t v) { return (v + 15) & ~(size_t)15; }

// shared-memory carve-up (dynamic):
//   bufA [max(src_rows_max, t2_rows_max) * S]  source band, later T2      (offset 0: the bulk-TMA destination)
//   taps2 [S], taps1 [rnd]
//   bufB [src_rows_max * rnd]  T1
//   bufC [y1_rows_max * rnd]   y1
template <bool TMA_STAGE>
__global__ void __launch_bounds__(kThreads) dim_fwd_kernel(const float* __restrict__ x, float* __restrict__ out, DimGeom gm) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t s_bar;
  const int S = gm.S, rnd = gm.rnd, R = gm.R, top = gm.top, left = gm.left, mode = gm.blend;
  const int a_rows = gm.src_rows_max > gm.t2_rows_max ? gm.src_rows_max : gm.t2_rows_max;
  float* bufA = reinterpret_cast<float*>(smem_raw);
  Tap* taps2 = reinterpret_cast<Tap*>(smem_raw + align16((size_t)a_rows * S * 4));
  Tap* taps1 = taps2 + S;
  float* bufB = reinterpret_cast<float*>(taps1 + rnd);
  float* bufC = bufB + (size_t)gm.src_rows_max * rnd;

  const int tid = threadIdx.x;
  const int oy0 = blockIdx.x * RB;
  const int oy1 = min(oy0 + RB, S) - 1;                 // inclusive
  const float* xp = x + (int64_t)blockIdx.y * S * S;
  float* op = out + (int64_t)blockIdx.y * S * S;

  const float scale2 = (float)R / (float)S, scale1 = (float)S / (float)rnd;
  for (int i = tid; i < S; i += kThreads) taps2[i] = make_tap(R, scale2, i);
  for (int i = tid; i < rnd; i += kThreads) taps1[i] = make_tap(S, scale1, i);
  if (TMA_STAGE && tid == 0) { mbar_init(&s_bar, 1); mbar_fence_init(); }
  __syncthreads();

  // rows of y2 (padded), y1 and x this band depends on; the y1 range is empty when the band maps entirely into the padding
  const int pr0 = taps2[oy0].i0, pr1 = taps2[oy1].i1;
  const int q0 = max(pr0 - top, 0), q1 = min(pr1 - top, rnd - 1);
  const bool any = q0 <= q1;
  int sr0 = 0, sr1 = -1;
  if (any) { sr0 = taps1[q0].i0; sr1 = taps1[q1].i1; }
  const int nsr = sr1 - sr0 + 1;

  if (any) {
    const float* src;
    if (TMA_STAGE) {
      if (tid == 0) {
        const uint32_t bytes = (uint32_t)(nsr * S * 4);
        mbar_expect_tx(&s_bar, bytes);
        tma_bulk_g2s(bufA, xp + (int64_t)sr0 * S, bytes, &s_bar);
      }
      mbar_wait(&s_bar, 0);
      src = bufA;
    } else {
      src = xp + (int64_t)sr0 * S;
    }
    // pass 1: T1[r][qx] = h-lerp of source row sr0 + r at y1 column qx
    for (int qx = tid; qx < rnd; qx += kThreads) {
      const Tap tw = taps1[qx];
      for (int r = 0; r < nsr; ++r) {
        const float* row = src + (int64_t)r * S;
        const float a = TMA_STAGE ? row[tw.i0] : __ldg(row + tw.i0);
        const float b = TMA_STAGE ? row[tw.i1] : __ldg(row + tw.i1);
        bufB[r * rnd + qx] = hlerp(mode, tw.l0, tw.l1, a, b);
      }
    }
    __syncthreads();
    // pass 2: y1[q][qx] = v-lerp of T1 rows
    for (int qx = tid; qx < rnd; qx += kThreads) {
      for (int q = q0; q <= q1; ++q) {
        const Tap th = taps1[q];
        bufC[(q - q0) * rnd + qx] = vlerp(mode, th.l0, th.l1, bufB[(th.i0 - sr0) * rnd + qx], bufB[(th.i1 - sr0) * rnd + qx]);
      }
    }
  }
  __syncthreads();
  // pass 3: T2[pr][ox] = h-lerp of the zero-padded y1 row pr at output column ox (the source band in bufA is dead now)
  for (int ox = tid; ox < S; ox += kThreads) {
    const Tap tw = taps2[ox];
    const int xa = tw.i0 - left, xb = tw.i1 - left;
    const bool xa_in = xa >= 0 && xa < rnd, xb_in = xb >= 0 && xb < rnd;
    for (int pr = pr0; pr <= pr1; ++pr) {
      const int yq = pr - top;
      const bool row_in = any && yq >= q0 && yq <= q1;
      const float a = (row_in && xa_in) ? bufC[(yq - q0) * rnd + xa] : 0.0f;
      const float b = (row_in && xb_in) ? bufC[(yq - q0) * rnd + xb] : 0.0f;
      bufA[(pr - pr0) * S + ox] = hlerp(mode, tw.l0, tw.l1, a, b);
    }
  }
  __syncthreads();
  // pass 4: out[oy][ox] = v-lerp of T2 rows (coalesced stores)
  for (int ox = tid; ox < S; ox += kThreads) {
    for (int oy = oy0; oy <= oy1; ++oy) {
      const Tap th = taps2[oy];
      op[(int64_t)oy * S + ox] = vlerp(mode, th.l0, th.l1, bufA[(th.i0 - pr0) * S + ox], bufA[(th.i1 - pr0) * S + ox]);
    }
  }
}

// ---- adjoint --------------------------------------------------------------------------------------------------------
// weight with which 1-D tap `t` (of some output index) reads input index `i`: l0 if i0 == i, plus l1 if i1 == i
__device__ __forceinline__ float tap_w(const Tap& t, int i) {
  float w = 0.0f;
  if (t.i0 == i) w = t.l0;
  if (t.i1 == i) w = add_rn(w, t.l1);
  return w;
}

constexpr int kMaxW = 6;   // weights of one inverse range kept in registers (bilinear at DIM's rates needs <= 4)

// smem: [taps2: S][taps1: rnd][inv2 lo/hi: 2R ints][inv1 lo/hi: 2S ints][bufU: max(nq*S, RB*rnd)][bufG: nq*rnd]
__global__ void __launch_bounds__(kThreads) dim_bwd_kernel(const float* __restrict__ gout, float* __restrict__ gin, DimGeom gm) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int S = gm.S, rnd = gm.rnd, R = gm.R, top = gm.top, left = gm.left;
  Tap* taps2 = reinterpret_cast<Tap*>(smem_raw);
  Tap* taps1 = taps2 + S;
  int* inv2_lo = reinterpret_cast<int*>(taps1 + rnd);
  int* inv2_hi = inv2_lo + R;
  int* inv1_lo = inv2_hi + R;
  int* inv1_hi = inv1_lo + S;
  float* bufU = reinterpret_cast<float*>(inv1_hi + S);
  const size_t u_elems = (size_t)gm.y1_rows_max * S > (size_t)RB * rnd ? (size_t)gm.y1_rows_max * S : (size_t)RB * rnd;
  float* bufG = bufU + u_elems;

  const int tid = threadIdx.x;
  const int sy0 = blockIdx.x * RB;
  const int sy1 = min(sy0 + RB, S) - 1;
  const float* gp = gout + (int64_t)blockIdx.y * S * S;
  float* ip = gin + (int64_t)blockIdx.y * S * S;

  const float scale2 = (float)R / (float)S, scale1 = (float)S / (float)rnd;
  for (int i = tid; i < S; i += kThreads) { taps2[i] = make_tap(R, scale2, i); inv1_lo[i] = 0x7fffffff; inv1_hi[i] = -1; }
  for (int i = tid; i < rnd; i += kThreads) taps1[i] = make_tap(S, scale1, i);
  for (int i = tid; i < R; i += kThreads) { inv2_lo[i] = 0x7fffffff; inv2_hi[i] = -1; }
  __syncthreads();
  // inverse ranges (min/max → order-independent): which outputs o read y2 index p; which y1 indices q read source s.
  // Taps are monotone, so every index inside [lo, hi] touches p.
  for (int o = tid; o < S; o += kThreads) {
    atomicMin(&inv2_lo[taps2[o].i0], o); atomicMax(&inv2_hi[taps2[o].i1], o);
    atomicMin(&inv2_lo[taps2[o].i1], o); atomicMax(&inv2_hi[taps2[o].i0], o);
  }
  for (int q = tid; q < rnd; q += kThreads) {
    atomicMin(&inv1_lo[taps1[q].i0], q); atomicMax(&inv1_hi[taps1[q].i1], q);
    atomicMin(&inv1_lo[taps1[q].i1], q); atomicMax(&inv1_hi[taps1[q].i0], q);
  }
  __syncthreads();

  // y1 rows feeding this band of source rows
  int q0 = 0x7fffffff, q1 = -1;
  for (int sy = sy0; sy <= sy1; ++sy) { q0 = min(q0, inv1_lo[sy]); q1 = max(q1, inv1_hi[sy]); }
  const bool any = q0 <= q1;

  if (any) {
    // pass a (adjoint of out's v-lerp): U[q][ox] = sum_{oy reads y2 row q+top} wy * gout[oy][ox]
    for (int ox = tid; ox < S; ox += kThreads) {
      for (int q = q0; q <= q1; ++q) {
        const int py = q + top;
        float acc = 0.0f;
        for (int oy = inv2_lo[py]; oy <= inv2_hi[py]; ++oy) acc = fmaf(tap_w(taps2[oy], py), __ldg(gp + (int64_t)oy * S + ox), acc);
        bufU[(q - q0) * S + ox] = acc;
      }
    }
    __syncthreads();
    // pass b (adjoint of T2's h-lerp, cropped to the pad window): g1[q][qx] = sum_{ox reads y2 col qx+left} wx * U[q][ox]
    for (int qx = tid; qx < rnd; qx += kThreads) {
      const int px = qx + left;
      const int lo = inv2_lo[px], cnt = inv2_hi[px] - lo + 1;
      float w[kMaxW];
#pragma unroll
      for (int k = 0; k < kMaxW; ++k) w[k] = (k < cnt) ? tap_w(taps2[lo + k], px) : 0.0f;
      for (int q = q0; q <= q1; ++q) {
        const float* row = bufU + (q - q0) * S;
        float acc = 0.0f;
#pragma unroll
        for (int k = 0; k < kMaxW; ++k) if (k < cnt) acc = fmaf(w[k], row[lo + k], acc);
        for (int k = kMaxW; k < cnt; ++k) acc = fmaf(tap_w(taps2[lo + k], px), row[lo + k], acc);
        bufG[(q - q0) * rnd + qx] = acc;
      }
    }
  }
  __syncthreads();
  // pass c (adjoint of y1's v-lerp): V[sy][qx] = sum_{q reads source row sy} wy * g1[q][qx]      (V overwrites U)
  for (int qx = tid; qx < rnd; qx += kThreads) {
    for (int sy = sy0; sy <= sy1; ++sy) {
      float acc = 0.0f;
      if (any)
        for (int q = inv1_lo[sy]; q <= inv1_hi[sy]; ++q) acc = fmaf(tap_w(taps1[q], sy), bufG[(q - q0) * rnd + qx], acc);
      bufU[(sy - sy0) * rnd + qx] = acc;
    }
  }
  __syncthreads();
  // pass d (adjoint of T1's h-lerp): gin[sy][sx] = sum_{qx reads source col sx} wx * V[sy][qx]     (coalesced stores)
  for (int sx = tid; sx < S; sx += kThreads) {
    const int lo = inv1_lo[sx], cnt = inv1_hi[sx] - lo + 1;
    float w[kMaxW];
#pragma unroll
    for (int k = 0; k < kMaxW; ++k) w[k] = (k < cnt) ? tap_w(taps1[lo + k], sx) : 0.0f;
    for (int sy = sy0; sy <= sy1; ++sy) {
      const float* row = bufU + (sy - sy0) * rnd;
      float acc = 0.0f;
#pragma unroll
      for (int k = 0; k < kMaxW; ++k) if (k < cnt) acc = fmaf(w[k], row[lo + k], acc);
      for (int k = kMaxW; k < cnt; ++k) acc = fmaf(tap_w(taps1[lo + k], sx), row[lo + k], acc);
      ip[(int64_t)sy * S + sx] = acc;
    }
  }
}

int check_geom(const char* who, int planes, int S, int rnd, int R, int top, int left) {
  TA_REQUIRE(planes > 0 && S > 0, "%s: empty shape", who);
  TA_REQUIRE(rnd >= 1 && R >= rnd && top >= 0 && left >= 0 && top + rnd <= R && left + rnd <= R,
             "%s: bad geometry S=%d rnd=%d R=%d top=%d left=%d", who, S, rnd, R, top, left);
  TA_REQUIRE(planes <= 65535, "%s: planes=%d exceeds 65535", who, planes);
  return TA_OK;
}

// conservative row bounds for the shared-memory bands
int band_rows(int rows_out, int in, int out) {   // input rows touched by `rows_out` consecutive output rows of an in->out resize
  return (int)((double)rows_out * (double)in / (double)out) + 3;
}

}  // namespace

extern "C" {

int ta_dim_fwd(const float* x, float* out, int planes, int S, int rnd, int R, int pad_top, int pad_left, ta_stream_t stream) {
  TA_REQUIRE(x && out, "ta_dim_fwd: null pointer");
  int rc = check_geom("ta_dim_fwd", planes, S, rnd, R, pad_top, pad_left);
  if (rc != TA_OK) return rc;
  DimGeom gm{S, rnd, R, pad_top, pad_left, 0, 0, 0, tune_get("dim.blend", 1)};
  gm.t2_rows_max = band_rows(RB, R, S);
  if (gm.t2_rows_max > R) gm.t2_rows_max = R;
  gm.y1_rows_max = gm.t2_rows_max < rnd ? gm.t2_rows_max : rnd;
  gm.src_rows_max = band_rows(gm.y1_rows_max, S, rnd);
  if (gm.src_rows_max > S) gm.src_rows_max = S;
  const bool can_tma = (S % 4 == 0) && aligned16(x) && tune_get("dim.tma", 1) != 0;
  const int a_rows = gm.src_rows_max > gm.t2_rows_max ? gm.src_rows_max : gm.t2_rows_max;
  const size_t smem = align16((size_t)a_rows * S * 4) + sizeof(Tap) * (size_t)(S + rnd) +
                      sizeof(float) * ((size_t)gm.src_rows_max * rnd + (size_t)gm.y1_rows_max * rnd);
  TA_REQUIRE(smem <= 200 * 1024, "ta_dim_fwd: image size S=%d needs %zu B of shared memory per CTA, more than the 204800 B limit", S, smem);
  auto k = can_tma ? dim_fwd_kernel<true> : dim_fwd_kernel<false>;
  static SmemOptIn optin_tma = {}, optin_ldg = {};
  rc = ensure_dyn_smem("ta_dim_fwd", k, smem, can_tma ? optin_tma : optin_ldg);
  if (rc != TA_OK) return rc;
  dim3 grid((unsigned)((S + RB - 1) / RB), (unsigned)planes);
  k<<<grid, kThreads, smem, (cudaStream_t)stream>>>(x, out, gm);
  count_launch();
  return check_launch("ta_dim_fwd");
}

int ta_dim_bwd(const float* gout, float* gin, int planes, int S, int rnd, int R, int pad_top, int pad_left, ta_stream_t stream) {
  TA_REQUIRE(gout && gin, "ta_dim_bwd: null pointer");
  int rc = check_geom("ta_dim_bwd", planes, S, rnd, R, pad_top, pad_left);
  if (rc != TA_OK) return rc;
  DimGeom gm{S, rnd, R, pad_top, pad_left, 0, 0, 0, 0};
  // y1 rows reading RB consecutive source rows of the S -> rnd resize
  gm.y1_rows_max = (int)((double)(RB + 1) * (double)rnd / (double)S) + 3;
  if (gm.y1_rows_max > rnd) gm.y1_rows_max = rnd;
  const size_t u_elems = (size_t)gm.y1_rows_max * S > (size_t)RB * rnd ? (size_t)gm.y1_rows_max * S : (size_t)RB * rnd;
  const size_t smem = sizeof(Tap) * (size_t)(S + rnd) + sizeof(int) * (size_t)(2 * R + 2 * S) +
                      sizeof(float) * (u_elems + (size_t)gm.y1_rows_max * rnd);
  TA_REQUIRE(smem <= 200 * 1024, "ta_dim_bwd: image size S=%d needs %zu B of shared memory per CTA, more than the 204800 B limit", S, smem);
  static SmemOptIn optin = {};
  rc = ensure_dyn_smem("ta_dim_bwd", dim_bwd_kernel, smem, optin);
  if (rc != TA_OK) return rc;
  dim3 grid((unsigned)((S + RB - 1) / RB), (unsigned)planes);
  dim_bwd_kernel<<<grid, kThreads, smem, (cudaStream_t)stream>>>(gout, gin, gm);
  count_launch();
  return check_launch("ta_dim_bwd");
}

// ---- with a caller-provided device workspace: the direct kernels of dim_direct.cu ---------------------------------------------
// ws: ta_dim_ws_bytes() bytes of DEVICE memory, 16-byte aligned, owned by the caller until the stream has passed the call
// (the per-call tap / inverse-range tables are uploaded into it in stream order). dim.impl: 1 (default) = direct kernels
// (dim.bwd: 0 (default) = gather + scatter into rotating accumulators, 1 = independent separable gather per element;
// dim.fwdtab: 0 (default) = forward tables as kernel parameters, 1 = in the workspace), 0 = the four-pass
// kernels above. Same results as ta_dim_fwd (bit-identical) / ta_dim_bwd (same sums, different association).
int64_t ta_dim_ws_bytes(void) { return (int64_t)dim_direct_ws_bytes(); }

int ta_dim_fwd_ws(const float* x, float* out, int planes, int S, int rnd, int R, int pad_top, int pad_left, void* ws,
                  ta_stream_t stream) {
  TA_REQUIRE(x && out, "ta_dim_fwd_ws: null pointer");
  int rc = check_geom("ta_dim_fwd_ws", planes, S, rnd, R, pad_top, pad_left);
  if (rc != TA_OK) return rc;
  if (ws && aligned16(ws) && tune_get("dim.impl", 2) != 0 && dim_direct_ok(S, rnd, R))
    return dim_fwd_direct(x, out, planes, S, rnd, R, pad_top, pad_left, tune_get("dim.blend", 1),
                          (S % 4 == 0) && aligned16(x) && tune_get("dim.tma", 1) != 0,
                          tune_get("dim.fwdtab", 0) != 0 ? ws : nullptr,      // forward: tables as kernel parameters by default
                          (cudaStream_t)stream);
  return ta_dim_fwd(x, out, planes, S, rnd, R, pad_top, pad_left, stream);
}

int ta_dim_bwd_ws(const float* gout, float* gin, int planes, int S, int rnd, int R, int pad_top, int pad_left, void* ws,
                  ta_stream_t stream) {
  TA_REQUIRE(gout && gin, "ta_dim_bwd_ws: null pointer");
  int rc = check_geom("ta_dim_bwd_ws", planes, S, rnd, R, pad_top, pad_left);
  if (rc != TA_OK) return rc;
  if (ws && aligned16(ws) && tune_get("dim.impl", 2) != 0 && dim_direct_ok(S, rnd, R))
    return dim_bwd_direct(gout, gin, planes, S, rnd, R, pad_top, pad_left,
                          (S % 4 == 0) && aligned16(gout) && tune_get("dim.tma", 1) != 0, tune_get("dim.bwd", 0) != 0, ws,
                          (cudaStream_t)stream);
  return ta_dim_bwd(gout, gin, planes, S, rnd, R, pad_top, pad_left, stream);
}


// ---- the draw in DEVICE memory: one captured CUDA graph serves every iteration's (coin, rnd, top, left) -----------------------
int64_t ta_dim_pack_bytes(void) { return (int64_t)sizeof(DimPack); }

int ta_dim_pack_build(void* host_pack, int S, int rnd, int R, int pad_top, int pad_left, int identity) {
  TA_REQUIRE(host_pack, "ta_dim_pack_build: null pointer");
  if (!identity) {
    const int rc = check_geom("ta_dim_pack_build", 1, S, rnd, R, pad_top, pad_left);
    if (rc != TA_OK) return rc;
    if (!dim_direct_ok(S, rnd, R)) { set_error("ta_dim_pack_build: S=%d R=%d beyond the direct kernels' tables (S <= %d, R <= %d)", S, R, kDimMaxS, kDimMaxR); return TA_EUNSUPPORTED; }
  }
  return dim_pack_build(reinterpret_cast<DimPack*>(host_pack), S, rnd, R, pad_top, pad_left, identity);
}

int ta_dim_fwd_dyn(const float* x, float* out, int planes, int S, int R, const void* packs, int n_packs, const int* it,
                   ta_stream_t stream) {
  TA_REQUIRE(x && out && packs && it && n_packs > 0 && planes > 0, "ta_dim_fwd_dyn: bad arguments");
  TA_REQUIRE(planes <= 65535, "ta_dim_fwd_dyn: planes=%d exceeds 65535", planes);
  if (!aligned16(packs)) { set_error("ta_dim_fwd_dyn: packs are not 16-byte aligned"); return TA_EUNSUPPORTED; }
  if (!dim_direct_ok(S, S, R)) {
    set_error("ta_dim_fwd_dyn: S=%d R=%d beyond the direct kernels' tables (S <= %d, R <= %d)", S, R, kDimMaxS, kDimMaxR);
    return TA_EUNSUPPORTED;
  }
  return dim_fwd_dyn(x, out, planes, S, R, reinterpret_cast<const DimPack*>(packs), n_packs, it,
                     (S % 4 == 0) && aligned16(x) && tune_get("dim.tma", 1) != 0, (cudaStream_t)stream);
}

int ta_dim_bwd_dyn(const float* gout, float* gin, int planes, int S, int R, const void* packs, int n_packs, const int* it,
                   ta_stream_t stream) {
  TA_REQUIRE(gout && gin && packs && it && n_packs > 0 && planes > 0, "ta_dim_bwd_dyn: bad arguments");
  TA_REQUIRE(planes <= 65535, "ta_dim_bwd_dyn: planes=%d exceeds 65535", planes);
  if (!aligned16(packs)) { set_error("ta_dim_bwd_dyn: packs are not 16-byte aligned"); return TA_EUNSUPPORTED; }
  if (!dim_direct_ok(S, S, R)) {
    set_error("ta_dim_bwd_dyn: S=%d R=%d beyond the direct kernels' tables (S <= %d, R <= %d)", S, R, kDimMaxS, kDimMaxR);
    return TA_EUNSUPPORTED;
  }
  return dim_bwd_dyn(gout, gin, planes, S, R, reinterpret_cast<const DimPack*>(packs), n_packs, it,
                     (S % 4 == 0) && aligned16(gout) && tune_get("dim.tma", 1) != 0, (cudaStream_t)stream);
}

}  // extern "C"
