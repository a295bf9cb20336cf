// Barlow Twins loss, forward + backward — replaces BarlowLoss.forward (reference utils/losses.py:127-142,
// call site models/barlow.py:90).
//
//   x~ = (x - mean_0) / std_0 (UNBIASED std, :136-137);  C = Xi~^T Xj~ / N (:138)
//   loss = sum_a (C_aa - 1)^2 + lambda * sum_{a != b} C_ab^2 (:139-142)
//   dC_aa = 2 (C_aa - 1), dC_ab = 2 lambda C_ab;  dXi~ = Xj~ dC^T / N;  dXj~ = Xi~ dC / N
//   dx = (dx~ - mean_0(dx~) - x~ * sum_0(dx~ . x~) / (N-1)) / std        [+ row-normalise backward if normalize]
//
// Forward, both views per launch: column statistics (shifted single pass) -> standardise to bf16 -> tcgen05 GEMM with
// both operands consumed MN-major in place (no transposed copies) and a fused epilogue that reduces the loss, emits dC in
// bf16 (the D x D fp32 matrix never reaches HBM) and takes the row / column sums of dC .* C -> one kernel that finishes
// the loss and q_i / q_j.
// Backward: ONE dual tcgen05 GEMM (dTi = Xj~ dC^T / n, dTj = Xi~ dC / n) whose epilogue applies the closed-form
// standardise-backward and writes dzi / dzj.  normalize = 1 (and the row-store epilogue) goes through fp32 dT instead:
// the dual GEMM writes dT (its epilogue also takes the column partials when they fit, else a separate reduction pass
// does) -> column finalize -> finish kernel with the row-normalise backward, both views per launch.
#include "gemm_host.cuh"

using namespace ssvb;

namespace {

constexpr int kColsPerBlock = 32;
constexpr int kRowSplit = 8;  // row stripes per column group (fills the SMs at D = 4096..8192)
constexpr int kStatSplit = 32;       // row stripes of the float4 statistics kernel (128 columns per block)
constexpr int kMaxFusedStripes = 256;  // fused backward column partials: one stripe per (128-row tile, epilogue warp)
constexpr int kMaxGemmCtas = 160;
// stripes of the backward column partials written by the GEMM epilogue (0: too many rows, separate reduction pass)
inline int fused_stripes(int64_t n) {
  const int64_t t = ceil_div(n, 128) * 4;
  return t <= kMaxFusedStripes ? static_cast<int>(t) : 0;
}

struct BarlowSaved {
  __nv_bfloat16 *xi, *xj;  // standardised operands [n x d]
  __nv_bfloat16* dC;       // [d x d]
  float *mean_i, *rstd_i, *mean_j, *rstd_j;  // [d]
  float *inv_i, *inv_j;                      // [n] row 1/norm (normalize=1)
  float *q_i, *q_j;  // [d] rstd * sum_n(dT x~)/(n-1), from the forward's dC .* C sums (closed-form backward, see below)
  size_t bytes;
};
BarlowSaved barlow_saved(void* base, int64_t n, int64_t d) {
  Carver c(base);
  BarlowSaved s;
  s.xi = c.take<__nv_bfloat16>(n * d);
  s.xj = c.take<__nv_bfloat16>(n * d);
  s.dC = c.take<__nv_bfloat16>(d * d);
  s.mean_i = c.take<float>(d);
  s.rstd_i = c.take<float>(d);
  s.mean_j = c.take<float>(d);
  s.rstd_j = c.take<float>(d);
  s.inv_i = c.take<float>(n);
  s.inv_j = c.take<float>(n);
  s.q_i = c.take<float>(d);
  s.q_j = c.take<float>(d);
  s.bytes = c.used();
  return s;
}
struct BarlowWs {
  float* colpart;        // [2 views][stripes][2][d], stripes = max(kStatSplit, fused_stripes(n), kRowSplit)
  int64_t view_stride;   // floats between the two views' partials
  float* loss_partials;  // [kMaxGemmCtas]
  float *dti, *dtj;      // backward: [n x d] fp32 each
  float* colred;         // [2 views][2][d]  (mean of dT, sum(dT x~)/(n-1))
  float* xrow;           // forward: [ceil(d/256)][d] row sums of dC .* C per column tile (GEMM epilogue)
  float* xcol;           // forward: [ceil(d/128) * 4][d] column sums of dC .* C per (row tile, epilogue warp)
  size_t bytes;
};
BarlowWs barlow_ws(void* base, int64_t n, int64_t d) {
  Carver c(base);
  BarlowWs w;
  int64_t stripes = kStatSplit > kRowSplit ? kStatSplit : kRowSplit;
  if (fused_stripes(n) > stripes) stripes = fused_stripes(n);
  w.view_stride = stripes * 2 * d;
  w.colpart = c.take<float>(2 * w.view_stride);
  w.loss_partials = c.take<float>(kMaxGemmCtas);
  w.dti = c.take<float>(n * d);
  w.dtj = c.take<float>(n * d);
  w.colred = c.take<float>(4 * d);
  w.xrow = c.take<float>(ceil_div(d, 256) * d);
  w.xcol = c.take<float>(ceil_div(d, 128) * 4 * d);
  w.bytes = c.used();
  return w;
}


// distributed: the saved blob holds only LOCAL rows; dC is a caller-visible tensor (it is all-gathered)
struct BarlowDistSaved {
  __nv_bfloat16 *xi, *xj;                    // standardised local rows [n_local x d]
  float *mean_i, *rstd_i, *mean_j, *rstd_j;  // [d] GLOBAL statistics
  float *inv_i, *inv_j;                      // [n_local]
  size_t bytes;
};
BarlowDistSaved barlow_dist_saved(void* base, int64_t n, int64_t d) {
  Carver c(base);
  BarlowDistSaved s;
  s.xi = c.take<__nv_bfloat16>(n * d);
  s.xj = c.take<__nv_bfloat16>(n * d);
  s.mean_i = c.take<float>(d);
  s.rstd_i = c.take<float>(d);
  s.mean_j = c.take<float>(d);
  s.rstd_j = c.take<float>(d);
  s.inv_i = c.take<float>(n);
  s.inv_j = c.take<float>(n);
  s.bytes = c.used();
  return s;
}
struct BarlowDistWs {
  float* colpart;   // [2 views][kRowSplit][2][d]
  float *dti, *dtj; // backward: [n_local x d] fp32 each (live between bwd_gemm and bwd_finish)
  float* colred;    // [2][2][d]
  size_t bytes;
};
constexpr int kEpiGridMax = 148 * 8;
BarlowDistWs barlow_dist_ws(void* base, int64_t n, int64_t d) {
  Carver c(base);
  BarlowDistWs w;
  w.colpart = c.take<float>(2 * kRowSplit * 2 * d);
  w.dti = c.take<float>(n * d);
  w.dtj = c.take<float>(n * d);
  w.colred = c.take<float>(4 * d);
  w.bytes = c.used();
  return w;
}

// row 1/max(||x||, eps): one warp per row
__global__ void row_invnorm_kernel(const float* __restrict__ x, int64_t n, int d, int64_t ld, float* __restrict__ inv) {
  const int64_t row = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n) return;
  const float4* xr = reinterpret_cast<const float4*>(x + row * ld);
  float s = 0.f;
  for (int c = lane; c < d / 4; c += 32) {
    const float4 v = __ldg(xr + c);
    s += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  s = warp_sum(s);
  if (lane == 0) inv[row] = 1.f / fmaxf(sqrtf(s), 1e-12f);
}

// Column partial sums over a row stripe.  MODE 0 (stats): f = v - v0, g = (v - v0)^2 with v0 = value of row 0
// (shift against cancellation).  MODE 1 (backward): f = dT, g = dT * x~.
// block (32, 8): threadIdx.x <-> column (coalesced 128-byte row segments), threadIdx.y <-> row phase.
template <int MODE>
__global__ void col_partials_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ inv_row,
                                    const float* __restrict__ dt, int64_t lddt, const float* __restrict__ mean,
                                    const float* __restrict__ rstd, int64_t n, int d, float* __restrict__ part) {
  const int col = blockIdx.x * kColsPerBlock + threadIdx.x;
  const int stripe = blockIdx.y;
  const int64_t rows_per = (n + gridDim.y - 1) / gridDim.y;
  const int64_t r0 = stripe * rows_per, r1 = min(n, r0 + rows_per);
  float s1 = 0.f, s2 = 0.f;
  if (col < d) {
    float v0 = 0.f, mu = 0.f, rs = 0.f;
    if (MODE == 0) v0 = x[col] * (inv_row ? inv_row[0] : 1.f);
    if (MODE == 1) { mu = mean[col]; rs = rstd[col]; }
    for (int64_t r = r0 + threadIdx.y; r < r1; r += blockDim.y) {
      const float v = x[r * ldx + col] * (inv_row ? inv_row[r] : 1.f);
      if (MODE == 0) {
        const float t = v - v0;
        s1 += t;
        s2 = fmaf(t, t, s2);
      } else {
        const float g = dt[r * lddt + col];
        s1 += g;
        s2 = fmaf(g, (v - mu) * rs, s2);
      }
    }
  }
  __shared__ float sh1[8][kColsPerBlock + 1], sh2[8][kColsPerBlock + 1];
  sh1[threadIdx.y][threadIdx.x] = s1;
  sh2[threadIdx.y][threadIdx.x] = s2;
  __syncthreads();
  if (threadIdx.y == 0 && col < d) {
    float a = 0.f, b = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { a += sh1[i][threadIdx.x]; b += sh2[i][threadIdx.x]; }
    part[(static_cast<int64_t>(stripe) * 2 + 0) * d + col] = a;
    part[(static_cast<int64_t>(stripe) * 2 + 1) * d + col] = b;
  }
}

// Forward statistics, float4 version of MODE 0: block (32, 8) covers 128 columns (one float4 per thread and row), eight
// rows in flight per thread; same shifted sums and the same partial layout [stripe][2][d].
__device__ __forceinline__ void col_stats4_body(const float* __restrict__ x, int64_t ldx, const float* __restrict__ inv_row,
                                                int64_t n, int d, float* __restrict__ part) {
  const int c4 = blockIdx.x * 32 + threadIdx.x;
  const int stripe = blockIdx.y;
  const int64_t rows_per = (n + gridDim.y - 1) / gridDim.y;
  const int64_t r0 = stripe * rows_per, r1 = min(n, r0 + rows_per);
  float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
  const bool ok = c4 * 4 < d;
  if (ok) {
    const float sc0 = inv_row ? inv_row[0] : 1.f;
    float4 v0 = __ldg(reinterpret_cast<const float4*>(x) + c4);
    v0 = make_float4(v0.x * sc0, v0.y * sc0, v0.z * sc0, v0.w * sc0);
    auto acc = [&](const float4 v, const float sc) {
      const float tx = v.x * sc - v0.x, ty = v.y * sc - v0.y, tz = v.z * sc - v0.z, tw = v.w * sc - v0.w;
      s1.x += tx; s1.y += ty; s1.z += tz; s1.w += tw;
      s2.x = fmaf(tx, tx, s2.x); s2.y = fmaf(ty, ty, s2.y); s2.z = fmaf(tz, tz, s2.z); s2.w = fmaf(tw, tw, s2.w);
    };
    int64_t r = r0 + threadIdx.y;
    for (; r + 56 < r1; r += 64) {  // eight rows (128 bytes per thread) in flight
      float4 v[8];
      float sc[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        v[u] = __ldg(reinterpret_cast<const float4*>(x + (r + 8 * u) * ldx) + c4);
        sc[u] = inv_row ? inv_row[r + 8 * u] : 1.f;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) acc(v[u], sc[u]);
    }
    for (; r < r1; r += 8) acc(__ldg(reinterpret_cast<const float4*>(x + r * ldx) + c4), inv_row ? inv_row[r] : 1.f);
  }
  __shared__ float4 sh1[8][32], sh2[8][32];
  sh1[threadIdx.y][threadIdx.x] = s1;
  sh2[threadIdx.y][threadIdx.x] = s2;
  __syncthreads();
  if (threadIdx.y == 0 && ok) {
    float4 a = sh1[0][threadIdx.x], b = sh2[0][threadIdx.x];
#pragma unroll
    for (int i = 1; i < 8; ++i) {
      const float4 u = sh1[i][threadIdx.x], w = sh2[i][threadIdx.x];
      a.x += u.x; a.y += u.y; a.z += u.z; a.w += u.w;
      b.x += w.x; b.y += w.y; b.z += w.z; b.w += w.w;
    }
    *reinterpret_cast<float4*>(part + (static_cast<int64_t>(stripe) * 2 + 0) * d + c4 * 4) = a;
    *reinterpret_cast<float4*>(part + (static_cast<int64_t>(stripe) * 2 + 1) * d + c4 * 4) = b;
  }
}

// Both views of the Barlow forward in ONE launch (view = blockIdx.z / blockIdx.y of the kernels below): the launch ramp,
// tail and dependency gap of three kernels are paid once instead of twice (profiles/r2_tuning_log.md §6).
struct TwoViews {
  const float *x0, *x1;      // [n x d] fp32 rows
  int64_t ld0, ld1;
  const float *inv0, *inv1;  // row 1/norm or nullptr
};
struct TwoStats {
  float *mean0, *rstd0, *mean1, *rstd1;  // [d] each
};
__global__ void __launch_bounds__(256)
col_stats4_x2_kernel(TwoViews v, int64_t n, int d, float* __restrict__ part, int64_t view_stride) {
  const bool second = blockIdx.z != 0;
  col_stats4_body(second ? v.x1 : v.x0, second ? v.ld1 : v.ld0, second ? v.inv1 : v.inv0, n, d,
                  part + (second ? view_stride : 0));
}

// forward statistics of both views: blockIdx.y = view
__global__ void col_finalize_x2_kernel(const float* __restrict__ part, int64_t view_stride, int nsplit, TwoViews v, int64_t n,
                                       int d, TwoStats st) {
  // block (32 columns x 8 stripe phases), fixed-order combine: 2 x d/32 CTAs instead of 2 x d/256 serial column loops
  __shared__ float sh1[8][33], sh2[8][33];
  const int col = blockIdx.x * 32 + threadIdx.x;
  const bool second = blockIdx.y != 0;
  part += second ? view_stride : 0;
  float s1 = 0.f, s2 = 0.f;
  if (col < d) {
#pragma unroll 4
    for (int i = threadIdx.y; i < nsplit; i += 8) {
      s1 += part[(static_cast<int64_t>(i) * 2 + 0) * d + col];
      s2 += part[(static_cast<int64_t>(i) * 2 + 1) * d + col];
    }
  }
  sh1[threadIdx.y][threadIdx.x] = s1;
  sh2[threadIdx.y][threadIdx.x] = s2;
  __syncthreads();
  if (threadIdx.y != 0 || col >= d) return;
  s1 = 0.f;
  s2 = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) { s1 += sh1[i][threadIdx.x]; s2 += sh2[i][threadIdx.x]; }
  const float* x = second ? v.x1 : v.x0;
  const float* inv_row = second ? v.inv1 : v.inv0;
  const float fn = static_cast<float>(n);
  const float v0 = x[col] * (inv_row ? inv_row[0] : 1.f);
  const float var = (s2 - s1 * s1 / fn) / (fn - 1.f);
  (second ? st.mean1 : st.mean0)[col] = v0 + s1 / fn;
  (second ? st.rstd1 : st.rstd0)[col] = rsqrtf(var);
}

// MODE 1 finalize for MANY stripes (the GEMM epilogue's partials: one stripe per 32 rows): block (32 columns x 8 stripe
// phases), fixed-order combine.  out0 = mean_0(dT), out1 = sum_0(dT x~) / (n - 1).
__global__ void col_finalize_wide_kernel(const float* __restrict__ part, int nsplit, int64_t n, int d,
                                         float* __restrict__ out0, float* __restrict__ out1, int64_t part_view_stride) {
  // blockIdx.y = view (two-view launch): partials `part_view_stride` apart, outputs [out0 | out1] pairs 2 * d apart
  part += blockIdx.y * part_view_stride;
  out0 += blockIdx.y * 2 * static_cast<int64_t>(d);
  out1 += blockIdx.y * 2 * static_cast<int64_t>(d);
  __shared__ float sh1[8][33], sh2[8][33];
  const int col = blockIdx.x * 32 + threadIdx.x;
  float s1 = 0.f, s2 = 0.f;
  if (col < d) {
    for (int i = threadIdx.y; i < nsplit; i += 8) {
      s1 += part[(static_cast<int64_t>(i) * 2 + 0) * d + col];
      s2 += part[(static_cast<int64_t>(i) * 2 + 1) * d + col];
    }
  }
  sh1[threadIdx.y][threadIdx.x] = s1;
  sh2[threadIdx.y][threadIdx.x] = s2;
  __syncthreads();
  if (threadIdx.y == 0 && col < d) {
    float a = 0.f, b = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { a += sh1[i][threadIdx.x]; b += sh2[i][threadIdx.x]; }
    const float fn = static_cast<float>(n);
    out0[col] = a / fn;
    out1[col] = b / (fn - 1.f);
  }
}

// x~ = (x * inv_row - mean) * rstd  -> bf16 [n x d]
__device__ __forceinline__ void standardize_body(const float* __restrict__ x, int64_t ldx, const float* __restrict__ inv_row,
                                                 const float* __restrict__ mean, const float* __restrict__ rstd, int64_t n,
                                                 int d4, __nv_bfloat16* __restrict__ out, int64_t ldo) {
  const int64_t total = n * d4;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = i / d4;
    const int c = static_cast<int>(i - r * d4);
    const float sc = inv_row ? inv_row[r] : 1.f;
    const float4 v = __ldg(reinterpret_cast<const float4*>(x + r * ldx) + c);
    const float4 mu = __ldg(reinterpret_cast<const float4*>(mean) + c);
    const float4 rs = __ldg(reinterpret_cast<const float4*>(rstd) + c);
    __nv_bfloat162 lo = __floats2bfloat162_rn((v.x * sc - mu.x) * rs.x, (v.y * sc - mu.y) * rs.y);
    __nv_bfloat162 hi = __floats2bfloat162_rn((v.z * sc - mu.z) * rs.z, (v.w * sc - mu.w) * rs.w);
    uint2 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&lo);
    pk.y = *reinterpret_cast<uint32_t*>(&hi);
    *reinterpret_cast<uint2*>(out + r * ldo + 4 * c) = pk;
  }
}

__global__ void standardize_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ inv_row,
                                   const float* __restrict__ mean, const float* __restrict__ rstd, int64_t n, int d4,
                                   __nv_bfloat16* __restrict__ out, int64_t ldo) {
  standardize_body(x, ldx, inv_row, mean, rstd, n, d4, out, ldo);
}
// both views: blockIdx.y = view; outputs `out_view_stride` elements apart
__global__ void standardize_x2_kernel(TwoViews v, TwoStats st, int64_t n, int d4, __nv_bfloat16* __restrict__ out,
                                      int64_t out_view_stride, int64_t ldo) {
  const bool second = blockIdx.y != 0;
  standardize_body(second ? v.x1 : v.x0, second ? v.ld1 : v.ld0, second ? v.inv1 : v.inv0, second ? st.mean1 : st.mean0,
                   second ? st.rstd1 : st.rstd0, n, d4, out + (second ? out_view_stride : 0), ldo);
}

// one block per row: dx^ = (dT - m1 - x~ m2) * rstd * grad_out, then (optionally) the row-normalise backward.
// float4 traffic throughout (d % 8 == 0 and 16-byte aligned rows are checked by the entry points).
__device__ __forceinline__ float4 barlow_g4(const float4 xv, const float4 dtv, const float4 mu, const float4 rs,
                                            const float4 a1, const float4 a2, float sc, float go, float4* xh_out) {
  float4 xh = make_float4(xv.x * sc, xv.y * sc, xv.z * sc, xv.w * sc);
  if (xh_out) *xh_out = xh;
  float4 g;
  g.x = (dtv.x - a1.x - (xh.x - mu.x) * rs.x * a2.x) * rs.x * go;
  g.y = (dtv.y - a1.y - (xh.y - mu.y) * rs.y * a2.y) * rs.y * go;
  g.z = (dtv.z - a1.z - (xh.z - mu.z) * rs.z * a2.z) * rs.z * go;
  g.w = (dtv.w - a1.w - (xh.w - mu.w) * rs.w * a2.w) * rs.w * go;
  return g;
}
__device__ __forceinline__ void barlow_finish_body(const float* __restrict__ x, int64_t ldx, const float* __restrict__ inv_row,
                                                   const float* __restrict__ mean, const float* __restrict__ rstd,
                                                   const float* __restrict__ dt, int64_t lddt, const float* __restrict__ m1,
                                                   const float* __restrict__ m2, int d, const float* __restrict__ grad_out,
                                                   float* __restrict__ dx, int64_t lddx) {
  const int64_t r = blockIdx.x;
  const float go = __ldg(grad_out);
  const float sc = inv_row ? inv_row[r] : 1.f;
  const int d4 = d >> 2;
  const float4* x4 = reinterpret_cast<const float4*>(x + r * ldx);
  const float4* dt4 = reinterpret_cast<const float4*>(dt + r * lddt);
  const float4* mu4 = reinterpret_cast<const float4*>(mean);
  const float4* rs4 = reinterpret_cast<const float4*>(rstd);
  const float4* a14 = reinterpret_cast<const float4*>(m1);
  const float4* a24 = reinterpret_cast<const float4*>(m2);
  float4* dx4 = reinterpret_cast<float4*>(dx + r * lddx);
  __shared__ float red[32];
  float dot = 0.f;
  if (inv_row) {
    for (int c = threadIdx.x; c < d4; c += blockDim.x) {
      float4 xh;
      const float4 g = barlow_g4(__ldg(x4 + c), __ldg(dt4 + c), __ldg(mu4 + c), __ldg(rs4 + c), __ldg(a14 + c),
                                 __ldg(a24 + c), sc, go, &xh);
      dot += (g.x * xh.x + g.y * xh.y) + (g.z * xh.z + g.w * xh.w);
    }
    dot = warp_sum(dot);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = dot;
    __syncthreads();
    float t = (threadIdx.x & 31) < (blockDim.x >> 5) ? red[threadIdx.x & 31] : 0.f;
    dot = warp_sum(t);
  }
  for (int c = threadIdx.x; c < d4; c += blockDim.x) {
    float4 xh;
    float4 g = barlow_g4(__ldg(x4 + c), __ldg(dt4 + c), __ldg(mu4 + c), __ldg(rs4 + c), __ldg(a14 + c), __ldg(a24 + c),
                         sc, go, &xh);
    if (inv_row) {
      g.x = (g.x - dot * xh.x) * sc; g.y = (g.y - dot * xh.y) * sc;
      g.z = (g.z - dot * xh.z) * sc; g.w = (g.w - dot * xh.w) * sc;
    }
    dx4[c] = g;
  }
}

__global__ void barlow_finish_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ inv_row,
                                     const float* __restrict__ mean, const float* __restrict__ rstd,
                                     const float* __restrict__ dt, int64_t lddt, const float* __restrict__ m1,
                                     const float* __restrict__ m2, int d, const float* __restrict__ grad_out,
                                     float* __restrict__ dx, int64_t lddx) {
  barlow_finish_body(x, ldx, inv_row, mean, rstd, dt, lddt, m1, m2, d, grad_out, dx, lddx);
}
// both views in one launch: blockIdx.y = view; colred = [m1_i | m2_i | m1_j | m2_j]
struct TwoGrads {
  const float *dt0, *dt1;  // [n x d] fp32, leading dimension lddt
  float *dx0, *dx1;
  int64_t lddx0, lddx1;
};
__global__ void barlow_finish_x2_kernel(TwoViews v, TwoStats st, TwoGrads g, int64_t lddt, const float* __restrict__ colred,
                                        int d, const float* __restrict__ grad_out) {
  const bool second = blockIdx.y != 0;
  const float* cr = colred + (second ? 2 * static_cast<int64_t>(d) : 0);
  barlow_finish_body(second ? v.x1 : v.x0, second ? v.ld1 : v.ld0, second ? v.inv1 : v.inv0, second ? st.mean1 : st.mean0,
                     second ? st.rstd1 : st.rstd0, second ? g.dt1 : g.dt0, lddt, cr, cr + d, d, grad_out,
                     second ? g.dx1 : g.dx0, second ? g.lddx1 : g.lddx0);
}


// ---- distributed (batch rows sharded over ranks) -------------------------------------------------------------
// local column statistics of one rank: out0 = local mean, out1 = local M2 = sum_r (x - mean_local)^2
__global__ void col_local_moments_kernel(const float* __restrict__ part, int nsplit, const float* __restrict__ x,
                                         const float* __restrict__ inv_row, int64_t n, int d, float* __restrict__ out0,
                                         float* __restrict__ out1) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= d) return;
  float s1 = 0.f, s2 = 0.f;
  for (int i = 0; i < nsplit; ++i) {
    s1 += part[(static_cast<int64_t>(i) * 2 + 0) * d + col];
    s2 += part[(static_cast<int64_t>(i) * 2 + 1) * d + col];
  }
  const float fn = static_cast<float>(n);
  const float v0 = x[col] * (inv_row ? inv_row[0] : 1.f);
  out0[col] = v0 + s1 / fn;
  out1[col] = fmaxf(s2 - s1 * s1 / fn, 0.f);
}

// Chan's pairwise combination of the per-rank (count, mean, M2) in RANK ORDER (identical on every rank) ->
// global mean and 1/std (unbiased over n_global = world * n_local rows).  stats_all: [world][2 views][2][d].
__global__ void col_combine_moments_kernel(const float* __restrict__ stats_all, int world, int64_t n_local, int d,
                                           int view, float* __restrict__ mean, float* __restrict__ rstd) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= d) return;
  const float nb = static_cast<float>(n_local);
  float na = 0.f, mu = 0.f, m2 = 0.f;
  for (int r = 0; r < world; ++r) {
    const float* blk = stats_all + (static_cast<int64_t>(r) * 2 + view) * 2 * d;
    const float mb = blk[col], m2b = blk[d + col];
    const float nt = na + nb, delta = mb - mu;
    mu += delta * (nb / nt);
    m2 += m2b + delta * delta * (na * nb / nt);
    na = nt;
  }
  mean[col] = mu;
  rstd[col] = rsqrtf(m2 / (na - 1.f));
}

// loss terms + dC (bf16) for `rows` rows (global rows row0 ..) of the SUMMED cross-correlation matrix
__global__ void xcorr_epilogue_kernel(const float* __restrict__ c, int64_t ldc, int64_t row0, int64_t rows, int d4,
                                      float lambda, __nv_bfloat16* __restrict__ dC, int64_t ld_dc,
                                      float* __restrict__ part) {
  float acc = 0.f;
  const int64_t total = rows * d4;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = i / d4;
    const int c4 = static_cast<int>(i - r * d4);
    const float4 v = __ldg(reinterpret_cast<const float4*>(c + r * ldc) + c4);
    const float e[4] = {v.x, v.y, v.z, v.w};
    float g[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const bool diag = (row0 + r) == static_cast<int64_t>(4 * c4 + j);
      const float t = diag ? e[j] - 1.f : e[j];
      const float w = diag ? 1.f : lambda;
      acc = fmaf(w * t, t, acc);
      g[j] = 2.f * w * t;
    }
    __nv_bfloat162 lo = __floats2bfloat162_rn(g[0], g[1]), hi = __floats2bfloat162_rn(g[2], g[3]);
    uint2 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&lo);
    pk.y = *reinterpret_cast<uint32_t*>(&hi);
    *reinterpret_cast<uint2*>(dC + r * ld_dc + 4 * c4) = pk;
  }
  __shared__ float red[32];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) part[blockIdx.x] = t;
  }
}

// raw column sums of the backward reductions: out0 = sum_0 dT, out1 = sum_0 dT x~  (local rows; all-reduced by the caller)
__global__ void col_sum_partials_kernel(const float* __restrict__ part, int nsplit, int d, float* __restrict__ out0,
                                        float* __restrict__ out1) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= d) return;
  float s1 = 0.f, s2 = 0.f;
  for (int i = 0; i < nsplit; ++i) {
    s1 += part[(static_cast<int64_t>(i) * 2 + 0) * d + col];
    s2 += part[(static_cast<int64_t>(i) * 2 + 1) * d + col];
  }
  out0[col] = s1;
  out1[col] = s2;
}
// m1 = sum / n_global, m2 = sum / (n_global - 1) for the 2 views x 2 reductions: colsum [2][2][d] -> colred [2][2][d]
__global__ void col_scale_sums_kernel(const float* __restrict__ colsum, int d, float inv_n, float inv_nm1,
                                      float* __restrict__ colred) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 4 * d) return;
  colred[i] = colsum[i] * (((i / d) & 1) ? inv_nm1 : inv_n);
}


// ---- column-sharded variant (all-gather of the standardised rows instead of an all-reduce of C) -------------------
// column sums over ALL n rows of a [n x ncols] fp32 slab dT and of dT * x~ (x~ = bf16 gathered rows, columns
// col0.. of a [n x ldx] matrix); same (32 columns, 8 row phases) x row-stripe layout as col_partials_kernel.
__global__ void slab_col_partials_kernel(const float* __restrict__ dt, int64_t lddt, const __nv_bfloat16* __restrict__ xt,
                                         int64_t ldx, int64_t n, int ncols, float* __restrict__ part) {
  const int col = blockIdx.x * kColsPerBlock + threadIdx.x;
  const int stripe = blockIdx.y;
  const int64_t rows_per = (n + gridDim.y - 1) / gridDim.y;
  const int64_t r0 = stripe * rows_per, r1 = min(n, r0 + rows_per);
  float s1 = 0.f, s2 = 0.f;
  if (col < ncols) {
    for (int64_t r = r0 + threadIdx.y; r < r1; r += blockDim.y) {
      const float g = dt[r * lddt + col];
      s1 += g;
      s2 = fmaf(g, __bfloat162float(xt[r * ldx + col]), s2);
    }
  }
  __shared__ float sh1[8][kColsPerBlock + 1], sh2[8][kColsPerBlock + 1];
  sh1[threadIdx.y][threadIdx.x] = s1;
  sh2[threadIdx.y][threadIdx.x] = s2;
  __syncthreads();
  if (threadIdx.y == 0 && col < ncols) {
    float a = 0.f, b = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { a += sh1[i][threadIdx.x]; b += sh2[i][threadIdx.x]; }
    part[(static_cast<int64_t>(stripe) * 2 + 0) * ncols + col] = a;
    part[(static_cast<int64_t>(stripe) * 2 + 1) * ncols + col] = b;
  }
}
// in place: dt[r, c] = (dt - m1_c - x~ m2_c) * rstd_c * grad_out, m1 = sum1 / n, m2 = sum2 / (n - 1)
__global__ void slab_finish_kernel(float* __restrict__ dt, int64_t lddt, const __nv_bfloat16* __restrict__ xt, int64_t ldx,
                                   const float* __restrict__ rstd, const float* __restrict__ part, int nsplit, int64_t n,
                                   int ncols, const float* __restrict__ grad_out) {
  const int col = blockIdx.x * kColsPerBlock + threadIdx.x;
  if (col >= ncols) return;
  float s1 = 0.f, s2 = 0.f;
  for (int i = 0; i < nsplit; ++i) {
    s1 += part[(static_cast<int64_t>(i) * 2 + 0) * ncols + col];
    s2 += part[(static_cast<int64_t>(i) * 2 + 1) * ncols + col];
  }
  const float m1 = s1 / static_cast<float>(n), m2 = s2 / static_cast<float>(n - 1);
  const float sc = rstd[col] * __ldg(grad_out);
  const int64_t rows_per = (n + gridDim.y - 1) / gridDim.y;
  const int64_t r0 = blockIdx.y * rows_per, r1 = min(n, r0 + rows_per);
  for (int64_t r = r0 + threadIdx.y; r < r1; r += blockDim.y) {
    const float g = dt[r * lddt + col];
    dt[r * lddt + col] = (g - m1 - __bfloat162float(xt[r * ldx + col]) * m2) * sc;
  }
}
// dx[n, q * ncols + c] = recv[q][n][c]  (+ row-normalise backward with x, inv_row); one block per local row
__global__ void slab_gather_rows_kernel(const float* __restrict__ recv, int world, int64_t n_local, int ncols,
                                        const float* __restrict__ x, int64_t ldx, const float* __restrict__ inv_row,
                                        float* __restrict__ dx, int64_t lddx) {
  const int64_t r = blockIdx.x;
  const int d = world * ncols;
  __shared__ float red[32];
  float dot = 0.f;
  const float sc = inv_row ? inv_row[r] : 1.f;
  if (inv_row) {
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
      const int q = c / ncols, cc = c - q * ncols;
      dot = fmaf(recv[(static_cast<int64_t>(q) * n_local + r) * ncols + cc], x[r * ldx + c] * sc, dot);
    }
    dot = warp_sum(dot);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = dot;
    __syncthreads();
    float t = (threadIdx.x & 31) < (blockDim.x >> 5) ? red[threadIdx.x & 31] : 0.f;
    dot = warp_sum(t);
  }
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    const int q = c / ncols, cc = c - q * ncols;
    float g = recv[(static_cast<int64_t>(q) * n_local + r) * ncols + cc];
    if (inv_row) g = (g - dot * x[r * ldx + c] * sc) * sc;
    dx[r * lddx + c] = g;
  }
}

int check_rows(const void* p, int64_t ld) {
  if (!p) return SSVB_ERR_INVALID;
  if ((reinterpret_cast<uintptr_t>(p) & 15) || (ld & 3)) return SSVB_ERR_ALIGNMENT;
  return SSVB_OK;
}
int check_shape(int64_t n, int64_t d) {
  if (n < 2 || d <= 0) return SSVB_ERR_INVALID;
  if (d % 8) return SSVB_ERR_ALIGNMENT;  // bf16 rows of x~ [n x d] and dC [d x d] must be 16-byte multiples
  if (n > (1 << 30) || d > (1 << 20)) return SSVB_ERR_UNSUPPORTED;
  return SSVB_OK;
}

// Closed-form backward of the batch standardisation.  With x~ = (x - mean) / std (unbiased) and dT = dL/dx~:
//   dx = (dT - mean_n(dT) - x~ * sum_n(dT x~) / (n - 1)) / std.
// Here dTi[n, a] = sum_b x~j[n, b] dC[a, b] / n, so mean_n(dTi[., a]) = sum_b dC[a, b] mean_n(x~j[., b]) = 0 (standardised
// columns have zero mean) and sum_n(dTi[n, a] x~i[n, a]) = sum_b dC[a, b] C[a, b]: both column statistics of the backward
// are known after the FORWARD GEMM - row sums (view i) / column sums (view j) of dC .* C, taken in its epilogue.  The
// backward GEMM epilogue can then turn each dT tile into the input gradient on its way out of TMEM: no fp32 dT round trip
// (2 x 67 MB written + read at 2048 x 8192), no column reduction, no finish pass.
// This kernel: blocks [0, ceil(d/32)) combine the partial sums in fixed order into q_i = rstd_i * m2_i, q_j = rstd_j * m2_j;
// the last block sums the loss partials (was sum_partials_kernel).
__global__ void barlow_fwd_finish_kernel(const float* __restrict__ xrow, int nrow, const float* __restrict__ xcol, int ncol,
                                         int d, float inv_nm1, const float* __restrict__ rstd_i,
                                         const float* __restrict__ rstd_j, float* __restrict__ q_i, float* __restrict__ q_j,
                                         const float* __restrict__ loss_part, int nloss, float* __restrict__ loss) {
  constexpr int kPh = 32;  // block (32 columns x 32 partial-row phases)
  __shared__ float sh1[kPh][33], sh2[kPh][33];
  const int tid = threadIdx.y * 32 + threadIdx.x;
  if (blockIdx.x == gridDim.x - 1) {
    float v = 0.f;
    for (int i = tid; i < nloss; i += 32 * kPh) v += loss_part[i];
    v = warp_sum(v);
    if (threadIdx.x == 0) sh1[threadIdx.y][0] = v;
    __syncthreads();
    if (tid == 0) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < kPh; ++i) t += sh1[i][0];
      loss[0] = t;
    }
    return;
  }
  const int col = blockIdx.x * 32 + threadIdx.x;
  float s1 = 0.f, s2 = 0.f;
  if (col < d) {
    for (int i = threadIdx.y; i < nrow; i += kPh) s1 += xrow[static_cast<int64_t>(i) * d + col];
#pragma unroll 8
    for (int i = threadIdx.y; i < ncol; i += kPh) s2 += xcol[static_cast<int64_t>(i) * d + col];
  }
  sh1[threadIdx.y][threadIdx.x] = s1;
  sh2[threadIdx.y][threadIdx.x] = s2;
  __syncthreads();
  if (threadIdx.y == 0 && col < d) {
    float a = 0.f, b = 0.f;
#pragma unroll
    for (int i = 0; i < kPh; ++i) { a += sh1[i][threadIdx.x]; b += sh2[i][threadIdx.x]; }
    q_i[col] = a * inv_nm1 * rstd_i[col];
    q_j[col] = b * inv_nm1 * rstd_j[col];
  }
}

// forward pre-pass of BOTH views in three launches (statistics, finalize, standardize); `xi` heads the two standardised
// operands (`x_view_stride` elements apart)
int standardize_both_views(const float* zi, int64_t ld_zi, const float* zj, int64_t ld_zj, int normalize, int64_t n,
                           int64_t d, float* inv_i, float* inv_j, TwoStats st, __nv_bfloat16* xi, int64_t x_view_stride,
                           float* colpart, int64_t part_view_stride, cudaStream_t s) {
  TwoViews v{zi, zj, ld_zi, ld_zj, nullptr, nullptr};
  if (normalize) {
    row_invnorm_kernel<<<static_cast<unsigned>(ceil_div(n, 8)), 256, 0, s>>>(zi, n, static_cast<int>(d), ld_zi, inv_i);
    SSVB_LAUNCH_CHECK();
    row_invnorm_kernel<<<static_cast<unsigned>(ceil_div(n, 8)), 256, 0, s>>>(zj, n, static_cast<int>(d), ld_zj, inv_j);
    SSVB_LAUNCH_CHECK();
    v.inv0 = inv_i;
    v.inv1 = inv_j;
  }
  dim3 grid(static_cast<unsigned>(ceil_div(d, 128)), kStatSplit, 2), block(32, 8);
  col_stats4_x2_kernel<<<grid, block, 0, s>>>(v, n, static_cast<int>(d), colpart, part_view_stride);
  SSVB_LAUNCH_CHECK();
  col_finalize_x2_kernel<<<dim3(static_cast<unsigned>(ceil_div(d, 32)), 2), dim3(32, 8), 0, s>>>(colpart, part_view_stride,
                                                                                                 kStatSplit, v, n,
                                                                                                 static_cast<int>(d), st);
  SSVB_LAUNCH_CHECK();
  const int64_t total = n * (d / 4);
  int64_t g = ceil_div(total, 256 * 4);
  const int64_t cap = static_cast<int64_t>(num_sms()) * 8;  // x 2 views = 16 resident-CTA waves' worth
  if (g > cap) g = cap;
  standardize_x2_kernel<<<dim3(static_cast<unsigned>(g), 2), 256, 0, s>>>(v, st, n, static_cast<int>(d / 4), xi, x_view_stride,
                                                                        d);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

}  // namespace

extern "C" {

size_t ssvb_barlow_saved_bytes(int64_t n, int64_t d) {
  if (n <= 0 || d <= 0) return 0;
  return barlow_saved(nullptr, n, d).bytes;
}
size_t ssvb_barlow_workspace_bytes(int64_t n, int64_t d) {
  if (n <= 0 || d <= 0) return 0;
  return barlow_ws(nullptr, n, d).bytes;
}

int ssvb_barlow_fwd(const float* zi, const float* zj, int64_t n, int64_t d, int64_t ld_zi, int64_t ld_zj,
                    int normalize, float lambda, float* loss, void* saved, void* workspace, size_t workspace_bytes,
                    void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(check_shape(n, d));
  SSVB_TRY(check_rows(zi, ld_zi));
  SSVB_TRY(check_rows(zj, ld_zj));
  if (!loss || !saved || !workspace) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_barlow_workspace_bytes(n, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BarlowSaved sv = barlow_saved(saved, n, d);
  BarlowWs ws = barlow_ws(workspace, n, d);
  SSVB_TRY(standardize_both_views(zi, ld_zi, zj, ld_zj, normalize, n, d, sv.inv_i, sv.inv_j,
                                  TwoStats{sv.mean_i, sv.rstd_i, sv.mean_j, sv.rstd_j}, sv.xi, sv.xj - sv.xi, ws.colpart,
                                  ws.view_stride, s));
  // C = Xi~^T Xj~ / n : contraction over the batch axis, both operands MN-major in place
  GemmParams p{};
  p.M = static_cast<int>(d);
  p.N = static_cast<int>(d);
  p.K = static_cast<int>(n);
  p.alpha = 1.f / static_cast<float>(n);
  p.lambda = lambda;
  p.dC = sv.dC;
  p.ld_dc = d;
  p.loss_partials = ws.loss_partials;
  p.bl_rowpart = ws.xrow;  // dC .* C sums for the closed-form backward (barlow_fwd_finish_kernel)
  p.bl_colpart = ws.xcol;
  SSVB_TRY(launch_gemm({sv.xi, d, true}, {sv.xj, d, true}, p, 256, EPI_BARLOW, kMaxGemmCtas, s));
  // every launched CTA wrote its partial (persistent kernel, grid = min(tiles, SMs)): sum exactly those, no memset
  barlow_fwd_finish_kernel<<<static_cast<unsigned>(ceil_div(d, 32) + 1), dim3(32, 32), 0, s>>>(
      ws.xrow, static_cast<int>(ceil_div(d, 256)), ws.xcol, static_cast<int>(ceil_div(d, 128) * 4), static_cast<int>(d),
      1.f / static_cast<float>(n - 1), sv.rstd_i, sv.rstd_j, sv.q_i, sv.q_j, ws.loss_partials,
      gemm_grid(ceil_div(d, 128) * ceil_div(d, 256), kMaxGemmCtas), loss);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

int ssvb_barlow_bwd(const float* zi, const float* zj, int64_t n, int64_t d, int64_t ld_zi, int64_t ld_zj,
                    int normalize, float lambda, const float* grad_out, const void* saved, float* dzi, float* dzj,
                    int64_t ld_dzi, int64_t ld_dzj, void* workspace, size_t workspace_bytes, void* stream) {
  (void)lambda;
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(check_shape(n, d));
  SSVB_TRY(check_rows(zi, ld_zi));
  SSVB_TRY(check_rows(zj, ld_zj));
  SSVB_TRY(check_rows(dzi, ld_dzi));
  SSVB_TRY(check_rows(dzj, ld_dzj));
  if (!grad_out || !saved || !workspace) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_barlow_workspace_bytes(n, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BarlowSaved sv = barlow_saved(const_cast<void*>(saved), n, d);
  BarlowWs ws = barlow_ws(workspace, n, d);

  GemmParams p{};
  p.M = static_cast<int>(n);
  p.N = static_cast<int>(d);
  p.K = static_cast<int>(d);
  p.alpha = 1.f / static_cast<float>(n);
  p.ldc = d;
  // dTi[n, a] = sum_b Xj~[n, b] dC[a, b]          (A K-major, B = dC rows K-major)
  // dTj[n, b] = sum_a Xi~[n, a] dC[a, b]          (A K-major, B = dC consumed MN-major)
  // ONE launch for both (a shared persistent tile queue: 2 x 512 tiles = 6.9 waves of 148 CTAs instead of 2 x 3.46),
  // and the epilogue leaves the column partials sum_n dT, sum_n dT x~ per (row tile, warp) beside the output
  const float* inv_i = normalize ? sv.inv_i : nullptr;
  const float* inv_j = normalize ? sv.inv_j : nullptr;
  if (!normalize && gemm_tma_store_allowed()) {
    // closed-form standardisation backward inside the GEMM epilogue (see barlow_fwd_finish_kernel): the two GEMMs write
    // dzi / dzj directly (rows are 16-byte aligned: check_rows above).  normalize = 1 also needs a per-row dot with the
    // finished gradient and keeps the dT + finish-kernel path below.
    p.out = dzi;
    p.ldc = ld_dzi;
    p.out2 = dzj;
    p.ldc2 = ld_dzj;
    p.xf = zi;  // x~ is rebuilt from the fp32 inputs: the bf16 operand copy would add 2^-9 to a term that largely cancels dT
    p.ldxf = ld_zi;
    p.xf2 = zj;
    p.ldxf2 = ld_zj;
    p.vm = sv.mean_i;
    p.vr = sv.rstd_i;
    p.vq = sv.q_i;
    p.vm2 = sv.mean_j;
    p.vr2 = sv.rstd_j;
    p.vq2 = sv.q_j;
    p.go = grad_out;
    const GemmOperand a2f{sv.xi, d, false}, b2f{sv.dC, d, true};
    return launch_gemm({sv.xj, d, false}, {sv.dC, d, false}, p, 256, EPI_BARLOW_BWD, 0, s, false, &a2f, &b2f);
  }
  float* part_i = ws.colpart;
  float* part_j = ws.colpart + ws.view_stride;
  int nsplit = fused_stripes(n);
  p.out = ws.dti;
  p.out2 = ws.dtj;
  if (nsplit && gemm_tma_store_allowed()) {
    p.colpart = part_i;
    p.colpart2 = part_j;
    p.xt = sv.xi;
    p.xt2 = sv.xj;
    p.ldx = d;
  } else {
    nsplit = 0;
  }
  const GemmOperand a2{sv.xi, d, false}, b2{sv.dC, d, true};
  SSVB_TRY(launch_gemm({sv.xj, d, false}, {sv.dC, d, false}, p, 256, EPI_STORE_F32, 0, s, false, &a2, &b2));
  if (!nsplit) {
    nsplit = kRowSplit;
    dim3 grid(static_cast<unsigned>(ceil_div(d, kColsPerBlock)), kRowSplit), block(32, 8);
    col_partials_kernel<1><<<grid, block, 0, s>>>(zi, ld_zi, inv_i, ws.dti, d, sv.mean_i, sv.rstd_i, n, static_cast<int>(d), part_i);
    SSVB_LAUNCH_CHECK();
    col_partials_kernel<1><<<grid, block, 0, s>>>(zj, ld_zj, inv_j, ws.dtj, d, sv.mean_j, sv.rstd_j, n, static_cast<int>(d), part_j);
    SSVB_LAUNCH_CHECK();
  }
  const unsigned fgrid = static_cast<unsigned>(ceil_div(d, 32));
  // both views per launch (colred = [mean dTi | sum dTi x~i | mean dTj | sum dTj x~j])
  col_finalize_wide_kernel<<<dim3(fgrid, 2), dim3(32, 8), 0, s>>>(part_i, nsplit, n, static_cast<int>(d), ws.colred,
                                                                  ws.colred + d, ws.view_stride);
  SSVB_LAUNCH_CHECK();
  barlow_finish_x2_kernel<<<dim3(static_cast<unsigned>(n), 2), 256, 0, s>>>(
      TwoViews{zi, zj, ld_zi, ld_zj, inv_i, inv_j}, TwoStats{sv.mean_i, sv.rstd_i, sv.mean_j, sv.rstd_j},
      TwoGrads{ws.dti, ws.dtj, dzi, dzj, ld_dzi, ld_dzj}, d, ws.colred, static_cast<int>(d), grad_out);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

// ------------------------------------------------------------------------------------------------------------
// Distributed Barlow Twins (SURVEY.md §8e): batch rows sharded over `world` ranks, n_local rows each; semantics =
// BarlowLoss on the rank-order concatenation (n_global = world * n_local rows).  See include/ssv_b200.h.
// ------------------------------------------------------------------------------------------------------------
size_t ssvb_barlow_dist_saved_bytes(int64_t n_local, int64_t d) {
  if (n_local <= 0 || d <= 0) return 0;
  return barlow_dist_saved(nullptr, n_local, d).bytes;
}
size_t ssvb_barlow_dist_workspace_bytes(int64_t n_local, int64_t d) {
  if (n_local <= 0 || d <= 0) return 0;
  return barlow_dist_ws(nullptr, n_local, d).bytes;
}

int ssvb_barlow_dist_stats(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi, int64_t ld_zj,
                           int normalize, float* stats_local, void* saved, void* workspace, size_t workspace_bytes,
                           void* stream) {
  SSVB_TRY(check_device_sm100());
  if (n_local < 1 || d <= 0) return SSVB_ERR_INVALID;
  if (d % 8) return SSVB_ERR_ALIGNMENT;
  SSVB_TRY(check_rows(zi, ld_zi));
  SSVB_TRY(check_rows(zj, ld_zj));
  if (!stats_local || !saved || !workspace) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_barlow_dist_workspace_bytes(n_local, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BarlowDistSaved sv = barlow_dist_saved(saved, n_local, d);
  BarlowDistWs ws = barlow_dist_ws(workspace, n_local, d);
  const int di = static_cast<int>(d);
  dim3 grid(static_cast<unsigned>(ceil_div(d, kColsPerBlock)), kRowSplit), block(32, 8);
  for (int v = 0; v < 2; ++v) {
    const float* x = v ? zj : zi;
    const int64_t ld = v ? ld_zj : ld_zi;
    float* inv_row = v ? sv.inv_j : sv.inv_i;
    const float* inv = nullptr;
    if (normalize) {
      row_invnorm_kernel<<<static_cast<unsigned>(ceil_div(n_local, 8)), 256, 0, s>>>(x, n_local, di, ld, inv_row);
      SSVB_LAUNCH_CHECK();
      inv = inv_row;
    }
    float* part = ws.colpart + v * kRowSplit * 2 * d;
    col_partials_kernel<0><<<grid, block, 0, s>>>(x, ld, inv, nullptr, 0, nullptr, nullptr, n_local, di, part);
    SSVB_LAUNCH_CHECK();
    col_local_moments_kernel<<<static_cast<unsigned>(ceil_div(d, 256)), 256, 0, s>>>(
        part, kRowSplit, x, inv, n_local, di, stats_local + (v * 2 + 0) * d, stats_local + (v * 2 + 1) * d);
    SSVB_LAUNCH_CHECK();
  }
  return SSVB_OK;
}

int ssvb_barlow_dist_xcorr(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi, int64_t ld_zj,
                           int normalize, const float* stats_all, int64_t world, float* c_partial, void* saved,
                           void* stream) {
  SSVB_TRY(check_device_sm100());
  if (n_local < 1 || d <= 0 || world < 1 || n_local * world < 2) return SSVB_ERR_INVALID;
  if (d % 8) return SSVB_ERR_ALIGNMENT;
  SSVB_TRY(check_rows(zi, ld_zi));
  SSVB_TRY(check_rows(zj, ld_zj));
  SSVB_TRY(check_rows(c_partial, d));
  if (!stats_all || !saved) return SSVB_ERR_INVALID;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BarlowDistSaved sv = barlow_dist_saved(saved, n_local, d);
  const int di = static_cast<int>(d);
  const unsigned cgrid = static_cast<unsigned>(ceil_div(d, 256));
  col_combine_moments_kernel<<<cgrid, 256, 0, s>>>(stats_all, static_cast<int>(world), n_local, di, 0, sv.mean_i, sv.rstd_i);
  SSVB_LAUNCH_CHECK();
  col_combine_moments_kernel<<<cgrid, 256, 0, s>>>(stats_all, static_cast<int>(world), n_local, di, 1, sv.mean_j, sv.rstd_j);
  SSVB_LAUNCH_CHECK();
  const int64_t total = n_local * (d / 4);
  int64_t g = ceil_div(total, 256 * 4);
  const int64_t cap = static_cast<int64_t>(num_sms()) * 16;
  if (g > cap) g = cap;
  standardize_kernel<<<static_cast<unsigned>(g), 256, 0, s>>>(zi, ld_zi, normalize ? sv.inv_i : nullptr, sv.mean_i,
                                                              sv.rstd_i, n_local, static_cast<int>(d / 4), sv.xi, d);
  SSVB_LAUNCH_CHECK();
  standardize_kernel<<<static_cast<unsigned>(g), 256, 0, s>>>(zj, ld_zj, normalize ? sv.inv_j : nullptr, sv.mean_j,
                                                              sv.rstd_j, n_local, static_cast<int>(d / 4), sv.xj, d);
  SSVB_LAUNCH_CHECK();
  // partial C_r = Xi~_r^T Xj~_r / n_global (fp32, summed over ranks by the caller's collective)
  GemmParams p{};
  p.M = di;
  p.N = di;
  p.K = static_cast<int>(n_local);
  p.alpha = 1.f / static_cast<float>(n_local * world);
  p.out = c_partial;
  p.ldc = d;
  SSVB_TRY(launch_gemm({sv.xi, d, true}, {sv.xj, d, true}, p, 256, EPI_STORE_F32, 0, s));
  return SSVB_OK;
}

int ssvb_barlow_dist_epilogue(const float* c_rows, int64_t row0, int64_t rows, int64_t d, float lambda, void* dC_rows,
                              float* loss_partial, void* workspace, size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  if (rows <= 0 || d <= 0 || row0 < 0 || row0 + rows > d) return SSVB_ERR_INVALID;
  if (d % 8) return SSVB_ERR_ALIGNMENT;
  SSVB_TRY(check_rows(c_rows, d));
  if (!dC_rows || !loss_partial || !workspace) return SSVB_ERR_INVALID;
  if (reinterpret_cast<uintptr_t>(dC_rows) & 15) return SSVB_ERR_ALIGNMENT;
  if (workspace_bytes < static_cast<size_t>(kEpiGridMax) * sizeof(float)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float* part = static_cast<float*>(workspace);
  int64_t g = ceil_div(rows * (d / 4), 256 * 4);
  if (g > kEpiGridMax) g = kEpiGridMax;
  xcorr_epilogue_kernel<<<static_cast<unsigned>(g), 256, 0, s>>>(c_rows, d, row0, rows, static_cast<int>(d / 4), lambda,
                                                                 static_cast<__nv_bfloat16*>(dC_rows), d, part);
  SSVB_LAUNCH_CHECK();
  sum_partials_kernel<<<1, 256, 0, s>>>(part, static_cast<int>(g), 1.f, loss_partial);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

int ssvb_barlow_dist_bwd_gemm(const float* zi, const float* zj, int64_t n_local, int64_t n_global, int64_t d,
                              int64_t ld_zi, int64_t ld_zj, int normalize, const void* dC, const void* saved,
                              float* colsum_local, void* workspace, size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  if (n_local < 1 || n_global < 2 || n_global < n_local || d <= 0) return SSVB_ERR_INVALID;
  if (d % 8) return SSVB_ERR_ALIGNMENT;
  SSVB_TRY(check_rows(zi, ld_zi));
  SSVB_TRY(check_rows(zj, ld_zj));
  if (!dC || !saved || !colsum_local || !workspace) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_barlow_dist_workspace_bytes(n_local, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BarlowDistSaved sv = barlow_dist_saved(const_cast<void*>(saved), n_local, d);
  BarlowDistWs ws = barlow_dist_ws(workspace, n_local, d);
  const int di = static_cast<int>(d);
  GemmParams p{};
  p.M = static_cast<int>(n_local);
  p.N = di;
  p.K = di;
  p.alpha = 1.f / static_cast<float>(n_global);
  p.ldc = d;
  p.out = ws.dti;  // dTi[n, a] = sum_b Xj~[n, b] dC[a, b]
  SSVB_TRY(launch_gemm({sv.xj, d, false}, {dC, d, false}, p, 256, EPI_STORE_F32, 0, s));
  p.out = ws.dtj;  // dTj[n, b] = sum_a Xi~[n, a] dC[a, b]
  SSVB_TRY(launch_gemm({sv.xi, d, false}, {dC, d, true}, p, 256, EPI_STORE_F32, 0, s));
  dim3 grid(static_cast<unsigned>(ceil_div(d, kColsPerBlock)), kRowSplit), block(32, 8);
  const unsigned fgrid = static_cast<unsigned>(ceil_div(d, 256));
  for (int v = 0; v < 2; ++v) {
    float* part = ws.colpart + v * kRowSplit * 2 * d;
    col_partials_kernel<1><<<grid, block, 0, s>>>(v ? zj : zi, v ? ld_zj : ld_zi,
                                                  normalize ? (v ? sv.inv_j : sv.inv_i) : nullptr, v ? ws.dtj : ws.dti, d,
                                                  v ? sv.mean_j : sv.mean_i, v ? sv.rstd_j : sv.rstd_i, n_local, di, part);
    SSVB_LAUNCH_CHECK();
    col_sum_partials_kernel<<<fgrid, 256, 0, s>>>(part, kRowSplit, di, colsum_local + (v * 2 + 0) * d,
                                                  colsum_local + (v * 2 + 1) * d);
    SSVB_LAUNCH_CHECK();
  }
  return SSVB_OK;
}

int ssvb_barlow_dist_bwd_finish(const float* zi, const float* zj, int64_t n_local, int64_t n_global, int64_t d,
                                int64_t ld_zi, int64_t ld_zj, int normalize, const float* colsum_global,
                                const float* grad_out, const void* saved, float* dzi, float* dzj, int64_t ld_dzi,
                                int64_t ld_dzj, void* workspace, size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  if (n_local < 1 || n_global < 2 || n_global < n_local || d <= 0) return SSVB_ERR_INVALID;
  if (d % 8) return SSVB_ERR_ALIGNMENT;
  SSVB_TRY(check_rows(zi, ld_zi));
  SSVB_TRY(check_rows(zj, ld_zj));
  SSVB_TRY(check_rows(dzi, ld_dzi));
  SSVB_TRY(check_rows(dzj, ld_dzj));
  if (!colsum_global || !grad_out || !saved || !workspace) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_barlow_dist_workspace_bytes(n_local, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BarlowDistSaved sv = barlow_dist_saved(const_cast<void*>(saved), n_local, d);
  BarlowDistWs ws = barlow_dist_ws(workspace, n_local, d);
  const int di = static_cast<int>(d);
  col_scale_sums_kernel<<<static_cast<unsigned>(ceil_div(4 * d, 256)), 256, 0, s>>>(
      colsum_global, di, 1.f / static_cast<float>(n_global), 1.f / static_cast<float>(n_global - 1), ws.colred);
  SSVB_LAUNCH_CHECK();
  barlow_finish_kernel<<<static_cast<unsigned>(n_local), 256, 0, s>>>(
      zi, ld_zi, normalize ? sv.inv_i : nullptr, sv.mean_i, sv.rstd_i, ws.dti, d, ws.colred, ws.colred + d, di, grad_out,
      dzi, ld_dzi);
  SSVB_LAUNCH_CHECK();
  barlow_finish_kernel<<<static_cast<unsigned>(n_local), 256, 0, s>>>(
      zj, ld_zj, normalize ? sv.inv_j : nullptr, sv.mean_j, sv.rstd_j, ws.dtj, d, ws.colred + 2 * d, ws.colred + 3 * d, di,
      grad_out, dzj, ld_dzj);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

// ------------------------------------------------------------------------------------------------------------
// Column-sharded distributed Barlow (the low-traffic alternative SURVEY.md §8e asks to measure): all-gather the
// standardised bf16 rows (N x D per view) instead of all-reducing the D x D fp32 matrix; rank r owns the column slab
// [col0, col0 + ncols) of C AND of C^T, so both gradient slabs come out complete and only an all-to-all of N*D/G
// floats per view remains.  See include/ssv_b200.h.
// ------------------------------------------------------------------------------------------------------------
int ssvb_barlow_dist_standardize(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi,
                                 int64_t ld_zj, int normalize, const float* stats_all, int64_t world, void* xt_i_slot,
                                 void* xt_j_slot, void* saved, void* stream) {
  SSVB_TRY(check_device_sm100());
  if (n_local < 1 || d <= 0 || world < 1 || n_local * world < 2) return SSVB_ERR_INVALID;
  if (d % 8) return SSVB_ERR_ALIGNMENT;
  SSVB_TRY(check_rows(zi, ld_zi));
  SSVB_TRY(check_rows(zj, ld_zj));
  if (!stats_all || !saved || !xt_i_slot || !xt_j_slot) return SSVB_ERR_INVALID;
  if ((reinterpret_cast<uintptr_t>(xt_i_slot) | reinterpret_cast<uintptr_t>(xt_j_slot)) & 15) return SSVB_ERR_ALIGNMENT;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BarlowDistSaved sv = barlow_dist_saved(saved, n_local, d);
  const int di = static_cast<int>(d);
  const unsigned cgrid = static_cast<unsigned>(ceil_div(d, 256));
  col_combine_moments_kernel<<<cgrid, 256, 0, s>>>(stats_all, static_cast<int>(world), n_local, di, 0, sv.mean_i, sv.rstd_i);
  SSVB_LAUNCH_CHECK();
  col_combine_moments_kernel<<<cgrid, 256, 0, s>>>(stats_all, static_cast<int>(world), n_local, di, 1, sv.mean_j, sv.rstd_j);
  SSVB_LAUNCH_CHECK();
  const int64_t total = n_local * (d / 4);
  int64_t g = ceil_div(total, 256 * 4);
  const int64_t cap = static_cast<int64_t>(num_sms()) * 16;
  if (g > cap) g = cap;
  standardize_kernel<<<static_cast<unsigned>(g), 256, 0, s>>>(zi, ld_zi, normalize ? sv.inv_i : nullptr, sv.mean_i, sv.rstd_i,
                                                              n_local, static_cast<int>(d / 4),
                                                              static_cast<__nv_bfloat16*>(xt_i_slot), d);
  SSVB_LAUNCH_CHECK();
  standardize_kernel<<<static_cast<unsigned>(g), 256, 0, s>>>(zj, ld_zj, normalize ? sv.inv_j : nullptr, sv.mean_j, sv.rstd_j,
                                                              n_local, static_cast<int>(d / 4),
                                                              static_cast<__nv_bfloat16*>(xt_j_slot), d);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

size_t ssvb_barlow_cs_workspace_bytes(int64_t n_global, int64_t d, int64_t ncols) {
  (void)n_global; (void)d;
  if (ncols <= 0) return 0;
  Carver c(nullptr);
  c.take<float>(kMaxGemmCtas);
  c.take<float>(kRowSplit * 2 * ncols);
  return c.used();
}

int ssvb_barlow_cs_fwd(const void* xa_all, const void* xb_all, int64_t n_global, int64_t d, int64_t col0, int64_t ncols,
                       float lambda, void* dc_slab, float* loss_partial, void* workspace, size_t workspace_bytes,
                       void* stream) {
  SSVB_TRY(check_device_sm100());
  if (!xa_all || !xb_all || !dc_slab || !workspace || n_global < 2 || d <= 0 || col0 < 0 || ncols <= 0 || col0 + ncols > d)
    return SSVB_ERR_INVALID;
  if ((d % 8) || (ncols % 8) || (col0 % 8)) return SSVB_ERR_ALIGNMENT;
  if (workspace_bytes < ssvb_barlow_cs_workspace_bytes(n_global, d, ncols)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Carver cv(workspace);
  float* lp = cv.take<float>(kMaxGemmCtas);
  // C[:, col0 .. col0+ncols) = Xa~^T Xb~[:, slab] / n : both operands MN-major in place, contraction over ALL n rows
  GemmParams p{};
  p.M = static_cast<int>(d);
  p.N = static_cast<int>(ncols);
  p.K = static_cast<int>(n_global);
  p.alpha = 1.f / static_cast<float>(n_global);
  p.lambda = lambda;
  p.dC = static_cast<__nv_bfloat16*>(dc_slab);
  p.ld_dc = ncols;
  p.loss_partials = lp;
  p.diag_off = static_cast<int>(col0);
  SSVB_CUDA(cudaMemsetAsync(lp, 0, kMaxGemmCtas * sizeof(float), s));
  SSVB_TRY(launch_gemm({xa_all, d, true}, {static_cast<const __nv_bfloat16*>(xb_all) + col0, d, true}, p, 256, EPI_BARLOW,
                       kMaxGemmCtas, s));
  if (loss_partial) {
    sum_partials_kernel<<<1, 256, 0, s>>>(lp, kMaxGemmCtas, 1.f, loss_partial);
    SSVB_LAUNCH_CHECK();
  }
  return SSVB_OK;
}

int ssvb_barlow_cs_bwd(const void* xa_all, const void* xb_all, const void* dc_slab, int64_t n_global, int64_t d,
                       int64_t col0, int64_t ncols, const void* saved, int64_t n_local, int view_b, const float* grad_out,
                       float* dxb_slab, void* workspace, size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  if (!xa_all || !xb_all || !dc_slab || !saved || !grad_out || !dxb_slab || !workspace || n_global < 2 || d <= 0 ||
      col0 < 0 || ncols <= 0 || col0 + ncols > d || n_local < 1 || (view_b != 0 && view_b != 1))
    return SSVB_ERR_INVALID;
  if ((d % 8) || (ncols % 8) || (col0 % 8)) return SSVB_ERR_ALIGNMENT;
  if (workspace_bytes < ssvb_barlow_cs_workspace_bytes(n_global, d, ncols)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BarlowDistSaved sv = barlow_dist_saved(const_cast<void*>(saved), n_local, d);
  Carver cv(workspace);
  cv.take<float>(kMaxGemmCtas);
  float* part = cv.take<float>(kRowSplit * 2 * ncols);
  // dT[n, c] = sum_k Xa~[n, k] dC[k, c] / n   (A K-major; B = the slab [d x ncols] consumed MN-major)
  GemmParams p{};
  p.M = static_cast<int>(n_global);
  p.N = static_cast<int>(ncols);
  p.K = static_cast<int>(d);
  p.alpha = 1.f / static_cast<float>(n_global);
  p.out = dxb_slab;
  p.ldc = ncols;
  SSVB_TRY(launch_gemm({xa_all, d, false}, {dc_slab, ncols, true}, p, 256, EPI_STORE_F32, 0, s));
  const __nv_bfloat16* xb = static_cast<const __nv_bfloat16*>(xb_all) + col0;
  dim3 grid(static_cast<unsigned>(ceil_div(ncols, kColsPerBlock)), kRowSplit), block(32, 8);
  slab_col_partials_kernel<<<grid, block, 0, s>>>(dxb_slab, ncols, xb, d, n_global, static_cast<int>(ncols), part);
  SSVB_LAUNCH_CHECK();
  slab_finish_kernel<<<grid, block, 0, s>>>(dxb_slab, ncols, xb, d, (view_b ? sv.rstd_j : sv.rstd_i) + col0, part, kRowSplit,
                                            n_global, static_cast<int>(ncols), grad_out);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

int ssvb_barlow_cs_finish(const float* recv, int64_t world, int64_t n_local, int64_t ncols, const float* x, int64_t ld_x,
                          int normalize, const void* saved, int view, float* dx, int64_t ld_dx, void* stream) {
  SSVB_TRY(check_device_sm100());
  if (!recv || !x || !saved || !dx || world < 1 || n_local < 1 || ncols <= 0 || (view != 0 && view != 1))
    return SSVB_ERR_INVALID;
  SSVB_TRY(check_rows(x, ld_x));
  SSVB_TRY(check_rows(dx, ld_dx));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BarlowDistSaved sv = barlow_dist_saved(const_cast<void*>(saved), n_local, world * ncols);
  slab_gather_rows_kernel<<<static_cast<unsigned>(n_local), 256, 0, s>>>(
      recv, static_cast<int>(world), n_local, static_cast<int>(ncols), x, ld_x,
      normalize ? (view ? sv.inv_j : sv.inv_i) : nullptr, dx, ld_dx);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

}  // extern "C"
