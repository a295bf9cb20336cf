// SwAV loss, forward + backward — replaces SwavLoss.forward (reference utils/losses.py:226-235, call site
// models/swav.py:140).
//
//   rows of both views = live batch rows followed by the bank rows (:227-229)
//   scores_v = z_v C^T (:231);  q_v = sinkhorn(scores_v) (no grad, :232);  p_v = log_softmax(scores_v / T) (:233)
//   loss = -1/2 mean_rows( sum_k q_1 p_2 + sum_k q_2 p_1 ) (:234)
//   dscores_2 = -(q_1 - softmax(s_2/T) * sum_k q_1) / (2 B' T), likewise 1 <-> 2
//   dz_v = dscores_v C (live rows only);  dC = dscores_1^T z_1 + dscores_2^T z_2
//
// Both views are stacked ([Z1; Z2], 2B' rows) so each contraction is ONE tcgen05 GEMM launch: scores (K-major x
// K-major), dz (B = prototypes consumed MN-major), dC (both operands MN-major, contraction over the 2B' rows).
// dscores are produced in forward (bf16) by the row-wise cross-entropy kernel and reused by both backward GEMMs.
#include "gemm_host.cuh"

namespace ssvb {
int sinkhorn_run(const float* scores, int64_t b, int64_t k, int64_t ld_scores, float eps, int n_iters, float* codes,
                 int64_t ld_codes, void* workspace, cudaStream_t s, int nprob, int64_t pstride_s, int64_t pstride_c);
size_t sinkhorn_ws_bytes(int64_t k);
bool sinkhorn_scaling_only(const float* scores, int64_t b, int64_t k, int64_t ld_scores, float eps, int n_iters, void* workspace,
                           cudaStream_t s, int64_t pstride_s, const float** alpha, const float** smax, int* kpad, int* rc);
}  // namespace ssvb

using namespace ssvb;

namespace {

struct SwavDims {
  int64_t nb, nbank, bp, k, d, dpad, kp4, kp8;
};
SwavDims dims(int64_t nb, int64_t nbank, int64_t k, int64_t d) {
  SwavDims s;
  s.nb = nb; s.nbank = nbank; s.bp = nb + nbank; s.k = k; s.d = d;
  s.dpad = round_up(d, 8);
  s.kp4 = round_up(k, 4);
  s.kp8 = round_up(k, 8);
  return s;
}
struct SwavSaved {
  __nv_bfloat16* z;   // [2B' x dpad]  (view 1 rows, then view 2 rows)
  __nv_bfloat16* c;   // [K x dpad]
  __nv_bfloat16* ds;  // [2B' x kp8]
  size_t bytes;
};
SwavSaved swav_saved(void* base, const SwavDims& m) {
  Carver c(base);
  SwavSaved s;
  s.z = c.take<__nv_bfloat16>(2 * m.bp * m.dpad);
  s.c = c.take<__nv_bfloat16>(m.k * m.dpad);
  s.ds = c.take<__nv_bfloat16>(2 * m.bp * m.kp8);
  s.bytes = c.used();
  return s;
}
struct SwavWs {
  float* scores;  // [2B' x kp4]
  float* codes;   // [2B' x kp4]
  float* loss_part;  // [B']
  float* dz;      // backward: [2B' x dpad] fp32
  float* dc;      // backward: [K x dpad] fp32
  void* sk;       // sinkhorn workspace
  size_t bytes;
};
SwavWs swav_ws(void* base, const SwavDims& m) {
  Carver c(base);
  SwavWs w;
  w.scores = c.take<float>(2 * m.bp * m.kp4);
  w.codes = c.take<float>(2 * m.bp * m.kp4);
  w.loss_part = c.take<float>(m.bp);
  w.dz = c.take<float>(2 * m.bp * m.dpad);
  w.dc = c.take<float>(m.k * m.dpad);
  w.sk = c.take<uint8_t>(sinkhorn_ws_bytes(m.k));
  w.bytes = c.used();
  return w;
}

__device__ __forceinline__ float block_reduce(float v, bool is_max, float* red) {
  v = is_max ? warp_max(v) : warp_sum(v);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  float t = lane < (blockDim.x >> 5) ? red[lane] : (is_max ? -INFINITY : 0.f);
  return is_max ? warp_max(t) : warp_sum(t);
}

// one block per sample row r (of B'): both views' cross-entropy terms and dscores.  Any K and any row alignment: the form
// for kp8 > 4096 and for score / code rows that are not 16-byte aligned.
__global__ void swav_ce_kernel(const float* __restrict__ scores, const float* __restrict__ codes, int64_t bp, int k,
                               int64_t ld, float inv_t, float coef /* 1/(2 B' T) */, float* __restrict__ loss_part,
                               __nv_bfloat16* __restrict__ ds, int64_t ldds) {
  __shared__ float red[32];
  const int64_t r = blockIdx.x;
  const float* s1 = scores + r * ld;
  const float* s2 = scores + (bp + r) * ld;
  const float* q1 = codes + r * ld;
  const float* q2 = codes + (bp + r) * ld;
  float m1 = -INFINITY, m2 = -INFINITY;
  for (int c = threadIdx.x; c < k; c += blockDim.x) {
    m1 = fmaxf(m1, s1[c]);
    m2 = fmaxf(m2, s2[c]);
  }
  m1 = block_reduce(m1, true, red) * inv_t;
  m2 = block_reduce(m2, true, red) * inv_t;
  float e1 = 0.f, e2 = 0.f, a12 = 0.f, a21 = 0.f, sq1 = 0.f, sq2 = 0.f;
  for (int c = threadIdx.x; c < k; c += blockDim.x) {
    const float t1 = s1[c] * inv_t, t2 = s2[c] * inv_t;
    e1 += __expf(t1 - m1);
    e2 += __expf(t2 - m2);
    const float a = q1[c], b = q2[c];
    a12 = fmaf(a, t2, a12);  // sum q1 * (s2/T)
    a21 = fmaf(b, t1, a21);
    sq1 += a;
    sq2 += b;
  }
  e1 = block_reduce(e1, false, red);
  e2 = block_reduce(e2, false, red);
  a12 = block_reduce(a12, false, red);
  a21 = block_reduce(a21, false, red);
  sq1 = block_reduce(sq1, false, red);
  sq2 = block_reduce(sq2, false, red);
  const float lse1 = m1 + __logf(e1), lse2 = m2 + __logf(e2);
  // sum_k q1 p2 = sum q1 (t2 - lse2) ; per-row loss term -1/2 (.. + ..)
  if (threadIdx.x == 0) loss_part[r] = -0.5f * ((a12 - sq1 * lse2) + (a21 - sq2 * lse1));
  __nv_bfloat16* d1 = ds + r * ldds;
  __nv_bfloat16* d2 = ds + (bp + r) * ldds;
  for (int c = threadIdx.x; c < ldds; c += blockDim.x) {
    float g1 = 0.f, g2 = 0.f;
    if (c < k) {
      g1 = -(q2[c] - __expf(s1[c] * inv_t - lse1) * sq2) * coef;  // d loss / d s1
      g2 = -(q1[c] - __expf(s2[c] * inv_t - lse2) * sq1) * coef;  // d loss / d s2
    }
    d1[c] = __float2bfloat16_rn(g1);
    d2[c] = __float2bfloat16_rn(g2);
  }
}

// Register-cached float4 form of swav_ce_kernel (16-byte aligned rows, ld % 4 == 0, ldds % 4 == 0, ldds <= 1024 * V):
// every score / code row is loaded ONCE and all statistics come from registers; the two maxima and the six sums are
// reduced together (two block reductions instead of eight).  The formulas of swav_ce_kernel, summed in another order.
// Thread t owns columns 4 * (t + 256 * e) .. + 3 (16-byte loads, 8-byte bf16 stores).
// The padding columns [k, ld) of the score / code rows are never written by their producers: masked per element.
template <int V>
__global__ void __launch_bounds__(256)
swav_ce_reg4_kernel(const float* __restrict__ scores, const float* __restrict__ codes, int64_t bp, int k, int64_t ld,
                    float inv_t, float coef /* 1/(2 B' T) */, float* __restrict__ loss_part, __nv_bfloat16* __restrict__ ds,
                    int64_t ldds) {
  __shared__ float red[8][6];
  const int64_t r = blockIdx.x;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float4* s1p = reinterpret_cast<const float4*>(scores + r * ld);
  const float4* s2p = reinterpret_cast<const float4*>(scores + (bp + r) * ld);
  const float4* q1p = reinterpret_cast<const float4*>(codes + r * ld);
  const float4* q2p = reinterpret_cast<const float4*>(codes + (bp + r) * ld);
  const int ld4 = static_cast<int>(ld >> 2);
  float t1[4 * V], t2[4 * V], q1[4 * V], q2[4 * V];
  float m1 = -INFINITY, m2 = -INFINITY;
  const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int e = 0; e < V; ++e) {
    const int c4 = threadIdx.x + e * 256;
    const bool in = c4 < ld4;
    const float4 a = in ? __ldg(s1p + c4) : z4, b = in ? __ldg(s2p + c4) : z4;
    const float4 x = in ? __ldg(q1p + c4) : z4, y = in ? __ldg(q2p + c4) : z4;
    const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
    const float xv[4] = {x.x, x.y, x.z, x.w}, yv[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const bool ok = c4 * 4 + i < k;
      t1[4 * e + i] = ok ? av[i] * inv_t : -INFINITY;
      t2[4 * e + i] = ok ? bv[i] * inv_t : -INFINITY;
      q1[4 * e + i] = ok ? xv[i] : 0.f;
      q2[4 * e + i] = ok ? yv[i] : 0.f;
      m1 = fmaxf(m1, t1[4 * e + i]);
      m2 = fmaxf(m2, t2[4 * e + i]);
    }
  }
  m1 = warp_max(m1);
  m2 = warp_max(m2);
  if (lane == 0) { red[w][0] = m1; red[w][1] = m2; }
  __syncthreads();
  m1 = red[0][0]; m2 = red[0][1];
#pragma unroll
  for (int i = 1; i < 8; ++i) { m1 = fmaxf(m1, red[i][0]); m2 = fmaxf(m2, red[i][1]); }
  __syncthreads();
  float v[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // e1, e2, a12, a21, sq1, sq2
#pragma unroll
  for (int e = 0; e < 4 * V; ++e) {
    if ((threadIdx.x + (e >> 2) * 256) * 4 + (e & 3) < k) {
      v[2] = fmaf(q1[e], t2[e], v[2]);  // sum q1 * (s2/T)
      v[3] = fmaf(q2[e], t1[e], v[3]);
    }
    t1[e] = __expf(t1[e] - m1);  // exp(-inf) = 0 on the padding
    t2[e] = __expf(t2[e] - m2);
    v[0] += t1[e];
    v[1] += t2[e];
    v[4] += q1[e];
    v[5] += q2[e];
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) v[i] = warp_sum(v[i]);
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < 6; ++i) red[w][i] = v[i];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    float t = 0.f;
#pragma unroll
    for (int ww = 0; ww < 8; ++ww) t += red[ww][i];
    v[i] = t;
  }
  const float lse1 = m1 + __logf(v[0]), lse2 = m2 + __logf(v[1]);
  if (threadIdx.x == 0) loss_part[r] = -0.5f * ((v[2] - v[4] * lse2) + (v[3] - v[5] * lse1));
  const float i1 = v[5] / v[0], i2 = v[4] / v[1];  // softmax(s/T) * sum(q of the other view)
  uint2* d1 = reinterpret_cast<uint2*>(ds + r * ldds);
  uint2* d2 = reinterpret_cast<uint2*>(ds + (bp + r) * ldds);
  const int ldds4 = static_cast<int>(ldds >> 2);
#pragma unroll
  for (int e = 0; e < V; ++e) {
    const int c4 = threadIdx.x + e * 256;
    if (c4 < ldds4) {
      float g1[4], g2[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const bool ok = c4 * 4 + i < k;
        g1[i] = ok ? -(q2[4 * e + i] - t1[4 * e + i] * i1) * coef : 0.f;  // d loss / d s1
        g2[i] = ok ? -(q1[4 * e + i] - t2[4 * e + i] * i2) * coef : 0.f;  // d loss / d s2
      }
      __nv_bfloat162 a0 = __floats2bfloat162_rn(g1[0], g1[1]), a1 = __floats2bfloat162_rn(g1[2], g1[3]);
      __nv_bfloat162 b0 = __floats2bfloat162_rn(g2[0], g2[1]), b1 = __floats2bfloat162_rn(g2[2], g2[3]);
      uint2 pa, pb;
      pa.x = *reinterpret_cast<uint32_t*>(&a0); pa.y = *reinterpret_cast<uint32_t*>(&a1);
      pb.x = *reinterpret_cast<uint32_t*>(&b0); pb.y = *reinterpret_cast<uint32_t*>(&b1);
      d1[c4] = pa;
      d2[c4] = pb;
    }
  }
}

// Cross-entropy with the codes rebuilt on the fly: q_v[r, c] = alpha_v[c] E_v[r, c] / sum_c alpha_v[c] E_v[r, c] with
// E_v = exp((s_v - smax_v) / eps) is exactly what the final Sinkhorn pass writes (sinkhorn.cu PHASE 2), so with the last
// scaling vectors in hand that pass and the fp32 code matrix (written, then read back here: 2 x 84 MB at 3512 x 3000) are
// not needed - the row sum of alpha E joins the first block reduction next to the softmax maxima.  Same layout / masks as
// swav_ce_reg4_kernel.  alpha = [2][kpad] (view 1, view 2), smax = [2].
template <int V>
__global__ void __launch_bounds__(256)
swav_ce_sk4_kernel(const float* __restrict__ scores, const float* __restrict__ alpha, const float* __restrict__ smax, int kpad,
                   float inv_eps_log2e, int64_t bp, int k, int64_t ld, float inv_t, float coef /* 1/(2 B' T) */,
                   float* __restrict__ loss_part, __nv_bfloat16* __restrict__ ds, int64_t ldds) {
  __shared__ float red[8][6];
  const int64_t r = blockIdx.x;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float4* s1p = reinterpret_cast<const float4*>(scores + r * ld);
  const float4* s2p = reinterpret_cast<const float4*>(scores + (bp + r) * ld);
  const float4* a1p = reinterpret_cast<const float4*>(alpha);
  const float4* a2p = reinterpret_cast<const float4*>(alpha + kpad);
  const int ld4 = static_cast<int>(ld >> 2), kp4 = kpad >> 2;
  const float sh1 = __ldg(smax) * inv_eps_log2e, sh2 = __ldg(smax + 1) * inv_eps_log2e;
  float t1[4 * V], t2[4 * V], q1[4 * V], q2[4 * V];
  float m1 = -INFINITY, m2 = -INFINITY, v1 = 0.f, v2 = 0.f;
  const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int e = 0; e < V; ++e) {
    const int c4 = threadIdx.x + e * 256;
    const bool in = c4 < ld4 && c4 < kp4;
    const float4 a = in ? __ldg(s1p + c4) : z4, b = in ? __ldg(s2p + c4) : z4;
    const float4 x = in ? __ldg(a1p + c4) : z4, y = in ? __ldg(a2p + c4) : z4;
    const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
    const float xv[4] = {x.x, x.y, x.z, x.w}, yv[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const bool ok = in && c4 * 4 + i < k;
      t1[4 * e + i] = ok ? av[i] * inv_t : -INFINITY;
      t2[4 * e + i] = ok ? bv[i] * inv_t : -INFINITY;
      q1[4 * e + i] = ok ? xv[i] * ex2f(fmaf(av[i], inv_eps_log2e, -sh1)) : 0.f;  // alpha E (un-normalised code)
      q2[4 * e + i] = ok ? yv[i] * ex2f(fmaf(bv[i], inv_eps_log2e, -sh2)) : 0.f;
      m1 = fmaxf(m1, t1[4 * e + i]);
      m2 = fmaxf(m2, t2[4 * e + i]);
      v1 += q1[4 * e + i];
      v2 += q2[4 * e + i];
    }
  }
  m1 = warp_max(m1);
  m2 = warp_max(m2);
  v1 = warp_sum(v1);
  v2 = warp_sum(v2);
  if (lane == 0) { red[w][0] = m1; red[w][1] = m2; red[w][2] = v1; red[w][3] = v2; }
  __syncthreads();
  m1 = red[0][0]; m2 = red[0][1]; v1 = red[0][2]; v2 = red[0][3];
#pragma unroll
  for (int i = 1; i < 8; ++i) {
    m1 = fmaxf(m1, red[i][0]); m2 = fmaxf(m2, red[i][1]);
    v1 += red[i][2]; v2 += red[i][3];
  }
  __syncthreads();
  const float iv1 = 1.f / v1, iv2 = 1.f / v2;
  float v[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // e1, e2, a12, a21, sq1, sq2
#pragma unroll
  for (int e = 0; e < 4 * V; ++e) {
    q1[e] *= iv1;  // codes_bk = alpha_k E_bk / v_b  (sinkhorn.cu PHASE 2)
    q2[e] *= iv2;
    if ((threadIdx.x + (e >> 2) * 256) * 4 + (e & 3) < k) {
      v[2] = fmaf(q1[e], t2[e], v[2]);  // sum q1 * (s2/T)
      v[3] = fmaf(q2[e], t1[e], v[3]);
    }
    t1[e] = __expf(t1[e] - m1);  // exp(-inf) = 0 on the padding
    t2[e] = __expf(t2[e] - m2);
    v[0] += t1[e];
    v[1] += t2[e];
    v[4] += q1[e];
    v[5] += q2[e];
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) v[i] = warp_sum(v[i]);
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < 6; ++i) red[w][i] = v[i];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    float t = 0.f;
#pragma unroll
    for (int ww = 0; ww < 8; ++ww) t += red[ww][i];
    v[i] = t;
  }
  const float lse1 = m1 + __logf(v[0]), lse2 = m2 + __logf(v[1]);
  if (threadIdx.x == 0) loss_part[r] = -0.5f * ((v[2] - v[4] * lse2) + (v[3] - v[5] * lse1));
  const float i1 = v[5] / v[0], i2 = v[4] / v[1];  // softmax(s/T) * sum(q of the other view)
  uint2* d1 = reinterpret_cast<uint2*>(ds + r * ldds);
  uint2* d2 = reinterpret_cast<uint2*>(ds + (bp + r) * ldds);
  const int ldds4 = static_cast<int>(ldds >> 2);
#pragma unroll
  for (int e = 0; e < V; ++e) {
    const int c4 = threadIdx.x + e * 256;
    if (c4 < ldds4) {
      float g1[4], g2[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const bool ok = c4 * 4 + i < k;
        g1[i] = ok ? -(q2[4 * e + i] - t1[4 * e + i] * i1) * coef : 0.f;  // d loss / d s1
        g2[i] = ok ? -(q1[4 * e + i] - t2[4 * e + i] * i2) * coef : 0.f;  // d loss / d s2
      }
      __nv_bfloat162 a0 = __floats2bfloat162_rn(g1[0], g1[1]), a1 = __floats2bfloat162_rn(g1[2], g1[3]);
      __nv_bfloat162 b0 = __floats2bfloat162_rn(g2[0], g2[1]), b1 = __floats2bfloat162_rn(g2[2], g2[3]);
      uint2 pa, pb;
      pa.x = *reinterpret_cast<uint32_t*>(&a0); pa.y = *reinterpret_cast<uint32_t*>(&a1);
      pb.x = *reinterpret_cast<uint32_t*>(&b0); pb.y = *reinterpret_cast<uint32_t*>(&b1);
      d1[c4] = pa;
      d2[c4] = pb;
    }
  }
}

// the three gradient outputs in one launch: segment g of (in, ldi, rows, out, ldo); out[r, c] = go * in[r, c], c < d
struct ScaleSeg {
  const float* in;
  float* out;
  int64_t ldi, ldo, rows;
};
struct ScaleSegs {
  ScaleSeg seg[3];
};
__global__ void scale_rows3_kernel(ScaleSegs sg, int d4, const float* __restrict__ grad_out) {
  const float go = __ldg(grad_out);
  const ScaleSeg& g = sg.seg[blockIdx.y];
  const int64_t total = g.rows * d4;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = i / d4;
    const int c = static_cast<int>(i - r * d4);
    float4 v = __ldg(reinterpret_cast<const float4*>(g.in + r * g.ldi) + c);
    v.x *= go; v.y *= go; v.z *= go; v.w *= go;
    reinterpret_cast<float4*>(g.out + r * g.ldo)[c] = v;
  }
}

int check_rows(const void* p, int64_t ld) {
  if (!p) return SSVB_ERR_INVALID;
  if ((reinterpret_cast<uintptr_t>(p) & 15) || (ld & 3)) return SSVB_ERR_ALIGNMENT;
  return SSVB_OK;
}
int check_shape(int64_t nb, int64_t nbank, int64_t k, int64_t d, float temperature) {
  if (nb <= 0 || nbank < 0 || k <= 0 || d <= 0 || !(temperature > 0.f)) return SSVB_ERR_INVALID;
  if (d % 4) return SSVB_ERR_ALIGNMENT;
  if (2 * (nb + nbank) > (1 << 30) || k > (1 << 24)) return SSVB_ERR_UNSUPPORTED;
  return SSVB_OK;
}
unsigned grid_for(int64_t total, int per_block) {
  int64_t g = ceil_div(total, per_block);
  const int64_t cap = static_cast<int64_t>(num_sms()) * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<unsigned>(g);
}


// One launch for the four operand conversions of the scores GEMM (one warp per source row): z1 -> Z[0, nb), z2 ->
// Z[bp, bp + nb), bank row j -> Z[nb + j] AND Z[bp + nb + j] (the bank closes both views, utils/losses.py:227-229),
// prototypes -> C.  fp32 [rows x d] -> bf16 [rows x dpad], zero padded.
__global__ void swav_stage_kernel(const float* __restrict__ z1, const float* __restrict__ z2, const float* __restrict__ bank,
                                  const float* __restrict__ proto, int64_t nb, int64_t nbank, int64_t k, int64_t bp, int d,
                                  int dpad, int64_t ld_z1, int64_t ld_z2, int64_t ld_bank, int64_t ld_proto,
                                  __nv_bfloat16* __restrict__ z, __nv_bfloat16* __restrict__ c) {
  int64_t row = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const float* src;
  __nv_bfloat16 *dst, *dst2 = nullptr;
  if (row < nb) {
    src = z1 + row * ld_z1;
    dst = z + row * dpad;
  } else if ((row -= nb) < nb) {
    src = z2 + row * ld_z2;
    dst = z + (bp + row) * dpad;
  } else if ((row -= nb) < nbank) {
    src = bank + row * ld_bank;
    dst = z + (nb + row) * dpad;
    dst2 = z + (bp + nb + row) * dpad;
  } else if ((row -= nbank) < k) {
    src = proto + row * ld_proto;
    dst = c + row * dpad;
  } else {
    return;
  }
  for (int col = lane * 4; col < dpad; col += 128) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (col < d) v = __ldg(reinterpret_cast<const float4*>(src + col));
    __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&lo);
    pk.y = *reinterpret_cast<uint32_t*>(&hi);
    *reinterpret_cast<uint2*>(dst + col) = pk;
    if (dst2) *reinterpret_cast<uint2*>(dst2 + col) = pk;
  }
}

// stage [Z1; Z2] (each = live rows then bank rows) and the prototypes as bf16, then scores[2B' x K] = [Z1; Z2] C^T
int stage_scores(const float* z1, const float* z2, const float* bank, const float* prototypes, const SwavDims& m,
                 int64_t ld_z1, int64_t ld_z2, int64_t ld_bank, int64_t ld_proto, const SwavSaved& sv, float* scores,
                 cudaStream_t s) {
  const int di = static_cast<int>(m.d), dp = static_cast<int>(m.dpad);
  const int64_t nb = m.nb, nbank = m.nbank, k = m.k;
  swav_stage_kernel<<<static_cast<unsigned>(ceil_div(2 * nb + nbank + k, 8)), 256, 0, s>>>(
      z1, z2, bank, prototypes, nb, nbank, k, m.bp, di, dp, ld_z1, ld_z2, ld_bank, ld_proto, sv.z, sv.c);
  SSVB_LAUNCH_CHECK();
  GemmParams p{};
  p.M = static_cast<int>(2 * m.bp);
  p.N = static_cast<int>(k);
  p.K = static_cast<int>(m.dpad);
  p.alpha = 1.f;
  p.out = scores;
  p.ldc = m.kp4;
  return launch_gemm({sv.z, m.dpad, false}, {sv.c, m.dpad, false}, p, 256, EPI_STORE_F32, 0, s);
}

// row-wise cross-entropy of both views: loss = sum of the local row terms / bp_total; dscores (bf16) carry the
// 1/(2 bp_total T) coefficient (bp_total = rows per view over ALL ranks; = m.bp on one GPU)
int stage_ce(const float* scores, const float* codes, const SwavDims& m, int64_t bp_total, float temperature,
             const SwavSaved& sv, float* loss_part, float* loss, cudaStream_t s) {
  const unsigned grid = static_cast<unsigned>(m.bp);
  const int ki = static_cast<int>(m.k);
  const float it = 1.f / temperature, coef = 0.5f / (static_cast<float>(bp_total) * temperature);
#define SSVB_CE4(V) swav_ce_reg4_kernel<V><<<grid, 256, 0, s>>>(scores, codes, m.bp, ki, m.kp4, it, coef, loss_part, sv.ds, m.kp8)
  // the float4 kernel needs 16-byte aligned score / code rows; a ssvb_swav_dist_ce caller may pass others
  const bool vec = !(reinterpret_cast<uintptr_t>(scores) & 15) && !(reinterpret_cast<uintptr_t>(codes) & 15) &&
                   !(reinterpret_cast<uintptr_t>(sv.ds) & 7);  // (kp4 % 4 == 0 and kp8 % 8 == 0 by construction)
  if (vec && m.kp8 <= 1 * 1024) SSVB_CE4(1);
  else if (vec && m.kp8 <= 2 * 1024) SSVB_CE4(2);
  else if (vec && m.kp8 <= 3 * 1024) SSVB_CE4(3);
  else if (vec && m.kp8 <= 4 * 1024) SSVB_CE4(4);
  else swav_ce_kernel<<<grid, 256, 0, s>>>(scores, codes, m.bp, ki, m.kp4, it, coef, loss_part, sv.ds, m.kp8);
#undef SSVB_CE4
  SSVB_LAUNCH_CHECK();
  sum_partials_kernel<<<1, 1024, 0, s>>>(loss_part, static_cast<int>(m.bp), 1.f / static_cast<float>(bp_total), loss);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

}  // namespace

extern "C" {

size_t ssvb_swav_saved_bytes(int64_t nb, int64_t nbank, int64_t k, int64_t d) {
  if (nb <= 0 || nbank < 0 || k <= 0 || d <= 0) return 0;
  return swav_saved(nullptr, dims(nb, nbank, k, d)).bytes;
}
size_t ssvb_swav_workspace_bytes(int64_t nb, int64_t nbank, int64_t k, int64_t d) {
  if (nb <= 0 || nbank < 0 || k <= 0 || d <= 0) return 0;
  return swav_ws(nullptr, dims(nb, nbank, k, d)).bytes;
}

int ssvb_swav_fwd(const float* z1, const float* z2, const float* bank, const float* prototypes, int64_t nb,
                  int64_t nbank, int64_t k, int64_t d, int64_t ld_z1, int64_t ld_z2, int64_t ld_bank,
                  int64_t ld_proto, float temperature, float eps, int n_iters, float* loss, void* saved,
                  void* workspace, size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(check_shape(nb, nbank, k, d, temperature));
  SSVB_TRY(check_rows(z1, ld_z1));
  SSVB_TRY(check_rows(z2, ld_z2));
  SSVB_TRY(check_rows(prototypes, ld_proto));
  if (nbank > 0) SSVB_TRY(check_rows(bank, ld_bank));
  if (!loss || !saved || !workspace || !(eps > 0.f) || n_iters < 0) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_swav_workspace_bytes(nb, nbank, k, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const SwavDims m = dims(nb, nbank, k, d);
  SwavSaved sv = swav_saved(saved, m);
  SwavWs ws = swav_ws(workspace, m);
  SSVB_TRY(stage_scores(z1, z2, bank, prototypes, m, ld_z1, ld_z2, ld_bank, ld_proto, sv, ws.scores, s));
  // codes per view (Sinkhorn normalises over the B' rows of ONE view)
  // the two views' code assignments (utils/losses.py:232) are independent problems of one shape: batched launches
  const float *alpha = nullptr, *smax = nullptr;
  int kpad = 0, rc = SSVB_OK;
  if (m.kp8 <= 4 * 1024 && !(reinterpret_cast<uintptr_t>(sv.ds) & 7) &&
      sinkhorn_scaling_only(ws.scores, m.bp, k, m.kp4, eps, n_iters, ws.sk, s, m.bp * m.kp4, &alpha, &smax, &kpad, &rc)) {
    // the iteration ran without its final pass: the cross-entropy kernel rebuilds each code row from the scaling vectors
    SSVB_TRY(rc);
    const unsigned grid = static_cast<unsigned>(m.bp);
    const float iel = SSVB_LOG2E / eps, it = 1.f / temperature, coef = 0.5f / (static_cast<float>(m.bp) * temperature);
#define SSVB_CESK(V)                                                                                                       \
  swav_ce_sk4_kernel<V><<<grid, 256, 0, s>>>(ws.scores, alpha, smax, kpad, iel, m.bp, static_cast<int>(k), m.kp4, it, coef, \
                                             ws.loss_part, sv.ds, m.kp8)
    if (m.kp8 <= 1 * 1024) SSVB_CESK(1);
    else if (m.kp8 <= 2 * 1024) SSVB_CESK(2);
    else if (m.kp8 <= 3 * 1024) SSVB_CESK(3);
    else SSVB_CESK(4);
#undef SSVB_CESK
    SSVB_LAUNCH_CHECK();
    sum_partials_kernel<<<1, 1024, 0, s>>>(ws.loss_part, static_cast<int>(m.bp), 1.f / static_cast<float>(m.bp), loss);
    SSVB_LAUNCH_CHECK();
    return SSVB_OK;
  }
  SSVB_TRY(sinkhorn_run(ws.scores, m.bp, k, m.kp4, eps, n_iters, ws.codes, m.kp4, ws.sk, s, 2, m.bp * m.kp4, m.bp * m.kp4));
  return stage_ce(ws.scores, ws.codes, m, m.bp, temperature, sv, ws.loss_part, loss, s);
}

// ---- distributed (sample rows sharded over ranks; prototypes replicated): see include/ssv_b200.h ----------------
int64_t ssvb_swav_kpad(int64_t k) { return k > 0 ? round_up(k, 4) : 0; }

int ssvb_swav_dist_scores(const float* z1, const float* z2, const float* bank, const float* prototypes, int64_t nb,
                          int64_t nbank, int64_t k, int64_t d, int64_t ld_z1, int64_t ld_z2, int64_t ld_bank,
                          int64_t ld_proto, float* scores, void* saved, void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(check_shape(nb, nbank, k, d, 1.f));
  SSVB_TRY(check_rows(z1, ld_z1));
  SSVB_TRY(check_rows(z2, ld_z2));
  SSVB_TRY(check_rows(prototypes, ld_proto));
  if (nbank > 0) SSVB_TRY(check_rows(bank, ld_bank));
  if (!scores || !saved) return SSVB_ERR_INVALID;
  if (reinterpret_cast<uintptr_t>(scores) & 15) return SSVB_ERR_ALIGNMENT;
  const SwavDims m = dims(nb, nbank, k, d);
  SwavSaved sv = swav_saved(saved, m);
  return stage_scores(z1, z2, bank, prototypes, m, ld_z1, ld_z2, ld_bank, ld_proto, sv, scores,
                      static_cast<cudaStream_t>(stream));
}

int ssvb_swav_dist_ce(const float* scores, const float* codes, int64_t nb, int64_t nbank, int64_t bp_global, int64_t k,
                      int64_t d, float temperature, float* loss_local, void* saved, void* workspace,
                      size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(check_shape(nb, nbank, k, d, temperature));
  if (!scores || !codes || !loss_local || !saved || !workspace || bp_global < nb + nbank) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_swav_workspace_bytes(nb, nbank, k, d)) return SSVB_ERR_WORKSPACE;
  const SwavDims m = dims(nb, nbank, k, d);
  SwavSaved sv = swav_saved(saved, m);
  SwavWs ws = swav_ws(workspace, m);
  return stage_ce(scores, codes, m, bp_global, temperature, sv, ws.loss_part, loss_local,
                  static_cast<cudaStream_t>(stream));
}

int ssvb_swav_bwd(const float* z1, const float* z2, const float* bank, const float* prototypes, int64_t nb,
                  int64_t nbank, int64_t k, int64_t d, int64_t ld_z1, int64_t ld_z2, int64_t ld_bank,
                  int64_t ld_proto, float temperature, const float* grad_out, const void* saved, float* dz1,
                  float* dz2, float* dproto, int64_t ld_dz1, int64_t ld_dz2, int64_t ld_dproto, void* workspace,
                  size_t workspace_bytes, void* stream) {
  (void)z1; (void)z2; (void)bank; (void)prototypes; (void)ld_z1; (void)ld_z2; (void)ld_bank; (void)ld_proto;
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(check_shape(nb, nbank, k, d, temperature));
  if (dz1) SSVB_TRY(check_rows(dz1, ld_dz1));
  if (dz2) SSVB_TRY(check_rows(dz2, ld_dz2));
  if (dproto) SSVB_TRY(check_rows(dproto, ld_dproto));
  if (!grad_out || !saved || !workspace) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_swav_workspace_bytes(nb, nbank, k, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const SwavDims m = dims(nb, nbank, k, d);
  SwavSaved sv = swav_saved(const_cast<void*>(saved), m);
  SwavWs ws = swav_ws(workspace, m);
  const int di = static_cast<int>(d);

  GemmParams pz{}, pc{};
  bool split_z = false, split_c = false;
  if (dz1 || dz2) {
    // dz[2B' x d] = ds[2B' x K] C[K x d]        (A K-major, B = prototypes consumed MN-major)
    pz.M = static_cast<int>(2 * m.bp);
    pz.N = static_cast<int>(m.dpad);
    pz.K = static_cast<int>(k);
    pz.alpha = 1.f;
    pz.out = ws.dz;
    pz.ldc = m.dpad;
    // 2B'/128 x 1 tiles (55 at the reference shape) for 148 SMs: split K over CTAs, partial products added by TMA
    split_z = gemm_will_split(pz.M, pz.N, pz.K, 128, ws.dz, m.dpad);
  }
  if (dproto) {
    // dC[K x d] = ds^T [K x 2B'] [Z1; Z2] [2B' x d]   (both operands MN-major, contraction over the stacked rows)
    pc.M = static_cast<int>(k);
    pc.N = static_cast<int>(m.dpad);
    pc.K = static_cast<int>(2 * m.bp);
    pc.alpha = 1.f;
    pc.out = ws.dc;
    pc.ldc = m.dpad;
    // K/128 x 1 tiles (24 at K = 3000): split the contraction over the stacked rows across CTAs
    split_c = gemm_will_split(pc.M, pc.N, pc.K, 128, ws.dc, m.dpad);
  }
  // split-K accumulators are zeroed up front; ws.dz and ws.dc are adjacent in the workspace: one memset node when both split
  const size_t zbytes = static_cast<size_t>(2 * m.bp) * m.dpad * sizeof(float), cbytes = static_cast<size_t>(k) * m.dpad * sizeof(float);
  if (split_z && split_c) {
    const size_t span = static_cast<size_t>(reinterpret_cast<uint8_t*>(ws.dc) - reinterpret_cast<uint8_t*>(ws.dz)) + cbytes;
    SSVB_CUDA(cudaMemsetAsync(ws.dz, 0, span, s));
  } else if (split_z) {
    SSVB_CUDA(cudaMemsetAsync(ws.dz, 0, zbytes, s));
  } else if (split_c) {
    SSVB_CUDA(cudaMemsetAsync(ws.dc, 0, cbytes, s));
  }
  if (dz1 || dz2) SSVB_TRY(launch_gemm({sv.ds, m.kp8, false}, {sv.c, m.dpad, true}, pz, 128, EPI_STORE_F32, 0, s, split_z));
  if (dproto) SSVB_TRY(launch_gemm({sv.ds, m.kp8, true}, {sv.z, m.dpad, true}, pc, 128, EPI_STORE_F32, 0, s, split_c));
  // grad_out scaling of every requested output in one launch
  ScaleSegs sg{};
  int nseg = 0;
  int64_t max_rows = 0;
  auto add = [&](const float* in, float* out, int64_t ldo, int64_t rows) {
    sg.seg[nseg++] = ScaleSeg{in, out, m.dpad, ldo, rows};
    if (rows > max_rows) max_rows = rows;
  };
  if (dz1) add(ws.dz, dz1, ld_dz1, nb);
  if (dz2) add(ws.dz + m.bp * m.dpad, dz2, ld_dz2, nb);
  if (dproto) add(ws.dc, dproto, ld_dproto, k);
  if (nseg) {
    scale_rows3_kernel<<<dim3(grid_for(max_rows * (d / 4), 256), static_cast<unsigned>(nseg)), 256, 0, s>>>(sg, di / 4, grad_out);
    SSVB_LAUNCH_CHECK();
  }
  return SSVB_OK;
}

}  // extern "C"
