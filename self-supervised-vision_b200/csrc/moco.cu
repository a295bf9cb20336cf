// MoCo InfoNCE loss, forward + backward — replaces MocoLoss.forward (reference utils/losses.py:56-72,
// call site models/moco.py:117).
//
//   l_a0 = qh_a . kh_a / tau          (positive: row dot, NOT the diagonal of a full N x N GEMM)
//   l_aj = qh_a . m_j / tau           (queue rows used as stored)
//   loss = mean_a [ LSE_{j=0..K} l_aj - l_a0 ]
//   d qh_a = [(p_a0 - 1) kh_a + sum_j p_aj m_j] / (N tau),  d kh_a = (p_a0 - 1) qh_a / (N tau)
// The N x K logits never reach HBM: the queue axis is split across CTAs (sim_fwd_kernel / sim_bwd_kernel
// in SIM_MOCO mode, online-max because stored queue rows are not guaranteed unit-norm).
#include "sim_host.cuh"

using namespace ssvb;

namespace {

struct MocoSaved {
  __nv_bfloat16* qhat;  // [npad x dpad]
  float *inv_q, *inv_k, *pos, *lse2;
  float* pm;  // [npad x dpad] fused path: sum_j p_aj m_j, produced by the FORWARD pass (backward never reads the queue)
  size_t bytes;
};
MocoSaved moco_saved(void* base, int64_t n, int64_t dpad) {
  Carver c(base);
  MocoSaved s;
  const int64_t npad = round_up(n, 128);
  s.qhat = c.take<__nv_bfloat16>(npad * dpad);
  s.inv_q = c.take<float>(npad);
  s.inv_k = c.take<float>(npad);
  s.pos = c.take<float>(npad);
  s.lse2 = c.take<float>(npad);
  s.pm = c.take<float>(npad * dpad);
  s.bytes = c.used();
  return s;
}

// Fused single-pass form (flash-attention shaped): when the queries are L2-normalised and the queue rows are unit-norm
// or zero (a MemoryBank: rows are normalised on enqueue, models/moco.py:31-36), every logit is bounded by 1/tau, a
// constant shift replaces the running max, and ONE pass over the queue yields both the row sums of exp (-> LSE, loss)
// and sum_j exp(l_aj) m_j (-> the gradient) as plain sums over column chunks.  The queue is read once per step
// instead of twice and the backward is a single row-wise kernel.
inline bool moco_fused(int normalize, int queue_unit_norm, float temperature) {
  return normalize && queue_unit_norm && (2.f * SSVB_LOG2E / temperature <= 120.f);
}

struct MocoWs {
  __nv_bfloat16* queue_bf16;  // [k x dpad] (only when no shadow is supplied)
  float *part_m, *part_l, *block_sums, *dacc;
  unsigned int* counter;
  size_t bytes;
};
void moco_plan(SimParams& p, int64_t n, int64_t k, float c, int BN, int min_tiles) {
  p = SimParams{};
  p.nseg = 1;
  p.seg_rows = static_cast<int>(n);
  p.seg_start[0] = 0;
  p.bps = static_cast<int>(ceil_div(n, 128));
  p.row_blocks = p.bps;
  p.cols = static_cast<int>(k);
  p.c = c;
  p.shift = 0.f;
  plan_chunks(p, BN, min_tiles);
}
MocoWs moco_ws(void* base, int64_t n, int64_t k, int64_t dpad) {
  Carver c(base);
  MocoWs w;
  const int64_t npad = round_up(n, 128);
  SimParams p, pb;
  moco_plan(p, n, k, 1.f, sim_fwd_bn(dpad), 512 / sim_fwd_bn(dpad));
  moco_plan(pb, n, k, 1.f, 128, 4);  // the fused single-pass form runs the backward-shaped kernel with its own chunk plan
  const int nch = p.nchunks > pb.nchunks ? p.nchunks : pb.nchunks;
  w.queue_bf16 = c.take<__nv_bfloat16>(k * dpad);
  w.part_m = c.take<float>(static_cast<size_t>(4 * nch) * npad);
  w.part_l = c.take<float>(static_cast<size_t>(4 * nch) * npad);
  w.block_sums = c.take<float>(ceil_div(npad, 8) + 8);
  w.counter = c.take<unsigned int>(4);
  w.dacc = c.take<float>(npad * dpad);
  w.bytes = c.used();
  return w;
}

// fp32 [k x d] -> bf16 [k x dpad] (zero padded), one warp per row
__global__ void queue_to_bf16_kernel(const float* __restrict__ q, int64_t k, int d, int64_t ld, int dpad,
                                     __nv_bfloat16* __restrict__ out) {
  const int64_t row = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= k) return;
  for (int c = lane * 4; c < dpad; c += 128) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < d) v = __ldg(reinterpret_cast<const float4*>(q + row * ld + c));
    __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&lo);
    pk.y = *reinterpret_cast<uint32_t*>(&hi);
    *reinterpret_cast<uint2*>(out + row * dpad + c) = pk;
  }
}

// the first kPartBatch lane-strided partials of row r (partial i lives at part[i * stride + r]) in registers: all loads
// in flight at once.  nparts <= 32 * kPartBatch covers every plan (<= 4 x 74 chunks); callers loop over the rest.
constexpr int kPartBatch = 12;
__device__ __forceinline__ void load_row_partials(const float* __restrict__ part, int nparts, int stride, int r, int lane,
                                                  float fill, float (&v)[kPartBatch]) {
#pragma unroll
  for (int u = 0; u < kPartBatch; ++u) {
    const int i = lane + 32 * u;
    v[u] = i < nparts ? part[static_cast<size_t>(i) * stride + r] : fill;
  }
}

// PIRL: BOTH InfoNCE heads from one read of the shared negatives' (max, sum) partials - head 0 = patch, head 1 = image
// (utils/losses.py:109-117) - and the combined loss w CE_0 + (1 - w) CE_1 in one deterministic reduction.
__global__ void pirl_finalize_kernel(const float* __restrict__ part_m, const float* __restrict__ part_l, int nparts,
                                     int stride, int nrows, const float* __restrict__ pos0,
                                     const float* __restrict__ pos1, float c, float* __restrict__ lse0,
                                     float* __restrict__ lse1, float w0, float w1, float* block_sums,
                                     unsigned int* counter, float loss_scale, float* loss) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  float term = 0.f;
  if (r < nrows) {
    float mv[kPartBatch], lv[kPartBatch];
    load_row_partials(part_m, nparts, stride, r, lane, -1e30f, mv);
    load_row_partials(part_l, nparts, stride, r, lane, 0.f, lv);
    const float p0 = pos0[r] * c, p1 = pos1[r] * c;
    float Mn = -1e30f;  // max over the negatives' partials
#pragma unroll
    for (int u = 0; u < kPartBatch; ++u) Mn = fmaxf(Mn, mv[u]);
    for (int i = lane + 32 * kPartBatch; i < nparts; i += 32) Mn = fmaxf(Mn, part_m[static_cast<size_t>(i) * stride + r]);
    Mn = warp_max(Mn);
    float Ln = 0.f;     // sum over the negatives relative to Mn
#pragma unroll
    for (int u = 0; u < kPartBatch; ++u) Ln += lv[u] * exp2f(mv[u] - Mn);
    for (int i = lane + 32 * kPartBatch; i < nparts; i += 32)
      Ln += part_l[static_cast<size_t>(i) * stride + r] * exp2f(part_m[static_cast<size_t>(i) * stride + r] - Mn);
    Ln = warp_sum(Ln);
    if (lane == 0) {
      const float M0 = fmaxf(Mn, p0), M1 = fmaxf(Mn, p1);
      const float l0 = M0 + log2f(Ln * exp2f(Mn - M0) + exp2f(p0 - M0));
      const float l1 = M1 + log2f(Ln * exp2f(Mn - M1) + exp2f(p1 - M1));
      lse0[r] = l0;
      lse1[r] = l1;
      term = (w0 * (l0 - p0) + w1 * (l1 - p1)) * SSVB_LN2;
    }
  }
  const float bt = block_sum_256(term);
  grid_sum_finish(bt, block_sums, counter, loss_scale, loss, false);
}

// fused path: combine the per-chunk row sums (fixed order), add the positive logit's term, emit lse2 / the loss term and
// turn the accumulated sum_j exp2(l_aj - shift) m_j into sum_j p_aj m_j.  One warp per query row.
__global__ void moco_fused_finalize_kernel(const float* __restrict__ part_l, int nparts, int stride, int nrows, int dpad,
                                           const float* __restrict__ pos, float c, float shift,
                                           const float* __restrict__ dacc, float* __restrict__ pm,
                                           float* __restrict__ lse2_out, float* block_sums, unsigned int* counter,
                                           float loss_scale, float* loss) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  float term = 0.f;
  if (r < nrows) {
    // every load of this row is issued before the first use (one memory round trip instead of ~10 dependent ones: the
    // partials of a row are `stride` floats apart); summation order unchanged (lane-strided, then the shuffle tree)
    float pv[kPartBatch];
    load_row_partials(part_l, nparts, stride, r, lane, 0.f, pv);
    const float4 acc0 = lane * 4 < dpad ? *reinterpret_cast<const float4*>(dacc + static_cast<size_t>(r) * dpad + lane * 4)
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
    const float pos_r = pos[r];
    float L = 0.f;
#pragma unroll
    for (int u = 0; u < kPartBatch; ++u) L += pv[u];
    for (int i = lane + 32 * kPartBatch; i < nparts; i += 32) L += part_l[static_cast<size_t>(i) * stride + r];
    L = warp_sum(L);
    const float p2 = pos_r * c;
    L += exp2f(p2 - shift);  // label-0 column of the reference's cat (utils/losses.py:70)
    const float lse2 = shift + log2f(L);
    const float inv = 1.f / L;
    for (int k = lane * 4; k < dpad; k += 128) {
      float4 v = k < 128 ? acc0 : *reinterpret_cast<const float4*>(dacc + static_cast<size_t>(r) * dpad + k);
      v.x *= inv; v.y *= inv; v.z *= inv; v.w *= inv;
      *reinterpret_cast<float4*>(pm + static_cast<size_t>(r) * dpad + k) = v;
    }
    if (lane == 0) {
      lse2_out[r] = lse2;
      term = (lse2 - p2) * SSVB_LN2;
    }
  }
  const float bt = block_sum_256(term);
  grid_sum_finish(bt, block_sums, counter, loss_scale, loss, false);
}

__global__ void moco_grad_finish_kernel(const float* __restrict__ q, const float* __restrict__ kk, int64_t ldq,
                                        int64_t ldk, int n, int d, const float* __restrict__ dacc, int ld_dacc,
                                        const MocoSaved sv, int normalize, float c, float inv_n_tau,
                                        const float* __restrict__ grad_out, float* __restrict__ dq,
                                        float* __restrict__ dk, int64_t lddq, int64_t lddk) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= n) return;
  const float scale = inv_n_tau * __ldg(grad_out);
  const float p0m1 = exp2f(sv.pos[row] * c - sv.lse2[row]) - 1.f;
  const float iq = normalize ? sv.inv_q[row] : 1.f, ik = normalize ? sv.inv_k[row] : 1.f;
  // d <= 256: up to two float4 per lane (columns lane * 4 and 128 + lane * 4)
  float gq[2][4], gk[2][4], qh[2][4], kh[2][4];
  float dq_dot = 0.f, dk_dot = 0.f;
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int k4 = it * 128 + lane * 4;
#pragma unroll
    for (int e = 0; e < 4; ++e) gq[it][e] = gk[it][e] = qh[it][e] = kh[it][e] = 0.f;
    if (k4 < d) {
      const float4 acc = *reinterpret_cast<const float4*>(dacc + static_cast<int64_t>(row) * ld_dacc + k4);
      const float4 vq = *reinterpret_cast<const float4*>(q + static_cast<int64_t>(row) * ldq + k4);
      const float4 vk = *reinterpret_cast<const float4*>(kk + static_cast<int64_t>(row) * ldk + k4);
      qh[it][0] = vq.x * iq; qh[it][1] = vq.y * iq; qh[it][2] = vq.z * iq; qh[it][3] = vq.w * iq;
      kh[it][0] = vk.x * ik; kh[it][1] = vk.y * ik; kh[it][2] = vk.z * ik; kh[it][3] = vk.w * ik;
      const float a[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        gq[it][e] = (p0m1 * kh[it][e] + a[e]) * scale;
        gk[it][e] = p0m1 * qh[it][e] * scale;
      }
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      dq_dot += gq[it][e] * qh[it][e];
      dk_dot += gk[it][e] * kh[it][e];
    }
  }
  if (normalize) {
    dq_dot = warp_sum(dq_dot);
    dk_dot = warp_sum(dk_dot);
#pragma unroll
    for (int it = 0; it < 2; ++it)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        gq[it][e] = (gq[it][e] - dq_dot * qh[it][e]) * iq;
        gk[it][e] = (gk[it][e] - dk_dot * kh[it][e]) * ik;
      }
  }
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int k4 = it * 128 + lane * 4;
    if (k4 < d) {
      if (dq) *reinterpret_cast<float4*>(dq + static_cast<int64_t>(row) * lddq + k4) = make_float4(gq[it][0], gq[it][1], gq[it][2], gq[it][3]);
      if (dk) *reinterpret_cast<float4*>(dk + static_cast<int64_t>(row) * lddk + k4) = make_float4(gk[it][0], gk[it][1], gk[it][2], gk[it][3]);
    }
  }
}

// ---- sharded queue (distributed) -----------------------------------------------------------------------------
// combine the per-chunk partials of the local shard into ONE (m, l) pair per global query row (one warp per row)
__global__ void shard_combine_kernel(const float* __restrict__ part_m, const float* __restrict__ part_l, int nparts,
                                     int stride, int nrows, float* __restrict__ out_m, float* __restrict__ out_l) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= nrows) return;
  float M = -1e30f;
  for (int i = lane; i < nparts; i += 32) M = fmaxf(M, part_m[static_cast<size_t>(i) * stride + r]);
  M = warp_max(M);
  float L = 0.f;
  for (int i = lane; i < nparts; i += 32)
    L += part_l[static_cast<size_t>(i) * stride + r] * exp2f(part_m[static_cast<size_t>(i) * stride + r] - M);
  L = warp_sum(L);
  if (lane == 0) {
    out_m[r] = M;
    out_l[r] = L;
  }
}
// part_all: [world] blocks of [m (n_global) | l (n_global) | pos of the block's own n_local rows]; combine in rank
// order with the positive logit (label-0 column) -> lse2_all and the global loss (identical on every rank).
__global__ void shard_finalize_kernel(const float* __restrict__ part_all, int world, int n_local, float c,
                                      float* __restrict__ lse2_all, float* block_sums, unsigned int* counter,
                                      float loss_scale, float* loss) {
  const int n_global = world * n_local;
  const int64_t blk = 2 * static_cast<int64_t>(n_global) + n_local;
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  float term = 0.f;
  if (r < n_global) {
    const float p2 = part_all[(r / n_local) * blk + 2 * n_global + (r % n_local)] * c;
    float M = p2;
    for (int w = 0; w < world; ++w) M = fmaxf(M, part_all[w * blk + r]);
    float L = exp2f(p2 - M);
    for (int w = 0; w < world; ++w) L += part_all[w * blk + n_global + r] * exp2f(part_all[w * blk + r] - M);
    const float lse2 = M + log2f(L);
    lse2_all[r] = lse2;
    term = (lse2 - p2) * SSVB_LN2;
  }
  const float bt = block_sum_256(term);
  grid_sum_finish(bt, block_sums, counter, loss_scale, loss, false);
}

// ---- PIRL (SURVEY §8f): two InfoNCE heads sharing the negatives; gradient only to the (normalised) key side ----------
struct PirlSaved {
  __nv_bfloat16* qhat;  // memory_pos rows as stored, bf16 [npad x dpad]
  float *inv_patch, *inv_img, *pos_patch, *pos_img, *lse_patch, *lse_img, *unused;
  size_t bytes;
};
PirlSaved pirl_saved(void* base, int64_t n, int64_t dpad) {
  Carver c(base);
  PirlSaved s;
  const int64_t npad = round_up(n, 128);
  s.qhat = c.take<__nv_bfloat16>(npad * dpad);
  s.inv_patch = c.take<float>(npad);
  s.inv_img = c.take<float>(npad);
  s.pos_patch = c.take<float>(npad);
  s.pos_img = c.take<float>(npad);
  s.lse_patch = c.take<float>(npad);
  s.lse_img = c.take<float>(npad);
  s.unused = c.take<float>(npad);
  s.bytes = c.used();
  return s;
}
// d v^_h = w_h (p0_h - 1) mem_pos / (N tau), chained through the row normalisation of v_h; one warp per row, both heads
__global__ void pirl_grad_kernel(const float* __restrict__ img, const float* __restrict__ patch,
                                 const float* __restrict__ mem_pos, int64_t ld_img, int64_t ld_patch, int64_t ld_pos, int n,
                                 int d, const PirlSaved sv, int normalize, float c, float inv_n_tau, float w,
                                 const float* __restrict__ grad_out, float* __restrict__ d_img, float* __restrict__ d_patch,
                                 int64_t ld_dimg, int64_t ld_dpatch) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= n) return;
  const float scale = inv_n_tau * __ldg(grad_out);
  // d <= 256: up to two float4 per lane (columns lane * 4 and 128 + lane * 4)
  float q[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int k4 = it * 128 + lane * 4;
    if (k4 < d) {
      const float4 v = *reinterpret_cast<const float4*>(mem_pos + static_cast<int64_t>(row) * ld_pos + k4);
      q[it][0] = v.x; q[it][1] = v.y; q[it][2] = v.z; q[it][3] = v.w;
    }
  }
#pragma unroll
  for (int h = 0; h < 2; ++h) {  // head 0: patch (weight w), head 1: img (weight 1 - w)
    float* dst = h ? d_img : d_patch;
    if (!dst) continue;
    const float* src = h ? img : patch;
    const int64_t lds = h ? ld_img : ld_patch, ldd = h ? ld_dimg : ld_dpatch;
    const float pos = h ? sv.pos_img[row] : sv.pos_patch[row];
    const float lse2 = h ? sv.lse_img[row] : sv.lse_patch[row];
    const float iv = normalize ? (h ? sv.inv_img[row] : sv.inv_patch[row]) : 1.f;
    const float coef = (exp2f(pos * c - lse2) - 1.f) * scale * (h ? 1.f - w : w);
    float g[2][4], xh[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    float dot = 0.f;
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int k4 = it * 128 + lane * 4;
      if (k4 < d) {
        const float4 v = *reinterpret_cast<const float4*>(src + static_cast<int64_t>(row) * lds + k4);
        xh[it][0] = v.x * iv; xh[it][1] = v.y * iv; xh[it][2] = v.z * iv; xh[it][3] = v.w * iv;
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        g[it][e] = coef * q[it][e];
        dot += g[it][e] * xh[it][e];
      }
    }
    if (normalize) {
      dot = warp_sum(dot);
#pragma unroll
      for (int it = 0; it < 2; ++it)
#pragma unroll
        for (int e = 0; e < 4; ++e) g[it][e] = (g[it][e] - dot * xh[it][e]) * iv;
    }
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int k4 = it * 128 + lane * 4;
      if (k4 < d)
        *reinterpret_cast<float4*>(dst + static_cast<int64_t>(row) * ldd + k4) = make_float4(g[it][0], g[it][1], g[it][2], g[it][3]);
    }
  }
}

int check_rows(const void* p, int64_t ld) {
  if (!p) return SSVB_ERR_INVALID;
  if ((reinterpret_cast<uintptr_t>(p) & 15) || (ld & 3)) return SSVB_ERR_ALIGNMENT;
  return SSVB_OK;
}
int check_shape(int64_t n, int64_t k, int64_t d, float temperature) {
  if (n <= 0 || k <= 0 || d <= 0 || !(temperature > 0.f)) return SSVB_ERR_INVALID;
  if (d % 4) return SSVB_ERR_ALIGNMENT;
  if (d > 256 || k > (1 << 30) || n > (1 << 30)) return SSVB_ERR_UNSUPPORTED;
  return SSVB_OK;
}

int get_queue_bf16(const float* queue, const void* shadow, int64_t k, int64_t d, int64_t ld, int64_t dpad,
                   MocoWs& ws, cudaStream_t s, const __nv_bfloat16** out) {
  if (shadow) {
    if (reinterpret_cast<uintptr_t>(shadow) & 15) return SSVB_ERR_ALIGNMENT;
    *out = static_cast<const __nv_bfloat16*>(shadow);
    return SSVB_OK;
  }
  SSVB_TRY(check_rows(queue, ld));
  queue_to_bf16_kernel<<<static_cast<unsigned>(ceil_div(k, 8)), 256, 0, s>>>(queue, k, static_cast<int>(d), ld,
                                                                             static_cast<int>(dpad), ws.queue_bf16);
  SSVB_LAUNCH_CHECK();
  *out = ws.queue_bf16;
  return SSVB_OK;
}

}  // namespace

extern "C" {

size_t ssvb_moco_saved_bytes(int64_t n, int64_t k, int64_t d) {
  (void)k;
  if (n <= 0 || d <= 0) return 0;
  return moco_saved(nullptr, n, sim_dpad(d)).bytes;
}
size_t ssvb_moco_workspace_bytes(int64_t n, int64_t k, int64_t d) {
  if (n <= 0 || k <= 0 || d <= 0) return 0;
  return moco_ws(nullptr, n, k, sim_dpad(d)).bytes;
}

int ssvb_moco_fwd(const float* query, const float* keys, const float* queue, const void* queue_bf16,
                  int queue_unit_norm, int64_t n, int64_t k, int64_t d, int64_t ld_q, int64_t ld_k, int64_t ld_queue,
                  int normalize, float temperature, float* loss, void* saved, void* workspace, size_t workspace_bytes,
                  void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(check_shape(n, k, d, temperature));
  SSVB_TRY(check_rows(query, ld_q));
  SSVB_TRY(check_rows(keys, ld_k));
  if (!loss || !saved || !workspace || (!queue && !queue_bf16)) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_moco_workspace_bytes(n, k, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t dpad = sim_dpad(d), npad = round_up(n, 128);
  MocoSaved sv = moco_saved(saved, n, dpad);
  MocoWs ws = moco_ws(workspace, n, k, dpad);
  const float c = SSVB_LOG2E / temperature;

  if (npad > n) SSVB_CUDA(cudaMemsetAsync(sv.qhat + n * dpad, 0, (npad - n) * dpad * sizeof(__nv_bfloat16), s));
  // the prep kernel also zeroes the last-block counter and (fused path) the P*M accumulator the column chunks add
  // into: no memset nodes in front of / between the kernels
  const bool fused_path = moco_fused(normalize, queue_unit_norm, temperature);
  pair_prep_kernel<<<static_cast<unsigned>(ceil_div(fused_path ? npad : n, 8)), 256, 0, s>>>(
      query, keys, static_cast<int>(n), static_cast<int>(d), ld_q, ld_k, normalize, 0, sv.qhat, nullptr,
      static_cast<int>(dpad), sv.inv_q, sv.inv_k, sv.pos, nullptr, -1, 1.f, ws.counter,
      fused_path ? ws.dacc : nullptr, static_cast<int>(dpad), static_cast<int>(npad));
  SSVB_LAUNCH_CHECK();
  const __nv_bfloat16* qb = nullptr;
  SSVB_TRY(get_queue_bf16(queue, queue_bf16, k, d, ld_queue, dpad, ws, s, &qb));

  SimParams p;
  if (moco_fused(normalize, queue_unit_norm, temperature)) {
    // one pass over the queue: S tile -> exp2(l - c) -> (row sums, W * M accumulated in TMEM) with the backward-shaped
    // kernel; the column chunks add into a zeroed accumulator
    moco_plan(p, n, k, c, 128, 4);
    p.shift = c;
    p.rowstat = nullptr;  // -> constant shift
    p.colstat = nullptr;
    p.part_l = ws.part_l;
    p.part_stride = static_cast<int>(npad);
    p.dacc = ws.dacc;
    p.ld_dacc = static_cast<int>(dpad);
    p.use_atomic = p.nchunks > 1;  // (ws.dacc was zeroed by the prep kernel)
    SSVB_TRY(launch_sim_bwd(SIM_MOCO, sv.qhat, npad, qb, k, dpad, p, s));
    moco_fused_finalize_kernel<<<static_cast<unsigned>(ceil_div(n, 8)), 256, 0, s>>>(
        ws.part_l, 4 * p.nchunks, p.part_stride, static_cast<int>(n), static_cast<int>(dpad), sv.pos, c, c, ws.dacc,
        sv.pm, sv.lse2, ws.block_sums, ws.counter, 1.f / static_cast<float>(n), loss);
    SSVB_LAUNCH_CHECK();
    return SSVB_OK;
  }
  moco_plan(p, n, k, c, sim_fwd_bn(dpad), 512 / sim_fwd_bn(dpad));
  p.part_m = ws.part_m;
  p.part_l = ws.part_l;
  p.part_stride = static_cast<int>(npad);
  SSVB_TRY(launch_sim_fwd(SIM_MOCO, sv.qhat, npad, qb, k, dpad, p, s));
  lse_finalize_wide_kernel<SIM_MOCO><<<static_cast<unsigned>(ceil_div(n, 8)), 256, 0, s>>>(
      ws.part_m, ws.part_l, 4 * p.nchunks, p.part_stride, static_cast<int>(n), sv.pos, c, sv.lse2, ws.block_sums,
      ws.counter, 1.f / static_cast<float>(n), loss);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

int ssvb_moco_bwd(const float* query, const float* keys, const float* queue, const void* queue_bf16,
                  int queue_unit_norm, int64_t n, int64_t k, int64_t d, int64_t ld_q, int64_t ld_k, int64_t ld_queue,
                  int normalize, float temperature, const float* grad_out, const void* saved, float* dquery,
                  float* dkeys, int64_t ld_dq, int64_t ld_dk, void* workspace, size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(check_shape(n, k, d, temperature));
  SSVB_TRY(check_rows(query, ld_q));
  SSVB_TRY(check_rows(keys, ld_k));
  if (dquery) SSVB_TRY(check_rows(dquery, ld_dq));
  if (dkeys) SSVB_TRY(check_rows(dkeys, ld_dk));
  if (!grad_out || !saved || !workspace || (!queue && !queue_bf16) || (!dquery && !dkeys)) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_moco_workspace_bytes(n, k, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t dpad = sim_dpad(d), npad = round_up(n, 128);
  MocoSaved sv = moco_saved(const_cast<void*>(saved), n, dpad);
  MocoWs ws = moco_ws(workspace, n, k, dpad);
  const float c = SSVB_LOG2E / temperature;
  if (moco_fused(normalize, queue_unit_norm, temperature)) {
    // sum_j p_aj m_j was produced by the forward pass: the backward is the row-wise finish only (no queue access)
    moco_grad_finish_kernel<<<static_cast<unsigned>(ceil_div(n, 8)), 256, 0, s>>>(
        query, keys, ld_q, ld_k, static_cast<int>(n), static_cast<int>(d), sv.pm, static_cast<int>(dpad), sv,
        normalize, c, 1.f / (static_cast<float>(n) * temperature), grad_out, dquery, dkeys, ld_dq, ld_dk);
    SSVB_LAUNCH_CHECK();
    return SSVB_OK;
  }
  const __nv_bfloat16* qb = nullptr;
  SSVB_TRY(get_queue_bf16(queue, queue_bf16, k, d, ld_queue, dpad, ws, s, &qb));

  SimParams p;
  moco_plan(p, n, k, c, 128, 4);
  p.rowstat = sv.lse2;
  p.colstat = nullptr;
  p.dacc = ws.dacc;
  p.ld_dacc = static_cast<int>(dpad);
  p.use_atomic = p.nchunks > 1;
  if (p.use_atomic) SSVB_CUDA(cudaMemsetAsync(ws.dacc, 0, npad * dpad * sizeof(float), s));
  SSVB_TRY(launch_sim_bwd(SIM_MOCO, sv.qhat, npad, qb, k, dpad, p, s));
  moco_grad_finish_kernel<<<static_cast<unsigned>(ceil_div(n, 8)), 256, 0, s>>>(
      query, keys, ld_q, ld_k, static_cast<int>(n), static_cast<int>(d), ws.dacc, static_cast<int>(dpad), sv,
      normalize, c, 1.f / (static_cast<float>(n) * temperature), grad_out, dquery, dkeys, ld_dq, ld_dk);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

// ------------------------------------------------------------------------------------------------------------
// MoCo with the queue sharded over ranks (SURVEY.md §8e).  See include/ssv_b200.h for the stage contract.
// ------------------------------------------------------------------------------------------------------------
int64_t ssvb_moco_dist_npad(int64_t n_global) { return n_global > 0 ? round_up(n_global, 128) : 0; }
size_t ssvb_moco_dist_workspace_bytes(int64_t n_global, int64_t k_local, int64_t d) {
  if (n_global <= 0 || k_local <= 0 || d <= 0) return 0;
  return moco_ws(nullptr, n_global, k_local, sim_dpad(d)).bytes;
}

int ssvb_moco_dist_prep(const float* query, const float* keys, int64_t n_local, int64_t d, int64_t ld_q, int64_t ld_k,
                        int normalize, int64_t world, int64_t rank, void* qhat_all, float* rowstat_local, void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(check_shape(n_local, 1, d, 1.f));
  SSVB_TRY(check_rows(query, ld_q));
  SSVB_TRY(check_rows(keys, ld_k));
  if (!qhat_all || !rowstat_local || world < 1 || rank < 0 || rank >= world) return SSVB_ERR_INVALID;
  if (reinterpret_cast<uintptr_t>(qhat_all) & 15) return SSVB_ERR_ALIGNMENT;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t dpad = sim_dpad(d), ng = n_local * world, npad = round_up(ng, 128);
  __nv_bfloat16* qh = static_cast<__nv_bfloat16*>(qhat_all);
  if (npad > ng) SSVB_CUDA(cudaMemsetAsync(qh + ng * dpad, 0, (npad - ng) * dpad * sizeof(__nv_bfloat16), s));
  pair_prep_kernel<<<static_cast<unsigned>(ceil_div(n_local, 8)), 256, 0, s>>>(
      query, keys, static_cast<int>(n_local), static_cast<int>(d), ld_q, ld_k, normalize, 0, qh + rank * n_local * dpad,
      nullptr, static_cast<int>(dpad), rowstat_local, rowstat_local + n_local, rowstat_local + 2 * n_local, nullptr);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

int ssvb_moco_dist_shard_fwd(const void* qhat_all, int64_t n_global, const float* queue_shard,
                             const void* queue_shard_bf16, int64_t k_local, int64_t d, int64_t ld_queue,
                             float temperature, const float* rowstat_local, int64_t n_local, float* part_local,
                             void* workspace, size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(check_shape(n_global, k_local, d, temperature));
  if (!qhat_all || !rowstat_local || !part_local || !workspace || (!queue_shard && !queue_shard_bf16) ||
      n_local <= 0 || n_local > n_global)
    return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_moco_dist_workspace_bytes(n_global, k_local, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t dpad = sim_dpad(d), npad = round_up(n_global, 128);
  MocoWs ws = moco_ws(workspace, n_global, k_local, dpad);
  const float c = SSVB_LOG2E / temperature;
  const __nv_bfloat16* qb = nullptr;
  SSVB_TRY(get_queue_bf16(queue_shard, queue_shard_bf16, k_local, d, ld_queue, dpad, ws, s, &qb));
  SimParams p;
  moco_plan(p, n_global, k_local, c, sim_fwd_bn(dpad), 512 / sim_fwd_bn(dpad));
  p.part_m = ws.part_m;
  p.part_l = ws.part_l;
  p.part_stride = static_cast<int>(npad);
  SSVB_TRY(launch_sim_fwd(SIM_MOCO, qhat_all, npad, qb, k_local, dpad, p, s));
  shard_combine_kernel<<<static_cast<unsigned>(ceil_div(n_global, 8)), 256, 0, s>>>(
      ws.part_m, ws.part_l, 4 * p.nchunks, p.part_stride, static_cast<int>(n_global), part_local, part_local + n_global);
  SSVB_LAUNCH_CHECK();
  SSVB_CUDA(cudaMemcpyAsync(part_local + 2 * n_global, rowstat_local + 2 * n_local, n_local * sizeof(float),
                            cudaMemcpyDeviceToDevice, s));
  return SSVB_OK;
}

int ssvb_moco_dist_finalize(const float* part_all, int64_t world, int64_t n_local, float temperature, float* lse2_all,
                            float* loss, void* workspace, size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  if (!part_all || !lse2_all || !loss || !workspace || world < 1 || n_local < 1 || !(temperature > 0.f))
    return SSVB_ERR_INVALID;
  const int64_t ng = world * n_local;
  const int64_t nblk = ceil_div(ng, 256);
  if (workspace_bytes < static_cast<size_t>(nblk + 8) * sizeof(float) + 256) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Carver cv(workspace);
  unsigned int* counter = cv.take<unsigned int>(4);
  float* block_sums = cv.take<float>(nblk + 8);
  SSVB_CUDA(cudaMemsetAsync(counter, 0, 16, s));
  shard_finalize_kernel<<<static_cast<unsigned>(nblk), 256, 0, s>>>(part_all, static_cast<int>(world),
                                                                    static_cast<int>(n_local), SSVB_LOG2E / temperature,
                                                                    lse2_all, block_sums, counter,
                                                                    1.f / static_cast<float>(ng), loss);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

int ssvb_moco_dist_shard_bwd(const void* qhat_all, int64_t n_global, const float* queue_shard,
                             const void* queue_shard_bf16, int64_t k_local, int64_t d, int64_t ld_queue,
                             float temperature, const float* lse2_all, float* dacc_partial, void* workspace,
                             size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(check_shape(n_global, k_local, d, temperature));
  if (!qhat_all || !lse2_all || !dacc_partial || !workspace || (!queue_shard && !queue_shard_bf16))
    return SSVB_ERR_INVALID;
  if (reinterpret_cast<uintptr_t>(dacc_partial) & 15) return SSVB_ERR_ALIGNMENT;
  if (workspace_bytes < ssvb_moco_dist_workspace_bytes(n_global, k_local, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t dpad = sim_dpad(d), npad = round_up(n_global, 128);
  MocoWs ws = moco_ws(workspace, n_global, k_local, dpad);
  const float c = SSVB_LOG2E / temperature;
  const __nv_bfloat16* qb = nullptr;
  SSVB_TRY(get_queue_bf16(queue_shard, queue_shard_bf16, k_local, d, ld_queue, dpad, ws, s, &qb));
  SimParams p;
  moco_plan(p, n_global, k_local, c, 128, 4);
  p.rowstat = const_cast<float*>(lse2_all);
  p.colstat = nullptr;
  p.dacc = dacc_partial;
  p.ld_dacc = static_cast<int>(dpad);
  p.use_atomic = p.nchunks > 1;
  if (p.use_atomic) SSVB_CUDA(cudaMemsetAsync(dacc_partial, 0, npad * dpad * sizeof(float), s));
  SSVB_TRY(launch_sim_bwd(SIM_MOCO, qhat_all, npad, qb, k_local, dpad, p, s));
  return SSVB_OK;
}

int ssvb_moco_dist_finish(const float* query, const float* keys, int64_t n_local, int64_t n_global, int64_t d,
                          int64_t ld_q, int64_t ld_k, int normalize, float temperature, const float* rowstat_local,
                          const float* lse2_local, const float* dacc_local, const float* grad_out, float* dquery,
                          float* dkeys, int64_t ld_dq, int64_t ld_dk, void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(check_shape(n_local, 1, d, temperature));
  SSVB_TRY(check_rows(query, ld_q));
  SSVB_TRY(check_rows(keys, ld_k));
  if (dquery) SSVB_TRY(check_rows(dquery, ld_dq));
  if (dkeys) SSVB_TRY(check_rows(dkeys, ld_dk));
  if (!rowstat_local || !lse2_local || !dacc_local || !grad_out || (!dquery && !dkeys) || n_global < n_local)
    return SSVB_ERR_INVALID;
  if (reinterpret_cast<uintptr_t>(dacc_local) & 15) return SSVB_ERR_ALIGNMENT;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t dpad = sim_dpad(d);
  MocoSaved sv{};
  sv.inv_q = const_cast<float*>(rowstat_local);
  sv.inv_k = const_cast<float*>(rowstat_local) + n_local;
  sv.pos = const_cast<float*>(rowstat_local) + 2 * n_local;
  sv.lse2 = const_cast<float*>(lse2_local);
  moco_grad_finish_kernel<<<static_cast<unsigned>(ceil_div(n_local, 8)), 256, 0, s>>>(
      query, keys, ld_q, ld_k, static_cast<int>(n_local), static_cast<int>(d), dacc_local, static_cast<int>(dpad), sv,
      normalize, SSVB_LOG2E / temperature, 1.f / (static_cast<float>(n_global) * temperature), grad_out, dquery, dkeys,
      ld_dq, ld_dk);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

// ------------------------------------------------------------------------------------------------------------
// PirlLoss (SURVEY.md §8f) — utils/losses.py:92-117, call site models/pirl.py:134.  See include/ssv_b200.h.
// ------------------------------------------------------------------------------------------------------------
size_t ssvb_pirl_saved_bytes(int64_t n, int64_t d) {
  if (n <= 0 || d <= 0) return 0;
  return pirl_saved(nullptr, n, sim_dpad(d)).bytes;
}
size_t ssvb_pirl_workspace_bytes(int64_t n, int64_t k, int64_t d) { return ssvb_moco_workspace_bytes(n, k, d); }

int ssvb_pirl_fwd(const float* img, const float* patch, const float* mem_pos, const float* mem_neg, int64_t n, int64_t k,
                  int64_t d, int64_t ld_img, int64_t ld_patch, int64_t ld_pos, int64_t ld_neg, int normalize,
                  float temperature, float loss_weight, float* loss, void* saved, void* workspace,
                  size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(check_shape(n, k, d, temperature));
  SSVB_TRY(check_rows(img, ld_img));
  SSVB_TRY(check_rows(patch, ld_patch));
  SSVB_TRY(check_rows(mem_pos, ld_pos));
  SSVB_TRY(check_rows(mem_neg, ld_neg));
  if (!loss || !saved || !workspace) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_pirl_workspace_bytes(n, k, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t dpad = sim_dpad(d), npad = round_up(n, 128);
  PirlSaved sv = pirl_saved(saved, n, dpad);
  MocoWs ws = moco_ws(workspace, n, k, dpad);
  const float c = SSVB_LOG2E / temperature;
  const int ni = static_cast<int>(n), di = static_cast<int>(d), dp = static_cast<int>(dpad);
  const unsigned pgrid = static_cast<unsigned>(ceil_div(n, 8));
  if (npad > n) SSVB_CUDA(cudaMemsetAsync(sv.qhat + n * dpad, 0, (npad - n) * dpad * sizeof(__nv_bfloat16), s));
  // "query" = memory_pos rows AS STORED (never normalised, :107-109); "keys" = patch / img rows (normalised if asked)
  const int mask = normalize ? 2 : 0;
  pair_prep_kernel<<<pgrid, 256, 0, s>>>(mem_pos, patch, ni, di, ld_pos, ld_patch, 0, 0, sv.qhat, nullptr, dp, sv.unused,
                                         sv.inv_patch, sv.pos_patch, nullptr, mask, 1.f, ws.counter);
  SSVB_LAUNCH_CHECK();
  pair_prep_kernel<<<pgrid, 256, 0, s>>>(mem_pos, img, ni, di, ld_pos, ld_img, 0, 0, nullptr, nullptr, dp, sv.unused,
                                         sv.inv_img, sv.pos_img, nullptr, mask);
  SSVB_LAUNCH_CHECK();
  const __nv_bfloat16* qb = nullptr;
  SSVB_TRY(get_queue_bf16(mem_neg, nullptr, k, d, ld_neg, dpad, ws, s, &qb));
  // the negatives' logits are shared by both heads (:109): one pass of the tensor-core kernel, one finalize for both
  SimParams p;
  moco_plan(p, n, k, c, sim_fwd_bn(dpad), 512 / sim_fwd_bn(dpad));
  p.part_m = ws.part_m;
  p.part_l = ws.part_l;
  p.part_stride = static_cast<int>(npad);
  SSVB_TRY(launch_sim_fwd(SIM_MOCO, sv.qhat, npad, qb, k, dpad, p, s));
  pirl_finalize_kernel<<<pgrid, 256, 0, s>>>(ws.part_m, ws.part_l, 4 * p.nchunks, p.part_stride, ni, sv.pos_patch,
                                             sv.pos_img, c, sv.lse_patch, sv.lse_img, loss_weight, 1.f - loss_weight,
                                             ws.block_sums, ws.counter, 1.f / static_cast<float>(n), loss);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

int ssvb_pirl_bwd(const float* img, const float* patch, const float* mem_pos, int64_t n, int64_t d, int64_t ld_img,
                  int64_t ld_patch, int64_t ld_pos, int normalize, float temperature, float loss_weight,
                  const float* grad_out, const void* saved, float* d_img, float* d_patch, int64_t ld_dimg,
                  int64_t ld_dpatch, void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(check_shape(n, 1, d, temperature));
  SSVB_TRY(check_rows(img, ld_img));
  SSVB_TRY(check_rows(patch, ld_patch));
  SSVB_TRY(check_rows(mem_pos, ld_pos));
  if (d_img) SSVB_TRY(check_rows(d_img, ld_dimg));
  if (d_patch) SSVB_TRY(check_rows(d_patch, ld_dpatch));
  if (!grad_out || !saved || (!d_img && !d_patch)) return SSVB_ERR_INVALID;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PirlSaved sv = pirl_saved(const_cast<void*>(saved), n, sim_dpad(d));
  pirl_grad_kernel<<<static_cast<unsigned>(ceil_div(n, 8)), 256, 0, s>>>(
      img, patch, mem_pos, ld_img, ld_patch, ld_pos, static_cast<int>(n), static_cast<int>(d), sv, normalize,
      SSVB_LOG2E / temperature, 1.f / (static_cast<float>(n) * temperature), loss_weight, grad_out, d_img, d_patch, ld_dimg,
      ld_dpatch);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

}  // extern "C"
