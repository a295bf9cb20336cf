// Sinkhorn-Knopp codes (SwAV) — replaces SwavLoss.compute_codes_sinkhorn (reference utils/losses.py:213-224).
//
// Scaling-vector form of the reference's dense iteration (never materialises Q or its transpose):
//   E_bk = exp((s_bk - smax)/eps)            (the global shift cancels in the first normalisation)
//   u_k  = sum_b E_bk * beta_b ;  alpha_k = (1/K) / u_k          (row / prototype normalisation, :219-220)
//   v_b  = sum_k alpha_k E_bk ;   beta_b  = (1/B) / v_b          (column / sample normalisation, :221)
//   codes_bk = alpha_k E_bk / v_b                                 (final column normalisation, :222-223)
// One pass over the scores per iteration (they stay L2-resident: 49 MB at 4096x3000): each warp stages the
// exp'd row in shared memory, reduces v_b with shuffles, then either feeds the next iteration's column sums
// (block-local shared accumulators -> per-block partial rows -> deterministic tree) or writes the codes.
#include "sim_host.cuh"

using namespace ssvb;

namespace {

struct SkWs {
  float* smax_part;  // [grid]
  float* smax;       // [1]
  float* upart;      // [grid x kpad]
  float* alpha;      // [kSkMaxProb x kpad]  (one scaling vector per batched problem)
  unsigned int* counter;
  size_t bytes;
  int grid;
  int kpad;
};
inline int sk_grid() { return num_sms() * 2; }
// Independent problems of one shape run in ONE launch per pass (SwAV: the two views' score matrices): problem p = blockIdx.y
// takes its own rows / alpha / smax / partial rows; the CTAs of a launch are split evenly between the problems.
constexpr int kSkMaxProb = 2;
SkWs sk_ws(void* base, int64_t k) {
  Carver c(base);
  SkWs w;
  w.grid = sk_grid();
  w.kpad = static_cast<int>(round_up(k, 4));
  w.smax_part = c.take<float>(w.grid);
  w.smax = c.take<float>(4);
  w.upart = c.take<float>(static_cast<size_t>(w.grid) * w.kpad);
  w.alpha = c.take<float>(static_cast<size_t>(kSkMaxProb) * w.kpad);
  w.counter = c.take<unsigned int>(4);
  w.bytes = c.used();
  return w;
}

__global__ void sk_max_kernel(const float* __restrict__ s, int64_t b, int k, int64_t ld, float* part,
                              unsigned int* counter, float* __restrict__ out) {
  float m = -INFINITY;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  for (int64_t r = gw; r < b; r += warps)
    for (int c = lane; c < k; c += 32) m = fmaxf(m, __ldg(s + r * ld + c));
  __shared__ float red[32];
  m = warp_max(m);
  if (lane == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : -INFINITY;
    t = warp_max(t);
    // last block to finish reduces the per-block maxima (max is order-independent -> deterministic)
    __shared__ bool is_last;
    if (threadIdx.x == 0) {
      part[blockIdx.x] = t;
      __threadfence();
      is_last = (atomicAdd(counter, 1u) == gridDim.x - 1);
    }
    __syncwarp();
    is_last = __shfl_sync(0xffffffffu, is_last ? 1 : 0, 0) != 0;
    if (is_last) {
      __threadfence();
      float m = -INFINITY;
      for (unsigned int i = threadIdx.x; i < gridDim.x; i += 32) m = fmaxf(m, __ldcg(part + i));
      m = warp_max(m);
      if (threadIdx.x == 0) {
        out[0] = m;
        *counter = 0;
      }
    }
  }
}
constexpr int kSkSlices = 32;  // row slices per column group in the alpha kernels (block = 32 x 32 threads)
// alpha_k = (1/K) / sum_g upart[g][k].  block (32 columns, kSkSlices row-slices): each thread sums every 8th partial row of
// its column (coalesced 128-byte row segments), fixed-order combine through shared memory -> ~94 CTAs instead of 12.
__global__ void sk_alpha_kernel(const float* __restrict__ upart, int grid, int kpad, int k, float* __restrict__ alpha,
                                int raw = 0) {
  pdl_launch_dependents();  // the next pass may start streaming score rows now; it waits before it reads alpha
  upart += static_cast<size_t>(blockIdx.y) * grid * kpad;  // batched problems: blockIdx.y (0 for a single problem)
  alpha += static_cast<size_t>(blockIdx.y) * kpad;
  __shared__ float sh[kSkSlices][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  float u = 0.f;
  if (c < k) {
#pragma unroll 6
    for (int g = threadIdx.y; g < grid; g += kSkSlices) u += upart[static_cast<size_t>(g) * kpad + c];
  }
  sh[threadIdx.y][threadIdx.x] = u;
  __syncthreads();
  if (threadIdx.y == 0 && c < k) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < kSkSlices; ++i) t += sh[i][threadIdx.x];
    alpha[c] = raw ? t : (1.f / static_cast<float>(k)) / t;  // raw: the column sums themselves (distributed path)
  }
}

// first alpha after the online-max PHASE 0 of the fast path: block partials carry their own reference maximum
__global__ void sk_alpha0_kernel(const float* __restrict__ upart, const float* __restrict__ mpart, int grid, int kpad,
                                 int k, float inv_eps_log2e, float* __restrict__ alpha, float* __restrict__ smax,
                                 int raw = 0) {
  pdl_launch_dependents();  // (see sk_alpha_kernel)
  upart += static_cast<size_t>(blockIdx.y) * grid * kpad;  // batched problems: blockIdx.y (0 for a single problem)
  mpart += static_cast<size_t>(blockIdx.y) * grid;
  alpha += static_cast<size_t>(blockIdx.y) * kpad;
  smax += blockIdx.y;
  __shared__ float sh[kSkSlices][33];
  __shared__ float msh[32];
  const int tid = threadIdx.y * 32 + threadIdx.x;
  float m = -INFINITY;
  for (int g = tid; g < grid; g += 32 * kSkSlices) m = fmaxf(m, mpart[g]);
  m = warp_max(m);
  if (threadIdx.x == 0) msh[threadIdx.y] = m;
  __syncthreads();
  float M = -INFINITY;
#pragma unroll
  for (int i = 0; i < kSkSlices; ++i) M = fmaxf(M, msh[i]);
  const int c = blockIdx.x * 32 + threadIdx.x;
  float u = 0.f;
  if (c < k) {
#pragma unroll 6
    for (int g = threadIdx.y; g < grid; g += kSkSlices) {
      const float mg = mpart[g];
      const float x = upart[static_cast<size_t>(g) * kpad + c];
      if (mg != -INFINITY) u = fmaf(x, ex2f((mg - M) * inv_eps_log2e), u);
    }
  }
  sh[threadIdx.y][threadIdx.x] = u;
  __syncthreads();
  if (threadIdx.y == 0 && c < k) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < kSkSlices; ++i) t += sh[i][threadIdx.x];
    alpha[c] = raw ? t : (1.f / static_cast<float>(k)) / t;
  }
  if (blockIdx.x == 0 && tid == 0) smax[0] = M;
}

// distributed: combine the gathered per-rank column sums u_all [world][k+1] (entry k of a PHASE-0 block = that rank's
// reference maximum) in RANK ORDER -> alpha_k = (1/K) / u_k and (PHASE 0) the global maximum.
__global__ void sk_dist_alpha_kernel(const float* __restrict__ u_all, int world, int64_t rank_stride, int k, int phase0,
                                     float inv_eps_log2e,
                                     float* __restrict__ alpha, float* __restrict__ smax) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  float M = -INFINITY;
  if (phase0)
    for (int r = 0; r < world; ++r) M = fmaxf(M, u_all[r * rank_stride + k]);
  if (c < k) {
    float u = 0.f;
    for (int r = 0; r < world; ++r) {
      const float* blk = u_all + r * rank_stride;
      if (phase0) {
        const float mr = blk[k];
        if (mr != -INFINITY) u = fmaf(blk[c], ex2f((mr - M) * inv_eps_log2e), u);
      } else {
        u += blk[c];
      }
    }
    alpha[c] = (1.f / static_cast<float>(k)) / u;
  }
  if (phase0 && blockIdx.x == 0 && threadIdx.x == 0) smax[0] = M;
}

// PHASE 0: u_k = sum_b E_bk                     (beta uniform: the reference's Q / sum(Q) scalar cancels)
// PHASE 1: v_b from alpha; u_k += E_bk / (B v_b) (middle iterations)
// PHASE 2: v_b from alpha; codes = alpha E / v_b (last pass)
// REGACC: column sums are accumulated in registers (thread <-> columns tid + 256 j, j < 16, i.e. K <= 4096)
// from the 8 rows the block's warps just staged in shared memory: no atomics, deterministic.  Otherwise
// (wide K) block-local shared-memory atomics.
constexpr int kSkJ = 16;
template <int PHASE, bool REGACC>
__global__ void sk_pass_kernel(const float* __restrict__ s, int64_t b, int k, int64_t ld, float inv_eps_log2e,
                               const float* __restrict__ smax, const float* __restrict__ alpha,
                               float* __restrict__ upart, int kpad, float* __restrict__ codes, int64_t ldc,
                               float inv_b) {
  extern __shared__ float sk_smem[];
  __shared__ float beta_s[32];
  const int nwarp = blockDim.x >> 5;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* uloc = sk_smem;                       // [kpad] (atomic path only)
  float* erow = sk_smem + kpad + w * kpad;     // this warp's exp'd row
  const float shift = smax[0] * inv_eps_log2e;
  float acc[kSkJ];
#pragma unroll
  for (int j = 0; j < kSkJ; ++j) acc[j] = 0.f;
  if (PHASE != 2 && !REGACC) {
    for (int c = threadIdx.x; c < kpad; c += blockDim.x) uloc[c] = 0.f;
    __syncthreads();
  }
  for (int64_t base = static_cast<int64_t>(blockIdx.x) * nwarp; base < b; base += static_cast<int64_t>(gridDim.x) * nwarp) {
    const int64_t r = base + w;
    if (r < b) {
      const float* row = s + r * ld;
      float v = 0.f;
      for (int c = lane; c < k; c += 32) {
        const float e = ex2f(fmaf(__ldg(row + c), inv_eps_log2e, -shift));
        erow[c] = e;
        if (PHASE != 0) v += e * alpha[c];
      }
      float beta = 1.f;
      if (PHASE != 0) {
        v = warp_sum(v);
        beta = inv_b / v;
      }
      __syncwarp();
      if (PHASE == 2) {
        const float iv = 1.f / v;
        float* out = codes + r * ldc;
        for (int c = lane; c < k; c += 32) out[c] = erow[c] * alpha[c] * iv;
        __syncwarp();
      } else if (!REGACC) {
        for (int c = lane; c < k; c += 32) atomicAdd(&uloc[c], erow[c] * beta);
        __syncwarp();
      } else if (lane == 0) {
        beta_s[w] = beta;
      }
    }
    if (PHASE != 2 && REGACC) {
      __syncthreads();
      const int nvalid = static_cast<int>(min(static_cast<int64_t>(nwarp), b - base));
#pragma unroll
      for (int j = 0; j < kSkJ; ++j) {
        const int c = threadIdx.x + j * blockDim.x;
        if (c < k) {
          float a = acc[j];
          for (int ww = 0; ww < nvalid; ++ww) a = fmaf(sk_smem[kpad + ww * kpad + c], beta_s[ww], a);
          acc[j] = a;
        }
      }
      __syncthreads();
    }
  }
  if (PHASE != 2) {
    if (REGACC) {
#pragma unroll
      for (int j = 0; j < kSkJ; ++j) {
        const int c = threadIdx.x + j * blockDim.x;
        if (c < k) upart[static_cast<size_t>(blockIdx.x) * kpad + c] = acc[j];
      }
    } else {
      __syncthreads();
      for (int c = threadIdx.x; c < k; c += blockDim.x) upart[static_cast<size_t>(blockIdx.x) * kpad + c] = uloc[c];
    }
  }
}

// float4 per lane of one score row held in registers by the fast path: K <= 32 * 4 * kSkNV = 3072
constexpr int kSkNV = 24;
constexpr int kSkConsumers = 7;  // + 1 producer warp = 8 warps: 2 per SM sub-partition, so 255 registers stay available

// Fast path (K <= 3072, K % 4 == 0, 16-byte aligned rows): the row stream is decoupled from the math by a TMA ring.
// One producer warp issues 1-D bulk copies (cp.async.bulk, one whole score row = K*4 bytes per copy, completion on an
// mbarrier) into a ring of `nst` row slots (up to 16 rows = 192 KB in flight per SM); the scaling vector alpha arrives
// by one more bulk copy (a serial LDG -> STS prologue cost 27 % of the kernel).  7 consumer warps take rows round
// robin, pull the row from shared memory into registers (24 float4 per lane), hand the slot straight back to the
// producer, and run the per-row math (online max in PHASE 0, column sums in registers).  The ring is reused for the
// fixed-order cross-warp combine at the end.
// Measured (profiles/r1_sinkhorn_tuning.md): a pass is bound by the ~6.5 TB/s the L2 -> SM fabric delivers (one row
// per warp every ~1.9 us while its math takes ~1 us), so caching exp() between passes or fusing the passes into one
// cooperative kernel (both tried) buys nothing; the remaining cost is the fixed ~3-4 us per launch.
template <int PHASE>
__global__ void __launch_bounds__((kSkConsumers + 1) * 32, 1)
sk_tma_kernel(const float* __restrict__ s, int64_t b, int k, int64_t ld, float inv_eps_log2e,
              const float* __restrict__ smax, const float* __restrict__ alpha, float* __restrict__ upart, int kpad,
              float* __restrict__ codes, int64_t ldc, float* __restrict__ mpart, float inv_b, int nst, int rowf,
              int64_t pstride_s, int64_t pstride_c) {
  extern __shared__ __align__(128) float sk_smem[];  // [nst][rowf] ring | [kpad] alpha | 2*nst + 1 mbarriers
  if (gridDim.y > 1) {  // batched independent problems (same b, k): problem blockIdx.y, gridDim.x CTAs each
    const size_t pb = blockIdx.y;
    s += pb * pstride_s;
    codes += pb * pstride_c;
    smax += pb;
    alpha += pb * kpad;
    upart += pb * gridDim.x * kpad;
    mpart += pb * gridDim.x;
  }
  float* ring = sk_smem;
  float* alpha_s = sk_smem + static_cast<size_t>(nst) * rowf;
  uint64_t* full = reinterpret_cast<uint64_t*>(alpha_s + kpad);
  uint64_t* empty = full + nst;
  uint64_t* abar = empty + nst;
  __shared__ float mw_s[kSkConsumers];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int k4 = k >> 2;
  const int n_my = blockIdx.x < b ? static_cast<int>((b - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0;
  if (threadIdx.x == 0) {
    for (int i = 0; i < nst; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(abar, 1);
    fence_barrier_init();
  }
  __syncthreads();

  float4 acc[kSkNV];
#pragma unroll
  for (int j = 0; j < kSkNV; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  // PHASE 0 needs no prior max pass: every warp keeps a running max Mw of the scores it has seen and rescales its
  // column sums when Mw grows (online, like a streaming softmax); blocks are combined with exp((M_blk - M)/eps) in
  // sk_alpha0_kernel, which also publishes the global max for the later passes.
  float Mw = -INFINITY;

  if (w == kSkConsumers) {
    // ---- producer: one elected lane streams this CTA's rows through the ring
    if (lane == 0) {
      const uint32_t bytes = static_cast<uint32_t>(k) * 4u;
      // the score rows do not depend on the previous kernel (the alpha kernel): when this pass was launched with
      // programmatic stream serialization the first ring-full of rows streams in while that kernel still runs
      const int pre = (PHASE != 0) ? (n_my < nst ? n_my : nst) : 0;
      for (int i = 0; i < pre; ++i) {
        const int64_t r = blockIdx.x + static_cast<int64_t>(i) * gridDim.x;
        mbar_expect_tx(&full[i], bytes);
        bulk_load_1d(ring + static_cast<size_t>(i) * rowf, s + r * ld, bytes, &full[i]);
      }
      if (PHASE != 0) {
        pdl_wait();
        mbar_expect_tx(abar, bytes);
        bulk_load_1d(alpha_s, alpha, bytes, abar);
      }
      for (int i = pre; i < n_my; ++i) {
        const int slot = i % nst;
        if (i >= nst) mbar_wait(&empty[slot], ((i / nst) - 1) & 1);
        const int64_t r = blockIdx.x + static_cast<int64_t>(i) * gridDim.x;
        mbar_expect_tx(&full[slot], bytes);
        bulk_load_1d(ring + static_cast<size_t>(slot) * rowf, s + r * ld, bytes, &full[slot]);
      }
    }
    if (PHASE != 0) pdl_wait();  // the whole producer warp takes part in the combine that overwrites upart
  } else {
    float shift = 0.f;
    if (PHASE != 0) {
      pdl_wait();  // smax / alpha come from the previous kernel
      shift = smax[0] * inv_eps_log2e;
      mbar_wait(abar, 0);
    }
    for (int i = w; i < n_my; i += kSkConsumers) {
      const int slot = i % nst;
      const int64_t r = blockIdx.x + static_cast<int64_t>(i) * gridDim.x;
      mbar_wait(&full[slot], (i / nst) & 1);
      const float4* row = reinterpret_cast<const float4*>(ring + static_cast<size_t>(slot) * rowf);
      float4 e[kSkNV];
#pragma unroll
      for (int j = 0; j < kSkNV; ++j) {
        const int c4 = lane + 32 * j;
        e[j] = (c4 < k4) ? row[c4] : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[slot]);  // the row now lives in registers: give the slot back
      if (PHASE == 0) {
        float rm = -INFINITY;
#pragma unroll
        for (int j = 0; j < kSkNV; ++j) rm = fmaxf(rm, fmaxf(fmaxf(e[j].x, e[j].y), fmaxf(e[j].z, e[j].w)));
        rm = warp_max(rm);
        if (rm > Mw) {  // warp-uniform
          const float sc = ex2f((Mw - rm) * inv_eps_log2e);  // 0 on the first row (Mw = -inf)
#pragma unroll
          for (int j = 0; j < kSkNV; ++j) { acc[j].x *= sc; acc[j].y *= sc; acc[j].z *= sc; acc[j].w *= sc; }
          Mw = rm;
        }
        shift = Mw * inv_eps_log2e;
      }
      float v = 0.f;
#pragma unroll
      for (int j = 0; j < kSkNV; ++j) {
        e[j].x = ex2f(fmaf(e[j].x, inv_eps_log2e, -shift));
        e[j].y = ex2f(fmaf(e[j].y, inv_eps_log2e, -shift));
        e[j].z = ex2f(fmaf(e[j].z, inv_eps_log2e, -shift));
        e[j].w = ex2f(fmaf(e[j].w, inv_eps_log2e, -shift));
        if (PHASE != 0) {
          const int c4 = lane + 32 * j;
          if (c4 < k4) {
            const float4 a = reinterpret_cast<const float4*>(alpha_s)[c4];
            v += (e[j].x * a.x + e[j].y * a.y) + (e[j].z * a.z + e[j].w * a.w);
          }
        }
      }
      if (PHASE == 0) {
#pragma unroll
        for (int j = 0; j < kSkNV; ++j) { acc[j].x += e[j].x; acc[j].y += e[j].y; acc[j].z += e[j].z; acc[j].w += e[j].w; }
      } else {
        v = warp_sum(v);
        if (PHASE == 1) {
          const float beta = inv_b / v;
#pragma unroll
          for (int j = 0; j < kSkNV; ++j) {
            acc[j].x = fmaf(e[j].x, beta, acc[j].x); acc[j].y = fmaf(e[j].y, beta, acc[j].y);
            acc[j].z = fmaf(e[j].z, beta, acc[j].z); acc[j].w = fmaf(e[j].w, beta, acc[j].w);
          }
        } else {
          const float iv = 1.f / v;
          float4* out = reinterpret_cast<float4*>(codes + r * ldc);
#pragma unroll
          for (int j = 0; j < kSkNV; ++j) {
            const int c4 = lane + 32 * j;
            if (c4 < k4) {
              const float4 a = reinterpret_cast<const float4*>(alpha_s)[c4];
              out[c4] = make_float4(e[j].x * a.x * iv, e[j].y * a.y * iv, e[j].z * a.z * iv, e[j].w * a.w * iv);
            }
          }
        }
      }
    }
  }
  if (PHASE != 2) {
    // every bulk copy has been consumed (each consumer waited on all of its rows): the ring is free for the combine
    __syncthreads();
    if (w < kSkConsumers) {
      float* mine = ring + static_cast<size_t>(w) * kpad;
#pragma unroll
      for (int j = 0; j < kSkNV; ++j) {
        const int c4 = lane + 32 * j;
        if (c4 < k4) reinterpret_cast<float4*>(mine)[c4] = acc[j];
      }
      if (PHASE == 0 && lane == 0) mw_s[w] = Mw;
    }
    __syncthreads();
    float wsc[kSkConsumers];
#pragma unroll
    for (int ww = 0; ww < kSkConsumers; ++ww) wsc[ww] = 1.f;
    if (PHASE == 0) {
      float mb = -INFINITY;
      for (int ww = 0; ww < kSkConsumers; ++ww) mb = fmaxf(mb, mw_s[ww]);
      for (int ww = 0; ww < kSkConsumers; ++ww)
        wsc[ww] = (mw_s[ww] == -INFINITY) ? 0.f : ex2f((mw_s[ww] - mb) * inv_eps_log2e);
      if (threadIdx.x == 0) mpart[blockIdx.x] = mb;
    }
    for (int c = threadIdx.x; c < k; c += blockDim.x) {
      float t = 0.f;
#pragma unroll
      for (int ww = 0; ww < kSkConsumers; ++ww) t = fmaf(ring[static_cast<size_t>(ww) * kpad + c], wsc[ww], t);
      upart[static_cast<size_t>(blockIdx.x) * kpad + c] = t;
    }
  }
}

// ring geometry of sk_tma_kernel for a K-column problem
struct SkRing {
  int nst, rowf;
  size_t smem;
};
inline SkRing sk_ring(int kpad) {
  SkRing g;
  g.rowf = static_cast<int>(round_up(kpad, 32));
  const size_t rowbytes = static_cast<size_t>(g.rowf) * 4, fixed = static_cast<size_t>(kpad) * 4 + 2 * 16 * 8 + 8 + 128;
  int nst = static_cast<int>((212 * 1024 - fixed) / rowbytes);
  if (nst > 16) nst = 16;
  g.nst = nst;  // >= 7 whenever kpad <= 3072 (the combine area needs kSkConsumers * kpad floats inside the ring)
  g.smem = static_cast<size_t>(nst) * rowbytes + static_cast<size_t>(kpad) * 4 + (2 * nst + 1) * 8 + 128;
  return g;
}
template <int PHASE>
int sk_launch_fast(int grid, cudaStream_t s, const float* scores, int64_t b, int k, int64_t ld, float iel, const SkWs& ws,
                   float* codes, int64_t ldc, float inv_b, bool pdl = false, int nprob = 1, int64_t pstride_s = 0,
                   int64_t pstride_c = 0) {
  const SkRing g = sk_ring(ws.kpad);
  SSVB_CUDA(cudaFuncSetAttribute(sk_tma_kernel<PHASE>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(g.smem)));
  if (pdl && PHASE != 0) {
    // programmatic dependent launch behind the alpha kernel: prologue + first ring-full of rows overlap it
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(grid), static_cast<unsigned>(nprob));
    cfg.blockDim = dim3((kSkConsumers + 1) * 32);
    cfg.dynamicSmemBytes = g.smem;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    const float* smax_c = ws.smax;
    const float* alpha_c = ws.alpha;
    SSVB_CUDA(cudaLaunchKernelEx(&cfg, sk_tma_kernel<PHASE>, scores, b, k, ld, iel, smax_c, alpha_c, ws.upart, ws.kpad, codes,
                                 ldc, ws.smax_part, inv_b, g.nst, g.rowf, pstride_s, pstride_c));
  } else {
    sk_tma_kernel<PHASE><<<dim3(static_cast<unsigned>(grid), static_cast<unsigned>(nprob)), (kSkConsumers + 1) * 32, g.smem, s>>>(
        scores, b, k, ld, iel, ws.smax, ws.alpha, ws.upart, ws.kpad, codes, ldc, ws.smax_part, inv_b, g.nst, g.rowf, pstride_s,
        pstride_c);
  }
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

template <int PHASE>
int sk_launch(bool regacc, int grid, int threads, size_t smem, cudaStream_t s, const float* scores, int64_t b, int k,
              int64_t ld, float iel, const SkWs& ws, float* codes, int64_t ldc, float inv_b) {
  if (regacc) {
    SSVB_CUDA(cudaFuncSetAttribute(sk_pass_kernel<PHASE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(smem)));
    sk_pass_kernel<PHASE, true><<<grid, threads, smem, s>>>(scores, b, k, ld, iel, ws.smax, ws.alpha, ws.upart,
                                                            ws.kpad, codes, ldc, inv_b);
  } else {
    SSVB_CUDA(cudaFuncSetAttribute(sk_pass_kernel<PHASE, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(smem)));
    sk_pass_kernel<PHASE, false><<<grid, threads, smem, s>>>(scores, b, k, ld, iel, ws.smax, ws.alpha, ws.upart,
                                                             ws.kpad, codes, ldc, inv_b);
  }
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

}  // namespace

namespace ssvb {
// shared with swav.cu: scores -> codes on `s`.  nprob > 1: that many independent problems of the same shape, problem p
// at scores + p * pstride_s / codes + p * pstride_c (elements).  On the fast path two problems share every launch (each
// pass and alpha kernel covers both: half of the CTAs per problem), which halves the number of dependent launches of
// SwAV's two code assignments (utils/losses.py:232); otherwise they run one after the other.
static int sinkhorn_run_impl(const float* scores, int64_t b, int64_t k, int64_t ld_scores, float eps, int n_iters, float* codes,
                             int64_t ld_codes, void* workspace, cudaStream_t s, int nprob, int64_t pstride_s,
                             int64_t pstride_c, bool scaling_only, bool* batched);
int sinkhorn_run(const float* scores, int64_t b, int64_t k, int64_t ld_scores, float eps, int n_iters, float* codes,
                 int64_t ld_codes, void* workspace, cudaStream_t s, int nprob, int64_t pstride_s, int64_t pstride_c) {
  return sinkhorn_run_impl(scores, b, k, ld_scores, eps, n_iters, codes, ld_codes, workspace, s, nprob, pstride_s, pstride_c,
                           false, nullptr);
}
// Two batched problems WITHOUT the final pass: runs the iterations (passes 0 .. n_iters - 1 and their alpha kernels) and
// hands back the last scaling vectors alpha [2][kpad] and the maxima smax [2] (both live in `workspace`), from which
// codes_bk = alpha_k E_bk / sum_k alpha_k E_bk can be rebuilt row by row (swav.cu: swav_ce_sk4_kernel).  Returns false -
// and launches nothing - when the batched fast path does not apply (the caller then uses sinkhorn_run).
bool sinkhorn_scaling_only(const float* scores, int64_t b, int64_t k, int64_t ld_scores, float eps, int n_iters, void* workspace,
                           cudaStream_t s, int64_t pstride_s, const float** alpha, const float** smax, int* kpad, int* rc) {
  bool batched = false;
  // (codes = scores: only its alignment is looked at on this path - nothing is written)
  *rc = sinkhorn_run_impl(scores, b, k, ld_scores, eps, n_iters, const_cast<float*>(scores), ld_scores, workspace, s, kSkMaxProb,
                          pstride_s, pstride_s, true, &batched);
  if (!batched) return false;
  const SkWs ws = sk_ws(workspace, k);
  *alpha = ws.alpha;
  *smax = ws.smax;
  *kpad = ws.kpad;
  return true;
}
static int sinkhorn_run_impl(const float* scores, int64_t b, int64_t k, int64_t ld_scores, float eps, int n_iters, float* codes,
                             int64_t ld_codes, void* workspace, cudaStream_t s, int nprob, int64_t pstride_s,
                             int64_t pstride_c, bool scaling_only, bool* batched) {
  SkWs ws = sk_ws(workspace, k);
  const int kk = static_cast<int>(k);
  const float iel = SSVB_LOG2E / eps;
  const float inv_b = 1.f / static_cast<float>(b);
  int nwarp = 8;
  while (nwarp > 1 && static_cast<size_t>(nwarp + 1) * ws.kpad * 4 > 200 * 1024) nwarp >>= 1;
  const size_t smem = static_cast<size_t>(nwarp + 1) * ws.kpad * 4;
  if (smem > 200 * 1024) return SSVB_ERR_UNSUPPORTED;
  const int threads = nwarp * 32;
  const bool regacc = (nwarp == 8) && (k <= static_cast<int64_t>(kSkJ) * threads);
  const bool fast = (k % 4 == 0) && (k <= 128 * kSkNV) && (ld_scores % 4 == 0) && (ld_codes % 4 == 0) &&
                    !(reinterpret_cast<uintptr_t>(scores) & 15) && !(reinterpret_cast<uintptr_t>(codes) & 15);
  static const bool no_batch = getenv("SSVB_SK_NO_BATCH") != nullptr;  // A/B switch
  const bool batch = fast && n_iters > 0 && nprob == kSkMaxProb && (pstride_s % 4 == 0) && (pstride_c % 4 == 0) && !no_batch;
  if (batched) *batched = batch;
  if (scaling_only && !batch) return SSVB_OK;  // nothing launched: the caller falls back to sinkhorn_run
  if (nprob > 1 && !batch) {
    for (int p = 0; p < nprob; ++p)
      SSVB_TRY(sinkhorn_run(scores + p * pstride_s, b, k, ld_scores, eps, n_iters, codes + p * pstride_c, ld_codes, workspace,
                            s, 1, 0, 0));
    return SSVB_OK;
  }
  const int np = batch ? nprob : 1;
  // one 8-warp CTA per SM; partial rows [np x fgrid x kpad] (batched: the SMs are split between the problems)
  const int fgrid = batch ? (num_sms() / np > 0 ? num_sms() / np : 1) : num_sms();
  if (!(fast && n_iters > 0)) {  // the fast path finds the max online inside its first pass
    SSVB_CUDA(cudaMemsetAsync(ws.counter, 0, 16, s));
    sk_max_kernel<<<ws.grid, 256, 0, s>>>(scores, b, kk, ld_scores, ws.smax_part, ws.counter, ws.smax);
    SSVB_LAUNCH_CHECK();
  }
  const unsigned agrid = static_cast<unsigned>(ceil_div(k, 256));  // (fill kernel: 256 columns per CTA)
  const dim3 alpha_grid(static_cast<unsigned>(ceil_div(k, 32)), static_cast<unsigned>(np)), alpha_block(32, kSkSlices);
  if (n_iters <= 0) {
    // no iterations: codes = E / rowsum(E)  (alpha = 1)
    fill_kernel<<<agrid, 256, 0, s>>>(ws.alpha, k, 1.f);
    SSVB_LAUNCH_CHECK();
  } else {
    if (fast) {
      SSVB_TRY(sk_launch_fast<0>(fgrid, s, scores, b, kk, ld_scores, iel, ws, codes, ld_codes, inv_b, false, np,
                                 pstride_s, pstride_c));
      sk_alpha0_kernel<<<alpha_grid, alpha_block, 0, s>>>(ws.upart, ws.smax_part, fgrid, ws.kpad, kk, iel, ws.alpha, ws.smax);
    } else {
      SSVB_TRY(sk_launch<0>(regacc, ws.grid, threads, smem, s, scores, b, kk, ld_scores, iel, ws, codes, ld_codes, inv_b));
      sk_alpha_kernel<<<alpha_grid, alpha_block, 0, s>>>(ws.upart, ws.grid, ws.kpad, kk, ws.alpha);
    }
    SSVB_LAUNCH_CHECK();
    for (int it = 1; it < n_iters; ++it) {
      if (fast)
        SSVB_TRY(sk_launch_fast<1>(fgrid, s, scores, b, kk, ld_scores, iel, ws, codes, ld_codes, inv_b, true, np,
                                   pstride_s, pstride_c));
      else SSVB_TRY(sk_launch<1>(regacc, ws.grid, threads, smem, s, scores, b, kk, ld_scores, iel, ws, codes, ld_codes, inv_b));
      sk_alpha_kernel<<<alpha_grid, alpha_block, 0, s>>>(ws.upart, fast ? fgrid : ws.grid, ws.kpad, kk, ws.alpha);
      SSVB_LAUNCH_CHECK();
    }
  }
  if (scaling_only) return SSVB_OK;
  // (n_iters == 0: the final pass follows a fill kernel without the launch_dependents trigger - plain launch)
  if (fast)
    SSVB_TRY(sk_launch_fast<2>(fgrid, s, scores, b, kk, ld_scores, iel, ws, codes, ld_codes, inv_b, n_iters > 0, np,
                               pstride_s, pstride_c));
  else SSVB_TRY(sk_launch<2>(regacc, ws.grid, threads, smem, s, scores, b, kk, ld_scores, iel, ws, codes, ld_codes, inv_b));
  return SSVB_OK;
}
// One pass of the row-sharded (distributed) iteration over this rank's b_local rows.  phase 0: u_local[0..k) = column
// sums of E relative to the LOCAL maximum, u_local[k] = that maximum; phase 1: column sums of E / (b_global v_b) with the
// global alpha / smax; phase 2: codes.  The caller all-gathers u_local and calls sinkhorn_dist_alpha between passes.
int sinkhorn_dist_pass(int phase, const float* scores, int64_t b, int64_t b_global, int64_t k, int64_t ld_scores,
                       float eps, const float* alpha, const float* smax, float* u_local, float* codes, int64_t ld_codes,
                       void* workspace, cudaStream_t s) {
  SkWs ws = sk_ws(workspace, k);
  const int kk = static_cast<int>(k);
  const float iel = SSVB_LOG2E / eps;
  const float inv_b = 1.f / static_cast<float>(b_global);
  int nwarp = 8;
  while (nwarp > 1 && static_cast<size_t>(nwarp + 1) * ws.kpad * 4 > 200 * 1024) nwarp >>= 1;
  const size_t smem = static_cast<size_t>(nwarp + 1) * ws.kpad * 4;
  if (smem > 200 * 1024) return SSVB_ERR_UNSUPPORTED;
  const int threads = nwarp * 32;
  const bool regacc = (nwarp == 8) && (k <= static_cast<int64_t>(kSkJ) * threads);
  // (`fast` must come out the same in all three phases: the caller passes the codes buffer every time)
  const bool fast = (k % 4 == 0) && (k <= 128 * kSkNV) && (ld_scores % 4 == 0) && !(reinterpret_cast<uintptr_t>(scores) & 15) &&
                    (ld_codes % 4 == 0) && !(reinterpret_cast<uintptr_t>(codes) & 15);
  const int fgrid = num_sms();
  const dim3 ablock(32, kSkSlices);
  const unsigned agrid = static_cast<unsigned>(ceil_div(k, 32));
  if (phase != 0) {  // global scaling vector / maximum from the caller
    ws.alpha = const_cast<float*>(alpha);
    ws.smax = const_cast<float*>(smax);
  }
  if (phase == 0) {
    if (fast) {
      SSVB_TRY(sk_launch_fast<0>(fgrid, s, scores, b, kk, ld_scores, iel, ws, codes, ld_codes, inv_b));
      sk_alpha0_kernel<<<agrid, ablock, 0, s>>>(ws.upart, ws.smax_part, fgrid, ws.kpad, kk, iel, u_local, u_local + k, 1);
    } else {
      SSVB_CUDA(cudaMemsetAsync(ws.counter, 0, 16, s));
      sk_max_kernel<<<ws.grid, 256, 0, s>>>(scores, b, kk, ld_scores, ws.smax_part, ws.counter, ws.smax);
      SSVB_LAUNCH_CHECK();
      SSVB_TRY(sk_launch<0>(regacc, ws.grid, threads, smem, s, scores, b, kk, ld_scores, iel, ws, nullptr, 0, inv_b));
      sk_alpha_kernel<<<agrid, ablock, 0, s>>>(ws.upart, ws.grid, ws.kpad, kk, u_local, 1);
      SSVB_LAUNCH_CHECK();
      SSVB_CUDA(cudaMemcpyAsync(u_local + k, ws.smax, sizeof(float), cudaMemcpyDeviceToDevice, s));
    }
    SSVB_LAUNCH_CHECK();
  } else if (phase == 1) {
    if (fast) SSVB_TRY(sk_launch_fast<1>(fgrid, s, scores, b, kk, ld_scores, iel, ws, codes, ld_codes, inv_b));
    else SSVB_TRY(sk_launch<1>(regacc, ws.grid, threads, smem, s, scores, b, kk, ld_scores, iel, ws, nullptr, 0, inv_b));
    sk_alpha_kernel<<<agrid, ablock, 0, s>>>(ws.upart, fast ? fgrid : ws.grid, ws.kpad, kk, u_local, 1);
    SSVB_LAUNCH_CHECK();
    fill_kernel<<<1, 32, 0, s>>>(u_local + k, 1, 0.f);
    SSVB_LAUNCH_CHECK();
  } else {
    if (fast) SSVB_TRY(sk_launch_fast<2>(fgrid, s, scores, b, kk, ld_scores, iel, ws, codes, ld_codes, inv_b));
    else SSVB_TRY(sk_launch<2>(regacc, ws.grid, threads, smem, s, scores, b, kk, ld_scores, iel, ws, codes, ld_codes, inv_b));
  }
  return SSVB_OK;
}
int sinkhorn_dist_alpha(const float* u_all, int64_t world, int64_t rank_stride, int64_t k, int phase0, float eps,
                        float* alpha, float* smax, cudaStream_t s) {
  sk_dist_alpha_kernel<<<static_cast<unsigned>(ceil_div(k, 256)), 256, 0, s>>>(
      u_all, static_cast<int>(world), rank_stride, static_cast<int>(k), phase0, SSVB_LOG2E / eps, alpha, smax);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}
size_t sinkhorn_ws_bytes(int64_t k) { return sk_ws(nullptr, k).bytes; }
}  // namespace ssvb

extern "C" {


size_t ssvb_sinkhorn_workspace_bytes(int64_t b, int64_t k) {
  (void)b;
  return k > 0 ? sk_ws(nullptr, k).bytes : 0;
}

int ssvb_sinkhorn(const float* scores, int64_t b, int64_t k, int64_t ld_scores, float eps, int n_iters, float* codes,
                  int64_t ld_codes, void* workspace, size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  if (!scores || !codes || !workspace || b <= 0 || k <= 0 || !(eps > 0.f) || n_iters < 0 || ld_scores < k ||
      ld_codes < k)
    return SSVB_ERR_INVALID;
  if (workspace_bytes < sk_ws(nullptr, k).bytes) return SSVB_ERR_WORKSPACE;
  return sinkhorn_run(scores, b, k, ld_scores, eps, n_iters, codes, ld_codes, workspace,
                      static_cast<cudaStream_t>(stream), 1, 0, 0);
}

// ---- distributed (sample rows sharded over ranks; SURVEY.md §8e): see include/ssv_b200.h
int ssvb_sinkhorn_dist_pass(int phase, const float* scores, int64_t b_local, int64_t b_global, int64_t k,
                            int64_t ld_scores, float eps, const float* alpha, const float* smax, float* u_local,
                            float* codes, int64_t ld_codes, void* workspace, size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  if (!scores || !workspace || b_local <= 0 || b_global < b_local || k <= 0 || !(eps > 0.f) || ld_scores < k ||
      phase < 0 || phase > 2)
    return SSVB_ERR_INVALID;
  if (phase != 0 && (!alpha || !smax)) return SSVB_ERR_INVALID;
  if (phase != 2 && !u_local) return SSVB_ERR_INVALID;
  if (!codes || ld_codes < k) return SSVB_ERR_INVALID;  // same buffer in every phase (it selects the kernel family)
  if (workspace_bytes < sk_ws(nullptr, k).bytes) return SSVB_ERR_WORKSPACE;
  return sinkhorn_dist_pass(phase, scores, b_local, b_global, k, ld_scores, eps, alpha, smax, u_local, codes, ld_codes,
                            workspace, static_cast<cudaStream_t>(stream));
}
int ssvb_sinkhorn_dist_alpha(const float* u_all, int64_t world, int64_t rank_stride, int64_t k, int phase0, float eps,
                             float* alpha, float* smax, void* stream) {
  SSVB_TRY(check_device_sm100());
  if (!u_all || !alpha || world <= 0 || k <= 0 || rank_stride < k + 1 || !(eps > 0.f) || (phase0 && !smax))
    return SSVB_ERR_INVALID;
  return sinkhorn_dist_alpha(u_all, world, rank_stride, k, phase0, eps, alpha, smax, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
