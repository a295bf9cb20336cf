// SURVEY.md §8(f) "next" rows built to the same bar as the hot path:
//   * multi-tensor EMA of the target / key / teacher network — models/moco.py:108-111, byol.py:120-123,
//     relic.py:119-122, dino.py:129-134:  t = m * t + (1 - m) * s   (bit-exact with the reference's three eager ops)
//   * DinoLoss forward + backward — utils/losses.py:75-89 (call site models/dino.py:161-162) and the centre EMA
//     (models/dino.py:136-141)
// Both are pure HBM-bandwidth kernels: coalesced float4 traffic, warp-shuffle / block reductions, fixed-order sums.
#include "gemm_host.cuh"

using namespace ssvb;

namespace {

// ------------------------------------------------------------------------------------------------ EMA
struct EmaChunk {
  float* t;
  const float* s;
  long long n;
};
constexpr int kEmaChunk = 8192;  // elements per table entry (host side splits tensors into chunks of this size)

// one block per chunk.  __fmul_rn / __fadd_rn keep the reference's rounding: m*t and (1-m)*s are rounded separately and
// then added (three eager ATen kernels), an FMA contraction would differ in the last bit.
__global__ void ema_kernel(const EmaChunk* __restrict__ table, float m, float om) {
  const EmaChunk c = table[blockIdx.x];
  const bool vec = ((reinterpret_cast<uintptr_t>(c.t) | reinterpret_cast<uintptr_t>(c.s)) & 15) == 0;
  if (vec) {
    const long long n4 = c.n >> 2;
    float4* t4 = reinterpret_cast<float4*>(c.t);
    const float4* s4 = reinterpret_cast<const float4*>(c.s);
    // 4 float4 of each operand per thread and trip: 8 independent 16-byte loads in flight before the first use
    // (r1 ncu: 54.7 % of DRAM throughput with long_scoreboard the top stall = too few bytes in flight)
    constexpr int U = 4;
    long long i = threadIdx.x;
    for (; i + (U - 1) * static_cast<long long>(blockDim.x) < n4; i += U * static_cast<long long>(blockDim.x)) {
      float4 a[U], b[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        a[u] = t4[i + u * blockDim.x];
        b[u] = __ldg(s4 + i + u * blockDim.x);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        float4 r;
        r.x = __fadd_rn(__fmul_rn(m, a[u].x), __fmul_rn(om, b[u].x));
        r.y = __fadd_rn(__fmul_rn(m, a[u].y), __fmul_rn(om, b[u].y));
        r.z = __fadd_rn(__fmul_rn(m, a[u].z), __fmul_rn(om, b[u].z));
        r.w = __fadd_rn(__fmul_rn(m, a[u].w), __fmul_rn(om, b[u].w));
        t4[i + u * blockDim.x] = r;
      }
    }
    for (; i < n4; i += blockDim.x) {
      const float4 a = t4[i];
      const float4 b = __ldg(s4 + i);
      float4 r;
      r.x = __fadd_rn(__fmul_rn(m, a.x), __fmul_rn(om, b.x));
      r.y = __fadd_rn(__fmul_rn(m, a.y), __fmul_rn(om, b.y));
      r.z = __fadd_rn(__fmul_rn(m, a.z), __fmul_rn(om, b.z));
      r.w = __fadd_rn(__fmul_rn(m, a.w), __fmul_rn(om, b.w));
      t4[i] = r;
    }
    for (long long i = (n4 << 2) + threadIdx.x; i < c.n; i += blockDim.x)
      c.t[i] = __fadd_rn(__fmul_rn(m, c.t[i]), __fmul_rn(om, __ldg(c.s + i)));
  } else {
    for (long long i = threadIdx.x; i < c.n; i += blockDim.x)
      c.t[i] = __fadd_rn(__fmul_rn(m, c.t[i]), __fmul_rn(om, __ldg(c.s + i)));
  }
}

// ------------------------------------------------------------------------------------------------ DINO
// One block per sample b.  teacher [bs][2][K], student [bs][nv][K], center [K].
//   T_g = softmax((teacher[b, g] - center) / temp_t)           g = 0, 1
//   logp_v = log_softmax(student[b, v] / temp_s)
//   loss = -(1 / (bs nv)) sum_b sum_v sum_k (T_0 + T_1) logp_v                   (utils/losses.py:86-89)
//   d student[b, v] = (2 softmax(student/temp_s) - (T_0 + T_1)) * grad_out / (temp_s bs nv)   (sum_k T_g = 1)
// The block first builds Tsum = T_0 + T_1 (in registers), then walks the nv student rows.
__device__ __forceinline__ float block_reduce_f(float v, bool is_max, float* red) {
  v = is_max ? warp_max(v) : warp_sum(v);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  float t = lane < (blockDim.x >> 5) ? red[lane] : (is_max ? -INFINITY : 0.f);
  return is_max ? warp_max(t) : warp_sum(t);
}

// Every row (K floats) is loaded ONCE into registers (EPT values per thread, coalesced: column = tid + e * 256) and the
// max / sum / dot / gradient passes run on the registers; one block reduction per statistic.
template <bool BWD, int EPT>
__global__ void __launch_bounds__(256)
dino_kernel(const float* __restrict__ teacher, int64_t ld_tb, int64_t ld_tv, const float* __restrict__ student,
            int64_t ld_sb, int64_t ld_sv, int nv, int k, const float* __restrict__ center, float inv_ts, float inv_tt,
            float* __restrict__ loss_part /* [bs] */, const float* __restrict__ grad_out, float coef,
            float* __restrict__ dstudent, int64_t ld_db, int64_t ld_dv) {
  __shared__ float red[32];
  const int64_t b = blockIdx.x;
  float tsum[EPT];
#pragma unroll
  for (int e = 0; e < EPT; ++e) tsum[e] = 0.f;
  for (int g = 0; g < 2; ++g) {
    const float* t = teacher + b * ld_tb + g * ld_tv;
    float x[EPT];
    float m = -INFINITY;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int c = threadIdx.x + e * 256;
      x[e] = c < k ? (t[c] - __ldg(center + c)) * inv_tt : -INFINITY;
      m = fmaxf(m, x[e]);
    }
    m = block_reduce_f(m, true, red);
    float z = 0.f;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      x[e] = __expf(x[e] - m);  // exp(-inf) = 0 for the padding
      z += x[e];
    }
    z = block_reduce_f(z, false, red);
    const float iz = 1.f / z;
#pragma unroll
    for (int e = 0; e < EPT; ++e) tsum[e] = fmaf(x[e], iz, tsum[e]);
  }
  float acc = 0.f;
  const float go = BWD ? __ldg(grad_out) * coef : 0.f;
  for (int v = 0; v < nv; ++v) {
    const float* s = student + b * ld_sb + v * ld_sv;
    float x[EPT];
    float m = -INFINITY;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int c = threadIdx.x + e * 256;
      x[e] = c < k ? s[c] * inv_ts : -INFINITY;
      m = fmaxf(m, x[e]);
    }
    m = block_reduce_f(m, true, red);
    float z = 0.f, dot = 0.f;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      if (!BWD && threadIdx.x + e * 256 < k) dot = fmaf(tsum[e], x[e], dot);
      x[e] = __expf(x[e] - m);
      z += x[e];
    }
    z = block_reduce_f(z, false, red);
    if (!BWD) {
      dot = block_reduce_f(dot, false, red);
      acc += dot - 2.f * (m + __logf(z));  // sum_k Tsum (x - lse) with sum_k Tsum = 2
    } else {
      const float iz = 2.f / z;
      float* d = dstudent + b * ld_db + v * ld_dv;
#pragma unroll
      for (int e = 0; e < EPT; ++e) {
        const int c = threadIdx.x + e * 256;
        if (c < k) d[c] = (x[e] * iz - tsum[e]) * go;
      }
    }
  }
  if (!BWD && threadIdx.x == 0) loss_part[b] = -acc;
}

// Large batches: one block per SAMPLE leaves bs blocks for 148 x 5 resident slots (1.4 waves at bs = 1024, the tail
// runs two latency-bound blocks per SM).  Split form: `dino_teacher_kernel` writes Tsum[b, :] = T_0 + T_1 once per sample,
// `dino_student_kernel` takes one (sample, view) ROW per block - bs x nv blocks, every row independent - and reads its
// Tsum row back (L2 / L1 resident: the nv rows of a sample are neighbouring blocks).
// V = 4: float4 accesses (K % 4 == 0, 16-byte aligned rows) - a warp-level LDG.128 moves 512 bytes per request slot
// where LDG.32 moves 128; the scalar form (V = 1) keeps arbitrary K / alignment working.  Thread t owns the V-wide
// column groups t + e * 256.
template <int V>
struct DinoVec;
template <>
struct DinoVec<1> {
  static __device__ __forceinline__ void load(const float* p, int c, float (&v)[1]) { v[0] = p[c]; }
  static __device__ __forceinline__ void store(float* p, int c, const float (&v)[1]) { p[c] = v[0]; }
};
template <>
struct DinoVec<4> {
  static __device__ __forceinline__ void load(const float* p, int c, float (&v)[4]) {
    const float4 t = *reinterpret_cast<const float4*>(p + c);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  static __device__ __forceinline__ void store(float* p, int c, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p + c) = make_float4(v[0], v[1], v[2], v[3]);
  }
};

template <int EPT, int V>
__global__ void __launch_bounds__(256)
dino_teacher_kernel(const float* __restrict__ teacher, int64_t ld_tb, int64_t ld_tv, int k,
                    const float* __restrict__ center, float inv_tt, float* __restrict__ tsum_out, int64_t ld_ts) {
  __shared__ float red[32];
  const int64_t b = blockIdx.x;
  float x[2][EPT][V];
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    const float* t = teacher + b * ld_tb + g * ld_tv;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int c = (threadIdx.x + e * 256) * V;
      if (c < k) {
        float cv[V];
        DinoVec<V>::load(t, c, x[g][e]);
        DinoVec<V>::load(center, c, cv);
#pragma unroll
        for (int i = 0; i < V; ++i) x[g][e][i] = (x[g][e][i] - cv[i]) * inv_tt;
      } else {
#pragma unroll
        for (int i = 0; i < V; ++i) x[g][e][i] = -INFINITY;
      }
    }
  }
  float tsum[EPT][V];
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    float m = -INFINITY;
#pragma unroll
    for (int e = 0; e < EPT; ++e)
#pragma unroll
      for (int i = 0; i < V; ++i) m = fmaxf(m, x[g][e][i]);
    m = block_reduce_f(m, true, red);
    float z = 0.f;
#pragma unroll
    for (int e = 0; e < EPT; ++e)
#pragma unroll
      for (int i = 0; i < V; ++i) {
        x[g][e][i] = __expf(x[g][e][i] - m);
        z += x[g][e][i];
      }
    z = block_reduce_f(z, false, red);
    const float iz = 1.f / z;
#pragma unroll
    for (int e = 0; e < EPT; ++e)
#pragma unroll
      for (int i = 0; i < V; ++i) tsum[e][i] = g == 0 ? x[g][e][i] * iz : fmaf(x[g][e][i], iz, tsum[e][i]);
  }
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    const int c = (threadIdx.x + e * 256) * V;
    if (c < k) DinoVec<V>::store(tsum_out + b * ld_ts, c, tsum[e]);
  }
}

template <bool BWD, int EPT, int V>
__global__ void __launch_bounds__(256, (EPT * V <= 16 ? 8 : 2))
dino_student_kernel(const float* __restrict__ student, int64_t ld_sb, int64_t ld_sv, int nv, int k,
                    const float* __restrict__ tsum_in, int64_t ld_ts, float inv_ts,
                    float* __restrict__ loss_part /* [bs * nv] */, const float* __restrict__ grad_out, float coef,
                    float* __restrict__ dstudent, int64_t ld_db, int64_t ld_dv) {
  __shared__ float red[32];
  const int64_t b = blockIdx.x / nv;
  const int v = static_cast<int>(blockIdx.x - b * nv);
  const float* s = student + b * ld_sb + v * ld_sv;
  const float* ts = tsum_in + b * ld_ts;
  // registers hold ONE row (x); the Tsum values are consumed at load time in the forward (dot) and re-read from L2 at
  // the end in the backward, so 8 blocks stay resident per SM (<= 32 registers / thread)
  float x[EPT][V];
  float m = -INFINITY, dot = 0.f;
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    const int c = (threadIdx.x + e * 256) * V;
    if (c < k) {
      DinoVec<V>::load(s, c, x[e]);
      float t[V];
      if (!BWD) DinoVec<V>::load(ts, c, t);
#pragma unroll
      for (int i = 0; i < V; ++i) {
        x[e][i] *= inv_ts;
        if (!BWD) dot = fmaf(t[i], x[e][i], dot);
        m = fmaxf(m, x[e][i]);
      }
    } else {
#pragma unroll
      for (int i = 0; i < V; ++i) x[e][i] = -INFINITY;
    }
  }
  m = block_reduce_f(m, true, red);
  float z = 0.f;
#pragma unroll
  for (int e = 0; e < EPT; ++e)
#pragma unroll
    for (int i = 0; i < V; ++i) {
      x[e][i] = __expf(x[e][i] - m);  // exp(-inf) = 0 for the padding
      z += x[e][i];
    }
  z = block_reduce_f(z, false, red);
  if (!BWD) {
    dot = block_reduce_f(dot, false, red);
    if (threadIdx.x == 0) loss_part[blockIdx.x] = -(dot - 2.f * (m + __logf(z)));
  } else {
    const float go = __ldg(grad_out) * coef;
    const float iz = 2.f / z;
    float* d = dstudent + b * ld_db + v * ld_dv;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int c = (threadIdx.x + e * 256) * V;
      if (c < k) {
        float g[V], t[V];
        DinoVec<V>::load(ts, c, t);
#pragma unroll
        for (int i = 0; i < V; ++i) g[i] = (x[e][i] * iz - t[i]) * go;
        DinoVec<V>::store(d, c, g);
      }
    }
  }
}

inline bool dino_split_path(int64_t bs, int64_t nv) { return bs * nv >= 4 * static_cast<int64_t>(num_sms()) && bs >= 128; }

template <bool BWD>
int dino_launch_split(const float* teacher, const float* student, const float* center, int64_t bs, int64_t nv, int64_t k,
                      float temp_s, float temp_t, float* tsum, float* part, const float* grad_out, float coef,
                      float* dstudent, cudaStream_t s) {
  const int ki = static_cast<int>(k), nvi = static_cast<int>(nv);
  const float its = 1.f / temp_s, itt = 1.f / temp_t;
  const unsigned g1 = static_cast<unsigned>(bs), g2 = static_cast<unsigned>(bs * nv);
#define SSVB_DINO2(E, V)                                                                                            \
  do {                                                                                                              \
    dino_teacher_kernel<E, V><<<g1, 256, 0, s>>>(teacher, 2 * k, k, ki, center, itt, tsum, k);                      \
    SSVB_LAUNCH_CHECK();                                                                                            \
    dino_student_kernel<BWD, E, V><<<g2, 256, 0, s>>>(student, nv * k, k, nvi, ki, tsum, k, its, part, grad_out,    \
                                                      coef, dstudent, nv * k, k);                                   \
  } while (0)
  const bool vec = (k % 4 == 0) && !((reinterpret_cast<uintptr_t>(teacher) | reinterpret_cast<uintptr_t>(student) |
                                      reinterpret_cast<uintptr_t>(center) | reinterpret_cast<uintptr_t>(tsum) |
                                      reinterpret_cast<uintptr_t>(dstudent)) & 15);
  if (vec) {
    if (k <= 1024) SSVB_DINO2(1, 4);
    else if (k <= 2048) SSVB_DINO2(2, 4);
    else if (k <= 4096) SSVB_DINO2(4, 4);
    else if (k <= 8192) SSVB_DINO2(8, 4);
    else return SSVB_ERR_UNSUPPORTED;
  } else {
    if (k <= 4 * 256) SSVB_DINO2(4, 1);
    else if (k <= 8 * 256) SSVB_DINO2(8, 1);
    else if (k <= 16 * 256) SSVB_DINO2(16, 1);
    else if (k <= 32 * 256) SSVB_DINO2(32, 1);
    else return SSVB_ERR_UNSUPPORTED;
  }
#undef SSVB_DINO2
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

// Wide heads (8192 < K <= 65536; DINO's published head is 65536 wide): a row no longer fits one CTA's registers, so it
// is split over a thread-block CLUSTER of C = ceil(K / 8192) CTAs.  CTA rank r keeps columns [8192 r, 8192 (r + 1)) in
// registers exactly as the split kernels above keep a whole row, and the row statistics meet in distributed shared
// memory:
//   * every thread folds its own values into (max m_t, sum exp(x - m_t)) - no block reduction - and a warp combines its
//     32 pairs with shuffles; lane 0 publishes one entry per warp in shared memory;
//   * one cluster barrier; then every warp of every CTA reads all 8 C entries through DSMEM and combines them with the
//     same fixed tree (entry L with entry L + 32 in lane L, then a butterfly), so all CTAs of the row hold bit-identical
//     statistics: deterministic, no second launch and no global round trip for the statistics;
//   * a second barrier (arrive once the DSMEM reads are done, wait just before exit) keeps each CTA's shared memory
//     alive until every peer has read it.
// Each row is still read once per kernel.  The combine is commutative bit for bit (explicit _rn operations, so no FMA
// contraction can order the two products differently), which is what makes every lane of a butterfly agree.
constexpr int kDinoSlice = 8192;    // columns per CTA: 256 threads x 32 floats
constexpr int kDinoMaxCluster = 8;  // the portable cluster size
constexpr int64_t kDinoMaxK = static_cast<int64_t>(kDinoSlice) * kDinoMaxCluster;

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_id_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_arrive_release() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_wait_acquire() {
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// 16-byte load from the shared memory of CTA `rank` of this cluster, at the offset `p` has in this CTA's
__device__ __forceinline__ float4 ld_dsmem_f4(const void* p, uint32_t rank) {
  uint32_t a;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(a) : "r"(smem_u32(p)), "r"(rank));
  float4 v;
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
  return v;
}

// (m, z) = (max, sum exp(x - m)) of a set of values; the empty set is (-inf, 0)
__device__ __forceinline__ float2 lse_merge(float2 a, float2 b) {
  const float m = fmaxf(a.x, b.x);
  if (m == -INFINITY) return make_float2(m, 0.f);
  return make_float2(m, __fadd_rn(__fmul_rn(a.y, __expf(a.x - m)), __fmul_rn(b.y, __expf(b.x - m))));
}
__device__ __forceinline__ float2 lse_warp_merge(float2 s) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
    s = lse_merge(s, make_float2(__shfl_xor_sync(0xffffffffu, s.x, o), __shfl_xor_sync(0xffffffffu, s.y, o)));
  return s;
}
// Lane L of a warp loads entries L and L + 32 of the cluster's 8 C published float4 (entry e = warp e % 8 of CTA e / 8);
// a missing entry reads as `none`.  The caller merges a with b and then across the warp: the fixed tree.
__device__ __forceinline__ void dino_cluster_load(const float4* pub, uint32_t csize, float4 none, float4& a, float4& b) {
  const int lane = threadIdx.x & 31, nent = static_cast<int>(csize) * 8;
  a = lane < nent ? ld_dsmem_f4(pub + (lane & 7), static_cast<uint32_t>(lane >> 3)) : none;
  b = lane + 32 < nent ? ld_dsmem_f4(pub + (lane & 7), static_cast<uint32_t>((lane + 32) >> 3)) : none;
}

// one cluster per sample: Tsum[b, slice] = T_0 + T_1
template <int EPT, int V>
__global__ void __launch_bounds__(256)
dino_teacher_cluster_kernel(const float* __restrict__ teacher, int64_t ld_tb, int64_t ld_tv, int k,
                            const float* __restrict__ center, float inv_tt, float* __restrict__ tsum_out, int64_t ld_ts) {
  static_assert(EPT * V * 256 == kDinoSlice, "one CTA owns one slice");
  __shared__ float4 pub[8];
  const uint32_t rank = cluster_ctarank(), csize = cluster_nctarank();
  const int64_t b = cluster_id_x();
  const int c0 = static_cast<int>(rank) * kDinoSlice;
  float x[2][EPT][V];
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    const float* t = teacher + b * ld_tb + g * ld_tv;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int c = c0 + (threadIdx.x + e * 256) * V;
      if (c < k) {
        float cv[V];
        DinoVec<V>::load(t, c, x[g][e]);
        DinoVec<V>::load(center, c, cv);
#pragma unroll
        for (int i = 0; i < V; ++i) x[g][e][i] = (x[g][e][i] - cv[i]) * inv_tt;
      } else {
#pragma unroll
        for (int i = 0; i < V; ++i) x[g][e][i] = -INFINITY;
      }
    }
  }
  float mt[2];  // this thread's own maxima: its exponentials are relative to them
  float2 w[2];
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    float m = -INFINITY;
#pragma unroll
    for (int e = 0; e < EPT; ++e)
#pragma unroll
      for (int i = 0; i < V; ++i) m = fmaxf(m, x[g][e][i]);
    const float ms = m == -INFINITY ? 0.f : m;  // a thread with padding only: exp(-inf) = 0, no NaN
    float z = 0.f;
#pragma unroll
    for (int e = 0; e < EPT; ++e)
#pragma unroll
      for (int i = 0; i < V; ++i) {
        x[g][e][i] = __expf(x[g][e][i] - ms);
        z += x[g][e][i];
      }
    mt[g] = m;
    w[g] = lse_warp_merge(make_float2(m, z));
  }
  if ((threadIdx.x & 31) == 0) pub[threadIdx.x >> 5] = make_float4(w[0].x, w[0].y, w[1].x, w[1].y);
  cluster_arrive_release();
  cluster_wait_acquire();
  float4 pa, pb;
  dino_cluster_load(pub, csize, make_float4(-INFINITY, 0.f, -INFINITY, 0.f), pa, pb);
  cluster_arrive_release();  // this thread's DSMEM reads are done
  const float2 r[2] = {lse_warp_merge(lse_merge(make_float2(pa.x, pa.y), make_float2(pb.x, pb.y))),
                       lse_warp_merge(lse_merge(make_float2(pa.z, pa.w), make_float2(pb.z, pb.w)))};
  float iz[2];
#pragma unroll
  for (int g = 0; g < 2; ++g) iz[g] = mt[g] == -INFINITY ? 0.f : __expf(mt[g] - r[g].x) / r[g].y;
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    const int c = c0 + (threadIdx.x + e * 256) * V;
    if (c < k) {
      float ts[V];
#pragma unroll
      for (int i = 0; i < V; ++i) ts[i] = fmaf(x[1][e][i], iz[1], x[0][e][i] * iz[0]);
      DinoVec<V>::store(tsum_out + b * ld_ts, c, ts);
    }
  }
  cluster_wait_acquire();  // no CTA leaves while a peer may still read its `pub`
}

// one cluster per (sample, view) row, sample-major: the nv rows of a sample are neighbours and share its Tsum row in L2.
// The forward fits 64 registers (4 CTAs / SM); the backward needs more than 64 without spilling (3 CTAs / SM at 72).
template <bool BWD, int EPT, int V>
__global__ void __launch_bounds__(256, BWD ? 2 : 4)
dino_student_cluster_kernel(const float* __restrict__ student, int64_t ld_sb, int64_t ld_sv, int nv, int k,
                            const float* __restrict__ tsum_in, int64_t ld_ts, float inv_ts,
                            float* __restrict__ loss_part /* [bs * nv] */, const float* __restrict__ grad_out,
                            float coef, float* __restrict__ dstudent, int64_t ld_db, int64_t ld_dv) {
  static_assert(EPT * V * 256 == kDinoSlice, "one CTA owns one slice");
  __shared__ float4 pub[8];
  const uint32_t rank = cluster_ctarank(), csize = cluster_nctarank();
  const int64_t row = cluster_id_x();
  const int64_t b = row / nv;
  const int v = static_cast<int>(row - b * nv);
  const int c0 = static_cast<int>(rank) * kDinoSlice;
  const float* s = student + b * ld_sb + v * ld_sv;
  const float* ts = tsum_in + b * ld_ts;
  float x[EPT][V];
  float m = -INFINITY, dot = 0.f;
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    const int c = c0 + (threadIdx.x + e * 256) * V;
    if (c < k) {
      DinoVec<V>::load(s, c, x[e]);
      float t[V];
      if (!BWD) DinoVec<V>::load(ts, c, t);
#pragma unroll
      for (int i = 0; i < V; ++i) {
        x[e][i] *= inv_ts;
        if (!BWD) dot = fmaf(t[i], x[e][i], dot);
        m = fmaxf(m, x[e][i]);
      }
    } else {
#pragma unroll
      for (int i = 0; i < V; ++i) x[e][i] = -INFINITY;
    }
  }
  const float ms = m == -INFINITY ? 0.f : m;
  float z = 0.f;
#pragma unroll
  for (int e = 0; e < EPT; ++e)
#pragma unroll
    for (int i = 0; i < V; ++i) {
      x[e][i] = __expf(x[e][i] - ms);
      z += x[e][i];
    }
  const float2 w = lse_warp_merge(make_float2(m, z));
  if (!BWD) dot = warp_sum(dot);
  if ((threadIdx.x & 31) == 0) pub[threadIdx.x >> 5] = make_float4(w.x, w.y, dot, 0.f);
  cluster_arrive_release();
  cluster_wait_acquire();
  float4 pa, pb;
  dino_cluster_load(pub, csize, make_float4(-INFINITY, 0.f, 0.f, 0.f), pa, pb);
  cluster_arrive_release();  // this thread's DSMEM reads are done
  const float2 r = lse_warp_merge(lse_merge(make_float2(pa.x, pa.y), make_float2(pb.x, pb.y)));
  if (!BWD) {
    const float dsum = warp_sum(pa.z + pb.z);
    if (rank == 0 && threadIdx.x == 0) loss_part[row] = -(dsum - 2.f * (r.x + __logf(r.y)));
  } else {
    const float go = __ldg(grad_out) * coef;
    const float iz = m == -INFINITY ? 0.f : 2.f * __expf(m - r.x) / r.y;
    float* d = dstudent + b * ld_db + v * ld_dv;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int c = c0 + (threadIdx.x + e * 256) * V;
      if (c < k) {
        float g[V], t[V];
        DinoVec<V>::load(ts, c, t);
#pragma unroll
        for (int i = 0; i < V; ++i) g[i] = (x[e][i] * iz - t[i]) * go;
        DinoVec<V>::store(d, c, g);
      }
    }
  }
  cluster_wait_acquire();  // no CTA leaves while a peer may still read its `pub`
}

template <typename... KArgs, typename... Args>
int launch_cluster(void (*kern)(KArgs...), int64_t clusters, unsigned csize, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(clusters * csize));
  cfg.blockDim = dim3(256);
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = csize;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  SSVB_CUDA(cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...));
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

template <bool BWD>
int dino_launch_cluster(const float* teacher, const float* student, const float* center, int64_t bs, int64_t nv,
                        int64_t k, float temp_s, float temp_t, float* tsum, float* part, const float* grad_out, float coef,
                        float* dstudent, cudaStream_t s) {
  const unsigned csize = static_cast<unsigned>(ceil_div(k, kDinoSlice));
  if (k > kDinoMaxK || bs * nv * csize > 0x7fffffffLL) return SSVB_ERR_UNSUPPORTED;
  const int ki = static_cast<int>(k), nvi = static_cast<int>(nv);
  const float its = 1.f / temp_s, itt = 1.f / temp_t;
#define SSVB_DINO_CL(E, V)                                                                                          \
  do {                                                                                                              \
    SSVB_TRY(launch_cluster(dino_teacher_cluster_kernel<E, V>, bs, csize, s, teacher, 2 * k, k, ki, center, itt,   \
                            tsum, k));                                                                              \
    SSVB_TRY(launch_cluster(dino_student_cluster_kernel<BWD, E, V>, bs * nv, csize, s, student, nv * k, k, nvi, ki, \
                            tsum, k, its, part, grad_out, coef, dstudent, nv * k, k));                              \
  } while (0)
  const bool vec = (k % 4 == 0) && !((reinterpret_cast<uintptr_t>(teacher) | reinterpret_cast<uintptr_t>(student) |
                                      reinterpret_cast<uintptr_t>(center) | reinterpret_cast<uintptr_t>(tsum) |
                                      reinterpret_cast<uintptr_t>(dstudent)) & 15);
  if (vec) SSVB_DINO_CL(8, 4);
  else SSVB_DINO_CL(32, 1);
#undef SSVB_DINO_CL
  return SSVB_OK;
}

template <bool BWD>
int dino_launch(const float* teacher, const float* student, const float* center, int64_t bs, int64_t nv, int64_t k,
                float temp_s, float temp_t, float* part, const float* grad_out, float coef, float* dstudent,
                cudaStream_t s) {
  const unsigned grid = static_cast<unsigned>(bs);
  const int ki = static_cast<int>(k), nvi = static_cast<int>(nv);
  const float its = 1.f / temp_s, itt = 1.f / temp_t;
#define SSVB_DINO(E)                                                                                                   \
  dino_kernel<BWD, E><<<grid, 256, 0, s>>>(teacher, 2 * k, k, student, nv * k, k, nvi, ki, center, its, itt, part, grad_out, \
                                           coef, dstudent, nv * k, k)
  if (k <= 4 * 256) SSVB_DINO(4);
  else if (k <= 8 * 256) SSVB_DINO(8);
  else if (k <= 16 * 256) SSVB_DINO(16);
  else if (k <= 32 * 256) SSVB_DINO(32);
  else return SSVB_ERR_UNSUPPORTED;
#undef SSVB_DINO
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

// centre EMA (models/dino.py:136-141): center = m * center + (1 - m) * mean_rows(teacher_fvecs); first call: plain mean.
// block (32 columns x 8 row phases), fixed-order combine -> deterministic.
__global__ void dino_center_kernel(const float* __restrict__ t, int64_t rows, int k, int64_t ld, float m, float om,
                                   int first, float* __restrict__ center) {
  __shared__ float sh[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  float s = 0.f;
  if (c < k)
    for (int64_t r = threadIdx.y; r < rows; r += 8) s += t[r * ld + c];
  sh[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && c < k) {
    float a = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) a += sh[i][threadIdx.x];
    const float mean = a / static_cast<float>(rows);
    center[c] = first ? mean : __fadd_rn(__fmul_rn(m, center[c]), __fmul_rn(om, mean));
  }
}

}  // namespace

extern "C" {

int64_t ssvb_ema_chunk_elems(void) { return kEmaChunk; }

int ssvb_ema_update(const void* chunk_table, int64_t n_chunks, float m, float one_minus_m, void* stream) {
  SSVB_TRY(check_device_sm100());
  if (n_chunks < 0 || (n_chunks > 0 && !chunk_table)) return SSVB_ERR_INVALID;
  if (n_chunks == 0) return SSVB_OK;
  if (n_chunks > 0x7fffffffLL) return SSVB_ERR_UNSUPPORTED;
  if (reinterpret_cast<uintptr_t>(chunk_table) & 7) return SSVB_ERR_ALIGNMENT;
  ema_kernel<<<static_cast<unsigned>(n_chunks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const EmaChunk*>(chunk_table), m, one_minus_m);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

// [bs * nv] loss partials + (split and cluster paths) Tsum [bs x k]
size_t ssvb_dino_workspace_bytes(int64_t bs, int64_t nv, int64_t k) {
  if (bs <= 0 || nv <= 0 || k <= 0) return 0;
  return (static_cast<size_t>(bs * nv) * sizeof(float) + 255) / 256 * 256 + static_cast<size_t>(bs * k) * sizeof(float) + 256;
}

int ssvb_dino_fwd(const float* teacher, const float* student, const float* center, int64_t bs, int64_t nv, int64_t k,
                  float temp_s, float temp_t, float* loss, void* workspace, size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  if (!teacher || !student || !center || !loss || !workspace || bs <= 0 || nv <= 0 || k <= 0 || !(temp_s > 0.f) ||
      !(temp_t > 0.f))
    return SSVB_ERR_INVALID;
  if (k > kDinoMaxK || bs > 0x7fffffffLL) return SSVB_ERR_UNSUPPORTED;
  if (workspace_bytes < ssvb_dino_workspace_bytes(bs, nv, k)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float* part = static_cast<float*>(workspace);
  float* tsum = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + (static_cast<size_t>(bs * nv) * sizeof(float) + 255) / 256 * 256);
  if (k > kDinoSlice) {
    SSVB_TRY(dino_launch_cluster<false>(teacher, student, center, bs, nv, k, temp_s, temp_t, tsum, part, nullptr, 0.f,
                                        nullptr, s));
    sum_partials_kernel<<<1, 1024, 0, s>>>(part, static_cast<int>(bs * nv), 1.f / static_cast<float>(bs * nv), loss);
    SSVB_LAUNCH_CHECK();
    return SSVB_OK;
  }
  if (dino_split_path(bs, nv)) {
    SSVB_TRY(dino_launch_split<false>(teacher, student, center, bs, nv, k, temp_s, temp_t, tsum, part, nullptr, 0.f,
                                      nullptr, s));
    sum_partials_kernel<<<1, 1024, 0, s>>>(part, static_cast<int>(bs * nv), 1.f / static_cast<float>(bs * nv), loss);
    SSVB_LAUNCH_CHECK();
    return SSVB_OK;
  }
  SSVB_TRY(dino_launch<false>(teacher, student, center, bs, nv, k, temp_s, temp_t, part, nullptr, 0.f, nullptr, s));
  sum_partials_kernel<<<1, 1024, 0, s>>>(part, static_cast<int>(bs), 1.f / static_cast<float>(bs * nv), loss);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

int ssvb_dino_bwd(const float* teacher, const float* student, const float* center, int64_t bs, int64_t nv, int64_t k,
                  float temp_s, float temp_t, const float* grad_out, float* dstudent, void* workspace,
                  size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  if (!teacher || !student || !center || !grad_out || !dstudent || bs <= 0 || nv <= 0 || k <= 0 || !(temp_s > 0.f) ||
      !(temp_t > 0.f))
    return SSVB_ERR_INVALID;
  if (k > kDinoMaxK || bs > 0x7fffffffLL) return SSVB_ERR_UNSUPPORTED;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (k > kDinoSlice) {
    if (!workspace || workspace_bytes < ssvb_dino_workspace_bytes(bs, nv, k)) return SSVB_ERR_WORKSPACE;
    float* tsum = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + (static_cast<size_t>(bs * nv) * sizeof(float) + 255) / 256 * 256);
    return dino_launch_cluster<true>(teacher, student, center, bs, nv, k, temp_s, temp_t, tsum, nullptr, grad_out,
                                     1.f / (temp_s * static_cast<float>(bs * nv)), dstudent, s);
  }
  if (dino_split_path(bs, nv)) {
    if (!workspace || workspace_bytes < ssvb_dino_workspace_bytes(bs, nv, k)) return SSVB_ERR_WORKSPACE;
    float* tsum = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + (static_cast<size_t>(bs * nv) * sizeof(float) + 255) / 256 * 256);
    return dino_launch_split<true>(teacher, student, center, bs, nv, k, temp_s, temp_t, tsum, nullptr, grad_out,
                                   1.f / (temp_s * static_cast<float>(bs * nv)), dstudent, s);
  }
  return dino_launch<true>(teacher, student, center, bs, nv, k, temp_s, temp_t, nullptr, grad_out,
                           1.f / (temp_s * static_cast<float>(bs * nv)), dstudent, s);
}

int ssvb_dino_center_update(const float* teacher_rows, int64_t rows, int64_t k, int64_t ld, float momentum,
                            float one_minus_m, int first, float* center, void* stream) {
  SSVB_TRY(check_device_sm100());
  if (!teacher_rows || !center || rows <= 0 || k <= 0 || ld < k) return SSVB_ERR_INVALID;
  dino_center_kernel<<<static_cast<unsigned>(ceil_div(k, 32)), dim3(32, 8), 0, static_cast<cudaStream_t>(stream)>>>(
      teacher_rows, rows, static_cast<int>(k), ld, momentum, one_minus_m, first, center);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

}  // extern "C"
