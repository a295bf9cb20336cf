// Host-side planning / launch of the similarity kernels + the small bandwidth kernels around them
// (row normalise -> bf16 staging, partial-LSE finalize, deterministic scalar reduction).
#pragma once
#include "host_util.h"
#include "sim_kernels.cuh"

namespace ssvb {

// staged row width: 64 or 128 columns for d <= 128, 256 for 128 < d <= 256 (KB = dpad / 64 = 1, 2 or 4 k-blocks)
inline int64_t sim_dpad(int64_t d) { return d <= 128 ? round_up(d, 64) : 256; }
inline int64_t sim_mpad(int64_t m) { return round_up(m, 256); }
// forward tile width for a staged row width (FwdCfg<KB>::BN) and the smallest number of tiles a column chunk may have
// (1024 columns)
inline int sim_fwd_bn(int64_t dpad) { return dpad > 128 ? 128 : kFwdBN; }
inline int sim_fwd_min_tiles(int64_t dpad) { return 1024 / sim_fwd_bn(dpad); }

// Choose the column chunking: (row block, chunk) units are statically strided over one CTA per SM, so the number
// of units should fill whole waves of `num_sms()` CTAs (tail effect) while every chunk keeps >= min_tiles tiles
// (amortises the A-tile load, the partial write / the accumulator drain).  No chunk is ever empty.
inline void plan_chunks_tiles(SimParams& p, int col_tiles, int min_tiles) {
  p.col_tiles = col_tiles;
  const int sms = num_sms();
  const int max_ch = p.col_tiles / min_tiles > 1 ? p.col_tiles / min_tiles : 1;
  int best = 1;
  double best_score = -1.0;
  for (int nch = 1; nch <= max_ch && nch <= 256; ++nch) {
    const int tpc = static_cast<int>(ceil_div(p.col_tiles, nch));
    const int real = static_cast<int>(ceil_div(p.col_tiles, tpc));
    if (real != nch) continue;  // would leave an empty chunk
    const int64_t units = static_cast<int64_t>(p.row_blocks) * nch;
    const int64_t waves = ceil_div(units, sms);
    // wave efficiency in tiles (the last chunk of a row block may be shorter), minus a small per-chunk overhead
    const double eff = static_cast<double>(p.row_blocks) * p.col_tiles / (static_cast<double>(waves) * sms * tpc);
    const double score = eff - 0.002 * nch;
    if (score > best_score) {
      best_score = score;
      best = nch;
    }
  }
  p.tiles_per_chunk = static_cast<int>(ceil_div(p.col_tiles, best));
  p.nchunks = static_cast<int>(ceil_div(p.col_tiles, p.tiles_per_chunk));
}
inline void plan_chunks(SimParams& p, int BN, int min_tiles) {
  plan_chunks_tiles(p, static_cast<int>(ceil_div(p.cols, BN)), min_tiles);
}
// symmetric forward (sim_fwd_sym_kernel): p.row_blocks = R row blocks of a square S; each takes a band of
// floor(R/2) + 1 128-column tiles, two per 256-column stage.  Returns the number of column partials per row
// ((R - 1) / 2, stored after the 4 * nchunks row partials).
inline int plan_sym(SimParams& p) {
  p.band = p.row_blocks / 2 + 1;
  plan_chunks_tiles(p, (p.band + 1) / 2, sim_fwd_min_tiles(128));
  return (p.row_blocks - 1) / 2;
}

template <int KB>
int launch_sim_fwd_sym_t(const CUtensorMap& tmA, const CUtensorMap& tmB, const SimParams& p, cudaStream_t s) {
  auto kern = sim_fwd_sym_kernel<KB, true>;
  constexpr int smem = SymCfg<KB>::SMEM;
  SSVB_TRY((set_smem_once<sim_fwd_sym_kernel<KB, true>>(smem)));
  const int nunits = p.row_blocks * p.nchunks;
  const int grid = nunits < num_sms() ? nunits : num_sms();
  const int slot = prof_begin(PROF_SIM_FWD, s);
  kern<<<grid, 640, smem, s>>>(tmA, tmB, p);
  prof_end(slot, s);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}
// Z: fp16 [z_rows x dpad] (unit-norm rows, pre-scaled; FIXED mode only), dpad <= 128
inline int launch_sim_fwd_sym(const void* Z, int64_t z_rows, int64_t dpad, const SimParams& p, cudaStream_t s) {
  if (!p.opf16 || dpad > 128) return SSVB_ERR_UNSUPPORTED;
  CUtensorMap tm;  // A and B are the same matrix, both in 128-row boxes
  SSVB_TRY(make_tmap_bf16(&tm, Z, z_rows, dpad, dpad, 128, true));
  return dpad == 64 ? launch_sim_fwd_sym_t<1>(tm, tm, p, s) : launch_sim_fwd_sym_t<2>(tm, tm, p, s);
}

template <int KB, int MODE, bool OPF16 = false>
int launch_sim_fwd_t(const CUtensorMap& tmA, const CUtensorMap& tmB, const SimParams& p, cudaStream_t s) {
  auto kern = sim_fwd_kernel<KB, MODE, OPF16>;
  constexpr int smem = FwdCfg<KB>::SMEM;
  SSVB_TRY((set_smem_once<sim_fwd_kernel<KB, MODE, OPF16>>(smem)));
  const int nunits = p.row_blocks * p.nchunks;
  const int grid = nunits < num_sms() ? nunits : num_sms();
  const int slot = prof_begin(PROF_SIM_FWD, s);
  kern<<<grid, 640, smem, s>>>(tmA, tmB, p);
  prof_end(slot, s);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}
template <int KB, int MODE, bool OPF16 = false>
int launch_sim_bwd_t(const CUtensorMap& tmA, const CUtensorMap& tmB, const SimParams& p, cudaStream_t s) {
  auto kern = sim_bwd_kernel<KB, MODE, OPF16>;
  constexpr int smem = BwdCfg<KB>::SMEM;
  SSVB_TRY((set_smem_once<sim_bwd_kernel<KB, MODE, OPF16>>(smem)));
  const int nunits = p.row_blocks * p.nchunks;
  const int grid = nunits < num_sms() ? nunits : num_sms();
  const int slot = prof_begin(PROF_SIM_BWD, s);
  kern<<<grid, 640, smem, s>>>(tmA, tmB, p);
  prof_end(slot, s);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

// A: bf16 [a_rows x dpad], B: bf16 [b_rows x dpad]
inline int launch_sim_fwd(int mode, const void* A, int64_t a_rows, const void* B, int64_t b_rows, int64_t dpad,
                          const SimParams& p, cudaStream_t s) {
  CUtensorMap tmA, tmB;
  SSVB_TRY(make_tmap_bf16(&tmA, A, a_rows, dpad, dpad, 128, p.opf16 != 0));
  SSVB_TRY(make_tmap_bf16(&tmB, B, b_rows, dpad, dpad, sim_fwd_bn(dpad), p.opf16 != 0));
  const int KB = static_cast<int>(dpad / 64);
#define SSVB_DISPATCH(KBV)                                                      \
  switch (mode) {                                                               \
    case SIM_NTX_FIXED:                                                         \
      if (p.opf16) return launch_sim_fwd_t<KBV, SIM_NTX_FIXED, true>(tmA, tmB, p, s);                   \
      return launch_sim_fwd_t<KBV, SIM_NTX_FIXED, false>(tmA, tmB, p, s);                               \
    case SIM_NTX_ONLINE:                                                        \
      if (p.opf16) return launch_sim_fwd_t<KBV, SIM_NTX_ONLINE, true>(tmA, tmB, p, s);                  \
      return launch_sim_fwd_t<KBV, SIM_NTX_ONLINE, false>(tmA, tmB, p, s);                              \
    case SIM_MOCO: return launch_sim_fwd_t<KBV, SIM_MOCO>(tmA, tmB, p, s);      \
    default: return SSVB_ERR_INVALID;                                           \
  }
  if (KB == 1) { SSVB_DISPATCH(1) }
  if (KB == 2) { SSVB_DISPATCH(2) }
  if (KB == 4) { SSVB_DISPATCH(4) }
#undef SSVB_DISPATCH
  return SSVB_ERR_UNSUPPORTED;
}
inline int launch_sim_bwd_half(int mode, const void* A, int64_t a_rows, const void* B, int64_t b_rows, int64_t dpad,
                               const SimParams& p, cudaStream_t s);
// dpad = 256: one launch per 128-column half of dZ (see BwdCfg::DP)
inline int launch_sim_bwd(int mode, const void* A, int64_t a_rows, const void* B, int64_t b_rows, int64_t dpad,
                          const SimParams& p, cudaStream_t s) {
  if (dpad <= 128) return launch_sim_bwd_half(mode, A, a_rows, B, b_rows, dpad, p, s);
  SimParams q = p;
  for (int h = 0; h < 2; ++h) {
    q.dhalf = h;
    SSVB_TRY(launch_sim_bwd_half(mode, A, a_rows, B, b_rows, dpad, q, s));
  }
  return SSVB_OK;
}
inline int launch_sim_bwd_half(int mode, const void* A, int64_t a_rows, const void* B, int64_t b_rows, int64_t dpad,
                          const SimParams& p, cudaStream_t s) {
  CUtensorMap tmA, tmB;
  SSVB_TRY(make_tmap_bf16(&tmA, A, a_rows, dpad, dpad, 128, p.opf16 != 0));
  SSVB_TRY(make_tmap_bf16(&tmB, B, b_rows, dpad, dpad, 128, p.opf16 != 0));
  const int KB = static_cast<int>(dpad / 64);
#define SSVB_DISPATCH(KBV)                                                      \
  switch (mode) {                                                               \
    case SIM_NTX_FIXED:                                                         \
      if (p.opf16) return launch_sim_bwd_t<KBV, SIM_NTX_FIXED, true>(tmA, tmB, p, s);  \
      return launch_sim_bwd_t<KBV, SIM_NTX_FIXED, false>(tmA, tmB, p, s);              \
    case SIM_NTX_ONLINE:                                                        \
      if (p.opf16) return launch_sim_bwd_t<KBV, SIM_NTX_ONLINE, true>(tmA, tmB, p, s); \
      return launch_sim_bwd_t<KBV, SIM_NTX_ONLINE, false>(tmA, tmB, p, s);             \
    case SIM_MOCO: return launch_sim_bwd_t<KBV, SIM_MOCO>(tmA, tmB, p, s);      \
    default: return SSVB_ERR_INVALID;                                           \
  }
  if (KB == 1) { SSVB_DISPATCH(1) }
  if (KB == 2) { SSVB_DISPATCH(2) }
  if (KB == 4) { SSVB_DISPATCH(4) }
#undef SSVB_DISPATCH
  return SSVB_ERR_UNSUPPORTED;
}

// ---------------------------------------------------------------------------------------------------
// pair_prep: one warp per row n of two [n x d] fp32 matrices.  Optionally L2-normalises
// (x / max(||x||, 1e-12), F.normalize semantics), writes bf16 rows (zero padded to dpad) and the
// row dot product of the two bf16-rounded rows (`pos`, exactly what the tensor cores will see).
// ---------------------------------------------------------------------------------------------------
static __global__ void pair_prep_kernel(const float* __restrict__ xi, const float* __restrict__ xj, int n, int d,
                                 int64_t ldi, int64_t ldj, int normalize, int f16, __nv_bfloat16* __restrict__ out_i,
                                 __nv_bfloat16* __restrict__ out_j, int dpad, float* __restrict__ inv_i,
                                 float* __restrict__ inv_j, float* __restrict__ pos_i, float* __restrict__ pos_j,
                                 int norm_mask = -1 /* >= 0: bit 0 normalises xi, bit 1 xj (overrides `normalize`) */,
                                 float prescale = 1.f /* staged rows = x_hat * prescale (NT-Xent FIXED mode:
                                 sqrt(log2(e)/tau), so the tensor-core accumulator is the log2-domain logit) */,
                                 unsigned int* zero_counter = nullptr /* 4 counters of the later last-block reductions:
                                 zeroed HERE (first kernel of the call) instead of by a memset node, which costs a
                                 2-4 us dependency gap in front of the first kernel of a CUDA graph */,
                                 float* zero_rows = nullptr, int zero_ld = 0, int zero_nrows = 0 /* fp32 accumulator
                                 rows [zero_nrows x zero_ld] that a later kernel adds into (red.global.add): warp w
                                 zeroes row w; the grid must cover max(n, zero_nrows) warps */) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (zero_counter && blockIdx.x == 0 && threadIdx.x < 4) zero_counter[threadIdx.x] = 0u;
  if (zero_rows && warp < zero_nrows)
    for (int k = lane * 4; k < zero_ld; k += 128)
      *reinterpret_cast<float4*>(zero_rows + static_cast<int64_t>(warp) * zero_ld + k) = make_float4(0.f, 0.f, 0.f, 0.f);
  if (warp >= n) return;
  const float* ri = xi + static_cast<int64_t>(warp) * ldi;
  const float* rj = xj + static_cast<int64_t>(warp) * ldj;
  const int nmask = norm_mask >= 0 ? norm_mask : (normalize ? 3 : 0);
  // dpad <= 256: up to two float4 per lane
  float4 a[2], b[2];
  float si = 0.f, sj = 0.f;
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int k = it * 128 + lane * 4;
    a[it] = make_float4(0.f, 0.f, 0.f, 0.f);
    b[it] = a[it];
    if (k < d) {
      a[it] = *reinterpret_cast<const float4*>(ri + k);
      b[it] = *reinterpret_cast<const float4*>(rj + k);
    }
    si += a[it].x * a[it].x + a[it].y * a[it].y + a[it].z * a[it].z + a[it].w * a[it].w;
    sj += b[it].x * b[it].x + b[it].y * b[it].y + b[it].z * b[it].z + b[it].w * b[it].w;
  }
  si = warp_sum(si);
  sj = warp_sum(sj);
  float ivi = 1.f, ivj = 1.f;
  if (nmask & 1) ivi = 1.f / fmaxf(sqrtf(si), 1e-12f);
  if (nmask & 2) ivj = 1.f / fmaxf(sqrtf(sj), 1e-12f);
  float dot = 0.f;
  const float si_ = ivi * prescale, sj_ = ivj * prescale;  // inv_norm outputs stay the plain 1/||x||
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int k = it * 128 + lane * 4;
    if (k < dpad) {
      uint2 vi, vj;
      vi.x = f16 ? pack_f16x2(a[it].x * si_, a[it].y * si_) : pack_bf16x2(a[it].x * si_, a[it].y * si_);
      vi.y = f16 ? pack_f16x2(a[it].z * si_, a[it].w * si_) : pack_bf16x2(a[it].z * si_, a[it].w * si_);
      vj.x = f16 ? pack_f16x2(b[it].x * sj_, b[it].y * sj_) : pack_bf16x2(b[it].x * sj_, b[it].y * sj_);
      vj.y = f16 ? pack_f16x2(b[it].z * sj_, b[it].w * sj_) : pack_bf16x2(b[it].z * sj_, b[it].w * sj_);
      const float2 fi01 = unpack_h2(vi.x, f16), fi23 = unpack_h2(vi.y, f16);
      const float2 fj01 = unpack_h2(vj.x, f16), fj23 = unpack_h2(vj.y, f16);
      dot += fi01.x * fj01.x + fi01.y * fj01.y + fi23.x * fj23.x + fi23.y * fj23.y;
      if (out_i) *reinterpret_cast<uint2*>(out_i + static_cast<int64_t>(warp) * dpad + k) = vi;
      if (out_j) *reinterpret_cast<uint2*>(out_j + static_cast<int64_t>(warp) * dpad + k) = vj;
    }
  }
  dot = warp_sum(dot);
  if (lane == 0) {
    if (inv_i) inv_i[warp] = ivi;
    if (inv_j) inv_j[warp] = ivj;
    if (pos_i) pos_i[warp] = dot;
    if (pos_j) pos_j[warp] = dot;
  }
}

// ---------------------------------------------------------------------------------------------------
// deterministic block-sum -> scalar: every block writes its partial, the last block to finish adds
// them in index order (no float atomics -> run-to-run bit-stable loss).
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ float block_sum_256(float v) {
  __shared__ float red[8];
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  float t = 0.f;
  if (w == 0) {
    t = lane < (blockDim.x >> 5) ? red[lane] : 0.f;
    t = warp_sum(t);
  }
  return t;  // valid in warp 0
}
__device__ __forceinline__ bool grid_sum_finish(float block_total, float* block_sums, unsigned int* counter,
                                                float scale, float* out, bool accumulate) {
  __shared__ bool is_last;
  if (counter == nullptr) {  // two-kernel form: the caller launches a one-block sum over block_sums afterwards
    if (threadIdx.x == 0) block_sums[blockIdx.x] = block_total;
    return false;
  }
  if (threadIdx.x == 0) {
    block_sums[blockIdx.x] = block_total;
    __threadfence();
    const unsigned int done = atomicAdd(counter, 1u);
    is_last = (done == gridDim.x - 1);
  }
  __syncthreads();
  if (is_last && threadIdx.x < 32) {
    __threadfence();
    float t = 0.f;
    for (unsigned int i = threadIdx.x; i < gridDim.x; i += 32) t += __ldcg(block_sums + i);
    t = warp_sum(t);
    if (threadIdx.x == 0) {
      if (accumulate)
        *out += t * scale;
      else
        *out = t * scale;
      *counter = 0;
    }
  }
  return is_last;  // block-uniform: true in the block that arrived last (all other blocks' writes are visible to it)
}

// ---- NVLink peer-memory transport helpers (symmetric arenas, generation flags; see ntxent.cu) ----
__device__ __forceinline__ void st_release_sys_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_volatile_u2(uint2* p, uint2 v) {
  asm volatile("st.volatile.global.v2.u32 [%0], {%1, %2};" ::"l"(p), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ uint2 ld_volatile_u2(const uint2* p) {
  uint2 v;
  asm volatile("ld.volatile.global.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
  return v;
}
// LL consumer: spin until the 8-byte {value, tag} pair carries generation `gen`; bounded like spin_wait_gen
__device__ __forceinline__ float ll_wait_value(const uint2* p, uint32_t gen) {
  uint2 v = ld_volatile_u2(p);
  if (v.y != gen) {
    const long long t0 = clock64();
    do {
      __nanosleep(32);
      v = ld_volatile_u2(p);
      if (clock64() - t0 > 60000000000LL) __trap();
    } while (v.y != gen);
  }
  return __uint_as_float(v.x);
}
// wait until a peer has published generation `gen` (monotonic counters, wrap-safe compare).  Bounded: a rank that
// never arrives turns into a CUDA error after ~30 s instead of a hung GPU.
__device__ __forceinline__ void spin_wait_gen(const uint32_t* flag, uint32_t gen) {
  const long long t0 = clock64();
  while (static_cast<int32_t>(ld_acquire_sys_u32(flag) - gen) < 0) {
    __nanosleep(64);
    if (clock64() - t0 > 60000000000LL) __trap();
  }
}
// 8-byte store to the same offset of EVERY rank's arena through the NVSwitch multicast mapping (one store on the
// wire instead of `world`)
__device__ __forceinline__ void multimem_st_v2(void* mc_addr, uint2 v) {
  asm volatile("multimem.st.relaxed.sys.global.v2.f32 [%0], {%1, %2};" ::"l"(mc_addr), "f"(__uint_as_float(v.x)),
               "f"(__uint_as_float(v.y))
               : "memory");
}

// ---------------------------------------------------------------------------------------------------
// lse_finalize: combine the per-chunk partials of every local row into its log2-domain LSE, emit the
// per-row statistic the backward needs (FIXED: 1/L', else lse2) and the loss sum.
//   MoCo: the positive logit joins the LSE (label-0 column of the reference's cat, utils/losses.py:70).
// ---------------------------------------------------------------------------------------------------
template <int MODE>
__global__ void lse_finalize_kernel(const float* __restrict__ part_m, const float* __restrict__ part_l, int nparts,
                                    int stride, int nrows, const float* __restrict__ pos, float c, float shift,
                                    float* __restrict__ stat, float* __restrict__ lse2_out,
                                    float* block_sums, unsigned int* counter, float loss_scale, float* loss,
                                    float* __restrict__ term_out = nullptr, float* const* __restrict__ peer_stat = nullptr,
                                    int world = 0, size_t peer_off = 0 /* elements (floats, or 8-byte pairs if gen) */,
                                    float wscale = 1.f, uint32_t gen = 0) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  float term = 0.f;
  if (r < nrows) {
    float lse2, st;
    const float p2 = pos[r] * c;
    if (MODE == SIM_NTX_FIXED) {
      // 8 partials in flight per trip (the plain loop issued one dependent-latency load at a time: 9-11 us for 36-64
      // partials per row on the multi-GPU path); the summation ORDER is unchanged (index order), so the result is too
      float L = 0.f;
      int i = 0;
      for (; i + 8 <= nparts; i += 8) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = __ldcg(part_l + static_cast<size_t>(i + u) * stride + r);
#pragma unroll
        for (int u = 0; u < 8; ++u) L += v[u];
      }
      for (; i < nparts; ++i) L += __ldcg(part_l + static_cast<size_t>(i) * stride + r);
      lse2 = shift + log2f(L);
      st = wscale / L;  // backward weight W = e^s (st_a + st_b): wscale = 2^k keeps W in fp16's normal range
    } else {
      float M = (MODE == SIM_MOCO) ? p2 : -1e30f;
      for (int i = 0; i < nparts; ++i) M = fmaxf(M, part_m[static_cast<size_t>(i) * stride + r]);
      float L = (MODE == SIM_MOCO) ? exp2f(p2 - M) : 0.f;
      for (int i = 0; i < nparts; ++i)
        L += part_l[static_cast<size_t>(i) * stride + r] * exp2f(part_m[static_cast<size_t>(i) * stride + r] - M);
      lse2 = M + log2f(L);
      st = lse2;
    }
    stat[r] = st;
    if (lse2_out) lse2_out[r] = lse2;
    term = (lse2 - p2) * SSVB_LN2;
    if (term_out) term_out[r] = term;
    if (peer_stat) {
      // fused all-gather of this rank's [lse2 | term] block into every peer's buffer.  `gen` != 0: "LL" form - every
      // value travels as ONE 8-byte store {value, generation}; 8-byte stores are single transactions, so the consumer
      // validates each element by its tag and neither a system fence nor a completion flag is needed (a fence after
      // remote stores costs ~8 us on NVLink: profiles/r2_stage_timing.md).  gen == 0: plain floats (the caller
      // separates the stages with a barrier).
      for (int pr = 0; pr < world; ++pr) {
        if (gen) {
          uint2* dst = reinterpret_cast<uint2*>(peer_stat[pr]) + peer_off;
          st_volatile_u2(dst + r, make_uint2(__float_as_uint(lse2), gen));
          st_volatile_u2(dst + nrows + r, make_uint2(__float_as_uint(term), gen));
        } else {
          float* dst = peer_stat[pr] + peer_off;
          dst[r] = lse2;
          dst[nrows + r] = term;
        }
      }
    }
  }
  const float bt = block_sum_256(term);
  grid_sum_finish(bt, block_sums, counter, loss_scale, loss, false);
}

// Same combine for MANY partials per row (MoCo: the queue axis is split into up to 128 chunks x 4 warpgroups):
// one warp per row, lanes stride over the partials, shuffle max / sum; 8 rows per block.
template <int MODE>
__global__ void lse_finalize_wide_kernel(const float* __restrict__ part_m, const float* __restrict__ part_l,
                                         int nparts, int stride, int nrows, const float* __restrict__ pos, float c,
                                         float* __restrict__ stat, float* block_sums, unsigned int* counter,
                                         float loss_scale, float* loss) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  float term = 0.f;
  if (r < nrows) {
    const float p2 = pos[r] * c;
    float M = (MODE == SIM_MOCO) ? p2 : -1e30f;
    for (int i = lane; i < nparts; i += 32) M = fmaxf(M, part_m[static_cast<size_t>(i) * stride + r]);
    M = warp_max(M);
    float L = 0.f;
    for (int i = lane; i < nparts; i += 32)
      L += part_l[static_cast<size_t>(i) * stride + r] * exp2f(part_m[static_cast<size_t>(i) * stride + r] - M);
    L = warp_sum(L);
    if (MODE == SIM_MOCO) L += exp2f(p2 - M);
    const float lse2 = M + log2f(L);
    if (lane == 0) {
      stat[r] = lse2;
      term = (lse2 - p2) * SSVB_LN2;
    }
  }
  const float bt = block_sum_256(term);
  grid_sum_finish(bt, block_sums, counter, loss_scale, loss, false);
}

static __global__ void fill_kernel(float* p, int64_t n, float v) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

}  // namespace ssvb
