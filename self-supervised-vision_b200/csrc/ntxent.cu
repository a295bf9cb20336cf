// NT-Xent (SimCLR) loss, forward + backward, single GPU and row-sharded multi-GPU pieces.
// Replaces SimclrLoss.forward (reference utils/losses.py:15-46) and the contrastive term of
// RelicLoss.forward (utils/losses.py:163-194).
//
// Math (SURVEY.md §8 a1): Z = [zi; zj] (M = 2N rows), s_ab = zh_a.zh_b / tau, partner(a) = a +- N,
//   loss = 1/M sum_a [ LSE_{b != a} s_ab - s_{a,partner(a)} ]
//   d zh_a = [ sum_{b != a} (P_ab + P_ba) zh_b - 2 zh_partner(a) ] / (M tau),  P_ab = exp(s_ab - lse_a)
//   d z_a  = (d zh_a - (d zh_a . zh_a) zh_a) / max(||z_a||, 1e-12)              (normalize=True)
// All exponentials run in the log2 domain: t = s * log2(e)/tau.
#include "sim_host.cuh"

using namespace ssvb;

namespace {

struct NtxPlan {
  int64_t n_glob, m, mpad, d, dpad;
  int mode;
  int normalize;
  float c, shift;   // what the kernels apply to the accumulator: x = s * c - shift
  float prescale;   // what pair_prep multiplies the staged rows with
  float wscale;     // FIXED mode: backward weights carry this power of two (fp16 normal range), undone in grad_finish
  float pos_c;      // log2-domain positive logit = pos * pos_c
};

int make_plan(NtxPlan& pl, int64_t n_glob, int64_t d, int normalize, float temperature) {
  if (n_glob <= 0 || d <= 0 || !(temperature > 0.f)) return SSVB_ERR_INVALID;
  if (d % 4) return SSVB_ERR_ALIGNMENT;
  if (d > 256) return SSVB_ERR_UNSUPPORTED;  // 128 < d <= 256: KB = 4 kernels (sim_kernels.cuh FwdCfg / BwdCfg)
  if (2 * n_glob > (1 << 30)) return SSVB_ERR_UNSUPPORTED;
  pl.n_glob = n_glob;
  pl.m = 2 * n_glob;
  pl.mpad = sim_mpad(pl.m);
  pl.d = d;
  pl.dpad = sim_dpad(d);
  pl.normalize = normalize ? 1 : 0;
  const float c = SSVB_LOG2E / temperature;
  // unit-norm rows bound |s| <= 1/tau, i.e. the log2-domain logits lie in [-c, c]: for c <= 32 (tau >= ~0.045)
  // exp2 needs neither a running max nor a shift (sums stay below 2^(32+30)); otherwise (or for raw inputs) online max.
  pl.mode = (normalize && 2.f * c <= 64.f) ? SIM_NTX_FIXED : SIM_NTX_ONLINE;
  if (pl.mode == SIM_NTX_FIXED) {
    // the staged fp16 rows are pre-scaled by sqrt(c): the tensor-core accumulator IS the log2-domain logit and the
    // exp loops carry no scale/shift instruction.
    pl.prescale = sqrtf(c);
    pl.c = 1.f;
    pl.shift = 0.f;
    pl.pos_c = 1.f;
    // W_ab = P_ab + P_ba is ~2/M: below fp16's normal range for M > 2^15.  Carry 2^k with k = floor(log2 M) - 4
    // (typical W -> 2^-3, largest possible W = 2 -> 2^(k+1) <= 32768 < 65504).
    int k = 0;
    while ((int64_t{2} << k) <= pl.m) ++k;  // k = floor(log2 M)
    k -= 4;
    if (k < 0) k = 0;
    if (k > 14) k = 14;
    pl.wscale = static_cast<float>(1 << k);
  } else {
    pl.prescale = 1.f;
    pl.c = c;
    pl.shift = c;
    pl.pos_c = c;
    pl.wscale = 1.f;
  }
  return SSVB_OK;
}

struct SavedLayout {  // single-GPU saved blob
  __nv_bfloat16* zhat;
  float* inv_norm;
  float* stat;
  size_t bytes;
};
SavedLayout saved_layout(void* base, int64_t mpad, int64_t dpad) {
  Carver c(base);
  SavedLayout s;
  s.zhat = c.take<__nv_bfloat16>(mpad * dpad);
  s.inv_norm = c.take<float>(mpad);
  s.stat = c.take<float>(mpad);
  s.bytes = c.used();
  return s;
}

struct WsLayout {
  float* pos;
  float* part_m;
  float* part_l;
  float* block_sums;
  unsigned int* counter;
  float* dacc;
  size_t bytes;
};
// `cols` = 2 * n_global: the partial buffers are sized from the same chunk plan the launch uses, and are
// at least mpad floats so rows_bwd can stage the per-column statistics in part_m.
WsLayout ws_layout(void* base, int64_t local_rows, int64_t row_blocks, int64_t cols, int64_t dpad) {
  Carver c(base);
  WsLayout w;
  const int64_t lr = round_up(local_rows, 256);
  SimParams p{};
  p.row_blocks = static_cast<int>(row_blocks);
  p.cols = static_cast<int>(cols);
  plan_chunks(p, sim_fwd_bn(dpad), sim_fwd_min_tiles(dpad));
  size_t part_elems = static_cast<size_t>(4 * p.nchunks + 2) * lr;
  if (local_rows == cols && dpad <= 128) {
    // single GPU: the symmetric forward's row partials, then its (R - 1) / 2 column partials per row
    SimParams q{};
    q.row_blocks = static_cast<int>(row_blocks);
    const int ncol = plan_sym(q);
    const size_t sym_elems = static_cast<size_t>(4 * q.nchunks + ncol) * lr;
    if (part_elems < sym_elems) part_elems = sym_elems;
  }
  if (part_elems < static_cast<size_t>(sim_mpad(cols))) part_elems = sim_mpad(cols);
  w.pos = c.take<float>(lr);
  w.part_m = c.take<float>(part_elems);
  w.part_l = c.take<float>(part_elems);
  w.block_sums = c.take<float>(ceil_div(lr, 256) + 8);
  w.counter = c.take<unsigned int>(4);
  w.dacc = c.take<float>(lr * dpad);
  w.bytes = c.used();
  return w;
}

// ---- gradient finish: partner term, 1/(M tau) * grad_out, normalise-backward --------------------------
__global__ void ntx_grad_finish_kernel(const float* __restrict__ zi, const float* __restrict__ zj, int64_t ldi,
                                       int64_t ldj, int n_view, int d, int row0,
                                       const float* __restrict__ dacc, int ld_dacc,
                                       const __nv_bfloat16* __restrict__ zhat, int dpad,
                                       const float* __restrict__ inv_norm, int normalize, float inv_m_tau,
                                       const float* __restrict__ grad_out, float* __restrict__ dzi,
                                       float* __restrict__ dzj, int64_t ld_dzi, int64_t ld_dzj,
                                       float acc_scale, float zp_scale) {
  // acc_scale / zp_scale undo the staging scales: dacc = wscale * prescale * sum_b W_ab zh_b, staged rows = prescale * zh
  const int lrow = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (lrow >= 2 * n_view) return;
  const int view = lrow >= n_view;
  const int r = lrow - view * n_view;
  const int a_glob = row0 + lrow;  // rank-major layout: [rank][view][row]
  const int partner = view ? a_glob - n_view : a_glob + n_view;
  const float* z = view ? zj + static_cast<int64_t>(r) * ldj : zi + static_cast<int64_t>(r) * ldi;
  float* out = view ? dzj + static_cast<int64_t>(r) * ld_dzj : dzi + static_cast<int64_t>(r) * ld_dzi;
  const float scale = inv_m_tau * __ldg(grad_out);
  const float inv = normalize ? inv_norm[lrow] : 1.f;
  // d <= 256: up to two float4 per lane (columns lane * 4 and 128 + lane * 4)
  float g[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}}, zh[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
  float dot = 0.f;
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int k = it * 128 + lane * 4;
    if (k < d) {
      const float4 acc = *reinterpret_cast<const float4*>(dacc + static_cast<int64_t>(lrow) * ld_dacc + k);
      const uint2 pz = *reinterpret_cast<const uint2*>(zhat + static_cast<int64_t>(partner) * dpad + k);
      const float2 p01 = unpack_h2(pz.x, normalize != 0), p23 = unpack_h2(pz.y, normalize != 0);  // fp16 iff normalised
      const float4 zz = *reinterpret_cast<const float4*>(z + k);
      const float za = -2.f * zp_scale;
      g[it][0] = fmaf(acc.x, acc_scale, za * p01.x) * scale;
      g[it][1] = fmaf(acc.y, acc_scale, za * p01.y) * scale;
      g[it][2] = fmaf(acc.z, acc_scale, za * p23.x) * scale;
      g[it][3] = fmaf(acc.w, acc_scale, za * p23.y) * scale;
      zh[it][0] = zz.x * inv; zh[it][1] = zz.y * inv; zh[it][2] = zz.z * inv; zh[it][3] = zz.w * inv;
    }
    dot += g[it][0] * zh[it][0] + g[it][1] * zh[it][1] + g[it][2] * zh[it][2] + g[it][3] * zh[it][3];
  }
  if (normalize) {
    dot = warp_sum(dot);
#pragma unroll
    for (int it = 0; it < 2; ++it)
#pragma unroll
      for (int i = 0; i < 4; ++i) g[it][i] = (g[it][i] - dot * zh[it][i]) * inv;
  }
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int k = it * 128 + lane * 4;
    if (k < d) *reinterpret_cast<float4*>(out + k) = make_float4(g[it][0], g[it][1], g[it][2], g[it][3]);
  }
}

int check_rows(const void* p, int64_t ld) {
  if (!p) return SSVB_ERR_INVALID;
  if ((reinterpret_cast<uintptr_t>(p) & 15) || (ld & 3)) return SSVB_ERR_ALIGNMENT;
  return SSVB_OK;
}

void fill_sim_params_rows(SimParams& p, const NtxPlan& pl, int nseg, int64_t seg_rows, int64_t s0, int64_t s1) {
  p = SimParams{};
  p.opf16 = pl.normalize ? 1 : 0;  // fp16 staging for unit-norm rows (3 more mantissa bits than bf16), bf16 otherwise
  p.nseg = nseg;
  p.seg_rows = static_cast<int>(seg_rows);
  p.seg_start[0] = static_cast<int>(s0);
  p.seg_start[1] = static_cast<int>(s1);
  p.bps = static_cast<int>(ceil_div(seg_rows, 128));
  p.row_blocks = nseg * p.bps;
  p.cols = static_cast<int>(pl.m);
  p.c = pl.c;
  p.shift = pl.shift;
}

}  // namespace

extern "C" {

int64_t ssvb_ntxent_dpad(int64_t d) { return sim_dpad(d); }
int64_t ssvb_ntxent_mpad(int64_t n_global) { return sim_mpad(2 * n_global); }

size_t ssvb_ntxent_saved_bytes(int64_t n, int64_t d) {
  if (n <= 0 || d <= 0) return 0;
  return saved_layout(nullptr, sim_mpad(2 * n), sim_dpad(d)).bytes;
}
size_t ssvb_ntxent_workspace_bytes(int64_t n, int64_t d) {
  if (n <= 0 || d <= 0) return 0;
  return ws_layout(nullptr, 2 * n, ceil_div(2 * n, 128), 2 * n, sim_dpad(d)).bytes;
}

int ssvb_ntxent_fwd(const float* zi, const float* zj, int64_t n, int64_t d, int64_t ld_zi, int64_t ld_zj,
                    int normalize, float temperature, float* loss, void* saved, void* workspace,
                    size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  NtxPlan pl;
  SSVB_TRY(make_plan(pl, n, d, normalize, temperature));
  SSVB_TRY(check_rows(zi, ld_zi));
  SSVB_TRY(check_rows(zj, ld_zj));
  if (!loss || !saved || !workspace) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_ntxent_workspace_bytes(n, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  SavedLayout sv = saved_layout(saved, pl.mpad, pl.dpad);
  WsLayout ws = ws_layout(workspace, pl.m, ceil_div(pl.m, 128), pl.m, pl.dpad);

  // zero the padding rows of the bf16 staging matrix and the reduction counter
  if (pl.mpad > pl.m)
    SSVB_CUDA(cudaMemsetAsync(sv.zhat + pl.m * pl.dpad, 0, (pl.mpad - pl.m) * pl.dpad * sizeof(__nv_bfloat16), s));
  {
    const int wpb = 8;  // (the prep kernel also zeroes the finalize kernel's last-block counter: no memset node)
    pair_prep_kernel<<<static_cast<unsigned>(ceil_div(n, wpb)), wpb * 32, 0, s>>>(
        zi, zj, static_cast<int>(n), static_cast<int>(d), ld_zi, ld_zj, normalize, normalize ? 1 : 0, sv.zhat,
        sv.zhat + n * pl.dpad,
        static_cast<int>(pl.dpad), sv.inv_norm, sv.inv_norm + n, ws.pos, ws.pos + n, -1, pl.prescale, ws.counter);
    SSVB_LAUNCH_CHECK();
  }
  SimParams p;
  fill_sim_params_rows(p, pl, 1, pl.m, 0, 0);
  p.part_m = ws.part_m;
  p.part_l = ws.part_l;
  p.part_stride = static_cast<int>(round_up(pl.m, 256));
  // FIXED mode needs no running max, so S = S^T is exploited: every tile is computed once and also yields the row
  // sums of its mirror (column partials after the row partials, summed by the finalize in index order)
  int nparts;
  if (pl.mode == SIM_NTX_FIXED && pl.dpad <= 128) {
    const int ncol = plan_sym(p);
    p.colpart = ws.part_l + static_cast<size_t>(4 * p.nchunks) * p.part_stride;
    nparts = 4 * p.nchunks + ncol;
    SSVB_TRY(launch_sim_fwd_sym(sv.zhat, pl.mpad, pl.dpad, p, s));
  } else {
    plan_chunks(p, sim_fwd_bn(pl.dpad), sim_fwd_min_tiles(pl.dpad));
    nparts = 4 * p.nchunks;
    SSVB_TRY(launch_sim_fwd(pl.mode, sv.zhat, pl.mpad, sv.zhat, pl.mpad, pl.dpad, p, s));
  }
  {
    const unsigned grid = static_cast<unsigned>(ceil_div(pl.m, 256));
    const float scale = 1.f / static_cast<float>(pl.m);
    if (pl.mode == SIM_NTX_FIXED)
      lse_finalize_kernel<SIM_NTX_FIXED><<<grid, 256, 0, s>>>(ws.part_m, ws.part_l, nparts, p.part_stride,
                                                            static_cast<int>(pl.m), ws.pos, pl.c, pl.shift,
                                                            sv.stat, nullptr, ws.block_sums, ws.counter, scale, loss,
                                                            nullptr, nullptr, 0, 0, pl.wscale);
    else
      lse_finalize_kernel<SIM_NTX_ONLINE><<<grid, 256, 0, s>>>(ws.part_m, ws.part_l, nparts, p.part_stride,
                                                             static_cast<int>(pl.m), ws.pos, pl.c, pl.shift,
                                                             sv.stat, nullptr, ws.block_sums, ws.counter, scale, loss);
    SSVB_LAUNCH_CHECK();
    if (pl.mpad > pl.m) {
      const float padv = pl.mode == SIM_NTX_FIXED ? 0.f : 1e30f;
      fill_kernel<<<static_cast<unsigned>(ceil_div(pl.mpad - pl.m, 256)), 256, 0, s>>>(sv.stat + pl.m,
                                                                                       pl.mpad - pl.m, padv);
      SSVB_LAUNCH_CHECK();
    }
  }
  return SSVB_OK;
}

int ssvb_ntxent_bwd(const float* zi, const float* zj, int64_t n, int64_t d, int64_t ld_zi, int64_t ld_zj,
                    int normalize, float temperature, const float* grad_out, const void* saved, float* dzi,
                    float* dzj, int64_t ld_dzi, int64_t ld_dzj, void* workspace, size_t workspace_bytes,
                    void* stream) {
  SSVB_TRY(check_device_sm100());
  NtxPlan pl;
  SSVB_TRY(make_plan(pl, n, d, normalize, temperature));
  SSVB_TRY(check_rows(zi, ld_zi));
  SSVB_TRY(check_rows(zj, ld_zj));
  SSVB_TRY(check_rows(dzi, ld_dzi));
  SSVB_TRY(check_rows(dzj, ld_dzj));
  if (!grad_out || !saved || !workspace) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_ntxent_workspace_bytes(n, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  SavedLayout sv = saved_layout(const_cast<void*>(saved), pl.mpad, pl.dpad);
  WsLayout ws = ws_layout(workspace, pl.m, ceil_div(pl.m, 128), pl.m, pl.dpad);

  SimParams p;
  fill_sim_params_rows(p, pl, 1, pl.m, 0, 0);
  plan_chunks(p, 128, 8);
  p.rowstat = sv.stat;
  p.colstat = sv.stat;
  p.dacc = ws.dacc;
  p.ld_dacc = static_cast<int>(pl.dpad);
  p.use_atomic = p.nchunks > 1;
  if (p.use_atomic) SSVB_CUDA(cudaMemsetAsync(ws.dacc, 0, pl.m * pl.dpad * sizeof(float), s));
  SSVB_TRY(launch_sim_bwd(pl.mode, sv.zhat, pl.mpad, sv.zhat, pl.mpad, pl.dpad, p, s));
  {
    const int wpb = 8;
    ntx_grad_finish_kernel<<<static_cast<unsigned>(ceil_div(pl.m, wpb)), wpb * 32, 0, s>>>(
        zi, zj, ld_zi, ld_zj, static_cast<int>(n), static_cast<int>(d), 0, ws.dacc,
        static_cast<int>(pl.dpad), sv.zhat, static_cast<int>(pl.dpad), sv.inv_norm, normalize,
        1.f / (static_cast<float>(pl.m) * temperature), grad_out, dzi, dzj, ld_dzi, ld_dzj,
        1.f / (pl.wscale * pl.prescale), 1.f / pl.prescale);
    SSVB_LAUNCH_CHECK();
  }
  return SSVB_OK;
}

// ------------------------------------------------------------------------------------ multi-GPU pieces
// Gathered layout is RANK-MAJOR: global row of (rank r, view v, local row i) = r*2L + v*L + i with L = n_local,
// so every rank owns ONE contiguous slot of zhat_all / stat_all (a single all-gather each) and the positive
// partner of a row is always on the same rank (a +- L).  NT-Xent is invariant to this row permutation.
size_t ssvb_ntxent_dist_workspace_bytes(int64_t world, int64_t n_local, int64_t d) {
  if (world <= 0 || n_local <= 0 || d <= 0) return 0;
  return ws_layout(nullptr, 2 * n_local, ceil_div(2 * n_local, 128), 2 * n_local * world, sim_dpad(d)).bytes;
}

namespace {
int dist_check(int64_t world, int64_t rank, int64_t n_local) {
  if (world <= 0 || rank < 0 || rank >= world || n_local <= 0) return SSVB_ERR_INVALID;
  return SSVB_OK;
}
}  // namespace

int ssvb_ntxent_dist_prep(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi,
                          int64_t ld_zj, int normalize, float temperature, int64_t world, int64_t rank,
                          void* zhat_all, float* inv_norm_local, float* pos_local, void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(dist_check(world, rank, n_local));
  NtxPlan pl;
  SSVB_TRY(make_plan(pl, n_local * world, d, normalize, temperature));
  SSVB_TRY(check_rows(zi, ld_zi));
  SSVB_TRY(check_rows(zj, ld_zj));
  if (!zhat_all || !inv_norm_local || !pos_local) return SSVB_ERR_INVALID;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  __nv_bfloat16* zh = static_cast<__nv_bfloat16*>(zhat_all);
  if (pl.mpad > pl.m)
    SSVB_CUDA(cudaMemsetAsync(zh + pl.m * pl.dpad, 0, (pl.mpad - pl.m) * pl.dpad * sizeof(__nv_bfloat16), s));
  const int64_t row0 = rank * 2 * n_local;
  const int wpb = 8;
  pair_prep_kernel<<<static_cast<unsigned>(ceil_div(n_local, wpb)), wpb * 32, 0, s>>>(
      zi, zj, static_cast<int>(n_local), static_cast<int>(d), ld_zi, ld_zj, normalize, normalize ? 1 : 0,
      zh + row0 * pl.dpad,
      zh + (row0 + n_local) * pl.dpad, static_cast<int>(pl.dpad), inv_norm_local, inv_norm_local + n_local,
      pos_local, pos_local + n_local, -1, pl.prescale);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

namespace {
int rows_fwd_impl(const void* zhat_all, int64_t world, int64_t rank, int64_t n_local, int64_t d, int normalize,
                  float temperature, const float* pos_local, float* stat_local, float* const* peer_stat,
                  float* loss_sum, void* workspace, size_t workspace_bytes, void* stream, size_t peer_stat_off = 0,
                  uint32_t gen = 0, unsigned int* counter = nullptr);
}
int ssvb_ntxent_dist_rows_fwd(const void* zhat_all, int64_t world, int64_t rank, int64_t n_local, int64_t d,
                              int normalize, float temperature, const float* pos_local, float* stat_local,
                              float* loss_sum, void* workspace, size_t workspace_bytes, void* stream) {
  if (!stat_local) return SSVB_ERR_INVALID;
  return rows_fwd_impl(zhat_all, world, rank, n_local, d, normalize, temperature, pos_local, stat_local, nullptr,
                       loss_sum, workspace, workspace_bytes, stream);
}
namespace {
int rows_fwd_impl(const void* zhat_all, int64_t world, int64_t rank, int64_t n_local, int64_t d, int normalize,
                  float temperature, const float* pos_local, float* stat_local, float* const* peer_stat,
                  float* loss_sum, void* workspace, size_t workspace_bytes, void* stream, size_t peer_stat_off,
                  uint32_t gen, unsigned int* counter) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(dist_check(world, rank, n_local));
  NtxPlan pl;
  SSVB_TRY(make_plan(pl, n_local * world, d, normalize, temperature));
  if (!zhat_all || !pos_local || !loss_sum || !workspace) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_ntxent_dist_workspace_bytes(world, n_local, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t lr = 2 * n_local;
  WsLayout ws = ws_layout(workspace, lr, ceil_div(lr, 128), pl.m, pl.dpad);
  // last-block counter of the finalize kernel: the workspace one needs zeroing (arbitrary contents); the peer-memory
  // transport passes one that lives in the zero-initialised arena and resets itself after every use (one launch less)
  if (!counter) {
    counter = ws.counter;
    SSVB_CUDA(cudaMemsetAsync(counter, 0, 16, s));
  }
  // local outputs either go to the caller's [2][2L] block or (push mode) into slot `rank` of every peer's buffer
  float* lse_out = stat_local;
  float* term_out = stat_local ? stat_local + lr : nullptr;
  // element offset of this rank's block inside every peer's buffer: plain floats, or 8-byte {value, generation} pairs
  const size_t peer_off = peer_stat_off / (gen ? sizeof(uint2) : sizeof(float)) + static_cast<size_t>(rank) * 2 * lr;
  SimParams p;
  fill_sim_params_rows(p, pl, 1, lr, rank * lr, 0);
  plan_chunks(p, sim_fwd_bn(pl.dpad), sim_fwd_min_tiles(pl.dpad));
  p.part_m = ws.part_m;
  p.part_l = ws.part_l;
  p.part_stride = static_cast<int>(round_up(lr, 256));
  SSVB_TRY(launch_sim_fwd(pl.mode, zhat_all, pl.mpad, zhat_all, pl.mpad, pl.dpad, p, s));
  const unsigned grid = static_cast<unsigned>(ceil_div(lr, 256));
  // stat_local always carries the log2-domain LSE (what gets all-gathered); the FIXED-mode 1/L' is
  // re-derived from it in rows_bwd.
  if (pl.mode == SIM_NTX_FIXED)
    lse_finalize_kernel<SIM_NTX_FIXED><<<grid, 256, 0, s>>>(ws.part_m, ws.part_l, 4 * p.nchunks, p.part_stride,
                                                          static_cast<int>(lr), pos_local, pl.c, pl.shift,
                                                          ws.dacc /*scratch*/, lse_out, ws.block_sums, counter,
                                                          1.f, loss_sum, term_out, peer_stat, static_cast<int>(world),
                                                          peer_off, 1.f, gen);
  else
    lse_finalize_kernel<SIM_NTX_ONLINE><<<grid, 256, 0, s>>>(ws.part_m, ws.part_l, 4 * p.nchunks, p.part_stride,
                                                           static_cast<int>(lr), pos_local, pl.c, pl.shift,
                                                           ws.dacc /*scratch*/, lse_out, ws.block_sums,
                                                           counter, 1.f, loss_sum, term_out, peer_stat,
                                                           static_cast<int>(world), peer_off, 1.f, gen);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}
}  // namespace

// global loss from the gathered per-row terms: loss = sum(stat_all[:, 1, :]) / (2 * world * L); fixed order
namespace {
__global__ void dist_loss_kernel(const float* __restrict__ g, int world, int lr, float scale, float* __restrict__ out) {
  // sum of the gathered per-row loss terms ([world][2][lr], second half of every block) in a FIXED order (identical on
  // every rank).  8 independent loads in flight per thread: the serial version (64 dependent-latency loads per thread)
  // took 29 us at world*lr = 65536.
  __shared__ float red[32];
  float acc[8];
#pragma unroll
  for (int u = 0; u < 8; ++u) acc[u] = 0.f;
  for (int r = 0; r < world; ++r) {
    const float* t = g + static_cast<size_t>(r) * 2 * lr + lr;
    int i = threadIdx.x;
    for (; i + 7 * static_cast<int>(blockDim.x) < lr; i += 8 * blockDim.x) {
#pragma unroll
      for (int u = 0; u < 8; ++u) acc[u] += t[i + u * blockDim.x];
    }
    for (; i < lr; i += blockDim.x) acc[0] += t[i];
  }
  float v = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) out[0] = t * scale;
  }
}
}  // namespace
int ssvb_ntxent_dist_loss(const float* stat_all, int64_t world, int64_t n_local, float* loss, void* stream) {
  SSVB_TRY(check_device_sm100());
  if (!stat_all || !loss || world <= 0 || n_local <= 0) return SSVB_ERR_INVALID;
  dist_loss_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(
      stat_all, static_cast<int>(world), static_cast<int>(2 * n_local), 1.f / static_cast<float>(2 * world * n_local),
      loss);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

namespace {
// lse2 (all rows) -> the column statistic the backward kernel consumes, with finite padding
// gathered layout: [world][2][2L] (per rank: 2L lse2 values, then 2L per-row loss terms)
__global__ void dist_stat_kernel(const float* __restrict__ gathered, float* __restrict__ stat, int m, int mpad, int lr,
                                 int fixed, float shift, float wscale) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= mpad) return;
  if (i < m) {
    const int r = i / lr;
    const float l2 = gathered[static_cast<size_t>(r) * 2 * lr + (i - r * lr)];
    stat[i] = fixed ? wscale * exp2f(shift - l2) : l2;
  } else {
    stat[i] = fixed ? 0.f : 1e30f;
  }
}
}  // namespace

namespace {
int rows_bwd_impl(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi, int64_t ld_zj,
                  int normalize, float temperature, int64_t world, int64_t rank, const void* zhat_all,
                  const float* stat_all, const float* colstat, const float* inv_norm_local, const float* grad_out,
                  float* dzi, float* dzj, int64_t ld_dzi, int64_t ld_dzj, void* workspace, size_t workspace_bytes,
                  void* stream);
}
int ssvb_ntxent_dist_rows_bwd(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi,
                              int64_t ld_zj, int normalize, float temperature, int64_t world, int64_t rank,
                              const void* zhat_all, const float* stat_all, const float* inv_norm_local,
                              const float* grad_out, float* dzi, float* dzj, int64_t ld_dzi, int64_t ld_dzj,
                              void* workspace, size_t workspace_bytes, void* stream) {
  if (!stat_all) return SSVB_ERR_INVALID;
  return rows_bwd_impl(zi, zj, n_local, d, ld_zi, ld_zj, normalize, temperature, world, rank, zhat_all, stat_all,
                       nullptr, inv_norm_local, grad_out, dzi, dzj, ld_dzi, ld_dzj, workspace, workspace_bytes, stream);
}
namespace {
int rows_bwd_impl(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi, int64_t ld_zj,
                  int normalize, float temperature, int64_t world, int64_t rank, const void* zhat_all,
                  const float* stat_all, const float* colstat, const float* inv_norm_local, const float* grad_out,
                  float* dzi, float* dzj, int64_t ld_dzi, int64_t ld_dzj, void* workspace, size_t workspace_bytes,
                  void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(dist_check(world, rank, n_local));
  NtxPlan pl;
  SSVB_TRY(make_plan(pl, n_local * world, d, normalize, temperature));
  SSVB_TRY(check_rows(zi, ld_zi));
  SSVB_TRY(check_rows(zj, ld_zj));
  SSVB_TRY(check_rows(dzi, ld_dzi));
  SSVB_TRY(check_rows(dzj, ld_dzj));
  if (!zhat_all || (!stat_all && !colstat) || !inv_norm_local || !grad_out || !workspace) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_ntxent_dist_workspace_bytes(world, n_local, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t lr = 2 * n_local;
  WsLayout ws = ws_layout(workspace, lr, ceil_div(lr, 128), pl.m, pl.dpad);
  const float* stat = colstat;  // peer-memory transport: already derived (and padded) by the statistics kernel
  if (!stat) {
    // column statistics for all M rows live in the (otherwise unused here) partial buffer
    dist_stat_kernel<<<static_cast<unsigned>(ceil_div(pl.mpad, 256)), 256, 0, s>>>(
        stat_all, ws.part_m, static_cast<int>(pl.m), static_cast<int>(pl.mpad), static_cast<int>(lr),
        pl.mode == SIM_NTX_FIXED, pl.shift, pl.wscale);
    SSVB_LAUNCH_CHECK();
    stat = ws.part_m;
  }

  SimParams p;
  fill_sim_params_rows(p, pl, 1, lr, rank * lr, 0);
  plan_chunks(p, 128, 8);
  p.rowstat = stat;
  p.colstat = stat;
  p.dacc = ws.dacc;
  p.ld_dacc = static_cast<int>(pl.dpad);
  p.use_atomic = p.nchunks > 1;
  if (p.use_atomic) SSVB_CUDA(cudaMemsetAsync(ws.dacc, 0, lr * pl.dpad * sizeof(float), s));
  SSVB_TRY(launch_sim_bwd(pl.mode, zhat_all, pl.mpad, zhat_all, pl.mpad, pl.dpad, p, s));
  const int wpb = 8;
  ntx_grad_finish_kernel<<<static_cast<unsigned>(ceil_div(lr, wpb)), wpb * 32, 0, s>>>(
      zi, zj, ld_zi, ld_zj, static_cast<int>(n_local), static_cast<int>(d), static_cast<int>(rank * lr), ws.dacc,
      static_cast<int>(pl.dpad), static_cast<const __nv_bfloat16*>(zhat_all), static_cast<int>(pl.dpad),
      inv_norm_local, normalize, 1.f / (static_cast<float>(pl.m) * temperature), grad_out, dzi, dzj, ld_dzi, ld_dzj,
        1.f / (pl.wscale * pl.prescale), 1.f / pl.prescale);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}
}  // namespace

}  // extern "C"

// =====================================================================================================
// NVLink peer-memory transport (fused compute + all-gather, no NCCL and no host-issued barrier on the data path).
// Every rank owns one SYMMETRIC arena (same layout everywhere, peer-mapped, e.g. torch symmetric memory):
//     zhat[2]  : 2 x (2L*world) x dpad 16-bit rows   - the gathered normalised rows, double-buffered by generation parity
//     stat[2]  : 2 x [world][2][2L] x 8 bytes         - the gathered [lse2 | per-row loss term] blocks, double-buffered
//     stat[2]  : (see above) every element is an 8-byte {value, generation} pair ("LL" form: an 8-byte store is one
//                transaction, the consumer validates each element by its tag - no fence, no completion flag)
//     flags    : [world] uint32                       - flags[r] = last generation whose ROWS rank r has completely
//                                                       published into THIS arena
//     counter  : 3 x uint32 (+ padding)               - self-resetting last-block counters (push / finalize / stat_loss)
// A forward of generation g:  p2p_prep_push (normalise, store own slot into every arena - unicast peer stores or one
// multicast store through the switch -, last block publishes flags[rank] = g everywhere)  ->  p2p_wait_copy (waits
// for flags[*] >= g, copies the gathered rows into a private matrix: the tensor-core kernels read ordinary device
// memory faster than a peer-mapped mapping)  ->  sim_fwd + finalize (stores tagged [lse2 | term] pairs into every
// arena)  ->  p2p_stat_loss (waits for every pair of generation g, derives the backward's column
// statistics and the global loss in a fixed order: bit-identical on every rank).  Backward needs no exchange.
// Double buffering makes the protocol barrier-free: a rank can only push generation g+2 (same parity as g) after it
// has seen every peer's generation g+1 statistics, which a peer publishes after it has finished reading generation g.
// =====================================================================================================
struct ArenaLayout {
  size_t zhat[2], stat[2], flags, counter, bytes;
};
ArenaLayout arena_layout(int64_t world, int64_t n_local, int64_t dpad) {
  ArenaLayout a;
  size_t off = 0;
  auto take = [&](size_t nbytes) {
    off = (off + 1023) & ~static_cast<size_t>(1023);
    const size_t r = off;
    off += nbytes;
    return r;
  };
  const size_t m = static_cast<size_t>(2 * n_local * world);
  for (int i = 0; i < 2; ++i) a.zhat[i] = take(m * dpad * sizeof(__nv_bfloat16));
  for (int i = 0; i < 2; ++i) a.stat[i] = take(m * 2 * sizeof(uint2));  // {value, generation} pairs
  a.flags = take(static_cast<size_t>(world) * sizeof(uint32_t));
  a.counter = take(64);
  a.bytes = (off + 1023) & ~static_cast<size_t>(1023);
  return a;
}

namespace {
// ROWS_PER_WARP row pairs per warp with all their loads issued up front (the one-row-per-warp form is latency-bound:
// one 16-byte load per lane in flight), 8 warps per CTA.
constexpr int P2P_RPW = 2;
__global__ void __launch_bounds__(256)
p2p_prep_push_kernel(const float* __restrict__ xi, const float* __restrict__ xj, int n, int d,
                                     int64_t ldi, int64_t ldj, int normalize, int f16, float prescale,
                                     uint8_t* const* __restrict__ peers, uint8_t* mc_base, size_t zoff, size_t flag_off,
                                     unsigned int* counter, int world, int rank, int64_t row_i, int64_t row_j, int dpad,
                                     float* __restrict__ inv_i, float* __restrict__ inv_j, float* __restrict__ pos_i,
                                     float* __restrict__ pos_j, uint32_t gen) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int r0 = warp * P2P_RPW;
  const int k = lane * 4;  // dpad <= 128: one float4 per lane and row
  float4 a[P2P_RPW], b[P2P_RPW];
#pragma unroll
  for (int j = 0; j < P2P_RPW; ++j) {
    a[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    b[j] = a[j];
    if (r0 + j < n && k < d) {
      a[j] = __ldg(reinterpret_cast<const float4*>(xi + static_cast<int64_t>(r0 + j) * ldi + k));
      b[j] = __ldg(reinterpret_cast<const float4*>(xj + static_cast<int64_t>(r0 + j) * ldj + k));
    }
  }
  // start at a different peer per CTA so the ranks do not all hit the same NVLink port at the same time
  const int p0 = static_cast<int>(blockIdx.x % static_cast<unsigned>(world));
#pragma unroll
  for (int j = 0; j < P2P_RPW; ++j) {
    const int row = r0 + j;
    if (row >= n) break;  // warp-uniform
    const float si = warp_sum(a[j].x * a[j].x + a[j].y * a[j].y + a[j].z * a[j].z + a[j].w * a[j].w);
    const float sj = warp_sum(b[j].x * b[j].x + b[j].y * b[j].y + b[j].z * b[j].z + b[j].w * b[j].w);
    float ivi = 1.f, ivj = 1.f;
    if (normalize) {
      ivi = 1.f / fmaxf(sqrtf(si), 1e-12f);
      ivj = 1.f / fmaxf(sqrtf(sj), 1e-12f);
    }
    const float si_ = ivi * prescale, sj_ = ivj * prescale;
    uint2 vi, vj;
    vi.x = f16 ? pack_f16x2(a[j].x * si_, a[j].y * si_) : pack_bf16x2(a[j].x * si_, a[j].y * si_);
    vi.y = f16 ? pack_f16x2(a[j].z * si_, a[j].w * si_) : pack_bf16x2(a[j].z * si_, a[j].w * si_);
    vj.x = f16 ? pack_f16x2(b[j].x * sj_, b[j].y * sj_) : pack_bf16x2(b[j].x * sj_, b[j].y * sj_);
    vj.y = f16 ? pack_f16x2(b[j].z * sj_, b[j].w * sj_) : pack_bf16x2(b[j].z * sj_, b[j].w * sj_);
    const float2 fi01 = unpack_h2(vi.x, f16), fi23 = unpack_h2(vi.y, f16);
    const float2 fj01 = unpack_h2(vj.x, f16), fj23 = unpack_h2(vj.y, f16);
    const float dot = warp_sum(fi01.x * fj01.x + fi01.y * fj01.y + fi23.x * fj23.x + fi23.y * fj23.y);
    if (k < dpad) {
      const size_t oi = zoff + (static_cast<size_t>(row_i + row) * dpad + k) * 2;
      const size_t oj = zoff + (static_cast<size_t>(row_j + row) * dpad + k) * 2;
      if (mc_base) {  // one store each through the NVSwitch multicast mapping reaches every rank's arena
        multimem_st_v2(mc_base + oi, vi);
        multimem_st_v2(mc_base + oj, vj);
      } else {
        for (int q = 0; q < world; ++q) {
          uint8_t* base = peers[(p0 + q) % world];
          *reinterpret_cast<uint2*>(base + oi) = vi;
          *reinterpret_cast<uint2*>(base + oj) = vj;
        }
      }
    }
    if (lane == 0) {
      inv_i[row] = ivi; inv_j[row] = ivj; pos_i[row] = dot; pos_j[row] = dot;
    }
  }
  // publish: CTA barrier, then ONE thread fences at system scope (cumulative over the stores it has observed through
  // the barrier - the cooperative-groups grid-sync idiom) and counts the CTA in; the last CTA raises this rank's flag
  // in every arena.
  __syncthreads();
  __shared__ bool is_last;
  if (threadIdx.x == 0) {
    __threadfence_system();
    const unsigned int done = atomicAdd(counter, 1u);
    is_last = (done == gridDim.x - 1);
    if (is_last) __threadfence();  // acquire side of the counter hand-off (device scope: the counter is local)
  }
  __syncthreads();
  if (is_last) {
    // every CTA fenced its stores at SYSTEM scope before counting in and this CTA has acquired all of those increments:
    // the system-scope release store below is ordered after all of them - no second system fence (each costs a
    // round trip over NVLink once remote stores are outstanding)
    if (threadIdx.x < world) {
      uint32_t* f = reinterpret_cast<uint32_t*>(peers[threadIdx.x] + flag_off);
      st_release_sys_u32(f + rank, gen);
    }
    if (threadIdx.x == 0) *counter = 0;
  }
}

// waits (per slot) until the owning rank has published generation `gen`, then copies that slot of the local arena
// into the private gathered matrix.  CTA b serves slot (b + rank) % world, so the local slot is handled first.
__global__ void p2p_wait_copy_kernel(const uint8_t* __restrict__ arena, size_t zoff, size_t flag_off, int world, int rank,
                                     uint32_t gen, uint4* __restrict__ dst, size_t slot_vecs) {
  const int slot = (static_cast<int>(blockIdx.x) + rank) % world;
  const int part = blockIdx.x / world, nparts = gridDim.x / world;
  if (part >= nparts) return;
  if (threadIdx.x == 0) spin_wait_gen(reinterpret_cast<const uint32_t*>(arena + flag_off) + slot, gen);
  __syncthreads();
  const uint4* src = reinterpret_cast<const uint4*>(arena + zoff) + static_cast<size_t>(slot) * slot_vecs;
  uint4* out = dst + static_cast<size_t>(slot) * slot_vecs;
  for (size_t i = static_cast<size_t>(part) * blockDim.x + threadIdx.x; i < slot_vecs;
       i += static_cast<size_t>(nparts) * blockDim.x)
    out[i] = __ldcg(src + i);
}

// waits for every rank's statistics of generation `gen`, then (a) column statistics of all M rows for the backward
// kernel (FIXED: wscale / L', else lse2; finite padding), (b) the global loss = fixed-order sum of the per-row terms.
__global__ void p2p_stat_loss_kernel(const uint8_t* arena, size_t soff, uint32_t gen, int lr, int m, int mpad, int fixed, float shift, float wscale,
                                     float* __restrict__ colstat, float* block_sums, unsigned int* counter, float scale,
                                     float* loss) {
  // every element arrives as an 8-byte {value, generation} pair: wait for the tag of THIS generation, element by element
  const uint2* g = reinterpret_cast<const uint2*>(arena + soff);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  float term = 0.f;
  if (i < mpad) {
    if (i < m) {
      const int r = i / lr;
      const size_t base = static_cast<size_t>(r) * 2 * lr + (i - r * lr);
      const float l2 = ll_wait_value(g + base, gen);
      term = ll_wait_value(g + base + lr, gen);
      colstat[i] = fixed ? wscale * exp2f(shift - l2) : l2;
    } else {
      colstat[i] = fixed ? 0.f : 1e30f;
    }
  }
  const float bt = block_sum_256(term);
  grid_sum_finish(bt, block_sums, counter, scale, loss, false);
}
}  // namespace

extern "C" {

size_t ssvb_ntxent_p2p_arena_bytes(int64_t world, int64_t n_local, int64_t d) {
  if (world <= 0 || n_local <= 0 || d <= 0) return 0;
  return arena_layout(world, n_local, sim_dpad(d)).bytes;
}

int ssvb_ntxent_p2p_prep_push(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi,
                              int64_t ld_zj, int normalize, float temperature, int64_t world, int64_t rank,
                              void* arena_local, void* const* peer_arenas, void* multicast_arena, int64_t gen,
                              float* inv_norm_local, float* pos_local, void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(dist_check(world, rank, n_local));
  if (world > 256 || d > 128) return SSVB_ERR_UNSUPPORTED;  // the push kernel moves one float4 per lane and row
  NtxPlan pl;
  SSVB_TRY(make_plan(pl, n_local * world, d, normalize, temperature));
  SSVB_TRY(check_rows(zi, ld_zi));
  SSVB_TRY(check_rows(zj, ld_zj));
  if (!arena_local || !peer_arenas || !inv_norm_local || !pos_local || gen <= 0) return SSVB_ERR_INVALID;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const ArenaLayout al = arena_layout(world, n_local, pl.dpad);
  const int64_t row0 = rank * 2 * n_local;
  const uint32_t g = static_cast<uint32_t>(gen);
  p2p_prep_push_kernel<<<static_cast<unsigned>(ceil_div(n_local, 8 * P2P_RPW)), 256, 0, s>>>(
      zi, zj, static_cast<int>(n_local), static_cast<int>(d), ld_zi, ld_zj, normalize, normalize ? 1 : 0, pl.prescale,
      reinterpret_cast<uint8_t* const*>(peer_arenas), static_cast<uint8_t*>(multicast_arena), al.zhat[g & 1], al.flags,
      reinterpret_cast<unsigned int*>(static_cast<uint8_t*>(arena_local) + al.counter), static_cast<int>(world),
      static_cast<int>(rank), row0, row0 + n_local, static_cast<int>(pl.dpad), inv_norm_local,
      inv_norm_local + n_local, pos_local, pos_local + n_local, g);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

int ssvb_ntxent_p2p_wait_copy(const void* arena_local, int64_t world, int64_t rank, int64_t n_local, int64_t d,
                              int64_t gen, void* zhat_all, void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(dist_check(world, rank, n_local));
  if (!arena_local || !zhat_all || gen <= 0 || d <= 0) return SSVB_ERR_INVALID;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t dpad = sim_dpad(d), m = 2 * n_local * world, mpad = sim_mpad(m);
  const ArenaLayout al = arena_layout(world, n_local, dpad);
  __nv_bfloat16* zh = static_cast<__nv_bfloat16*>(zhat_all);
  if (mpad > m) SSVB_CUDA(cudaMemsetAsync(zh + m * dpad, 0, (mpad - m) * dpad * sizeof(__nv_bfloat16), s));
  const size_t slot_vecs = static_cast<size_t>(2 * n_local) * dpad * 2 / 16;  // dpad % 64 == 0: whole 16-byte vectors
  // enough CTAs to run at copy bandwidth, a whole number of them per slot, all co-resident (they spin on flags)
  int parts = static_cast<int>(ceil_div(2 * num_sms(), world));
  const int64_t max_parts = ceil_div(static_cast<int64_t>(slot_vecs), 256);
  if (parts > max_parts) parts = static_cast<int>(max_parts);
  if (parts < 1) parts = 1;
  p2p_wait_copy_kernel<<<static_cast<unsigned>(parts * world), 256, 0, s>>>(
      static_cast<const uint8_t*>(arena_local), al.zhat[static_cast<uint32_t>(gen) & 1], al.flags,
      static_cast<int>(world), static_cast<int>(rank), static_cast<uint32_t>(gen), reinterpret_cast<uint4*>(zhat_all),
      slot_vecs);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

int ssvb_ntxent_p2p_rows_fwd(const void* zhat_all, int64_t world, int64_t rank, int64_t n_local, int64_t d,
                             int normalize, float temperature, const float* pos_local, void* arena_local,
                             void* const* peer_arenas, int64_t gen, float* loss_sum, void* workspace,
                             size_t workspace_bytes, void* stream) {
  if (!arena_local || !peer_arenas || gen <= 0 || d <= 0) return SSVB_ERR_INVALID;
  const ArenaLayout al = arena_layout(world, n_local, sim_dpad(d));
  return rows_fwd_impl(zhat_all, world, rank, n_local, d, normalize, temperature, pos_local, nullptr,
                       reinterpret_cast<float* const*>(peer_arenas), loss_sum, workspace, workspace_bytes, stream,
                       al.stat[static_cast<uint32_t>(gen) & 1], static_cast<uint32_t>(gen),
                       reinterpret_cast<unsigned int*>(static_cast<uint8_t*>(arena_local) + al.counter) + 1);
}

int ssvb_ntxent_p2p_stat_loss(void* arena_local, int64_t world, int64_t rank, int64_t n_local, int64_t d,
                              int normalize, float temperature, int64_t gen, float* colstat, float* loss,
                              void* workspace, size_t workspace_bytes, void* stream) {
  SSVB_TRY(check_device_sm100());
  SSVB_TRY(dist_check(world, rank, n_local));
  NtxPlan pl;
  SSVB_TRY(make_plan(pl, n_local * world, d, normalize, temperature));
  if (!arena_local || !colstat || !loss || !workspace || gen <= 0 || world > 256) return SSVB_ERR_INVALID;
  if (workspace_bytes < ssvb_ntxent_dist_workspace_bytes(world, n_local, d)) return SSVB_ERR_WORKSPACE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t lr = 2 * n_local;
  WsLayout ws = ws_layout(workspace, lr, ceil_div(lr, 128), pl.m, pl.dpad);
  const ArenaLayout al = arena_layout(world, n_local, pl.dpad);
  // block partials: part_l is free again once the finalize kernel of this forward has run (same stream)
  float* block_sums = ws.part_l;
  p2p_stat_loss_kernel<<<static_cast<unsigned>(ceil_div(pl.mpad, 256)), 256, 0, s>>>(
      static_cast<const uint8_t*>(arena_local), al.stat[static_cast<uint32_t>(gen) & 1],
      static_cast<uint32_t>(gen), static_cast<int>(lr), static_cast<int>(pl.m),
      static_cast<int>(pl.mpad), pl.mode == SIM_NTX_FIXED, pl.shift, pl.wscale, colstat, block_sums,
      reinterpret_cast<unsigned int*>(const_cast<uint8_t*>(static_cast<const uint8_t*>(arena_local)) + al.counter) + 2,
      1.f / static_cast<float>(pl.m), loss);
  SSVB_LAUNCH_CHECK();
  return SSVB_OK;
}

// The four forward stages in ONE call (the product path of DistributedSimclrLoss): at 8 GPUs the whole step is ~0.4 ms,
// so every host microsecond between the launches shows; one ctypes crossing instead of four.
int ssvb_ntxent_p2p_forward(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi, int64_t ld_zj,
                            int normalize, float temperature, int64_t world, int64_t rank, void* arena_local,
                            void* const* peer_arenas, void* multicast_arena, int64_t gen, void* zhat_all,
                            float* inv_norm_local, float* pos_local, float* colstat, float* loss_sum, float* loss,
                            void* workspace, size_t workspace_bytes, void* stream) {
  SSVB_TRY(ssvb_ntxent_p2p_prep_push(zi, zj, n_local, d, ld_zi, ld_zj, normalize, temperature, world, rank, arena_local,
                                     peer_arenas, multicast_arena, gen, inv_norm_local, pos_local, stream));
  SSVB_TRY(ssvb_ntxent_p2p_wait_copy(arena_local, world, rank, n_local, d, gen, zhat_all, stream));
  SSVB_TRY(ssvb_ntxent_p2p_rows_fwd(zhat_all, world, rank, n_local, d, normalize, temperature, pos_local, arena_local,
                                    peer_arenas, gen, loss_sum, workspace, workspace_bytes, stream));
  return ssvb_ntxent_p2p_stat_loss(arena_local, world, rank, n_local, d, normalize, temperature, gen, colstat, loss,
                                   workspace, workspace_bytes, stream);
}

int ssvb_ntxent_p2p_rows_bwd(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi,
                             int64_t ld_zj, int normalize, float temperature, int64_t world, int64_t rank,
                             const void* zhat_all, const float* colstat, const float* inv_norm_local,
                             const float* grad_out, float* dzi, float* dzj, int64_t ld_dzi, int64_t ld_dzj,
                             void* workspace, size_t workspace_bytes, void* stream) {
  if (!colstat) return SSVB_ERR_INVALID;
  return rows_bwd_impl(zi, zj, n_local, d, ld_zi, ld_zj, normalize, temperature, world, rank, zhat_all, nullptr,
                       colstat, inv_norm_local, grad_out, dzi, dzj, ld_dzi, ld_dzj, workspace, workspace_bytes, stream);
}

}  // extern "C"
