/* ssv_b200 — C ABI of the B200-native self-supervised loss hot path.
 *
 * Drop-in boundary for the loss layer of NightShade99/Self-Supervised-Vision
 * (reference `utils/losses.py` + the ring buffers of `models/moco.py`, `models/swav.py`).
 * The reference is pure Python/PyTorch and has no FFI of its own; these entry points are
 * what a `ctypes` binding added to the reference's `utils/losses.py` would bind (see
 * INTEGRATION.md).  Every entry point cites the reference interface it replaces.
 *
 * Conventions
 *  - all pointers are DEVICE pointers (current device), fp32 row-major unless noted;
 *    `ld*` are leading dimensions in ELEMENTS; rows must be 16-byte aligned
 *    (pointer % 16 == 0, ld % 4 == 0);
 *  - the caller owns every buffer (inputs, outputs, `saved`, `workspace`); the library never
 *    allocates or frees device memory and keeps no pointer after returning;
 *  - `saved` is an opaque blob written by `*_fwd` and read by the matching `*_bwd`
 *    (size from `*_saved_bytes`); `workspace` is scratch (size from `*_workspace_bytes`);
 *  - all work is enqueued asynchronously on `stream` (a `cudaStream_t`); no host sync, no
 *    global mutable state that affects results: entry points are re-entrant (autograd calls bwd from its own thread;
 *    the library only memoises - a per-thread cache of encoded TMA descriptors, per-kernel attribute bits - and
 *    keeps the opt-in profiling counters of ssvb_profile_enable).  One switch for tests is read from the environment
 *    once per process: SSVB_GEMM_NO_TMA_STORE forces the per-thread row-store GEMM epilogue that rows without 16-byte
 *    alignment take, same results within rounding; unset = the shipped path;
 *  - `loss` and `grad_out` are device scalars (fp32) so no device->host sync is ever needed;
 *  - return 0 on success, <0 for argument errors detected before launch (see codes),
 *    >0 = a `cudaError_t`.  No exceptions, no exit(), no CPU fallback: on a non-sm_100
 *    device every compute entry point returns SSVB_ERR_ARCH.
 */
#ifndef SSV_B200_H_
#define SSV_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSVB_VERSION 110 /* 110: multi-GPU stage entry points, next rows (EMA, DINO, PIRL) */

enum {
  SSVB_OK = 0,
  SSVB_ERR_INVALID = -1,     /* null pointer / non-positive size / bad flag */
  SSVB_ERR_ALIGNMENT = -2,   /* pointer or leading dimension not 16-byte aligned */
  SSVB_ERR_UNSUPPORTED = -3, /* shape outside what the sm_100a kernels cover (e.g. d > 256 for tensor-core losses) */
  SSVB_ERR_WORKSPACE = -4,   /* workspace / saved buffer too small */
  SSVB_ERR_ARCH = -5,        /* current device is not compute capability 10.x */
  SSVB_ERR_DRIVER = -6       /* cuTensorMapEncodeTiled unavailable / failed */
};

int ssvb_version(void);
const char* ssvb_strerror(int rc);
/* 0 if the current device can run the kernels (compute capability 10.x) */
int ssvb_device_check(void);

/* ---------------------------------------------------------------------------------------
 * a1  SimCLR NT-Xent — replaces SimclrLoss.forward (utils/losses.py:15-46; ctor :10-13;
 *     call site models/simclr.py:90) and the contrastive term of RelicLoss (:163-194).
 *     zi, zj: [n x d].  loss = mean over 2n rows of (LSE_{b != a} s_ab - s_{a,partner(a)}),
 *     s = Zhat Zhat^T / temperature.  The 2n x 2n similarity matrix is never written to HBM.
 *     d <= 256: zero-padded internally to 64 / 128 columns (d <= 128, the tuned path: whole rows per tile) or to 256
 *     (128 < d <= 256: four 64-wide k-blocks per tile, two-stage ring, backward in two 128-column halves).
 * ------------------------------------------------------------------------------------- */
size_t ssvb_ntxent_saved_bytes(int64_t n, int64_t d);
size_t ssvb_ntxent_workspace_bytes(int64_t n, int64_t d);
int ssvb_ntxent_fwd(const float* zi, const float* zj, int64_t n, int64_t d, int64_t ld_zi, int64_t ld_zj,
                    int normalize, float temperature, float* loss, void* saved, void* workspace,
                    size_t workspace_bytes, void* stream);
/* dzi/dzj: [n x d] gradients (overwritten).  grad_out: device scalar dL/dloss. */
int ssvb_ntxent_bwd(const float* zi, const float* zj, int64_t n, int64_t d, int64_t ld_zi, int64_t ld_zj,
                    int normalize, float temperature, const float* grad_out, const void* saved, float* dzi,
                    float* dzj, int64_t ld_dzi, int64_t ld_dzj, void* workspace, size_t workspace_bytes,
                    void* stream);

/* ---------------------------------------------------------------------------------------
 * a1/e  Global-batch NT-Xent, row-sharded over `world` ranks (SURVEY.md §8e; the reference has no
 *     multi-GPU path: semantics = SimclrLoss on the concatenation of all ranks' inputs, each rank
 *     receiving the gradient rows of its own inputs).  Every rank holds n_local rows per view.
 *     The gathered matrices are RANK-MAJOR: global row of (rank r, view v, row i) = r*2L + v*L + i
 *     (L = n_local), so each rank owns one contiguous slot and a single all-gather fills the rest;
 *     NT-Xent is invariant to this row permutation (the positive partner is a +- L, same rank).
 *     Stage 1 (prep):     normalise the local rows of both views into this rank's slot of `zhat_all`
 *                         (bf16 [mpad x dpad], mpad = ssvb_ntxent_mpad(world*L)) + local positives.
 *                         -> caller all-gathers the slots (2L*dpad bf16 per rank).
 *     Stage 2 (rows_fwd): local rows against ALL columns -> `stat_local` [2][2L]: the log2-domain LSE of
 *                         the local rows, then their per-row loss terms (lse - pos, natural log); also the
 *                         local loss sum.  ONE all-gather of stat_local into stat_all [world][2][2L] gives
 *                         every rank both the column statistics for backward and (summing the term halves,
 *                         divided by 2*world*L) the global loss - no separate all-reduce.
 *     Stage 3 (rows_bwd): complete gradient of the local rows; no reduce-scatter of gradients is
 *                         needed because W_ab = P_ab + P_ba is computable from s_ab, lse_a, lse_b.
 * ------------------------------------------------------------------------------------- */
int64_t ssvb_ntxent_dpad(int64_t d);                 /* padded feature dim of zhat_all */
int64_t ssvb_ntxent_mpad(int64_t n_global);          /* padded row count of zhat_all (n_global = world*L) */
size_t ssvb_ntxent_dist_workspace_bytes(int64_t world, int64_t n_local, int64_t d);
int ssvb_ntxent_dist_prep(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi,
                          int64_t ld_zj, int normalize, float temperature, int64_t world, int64_t rank,
                          void* zhat_all /* bf16 [mpad x dpad] */, float* inv_norm_local /* [2L] */,
                          float* pos_local /* [2L] */, void* stream);
int ssvb_ntxent_dist_rows_fwd(const void* zhat_all, int64_t world, int64_t rank, int64_t n_local, int64_t d,
                              int normalize, float temperature, const float* pos_local, float* stat_local,
                              float* loss_sum, void* workspace, size_t workspace_bytes, void* stream);
int ssvb_ntxent_dist_loss(const float* stat_all, int64_t world, int64_t n_local, float* loss, void* stream);

/* ---- NVLink peer-memory transport with generation flags (no NCCL, no host-issued barrier on the data path).
 * Multi-GPU form of SimclrLoss.forward (reference utils/losses.py:15-46 on the rank-order concatenation, SURVEY.md
 * §8e).  Every rank owns one SYMMETRIC arena of ssvb_ntxent_p2p_arena_bytes() bytes (zero-initialised once, then a
 * group barrier); `peer_arenas` is a DEVICE array of the `world` peer-mapped arena base pointers (index = rank,
 * including this rank's own), `arena_local` this rank's base, `multicast_arena` the NVSwitch multicast mapping of the
 * same allocation or NULL (then unicast peer stores are used).  `gen` = 1, 2, 3, ... is the forward's generation,
 * identical on every rank; buffers inside the arena are double-buffered by its parity.
 *   prep_push : normalise + stage this rank's rows into EVERY arena, then publish flag[rank] = gen everywhere
 *   wait_copy : wait for every rank's rows of `gen`, copy the gathered matrix into private memory `zhat_all`
 *   rows_fwd  : similarity rows of this rank -> [lse | term] stored into every arena as 8-byte {value, gen} pairs
 *   stat_loss : wait for every pair of generation `gen`, write the backward's column statistics `colstat` [mpad] and the
 *               global loss (fixed summation order: bit-identical on every rank)
 *   rows_bwd  : complete gradient of this rank's rows from zhat_all + colstat (no exchange) */
size_t ssvb_ntxent_p2p_arena_bytes(int64_t world, int64_t n_local, int64_t d);
int ssvb_ntxent_p2p_prep_push(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi,
                              int64_t ld_zj, int normalize, float temperature, int64_t world, int64_t rank,
                              void* arena_local, void* const* peer_arenas, void* multicast_arena, int64_t gen,
                              float* inv_norm_local, float* pos_local, void* stream);
int ssvb_ntxent_p2p_wait_copy(const void* arena_local, int64_t world, int64_t rank, int64_t n_local, int64_t d,
                              int64_t gen, void* zhat_all, void* stream);
int ssvb_ntxent_p2p_rows_fwd(const void* zhat_all, int64_t world, int64_t rank, int64_t n_local, int64_t d,
                             int normalize, float temperature, const float* pos_local, void* arena_local,
                             void* const* peer_arenas, int64_t gen, float* loss_sum, void* workspace,
                             size_t workspace_bytes, void* stream);
int ssvb_ntxent_p2p_stat_loss(void* arena_local, int64_t world, int64_t rank, int64_t n_local, int64_t d,
                              int normalize, float temperature, int64_t gen, float* colstat, float* loss,
                              void* workspace, size_t workspace_bytes, void* stream);
/* prep_push + wait_copy + rows_fwd + stat_loss in one call (same arguments, same order of launches). */
int ssvb_ntxent_p2p_forward(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi, int64_t ld_zj,
                            int normalize, float temperature, int64_t world, int64_t rank, void* arena_local,
                            void* const* peer_arenas, void* multicast_arena, int64_t gen, void* zhat_all,
                            float* inv_norm_local, float* pos_local, float* colstat, float* loss_sum, float* loss,
                            void* workspace, size_t workspace_bytes, void* stream);
int ssvb_ntxent_p2p_rows_bwd(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi,
                             int64_t ld_zj, int normalize, float temperature, int64_t world, int64_t rank,
                             const void* zhat_all, const float* colstat, const float* inv_norm_local,
                             const float* grad_out, float* dzi, float* dzj, int64_t ld_dzi, int64_t ld_dzj,
                             void* workspace, size_t workspace_bytes, void* stream);
int ssvb_ntxent_dist_rows_bwd(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi,
                              int64_t ld_zj, int normalize, float temperature, int64_t world, int64_t rank,
                              const void* zhat_all, const float* stat_all /* [world][2][2L] */,
                              const float* inv_norm_local, const float* grad_out, float* dzi, float* dzj,
                              int64_t ld_dzi, int64_t ld_dzj, void* workspace, size_t workspace_bytes,
                              void* stream);

/* ---------------------------------------------------------------------------------------
 * a2  MoCo InfoNCE — replaces MocoLoss.forward (utils/losses.py:56-72; call models/moco.py:117).
 *     query, keys: [n x d]; queue: [k x d] rows used AS STORED (no re-normalisation, no grad).
 *     queue_bf16 (optional, may be NULL): a bf16 shadow [k x dpad] (dpad = ssvb_ntxent_dpad(d),
 *     zero padded) maintained by ssvb_ring_enqueue; when NULL the fp32 queue is converted
 *     into the workspace on every call.
 * ------------------------------------------------------------------------------------- */
size_t ssvb_moco_saved_bytes(int64_t n, int64_t k, int64_t d);
size_t ssvb_moco_workspace_bytes(int64_t n, int64_t k, int64_t d);
/* queue_unit_norm != 0 asserts that every queue row is unit-norm or zero (a MemoryBank: rows are normalised on enqueue,
 * models/moco.py:31-36).  With normalize != 0 that bounds every logit by 1/tau and selects the fused single-pass form:
 * the forward reads the queue ONCE and also produces sum_j p_aj m_j (kept in `saved`), the backward is one row-wise
 * kernel that never touches the queue.  Pass 0 for arbitrary `memory_vectors` (two-pass online-max form). */
int ssvb_moco_fwd(const float* query, const float* keys, const float* queue, const void* queue_bf16,
                  int queue_unit_norm, int64_t n, int64_t k, int64_t d, int64_t ld_q, int64_t ld_k, int64_t ld_queue,
                  int normalize, float temperature, float* loss, void* saved, void* workspace, size_t workspace_bytes,
                  void* stream);
int ssvb_moco_bwd(const float* query, const float* keys, const float* queue, const void* queue_bf16,
                  int queue_unit_norm, int64_t n, int64_t k, int64_t d, int64_t ld_q, int64_t ld_k, int64_t ld_queue,
                  int normalize, float temperature, const float* grad_out, const void* saved, float* dquery,
                  float* dkeys, int64_t ld_dq, int64_t ld_dk, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * a2/e  MoCo with the queue SHARDED over `world` ranks (SURVEY.md §8e; semantics = MocoLoss on the rank-order
 *     concatenation of all ranks' queries / keys against the whole queue; every rank gets the gradients of its own
 *     rows).  Rank s owns k_local consecutive queue rows; every rank has n_local queries (n_global = world*n_local).
 *     1 prep:       normalise the local rows; bf16 queries into slot `rank` of qhat_all
 *                   [ssvb_moco_dist_npad(n_global) x ssvb_ntxent_dpad(d)]; rowstat_local [3][n_local] = 1/|q|, 1/|k|,
 *                   positive logit (unscaled).            -> caller ALL-GATHERS the qhat slots
 *     2 shard_fwd:  all n_global queries against this rank's shard -> part_local
 *                   [m (n_global) | l (n_global) | pos (n_local)] (log2-domain max / sum of exponentials over the shard)
 *                                                          -> caller ALL-GATHERS part_local into part_all [world][..]
 *     3 finalize:   combine the shards in rank order + the positive -> lse2_all [npad] and the global loss
 *                   (identical on every rank: no all-reduce)
 *     4 shard_bwd:  dacc_partial [npad x dpad] fp32 = sum_{j in shard} p_aj m_j for every global query
 *                                                          -> caller REDUCE-SCATTERS (sum) the first n_global rows
 *     5 finish:     gradients of the local query / key rows from the reduced dacc_local [n_local x dpad].
 * ------------------------------------------------------------------------------------- */
int64_t ssvb_moco_dist_npad(int64_t n_global);
size_t ssvb_moco_dist_workspace_bytes(int64_t n_global, int64_t k_local, int64_t d);
int ssvb_moco_dist_prep(const float* query, const float* keys, int64_t n_local, int64_t d, int64_t ld_q,
                        int64_t ld_k, int normalize, int64_t world, int64_t rank, void* qhat_all,
                        float* rowstat_local, void* stream);
int ssvb_moco_dist_shard_fwd(const void* qhat_all, int64_t n_global, const float* queue_shard,
                             const void* queue_shard_bf16, int64_t k_local, int64_t d, int64_t ld_queue,
                             float temperature, const float* rowstat_local, int64_t n_local, float* part_local,
                             void* workspace, size_t workspace_bytes, void* stream);
int ssvb_moco_dist_finalize(const float* part_all, int64_t world, int64_t n_local, float temperature,
                            float* lse2_all, float* loss, void* workspace, size_t workspace_bytes, void* stream);
int ssvb_moco_dist_shard_bwd(const void* qhat_all, int64_t n_global, const float* queue_shard,
                             const void* queue_shard_bf16, int64_t k_local, int64_t d, int64_t ld_queue,
                             float temperature, const float* lse2_all, float* dacc_partial, void* workspace,
                             size_t workspace_bytes, void* stream);
int ssvb_moco_dist_finish(const float* query, const float* keys, int64_t n_local, int64_t n_global, int64_t d,
                          int64_t ld_q, int64_t ld_k, int normalize, float temperature, const float* rowstat_local,
                          const float* lse2_local, const float* dacc_local, const float* grad_out, float* dquery,
                          float* dkeys, int64_t ld_dq, int64_t ld_dk, void* stream);

/* ---------------------------------------------------------------------------------------
 * a3/a7  Ring-buffer enqueue — replaces MemoryBank.add_batch (models/moco.py:31-36,
 *     normalize=1) and FeatureBank.add_vectors (models/swav.py:70-75, normalize=0).
 *     Row i of `batch` is written to bank row (ptr + i) mod size; when n > size only the
 *     last writer of each slot survives (same as the reference's sequential loop).
 *     bank_bf16 (optional): bf16 shadow [size x dpad] kept in sync.  The new pointer
 *     (ptr + n) mod size is returned through *new_ptr (HOST int64, bit-exact bookkeeping).
 * ------------------------------------------------------------------------------------- */
int ssvb_ring_enqueue(float* bank, void* bank_bf16, int64_t size, int64_t d, int64_t ld_bank,
                      const float* batch, int64_t n, int64_t ld_batch, int64_t ptr, int normalize,
                      int64_t* new_ptr, void* stream);

/* Sharded ring (MoCo queue range-partitioned over ranks, SURVEY.md §8e): `bank_shard` holds global rows
 * [shard_lo, shard_lo + shard_rows) of a ring of `size` rows; `batch` is the GLOBAL batch (every rank's keys in rank
 * order, all-gathered by the caller); only rows whose slot falls into this shard are written.  The pointer arithmetic
 * is the single-process ring's and identical on every rank (bit-exact bookkeeping). */
int ssvb_ring_enqueue_shard(float* bank_shard, void* bank_shard_bf16, int64_t size, int64_t shard_lo,
                            int64_t shard_rows, int64_t d, int64_t ld_bank, const float* batch, int64_t n,
                            int64_t ld_batch, int64_t ptr, int normalize, int64_t* new_ptr, void* stream);

/* ---------------------------------------------------------------------------------------
 * a4  Barlow Twins — replaces BarlowLoss.forward (utils/losses.py:127-142; call models/barlow.py:90).
 *     z_i, z_j: [n x d]; unbiased column standardisation, C = Xi^T Xj / n,
 *     loss = sum_a (C_aa-1)^2 + lambda * sum_{a!=b} C_ab^2.  d % 8 == 0, n % 8 == 0.
 * ------------------------------------------------------------------------------------- */
size_t ssvb_barlow_saved_bytes(int64_t n, int64_t d);
size_t ssvb_barlow_workspace_bytes(int64_t n, int64_t d);
int ssvb_barlow_fwd(const float* zi, const float* zj, int64_t n, int64_t d, int64_t ld_zi, int64_t ld_zj,
                    int normalize, float lambda, float* loss, void* saved, void* workspace,
                    size_t workspace_bytes, void* stream);
int ssvb_barlow_bwd(const float* zi, const float* zj, int64_t n, int64_t d, int64_t ld_zi, int64_t ld_zj,
                    int normalize, float lambda, const float* grad_out, const void* saved, float* dzi,
                    float* dzj, int64_t ld_dzi, int64_t ld_dzj, void* workspace, size_t workspace_bytes,
                    void* stream);

/* ---------------------------------------------------------------------------------------
 * a4/e  Distributed Barlow Twins (SURVEY.md §8e; the reference has no multi-GPU path: semantics =
 *     BarlowLoss on the rank-order concatenation of all ranks' rows, n_global = world * n_local, every
 *     rank receiving the gradient rows of its own inputs).  Batch rows are sharded; the exchange steps are
 *     the caller's collectives (NCCL through torch.distributed), the stages below are everything between:
 *     1 stats:     local column (mean, M2) of both views -> stats_local [2 views][2][d]
 *                  -> caller ALL-GATHERS into stats_all [world][2][2][d]
 *     2 xcorr:     Chan-combine in rank order -> global mean / unbiased std; standardise the local rows (bf16);
 *                  c_partial [d x d] fp32 = Xi~_r^T Xj~_r / n_global
 *                  -> caller REDUCE-SCATTERS (or all-reduces) c_partial: the cross-correlation all-reduce
 *     3 epilogue:  loss terms + dC (bf16) of a row slab [row0, row0+rows) of the summed matrix
 *                  -> caller ALL-GATHERS the dC slabs (the second half of the all-reduce, in bf16) and
 *                  all-reduces the scalar loss partials
 *     4 bwd_gemm:  dT_i = Xj~ dC^T / n_global, dT_j = Xi~ dC / n_global for the local rows (kept in `workspace`)
 *                  and their local column sums colsum_local [2 views][2][d] (sum dT, sum dT*x~)
 *                  -> caller ALL-REDUCES colsum (sum)
 *     5 bwd_finish: standardise (+ row-normalise) backward with the global reductions -> dzi, dzj.
 *     The same `workspace` buffer must be passed to bwd_gemm and bwd_finish without other use in between.
 * ------------------------------------------------------------------------------------- */
size_t ssvb_barlow_dist_saved_bytes(int64_t n_local, int64_t d);
size_t ssvb_barlow_dist_workspace_bytes(int64_t n_local, int64_t d);
int ssvb_barlow_dist_stats(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi,
                           int64_t ld_zj, int normalize, float* stats_local, void* saved, void* workspace,
                           size_t workspace_bytes, void* stream);
int ssvb_barlow_dist_xcorr(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi,
                           int64_t ld_zj, int normalize, const float* stats_all, int64_t world, float* c_partial,
                           void* saved, void* stream);
int ssvb_barlow_dist_epilogue(const float* c_rows, int64_t row0, int64_t rows, int64_t d, float lambda,
                              void* dC_rows /* bf16 [rows x d] */, float* loss_partial, void* workspace,
                              size_t workspace_bytes, void* stream);
int ssvb_barlow_dist_bwd_gemm(const float* zi, const float* zj, int64_t n_local, int64_t n_global, int64_t d,
                              int64_t ld_zi, int64_t ld_zj, int normalize, const void* dC /* bf16 [d x d] */,
                              const void* saved, float* colsum_local, void* workspace, size_t workspace_bytes,
                              void* stream);
int ssvb_barlow_dist_bwd_finish(const float* zi, const float* zj, int64_t n_local, int64_t n_global, int64_t d,
                                int64_t ld_zi, int64_t ld_zj, int normalize, const float* colsum_global,
                                const float* grad_out, const void* saved, float* dzi, float* dzj, int64_t ld_dzi,
                                int64_t ld_dzj, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * a5  Sinkhorn-Knopp codes — replaces SwavLoss.compute_codes_sinkhorn (utils/losses.py:213-224).
 *     scores: [b x k] -> codes [b x k] (rows sum to 1).  ld % 4 == 0 not required.
 * ------------------------------------------------------------------------------------- */
size_t ssvb_sinkhorn_workspace_bytes(int64_t b, int64_t k);
int ssvb_sinkhorn(const float* scores, int64_t b, int64_t k, int64_t ld_scores, float eps, int n_iters,
                  float* codes, int64_t ld_codes, void* workspace, size_t workspace_bytes, void* stream);

/* a4/e (alternative)  Column-sharded distributed Barlow — what SURVEY.md §8e asks to measure next to the all-reduce:
 *     the D x D matrix never crosses NVLink.  After the same stats exchange, every rank standardises its rows into its
 *     slot of two gathered bf16 matrices Xi~, Xj~ [n_global x d] (caller ALL-GATHERS them: 2 * n_global * d * 2 bytes),
 *     then owns the column slab [col0, col0+ncols) of BOTH C = Xi~^T Xj~ / n and C^T:
 *       cs_fwd(xa, xb):  slab of xa^T xb / n with the fused loss / dC epilogue -> dc_slab bf16 [d x ncols] and (optional)
 *                        the slab's loss terms; called as (Xi~, Xj~) [loss counted here] and (Xj~, Xi~) [C^T, no loss];
 *       cs_bwd(xa, xb, dc_slab): dT = xa dc_slab / n for ALL n_global rows, then the standardisation backward of the
 *                        slab's columns (their reductions over the batch are local now) -> dxb_slab fp32
 *                        [n_global x ncols], complete; called as (Xi~, Xj~, dC slab, view 1) and (Xj~, Xi~, dC^T slab, 0);
 *       caller ALL-TO-ALLs the row blocks of the slabs to their owners (n_local x ncols floats per pair);
 *       cs_finish: reassemble [world][n_local x ncols] into the local gradient rows (+ row-normalise backward).
 *     `saved` is the ssvb_barlow_dist_* blob of this rank (global mean / rstd, local row norms). */
int ssvb_barlow_dist_standardize(const float* zi, const float* zj, int64_t n_local, int64_t d, int64_t ld_zi,
                                 int64_t ld_zj, int normalize, const float* stats_all, int64_t world,
                                 void* xt_i_slot /* bf16 [n_local x d] */, void* xt_j_slot, void* saved, void* stream);
size_t ssvb_barlow_cs_workspace_bytes(int64_t n_global, int64_t d, int64_t ncols);
int ssvb_barlow_cs_fwd(const void* xa_all, const void* xb_all, int64_t n_global, int64_t d, int64_t col0,
                       int64_t ncols, float lambda, void* dc_slab, float* loss_partial, void* workspace,
                       size_t workspace_bytes, void* stream);
int ssvb_barlow_cs_bwd(const void* xa_all, const void* xb_all, const void* dc_slab, int64_t n_global, int64_t d,
                       int64_t col0, int64_t ncols, const void* saved, int64_t n_local, int view_b,
                       const float* grad_out, float* dxb_slab, void* workspace, size_t workspace_bytes, void* stream);
int ssvb_barlow_cs_finish(const float* recv /* [world][n_local x ncols] */, int64_t world, int64_t n_local,
                          int64_t ncols, const float* x, int64_t ld_x, int normalize, const void* saved, int view,
                          float* dx, int64_t ld_dx, void* stream);

/* a5/e  Distributed Sinkhorn (SURVEY.md §8e): the B sample rows are sharded (b_local per rank, b_global in total),
 *     prototypes / columns replicated.  The only cross-rank quantity is the K-vector of prototype marginals:
 *       pass(phase 0): u_local[0..k) = sum_b E_bk relative to this rank's maximum, u_local[k] = that maximum;
 *       pass(phase 1): u_local[0..k) = sum_b E_bk / (b_global v_b)  (needs the global alpha [k] and smax [1]);
 *       pass(phase 2): codes of the local rows.
 *     `codes` must be the SAME buffer in all three phases (its alignment selects the kernel family); it is written
 *     in phase 2 only.
 *     Between passes the caller ALL-GATHERS u_local (k+1 floats per rank) and calls ssvb_sinkhorn_dist_alpha, which
 *     combines the blocks in rank order (identical on every rank: the all-reduce of the marginals) into
 *     alpha_k = (1/K)/u_k and, after phase 0, the global maximum.  n_iters iterations = phase 0, (n_iters-1) x
 *     phase 1, phase 2 — the same schedule as ssvb_sinkhorn. */
int ssvb_sinkhorn_dist_pass(int phase, const float* scores, int64_t b_local, int64_t b_global, int64_t k,
                            int64_t ld_scores, float eps, const float* alpha, const float* smax, float* u_local,
                            float* codes, int64_t ld_codes, void* workspace, size_t workspace_bytes, void* stream);
int ssvb_sinkhorn_dist_alpha(const float* u_all /* world blocks of k+1 floats, rank_stride floats apart */,
                             int64_t world, int64_t rank_stride, int64_t k, int phase0, float eps, float* alpha,
                             float* smax, void* stream);

/* ---------------------------------------------------------------------------------------
 * a6  SwAV loss — replaces SwavLoss.forward (utils/losses.py:226-235; call models/swav.py:140).
 *     z1, z2: [nb x d] live rows; bank: [nbank x d] or NULL (appended under both views, no grad);
 *     prototypes: [k x d].
 * ------------------------------------------------------------------------------------- */
size_t ssvb_swav_saved_bytes(int64_t nb, int64_t nbank, int64_t k, int64_t d);
size_t ssvb_swav_workspace_bytes(int64_t nb, int64_t nbank, int64_t k, int64_t d);
int ssvb_swav_fwd(const float* z1, const float* z2, const float* bank, const float* prototypes, int64_t nb,
                  int64_t nbank, int64_t k, int64_t d, int64_t ld_z1, int64_t ld_z2, int64_t ld_bank,
                  int64_t ld_proto, float temperature, float eps, int n_iters, float* loss, void* saved,
                  void* workspace, size_t workspace_bytes, void* stream);
int ssvb_swav_bwd(const float* z1, const float* z2, const float* bank, const float* prototypes, int64_t nb,
                  int64_t nbank, int64_t k, int64_t d, int64_t ld_z1, int64_t ld_z2, int64_t ld_bank,
                  int64_t ld_proto, float temperature, const float* grad_out, const void* saved, float* dz1,
                  float* dz2, float* dproto, int64_t ld_dz1, int64_t ld_dz2, int64_t ld_dproto, void* workspace,
                  size_t workspace_bytes, void* stream);

/* a6/e  Distributed SwAV loss: every rank holds nb live rows (+ nbank bank rows) per view; B' is summed over ranks
 *     (bp_global).  scores (caller buffer, fp32 [2*(nb+nbank) x ssvb_swav_kpad(k)], view 1 rows then view 2 rows) ->
 *     caller runs the distributed Sinkhorn passes on each view's half -> codes (same layout) -> dist_ce writes this
 *     rank's share of the loss (sum of local row terms / bp_global; the caller all-reduces it) and the dscores used by
 *     ssvb_swav_bwd (unchanged; its dproto is this rank's partial: the caller all-reduces it). */
int64_t ssvb_swav_kpad(int64_t k);
int ssvb_swav_dist_scores(const float* z1, const float* z2, const float* bank, const float* prototypes, int64_t nb,
                          int64_t nbank, int64_t k, int64_t d, int64_t ld_z1, int64_t ld_z2, int64_t ld_bank,
                          int64_t ld_proto, float* scores, void* saved, void* stream);
int ssvb_swav_dist_ce(const float* scores, const float* codes, int64_t nb, int64_t nbank, int64_t bp_global,
                      int64_t k, int64_t d, float temperature, float* loss_local, void* saved, void* workspace,
                      size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * a8/a9  Row-dot regression losses.
 *     kind 0: BYOL nn.MSELoss() mean((o-t)^2)            (models/byol.py:89,129-130)
 *     kind 1: SimSiamLoss -mean_n sum_k o*t              (utils/losses.py:150-151; models/simsiam.py:126)
 *     o, t: [n x d].  d_o / d_t may be NULL (no gradient wanted for that operand).
 * ------------------------------------------------------------------------------------- */
size_t ssvb_rowdot_workspace_bytes(int64_t n, int64_t d);
int ssvb_rowdot_fwd(int kind, const float* o, const float* t, int64_t n, int64_t d, int64_t ld_o, int64_t ld_t,
                    float* loss, void* workspace, size_t workspace_bytes, void* stream);
int ssvb_rowdot_bwd(int kind, const float* o, const float* t, int64_t n, int64_t d, int64_t ld_o, int64_t ld_t,
                    const float* grad_out, float* d_o, float* d_t, int64_t ld_do, int64_t ld_dt, void* stream);

/* f1 (SURVEY.md §8f rank 1): the same two losses taken on the RAW projection-head outputs, with the head's final
 * F.normalize (models/byol.py:47,59; models/simsiam.py:48,69) fused into the loss: one pass forward (row norms + row
 * dot), one pass backward (normalise-backward projection from three saved scalars per row) instead of the reference's
 * normalise fwd / loss fwd / loss bwd / normalise bwd passes.  normalize_o / normalize_t select which operand is
 * normalised inside (the other is taken as given).  Value and gradients equal loss(F.normalize(o), F.normalize(t)). */
size_t ssvb_rowdot_norm_saved_bytes(int64_t n);
int ssvb_rowdot_norm_fwd(int kind, const float* o, const float* t, int64_t n, int64_t d, int64_t ld_o, int64_t ld_t,
                         int normalize_o, int normalize_t, float* loss, void* saved, void* workspace,
                         size_t workspace_bytes, void* stream);
int ssvb_rowdot_norm_bwd(int kind, const float* o, const float* t, int64_t n, int64_t d, int64_t ld_o, int64_t ld_t,
                         int normalize_o, int normalize_t, const float* grad_out, const void* saved, float* d_o,
                         float* d_t, int64_t ld_do, int64_t ld_dt, void* stream);

/* ---------------------------------------------------------------------------------------
 * a10  ReLIC KL term — the `alpha * kl_div_loss` part of RelicLoss.forward
 *     (utils/losses.py:196-201; call models/relic.py:129), reproducing the reference quirk:
 *     KL = sum_n exp(lq_n) * (lq_n - p_n), p = softmax_n(zi_n.zo_n/tau), lq = log_softmax_n(zj_n.zo_n/tau).
 *     `kl` receives alpha*KL.  The contrastive term is ssvb_ntxent_*.
 * ------------------------------------------------------------------------------------- */
size_t ssvb_relic_kl_saved_bytes(int64_t n);
size_t ssvb_relic_kl_workspace_bytes(int64_t n);
int ssvb_relic_kl_fwd(const float* zi, const float* zj, const float* zo, int64_t n, int64_t d, int64_t ld_zi,
                      int64_t ld_zj, int64_t ld_zo, int normalize, float temperature, float alpha, float* kl,
                      void* saved, void* workspace, size_t workspace_bytes, void* stream);
/* ACCUMULATES into dzi/dzj (so it composes with ssvb_ntxent_bwd) and overwrites dzo. */
int ssvb_relic_kl_bwd(const float* zi, const float* zj, const float* zo, int64_t n, int64_t d, int64_t ld_zi,
                      int64_t ld_zj, int64_t ld_zo, int normalize, float temperature, float alpha,
                      const float* grad_out, const void* saved, float* dzi, float* dzj, float* dzo,
                      int64_t ld_dzi, int64_t ld_dzj, int64_t ld_dzo, void* stream);
/* The whole RelicLoss.forward / backward (utils/losses.py:162-201) in one call each: ssvb_ntxent_fwd on (zi, zj) followed by
 * the KL term; `loss` = contrastive + alpha*KL.  saved_ntxent: ssvb_ntxent_saved_bytes(n, d); saved_kl:
 * ssvb_relic_kl_saved_bytes(n); workspace: ssvb_ntxent_workspace_bytes(n, d). */
int ssvb_relic_fwd(const float* zi, const float* zj, const float* zo, int64_t n, int64_t d, int64_t ld_zi, int64_t ld_zj,
                   int64_t ld_zo, int normalize, float temperature, float alpha, float* loss, void* saved_ntxent,
                   void* saved_kl, void* workspace, size_t workspace_bytes, void* stream);
int ssvb_relic_bwd(const float* zi, const float* zj, const float* zo, int64_t n, int64_t d, int64_t ld_zi, int64_t ld_zj,
                   int64_t ld_zo, int normalize, float temperature, float alpha, const float* grad_out,
                   const void* saved_ntxent, const void* saved_kl, float* dzi, float* dzj, float* dzo, int64_t ld_dzi,
                   int64_t ld_dzj, int64_t ld_dzo, void* workspace, size_t workspace_bytes, void* stream);

/* Multi-GPU ReLIC-KL (SURVEY.md §8e last row): the KL's softmaxes run over the batch axis (utils/losses.py:196-200),
 * so the per-row logits of all ranks are all-gathered between two stages.  dist_dots writes this rank's a_n, b_n into
 * `saved` and into ab_local [2][n_local]; the caller all-gathers ab_local into ab_all [world][2][n_local]; dist_reduce
 * derives the global softmax statistics (into `saved`) and alpha*KL (identical on every rank); ssvb_relic_kl_bwd then
 * yields the gradient rows of this rank's inputs.  The contrastive term is ssvb_ntxent_dist_* / ssvb_ntxent_p2p_*. */
int ssvb_relic_kl_dist_dots(const float* zi, const float* zj, const float* zo, int64_t n_local, int64_t d,
                            int64_t ld_zi, int64_t ld_zj, int64_t ld_zo, int normalize, float temperature,
                            void* saved, float* ab_local, void* stream);
int ssvb_relic_kl_dist_reduce(const float* ab_all, int64_t world, int64_t n_local, float alpha, void* saved, float* kl,
                              void* stream);

/* ---------------------------------------------------------------------------------------
 * Row L2-normalise (F.normalize(x, p=2, dim=-1), eps 1e-12) forward / backward —
 * Prototypes.forward (models/swav.py:51-54) and the projection-head epilogues.
 * ------------------------------------------------------------------------------------- */
int ssvb_l2norm_fwd(const float* x, int64_t n, int64_t d, int64_t ld_x, float* y, int64_t ld_y,
                    float* inv_norm /* [n] */, void* stream);
int ssvb_l2norm_bwd(const float* dy, const float* y, const float* inv_norm, int64_t n, int64_t d, int64_t ld_dy,
                    int64_t ld_y, float* dx, int64_t ld_dx, void* stream);

/* ---------------------------------------------------------------------------------------
 * (f) "next" rows of SURVEY.md §8, built to the same parity + measurement bar.
 *
 * EMA of the momentum (key / target / teacher) network — models/moco.py:108-111, byol.py:120-123,
 *     relic.py:119-122, dino.py:129-134:  t = m*t + (1-m)*s for every parameter, ONE launch for the whole network.
 *     chunk_table: DEVICE array of n_chunks entries {float* t; const float* s; int64 n} (24 bytes each), every tensor
 *     split by the caller into chunks of <= ssvb_ema_chunk_elems() elements (one CTA per chunk).  `m` and
 *     `one_minus_m` are passed separately so the caller's double-precision (1.0 - m) is rounded exactly as the
 *     reference's scalar is; products and sum are rounded separately (no FMA): bit-exact with the eager ops.
 * ------------------------------------------------------------------------------------- */
int64_t ssvb_ema_chunk_elems(void);
int ssvb_ema_update(const void* chunk_table, int64_t n_chunks, float m, float one_minus_m, void* stream);

/* ---------------------------------------------------------------------------------------
 * SeLA self-labelling (SURVEY.md §8f rank 4) - the per-batch body of SeLA.self_label_step
 * (reference models/sela.py:146-166): P = pow(log_softmax(logits, -1), lambda)^T [K x B];
 * num_iters x { alpha = 1 / (P beta); beta = 1 / (alpha^T P)^T }; labels_b = argmax_k alpha_k P_kb beta_b.
 * alpha [k] and beta [b] are the state carried from batch to batch (sela.py:72-73), updated in place.
 * logits: [b x k] fp32 row-major (leading dimension ld); labels: int64 [b]; one launch for the whole step.
 * ------------------------------------------------------------------------------------- */
size_t ssvb_sela_workspace_bytes(int64_t b, int64_t k);
int ssvb_sela_self_label(const float* logits, int64_t b, int64_t k, int64_t ld, float lambda, int64_t num_iters,
                         float* alpha, float* beta, int64_t* labels, void* workspace, size_t workspace_bytes,
                         void* stream);

/* ---------------------------------------------------------------------------------------
 * DinoLoss — replaces DinoLoss.forward (utils/losses.py:80-89; call site models/dino.py:161-162).
 *     teacher: [bs x 2 x k] contiguous, student: [bs x nv x k] contiguous, center: [k].
 *     loss = -(1/(bs nv)) sum_{b,v,k} (T_0 + T_1) log_softmax(student/temp_s),  T_g = softmax((teacher_g - center)/temp_t);
 *     gradient to the student only (the teacher runs under no_grad, models/dino.py:151-152).
 *     Envelope: 1 <= k <= 65536.  k <= 8192: one CTA per sample, or (large batches) one per (sample, view) row;
 *     8192 < k <= 65536: one thread-block cluster of ceil(k / 8192) CTAs per row, each CTA holding one 8192-column
 *     slice, the row statistics combined through distributed shared memory.  k > 65536: SSVB_ERR_UNSUPPORTED.
 *     The split and cluster forms use float4 accesses when k % 4 == 0 and every pointer is 16-byte aligned, scalar
 *     accesses otherwise.
 *     Workspace: [bs * nv] fp32 loss partials (padded to 256 bytes), then Tsum = T_0 + T_1 [bs x k] fp32.  The
 *     backward needs it whenever bs and nv select the split form or k > 8192; the forward always.
 *     ssvb_dino_center_update: models/dino.py:136-141 (first != 0: center = mean of the rows), any k.
 * ------------------------------------------------------------------------------------- */
size_t ssvb_dino_workspace_bytes(int64_t bs, int64_t nv, int64_t k);
int ssvb_dino_fwd(const float* teacher, const float* student, const float* center, int64_t bs, int64_t nv, int64_t k,
                  float temp_s, float temp_t, float* loss, void* workspace, size_t workspace_bytes, void* stream);
int ssvb_dino_bwd(const float* teacher, const float* student, const float* center, int64_t bs, int64_t nv, int64_t k,
                  float temp_s, float temp_t, const float* grad_out, float* dstudent, void* workspace,
                  size_t workspace_bytes, void* stream);
int ssvb_dino_center_update(const float* teacher_rows, int64_t rows, int64_t k, int64_t ld, float momentum,
                            float one_minus_m, int first, float* center, void* stream);

/* ---------------------------------------------------------------------------------------
 * PirlLoss — replaces PirlLoss.forward (utils/losses.py:100-117; call site models/pirl.py:134).
 *     img, patch, mem_pos: [n x d]; mem_neg: [k x d].  Two InfoNCE heads over the SAME negatives:
 *     logits_h = [mem_pos . v_h / tau | mem_pos mem_neg^T / tau], v_0 = patch, v_1 = img (L2-normalised when
 *     `normalize`; the memory rows are used as stored), loss = w CE_0 + (1 - w) CE_1 (label 0).
 *     `loss` receives w CE_0 + (1 - w) CE_1 (one deterministic reduction over both heads).  The memory rows carry no
 *     gradient (models/pirl.py:131-133 reads them from the bank), so backward is one row-wise kernel.  d <= 256.
 *     ssvb_bank_scatter / ssvb_bank_gather: the per-sample momentum bank of models/pirl.py:22-46
 *     (mode 0 initialize_vectors, mode 1 update_vectors; indices: DEVICE int64).
 * ------------------------------------------------------------------------------------- */
size_t ssvb_pirl_saved_bytes(int64_t n, int64_t d);
size_t ssvb_pirl_workspace_bytes(int64_t n, int64_t k, int64_t d);
int ssvb_pirl_fwd(const float* img, const float* patch, const float* mem_pos, const float* mem_neg, int64_t n,
                  int64_t k, int64_t d, int64_t ld_img, int64_t ld_patch, int64_t ld_pos, int64_t ld_neg,
                  int normalize, float temperature, float loss_weight, float* loss, void* saved, void* workspace,
                  size_t workspace_bytes, void* stream);
int ssvb_pirl_bwd(const float* img, const float* patch, const float* mem_pos, int64_t n, int64_t d, int64_t ld_img,
                  int64_t ld_patch, int64_t ld_pos, int normalize, float temperature, float loss_weight,
                  const float* grad_out, const void* saved, float* d_img, float* d_patch, int64_t ld_dimg,
                  int64_t ld_dpatch, void* stream);
int ssvb_bank_scatter(float* bank, int64_t size, int64_t d, int64_t ld_bank, const int64_t* indices, int64_t n,
                      const float* vectors, int64_t ld_vectors, float momentum, float one_minus_m, int mode,
                      void* stream);
int ssvb_bank_gather(const float* bank, int64_t size, int64_t d, int64_t ld_bank, const int64_t* indices, int64_t n,
                     float* out, int64_t ld_out, void* stream);

/* ---------------------------------------------------------------------------------------
 * Measurement hooks (bench.py only; OFF by default, not on the loss path).
 *   ssvb_launch_count: number of kernels this library has launched (reset != 0 zeroes it).
 *   ssvb_profile_enable(1): record a CUDA-event pair around every tensor-core kernel launch, on
 *   the stream it is launched on; ssvb_profile_summary(kind, &ms, &n) sums them
 *   (kind 0 = sim_fwd_kernel, 1 = sim_bwd_kernel, 2 = gemm kernels).
 * ------------------------------------------------------------------------------------- */
long long ssvb_launch_count(int reset);
int ssvb_profile_enable(int on);
int ssvb_profile_summary(int kind, double* total_ms, long long* count);

#ifdef __cplusplus
}
#endif
#endif /* SSV_B200_H_ */
