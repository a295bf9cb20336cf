// Flash-style similarity-matrix kernels for NT-Xent (SimCLR / ReLIC) and MoCo InfoNCE.
//
//   sim_fwd_kernel : S tile = A_I * B_J^T on tcgen05 (bf16 operands via TMA, fp32 accumulators in TMEM),
//                    streamed through exp2 / row-sum in registers -> per-(row, column-chunk) partial
//                    (max, sum) pairs.  S never touches HBM.
//   sim_bwd_kernel : recompute the S tile, turn it into the softmax weight tile W (bf16, written back to
//                    TMEM), second tcgen05 GEMM dA_I += W * B_J with W as the TMEM A-operand and the SAME
//                    smem B tile read MN-major.  Accumulator stays in TMEM for the whole row block.
//
// Warp roles (320 threads, 1 CTA / SM): warp 0 = TMA producer, warp 1 = MMA issuer, warps 2..9 = two
// softmax warpgroups (TMEM lane quarter = warp % 4).  All hand-offs are mbarriers; every wait is bounded.
#pragma once
#include "common.cuh"

namespace ssvb {

enum SimMode { SIM_NTX_FIXED = 0, SIM_NTX_ONLINE = 1, SIM_MOCO = 2 };

struct SimParams {
  // A rows: `nseg` segments of `seg_rows` rows starting at global rows seg_start[s] of the A tensor map.
  // Local row index (partials / dacc / MoCo rowstat) = seg * seg_rows + row-in-segment.
  int nseg, seg_rows, seg_start[2];
  int bps;         // 128-row blocks per segment
  int row_blocks;  // nseg * bps
  int cols;        // valid columns (rows of B)
  int col_tiles;   // ceil(cols / BN)
  int nchunks, tiles_per_chunk;
  float c;      // log2(e) / temperature
  float shift;  // FIXED mode: constant log2-domain shift (= c, the largest possible logit)
  // forward outputs: [4 * nchunks][part_stride] (one partial per softmax warpgroup and column chunk)
  float* part_m;
  float* part_l;
  int part_stride;
  // symmetric forward (sim_fwd_sym_kernel): band tiles per row block, column partials [(R - 1) / 2][part_stride]
  int band;
  float* colpart;
  // backward inputs / outputs
  const float* rowstat;  // NT-Xent: indexed by global row; MoCo: by local row
  const float* colstat;  // NT-Xent: fp32 column statistic (FIXED: 1/L', ONLINE: lse2), padded to a multiple of 128
  float* dacc;           // [local rows x ld_dacc] fp32
  int ld_dacc;
  int use_atomic;  // nchunks > 1: red.add into a zeroed dacc
  int opf16;  // similarity operands staged as fp16 (normalised rows) instead of bf16
  int dhalf;  // backward, dpad = 256 only: which 128-column half of dZ this launch produces
};

__device__ __forceinline__ uint8_t* align1024(uint8_t* p) {
  return reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(p) + 1023) & ~static_cast<uintptr_t>(1023));
}

// wait::ld with the destination registers as in/out operands so no consumer is scheduled above it
__device__ __forceinline__ void tmem_ld_wait_regs(uint32_t (&v)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                 "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]),
                 "+r"(v[15]), "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]),
                 "+r"(v[22]), "+r"(v[23]), "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]),
                 "+r"(v[29]), "+r"(v[30]), "+r"(v[31])::"memory");
}

struct UnitInfo {
  int g0;      // global A row of the block's first row
  int lrow0;   // local row index of the block's first row
  int nvalid;  // valid rows in the block
  int t0, t1;  // column-tile range of the chunk
  int ch;
};
__device__ __forceinline__ UnitInfo decode_unit(const SimParams& p, int u) {
  UnitInfo ui;
  const int rb = u / p.nchunks;
  ui.ch = u - rb * p.nchunks;
  const int seg = rb / p.bps;
  const int rbi = rb - seg * p.bps;
  ui.g0 = p.seg_start[seg] + rbi * 128;
  ui.lrow0 = seg * p.seg_rows + rbi * 128;
  ui.nvalid = min(128, p.seg_rows - rbi * 128);
  ui.t0 = ui.ch * p.tiles_per_chunk;
  ui.t1 = min(p.col_tiles, ui.t0 + p.tiles_per_chunk);
  return ui;
}

// FIXED mode hot loops: of every kPolyFwdPeriod (forward) / kPolyBwdPeriod (backward) consecutive PAIRS of
// exponentials, the first takes the packed polynomial exp2 and the rest two MUFU.EX2.  MUFU issues through the MIO
// queue at 16 / clk / SM and is co-critical with the tensor pipe in both kernels (ncu: mio_throttle on MUFU.EX2), so a
// share of the exponentials moves to the FMA pipe (shares measured in profiles/r2_tuning_log.md).
constexpr int kPolyFwdPeriod = 2;
constexpr int kPolyBwdPeriod = 3;

// exp2 of two values on the FMA pipe with packed instructions (Cody-Waite split + degree-3 minimax, max rel. error
// 7.5e-5): 6 FADD2/FFMA2 + 2 IMAD per pair = 4 issue slots per element and no MUFU slot.  Valid for x > -126.
__device__ __forceinline__ unsigned long long ex2_poly3_x2(unsigned long long x2) {
  const unsigned long long magic2 = pack_f32x2(12582912.f, 12582912.f);
  const unsigned long long nmagic2 = pack_f32x2(-12582912.f, -12582912.f);
  const unsigned long long r2 = add_f32x2(x2, magic2);      // low mantissa bits = round(x)
  const unsigned long long t2 = add_f32x2(r2, nmagic2);     // round(x) as a float (exact)
  const unsigned long long f2 = fma_f32x2(t2, pack_f32x2(-1.f, -1.f), x2);  // f in [-0.5, 0.5]
  unsigned long long q2 = fma_f32x2(f2, pack_f32x2(5.517166745e-2f, 5.517166745e-2f),
                                    pack_f32x2(2.426111221e-1f, 2.426111221e-1f));
  q2 = fma_f32x2(q2, f2, pack_f32x2(6.932609858e-1f, 6.932609858e-1f));
  q2 = fma_f32x2(q2, f2, pack_f32x2(9.999280736e-1f, 9.999280736e-1f));
  float q0, q1, r0, r1;
  unpack_f32x2(q2, q0, q1);
  unpack_f32x2(r2, r0, r1);
  const float e0 = __int_as_float(__float_as_int(q0) + (__float_as_int(r0) << 23));
  const float e1 = __int_as_float(__float_as_int(q1) + (__float_as_int(r1) << 23));
  return pack_f32x2(e0, e1);
}
// 16-byte shared-memory load from a 32-bit shared address (the generic-pointer form costs two address instructions
// per load plus a generic->shared window computation per call site)
__device__ __forceinline__ void lds_v4(uint32_t saddr, unsigned long long& lo, unsigned long long& hi) {
  asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(lo), "=l"(hi) : "r"(saddr));
}

// =====================================================================================================
// forward
// =====================================================================================================
// Forward tile width.  256: two 256-column S buffers, a warpgroup PAIR shares a tile (one 128-column half each) and the
// buffer is handed back after 3/4 of the pair's math.  128: FOUR 128-column S buffers, each softmax warpgroup owns a
// whole tile in its own buffer (more independent MMA -> softmax streams).  Measured (profiles/r2_tuning_log.md): 128 is
// 4 % slower (16 instead of 8 MMAs + commits per 256 columns on the one issuing thread).
constexpr int kFwdBN = 256;
template <int KB>
struct FwdCfg {
  // d <= 128 (KB <= 2): BN = kFwdBN.  128 < d <= 256 (KB = 4, dpad = 256): 128-column tiles (four S buffers) and a
  // 2-stage ring - a 64 KB A tile + 2 x 64 KB B tiles is what fits in 227 KB; functional coverage, not the tuned path.
  static constexpr int BN = (KB > 2) ? 128 : kFwdBN;
  static constexpr int NBUF = 512 / BN;  // S buffers in TMEM
  static constexpr int A_BYTES = 128 * 128 * KB;
  static constexpr int B_BYTES = BN * 128 * KB;
  static constexpr int NSTAGE = (KB > 2) ? 2 : ((KB == 1) ? 6 : 3) * (256 / BN);  // deep enough to cover the TMA latency
  static constexpr int NBARS = 4 + 2 * NSTAGE + 2 * NBUF;
  static constexpr int SMEM = 1024 + A_BYTES + NSTAGE * B_BYTES + NBARS * 8 + 16;
};

template <int MODE, bool MASKED>
__device__ __forceinline__ void fwd_tile(uint32_t taddr, const SimParams& p, int a_glob, int j0, float& m,
                                         float (&l)[4], uint32_t s_empty_bar, int lane) {
  uint32_t v[2][32];
  unsigned long long l2[2] = {pack_f32x2(0.f, 0.f), pack_f32x2(0.f, 0.f)};  // packed row-sum accumulators
  tmem_ld_x32(taddr, v[0]);
#pragma unroll
  for (int cc = 0; cc < 4; ++cc) {
    uint32_t(&cur)[32] = v[cc & 1];
    tmem_ld_wait_regs(cur);
    if (cc < 3) {
      tmem_ld_x32(taddr + (cc + 1) * 32, v[(cc + 1) & 1]);
    } else {
      // the S buffer is fully in registers: hand it back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_a(s_empty_bar);
    }
    const int colbase = j0 + cc * 32;
    if (MODE == SIM_NTX_FIXED && !MASKED) {
      // FIXED mode operands are pre-scaled by sqrt(log2(e)/tau) (pair_prep), so the accumulator IS the log2-domain
      // logit: no scale/shift FFMA.  Per pair: two MUFU.EX2 or one packed polynomial, one packed row-sum FADD2.
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        unsigned long long e2;
        if (i % kPolyFwdPeriod == 0) {
          e2 = ex2_poly3_x2(pack_f32x2(__uint_as_float(cur[2 * i]), __uint_as_float(cur[2 * i + 1])));
        } else {
          e2 = pack_f32x2(ex2f(__uint_as_float(cur[2 * i])), ex2f(__uint_as_float(cur[2 * i + 1])));
        }
        l2[i & 1] = add_f32x2(l2[i & 1], e2);
      }
    } else if (MODE == SIM_NTX_FIXED) {
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        float t = fmaf(__uint_as_float(cur[i]), p.c, -p.shift);
        if (MASKED) {
          const int col = colbase + i;
          if (col == a_glob || col >= p.cols) t = -INFINITY;
        }
        l[i & 3] += ex2f(t);
      }
    } else {
      float x[32];
      float cm = -INFINITY;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        float t = __uint_as_float(cur[i]) * p.c;
        if (MASKED) {
          const int col = colbase + i;
          if ((MODE != SIM_MOCO && col == a_glob) || col >= p.cols) t = -INFINITY;
        }
        x[i] = t;
        cm = fmaxf(cm, t);
      }
      const float mn = fmaxf(m, cm);
      const float sc = ex2f(m - mn);
      m = mn;
#pragma unroll
      for (int i = 0; i < 4; ++i) l[i] *= sc;
#pragma unroll
      for (int i = 0; i < 32; ++i) l[i & 3] += ex2f(x[i] - mn);
    }
  }
  if (MODE == SIM_NTX_FIXED && !MASKED) {
    float a0, a1, b0, b1;
    unpack_f32x2(l2[0], a0, a1);
    unpack_f32x2(l2[1], b0, b1);
    l[0] += a0; l[1] += a1; l[2] += b0; l[3] += b1;
  }
}


// 640 threads: warpgroup 0 = {TMA producer, MMA issuer, 2 idle warps} shrinks to 40 registers/thread; warps 4..19 are
// FOUR softmax warpgroups (TMEM lane quarter = warp % 4): tile t belongs to the warpgroup pair (t & 1) (= its S
// buffer), and within the pair each warpgroup streams one 128-column half.  Four math warps per scheduler keep the
// MUFU and FMA pipes (polynomial exp2) busy at the same time.
template <int KB, int MODE, bool OPF16 = false>
__global__ void __launch_bounds__(640, 1)
sim_fwd_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const SimParams p) {
  using C = FwdCfg<KB>;
  constexpr int BN = C::BN, NSTAGE = C::NSTAGE, NBUF = C::NBUF;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align1024(smem_raw);
  uint8_t* sA = smem;
  uint8_t* sB = smem + C::A_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + NSTAGE * C::B_BYTES);
  uint64_t* a_full = bars;
  uint64_t* a_empty = bars + 2;
  uint64_t* b_full = bars + 4;
  uint64_t* b_empty = b_full + NSTAGE;
  uint64_t* s_full = b_empty + NSTAGE;
  uint64_t* s_empty = s_full + NBUF;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_empty + NBUF);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&a_full[i], 1);
      mbar_init(&a_empty[i], 1);
    }
    for (int i = 0; i < NBUF; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&s_empty[i], 16 / NBUF);  // the warps that drain one S buffer: a warpgroup pair (8) or one warpgroup (4)
    }
    for (int i = 0; i < NSTAGE; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int nunits = p.row_blocks * p.nchunks;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
  // Producer / issuer loops are executed by the WHOLE warp (warp-uniform control flow and operands, so the TMA /
  // UMMA operands stay in uniform registers); only the issue instructions sit behind elect_one().
  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    int ucount = 0, gt = 0;
    for (int u = blockIdx.x; u < nunits; u += gridDim.x, ++ucount) {
      const UnitInfo ui = decode_unit(p, u);
      mbar_wait(&a_empty[0], (ucount & 1) ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&a_full[0], C::A_BYTES);
#pragma unroll
        for (int kb = 0; kb < KB; ++kb) tma_load_2d(sA + kb * (128 * 128), &tmA, &a_full[0], kb * 64, ui.g0);
      }
      __syncwarp();
      for (int t = ui.t0; t < ui.t1; ++t, ++gt) {
        const int st = gt % NSTAGE;
        mbar_wait(&b_empty[st], ((gt / NSTAGE) & 1) ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&b_full[st], C::B_BYTES);
#pragma unroll
          for (int kb = 0; kb < KB; ++kb)
            tma_load_2d(sB + st * C::B_BYTES + kb * (BN * 128), &tmB, &b_full[st], kb * 64, t * BN);
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t IDESC = make_idesc(128, BN, 0, 0, OPF16 ? 0 : 1);
    const uint32_t abase = smem_u32(sA);
    int ucount = 0, gt = 0;
    for (int u = blockIdx.x; u < nunits; u += gridDim.x, ++ucount) {
      const UnitInfo ui = decode_unit(p, u);
      mbar_wait(&a_full[0], ucount & 1);
      for (int t = ui.t0; t < ui.t1; ++t, ++gt) {
        const int st = gt % NSTAGE, buf = gt % NBUF;
        mbar_wait(&b_full[st], (gt / NSTAGE) & 1);
        mbar_wait(&s_empty[buf], ((gt / NBUF) & 1) ^ 1);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t bbase = smem_u32(sB + st * C::B_BYTES);
#pragma unroll
          for (int kb = 0; kb < KB; ++kb)
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4)
              umma_ss(tmem + buf * BN, desc_kmajor(abase + kb * (128 * 128) + k4 * 32),
                      desc_kmajor(bbase + kb * (BN * 128) + k4 * 32), IDESC, (kb | k4) != 0);
          umma_commit(&b_empty[st]);
          umma_commit(&s_full[buf]);
          if (t == ui.t1 - 1) umma_commit(&a_empty[0]);
        }
        __syncwarp();
      }
    }
  }
  } else {
    // ------------------------------------------------------------------ softmax warpgroups
    asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
    const int wgi = (warp - 4) >> 2;  // 0..3
    const int pair = wgi >> 1, half = wgi & 1;
    const int q = warp & 3;
    const int row_l = q * 32 + lane;
    const uint32_t tlane = static_cast<uint32_t>(q * 32) << 16;
    int gt = 0;
    const int my_buf = NBUF == 2 ? pair : wgi;
    const uint32_t a_s_full = smem_u32(&s_full[my_buf]), a_s_empty = smem_u32(&s_empty[my_buf]);  // hoisted (see bwd)
    for (int u = blockIdx.x; u < nunits; u += gridDim.x) {
      const UnitInfo ui = decode_unit(p, u);
      const int a_glob = ui.g0 + row_l;
      float m = -1e30f;
      float l[4] = {0.f, 0.f, 0.f, 0.f};
      for (int t = ui.t0; t < ui.t1; ++t, ++gt) {
        // BN = 256: tile t belongs to the warpgroup pair (t & 1), each warpgroup of the pair streams one 128-column half;
        // BN = 128: tile t belongs to warpgroup (t & 3) alone (its own S buffer)
        if (NBUF == 2 ? ((gt & 1) != pair) : ((gt & 3) != wgi)) continue;
        const int buf = NBUF == 2 ? pair : wgi;
        mbar_wait_a(a_s_full, (gt / NBUF) & 1);
        tc_fence_after();
        const int j0 = t * BN + (NBUF == 2 ? half * 128 : 0);
        const bool special = (MODE != SIM_MOCO && j0 < ui.g0 + 128 && j0 + 128 > ui.g0) || (j0 + 128 > p.cols);
        const uint32_t taddr = tmem + tlane + buf * BN + (NBUF == 2 ? half * 128 : 0);
        if (special)
          fwd_tile<MODE, true>(taddr, p, a_glob, j0, m, l, a_s_empty, lane);
        else
          fwd_tile<MODE, false>(taddr, p, a_glob, j0, m, l, a_s_empty, lane);
      }
      if (row_l < ui.nvalid) {
        const size_t o = static_cast<size_t>(ui.ch * 4 + wgi) * p.part_stride + ui.lrow0 + row_l;
        p.part_l[o] = (l[0] + l[1]) + (l[2] + l[3]);
        if (MODE != SIM_NTX_FIXED) p.part_m[o] = m;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem);
}

// =====================================================================================================
// symmetric forward (single GPU, FIXED mode, dpad <= 128): S = Z Z^T, so each 128 x 128 tile is computed once
// =====================================================================================================
// Row block i (R = row_blocks) takes the cyclic band of column blocks b = (i + o) mod R, o = 0 .. floor(R/2)
// (p.band = floor(R/2) + 1 tiles):
//   o = 0          diagonal tile: row sums only, diagonal element masked;
//   1 <= o < R/2   full tile: row sums -> block i, column sums -> block b (p.colpart[o - 1][b * 128 + col]);
//   o = R/2        (R even) antipodal tile, reached from both partners: each takes row sums only.
// So exp2(t_ab) enters L_a exactly once for every pair of valid rows a != b.  A 256-column stage holds the tiles
// o = 2t and 2t + 1 (two 128-row TMA boxes, block coordinates taken mod R); when the band length is odd the second half
// of the last stage is loaded and multiplied but not read.  Staged rows >= M are zero (logit 0, exp2 = 1): they are
// masked out of both sums.
//
// Column sums: the softmax warps read S with tcgen05.ld.16x256b (the mma accumulator fragment: thread 4g + c holds
// rows g, g + 8 (+16, +24 from the second load) and columns 8k + 2c, 8k + 2c + 1), so one thread covers 4 rows and the
// rows of a column are spread over 8 lanes instead of 32.  Per pair of exponentials: one packed add into the row
// accumulator and one into the column accumulator.  Each warp stores its per-lane column partials (8 floats per 32
// columns) to shared memory; after a warpgroup barrier two warps sum the 32 partials of each column in a fixed order
// and write one 128-float partial per tile (deterministic: no float atomics).
template <int KB>
struct SymCfg {
  static constexpr int BN = 256;
  static constexpr int A_BYTES = 128 * 128 * KB;
  static constexpr int B_BYTES = BN * 128 * KB;
  // d = 128: a 2-stage ring is what leaves room for the 64 KB of column-partial buffers in 227 KB
  static constexpr int NSTAGE = (KB == 1) ? 4 : 2;
  static constexpr int CP_BYTES = 4 * 16384;  // per softmax warpgroup: [chunk 4][warp 4][g 8][32 floats]
  static constexpr int NBARS = 4 + 2 * NSTAGE + 4;
  static constexpr int SMEM = 1024 + A_BYTES + NSTAGE * B_BYTES + CP_BYTES + NBARS * 8 + 16;
};

// TMEM -> registers, 16 lanes x 8 columns x 4 repetitions (see the layout note above)
__device__ __forceinline__ void tmem_ld_16x256b_x4(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// one 128 x 128 tile (this warp: 32 rows).  COLS: also store the column partials of each 32-column chunk to `cp`
// (this warp's slot of the warpgroup buffer).  MASKED: diag = diagonal tile; rows / columns >= p.cols are padding.
template <bool MASKED, bool COLS>
__device__ __forceinline__ void sym_tile(uint32_t taddr, const SimParams& p, unsigned long long (&racc)[4],
                                         uint32_t a_s_empty, int lane, uint32_t cp_st0, uint32_t cp_st1, int barid,
                                         int row_w, int col_t, bool diag) {
  uint32_t v[2][32];
  tmem_ld_16x256b_x4(taddr, v[0]);
  tmem_ld_16x256b_x4(taddr + (16u << 16), v[0] + 16);
  const int g = lane >> 2, c4 = lane & 3;
#pragma unroll
  for (int cc = 0; cc < 4; ++cc) {
    uint32_t(&cur)[32] = v[cc & 1];
    tmem_ld_wait_regs(cur);
    if (cc < 3) {
      tmem_ld_16x256b_x4(taddr + (cc + 1) * 32, v[(cc + 1) & 1]);
      tmem_ld_16x256b_x4(taddr + (16u << 16) + (cc + 1) * 32, v[(cc + 1) & 1] + 16);
    } else {
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_a(a_s_empty);
    }
    unsigned long long cacc[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
      for (int r = 0; r < 4; ++r) {  // row slot r: row g + 8 r of this warp's 32
        const int idx = 16 * (r >> 1) + 4 * k + 2 * (r & 1);
        unsigned long long e2;
        if (MASKED) {
          const int row = row_w + g + 8 * r, col = col_t + cc * 32 + 8 * k + 2 * c4;
          float e[2];
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const bool off = (diag && row == col + j) || row >= p.cols || col + j >= p.cols;
            e[j] = ex2f(off ? -INFINITY : __uint_as_float(cur[idx + j]));
          }
          e2 = pack_f32x2(e[0], e[1]);
        } else if ((4 * k + r) % kPolyFwdPeriod == 0) {
          e2 = ex2_poly3_x2(pack_f32x2(__uint_as_float(cur[idx]), __uint_as_float(cur[idx + 1])));
        } else {
          e2 = pack_f32x2(ex2f(__uint_as_float(cur[idx])), ex2f(__uint_as_float(cur[idx + 1])));
        }
        racc[r] = add_f32x2(racc[r], e2);
        if (COLS) cacc[k] = r == 0 ? e2 : add_f32x2(cacc[k], e2);
      }
    }
    if (COLS) {
      // the two readers of the previous tile's partials are done before the first store of this tile
      if (cc == 0) named_bar_sync(barid, 128);
      const uint32_t o = cc * 4096;
      asm volatile("st.shared.v2.b64 [%0], {%1, %2};" ::"r"(cp_st0 + o), "l"(cacc[0]), "l"(cacc[1]) : "memory");
      asm volatile("st.shared.v2.b64 [%0], {%1, %2};" ::"r"(cp_st1 + o), "l"(cacc[2]), "l"(cacc[3]) : "memory");
    }
  }
}

template <int KB, bool OPF16>
__global__ void __launch_bounds__(640, 1)
sim_fwd_sym_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const SimParams p) {
  using C = SymCfg<KB>;
  constexpr int BN = C::BN, NSTAGE = C::NSTAGE, NBUF = 2;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align1024(smem_raw);
  uint8_t* sA = smem;
  uint8_t* sB = smem + C::A_BYTES;
  uint8_t* sCP = sB + NSTAGE * C::B_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sCP + C::CP_BYTES);
  uint64_t* a_full = bars;
  uint64_t* a_empty = bars + 2;
  uint64_t* b_full = bars + 4;
  uint64_t* b_empty = b_full + NSTAGE;
  uint64_t* s_full = b_empty + NSTAGE;
  uint64_t* s_empty = s_full + NBUF;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_empty + NBUF);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int R = p.row_blocks;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(&a_full[0], 1);
    mbar_init(&a_empty[0], 1);
    for (int i = 0; i < NBUF; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&s_empty[i], 8);  // the warpgroup pair that drains the buffer
    }
    for (int i = 0; i < NSTAGE; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int nunits = p.row_blocks * p.nchunks;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == 0) {
      // ---------------------------------------------------------------- TMA producer
      int ucount = 0, gt = 0;
      for (int u = blockIdx.x; u < nunits; u += gridDim.x, ++ucount) {
        const UnitInfo ui = decode_unit(p, u);
        const int rb = ui.g0 >> 7;
        mbar_wait(&a_empty[0], (ucount & 1) ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&a_full[0], C::A_BYTES);
#pragma unroll
          for (int kb = 0; kb < KB; ++kb) tma_load_2d(sA + kb * (128 * 128), &tmA, &a_full[0], kb * 64, ui.g0);
        }
        __syncwarp();
        for (int t = ui.t0; t < ui.t1; ++t, ++gt) {
          const int st = gt % NSTAGE;
          mbar_wait(&b_empty[st], ((gt / NSTAGE) & 1) ^ 1);
          if (elect_one()) {
            mbar_expect_tx(&b_full[st], C::B_BYTES);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int b = (rb + 2 * t + h) % R;
#pragma unroll
              for (int kb = 0; kb < KB; ++kb)
                tma_load_2d(sB + st * C::B_BYTES + kb * (BN * 128) + h * (128 * 128), &tmB, &b_full[st], kb * 64,
                            b * 128);
            }
          }
          __syncwarp();
        }
      }
    } else if (warp == 1) {
      // ---------------------------------------------------------------- MMA issuer
      constexpr uint32_t IDESC = make_idesc(128, BN, 0, 0, OPF16 ? 0 : 1);
      const uint32_t abase = smem_u32(sA);
      int ucount = 0, gt = 0;
      for (int u = blockIdx.x; u < nunits; u += gridDim.x, ++ucount) {
        const UnitInfo ui = decode_unit(p, u);
        mbar_wait(&a_full[0], ucount & 1);
        for (int t = ui.t0; t < ui.t1; ++t, ++gt) {
          const int st = gt % NSTAGE, buf = gt % NBUF;
          mbar_wait(&b_full[st], (gt / NSTAGE) & 1);
          mbar_wait(&s_empty[buf], ((gt / NBUF) & 1) ^ 1);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t bbase = smem_u32(sB + st * C::B_BYTES);
#pragma unroll
            for (int kb = 0; kb < KB; ++kb)
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4)
                umma_ss(tmem + buf * BN, desc_kmajor(abase + kb * (128 * 128) + k4 * 32),
                        desc_kmajor(bbase + kb * (BN * 128) + k4 * 32), IDESC, (kb | k4) != 0);
            umma_commit(&b_empty[st]);
            umma_commit(&s_full[buf]);
            if (t == ui.t1 - 1) umma_commit(&a_empty[0]);
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ softmax warpgroups
    asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
    const int wgi = (warp - 4) >> 2;  // 0..3
    const int pair = wgi >> 1, half = wgi & 1;
    const int q = warp & 3;
    const int g = lane >> 2, c4 = lane & 3;
    const uint32_t tlane = static_cast<uint32_t>(q * 32) << 16;
    const uint32_t a_s_full = smem_u32(&s_full[pair]), a_s_empty = smem_u32(&s_empty[pair]);
    const int barid = 1 + wgi;
    // column partial buffer of this warpgroup: [chunk][warp q][g][c4 * 8 + k * 2 + j]; the two 16-byte halves of a
    // thread's 32 bytes are swapped for odd g (conflict-free stores), the readers undo it
    const uint32_t cp_wg = smem_u32(sCP) + wgi * 16384;
    const uint32_t cp_st = cp_wg + (q * 8 + g) * 128 + c4 * 32;
    const uint32_t cp_st0 = cp_st + ((g & 1) << 4), cp_st1 = cp_st + (((g & 1) ^ 1) << 4);
    const int H = (R - 1) >> 1;  // full tiles per row block
    const bool ragged = (p.cols & 127) != 0;
    int gt = 0;
    for (int u = blockIdx.x; u < nunits; u += gridDim.x) {
      const UnitInfo ui = decode_unit(p, u);
      const int rb = ui.g0 >> 7;
      unsigned long long racc[4] = {0ull, 0ull, 0ull, 0ull};
      for (int t = ui.t0; t < ui.t1; ++t, ++gt) {
        if ((gt & 1) != pair) continue;
        mbar_wait_a(a_s_full, (gt >> 1) & 1);
        tc_fence_after();
        const int o = 2 * t + half;
        const uint32_t taddr = tmem + tlane + pair * BN + half * 128;
        if (o >= p.band) {  // odd band: the second half of the last stage is not part of it
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_a(a_s_empty);
          continue;
        }
        const int b = (rb + o) % R;
        const bool cols = o >= 1 && o <= H;
        const bool masked = o == 0 || (ragged && (rb == R - 1 || b == R - 1));
        const int row_w = ui.g0 + q * 32;  // global rows / columns: padding test against p.cols
        if (!cols) {
          sym_tile<true, false>(taddr, p, racc, a_s_empty, lane, 0, 0, barid, row_w, b * 128, o == 0);
          continue;
        }
        if (masked)
          sym_tile<true, true>(taddr, p, racc, a_s_empty, lane, cp_st0, cp_st1, barid, row_w, b * 128, false);
        else
          sym_tile<false, true>(taddr, p, racc, a_s_empty, lane, cp_st0, cp_st1, barid, row_w, b * 128, false);
        named_bar_sync(barid, 128);
        if (q < 2) {
          // readers: column pair rd = q * 32 + lane of the tile (chunk rd >> 4, k = (rd >> 2) & 3, c4 = rd & 3), its
          // 32 partials (4 warps x 8 lane groups) summed in a fixed order
          const int rd = q * 32 + lane;
          const int rd_k = (rd >> 2) & 3;
          const uint32_t cp_rd = cp_wg + (rd >> 4) * 4096 + (rd & 3) * 32;
          const int rd_col = (rd >> 4) * 32 + 8 * rd_k + 2 * (rd & 3);
          unsigned long long s2 = pack_f32x2(0.f, 0.f);
#pragma unroll
          for (int w = 0; w < 4; ++w)
#pragma unroll
            for (int gg = 0; gg < 8; ++gg) {
              unsigned long long x;
              asm volatile("ld.shared.b64 %0, [%1];"
                           : "=l"(x)
                           : "r"(cp_rd + (w * 8 + gg) * 128 + ((rd_k * 8) ^ ((gg & 1) << 4))));
              s2 = add_f32x2(s2, x);
            }
          float c0, c1;
          unpack_f32x2(s2, c0, c1);
          *reinterpret_cast<float2*>(p.colpart + static_cast<size_t>(o - 1) * p.part_stride + b * 128 + rd_col) =
              make_float2(c0, c1);
        }
      }
      // row sums: the packed halves, then the 4 lanes of a row group (butterfly: identical bits in all four)
      float rs[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        float x0, x1;
        unpack_f32x2(racc[r], x0, x1);
        rs[r] = x0 + x1;
        rs[r] += __shfl_xor_sync(0xffffffffu, rs[r], 1);
        rs[r] += __shfl_xor_sync(0xffffffffu, rs[r], 2);
      }
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int row_l = q * 32 + g + 8 * r;
        if (c4 == r && row_l < ui.nvalid)
          p.part_l[static_cast<size_t>(ui.ch * 4 + wgi) * p.part_stride + ui.lrow0 + row_l] = rs[r];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem);
}

// =====================================================================================================
// backward
// =====================================================================================================
// TMEM plan (512 columns): S0 @0, S1 @128 (fp32 similarity tiles), dZ @256 (DP-column gradient accumulator),
// W0 @384, W1 @448 (bf16 weight tiles, the TMEM A-operand of the second GEMM).
// Decoupling: a weight warpgroup pulls its WHOLE S tile into registers first and hands the S buffer straight back,
// and the MMA thread never blocks on a single barrier — it polls "next S issuable" and "next dZ issuable" and issues
// whichever is ready — so the similarity GEMM of tile t+2 runs while W(t) is still being computed and the
// W -> dZ latency is off the critical path of the exp warps.
template <int KB>
struct BwdCfg {
  static constexpr int BN = 128;
  // output columns of one launch: the whole row for d <= 128; for KB = 4 (dpad = 256) the dZ accumulator holds ONE
  // 128-column half (TMEM: S0 S1 dZ W0 W1 = 512 columns) and the host launches the kernel once per half (p.dhalf) -
  // S and the weights are recomputed, the second GEMM reads k-blocks {2 dhalf, 2 dhalf + 1} of the same B tile
  static constexpr int DP = (KB >= 2) ? 128 : 64;
  static constexpr int A_BYTES = 128 * 128 * KB;
  static constexpr int B_BYTES = BN * 128 * KB;
  static constexpr int CS_BYTES = BN * 4;  // per-stage column statistics (fp32)
  static constexpr int NSTAGE = (KB == 1) ? 8 : (KB == 2 ? 5 : 2);
  static constexpr int NBARS = 2 + 2 * NSTAGE + 8 + 2;
  static constexpr int SMEM = 1024 + A_BYTES + NSTAGE * (B_BYTES + CS_BYTES) + NBARS * 8 + 16;
  static constexpr int T_S = 0;
  static constexpr int T_DZ = 256;
  static constexpr int T_W = 384;
};

// weights of 32 consecutive columns [cb, cb+32) of one row: sv = S values, pk = packed bf16 pairs out
template <int MODE, bool MASKED, bool OPF16>
__device__ __forceinline__ void bwd_weights32(const uint32_t (&sv)[32], uint32_t (&pk)[16], const SimParams& p,
                                              int a_glob, int colbase, float rs, uint32_t cs32, float& wsum) {
  if (MODE == SIM_NTX_FIXED && !MASKED) {
    // issue-bound loop.  Operands are pre-scaled (the S accumulator is the log2-domain logit): per pair two MUFU.EX2
    // (or one packed polynomial), FADD2 (row + column factor), FMUL2, one pack -> 2.5 issue slots per element.
    // Column factors: fp32 pairs straight from shared memory (LDS.128 = 2 pairs, 32-bit shared address).
    const unsigned long long rs2 = pack_f32x2(rs, rs);
#pragma unroll
    for (int i2 = 0; i2 < 8; ++i2) {
      unsigned long long cu[2];  // column factors of 4 consecutive columns
      lds_v4(cs32 + i2 * 16, cu[0], cu[1]);
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int i = i2 * 2 + e;  // pair index: columns 2i, 2i+1
        unsigned long long e2;
        if (i % kPolyBwdPeriod == 0) {
          e2 = ex2_poly3_x2(pack_f32x2(__uint_as_float(sv[2 * i]), __uint_as_float(sv[2 * i + 1])));
        } else {
          e2 = pack_f32x2(ex2f(__uint_as_float(sv[2 * i])), ex2f(__uint_as_float(sv[2 * i + 1])));
        }
        const unsigned long long w2 = mul_f32x2(e2, add_f32x2(rs2, cu[e]));
        float w0, w1;
        unpack_f32x2(w2, w0, w1);
        pk[i] = pack_h2<OPF16>(w0, w1);
      }
    }
    return;
  }
#pragma unroll
  for (int i4 = 0; i4 < 8; ++i4) {
    float csv[4] = {0.f, 0.f, 0.f, 0.f};
    if (MODE != SIM_MOCO) {
      unsigned long long c01, c23;
      lds_v4(cs32 + i4 * 16, c01, c23);
      unpack_f32x2(c01, csv[0], csv[1]);
      unpack_f32x2(c23, csv[2], csv[3]);
    }
    float w[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int i = i4 * 4 + e;
      const float s = __uint_as_float(sv[i]);
      float wv;
      if (MODE == SIM_NTX_FIXED) {
        const float x = fmaf(s, p.c, -p.shift);
        wv = ex2f(x) * (rs + csv[e]);
      } else if (MODE == SIM_NTX_ONLINE) {
        const float t = s * p.c;
        wv = ex2f(t - rs) + ex2f(t - csv[e]);
      } else {
        wv = ex2f(fmaf(s, p.c, -rs));
      }
      if (MASKED && MODE != SIM_MOCO && (colbase + i == a_glob)) wv = 0.f;
      if (MASKED && MODE == SIM_MOCO && (colbase + i >= p.cols)) wv = 0.f;  // queue tail (zero-filled B rows)
      if (MODE == SIM_MOCO) wsum += wv;  // fused MoCo forward: row sums of the un-normalised weights
      w[e] = wv;
    }
    pk[i4 * 2] = pack_h2<OPF16>(w[0], w[1]);
    pk[i4 * 2 + 1] = pack_h2<OPF16>(w[2], w[3]);
  }
}

// 640 threads: warpgroup 0 = {TMA producer, MMA issuer, 2 idle warps} at 40 registers/thread; warps 4..19 = FOUR weight
// warpgroups.  Tile t is processed by the warpgroup pair (t & 1); within the pair each warpgroup owns one 64-column
// half of the 128 x 128 tile (thread = row, TMEM lane quarter = warp % 4).  Four resident math warps per scheduler
// (instead of two) hide the TMEM-load / barrier / MUFU latencies of each other.
template <int KB, int MODE, bool OPF16 = false>
__global__ void __launch_bounds__(640, 1)
sim_bwd_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const SimParams p) {
  using C = BwdCfg<KB>;
  constexpr int BN = C::BN, NSTAGE = C::NSTAGE, DP = C::DP;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align1024(smem_raw);
  uint8_t* sA = smem;
  uint8_t* sB = smem + C::A_BYTES;
  uint8_t* sC = sB + NSTAGE * C::B_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sC + NSTAGE * C::CS_BYTES);
  uint64_t* a_full = bars;
  uint64_t* a_empty = bars + 1;
  uint64_t* b_full = bars + 2;
  uint64_t* b_empty = b_full + NSTAGE;
  uint64_t* s_full = b_empty + NSTAGE;
  uint64_t* s_empty = s_full + 2;
  uint64_t* w_full = s_empty + 2;
  uint64_t* w_empty = w_full + 2;
  uint64_t* dz_full = w_empty + 2;
  uint64_t* dz_empty = dz_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(dz_empty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(a_full, 1);
    mbar_init(a_empty, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&s_empty[i], 8);
      mbar_init(&w_full[i], 8);
      mbar_init(&w_empty[i], 1);
    }
    for (int i = 0; i < NSTAGE; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    mbar_init(dz_full, 1);
    mbar_init(dz_empty, 16);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int nunits = p.row_blocks * p.nchunks;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == 0) {
      // ---------------------------------------------------------------- TMA producer (whole warp, elect_one issues)
      int ucount = 0, gt = 0;
      for (int u = blockIdx.x; u < nunits; u += gridDim.x, ++ucount) {
        const UnitInfo ui = decode_unit(p, u);
        mbar_wait(a_empty, (ucount & 1) ^ 1);
        if (elect_one()) {
          mbar_expect_tx(a_full, C::A_BYTES);
#pragma unroll
          for (int kb = 0; kb < KB; ++kb) tma_load_2d(sA + kb * (128 * 128), &tmA, a_full, kb * 64, ui.g0);
        }
        __syncwarp();
        for (int t = ui.t0; t < ui.t1; ++t, ++gt) {
          const int st = gt % NSTAGE;
          mbar_wait(&b_empty[st], ((gt / NSTAGE) & 1) ^ 1);
          if (elect_one()) {
            constexpr int CSB = (MODE != SIM_MOCO) ? BN * 4 : 0;
            mbar_expect_tx(&b_full[st], C::B_BYTES + CSB);
#pragma unroll
            for (int kb = 0; kb < KB; ++kb)
              tma_load_2d(sB + st * C::B_BYTES + kb * (BN * 128), &tmB, &b_full[st], kb * 64, t * BN);
            if (MODE != SIM_MOCO) bulk_load_1d(sC + st * C::CS_BYTES, p.colstat + t * BN, CSB, &b_full[st]);
          }
          __syncwarp();
        }
      }
    } else if (warp == 1) {
      // ---------------------------------------------------------------- S-GEMM issuer (whole warp, elect_one issues).
      // The two GEMMs have their own issuer warps: a tile needs 16 tcgen05.mma of only 64 tensor-cycles each, and one
      // thread cannot issue them (plus commits and barrier waits) fast enough to keep the pipe full.
      constexpr uint32_t IDESC_S = make_idesc(128, BN, 0, 0, OPF16 ? 0 : 1);
      const uint32_t abase = smem_u32(sA);
      int ucount = 0, gt = 0;
      for (int u = blockIdx.x; u < nunits; u += gridDim.x, ++ucount) {
        const UnitInfo ui = decode_unit(p, u);
        mbar_wait(a_full, ucount & 1);
        for (int t = ui.t0; t < ui.t1; ++t, ++gt) {
          const int st = gt % NSTAGE, buf = gt & 1;
          mbar_wait(&b_full[st], (gt / NSTAGE) & 1);
          mbar_wait(&s_empty[buf], ((gt >> 1) & 1) ^ 1);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t bbase = smem_u32(sB + st * C::B_BYTES);
#pragma unroll
            for (int kb = 0; kb < KB; ++kb)
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4)
                umma_ss(tmem + C::T_S + buf * BN, desc_kmajor(abase + kb * (128 * 128) + k4 * 32),
                        desc_kmajor(bbase + kb * (BN * 128) + k4 * 32), IDESC_S, (kb | k4) != 0);
            umma_commit(&s_full[buf]);
            if (t == ui.t1 - 1) umma_commit(a_empty);  // last reader of this unit's A tile
          }
          __syncwarp();
        }
      }
    } else if (warp == 2) {
      // ---------------------------------------------------------------- dZ-GEMM issuer
      constexpr uint32_t IDESC_D = make_idesc(128, DP, 0, 1, OPF16 ? 0 : 1);  // A = W from TMEM, B = smem tile MN-major
      int ucount = 0, gt = 0;
      for (int u = blockIdx.x; u < nunits; u += gridDim.x, ++ucount) {
        const UnitInfo ui = decode_unit(p, u);
        mbar_wait(dz_empty, (ucount & 1) ^ 1);
        for (int t = ui.t0; t < ui.t1; ++t, ++gt) {
          const int st = gt % NSTAGE, buf = gt & 1;
          mbar_wait(&w_full[buf], (gt >> 1) & 1);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t bbase = smem_u32(sB + st * C::B_BYTES);
#pragma unroll
            for (int k = 0; k < BN / 16; ++k)
              umma_ts(tmem + C::T_DZ, tmem + C::T_W + buf * 64 + k * 8,
                      desc_mnmajor(bbase + (KB > 2 ? p.dhalf * 2 * (BN * 128) : 0) + k * (16 * 128), BN * 128), IDESC_D,
                      (t > ui.t0 || k > 0) ? 1u : 0u);
            umma_commit(&b_empty[st]);
            umma_commit(&w_empty[buf]);
            if (t == ui.t1 - 1) umma_commit(dz_full);
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ weight warpgroups + epilogue
    asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
    const int wgi = (warp - 4) >> 2;  // 0..3
    const int pair = wgi >> 1;        // which tiles (parity) / which S and W buffer
    const int half = wgi & 1;         // which 64-column half of the tile
    const int q = warp & 3;
    const int row_l = q * 32 + lane;
    const uint32_t tlane = static_cast<uint32_t>(q * 32) << 16;
    int gt = 0, ucount = 0;
    // barrier addresses in the shared window, computed once (a generic pointer costs a cvta sequence per use)
    const uint32_t a_s_full = smem_u32(&s_full[pair]), a_s_empty = smem_u32(&s_empty[pair]);
    const uint32_t a_w_full = smem_u32(&w_full[pair]), a_w_empty = smem_u32(&w_empty[pair]);
    const uint32_t a_dz_full = smem_u32(dz_full), a_dz_empty = smem_u32(dz_empty);
    const uint32_t a_sC = smem_u32(sC) + half * 64 * 4;
    for (int u = blockIdx.x; u < nunits; u += gridDim.x, ++ucount) {
      const UnitInfo ui = decode_unit(p, u);
      const int a_glob = ui.g0 + row_l;
      const bool valid = row_l < ui.nvalid;
      float rs = 0.f;
      if (valid) rs = (MODE == SIM_MOCO) ? (p.rowstat ? p.rowstat[ui.lrow0 + row_l] : p.shift) : p.rowstat[a_glob];
      float lsum = 0.f;  // SIM_MOCO with p.part_l: sum over this unit's columns of exp2(l - shift) (fused forward)
      for (int t = ui.t0; t < ui.t1; ++t, ++gt) {
        if ((gt & 1) != pair) continue;
        const int st = gt % NSTAGE;
        // no separate wait on b_full: S(t) was issued only after the MMA warp observed b_full[st], so observing
        // s_full(t) also orders this warp after the TMA / bulk-copy writes of the B tile and its column statistics
        mbar_wait_a(a_s_full, (gt >> 1) & 1);
        tc_fence_after();
        const uint32_t t_s = tmem + tlane + C::T_S + pair * BN + half * 64;
        uint32_t sv[2][32];
        tmem_ld_x32(t_s, sv[0]);
        tmem_ld_x32(t_s + 32, sv[1]);
        tmem_ld_wait_regs(sv[0]);
        tmem_ld_wait_regs(sv[1]);
        // this half of the S tile is in registers: give the buffer back so S(t+2) can be issued right away
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_a(a_s_empty);
        const int j0 = t * BN + half * 64;
        const bool special = (MODE != SIM_MOCO) ? ((j0 < ui.g0 + 128) && (j0 + 64 > ui.g0)) : (j0 + 64 > p.cols);
        const uint32_t t_w = tmem + tlane + C::T_W + pair * 64 + half * 32;
        const uint32_t cs = a_sC + st * C::CS_BYTES;
        constexpr int CSTEP = 32 * 4;
        // all 64 weights are computed and packed before waiting for the W buffer (the dZ GEMM of tile t-2 may still
        // be reading it): that wait is off the critical path unless the tensor pipe is the bottleneck
        uint32_t pk[2][16];
        if (special) {
          bwd_weights32<MODE, true, OPF16>(sv[0], pk[0], p, a_glob, j0, rs, cs, lsum);
          bwd_weights32<MODE, true, OPF16>(sv[1], pk[1], p, a_glob, j0 + 32, rs, cs + CSTEP, lsum);
        } else {
          bwd_weights32<MODE, false, OPF16>(sv[0], pk[0], p, a_glob, j0, rs, cs, lsum);
          bwd_weights32<MODE, false, OPF16>(sv[1], pk[1], p, a_glob, j0 + 32, rs, cs + CSTEP, lsum);
        }
        mbar_wait_a(a_w_empty, ((gt >> 1) & 1) ^ 1);
        tc_fence_after();
        tmem_st_x16(t_w, pk[0]);
        tmem_st_x16(t_w + 16, pk[1]);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_a(a_w_full);
      }
      if (MODE == SIM_MOCO && p.part_l != nullptr && valid)
        p.part_l[static_cast<size_t>(ui.ch * 4 + wgi) * p.part_stride + ui.lrow0 + row_l] = lsum;
      // ---- epilogue: the four warpgroups drain DP/4 accumulator columns each (DP = 64: only two of them have work)
      mbar_wait_a(a_dz_full, ucount & 1);
      tc_fence_after();
      if (DP == 128 || wgi < 2) {
        const int col0 = wgi * 32;
        uint32_t v[32];
        tmem_ld_x32(tmem + tlane + C::T_DZ + col0, v);
        tmem_ld_wait_regs(v);
        if (valid) {
          float* dst = p.dacc + static_cast<size_t>(ui.lrow0 + row_l) * p.ld_dacc + col0 + (KB > 2 ? p.dhalf * 128 : 0);
          if (p.use_atomic) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
              red_add_v4(dst + 4 * i, __uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]),
                         __uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3]));
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i)
              reinterpret_cast<float4*>(dst)[i] =
                  make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]),
                              __uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3]));
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_a(a_dz_empty);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem);
}

}  // namespace ssvb
