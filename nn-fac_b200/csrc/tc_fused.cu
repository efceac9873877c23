// Fused X pass (rank <= 64): the model tile K = W H is formed on tcgen05, consumed in registers,
// and never reaches HBM.
//
// For one 128-row tile of an X plane and each 64-column stage:
//   GEMM-1   D1[128 x 64] = A1[128 x 64] * Fk^T          A1 = rows of the factor aligned with X's rows,
//                                                         Fk = 64 rows of the other factor (rank contiguous)
//   transform (16 warps)   MODE_MU  : Q = X / K  (mu.py:84), written to tensor memory as the A operand of GEMM-2;
//                                     cost partial += X log2(X / K); KL(X | K) = ln2 * that - sum(X) + sum(K)
//                                     with sum(K) = <column sums of U, row sums of V>     (beta_divergence.py:45-48)
//                          MODE_RES : cost += (X - K)^2                                (nmf.py:452)
//   GEMM-2   D2[128 x r]  += A2[128 x 64] * Fn^T          A2 = Q (MU, mu.py:88) or X (HALS cross product, nmf.py:408)
// so one pass over X yields the contraction the update needs AND the cost of the factors it started
// from (the reference re-forms U V in a third pass for that).  All products are bf16 hi/lo splits
// (3 MMAs each) with fp32 accumulation in TMEM; D2 chains are cut every `drain` stages and summed in
// registers because the tensor core accumulates with truncation.
//
// General beta (MODE_BETA0 / _BETAI / _BETAG: beta = 0, integer beta >= 3, any other beta; 2 planes, rank <= 64), mu.py:84-97:
//   transform   Q_num = x k^(beta-2), Q_den = k^(beta-1) (both 0 where k = 0: padding), cost += k^beta h_beta(x / k)
//   GEMM-2      two chains per stage against the same factor slab: D2_num += Q_num Fn^T, D2_den += Q_den Fn^T
// Tensor memory: D1 2 x 64 | D2_num 2 x 64 | D2_den 2 x 64 | Q_num 64 | Q_den 64 = 512 columns.  A1 is not copied to tensor
// memory: the model GEMM reads it from its shared-memory staging buffer (SS form), so the next unit's A1 is only loaded once
// the unit's last model GEMM has retired.  The ratio tiles are single-buffered: the transform of stage i + 1 writes them
// after the contraction of stage i has retired.
#include "tc_plan.cuh"

#include <string.h>

namespace {
using namespace tcplan;

constexpr int NSP = 4;               // column splits of a stage among the transform warps
constexpr int CW = 64 / NSP;         // X columns per transform thread and stage
constexpr int NCHK = CW / 8;         // 16-byte chunks per thread, plane and stage
constexpr int NWT = 4 * NSP;         // transform warps: 4 TMEM lane quadrants x NSP column parts
constexpr int FUSED_THREADS = 128 + 32 * NWT;   // warp0 TMA, warps 1/3 MMA issuers, warp2 TMEM, then transform warps
static_assert(CW == 16, "the transform below moves 16 columns per tcgen05.ld / 8 words per tcgen05.st");
constexpr uint32_t X_BYTES = TILE_ROWS * BK * sizeof(bf16);   // 16 KiB per plane tile
constexpr int MODE_RES = 0, MODE_MU = 1, MODE_BETA0 = 2, MODE_BETAI = 3, MODE_BETAG = 4;
#ifndef FUSED_PREFETCH
#define FUSED_PREFETCH 0             // 1: fetch the model tile of stage i + 1 from tensor memory while stage i is transformed (measured: 9-13 % slower)
#endif
#ifndef FUSED_PACKED
#define FUSED_PACKED 1               // element-wise math on packed fp32 pairs (FADD2 / FMUL2 / FFMA2)
#endif
#ifndef FUSED_DEFER_COST
#define FUSED_DEFER_COST 1           // beta = 1 pass with cost: the log terms are computed AFTER the ratio tile has been handed to the contraction GEMM
#endif
constexpr int DRAIN = 2;             // stages per TMEM accumulation chain of the contraction GEMM (the tensor core accumulates with truncation)

// Per padded rank RK (64 or 128).  RK = 128 (ranks 65..128, MODE_RES only): the factor slab of a stage is two 64-rank
// atoms per plane (64 KiB stages, 3 of them), the contraction GEMM is 128 wide, and the rows of the aligned factor go
// global -> registers -> tensor memory (no 64 KiB staging buffer); tensor memory: D1 2 x 64 | D2 2 x 128 | A1 128.
//
// PLANES = 3 (rank <= 64): X, the factor slabs and A1 are hi/mid/lo planes, every product is six MMAs (five for the ratio tile
// of MU, which stays hi/lo).  Residual pass: stages of 3 x 16 KiB X + 3 x 8 KiB slab = 72 KiB, two of them after the 48 KiB A1
// staging buffer.  beta = 1 (X from its fp32 copy): 56 KiB stages, three of them; tensor memory D1 2 x 64 | D2 2 x 64 | A1 96 |
// Q 128 = 480 columns (ND1 = 2: three model-tile buffers would need 544).
template <int RK, int PLANES = 2, bool XF32 = false>
struct Cfg {
  static constexpr int KR = RK / 64;                                              // 64-rank atoms
  static constexpr uint32_t FK_BYTES = (uint32_t)KR * 64 * BK * sizeof(bf16);     // one plane of the slab: 64 columns of X x RK ranks
  static constexpr uint32_t XB = (PLANES == 3 && !XF32 ? 3 : 2) * X_BYTES;        // X part of a stage (XF32: one fp32 tile = 2 x 16 KiB)
  static constexpr uint32_t STAGE_BYTES = XB + PLANES * FK_BYTES;                 // 48 / 64 KiB (3 planes: 72 / 56 KiB)
  static constexpr int FSTAGES = PLANES == 3 ? (XF32 ? 3 : 2) : RK == 64 ? 4 : 3;
  static constexpr int ND1 = PLANES == 3 && XF32 ? 2 : RK == 64 ? 3 : 2;   // model-tile buffers in tensor memory: the model GEMM runs up to ND1 - 1 stages ahead of the transform
  static constexpr uint32_t A1_BYTES = RK == 64 ? PLANES * X_BYTES : 0;
  static constexpr int CWD = RK / NSP;           // D2 columns per transform thread
  static constexpr size_t SMEM = A1_BYTES + (size_t)FSTAGES * STAGE_BYTES + 512;
};

struct FusedParams {
  int r_pad, splits, stages_per_unit, num_units, drain, want_cost, tiles, split_major;
  int64_t ld_partial;
  float* partial;
  double* cost_part;
  const bf16 *a1h, *a1l;   // RK = 128: rank-contiguous planes [R x RK] of the factor aligned with the rows of this side
  int64_t R;               // rows of this side
  // push_chunk > 0 (column-sharded path, side 0): the partial of row tile t goes to rank q = 128 t / push_chunk, slab
  // (push_src * splits + split) of its inbox push[q] = [world * splits][r_pad][push_chunk] -- the reduce-scatter of the U side
  // happens in this kernel's epilogue, tile by tile, over NVLink
  float* push[NNFAC_MAX_PEERS];
  int64_t push_chunk;
  int push_src;
};

// Constants of a general-beta pass (MODE_BETA*), a kernel argument of its own behind the others.  hc[i] = c_(i+2), the
// coefficients of h_beta(1 + d) = sum_n c_n d^n (n >= 2): c_2 = 1/2, c_(n+1) = c_n (beta - n) / (n + 1).
constexpr int NHC = 11;            // d^2 .. d^12: truncation < 4e-8 relative for |d| < 1/4 and 0 <= beta <= 5
struct BetaParams {
  float* den;                      // [splits][r_pad][ld_partial]: split partials of the denominator contraction
  float beta, bm2;                 // beta, beta - 2
  int ibm2, ibeta;                 // MODE_BETAI: beta - 2 and beta as integers
  float inv_bb1, inv_beta;         // 1 / (beta (beta - 1)), 1 / beta
  float hc[NHC];
  int kb_per_slab;                 // NTF middle-mode views (AMODE 2): 64-wide k-blocks per slab of the 3-D map.  Kept here, behind
                                   // every field the other passes read, so that their kernels compile as before
};

__device__ __forceinline__ float rcp_approx(float x) {   // MUFU.RCP, <= 1 ulp: no IEEE fix-up branch
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2_approx(float x) {   // MUFU.LG2 without the denormal pre-scaling (arguments are >= 1e-30)
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// g(q) = q ln q - q + 1 >= 0, so that KL(x | k) = k g(x / k) element by element: a sum of non-negative terms, accurate also when
// x / k is within 1e-3 of 1 (series of g in d = q - 1 there; the cost of the 3-plane beta = 1 pass).  q = 0 (x = 0) gives 1.
__device__ __forceinline__ float kl_g(float q) {
  const float d = q - 1.f;
  if (fabsf(d) < 0.0625f) {
    float c = fmaf(d, -1.f / 42.f, 1.f / 30.f);
    c = fmaf(d, c, -1.f / 20.f);
    c = fmaf(d, c, 1.f / 12.f);
    c = fmaf(d, c, -1.f / 6.f);
    c = fmaf(d, c, 0.5f);
    return d * d * c;
  }
  return fmaf(q, lg2_approx(q + 1e-30f) * 0.6931471805599453f, -d);
}
__device__ __forceinline__ float ex2_approx(float x) {    // MUFU.EX2
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float ipow(float b, int n) {   // b^n, n >= 0: products only
  float r = 1.f;
  for (; n; n >>= 1, b *= b)
    if (n & 1) r *= b;
  return r;
}
// k^beta h_beta(x / k), h_beta(q) = (q^beta - beta q + beta - 1) / (beta (beta - 1)) >= 0 (beta = 0: q - 1 - ln q), so that the
// beta-divergence is a sum of non-negative terms (no cancellation against the sums of x^beta and k^beta); near q = 1 the series
// of h_beta in d = q - 1.  kb = k^beta, ik = 1 / k.  Padding (k = 0) contributes 0; x = 0 contributes what
// beta_divergence.py:49-52 gives there: k^beta / beta, and -1 at beta = 0 (its masked logarithm).
template <int MODE>
__device__ __forceinline__ float beta_cost(float x, float k, float kb, float ik, const BetaParams& bp) {
  if (!(k > 0.f)) return 0.f;
  if (x == 0.f) return MODE == MODE_BETA0 ? -1.f : kb * bp.inv_beta;
  const float q = x * ik, d = q - 1.f;
  float h;
  if (fabsf(d) < 0.25f) {
    float c = bp.hc[NHC - 1];
#pragma unroll
    for (int i = NHC - 2; i >= 0; --i) c = fmaf(d, c, bp.hc[i]);
    h = d * d * c;
  } else if (MODE == MODE_BETA0) {
    h = fmaf(lg2_approx(q), -0.6931471805599453f, d);
  } else {
    const float qb = MODE == MODE_BETAI ? ipow(q, bp.ibeta) : ex2_approx(bp.beta * lg2_approx(q));
    h = (fmaf(-bp.beta, q, qb) + (bp.beta - 1.f)) * bp.inv_bb1;
  }
  return kb * h;
}
__device__ __forceinline__ float bf_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }

// map_xm / map_fkm / map_a1m: the middle planes (PLANES = 3 only).
//
// KRAO (NTF: one-sided plans and views, MODE_MU / MODE_BETA*, rank <= 64, 2 planes): the factor slab of a stage is 64 columns of
// the Khatri-Rao operand as set_krao writes it, the K-major planes [r_pad x ld] of side 0 (a 64 x 64 box; ranks beyond r_pad read
// as zeros): the contraction GEMM reads it K-major, the model GEMM MN-major.  AMODE addresses X as tc_cross_kernel does:
// 0 rows of a 2-D map; 2 a middle mode through the 3-D map {right, I, left} (the same 128 x 64 K-major tile); 1 the last mode,
// two 64 x 64 boxes of the planes read as [left x I] (an MN-major tile: the transform reads its row's columns transposed).
// X only passes through registers there, so its addressing changes nothing else.
template <int MODE, bool COST, bool XF32, int RK, int PLANES = 2, int AMODE = 0, bool KRAO = false>
__global__ void __launch_bounds__(FUSED_THREADS, 1)
tc_fused_kernel(const __grid_constant__ CUtensorMap map_xh, const __grid_constant__ CUtensorMap map_xl,
                const __grid_constant__ CUtensorMap map_fkh, const __grid_constant__ CUtensorMap map_fkl,
                const __grid_constant__ CUtensorMap map_a1h, const __grid_constant__ CUtensorMap map_a1l,
                const FusedParams p, const __grid_constant__ CUtensorMap map_xm, const __grid_constant__ CUtensorMap map_fkm,
                const __grid_constant__ CUtensorMap map_a1m, const BetaParams bp) {
  using C = Cfg<RK, PLANES, PLANES == 3 && XF32>;
  constexpr bool BETA = MODE >= MODE_BETA0;
  static_assert(!BETA || (RK == 64 && PLANES == 2), "general beta: 2 planes, rank <= 64");
  static_assert(RK == 64 || (MODE == MODE_RES && !XF32), "rank 65..128: residual + cross-product pass only");
  static_assert(PLANES == 2 || (RK == 64 && (MODE == MODE_RES) != XF32), "3 planes: rank <= 64; beta = 1 reads X from its fp32 copy");
  static_assert(!KRAO || (RK == 64 && PLANES == 2 && !XF32 && MODE != MODE_RES), "Khatri-Rao operand: MU / general beta, 2 planes, rank <= 64");
  static_assert(AMODE == 0 || KRAO, "X addressing modes 1 and 2: NTF views only");
  constexpr int FSTAGES = C::FSTAGES, ND1 = BETA ? 2 : C::ND1, CWD = C::CWD;
  constexpr int NQ = BETA ? 1 : 2;     // ratio-tile buffers in tensor memory
  // 3 planes: one stage per contraction chain (24 MMAs, as many as two stages of the 2-plane products), drained two stages late
  constexpr int DRAIN_P = PLANES == 3 ? 1 : DRAIN;
  constexpr uint32_t FK_BYTES = C::FK_BYTES, STAGE_BYTES = C::STAGE_BYTES, A1_BYTES = C::A1_BYTES, XB = C::XB;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* a1 = smem;                                   // [hi | lo (| mid)]  (RK = 64 only)
  uint8_t* ring = smem + A1_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(ring + (size_t)FSTAGES * STAGE_BYTES);
  uint64_t* full = bars;                 // [4]
  uint64_t* empty = bars + 4;            // [4]  count NWT + 1: GEMM-2 commit + the transform warps
  uint64_t* a1_full = bars + 9;
  uint64_t* a1_empty = bars + 10;
  uint64_t* d1_full = bars + 11;         // [ND1]
  uint64_t* d1_empty = bars + 14;        // [ND1] count NWT
  uint64_t* d2_full = bars + 17;         // [2]
  uint64_t* d2_empty = bars + 19;        // [2] count NWT
  uint64_t* a1t_ready = bars + 21;       // A1 copied into tensor memory (count NWT)
  uint64_t* a1t_free = bars + 22;        // every model GEMM of the unit has retired
  uint64_t* q_ready = bars + 23;         // [2] count NWT: ratio tile written to tensor memory
  uint64_t* q_free = bars + 25;          // [2] contraction GEMM that read it has retired
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 27);
  double* cost_sh = reinterpret_cast<double*>(bars + 28);   // [2 * NWT]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tc::prefetch_tmap(&map_xh); tc::prefetch_tmap(&map_xl);
    tc::prefetch_tmap(&map_fkh); tc::prefetch_tmap(&map_fkl);
    if (RK == 64) { tc::prefetch_tmap(&map_a1h); tc::prefetch_tmap(&map_a1l); }
    if (PLANES == 3) { if (!XF32) tc::prefetch_tmap(&map_xm); tc::prefetch_tmap(&map_fkm); tc::prefetch_tmap(&map_a1m); }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < FSTAGES; ++s) { tc::mbar_init(&full[s], 1); tc::mbar_init(&empty[s], NWT + 1); }
    tc::mbar_init(a1_full, 1); tc::mbar_init(a1_empty, BETA ? 1 : NWT);   // BETA: released by the unit's last model GEMM
    tc::mbar_init(a1t_ready, NWT); tc::mbar_init(a1t_free, 1);
    for (int b = 0; b < 2; ++b) { tc::mbar_init(&q_ready[b], NWT); tc::mbar_init(&q_free[b], 1); }
    for (int b = 0; b < ND1; ++b) { tc::mbar_init(&d1_full[b], 1); tc::mbar_init(&d1_empty[b], NWT); }
    for (int b = 0; b < 2; ++b) { tc::mbar_init(&d2_full[b], 1); tc::mbar_init(&d2_empty[b], NWT); }
    tc::fence_barrier_init();
  }
  if (warp == 2) tc::tmem_alloc(tmem_slot, 512);
  tc::tcgen05_fence_before();
  __syncthreads();
  tc::tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // tensor-memory map (columns): D1 ND1 x 64 | D2 2 x RK | A1 hi RK/2 + lo RK/2 (+ mid RK/2) | Q 2 x (hi 32 + lo 32) (MU)  (512 in all)
  // BETA: D1 2 x 64 | D2 (numerator) 2 x 64 | D2D (denominator) 2 x 64 | Q_num (hi 32 + lo 32) | Q_den (hi 32 + lo 32)
  const uint32_t D1 = tmem_base, D2 = tmem_base + 64 * ND1, A1T = D2 + 2 * RK, QT = BETA ? A1T + 2 * RK : A1T + PLANES * (RK / 2);
  const uint32_t D2D = A1T;
  const int S = p.stages_per_unit;

  if (warp == 0 && lane == 0) {
    // ===================== TMA producer =====================
    int stage = 0; uint32_t phase = 0, a1_phase = 0;
    for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
      const int tile = p.split_major ? u % p.tiles : u / p.splits, split = p.split_major ? u / p.tiles : u % p.splits;
      const int row0 = tile * TILE_ROWS, k0 = split * S * BK;
      if (RK == 64) {
        tc::mbar_wait(a1_empty, a1_phase ^ 1);
        a1_phase ^= 1;
        tc::mbar_arrive_expect_tx(a1_full, A1_BYTES);
        tc::tma_load_2d_hint(a1, &map_a1h, a1_full, 0, row0, tc::kEvictLast);
        tc::tma_load_2d_hint(a1 + X_BYTES, &map_a1l, a1_full, 0, row0, tc::kEvictLast);
        if (PLANES == 3) tc::tma_load_2d_hint(a1 + 2 * X_BYTES, &map_a1m, a1_full, 0, row0, tc::kEvictLast);
      }
      for (int ks = 0; ks < S; ++ks) {
        tc::mbar_wait(&empty[stage], phase ^ 1);
        uint8_t* st = ring + (size_t)stage * STAGE_BYTES;
        tc::mbar_arrive_expect_tx(&full[stage], STAGE_BYTES);
        const int c = k0 + ks * BK;
        if constexpr (AMODE == 1) {
#pragma unroll
          for (int mb = 0; mb < 2; ++mb) {             // rows row0 + 64 mb .. + 63 of the tile, columns c .. c + 63
            tc::tma_load_2d_hint(st + mb * 8192, &map_xh, &full[stage], row0 + 64 * mb, c, tc::kEvictFirst);
            tc::tma_load_2d_hint(st + X_BYTES + mb * 8192, &map_xl, &full[stage], row0 + 64 * mb, c, tc::kEvictFirst);
          }
        } else if constexpr (AMODE == 2) {
          const int b = c / BK, slab = b / bp.kb_per_slab, off = (b - slab * bp.kb_per_slab) * BK;
          tc::tma_load_3d_hint(st, &map_xh, &full[stage], off, row0, slab, tc::kEvictFirst);
          tc::tma_load_3d_hint(st + X_BYTES, &map_xl, &full[stage], off, row0, slab, tc::kEvictFirst);
        } else {
        // XF32: map_xh is the fp32 copy of X; the two 16 KiB halves of the tile are its columns [c, c+32) and [c+32, c+64)
        tc::tma_load_2d_hint(st, &map_xh, &full[stage], c, row0, tc::kEvictFirst);
        tc::tma_load_2d_hint(st + X_BYTES, XF32 ? &map_xh : &map_xl, &full[stage], XF32 ? c + 32 : c, row0, tc::kEvictFirst);
        if (PLANES == 3 && !XF32) tc::tma_load_2d_hint(st + 2 * X_BYTES, &map_xm, &full[stage], c, row0, tc::kEvictFirst);
        }
        if constexpr (KRAO) {                          // ranks 0 .. 63 x columns c .. c + 63 of the Khatri-Rao planes
          tc::tma_load_2d_hint(st + XB, &map_fkh, &full[stage], c, 0, tc::kEvictLast);
          tc::tma_load_2d_hint(st + XB + FK_BYTES, &map_fkl, &full[stage], c, 0, tc::kEvictLast);
        } else {
#pragma unroll
        for (int kr = 0; kr < C::KR; ++kr) {   // 64 columns of X x 64 ranks per box
          tc::tma_load_2d_hint(st + XB + kr * 8192, &map_fkh, &full[stage], kr * 64, c, tc::kEvictLast);
          tc::tma_load_2d_hint(st + XB + FK_BYTES + kr * 8192, &map_fkl, &full[stage], kr * 64, c, tc::kEvictLast);
          if (PLANES == 3) tc::tma_load_2d_hint(st + XB + 2 * FK_BYTES + kr * 8192, &map_fkm, &full[stage], kr * 64, c, tc::kEvictLast);
        }
        }
        if (++stage == FSTAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer 1: model GEMM  D1 = A1 * Fk^T =====================
    // (two issuing warps, each running its loop converged with one elected lane issuing: see tc::elect_one)
    // KRAO: the slab is [ranks x columns], columns contiguous -> B operand MN-major, a K step (16 ranks) is 16 rows of 128 B
    const uint32_t idesc1 = tc::umma_idesc_bf16(TILE_ROWS, 64) | (KRAO ? (1u << 16) : 0u);
    const int ksteps = p.r_pad / UMMA_K;             // the planes are zero beyond r_pad: shorter contraction for small ranks
    int st1 = 0; uint32_t ph1 = 0;
    int b1 = 0; uint32_t b1_phase = 0;
    uint32_t a1_phase = 0;
    for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
      tc::mbar_wait(BETA ? a1_full : a1t_ready, a1_phase);
      a1_phase ^= 1;
      for (int i = 0; i < S; ++i) {
        tc::mbar_wait(&full[st1], ph1);
        tc::mbar_wait(&d1_empty[b1], b1_phase ^ 1);
        tc::tcgen05_fence_after();
        if (tc::elect_one()) {
          const uint32_t sb = tc::smem_u32(ring + (size_t)st1 * STAGE_BYTES);
          const uint64_t fkh = KRAO ? tc::umma_desc_mn_sw128(sb + XB) : tc::umma_desc_k_sw128(sb + XB);
          const uint64_t fkl = KRAO ? tc::umma_desc_mn_sw128(sb + XB + FK_BYTES) : tc::umma_desc_k_sw128(sb + XB + FK_BYTES);
          const uint32_t d = D1 + (uint32_t)b1 * 64;
          if constexpr (PLANES == 3) {
            // the five small products over the whole contraction first, the hi * hi ones last (truncating accumulation)
            const uint64_t fkm = tc::umma_desc_k_sw128(sb + XB + 2 * FK_BYTES);
            const uint32_t ah = A1T, al = A1T + RK / 2, am = A1T + RK;
#pragma unroll
            for (int k = 0; k < RK / UMMA_K; ++k) {
              if (k < ksteps) {
                const uint64_t bo = (uint64_t)((k & 3) * 2);
                tc::umma_bf16_ts(d, al + 8 * k, fkh + bo, idesc1, k != 0);   // order 2^-16
                tc::umma_bf16_ts(d, am + 8 * k, fkm + bo, idesc1, true);
                tc::umma_bf16_ts(d, ah + 8 * k, fkl + bo, idesc1, true);
                tc::umma_bf16_ts(d, am + 8 * k, fkh + bo, idesc1, true);     // order 2^-8
                tc::umma_bf16_ts(d, ah + 8 * k, fkm + bo, idesc1, true);
              }
            }
#pragma unroll
            for (int k = 0; k < RK / UMMA_K; ++k)
              if (k < ksteps) tc::umma_bf16_ts(d, ah + 8 * k, fkh + (uint64_t)((k & 3) * 2), idesc1, true);
          } else if constexpr (BETA) {
            // A1 from its shared-memory staging buffer (K-major, like an X tile)
            const uint64_t ah = tc::umma_desc_k_sw128(tc::smem_u32(a1)), al = tc::umma_desc_k_sw128(tc::smem_u32(a1 + X_BYTES));
#pragma unroll
            for (int k = 0; k < RK / UMMA_K; ++k) {
              if (k < ksteps) {
                const uint64_t ko = (uint64_t)(k * 2), bo = KRAO ? (uint64_t)(k * 128) : (uint64_t)((k & 3) * 2);
                tc::umma_bf16(d, ah + ko, fkh + bo, idesc1, k != 0);
                tc::umma_bf16(d, al + ko, fkh + bo, idesc1, true);
                tc::umma_bf16(d, ah + ko, fkl + bo, idesc1, true);
              }
            }
          } else {
#pragma unroll
          for (int k = 0; k < RK / UMMA_K; ++k) {
            if (k < ksteps) {
              const uint64_t bo = KRAO ? (uint64_t)(k * 128)                             // 16 rank rows of 128 B
                                       : (uint64_t)((k >> 2) * (8192 >> 4) + (k & 3) * 2);   // 64-rank atom, 32 B inside its 128 B row
              tc::umma_bf16_ts(d, A1T + 8 * k, fkh + bo, idesc1, k != 0);
              tc::umma_bf16_ts(d, A1T + RK / 2 + 8 * k, fkh + bo, idesc1, true);
              tc::umma_bf16_ts(d, A1T + 8 * k, fkl + bo, idesc1, true);
            }
          }
          }
          tc::umma_commit(&d1_full[b1]);
          if (i == S - 1) tc::umma_commit(BETA ? a1_empty : a1t_free);
        }
        __syncwarp();
        if (++b1 == ND1) { b1 = 0; b1_phase ^= 1; }
        if (++st1 == FSTAGES) { st1 = 0; ph1 ^= 1; }
      }
    }
  } else if (warp == 3) {
    // ===================== MMA issuer 2: contraction GEMM  D2 += A2 * Fn^T =====================
    // B operand MN-major (the rank-contiguous slab); KRAO: K-major (the Khatri-Rao planes, columns contiguous)
    const uint32_t idesc2 = tc::umma_idesc_bf16(TILE_ROWS, p.r_pad) | (KRAO ? 0u : (1u << 16));
    int qb = 0; uint32_t qb_phase = 0;      // Q buffer (MU)
    int st2 = 0; uint32_t ph2 = 0;
    int b2 = 0; uint32_t b2_phase = 0;      // D2 buffer
    for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
      for (int j = 0; j < S; ++j) {
        const bool chain_start = (j % DRAIN_P) == 0;
        const bool chain_end = ((j + 1) % DRAIN_P) == 0 || j == S - 1;
        tc::mbar_wait(&full[st2], ph2);
        if (MODE == MODE_MU || BETA) tc::mbar_wait(&q_ready[qb], qb_phase);
        if (chain_start) tc::mbar_wait(&d2_empty[b2], b2_phase ^ 1);
        tc::tcgen05_fence_after();
        if (tc::elect_one()) {
          const uint32_t sb = tc::smem_u32(ring + (size_t)st2 * STAGE_BYTES);
          const uint64_t xh = tc::umma_desc_k_sw128(sb), xl = tc::umma_desc_k_sw128(sb + X_BYTES);
          // B operand = the SAME 64-column slab of the other factor that the model GEMM reads K-major, addressed
          // MN-major here (rank contiguous = N, columns = K): no second copy of the factor travels through L2
          const uint64_t fnh = KRAO ? tc::umma_desc_k_sw128(sb + XB) : tc::umma_desc_mn_sw128(sb + XB);
          const uint64_t fnl = KRAO ? tc::umma_desc_k_sw128(sb + XB + FK_BYTES) : tc::umma_desc_mn_sw128(sb + XB + FK_BYTES);
          const uint32_t d = D2 + (uint32_t)b2 * RK;
          if constexpr (PLANES == 3) {
            // small products of the stage first, hi * hi last (see the model GEMM)
            const uint64_t fnm = tc::umma_desc_mn_sw128(sb + XB + 2 * FK_BYTES);
            const uint64_t xm = tc::umma_desc_k_sw128(sb + 2 * X_BYTES);
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              const uint64_t ko = (uint64_t)(k * 2), kb = (uint64_t)(k * 128);
              const bool acc0 = !(chain_start && k == 0);
              if (MODE == MODE_MU) {
                const uint32_t qa = QT + (uint32_t)qb * 64 + 8 * k;   // ratio tile: hi at qa, lo at qa + 32
                tc::umma_bf16_ts(d, qa, fnl + kb, idesc2, acc0);        // order 2^-16
                tc::umma_bf16_ts(d, qa + 32, fnm + kb, idesc2, true);
                tc::umma_bf16_ts(d, qa, fnm + kb, idesc2, true);        // order 2^-8
                tc::umma_bf16_ts(d, qa + 32, fnh + kb, idesc2, true);
              } else {
                tc::umma_bf16(d, xl + ko, fnh + kb, idesc2, acc0);      // order 2^-16
                tc::umma_bf16(d, xm + ko, fnm + kb, idesc2, true);
                tc::umma_bf16(d, xh + ko, fnl + kb, idesc2, true);
                tc::umma_bf16(d, xm + ko, fnh + kb, idesc2, true);      // order 2^-8
                tc::umma_bf16(d, xh + ko, fnm + kb, idesc2, true);
              }
            }
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              if (MODE == MODE_MU) tc::umma_bf16_ts(d, QT + (uint32_t)qb * 64 + 8 * k, fnh + (uint64_t)(k * 128), idesc2, true);
              else tc::umma_bf16(d, xh + (uint64_t)(k * 2), fnh + (uint64_t)(k * 128), idesc2, true);
            }
          } else if constexpr (BETA) {
            // two chains against the same slab: numerator into D2, denominator into D2D
            const uint32_t dd = D2D + (uint32_t)b2 * RK;
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              const uint64_t kb = KRAO ? (uint64_t)(k * 2) : (uint64_t)(k * 128);   // KRAO: 16 columns = 32 B inside the 128 B row
              const uint32_t qa = QT + 8 * k, qd = qa + 64;
              const bool acc0 = !(chain_start && k == 0);
              tc::umma_bf16_ts(d, qa, fnh + kb, idesc2, acc0);
              tc::umma_bf16_ts(d, qa + 32, fnh + kb, idesc2, true);
              tc::umma_bf16_ts(d, qa, fnl + kb, idesc2, true);
              tc::umma_bf16_ts(dd, qd, fnh + kb, idesc2, acc0);
              tc::umma_bf16_ts(dd, qd + 32, fnh + kb, idesc2, true);
              tc::umma_bf16_ts(dd, qd, fnl + kb, idesc2, true);
            }
          } else {
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            const uint64_t ko = (uint64_t)(k * 2);            // A (K-major): 16 bf16 = 32 B inside the 128 B row
            const uint64_t kb = KRAO ? (uint64_t)(k * 2)      // B (KRAO, K-major): 32 B inside the 128 B row
                                     : (uint64_t)(k * 128);   // B (MN-major): 16 rows of 128 B = 2048 B
            if (MODE == MODE_MU) {
              const uint32_t qa = QT + (uint32_t)qb * 64 + 8 * k;
              tc::umma_bf16_ts(d, qa, fnh + kb, idesc2, !(chain_start && k == 0));
              tc::umma_bf16_ts(d, qa + 32, fnh + kb, idesc2, true);
              tc::umma_bf16_ts(d, qa, fnl + kb, idesc2, true);
            } else {
              tc::umma_bf16(d, xh + ko, fnh + kb, idesc2, !(chain_start && k == 0));
              tc::umma_bf16(d, xl + ko, fnh + kb, idesc2, true);
              tc::umma_bf16(d, xh + ko, fnl + kb, idesc2, true);
            }
          }
          }
          tc::umma_commit(&empty[st2]);
          if (MODE == MODE_MU || BETA) tc::umma_commit(&q_free[qb]);
          if (chain_end) tc::umma_commit(&d2_full[b2]);
        }
        __syncwarp();
        if (MODE == MODE_MU || BETA) { if (++qb == NQ) { qb = 0; qb_phase ^= 1; } }
        if (chain_end) { if (++b2 == 2) { b2 = 0; b2_phase ^= 1; } }
        if (++st2 == FSTAGES) { st2 = 0; ph2 ^= 1; }
      }
    }
  } else if (warp >= 4) {
    // ===================== transform + epilogue warps =====================
    const int q = warp & 3, part = (warp - 4) >> 2;           // TMEM lane quadrant, column part (0..NSP-1)
    const int row = q * 32 + lane;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    int st = 0; uint32_t ph = 0;
    int b1 = 0; uint32_t b1_phase = 0;
    int b2 = 0; uint32_t b2_phase = 0;
    int qb = 0; uint32_t qb_phase = 0;
    uint32_t a1_phase = 0;
    double cost = 0.0, costk = 0.0;
    for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
      const int tile = p.split_major ? u % p.tiles : u / p.splits, split = p.split_major ? u / p.tiles : u % p.splits;
      float sum[CWD], sumd[BETA ? CWD : 1];     // sumd: denominator (BETA)
#pragma unroll
      for (int j = 0; j < CWD; ++j) sum[j] = 0.f;
      if (BETA) {
#pragma unroll
        for (int j = 0; j < CWD; ++j) sumd[BETA ? j : 0] = 0.f;
      } else if (RK == 64) {
        // A1 (this unit's rows of the aligned factor): shared memory -> tensor memory, this thread's row and K part
        tc::mbar_wait(a1_full, a1_phase);
        tc::mbar_wait(a1t_free, a1_phase ^ 1);
        a1_phase ^= 1;
        tc::tcgen05_fence_after();
#pragma unroll
        for (int pl = 0; pl < PLANES; ++pl) {
          uint32_t w[4 * NCHK];
#pragma unroll
          for (int cc = 0; cc < NCHK; ++cc) {
            const int chunk = NCHK * part + cc;
            const uint4 v4 = *reinterpret_cast<const uint4*>(a1 + pl * X_BYTES + (uint32_t)row * 128u + (uint32_t)((chunk ^ (row & 7)) << 4));
            w[4 * cc] = v4.x; w[4 * cc + 1] = v4.y; w[4 * cc + 2] = v4.z; w[4 * cc + 3] = v4.w;
          }
          tc::tmem_st8(A1T + lane_base + 32 * pl + (CW / 2) * part, w);
        }
        tc::tmem_st_wait();
        tc::tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) { tc::mbar_arrive(a1t_ready); tc::mbar_arrive(a1_empty); }
      } else {
        // rank 65..128: this thread's row of the aligned factor, ranks [32 part, 32 part + 32) of both planes, straight from
        // the rank-contiguous planes in global memory (64 B per plane) into tensor memory
        const int64_t grow = (int64_t)tile * TILE_ROWS + row;
        uint32_t w[2][16];
#pragma unroll
        for (int pl = 0; pl < 2; ++pl) {
          const uint4* src = reinterpret_cast<const uint4*>((pl ? p.a1l : p.a1h) + grow * RK + part * (RK / 4));
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const uint4 v4 = grow < p.R ? __ldg(src + c) : make_uint4(0u, 0u, 0u, 0u);
            w[pl][4 * c] = v4.x; w[pl][4 * c + 1] = v4.y; w[pl][4 * c + 2] = v4.z; w[pl][4 * c + 3] = v4.w;
          }
        }
        tc::mbar_wait(a1t_free, a1_phase ^ 1);
        a1_phase ^= 1;
        tc::tcgen05_fence_after();
        tc::tmem_st16(A1T + lane_base + (RK / 8) * part, w[0]);
        tc::tmem_st16(A1T + lane_base + RK / 2 + (RK / 8) * part, w[1]);
        tc::tmem_st_wait();
        tc::tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(a1t_ready);
      }
      auto drain_chain = [&]() {
        tc::mbar_wait(&d2_full[b2], b2_phase);
        tc::tcgen05_fence_after();
#pragma unroll
        for (int c0 = 0; c0 < CWD; c0 += 16) {
          if (CWD * part + c0 < p.r_pad) {                       // r_pad is a multiple of 16; warp-uniform
            uint32_t v[16];
            tc::tmem_ld16(D2 + (uint32_t)b2 * RK + lane_base + CWD * part + c0, v);
            tc::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) sum[c0 + j] += __uint_as_float(v[j]);
            if (BETA) {
              tc::tmem_ld16(D2D + (uint32_t)b2 * RK + lane_base + CWD * part + c0, v);
              tc::tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < 16; ++j) sumd[BETA ? c0 + j : 0] += __uint_as_float(v[j]);
            }
          }
        }
        tc::tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&d2_empty[b2]);
        if (++b2 == 2) { b2 = 0; b2_phase ^= 1; }
      };
      int drained = 0;
      // fp32 partial sums of up to 8 stages (128 elements) per lane pair; FP64 adds are scarce on this part.  The element-wise
      // math runs on PACKED fp32 pairs (FADD2 / FMUL2 / FFMA2 of sm_100): two columns per instruction.
      float2 acc2 = make_float2(0.f, 0.f), acck2 = make_float2(0.f, 0.f);
      const float2 neg1 = make_float2(-1.f, -1.f), tiny2 = make_float2(1e-30f, 1e-30f);
      // The model tile of stage i + 1 is fetched from tensor memory WHILE stage i is transformed (tcgen05.ld is asynchronous
      // until its wait): the 16 transform warps read 32 KiB of tensor memory per stage, which otherwise sits on the critical path.
      uint32_t kn[CW];
      int bf = b1; uint32_t bf_phase = b1_phase;                 // buffer of the next fetch
      auto fetch_d1 = [&]() {
        tc::mbar_wait(&d1_full[bf], bf_phase);
        tc::tcgen05_fence_after();
        tc::tmem_ld16(D1 + (uint32_t)bf * 64 + lane_base + CW * part, kn);
        if (++bf == ND1) { bf = 0; bf_phase ^= 1; }
      };
#if FUSED_PREFETCH
      fetch_d1();
#endif
      for (int i = 0; i < S; ++i) {
        // ---- model tile for this stage ----
#if !FUSED_PREFETCH
        fetch_d1();
#endif
        tc::tmem_ld_wait16(kn);
        uint32_t kk[CW];
#pragma unroll
        for (int j = 0; j < CW; ++j) kk[j] = kn[j];
        tc::tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&d1_empty[b1]);
        if (++b1 == ND1) { b1 = 0; b1_phase ^= 1; }
#if FUSED_PREFETCH
        if (i + 1 < S) fetch_d1();
#endif
        // the stage's TMA data is visible to the MMA issuers; this thread must observe the barrier too
        // before reading X through the generic proxy
        tc::mbar_wait(&full[st], ph);
        uint8_t* xh = ring + (size_t)st * STAGE_BYTES;
        uint8_t* xl = xh + X_BYTES;
        uint32_t qhw[4 * NCHK], qlw[4 * NCHK];
        // deferred cost (FUSED_DEFER_COST): x and the ratio q of this thread's 16 elements stay in registers until the ratio tile
        // is on its way to the contraction GEMM; only then are the MUFU.LG2 terms computed (nothing waits for them)
        constexpr bool DEFER = FUSED_DEFER_COST && FUSED_PACKED && MODE == MODE_MU && COST;
        float2 xs[DEFER ? 4 * NCHK : 1], qs[DEFER ? 4 * NCHK : 1];
        uint32_t dhw[BETA ? 4 * NCHK : 1], dlw[BETA ? 4 * NCHK : 1];   // BETA: denominator operand (qhw / qlw: numerator)
#pragma unroll
        for (int cc = 0; cc < NCHK; ++cc) {
          float2 xv[4];
          if (XF32) {
            // fp32 tile: half (part >> 1) holds 32 columns = 8 chunks of 4 floats per row; this thread's 16 columns are
            // chunks 4 (part & 1) .. +3, two of them per iteration
            const uint8_t* xb = xh + (size_t)(part >> 1) * X_BYTES + (uint32_t)row * 128u;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int chunk = 4 * (part & 1) + 2 * cc + h;
              const float4 v4 = *reinterpret_cast<const float4*>(xb + ((chunk ^ (row & 7)) << 4));
              xv[2 * h] = make_float2(v4.x, v4.y); xv[2 * h + 1] = make_float2(v4.z, v4.w);
            }
          } else if constexpr (AMODE == 1) {
            // MN-major tile: this thread's row is element (row & 63) of the 128 B rows of box (row >> 6), one row per column.  The
            // 32 lanes of a warp read 64 neighbouring bytes of the same row: no bank conflict.
            const uint8_t* xb = xh + (row >> 6) * 8192 + (row & 7) * 2;
            const int rc = (row & 63) >> 3;
#pragma unroll
            for (int w = 0; w < 4; ++w) {
              float v[2];
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                const int col = CW * part + 8 * cc + 2 * w + h;
                const uint32_t off = (uint32_t)col * 128u + (uint32_t)((rc ^ (col & 7)) << 4);
                const uint32_t hb = *reinterpret_cast<const uint16_t*>(xb + off), lb = *reinterpret_cast<const uint16_t*>(xb + X_BYTES + off);
                v[h] = __uint_as_float(hb << 16) + __uint_as_float(lb << 16);
              }
              xv[w] = make_float2(v[0], v[1]);
            }
          } else {
            const int chunk = NCHK * part + cc;
            const uint32_t off = (uint32_t)row * 128u + (uint32_t)((chunk ^ (row & 7)) << 4);
            const uint4 h4 = *reinterpret_cast<const uint4*>(xh + off);
            const uint4 l4 = *reinterpret_cast<const uint4*>(xl + off);
            const uint32_t hw[4] = {h4.x, h4.y, h4.z, h4.w}, lw[4] = {l4.x, l4.y, l4.z, l4.w};
            if constexpr (PLANES == 3) {
              // x = hi + (mid + lo): mid + lo is the exact remainder x - hi, so x is the caller's fp32 value (hi + mid can overflow
              // near the largest float)
              const uint4 m4 = *reinterpret_cast<const uint4*>(xl + X_BYTES + off);
              const uint32_t mw[4] = {m4.x, m4.y, m4.z, m4.w};
#pragma unroll
              for (int w = 0; w < 4; ++w)
                xv[w] = __fadd2_rn(make_float2(bf_lo(hw[w]), bf_hi(hw[w])),
                                   __fadd2_rn(make_float2(bf_lo(mw[w]), bf_hi(mw[w])), make_float2(bf_lo(lw[w]), bf_hi(lw[w]))));
            } else {
#pragma unroll
            for (int w = 0; w < 4; ++w)
#if FUSED_PACKED
              xv[w] = __fadd2_rn(make_float2(bf_lo(hw[w]), bf_hi(hw[w])), make_float2(bf_lo(lw[w]), bf_hi(lw[w])));
#else
              xv[w] = make_float2(bf_lo(hw[w]) + bf_lo(lw[w]), bf_hi(hw[w]) + bf_hi(lw[w]));
#endif
            }
          }
          if constexpr (BETA) {
#pragma unroll
            for (int w = 0; w < 4; ++w) {
              float an[2], ad[2];
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                const float x = h ? xv[w].y : xv[w].x, k = __uint_as_float(kk[cc * 8 + 2 * w + h]);
                float ik = 0.f, pk, kb = 1.f;                                  // pk = k^(beta - 2), kb = k^beta
                if (MODE == MODE_BETA0) {
                  ik = rcp_approx(k);
                  pk = ik * ik;
                  ad[h] = ik;
                } else {
                  pk = MODE == MODE_BETAI ? ipow(k, bp.ibm2) : ex2_approx(bp.bm2 * lg2_approx(k));
                  ad[h] = pk * k;
                  if (COST) { ik = rcp_approx(k); kb = ad[h] * k; }
                }
                an[h] = x * pk;
                if (!(k > 0.f)) { an[h] = 0.f; ad[h] = 0.f; }                   // padding: never 0 * inf
                if (COST) acc2.x += beta_cost<MODE>(x, k, kb, ik, bp);
              }
              // hi / lo bf16 pairs: lo = bf16(v - hi), exact remainder
              const __nv_bfloat162 hn = __floats2bfloat162_rn(an[0], an[1]), hd = __floats2bfloat162_rn(ad[0], ad[1]);
              const uint32_t hnw = *reinterpret_cast<const uint32_t*>(&hn), hdw = *reinterpret_cast<const uint32_t*>(&hd);
              const __nv_bfloat162 ln = __floats2bfloat162_rn(an[0] - bf_lo(hnw), an[1] - bf_hi(hnw));
              const __nv_bfloat162 ld = __floats2bfloat162_rn(ad[0] - bf_lo(hdw), ad[1] - bf_hi(hdw));
              qhw[4 * cc + w] = hnw;
              qlw[4 * cc + w] = *reinterpret_cast<const uint32_t*>(&ln);
              dhw[BETA ? 4 * cc + w : 0] = hdw;
              dlw[BETA ? 4 * cc + w : 0] = *reinterpret_cast<const uint32_t*>(&ld);
            }
          } else {
#if FUSED_PACKED
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            const float2 x2 = xv[w];
            const float2 k2 = make_float2(__uint_as_float(kk[cc * 8 + 2 * w]), __uint_as_float(kk[cc * 8 + 2 * w + 1]));
            if (MODE == MODE_RES) {
              const float2 r2 = __ffma2_rn(k2, neg1, x2);            // x - k
              acc2 = __ffma2_rn(r2, r2, acc2);
            } else {
              // padded rows / columns have x = 0 and k = 0: k + 1e-30 keeps 0 * (1/k) = 0 there and changes no real k
              // (k >= r * 1e-24 through the 1e-12 floor of the factors)
              const float2 kt = __fadd2_rn(k2, tiny2);
              const float2 q2 = __fmul2_rn(x2, make_float2(rcp_approx(kt.x), rcp_approx(kt.y)));
              if (COST) {
                // sum of x log2(x / k) and sum of k (the model tile as the tensor core produced it, so that the two terms
                // stay consistent); the sum of x is a constant of the plan (see kl_cost_finish_kernel).  x = 0: 0 * log2(1e-30).
                if (DEFER) {
                  xs[DEFER ? 4 * cc + w : 0] = x2; qs[DEFER ? 4 * cc + w : 0] = q2;
                } else {
                  const float2 qt = __fadd2_rn(q2, tiny2);
                  acc2 = __ffma2_rn(x2, make_float2(lg2_approx(qt.x), lg2_approx(qt.y)), acc2);
                }
                acck2 = __fadd2_rn(acck2, k2);
              }
              const __nv_bfloat162 hq = __floats2bfloat162_rn(q2.x, q2.y);
              const uint32_t hqw = *reinterpret_cast<const uint32_t*>(&hq);
              const float2 rem = __ffma2_rn(make_float2(bf_lo(hqw), bf_hi(hqw)), neg1, q2);    // q - hi(q), exact
              const __nv_bfloat162 lq = __floats2bfloat162_rn(rem.x, rem.y);
              qhw[4 * cc + w] = hqw;
              qlw[4 * cc + w] = *reinterpret_cast<const uint32_t*>(&lq);
            }
          }
#else
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            const float x0 = xv[w].x, x1 = xv[w].y;
            const float k0 = __uint_as_float(kk[cc * 8 + 2 * w]), k1 = __uint_as_float(kk[cc * 8 + 2 * w + 1]);
            if (MODE == MODE_RES) {
              const float r0 = x0 - k0, r1 = x1 - k1;
              acc2.x = fmaf(r0, r0, acc2.x);
              acc2.y = fmaf(r1, r1, acc2.y);
            } else {
              const float i0 = rcp_approx(fmaxf(k0, 1e-30f)), i1 = rcp_approx(fmaxf(k1, 1e-30f));
              const float q0 = x0 * i0, q1 = x1 * i1;
              if (COST) {
                acc2.x = fmaf(x0, lg2_approx(fmaxf(q0, 1e-30f)), acc2.x);
                acc2.y = fmaf(x1, lg2_approx(fmaxf(q1, 1e-30f)), acc2.y);
                acck2.x += k0; acck2.y += k1;
              }
              const __nv_bfloat162 hq = __floats2bfloat162_rn(q0, q1);
              const uint32_t hqw = *reinterpret_cast<const uint32_t*>(&hq);
              const __nv_bfloat162 lq = __floats2bfloat162_rn(q0 - bf_lo(hqw), q1 - bf_hi(hqw));
              qhw[4 * cc + w] = hqw;
              qlw[4 * cc + w] = *reinterpret_cast<const uint32_t*>(&lq);
            }
          }
#endif
          }
        }
        auto flush_cost = [&]() {
          if (COST && ((i & 7) == 7 || i == S - 1)) {
            cost += (double)(acc2.x + acc2.y);
            acc2 = make_float2(0.f, 0.f);
            if (MODE == MODE_MU) { costk += (double)(acck2.x + acck2.y); acck2 = make_float2(0.f, 0.f); }
          }
        };
        if (!DEFER) flush_cost();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&empty[st]);          // done with the stage's X tile
        if (++st == FSTAGES) { st = 0; ph ^= 1; }
        if (MODE == MODE_MU) {
          // ratio tile -> tensor memory (A operand of the contraction GEMM): hi 32 columns, lo 32 columns
          tc::mbar_wait(&q_free[qb], qb_phase ^ 1);
          tc::tcgen05_fence_after();
          const uint32_t qa = QT + (uint32_t)qb * 64 + lane_base + (CW / 2) * part;
          tc::tmem_st8(qa, qhw);
          tc::tmem_st8(qa + 32, qlw);
          tc::tmem_st_wait();
          tc::tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) tc::mbar_arrive(&q_ready[qb]);
          if (++qb == NQ) { qb = 0; qb_phase ^= 1; }
          if (DEFER) {
#pragma unroll
            for (int e = 0; e < 4 * NCHK; ++e) {
              if constexpr (PLANES == 3) {     // the KL terms themselves, k g(q): no cancellation against sum(x) - sum(k)
                const float2 k2 = make_float2(__uint_as_float(kk[2 * e]), __uint_as_float(kk[2 * e + 1]));
                acc2 = __ffma2_rn(k2, make_float2(kl_g(qs[DEFER ? e : 0].x), kl_g(qs[DEFER ? e : 0].y)), acc2);
              } else {
                const float2 qt = __fadd2_rn(qs[DEFER ? e : 0], tiny2);
                acc2 = __ffma2_rn(xs[DEFER ? e : 0], make_float2(lg2_approx(qt.x), lg2_approx(qt.y)), acc2);
              }
            }
            flush_cost();
          }
        }
        if constexpr (BETA) {
          // numerator and denominator operands -> tensor memory (single buffer: the contraction of the previous stage has retired)
          tc::mbar_wait(&q_free[0], qb_phase ^ 1);
          tc::tcgen05_fence_after();
          const uint32_t qa = QT + lane_base + (CW / 2) * part;
          tc::tmem_st8(qa, qhw);
          tc::tmem_st8(qa + 32, qlw);
          tc::tmem_st8(qa + 64, dhw);
          tc::tmem_st8(qa + 96, dlw);
          tc::tmem_st_wait();
          tc::tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) tc::mbar_arrive(&q_ready[0]);
          qb_phase ^= 1;
        }
        // drain with a lag of one more stage: chain (i-3)/2 ended with stage i-2, its GEMMs have retired by now, and
        // its TMEM buffer is only needed again by the chain that starts with stage i+1
        if (DRAIN_P == 2 ? (i >= 3 && (i & 1)) : i >= 2) { drain_chain(); ++drained; }
      }
      for (; drained < (S + DRAIN_P - 1) / DRAIN_P; ++drained) drain_chain();
      if (p.push_chunk > 0) {
        const int64_t row0 = (int64_t)tile * TILE_ROWS;
        const int q = (int)(row0 / p.push_chunk);                          // owner of these rows of U (warp-uniform)
        float* out = p.push[q] + (((int64_t)p.push_src * p.splits + split) * p.r_pad + CWD * part) * p.push_chunk + (row0 - q * p.push_chunk) + row;
#pragma unroll
        for (int j = 0; j < CWD; ++j)
          if (CWD * part + j < p.r_pad) out[(int64_t)j * p.push_chunk] = sum[j];
      } else {
        float* out = p.partial + ((int64_t)split * p.r_pad + CWD * part) * p.ld_partial + (int64_t)tile * TILE_ROWS + row;
#pragma unroll
        for (int j = 0; j < CWD; ++j)
          if (CWD * part + j < p.r_pad) out[(int64_t)j * p.ld_partial] = sum[j];
        if (BETA) {     // the denominator partials, same layout
          float* outd = bp.den + ((int64_t)split * p.r_pad + CWD * part) * p.ld_partial + (int64_t)tile * TILE_ROWS + row;
#pragma unroll
          for (int j = 0; j < CWD; ++j)
            if (CWD * part + j < p.r_pad) outd[(int64_t)j * p.ld_partial] = sumd[BETA ? j : 0];
        }
      }
    }
    // per-CTA cost partials (fixed order): [blockIdx] = sum of squares or sum of x log2(x/k); [512 + blockIdx] = sum of k
    if (COST) {
      cost = warp_sum(cost);
      if (MODE == MODE_MU) costk = warp_sum(costk);
      if (lane == 0) { cost_sh[warp - 4] = cost; cost_sh[NWT + warp - 4] = costk; }
      asm volatile("bar.sync 1, %0;" ::"n"(32 * NWT) : "memory");
      if (warp == 4 && lane == 0) {
        double t = 0.0, tk = 0.0;
        for (int w = 0; w < NWT; ++w) { t += cost_sh[w]; tk += cost_sh[NWT + w]; }
        p.cost_part[blockIdx.x] = t;
        p.cost_part[512 + blockIdx.x] = tk;
      }
    }
  }
  tc::tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) tc::tmem_dealloc(tmem_base, 512);
}

// One pass that finishes a factor update and installs the factor in the plan:
//   APPLY: F = max(F_in * (sum of the split partials of the last fused pass) / den[k], floor)      (mu.py:84-88)
//          DENP (general beta): F = max(F_in * (num / den)^gamma, floor), den = the sum of the denominator partials
//          `den` of the same pass ([splits][r_pad][ldp], summed in the order of the numerator)          (mu.py:84-97)
//   else : F = F_in                                                                                 (after a HALS solve)
// and writes F (fp32, rank-major), its K-major bf16 hi/lo planes [r_pad x ld_plane] (operand of the cross product)
// and its rank-contiguous planes [R x 64] (operands of the fused pass).  Block = 32 columns x all ranks.
struct PeerG {                      // PULL: slice s of the factor lives in p[s] ([r x ld_in], the peers' send buffers mapped here)
  const float* p[NNFAC_MAX_PEERS];
  const unsigned long long* flags;  // local flag block of the exchange region: the kernel waits until every rank's
  int world;                        // sequence number of phase 1 (send buffer complete) has reached `seq`
  unsigned long long seq;
};

// PLANES = 3: the middle planes go to fm / rowm.  KPLANES = false (one-sided plans and views, nnfac_nmf_plan_mu_finish_rows):
// no K-major planes; the factor is the one aligned with the rows of side 0, installed as its row planes only.
template <bool APPLY, int RK, bool PULL, int PLANES = 2, bool DENP = false, bool KPLANES = true>
__global__ void __launch_bounds__(256) factor_finish_kernel(const float* __restrict__ partial, int splits, int r, int r_pad, int64_t R,
                                                            int64_t ldp, const float* __restrict__ F_in, int64_t ld_in,
                                                            int64_t in_chunk, int64_t in_slab, const PeerG G,
                                                            const float* __restrict__ den, float floor_value, float* __restrict__ F_out,
                                                            int64_t ld_out, bf16* __restrict__ fh, bf16* __restrict__ fl, int64_t ld_plane,
                                                            bf16* __restrict__ rowh, bf16* __restrict__ rowl,
                                                            bf16* __restrict__ fm = nullptr, bf16* __restrict__ rowm = nullptr,
                                                            float gamma = 1.f) {
  __shared__ float tile[RK][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  if (PULL && G.flags != nullptr) {
    if ((int)threadIdx.x < G.world) {
      const unsigned long long* f = G.flags + NNFAC_MAX_PEERS + threadIdx.x;      // [phase 1][rank]
      unsigned long long v, spins = 0;
      do {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
        if (++spins > (1ull << 27)) __trap();
      } while (v < G.seq);
    }
    __syncthreads();
  }
  const int64_t c0 = (int64_t)blockIdx.x * 32, c = c0 + tx;
  // in_chunk > 0: F_in is the output of an all-gather of column slices, [slice][r][in_chunk] with slab pitch in_slab
  const int64_t cin = in_chunk > 0 ? (c / in_chunk) * in_slab + (c % in_chunk) : c;
  // PULL: this thread's RK / 8 loads from the owner's send buffer (over NVLink) are all issued before the first is used
  float pulled[PULL ? RK / 8 : 1];
  if (PULL) {
    const float* src = c < R ? G.p[c / in_chunk] + (c % in_chunk) : nullptr;
#pragma unroll
    for (int i = 0; i < RK / 8; ++i) {
      const int k = ty + 8 * i;
      pulled[i] = (k < r && c < R) ? __ldcv(src + (int64_t)k * ld_in) : 0.f;
    }
  }
#pragma unroll
  for (int k = ty; k < RK; k += 8) {
    float f = 0.f;
    if (k < r && c < R) {
      f = PULL ? pulled[PULL ? (k - ty) / 8 : 0] : F_in[(int64_t)k * ld_in + cin];
      if (APPLY) {
        auto sum_splits = [&](const float* __restrict__ part) {
          float s = 0.f;                            // fixed order; loads issued eight at a time (few blocks, many splits
          int sp = 0;                               // when the other dimension is short: NTD has 64 splits for 256 rows)
          for (; sp + 8 <= splits; sp += 8) {
            float t[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) t[u] = part[((int64_t)(sp + u) * r_pad + k) * ldp + c];
#pragma unroll
            for (int u = 0; u < 8; ++u) s += t[u];
          }
          for (; sp < splits; ++sp) s += part[((int64_t)sp * r_pad + k) * ldp + c];
          return s;
        };
        const float num = sum_splits(partial);
        float v;
        if constexpr (DENP) {
          float ratio = num / sum_splits(den);
          if (gamma == 0.5f) ratio = sqrtf(ratio);  // beta = 0 (gamma_beta, beta_divergence.py:75-80)
          else if (gamma != 1.f) ratio = powf(ratio, gamma);
          v = f * ratio;
        } else {
          v = f * (num / den[k]);
        }
        f = v > floor_value ? v : floor_value;      // np.maximum(., epsilon); NaN propagates like numpy
        if (v != v) f = v;
      }
      if (F_out) F_out[(int64_t)k * ld_out + c] = f;
      if constexpr (KPLANES) {
      bf16 h, l;
      if constexpr (PLANES == 3) {
        bf16 md;
        tc::split3_bf16(f, h, md, l);
        fm[(int64_t)k * ld_plane + c] = md;
      } else {
        tc::split_bf16(f, h, l);
      }
      fh[(int64_t)k * ld_plane + c] = h;
      fl[(int64_t)k * ld_plane + c] = l;
      }
    }
    tile[k][tx] = f;
  }
  if (rowh == nullptr) return;
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int64_t cc = c0 + i;
    if (cc < R) {
#pragma unroll
      for (int h2 = 0; h2 < RK / 32; ++h2) {
        const int k = tx + 32 * h2;
        bf16 h, l;
        if constexpr (PLANES == 3) {
          bf16 md;
          tc::split3_bf16(tile[k][i], h, md, l);
          rowm[cc * RK + k] = md;
        } else {
          tc::split_bf16(tile[k][i], h, l);
        }
        rowh[cc * RK + k] = h;
        rowl[cc * RK + k] = l;
      }
    }
  }
}

__global__ void sum_cost_parts_kernel(const double* part, int n, double* out) {
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < n; ++i) s += part[i];
    out[0] = s;
  }
}

// KL(X | U V) = sum x ln(x / k) - sum x + sum k   (beta_divergence.py:45-48; terms with x = 0 contribute k).
// part[0..n): per-CTA sums of x log2(x / k); part[512..512+n): per-CTA sums of k; sums[0] = sum of X (constant of the plan).
//
// MUFU.LG2 (lg2.approx.ftz.f32) is not centred: on sm_100 its mean error is +6.05e-8 - 4.0e-8 * log2(q) for q in
// [0.5, 2] (tools/micro/lg2_bias.cu; residual of that fit 1.4e-8 rms).  Weighted by x and summed over 10^8..10^9
// elements this bias -- not the rounding noise -- is what limits the cost when the fit is good (cost << sum of X), so
// it is taken out of the SUM here (no per-element work):  sum x (y - a0 - a1 y) = (1 - a1) S - a0 sum(x).
__global__ void kl_cost_finish_kernel(const double* part, int n, const double* sums, double* out) {
  if (threadIdx.x == 0) {
    double s = 0.0, sk = 0.0;
    for (int i = 0; i < n; ++i) { s += part[i]; sk += part[512 + i]; }
    constexpr double a0 = 6.05e-8, a1 = -4.0e-8;
    s = (1.0 - a1) * s - a0 * sums[0];
    out[0] = 0.6931471805599453 * s - sums[0] + sk;
  }
}

// fp32 copy of a plane pair: out = hi + lo (exact: 16 significant bits), [rows x ld].  PLANES = 3: out = hi + (mid + lo),
// the fp32 value the planes were split from (mid + lo is its exact remainder x - hi).
template <int PLANES>
__global__ void __launch_bounds__(256) planes_to_f32_kernel(const bf16* __restrict__ hi, const bf16* __restrict__ lo, int64_t count,
                                                            float* __restrict__ out, const bf16* __restrict__ mid) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x * 2;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 2; i < count; i += stride) {
    const uint32_t h = *reinterpret_cast<const uint32_t*>(hi + i), l = *reinterpret_cast<const uint32_t*>(lo + i);
    if constexpr (PLANES == 3) {
      const uint32_t md = *reinterpret_cast<const uint32_t*>(mid + i);
      *reinterpret_cast<float2*>(out + i) = make_float2(bf_lo(h) + (bf_lo(md) + bf_lo(l)), bf_hi(h) + (bf_hi(md) + bf_hi(l)));
    } else {
      *reinterpret_cast<float2*>(out + i) = make_float2(bf_lo(h) + bf_lo(l), bf_hi(h) + bf_hi(l));
    }
  }
}

}  // namespace

static int finish_factor(nnfac_nmf_plan* p, int which, bool apply, const float* F_in, int64_t ld_in, int64_t in_chunk, int64_t in_slab,
                         const float* den, float floor_value, float* F_out, int64_t ld_out, cudaStream_t st, const PeerG* pulled = nullptr) {
  const int64_t len = which == 0 ? p->m : p->n;
  Side* cs = &p->side[which == 0 ? 1 : 0];        // U^T planes are the Fn operand of side 1, V planes of side 0
  Side* ps = &p->side[which];                     // the pass whose partials feed this factor
  const unsigned grid = (unsigned)ceil_div64(len, 32);
  bf16* rh = p->fused_ok ? p->rowp_h[which] : nullptr;
  bf16* rl = p->fused_ok ? p->rowp_l[which] : nullptr;
  PeerG none;
  memset(&none, 0, sizeof(none));
  if (p->planes == 3) {     // plain install only (the writers that would apply or pull refuse a 3-plane plan)
    factor_finish_kernel<false, 64, false, 3><<<grid, 256, 0, st>>>(nullptr, 0, p->r, p->r_pad, len, 0, F_in, ld_in, in_chunk, in_slab,
        none, nullptr, 0.f, F_out, ld_out, cs->fh, cs->fl, cs->ld, rh, rl, cs->fm, p->rowp_m[which]);
    NNFAC_LAUNCH_CHECK(p->ctx);
    return NNFAC_OK;
  }
#define NNFAC_FINISH(RKV)                                                                                                          \
  do {                                                                                                                             \
    if (pulled)                                                                                                                    \
      factor_finish_kernel<false, RKV, true><<<grid, 256, 0, st>>>(nullptr, 0, p->r, p->r_pad, len, 0, nullptr, ld_in, in_chunk,  \
          in_slab, *pulled, nullptr, 0.f, F_out, ld_out, cs->fh, cs->fl, cs->ld, rh, rl);                                          \
    else if (apply)                                                                                                                \
      factor_finish_kernel<true, RKV, false><<<grid, 256, 0, st>>>(p->partial, ps->cp.splits, p->r, p->r_pad, len,                \
          ps->cp.ld_partial, F_in, ld_in, in_chunk, in_slab, none, den, floor_value, F_out, ld_out, cs->fh, cs->fl, cs->ld, rh,    \
          rl);                                                                                                                     \
    else                                                                                                                           \
      factor_finish_kernel<false, RKV, false><<<grid, 256, 0, st>>>(nullptr, 0, p->r, p->r_pad, len, 0, F_in, ld_in, in_chunk,    \
          in_slab, none, nullptr, 0.f, F_out, ld_out, cs->fh, cs->fl, cs->ld, rh, rl);                                             \
  } while (0)
  if (p->rk == 64) NNFAC_FINISH(64); else NNFAC_FINISH(128);
#undef NNFAC_FINISH
  NNFAC_LAUNCH_CHECK(p->ctx);
  return NNFAC_OK;
}

static FusedParams fused_params(const nnfac_nmf_plan* p, int side, bool want_cost) {
  const Side* s = &p->side[side];
  FusedParams fp;
  fp.r_pad = p->r_pad; fp.splits = s->cp.splits; fp.stages_per_unit = s->cp.stages_per_unit; fp.num_units = s->cp.num_units;
  fp.drain = DRAIN; fp.want_cost = want_cost ? 1 : 0;
  fp.tiles = s->cp.tiles; fp.split_major = s->cp.split_major;
  fp.ld_partial = s->cp.ld_partial; fp.partial = p->partial; fp.cost_part = p->cost_part;
  fp.a1h = p->rowp_h[side]; fp.a1l = p->rowp_l[side]; fp.R = s->R;
  fp.push_chunk = 0; fp.push_src = 0;
  for (int q = 0; q < NNFAC_MAX_PEERS; ++q) fp.push[q] = nullptr;
  return fp;
}

// The MU / general-beta pass of a one-sided plan or a view (NTF): X of side 0 as the plan addresses it, the Khatri-Rao operand
// from the K-major planes of side 0 (nnfac_nmf_plan_set_krao), A1 from the row planes of factor 0.
template <int M, bool C, int AM>
static cudaError_t launch_krao_am(const nnfac_nmf_plan* p, const FusedParams& fp, const BetaParams& bp, cudaStream_t st) {
  const Side* s = &p->side[0];
  const size_t smem = Cfg<64>::SMEM;
  const cudaError_t e = cudaFuncSetAttribute(tc_fused_kernel<M, C, false, 64, 2, AM, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  tc_fused_kernel<M, C, false, 64, 2, AM, true><<<s->grid, FUSED_THREADS, smem, st>>>(s->map_xh, s->map_xl, s->map_kh, s->map_kl,
      p->map_row_a_h[0], p->map_row_a_l[0], fp, s->map_xh, s->map_kh, p->map_row_a_h[0], bp);
  return cudaSuccess;
}
template <int M, bool C>
static cudaError_t launch_krao(const nnfac_nmf_plan* p, const FusedParams& fp, BetaParams bp, cudaStream_t st) {
  const CrossParams& cp = p->side[0].cp;
  bp.kb_per_slab = cp.kb_per_slab;
  return cp.amode == 1 ? launch_krao_am<M, C, 1>(p, fp, bp, st) : cp.amode == 2 ? launch_krao_am<M, C, 2>(p, fp, bp, st)
                                                                                 : launch_krao_am<M, C, 0>(p, fp, bp, st);
}

extern "C" {

// fp32 copies of X for the beta = 1 fused pass (see nnfac_nmf_plan::xf): `workspace` (256-byte aligned, caller-owned,
// >= nnfac_nmf_plan_f32_bytes) receives X and X^T as fp32; call after the ingest.  Optional for 2-plane plans: without it
// the pass reconstructs x = hi + lo from the bf16 planes.  A 3-plane plan's beta = 1 pass needs it; its copies are the
// caller's fp32 values (hi + mid + lo).
int nnfac_nmf_plan_f32_bytes(const nnfac_nmf_plan* p, size_t* bytes) {
  NNFAC_ARG(p && bytes, "nnfac_nmf_plan_f32_bytes: NULL argument");
  size_t tot = 0;
  for (int i = 0; i < 2; ++i) tot += (((size_t)p->side[i].R * p->side[i].ld * sizeof(float)) + 255) & ~(size_t)255;
  *bytes = tot;
  return NNFAC_OK;
}

int nnfac_nmf_plan_enable_f32(nnfac_nmf_plan* p, void* workspace, size_t workspace_bytes, void* stream) {
  NNFAC_ARG(p && workspace && (((uintptr_t)workspace) & 255) == 0, "nnfac_nmf_plan_enable_f32: bad argument");
  size_t need = 0;
  nnfac_nmf_plan_f32_bytes(p, &need);
  NNFAC_ARG(workspace_bytes >= need, "nnfac_nmf_plan_enable_f32: workspace of %zu bytes needed, got %zu", need, workspace_bytes);
  NNFAC_ARG(p->sides == 3, "nnfac_nmf_plan_enable_f32: needs a two-sided plan");
  if (!p->fused_ok || p->rk != 64) { nnfac_set_error("nnfac_nmf_plan_enable_f32: rank %d > 64 is not covered by the beta = 1 fused pass", p->r); return NNFAC_ERR_UNSUPPORTED; }
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* base = (uint8_t*)workspace;
  for (int i = 0; i < 2; ++i) {
    Side* s = &p->side[i];
    p->xf[i] = (float*)base;
    const int64_t count = s->R * s->ld;                       // ld is a multiple of 64: pairs never straddle rows
    base += (((size_t)count * sizeof(float)) + 255) & ~(size_t)255;
    if (p->planes == 3) planes_to_f32_kernel<3><<<p->ctx->sm_count * 16, 256, 0, st>>>(s->xh, s->xl, count, p->xf[i], s->xm);
    else planes_to_f32_kernel<2><<<p->ctx->sm_count * 16, 256, 0, st>>>(s->xh, s->xl, count, p->xf[i], nullptr);
    NNFAC_LAUNCH_CHECK(p->ctx);
    const int rc = make_map_f32(&p->map_xf[i], p->xf[i], s->R, s->C, s->ld);
    if (rc) return rc;
  }
  p->xf_ready = 1;
  return NNFAC_OK;
}

// which = 0: U given as U^T (r x m); which = 1: V (r x n).  Builds every bf16 operand plane of that factor.
int nnfac_nmf_plan_set_factor(nnfac_nmf_plan* p, int which, const float* Ft, int64_t ld, void* stream) {
  NNFAC_ARG(p && Ft && (which == 0 || which == 1), "nnfac_nmf_plan_set_factor: bad argument");
  NNFAC_ARG(!p->base, "nnfac_nmf_plan_set_factor: not available on a view plan");
  const int64_t len = which == 0 ? p->m : p->n;
  NNFAC_ARG(ld >= len, "nnfac_nmf_plan_set_factor: leading dimension too small");
  return finish_factor(p, which, false, Ft, ld, 0, 0, nullptr, 0.f, nullptr, 0, (cudaStream_t)stream);
}

// The same from the output of an all-gather of column slices: G = [slices][r][chunk] (slice s holds columns
// [s * chunk, (s + 1) * chunk) of the factor, the last slice may be short).  Also writes the factor itself, rank-major,
// into Ft_out (r x len, leading dimension ld_out) -- one kernel instead of an un-permuting copy followed by set_factor.
int nnfac_nmf_plan_set_factor_gathered(nnfac_nmf_plan* p, int which, const float* G, int64_t chunk, float* Ft_out, int64_t ld_out,
                                       void* stream) {
  NNFAC_ARG(p && G && Ft_out && chunk > 0 && (which == 0 || which == 1), "nnfac_nmf_plan_set_factor_gathered: bad argument");
  const int64_t len = which == 0 ? p->m : p->n;
  NNFAC_ARG(ld_out >= len, "nnfac_nmf_plan_set_factor_gathered: leading dimension too small");
  if (p->planes != 2) { nnfac_set_error("nnfac_nmf_plan_set_factor_gathered: writes two planes, the plan has %d", p->planes); return NNFAC_ERR_UNSUPPORTED; }
  return finish_factor(p, which, false, G, chunk, chunk, (int64_t)p->r * chunk, nullptr, 0.f, Ft_out, ld_out, (cudaStream_t)stream);
}

// The same straight from the peers' send buffers of an exchange region (csrc/peer_xchg.cu): slice s = columns
// [s * chunk, (s + 1) * chunk) of the factor is read from rank s's send buffer ([r x pitch], mapped here) over NVLink -- the
// all-gather, the un-permute and the construction of the operand planes in one kernel.  Call after this rank's
// nnfac_xchg_post(x, 1): the kernel itself waits until every rank has posted as often.
const float* nnfac_xchg_peer_send(const nnfac_xchg* x, int q);
int nnfac_xchg_world(const nnfac_xchg* x);
void nnfac_xchg_wait_args(const nnfac_xchg* x, int phase, const unsigned long long** flags, int* world, unsigned long long* seq);
int nnfac_nmf_plan_set_factor_pulled(nnfac_nmf_plan* p, int which, const nnfac_xchg* x, int64_t chunk, int64_t pitch, float* Ft_out,
                                     int64_t ld_out, void* stream) {
  NNFAC_ARG(p && x && Ft_out && chunk > 0 && pitch >= chunk && (which == 0 || which == 1), "nnfac_nmf_plan_set_factor_pulled: bad argument");
  NNFAC_ARG(!p->base, "nnfac_nmf_plan_set_factor_pulled: not available on a view plan");
  if (p->planes != 2) { nnfac_set_error("nnfac_nmf_plan_set_factor_pulled: writes two planes, the plan has %d", p->planes); return NNFAC_ERR_UNSUPPORTED; }
  const int64_t len = which == 0 ? p->m : p->n;
  const int world = nnfac_xchg_world(x);
  NNFAC_ARG(ld_out >= len && (int64_t)world * chunk >= len, "nnfac_nmf_plan_set_factor_pulled: %d slices of %lld columns do not cover %lld",
            world, (long long)chunk, (long long)len);
  PeerG g;
  for (int q = 0; q < NNFAC_MAX_PEERS; ++q) g.p[q] = nnfac_xchg_peer_send(x, q);
  nnfac_xchg_wait_args(x, 1, &g.flags, &g.world, &g.seq);
  return finish_factor(p, which, false, nullptr, pitch, chunk, 0, nullptr, 0.f, Ft_out, ld_out, (cudaStream_t)stream, &g);
}

// HALS solve of factor `which` (nnls.py:24-198, deterministic rule) that also installs the result in the plan:
// F_out = hals_nnls_acc(UtM, UtU, F_in) and every operand plane of F_out, written by the sweep kernel itself.
// Returns NNFAC_ERR_UNSUPPORTED (no error text) when the shape is outside the tensor-core sweep's envelope, or for a 3-plane plan
// (the sweep writes two planes); the caller then runs nnfac_hals_nnls + nnfac_nmf_plan_set_factor.
int nnfac_nmf_plan_hals_solve(nnfac_nmf_plan* p, int which, const float* UtM, int64_t ld_utm, const float* UtU, int64_t ld_utu,
                              const float* F_in, int64_t ld_in, float* F_out, int64_t ld_out, int maxiter, double delta,
                              double sparsity, double* result, void* stream) {
  NNFAC_ARG(p && UtU && F_in && F_out && result && (which == 0 || which == 1), "nnfac_nmf_plan_hals_solve: bad argument");
  NNFAC_ARG(!p->base, "nnfac_nmf_plan_hals_solve: not available on a view plan");
  if (p->planes != 2) return NNFAC_ERR_UNSUPPORTED;
  const int64_t len = which == 0 ? p->m : p->n;
  NNFAC_ARG((!UtM || ld_utm >= len) && ld_in >= len && ld_out >= len && ld_utu >= p->r, "nnfac_nmf_plan_hals_solve: leading dimension too small");
  // UtM == NULL: the right-hand side is what the last X pass over side `which` left in the plan as split-K partials
  // (nnfac_nmf_plan_fused / _cross with out = NULL); the solve adds them up itself, in the order of the reduction kernel
  int nsplit = 1;
  int64_t split_stride = 0;
  if (!UtM) {
    const CrossParams& cp = p->side[which].cp;
    UtM = p->partial; ld_utm = cp.ld_partial; nsplit = cp.splits; split_stride = (int64_t)p->r_pad * cp.ld_partial;
  }
  Side* cs = &p->side[which == 0 ? 1 : 0];
  nnfac_sweep_planes pl;
  pl.fh = cs->fh; pl.fl = cs->fl; pl.ld_plane = cs->ld; pl.r_pad = p->r_pad;
  pl.rowh = p->fused_ok ? p->rowp_h[which] : nullptr;
  pl.rowl = p->fused_ok ? p->rowp_l[which] : nullptr;
  pl.row_pitch = p->rk;
  return nnfac_tc_sweep_run(p->ctx, UtM, ld_utm, UtU, ld_utu, F_in, ld_in, F_out, ld_out, p->r, len, maxiter, delta, sparsity,
                            result, &pl, (cudaStream_t)stream, nsplit, split_stride);
}

// Column-sharded path, U side: from now on a fused pass over side 0 that keeps its partials (out = NULL) writes them into the
// inbox of the rank that owns those rows of U instead of the plan's own buffer: x's stage buffer on rank q, `inbox_off`
// floats in, laid out [world * splits][r_pad][chunk] (slab = source rank * splits + split); chunk = rows of U per rank, a
// multiple of 128.  x == NULL switches it off.  *slabs / *slab_stride (optional) receive world * splits and r_pad * chunk: what
// the owner's solve (nnfac_hals_solve_slabs_f32) or update (nnfac_xchg_inbox_mu_apply) needs to add the slabs up.
void* nnfac_xchg_peer_stage(const nnfac_xchg* x, int q);
int nnfac_xchg_rank(const nnfac_xchg* x);
int64_t nnfac_xchg_stage_floats(const nnfac_xchg* x);
int nnfac_nmf_plan_set_push(nnfac_nmf_plan* p, const nnfac_xchg* x, int64_t inbox_off, int64_t chunk, int* slabs, int64_t* slab_stride) {
  NNFAC_ARG(p, "nnfac_nmf_plan_set_push: NULL plan");
  if (!x) { p->push_chunk = 0; return NNFAC_OK; }
  NNFAC_ARG(!p->base && p->fused_ok, "nnfac_nmf_plan_set_push: needs a plan with the fused pass");
  if (p->planes != 2) { nnfac_set_error("nnfac_nmf_plan_set_push: not available on a 3-plane plan"); return NNFAC_ERR_UNSUPPORTED; }
  const int world = nnfac_xchg_world(x);
  const int splits = p->side[0].cp.splits;
  NNFAC_ARG(chunk > 0 && chunk % TILE_ROWS == 0 && (int64_t)world * chunk >= p->m && inbox_off >= 0,
            "nnfac_nmf_plan_set_push: %d slices of %lld rows (multiple of 128) must cover %lld", world, (long long)chunk, (long long)p->m);
  NNFAC_ARG(inbox_off + (int64_t)world * splits * p->r_pad * chunk <= nnfac_xchg_stage_floats(x),
            "nnfac_nmf_plan_set_push: the stage buffer is too small for %d x %d slabs of %d x %lld", world, splits, p->r_pad, (long long)chunk);
  for (int q = 0; q < world; ++q) p->push[q] = (float*)nnfac_xchg_peer_stage(x, q) + inbox_off;
  p->push_chunk = chunk; p->push_src = nnfac_xchg_rank(x); p->push_world = world;
  if (slabs) *slabs = world * splits;
  if (slab_stride) *slab_stride = (int64_t)p->r_pad * chunk;
  return NNFAC_OK;
}

// out (r x n) = sum of nslabs slabs ([r_pad x ld] each, r_pad * ld floats apart), in slab order: the partials a rank finds in its
// inbox (nnfac_nmf_plan_set_push) when a plain sum is what the update needs (beta = 2 numerator)
int nnfac_reduce_slabs_f32(nnfac_ctx* ctx, const float* slabs, int64_t ld, int nslabs, int r, int r_pad, int64_t n, float* out,
                           int64_t ld_out, void* stream) {
  NNFAC_ARG(ctx && slabs && out && nslabs >= 1 && r >= 1 && r_pad >= r && n >= 1 && ld >= n && ld_out >= n, "nnfac_reduce_slabs_f32: bad argument");
  nnfac_reduce_partials(slabs, nslabs, r, r_pad, n, ld, out, ld_out, ctx->sm_count, (cudaStream_t)stream);
  NNFAC_LAUNCH_CHECK(ctx);
  return NNFAC_OK;
}

// Sum the split-K partials the last X pass over `side` left in the plan into out (r x R): what nnfac_nmf_plan_fused /
// _cross do themselves when they are given an output.
int nnfac_nmf_plan_reduce(nnfac_nmf_plan* p, int side, float* out, int64_t ld_out, void* stream) {
  NNFAC_ARG(p && out && (side == 0 || side == 1), "nnfac_nmf_plan_reduce: bad argument");
  Side* s = &p->side[side];
  NNFAC_ARG(ld_out >= s->R, "nnfac_nmf_plan_reduce: leading dimension too small");
  nnfac_reduce_partials(p->partial, s->cp.splits, p->r, p->r_pad, s->R, s->cp.ld_partial, out, ld_out, p->ctx->sm_count, (cudaStream_t)stream);
  NNFAC_LAUNCH_CHECK(p->ctx);
  return NNFAC_OK;
}

// The same sum of a partial set the caller owns, laid out as the plan's own for `side` ([splits][r_pad][ld_partial]): the
// denominator partials nnfac_nmf_plan_fused_beta leaves in den_partial, summed as a matrix.
int nnfac_nmf_plan_reduce_partials(nnfac_nmf_plan* p, int side, const float* partial, float* out, int64_t ld_out, void* stream) {
  NNFAC_ARG(p && partial && out && (side == 0 || side == 1), "nnfac_nmf_plan_reduce_partials: bad argument");
  Side* s = &p->side[side];
  NNFAC_ARG(ld_out >= s->R, "nnfac_nmf_plan_reduce_partials: leading dimension too small");
  nnfac_reduce_partials(partial, s->cp.splits, p->r, p->r_pad, s->R, s->cp.ld_partial, out, ld_out, p->ctx->sm_count, (cudaStream_t)stream);
  NNFAC_LAUNCH_CHECK(p->ctx);
  return NNFAC_OK;
}

// The sum of nnfac_nmf_plan_reduce, written as the send buffer of a reduce-scatter over `slabs` ranks (see the kernel in
// tc_nmf.cu): out = [slabs][r][chunk + tail_cols], `tail` (r x tail_cols, may be NULL with tail_cols = 0) copied behind
// every chunk.  Replaces a reduction + a permuting copy + a broadcast copy by one kernel.
int nnfac_nmf_plan_reduce_chunked(nnfac_nmf_plan* p, int side, float* out, int64_t chunk, int slabs, const float* tail, int64_t ld_tail,
                                  int tail_cols, void* stream) {
  NNFAC_ARG(p && out && (side == 0 || side == 1) && chunk > 0 && slabs > 0 && tail_cols >= 0 && (tail || tail_cols == 0),
            "nnfac_nmf_plan_reduce_chunked: bad argument");
  Side* s = &p->side[side];
  NNFAC_ARG((int64_t)slabs * chunk >= s->R, "nnfac_nmf_plan_reduce_chunked: %d slabs of %lld columns do not cover %lld", slabs,
            (long long)chunk, (long long)s->R);
  nnfac_reduce_partials_chunked(p->partial, s->cp.splits, p->r, p->r_pad, s->R, s->cp.ld_partial, out, chunk, slabs, tail, ld_tail,
                                tail_cols, p->ctx->sm_count, (cudaStream_t)stream);
  NNFAC_LAUNCH_CHECK(p->ctx);
  return NNFAC_OK;
}

// beta = 1 multiplicative update of factor `which` from the numerator partials the last fused pass over side `which`
// left in the plan (call nnfac_nmf_plan_fused with out = NULL): F_out = max(F_in * num / den[k], floor), mu.py:84-88,
// and F_out is installed in the plan (as nnfac_nmf_plan_set_factor would).  den: r row sums of the other factor.
int nnfac_nmf_plan_mu_finish(nnfac_nmf_plan* p, int which, const float* F_in, int64_t ld_in, const float* den, double floor_value,
                             float* F_out, int64_t ld_out, void* stream) {
  NNFAC_ARG(p && F_in && den && F_out && (which == 0 || which == 1), "nnfac_nmf_plan_mu_finish: bad argument");
  const int64_t len = which == 0 ? p->m : p->n;
  NNFAC_ARG(ld_in >= len && ld_out >= len, "nnfac_nmf_plan_mu_finish: leading dimension too small");
  if (!p->fused_ok) { nnfac_set_error("nnfac_nmf_plan_mu_finish: rank %d > 128 is not covered by the fused pass", p->r); return NNFAC_ERR_UNSUPPORTED; }
  if (p->base) { nnfac_set_error("nnfac_nmf_plan_mu_finish: a view has no side-1 planes (nnfac_nmf_plan_mu_finish_rows)"); return NNFAC_ERR_UNSUPPORTED; }
  if (p->planes != 2) { nnfac_set_error("nnfac_nmf_plan_mu_finish: writes two planes, the plan has %d (apply + set_factor)", p->planes); return NNFAC_ERR_UNSUPPORTED; }
  return finish_factor(p, which, true, F_in, ld_in, 0, 0, den, (float)floor_value, F_out, ld_out, (cudaStream_t)stream);
}

// One fused pass over side `side` (0: planes of X, rows = m; 1: planes of X^T, rows = n).
//   mode 0: out (r x R) = Fn X-plane^T (the HALS cross product), cost = ||X - U V||_F^2
//   mode 1: out (r x R) = Fn (X / (U V))^T (the beta=1 MU numerator), cost = KL(X | U V) when want_cost
// Uses the factor planes installed by nnfac_nmf_plan_set_factor for BOTH factors.
int nnfac_nmf_plan_fused(nnfac_nmf_plan* p, int side, int mode, int want_cost, float* out, int64_t ld_out, double* cost_out,
                         void* stream) {
  NNFAC_ARG(p && (side == 0 || side == 1) && (mode == 0 || mode == 1), "nnfac_nmf_plan_fused: bad argument");
  NNFAC_ARG((p->sides >> side) & 1, "nnfac_nmf_plan_fused: this plan keeps no planes of side %d", side);
  if (!p->fused_ok) { nnfac_set_error("nnfac_nmf_plan_fused: not covered by the fused pass (rank %d > 128, or a view plan of rank > 64)", p->r); return NNFAC_ERR_UNSUPPORTED; }
  if (mode == 1 && p->rk != 64) { nnfac_set_error("nnfac_nmf_plan_fused: the beta = 1 pass covers rank <= 64 (rank %d)", p->r); return NNFAC_ERR_UNSUPPORTED; }
  if (mode == 0 && p->base) { nnfac_set_error("nnfac_nmf_plan_fused: the residual pass reads row planes a view does not have (set_krao_rows)"); return NNFAC_ERR_UNSUPPORTED; }
  if (mode == 1 && p->planes == 3 && !p->xf_ready) { nnfac_set_error("nnfac_nmf_plan_fused: the beta = 1 pass of a 3-plane plan reads X from its fp32 copies (nnfac_nmf_plan_enable_f32)"); return NNFAC_ERR_UNSUPPORTED; }
  Side* s = &p->side[side];
  NNFAC_ARG(!out || ld_out >= s->R, "nnfac_nmf_plan_fused: leading dimension too small");
  cudaStream_t st = (cudaStream_t)stream;
  FusedParams fp = fused_params(p, side, mode == 0 || want_cost);
  BetaParams bp;
  memset(&bp, 0, sizeof(bp));
  if (side == 0 && !out && p->push_chunk > 0) {       // sharded U side: partials go straight to their owners' inboxes
    fp.push_chunk = p->push_chunk; fp.push_src = p->push_src;
    for (int q = 0; q < p->push_world; ++q) fp.push[q] = p->push[q];
  }
  const int other = 1 - side;
  const bool krao = mode == 1 && p->sides == 1;       // one-sided plan or view: the Khatri-Rao operand of set_krao
  if (krao && p->push_chunk > 0) { nnfac_set_error("nnfac_nmf_plan_fused: no push exchange on a one-sided plan"); return NNFAC_ERR_UNSUPPORTED; }
#define NNFAC_LAUNCH_FUSED(M, C, XF, RKV, MAPH, MAPL)                                                                             \
  do {                                                                                                                        \
    const size_t smem = Cfg<RKV>::SMEM;                                                                                       \
    NNFAC_CUDA(cudaFuncSetAttribute(tc_fused_kernel<M, C, XF, RKV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    tc_fused_kernel<M, C, XF, RKV><<<s->grid, FUSED_THREADS, smem, st>>>(MAPH, MAPL, p->map_row_b_h[other],                  \
        p->map_row_b_l[other], p->map_row_a_h[side], p->map_row_a_l[side], fp, MAPH, p->map_row_b_h[other],                  \
        p->map_row_a_h[side], bp);                                                                                            \
  } while (0)
#define NNFAC_LAUNCH_FUSED3(M, C, XF, MAPH, MAPL)                                                                                \
  do {                                                                                                                        \
    const size_t smem = Cfg<64, 3, XF>::SMEM;                                                                                 \
    NNFAC_CUDA(cudaFuncSetAttribute(tc_fused_kernel<M, C, XF, 64, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    tc_fused_kernel<M, C, XF, 64, 3><<<s->grid, FUSED_THREADS, smem, st>>>(MAPH, MAPL, p->map_row_b_h[other],                \
        p->map_row_b_l[other], p->map_row_a_h[side], p->map_row_a_l[side], fp, s->map_xm, p->map_row_b_m[other],             \
        p->map_row_a_m[side], bp);                                                                                            \
  } while (0)
  if (krao) {
    NNFAC_CUDA((fp.want_cost ? launch_krao<MODE_MU, true>(p, fp, bp, st) : launch_krao<MODE_MU, false>(p, fp, bp, st)));
  } else if (p->planes == 3) {
    if (mode == 0) NNFAC_LAUNCH_FUSED3(MODE_RES, true, false, s->map_xh, s->map_xl);
    else if (fp.want_cost) NNFAC_LAUNCH_FUSED3(MODE_MU, true, true, p->map_xf[side], p->map_xf[side]);
    else NNFAC_LAUNCH_FUSED3(MODE_MU, false, true, p->map_xf[side], p->map_xf[side]);
  } else if (mode == 0 && p->rk == 128) NNFAC_LAUNCH_FUSED(MODE_RES, true, false, 128, s->map_xh, s->map_xl);
  else if (mode == 0) NNFAC_LAUNCH_FUSED(MODE_RES, true, false, 64, s->map_xh, s->map_xl);
  else if (p->xf_ready) {   // beta = 1: X only travels through registers -> read its fp32 copy
    if (fp.want_cost) NNFAC_LAUNCH_FUSED(MODE_MU, true, true, 64, p->map_xf[side], p->map_xf[side]);
    else NNFAC_LAUNCH_FUSED(MODE_MU, false, true, 64, p->map_xf[side], p->map_xf[side]);
  } else {
    if (fp.want_cost) NNFAC_LAUNCH_FUSED(MODE_MU, true, false, 64, s->map_xh, s->map_xl);
    else NNFAC_LAUNCH_FUSED(MODE_MU, false, false, 64, s->map_xh, s->map_xl);
  }
#undef NNFAC_LAUNCH_FUSED
#undef NNFAC_LAUNCH_FUSED3
  NNFAC_LAUNCH_CHECK(p->ctx);
  if (out) {      // out == NULL: the split partials stay in the plan for nnfac_nmf_plan_mu_finish
    nnfac_reduce_partials(p->partial, fp.splits, p->r, p->r_pad, s->R, fp.ld_partial, out, ld_out, p->ctx->sm_count, st);
    NNFAC_LAUNCH_CHECK(p->ctx);
  }
  if (cost_out && fp.want_cost) {
    if (mode == 0 || p->planes == 3)     // 3 planes, mode 1: the pass summed the KL terms themselves
      sum_cost_parts_kernel<<<1, 32, 0, st>>>(p->cost_part, s->grid, cost_out);
    else
      kl_cost_finish_kernel<<<1, 32, 0, st>>>(p->cost_part, s->grid, p->sums, cost_out);
    NNFAC_LAUNCH_CHECK(p->ctx);
  }
  return NNFAC_OK;
}

// Bytes of the caller-owned buffer that receives the denominator partials of nnfac_nmf_plan_fused_beta (either side).
int nnfac_nmf_plan_fused_beta_bytes(const nnfac_nmf_plan* p, size_t* bytes) {
  NNFAC_ARG(p && bytes, "nnfac_nmf_plan_fused_beta_bytes: NULL argument");
  *bytes = p->partial_bytes;
  return NNFAC_OK;
}

// General-beta pass (beta >= 0 other than 1 and 2) over side `side`: numerator partials of (K^(beta-2) * X) Fn^T into the
// plan's partial buffer, denominator partials of K^(beta-1) Fn^T into den_partial, cost_out = beta-divergence(X | U V).
int nnfac_nmf_plan_fused_beta(nnfac_nmf_plan* p, int side, double beta, int want_cost, float* den_partial, double* cost_out,
                              void* stream) {
  NNFAC_ARG(p && den_partial && (side == 0 || side == 1), "nnfac_nmf_plan_fused_beta: bad argument");
  NNFAC_ARG(beta >= 0.0, "nnfac_nmf_plan_fused_beta: beta must be >= 0 (got %g)", beta);
  NNFAC_ARG((p->sides >> side) & 1, "nnfac_nmf_plan_fused_beta: this plan keeps no planes of side %d", side);
  if (beta == 1.0 || beta == 2.0) { nnfac_set_error("nnfac_nmf_plan_fused_beta: beta = %g is the mode-1 / cross-product pass", beta); return NNFAC_ERR_UNSUPPORTED; }
  if (!p->fused_ok || p->rk != 64) { nnfac_set_error("nnfac_nmf_plan_fused_beta: covers rank <= 64 (rank %d)", p->r); return NNFAC_ERR_UNSUPPORTED; }
  if (p->planes != 2) { nnfac_set_error("nnfac_nmf_plan_fused_beta: covers 2-plane plans (the plan has %d)", p->planes); return NNFAC_ERR_UNSUPPORTED; }
  if (p->push_chunk > 0) { nnfac_set_error("nnfac_nmf_plan_fused_beta: not available with the push exchange (nnfac_nmf_plan_set_push)"); return NNFAC_ERR_UNSUPPORTED; }
  Side* s = &p->side[side];
  cudaStream_t st = (cudaStream_t)stream;
  const FusedParams fp = fused_params(p, side, want_cost != 0);
  BetaParams bp;
  memset(&bp, 0, sizeof(bp));
  bp.den = den_partial;
  bp.beta = (float)beta; bp.bm2 = (float)(beta - 2.0);
  bp.ibm2 = (int)beta - 2; bp.ibeta = (int)beta;
  bp.inv_bb1 = (float)(1.0 / (beta * (beta - 1.0))); bp.inv_beta = beta > 0.0 ? (float)(1.0 / beta) : 0.f;
  double c = 0.5;
  for (int i = 0; i < NHC; ++i) { bp.hc[i] = (float)c; c *= (beta - (i + 2)) / (i + 3); }
  const bool integral = beta >= 3.0 && beta == (double)(int)beta;
  const int other = 1 - side;
#define NNFAC_LAUNCH_BETA(M, C, XF, MAPH, MAPL)                                                                                \
  do {                                                                                                                        \
    const size_t smem = Cfg<64>::SMEM;                                                                                        \
    NNFAC_CUDA(cudaFuncSetAttribute(tc_fused_kernel<M, C, XF, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));  \
    tc_fused_kernel<M, C, XF, 64><<<s->grid, FUSED_THREADS, smem, st>>>(MAPH, MAPL, p->map_row_b_h[other],                    \
        p->map_row_b_l[other], p->map_row_a_h[side], p->map_row_a_l[side], fp, MAPH, p->map_row_b_h[other],                  \
        p->map_row_a_h[side], bp);                                                                                            \
  } while (0)
#define NNFAC_LAUNCH_BETA_X(M, C)                                                                                              \
  do {                                                                                                                        \
    if (p->xf_ready) NNFAC_LAUNCH_BETA(M, C, true, p->map_xf[side], p->map_xf[side]);                                         \
    else NNFAC_LAUNCH_BETA(M, C, false, s->map_xh, s->map_xl);                                                                \
  } while (0)
  if (p->sides == 1) {      // one-sided plan or view: the Khatri-Rao operand of set_krao
    if (side != 0) { nnfac_set_error("nnfac_nmf_plan_fused_beta: a one-sided plan passes over side 0"); return NNFAC_ERR_UNSUPPORTED; }
    const bool wc = fp.want_cost != 0;
    if (beta == 0.0) NNFAC_CUDA((wc ? launch_krao<MODE_BETA0, true>(p, fp, bp, st) : launch_krao<MODE_BETA0, false>(p, fp, bp, st)));
    else if (integral) NNFAC_CUDA((wc ? launch_krao<MODE_BETAI, true>(p, fp, bp, st) : launch_krao<MODE_BETAI, false>(p, fp, bp, st)));
    else NNFAC_CUDA((wc ? launch_krao<MODE_BETAG, true>(p, fp, bp, st) : launch_krao<MODE_BETAG, false>(p, fp, bp, st)));
  } else if (beta == 0.0) { if (fp.want_cost) NNFAC_LAUNCH_BETA_X(MODE_BETA0, true); else NNFAC_LAUNCH_BETA_X(MODE_BETA0, false); }
  else if (integral) { if (fp.want_cost) NNFAC_LAUNCH_BETA_X(MODE_BETAI, true); else NNFAC_LAUNCH_BETA_X(MODE_BETAI, false); }
  else { if (fp.want_cost) NNFAC_LAUNCH_BETA_X(MODE_BETAG, true); else NNFAC_LAUNCH_BETA_X(MODE_BETAG, false); }
#undef NNFAC_LAUNCH_BETA_X
#undef NNFAC_LAUNCH_BETA
  NNFAC_LAUNCH_CHECK(p->ctx);
  if (cost_out && fp.want_cost) {
    sum_cost_parts_kernel<<<1, 32, 0, st>>>(p->cost_part, s->grid, cost_out);
    NNFAC_LAUNCH_CHECK(p->ctx);
  }
  return NNFAC_OK;
}

// General-beta multiplicative update of factor `which` from the partials of the last nnfac_nmf_plan_fused_beta pass over side
// `which`: F_out = max(F_in * (num / den)^gamma, floor_value) (mu.py:84-97), installed in the plan.  One kernel.
int nnfac_nmf_plan_mu_finish_beta(nnfac_nmf_plan* p, int which, const float* F_in, int64_t ld_in, const float* den_partial, double gamma,
                                  double floor_value, float* F_out, int64_t ld_out, void* stream) {
  NNFAC_ARG(p && F_in && den_partial && F_out && (which == 0 || which == 1), "nnfac_nmf_plan_mu_finish_beta: bad argument");
  const int64_t len = which == 0 ? p->m : p->n;
  NNFAC_ARG(ld_in >= len && ld_out >= len, "nnfac_nmf_plan_mu_finish_beta: leading dimension too small");
  if (p->base || !p->fused_ok || p->rk != 64 || p->planes != 2) {
    nnfac_set_error("nnfac_nmf_plan_mu_finish_beta: covers the plans of nnfac_nmf_plan_fused_beta (rank <= 64, 2 planes, no view)");
    return NNFAC_ERR_UNSUPPORTED;
  }
  const Side* cs = &p->side[which == 0 ? 1 : 0];
  const Side* ps = &p->side[which];
  PeerG none;
  memset(&none, 0, sizeof(none));
  factor_finish_kernel<true, 64, false, 2, true><<<(unsigned)ceil_div64(len, 32), 256, 0, (cudaStream_t)stream>>>(
      p->partial, ps->cp.splits, p->r, p->r_pad, len, ps->cp.ld_partial, F_in, ld_in, 0, 0, none, den_partial, (float)floor_value,
      F_out, ld_out, cs->fh, cs->fl, cs->ld, p->rowp_h[which], p->rowp_l[which], nullptr, nullptr, (float)gamma);
  NNFAC_LAUNCH_CHECK(p->ctx);
  return NNFAC_OK;
}

// Factor 0 of a one-sided plan or view (rank <= 64; F^T, r x m) installed as its row planes only: the A1 operand of the MU pass
// (a view has no side-1 planes, and that pass reads no others).
int nnfac_nmf_plan_set_factor_rows(nnfac_nmf_plan* p, const float* Ft, int64_t ld, void* stream) {
  NNFAC_ARG(p && Ft && ld >= p->m, "nnfac_nmf_plan_set_factor_rows: bad argument");
  if (p->sides != 1 || !p->fused_ok || p->rk != 64 || p->planes != 2) {
    nnfac_set_error("nnfac_nmf_plan_set_factor_rows: covers one-sided plans and views of rank <= 64 with 2 planes");
    return NNFAC_ERR_UNSUPPORTED;
  }
  PeerG none;
  memset(&none, 0, sizeof(none));
  factor_finish_kernel<false, 64, false, 2, false, false><<<(unsigned)ceil_div64(p->m, 32), 256, 0, (cudaStream_t)stream>>>(
      nullptr, 0, p->r, p->r_pad, p->m, 0, Ft, ld, 0, 0, none, nullptr, 0.f, nullptr, 0, nullptr, nullptr, 0, p->rowp_h[0], p->rowp_l[0]);
  NNFAC_LAUNCH_CHECK(p->ctx);
  return NNFAC_OK;
}

// Multiplicative update of factor 0 of a one-sided plan or view (the NTF factor of the plan's mode) from the partials of the last
// MU pass over side 0: F_out = max(F_in * num / den[k], floor) after nnfac_nmf_plan_fused(mode 1) with `den` = r floats (the
// column sums of the Khatri-Rao operand), or F_out = max(F_in * (num / den)^gamma, floor) after nnfac_nmf_plan_fused_beta with
// `den_partial` its denominator partials; exactly one of the two.  F_out is installed as the row planes of factor 0 only.
int nnfac_nmf_plan_mu_finish_rows(nnfac_nmf_plan* p, const float* F_in, int64_t ld_in, const float* den, const float* den_partial,
                                  double gamma, double floor_value, float* F_out, int64_t ld_out, void* stream) {
  NNFAC_ARG(p && F_in && F_out && (den == nullptr) != (den_partial == nullptr), "nnfac_nmf_plan_mu_finish_rows: bad argument");
  NNFAC_ARG(ld_in >= p->m && ld_out >= p->m, "nnfac_nmf_plan_mu_finish_rows: leading dimension too small");
  if (p->sides != 1 || !p->fused_ok || p->rk != 64 || p->planes != 2) {
    nnfac_set_error("nnfac_nmf_plan_mu_finish_rows: covers one-sided plans and views of rank <= 64 with 2 planes");
    return NNFAC_ERR_UNSUPPORTED;
  }
  const Side* s = &p->side[0];
  const unsigned grid = (unsigned)ceil_div64(p->m, 32);
  cudaStream_t st = (cudaStream_t)stream;
  PeerG none;
  memset(&none, 0, sizeof(none));
  if (den)
    factor_finish_kernel<true, 64, false, 2, false, false><<<grid, 256, 0, st>>>(p->partial, s->cp.splits, p->r, p->r_pad, p->m,
        s->cp.ld_partial, F_in, ld_in, 0, 0, none, den, (float)floor_value, F_out, ld_out, nullptr, nullptr, 0, p->rowp_h[0], p->rowp_l[0]);
  else
    factor_finish_kernel<true, 64, false, 2, true, false><<<grid, 256, 0, st>>>(p->partial, s->cp.splits, p->r, p->r_pad, p->m,
        s->cp.ld_partial, F_in, ld_in, 0, 0, none, den_partial, (float)floor_value, F_out, ld_out, nullptr, nullptr, 0, p->rowp_h[0],
        p->rowp_l[0], nullptr, nullptr, (float)gamma);
  NNFAC_LAUNCH_CHECK(p->ctx);
  return NNFAC_OK;
}

}  // extern "C"
