// fp32 headline path for NMF: X resident in HBM as bf16 hi/lo planes (4 bytes per element, the
// same HBM bytes as fp32, ~17 mantissa bits) in BOTH orientations, so that each of the two
// X passes of an outer iteration streams K-major tiles through TMA into tcgen05.mma.
//
//   cross(which=0):  VMt (r x m) = V  X^T   (nmf.py:408)   contraction over n, planes of X   [m x n]
//   cross(which=1):  UtM (r x n) = U^T X    (nmf.py:433)   contraction over m, planes of X^T [n x m]
//
// Each product runs as 3 bf16 MMAs (hi*hi + lo*hi + hi*lo) with fp32 accumulation in TMEM; the
// dropped lo*lo term is 2^-18 relative.  Work is cut into units of (128 rows of the X plane) x
// (a fixed range of the contraction axis); every unit writes its own fp32 partial, and a
// fixed-order reduction sums the partials, so results are deterministic.
#include "tc_plan.cuh"

#include <stdlib.h>

namespace {
using namespace tcplan;

// ---- ingest: fp32 -> bf16 hi/lo planes (PLANES = 3: hi/mid/lo, `mid` is the middle plane) ------------------------------
template <int PLANES>
__global__ void split_planes_kernel(const float* __restrict__ in, int64_t ld_in, int64_t rows, int64_t cols,
                                    bf16* __restrict__ hi, bf16* __restrict__ lo, int64_t ld_out, bf16* __restrict__ mid) {
  const int64_t total = rows * cols;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cols, c = i % cols;
    bf16 h, l;
    if constexpr (PLANES == 3) {
      bf16 md;
      tc::split3_bf16(in[r * ld_in + c], h, md, l);
      mid[r * ld_out + c] = md;
    } else {
      tc::split_bf16(in[r * ld_in + c], h, l);
    }
    hi[r * ld_out + c] = h;
    lo[r * ld_out + c] = l;
  }
}

// The factor operand read from a strided tensor: B is the C-order array (left, r, right) and plane row q = blockIdx.y holds
// V[q][l * right + rr] = B[l][q][rr] (right > 1: runs of `right` contiguous values; the last mode, right == 1, takes the tiled
// transpose below).  The same split as split_planes_kernel<2>, so that for the same values both write the same bits.  The plans
// keep every extent below 2^31, so the column index is split with 32-bit arithmetic.
__global__ void split_planes_strided_kernel(const float* __restrict__ B, int cols, int r, int right, bf16* __restrict__ hi,
                                            bf16* __restrict__ lo, int64_t ld_out) {
  const int q = blockIdx.y;
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < cols; c += gridDim.x * blockDim.x) {
    const int l = c / right, rr = c - l * right;
    bf16 h, l16;
    tc::split_bf16(B[((int64_t)l * r + q) * right + rr], h, l16);
    hi[q * ld_out + c] = h;
    lo[q * ld_out + c] = l16;
  }
}

// out planes hold in^T: hiT/loT (/midT) are [cols x rows] with leading dimension ld_out
template <int PLANES>
__global__ void split_planes_transposed_kernel(const float* __restrict__ in, int64_t ld_in, int64_t rows, int64_t cols,
                                               bf16* __restrict__ hiT, bf16* __restrict__ loT, int64_t ld_out,
                                               bf16* __restrict__ midT) {
  __shared__ float tile[32][33];
  const int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int64_t r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? in[r * ld_in + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int64_t c = c0 + i, r = r0 + threadIdx.x;
    if (r < rows && c < cols) {
      bf16 h, l;
      if constexpr (PLANES == 3) {
        bf16 md;
        tc::split3_bf16(tile[threadIdx.x][i], h, md, l);
        midT[c * ld_out + r] = md;
      } else {
        tc::split_bf16(tile[threadIdx.x][i], h, l);
      }
      hiT[c * ld_out + r] = h;
      loT[c * ld_out + r] = l;
    }
  }
}

// AMODE: how the X operand is addressed (CrossParams::amode).  0: the planes hold the rows of X K-major (TMA 2-D, 128-row box);
// 1: the planes hold X^T -- contraction index = plane row, the 128 output rows of a tile are contiguous in memory -- and the
// tile is an MN-major UMMA operand (two 64-wide M blocks per plane, each a 64 x 64 TMA box): the LAST mode of a C-order tensor;
// 2: as 0 through a 3-D map, k-block b = (slab b / kb_per_slab, offset 64 (b % kb_per_slab)): a MIDDLE mode.
// PLANES = 3 (AMODE 0 only): X and the factor as hi/mid/lo planes (map_xm / map_fm: the middle ones), six MMAs per k step.
template <int MAX_RPAD, int AMODE, int PLANES>
__global__ void __launch_bounds__(NTHREADS, 1)
tc_cross_kernel(const __grid_constant__ CUtensorMap map_xh, const __grid_constant__ CUtensorMap map_xl,
                const __grid_constant__ CUtensorMap map_fh, const __grid_constant__ CUtensorMap map_fl,
                const CrossParams p, const __grid_constant__ CUtensorMap map_xm, const __grid_constant__ CUtensorMap map_fm) {
  static_assert(PLANES == 2 || (PLANES == 3 && AMODE == 0 && MAX_RPAD == 64), "3 planes: rank <= 64, rows K-major");
  extern __shared__ __align__(1024) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t x_bytes = TILE_ROWS * BK * sizeof(bf16);        // 16 KiB
  const uint32_t f_bytes = (uint32_t)p.r_pad * BK * sizeof(bf16);
  const uint32_t stage_bytes = PLANES * (x_bytes + f_bytes);   // [X planes | factor planes], plane order hi, lo(, mid)
  uint8_t* ring = smem;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)p.num_stages * stage_bytes);
  uint64_t* empty = full + p.num_stages;
  uint64_t* acc_full = empty + p.num_stages;   // [2]
  uint64_t* acc_empty = acc_full + 2;          // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  const uint32_t acc_cols = (uint32_t)p.r_pad;  // fp32 accumulator columns per buffer
  uint32_t tmem_cols = 32;
  while (tmem_cols < 2 * acc_cols) tmem_cols <<= 1;

  if (warp == 0 && lane == 0) {
    tc::prefetch_tmap(&map_xh); tc::prefetch_tmap(&map_xl); tc::prefetch_tmap(&map_fh); tc::prefetch_tmap(&map_fl);
    if (PLANES == 3) { tc::prefetch_tmap(&map_xm); tc::prefetch_tmap(&map_fm); }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < p.num_stages; ++s) { tc::mbar_init(&full[s], 1); tc::mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { tc::mbar_init(&acc_full[a], 1); tc::mbar_init(&acc_empty[a], 4); }
    tc::fence_barrier_init();
  }
  if (warp == 2) tc::tmem_alloc(tmem_slot, tmem_cols);
  tc::tcgen05_fence_before();
  __syncthreads();
  tc::tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0 && lane == 0) {
    // ===== TMA producer =====
    int stage = 0; uint32_t phase = 0;
    for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
      const int tile = p.split_major ? u % p.tiles : u / p.splits, split = p.split_major ? u / p.tiles : u % p.splits;
      const int row0 = tile * TILE_ROWS;
      const int k0 = split * p.stages_per_unit * BK;
      for (int ks = 0; ks < p.stages_per_unit; ++ks) {
        tc::mbar_wait(&empty[stage], phase ^ 1);
        uint8_t* st = ring + (size_t)stage * stage_bytes;
        tc::mbar_arrive_expect_tx(&full[stage], stage_bytes);
        const int c = k0 + ks * BK;
        if (AMODE == 0) {
          tc::tma_load_2d_hint(st, &map_xh, &full[stage], c, row0, tc::kEvictFirst);
          tc::tma_load_2d_hint(st + x_bytes, &map_xl, &full[stage], c, row0, tc::kEvictFirst);
          if (PLANES == 3) tc::tma_load_2d_hint(st + 2 * x_bytes, &map_xm, &full[stage], c, row0, tc::kEvictFirst);
        } else if (AMODE == 1) {
#pragma unroll
          for (int mb = 0; mb < 2; ++mb) {             // M block mb: output rows row0 + 64 mb .. + 63, contraction rows c .. c + 63
            tc::tma_load_2d_hint(st + mb * 8192, &map_xh, &full[stage], row0 + 64 * mb, c, tc::kEvictFirst);
            tc::tma_load_2d_hint(st + x_bytes + mb * 8192, &map_xl, &full[stage], row0 + 64 * mb, c, tc::kEvictFirst);
          }
        } else {
          const int b = c / BK, slab = b / p.kb_per_slab, off = (b - slab * p.kb_per_slab) * BK;
          tc::tma_load_3d_hint(st, &map_xh, &full[stage], off, row0, slab, tc::kEvictFirst);
          tc::tma_load_3d_hint(st + x_bytes, &map_xl, &full[stage], off, row0, slab, tc::kEvictFirst);
        }
        tc::tma_load_2d_hint(st + PLANES * x_bytes, &map_fh, &full[stage], c, 0, tc::kEvictLast);
        tc::tma_load_2d_hint(st + PLANES * x_bytes + f_bytes, &map_fl, &full[stage], c, 0, tc::kEvictLast);
        if (PLANES == 3) tc::tma_load_2d_hint(st + 3 * x_bytes + 2 * f_bytes, &map_fm, &full[stage], c, 0, tc::kEvictLast);
        if (++stage == p.num_stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (the warp runs converged, one elected lane issues: see tc::elect_one) =====
    // The tensor core adds into the fp32 accumulator with truncation, so a long chain drifts low
    // (measured: -1.9e-5 relative over 768 accumulations).  Chains are therefore cut every
    // `drain` stages; the epilogue warps sum the chain results in registers (round-to-nearest).
    const uint32_t idesc = tc::umma_idesc_bf16(TILE_ROWS, p.r_pad) | (AMODE == 1 ? (1u << 15) : 0u);   // bit 15: A operand MN-major
    int stage = 0; uint32_t phase = 0;
    int acc = 0; uint32_t acc_phase = 0;
    for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
      for (int ks0 = 0; ks0 < p.stages_per_unit; ks0 += p.drain) {
        tc::mbar_wait(&acc_empty[acc], acc_phase ^ 1);
        tc::tcgen05_fence_after();
        const uint32_t d = tmem_base + (uint32_t)acc * acc_cols;
        const int ks1 = ks0 + p.drain < p.stages_per_unit ? ks0 + p.drain : p.stages_per_unit;
        for (int ks = ks0; ks < ks1; ++ks) {
          tc::mbar_wait(&full[stage], phase);
          tc::tcgen05_fence_after();
          if (tc::elect_one()) {
            const uint32_t st = tc::smem_u32(ring + (size_t)stage * stage_bytes);
            if constexpr (PLANES == 3) {
              // the five small products of the whole stage first, then the four hi*hi: the truncating adds of the small terms
              // then act on a partial sum 2^8 smaller than the result
              const uint32_t fb = st + 3 * x_bytes;
#pragma unroll
              for (int k = 0; k < BK / UMMA_K; ++k) {
                const uint32_t koff = k * UMMA_K * sizeof(bf16);
                const uint64_t xh = tc::umma_desc_k_sw128(st + koff), xl = tc::umma_desc_k_sw128(st + x_bytes + koff);
                const uint64_t xm = tc::umma_desc_k_sw128(st + 2 * x_bytes + koff);
                const uint64_t fh = tc::umma_desc_k_sw128(fb + koff), fl = tc::umma_desc_k_sw128(fb + f_bytes + koff);
                const uint64_t fm = tc::umma_desc_k_sw128(fb + 2 * f_bytes + koff);
                tc::umma_bf16(d, xl, fh, idesc, (ks != ks0) || (k != 0));   // order 2^-16
                tc::umma_bf16(d, xm, fm, idesc, true);
                tc::umma_bf16(d, xh, fl, idesc, true);
                tc::umma_bf16(d, xm, fh, idesc, true);                      // order 2^-8
                tc::umma_bf16(d, xh, fm, idesc, true);
              }
#pragma unroll
              for (int k = 0; k < BK / UMMA_K; ++k) {
                const uint32_t koff = k * UMMA_K * sizeof(bf16);
                tc::umma_bf16(d, tc::umma_desc_k_sw128(st + koff), tc::umma_desc_k_sw128(fb + koff), idesc, true);
              }
            } else {
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              const uint32_t koff = k * UMMA_K * sizeof(bf16);   // 32 B inside the 128 B swizzle row
              // MN-major A: a K step is 16 rows of 128 B inside each 64-wide M block
              const uint64_t xh = AMODE == 1 ? tc::umma_desc_mn_sw128(st + k * 2048) : tc::umma_desc_k_sw128(st + koff);
              const uint64_t xl = AMODE == 1 ? tc::umma_desc_mn_sw128(st + x_bytes + k * 2048) : tc::umma_desc_k_sw128(st + x_bytes + koff);
              const uint64_t fh = tc::umma_desc_k_sw128(st + 2 * x_bytes + koff);
              const uint64_t fl = tc::umma_desc_k_sw128(st + 2 * x_bytes + f_bytes + koff);
              tc::umma_bf16(d, xh, fh, idesc, (ks != ks0) || (k != 0));
              tc::umma_bf16(d, xl, fh, idesc, true);
              tc::umma_bf16(d, xh, fl, idesc, true);
            }
            }
            tc::umma_commit(&empty[stage]);                      // frees the smem slot when the MMAs retire
            if (ks == ks1 - 1) tc::umma_commit(&acc_full[acc]);  // chain result ready for the epilogue
          }
          __syncwarp();
          if (++stage == p.num_stages) { stage = 0; phase ^= 1; }
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 4) {
    // ===== epilogue: TMEM chains -> register sums -> partial[split][k][row] (coalesced along rows) =====
    const int q = warp & 3;                                  // TMEM lane quadrant of this warp
    int acc = 0; uint32_t acc_phase = 0;
    for (int u = blockIdx.x; u < p.num_units; u += gridDim.x) {
      const int tile = p.split_major ? u % p.tiles : u / p.splits, split = p.split_major ? u / p.tiles : u % p.splits;
      const int64_t row = (int64_t)tile * TILE_ROWS + q * 32 + lane;
      float* out = p.partial + (int64_t)split * p.r_pad * p.ld_partial + row;
      float sum[MAX_RPAD];
#pragma unroll
      for (int j = 0; j < MAX_RPAD; ++j) sum[j] = 0.f;
      for (int ks0 = 0; ks0 < p.stages_per_unit; ks0 += p.drain) {
        tc::mbar_wait(&acc_full[acc], acc_phase);
        tc::tcgen05_fence_after();
        const uint32_t taddr = tmem_base + (uint32_t)acc * acc_cols + ((uint32_t)(q * 32) << 16);
#pragma unroll
        for (int c0 = 0; c0 < MAX_RPAD; c0 += 16) {
          if (c0 < p.r_pad) {
            uint32_t v[16];
            tc::tmem_ld16(taddr + c0, v);
            tc::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) sum[c0 + j] += __uint_as_float(v[j]);
          }
        }
        tc::tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&acc_empty[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
#pragma unroll
      for (int j = 0; j < MAX_RPAD; ++j)
        if (j < p.r_pad) out[(int64_t)j * p.ld_partial] = sum[j];
    }
  }
  tc::tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) tc::tmem_dealloc(tmem_base, tmem_cols);
}

__global__ void reduce_partials_kernel(const float* __restrict__ partial, int splits, int r, int r_pad, int64_t R,
                                       int64_t ld_partial, float* __restrict__ out, int64_t ld_out) {
  const int64_t total = (int64_t)r * R;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t k = i / R, row = i % R;
    float s = 0.f;
    for (int sp = 0; sp < splits; ++sp) s += partial[((int64_t)sp * r_pad + k) * ld_partial + row];   // fixed order
    out[k * ld_out + row] = s;
  }
}

// The same sum written in the send layout of a reduce-scatter over `slabs` ranks: column `row` of the (r x R) result goes to
// out[row / chunk][k][row % chunk] (slab pitch `slab`, row pitch `pitch` >= chunk + tail_cols), columns beyond R are zero, and
// every slab also receives a copy of the small matrix `tail` (r x tail_cols: the partial Gram) behind its chunk.
__global__ void reduce_partials_chunked_kernel(const float* __restrict__ partial, int splits, int r, int r_pad, int64_t R,
                                               int64_t ld_partial, float* __restrict__ out, int64_t chunk, int64_t pitch, int64_t slab,
                                               int slabs, const float* __restrict__ tail, int64_t ld_tail, int tail_cols) {
  const int64_t width = chunk + tail_cols, total = (int64_t)slabs * r * width;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t c = i % width, k = (i / width) % r, s = i / (width * r);
    float v = 0.f;
    if (c < chunk) {
      const int64_t row = s * chunk + c;
      if (row < R)
        for (int sp = 0; sp < splits; ++sp) v += partial[((int64_t)sp * r_pad + k) * ld_partial + row];   // fixed order
    } else {
      v = tail[k * ld_tail + (c - chunk)];
    }
    out[s * slab + k * pitch + c] = v;
  }
}

}  // namespace

namespace {

int64_t round_up(int64_t a, int64_t b) { return (a + b - 1) / b * b; }

void choose_partition(int sm, int64_t R, int64_t C, int r_pad, int planes, Side* s) {
  const int64_t tiles = ceil_div64(R, TILE_ROWS), kblocks = ceil_div64(C, BK);
  int best_s = 1;
  double best_eff = -1.0;
  for (int S = 1; S <= 64; ++S) {
    if (S > 1 && kblocks / S < 8) break;
    const int64_t units = tiles * S;
    const int64_t waves = ceil_div64(units, sm);
    // efficiency of the last wave, discounted by the extra partial traffic of more splits
    const double eff = (double)units / (double)(waves * sm) - 0.002 * S;
    if (eff > best_eff + 1e-9) { best_eff = eff; best_s = S; }
  }
  s->cp.r_pad = r_pad;
  s->cp.splits = best_s;
  s->cp.stages_per_unit = (int)ceil_div64(kblocks, best_s);
  s->cp.splits = (int)ceil_div64(kblocks, s->cp.stages_per_unit);
  s->cp.num_units = (int)(tiles * s->cp.splits);
  s->cp.tiles = (int)tiles;
  s->cp.amode = 0;
  s->cp.kb_per_slab = 1;
  // factor planes of this side: r_pad x ld, `planes` of them.  When they do not fit L2 comfortably, order the units split-major
  s->cp.split_major = ((size_t)r_pad * (size_t)round_up(C, 64) * 2 * planes > ((size_t)32 << 20) && tiles <= sm) ? 1 : 0;
  const size_t stage_bytes = (size_t)planes * ((size_t)TILE_ROWS * BK * 2 + (size_t)r_pad * BK * 2);
  int stages = (int)((200 * 1024) / stage_bytes);
  if (stages > 6) stages = 6;
  if (stages < 2) stages = 2;
  s->cp.num_stages = stages;
  s->cp.drain = planes == 3 ? 1 : 2;    // 3 planes: 24 MMAs per stage already
  s->cp.ld_partial = round_up(R, TILE_ROWS);
  s->smem = (size_t)stages * stage_bytes + (2 * stages + 4) * sizeof(uint64_t) + 16;
  s->grid = s->cp.num_units < sm ? s->cp.num_units : sm;
}

// Sum of hi + lo (+ mid) over an [rows x cols] plane pair (triple): per-block fp64 partials (rows are dealt round-robin to the
// blocks).
template <int PLANES>
__global__ void __launch_bounds__(256) plane_total_kernel(const bf16* __restrict__ hi, const bf16* __restrict__ lo, int64_t ld,
                                                          int64_t rows, int64_t cols, double* part, const bf16* __restrict__ mid) {
  __shared__ double sh[33];
  double s = 0.0;
  for (int64_t r = blockIdx.x; r < rows; r += gridDim.x) {
    const bf16* h = hi + r * ld;
    const bf16* l = lo + r * ld;
    float t = 0.f;
    int cnt = 0;
    for (int64_t c = threadIdx.x; c < cols; c += 256) {
      if constexpr (PLANES == 3)
        t += __bfloat162float(h[c]) + (__bfloat162float(mid[r * ld + c]) + __bfloat162float(l[c]));
      else
        t += __bfloat162float(h[c]) + __bfloat162float(l[c]);
      if (++cnt == 16) { s += (double)t; t = 0.f; cnt = 0; }
    }
    s += (double)t;
  }
  s = block_sum(s, sh);
  if (threadIdx.x == 0) part[blockIdx.x] = s;
}
__global__ void plane_total_finish_kernel(const double* part, int n, double* out) {
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < n; ++i) s += part[i];
    out[0] = s;
  }
}

// K-major bf16 hi/lo planes of a Khatri-Rao product, never materialised in fp32: plane[q][a * J + b] = At[q][a] * Bt[q][b]
// (ntf.py:448: the first kept factor's row index is the slow one).  One thread per column, rank loop inside.
__global__ void __launch_bounds__(256) krao_planes_kernel(const float* __restrict__ At, int64_t lda, int64_t I, const float* __restrict__ Bt,
                                                          int64_t ldb, int64_t J, int r, bf16* __restrict__ hi, bf16* __restrict__ lo,
                                                          int64_t ld_out) {
  const int64_t total = I * J;
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < total; c += (int64_t)gridDim.x * blockDim.x) {
    const int64_t a = c / J, b = c - a * J;
    for (int q = 0; q < r; ++q) {
      const float v = At[(int64_t)q * lda + a] * Bt[(int64_t)q * ldb + b];
      bf16 h, l;
      tc::split_bf16(v, h, l);
      hi[(int64_t)q * ld_out + c] = h;
      lo[(int64_t)q * ld_out + c] = l;
    }
  }
}

// The same Khatri-Rao product as RANK-CONTIGUOUS bf16 hi/lo planes [I*J x rk] (the "row planes" the fused pass reads its
// factor slabs from): row c = a * J + b holds At[q][a] * Bt[q][b], q < r; ranks r .. rk stay zero.  One thread per row.
__global__ void __launch_bounds__(256) krao_row_planes_kernel(const float* __restrict__ At, int64_t lda, int64_t I, const float* __restrict__ Bt,
                                                              int64_t ldb, int64_t J, int r, int rk, bf16* __restrict__ hi, bf16* __restrict__ lo) {
  const int64_t total = I * J;
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < total; c += (int64_t)gridDim.x * blockDim.x) {
    const int64_t a = c / J, b = c - a * J;
    for (int q0 = 0; q0 < r; q0 += 8) {
      uint32_t hw[4], lw[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int q = q0 + 2 * j;
        const float v0 = q < r ? At[(int64_t)q * lda + a] * Bt[(int64_t)q * ldb + b] : 0.f;
        const float v1 = q + 1 < r ? At[(int64_t)(q + 1) * lda + a] * Bt[(int64_t)(q + 1) * ldb + b] : 0.f;
        const __nv_bfloat162 h = __floats2bfloat162_rn(v0, v1);
        hw[j] = *reinterpret_cast<const uint32_t*>(&h);
        const __nv_bfloat162 l = __floats2bfloat162_rn(v0 - __uint_as_float(hw[j] << 16), v1 - __uint_as_float(hw[j] & 0xffff0000u));
        lw[j] = *reinterpret_cast<const uint32_t*>(&l);
      }
      *reinterpret_cast<uint4*>(hi + c * rk + q0) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
      *reinterpret_cast<uint4*>(lo + c * rk + q0) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
    }
  }
}

}  // namespace

void nnfac_split_planes(const float* in, int64_t ld_in, int64_t rows, int64_t cols, __nv_bfloat16* hi, __nv_bfloat16* lo,
                        int64_t ld_out, int grid, cudaStream_t st) {
  split_planes_kernel<2><<<grid, 256, 0, st>>>(in, ld_in, rows, cols, hi, lo, ld_out, nullptr);
}

void nnfac_split_planes_transposed(const float* in, int64_t ld_in, int64_t rows, int64_t cols, __nv_bfloat16* hiT,
                                   __nv_bfloat16* loT, int64_t ld_out, cudaStream_t st) {
  dim3 g((unsigned)ceil_div64(cols, 32), (unsigned)ceil_div64(rows, 32)), b(32, 8);
  split_planes_transposed_kernel<2><<<g, b, 0, st>>>(in, ld_in, rows, cols, hiT, loT, ld_out, nullptr);
}

void nnfac_reduce_partials(const float* partial, int splits, int r, int r_pad, int64_t R, int64_t ld_partial, float* out,
                           int64_t ld_out, int sm_count, cudaStream_t st) {
  const int64_t total = (int64_t)r * R;
  const int grid = (int)(ceil_div64(total, 256) < (int64_t)sm_count * 8 ? ceil_div64(total, 256) : (int64_t)sm_count * 8);
  reduce_partials_kernel<<<grid, 256, 0, st>>>(partial, splits, r, r_pad, R, ld_partial, out, ld_out);
}

void nnfac_reduce_partials_chunked(const float* partial, int splits, int r, int r_pad, int64_t R, int64_t ld_partial, float* out,
                                   int64_t chunk, int slabs, const float* tail, int64_t ld_tail, int tail_cols, int sm_count,
                                   cudaStream_t st) {
  const int64_t total = (int64_t)slabs * r * (chunk + tail_cols);
  const int grid = (int)(ceil_div64(total, 256) < (int64_t)sm_count * 8 ? ceil_div64(total, 256) : (int64_t)sm_count * 8);
  reduce_partials_chunked_kernel<<<grid, 256, 0, st>>>(partial, splits, r, r_pad, R, ld_partial, out, chunk, chunk + tail_cols,
                                                       (int64_t)r * (chunk + tail_cols), slabs, tail, ld_tail, tail_cols);
}

// every variant of the cross-product kernel: padded rank <= 64 / <= 128 x addressing mode of the X operand (+ the 3-plane one)
template <int AMODE>
static cudaError_t cross_set_smem(int r_pad, size_t smem) {
  return r_pad <= 64 ? cudaFuncSetAttribute(tc_cross_kernel<64, AMODE, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                     : cudaFuncSetAttribute(tc_cross_kernel<128, AMODE, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}
static cudaError_t cross_prepare(const Side* s, int r_pad, int planes) {
  if (planes == 3) return cudaFuncSetAttribute(tc_cross_kernel<64, 0, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->smem);
  return s->cp.amode == 0 ? cross_set_smem<0>(r_pad, s->smem) : s->cp.amode == 1 ? cross_set_smem<1>(r_pad, s->smem) : cross_set_smem<2>(r_pad, s->smem);
}
template <int AMODE>
static void cross_launch_mode(const Side* s, const CrossParams& cp, int r_pad, cudaStream_t st) {
  if (r_pad <= 64)
    tc_cross_kernel<64, AMODE, 2><<<s->grid, NTHREADS, s->smem, st>>>(s->map_xh, s->map_xl, s->map_fh, s->map_fl, cp, s->map_xh, s->map_fh);
  else
    tc_cross_kernel<128, AMODE, 2><<<s->grid, NTHREADS, s->smem, st>>>(s->map_xh, s->map_xl, s->map_fh, s->map_fl, cp, s->map_xh, s->map_fh);
}
static void cross_launch(const Side* s, const CrossParams& cp, int r_pad, int planes, cudaStream_t st) {
  if (planes == 3) tc_cross_kernel<64, 0, 3><<<s->grid, NTHREADS, s->smem, st>>>(s->map_xh, s->map_xl, s->map_fh, s->map_fl, cp, s->map_xm, s->map_fm);
  else if (cp.amode == 0) cross_launch_mode<0>(s, cp, r_pad, st);
  else if (cp.amode == 1) cross_launch_mode<1>(s, cp, r_pad, st);
  else cross_launch_mode<2>(s, cp, r_pad, st);
}

extern "C" {

int nnfac_nmf_plan_destroy(nnfac_nmf_plan* p) {
  if (!p) return NNFAC_OK;
  if (p->owns_buffer) cudaFree(p->buffer);
  free(p);
  return NNFAC_OK;
}

// Every device buffer of a plan is carved out of ONE allocation (256-byte aligned pieces): either the caller's
// workspace (`buffer`, at least nnfac_nmf_plan_bytes() bytes -- e.g. a block of a caching allocator, so that repeated
// factorisations of same-shaped data never reach cudaMalloc / cudaFree) or one cudaMalloc owned by the plan.
static int plan_build(nnfac_ctx* ctx, int64_t m, int64_t n, int r, int sides, int planes, void* buffer, size_t buffer_bytes,
                      cudaStream_t st, nnfac_nmf_plan** out, size_t* bytes_out) {
  NNFAC_ARG(ctx && m > 0 && n > 0 && r > 0 && sides >= 1 && sides <= 3 && (planes == 2 || planes == 3), "nnfac_nmf_plan_create: bad argument");
  if (r > 128) { nnfac_set_error("nnfac_nmf_plan_create: rank %d > 128 is not covered by the tensor-core path", r); return NNFAC_ERR_UNSUPPORTED; }
  if (planes == 3 && r > 64) { nnfac_set_error("nnfac_nmf_plan_create: 3-plane plans cover rank <= 64 (rank %d)", r); return NNFAC_ERR_UNSUPPORTED; }
  if (m >= (1ll << 31) - 256 || n >= (1ll << 31) - 256) { nnfac_set_error("nnfac_nmf_plan_create: dimension too large"); return NNFAC_ERR_UNSUPPORTED; }
  nnfac_nmf_plan* p = (nnfac_nmf_plan*)calloc(1, sizeof(nnfac_nmf_plan));
  if (!p) return NNFAC_ERR_ALLOC;
  p->ctx = ctx; p->m = m; p->n = n; p->r = r;
  p->sides = sides;
  p->planes = planes;
  p->r_pad = (int)round_up(r, 16);
  p->rk = p->r_pad <= 64 ? 64 : 128;
  p->fused_ok = 1;                       // rank <= 128: residual pass; the beta = 1 pass needs rk == 64
  // ---- sizes ----
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
  size_t o_xh[2], o_xl[2], o_fh[2], o_fl[2], o_xm[2], o_fm[2], o_rh[2] = {0, 0}, o_rl[2] = {0, 0}, o_rm[2] = {0, 0}, xb[2], fb[2],
         rb[2] = {0, 0};
  const size_t mid = planes == 3 ? 1 : 0;    // the middle planes exist in 3-plane plans only
  size_t partial_bytes = 0;
  for (int i = 0; i < 2; ++i) {
    Side* s = &p->side[i];
    s->R = i == 0 ? m : n;
    s->C = i == 0 ? n : m;
    s->ld = round_up(s->C, 64);
    xb[i] = (sides >> i) & 1 ? (size_t)s->R * s->ld * sizeof(bf16) : 0;     // an absent side keeps no planes of X
    fb[i] = (size_t)p->r_pad * s->ld * sizeof(bf16);
    o_xh[i] = take(xb[i]); o_xl[i] = take(xb[i]); o_fh[i] = take(fb[i]); o_fl[i] = take(fb[i]);
    o_xm[i] = take(mid * xb[i]); o_fm[i] = take(mid * fb[i]);
    choose_partition(ctx->sm_count, s->R, s->C, p->r_pad, planes, s);
    const size_t pb = (size_t)s->cp.splits * p->r_pad * s->cp.ld_partial * sizeof(float);
    if (((sides >> i) & 1) && pb > partial_bytes) partial_bytes = pb;
  }
  const size_t o_partial = take(partial_bytes);
  if (p->fused_ok)
    for (int i = 0; i < 2; ++i) {
      rb[i] = (size_t)(i == 0 ? m : n) * p->rk * sizeof(bf16);
      o_rh[i] = take(rb[i]); o_rl[i] = take(rb[i]); o_rm[i] = take(mid * rb[i]);
    }
  const size_t o_cost = take(sizeof(double) * 2048);
  if (bytes_out) *bytes_out = off;
  if (!out) { free(p); return NNFAC_OK; }      // size query only
  // ---- memory ----
  if (buffer) {
    if (buffer_bytes < off || ((uintptr_t)buffer & 255)) {
      nnfac_set_error("nnfac_nmf_plan_create_in: workspace of %zu bytes (256-byte aligned) needed, got %zu", off, buffer_bytes);
      free(p);
      return NNFAC_ERR_ARG;
    }
    p->buffer = buffer;
  } else {
    if (cudaMalloc(&p->buffer, off) != cudaSuccess) {
      cudaGetLastError();
      nnfac_set_error("nnfac_nmf_plan_create: out of device memory (%zu bytes)", off);
      free(p);
      return NNFAC_ERR_ALLOC;
    }
    p->owns_buffer = 1;
  }
  p->buffer_bytes = off;
  uint8_t* base = (uint8_t*)p->buffer;
  for (int i = 0; i < 2; ++i) {
    Side* s = &p->side[i];
    s->xh = (bf16*)(base + o_xh[i]); s->xl = (bf16*)(base + o_xl[i]);
    s->fh = (bf16*)(base + o_fh[i]); s->fl = (bf16*)(base + o_fl[i]);
    cudaMemsetAsync(s->fh, 0, fb[i], st);
    cudaMemsetAsync(s->fl, 0, fb[i], st);
    int rc = make_map(&s->map_xh, s->xh, s->R, s->C, s->ld, TILE_ROWS);
    if (!rc) rc = make_map(&s->map_xl, s->xl, s->R, s->C, s->ld, TILE_ROWS);
    if (!rc) rc = make_map(&s->map_fh, s->fh, p->r_pad, s->C, s->ld, p->r_pad);
    if (!rc) rc = make_map(&s->map_fl, s->fl, p->r_pad, s->C, s->ld, p->r_pad);
    if (planes == 3) {
      s->xm = (bf16*)(base + o_xm[i]); s->fm = (bf16*)(base + o_fm[i]);
      cudaMemsetAsync(s->fm, 0, fb[i], st);
      if (!rc) rc = make_map(&s->map_xm, s->xm, s->R, s->C, s->ld, TILE_ROWS);
      if (!rc) rc = make_map(&s->map_fm, s->fm, p->r_pad, s->C, s->ld, p->r_pad);
    }
    if (i == 0 && sides == 1 && planes == 2 && p->rk == 64) {
      if (!rc) rc = make_map(&s->map_kh, s->fh, p->r_pad, s->C, s->ld, 64);
      if (!rc) rc = make_map(&s->map_kl, s->fl, p->r_pad, s->C, s->ld, 64);
    }
    if (rc) { nnfac_nmf_plan_destroy(p); return rc; }
    cudaError_t e = cross_prepare(s, p->r_pad, planes);
    if (e != cudaSuccess) { nnfac_set_error("cudaFuncSetAttribute(smem=%zu): %s", s->smem, cudaGetErrorString(e)); nnfac_nmf_plan_destroy(p); return NNFAC_ERR_CUDA; }
  }
  p->partial = (float*)(base + o_partial);
  p->partial_bytes = partial_bytes;
  // fused passes: row planes of both factors (rank axis contiguous, padded to 64) and per-CTA cost partials
  if (p->fused_ok) {
    for (int i = 0; i < 2; ++i) {
      const int64_t len = i == 0 ? m : n;
      p->rowp_h[i] = (bf16*)(base + o_rh[i]); p->rowp_l[i] = (bf16*)(base + o_rl[i]);
      cudaMemsetAsync(p->rowp_h[i], 0, rb[i], st);
      cudaMemsetAsync(p->rowp_l[i], 0, rb[i], st);
      int rc = make_map(&p->map_row_a_h[i], p->rowp_h[i], len, p->rk, p->rk, TILE_ROWS);
      if (!rc) rc = make_map(&p->map_row_a_l[i], p->rowp_l[i], len, p->rk, p->rk, TILE_ROWS);
      if (!rc) rc = make_map(&p->map_row_b_h[i], p->rowp_h[i], len, p->rk, p->rk, 64);
      if (!rc) rc = make_map(&p->map_row_b_l[i], p->rowp_l[i], len, p->rk, p->rk, 64);
      if (planes == 3) {
        p->rowp_m[i] = (bf16*)(base + o_rm[i]);
        cudaMemsetAsync(p->rowp_m[i], 0, rb[i], st);
        if (!rc) rc = make_map(&p->map_row_a_m[i], p->rowp_m[i], len, p->rk, p->rk, TILE_ROWS);
        if (!rc) rc = make_map(&p->map_row_b_m[i], p->rowp_m[i], len, p->rk, p->rk, 64);
      }
      if (rc) { nnfac_nmf_plan_destroy(p); return rc; }
    }
  }
  p->cost_part = (double*)(base + o_cost);
  cudaMemsetAsync(p->cost_part, 0, sizeof(double) * 2048, st);
  p->sums = p->cost_part + 1024;
  if (cudaGetLastError() != cudaSuccess) { nnfac_set_error("nnfac_nmf_plan_create: clearing the workspace failed"); nnfac_nmf_plan_destroy(p); return NNFAC_ERR_CUDA; }
  *out = p;
  return NNFAC_OK;
}

int nnfac_nmf_plan_create(nnfac_ctx* ctx, int64_t m, int64_t n, int r, nnfac_nmf_plan** out) {
  NNFAC_ARG(out != nullptr, "nnfac_nmf_plan_create: out is NULL");
  return plan_build(ctx, m, n, r, 3, 2, nullptr, 0, (cudaStream_t)0, out, nullptr);
}

int nnfac_nmf_plan_bytes(nnfac_ctx* ctx, int64_t m, int64_t n, int r, size_t* bytes) {
  NNFAC_ARG(bytes != nullptr, "nnfac_nmf_plan_bytes: bytes is NULL");
  return plan_build(ctx, m, n, r, 3, 2, nullptr, 0, (cudaStream_t)0, nullptr, bytes);
}

int nnfac_nmf_plan_create_in(nnfac_ctx* ctx, int64_t m, int64_t n, int r, void* workspace, size_t workspace_bytes,
                             void* stream, nnfac_nmf_plan** out) {
  NNFAC_ARG(out != nullptr && workspace != nullptr, "nnfac_nmf_plan_create_in: NULL argument");
  return plan_build(ctx, m, n, r, 3, 2, workspace, workspace_bytes, (cudaStream_t)stream, out, nullptr);
}

// One-sided plans: sides = 1 keeps only the planes of X (passes over side 0: V X^T, the MTTKRP of an unfolding),
// sides = 2 only those of X^T, 3 both.  A pass over an absent side is refused.
int nnfac_nmf_plan_bytes_sided(nnfac_ctx* ctx, int64_t m, int64_t n, int r, int sides, size_t* bytes) {
  NNFAC_ARG(bytes != nullptr, "nnfac_nmf_plan_bytes_sided: bytes is NULL");
  return plan_build(ctx, m, n, r, sides, 2, nullptr, 0, (cudaStream_t)0, nullptr, bytes);
}

int nnfac_nmf_plan_create_sided(nnfac_ctx* ctx, int64_t m, int64_t n, int r, int sides, void* workspace, size_t workspace_bytes,
                                void* stream, nnfac_nmf_plan** out) {
  NNFAC_ARG(out != nullptr && workspace != nullptr, "nnfac_nmf_plan_create_sided: NULL argument");
  return plan_build(ctx, m, n, r, sides, 2, workspace, workspace_bytes, (cudaStream_t)stream, out, nullptr);
}

// The same with `planes` bf16 planes per value: 2 (as above) or 3 (hi + mid + lo: every fp32 value of X and of the factors
// exactly; rank <= 64).  The plane count is fixed here because the planes are carved from the one workspace.
int nnfac_nmf_plan_bytes_planes(nnfac_ctx* ctx, int64_t m, int64_t n, int r, int sides, int planes, size_t* bytes) {
  NNFAC_ARG(bytes != nullptr, "nnfac_nmf_plan_bytes_planes: bytes is NULL");
  return plan_build(ctx, m, n, r, sides, planes, nullptr, 0, (cudaStream_t)0, nullptr, bytes);
}

int nnfac_nmf_plan_create_planes(nnfac_ctx* ctx, int64_t m, int64_t n, int r, int sides, int planes, void* workspace,
                                 size_t workspace_bytes, void* stream, nnfac_nmf_plan** out) {
  NNFAC_ARG(out != nullptr && workspace != nullptr, "nnfac_nmf_plan_create_planes: NULL argument");
  return plan_build(ctx, m, n, r, sides, planes, workspace, workspace_bytes, (cudaStream_t)stream, out, nullptr);
}

// View plan: the unfolding of another mode of the C-order tensor whose mode-0 unfolding `base` holds (base: I_0 x rest, planes
// without row padding).  The tensor is (left, I, right) with left * I * right = I_0 * rest; the view is the I x (left * right)
// unfolding of the middle axis (ntf.py:309-311 makes a COPY of the tensor for it; here it is a TMA map over the same planes):
//   right == 1 (last mode):   the planes read as [left x I] hold the unfolding transposed -> MN-major operand (amode 1)
//   otherwise (middle modes): 3-D map {right, I, left}, contraction index c = l * right + rr (amode 2; right % 64 == 0)
// A view supports nnfac_nmf_plan_set_krao / _cross(which = 0) / _reduce / _info; its workspace holds the factor planes and the
// split-K partials, and at rank <= 64 also the row planes of factor 0 [I x 64] and the cost partials of the MU passes
// (nnfac_nmf_plan_set_factor_rows / _fused(mode 1) / _fused_beta / _mu_finish_rows).
static int view_build(nnfac_ctx* ctx, const nnfac_nmf_plan* base, int64_t left, int64_t I, int64_t right, int r, void* buffer,
                      size_t buffer_bytes, cudaStream_t st, nnfac_nmf_plan** out, size_t* bytes_out) {
  NNFAC_ARG(ctx && base && left >= 1 && I >= 1 && right >= 1 && r > 0 && r <= 128, "nnfac_nmf_plan_view: bad argument");
  NNFAC_ARG(!base->base && (base->sides & 1), "nnfac_nmf_plan_view: the base plan must own the planes of side 0");
  if (base->planes != 2) { nnfac_set_error("nnfac_nmf_plan_view: views of 3-plane plans are not built"); return NNFAC_ERR_UNSUPPORTED; }
  NNFAC_ARG(left * I * right == base->m * base->n, "nnfac_nmf_plan_view: %lld x %lld x %lld is not the base tensor", (long long)left,
            (long long)I, (long long)right);
  if (left == 1 || base->side[0].ld != base->n || (right == 1 ? (I % 8 != 0) : (right % 64 != 0)) || left * right >= (1ll << 31) - 256) {
    nnfac_set_error("nnfac_nmf_plan_view: this unfolding cannot be addressed in place (mode 0, padded planes, or misaligned extents)");
    return NNFAC_ERR_UNSUPPORTED;
  }
  nnfac_nmf_plan* p = (nnfac_nmf_plan*)calloc(1, sizeof(nnfac_nmf_plan));
  if (!p) return NNFAC_ERR_ALLOC;
  p->ctx = ctx; p->base = base; p->m = I; p->n = left * right; p->r = r; p->sides = 1; p->planes = 2;
  p->r_pad = (int)round_up(r, 16);
  p->rk = p->r_pad <= 64 ? 64 : 128;
  p->fused_ok = p->rk == 64;
  Side* s = &p->side[0];
  s->R = I; s->C = left * right; s->ld = round_up(s->C, 64);
  choose_partition(ctx->sm_count, s->R, s->C, p->r_pad, 2, s);
  s->cp.amode = right == 1 ? 1 : 2;
  s->cp.kb_per_slab = right == 1 ? 1 : (int)(right / 64);
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
  const size_t fb = (size_t)p->r_pad * s->ld * sizeof(bf16);
  const size_t o_fh = take(fb), o_fl = take(fb);
  const size_t partial_bytes = (size_t)s->cp.splits * p->r_pad * s->cp.ld_partial * sizeof(float);
  const size_t o_partial = take(partial_bytes);
  const size_t rb = p->fused_ok ? (size_t)I * p->rk * sizeof(bf16) : 0;
  const size_t o_rh = take(rb), o_rl = take(rb), o_cost = take(p->fused_ok ? sizeof(double) * 1024 : 0);
  if (bytes_out) *bytes_out = off;
  if (!out) { free(p); return NNFAC_OK; }
  if (!buffer || buffer_bytes < off || ((uintptr_t)buffer & 255)) {
    nnfac_set_error("nnfac_nmf_plan_create_view: workspace of %zu bytes (256-byte aligned) needed, got %zu", off, buffer_bytes);
    free(p);
    return NNFAC_ERR_ARG;
  }
  p->buffer = buffer; p->buffer_bytes = off; p->owns_buffer = 0;
  uint8_t* mem = (uint8_t*)buffer;
  s->xh = base->side[0].xh; s->xl = base->side[0].xl;
  s->fh = (bf16*)(mem + o_fh); s->fl = (bf16*)(mem + o_fl);
  p->partial = (float*)(mem + o_partial); p->partial_bytes = partial_bytes;
  cudaMemsetAsync(s->fh, 0, fb, st);
  cudaMemsetAsync(s->fl, 0, fb, st);
  int rc = NNFAC_OK;
  if (p->fused_ok) {
    p->rowp_h[0] = (bf16*)(mem + o_rh); p->rowp_l[0] = (bf16*)(mem + o_rl);
    cudaMemsetAsync(p->rowp_h[0], 0, rb, st);
    cudaMemsetAsync(p->rowp_l[0], 0, rb, st);
    p->cost_part = (double*)(mem + o_cost);
    cudaMemsetAsync(p->cost_part, 0, sizeof(double) * 1024, st);
    p->sums = base->sums;     // sum of X: the same tensor
    rc = make_map(&p->map_row_a_h[0], p->rowp_h[0], I, p->rk, p->rk, TILE_ROWS);
    if (!rc) rc = make_map(&p->map_row_a_l[0], p->rowp_l[0], I, p->rk, p->rk, TILE_ROWS);
    if (!rc) rc = make_map(&s->map_kh, s->fh, p->r_pad, s->C, s->ld, 64);
    if (!rc) rc = make_map(&s->map_kl, s->fl, p->r_pad, s->C, s->ld, 64);
  }
  if (!rc && right == 1) {           // planes as [left x I]: box = 64 contraction rows x 64 output rows
    rc = make_map(&s->map_xh, s->xh, left, I, I, 64);
    if (!rc) rc = make_map(&s->map_xl, s->xl, left, I, I, 64);
  } else if (!rc) {
    rc = make_map_3d(&s->map_xh, s->xh, right, I, left, right, I * right, TILE_ROWS);
    if (!rc) rc = make_map_3d(&s->map_xl, s->xl, right, I, left, right, I * right, TILE_ROWS);
  }
  if (!rc) rc = make_map(&s->map_fh, s->fh, p->r_pad, s->C, s->ld, p->r_pad);
  if (!rc) rc = make_map(&s->map_fl, s->fl, p->r_pad, s->C, s->ld, p->r_pad);
  if (!rc && cross_prepare(s, p->r_pad, 2) != cudaSuccess) { nnfac_set_error("cudaFuncSetAttribute failed for a view plan"); rc = NNFAC_ERR_CUDA; }
  if (!rc && cudaGetLastError() != cudaSuccess) { nnfac_set_error("nnfac_nmf_plan_create_view: clearing the workspace failed"); rc = NNFAC_ERR_CUDA; }
  if (rc) { free(p); return rc; }
  *out = p;
  return NNFAC_OK;
}

int nnfac_nmf_plan_view_bytes(nnfac_ctx* ctx, const nnfac_nmf_plan* base, int64_t left, int64_t I, int64_t right, int r, size_t* bytes) {
  NNFAC_ARG(bytes != nullptr, "nnfac_nmf_plan_view_bytes: bytes is NULL");
  return view_build(ctx, base, left, I, right, r, nullptr, 0, (cudaStream_t)0, nullptr, bytes);
}

int nnfac_nmf_plan_create_view(nnfac_ctx* ctx, const nnfac_nmf_plan* base, int64_t left, int64_t I, int64_t right, int r,
                               void* workspace, size_t workspace_bytes, void* stream, nnfac_nmf_plan** out) {
  NNFAC_ARG(out != nullptr && workspace != nullptr, "nnfac_nmf_plan_create_view: NULL argument");
  return view_build(ctx, base, left, I, right, r, workspace, workspace_bytes, (cudaStream_t)stream, out, nullptr);
}

// Rows [row0, row0 + rows) of X (device fp32, `Xrows` points at row row0): both plane orientations of that slab.
// Lets the host pipeline the upload of X with its ingest (see NMFPlan.load_host in nn_fac/_ops.py).
int nnfac_nmf_plan_load_x_rows(nnfac_nmf_plan* p, const float* Xrows, int64_t ldx, int64_t row0, int64_t rows, void* stream) {
  NNFAC_ARG(p && Xrows && ldx >= p->n && row0 >= 0 && rows > 0 && row0 + rows <= p->m, "nnfac_nmf_plan_load_x_rows: bad argument");
  NNFAC_ARG(!p->base, "nnfac_nmf_plan_load_x_rows: a view plan has no planes of its own");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t total = rows * p->n;
  int grid = (int)(ceil_div64(total, 256) < (int64_t)p->ctx->sm_count * 32 ? ceil_div64(total, 256) : (int64_t)p->ctx->sm_count * 32);
  const Side* s0 = &p->side[0];
  const Side* s1 = &p->side[1];
  if (p->sides & 1) {
    if (p->planes == 3)
      split_planes_kernel<3><<<grid, 256, 0, st>>>(Xrows, ldx, rows, p->n, s0->xh + row0 * s0->ld, s0->xl + row0 * s0->ld, s0->ld,
                                                   s0->xm + row0 * s0->ld);
    else
      split_planes_kernel<2><<<grid, 256, 0, st>>>(Xrows, ldx, rows, p->n, s0->xh + row0 * s0->ld, s0->xl + row0 * s0->ld, s0->ld,
                                                   nullptr);
    NNFAC_LAUNCH_CHECK(p->ctx);
  }
  // grid.y is limited to 65535 blocks of 32 rows: walk the rows in slabs
  const int64_t slab = 65535ll * 32;
  for (int64_t r0 = 0; (p->sides & 2) && r0 < rows; r0 += slab) {
    const int64_t nr = rows - r0 < slab ? rows - r0 : slab;
    dim3 g((unsigned)ceil_div64(p->n, 32), (unsigned)ceil_div64(nr, 32)), b(32, 8);
    if (p->planes == 3)
      split_planes_transposed_kernel<3><<<g, b, 0, st>>>(Xrows + r0 * ldx, ldx, nr, p->n, s1->xh + row0 + r0, s1->xl + row0 + r0,
                                                         s1->ld, s1->xm + row0 + r0);
    else
      split_planes_transposed_kernel<2><<<g, b, 0, st>>>(Xrows + r0 * ldx, ldx, nr, p->n, s1->xh + row0 + r0, s1->xl + row0 + r0,
                                                         s1->ld, nullptr);
    NNFAC_LAUNCH_CHECK(p->ctx);
  }
  return NNFAC_OK;
}

// After the last slab: constants of the data that the passes need (sum of X for the KL cost).
int nnfac_nmf_plan_load_x_done(nnfac_nmf_plan* p, void* stream) {
  NNFAC_ARG(p != nullptr, "nnfac_nmf_plan_load_x_done: plan is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  if (p->fused_ok && (p->sides & 1)) {
    // sum of X as the passes see it (hi + lo (+ mid) planes), fp64, fixed order: the constant term of the KL cost
    const int blocks = p->ctx->sm_count * 4;
    const int grc = nnfac_guard_enter(p->ctx, NNFAC_GUARD_RED, st);
    if (grc) return grc;
    if (p->planes == 3)
      plane_total_kernel<3><<<blocks, 256, 0, st>>>(p->side[0].xh, p->side[0].xl, p->side[0].ld, p->m, p->n, p->ctx->red, p->side[0].xm);
    else
      plane_total_kernel<2><<<blocks, 256, 0, st>>>(p->side[0].xh, p->side[0].xl, p->side[0].ld, p->m, p->n, p->ctx->red, nullptr);
    NNFAC_LAUNCH_CHECK(p->ctx);
    plane_total_finish_kernel<<<1, 32, 0, st>>>(p->ctx->red, blocks, p->sums);
    NNFAC_LAUNCH_CHECK(p->ctx);
  }
  return NNFAC_OK;
}

int nnfac_nmf_plan_load_x(nnfac_nmf_plan* p, const float* X, int64_t ldx, void* stream) {
  NNFAC_ARG(p && X && ldx >= p->n, "nnfac_nmf_plan_load_x: bad argument");
  const int rc = nnfac_nmf_plan_load_x_rows(p, X, ldx, 0, p->m, stream);
  return rc ? rc : nnfac_nmf_plan_load_x_done(p, stream);
}

int nnfac_nmf_plan_cross(nnfac_nmf_plan* p, int which, const float* F, int64_t ldf, float* out, int64_t ld_out,
                         void* stream) {
  NNFAC_ARG(p && (which == 0 || which == 1), "nnfac_nmf_plan_cross: bad argument");
  NNFAC_ARG((p->sides >> which) & 1, "nnfac_nmf_plan_cross: this plan keeps no planes of side %d", which);
  Side* s = &p->side[which];
  NNFAC_ARG((!F || ldf >= s->C) && (!out || ld_out >= s->R), "nnfac_nmf_plan_cross: leading dimension too small");
  cudaStream_t st = (cudaStream_t)stream;
  int grid;
  if (F) {   // F == NULL: the operand planes of the factor installed by nnfac_nmf_plan_set_factor / _mu_finish are current
    const int64_t total = (int64_t)p->r * s->C;
    grid = (int)(ceil_div64(total, 256) < (int64_t)p->ctx->sm_count * 8 ? ceil_div64(total, 256) : (int64_t)p->ctx->sm_count * 8);
    if (p->planes == 3) split_planes_kernel<3><<<grid, 256, 0, st>>>(F, ldf, p->r, s->C, s->fh, s->fl, s->ld, s->fm);
    else split_planes_kernel<2><<<grid, 256, 0, st>>>(F, ldf, p->r, s->C, s->fh, s->fl, s->ld, nullptr);
    NNFAC_LAUNCH_CHECK(p->ctx);
  }
  CrossParams cp = s->cp;
  cp.partial = p->partial;
  cross_launch(s, cp, p->r_pad, p->planes, st);
  NNFAC_LAUNCH_CHECK(p->ctx);
  if (!out) return NNFAC_OK;     // the split-K partials stay in the plan (nnfac_nmf_plan_hals_solve / _reduce)
  const int64_t tot2 = (int64_t)p->r * s->R;
  grid = (int)(ceil_div64(tot2, 256) < (int64_t)p->ctx->sm_count * 8 ? ceil_div64(tot2, 256) : (int64_t)p->ctx->sm_count * 8);
  reduce_partials_kernel<<<grid, 256, 0, st>>>(p->partial, cp.splits, p->r, p->r_pad, s->R, cp.ld_partial, out, ld_out);
  NNFAC_LAUNCH_CHECK(p->ctx);
  return NNFAC_OK;
}

// Install the Khatri-Rao product of two rank-major factors At (r x I) and Bt (r x J) as the r x (I*J) factor of
// nnfac_nmf_plan_cross(which = 0, F = NULL): the MTTKRP operand of ntf.py:448-449, written straight into its bf16 operand
// planes (no fp32 Khatri-Rao matrix, no transpose, no separate split pass).  Requires I * J == n of the plan.
int nnfac_nmf_plan_set_krao(nnfac_nmf_plan* p, const float* At, int64_t lda, int64_t I, const float* Bt, int64_t ldb, int64_t J,
                            void* stream) {
  NNFAC_ARG(p && At && Bt && I > 0 && J > 0 && I * J == p->n && lda >= I && ldb >= J, "nnfac_nmf_plan_set_krao: bad argument");
  if (p->planes != 2) { nnfac_set_error("nnfac_nmf_plan_set_krao: writes two planes, the plan has %d", p->planes); return NNFAC_ERR_UNSUPPORTED; }
  Side* s = &p->side[0];
  const int64_t total = I * J;
  const int grid = (int)(ceil_div64(total, 256) < (int64_t)p->ctx->sm_count * 16 ? ceil_div64(total, 256) : (int64_t)p->ctx->sm_count * 16);
  krao_planes_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(At, lda, I, Bt, ldb, J, p->r, s->fh, s->fl, s->ld);
  NNFAC_LAUNCH_CHECK(p->ctx);
  return NNFAC_OK;
}

// Install the r x (left * right) factor V[q][l * right + rr] = B[l][q][rr] of a C-order fp32 array B (left, r, right) into the
// K-major planes of side 0 that nnfac_nmf_plan_cross(which = 0, F = NULL) and, on one-sided plans and views, the MU passes read
// (where nnfac_nmf_plan_set_krao writes): the operand of an NTD unfolding, B = G x_{j != n} F_j, without its unfolded copy.
int nnfac_nmf_plan_set_operand(nnfac_nmf_plan* p, const float* B, int64_t left, int r, int64_t right, void* stream) {
  NNFAC_ARG(p && B && left > 0 && r > 0 && right > 0, "nnfac_nmf_plan_set_operand: bad argument");
  NNFAC_ARG(p->sides & 1, "nnfac_nmf_plan_set_operand: this plan keeps no planes of side 0");
  if (p->planes != 2) { nnfac_set_error("nnfac_nmf_plan_set_operand: writes two planes, the plan has %d", p->planes); return NNFAC_ERR_UNSUPPORTED; }
  Side* s = &p->side[0];
  NNFAC_ARG(r == p->r && left * right == s->C, "nnfac_nmf_plan_set_operand: (%lld, %d, %lld) is not an operand of this %d x %lld plan",
            (long long)left, r, (long long)right, p->r, (long long)s->C);
  cudaStream_t st = (cudaStream_t)stream;
  if (right == 1) {     // V = B^T, B read as [left x r]: grid.y is limited to 65535 blocks of 32 rows, walk the rows in slabs
    for (int64_t r0 = 0; r0 < left; r0 += 65535ll * 32) {
      const int64_t nr = left - r0 < 65535ll * 32 ? left - r0 : 65535ll * 32;
      dim3 g((unsigned)ceil_div64(r, 32), (unsigned)ceil_div64(nr, 32)), b(32, 8);
      split_planes_transposed_kernel<2><<<g, b, 0, st>>>(B + r0 * r, r, nr, r, s->fh + r0, s->fl + r0, s->ld, nullptr);
      NNFAC_LAUNCH_CHECK(p->ctx);
    }
    return NNFAC_OK;
  }
  const int64_t bx = ceil_div64(s->C, 256) < 1024 ? ceil_div64(s->C, 256) : 1024;
  split_planes_strided_kernel<<<dim3((unsigned)bx, (unsigned)r), 256, 0, st>>>(B, (int)s->C, r, (int)right, s->fh, s->fl, s->ld);
  NNFAC_LAUNCH_CHECK(p->ctx);
  return NNFAC_OK;
}

// The same operand for the FUSED pass over side 0 (nnfac_nmf_plan_fused(plan, 0, 0, ...)): the Khatri-Rao product installed as
// the rank-contiguous planes of factor 1 ("V^T", [n x rk]).  With the mode's own factor installed as factor 0
// (nnfac_nmf_plan_set_factor(plan, 0, F^T)) that pass yields the MTTKRP of ntf.py:449 AND ||unfold(T, mode) - F krao^T||^2, the
// direct residual of the CP model, in one pass over the tensor.
int nnfac_nmf_plan_set_krao_rows(nnfac_nmf_plan* p, const float* At, int64_t lda, int64_t I, const float* Bt, int64_t ldb, int64_t J,
                                 void* stream) {
  NNFAC_ARG(p && At && Bt && I > 0 && J > 0 && I * J == p->n && lda >= I && ldb >= J, "nnfac_nmf_plan_set_krao_rows: bad argument");
  NNFAC_ARG(p->fused_ok && !p->base, "nnfac_nmf_plan_set_krao_rows: the plan has no row planes");
  if (p->planes != 2) { nnfac_set_error("nnfac_nmf_plan_set_krao_rows: writes two planes, the plan has %d", p->planes); return NNFAC_ERR_UNSUPPORTED; }
  const int64_t total = I * J;
  const int grid = (int)(ceil_div64(total, 256) < (int64_t)p->ctx->sm_count * 16 ? ceil_div64(total, 256) : (int64_t)p->ctx->sm_count * 16);
  krao_row_planes_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(At, lda, I, Bt, ldb, J, p->r, p->rk, p->rowp_h[1], p->rowp_l[1]);
  NNFAC_LAUNCH_CHECK(p->ctx);
  return NNFAC_OK;
}

int nnfac_nmf_plan_info(const nnfac_nmf_plan* p, int which, int* splits, int* stages_per_unit, int* num_units,
                        int* num_stages, int* grid) {
  NNFAC_ARG(p && (which == 0 || which == 1), "nnfac_nmf_plan_info: bad argument");
  const Side* s = &p->side[which];
  if (splits) *splits = s->cp.splits;
  if (stages_per_unit) *stages_per_unit = s->cp.stages_per_unit;
  if (num_units) *num_units = s->cp.num_units;
  if (num_stages) *num_stages = s->cp.num_stages;
  if (grid) *grid = s->grid;
  return NNFAC_OK;
}

}  // extern "C"
