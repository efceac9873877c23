// Tensor-core HALS sweep (fp32 path, rank <= 64): blocked Gauss-Seidel that reproduces the exact
// row-by-row recurrence of nn_fac/update_rules/nnls.py:158-170.
//
// Formulation: the kernel keeps the scaled, sparsity-shifted residual  W[k] = (UtM[k] - sp - UtU[k,:] V) / UtU[k,k]
// of every column in a tensor-memory accumulator for the whole call and updates it incrementally.  For a block
// of 16 rows the step of row k is  d_k = max(W[k], -V[k])  (nnls.py:163/167); inside the block the rows see each
// other's steps through 120 FMAs per column whose operands (-UtU[k2,k] / UtU[k2,k2]) come from __constant__
// memory (the same for every column); once the 16 steps of a block are known, ONE rank-16 update
//        W[:, col] -= (UtU / diag)[:, block] d[block]
// runs on tcgen05 ([128 columns x 16] x [16 x 64] per column tile, accumulated into TMEM).  The initial residual
// uses 3-term bf16 splits of V and of the Gram (6 of 9 products: fp32-equivalent).  In the loop the operand of the
// tensor core is the STEP (not V), so rounding is relative to the step and the accumulator error relative to the
// residual: two terms of the step against two of the Gram (3 products) suffice -- the solve stops once the steps have
// shrunk by a factor 10 -- and the result is more accurate than re-forming UtM - UtU V each time.
//
// One thread owns one column of V.  The fp32 masters of V and the residual both live in tensor memory
// (2 x 64 columns per 128-column tile); shared memory only holds the operand planes.  A CTA carries up
// to 4 column tiles (512 update threads) plus one MMA-issuing warp per tile, so issuing never competes
// with the update chain.  The per-sweep stop test (nnls.py:156) is an all-to-all exchange of the CTAs'
// partial sums through tagged 64-bit mailboxes (one L2 hop, no atomics), summed in a fixed order so that
// every CTA takes the same decision; the first three blocks of the next sweep run speculatively meanwhile.
// The final write-out also produces the bf16 operand planes of the result for the NMF plan (optional).
#include <stdlib.h>
#include <type_traits>

#include "common.cuh"
#include "tc_common.cuh"

namespace {

using bf16 = __nv_bfloat16;

#ifndef SWEEP_POSTER4
#define SWEEP_POSTER4 0          // 1: posting warp in the four-tile variant too (672 threads -> 80 registers, spills: 5.39 against 5.15 us per sweep at n = 65536)
#endif
constexpr int BLK = 16;           // rows per Gauss-Seidel block (K extent of the rank update)
constexpr int TILE = 128;         // columns per tile (UMMA M)
constexpr uint32_t PLANE_BYTES = TILE * 64 * sizeof(bf16);   // 16 KiB: one 64-wide K atom of an operand plane of a tile
constexpr int NPLANES = 3;
constexpr int XMAXW = 8;          // ranks of a collective solve (cross-GPU stop scalar)
constexpr int XMAXG = 160;        // board entries per rank (>= CTAs of a solve)

// Per padded rank RP (64 or 128): a tile keeps RP residual + RP master columns in tensor memory, so a CTA carries
// up to 256 / RP tiles; the Gram operand planes are RP / 64 K atoms of [RP rows x 128 B].
// MT = tiles a CTA of this variant carries at most; LAG = the stop test lags one sweep (see the main loop).
template <int RP, int MT, bool LAG>
struct Cfg {
  static_assert(MT * RP <= 256, "512 tensor-memory columns: RP residual + RP master columns per tile");
  static constexpr int NBLK = RP / BLK;
  static constexpr int KR = RP / 64;
  static constexpr int MAX_TILES = MT;
  static constexpr int UPD_THREADS = MAX_TILES * TILE;
  // The partial sums of a sweep are posted by a warp of their own, except in the four-tile variant (rank <= 64, more than
  // 256 columns per CTA: 640 threads already sit at the register limit of the update chain; it keeps the update threads
  // posting after a CTA-wide barrier)
  static constexpr bool POSTER = SWEEP_POSTER4 || !(RP == 64 && MT == 4);
  static constexpr int NTHREADS = UPD_THREADS + MAX_TILES * 32 + (POSTER ? 32 : 0);   // + one issuing warp per tile (+ the posting warp)
  static constexpr int TMEM_PER_TILE = 2 * RP;
  static constexpr uint32_t G_ATOM_BYTES = RP * 128;               // [RP rows x 64 K] bf16
  static constexpr uint32_t G_PLANE_BYTES = KR * G_ATOM_BYTES;     // 8 / 32 KiB
  // blocks of the next sweep that run speculatively while the stop scalar travels: the masters they overwrite are parked in
  // shared memory (blocks 0 .. NSM-1: the idle third operand plane holds two blocks per column, an extra region two more)
  // and in registers (blocks NSM .. NSPEC-1).  Without lag, RP = 64: 3 of 4 blocks (96 of the 102 registers of a 640-thread
  // CTA are taken); RP = 128: 6 of 8.  With lag the WHOLE next sweep is speculative (NSPEC = NBLK): RP = 64 with at most two
  // tiles per CTA (320 threads, 204 registers), RP = 128 with four blocks in shared memory.
  static constexpr int NSPEC = LAG ? NBLK : (RP == 64 ? 3 : 6);
  static constexpr int NSM = (LAG && RP == 128) ? 4 : 2;
  static constexpr uint32_t BK_EXTRA_BYTES = (NSM - 2) * (BLK * 4) * UPD_THREADS;   // 64 B per column and block beyond the first two
  static constexpr size_t SMEM = NPLANES * G_PLANE_BYTES + (size_t)MAX_TILES * NPLANES * PLANE_BYTES + BK_EXTRA_BYTES + 512;
  static constexpr int MBANKS = LAG ? 4 : 2;                       // mailbox / board banks per call (by sweep number)
};

template <int RP>
struct alignas(16) SweepConst {
  float nh[RP / BLK][BLK][BLK]; // [B][e][e2] = -UtU[k2][k] / UtU[k2][k2] (source row k = 16B+e, target row k2 = 16B+e2)
  float invd[RP];               // 1 / UtU[k][k], 0 when the diagonal entry is 0 or k >= r
  int has_zero_diag;            // some row k < r has UtU[k][k] == 0
};
// One bank per padded rank and device.  It is written by a one-block kernel on the stream of the solve, right before the
// solve; solves of one context on different streams are ordered by the context's scratch guard (nnfac_guard_enter).
__constant__ SweepConst<64> c_sw64;
__constant__ SweepConst<128> c_sw128;
template <int RP>
__device__ __forceinline__ const SweepConst<RP>& csw() {
  if constexpr (RP == 64) return c_sw64; else return c_sw128;
}

// Per-call preparation (one block): the constants of the in-block recurrence, and the call generation of the mailbox
// tags.  The generation lives in device memory and is advanced HERE, not on the host, so that a solve captured into a
// CUDA graph gets a fresh generation on every replay (a host-side counter would be frozen into the graph and the tags
// of the previous replay would match).  When the 16-bit generation wraps, the mailboxes are cleared first.
template <int RP>
__global__ void sweep_prep_kernel(const float* __restrict__ G, int64_t ld_g, int r, SweepConst<RP>* out, unsigned* gen,
                                  unsigned long long* mail, size_t mail_count) {
  constexpr int NBLK = RP / BLK;
  __shared__ unsigned next_gen;
  if (threadIdx.x == 0) next_gen = (*gen + 1u) & 0xffffu;
  __syncthreads();
  if (next_gen == 0u) {
    for (size_t i = threadIdx.x; i < mail_count; i += blockDim.x) mail[i] = 0ull;
    __syncthreads();
  }
  if (threadIdx.x == 0) *gen = next_gen == 0u ? 1u : next_gen;
  for (int idx = threadIdx.x; idx < NBLK * BLK * BLK; idx += blockDim.x) {
    const int B = idx / (BLK * BLK), e = (idx / BLK) % BLK, e2 = idx % BLK;
    const int k = B * BLK + e, k2 = B * BLK + e2;
    const float d2 = k2 < r ? G[(int64_t)k2 * ld_g + k2] : 0.f;
    out->nh[B][e][e2] = (k < r && k2 < r && d2 != 0.f && e2 > e) ? -G[(int64_t)k2 * ld_g + k] * (1.f / d2) : 0.f;
  }
  for (int k = threadIdx.x; k < RP; k += blockDim.x) {
    const float d = k < r ? G[(int64_t)k * ld_g + k] : 0.f;
    out->invd[k] = d != 0.f ? 1.f / d : 0.f;
  }
  if (threadIdx.x == 0) {
    int z = 0;
    for (int k = 0; k < r; ++k) z |= (G[(int64_t)k * ld_g + k] == 0.f);
    out->has_zero_diag = z;
  }
}

struct TcSweepArgs {
  const float* b;   // UtM r x n
  const float* G;   // UtU r x r
  const float* Vin; // r x n start values (may alias V)
  float* V;         // r x n result
  int64_t ld_b, ld_g, ld_v, ld_vin, n;
  int nsplit;              // UtM = sum of nsplit slabs b + s * split_stride (split-K partials of an X pass), summed in order
  int64_t split_stride;
  // optional: bf16 hi/lo operand planes of the result for the NMF plan (nnfac_nmf_plan_hals_solve)
  bf16 *fh, *fl;    // [r_pad x ld_plane], K-major (rank rows)
  bf16 *rowh, *rowl;// [n x row_pitch], rank contiguous (may be NULL)
  int64_t ld_plane;
  int r_pad, row_pitch;
  int r, maxiter, cols_per_cta;
  double delta;
  float sp;
  unsigned long long* mail;   // [2][grid][grid] tagged partial sums (tag = generation << 16 | sweep)
  const unsigned* gen;        // call generation (device word, advanced by sweep_prep_kernel): stale mailbox contents of
                              // earlier calls never match
  double* result;
  // Collective solve (several GPUs, one slice of the columns each): the stop test of nnls.py:156 sums the squared steps
  // over ALL columns.  Every CTA posts its partial on the board of every rank (peer-mapped memory, one 8-byte store
  // each over NVLink) and adds up all P x grid partials it finds on its own board, in (rank, CTA) order, so that every
  // CTA of every GPU obtains the same bits (a group of one GPU too).  xworld = 0: not collective, exchange through the private
  // mailboxes above.
  int xworld, xrank;
  unsigned xgen;                              // collective call counter (host side, the same on every rank)
  unsigned long long* xboard[XMAXW];          // [q]: board of rank q as mapped here; [xrank]: the local one
  int xgrid[XMAXW];                           // CTAs of rank q's solve
};

using tc::tmem_st16;
using tc::tmem_st_wait;

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  const __nv_bfloat162 p = __floats2bfloat162_rn(a, b);   // .x = a (low half), .y = b
  return *reinterpret_cast<const uint32_t*>(&p);
}

// Write 8 consecutive K-elements (one 16-byte chunk) of row `row` into the three K-major SW128 planes
// (hi, mid, lo: x = hi + mid + lo exactly for normal fp32 values, i.e. fp32 operands for the tensor core).
// Two values per conversion (cvt.rn.bf16x2.f32); the halves are widened back with a shift / a mask.
__device__ __forceinline__ void store_chunk(uint8_t* plane_hi, int row, int chunk, const float* x, uint32_t plane_stride) {
  uint32_t h[4], m[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float a = x[2 * i], b = x[2 * i + 1];
    h[i] = pack_bf16(a, b);
    const float a1 = a - __uint_as_float(h[i] << 16), b1 = b - __uint_as_float(h[i] & 0xffff0000u);
    m[i] = pack_bf16(a1, b1);
    const float a2 = a1 - __uint_as_float(m[i] << 16), b2 = b1 - __uint_as_float(m[i] & 0xffff0000u);
    l[i] = pack_bf16(a2, b2);
  }
  uint8_t* p = plane_hi + (uint32_t)row * 128u + (uint32_t)((chunk ^ (row & 7)) << 4);
  *reinterpret_cast<uint4*>(p) = make_uint4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<uint4*>(p + plane_stride) = make_uint4(m[0], m[1], m[2], m[3]);
  *reinterpret_cast<uint4*>(p + 2 * plane_stride) = make_uint4(l[0], l[1], l[2], l[3]);
}

// Two-term variant (hi, mid) for the steps: |x - hi - mid| <= 2^-17 |x|.
__device__ __forceinline__ void store_chunk2(uint8_t* plane_hi, int row, int chunk, const float* x, uint32_t plane_stride) {
  uint32_t h[4], m[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float a = x[2 * i], b = x[2 * i + 1];
    h[i] = pack_bf16(a, b);
    m[i] = pack_bf16(a - __uint_as_float(h[i] << 16), b - __uint_as_float(h[i] & 0xffff0000u));
  }
  uint8_t* p = plane_hi + (uint32_t)row * 128u + (uint32_t)((chunk ^ (row & 7)) << 4);
  *reinterpret_cast<uint4*>(p) = make_uint4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<uint4*>(p + plane_stride) = make_uint4(m[0], m[1], m[2], m[3]);
}

__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

using tc::elect_one;

__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// The six partial products of one 16-wide K slice:  acc += (a_hi + a_mid + a_lo) (g_hi + g_mid + g_lo)^T
// without the three terms below 2^-24.  `koff` is the K offset inside the 128-byte swizzled row (>> 4).
// Rank update of one block inside the sweep: the operand is the STEP of the block, whose rounding only has to
// be small against the step itself (the solve stops when the steps have shrunk by a factor 10, nnls.py:156):
// two terms of the step against two terms of the Gram, three products (error 2^-16 of the update).
// `a_hi` / `g_hi`: descriptors of the hi planes, already advanced to the 16-wide K slice; AP / GP: plane pitches (>> 4).
__device__ __forceinline__ void issue_step_update(uint64_t a_hi, uint64_t g_hi, uint32_t d, uint32_t idesc, uint64_t GP) {
  constexpr uint64_t AP = PLANE_BYTES >> 4;
  tc::umma_bf16(d, a_hi, g_hi, idesc, true);
  tc::umma_bf16(d, a_hi, g_hi + GP, idesc, true);
  tc::umma_bf16(d, a_hi + AP, g_hi, idesc, true);
}

__device__ __forceinline__ void issue_kslice(uint64_t a_hi, uint64_t g_hi, uint32_t d, uint32_t idesc, uint64_t GP) {
  constexpr uint64_t AP = PLANE_BYTES >> 4;
  tc::umma_bf16(d, a_hi, g_hi, idesc, true);
  tc::umma_bf16(d, a_hi, g_hi + GP, idesc, true);
  tc::umma_bf16(d, a_hi + AP, g_hi, idesc, true);
  tc::umma_bf16(d, a_hi, g_hi + 2 * GP, idesc, true);
  tc::umma_bf16(d, a_hi + AP, g_hi + GP, idesc, true);
  tc::umma_bf16(d, a_hi + 2 * AP, g_hi, idesc, true);
}

// compile-time loop over the blocks of a sweep
template <int B, int N>
struct BlockLoop {
  template <class F>
  static __device__ __forceinline__ void run(F& f) {
    f(std::integral_constant<int, B>{});
    BlockLoop<B + 1, N>::run(f);
  }
};
template <int N>
struct BlockLoop<N, N> {
  template <class F>
  static __device__ __forceinline__ void run(F&) {}
};

template <int RP, int MT, bool LAG>
__global__ void __launch_bounds__(Cfg<RP, MT, LAG>::NTHREADS, 1) tc_sweep_kernel(const TcSweepArgs a) {
  using C = Cfg<RP, MT, LAG>;
  constexpr int MAX_TILES = C::MAX_TILES, UPD_THREADS = C::UPD_THREADS, TMEM_PER_TILE = C::TMEM_PER_TILE, KR = C::KR;
  constexpr uint32_t G_PLANE_BYTES = C::G_PLANE_BYTES, G_ATOM_BYTES = C::G_ATOM_BYTES;
  constexpr uint64_t GP = G_PLANE_BYTES >> 4;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* g_planes = smem;                                            // -UtU / diag: hi | mid | lo, [K atom][row j][128 B]
  uint8_t* v_planes = smem + NPLANES * G_PLANE_BYTES;                  // [tile][hi|mid|lo][16 KiB]
  uint8_t* bk_extra = v_planes + (size_t)MAX_TILES * NPLANES * PLANE_BYTES;   // parked masters of blocks 2 .. NSM-1 (LAG, RP = 128)
  uint8_t* tail = bk_extra + C::BK_EXTRA_BYTES;
  uint64_t* s_full = reinterpret_cast<uint64_t*>(tail);                // [MAX_TILES] MMA batch complete
  uint64_t* s_ready = s_full + MAX_TILES;                              // [MAX_TILES] operand planes of a tile rewritten
  float* redf = reinterpret_cast<float*>(s_ready + MAX_TILES);         // [48]: per-warp partials of a post (2 x 16, by parity), of a collect (16)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(redf + 48);
  volatile uint32_t* s_done = tmem_slot + 1;                            // [MAX_TILES]
  volatile uint32_t* s_quit = s_done + MAX_TILES;                       // the solve has ended: the posting warp leaves
  volatile uint32_t* s_posted = s_quit + 1;                             // posts the posting warp has completed

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = a.r;
  const int nblk = (r + BLK - 1) / BLK;
  const int64_t cta_col0 = (int64_t)blockIdx.x * a.cols_per_cta;
  int64_t cta_cols = a.n - cta_col0;
  if (cta_cols > a.cols_per_cta) cta_cols = a.cols_per_cta;
  const int ntiles = (int)((cta_cols + TILE - 1) / TILE);

  if (warp == 0) {
    if (lane == 0) {
      for (int t = 0; t < MAX_TILES; ++t) {
        tc::mbar_init(&s_full[t], 1);
        tc::mbar_init(&s_ready[t], TILE);
      }
      for (int t = 0; t < MAX_TILES; ++t) s_done[t] = 0;
      *s_quit = 0;
      *s_posted = 0;
      tc::fence_barrier_init();
    }
    __syncwarp();
    tc::tmem_alloc(tmem_slot, 512);
  }
  // Operand planes of -UtU[j][:] / UtU[j][j] (K-major, 128B swizzle): row j = output row of the rank update, K = source
  // row.  With the rows scaled by the diagonal the accumulator holds the SCALED residual, i.e. the unclamped step.
  if (threadIdx.x < UPD_THREADS) {
    for (int idx = threadIdx.x; idx < RP * (RP / 8); idx += UPD_THREADS) {
      const int j = idx / (RP / 8), c = idx % (RP / 8);                // row j, 16-byte chunk c = source rows 8c .. 8c+7
      const float dj = j < r ? a.G[(int64_t)j * a.ld_g + j] : 0.f;
      const float sj = dj != 0.f ? -1.f / dj : 0.f;
      float x[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int l = c * 8 + i;
        x[i] = (j < r && l < r) ? a.G[(int64_t)j * a.ld_g + l] * sj : 0.f;
      }
      store_chunk(g_planes + (c >> 3) * G_ATOM_BYTES, j, c & 7, x, G_PLANE_BYTES);
    }
  }
  tc::fence_proxy_async_smem();
  tc::tcgen05_fence_before();
  __syncthreads();
  tc::tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t idesc = tc::umma_idesc_bf16(TILE, RP);
  const uint64_t g_desc = tc::umma_desc_k_sw128(tc::smem_u32(g_planes));

  // ------------------------------------------------------------------------------------------------
  // MMA-issuing warps: one per tile.  Every arrival of the tile's 128 update threads on s_ready hands
  // over one operand set: first V (initial residual; one 64-row K atom per hand-over), then one 16-row
  // block of steps each.
  // ------------------------------------------------------------------------------------------------
  if (C::POSTER && warp == UPD_THREADS / 32 + MAX_TILES) {
    // ----------------------------------------------------------------------------------------------
    // Posting warp: after every sweep the update warps leave their partial sums of squared steps in shared memory and
    // ARRIVE on named barrier 2 without waiting; this warp adds them up in a fixed order and posts the CTA's partial sum
    // to every CTA (mailboxes) or, in a collective solve, to the board of every rank (one 8-byte sys-scope store each
    // over NVLink).  Stores to peer memory can hold the issuing warp for the better part of a microsecond: on a warp of
    // its own they no longer sit on the update chain (nor does the CTA-wide barrier the update warps used to wait on).
    // ----------------------------------------------------------------------------------------------
    constexpr unsigned MB = C::MBANKS;
    const unsigned nb = gridDim.x;
    const unsigned gen = *a.gen;
    const bool collective = a.xworld > 0;
    for (unsigned e = 0;; ++e) {
      named_bar_sync(2, UPD_THREADS + 32);
      if (*s_quit) break;
      float sum = 0.f;
#pragma unroll
      for (int w = 0; w < UPD_THREADS / 32; ++w) sum += redf[(e & 1u) * 16 + w];
      const unsigned tag = collective ? ((a.xgen & 0xffffu) << 16) | (e + 1u) : (gen << 16) | (e + 1u);
      const unsigned long long bits = ((unsigned long long)tag << 32) | __float_as_uint(sum);
      if (collective) {
        // 8 banks of XMAXW x XMAXG entries, bank = 4 (call parity) + sweep number mod MBANKS, so that a rank that is ahead
        // (by up to a sweep, with LAG by up to three, or by the start of the next call) never overwrites an entry a slower
        // rank still has to read
        const size_t xbank = (size_t)((a.xgen & 1u) * 4u + (e % MB)) * (XMAXW * XMAXG);
        if (lane < a.xworld) st_relaxed_sys_u64(a.xboard[lane] + xbank + (size_t)a.xrank * XMAXG + blockIdx.x, bits);
      } else if (nb > 1) {
        for (unsigned t = lane; t < nb; t += 32) st_relaxed_u64(a.mail + ((size_t)(e % MB) * nb + t) * nb + blockIdx.x, bits);
      }
      __syncwarp();
      if (lane == 0) *s_posted = e + 1u;
    }
  } else if (warp >= UPD_THREADS / 32) {
    // warp-uniform by construction (shuffle), so that descriptors live in uniform registers
    const int tile = __shfl_sync(0xffffffffu, warp, 0) - UPD_THREADS / 32;
    if (tile < ntiles) {
      const uint64_t a_desc = tc::umma_desc_k_sw128(tc::smem_u32(v_planes + (size_t)tile * NPLANES * PLANE_BYTES));
      const uint32_t d = tmem_base + (uint32_t)(tile * TMEM_PER_TILE);
      uint32_t phase = 0;
      for (int kr = 0; kr < KR; ++kr) {
        if (kr * 4 >= nblk) break;
        tc::mbar_wait(&s_ready[tile], phase);
        phase ^= 1;
        tc::tcgen05_fence_after();
        if (elect_one()) {
          for (int ks = 0; ks < 4 && kr * 4 + ks < nblk; ++ks)
            issue_kslice(a_desc + (uint64_t)(ks * 2), g_desc + (uint64_t)(kr * (G_ATOM_BYTES >> 4) + ks * 2), d, idesc, GP);
          tc::umma_commit(&s_full[tile]);
        }
        __syncwarp();
      }
      for (int B = 0;; B = (B + 1 < nblk) ? B + 1 : 0) {
        tc::mbar_wait(&s_ready[tile], phase);
        phase ^= 1;
        if (s_done[tile]) break;
        tc::tcgen05_fence_after();
        if (elect_one()) {
          issue_step_update(a_desc + (uint64_t)((B & 3) * 2), g_desc + (uint64_t)((B >> 2) * (G_ATOM_BYTES >> 4) + (B & 3) * 2), d, idesc, GP);
          tc::umma_commit(&s_full[tile]);
        }
        __syncwarp();
      }
    }
  } else {
    // ----------------------------------------------------------------------------------------------
    // Update threads: one per column; 4 warps (= 128 TMEM lanes) per tile.
    // ----------------------------------------------------------------------------------------------
    const int tile = warp >> 2, q = warp & 3;
    const bool active = tile < ntiles;
    const int row = q * 32 + lane;                                       // row of the A tile == TMEM lane
    const int64_t col = cta_col0 + (int64_t)tile * TILE + row;
    const bool valid = active && (int64_t)tile * TILE + row < cta_cols;
    uint8_t* vh = v_planes + (size_t)tile * NPLANES * PLANE_BYTES;
    const uint32_t t_w = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(tile * TMEM_PER_TILE);
    const uint32_t t_v = t_w + RP;
    uint32_t s_phase = 0;

    if (active) {
      // UtM - sp -> residual accumulator, for ALL rank rows before the first hand-over (the products of the first K atom
      // already add -UtU[:, atom] V[atom] into every one of the RP residual columns)
#pragma unroll
      for (int c0 = 0; c0 < RP; c0 += 16) {
        uint32_t w[16];
        if (c0 < nblk * BLK) {
          // right-hand side: 16 independent loads in flight per slab (a loop over the slabs INSIDE the row loop serialises
          // them: measured +0.07 ms per solve); the slabs of split-K partials are added in order, like the reduction kernel
          float bv[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) bv[j] = (valid && c0 + j < r) ? a.b[(int64_t)(c0 + j) * a.ld_b + col] : 0.f;
          for (int sp = 1; sp < a.nsplit; ++sp) {
            float t[16];
#pragma unroll
            for (int j = 0; j < 16; ++j)
              t[j] = (valid && c0 + j < r) ? a.b[(int64_t)sp * a.split_stride + (int64_t)(c0 + j) * a.ld_b + col] : 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) bv[j] += t[j];
          }
#pragma unroll
          for (int j = 0; j < 16; ++j) w[j] = __float_as_uint((valid && c0 + j < r) ? (bv[j] - a.sp) * csw<RP>().invd[c0 + j] : 0.f);
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) w[j] = 0u;
        }
        tmem_st16(t_w + c0, w);
      }
      // V -> TMEM masters and operand planes, one 64-row K atom per hand-over (the issuer adds -UtU[:, atom] V[atom])
#pragma unroll
      for (int kr = 0; kr < KR; ++kr) {
        if (kr * 4 < nblk) {
          if (kr > 0) {                                                  // the planes are reused: the products of the previous
            tc::mbar_wait(&s_full[tile], s_phase);                       // K atom must have retired
            s_phase ^= 1;
          }
#pragma unroll
          for (int c1 = 0; c1 < 64; c1 += 16) {
            const int c0 = kr * 64 + c1;
            float x[16];
            uint32_t w[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) x[j] = (valid && c0 + j < r) ? a.Vin[(int64_t)(c0 + j) * a.ld_vin + col] : 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) w[j] = __float_as_uint(csw<RP>().invd[c0 + j] != 0.f ? x[j] : 0.f);   // skipped rows: master 0
            tmem_st16(t_v + c0, w);
            store_chunk(vh, row, c1 / 8, &x[0], PLANE_BYTES);
            store_chunk(vh, row, c1 / 8 + 1, &x[8], PLANE_BYTES);
          }
          tmem_st_wait();
          tc::fence_proxy_async_smem();
          tc::tcgen05_fence_before();
          tc::mbar_arrive(&s_ready[tile]);
        } else {
          uint32_t z[16];                                                // rank rows beyond the last block: masters are zero
#pragma unroll
          for (int j = 0; j < 16; ++j) z[j] = 0u;
#pragma unroll
          for (int c1 = 0; c1 < 64; c1 += 16) tmem_st16(t_v + kr * 64 + c1, z);
          tmem_st_wait();
        }
      }
    }

    uint8_t* bkrow = vh + 2 * PLANE_BYTES + (uint32_t)row * 128u;       // 128 B: masters of up to 2 speculative blocks
    uint8_t* bkrow2 = bk_extra + (uint32_t)(tile * TILE + row) * (uint32_t)((C::NSM - 2) * BLK * 4);   // blocks 2 .. NSM-1
    (void)bkrow2;
#ifdef SWEEP_PROF
    long long prof[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#define PROF_T(i) { const long long t__ = clock64(); prof[i] += t__ - tp; tp = t__; }
#define PROF_START long long tp = clock64();
#else
#define PROF_T(i)
#define PROF_START
#endif
    // One Gauss-Seidel block (16 rows) of this thread's column: wait for the rank update that precedes it,
    // run the in-block recurrence, write the new masters and the operand planes of the 16 steps and hand
    // them to the issuing warp.  Returns the squared step of the block (nnls.py:170).  `keep` receives the
    // masters the block overwrote (needed to undo a speculative block).
    constexpr int NSM = C::NSM;
    uint32_t bkreg[C::NSPEC - NSM][BLK];                                // masters the speculative blocks NSM .. NSPEC-1 overwrote
    auto block_update = [&](auto Bc, auto Backup) -> float {
      constexpr int B = decltype(Bc)::value;
      constexpr bool BACKUP = decltype(Backup)::value;
      float nd = 0.f;
      PROF_START
      uint32_t wb[BLK], keep[BLK];
      tc::tmem_ld16(t_v + B * BLK, keep);                              // masters: do not wait for the MMA
      tc::mbar_wait(&s_full[tile], s_phase);
      s_phase ^= 1;
      tc::tcgen05_fence_after();
      PROF_T(0)
      tc::tmem_ld16(t_w + B * BLK, wb);
      tc::tmem_ld_wait();
      if (BACKUP && B < 2) {
        // speculative block: the masters it overwrites go to this thread's row of the (now unused) third operand plane
#pragma unroll
        for (int c = 0; c < 4; ++c)
          *reinterpret_cast<uint4*>(bkrow + (((B * 4 + c) ^ (row & 7)) << 4)) = make_uint4(keep[4 * c], keep[4 * c + 1], keep[4 * c + 2], keep[4 * c + 3]);
      }
      if (BACKUP && B >= 2 && B < NSM) {                               // NSM = 4: 128 B per column in the extra region, same swizzle
#pragma unroll
        for (int c = 0; c < 4; ++c)
          *reinterpret_cast<uint4*>(bkrow2 + ((((B - 2) * 4 + c) ^ (row & 7)) << 4)) = make_uint4(keep[4 * c], keep[4 * c + 1], keep[4 * c + 2], keep[4 * c + 3]);
      }
      if (BACKUP && B >= NSM && B < C::NSPEC) {                        // ... the others' stay in registers
#pragma unroll
        for (int e = 0; e < BLK; ++e) bkreg[B >= NSM && B < C::NSPEC ? B - NSM : 0][e] = keep[e];
      }
      float u[BLK];
#pragma unroll
      for (int e = 0; e < BLK; ++e) u[e] = __uint_as_float(wb[e]);
      PROF_T(1)
      // In-block Gauss-Seidel recurrence (nnls.py:158-170) on the scaled residuals: the step of row k is
      // max(u, -V[k]) and every later row of the block sees it through -UtU[k2][k] / UtU[k2][k2].
      float dd[BLK];
      uint32_t vn[BLK];
#ifdef SWEEP_SCALAR_FMA
#pragma unroll
      for (int e = 0; e < BLK; ++e) {
        const float cur = __uint_as_float(keep[e]);
        const float d = fmaxf(u[e], -cur);
        if (e + 1 < BLK) u[e + 1] = fmaf(csw<RP>().nh[B][e][e + 1], d, u[e + 1]);
        dd[e] = d;
        vn[e] = __float_as_uint(cur + d);
        nd = fmaf(d, d, nd);                                           // nnls.py:170
#pragma unroll
        for (int e2 = e + 2; e2 < BLK; ++e2) u[e2] = fmaf(csw<RP>().nh[B][e][e2], d, u[e2]);
      }
#else
      // the same recurrence with the off-chain updates on PACKED fp32 pairs (FFMA2): rows (e2, e2 + 1), e2 even, take
      // u[e2 .. e2+1] += nh[B][e][e2 .. e2+1] * (d, d) in one instruction; the update of the NEXT row stays scalar and
      // first, it is the dependent chain.  Same products and sums as the scalar form, element for element.
#pragma unroll
      for (int e = 0; e < BLK; ++e) {
        const float cur = __uint_as_float(keep[e]);
        // nnls.py:163/167.  A skipped row (zero diagonal, nnls.py:160) has u = 0 and a master of 0 (its true value only
        // enters the initial residual and is left untouched in memory), so its step is max(0, -0) = 0.
        const float d = fmaxf(u[e], -cur);
        if (e + 1 < BLK) u[e + 1] = fmaf(csw<RP>().nh[B][e][e + 1], d, u[e + 1]);
        dd[e] = d;
        vn[e] = __float_as_uint(cur + d);
        nd = fmaf(d, d, nd);                                           // nnls.py:170
        const float2 d2 = make_float2(d, d);
        constexpr int dummy = 0; (void)dummy;
        if (((e + 2) & 1) && e + 2 < BLK) u[e + 2] = fmaf(csw<RP>().nh[B][e][e + 2], d, u[e + 2]);
#pragma unroll
        for (int e2 = (e + 2 + 1) & ~1; e2 + 1 < BLK; e2 += 2) {
          const float2 c2 = *reinterpret_cast<const float2*>(&csw<RP>().nh[B][e][e2]);
          const float2 r2 = __ffma2_rn(c2, d2, make_float2(u[e2], u[e2 + 1]));
          u[e2] = r2.x; u[e2 + 1] = r2.y;
        }
      }
#endif
      PROF_T(2)
      tmem_st16(t_v + B * BLK, vn);
      store_chunk2(vh, row, 2 * (B & 3), &dd[0], PLANE_BYTES);
      store_chunk2(vh, row, 2 * (B & 3) + 1, &dd[8], PLANE_BYTES);
      PROF_T(3)
      tc::fence_proxy_async_smem();
      tmem_st_wait();
      tc::tcgen05_fence_before();
      tc::mbar_arrive(&s_ready[tile]);
      PROF_T(4)
      return nd;
    };

    float thr = 0.f, epsf = 1.f;
    int cnt = 1;
    unsigned epoch = 0;
    const unsigned nb = gridDim.x;
    const unsigned gen = *a.gen;
    const bool collective = a.xworld > 0;
    // Stop test of nnls.py:156: it needs the sum of squared steps over ALL columns after every sweep.  Every CTA posts
    // its partial into the mailbox of every CTA (one 64-bit store each, tag | value) and adds the partials it receives
    // in a fixed order, so that all CTAs obtain the same bits and take the same decision.  While the partials travel,
    // the first blocks of the coming sweep are run SPECULATIVELY (the masters they overwrite are kept aside), which
    // hides the L2 round trip; if the test ends the solve they are undone.
    constexpr int NSPEC = C::NSPEC;
    int nspec = 0;                                                        // speculative blocks of the current sweep already done
    float nd_spec = 0.f;
    std::integral_constant<bool, false> plain;
    std::integral_constant<bool, true> backup;
    constexpr unsigned MBANKS = C::MBANKS;
    // hand the squared steps of this warp's columns in sweep e + 1 to the posting warp (no wait: the barrier is only arrived on)
    // (fp32 trees: every CTA adds the same numbers in the same order)
    unsigned nposts = 0;
    auto post = [&](float nd, unsigned e) {
      const float t = warp_sum_f(nd);
      ++nposts;
      if constexpr (C::POSTER) {
        if (lane == 0) {
          // the posting warp has long finished post e - 1 (a sweep ago); waiting for it makes the double-buffered slots and the
          // one-phase-at-a-time use of the named barrier safe by construction
          while (*s_posted < e) {}
          redf[(e & 1u) * 16 + warp] = t;
        }
        __syncwarp();
        asm volatile("bar.arrive 2, %0;" ::"n"(UPD_THREADS + 32) : "memory");
      } else {
        // no posting warp: CTA-wide barrier, then the first threads post (one store each)
        if (lane == 0) redf[(e & 1u) * 16 + warp] = t;
        named_bar_sync(1, UPD_THREADS);
        const unsigned tag = collective ? ((a.xgen & 0xffffu) << 16) | (e + 1u) : (gen << 16) | (e + 1u);
        if (collective ? threadIdx.x < (unsigned)a.xworld : (nb > 1 && threadIdx.x < nb)) {
          float sum = 0.f;
#pragma unroll
          for (int w = 0; w < UPD_THREADS / 32; ++w) sum += redf[(e & 1u) * 16 + w];
          const unsigned long long bits = ((unsigned long long)tag << 32) | __float_as_uint(sum);
          if (collective)
            st_relaxed_sys_u64(a.xboard[threadIdx.x] + (size_t)((a.xgen & 1u) * 4u + (e % MBANKS)) * (XMAXW * XMAXG) + (size_t)a.xrank * XMAXG + blockIdx.x, bits);
          else
            st_relaxed_u64(a.mail + ((size_t)(e % MBANKS) * nb + threadIdx.x) * nb + blockIdx.x, bits);
        }
      }
    };
    const bool poller = !collective && nb > 1 && threadIdx.x < nb;
    auto slot_of = [&](unsigned e) { return a.mail + ((size_t)(e % MBANKS) * nb + blockIdx.x) * nb + threadIdx.x; };
    // collective solves: the entries of the local board this thread adds up (entries t, t + UPD_THREADS, ... rank-major)
    constexpr int MAXE = (XMAXW * XMAXG + UPD_THREADS - 1) / UPD_THREADS;
    bool want[MAXE];
#pragma unroll
    for (int j = 0; j < MAXE; ++j) {
      const int en = threadIdx.x + j * UPD_THREADS;
      const int qr = en / XMAXG, c = en - qr * XMAXG;
      want[j] = collective && en < a.xworld * XMAXG && c < a.xgrid[qr < XMAXW ? qr : 0];
    }
    auto board_of = [&](unsigned e) { return a.xboard[a.xrank] + (size_t)((a.xgen & 1u) * 4u + (e % MBANKS)) * (XMAXW * XMAXG); };
    // a first look at the partial sums of sweep e + 1 (issued under the last speculative block: the L2 round trip of the
    // loads runs under that block)
    unsigned long long early_x[MAXE];
    auto peek = [&](unsigned e, unsigned long long& early) {
      if (poller) early = ld_relaxed_u64(slot_of(e));
      if (collective) {
        const unsigned long long* board = board_of(e);
#pragma unroll
        for (int j = 0; j < MAXE; ++j) early_x[j] = want[j] ? ld_relaxed_sys_u64(board + threadIdx.x + j * UPD_THREADS) : 0ull;
      }
    };
    // the total of sweep e + 1 over all CTAs (and ranks); `early` / early_x: the first look taken by peek(e), if `peeked`
    auto collect = [&](unsigned e, unsigned long long early, bool peeked) -> float {
#ifdef SWEEP_PROF
      const long long tg0 = clock64();
#endif
      const unsigned tag = collective ? ((a.xgen & 0xffffu) << 16) | (e + 1u) : (gen << 16) | (e + 1u);
      float totf = 0.f;
      if (collective) {
        // every entry of the local board, then the usual trees.  All loads of a thread are issued before the first one is
        // looked at (independent L2 round trips), then only the entries that had not arrived yet are polled again
        float got = 0.f;
        const unsigned long long* board = board_of(e);
        unsigned long long bits[MAXE];
#pragma unroll
        for (int j = 0; j < MAXE; ++j) bits[j] = peeked ? early_x[j] : (want[j] ? ld_relaxed_sys_u64(board + threadIdx.x + j * UPD_THREADS) : 0ull);
#pragma unroll
        for (int j = 0; j < MAXE; ++j) {
          if (want[j]) {
            uint32_t spins = 0;
            while ((unsigned)(bits[j] >> 32) != tag) {
              bits[j] = ld_relaxed_sys_u64(board + threadIdx.x + j * UPD_THREADS);
              if (++spins > (1u << 26)) __trap();
            }
            got += __uint_as_float((unsigned)bits[j]);
          }
        }
        got = warp_sum_f(got);
        if (lane == 0) redf[32 + warp] = got;
        named_bar_sync(1, UPD_THREADS);
#pragma unroll
        for (int w = 0; w < UPD_THREADS / 32; ++w) totf += redf[32 + w];
      } else if (nb > 1) {
        float got = 0.f;
        if (poller) {
          const unsigned long long* slot = slot_of(e);
          unsigned long long bits = peeked ? early : ld_relaxed_u64(slot);
          uint32_t spins = 0;
          while ((unsigned)(bits >> 32) != tag) {
            bits = ld_relaxed_u64(slot);
            if (++spins > (1u << 24)) __trap();
          }
          got = __uint_as_float((unsigned)bits);
        }
        got = warp_sum_f(got);
        if (lane == 0) redf[32 + warp] = got;
        named_bar_sync(1, UPD_THREADS);
#pragma unroll
        for (int w = 0; w < UPD_THREADS / 32; ++w) totf += redf[32 + w];
      } else {
        if (C::POSTER) named_bar_sync(1, UPD_THREADS);                  // one CTA, no exchange: the partials of post e are all there
#pragma unroll
        for (int w = 0; w < UPD_THREADS / 32; ++w) totf += redf[(e & 1u) * 16 + w];
      }
#ifdef SWEEP_PROF
      prof[6] += clock64() - tg0;
#endif
      return totf;
    };
    // nnls.py:156 after a sweep whose total squared step is totf; returns true when the solve ends
    auto decide = [&](float totf) -> bool {
      if (cnt == 1) {
        // eps >= delta * eps0 (nnls.py:156, evaluated in double) <=> totf >= thr with thr = delta * eps0 rounded UP to
        // fp32: the per-sweep test then needs no FP64 instruction (scarce on this part)
        const double thr_d = a.delta * (double)totf;
        thr = (float)thr_d;
        if ((double)thr < thr_d) thr = __uint_as_float(__float_as_uint(thr) + 1u);   // thr_d >= 0: next float up
      }
      epsf = totf;
      ++cnt;
      bool stop = !(epsf >= thr && cnt <= a.maxiter);
      if (totf == 0.f) {
        // every further sweep is a no-op.  nnls.py:156 keeps looping on `0 >= delta * 0` only when the FIRST sweep already
        // moved nothing (eps0 == 0): then it burns all maxiter sweeps and returns cnt = maxiter + 1; otherwise
        // 0 >= delta * eps0 is false and the loop ends with the current count.
        if (thr == 0.f && cnt < a.maxiter + 1) cnt = a.maxiter + 1;
        stop = true;
      }
      return stop;
    };
    if constexpr (LAG) {
      // Stop test with a LAG of one sweep: the partial sums of sweep k are posted, then the WHOLE sweep k + 1 runs
      // speculatively (every master it overwrites is parked) and is posted too, and only then is the total of sweep k
      // collected -- it has been travelling for a full sweep, so neither the L2 nor an NVLink round trip (collective solves)
      // is waited for.  If the test ends the solve after sweep k, sweep k + 1 is undone (one wasted sweep per solve).  Posts
      // are not gated by collects here: a CTA can be up to three sweeps ahead of the slowest reader, hence four banks.
      // The host never takes this variant for a single CTA outside a collective solve (nothing to wait for there).
      float nd = 0.f;
      if (active) {
        auto body = [&](auto Bc) {
          constexpr int B = decltype(Bc)::value;
          if (B < nblk) nd += block_update(Bc, plain);
        };
        BlockLoop<0, C::NBLK>::run(body);
      }
      post(nd, 0u);
      while (true) {
        // here: sweeps 1 .. cnt are done and posted, the totals up to sweep cnt - 1 are known (epoch = cnt - 1)
        unsigned long long early = 0ull;
        nspec = 0;
        if (cnt + 1 <= a.maxiter) {
          nspec = nblk;
          float nd2 = 0.f;
          auto spec = [&](auto Bc) {
            constexpr int B = decltype(Bc)::value;
            if (B < nblk) {
              if (B == nblk - 1) peek(epoch, early);                                  // first look, under the last block
              if (active) nd2 += block_update(Bc, backup);
            }
          };
          BlockLoop<0, C::NBLK>::run(spec);
          post(nd2, epoch + 1u);
        }
        const float totf = collect(epoch, early, nspec > 0);
        ++epoch;
        if (decide(totf)) break;
      }
    } else {
    while (true) {
      float nd = nd_spec;
      if (active) {
        auto body = [&](auto Bc) {
          constexpr int B = decltype(Bc)::value;
          if (B < nblk && B >= nspec) nd += block_update(Bc, plain);
        };
        BlockLoop<0, C::NBLK>::run(body);
      }
      post(nd, epoch);
      // ---- speculative blocks of the next sweep; the first look into the mailbox is issued before the last of them,
      //      so that its L2 round trip runs under that block ----
      unsigned long long early = 0ull;
      nspec = 0;
      nd_spec = 0.f;
      if (cnt + 1 <= a.maxiter) {
        nspec = nblk < NSPEC ? nblk : NSPEC;
        auto spec = [&](auto Bc) {
          constexpr int B = decltype(Bc)::value;
          if (B < nspec) {
            if (B == nspec - 1) peek(epoch, early);                                  // first look, under the last speculative block
            if (active) nd_spec += block_update(Bc, backup);
          }
        };
        BlockLoop<0, NSPEC>::run(spec);
      }
      // ---- collect the total ----
      const float totf = collect(epoch, early, nspec > 0);
      ++epoch;
      if (decide(totf)) break;
    }
    }
    if constexpr (C::POSTER) {
      if (lane == 0) {
        while (*s_posted < nposts) {}                                     // every post has been made: the barrier is between phases
        if (threadIdx.x == 0) *s_quit = 1;                                // releases the posting warp
      }
      __syncwarp();
      asm volatile("bar.arrive 2, %0;" ::"n"(UPD_THREADS + 32) : "memory");
    }
    if (active) {
      tc::mbar_wait(&s_full[tile], s_phase);                              // drain the last rank update
      tc::tcgen05_fence_after();
      if (lane == 0 && q == 0) s_done[tile] = 1;
      __threadfence_block();
      tc::mbar_arrive(&s_ready[tile]);                                    // releases the issuing warp
    }
    if (active) {                                                         // tcgen05.ld is warp-collective: no per-lane branch around it
#pragma unroll
      for (int c0 = 0; c0 < RP; c0 += 16) {
        if (c0 < nblk * BLK) {
          uint32_t w[16];
          tc::tmem_ld16(t_v + c0, w);
          tc::tmem_ld_wait();
          if (c0 / BLK >= NSM && c0 / BLK < NSPEC && c0 / BLK < nspec) {      // undo the speculative blocks
#pragma unroll
            for (int e = 0; e < BLK; ++e) w[e] = bkreg[c0 / BLK >= NSM && c0 / BLK < NSPEC ? c0 / BLK - NSM : 0][e];
          } else if (c0 / BLK >= 2 && c0 / BLK < NSM && c0 / BLK < nspec) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const uint4 b4 = *reinterpret_cast<const uint4*>(bkrow2 + ((((c0 / BLK - 2) * 4 + c) ^ (row & 7)) << 4));
              w[4 * c] = b4.x; w[4 * c + 1] = b4.y; w[4 * c + 2] = b4.z; w[4 * c + 3] = b4.w;
            }
          } else if (c0 / BLK < 2 && c0 / BLK < nspec) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const uint4 b4 = *reinterpret_cast<const uint4*>(bkrow + ((((c0 / BLK) * 4 + c) ^ (row & 7)) << 4));
              w[4 * c] = b4.x; w[4 * c + 1] = b4.y; w[4 * c + 2] = b4.z; w[4 * c + 3] = b4.w;
            }
          }
          float x[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            x[j] = __uint_as_float(w[j]);
            // a skipped row (zero diagonal) keeps its start value (its master was a placeholder 0)
            if (csw<RP>().has_zero_diag && valid && c0 + j < r && csw<RP>().invd[c0 + j] == 0.f) x[j] = a.Vin[(int64_t)(c0 + j) * a.ld_vin + col];
            if (valid && c0 + j < r) a.V[(int64_t)(c0 + j) * a.ld_v + col] = x[j];
          }
          if (a.fh != nullptr) {
            // operand planes of the new factor, straight from the registers (replaces a separate pass over the factor)
            uint32_t hw[8], lw[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float p0 = (valid && c0 + 2 * j < r) ? x[2 * j] : 0.f, p1 = (valid && c0 + 2 * j + 1 < r) ? x[2 * j + 1] : 0.f;
              hw[j] = pack_bf16(p0, p1);
              lw[j] = pack_bf16(p0 - __uint_as_float(hw[j] << 16), p1 - __uint_as_float(hw[j] & 0xffff0000u));
            }
            if (valid) {
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                if (c0 + j < a.r_pad) {
                  const uint32_t h = (j & 1) ? (hw[j >> 1] >> 16) : (hw[j >> 1] & 0xffffu), l = (j & 1) ? (lw[j >> 1] >> 16) : (lw[j >> 1] & 0xffffu);
                  reinterpret_cast<unsigned short*>(a.fh)[(int64_t)(c0 + j) * a.ld_plane + col] = (unsigned short)h;
                  reinterpret_cast<unsigned short*>(a.fl)[(int64_t)(c0 + j) * a.ld_plane + col] = (unsigned short)l;
                }
              }
              if (a.rowh != nullptr) {
                uint4* rh = reinterpret_cast<uint4*>(a.rowh + col * a.row_pitch + c0);
                uint4* rl = reinterpret_cast<uint4*>(a.rowl + col * a.row_pitch + c0);
                rh[0] = make_uint4(hw[0], hw[1], hw[2], hw[3]); rh[1] = make_uint4(hw[4], hw[5], hw[6], hw[7]);
                rl[0] = make_uint4(lw[0], lw[1], lw[2], lw[3]); rl[1] = make_uint4(lw[4], lw[5], lw[6], lw[7]);
              }
            }
          }
        }
      }
    }
#ifdef SWEEP_PROF
    if (blockIdx.x == 1 && (threadIdx.x == 0 || threadIdx.x == 32)) {
      printf("sweep prof (cycles/sweep) thr %d: mma_wait %lld tmem_ld %lld chain %lld split_store %lld fence_arrive %lld grid %lld\n",
             threadIdx.x, prof[0] / (cnt - 1), prof[1] / (cnt - 1), prof[2] / (cnt - 1), prof[3] / (cnt - 1), prof[4] / (cnt - 1),
             prof[6] / (cnt - 1));
    }
#endif
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      a.result[0] = (double)epsf;
      a.result[1] = (double)cnt;
      a.result[2] = -1.0;
      a.result[3] = (double)(cnt - 1);
    }
  }
  tc::tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem_base, 512);
}

}  // namespace

template <int RP, int MT, bool LAG>
static int sweep_launch(nnfac_ctx* ctx, TcSweepArgs& a, const float* UtU, int64_t ld_utu, int64_t grid, cudaStream_t st) {
  using C = Cfg<RP, MT, LAG>;
  // the per-call constants are written straight into the __constant__ bank of this device by a one-block kernel (constant
  // caches are invalidated at kernel boundaries, and the stream orders it before the sweep); the bank address is resolved
  // once per context, i.e. per device
  void*& bank = ctx->sweep_const[RP == 64 ? 0 : 1];
  if (!bank) {
    if (RP == 64) NNFAC_CUDA(cudaGetSymbolAddress(&bank, c_sw64));
    else NNFAC_CUDA(cudaGetSymbolAddress(&bank, c_sw128));
  }
  unsigned* gen_dev = reinterpret_cast<unsigned*>(ctx->mail + ctx->mail_count);
  sweep_prep_kernel<RP><<<1, 256, 0, st>>>(UtU, ld_utu, a.r, (SweepConst<RP>*)bank, gen_dev, ctx->mail, ctx->mail_count);
  NNFAC_LAUNCH_CHECK(ctx);
  a.mail = ctx->mail; a.gen = gen_dev;
  NNFAC_CUDA(cudaFuncSetAttribute(tc_sweep_kernel<RP, MT, LAG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
  // every CTA waits for every other one once per sweep: the cooperative launch guarantees that all of them are resident
  // (a plain launch was measured: no difference in launch cost)
  void* params[] = {&a};
  NNFAC_CUDA(cudaLaunchCooperativeKernel((const void*)tc_sweep_kernel<RP, MT, LAG>, dim3((unsigned)grid), dim3(C::NTHREADS), params, C::SMEM, st));
  ctx->launches++;
  return NNFAC_OK;
}

// Returns NNFAC_ERR_UNSUPPORTED (without setting an error) when the shape is outside this kernel's
// envelope, so that the caller can use the FMA kernel instead.  `planes` (optional) receives the bf16 operand planes
// of the result (see TcSweepArgs); Vin may alias V.
int nnfac_tc_sweep_run(nnfac_ctx* ctx, const float* UtM, int64_t ld_utm, const float* UtU, int64_t ld_utu, const float* Vin,
                       int64_t ld_vin, float* V, int64_t ld_v, int r, int64_t n, int maxiter, double delta, double sparsity,
                       double* result, const nnfac_sweep_planes* planes, cudaStream_t st, int nsplit, int64_t split_stride) {
  if (r > 128 || maxiter < 1 || n < 1) return NNFAC_ERR_UNSUPPORTED;
  const int rp = r <= 64 ? 64 : 128;
  const int max_cols = (256 / rp) * TILE;                  // columns a CTA can keep in tensor memory
  int64_t cols = ceil_div64(n, ctx->sm_count);
  cols = ceil_div64(cols, 32) * 32;
  if (const char* force = getenv("NNFAC_SWEEP_COLS")) {   // experiment switch: columns per CTA (multiple of 32)
    const int64_t f = atoll(force);
    if (f >= 32 && f % 32 == 0 && f > cols) cols = f;
  }
  const nnfac_peer_group* pg = ctx->collective ? &ctx->peers : nullptr;
  if (pg) {
    // collective solve: every rank must take the same kernel; the widest slice decides whether the shape fits
    int64_t widest = n;
    for (int q = 0; q < pg->world; ++q) if (ctx->collective_n[q] > widest) widest = ctx->collective_n[q];
    int64_t wc = ceil_div64(ceil_div64(widest, ctx->sm_count), 32) * 32;
    if (wc > max_cols) { nnfac_set_error("collective HALS solve: a slice of %lld columns at rank %d exceeds the tensor-core sweep", (long long)widest, r); return NNFAC_ERR_UNSUPPORTED; }
  }
  if (cols > max_cols) return NNFAC_ERR_UNSUPPORTED;
  const int64_t grid = ceil_div64(n, cols);
  if ((size_t)(4 * grid * grid) > ctx->mail_count || maxiter > 65000 || grid > XMAXG) return NNFAC_ERR_UNSUPPORTED;
  int rc = nnfac_guard_enter(ctx, NNFAC_GUARD_SWEEP, st);
  if (rc) return rc;
  TcSweepArgs a;
  a.b = UtM; a.G = UtU; a.Vin = Vin; a.V = V; a.ld_b = ld_utm; a.ld_g = ld_utu; a.ld_v = ld_v; a.ld_vin = ld_vin; a.n = n;
  a.r = r; a.maxiter = maxiter; a.cols_per_cta = (int)cols; a.delta = delta; a.sp = (float)sparsity;
  a.nsplit = nsplit > 0 ? nsplit : 1; a.split_stride = split_stride;
  a.fh = a.fl = a.rowh = a.rowl = nullptr; a.ld_plane = 0; a.r_pad = 0; a.row_pitch = 64;
  if (planes) {
    a.fh = (bf16*)planes->fh; a.fl = (bf16*)planes->fl; a.rowh = (bf16*)planes->rowh; a.rowl = (bf16*)planes->rowl;
    a.ld_plane = planes->ld_plane; a.r_pad = planes->r_pad; a.row_pitch = planes->row_pitch;
  }
  a.result = result;
  a.xworld = 0; a.xrank = 0; a.xgen = 0;
  for (int q = 0; q < XMAXW; ++q) { a.xboard[q] = nullptr; a.xgrid[q] = 0; }
  if (pg) {
    a.xworld = pg->world; a.xrank = pg->rank; a.xgen = ++ctx->collective_gen;
    for (int q = 0; q < pg->world; ++q) {
      a.xboard[q] = (unsigned long long*)pg->board[q];
      const int64_t nq = ctx->collective_n[q];
      int64_t cq = ceil_div64(ceil_div64(nq, ctx->sm_count), 32) * 32;
      a.xgrid[q] = nq > 0 ? (int)ceil_div64(nq, cq) : 0;
    }
    if (a.xgrid[pg->rank] != (int)grid) { nnfac_set_error("collective HALS solve: slice length %lld does not match the announced one", (long long)n); return NNFAC_ERR_ARG; }
  }
  // mailbox tags carry a call generation (device-side, see sweep_prep_kernel), so that the slots never need clearing
  // Variant.  The lagged stop test (whole next sweep speculative) needs room to park every master (rank <= 64: at most two
  // tiles per CTA) and something to wait for (more than one CTA, or a collective solve).  Measured with the posting warp
  // (tools/time_sweeps_lag.py, tools/time_sweeps_collective.py; us per sweep, plain -> lagged; results bit-identical on one
  // GPU): collective solves on 2 GPUs, rank 64: 5.20 -> 3.63 (8192 columns per rank, one tile per CTA), 5.04 -> 3.57 (4096),
  // 4.48 -> 4.34 (32768, two tiles); rank 128: 8.59 -> 8.15 -- the lagged variant runs a collective solve at the per-sweep
  // cost of a single-GPU solve (3.50 / 8.24), the NVLink round trip is off the chain.  One GPU: 3.50 -> 3.47 at one tile
  // per CTA on 128 CTAs (3.42 -> 3.14 before the posting warp existed), no gain with two tiles per CTA or a handful of
  // CTAs.  So "auto" takes it for every collective solve and for single-GPU solves with one tile per CTA on at least 64
  // CTAs.  Every rank of a collective solve takes the same variant: the widest slice decides.
  // NNFAC_SWEEP_LAG / nnfac_ctx_sweep_variant: 0 never, 1 auto, 2 wherever possible.
  static const int lag_env = [] { const char* e = getenv("NNFAC_SWEEP_LAG"); return e ? atoi(e) : 1; }();
  const int lag_mode = ctx->sweep_lag >= 0 ? ctx->sweep_lag : lag_env;     // nnfac_ctx_sweep_variant overrides the environment
  int64_t decide_cols = cols;
  if (pg) {
    int64_t widest = n;
    for (int q = 0; q < pg->world; ++q) if (ctx->collective_n[q] > widest) widest = ctx->collective_n[q];
    decide_cols = ceil_div64(ceil_div64(widest, ctx->sm_count), 32) * 32;
  }
  const bool lag_possible = (pg != nullptr || grid > 1) && (rp == 128 || decide_cols <= 2 * TILE);
  const bool lag_pays = pg != nullptr || (decide_cols <= TILE && grid >= 64);
  const bool lag = lag_possible && (lag_mode >= 2 || (lag_mode == 1 && lag_pays));
  if (rp == 64) {
    if (lag) rc = sweep_launch<64, 2, true>(ctx, a, UtU, ld_utu, grid, st);
    else if (decide_cols <= 2 * TILE) rc = sweep_launch<64, 2, false>(ctx, a, UtU, ld_utu, grid, st);
    else rc = sweep_launch<64, 4, false>(ctx, a, UtU, ld_utu, grid, st);
  } else {
    rc = lag ? sweep_launch<128, 2, true>(ctx, a, UtU, ld_utu, grid, st) : sweep_launch<128, 2, false>(ctx, a, UtU, ld_utu, grid, st);
  }
  return rc;
}

int nnfac_tc_sweep_try(nnfac_ctx* ctx, const float* UtM, int64_t ld_utm, const float* UtU, int64_t ld_utu, float* V,
                       int64_t ld_v, int r, int64_t n, int maxiter, double delta, double sparsity, double* result,
                       cudaStream_t st) {
  return nnfac_tc_sweep_run(ctx, UtM, ld_utm, UtU, ld_utu, V, ld_v, V, ld_v, r, n, maxiter, delta, sparsity, result, nullptr, st, 1, 0);
}
