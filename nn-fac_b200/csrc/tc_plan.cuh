// Shared declarations of the NMF plan (tensor-core path): X planes, factor planes, TMA maps, work partition.
#pragma once
#include "common.cuh"
#include "tc_common.cuh"

namespace tcplan {

using bf16 = __nv_bfloat16;

constexpr int TILE_ROWS = 128;   // UMMA M
constexpr int BK = 64;           // bf16 elements per 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int NTHREADS = 256;    // warp0 TMA, warp1 MMA, warp2 TMEM alloc, warps 4-7 epilogue

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// 2-D bf16 row-major [rows x cols] (leading dimension ld elements), box = box_rows x 64, 128B swizzle.
inline int make_map(CUtensorMap* map, const bf16* base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { nnfac_set_error("cuTensorMapEncodeTiled is not available from the driver"); return NNFAC_ERR_CUDA; }
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)ld * sizeof(bf16)};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult rc = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)base, gdim, gstr, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) { nnfac_set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)rc); return NNFAC_ERR_CUDA; }
  return NNFAC_OK;
}

// 3-D bf16 tensor [d2][d1][d0] (d0 contiguous; pitches p1, p2 in elements), box = 1 x box_rows x 64, 128B swizzle: the unfolding
// of a MIDDLE mode of a C-order tensor without a copy (d0 = trailing modes, d1 = the mode, d2 = leading modes).
inline int make_map_3d(CUtensorMap* map, const bf16* base, int64_t d0, int64_t d1, int64_t d2, int64_t p1, int64_t p2, int box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { nnfac_set_error("cuTensorMapEncodeTiled is not available from the driver"); return NNFAC_ERR_CUDA; }
  cuuint64_t gdim[3] = {(cuuint64_t)d0, (cuuint64_t)d1, (cuuint64_t)d2};
  cuuint64_t gstr[2] = {(cuuint64_t)p1 * sizeof(bf16), (cuuint64_t)p2 * sizeof(bf16)};
  cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)box_rows, 1u};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult rc = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, (void*)base, gdim, gstr, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) { nnfac_set_error("cuTensorMapEncodeTiled(3d) failed with CUresult %d", (int)rc); return NNFAC_ERR_CUDA; }
  return NNFAC_OK;
}

// 2-D fp32 row-major [rows x cols], box = 128 rows x 32 columns (128 bytes), 128B swizzle.
inline int make_map_f32(CUtensorMap* map, const float* base, int64_t rows, int64_t cols, int64_t ld) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { nnfac_set_error("cuTensorMapEncodeTiled is not available from the driver"); return NNFAC_ERR_CUDA; }
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)ld * sizeof(float)};
  cuuint32_t box[2] = {32u, (cuuint32_t)TILE_ROWS};
  cuuint32_t estr[2] = {1, 1};
  CUresult rc = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstr, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) { nnfac_set_error("cuTensorMapEncodeTiled(f32) failed with CUresult %d", (int)rc); return NNFAC_ERR_CUDA; }
  return NNFAC_OK;
}

// ---- the cross-product kernel --------------------------------------------------------------------
struct CrossParams {
  int r_pad;            // UMMA N (multiple of 16)
  int splits;           // S: contraction ranges per row tile
  int stages_per_unit;  // 64-wide k-blocks per unit
  int num_units;        // row_tiles * splits
  int num_stages;       // smem ring depth
  int drain;            // stages per TMEM accumulation chain (the tensor core accumulates with truncation)
  int amode;            // how the X operand of this side is addressed (see tc_cross_kernel): 0 rows K-major (2-D map);
                        // 1 MN-major: the planes hold X^T, rows = contraction index, output rows contiguous (last mode of a
                        // tensor); 2 rows K-major through a 3-D map, contraction index = (slab, position in slab) (middle modes)
  int kb_per_slab;      // amode 2: 64-wide k-blocks per slab
  int tiles;            // row tiles
  int split_major;      // unit u = split * tiles + tile instead of tile * splits + split: concurrent CTAs then share the factor
                        // columns of one split (the factor planes are re-read per tile; beyond the L2 size that order decides
                        // whether they come from L2 or from HBM)
  int64_t ld_partial;   // row pitch of the partial buffer (multiple of 128)
  float* partial;       // [splits][r_pad][ld_partial]
};

struct Side {           // one orientation of X
  int64_t R, C, ld;     // plane is [R x C], leading dimension ld
  bf16 *xh, *xl;        // X planes
  bf16 *fh, *fl;        // factor planes [r_pad x ld]
  bf16 *xm, *fm;        // 3-plane plans: the middle planes (x = xh + xm + xl); NULL otherwise
  CUtensorMap map_xh, map_xl, map_fh, map_fl, map_xm, map_fm;
  CUtensorMap map_kh, map_kl;   // side 0 of a one-sided plan or view of rank <= 64: fh / fl in 64 x 64 boxes (Khatri-Rao operand of
                                // the NTF MU pass; ranks beyond r_pad read as zeros)
  CrossParams cp;
  int grid;
  size_t smem;
};

}  // namespace tcplan

struct nnfac_nmf_plan {
  nnfac_ctx* ctx;
  int64_t m, n;
  int r, r_pad;
  tcplan::Side side[2];         // [0]: planes of X (m x n), used for V X^T;  [1]: planes of X^T (n x m), used for U^T X
  float* partial;
  size_t partial_bytes;
  // fused passes: factor "row planes" with the rank axis contiguous, padded to rk = 64 (rank <= 64) or 128:
  //   rowp[0] = U [m x rk], rowp[1] = V^T [n x rk]; map_row_a: 128-row boxes (A operand of the model GEMM, rk = 64 only),
  //   map_row_b: boxes of 64 rows x 64 ranks (B operand of the model GEMM)
  int rk;
  __nv_bfloat16 *rowp_h[2], *rowp_l[2], *rowp_m[2];
  CUtensorMap map_row_a_h[2], map_row_a_l[2], map_row_b_h[2], map_row_b_l[2], map_row_a_m[2], map_row_b_m[2];
  // bf16 planes per value, fixed at creation: 2 (hi + lo, 16 significant bits) or 3 (hi + mid + lo, the fp32 value
  // itself; rank <= 64; products of six MMAs).  Writers that only know two planes refuse a 3-plane plan.
  int planes;
  double* cost_part;    // [1024] per-CTA cost partials of a fused pass ([512 + i]: second partial of CTA i)
  double* sums;         // cost_part + 1024: [0] sum of X (as stored in the planes)
  int fused_ok;
  const nnfac_nmf_plan* base;   // view plans (nnfac_nmf_plan_create_view): the X planes belong to this plan
  int sides;            // bit i: the planes of side i exist (one-sided plans: the MTTKRP of a tensor unfolding only reads side 0)
  void* buffer;         // the one device allocation every pointer above points into
  size_t buffer_bytes;
  int owns_buffer;      // 0: caller's workspace (nnfac_nmf_plan_create_in)
  // optional fp32 copies of X (= hi + lo) in both orientations: the beta = 1 fused pass never needs X as a tensor-core
  // operand, only in registers, and reads it 3 instructions per element cheaper from fp32 (nnfac_nmf_plan_enable_f32)
  float* xf[2];
  CUtensorMap map_xf[2];
  int xf_ready;
  // column-sharded path, U side: the fused pass over side 0 writes its split partials straight into the INBOX of the rank
  // that owns those rows of U (peer-mapped memory, nnfac_nmf_plan_set_push): [source rank][split][r_pad][push_chunk]
  float* push[NNFAC_MAX_PEERS];
  int64_t push_chunk;   // rows of U per rank (multiple of 128); 0: off
  int push_src, push_world;
};


// helpers shared between tc_nmf.cu and tc_fused.cu (defined in tc_nmf.cu)
void nnfac_split_planes(const float* in, int64_t ld_in, int64_t rows, int64_t cols, __nv_bfloat16* hi, __nv_bfloat16* lo,
                        int64_t ld_out, int grid, cudaStream_t st);
void nnfac_split_planes_transposed(const float* in, int64_t ld_in, int64_t rows, int64_t cols, __nv_bfloat16* hiT,
                                   __nv_bfloat16* loT, int64_t ld_out, cudaStream_t st);
void nnfac_reduce_partials(const float* partial, int splits, int r, int r_pad, int64_t R, int64_t ld_partial, float* out,
                           int64_t ld_out, int sm_count, cudaStream_t st);
void nnfac_reduce_partials_chunked(const float* partial, int splits, int r, int r_pad, int64_t R, int64_t ld_partial, float* out,
                                   int64_t chunk, int slabs, const float* tail, int64_t ld_tail, int tail_cols, int sm_count,
                                   cudaStream_t st);
