// C-ABI entry of the HALS NNLS solver; dispatches on dtype and padded rank.
#include "hals_sweep.cuh"
#include <stdlib.h>
#include <string.h>

#define DECL(tag, T, rp) int nnfac_sweep_##tag##_##rp(nnfac_ctx*, hals::SweepArgs<T>, cudaStream_t);
DECL(f32, float, 16) DECL(f32, float, 32) DECL(f32, float, 64) DECL(f32, float, 128)
DECL(f64, double, 16) DECL(f64, double, 32) DECL(f64, double, 64) DECL(f64, double, 128)
#undef DECL

int nnfac_tc_sweep_try(nnfac_ctx* ctx, const float* UtM, int64_t ld_utm, const float* UtU, int64_t ld_utu, float* V,
                       int64_t ld_v, int r, int64_t n, int maxiter, double delta, double sparsity, double* result,
                       cudaStream_t st);
// any rank, any number of columns, every option (csrc/hals_general.cu): the fallback behind the specialised kernels
int nnfac_sweep_general(nnfac_ctx* ctx, int dtype, const void* UtM, int64_t ld_utm, const void* UtU, int64_t ld_utu, void* V,
                        int64_t ld_v, int r, int64_t n, int maxiter, double delta, double sparsity, unsigned flags, double* result,
                        cudaStream_t st);

void nnfac_reduce_partials(const float* partial, int splits, int r, int r_pad, int64_t R, int64_t ld_partial, float* out,
                           int64_t ld_out, int sm_count, cudaStream_t st);       // csrc/tc_nmf.cu

namespace {
template <typename T>
hals::SweepArgs<T> make_args(const void* UtM, int64_t ld_utm, const void* UtU, int64_t ld_utu, void* V,
                             int64_t ld_v, int r, int64_t n, int maxiter, double delta, double sparsity,
                             unsigned flags, double* result) {
  hals::SweepArgs<T> a;
  a.b = (const T*)UtM; a.G = (const T*)UtU; a.V = (T*)V;
  a.ld_b = ld_utm; a.ld_g = ld_utu; a.ld_v = ld_v; a.n = n;
  a.r = r; a.maxiter = maxiter; a.delta = delta; a.sp = (T)sparsity; a.flags = flags;
  a.nbatch = 1; a.slab_ld = 0; a.part = nullptr; a.counter = nullptr; a.result = result;
  return a;
}
}  // namespace

extern "C" int nnfac_hals_nnls(nnfac_ctx* ctx, int dtype, const void* UtM, int64_t ld_utm,
                               const void* UtU, int64_t ld_utu, void* V, int64_t ld_v, int r,
                               int64_t n, int maxiter, double delta, double sparsity, unsigned flags,
                               double* result, void* stream) {
  NNFAC_ARG(ctx && UtM && UtU && V && result, "nnfac_hals_nnls: NULL argument");
  NNFAC_ARG(r > 0 && n > 0, "nnfac_hals_nnls: empty problem (r=%d, n=%lld)", r, (long long)n);
  NNFAC_ARG(ld_utm >= n && ld_v >= n && ld_utu >= r, "nnfac_hals_nnls: leading dimension too small");
  NNFAC_ARG(dtype == NNFAC_F32 || dtype == NNFAC_F64, "nnfac_hals_nnls: bad dtype %d", dtype);
  NNFAC_ARG(maxiter >= 0, "nnfac_hals_nnls: negative maxiter");
  cudaStream_t st = (cudaStream_t)stream;
  static const bool force_general = getenv("NNFAC_SWEEP") && !strcmp(getenv("NNFAC_SWEEP"), "general");
  if (r > 128 || force_general)       // beyond the specialised kernels (the reference has no rank limit)
    return nnfac_sweep_general(ctx, dtype, UtM, ld_utm, UtU, ld_utu, V, ld_v, r, n, maxiter, delta, sparsity, flags, result, st);
  const int rp = r <= 16 ? 16 : r <= 32 ? 32 : r <= 64 ? 64 : 128;
  if (dtype == NNFAC_F32 && flags == 0) {   // (NNFAC_HALS_NO_TC makes flags != 0: no tensor-core sweep)
    // tensor-core blocked sweep when the shape fits (rank <= 64, n <= 512 columns per SM); NNFAC_SWEEP=fma disables it
    static const bool force_fma = getenv("NNFAC_SWEEP") && !strcmp(getenv("NNFAC_SWEEP"), "fma");
    if (!force_fma) {
      const int rc = nnfac_tc_sweep_try(ctx, (const float*)UtM, ld_utm, (const float*)UtU, ld_utu, (float*)V, ld_v, r, n,
                                        maxiter, delta, sparsity, result, st);
      if (rc != NNFAC_ERR_UNSUPPORTED) return rc;
    }
  }
  int rc;
  if (dtype == NNFAC_F32) {
    auto a = make_args<float>(UtM, ld_utm, UtU, ld_utu, V, ld_v, r, n, maxiter, delta, sparsity, flags, result);
    switch (rp) {
      case 16: rc = nnfac_sweep_f32_16(ctx, a, st); break;
      case 32: rc = nnfac_sweep_f32_32(ctx, a, st); break;
      case 64: rc = nnfac_sweep_f32_64(ctx, a, st); break;
      default: rc = nnfac_sweep_f32_128(ctx, a, st); break;
    }
  } else {
    auto a = make_args<double>(UtM, ld_utm, UtU, ld_utu, V, ld_v, r, n, maxiter, delta, sparsity, flags, result);
    switch (rp) {
      case 16: rc = nnfac_sweep_f64_16(ctx, a, st); break;
      case 32: rc = nnfac_sweep_f64_32(ctx, a, st); break;
      case 64: rc = nnfac_sweep_f64_64(ctx, a, st); break;
      default: rc = nnfac_sweep_f64_128(ctx, a, st); break;
    }
  }
  // outside the register-resident kernel's envelope (row-wise options on more columns than it keeps resident, ...): the
  // general sweep takes anything
  if (rc == NNFAC_ERR_UNSUPPORTED)
    rc = nnfac_sweep_general(ctx, dtype, UtM, ld_utm, UtU, ld_utu, V, ld_v, r, n, maxiter, delta, sparsity, flags, result, st);
  return rc;
}

// Out-of-place fp32 solve: Vout (r x n) = hals_nnls_acc(UtM, UtU, Vin) with Vin untouched (the copy of nnls.py:147 happens
// inside the kernel: the tensor-core sweep reads its start values from Vin and writes the result to Vout).  Used for the
// slice solves of the sharded path, whose input is a strided view of the full factor and whose output is the contiguous
// send buffer of the all-gather.  Shapes outside the tensor-core sweep: a strided copy, then the in-place solver.
//
// nnfac_hals_solve_slabs_f32: the right-hand side is the sum of `nslabs` slabs UtM + s * slab_stride ([>= r rows x ld_utm] each:
// split-K partials of an X pass, or the inbox the peers' fused passes pushed their partials into), added up in slab order by the
// solve itself.  Shapes outside the tensor-core sweep: the slabs are first summed into `scratch` (r x n floats, caller's).
extern "C" int nnfac_hals_solve_slabs_f32(nnfac_ctx* ctx, const float* UtM, int64_t ld_utm, int nslabs, int64_t slab_stride, int r_pad,
                                          float* scratch, const float* UtU, int64_t ld_utu, const float* Vin, int64_t ld_vin, float* Vout,
                                          int64_t ld_vout, int r, int64_t n, int maxiter, double delta, double sparsity, double* result,
                                          void* stream) {
  NNFAC_ARG(ctx && UtM && UtU && Vin && Vout && result && scratch, "nnfac_hals_solve_slabs_f32: NULL argument");
  NNFAC_ARG(r > 0 && n > 0 && nslabs >= 1 && r_pad >= r, "nnfac_hals_solve_slabs_f32: empty problem (r=%d, n=%lld, %d slabs)", r, (long long)n, nslabs);
  NNFAC_ARG(ld_utm >= n && ld_vin >= n && ld_vout >= n && ld_utu >= r && slab_stride == (int64_t)r_pad * ld_utm,
            "nnfac_hals_solve_slabs_f32: leading dimension too small");
  cudaStream_t st = (cudaStream_t)stream;
  static const bool force_fma = getenv("NNFAC_SWEEP") && !strcmp(getenv("NNFAC_SWEEP"), "fma");
  if (!force_fma) {
    const int rc = nnfac_tc_sweep_run(ctx, UtM, ld_utm, UtU, ld_utu, Vin, ld_vin, Vout, ld_vout, r, n, maxiter, delta, sparsity,
                                      result, nullptr, st, nslabs, slab_stride);
    if (rc != NNFAC_ERR_UNSUPPORTED) return rc;
  }
  nnfac_reduce_partials(UtM, nslabs, r, r_pad, n, ld_utm, scratch, n, ctx->sm_count, st);
  NNFAC_LAUNCH_CHECK(ctx);
  if (Vin != Vout)
    NNFAC_CUDA(cudaMemcpy2DAsync(Vout, ld_vout * sizeof(float), Vin, ld_vin * sizeof(float), n * sizeof(float), r,
                                 cudaMemcpyDeviceToDevice, st));
  return nnfac_hals_nnls(ctx, NNFAC_F32, scratch, n, UtU, ld_utu, Vout, ld_vout, r, n, maxiter, delta, sparsity, 0u, result, stream);
}

extern "C" int nnfac_hals_solve_f32(nnfac_ctx* ctx, const float* UtM, int64_t ld_utm, const float* UtU, int64_t ld_utu,
                                    const float* Vin, int64_t ld_vin, float* Vout, int64_t ld_vout, int r, int64_t n, int maxiter,
                                    double delta, double sparsity, double* result, void* stream) {
  NNFAC_ARG(ctx && UtM && UtU && Vin && Vout && result, "nnfac_hals_solve_f32: NULL argument");
  NNFAC_ARG(r > 0 && n > 0, "nnfac_hals_solve_f32: empty problem (r=%d, n=%lld)", r, (long long)n);
  NNFAC_ARG(ld_utm >= n && ld_vin >= n && ld_vout >= n && ld_utu >= r, "nnfac_hals_solve_f32: leading dimension too small");
  cudaStream_t st = (cudaStream_t)stream;
  static const bool force_fma = getenv("NNFAC_SWEEP") && !strcmp(getenv("NNFAC_SWEEP"), "fma");
  if (!force_fma) {
    const int rc = nnfac_tc_sweep_run(ctx, UtM, ld_utm, UtU, ld_utu, Vin, ld_vin, Vout, ld_vout, r, n, maxiter, delta, sparsity,
                                      result, nullptr, st, 1, 0);
    if (rc != NNFAC_ERR_UNSUPPORTED) return rc;
  }
  if (Vin != Vout)
    NNFAC_CUDA(cudaMemcpy2DAsync(Vout, ld_vout * sizeof(float), Vin, ld_vin * sizeof(float), n * sizeof(float), r,
                                 cudaMemcpyDeviceToDevice, st));
  return nnfac_hals_nnls(ctx, NNFAC_F32, UtM, ld_utm, UtU, ld_utu, Vout, ld_vout, r, n, maxiter, delta, sparsity, 0u, result, stream);
}
