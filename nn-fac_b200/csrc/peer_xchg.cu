// Exchange steps of the column-sharded path over peer-mapped memory (NVLink / NVSwitch), one process per GPU.
//
// Per outer iteration the sharded NMF has one exchange on the U side: the partial cross products V_p X_p^T (r x m) and
// Grams of all ranks are summed, rank p needing only ITS m/P columns (a reduce-scatter), and after the slice solves
// every rank needs all slices (an all-gather).  With NCCL each of the two costs 0.1-0.2 ms at C2 on 8 GPUs whatever the
// size (16.8 MB): launch + protocol latency.  Here every rank owns an exchange region in device memory (cudaMalloc,
// exported with CUDA IPC, mapped by every peer):
//     [ flags | stage: tail block r x tpad, inbox (P * splits) x r_pad x chunk | send: r x (chunk + tpad) ]
// * the fused X pass of every rank writes its partial of each row tile straight into the inbox of the rank that owns those
//   rows of U (nnfac_nmf_plan_set_push, tc_fused.cu); the rank's small partial sums (Gram / row sums of V) go into its own tail
//   block; then `post` raises a sequence number in every peer's flag block (one st.release.sys each);
// * the consumers wait for the flags themselves: the slice solve and `inbox_mu_apply` add the slabs of the local inbox in slab
//   order, `pull_tail` sums the tail blocks of all P ranks in rank order over NVLink -- deterministic;
// * the slice solve writes into `send` (the slice's Gram behind it); after the next `post`, the kernel that installs the new
//   factor in the plan reads the P slices directly from the peers' `send` regions (nnfac_nmf_plan_set_factor_pulled): the
//   all-gather, the un-permute and the operand-plane construction in ONE kernel.
// Nothing is overwritten early: a rank writes into the inboxes and its tail block again only after its own install, which
// waited for every peer's second post (hence for every peer's solve and tail pull); it rewrites its send only after its own
// wait on the first posts of the next iteration (hence after every peer's install and Gram pull).
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

struct nnfac_xchg {
  nnfac_ctx* ctx;
  void* region;                 // local allocation
  size_t bytes, stage_off, send_off;
  int world, rank;
  void* peer[NNFAC_MAX_PEERS];  // mapped regions (peer[rank] == region)
  unsigned long long seq[2];    // posts made so far per phase
};

namespace {

constexpr size_t FLAG_BYTES = 256;   // [phase][rank] u64

struct PeerPtrs {
  const float* p[NNFAC_MAX_PEERS];
};
struct FlagPtrs {
  unsigned long long* p[NNFAC_MAX_PEERS];
};

// optional: tail_dst[k * tail_pitch] = tail_src[k], k < tail_count (a column of partial sums that travels with the buffer),
// written by this block before the flags are raised
__global__ void xchg_post_kernel(FlagPtrs flags, int world, int phase, int my_rank, unsigned long long seq, const float* tail_src,
                                 float* tail_dst, int64_t tail_pitch, int tail_count) {
  for (int k = threadIdx.x; k < tail_count; k += blockDim.x) tail_dst[(int64_t)k * tail_pitch] = tail_src[k];
  __syncthreads();
  if ((int)threadIdx.x < world) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flags.p[threadIdx.x] + phase * NNFAC_MAX_PEERS + my_rank), "l"(seq) : "memory");
  }
}

// Block-level wait inside a consumer kernel: every rank has posted `seq` times on `phase` (flags = the local flag block).
__device__ __forceinline__ void xchg_block_wait(const unsigned long long* flags, int world, int phase, unsigned long long seq) {
  if (flags != nullptr) {
    if ((int)threadIdx.x < world) {
      const unsigned long long* f = flags + phase * NNFAC_MAX_PEERS + threadIdx.x;
      unsigned long long v;
      unsigned long long spins = 0;
      do {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
        if (++spins > (1ull << 27)) __trap();   // a protocol bug fails the launch instead of hanging the GPU
      } while (v < seq);
    }
    __syncthreads();
  }
}

// sum_q src_q[off] in the fixed order q = 0 .. world-1 (the loads of all ranks are issued together)
__device__ __forceinline__ float pull_sum(const PeerPtrs& src, int world, int64_t off) {
  float v[NNFAC_MAX_PEERS];
#pragma unroll
  for (int q = 0; q < NNFAC_MAX_PEERS; ++q) v[q] = q < world ? __ldcv(src.p[q] + off) : 0.f;
  float s = 0.f;
#pragma unroll
  for (int q = 0; q < NNFAC_MAX_PEERS; ++q) if (q < world) s += v[q];
  return s;
}

// out[k][j] = sum_q src_q[k * pitch + col + j]  (j < tail), after waiting for every rank's post.  grid = r.
__global__ void __launch_bounds__(256) xchg_pull_tail_kernel(PeerPtrs src, int world, int64_t pitch, int64_t col, int tail,
                                                             float* __restrict__ out, int64_t ld_out, const unsigned long long* flags,
                                                             int phase, unsigned long long seq) {
  xchg_block_wait(flags, world, phase, seq);
  const int64_t k = blockIdx.x;
  for (int j = threadIdx.x; j < tail; j += blockDim.x) out[k * ld_out + j] = pull_sum(src, world, k * pitch + col + j);
}

// beta = 1 multiplicative update (mu.py:84-88): max(f * (num / den), floor), NaN propagating like numpy
__device__ __forceinline__ float mu_rule(float f, float num, float den, float floor_value) {
  const float v = f * (num / den);
  return v != v ? v : (v > floor_value ? v : floor_value);
}

// The update of this rank's rows of U when the partial numerators were PUSHED into this rank's inbox by the peers' fused passes
// (nnfac_nmf_plan_set_push): numerator = sum of the nslabs local slabs [r_pad x chunk] in slab order (rank-major, then split),
// denominator = sum over the ranks of column 0 of their tail blocks ([r x tail_pitch] at the start of every stage, read over
// NVLink: r floats per rank).  grid = (column blocks, r).
__global__ void __launch_bounds__(256) xchg_inbox_mu_apply_kernel(PeerPtrs stage, int world, const float* __restrict__ inbox, int nslabs,
                                                                  int64_t slab_stride, int64_t chunk, int64_t tail_pitch, int64_t lo,
                                                                  int64_t ncols, const float* __restrict__ F, int64_t ld_f,
                                                                  float floor_value, float* __restrict__ send, int64_t ld_send,
                                                                  const unsigned long long* flags, unsigned long long seq) {
  __shared__ float den_s;
  xchg_block_wait(flags, world, 0, seq);
  const int64_t k = blockIdx.y;
  if (threadIdx.x == 0) den_s = pull_sum(stage, world, k * tail_pitch);
  __syncthreads();
  const float den = den_s;
  const float* src = inbox + k * chunk;
  const int64_t nquad = (ncols + 3) / 4;           // chunk is a multiple of 128: quads never straddle the padding
  for (int64_t q0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q0 < nquad; q0 += (int64_t)gridDim.x * blockDim.x) {
    const int64_t c = q0 * 4;
    float4 num = make_float4(0.f, 0.f, 0.f, 0.f);
    int s = 0;
    for (; s + 4 <= nslabs; s += 4) {             // four slabs in flight, added in slab order
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = __ldcv(reinterpret_cast<const float4*>(src + (int64_t)(s + u) * slab_stride + c));
#pragma unroll
      for (int u = 0; u < 4; ++u) { num.x += v[u].x; num.y += v[u].y; num.z += v[u].z; num.w += v[u].w; }
    }
    for (; s < nslabs; ++s) {
      const float4 v = __ldcv(reinterpret_cast<const float4*>(src + (int64_t)s * slab_stride + c));
      num.x += v.x; num.y += v.y; num.z += v.z; num.w += v.w;
    }
    const float nv[4] = {num.x, num.y, num.z, num.w};
    for (int e = 0; e < 4 && c + e < ncols; ++e)
      send[k * ld_send + c + e] = mu_rule(F[k * ld_f + lo + c + e], nv[e], den, floor_value);
  }
}

}  // namespace

extern "C" {

int nnfac_xchg_create(nnfac_ctx* ctx, int64_t stage_floats, int64_t send_floats, nnfac_xchg** out) {
  NNFAC_ARG(ctx && out && stage_floats > 0 && send_floats > 0, "nnfac_xchg_create: bad argument");
  NNFAC_CUDA(cudaSetDevice(ctx->device));
  nnfac_xchg* x = (nnfac_xchg*)calloc(1, sizeof(nnfac_xchg));
  if (!x) return NNFAC_ERR_ALLOC;
  x->ctx = ctx;
  x->stage_off = FLAG_BYTES;
  x->send_off = x->stage_off + (((size_t)stage_floats * sizeof(float) + 255) & ~(size_t)255);
  x->bytes = x->send_off + (((size_t)send_floats * sizeof(float) + 255) & ~(size_t)255);
  if (cudaMalloc(&x->region, x->bytes) != cudaSuccess) {
    cudaGetLastError();
    nnfac_set_error("nnfac_xchg_create: out of device memory (%zu bytes)", x->bytes);
    free(x);
    return NNFAC_ERR_ALLOC;
  }
  NNFAC_CUDA(cudaMemset(x->region, 0, x->bytes));
  NNFAC_CUDA(cudaDeviceSynchronize());
  x->world = 1;
  x->peer[0] = x->region;
  *out = x;
  return NNFAC_OK;
}

int nnfac_xchg_export(nnfac_xchg* x, void* handle_out) {
  NNFAC_ARG(x && handle_out, "nnfac_xchg_export: NULL argument");
  cudaIpcMemHandle_t h;
  NNFAC_CUDA(cudaIpcGetMemHandle(&h, x->region));
  memcpy(handle_out, &h, sizeof(h));
  return NNFAC_OK;
}

int nnfac_xchg_attach(nnfac_xchg* x, int world, int rank, const void* handles) {
  NNFAC_ARG(x && handles && world >= 1 && world <= NNFAC_MAX_PEERS && rank >= 0 && rank < world, "nnfac_xchg_attach: bad argument");
  NNFAC_CUDA(cudaSetDevice(x->ctx->device));
  for (int q = 0; q < world; ++q) {
    if (q == rank) { x->peer[q] = x->region; continue; }
    cudaIpcMemHandle_t h;
    memcpy(&h, (const char*)handles + (size_t)q * sizeof(h), sizeof(h));
    NNFAC_CUDA(cudaIpcOpenMemHandle(&x->peer[q], h, cudaIpcMemLazyEnablePeerAccess));
  }
  x->world = world;
  x->rank = rank;
  return NNFAC_OK;
}

int nnfac_xchg_destroy(nnfac_xchg* x) {
  if (!x) return NNFAC_OK;
  cudaSetDevice(x->ctx->device);
  for (int q = 0; q < x->world; ++q)
    if (q != x->rank && x->peer[q]) cudaIpcCloseMemHandle(x->peer[q]);
  cudaFree(x->region);
  free(x);
  return NNFAC_OK;
}

// local device pointer of the stage (which = 0) or send (which = 1) buffer
void* nnfac_xchg_ptr(nnfac_xchg* x, int which) {
  if (!x) return nullptr;
  return (char*)x->region + (which == 0 ? x->stage_off : x->send_off);
}

// "what this rank wrote into its stage / send buffer so far (on `stream`) is complete": raises the sequence number of
// `phase` (0: stage, 1: send) in every rank's flag block.
int nnfac_xchg_post(nnfac_xchg* x, int phase, void* stream) {
  NNFAC_ARG(x && (phase == 0 || phase == 1), "nnfac_xchg_post: bad argument");
  FlagPtrs f;
  for (int q = 0; q < NNFAC_MAX_PEERS; ++q) f.p[q] = q < x->world ? (unsigned long long*)x->peer[q] : nullptr;
  xchg_post_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(f, x->world, phase, x->rank, ++x->seq[phase], nullptr, nullptr, 0, 0);
  NNFAC_LAUNCH_CHECK(x->ctx);
  return NNFAC_OK;
}

// nnfac_xchg_post(x, 0, stream) after writing column `col` of the stage ([rows x pitch]) from tail_src[0 .. rows): the small
// partial sums that travel behind the big ones (row sums of V for the beta = 1 update) without a copy kernel of their own
int nnfac_xchg_post_tail(nnfac_xchg* x, const float* tail_src, int rows, int64_t pitch, int64_t col, void* stream) {
  NNFAC_ARG(x && tail_src && rows > 0 && col >= 0 && col < pitch, "nnfac_xchg_post_tail: bad argument");
  NNFAC_ARG((size_t)rows * (size_t)pitch * sizeof(float) <= x->send_off - x->stage_off, "nnfac_xchg_post_tail: beyond the stage buffer");
  FlagPtrs f;
  for (int q = 0; q < NNFAC_MAX_PEERS; ++q) f.p[q] = q < x->world ? (unsigned long long*)x->peer[q] : nullptr;
  float* stage = (float*)((char*)x->region + x->stage_off);
  xchg_post_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(f, x->world, 0, x->rank, ++x->seq[0], tail_src, stage + col, pitch, rows);
  NNFAC_LAUNCH_CHECK(x->ctx);
  return NNFAC_OK;
}

// flag block, world and the number of posts this rank has made on `phase`: what a consumer kernel needs to wait by itself
void nnfac_xchg_wait_args(const nnfac_xchg* x, int phase, const unsigned long long** flags, int* world, unsigned long long* seq) {
  *flags = (const unsigned long long*)x->region;
  *world = x->world;
  *seq = x->seq[phase];
}

// out[k][j] = sum over the ranks, in rank order, of element k * pitch + col + j of their buffer `which` ([r x pitch] each;
// k < r, j < tail).  Call after this rank's nnfac_xchg_post(x, which): the kernel itself waits until every rank has posted as
// often.
int nnfac_xchg_pull_tail(nnfac_xchg* x, int which, float* out, int64_t ld_out, int r, int64_t pitch, int64_t col, int tail,
                         void* stream) {
  NNFAC_ARG(x && out && (which == 0 || which == 1) && r > 0 && tail > 0 && ld_out >= tail && col >= 0 && col + tail <= pitch,
            "nnfac_xchg_pull_tail: bad argument");
  const size_t off = which == 0 ? x->stage_off : x->send_off;
  const size_t end = which == 0 ? x->send_off : x->bytes;
  NNFAC_ARG((size_t)r * (size_t)pitch * sizeof(float) <= end - off, "nnfac_xchg_pull_tail: beyond the buffer");
  PeerPtrs src;
  for (int q = 0; q < NNFAC_MAX_PEERS; ++q) src.p[q] = q < x->world ? (const float*)((const char*)x->peer[q] + off) : nullptr;
  xchg_pull_tail_kernel<<<(unsigned)r, 256, 0, (cudaStream_t)stream>>>(src, x->world, pitch, col, tail, out, ld_out,
                                                                       (const unsigned long long*)x->region, which, x->seq[which]);
  NNFAC_LAUNCH_CHECK(x->ctx);
  return NNFAC_OK;
}

// The U update of the column-sharded beta = 1 rule when the peers' fused passes pushed their partial numerators into this rank's
// inbox (nnfac_nmf_plan_set_push; inbox_off floats into the stage buffer, nslabs slabs of slab_stride floats, row pitch chunk),
// after this rank's post on phase 0 (nnfac_xchg_post_tail with pitch = tail_pitch, col = 0: the partial row sums of V sit in
// column 0 of the [r x tail_pitch] block at the start of every stage).  Writes the new rows [lo, lo + ncols) of U^T into this
// rank's send buffer ([r x ld_send]).
int nnfac_xchg_inbox_mu_apply(nnfac_xchg* x, int64_t inbox_off, int nslabs, int64_t slab_stride, int64_t chunk, int64_t tail_pitch,
                              const float* F, int64_t ld_f, int r, int64_t lo, int64_t ncols, double floor_value, int64_t ld_send,
                              void* stream) {
  NNFAC_ARG(x && F && r > 0 && nslabs > 0 && ncols >= 0 && ncols <= chunk && chunk % 4 == 0 && inbox_off % 4 == 0 && slab_stride % 4 == 0 &&
                tail_pitch > 0 && inbox_off >= (int64_t)r * tail_pitch && ld_send >= ncols && lo >= 0 && ld_f >= lo + ncols,
            "nnfac_xchg_inbox_mu_apply: bad argument");
  NNFAC_ARG((size_t)(inbox_off + (int64_t)nslabs * slab_stride) * sizeof(float) <= x->send_off - x->stage_off,
            "nnfac_xchg_inbox_mu_apply: beyond the stage buffer");
  NNFAC_ARG((size_t)r * (size_t)ld_send * sizeof(float) <= x->bytes - x->send_off, "nnfac_xchg_inbox_mu_apply: beyond the send buffer");
  if (ncols == 0) return NNFAC_OK;
  PeerPtrs src;
  for (int q = 0; q < NNFAC_MAX_PEERS; ++q) src.p[q] = q < x->world ? (const float*)((const char*)x->peer[q] + x->stage_off) : nullptr;
  const int64_t gx = ceil_div64(ceil_div64(ncols, 4), 256);
  xchg_inbox_mu_apply_kernel<<<dim3((unsigned)gx, (unsigned)r), 256, 0, (cudaStream_t)stream>>>(
      src, x->world, (const float*)((const char*)x->region + x->stage_off) + inbox_off, nslabs, slab_stride, chunk, tail_pitch, lo, ncols,
      F, ld_f, (float)floor_value, (float*)((char*)x->region + x->send_off), ld_send, (const unsigned long long*)x->region, x->seq[0]);
  NNFAC_LAUNCH_CHECK(x->ctx);
  return NNFAC_OK;
}

// peer q's send buffer as mapped here (for nnfac_nmf_plan_set_factor_pulled)
const float* nnfac_xchg_peer_send(const nnfac_xchg* x, int q) {
  if (!x || q < 0 || q >= x->world) return nullptr;
  return (const float*)((const char*)x->peer[q] + x->send_off);
}
int nnfac_xchg_world(const nnfac_xchg* x) { return x ? x->world : 0; }
int nnfac_xchg_rank(const nnfac_xchg* x) { return x ? x->rank : 0; }
void* nnfac_xchg_peer_stage(const nnfac_xchg* x, int q) {
  if (!x || q < 0 || q >= x->world) return nullptr;
  return (char*)x->peer[q] + x->stage_off;
}
int64_t nnfac_xchg_stage_floats(const nnfac_xchg* x) { return x ? (int64_t)((x->send_off - x->stage_off) / sizeof(float)) : 0; }

}  // extern "C"
