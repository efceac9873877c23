// Context management and error reporting for the C ABI (include/nnfac_b200.h).
#include "common.cuh"
#include <stdlib.h>
#include <string.h>

static thread_local char g_err[512] = "";

void nnfac_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int nnfac_ws_reserve(nnfac_ctx* ctx, size_t bytes, cudaStream_t st) {
  if (bytes <= ctx->ws_bytes) return NNFAC_OK;
  // growing the scratch buffer is rare: drain the stream that may still be using the old one
  NNFAC_CUDA(cudaStreamSynchronize(st));
  if (ctx->ws) NNFAC_CUDA(cudaFree(ctx->ws));
  ctx->ws = nullptr;
  ctx->ws_bytes = 0;
  size_t want = bytes + (bytes >> 2);
  if (cudaMalloc(&ctx->ws, want) != cudaSuccess) {
    cudaGetLastError();
    nnfac_set_error("workspace allocation of %zu bytes failed", want);
    return NNFAC_ERR_ALLOC;
  }
  ctx->ws_bytes = want;
  return NNFAC_OK;
}

int nnfac_guard_enter(nnfac_ctx* ctx, int which, cudaStream_t st) {
  nnfac_guard* g = &ctx->guard[which];
  if (g->valid && g->last != st) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) cudaGetLastError();
    if (cs != cudaStreamCaptureStatusNone) return NNFAC_OK;       // a captured sequence is single-stream by construction
    if (!g->ev) NNFAC_CUDA(cudaEventCreateWithFlags(&g->ev, cudaEventDisableTiming));
    if (cudaEventRecord(g->ev, g->last) == cudaSuccess) {
      NNFAC_CUDA(cudaStreamWaitEvent(st, g->ev, 0));
    } else {
      cudaGetLastError();                                          // the last user's stream is gone: drain the device instead
      NNFAC_CUDA(cudaDeviceSynchronize());
    }
  }
  g->last = st;
  g->valid = 1;
  return NNFAC_OK;
}

// layout of a stop-scalar board: 8 banks x NNFAC_MAX_PEERS ranks x 160 CTAs of 8 bytes (see csrc/tc_sweep.cu)
static const size_t kBoardBytes = (size_t)8 * NNFAC_MAX_PEERS * 160 * sizeof(unsigned long long);

extern "C" {

int nnfac_abi_version(void) { return NNFAC_ABI_VERSION; }

const char* nnfac_last_error(void) { return g_err; }

int nnfac_ctx_create(int device, nnfac_ctx** out) {
  NNFAC_ARG(out != nullptr, "nnfac_ctx_create: out is NULL");
  int ndev = 0;
  NNFAC_CUDA(cudaGetDeviceCount(&ndev));
  NNFAC_ARG(device >= 0 && device < ndev, "nnfac_ctx_create: device %d out of range (%d visible)", device, ndev);
  NNFAC_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  NNFAC_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    nnfac_set_error("nnfac_b200 is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
    return NNFAC_ERR_UNSUPPORTED;
  }
  nnfac_ctx* c = (nnfac_ctx*)calloc(1, sizeof(nnfac_ctx));
  if (c) c->sweep_lag = -1;
  if (!c) return NNFAC_ERR_ALLOC;
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  c->red_count = 1 << 16;
  NNFAC_CUDA(cudaMalloc(&c->red, c->red_count * sizeof(double)));
  NNFAC_CUDA(cudaMalloc(&c->sync, 64 * sizeof(unsigned)));
  NNFAC_CUDA(cudaMemset(c->sync, 0, 64 * sizeof(unsigned)));
  c->mail_count = (size_t)1 << 18;
  // one extra word behind the mailboxes holds the call generation (advanced on the device, see csrc/tc_sweep.cu)
  NNFAC_CUDA(cudaMalloc(&c->mail, (c->mail_count + 1) * sizeof(unsigned long long)));
  NNFAC_CUDA(cudaMemset(c->mail, 0, (c->mail_count + 1) * sizeof(unsigned long long)));
  c->ws_bytes = (size_t)64 << 20;
  NNFAC_CUDA(cudaMalloc(&c->ws, c->ws_bytes));
  *out = c;
  return NNFAC_OK;
}

int nnfac_ctx_destroy(nnfac_ctx* ctx) {
  if (!ctx) return NNFAC_OK;
  cudaSetDevice(ctx->device);
  cudaFree(ctx->ws);
  cudaFree(ctx->red);
  cudaFree(ctx->sync);
  cudaFree(ctx->mail);
  for (int q = 0; q < ctx->peers.world; ++q)
    if (q != ctx->peers.rank && ctx->peers.board[q]) cudaIpcCloseMemHandle(ctx->peers.board[q]);
  cudaFree(ctx->board);
  for (int i = 0; i < NNFAC_NGUARD; ++i)
    if (ctx->guard[i].ev) cudaEventDestroy(ctx->guard[i].ev);
  free(ctx);
  return NNFAC_OK;
}

// ---- collective HALS solves over several GPUs (one process each) -------------------------------------------------
// 1. every rank: nnfac_ctx_board_export -> 64-byte IPC handle of its board; 2. exchange the handles (any transport);
// 3. every rank: nnfac_ctx_board_attach(world, rank, handles); 4. around a solve that is one slice of a joint solve:
// nnfac_ctx_collective(ctx, 1, slice_lengths) ... nnfac_ctx_collective(ctx, 0, NULL).
int nnfac_ctx_sweep_variant(nnfac_ctx* ctx, int mode) {
  NNFAC_ARG(ctx && mode >= -1 && mode <= 2, "nnfac_ctx_sweep_variant: mode must be -1, 0, 1 or 2");
  ctx->sweep_lag = mode;
  return NNFAC_OK;
}

int nnfac_ctx_board_export(nnfac_ctx* ctx, void* handle_out) {
  NNFAC_ARG(ctx && handle_out, "nnfac_ctx_board_export: NULL argument");
  NNFAC_CUDA(cudaSetDevice(ctx->device));
  if (!ctx->board) {
    NNFAC_CUDA(cudaMalloc(&ctx->board, kBoardBytes));
    NNFAC_CUDA(cudaMemset(ctx->board, 0, kBoardBytes));
    NNFAC_CUDA(cudaDeviceSynchronize());
  }
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  cudaIpcMemHandle_t h;
  NNFAC_CUDA(cudaIpcGetMemHandle(&h, ctx->board));
  memcpy(handle_out, &h, sizeof(h));
  return NNFAC_OK;
}

int nnfac_ctx_board_attach(nnfac_ctx* ctx, int world, int rank, const void* handles) {
  NNFAC_ARG(ctx && handles && world >= 1 && world <= NNFAC_MAX_PEERS && rank >= 0 && rank < world, "nnfac_ctx_board_attach: bad argument");
  NNFAC_ARG(ctx->board != nullptr, "nnfac_ctx_board_attach: call nnfac_ctx_board_export first");
  NNFAC_CUDA(cudaSetDevice(ctx->device));
  for (int q = 0; q < ctx->peers.world; ++q)
    if (q != ctx->peers.rank && ctx->peers.board[q]) cudaIpcCloseMemHandle(ctx->peers.board[q]);
  memset(&ctx->peers, 0, sizeof(ctx->peers));
  for (int q = 0; q < world; ++q) {
    if (q == rank) { ctx->peers.board[q] = ctx->board; continue; }
    cudaIpcMemHandle_t h;
    memcpy(&h, (const char*)handles + (size_t)q * sizeof(h), sizeof(h));
    NNFAC_CUDA(cudaIpcOpenMemHandle(&ctx->peers.board[q], h, cudaIpcMemLazyEnablePeerAccess));
  }
  ctx->peers.world = world;
  ctx->peers.rank = rank;
  return NNFAC_OK;
}

int nnfac_ctx_collective(nnfac_ctx* ctx, int on, const int64_t* slice_lengths) {
  NNFAC_ARG(ctx != nullptr, "nnfac_ctx_collective: ctx is NULL");
  if (!on) { ctx->collective = 0; return NNFAC_OK; }
  // a group of one is a group: its solves take the board protocol too (which is how that protocol is checked on one GPU)
  NNFAC_ARG(ctx->peers.world >= 1 && slice_lengths, "nnfac_ctx_collective: no peer group attached");
  for (int q = 0; q < ctx->peers.world; ++q) ctx->collective_n[q] = slice_lengths[q];
  ctx->collective = 1;
  return NNFAC_OK;
}

int nnfac_ctx_sm_count(const nnfac_ctx* ctx) { return ctx ? ctx->sm_count : 0; }
int64_t nnfac_ctx_launch_count(const nnfac_ctx* ctx) { return ctx ? ctx->launches : 0; }

}  // extern "C"
