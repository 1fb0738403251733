// ctx.cu -- context, memory, timers, error plumbing of libigneous_b200
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

namespace ign {

static thread_local std::string g_err;

void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
}

int activate(ign_ctx* ctx) {
  IGN_REQUIRE(ctx != nullptr, IGN_ERR_INVALID, "null ign_ctx");
  IGN_CUDA(cudaSetDevice(ctx->device));
  return IGN_OK;
}

// replaces *buf by a fresh allocation of exactly `bytes`
static int realloc_buffer(ign_ctx* ctx, char** buf, size_t* have, size_t bytes, const char* what) {
  IGN_CUDA(cudaStreamSynchronize(ctx->stream));
  if (*buf) IGN_CUDA(cudaFree(*buf));
  *buf = nullptr;
  *have = 0;
  cudaError_t e = cudaMalloc((void**)buf, bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("%s: cudaMalloc(%zu) failed: %s", what, bytes, cudaGetErrorString(e));
    return IGN_ERR_NOMEM;
  }
  *have = bytes;
  return IGN_OK;
}

int grow_buffer(ign_ctx* ctx, char** buf, size_t* have, size_t need, const char* what) {
  if (*have >= need) return IGN_OK;
  return realloc_buffer(ctx, buf, have, need + need / 4, what);
}

int Scratch::reserve(size_t bytes) {
  if (!owner()) return IGN_OK;
  bytes = align_up(bytes + 4096, 1 << 20);
  if (bytes <= ctx_->scratch_bytes) return IGN_OK;
  return realloc_buffer(ctx_, &ctx_->scratch, &ctx_->scratch_bytes, bytes, "scratch arena");
}

void* Scratch::take_bytes(size_t bytes) {
  const size_t off = align_up(ctx_->scratch_used, 256);
  if (off + bytes > ctx_->scratch_bytes) {
    ok_ = false;
    return nullptr;
  }
  ctx_->scratch_used = off + bytes;
  return ctx_->scratch + off;
}

void Scratch::rewind() {
  ctx_->scratch_used = base_;
  ok_ = true;
}

int Staging::stage() {
  size_t total = 0;
  for (const Slot& s : slots_) total += align_up(s.bytes, 256);
  IGN_TRY(grow_buffer(ctx_, &ctx_->stage, &ctx_->stage_bytes, total, "staging buffer"));
  size_t off = 0;
  for (const Slot& s : slots_) {
    *s.dev = s.bytes ? ctx_->stage + off : nullptr;
    if (s.host && s.bytes) IGN_CUDA(cudaMemcpyAsync(*s.dev, s.host, s.bytes, cudaMemcpyHostToDevice, ctx_->stream));
    off += align_up(s.bytes, 256);
  }
  return IGN_OK;
}

int Staging::back(void* host, const void* dev, size_t bytes) {
  if (bytes) IGN_CUDA(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx_->stream));
  return IGN_OK;
}

int Staging::sync() {
  IGN_CUDA(cudaStreamSynchronize(ctx_->stream));
  return IGN_OK;
}

template <typename T>
__global__ void __launch_bounds__(256)
    k_copy_box(const T* __restrict__ src, uint64_t sx, uint64_t sy, uint64_t x0, uint64_t y0,
               uint64_t z0, uint64_t bx, uint64_t by, uint64_t total, T* __restrict__ dst) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const uint64_t x = i % bx, r = i / bx, y = r % by, z = r / by;
  dst[i] = src[((z0 + z) * sy + (y0 + y)) * sx + (x0 + x)];
}

// ---- mapped pinned window (small control transfers)
enum : size_t { WIN_FETCH_BYTES = 256 << 10, WIN_PUSH_BYTES = 768 << 10 };

__global__ void __launch_bounds__(256) k_copy_small(void* __restrict__ dst, const void* __restrict__ src,
                                                    uint32_t n_words, uint32_t tail_bytes) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_words) ((uint32_t*)dst)[i] = ((const uint32_t*)src)[i];
  if (i < tail_bytes) ((uint8_t*)dst)[4ull * n_words + i] = ((const uint8_t*)src)[4ull * n_words + i];
}

static int copy_small_launch(ign_ctx* ctx, void* dst, const void* src, size_t bytes);

// Device -> pinned host copy by a kernel (stores to mapped host memory) instead of the D2H copy engine.
// The engine serves one copy at a time: a MeshTask's fragment export queued behind a multi-gigabyte
// label download waits for it, and with it the task's stream (measured on the streamed 2048^3 step:
// +0.38 s).  Stores issued by SMs share the PCIe link with the DMA but are not queued behind it.
__global__ void __launch_bounds__(256) k_copy_to_host(uint4* __restrict__ dst, const uint4* __restrict__ src, uint64_t n16) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n16; i += (uint64_t)gridDim.x * blockDim.x)
    dst[i] = src[i];
}

int d2h_by_kernel(ign_ctx* ctx, void* host_dst, const void* dev_src, size_t bytes) {
  cudaPointerAttributes at;
  const bool pinned = cudaPointerGetAttributes(&at, host_dst) == cudaSuccess && at.type == cudaMemoryTypeHost &&
                      at.devicePointer != nullptr;
  cudaGetLastError();
  if (!pinned || ((uintptr_t)at.devicePointer % 16) != 0 || ((uintptr_t)dev_src % 16) != 0) {
    IGN_CUDA(cudaMemcpyAsync(host_dst, dev_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return IGN_OK;
  }
  const uint64_t n16 = bytes / 16;
  if (n16) {
    const unsigned grid = (unsigned)(blocks_for(n16, 256) < (uint64_t)ctx->sm_count * 2 ? blocks_for(n16, 256) : (uint64_t)ctx->sm_count * 2);
    IGN_LAUNCH(ctx, k_copy_to_host, grid, 256, 0, (uint4*)at.devicePointer, (const uint4*)dev_src, n16);
  }
  if (bytes % 16)
    IGN_TRY(copy_small_launch(ctx, (char*)at.devicePointer + 16 * n16, (const char*)dev_src + 16 * n16, bytes % 16));
  return IGN_OK;
}

static int copy_small_launch(ign_ctx* ctx, void* dst, const void* src, size_t bytes) {
  const bool words = ((uintptr_t)dst % 4 == 0) && ((uintptr_t)src % 4 == 0);
  const uint32_t nw = words ? (uint32_t)(bytes / 4) : 0;
  const uint32_t tail = (uint32_t)(bytes - 4ull * nw);
  const uint32_t work = nw > tail ? nw : tail;
  IGN_LAUNCH(ctx, k_copy_small, blocks_for(work, 256), 256, 0, dst, src, nw, tail);
  return IGN_OK;
}

int small_d2h(ign_ctx* ctx, void* host_dst, const void* dev_src, size_t bytes) {
  if (bytes == 0) return IGN_OK;
  const size_t off = align_up(ctx->win_fetch_used, 16);
  if (!ctx->win || ctx->fetch_n == 32 || off + bytes > WIN_FETCH_BYTES) {
    IGN_CUDA(cudaMemcpyAsync(host_dst, dev_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return IGN_OK;
  }
  IGN_TRY(copy_small_launch(ctx, ctx->win_dev + off, dev_src, bytes));
  ctx->fetch[ctx->fetch_n++] = {host_dst, off, bytes};
  ctx->win_fetch_used = off + bytes;
  return IGN_OK;
}

int small_sync(ign_ctx* ctx) {
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  if (e == cudaSuccess)
    for (int i = 0; i < ctx->fetch_n; i++)
      memcpy(ctx->fetch[i].dst, ctx->win + ctx->fetch[i].off, ctx->fetch[i].bytes);
  ctx->fetch_n = 0;
  ctx->win_fetch_used = 0;
  ctx->win_push_used = 0;  // every queued push kernel has run
  IGN_CUDA(e);
  return IGN_OK;
}

int small_h2d(ign_ctx* ctx, void* dev_dst, const void* host_src, size_t bytes) {
  if (bytes == 0) return IGN_OK;
  if (!ctx->win || bytes > WIN_PUSH_BYTES) {
    IGN_CUDA(cudaMemcpyAsync(dev_dst, host_src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return IGN_OK;
  }
  size_t off = align_up(ctx->win_push_used, 16);
  if (off + bytes > WIN_PUSH_BYTES) {  // window full: wait until the queued copy kernels have read it
    IGN_CUDA(cudaStreamSynchronize(ctx->stream));
    off = 0;
  }
  char* stage = ctx->win + WIN_FETCH_BYTES + off;
  memcpy(stage, host_src, bytes);
  ctx->win_push_used = off + bytes;
  return copy_small_launch(ctx, dev_dst, ctx->win_dev + WIN_FETCH_BYTES + off, bytes);
}

int prof_begin(ign_ctx* ctx, int cls) {
  if (!ctx->prof_on) return -1;
  if (ctx->prof_n == ctx->prof_cap) {
    const int ncap = ctx->prof_cap ? ctx->prof_cap * 2 : 256;
    ign_ctx::ProfRec* np = (ign_ctx::ProfRec*)realloc(ctx->prof, sizeof(ign_ctx::ProfRec) * ncap);
    if (!np) return -1;
    for (int i = ctx->prof_cap; i < ncap; i++) {
      cudaEventCreate(&np[i].a);
      cudaEventCreate(&np[i].b);
    }
    ctx->prof = np;
    ctx->prof_cap = ncap;
  }
  const int slot = ctx->prof_n++;
  ctx->prof[slot].cls = cls;
  cudaEventRecord(ctx->prof[slot].a, ctx->stream);
  return slot;
}

void prof_end(ign_ctx* ctx, int slot) {
  if (slot >= 0) cudaEventRecord(ctx->prof[slot].b, ctx->stream);
}

}  // namespace ign

using namespace ign;

extern "C" {

int ign_version(void) { return 100; }

const char* ign_last_error(void) { return g_err.c_str(); }

int ign_device_count(int* n) {
  IGN_REQUIRE(n, IGN_ERR_INVALID, "null out pointer");
  cudaError_t e = cudaGetDeviceCount(n);
  if (e != cudaSuccess) {
    *n = 0;
    set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e));
    cudaGetLastError();
    return IGN_ERR_CUDA;
  }
  return IGN_OK;
}

int ign_init(int device, ign_ctx** out) {
  IGN_REQUIRE(out, IGN_ERR_INVALID, "null out pointer");
  *out = nullptr;
  int n = 0;
  IGN_TRY(ign_device_count(&n));
  IGN_REQUIRE(n > 0, IGN_ERR_CUDA, "no CUDA device visible (this library has no CPU fallback)");
  IGN_REQUIRE(device >= 0 && device < n, IGN_ERR_INVALID, "device %d out of range [0,%d)", device, n);
  IGN_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  IGN_CUDA(cudaGetDeviceProperties(&prop, device));
  IGN_REQUIRE(prop.major >= 10, IGN_ERR_UNSUPPORTED,
              "device %d is sm_%d%d; libigneous_b200 is built for sm_100a only", device,
              prop.major, prop.minor);
  ign_ctx* ctx = new ign_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  ctx->scratch = nullptr;
  ctx->scratch_bytes = ctx->scratch_used = 0;
  ctx->stage = nullptr;
  ctx->stage_bytes = 0;
  ctx->launches = 0;
  ctx->prof_on = 0;
  ctx->prof = nullptr;
  ctx->prof_n = ctx->prof_cap = 0;
  ctx->mesh_pool = nullptr;
  ctx->mesh_pool_bytes = 0;
  ctx->mesh_pool_busy = 0;
  IGN_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  IGN_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  ctx->pinned_bytes = 1 << 20;
  IGN_CUDA(cudaHostAlloc((void**)&ctx->pinned, ctx->pinned_bytes, cudaHostAllocDefault));
  for (int i = 0; i < IGN_TIMER_SLOTS; i++) {
    IGN_CUDA(cudaEventCreate(&ctx->timers[i][0]));
    IGN_CUDA(cudaEventCreate(&ctx->timers[i][1]));
  }
  ctx->win = ctx->win_dev = nullptr;
  ctx->win_fetch_used = ctx->win_push_used = 0;
  ctx->fetch_n = 0;
  if (cudaHostAlloc((void**)&ctx->win, WIN_FETCH_BYTES + WIN_PUSH_BYTES,
                    cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess ||
      cudaHostGetDevicePointer((void**)&ctx->win_dev, ctx->win, 0) != cudaSuccess) {
    // no mapped host memory: small transfers use the copy engines
    cudaGetLastError();
    if (ctx->win) cudaFreeHost(ctx->win);
    ctx->win = ctx->win_dev = nullptr;
  }
  *out = ctx;
  return IGN_OK;
}

int ign_destroy(ign_ctx* ctx) {
  if (!ctx) return IGN_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->scratch) cudaFree(ctx->scratch);
  if (ctx->stage) cudaFree(ctx->stage);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  if (ctx->win) cudaFreeHost(ctx->win);
  if (ctx->mesh_pool) cudaFree(ctx->mesh_pool);
  for (int i = 0; i < IGN_TIMER_SLOTS; i++) {
    cudaEventDestroy(ctx->timers[i][0]);
    cudaEventDestroy(ctx->timers[i][1]);
  }
  cudaStreamDestroy(ctx->stream);
  cudaStreamDestroy(ctx->copy_stream);
  delete ctx;
  return IGN_OK;
}

int ign_sync(ign_ctx* ctx) {
  IGN_TRY(activate(ctx));
  IGN_CUDA(cudaStreamSynchronize(ctx->stream));
  return IGN_OK;
}

int ign_launch_count(ign_ctx* ctx, uint64_t* n) {
  IGN_REQUIRE(ctx && n, IGN_ERR_INVALID, "null argument");
  *n = ctx->launches;
  return IGN_OK;
}

int ign_stream(ign_ctx* ctx, void** stream) {
  IGN_REQUIRE(ctx && stream, IGN_ERR_INVALID, "null argument");
  *stream = (void*)ctx->stream;
  return IGN_OK;
}

int ign_dev_alloc(ign_ctx* ctx, uint64_t bytes, void** dptr) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(dptr, IGN_ERR_INVALID, "null out pointer");
  *dptr = nullptr;
  cudaError_t e = cudaMalloc(dptr, bytes ? bytes : 1);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("cudaMalloc(%llu) failed: %s", (unsigned long long)bytes, cudaGetErrorString(e));
    return IGN_ERR_NOMEM;
  }
  return IGN_OK;
}

int ign_dev_free(ign_ctx* ctx, void* dptr) {
  IGN_TRY(activate(ctx));
  IGN_CUDA(cudaStreamSynchronize(ctx->stream));
  IGN_CUDA(cudaFree(dptr));
  return IGN_OK;
}

int ign_host_alloc(ign_ctx* ctx, uint64_t bytes, void** hptr) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(hptr, IGN_ERR_INVALID, "null out pointer");
  cudaError_t e = cudaHostAlloc(hptr, bytes ? bytes : 1, cudaHostAllocDefault);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("cudaHostAlloc(%llu) failed: %s", (unsigned long long)bytes, cudaGetErrorString(e));
    return IGN_ERR_NOMEM;
  }
  return IGN_OK;
}

int ign_host_free(ign_ctx* ctx, void* hptr) {
  IGN_TRY(activate(ctx));
  IGN_CUDA(cudaFreeHost(hptr));
  return IGN_OK;
}

// Bulk copies are issued in 64 MiB pieces so that transfers of other contexts sharing
// the copy engines (mesh fragment exports) interleave instead of waiting for a
// multi-GB transfer to drain.
static const uint64_t BULK_PIECE = 64ull << 20;

// Bulk host copies are queued in BULK_PIECE pieces (copies of other streams can be served in between).
static int bulk_copy(ign_ctx* ctx, void* dst, const void* src, uint64_t bytes, cudaMemcpyKind kind) {
  for (uint64_t at = 0; at < bytes; at += BULK_PIECE) {
    const uint64_t nb = bytes - at < BULK_PIECE ? bytes - at : BULK_PIECE;
    IGN_CUDA(cudaMemcpyAsync((char*)dst + at, (const char*)src + at, nb, kind, ctx->stream));
  }
  return IGN_OK;
}

int ign_h2d(ign_ctx* ctx, void* dst, const void* src, uint64_t bytes) {
  IGN_TRY(activate(ctx));
  return bulk_copy(ctx, dst, src, bytes, cudaMemcpyHostToDevice);
}

int ign_d2h(ign_ctx* ctx, void* dst, const void* src, uint64_t bytes) {
  IGN_TRY(activate(ctx));
  return bulk_copy(ctx, dst, src, bytes, cudaMemcpyDeviceToHost);
}

int ign_d2d(ign_ctx* ctx, void* dst, const void* src, uint64_t bytes) {
  IGN_TRY(activate(ctx));
  IGN_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
  return IGN_OK;
}

int ign_memset(ign_ctx* ctx, void* dst, int byte, uint64_t bytes) {
  IGN_TRY(activate(ctx));
  IGN_CUDA(cudaMemsetAsync(dst, byte, bytes, ctx->stream));
  return IGN_OK;
}

int ign_prof_enable(ign_ctx* ctx, int on) {
  IGN_REQUIRE(ctx, IGN_ERR_INVALID, "null ctx");
  ctx->prof_on = on ? 1 : 0;
  ctx->prof_n = 0;
  return IGN_OK;
}

// sums the recorded launches of one kernel class since ign_prof_enable(ctx,1)
int ign_prof_read(ign_ctx* ctx, int cls, float* total_ms, uint64_t* launches) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(total_ms && launches, IGN_ERR_INVALID, "null argument");
  IGN_CUDA(cudaStreamSynchronize(ctx->stream));
  float sum = 0;
  uint64_t cnt = 0;
  for (int i = 0; i < ctx->prof_n; i++) {
    if (ctx->prof[i].cls != cls) continue;
    float ms = 0;
    IGN_CUDA(cudaEventElapsedTime(&ms, ctx->prof[i].a, ctx->prof[i].b));
    sum += ms;
    cnt++;
  }
  *total_ms = sum;
  *launches = cnt;
  return IGN_OK;
}

// strided 3-D sub-box copy between device volumes (Fortran order).  A plain
// coalesced kernel: cudaMemcpy3D takes a slow path for rows of ~1 KB.
int ign_copy_box_dev(ign_ctx* ctx, const void* src, int dtype, uint64_t sx, uint64_t sy, uint64_t sz,
                     uint64_t x0, uint64_t y0, uint64_t z0, uint64_t bx, uint64_t by, uint64_t bz,
                     void* dst) {
  IGN_TRY(activate(ctx));
  const size_t es = dtype_size(dtype);
  IGN_REQUIRE(src && dst && es > 0, IGN_ERR_INVALID, "bad copy_box argument");
  IGN_REQUIRE(x0 + bx <= sx && y0 + by <= sy && z0 + bz <= sz, IGN_ERR_INVALID, "box outside the volume");
  const uint64_t total = bx * by * bz;
  if (total == 0) return IGN_OK;
  const unsigned g = blocks_for(total, 256);
  switch (es) {
    case 1: IGN_LAUNCH(ctx, (k_copy_box<uint8_t>), g, 256, 0, (const uint8_t*)src, sx, sy, x0, y0, z0, bx, by, total, (uint8_t*)dst); break;
    case 2: IGN_LAUNCH(ctx, (k_copy_box<uint16_t>), g, 256, 0, (const uint16_t*)src, sx, sy, x0, y0, z0, bx, by, total, (uint16_t*)dst); break;
    case 4: IGN_LAUNCH(ctx, (k_copy_box<uint32_t>), g, 256, 0, (const uint32_t*)src, sx, sy, x0, y0, z0, bx, by, total, (uint32_t*)dst); break;
    default: IGN_LAUNCH(ctx, (k_copy_box<uint64_t>), g, 256, 0, (const uint64_t*)src, sx, sy, x0, y0, z0, bx, by, total, (uint64_t*)dst); break;
  }
  return IGN_OK;
}

// make `waiter`'s stream wait for the point where `producer` last called
// ign_timer_start(producer, slot) -- cross-stream ordering without a host sync
int ign_stream_wait_mark(ign_ctx* waiter, ign_ctx* producer, int slot) {
  IGN_REQUIRE(waiter && producer && slot >= 0 && slot < IGN_TIMER_SLOTS, IGN_ERR_INVALID, "bad stream_wait argument");
  IGN_TRY(activate(waiter));
  IGN_CUDA(cudaStreamWaitEvent(waiter->stream, producer->timers[slot][0], 0));
  return IGN_OK;
}

int ign_stream_priority(ign_ctx* ctx, int high) {
  IGN_TRY(activate(ctx));
  int least = 0, greatest = 0;
  IGN_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
  IGN_CUDA(cudaStreamSynchronize(ctx->stream));
  cudaStream_t fresh;
  IGN_CUDA(cudaStreamCreateWithPriority(&fresh, cudaStreamNonBlocking, high ? greatest : least));
  cudaStreamDestroy(ctx->stream);
  ctx->stream = fresh;
  return IGN_OK;
}

int ign_timer_start(ign_ctx* ctx, int slot) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(slot >= 0 && slot < IGN_TIMER_SLOTS, IGN_ERR_INVALID, "timer slot %d out of range", slot);
  IGN_CUDA(cudaEventRecord(ctx->timers[slot][0], ctx->stream));
  return IGN_OK;
}

int ign_timer_stop(ign_ctx* ctx, int slot) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(slot >= 0 && slot < IGN_TIMER_SLOTS, IGN_ERR_INVALID, "timer slot %d out of range", slot);
  IGN_CUDA(cudaEventRecord(ctx->timers[slot][1], ctx->stream));
  return IGN_OK;
}

int ign_timer_ms(ign_ctx* ctx, int slot, float* ms) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(slot >= 0 && slot < IGN_TIMER_SLOTS && ms, IGN_ERR_INVALID, "bad timer argument");
  IGN_CUDA(cudaEventSynchronize(ctx->timers[slot][1]));
  IGN_CUDA(cudaEventElapsedTime(ms, ctx->timers[slot][0], ctx->timers[slot][1]));
  return IGN_OK;
}

}  // extern "C"
