// common.cuh -- shared host/device helpers for libigneous_b200 (sm_100a only)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/igneous_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libigneous_b200 targets sm_100a (Blackwell B200) only"
#endif

namespace ign {

void set_error(const char* fmt, ...);

#define IGN_CUDA(call)                                                          \
  do {                                                                          \
    cudaError_t _e = (call);                                                    \
    if (_e != cudaSuccess) {                                                    \
      ign::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call,              \
                     cudaGetErrorString(_e));                                   \
      return IGN_ERR_CUDA;                                                      \
    }                                                                           \
  } while (0)

#define IGN_TRY(call)                 \
  do {                                \
    int _s = (call);                  \
    if (_s != IGN_OK) return _s;      \
  } while (0)

#define IGN_REQUIRE(cond, status, ...)   \
  do {                                   \
    if (!(cond)) {                       \
      ign::set_error(__VA_ARGS__);       \
      return (status);                   \
    }                                    \
  } while (0)

static inline int dtype_size(int dt) {
  switch (dt) {
    case IGN_U8: return 1;
    case IGN_U16: return 2;
    case IGN_U32: return 4;
    case IGN_U64: return 8;
    case IGN_F32: return 4;
    default: return 0;
  }
}

}  // namespace ign

constexpr int IGN_TIMER_SLOTS = 64;  // CUDA event pairs per context: timers and cross-stream marks

struct ign_ctx {
  int device;
  int sm_count;
  cudaStream_t stream;
  cudaStream_t copy_stream;
  // grow-only device scratch arena, bump allocated through ign::Scratch
  char* scratch;
  size_t scratch_bytes;
  size_t scratch_used;
  // grow-only device copies of the host-buffer entry points' arrays (ign::Staging)
  char* stage;
  size_t stage_bytes;
  char* pinned;  // staging for scalars / small results
  size_t pinned_bytes;
  cudaEvent_t timers[IGN_TIMER_SLOTS][2];
  uint64_t launches;
  // optional per-kernel-class profiling (ign_prof_enable): CUDA events recorded
  // on the ctx stream around selected launches
  int prof_on;
  struct ProfRec { int cls; cudaEvent_t a, b; };
  ProfRec* prof;
  int prof_n, prof_cap;
  // grow-only pool for the result buffers of the (normally single) live mesher:
  // cudaMalloc/cudaFree per task serialise on the driver lock
  char* mesh_pool;
  size_t mesh_pool_bytes;
  int mesh_pool_busy;
  // mapped pinned window for small control transfers (see ign::small_d2h)
  char* win;      // host address
  char* win_dev;  // the same bytes as seen by kernels
  size_t win_fetch_used, win_push_used;
  struct FetchRec { void* dst; size_t off, bytes; };
  FetchRec fetch[32];
  int fetch_n;
};

enum { IGN_PROF_CCL_LOCAL = 0, IGN_PROF_CCL_MERGE = 1, IGN_PROF_CCL_LABEL = 2, IGN_PROF_POOL = 3,
       IGN_PROF_MC = 4, IGN_PROF_SIMP = 5, IGN_PROF_CLASSES = 8 };

namespace ign {

// Make `ctx->device` current (one ctx per process is the contract, but be safe).
int activate(ign_ctx* ctx);

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Grow a grow-only device buffer to at least `need` bytes (plus a quarter, so that slowly rising
// sizes do not reallocate every call).  The contents are dropped; work queued on ctx->stream is
// waited for first, since it may still use the old buffer.
int grow_buffer(ign_ctx* ctx, char** buf, size_t* have, size_t need, const char* what);

// One function's use of the scratch arena.  Construct it at the top of every function that takes
// from the arena; its destructor gives the bytes back on every return path.  The scope owns the
// arena iff nothing is held below it: the outermost call, with no CCL volume open.  Only the owner
// grows the arena, since growing moves it; a nested scope lives in the room its caller reserved.
class Scratch {
 public:
  explicit Scratch(ign_ctx* ctx) : Scratch(ctx, ctx->scratch_used) {}
  // adopts the bytes a kept scope with this base still holds: they are released with this scope
  Scratch(ign_ctx* ctx, size_t base) : ctx_(ctx), base_(base) {}
  ~Scratch() {
    if (!kept_) ctx_->scratch_used = base_;
  }
  Scratch(const Scratch&) = delete;
  Scratch& operator=(const Scratch&) = delete;

  bool owner() const { return base_ == 0; }
  // owner: make the arena at least `bytes` (call before the first take); nested: nothing
  int reserve(size_t bytes);
  // `count` elements, 256 B aligned; nullptr when they do not fit, and ok() turns false
  template <typename T = char>
  T* take(size_t count) { return (T*)take_bytes(count * sizeof(T)); }
  bool ok() const { return ok_; }
  // back to the base: every take of this scope is released
  void rewind();
  // leave the bytes held past this scope; returns the base to release them to later
  size_t keep() {
    kept_ = true;
    return base_;
  }

 private:
  void* take_bytes(size_t bytes);
  ign_ctx* ctx_;
  size_t base_;
  bool ok_ = true, kept_ = false;
};

// Device copies of a host-buffer entry point's arrays, in the context's grow-only staging buffer.
// They sit outside the scratch arena, so the _dev function the entry point calls sizes its own
// arena use.  add() every slot, stage(), call the _dev function, back() its results, sync().
class Staging {
 public:
  explicit Staging(ign_ctx* ctx) : ctx_(ctx) {}
  // a device slot of `bytes` (nullptr if 0), filled from `host` unless that is null
  void add(void** dev, size_t bytes, const void* host = nullptr) { slots_.push_back({dev, bytes, host}); }
  // grows the buffer, sets every slot pointer and queues the host -> device copies
  int stage();
  // queues a device -> host copy of a result
  int back(void* host, const void* dev, size_t bytes);
  // waits for the copies
  int sync();

 private:
  struct Slot {
    void** dev;
    size_t bytes;
    const void* host;
  };
  ign_ctx* ctx_;
  std::vector<Slot> slots_;
};

// Small control transfers (counters, per-label offset tables) that sit between kernels
// of one call.  cudaMemcpyAsync would put them on a copy engine, where they queue behind
// multi-GB transfers issued by other contexts of the same device (the volume upload /
// label download that overlap the mesh stage).  Instead a copy kernel on the ctx stream
// moves them through a mapped pinned window, so only the SMs and the stream order are
// involved.  Transfers that do not fit the window fall back to cudaMemcpyAsync.
//   small_d2h: host_dst is valid after small_sync().
//   small_h2d: host_src is consumed before the call returns.
//   small_sync: cudaStreamSynchronize(ctx->stream) + delivery of pending small_d2h results.
int small_d2h(ign_ctx* ctx, void* host_dst, const void* dev_src, size_t bytes);
// bulk device -> pinned host copy issued as a kernel on the ctx stream (falls back to the copy engine for pageable memory)
int d2h_by_kernel(ign_ctx* ctx, void* host_dst, const void* dev_src, size_t bytes);
int small_h2d(ign_ctx* ctx, void* dev_dst, const void* host_src, size_t bytes);
int small_sync(ign_ctx* ctx);

// launch bookkeeping: every kernel launch in this library goes through
// IGN_LAUNCH so ign_launch_count() is exact.
#define IGN_LAUNCH(ctx, kernel, grid, block, smem, ...)                          \
  do {                                                                           \
    kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);             \
    (ctx)->launches++;                                                           \
    IGN_CUDA(cudaGetLastError());                                                \
  } while (0)

// profiled launch: like IGN_LAUNCH, plus an event pair when profiling is on
int prof_begin(ign_ctx* ctx, int cls);
void prof_end(ign_ctx* ctx, int slot);
#define IGN_LAUNCH_PROF(ctx, cls, kernel, grid, block, smem, ...)                 \
  do {                                                                           \
    const int _slot = ign::prof_begin((ctx), (cls));                             \
    kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);             \
    (ctx)->launches++;                                                           \
    ign::prof_end((ctx), _slot);                                                 \
    IGN_CUDA(cudaGetLastError());                                                \
  } while (0)

static inline unsigned blocks_for(uint64_t n, unsigned threads) {
  return (unsigned)((n + threads - 1) / threads);
}

}  // namespace ign

// ------------------------------------------------------------------ device
#ifdef __CUDACC__
namespace ign {

__device__ __forceinline__ uint4 ld_stream(const void* p) {
  // streaming 128-bit load: read-only path, do not allocate in L1
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream(void* p, uint4 v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x),
               "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}
__device__ __forceinline__ void st_stream(void* p, uint2 v) {
  asm volatile("st.global.L1::no_allocate.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(v.x), "r"(v.y)
               : "memory");
}

__device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

}  // namespace ign
#endif
