// remap.cu -- label glue kernels (K6, K7): renumber / remap / unique / mask /
// inverse_component_map, replacing the `fastremap` calls on the igneous hot
// path (igneous/tasks/mesh/mesh.py:201-207,318-320,368-369;
// igneous/tasks/image/ccl.py:280,346).
//
// All of them are one or two streaming passes over the volume around a small
// open-addressing hash table (64-bit keys, linear probing, atomicCAS claims)
// that lives in L2 for realistic label counts.  Roofline: HBM, algorithmic
// bytes = read + write of the volume.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace ign {

constexpr uint64_t HT_EMPTY = ~0ull;
constexpr uint32_t HT_NONE = 0xFFFFFFFFu;
constexpr unsigned FULLM = 0xFFFFFFFFu;

// The key HT_EMPTY (2^64-1) marks a free slot, so it cannot be stored in keys[]; it gets a
// side slot instead: index mask + 1, present when *side != 0, payload vals[mask + 1].  Every
// lookup of that key goes through the side slot, so all 2^64 labels are valid keys.
struct HashTable {
  uint64_t* keys;  // [cap]
  uint64_t* vals;  // [cap + 1] payload (first index / count / mapped value)
  uint32_t* side;  // present flag of the key HT_EMPTY
  uint32_t mask;   // cap - 1
};

__device__ __forceinline__ uint32_t ht_hash(uint64_t key, uint32_t mask) {
  return (uint32_t)(mix64(key) >> 17) & mask;
}

// key stored in slot s (s <= mask + 1); only meaningful for an occupied slot
__device__ __forceinline__ uint64_t ht_key(const HashTable& t, uint32_t s) {
  return s > t.mask ? HT_EMPTY : t.keys[s];
}
__device__ __forceinline__ bool ht_occupied(const HashTable& t, uint32_t s) {
  return s <= t.mask ? t.keys[s] != HT_EMPTY : (s == t.mask + 1 && *t.side != 0);
}

// returns slot of key, inserting it if absent; HT_NONE when the table is full
__device__ __forceinline__ uint32_t ht_insert(const HashTable& t, uint64_t key, uint32_t* counters) {
  if (key == HT_EMPTY) {
    if (((volatile uint32_t*)t.side)[0] == 0 && atomicExch(t.side, 1u) == 0) atomicAdd(&counters[0], 1u);
    return t.mask + 1;
  }
  uint32_t h = ht_hash(key, t.mask);
  for (uint32_t probes = 0; probes <= t.mask; probes++) {
    const uint64_t cur = ((volatile uint64_t*)t.keys)[h];
    if (cur == key) return h;
    if (cur == HT_EMPTY) {
      const uint64_t old = atomicCAS((unsigned long long*)&t.keys[h], (unsigned long long)HT_EMPTY,
                                     (unsigned long long)key);
      if (old == HT_EMPTY) {
        atomicAdd(&counters[0], 1u);
        return h;
      }
      if (old == key) return h;
    }
    h = (h + 1) & t.mask;
  }
  counters[1] = 1;  // overflow
  return HT_NONE;
}

__device__ __forceinline__ uint32_t ht_find(const HashTable& t, uint64_t key) {
  if (key == HT_EMPTY) return *t.side ? t.mask + 1 : HT_NONE;
  uint32_t h = ht_hash(key, t.mask);
  for (uint32_t probes = 0; probes <= t.mask; probes++) {
    const uint64_t cur = t.keys[h];
    if (cur == key) return h;
    if (cur == HT_EMPTY) return HT_NONE;
    h = (h + 1) & t.mask;
  }
  return HT_NONE;
}

template <typename T>
__device__ __forceinline__ uint64_t load_key(const void* p, uint64_t i) {
  return (uint64_t)((const T*)p)[i];
}

// ---- renumber pass 1: first index of every label (run heads only)
template <typename T>
__global__ void __launch_bounds__(256)
    k_first_index(const T* __restrict__ in, uint64_t n, HashTable t, uint32_t* counters) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const T v = in[i];
  if (i > 0 && in[i - 1] == v) return;
  const uint32_t h = ht_insert(t, (uint64_t)v, counters);
  if (h != HT_NONE) atomicMin((unsigned long long*)&t.vals[h], (unsigned long long)i);
}

// occupied slots (side slot included: launch over cap + 1 threads) -> (first index, slot) lists
__global__ void __launch_bounds__(256)
    k_compact_slots(HashTable t, uint64_t* __restrict__ firsts, uint32_t* __restrict__ slots,
                    uint32_t* counters) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t lane = threadIdx.x & 31;
  const bool occ = ht_occupied(t, s);
  const uint32_t m = __ballot_sync(FULLM, occ);
  if (m) {
    const int leader = __ffs(m) - 1;
    uint32_t base = 0;
    if ((int)lane == leader) base = atomicAdd(&counters[3], (uint32_t)__popc(m));
    base = __shfl_sync(FULLM, base, leader);
    if (occ) {
      const uint32_t pos = base + __popc(m & ((1u << lane) - 1u));
      firsts[pos] = t.vals[s];
      slots[pos] = s;
    }
  }
}

__global__ void __launch_bounds__(256)
    k_find_zero(HashTable t, const uint32_t* __restrict__ slots_sorted, uint32_t k,
                uint32_t* counters) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < k && ht_key(t, slots_sorted[j]) == 0) counters[4] = j;
}

__global__ void __launch_bounds__(256)
    k_assign_ids(HashTable t, const uint32_t* __restrict__ slots_sorted, uint32_t k,
                 const uint32_t* __restrict__ counters, uint64_t* __restrict__ uniq,
                 uint64_t uniq_cap) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= k) return;
  const uint32_t zero_pos = counters[4];
  const uint32_t s = slots_sorted[j];
  const uint64_t key = ht_key(t, s);
  uint64_t id = 0;
  if (key != 0) {
    id = (uint64_t)j + 1 - ((zero_pos != HT_NONE && j > zero_pos) ? 1 : 0);
    if (uniq != nullptr && id - 1 < uniq_cap) uniq[id - 1] = key;
  }
  t.vals[s] = id;
}

template <typename T, typename O>
__global__ void __launch_bounds__(256)
    k_gather(const T* __restrict__ in, uint64_t n, HashTable t, O* __restrict__ out) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t h = ht_find(t, (uint64_t)in[i]);
  out[i] = (h == HT_NONE) ? (O)0 : (O)t.vals[h];
}

// ---- remap / mask table build from (device) key / value lists
__global__ void __launch_bounds__(256)
    k_table_build(const uint64_t* __restrict__ keys, const uint64_t* __restrict__ vals, uint64_t nk,
                  HashTable t, uint32_t* counters) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= nk) return;
  const uint32_t h = ht_insert(t, keys[i], counters);
  if (h != HT_NONE) t.vals[h] = vals ? vals[i] : 1;
}

template <typename T>
__global__ void __launch_bounds__(256)
    k_remap(T* __restrict__ arr, uint64_t n, HashTable t, int preserve_missing, uint32_t* counters,
            uint64_t* missing) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const T v = arr[i];
  const uint32_t h = ht_find(t, (uint64_t)v);
  if (h != HT_NONE) {
    arr[i] = (T)t.vals[h];
  } else if (!preserve_missing) {
    if (atomicExch(&counters[5], 1u) == 0) *missing = (uint64_t)v;
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
    k_mask(T* __restrict__ arr, uint64_t n, HashTable t, int except, T value) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const bool hit = ht_find(t, (uint64_t)arr[i]) != HT_NONE;
  if (hit != (except != 0)) arr[i] = value;
}

// ---- unique with counts: one atomicAdd per run of equal values in a warp
template <typename T>
__global__ void __launch_bounds__(256)
    k_count(const T* __restrict__ in, uint64_t n, HashTable t, uint32_t* counters) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  const uint32_t lane = threadIdx.x & 31;
  const bool inb = i < n;
  const T v = inb ? in[i] : (T)0;
  unsigned long long vv = (unsigned long long)v;
  const unsigned long long vl = __shfl_up_sync(FULLM, vv, 1);
  const bool head = inb && (lane == 0 || vl != vv);
  const uint32_t hm = __ballot_sync(FULLM, head || !inb);
  if (head) {
    const uint32_t above = (lane == 31) ? 0u : (hm & ~((2u << lane) - 1u));
    const uint32_t end = above ? (uint32_t)(__ffs(above) - 1) : 32u;
    const uint32_t h = ht_insert(t, (uint64_t)v, counters);
    if (h != HT_NONE) atomicAdd((unsigned long long*)&t.vals[h], (unsigned long long)(end - lane));
  }
}

__global__ void __launch_bounds__(256)
    k_compact_kv(HashTable t, uint64_t* __restrict__ keys, uint64_t* __restrict__ vals,
                 uint32_t* counters) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t lane = threadIdx.x & 31;
  const bool occ = ht_occupied(t, s);
  const uint32_t m = __ballot_sync(FULLM, occ);
  if (m) {
    const int leader = __ffs(m) - 1;
    uint32_t base = 0;
    if ((int)lane == leader) base = atomicAdd(&counters[3], (uint32_t)__popc(m));
    base = __shfl_sync(FULLM, base, leader);
    if (occ) {
      const uint32_t pos = base + __popc(m & ((1u << lane) - 1u));
      keys[pos] = ht_key(t, s);
      vals[pos] = t.vals[s];
    }
  }
}

// ---- casts
template <typename A, typename B>
__global__ void __launch_bounds__(256) k_cast(const A* __restrict__ in, B* __restrict__ out, uint64_t n) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = (B)in[i];
}

// ---- inverse_component_map helpers
template <typename T>
__global__ void __launch_bounds__(256)
    k_widen_pairs(const T* __restrict__ p, const T* __restrict__ c, uint64_t n,
                  uint64_t* __restrict__ po, uint64_t* __restrict__ co) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i < n) {
    po[i] = (uint64_t)p[i];
    co[i] = (uint64_t)c[i];
  }
}

__global__ void __launch_bounds__(256)
    k_pair_heads(const uint64_t* __restrict__ p, const uint64_t* __restrict__ c, uint64_t n,
                 uint32_t* __restrict__ flags) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i < n) flags[i] = (i == 0 || p[i] != p[i - 1] || c[i] != c[i - 1]) ? 1u : 0u;
}

__global__ void __launch_bounds__(256)
    k_pair_scatter(const uint64_t* __restrict__ p, const uint64_t* __restrict__ c,
                   const uint32_t* __restrict__ flags, const uint32_t* __restrict__ pos, uint64_t n,
                   uint64_t* __restrict__ out, uint64_t cap) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i < n && flags[i] && pos[i] < cap) {
    out[2 * (uint64_t)pos[i]] = p[i];
    out[2 * (uint64_t)pos[i] + 1] = c[i];
  }
}

// ------------------------------------------------------------- host helpers
static uint32_t pow2_at_least(uint64_t v) {
  uint64_t c = 1024;
  while (c < v && c < (1ull << 31)) c <<= 1;
  return (uint32_t)c;
}

static int table_alloc(ign_ctx* ctx, Scratch& sc, uint32_t cap, uint64_t val_init_byte, HashTable& t,
                       uint32_t** counters) {
  t.keys = sc.take<uint64_t>(cap);
  t.vals = sc.take<uint64_t>((size_t)cap + 1);
  *counters = sc.take<uint32_t>(64);
  IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small for hash table");
  t.side = *counters + 2;
  t.mask = cap - 1;
  IGN_CUDA(cudaMemsetAsync(t.keys, 0xFF, (size_t)cap * 8, ctx->stream));
  IGN_CUDA(cudaMemsetAsync(t.vals, (int)val_init_byte, ((size_t)cap + 1) * 8, ctx->stream));
  IGN_CUDA(cudaMemsetAsync(*counters, 0, 256, ctx->stream));
  IGN_CUDA(cudaMemsetAsync(*counters + 4, 0xFF, 4, ctx->stream));  // zero_pos = NONE
  return IGN_OK;
}

static int read_counters(ign_ctx* ctx, const uint32_t* counters, uint32_t* h8) {
  IGN_TRY(small_d2h(ctx, h8, counters, 32));
  return small_sync(ctx);
}

#define DISPATCH_UINT(dtype, FN, ...)                                      \
  switch (dtype) {                                                         \
    case IGN_U8: FN(uint8_t, __VA_ARGS__); break;                          \
    case IGN_U16: FN(uint16_t, __VA_ARGS__); break;                        \
    case IGN_U32: FN(uint32_t, __VA_ARGS__); break;                        \
    case IGN_U64: FN(uint64_t, __VA_ARGS__); break;                        \
    default: set_error("unsupported label dtype %d", dtype); return IGN_ERR_UNSUPPORTED; \
  }

static size_t sort_tmp_bytes_u64(uint32_t n) {
  size_t a = 0, b = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, a, (const uint64_t*)nullptr, (uint64_t*)nullptr,
                                  (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)n);
  cub::DeviceRadixSort::SortPairs(nullptr, b, (const uint64_t*)nullptr, (uint64_t*)nullptr,
                                  (const uint64_t*)nullptr, (uint64_t*)nullptr, (int)n);
  return (a > b ? a : b) + 256;
}

// Builds the first-appearance table for `in` and assigns ids; leaves table in t.
// Retries with a larger table on overflow.  The table lives in the caller's scope `sc`.
static int renumber_table(ign_ctx* ctx, Scratch& sc, const void* in, int dtype, uint64_t n, HashTable& t,
                          uint32_t** counters_out, uint64_t* uniq_dev, uint64_t uniq_cap,
                          uint64_t* k_out) {
  IGN_REQUIRE(n < 0xFFFFFFFFull, IGN_ERR_OVERFLOW, "renumber: more than 2^32 elements");
  uint32_t cap = pow2_at_least(n < (1u << 19) ? 2 * n + 16 : (1u << 20));
  const uint32_t cap_max = pow2_at_least(2 * n + 16);
  while (true) {
    sc.rewind();
    const size_t need = (size_t)cap * 16 + (size_t)cap * (8 + 4 + 8 + 4) + sort_tmp_bytes_u64(cap) + 8192;
    IGN_TRY(sc.reserve(need));
    uint32_t* counters;
    IGN_TRY(table_alloc(ctx, sc, cap, 0xFF, t, &counters));
#define RUN_FIRST(T, dummy) IGN_LAUNCH(ctx, (k_first_index<T>), blocks_for(n, 256), 256, 0, (const T*)in, n, t, counters)
    DISPATCH_UINT(dtype, RUN_FIRST, 0)
#undef RUN_FIRST
    uint32_t h[8];
    IGN_TRY(read_counters(ctx, counters, h));
    if (h[1] != 0 || h[0] > cap / 2) {
      IGN_REQUIRE(cap < cap_max, IGN_ERR_OVERFLOW, "renumber: hash table overflow at maximum capacity");
      cap = (cap > cap_max / 8) ? cap_max : cap * 8;
      continue;
    }
    const uint32_t total = h[0];
    uint64_t* firsts = sc.take<uint64_t>((size_t)total + 1);
    uint32_t* slots = sc.take<uint32_t>((size_t)total + 1);
    uint64_t* firsts_s = sc.take<uint64_t>((size_t)total + 1);
    uint32_t* slots_s = sc.take<uint32_t>((size_t)total + 1);
    size_t tmp_bytes = sort_tmp_bytes_u64(total ? total : 1);
    void* tmp = sc.take(tmp_bytes);
    IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small (renumber)");
    uint64_t k = 0;
    if (total > 0) {
      IGN_LAUNCH(ctx, k_compact_slots, blocks_for((uint64_t)cap + 1, 256), 256, 0, t, firsts, slots, counters);
      int end_bit = 1;
      while (end_bit < 64 && (1ull << end_bit) < n) end_bit++;
      IGN_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, firsts, firsts_s, slots, slots_s,
                                               (int)total, 0, end_bit, ctx->stream));
      ctx->launches += 2;
      IGN_LAUNCH(ctx, k_find_zero, blocks_for(total, 256), 256, 0, t, slots_s, total, counters);
      IGN_LAUNCH(ctx, k_assign_ids, blocks_for(total, 256), 256, 0, t, slots_s, total, counters, uniq_dev, uniq_cap);
      IGN_TRY(read_counters(ctx, counters, h));
      k = total - (h[4] != HT_NONE ? 1 : 0);
    }
    *k_out = k;
    *counters_out = counters;
    return IGN_OK;
  }
}

}  // namespace ign

using namespace ign;

extern "C" {

int ign_cast_dev(ign_ctx* ctx, const void* in, int in_dtype, void* out, int out_dtype, uint64_t n) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(in && out, IGN_ERR_INVALID, "null buffer");
  if (n == 0) return IGN_OK;
  const unsigned g = blocks_for(n, 256);
#define CAST2(A, B) IGN_LAUNCH(ctx, (k_cast<A, B>), g, 256, 0, (const A*)in, (B*)out, n)
#define CAST1(A, dummy)                                  \
  switch (out_dtype) {                                   \
    case IGN_U8: CAST2(A, uint8_t); break;               \
    case IGN_U16: CAST2(A, uint16_t); break;             \
    case IGN_U32: CAST2(A, uint32_t); break;             \
    case IGN_U64: CAST2(A, uint64_t); break;             \
    default: set_error("cast: unsupported out dtype %d", out_dtype); return IGN_ERR_UNSUPPORTED; \
  }
  DISPATCH_UINT(in_dtype, CAST1, 0)
#undef CAST1
#undef CAST2
  return IGN_OK;
}

int ign_renumber_dev(ign_ctx* ctx, const void* in, int dtype, uint64_t n, uint32_t* out,
                     uint64_t* uniq_dev, uint64_t uniq_capacity, uint64_t* k) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(in && out && k, IGN_ERR_INVALID, "null argument");
  *k = 0;
  if (n == 0) return IGN_OK;
  Scratch sc(ctx);
  HashTable t;
  uint32_t* counters;
  IGN_TRY(renumber_table(ctx, sc, in, dtype, n, t, &counters, uniq_dev, uniq_capacity, k));
#define RUN_GATHER(T, dummy) IGN_LAUNCH(ctx, (k_gather<T, uint32_t>), blocks_for(n, 256), 256, 0, (const T*)in, n, t, out)
  DISPATCH_UINT(dtype, RUN_GATHER, 0)
#undef RUN_GATHER
  return IGN_OK;
}

int ign_renumber(ign_ctx* ctx, const void* in, int dtype, uint64_t n, uint32_t* out, uint64_t* uniq,
                 uint64_t uniq_capacity, uint64_t* k) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(in && out && k, IGN_ERR_INVALID, "null argument");
  *k = 0;
  if (n == 0) return IGN_OK;
  const int es = dtype_size(dtype);
  IGN_REQUIRE(es > 0 && dtype != IGN_F32, IGN_ERR_UNSUPPORTED, "unsupported dtype %d", dtype);
  IGN_REQUIRE(n < 0xFFFFFFFFull, IGN_ERR_OVERFLOW, "renumber: more than 2^32 elements");
  Staging st(ctx);
  void *d_in, *d_out, *d_uniq;
  st.add(&d_in, n * es, in);
  st.add(&d_out, n * 4);
  st.add(&d_uniq, uniq_capacity * 8);
  IGN_TRY(st.stage());
  IGN_TRY(ign_renumber_dev(ctx, d_in, dtype, n, (uint32_t*)d_out, (uint64_t*)d_uniq, uniq_capacity, k));
  IGN_TRY(st.back(out, d_out, n * 4));
  if (uniq) IGN_TRY(st.back(uniq, d_uniq, (*k < uniq_capacity ? *k : uniq_capacity) * 8));
  return st.sync();
}

// keys/vals are HOST arrays (the table is small); arr is a DEVICE array
int ign_remap_dev(ign_ctx* ctx, void* arr, int dtype, uint64_t n, const uint64_t* keys_host,
                  const uint64_t* vals_host, uint64_t n_keys, int preserve_missing) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(arr && (n_keys == 0 || (keys_host && vals_host)), IGN_ERR_INVALID, "null argument");
  if (n == 0) return IGN_OK;
  Scratch sc(ctx);
  const uint32_t cap = pow2_at_least(2 * n_keys + 16);
  IGN_TRY(sc.reserve((size_t)cap * 16 + n_keys * 16 + 8192));
  HashTable t;
  uint32_t* counters;
  IGN_TRY(table_alloc(ctx, sc, cap, 0, t, &counters));
  uint64_t* dk = sc.take<uint64_t>(n_keys + 1);
  uint64_t* dv = sc.take<uint64_t>(n_keys + 1);
  uint64_t* dmiss = sc.take<uint64_t>(1);
  IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small (remap)");
  if (n_keys) {
    IGN_CUDA(cudaMemcpyAsync(dk, keys_host, n_keys * 8, cudaMemcpyHostToDevice, ctx->stream));
    IGN_CUDA(cudaMemcpyAsync(dv, vals_host, n_keys * 8, cudaMemcpyHostToDevice, ctx->stream));
    IGN_LAUNCH(ctx, k_table_build, blocks_for(n_keys, 256), 256, 0, dk, dv, n_keys, t, counters);
  }
#define RUN_REMAP(T, dummy) IGN_LAUNCH(ctx, (k_remap<T>), blocks_for(n, 256), 256, 0, (T*)arr, n, t, preserve_missing, counters, dmiss)
  DISPATCH_UINT(dtype, RUN_REMAP, 0)
#undef RUN_REMAP
  uint32_t h[8];
  IGN_TRY(read_counters(ctx, counters, h));
  if (h[5] != 0) {
    uint64_t miss = 0;
    IGN_CUDA(cudaMemcpy(&miss, dmiss, 8, cudaMemcpyDeviceToHost));
    set_error("%llu", (unsigned long long)miss);  // KeyError(label), as fastremap.remap
    return IGN_ERR_KEY;
  }
  return IGN_OK;
}

int ign_remap(ign_ctx* ctx, void* arr, int dtype, uint64_t n, const uint64_t* keys,
              const uint64_t* vals, uint64_t n_keys, int preserve_missing) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(arr, IGN_ERR_INVALID, "null argument");
  if (n == 0) return IGN_OK;
  const int es = dtype_size(dtype);
  IGN_REQUIRE(es > 0 && dtype != IGN_F32, IGN_ERR_UNSUPPORTED, "unsupported dtype %d", dtype);
  Staging st(ctx);
  void* d;
  st.add(&d, n * es, arr);
  IGN_TRY(st.stage());
  IGN_TRY(ign_remap_dev(ctx, d, dtype, n, keys, vals, n_keys, preserve_missing));
  IGN_TRY(st.back(arr, d, n * es));
  return st.sync();
}

int ign_mask(ign_ctx* ctx, void* arr, int dtype, uint64_t n, const uint64_t* labels,
             uint64_t n_labels, int except, uint64_t value) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(arr && (n_labels == 0 || labels), IGN_ERR_INVALID, "null argument");
  if (n == 0) return IGN_OK;
  const int es = dtype_size(dtype);
  IGN_REQUIRE(es > 0 && dtype != IGN_F32, IGN_ERR_UNSUPPORTED, "unsupported dtype %d", dtype);
  Staging st(ctx);
  void* d;
  st.add(&d, n * es, arr);
  IGN_TRY(st.stage());
  Scratch sc(ctx);
  const uint32_t cap = pow2_at_least(2 * n_labels + 16);
  IGN_TRY(sc.reserve((size_t)cap * 16 + n_labels * 8 + 16384));
  HashTable t;
  uint32_t* counters;
  IGN_TRY(table_alloc(ctx, sc, cap, 0, t, &counters));
  uint64_t* dk = sc.take<uint64_t>(n_labels + 1);
  IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small (mask)");
  if (n_labels) {
    IGN_CUDA(cudaMemcpyAsync(dk, labels, n_labels * 8, cudaMemcpyHostToDevice, ctx->stream));
    IGN_LAUNCH(ctx, k_table_build, blocks_for(n_labels, 256), 256, 0, dk, (const uint64_t*)nullptr, n_labels, t, counters);
  }
#define RUN_MASK(T, dummy) IGN_LAUNCH(ctx, (k_mask<T>), blocks_for(n, 256), 256, 0, (T*)d, n, t, except, (T)value)
  DISPATCH_UINT(dtype, RUN_MASK, 0)
#undef RUN_MASK
  IGN_TRY(st.back(arr, d, n * es));
  return st.sync();
}

int ign_unique(ign_ctx* ctx, const void* in, int dtype, uint64_t n, uint64_t* uniq, uint64_t* counts,
               uint64_t capacity, uint64_t* k) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(in && k, IGN_ERR_INVALID, "null argument");
  *k = 0;
  if (n == 0) return IGN_OK;
  const int es = dtype_size(dtype);
  IGN_REQUIRE(es > 0 && dtype != IGN_F32, IGN_ERR_UNSUPPORTED, "unsupported dtype %d", dtype);
  IGN_REQUIRE(n < 0xFFFFFFFFull, IGN_ERR_OVERFLOW, "unique: more than 2^32 elements");
  Staging st(ctx);
  void* d_in;
  st.add(&d_in, n * es, in);
  IGN_TRY(st.stage());
  Scratch sc(ctx);
  uint32_t cap = pow2_at_least(n < (1u << 19) ? 2 * n + 16 : (1u << 20));
  const uint32_t cap_max = pow2_at_least(2 * n + 16);
  while (true) {
    sc.rewind();
    IGN_TRY(sc.reserve((size_t)cap * 16 + (size_t)cap * 32 + sort_tmp_bytes_u64(cap) + 16384));
    HashTable t;
    uint32_t* counters;
    IGN_TRY(table_alloc(ctx, sc, cap, 0, t, &counters));
#define RUN_COUNT(T, dummy) IGN_LAUNCH(ctx, (k_count<T>), blocks_for(n, 256), 256, 0, (const T*)d_in, n, t, counters)
    DISPATCH_UINT(dtype, RUN_COUNT, 0)
#undef RUN_COUNT
    uint32_t h[8];
    IGN_TRY(read_counters(ctx, counters, h));
    if (h[1] != 0 || h[0] > cap / 2) {
      IGN_REQUIRE(cap < cap_max, IGN_ERR_OVERFLOW, "unique: hash table overflow");
      cap = (cap > cap_max / 8) ? cap_max : cap * 8;
      continue;
    }
    const uint32_t total = h[0];
    *k = total;
    if (uniq != nullptr && total > 0) {
      uint64_t* ck = sc.take<uint64_t>(total);
      uint64_t* cv = sc.take<uint64_t>(total);
      uint64_t* sk = sc.take<uint64_t>(total);
      uint64_t* sv = sc.take<uint64_t>(total);
      size_t tmp_bytes = sort_tmp_bytes_u64(total);
      void* tmp = sc.take(tmp_bytes);
      IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small (unique)");
      IGN_LAUNCH(ctx, k_compact_kv, blocks_for((uint64_t)cap + 1, 256), 256, 0, t, ck, cv, counters);
      IGN_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, ck, sk, cv, sv, (int)total, 0, 64, ctx->stream));
      ctx->launches += 2;
      const uint64_t m = total < capacity ? total : capacity;
      IGN_TRY(st.back(uniq, sk, m * 8));
      if (counts) IGN_TRY(st.back(counts, sv, m * 8));
      IGN_TRY(st.sync());
    }
    return IGN_OK;
  }
}

int ign_inverse_component_map(ign_ctx* ctx, const void* parents, const void* components, int dtype,
                              uint64_t n, uint64_t* pairs, uint64_t* n_pairs) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(parents && components && n_pairs, IGN_ERR_INVALID, "null argument");
  const uint64_t capacity = *n_pairs;
  *n_pairs = 0;
  if (n == 0) return IGN_OK;
  const int es = dtype_size(dtype);
  IGN_REQUIRE(es > 0 && dtype != IGN_F32, IGN_ERR_UNSUPPORTED, "unsupported dtype %d", dtype);
  IGN_REQUIRE(n < 0x7FFFFFFFull, IGN_ERR_OVERFLOW, "inverse_component_map: too many elements");
  Staging st(ctx);
  void *dp, *dc;
  st.add(&dp, n * es, parents);
  st.add(&dc, n * es, components);
  IGN_TRY(st.stage());
  Scratch sc(ctx);
  size_t scan_bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)n);
  const size_t tmp_bytes = sort_tmp_bytes_u64((uint32_t)n) + scan_bytes;
  IGN_TRY(sc.reserve(4 * align_up(n * 8, 256) + 2 * align_up(n * 4, 256) + align_up(n * 16, 256) + tmp_bytes + 16384));
  uint64_t* p0 = sc.take<uint64_t>(n);
  uint64_t* c0 = sc.take<uint64_t>(n);
  uint64_t* p1 = sc.take<uint64_t>(n);
  uint64_t* c1 = sc.take<uint64_t>(n);
  uint32_t* flags = sc.take<uint32_t>(n);
  uint32_t* pos = sc.take<uint32_t>(n + 1);
  uint64_t* dout = sc.take<uint64_t>(2 * n);
  void* tmp = sc.take(tmp_bytes);
  IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small (inverse_component_map)");
#define RUN_WIDEN(T, dummy) IGN_LAUNCH(ctx, (k_widen_pairs<T>), blocks_for(n, 256), 256, 0, (const T*)dp, (const T*)dc, n, p0, c0)
  DISPATCH_UINT(dtype, RUN_WIDEN, 0)
#undef RUN_WIDEN
  // LSD: stable sort by component, then by parent
  size_t tb = tmp_bytes;
  IGN_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tb, c0, c1, p0, p1, (int)n, 0, 64, ctx->stream));
  tb = tmp_bytes;
  IGN_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tb, p1, p0, c1, c0, (int)n, 0, 64, ctx->stream));
  ctx->launches += 4;
  IGN_LAUNCH(ctx, k_pair_heads, blocks_for(n, 256), 256, 0, p0, c0, n, flags);
  tb = tmp_bytes;
  IGN_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, flags, pos, (int)n, ctx->stream));
  ctx->launches += 1;
  IGN_LAUNCH(ctx, k_pair_scatter, blocks_for(n, 256), 256, 0, p0, c0, flags, pos, n, dout, capacity);
  uint32_t last[2];
  IGN_CUDA(cudaMemcpyAsync(&last[0], pos + (n - 1), 4, cudaMemcpyDeviceToHost, ctx->stream));
  IGN_CUDA(cudaMemcpyAsync(&last[1], flags + (n - 1), 4, cudaMemcpyDeviceToHost, ctx->stream));
  IGN_CUDA(cudaStreamSynchronize(ctx->stream));
  const uint64_t total = (uint64_t)last[0] + last[1];
  *n_pairs = total;
  if (pairs) {
    const uint64_t m = total < capacity ? total : capacity;
    IGN_CUDA(cudaMemcpy(pairs, dout, m * 16, cudaMemcpyDeviceToHost));
  }
  return IGN_OK;
}

}  // extern "C"
