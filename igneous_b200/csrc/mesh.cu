// mesh.cu -- multi-label marching cubes (K8) + per-label vertex welding (K9)
//
// Replaces zmesh.Mesher.mesh / ids / get as called from
// igneous/tasks/mesh/mesh.py:151,245,371-383.
//
//   renumber   labels -> dense 1..K (shares remap.cu's hash table kernels)
//   count      one thread per 2x2x2 cube (x fastest, corners through L1): for
//              every distinct non-zero corner label the 256-case table gives a
//              triangle count; warp-reduced, one atomicAdd per warp.
//   emit       same walk; a warp prefix-sum + ONE atomicAdd per warp reserves a
//              contiguous slice of the compacted triangle buffer
//              (warp-aggregated atomics); records are 64-bit keys
//              [label | cube | t] + the 8-bit case index.
//   sort       radix sort of the keys -> per label, cube raster order
//              (deterministic whatever order the atomics resolved in).
//   weld       3 vertex keys [label | z | y | x] (half-voxel lattice) per
//              triangle, radix sorted; heads of runs are the unique vertices;
//              an exclusive scan ranks them; faces index them per label.
// Roofline: HBM-bound streaming over the label volume for count/emit
// (algorithmic bytes = sizeof(label) per voxel); the sorts are bound by the
// surface size, not the volume.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <atomic>
#include <memory>
#include <vector>

#include "common.cuh"
#include "mc_table.h"

namespace ign {

constexpr unsigned MFULL = 0xFFFFFFFFu;
constexpr int TRI_T_BITS = 3, TRI_CUBE_BITS = 30;
constexpr int V_COORD_BITS = 11;
constexpr int V_LABEL_SHIFT = 3 * V_COORD_BITS;  // 33
constexpr int TRI_LABEL_SHIFT = TRI_T_BITS + TRI_CUBE_BITS;  // 33

__constant__ int8_t c_edge_mid[12][3] = {{1, 0, 0}, {2, 1, 0}, {1, 2, 0}, {0, 1, 0},
                                         {1, 0, 2}, {2, 1, 2}, {1, 2, 2}, {0, 1, 2},
                                         {0, 0, 1}, {2, 0, 1}, {2, 2, 1}, {0, 2, 1}};

struct McTables {
  int8_t tri[256][16];
  uint8_t ntri[256];
};
__constant__ McTables c_mc;

// corner k of Bourke's numbering -> offset (dx,dy,dz)
__device__ __forceinline__ void cube_corners(const uint32_t* __restrict__ lab, uint32_t sx,
                                             uint32_t sxy, uint32_t base, uint32_t (&c)[8]) {
  c[0] = lab[base];
  c[1] = lab[base + 1];
  c[2] = lab[base + 1 + sx];
  c[3] = lab[base + sx];
  c[4] = lab[base + sxy];
  c[5] = lab[base + 1 + sxy];
  c[6] = lab[base + 1 + sx + sxy];
  c[7] = lab[base + sx + sxy];
}

// EMIT=false: count triangles; EMIT=true: write records
template <bool EMIT>
__global__ void __launch_bounds__(256)
    k_mc(const uint32_t* __restrict__ lab, uint32_t sx, uint32_t sy, uint32_t sz,
         unsigned long long* total, uint64_t* __restrict__ keys, uint8_t* __restrict__ cases,
         uint64_t capacity) {
  __shared__ uint8_t s_ntri[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_ntri[i] = c_mc.ntri[i];
  __syncthreads();
  const uint32_t cx = sx - 1, cy = sy - 1, cz = sz - 1;
  const uint64_t ncubes = (uint64_t)cx * cy * cz;
  const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  const uint32_t lane = threadIdx.x & 31;
  uint32_t mine = 0;
  uint32_t c[8];
  uint32_t x = 0, y = 0, z = 0;
  bool active = false;
  if (t < ncubes) {
    x = (uint32_t)(t % cx);
    y = (uint32_t)((t / cx) % cy);
    z = (uint32_t)(t / ((uint64_t)cx * cy));
    cube_corners(lab, sx, sx * sy, (z * sy + y) * sx + x, c);
    const uint32_t o = c[0] | c[1] | c[2] | c[3] | c[4] | c[5] | c[6] | c[7];
    const bool same = (c[0] == c[1]) & (c[0] == c[2]) & (c[0] == c[3]) & (c[0] == c[4]) &
                      (c[0] == c[5]) & (c[0] == c[6]) & (c[0] == c[7]);
    active = (o != 0) && !same;
  }
  uint8_t idxs[8];
  if (active) {
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const uint32_t L = c[k];
      bool first = (L != 0);
#pragma unroll
      for (int j = 0; j < 8; j++)
        if (j < k) first = first && (c[j] != L);
      uint32_t idx = 0;
#pragma unroll
      for (int j = 0; j < 8; j++) idx |= (uint32_t)(c[j] == L) << j;
      idxs[k] = first ? (uint8_t)idx : 0;  // case 0 emits nothing
      mine += s_ntri[idxs[k]];
    }
  }
  if (!EMIT) {
    uint32_t s = mine;
    for (int d = 16; d > 0; d >>= 1) s += __shfl_down_sync(MFULL, s, d);
    if (lane == 0 && s) atomicAdd(total, (unsigned long long)s);
    return;
  }
  // warp-aggregated reservation
  uint32_t incl = mine;
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t v = __shfl_up_sync(MFULL, incl, d);
    if (lane >= d) incl += v;
  }
  const uint32_t warp_total = __shfl_sync(MFULL, incl, 31);
  if (warp_total == 0) return;
  unsigned long long base = 0;
  if (lane == 31) base = atomicAdd(total, (unsigned long long)warp_total);
  base = __shfl_sync(MFULL, base, 31);
  uint64_t pos = base + (incl - mine);
  if (active) {
    const uint64_t cube = (uint64_t)t;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const uint32_t n = s_ntri[idxs[k]];
      for (uint32_t tt = 0; tt < n; tt++) {
        if (pos < capacity) {
          keys[pos] = ((uint64_t)c[k] << TRI_LABEL_SHIFT) | (cube << TRI_T_BITS) | tt;
          cases[pos] = idxs[k];
        }
        pos++;
      }
    }
  }
}

// triangle records (sorted) -> 3 vertex keys each
__global__ void __launch_bounds__(256)
    k_tri_vertices(const uint64_t* __restrict__ keys, const uint8_t* __restrict__ cases, uint64_t T,
                   uint32_t cx, uint32_t cy, uint64_t* __restrict__ vkeys,
                   uint32_t* __restrict__ corner) {
  const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (t >= T) return;
  const uint64_t key = keys[t];
  const uint64_t label = key >> TRI_LABEL_SHIFT;
  const uint64_t cube = (key >> TRI_T_BITS) & ((1ull << TRI_CUBE_BITS) - 1);
  const uint32_t tt = (uint32_t)(key & ((1u << TRI_T_BITS) - 1));
  const uint32_t x = (uint32_t)(cube % cx), y = (uint32_t)((cube / cx) % cy),
                 z = (uint32_t)(cube / ((uint64_t)cx * cy));
  const int8_t* row = c_mc.tri[cases[t]];
#pragma unroll
  for (int v = 0; v < 3; v++) {
    // table winds clockwise seen from outside for "bit = inside"; reverse it so
    // that normals point out of the label (oracle.marching_cubes flip=True)
    const int e = row[3 * tt + (2 - v)];
    const uint64_t vx = 2 * x + c_edge_mid[e][0], vy = 2 * y + c_edge_mid[e][1],
                   vz = 2 * z + c_edge_mid[e][2];
    vkeys[3 * t + v] = (label << V_LABEL_SHIFT) | (vz << (2 * V_COORD_BITS)) | (vy << V_COORD_BITS) | vx;
    corner[3 * t + v] = (uint32_t)(3 * t + v);
  }
}

// boundaries in a sorted array of keys -> per-label [start) markers
__global__ void __launch_bounds__(256)
    k_label_starts(const uint64_t* __restrict__ keys, uint64_t n, int shift,
                   uint32_t* __restrict__ start /* [K+2], prefilled with n */) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t label = keys[i] >> shift;
  if (i == 0 || (keys[i - 1] >> shift) != label) start[label] = (uint32_t)i;
}

__global__ void __launch_bounds__(256) k_fill_u32(uint32_t* a, uint32_t value, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] = value;
}

__global__ void __launch_bounds__(256)
    k_vertex_heads(const uint64_t* __restrict__ vkeys_sorted, uint64_t n, uint32_t* __restrict__ heads) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i < n) heads[i] = (i == 0 || vkeys_sorted[i - 1] != vkeys_sorted[i]) ? 1u : 0u;
}

// heads + exclusive scan -> unique vertex list and global vertex id per corner
__global__ void __launch_bounds__(256)
    k_vertex_assign(const uint64_t* __restrict__ vkeys_sorted, const uint32_t* __restrict__ corner_sorted,
                    const uint32_t* __restrict__ heads, const uint32_t* __restrict__ rank, uint64_t n,
                    uint64_t* __restrict__ uniq_vkeys, uint32_t* __restrict__ face_global) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t id = rank[i] + heads[i] - 1;  // inclusive rank - 1
  if (heads[i]) uniq_vkeys[id] = vkeys_sorted[i];
  face_global[corner_sorted[i]] = id;
}

// global vertex ids -> ids local to the label
__global__ void __launch_bounds__(256)
    k_faces_local(const uint64_t* __restrict__ tri_keys, const uint32_t* __restrict__ vert_off,
                  uint64_t T, uint32_t* __restrict__ faces) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= 3 * T) return;
  const uint64_t label = tri_keys[i / 3] >> TRI_LABEL_SHIFT;
  faces[i] -= vert_off[label];
}

__global__ void __launch_bounds__(256)
    k_vertex_positions(const uint64_t* __restrict__ uniq_vkeys, uint64_t first, uint64_t count,
                       float rx, float ry, float rz, float shift, float* __restrict__ out) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= count) return;
  const uint64_t k = uniq_vkeys[first + i];
  const float x = (float)(k & ((1u << V_COORD_BITS) - 1));
  const float y = (float)((k >> V_COORD_BITS) & ((1u << V_COORD_BITS) - 1));
  const float z = (float)((k >> (2 * V_COORD_BITS)) & ((1u << V_COORD_BITS) - 1));
  out[3 * i + 0] = __fmul_rn(__fadd_rn(__fmul_rn(x, 0.5f), shift), rx);
  out[3 * i + 1] = __fmul_rn(__fadd_rn(__fmul_rn(y, 0.5f), shift), ry);
  out[3 * i + 2] = __fmul_rn(__fadd_rn(__fmul_rn(z, 0.5f), shift), rz);
}

}  // namespace ign

#include "mesher.h"

namespace ign {
int simp_export_positions(ign_ctx* ctx, const float* pos_f, uint64_t first, uint64_t count,
                          const float shift[3], float* d_out);
}
using namespace ign;

// positions of vertices [first, first+count) into d_out (device), whichever form the mesher holds
static int mesher_positions(ign_mesher* m, uint64_t first, uint64_t count, const float resolution[3],
                            int voxel_centered, float* d_out) {
  ign_ctx* ctx = m->ctx;
  if (m->simplified) {
    IGN_REQUIRE(resolution[0] == m->res[0] && resolution[1] == m->res[1] && resolution[2] == m->res[2],
                IGN_ERR_INVALID, "resolution differs from the one the mesher was simplified with");
    const float shift[3] = {voxel_centered ? 0.5f * m->res[0] : 0.0f, voxel_centered ? 0.5f * m->res[1] : 0.0f,
                            voxel_centered ? 0.5f * m->res[2] : 0.0f};
    return simp_export_positions(ctx, m->d_pos_f, first, count, shift, d_out);
  }
  IGN_LAUNCH(ctx, k_vertex_positions, blocks_for(count, 256), 256, 0, m->d_uniq_vkeys, first, count,
             resolution[0], resolution[1], resolution[2], voxel_centered ? 0.5f : 0.0f, d_out);
  return IGN_OK;
}

// one flag per device; set after the upload has completed (mesh streams of one device share it)
static std::atomic<bool> g_tables_loaded[64];

static int load_tables(ign_ctx* ctx) {
  if (ctx->device < 64 && g_tables_loaded[ctx->device]) return IGN_OK;
  McTables h;
  memcpy(h.tri, mc_tri_table, sizeof(h.tri));
  memcpy(h.ntri, mc_tri_count, sizeof(h.ntri));
  IGN_CUDA(cudaMemcpyToSymbolAsync(c_mc, &h, sizeof(h), 0, cudaMemcpyHostToDevice, ctx->stream));
  IGN_CUDA(cudaStreamSynchronize(ctx->stream));
  if (ctx->device < 64) g_tables_loaded[ctx->device] = true;
  return IGN_OK;
}

static int bits_for(uint64_t v) {
  int b = 1;
  while (b < 64 && (1ull << b) <= v) b++;
  return b;
}

extern "C" {

int ign_mesh_free(ign_mesher* m) {
  if (!m) return IGN_OK;
  cudaSetDevice(m->ctx->device);
  if (m->pooled) {
    m->ctx->mesh_pool_busy = 0;
  } else {
    if (m->d_uniq_vkeys) cudaFree(m->d_uniq_vkeys);
    if (m->d_faces) cudaFree(m->d_faces);
  }
  delete m;
  return IGN_OK;
}

// frees a mesher that ign_mesh_begin_dev could not finish
struct MesherFree {
  void operator()(ign_mesher* m) const { ign_mesh_free(m); }
};

int ign_mesh_begin_dev(ign_ctx* ctx, const void* labels, int dtype, uint64_t sx, uint64_t sy,
                       uint64_t sz, ign_mesher** out) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(labels && out, IGN_ERR_INVALID, "null argument");
  *out = nullptr;
  IGN_REQUIRE(sx >= 1 && sy >= 1 && sz >= 1, IGN_ERR_INVALID, "empty volume");
  IGN_REQUIRE(sx <= 1023 && sy <= 1023 && sz <= 1023, IGN_ERR_UNSUPPORTED,
              "mesher: task of %llux%llux%llu exceeds the 1023^3 limit of the packed vertex format",
              (unsigned long long)sx, (unsigned long long)sy, (unsigned long long)sz);
  IGN_TRY(load_tables(ctx));
  const uint64_t n = sx * sy * sz;
  Scratch sc(ctx);

  std::unique_ptr<ign_mesher, MesherFree> m(new ign_mesher());
  m->ctx = ctx;
  m->K = m->T = m->U = 0;
  m->d_uniq_vkeys = nullptr;
  m->d_faces = nullptr;
  m->pooled = false;
  m->simplified = false;
  m->d_pos_f = nullptr;
  m->simp_factor = 0;
  m->simp_max_error = 0;
  m->simp_rounds = 0;

  // ---- dense labels
  uint64_t cap2 = 1024;
  while (cap2 < 2 * n + 16 && cap2 < (1ull << 31)) cap2 <<= 1;
  const size_t renumber_need = cap2 * 40 + (1 << 20);
  IGN_TRY(sc.reserve(align_up(n * 4, 256) + align_up(n * 8, 256) + renumber_need + (64 << 20)));
  uint32_t* d_lab = sc.take<uint32_t>(n);
  uint64_t* d_uniq = sc.take<uint64_t>(n);
  IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small (mesher labels)");
  uint64_t K = 0;
  IGN_TRY(ign_renumber_dev(ctx, labels, dtype, n, d_lab, d_uniq, n, &K));
  m->K = K;
  m->ids.resize(K);
  if (K) {
    IGN_TRY(small_d2h(ctx, m->ids.data(), d_uniq, K * 8));
    IGN_TRY(small_sync(ctx));
  }
  m->tri_off.assign(K + 2, 0);
  m->vert_off.assign(K + 2, 0);
  if (K == 0 || sx < 2 || sy < 2 || sz < 2) {
    *out = m.release();
    return IGN_OK;
  }
  IGN_REQUIRE(K < (1ull << 31), IGN_ERR_OVERFLOW, "mesher: too many labels");
  // the arena below d_uniq is reusable now: only d_lab must survive
  sc.rewind();
  d_lab = sc.take<uint32_t>(n);

  // ---- count
  unsigned long long* d_total = sc.take<unsigned long long>(32);
  const uint64_t ncubes = (sx - 1) * (sy - 1) * (sz - 1);
  const unsigned grid = blocks_for(ncubes, 256);
  unsigned long long T = 0;
  IGN_CUDA(cudaMemsetAsync(d_total, 0, 8, ctx->stream));
  IGN_LAUNCH(ctx, (k_mc<false>), grid, 256, 0, d_lab, (uint32_t)sx, (uint32_t)sy, (uint32_t)sz, d_total,
             (uint64_t*)nullptr, (uint8_t*)nullptr, 0ull);
  IGN_TRY(small_d2h(ctx, &T, d_total, 8));
  IGN_TRY(small_sync(ctx));
  m->T = T;
  if (T == 0) {
    *out = m.release();
    return IGN_OK;
  }
  IGN_REQUIRE(3 * T < 0xFFFFFFFFull, IGN_ERR_OVERFLOW, "mesher: %llu triangles exceed 32-bit corner indices", T);

  // ---- arena plan for emit + sort + weld
  size_t sort1 = 0, sort2 = 0, scanb = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort1, (const uint64_t*)nullptr, (uint64_t*)nullptr,
                                  (const uint8_t*)nullptr, (uint8_t*)nullptr, (int)T);
  cub::DeviceRadixSort::SortPairs(nullptr, sort2, (const uint64_t*)nullptr, (uint64_t*)nullptr,
                                  (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)(3 * T));
  cub::DeviceScan::ExclusiveSum(nullptr, scanb, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)(3 * T));
  size_t tmp_bytes = sort1 > sort2 ? sort1 : sort2;
  if (scanb > tmp_bytes) tmp_bytes = scanb;
  const size_t need = align_up(n * 4, 256) + 2 * align_up(T * 8, 256) + 2 * align_up(T, 256) +
                      2 * align_up(3 * T * 8, 256) + 4 * align_up(3 * T * 4, 256) +
                      2 * align_up((K + 2) * 4, 256) + tmp_bytes + (1 << 20);
  if (sc.owner() && need > ctx->scratch_bytes) {
    // growing the arena invalidates d_lab: re-run the (cheap) renumber into the new arena
    sc.rewind();
    IGN_TRY(sc.reserve(need + renumber_need + align_up(n * 8, 256)));
    d_lab = sc.take<uint32_t>(n);
    uint64_t* d_uniq2 = sc.take<uint64_t>(n);
    uint64_t K2 = 0;
    IGN_TRY(ign_renumber_dev(ctx, labels, dtype, n, d_lab, d_uniq2, n, &K2));
    sc.rewind();
    d_lab = sc.take<uint32_t>(n);
    d_total = sc.take<unsigned long long>(32);
  }
  uint64_t* keys = sc.take<uint64_t>(T);
  uint64_t* keys_s = sc.take<uint64_t>(T);
  uint8_t* cases = sc.take<uint8_t>(T);
  uint8_t* cases_s = sc.take<uint8_t>(T);
  uint64_t* vkeys = sc.take<uint64_t>(3 * T);
  uint64_t* vkeys_s = sc.take<uint64_t>(3 * T);
  uint32_t* corner = sc.take<uint32_t>(3 * T);
  uint32_t* corner_s = sc.take<uint32_t>(3 * T);
  uint32_t* heads = sc.take<uint32_t>(3 * T);
  uint32_t* rank = sc.take<uint32_t>(3 * T);
  uint32_t* d_tri_off = sc.take<uint32_t>(K + 2);
  uint32_t* d_vert_off = sc.take<uint32_t>(K + 2);
  void* tmp = sc.take(tmp_bytes);
  IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small (mesher: %llu triangles)", T);

  // ---- emit + sort
  IGN_CUDA(cudaMemsetAsync(d_total, 0, 8, ctx->stream));
  IGN_LAUNCH(ctx, (k_mc<true>), grid, 256, 0, d_lab, (uint32_t)sx, (uint32_t)sy, (uint32_t)sz, d_total, keys,
             cases, (uint64_t)T);
  const int label_bits = bits_for(K);
  size_t tb = tmp_bytes;
  IGN_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tb, keys, keys_s, cases, cases_s, (int)T, 0,
                                           TRI_LABEL_SHIFT + label_bits, ctx->stream));
  ctx->launches += 4;

  // ---- weld
  IGN_LAUNCH(ctx, k_tri_vertices, blocks_for(T, 256), 256, 0, keys_s, cases_s, (uint64_t)T, (uint32_t)(sx - 1),
             (uint32_t)(sy - 1), vkeys, corner);
  tb = tmp_bytes;
  IGN_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tb, vkeys, vkeys_s, corner, corner_s, (int)(3 * T), 0,
                                           V_LABEL_SHIFT + label_bits, ctx->stream));
  ctx->launches += 4;
  IGN_LAUNCH(ctx, k_vertex_heads, blocks_for(3 * T, 256), 256, 0, vkeys_s, (uint64_t)(3 * T), heads);
  tb = tmp_bytes;
  IGN_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, heads, rank, (int)(3 * T), ctx->stream));
  ctx->launches += 2;
  uint32_t last[2];
  IGN_TRY(small_d2h(ctx, &last[0], rank + (3 * T - 1), 4));
  IGN_TRY(small_d2h(ctx, &last[1], heads + (3 * T - 1), 4));
  IGN_TRY(small_sync(ctx));
  const uint64_t U = (uint64_t)last[0] + last[1];
  m->U = U;
  {
    const size_t fbytes = align_up(3 * T * 4, 256), vbytes = align_up(U * 12, 256);  // 12: float3 after simplify
    if (!ctx->mesh_pool_busy) {
      IGN_TRY(grow_buffer(ctx, &ctx->mesh_pool, &ctx->mesh_pool_bytes, fbytes + vbytes, "mesh pool"));
      m->d_faces = (uint32_t*)ctx->mesh_pool;
      m->d_uniq_vkeys = (uint64_t*)(ctx->mesh_pool + fbytes);
      m->pooled = true;
      ctx->mesh_pool_busy = 1;
    } else {
      IGN_CUDA(cudaMalloc((void**)&m->d_faces, 3 * T * 4));
      IGN_CUDA(cudaMalloc((void**)&m->d_uniq_vkeys, U * 12));  // 12: float3 positions after simplification
    }
  }
  IGN_LAUNCH(ctx, k_vertex_assign, blocks_for(3 * T, 256), 256, 0, vkeys_s, corner_s, heads, rank,
             (uint64_t)(3 * T), m->d_uniq_vkeys, m->d_faces);

  // ---- per-label offsets (labels are 1..K; slot K+1 is the end sentinel)
  IGN_LAUNCH(ctx, k_fill_u32, blocks_for(K + 2, 256), 256, 0, d_tri_off, (uint32_t)T, (uint32_t)(K + 2));
  IGN_LAUNCH(ctx, k_fill_u32, blocks_for(K + 2, 256), 256, 0, d_vert_off, (uint32_t)U, (uint32_t)(K + 2));
  IGN_LAUNCH(ctx, k_label_starts, blocks_for(T, 256), 256, 0, keys_s, (uint64_t)T, TRI_LABEL_SHIFT, d_tri_off);
  IGN_LAUNCH(ctx, k_label_starts, blocks_for(U, 256), 256, 0, m->d_uniq_vkeys, U, V_LABEL_SHIFT, d_vert_off);
  IGN_TRY(small_d2h(ctx, m->tri_off.data(), d_tri_off, (K + 2) * 4));
  IGN_TRY(small_d2h(ctx, m->vert_off.data(), d_vert_off, (K + 2) * 4));
  IGN_TRY(small_sync(ctx));
  // absent labels hold the end marker: a suffix minimum turns starts into offsets
  for (int64_t l = (int64_t)K; l >= 0; l--) {
    if (m->tri_off[l] > m->tri_off[l + 1]) m->tri_off[l] = m->tri_off[l + 1];
    if (m->vert_off[l] > m->vert_off[l + 1]) m->vert_off[l] = m->vert_off[l + 1];
  }
  IGN_TRY(small_h2d(ctx, d_vert_off, m->vert_off.data(), (K + 2) * 4));
  IGN_LAUNCH(ctx, k_faces_local, blocks_for(3 * T, 256), 256, 0, keys_s, d_vert_off, (uint64_t)T, m->d_faces);
  IGN_CUDA(cudaStreamSynchronize(ctx->stream));
  for (uint64_t l = 1; l <= K; l++)
    if (m->tri_off[l + 1] > m->tri_off[l]) m->present.push_back(m->ids[l - 1]);
  *out = m.release();
  return IGN_OK;
}

int ign_mesh_begin(ign_ctx* ctx, const void* labels, int dtype, uint64_t sx, uint64_t sy, uint64_t sz,
                   ign_mesher** out) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(labels && out, IGN_ERR_INVALID, "null argument");
  const int es = dtype_size(dtype);
  IGN_REQUIRE(es > 0 && dtype != IGN_F32, IGN_ERR_UNSUPPORTED, "unsupported dtype %d", dtype);
  Staging st(ctx);
  void* d;
  st.add(&d, sx * sy * sz * es, labels);
  IGN_TRY(st.stage());
  IGN_TRY(ign_mesh_begin_dev(ctx, d, dtype, sx, sy, sz, out));
  return st.sync();
}

int ign_mesh_num_ids(ign_mesher* m, uint64_t* n) {
  IGN_REQUIRE(m && n, IGN_ERR_INVALID, "null argument");
  *n = m->present.size();
  return IGN_OK;
}

int ign_mesh_ids(ign_mesher* m, uint64_t* ids, uint64_t capacity) {
  IGN_REQUIRE(m && ids, IGN_ERR_INVALID, "null argument");
  const uint64_t k = m->present.size() < capacity ? m->present.size() : capacity;
  for (uint64_t i = 0; i < k; i++) ids[i] = m->present[i];
  return IGN_OK;
}

int ign_mesh_totals(ign_mesher* m, uint64_t* nv, uint64_t* nf) {
  IGN_REQUIRE(m && nv && nf, IGN_ERR_INVALID, "null argument");
  *nv = m->U;
  *nf = m->T;
  return IGN_OK;
}

static int64_t dense_of(ign_mesher* m, uint64_t id) {
  // ids[] is in first-appearance order, not sorted: linear scan is fine for the
  // per-id API (bulk export does not need it)
  for (uint64_t i = 0; i < m->ids.size(); i++)
    if (m->ids[i] == id) return (int64_t)i + 1;
  return -1;
}

int ign_mesh_counts(ign_mesher* m, uint64_t id, uint64_t* nv, uint64_t* nf) {
  IGN_REQUIRE(m && nv && nf, IGN_ERR_INVALID, "null argument");
  const int64_t l = dense_of(m, id);
  IGN_REQUIRE(l > 0, IGN_ERR_KEY, "%llu", (unsigned long long)id);
  *nv = m->vert_off[l + 1] - m->vert_off[l];
  *nf = m->tri_off[l + 1] - m->tri_off[l];
  return IGN_OK;
}

int ign_mesh_get(ign_mesher* m, uint64_t id, const float resolution[3], int reduction_factor,
                 float max_error, int voxel_centered, float* vertices, uint32_t* faces, uint64_t* nv,
                 uint64_t* nf) {
  IGN_REQUIRE(m && resolution && nv && nf, IGN_ERR_INVALID, "null argument");
  ign_ctx* ctx = m->ctx;
  IGN_TRY(activate(ctx));
  if (reduction_factor > 0 && !m->simplified) IGN_TRY(ign_mesh_simplify(m, resolution, reduction_factor, max_error));
  if (m->simplified) {
    IGN_REQUIRE(reduction_factor == m->simp_factor && max_error == m->simp_max_error, IGN_ERR_INVALID,
                "mesher was simplified with reduction_factor=%d max_error=%g; call mesh() again to change",
                m->simp_factor, (double)m->simp_max_error);
  }
  const int64_t l = dense_of(m, id);
  IGN_REQUIRE(l > 0, IGN_ERR_KEY, "%llu", (unsigned long long)id);
  const uint64_t v0 = m->vert_off[l], v1 = m->vert_off[l + 1];
  const uint64_t t0 = m->tri_off[l], t1 = m->tri_off[l + 1];
  *nv = v1 - v0;
  *nf = t1 - t0;
  if (*nv == 0 || vertices == nullptr || faces == nullptr) return IGN_OK;
  Scratch sc(ctx);
  IGN_TRY(sc.reserve((v1 - v0) * 12 + 4096));
  float* d_pos = sc.take<float>((v1 - v0) * 3);
  IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small (mesh positions)");
  IGN_TRY(mesher_positions(m, v0, v1 - v0, resolution, voxel_centered, d_pos));
  IGN_CUDA(cudaMemcpyAsync(vertices, d_pos, (v1 - v0) * 12, cudaMemcpyDeviceToHost, ctx->stream));
  IGN_CUDA(cudaMemcpyAsync(faces, m->d_faces + 3 * t0, (t1 - t0) * 12, cudaMemcpyDeviceToHost, ctx->stream));
  IGN_CUDA(cudaStreamSynchronize(ctx->stream));
  return IGN_OK;
}

int ign_mesh_export(ign_mesher* m, const float resolution[3], int voxel_centered, float* vertices,
                    uint32_t* faces, uint64_t* vert_offsets, uint64_t* face_offsets) {
  IGN_REQUIRE(m && resolution && vert_offsets && face_offsets, IGN_ERR_INVALID, "null argument");
  ign_ctx* ctx = m->ctx;
  IGN_TRY(activate(ctx));
  uint64_t j = 0;
  for (uint64_t l = 1; l <= m->K; l++) {
    if (m->tri_off[l + 1] > m->tri_off[l]) {
      vert_offsets[j] = m->vert_off[l];
      face_offsets[j] = m->tri_off[l];
      j++;
    }
  }
  vert_offsets[j] = m->U;
  face_offsets[j] = m->T;
  if (m->U == 0 || vertices == nullptr || faces == nullptr) return IGN_OK;
  Scratch sc(ctx);
  IGN_TRY(sc.reserve(m->U * 12 + 4096));
  float* d_pos = sc.take<float>(m->U * 3);
  IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small (mesh positions)");
  IGN_TRY(mesher_positions(m, 0, m->U, resolution, voxel_centered, d_pos));
  IGN_TRY(d2h_by_kernel(ctx, vertices, d_pos, m->U * 12));
  IGN_TRY(d2h_by_kernel(ctx, faces, m->d_faces, m->T * 12));
  IGN_CUDA(cudaStreamSynchronize(ctx->stream));
  return IGN_OK;
}

}  // extern "C"
