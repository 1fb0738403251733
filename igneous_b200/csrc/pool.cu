// pool.cu -- 2x2x1 mode / average pooling pyramids (K1, K2)
//
// Replaces tinybrain.downsample_segmentation / downsample_with_averaging as
// called from igneous/tasks/image/image.py:46-55,91.
//
// Roofline: HBM.  Algorithmic bytes per input voxel for a fused k-mip launch
// = sizeof(T) * (1 + sum_{i=1..k} 4^-i)   (u32, 2 mips: 5.3125 B/vx).
//
// Fast path ("fused"): one thread owns a VEC x 2^NM input patch of one z-slice
// (VEC = 16 B / sizeof(T) voxels, i.e. one 128-bit load per row, rows
// independent -> 2^NM loads in flight per thread, warps read 512 contiguous
// bytes per row), reduces it NM levels deep in registers and writes every
// level once.  No shared memory: there is no inter-thread reuse in a 2x2x1
// pooling pyramid once a thread owns the whole patch.
// Generic path: one thread per output voxel, any extent (odd edges), sparse
// mode, float32.
#include <type_traits>

#include "common.cuh"

namespace ign {

// ------------------------------------------------------------------ helpers
template <typename T>
__device__ __forceinline__ T mode4(T a, T b, T c, T d) {
  // COUNTLESS 2-D: a=(x,y) b=(x+1,y) c=(x,y+1) d=(x+1,y+1)
  return (a == b || a == c) ? a : ((b == c) ? b : d);
}

template <typename T>
__device__ __forceinline__ T mode4_sparse(T a, T b, T c, T d, bool hx, bool hy) {
  T v[4];
  int n = 0;
  if (a) v[n++] = a;
  if (hx && b) v[n++] = b;
  if (hy && c) v[n++] = c;
  if (hx && hy && d) v[n++] = d;
  if (n == 0) return 0;
  if (n <= 2) return v[0];
  if (n == 3) return (v[0] == v[1] || v[0] == v[2]) ? v[0] : ((v[1] == v[2]) ? v[1] : v[0]);
  return (v[0] == v[1] || v[0] == v[2]) ? v[0] : ((v[1] == v[2]) ? v[1] : v[3]);
}

template <typename A>
__device__ __forceinline__ A render(A acc, int shift, int rounding) {
  if (rounding == IGN_ROUND_FLOOR) return acc >> shift;
  const A half = A(1) << (shift - 1);
  if (rounding == IGN_ROUND_HALF_UP) return (acc + half) >> shift;
  A q = acc >> shift;
  const A rem = acc & ((A(1) << shift) - 1);
  if (rem > half || (rem == half && (q & 1))) q++;
  return q;
}

template <typename T, int W>
__device__ __forceinline__ void store_row(T* dst, const T (&v)[W]) {
  constexpr int B = W * (int)sizeof(T);
  union {
    T e[W];
    uint4 q4;
    uint2 q2;
    uint32_t q1;
    uint16_t h;
    uint8_t b;
  } u;
#pragma unroll
  for (int i = 0; i < W; i++) u.e[i] = v[i];
  if constexpr (B == 16) st_stream(dst, u.q4);
  else if constexpr (B == 8) st_stream(dst, u.q2);
  else if constexpr (B == 4) *reinterpret_cast<uint32_t*>(dst) = u.q1;
  else if constexpr (B == 2) *reinterpret_cast<uint16_t*>(dst) = u.h;
  else *reinterpret_cast<uint8_t*>(dst) = u.b;
}

template <typename T, int H, int W>
__device__ __forceinline__ void mode_level(const T (&s)[H][W], T (&d)[H / 2][W / 2]) {
#pragma unroll
  for (int y = 0; y < H / 2; y++)
#pragma unroll
    for (int x = 0; x < W / 2; x++)
      d[y][x] = mode4(s[2 * y][2 * x], s[2 * y][2 * x + 1], s[2 * y + 1][2 * x],
                      s[2 * y + 1][2 * x + 1]);
}

template <typename S, typename A, int H, int W>
__device__ __forceinline__ void sum_level(const S (&s)[H][W], A (&d)[H / 2][W / 2]) {
#pragma unroll
  for (int y = 0; y < H / 2; y++)
#pragma unroll
    for (int x = 0; x < W / 2; x++)
      d[y][x] = (A)s[2 * y][2 * x] + (A)s[2 * y][2 * x + 1] + (A)s[2 * y + 1][2 * x] +
                (A)s[2 * y + 1][2 * x + 1];
}

template <typename T, typename A, int H, int W>
__device__ __forceinline__ void render_store(const A (&s)[H][W], T* out, uint64_t osx, uint64_t osy,
                                             uint64_t z, uint64_t ty, uint64_t tx, int shift,
                                             int rounding) {
  if (out == nullptr) return;
#pragma unroll
  for (int y = 0; y < H; y++) {
    T row[W];
#pragma unroll
    for (int x = 0; x < W; x++) row[x] = (T)render<A>(s[y][x], shift, rounding);
    store_row<T, W>(out + ((z * osy + ty * H + y) * osx + tx * W), row);
  }
}

template <typename T, int H, int W>
__device__ __forceinline__ void store_tile(const T (&s)[H][W], T* out, uint64_t osx, uint64_t osy,
                                           uint64_t z, uint64_t ty, uint64_t tx) {
#pragma unroll
  for (int y = 0; y < H; y++) store_row<T, W>(out + ((z * osy + ty * H + y) * osx + tx * W), s[y]);
}

template <typename T, int E, int VEC>
__device__ __forceinline__ void load_patch(const T* __restrict__ p, uint64_t sx, T (&a)[E][VEC]) {
  uint4 q[E];
#pragma unroll
  for (int j = 0; j < E; j++) q[j] = ld_stream(p + (uint64_t)j * sx);
#pragma unroll
  for (int j = 0; j < E; j++) {
    union {
      uint4 q;
      T e[VEC];
    } u;
    u.q = q[j];
#pragma unroll
    for (int i = 0; i < VEC; i++) a[j][i] = u.e[i];
  }
}

// --------------------------------------------------------------- fused mode
template <typename T, int NM>
__global__ void __launch_bounds__(256)
    k_mode_fused(const T* __restrict__ in, uint64_t sx, uint64_t sy, uint64_t tiles_x,
                 uint64_t tiles_y, uint64_t total, T* __restrict__ o1, T* __restrict__ o2,
                 T* __restrict__ o3, T* __restrict__ o4) {
  constexpr int VEC = 16 / (int)sizeof(T);
  constexpr int E = 1 << NM;
  static_assert(E <= VEC, "patch wider than one 128-bit load");
  const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (t >= total) return;
  const uint64_t tx = t % tiles_x, r = t / tiles_x, ty = r % tiles_y, z = r / tiles_y;
  T a[E][VEC];
  load_patch<T, E, VEC>(in + ((z * sy + ty * E) * sx + tx * VEC), sx, a);

  T l1[E / 2][VEC / 2];
  mode_level(a, l1);
  store_tile(l1, o1, sx >> 1, sy >> 1, z, ty, tx);
  if constexpr (NM >= 2) {
    T l2[E / 4][VEC / 4];
    mode_level(l1, l2);
    store_tile(l2, o2, sx >> 2, sy >> 2, z, ty, tx);
    if constexpr (NM >= 3) {
      T l3[E / 8][VEC / 8];
      mode_level(l2, l3);
      store_tile(l3, o3, sx >> 3, sy >> 3, z, ty, tx);
      if constexpr (NM >= 4) {
        T l4[E / 16][VEC / 16];
        mode_level(l3, l4);
        store_tile(l4, o4, sx >> 4, sy >> 4, z, ty, tx);
      }
    }
  }
}

// ------------------------------------------------------------ fused average
// Exact sums of the original samples for every level of the group; rendered
// as sum >> 2k (igneous/tasks/image/image.py:50-51 -> tinybrain averaging).
template <typename T, typename A, int NM>
__global__ void __launch_bounds__(256)
    k_avg_fused(const T* __restrict__ in, uint64_t sx, uint64_t sy, uint64_t tiles_x,
                uint64_t tiles_y, uint64_t total, int rounding, T* __restrict__ o1,
                T* __restrict__ o2, T* __restrict__ o3, T* __restrict__ o4) {
  constexpr int VEC = 16 / (int)sizeof(T);
  constexpr int E = 1 << NM;
  static_assert(E <= VEC, "patch wider than one 128-bit load");
  const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (t >= total) return;
  const uint64_t tx = t % tiles_x, r = t / tiles_x, ty = r % tiles_y, z = r / tiles_y;
  T a[E][VEC];
  load_patch<T, E, VEC>(in + ((z * sy + ty * E) * sx + tx * VEC), sx, a);

  A s1[E / 2][VEC / 2];
  sum_level(a, s1);
  render_store<T, A>(s1, o1, sx >> 1, sy >> 1, z, ty, tx, 2, rounding);
  if constexpr (NM >= 2) {
    A s2[E / 4][VEC / 4];
    sum_level(s1, s2);
    render_store<T, A>(s2, o2, sx >> 2, sy >> 2, z, ty, tx, 4, rounding);
    if constexpr (NM >= 3) {
      A s3[E / 8][VEC / 8];
      sum_level(s2, s3);
      render_store<T, A>(s3, o3, sx >> 3, sy >> 3, z, ty, tx, 6, rounding);
      if constexpr (NM >= 4) {
        A s4[E / 16][VEC / 16];
        sum_level(s3, s4);
        render_store<T, A>(s4, o4, sx >> 4, sy >> 4, z, ty, tx, 8, rounding);
      }
    }
  }
}

// ------------------------------------------------------------ generic paths
template <typename T>
__global__ void __launch_bounds__(256)
    k_mode_generic(const T* __restrict__ in, uint64_t sx, uint64_t sy, uint64_t nz,
                   T* __restrict__ out, int sparse) {
  const uint64_t ox = (sx + 1) >> 1, oy = (sy + 1) >> 1;
  const uint64_t total = ox * oy * nz;
  const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (t >= total) return;
  const uint64_t x = t % ox, r = t / ox, y = r % oy, z = r / oy;
  const uint64_t x0 = 2 * x, y0 = 2 * y;
  const bool hx = x0 + 1 < sx, hy = y0 + 1 < sy;
  const T* p = in + (z * sy + y0) * sx + x0;
  const T a = p[0];
  const T b = hx ? p[1] : a;
  const T c = hy ? p[sx] : a;
  const T d = (hx && hy) ? p[sx + 1] : a;
  T res;
  if (sparse) res = mode4_sparse(a, b, c, d, hx, hy);
  else res = (hx && hy) ? mode4(a, b, c, d) : a;
  out[t] = res;
}

// one averaging level: reads TI (original samples or accumulators), writes the
// accumulator (mirrored odd edges) and the rendered output.
template <typename TI, typename A, typename T>
__global__ void __launch_bounds__(256)
    k_avg_generic(const TI* __restrict__ in, uint64_t sx, uint64_t sy, uint64_t nz,
                  A* __restrict__ acc_out, T* __restrict__ out, int shift, int rounding) {
  const uint64_t ox = (sx + 1) >> 1, oy = (sy + 1) >> 1;
  const uint64_t total = ox * oy * nz;
  const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (t >= total) return;
  const uint64_t x = t % ox, r = t / ox, y = r % oy, z = r / oy;
  const uint64_t x0 = 2 * x, y0 = 2 * y;
  const uint64_t x1 = (x0 + 1 < sx) ? x0 + 1 : x0, y1 = (y0 + 1 < sy) ? y0 + 1 : y0;
  const TI* p = in + z * sy * sx;
  const A acc = (A)p[y0 * sx + x0] + (A)p[y0 * sx + x1] + (A)p[y1 * sx + x0] + (A)p[y1 * sx + x1];
  if (acc_out) acc_out[t] = acc;
  out[t] = (T)render<A>(acc, shift, rounding);
}

__global__ void __launch_bounds__(256)
    k_avg_f32_generic(const float* __restrict__ in, uint64_t sx, uint64_t sy, uint64_t nz,
                      float* __restrict__ out) {
  const uint64_t ox = (sx + 1) >> 1, oy = (sy + 1) >> 1;
  const uint64_t total = ox * oy * nz;
  const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (t >= total) return;
  const uint64_t x = t % ox, r = t / ox, y = r % oy, z = r / oy;
  const uint64_t x0 = 2 * x, y0 = 2 * y;
  const uint64_t x1 = (x0 + 1 < sx) ? x0 + 1 : x0, y1 = (y0 + 1 < sy) ? y0 + 1 : y0;
  const float* p = in + z * sy * sx;
  const float a = p[y0 * sx + x0], b = p[y0 * sx + x1], c = p[y1 * sx + x0], d = p[y1 * sx + x1];
  out[t] = __fmul_rn(__fadd_rn(__fadd_rn(a, b), __fadd_rn(c, d)), 0.25f);
}

// min / max pooling and striding over fx x fy x fz blocks (factors 1 or 2 per axis;
// partial edge blocks reduce over the samples that exist).  op: 0 min, 1 max, 2 striding.
template <typename T>
__global__ void __launch_bounds__(256)
    k_pool_select(const T* __restrict__ in, uint64_t sx, uint64_t sy, uint64_t sz, uint32_t fx,
                  uint32_t fy, uint32_t fz, int op, T* __restrict__ out) {
  const uint64_t ox = (sx + fx - 1) / fx, oy = (sy + fy - 1) / fy, oz = (sz + fz - 1) / fz;
  const uint64_t total = ox * oy * oz;
  const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (t >= total) return;
  const uint64_t x = t % ox, r = t / ox, y = r % oy, z = r / oy;
  const uint64_t x0 = x * fx, y0 = y * fy, z0 = z * fz;
  T acc = in[(z0 * sy + y0) * sx + x0];
  if (op != 2) {
    for (uint32_t dz = 0; dz < fz && z0 + dz < sz; dz++)
      for (uint32_t dy = 0; dy < fy && y0 + dy < sy; dy++)
        for (uint32_t dx = 0; dx < fx && x0 + dx < sx; dx++) {
          const T v = in[((z0 + dz) * sy + (y0 + dy)) * sx + (x0 + dx)];
          acc = (op == 0) ? (v < acc ? v : acc) : (v > acc ? v : acc);
        }
  }
  out[t] = acc;
}

// mode / average over fx x fy x fz blocks (factors 1 or 2 per axis), one thread per
// output voxel -- the non-(2,2,1) factors of tinybrain.downsample_segmentation /
// downsample_with_averaging (2x2x2 for --volumetric).  Rules: oracle/igneous_oracle.c
// "Block pooling" (samples visited x fastest; planar factor with four samples left ->
// COUNTLESS 2-D pick, otherwise highest count with ties to the earliest sample; averages
// count the lone row/column/slice of an odd extent twice).
template <typename T>
__global__ void __launch_bounds__(256)
    k_block_mode(const T* __restrict__ in, uint64_t sx, uint64_t sy, uint64_t sz, uint32_t fx,
                 uint32_t fy, uint32_t fz, int sparse, T* __restrict__ out) {
  const uint64_t ox = (sx + fx - 1) / fx, oy = (sy + fy - 1) / fy, oz = (sz + fz - 1) / fz;
  const uint64_t total = ox * oy * oz;
  const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (t >= total) return;
  const uint64_t x = t % ox, r = t / ox, y = r % oy, z = r / oy;
  const uint64_t x0 = x * fx, y0 = y * fy, z0 = z * fz;
  T v[8];
  int n = 0;
#pragma unroll
  for (uint32_t dz = 0; dz < 2; dz++)
#pragma unroll
    for (uint32_t dy = 0; dy < 2; dy++)
#pragma unroll
      for (uint32_t dx = 0; dx < 2; dx++) {
        if (dx < fx && dy < fy && dz < fz && x0 + dx < sx && y0 + dy < sy && z0 + dz < sz) {
          const T s = in[((z0 + dz) * sy + (y0 + dy)) * sx + (x0 + dx)];
          if (!sparse || s != 0) v[n++] = s;
        }
      }
  T res = 0;
  if (fx * fy * fz == 4 && n == 4) {
    res = mode4(v[0], v[1], v[2], v[3]);
  } else {
    int best = 0;
    for (int a = 0; a < n; a++) {
      int ct = 0;
      for (int b = 0; b < n; b++) ct += (v[b] == v[a]);
      if (ct > best) {
        best = ct;
        res = v[a];
      }
    }
  }
  out[t] = res;
}

// acc / n with the rounding enum (n = number of non-zero samples of a sparse average)
template <typename A>
__device__ __forceinline__ A render_div(A acc, A n, int rounding) {
  A q = acc / n;
  const A rem2 = 2 * (acc - q * n);
  if (rounding == IGN_ROUND_HALF_UP) q += (rem2 >= n);
  else if (rounding == IGN_ROUND_HALF_EVEN) q += (rem2 > n || (rem2 == n && (q & 1)));
  return q;
}

template <typename T, typename A>
__global__ void __launch_bounds__(256)
    k_block_avg(const T* __restrict__ in, uint64_t sx, uint64_t sy, uint64_t sz, uint32_t fx,
                uint32_t fy, uint32_t fz, int rounding, int sparse, T* __restrict__ out) {
  const uint64_t ox = (sx + fx - 1) / fx, oy = (sy + fy - 1) / fy, oz = (sz + fz - 1) / fz;
  const uint64_t total = ox * oy * oz;
  const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (t >= total) return;
  const uint64_t x = t % ox, r = t / ox, y = r % oy, z = r / oy;
  A acc = 0, nonzero = 0;
  for (uint32_t dz = 0; dz < fz; dz++)
    for (uint32_t dy = 0; dy < fy; dy++)
      for (uint32_t dx = 0; dx < fx; dx++) {
        uint64_t xx = x * fx + dx, yy = y * fy + dy, zz = z * fz + dz;
        xx = xx < sx ? xx : sx - 1;
        yy = yy < sy ? yy : sy - 1;
        zz = zz < sz ? zz : sz - 1;
        const A v = (A)in[(zz * sy + yy) * sx + xx];
        acc += v;
        nonzero += (v != 0);
      }
  if (sparse) {  // mean of the non-zero samples
    out[t] = (T)(nonzero ? render_div<A>(acc, nonzero, rounding) : A(0));
    return;
  }
  const int shift = (fx == 2) + (fy == 2) + (fz == 2);
  out[t] = (T)(shift ? render<A>(acc, shift, rounding) : acc);
}

__global__ void __launch_bounds__(256)
    k_block_avg_f32(const float* __restrict__ in, uint64_t sx, uint64_t sy, uint64_t sz, uint32_t fx,
                    uint32_t fy, uint32_t fz, int sparse, float* __restrict__ out) {
  const uint64_t ox = (sx + fx - 1) / fx, oy = (sy + fy - 1) / fy, oz = (sz + fz - 1) / fz;
  const uint64_t total = ox * oy * oz;
  const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (t >= total) return;
  const uint64_t x = t % ox, r = t / ox, y = r % oy, z = r / oy;
  float zs[2] = {0.0f, 0.0f};
  int nonzero = 0;
  for (uint32_t dz = 0; dz < fz; dz++) {
    float ys[2] = {0.0f, 0.0f};
    for (uint32_t dy = 0; dy < fy; dy++) {
      float xs[2] = {0.0f, 0.0f};
      for (uint32_t dx = 0; dx < fx; dx++) {
        uint64_t xx = x * fx + dx, yy = y * fy + dy, zz = z * fz + dz;
        xx = xx < sx ? xx : sx - 1;
        yy = yy < sy ? yy : sy - 1;
        zz = zz < sz ? zz : sz - 1;
        xs[dx] = in[(zz * sy + yy) * sx + xx];
        nonzero += (xs[dx] != 0.0f);
      }
      ys[dy] = (fx == 2) ? __fadd_rn(xs[0], xs[1]) : xs[0];
    }
    zs[dz] = (fy == 2) ? __fadd_rn(ys[0], ys[1]) : ys[0];
  }
  const float sum = (fz == 2) ? __fadd_rn(zs[0], zs[1]) : zs[0];
  if (sparse) out[t] = nonzero ? __fdiv_rn(sum, (float)nonzero) : 0.0f;
  else out[t] = __fmul_rn(sum, 1.0f / (float)(fx * fy * fz));
}

template <typename A>
__global__ void __launch_bounds__(256)
    k_widen_from(const void* __restrict__ in, int dtype, uint64_t n, A* __restrict__ out) {
  const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (t >= n) return;
  A v;
  switch (dtype) {
    case IGN_U8: v = ((const uint8_t*)in)[t]; break;
    case IGN_U16: v = ((const uint16_t*)in)[t]; break;
    case IGN_U32: v = ((const uint32_t*)in)[t]; break;
    default: v = (A)((const uint64_t*)in)[t]; break;
  }
  out[t] = v;
}

// ------------------------------------------------------------ host drivers
static int ilog2(int v) {
  int r = 0;
  while ((1 << (r + 1)) <= v) r++;
  return r;
}

template <typename T>
static int mode_pyramid(ign_ctx* ctx, const T* in, uint64_t sx, uint64_t sy, uint64_t nz,
                        int num_mips, int sparse, void* const* outs) {
  constexpr int VEC = 16 / (int)sizeof(T);
  const T* cur = in;
  int m = 0;
  while (m < num_mips) {
    int nm = 0;
    if (!sparse && sx % VEC == 0 && ((uintptr_t)cur % 16) == 0) {
      nm = ilog2(VEC);
      if (nm > num_mips - m) nm = num_mips - m;
      while (nm > 0 && (sy % (1ull << nm)) != 0) nm--;
    }
    if (nm > 0) {
      const uint64_t tiles_x = sx / VEC, tiles_y = sy >> nm, total = tiles_x * tiles_y * nz;
      T* o[4] = {nullptr, nullptr, nullptr, nullptr};
      for (int k = 0; k < nm; k++) o[k] = (T*)outs[m + k];
      const unsigned grid = blocks_for(total, 256);
      if (total > 0) {
        switch (nm) {
          case 1: IGN_LAUNCH_PROF(ctx, IGN_PROF_POOL, (k_mode_fused<T, 1>), grid, 256, 0, cur, sx, sy, tiles_x, tiles_y, total, o[0], o[1], o[2], o[3]); break;
          case 2:
            if constexpr (VEC >= 4) { IGN_LAUNCH_PROF(ctx, IGN_PROF_POOL, (k_mode_fused<T, 2>), grid, 256, 0, cur, sx, sy, tiles_x, tiles_y, total, o[0], o[1], o[2], o[3]); }
            break;
          case 3:
            if constexpr (VEC >= 8) { IGN_LAUNCH_PROF(ctx, IGN_PROF_POOL, (k_mode_fused<T, 3>), grid, 256, 0, cur, sx, sy, tiles_x, tiles_y, total, o[0], o[1], o[2], o[3]); }
            break;
          default:
            if constexpr (VEC >= 16) { IGN_LAUNCH_PROF(ctx, IGN_PROF_POOL, (k_mode_fused<T, 4>), grid, 256, 0, cur, sx, sy, tiles_x, tiles_y, total, o[0], o[1], o[2], o[3]); }
            break;
        }
      }
      sx >>= nm;
      sy >>= nm;
      m += nm;
      cur = (const T*)outs[m - 1];
    } else {
      const uint64_t ox = (sx + 1) >> 1, oy = (sy + 1) >> 1, total = ox * oy * nz;
      if (total > 0)
        IGN_LAUNCH(ctx, (k_mode_generic<T>), blocks_for(total, 256), 256, 0, cur, sx, sy, nz,
                   (T*)outs[m], sparse);
      sx = ox;
      sy = oy;
      cur = (const T*)outs[m];
      m++;
    }
  }
  return IGN_OK;
}

// worst-case scratch needed by the averaging generic path
static size_t avg_scratch_bytes(uint64_t sx, uint64_t sy, uint64_t nz) {
  const uint64_t ox = (sx + 1) >> 1, oy = (sy + 1) >> 1;
  return align_up(ox * oy * nz * 8, 256) * 5 / 4 + 4096;
}

// A: accumulator type wide enough for 256 * max(T)
template <typename T, typename A>
static int avg_pyramid(ign_ctx* ctx, const T* in, uint64_t sx, uint64_t sy, uint64_t nz,
                       int num_mips, int rounding, void* const* outs) {
  constexpr int VEC = 16 / (int)sizeof(T);
  Scratch sc(ctx);
  IGN_TRY(sc.reserve(avg_scratch_bytes(sx, sy, nz)));
  const T* cur = in;
  int m = 0;
  while (m < num_mips) {
    // one group of up to four levels is rendered from exact sums
    const int g = (num_mips - m) < 4 ? (num_mips - m) : 4;
    const bool fused_ok = (g <= ilog2(VEC)) && sx % VEC == 0 && (sy % (1ull << g)) == 0 &&
                          ((uintptr_t)cur % 16) == 0;
    if (fused_ok) {
      const uint64_t tiles_x = sx / VEC, tiles_y = sy >> g, total = tiles_x * tiles_y * nz;
      T* o[4] = {nullptr, nullptr, nullptr, nullptr};
      for (int k = 0; k < g; k++) o[k] = (T*)outs[m + k];
      const unsigned grid = blocks_for(total, 256);
      if (total > 0) {
        switch (g) {
          case 1: IGN_LAUNCH_PROF(ctx, IGN_PROF_POOL, (k_avg_fused<T, A, 1>), grid, 256, 0, cur, sx, sy, tiles_x, tiles_y, total, rounding, o[0], o[1], o[2], o[3]); break;
          case 2:
            if constexpr (VEC >= 4) { IGN_LAUNCH_PROF(ctx, IGN_PROF_POOL, (k_avg_fused<T, A, 2>), grid, 256, 0, cur, sx, sy, tiles_x, tiles_y, total, rounding, o[0], o[1], o[2], o[3]); }
            break;
          case 3:
            if constexpr (VEC >= 8) { IGN_LAUNCH_PROF(ctx, IGN_PROF_POOL, (k_avg_fused<T, A, 3>), grid, 256, 0, cur, sx, sy, tiles_x, tiles_y, total, rounding, o[0], o[1], o[2], o[3]); }
            break;
          default:
            if constexpr (VEC >= 16) { IGN_LAUNCH_PROF(ctx, IGN_PROF_POOL, (k_avg_fused<T, A, 4>), grid, 256, 0, cur, sx, sy, tiles_x, tiles_y, total, rounding, o[0], o[1], o[2], o[3]); }
            break;
        }
      }
      sx >>= g;
      sy >>= g;
    } else {
      // level by level with explicit accumulator arrays (ping-pong in scratch)
      const uint64_t ox1 = (sx + 1) >> 1, oy1 = (sy + 1) >> 1;
      const size_t acc_bytes = align_up(ox1 * oy1 * nz * sizeof(A), 256);
      sc.rewind();
      A* acc[2] = {nullptr, nullptr};
      if (g > 1) {
        acc[0] = (A*)sc.take(acc_bytes);
        acc[1] = (A*)sc.take(acc_bytes / 4 + 256);
        IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small for averaging accumulators");
      }
      for (int k = 0; k < g; k++) {
        const uint64_t ox = (sx + 1) >> 1, oy = (sy + 1) >> 1, total = ox * oy * nz;
        A* acc_out = (k + 1 < g) ? acc[k & 1] : nullptr;
        if (total > 0) {
          if (k == 0)
            IGN_LAUNCH(ctx, (k_avg_generic<T, A, T>), blocks_for(total, 256), 256, 0, cur, sx, sy, nz, acc_out, (T*)outs[m + k], 2, rounding);
          else
            IGN_LAUNCH(ctx, (k_avg_generic<A, A, T>), blocks_for(total, 256), 256, 0, (const A*)acc[(k - 1) & 1], sx, sy, nz, acc_out, (T*)outs[m + k], 2 * (k + 1), rounding);
        }
        sx = ox;
        sy = oy;
      }
    }
    m += g;
    cur = (const T*)outs[m - 1];
  }
  return IGN_OK;
}

static int avg_f32_pyramid(ign_ctx* ctx, const float* in, uint64_t sx, uint64_t sy, uint64_t nz,
                           int num_mips, void* const* outs) {
  const float* cur = in;
  for (int m = 0; m < num_mips; m++) {
    const uint64_t ox = (sx + 1) >> 1, oy = (sy + 1) >> 1, total = ox * oy * nz;
    if (total > 0)
      IGN_LAUNCH(ctx, k_avg_f32_generic, blocks_for(total, 256), 256, 0, cur, sx, sy, nz, (float*)outs[m]);
    cur = (const float*)outs[m];
    sx = ox;
    sy = oy;
  }
  return IGN_OK;
}

static int check_pool_args(const void* in, int dtype, uint64_t sx, uint64_t sy, uint64_t nz,
                           int num_mips, void* const* outs) {
  IGN_REQUIRE(in && outs, IGN_ERR_INVALID, "null buffer");
  IGN_REQUIRE(dtype_size(dtype) > 0, IGN_ERR_UNSUPPORTED, "unsupported dtype %d", dtype);
  IGN_REQUIRE(num_mips >= 1 && num_mips <= 32, IGN_ERR_INVALID, "num_mips=%d out of range", num_mips);
  IGN_REQUIRE(sx > 0 && sy > 0 && nz > 0, IGN_ERR_INVALID, "empty volume");
  return IGN_OK;
}

// accumulator wide enough for eight samples
template <typename T> struct BlockAcc { using type = uint32_t; };
template <> struct BlockAcc<uint32_t> { using type = uint64_t; };

// ops: 0 min, 1 max, 2 striding, 3 mode, 4 sparse mode, 5/6/7 average with
// IGN_ROUND_FLOOR / HALF_UP / HALF_EVEN, 8/9/10 sparse average (mean of the non-zero
// samples) with the same roundings.  Every mip is computed from the previous one.
template <typename T>
static int select_pyramid(ign_ctx* ctx, const void* in, uint64_t sx, uint64_t sy, uint64_t sz, uint32_t fx,
                          uint32_t fy, uint32_t fz, int num_mips, int op, void* const* outs) {
  const T* cur = (const T*)in;
  for (int m = 0; m < num_mips; m++) {
    const uint64_t ox = (sx + fx - 1) / fx, oy = (sy + fy - 1) / fy, oz = (sz + fz - 1) / fz;
    const uint64_t total = ox * oy * oz;
    if (total > 0) {
      const unsigned grid = blocks_for(total, 256);
      if (op <= 2) {
        IGN_LAUNCH(ctx, (k_pool_select<T>), grid, 256, 0, cur, sx, sy, sz, fx, fy, fz, op, (T*)outs[m]);
      } else if (op <= 4) {
        if constexpr (std::is_same<T, float>::value) {  // bit patterns: equality is all the mode needs
          IGN_LAUNCH(ctx, (k_block_mode<uint32_t>), grid, 256, 0, (const uint32_t*)cur, sx, sy, sz, fx, fy, fz,
                     op == 4, (uint32_t*)outs[m]);
        } else {
          IGN_LAUNCH(ctx, (k_block_mode<T>), grid, 256, 0, cur, sx, sy, sz, fx, fy, fz, op == 4, (T*)outs[m]);
        }
      } else {
        if constexpr (std::is_same<T, float>::value) {
          IGN_LAUNCH(ctx, k_block_avg_f32, grid, 256, 0, cur, sx, sy, sz, fx, fy, fz, op >= 8, (float*)outs[m]);
        } else if constexpr (std::is_same<T, uint64_t>::value) {
          set_error("averaging: uint64 images are not supported");
          return IGN_ERR_UNSUPPORTED;
        } else {
          using A = typename BlockAcc<T>::type;
          IGN_LAUNCH(ctx, (k_block_avg<T, A>), grid, 256, 0, cur, sx, sy, sz, fx, fy, fz, (op - 5) % 3, op >= 8,
                     (T*)outs[m]);
        }
      }
    }
    cur = (const T*)outs[m];
    sx = ox; sy = oy; sz = oz;
  }
  return IGN_OK;
}

}  // namespace ign

using namespace ign;

// host buffers: stage `in` and one output slot per mip, run the _dev function, copy the mips back
template <typename Run>
static int pool_host(ign_ctx* ctx, const void* in, uint64_t in_bytes, const uint64_t* out_bytes, int num_mips,
                     void* const* outs, const Run& run) {
  Staging st(ctx);
  void* d_in;
  void* d_out[32];
  st.add(&d_in, in_bytes, in);
  for (int m = 0; m < num_mips; m++) st.add(&d_out[m], out_bytes[m]);
  IGN_TRY(st.stage());
  IGN_TRY(run(d_in, d_out));
  for (int m = 0; m < num_mips; m++) IGN_TRY(st.back(outs[m], d_out[m], out_bytes[m]));
  return st.sync();
}

extern "C" {

int ign_pool_mode_2x2x1_dev(ign_ctx* ctx, const void* in, int dtype, uint64_t sx, uint64_t sy,
                            uint64_t sz, int num_mips, int sparse, void* const* outs) {
  IGN_TRY(activate(ctx));
  IGN_TRY(check_pool_args(in, dtype, sx, sy, sz, num_mips, outs));
  switch (dtype) {
    case IGN_U8: return mode_pyramid<uint8_t>(ctx, (const uint8_t*)in, sx, sy, sz, num_mips, sparse, outs);
    case IGN_U16: return mode_pyramid<uint16_t>(ctx, (const uint16_t*)in, sx, sy, sz, num_mips, sparse, outs);
    case IGN_U32:
    case IGN_F32: return mode_pyramid<uint32_t>(ctx, (const uint32_t*)in, sx, sy, sz, num_mips, sparse, outs);
    case IGN_U64: return mode_pyramid<uint64_t>(ctx, (const uint64_t*)in, sx, sy, sz, num_mips, sparse, outs);
  }
  set_error("unsupported dtype %d", dtype);
  return IGN_ERR_UNSUPPORTED;
}

int ign_pool_avg_2x2x1_dev(ign_ctx* ctx, const void* in, int dtype, uint64_t sx, uint64_t sy,
                           uint64_t sz, int num_mips, int rounding, void* const* outs) {
  IGN_TRY(activate(ctx));
  IGN_TRY(check_pool_args(in, dtype, sx, sy, sz, num_mips, outs));
  IGN_REQUIRE(rounding >= 0 && rounding <= 2, IGN_ERR_INVALID, "bad rounding mode %d", rounding);
  switch (dtype) {
    case IGN_U8: return avg_pyramid<uint8_t, uint32_t>(ctx, (const uint8_t*)in, sx, sy, sz, num_mips, rounding, outs);
    case IGN_U16: return avg_pyramid<uint16_t, uint32_t>(ctx, (const uint16_t*)in, sx, sy, sz, num_mips, rounding, outs);
    case IGN_U32: return avg_pyramid<uint32_t, uint64_t>(ctx, (const uint32_t*)in, sx, sy, sz, num_mips, rounding, outs);
    case IGN_F32: return avg_f32_pyramid(ctx, (const float*)in, sx, sy, sz, num_mips, outs);
  }
  set_error("averaging: unsupported dtype %d", dtype);
  return IGN_ERR_UNSUPPORTED;
}

int ign_pool_select_dev(ign_ctx* ctx, const void* in, int dtype, uint64_t sx, uint64_t sy, uint64_t sz,
                        uint32_t fx, uint32_t fy, uint32_t fz, int num_mips, int op, void* const* outs) {
  IGN_TRY(activate(ctx));
  IGN_TRY(check_pool_args(in, dtype, sx, sy, sz, num_mips, outs));
  IGN_REQUIRE(fx >= 1 && fx <= 2 && fy >= 1 && fy <= 2 && fz >= 1 && fz <= 2, IGN_ERR_UNSUPPORTED,
              "pooling factors must be 1 or 2 per axis (got %u,%u,%u)", fx, fy, fz);
  IGN_REQUIRE(op >= 0 && op <= 10, IGN_ERR_INVALID,
              "op must be 0 min, 1 max, 2 striding, 3 mode, 4 sparse mode, 5-7 average or 8-10 sparse average "
              "(floor / half-up / half-even)");
  switch (dtype) {
    case IGN_U8: return select_pyramid<uint8_t>(ctx, in, sx, sy, sz, fx, fy, fz, num_mips, op, outs);
    case IGN_U16: return select_pyramid<uint16_t>(ctx, in, sx, sy, sz, fx, fy, fz, num_mips, op, outs);
    case IGN_U32: return select_pyramid<uint32_t>(ctx, in, sx, sy, sz, fx, fy, fz, num_mips, op, outs);
    case IGN_U64: return select_pyramid<uint64_t>(ctx, in, sx, sy, sz, fx, fy, fz, num_mips, op, outs);
    case IGN_F32: return select_pyramid<float>(ctx, in, sx, sy, sz, fx, fy, fz, num_mips, op, outs);
  }
  set_error("unsupported dtype %d", dtype);
  return IGN_ERR_UNSUPPORTED;
}

int ign_pool_select(ign_ctx* ctx, const void* in, int dtype, uint64_t sx, uint64_t sy, uint64_t sz,
                    uint32_t fx, uint32_t fy, uint32_t fz, int num_mips, int op, void* const* outs) {
  IGN_TRY(activate(ctx));
  IGN_TRY(check_pool_args(in, dtype, sx, sy, sz, num_mips, outs));
  IGN_REQUIRE(fx >= 1 && fx <= 2 && fy >= 1 && fy <= 2 && fz >= 1 && fz <= 2, IGN_ERR_UNSUPPORTED,
              "pooling factors must be 1 or 2 per axis (got %u,%u,%u)", fx, fy, fz);
  const size_t es = dtype_size(dtype);
  uint64_t ob[32];
  uint64_t x = sx, y = sy, z = sz;
  for (int m = 0; m < num_mips; m++) {
    x = (x + fx - 1) / fx; y = (y + fy - 1) / fy; z = (z + fz - 1) / fz;
    ob[m] = x * y * z * es;
  }
  return pool_host(ctx, in, sx * sy * sz * es, ob, num_mips, outs, [&](const void* d_in, void* const* d_out) {
    return ign_pool_select_dev(ctx, d_in, dtype, sx, sy, sz, fx, fy, fz, num_mips, op, d_out);
  });
}

// 2x2x1 pyramids: every mip halves x and y
static int pool_2x2x1_host(ign_ctx* ctx, bool mode, const void* in, int dtype, uint64_t sx, uint64_t sy,
                           uint64_t sz, int num_mips, int flag, void* const* outs) {
  IGN_TRY(activate(ctx));
  IGN_TRY(check_pool_args(in, dtype, sx, sy, sz, num_mips, outs));
  const size_t es = dtype_size(dtype);
  uint64_t ob[32];
  uint64_t x = sx, y = sy;
  for (int m = 0; m < num_mips; m++) {
    x = (x + 1) >> 1;
    y = (y + 1) >> 1;
    ob[m] = x * y * sz * es;
  }
  return pool_host(ctx, in, sx * sy * sz * es, ob, num_mips, outs, [&](const void* d_in, void* const* d_out) {
    return mode ? ign_pool_mode_2x2x1_dev(ctx, d_in, dtype, sx, sy, sz, num_mips, flag, d_out)
                : ign_pool_avg_2x2x1_dev(ctx, d_in, dtype, sx, sy, sz, num_mips, flag, d_out);
  });
}

int ign_pool_mode_2x2x1(ign_ctx* ctx, const void* in, int dtype, uint64_t sx, uint64_t sy,
                        uint64_t sz, int num_mips, int sparse, void* const* outs) {
  return pool_2x2x1_host(ctx, true, in, dtype, sx, sy, sz, num_mips, sparse, outs);
}

int ign_pool_avg_2x2x1(ign_ctx* ctx, const void* in, int dtype, uint64_t sx, uint64_t sy,
                       uint64_t sz, int num_mips, int rounding, void* const* outs) {
  return pool_2x2x1_host(ctx, false, in, dtype, sx, sy, sz, num_mips, rounding, outs);
}

}  // extern "C"
