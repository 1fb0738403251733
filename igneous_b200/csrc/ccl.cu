// ccl.cu -- 6-connected multi-label connected components (K3), dust (K4)
//
// Replaces cc3d.connected_components(labels, connectivity=6, out_dtype=uint64)
// and cc3d.dust as called from igneous/tasks/image/ccl.py:169-175,231-240,335-344,
// and fuses the surrounding passes of CCLFacesTask (threshold_image :89-101,
// blackout_non_face_rails :103-124, `+= label_offset`, `[labels==0] = 0`
// :174-175) into the same kernels.
//
// Algorithm: union-find over x-RUNS described by per-voxel BIT MASKS.  Voxels
// are touched by two streaming passes only (A reads them once, C writes them
// once); everything in between works on 0.625 bytes per voxel of masks and on
// one u32 per run (a run = maximal x-segment of equal non-zero labels; typical
// segmentation has ~40 voxels per run).
//
//   A  masks   k_ccl_masks: persistent CTAs stage (128+halo) x 9 x 9 voxel tiles
//              in shared memory -- one cp.async.bulk.tensor.3d (TMA) per tile into
//              a double buffer, completion on an mbarrier, out-of-volume halo
//              zero-filled by the copy engine, so the compute loop has no address
//              arithmetic and no bounds predicates (volumes whose row pitch is
//              not a multiple of 16 bytes -- igneous's own 513^3 task shape --
//              take a cooperative-load fill of the same tile).  Per 32-voxel
//              word four ballots: S run starts (v != 0 && v != left), Z non-zero,
//              Ey / Ez equal to the y-1 / z-1 neighbour.  threshold_image and
//              blackout_non_face_rails are applied to the staged tile in place.  For rows of
//              2048+ voxels a CTA takes x-adjacent tile PAIRS and stores whole 32-byte mask
//              sectors (half sectors written apart did not survive in L2 at that size).
//      scan    exclusive sum of popc(S): the id of the first run starting in each
//              word.  Run ids therefore follow voxel raster order.
//   B  tiles   k_ccl_tiles: a CTA owns all words of 8 x 8 rows; the runs of the tile
//              are united along y and z on a union-find in SHARED memory (one
//              union per stretch of Ey / Ez in which neither row starts a new run),
//              then every run's parent (global run id of its tile root) is written.
//      merge   k_ccl_merge: the rows on tile faces do the same unions on the global
//              parent array (atomicMin union-find, path halving).
//   R  roots   flatten, then an exclusive scan over (parent[r] == r): roots are run
//              ids in raster order, so the scan IS cc3d's numbering (rank of the
//              component's first voxel); no sort.
//   C  expand  k_ccl_expand: label of voxel = label[run base of its word +
//              popc(S below it) - 1], 0 where Z is clear; optional offset /
//              lookup table (dust, multi-GPU relabelling); u16 / u32 / u64.
// HBM traffic ~ in + 0.625 (A) + ~0.6 (B, R: masks + runs) + 0.25 + out (C)
// bytes/voxel; algorithmic bytes (cc3d contract) = in + out.
#include <cub/device/device_scan.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>
#include <cuda.h>

#include <stdlib.h>
#include <string.h>

#include <memory>
#include <type_traits>
#include <vector>

#include "group.h"

namespace ign {

constexpr unsigned FULL = 0xFFFFFFFFu;

// ----------------------------------------------------------------- reader
// How a voxel value becomes a label: raw, or threshold_image() -> {0,1}; the
// rails of the +1 overlap shell are blacked out (ccl.py:103-124).
template <typename T, bool THR>
struct Reader {
  using value_type = T;
  static constexpr bool thresholded = THR;
  const T* in;
  double gte, lte;
  int use_gte, use_lte;
  uint32_t rx, ry, rz;  // rail coordinates (0xFFFFFFFF = none)
  __host__ __device__ __forceinline__ bool has_rails() const { return (rx & ry & rz) != 0xFFFFFFFFu; }
  // label stored back in the staged tile (type T: 0 / 1 when thresholded)
  __device__ __forceinline__ T label(T raw, uint32_t x, uint32_t y, uint32_t z) const {
    T v = raw;
    if constexpr (THR) {
      bool ok = true;
      if constexpr (std::is_same<T, float>::value) {
        if (use_gte) ok = ok && (raw >= (float)gte);
        if (use_lte) ok = ok && (raw <= (float)lte);
      } else {
        if (use_gte) ok = ok && ((double)raw >= gte);
        if (use_lte) ok = ok && ((double)raw <= lte);
      }
      v = ok ? (T)1 : (T)0;
    }
    const int on = (int)(x == rx) + (int)(y == ry) + (int)(z == rz);
    if (on >= 2) v = (T)0;
    return v;
  }
};

// ------------------------------------------------------------- union-find
// works on shared and on global memory (generic pointers)
__device__ __forceinline__ uint32_t uf_find(volatile uint32_t* P, uint32_t i) {
  uint32_t cur = i, p = P[cur];
  while (p != cur) {
    const uint32_t gp = P[p];
    if (gp != p) P[cur] = gp;  // path halving; cur is not a root here
    cur = p;
    p = gp;
  }
  return cur;
}

__device__ __forceinline__ void uf_union(uint32_t* P, uint32_t a, uint32_t b) {
  while (true) {
    a = uf_find(P, a);
    b = uf_find(P, b);
    if (a == b) return;
    if (a < b) {
      const uint32_t t = a;
      a = b;
      b = t;
    }
    const uint32_t old = atomicMin(&P[a], b);  // hook the larger root under the smaller
    if (old == a) return;
    a = old;  // lost a race: a had a parent already; unite that with b
  }
}

// ---------------------------------------------------------------- TMA / mbarrier
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// ------------------------------------------------------------------ pass A
// tile of the mask kernel: MT_BX x MT_BY x bz voxels (+1 halo row / plane on the low
// side, +16 bytes of halo on the low x side: TMA boxes are multiples of 16 bytes)
constexpr int MT_BX = 128, MT_BY = 8;
constexpr int MT_THREADS = 512;
#ifndef MT_BZ_OVERRIDE
#define MT_BZ_OVERRIDE 0
#endif
template <typename T> struct MaskTile {
  static constexpr int BZ = MT_BZ_OVERRIDE ? MT_BZ_OVERRIDE : (sizeof(T) == 8 ? 4 : 8);
  static constexpr int HX = 16 / (int)sizeof(T);
  static constexpr int PITCH = MT_BX + HX;             // elements per tile row
  static constexpr int ROWS = (MT_BY + 1) * (BZ + 1);  // rows incl. halo
  static constexpr int ELEMS = PITCH * ROWS;
  static constexpr size_t BYTES = ((size_t)ELEMS * sizeof(T) + 127) / 128 * 128;
};

struct MaskArgs {
  uint32_t sx, sy, sz, wpr;
  uint32_t ntx, nty, ntz, nby, nbz;  // tiles per axis; 8x8 blocks of (y,z) tile columns
  uint32_t ncols;                    // padded number of (y,z) columns = nby*nbz*64
  uint32_t pair;                     // 1: a CTA takes x-adjacent tile PAIRS and writes whole 32-byte mask sectors
  uint32_t *S, *Z, *Ey, *Ez;
};

// tile index -> tile coordinates (x fastest, then 8x8 blocks of (y,z) columns so that
// the halo rows / planes a tile re-reads are still in L2); false = padding, skip
__device__ __forceinline__ bool mask_tile_coords(const MaskArgs& a, uint64_t t, uint32_t* tx, uint32_t* ty,
                                                 uint32_t* tz) {
  *tx = (uint32_t)(t % a.ntx);
  const uint32_t c = (uint32_t)(t / a.ntx);
  const uint32_t b = c >> 6, r = c & 63u;
  *ty = (b % a.nby) * 8 + (r & 7u);
  *tz = (b / a.nby) * 8 + (r >> 3);
  return *ty < a.nty && *tz < a.ntz;
}

template <typename T, bool THR, bool TMA, bool PAIR>
__global__ void __launch_bounds__(MT_THREADS)
    k_ccl_masks(const __grid_constant__ CUtensorMap tmap, const Reader<T, THR> rd, const MaskArgs a) {
  using MT = MaskTile<T>;
  extern __shared__ __align__(128) unsigned char mt_smem[];
  __shared__ __align__(8) uint64_t bars[2];
  T* buf[2] = {(T*)mt_smem, (T*)(mt_smem + MT::BYTES)};
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const uint64_t ntiles = (uint64_t)a.ntx * a.ncols;
  const bool transform = THR || rd.has_rails();

  uint32_t tx = 0, ty = 0, tz = 0;
  // Tile sequence of this CTA.  Unpaired: tiles blockIdx, blockIdx + grid, ... (padding columns are
  // skipped).  Paired: the same over PAIRS of x-adjacent tiles (2p, 2p + 1), first the even one.
  auto first_from = [&](uint64_t unit) {  // first valid unit >= `unit` in this CTA's stride class -> tile id
    const uint64_t step = PAIR ? 2 : 1;
    uint64_t q = unit * step;
    while (q < ntiles && !mask_tile_coords(a, q, &tx, &ty, &tz)) q += gridDim.x * step;
    return q;
  };
  auto advance = [&](uint64_t cur) -> uint64_t {  // tile after `cur` (sets tx / ty / tz)
    if (PAIR) {
      if (!(cur & 1u)) {
        mask_tile_coords(a, cur + 1, &tx, &ty, &tz);  // same column as its partner: valid
        return cur + 1;
      }
      return first_from((cur >> 1) + gridDim.x);
    }
    return first_from(cur + gridDim.x);
  };
  // masks of the even tile of a pair wait here for the odd one: [warp][row][S, Z, Ey, Ez]
  __shared__ uint4 stash[PAIR ? MT_THREADS / 32 : 1][PAIR ? MT_BY : 1][4];
  uint64_t t = first_from(blockIdx.x);
  if constexpr (TMA) {
    if (tid == 0) {
      mbar_init(&bars[0], 1);
      mbar_init(&bars[1], 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0 && t < ntiles) {
      mbar_expect_tx(&bars[0], (uint32_t)(MT::ELEMS * sizeof(T)));
      tma_load_3d(buf[0], &tmap, &bars[0], (int)(tx * MT_BX) - MT::HX, (int)(ty * MT_BY) - 1, (int)(tz * MT::BZ) - 1);
    }
  }
  uint32_t it = 0;
  while (t < ntiles) {
    const uint32_t cur = TMA ? (it & 1u) : 0u;  // the cooperative fill is synchronous: one buffer
    const uint32_t x0 = tx * MT_BX, y0 = ty * MT_BY, z0 = tz * MT::BZ;
    // next tile of this CTA (its coordinates replace tx/ty/tz from here on)
    const uint64_t tn = advance(t);
    T* tile = (T*)(mt_smem + (size_t)cur * MT::BYTES);
    if constexpr (TMA) {
      if (tid == 0 && tn < ntiles) {  // the other buffer was released by the barrier that ended the previous iteration
        mbar_expect_tx(&bars[cur ^ 1u], (uint32_t)(MT::ELEMS * sizeof(T)));
        tma_load_3d(buf[cur ^ 1u], &tmap, &bars[cur ^ 1u], (int)(tx * MT_BX) - MT::HX, (int)(ty * MT_BY) - 1,
                    (int)(tz * MT::BZ) - 1);
      }
      mbar_wait(&bars[cur], (it >> 1) & 1u);
    } else {
      // cooperative fill (row pitch not 16-byte aligned): a warp per tile row, zero outside the volume
      for (uint32_t r = warp; r < (uint32_t)MT::ROWS; r += MT_THREADS / 32) {
        const uint32_t iy = r % (MT_BY + 1), iz = r / (MT_BY + 1);
        const int64_t gy = (int64_t)y0 + iy - 1, gz = (int64_t)z0 + iz - 1;
        const bool rok = gy >= 0 && gz >= 0 && gy < (int64_t)a.sy && gz < (int64_t)a.sz;
        const T* src = rd.in + ((uint64_t)(rok ? gz : 0) * a.sy + (uint64_t)(rok ? gy : 0)) * a.sx;
        for (uint32_t ix = MT::HX - 1 + lane; ix < (uint32_t)MT::PITCH; ix += 32) {
          const int64_t gx = (int64_t)x0 + ix - MT::HX;
          tile[r * MT::PITCH + ix] = (rok && gx >= 0 && gx < (int64_t)a.sx) ? src[gx] : (T)0;
        }
      }
      __syncthreads();
    }
    if (transform) {  // threshold_image / rails on the staged tile, in place
      for (uint32_t r = warp; r < (uint32_t)MT::ROWS; r += MT_THREADS / 32) {
        const uint32_t iy = r % (MT_BY + 1), iz = r / (MT_BY + 1);
        const uint32_t gy = y0 + iy - 1, gz = z0 + iz - 1;  // wraps to huge values in the low halo: out of range
        const bool rok = gy < a.sy && gz < a.sz;
        for (uint32_t ix = MT::HX - 1 + lane; ix < (uint32_t)MT::PITCH; ix += 32) {
          const uint32_t gx = x0 + ix - MT::HX;
          const T raw = tile[r * MT::PITCH + ix];
          tile[r * MT::PITCH + ix] = (rok && gx < a.sx) ? rd.label(raw, gx, gy, gz) : (T)0;
        }
      }
      if constexpr (TMA) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncthreads();
    }
    // ---- masks: warp w owns plane w % BZ and RPW of its rows.  Straight-line code: rows /
    // planes outside the volume are zero in the tile, so only the STORES are predicated and
    // every ballot runs in converged code.
    {
      constexpr int WPP = (MT_THREADS / 32) / MT::BZ;  // warps per plane
      constexpr int RPW = MT_BY / WPP;                 // rows per warp
      constexpr int NXW = MT_BX / 32;
      constexpr uint32_t PLANE = (MT_BY + 1) * MT::PITCH;
      const T* ts = (const T*)(mt_smem + (size_t)cur * MT::BYTES);  // shared-space addressing
      const uint32_t iz = warp % MT::BZ + 1;
      const uint32_t ry0 = (warp / MT::BZ) * RPW;
      const uint32_t gz = z0 + iz - 1;
      const uint32_t e0 = (iz * (MT_BY + 1) + ry0) * MT::PITCH + MT::HX + lane;  // row above the warp's first row
      T upv[NXW];  // the previous row stays in registers
#pragma unroll
      for (int xw = 0; xw < NXW; xw++) upv[xw] = ts[e0 + xw * 32];
      const uint32_t w0 = x0 / 32;
      const bool vec_ok = (a.wpr % NXW == 0);  // 16-byte aligned mask rows: one vector store per mask
#pragma unroll
      for (int k = 0; k < RPW; k++) {
        const uint32_t e = e0 + (k + 1) * MT::PITCH;
        uint32_t bS[NXW], bZ[NXW], bY[NXW], bB[NXW];
#pragma unroll
        for (int xw = 0; xw < NXW; xw++) {
          const T v = ts[e + xw * 32], left = ts[e + xw * 32 - 1], back = ts[e + xw * 32 - PLANE];
          const bool nz = v != (T)0;
          bS[xw] = __ballot_sync(FULL, nz && v != left);
          bZ[xw] = __ballot_sync(FULL, nz);
          bY[xw] = __ballot_sync(FULL, nz && v == upv[xw]);
          bB[xw] = __ballot_sync(FULL, nz && v == back);
          upv[xw] = v;
        }
        const uint32_t gy = y0 + ry0 + k;
        if (lane == 0 && gz < a.sz && gy < a.sy) {
          const uint64_t wi = ((uint64_t)gz * a.sy + gy) * a.wpr + w0;
          if (PAIR) {
            // (handled below by lanes 0 and 1 together)
          } else if (vec_ok) {
            static_assert(NXW == 4, "vector stores cover 4 words");
            *(uint4*)(a.S + wi) = make_uint4(bS[0], bS[1], bS[2], bS[3]);
            *(uint4*)(a.Z + wi) = make_uint4(bZ[0], bZ[1], bZ[2], bZ[3]);
            *(uint4*)(a.Ey + wi) = make_uint4(bY[0], bY[1], bY[2], bY[3]);
            *(uint4*)(a.Ez + wi) = make_uint4(bB[0], bB[1], bB[2], bB[3]);
          } else {
#pragma unroll
            for (int xw = 0; xw < NXW; xw++)
              if (w0 + xw < a.wpr) {
                a.S[wi + xw] = bS[xw]; a.Z[wi + xw] = bZ[xw]; a.Ey[wi + xw] = bY[xw]; a.Ez[wi + xw] = bB[xw];
              }
          }
        }
        if (PAIR) {
          // A 128-voxel tile yields 16 bytes per mask and row: half a 32-byte sector.  Written alone,
          // the half sectors were evicted from L2 before the x-neighbour's half arrived (2048^3:
          // 7.9 GB of DRAM writes for 4.3 GB of masks plus the fills).  The even tile parks its words
          // in shared memory; with the odd tile lanes 0 / 1 store both halves in one instruction.
          const bool rowok = gz < a.sz && gy < a.sy;
          const uint4 cS = make_uint4(bS[0], bS[1], bS[2], bS[3]), cZ = make_uint4(bZ[0], bZ[1], bZ[2], bZ[3]);
          const uint4 cY = make_uint4(bY[0], bY[1], bY[2], bY[3]), cB = make_uint4(bB[0], bB[1], bB[2], bB[3]);
          if (!(t & 1u)) {
            if (lane == 0) {
              stash[warp][k][0] = cS; stash[warp][k][1] = cZ; stash[warp][k][2] = cY; stash[warp][k][3] = cB;
            }
          } else if (lane < 2 && rowok) {
            const uint64_t wi = ((uint64_t)gz * a.sy + gy) * a.wpr + w0 - 4u + 4u * lane;  // lane 0: the even tile's words
            *(uint4*)(a.S + wi) = lane ? cS : stash[warp][k][0];
            *(uint4*)(a.Z + wi) = lane ? cZ : stash[warp][k][1];
            *(uint4*)(a.Ey + wi) = lane ? cY : stash[warp][k][2];
            *(uint4*)(a.Ez + wi) = lane ? cB : stash[warp][k][3];
          }
        }
      }
    }
    __syncthreads();  // tile consumed: its buffer may be refilled
    t = tn;
    it++;
  }
}

// ------------------------------------------------------------------ pass B
constexpr int TB_WMAX = 4096;   // words of a tile (all words of TY x TZ rows)
constexpr int TB_RCAP = 8192;   // runs of a tile resolved in shared memory
constexpr int TB_THREADS = 1024;
constexpr int TB_QCAP = 128;    // per-warp queue of union tasks (4 per lane per round)
constexpr uint32_t TB_GFLAG = 0x80000000u;

struct TileArgs {
  uint32_t sx, sy, sz, wpr, TY, TZ, nty, ntz, wcap;  // wcap: words of a full tile (shared-memory layout)
  uint32_t wpr_shift, ty_shift;                     // log2(wpr), log2(TY) when wpr is a power of two, else 0xFFFFFFFF
  const uint32_t *S, *Ey, *Ez, *rbase;
  uint32_t* parent;
};

__device__ __forceinline__ uint32_t mask_le(uint32_t p) { return 0xFFFFFFFFu >> (31u - p); }

// positions of one word that need a union with the same word of a neighbour row: one per
// stretch of E in which neither row starts a new run
__device__ __forceinline__ uint32_t union_candidates(uint32_t E, uint32_t Eprev_bit31, uint32_t S, uint32_t Sn) {
  return E & (S | Sn | ~((E << 1) | Eprev_bit31));
}
// base / nbase: id of the first run that starts in the word (own row / neighbour row)
template <typename UNION>
__device__ __forceinline__ void word_unions(uint32_t E, uint32_t Eprev_bit31, uint32_t S, uint32_t Sn, uint32_t base,
                                            uint32_t nbase, UNION&& unite) {
  uint32_t cand = union_candidates(E, Eprev_bit31, S, Sn);
  while (cand) {
    const uint32_t p = __ffs(cand) - 1;
    cand &= cand - 1;
    const uint32_t le = mask_le(p);
    unite(base + __popc(S & le) - 1, nbase + __popc(Sn & le) - 1);
  }
}

__global__ void __launch_bounds__(TB_THREADS) k_ccl_tiles(const TileArgs a) {
  extern __shared__ __align__(16) uint32_t tb_smem[];
  uint32_t* sS = tb_smem;
  uint32_t* sEy = sS + a.wcap;
  uint32_t* sEz = sEy + a.wcap;
  uint32_t* par = sEz + a.wcap;                                        // [TB_RCAP]
  uint32_t* queue = par + TB_RCAP;                                     // [warps][TB_QCAP] packed (a << 16 | b)
  uint16_t* lbase = (uint16_t*)(queue + (TB_THREADS / 32) * TB_QCAP);  // [wcap]
  __shared__ uint32_t warp_sums[TB_THREADS / 32];
  __shared__ uint32_t total_runs;
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const uint32_t ty = blockIdx.x % a.nty, tz = blockIdx.x / a.nty;
  const uint32_t y0 = ty * a.TY, z0 = tz * a.TZ;
  const uint32_t ny = min(a.TY, a.sy - y0), nz = min(a.TZ, a.sz - z0);
  const uint32_t wpr = a.wpr, rowsw = ny * wpr, W = rowsw * nz;
  // local word -> (plane, row, word in row): shifts when the tile is full and wpr a power of two (the
  // kernel is instruction bound: three integer divisions per word and pass were ~15 % of it)
  const bool p2 = a.wpr_shift != 0xFFFFFFFFu && ny == a.TY;
  const uint32_t rshift = a.wpr_shift + a.ty_shift;
  auto split = [&](uint32_t lw, uint32_t* lz, uint32_t* ly, uint32_t* xw) {
    if (p2) {
      *lz = lw >> rshift;
      *ly = (lw >> a.wpr_shift) & (a.TY - 1u);
      *xw = lw & (wpr - 1u);
    } else {
      const uint32_t z = lw / rowsw, r = lw - z * rowsw, y = r / wpr;
      *lz = z; *ly = y; *xw = r - y * wpr;
    }
  };
  auto gword = [&](uint32_t lw) -> uint64_t {  // local word -> global word
    const uint32_t lz = p2 ? lw >> rshift : lw / rowsw, r = lw - lz * rowsw;
    return ((uint64_t)(z0 + lz) * a.sy + y0) * wpr + r;
  };
  // ---- load the masks (the ny rows of one plane are contiguous words)
  for (uint32_t lw = tid; lw < W; lw += TB_THREADS) {
    const uint64_t g = gword(lw);
    sS[lw] = a.S[g];
    sEy[lw] = a.Ey[g];
    sEz[lw] = a.Ez[g];
  }
  __syncthreads();
  // ---- local run numbering: exclusive scan of popc(S) over the tile's words
  constexpr int WPT = TB_WMAX / TB_THREADS;  // 16 consecutive words per thread
  uint32_t cnt = 0;
#pragma unroll
  for (int k = 0; k < WPT; k++) {
    const uint32_t lw = tid * WPT + k;
    if (lw < W) cnt += __popc(sS[lw]);
  }
  uint32_t inc = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t o = __shfl_up_sync(FULL, inc, d);
    if ((int)lane >= d) inc += o;
  }
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  uint32_t woff = 0;
  for (uint32_t w = 0; w < warp; w++) woff += warp_sums[w];
  if (tid == TB_THREADS - 1) total_runs = woff + inc;
  uint32_t run = woff + inc - cnt;
  __syncthreads();
  const uint32_t RL = total_runs;
  const bool fits = RL <= (uint32_t)TB_RCAP;
  if (!fits) {
    // too many runs for shared memory (noise-like data): every union goes to the global array
    for (uint32_t lw = tid; lw < W; lw += TB_THREADS) {
      const uint32_t b = a.rbase[gword(lw)], c = __popc(sS[lw]);
      for (uint32_t k = 0; k < c; k++) a.parent[b + k] = b + k;
    }
    __syncthreads();
    for (uint32_t lw = tid; lw < W; lw += TB_THREADS) {
      uint32_t lz, ly, xw;
      split(lw, &lz, &ly, &xw);
      const uint32_t ey = ly > 0 ? sEy[lw] : 0u, ez = lz > 0 ? sEz[lw] : 0u;
      if (!(ey | ez)) continue;
      const uint32_t S = sS[lw], base = a.rbase[gword(lw)];
      auto un = [&](uint32_t x, uint32_t y) { uf_union(a.parent, x, y); };
      if (ey) word_unions(ey, xw > 0 ? sEy[lw - 1] >> 31 : 0u, S, sS[lw - wpr], base, a.rbase[gword(lw - wpr)], un);
      if (ez) word_unions(ez, xw > 0 ? sEz[lw - 1] >> 31 : 0u, S, sS[lw - rowsw], base, a.rbase[gword(lw - rowsw)], un);
    }
    return;
  }
#pragma unroll
  for (int k = 0; k < WPT; k++) {
    const uint32_t lw = tid * WPT + k;
    if (lw < W) {
      lbase[lw] = (uint16_t)run;
      run += __popc(sS[lw]);
    }
  }
  for (uint32_t i = tid; i < RL; i += TB_THREADS) par[i] = i;
  __syncthreads();
  // ---- unions along y and z inside the tile.  A warp takes 32 words; the lanes queue their
  // union tasks (4 per lane per round) and the warp then runs the queue on dense lanes.
  {
    uint32_t* q = queue + warp * TB_QCAP;
    for (uint32_t base0 = warp * 32; base0 < W; base0 += TB_THREADS) {
      const uint32_t lw = base0 + lane;
      uint32_t cy = 0, cz = 0, S = 0, Sy = 0, Sz = 0, lb = 0, lby = 0, lbz = 0;
      if (lw < W) {
        uint32_t lz, ly, xw;
        split(lw, &lz, &ly, &xw);
        S = sS[lw];
        lb = lbase[lw];
        if (ly > 0) {
          const uint32_t E = sEy[lw];
          if (E) {
            Sy = sS[lw - wpr];
            lby = lbase[lw - wpr];
            cy = union_candidates(E, xw > 0 ? sEy[lw - 1] >> 31 : 0u, S, Sy);
          }
        }
        if (lz > 0) {
          const uint32_t E = sEz[lw];
          if (E) {
            Sz = sS[lw - rowsw];
            lbz = lbase[lw - rowsw];
            cz = union_candidates(E, xw > 0 ? sEz[lw - 1] >> 31 : 0u, S, Sz);
          }
        }
      }
      while (__any_sync(FULL, (cy | cz) != 0)) {
        uint32_t t[4], nt = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
          if (cy) {
            const uint32_t p = __ffs(cy) - 1, le = mask_le(p);
            cy &= cy - 1;
            t[nt++] = ((lb + __popc(S & le) - 1) << 16) | (lby + __popc(Sy & le) - 1);
          } else if (cz) {
            const uint32_t p = __ffs(cz) - 1, le = mask_le(p);
            cz &= cz - 1;
            t[nt++] = ((lb + __popc(S & le) - 1) << 16) | (lbz + __popc(Sz & le) - 1);
          }
        }
        uint32_t off = nt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const uint32_t o = __shfl_up_sync(FULL, off, d);
          if ((int)lane >= d) off += o;
        }
        const uint32_t total = __shfl_sync(FULL, off, 31);
        off -= nt;
#pragma unroll
        for (int k = 0; k < 4; k++)
          if (k < (int)nt) q[off + k] = t[k];
        __syncwarp();
        for (uint32_t j = lane; j < total; j += 32) {
          const uint32_t e = q[j];
          uf_union(par, e >> 16, e & 0xFFFFu);
        }
        __syncwarp();
      }
    }
  }
  __syncthreads();
  // ---- flatten; roots take their global id (flagged); every run then stores the global id of its root
  // (read-only walks: a path-halving write of another thread could otherwise replace an entry
  // that already holds its root by a mere ancestor)
  for (uint32_t i = tid; i < RL; i += TB_THREADS) {
    volatile uint32_t* P = par;
    uint32_t cur = i, p = P[cur];
    while (p != cur) {
      cur = p;
      p = P[cur];
    }
    if (cur != i) P[i] = cur;
  }
  __syncthreads();
  for (uint32_t lw = tid; lw < W; lw += TB_THREADS) {
    const uint32_t c = __popc(sS[lw]);
    if (c == 0) continue;
    const uint32_t lb = lbase[lw], gb = a.rbase[gword(lw)];
    sEy[lw] = gb;  // the E masks are dead: keep the word's global run base
    for (uint32_t k = 0; k < c; k++)
      if (par[lb + k] == lb + k) par[lb + k] = TB_GFLAG | (gb + k);
  }
  __syncthreads();
  for (uint32_t lw = tid; lw < W; lw += TB_THREADS) {
    const uint32_t c = __popc(sS[lw]);
    if (c == 0) continue;
    const uint32_t lb = lbase[lw], gb = sEy[lw];
    for (uint32_t k = 0; k < c; k++) {
      uint32_t v = par[lb + k];
      if (!(v & TB_GFLAG)) v = par[v];  // flattened: v is a root, its entry is flagged
      a.parent[gb + k] = v & ~TB_GFLAG;
    }
  }
}

// rows on tile faces: the same unions on the global parent array
struct MergeArgs {
  uint32_t sx, sy, sz, wpr, TY, TZ, nty, ntz;
  uint64_t words_y, words_z;  // work items of the y-face rows / z-face rows
  const uint32_t *S, *Ey, *Ez, *rbase;
  uint32_t* parent;
};

// Latency bound (dependent loads, a handful of unions): a thread owns MG_W consecutive words of a
// face row and issues all their loads before the first union.
constexpr int MG_W = 4;

__global__ void __launch_bounds__(256) k_ccl_merge(const MergeArgs a) {
  const uint32_t gpr = (a.wpr + MG_W - 1) / MG_W;  // word groups per row
  const uint64_t rows_y = (uint64_t)(a.nty - 1) * a.sz, rows_z = (uint64_t)(a.ntz - 1) * a.sy;
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= (rows_y + rows_z) * gpr) return;
  const uint64_t r = i / gpr;
  const uint32_t xw0 = (uint32_t)(i - r * gpr) * MG_W;
  uint32_t y, z;
  bool ydir;
  if (r < rows_y) {  // rows y = k*TY (k >= 1), every z
    ydir = true;
    y = ((uint32_t)(r % (a.nty - 1)) + 1) * a.TY;
    z = (uint32_t)(r / (a.nty - 1));
  } else {  // rows of planes z = k*TZ (k >= 1), every y
    ydir = false;
    const uint64_t j = r - rows_y;
    y = (uint32_t)(j % a.sy);
    z = ((uint32_t)(j / a.sy) + 1) * a.TZ;
  }
  const uint64_t g0 = ((uint64_t)z * a.sy + y) * a.wpr + xw0;
  const uint64_t n0 = ydir ? g0 - a.wpr : g0 - (uint64_t)a.sy * a.wpr;
  const uint32_t* Em = ydir ? a.Ey : a.Ez;
  uint32_t E[MG_W], S[MG_W], Sn[MG_W], rb[MG_W], rn[MG_W];
  uint32_t prev = xw0 > 0 ? Em[g0 - 1] >> 31 : 0u;
#pragma unroll
  for (int k = 0; k < MG_W; k++) {
    const bool in = xw0 + k < a.wpr;
    E[k] = in ? Em[g0 + k] : 0u;
    S[k] = in ? a.S[g0 + k] : 0u;
    Sn[k] = in ? a.S[n0 + k] : 0u;
    rb[k] = in ? a.rbase[g0 + k] : 0u;
    rn[k] = in ? a.rbase[n0 + k] : 0u;
  }
  auto un = [&](uint32_t x, uint32_t yv) { uf_union(a.parent, x, yv); };
#pragma unroll
  for (int k = 0; k < MG_W; k++) {
    if (E[k]) word_unions(E[k], prev, S[k], Sn[k], rb[k], rn[k], un);
    prev = E[k] >> 31;
  }
}

// ------------------------------------------------------------------ runs
__global__ void __launch_bounds__(256) k_ccl_flatten(uint32_t* parent, uint32_t R) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  volatile uint32_t* P = parent;
  uint32_t cur = r, p = P[cur];
  while (p != cur) {
    cur = p;
    p = P[cur];
  }
  P[r] = cur;
}

struct IsRootOp {
  const uint32_t* parent;
  __host__ __device__ __forceinline__ uint32_t operator()(uint32_t r) const { return parent[r] == r ? 1u : 0u; }
};
struct PopcOp {
  __host__ __device__ __forceinline__ uint32_t operator()(uint32_t w) const {
#ifdef __CUDA_ARCH__
    return __popc(w);
#else
    return (uint32_t)__builtin_popcount(w);
#endif
  }
};

// parent[r] (flattened) -> label of the run: rank of its root + 1
__global__ void __launch_bounds__(256)
    k_ccl_runlabel(uint32_t* parent, const uint32_t* __restrict__ rank, uint32_t R) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  parent[r] = rank[parent[r]] + 1;
}
__global__ void __launch_bounds__(256)
    k_ccl_relabel_runs(uint32_t* label, uint32_t R, const uint32_t* __restrict__ lut) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < R) label[r] = lut[label[r]];
}

// ------------------------------------------------------------------ pass C
struct ExpandArgs {
  uint32_t sx, wpr;
  uint64_t rows;    // sy * sz
  uint64_t offset;  // added to every non-zero label
  const uint32_t *S, *Z, *rbase, *label;
};

// The expansion is two dependent loads (masks -> run label) followed by a store, so a warp
// keeps EX_G independent 128-voxel groups in flight (a single group per warp is latency bound:
// 2.2 TB/s measured).  A lane owns 4 consecutive voxels of each group (one vector store).
constexpr int EX_G = 4;

template <typename OUT>
__device__ __forceinline__ void ex_store4(OUT* dst, const OUT* v) {
  if constexpr (sizeof(OUT) == 2) {
    *(uint2*)dst = make_uint2((uint32_t)v[0] | ((uint32_t)v[1] << 16), (uint32_t)v[2] | ((uint32_t)v[3] << 16));
  } else if constexpr (sizeof(OUT) == 4) {
    st_stream(dst, make_uint4((uint32_t)v[0], (uint32_t)v[1], (uint32_t)v[2], (uint32_t)v[3]));
  } else {
    st_stream(dst, make_uint4((uint32_t)v[0], (uint32_t)((uint64_t)v[0] >> 32), (uint32_t)v[1], (uint32_t)((uint64_t)v[1] >> 32)));
    st_stream(dst + 2, make_uint4((uint32_t)v[2], (uint32_t)((uint64_t)v[2] >> 32), (uint32_t)v[3], (uint32_t)((uint64_t)v[3] >> 32)));
  }
}

template <typename OUT>
__global__ void __launch_bounds__(256) k_ccl_expand4(const ExpandArgs a, OUT* __restrict__ out) {
  const uint32_t lane = threadIdx.x & 31u;
  // a warp owns EX_G consecutive 128-voxel groups of ONE row (chunk c of the row)
  const uint32_t gpr = (a.wpr + 3) / 4;               // groups per row
  const uint32_t cpr = (gpr + EX_G - 1) / EX_G;       // warp chunks per row
  const uint64_t wid = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
  const uint64_t row = wid / cpr;
  if (row >= a.rows) return;
  const uint32_t chunk = (uint32_t)(wid - row * cpr);
  const uint32_t b0 = (lane & 7u) * 4;
  const uint32_t xw0 = chunk * (EX_G * 4) + (lane >> 3);
  const uint32_t* Sr = a.S + row * a.wpr;
  const uint32_t* Zr = a.Z + row * a.wpr;
  const uint32_t* Rr = a.rbase + row * a.wpr;
  OUT* orow = out + row * a.sx;
  uint32_t S[EX_G], Z[EX_G], rb[EX_G], lab[EX_G], idx0[EX_G];
  bool ok[EX_G];
#pragma unroll
  for (int g = 0; g < EX_G; g++) {
    const uint32_t xw = xw0 + g * 4;
    ok[g] = xw < a.wpr && xw * 32 + b0 < a.sx;  // sx % 4 == 0: a quad is all in or all out
    S[g] = ok[g] ? Sr[xw] : 0u;
    Z[g] = ok[g] ? Zr[xw] : 0u;
    rb[g] = ok[g] ? Rr[xw] : 0u;
  }
#pragma unroll
  for (int g = 0; g < EX_G; g++) {  // the label of the first non-zero voxel of the quad (usually of all four)
    const uint32_t zq = (Z[g] >> b0) & 15u;
    const uint32_t first = zq ? b0 + (uint32_t)__ffs(zq) - 1 : b0;
    idx0[g] = rb[g] + __popc(S[g] & mask_le(first)) - 1;
    lab[g] = zq ? a.label[idx0[g]] : 0u;
  }
#pragma unroll
  for (int g = 0; g < EX_G; g++) {
    if (!ok[g]) continue;
    OUT v[4];
    const uint32_t zq = (Z[g] >> b0) & 15u, sq = (S[g] >> b0) & 15u;
    const OUT l0 = lab[g] ? (OUT)(lab[g] + a.offset) : (OUT)0;
    // no run starts after the quad's first non-zero voxel: its non-zero voxels are one run
    if (zq == 0 || (sq >> __ffs(zq)) == 0) {
#pragma unroll
      for (int j = 0; j < 4; j++) v[j] = ((zq >> j) & 1u) ? l0 : (OUT)0;
    } else {
      uint32_t cur_idx = idx0[g], cur_lab = lab[g];
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const uint32_t b = b0 + j;
        OUT o = 0;
        if ((Z[g] >> b) & 1u) {
          const uint32_t idx = rb[g] + __popc(S[g] & mask_le(b)) - 1;
          if (idx != cur_idx) {  // another run inside the quad
            cur_idx = idx;
            cur_lab = a.label[idx];
          }
          o = cur_lab ? (OUT)(cur_lab + a.offset) : (OUT)0;
        }
        v[j] = o;
      }
    }
    ex_store4(orow + (xw0 + g * 4) * 32 + b0, v);
  }
}

// any row pitch: a lane owns one voxel of each of EX_G consecutive words
template <typename OUT>
__global__ void __launch_bounds__(256) k_ccl_expand1(const ExpandArgs a, OUT* __restrict__ out) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t total = a.rows * a.wpr;
  const uint64_t w0 = ((blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5) * EX_G;
  if (w0 >= total) return;
  uint32_t lab[EX_G];
  uint64_t at[EX_G];
  bool ok[EX_G], nz[EX_G];
#pragma unroll
  for (int g = 0; g < EX_G; g++) {
    const uint64_t wi = w0 + g;
    const uint64_t row = wi / a.wpr;
    const uint32_t x = (uint32_t)(wi - row * a.wpr) * 32 + lane;
    ok[g] = wi < total && x < a.sx;
    at[g] = row * a.sx + x;
    const uint32_t S = ok[g] ? a.S[wi] : 0u, Z = ok[g] ? a.Z[wi] : 0u;
    nz[g] = (Z >> lane) & 1u;
    lab[g] = nz[g] ? a.rbase[wi] + __popc(S & mask_le(lane)) - 1 : 0u;  // run id for now
  }
#pragma unroll
  for (int g = 0; g < EX_G; g++) lab[g] = nz[g] ? a.label[lab[g]] : 0u;
#pragma unroll
  for (int g = 0; g < EX_G; g++)
    if (ok[g]) out[at[g]] = lab[g] ? (OUT)(lab[g] + a.offset) : (OUT)0;
}

// one z-plane: voxel values widened to u64 and run labels (multi-GPU face exchange)
template <typename T>
__global__ void __launch_bounds__(256)
    k_ccl_plane(const T* __restrict__ in, const ExpandArgs a, uint64_t z, uint32_t sy, uint64_t* __restrict__ values,
                uint32_t* __restrict__ labels) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  const uint64_t np = (uint64_t)a.sx * sy;
  if (i >= np) return;
  const uint32_t y = (uint32_t)(i / a.sx), x = (uint32_t)(i - (uint64_t)y * a.sx);
  const uint64_t row = z * sy + y;
  const uint64_t wi = row * a.wpr + (x >> 5);
  const uint32_t b = x & 31u;
  values[i] = (uint64_t)in[row * a.sx + x];
  uint32_t l = 0;
  if ((a.Z[wi] >> b) & 1u) l = a.label[a.rbase[wi] + __popc(a.S[wi] & mask_le(b)) - 1];
  labels[i] = l;
}

// ------------------------------------------------------------------- dust
// voxels per component: every x-segment of a run inside a word adds its length once
__global__ void __launch_bounds__(256) k_ccl_count(const ExpandArgs a, uint32_t* __restrict__ counts) {
  const uint64_t wi = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (wi >= a.rows * a.wpr) return;
  const uint32_t S = a.S[wi], Z = a.Z[wi];
  if (!Z) return;
  const uint32_t rb = a.rbase[wi];
  // segment heads: a start, or a non-zero voxel at bit 0 (run continuing from the previous word)
  uint32_t heads = S | (Z & 1u);
  while (heads) {
    const uint32_t p = __ffs(heads) - 1;
    heads &= heads - 1;
    // the segment ends before the next start or the next zero voxel
    const uint32_t stop = (p == 31) ? 0u : ((S | ~Z) & ~mask_le(p));
    const uint32_t q = stop ? (uint32_t)(__ffs(stop) - 1) : 32u;
    const uint32_t l = a.label[rb + __popc(S & mask_le(p)) - 1];
    atomicAdd(&counts[l], q - p);
  }
}

__global__ void __launch_bounds__(256)
    k_dust_flags(const uint32_t* __restrict__ counts, uint32_t n, uint64_t threshold, uint32_t* __restrict__ keep) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i <= n + 1) keep[i] = (i >= 1 && i <= n && (uint64_t)counts[i] >= threshold) ? 1u : 0u;
}

// keep[] (0/1) and its exclusive scan -> lut: old label -> new label (0 = removed)
__global__ void __launch_bounds__(256)
    k_dust_lut(const uint32_t* __restrict__ keep, const uint32_t* __restrict__ scan, uint32_t n,
               uint32_t* __restrict__ lut) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i <= n) lut[i] = keep[i] ? scan[i] + 1 : 0u;
}

// cc3d.dust(in_place=True): zero the voxels of removed components in the input array
template <typename T>
__global__ void __launch_bounds__(256) k_dust_apply(const ExpandArgs a, T* __restrict__ labels) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t wi = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
  if (wi >= a.rows * a.wpr) return;
  const uint64_t row = wi / a.wpr;
  const uint32_t xw = (uint32_t)(wi - row * a.wpr);
  const uint32_t x = xw * 32 + lane;
  if (x >= a.sx) return;
  const uint32_t S = a.S[wi], Z = a.Z[wi];
  if (!((Z >> lane) & 1u)) return;
  if (a.label[a.rbase[wi] + __popc(S & mask_le(lane)) - 1] == 0) labels[row * a.sx + x] = (T)0;
}

// equivalence pairs between two facing planes (same x,y; adjacent z)
__global__ void __launch_bounds__(256)
    k_ccl_link(const uint64_t* __restrict__ va, const uint32_t* __restrict__ la, uint64_t offa,
               const uint64_t* __restrict__ vb, const uint32_t* __restrict__ lb, uint64_t offb,
               uint64_t nplane, uint64_t* __restrict__ pairs, uint32_t cap, uint32_t* counters) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  const uint32_t lane = threadIdx.x & 31;
  bool emit = false;
  uint64_t a = 0, b = 0;
  if (i < nplane) {
    const uint64_t v = va[i];
    if (v != 0 && v == vb[i]) {
      a = offa + la[i];
      b = offb + lb[i];
      // runs of the same pair along x are emitted once
      emit = !(i > 0 && la[i - 1] == la[i] && lb[i - 1] == lb[i] && va[i - 1] == v && vb[i - 1] == v);
    }
  }
  const uint32_t m = __ballot_sync(FULL, emit);
  if (m) {
    const int leader = __ffs(m) - 1;
    uint32_t base = 0;
    if ((int)lane == leader) base = atomicAdd(&counters[0], (uint32_t)__popc(m));
    base = __shfl_sync(FULL, base, leader);
    if (emit) {
      const uint32_t pos = base + __popc(m & ((1u << lane) - 1u));
      if (pos < cap) {
        pairs[2 * (uint64_t)pos] = a;
        pairs[2 * (uint64_t)pos + 1] = b;
      }
    }
  }
}

// multi-GPU merge on the device: the equivalences between two facing planes go straight into
// a union-find over the dataset-wide provisional ids (offset + volume-local id)
__global__ void __launch_bounds__(256)
    k_ccl_link_union(const uint64_t* __restrict__ va, const uint32_t* __restrict__ la, uint32_t offa,
                     const uint64_t* __restrict__ vb, const uint32_t* __restrict__ lb, uint32_t offb,
                     uint64_t nplane, uint32_t* parent) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= nplane) return;
  const uint64_t v = va[i];
  if (v == 0 || v != vb[i]) return;
  // runs of the same pair along x unite once
  if (i > 0 && la[i - 1] == la[i] && lb[i - 1] == lb[i] && va[i - 1] == v && vb[i - 1] == v) return;
  uf_union(parent, offa + la[i], offb + lb[i]);
}
__global__ void __launch_bounds__(256) k_iota_u32(uint32_t* p, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = i;
}
// parent[i] (flattened) -> rank of its root; id 0 is a root of its own and ranks 0
__global__ void __launch_bounds__(256)
    k_ccl_rank_of_root(uint32_t* parent, const uint32_t* __restrict__ rank, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) parent[i] = rank[parent[i]];
}

// ------------------------------------------------------------- host driver
// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
    else
      cudaGetLastError();
  }
  return fn;
}

template <typename T> static CUtensorMapDataType tmap_dtype() {
  if (std::is_same<T, float>::value) return CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  switch (sizeof(T)) {
    case 1: return CU_TENSOR_MAP_DATA_TYPE_UINT8;
    case 2: return CU_TENSOR_MAP_DATA_TYPE_UINT16;
    case 4: return CU_TENSOR_MAP_DATA_TYPE_UINT32;
    default: return CU_TENSOR_MAP_DATA_TYPE_UINT64;
  }
}

// the structure of one CCL call, all device pointers inside the scratch arena
struct CclPlan {
  uint32_t sx, sy, sz, wpr;
  uint64_t n, W;  // voxels, words
  uint32_t *S, *Z, *Ey, *Ez, *rbase;
  uint32_t R;       // runs
  uint32_t* label;  // [R+1]: parent during the build, then the label of every run
  uint32_t* rank;   // [R+1] scratch of the build
  uint32_t ncomp;
  void* cub_tmp;
  size_t cub_bytes;
  ExpandArgs expand_args(uint64_t offset) const {
    ExpandArgs e;
    e.sx = sx; e.wpr = wpr; e.rows = (uint64_t)sy * sz; e.offset = offset;
    e.S = S; e.Z = Z; e.rbase = rbase; e.label = label;
    return e;
  }
};

static int check_ccl_dims(uint64_t sx, uint64_t sy, uint64_t sz) {
  IGN_REQUIRE(sx > 0 && sy > 0 && sz > 0, IGN_ERR_INVALID, "empty volume");
  IGN_REQUIRE(sx < (1ull << 31) && sy < (1ull << 31) && sz < (1ull << 31), IGN_ERR_OVERFLOW, "CCL extent too large");
  const uint64_t wpr = (sx + 31) / 32;
  IGN_REQUIRE(wpr <= (uint64_t)TB_WMAX, IGN_ERR_OVERFLOW, "CCL rows longer than %d voxels are not supported", TB_WMAX * 32);
  IGN_REQUIRE(sy * sz < (1ull << 40) && wpr * sy * sz < 0x7FFFFFF0ull, IGN_ERR_OVERFLOW,
              "CCL volume of %llu voxels exceeds the 2^36 voxel limit; split it into tasks (igneous uses 512^3)",
              (unsigned long long)(sx * sy * sz));
  return IGN_OK;
}

static size_t ccl_cub_bytes(uint64_t items) {
  size_t b = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, b, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)items);
  return b + 256;
}
// arena bytes of a CCL with W mask words whose runs fit rcap
static size_t ccl_scratch_bytes(uint64_t W, uint64_t rcap) {
  const uint64_t items = (W + 1 > rcap + 1 ? W + 1 : rcap + 1);
  return 5 * align_up((W + 2) * 4, 256) + 2 * align_up((rcap + 2) * 4, 256) + align_up(ccl_cub_bytes(items), 256) + 8192;
}
static uint64_t default_rcap(uint64_t n) { return n / 8 + 4096; }

// Pass A .. run labels.  On success plan.label[r] = component id (1..ncomp, cc3d numbering)
// of every run and plan.ncomp is on the host.  `rcap` = run capacity reserved in the arena;
// *need_rcap > rcap on return means the volume has more runs (nothing else is valid).
template <typename R>
static int ccl_structure(ign_ctx* ctx, Scratch& sc, const R& rd, uint32_t sx, uint32_t sy, uint32_t sz, uint64_t rcap,
                         CclPlan& p, uint64_t* need_rcap) {
  using T = typename R::value_type;
  using MT = MaskTile<T>;
  p.sx = sx; p.sy = sy; p.sz = sz;
  p.wpr = (sx + 31) / 32;
  p.n = (uint64_t)sx * sy * sz;
  p.W = (uint64_t)p.wpr * sy * sz;
  p.R = 0;
  p.ncomp = 0;
  const uint64_t W = p.W;
  p.S = sc.take<uint32_t>(W + 2);
  p.Z = sc.take<uint32_t>(W + 2);
  p.Ey = sc.take<uint32_t>(W + 2);
  p.Ez = sc.take<uint32_t>(W + 2);
  p.rbase = sc.take<uint32_t>(W + 2);
  p.label = sc.take<uint32_t>(rcap + 2);
  p.rank = sc.take<uint32_t>(rcap + 2);
  const uint64_t items = (W + 1 > rcap + 1 ? W + 1 : rcap + 1);
  p.cub_bytes = ccl_cub_bytes(items);
  p.cub_tmp = sc.take(p.cub_bytes);
  IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "CCL scratch arena too small");
  *need_rcap = 0;

  // ---- pass A
  MaskArgs ma;
  ma.sx = sx; ma.sy = sy; ma.sz = sz; ma.wpr = p.wpr;
  ma.ntx = (sx + MT_BX - 1) / MT_BX;
  ma.nty = (sy + MT_BY - 1) / MT_BY;
  ma.ntz = (sz + MT::BZ - 1) / MT::BZ;
  ma.nby = (ma.nty + 7) / 8;
  ma.nbz = (ma.ntz + 7) / 8;
  ma.ncols = ma.nby * ma.nbz * 64;
  ma.S = p.S; ma.Z = p.Z; ma.Ey = p.Ey; ma.Ez = p.Ez;
  // whole-sector mask writes pay off where L2 no longer merges the half sectors of x-neighbours: rows of
  // 16+ tiles (measured at 2048^3: 12.7 vs 16.3 ms; at 1024^3 the unpaired kernel is faster, 1.27 vs 1.60 ms)
  ma.pair = (p.wpr % 8 == 0 && sx % MT_BX == 0 && ma.ntx >= 16) ? 1u : 0u;
  if (const char* e = getenv("IGN_CCL_PAIR")) ma.pair = (atoi(e) != 0 && p.wpr % 8 == 0 && sx % MT_BX == 0) ? 1u : 0u;
  const uint64_t ntiles = (uint64_t)ma.ntx * ma.ncols;
  const size_t es = sizeof(T);
  CUtensorMap tmap;
  memset(&tmap, 0, sizeof(tmap));
  const bool use_tma = ((uint64_t)sx * es) % 16 == 0 && ((uintptr_t)rd.in % 16) == 0 && getenv("IGN_CCL_NO_TMA") == nullptr;
  if (use_tma) {
    EncodeTiledFn enc = encode_tiled_fn();
    IGN_REQUIRE(enc != nullptr, IGN_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    const cuuint64_t gdim[3] = {sx, sy, sz};
    const cuuint64_t gstr[2] = {(cuuint64_t)sx * es, (cuuint64_t)sx * sy * es};
    const cuuint32_t box[3] = {(cuuint32_t)MT::PITCH, MT_BY + 1, (cuuint32_t)MT::BZ + 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_128B;
    if (const char* e = getenv("IGN_CCL_L2PROMO")) promo = atoi(e) == 256 ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B : (atoi(e) == 64 ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B : (atoi(e) == 0 ? CU_TENSOR_MAP_L2_PROMOTION_NONE : promo));
    const CUresult r = enc(&tmap, tmap_dtype<T>(), 3, (void*)rd.in, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_NONE, promo,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    IGN_REQUIRE(r == CUDA_SUCCESS, IGN_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for %ux%ux%u", (int)r, sx, sy, sz);
  }
  {
    const size_t smem = (use_tma ? 2 : 1) * MT::BYTES;
    unsigned per_sm = (unsigned)(200 * 1024 / (smem + 1024)) < 8u ? (unsigned)(200 * 1024 / (smem + 1024)) : 8u;
    if (const char* e = getenv("IGN_CCL_MASK_CTAS")) per_sm = (unsigned)atoi(e) ? (unsigned)atoi(e) : per_sm;
    const uint64_t cap = (uint64_t)ctx->sm_count * (per_sm ? per_sm : 1);
    const uint64_t units = ma.pair ? ntiles / 2 : ntiles;  // tile pairs when the CTAs write whole mask sectors
    const unsigned grid = (unsigned)(units < cap ? units : cap);
    IGN_CUDA(cudaMemsetAsync(p.S + W, 0, 8, ctx->stream));  // sentinel words S[W], S[W+1]
    auto launch = [&](auto kern) -> int {
      IGN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      IGN_LAUNCH_PROF(ctx, IGN_PROF_CCL_LOCAL, kern, grid, MT_THREADS, smem, tmap, rd, ma);
      return IGN_OK;
    };
    if (use_tma) {
      if (ma.pair) IGN_TRY(launch(k_ccl_masks<T, R::thresholded, true, true>));
      else IGN_TRY(launch(k_ccl_masks<T, R::thresholded, true, false>));
    } else {
      if (ma.pair) IGN_TRY(launch(k_ccl_masks<T, R::thresholded, false, true>));
      else IGN_TRY(launch(k_ccl_masks<T, R::thresholded, false, false>));
    }
  }
  // ---- run ids: exclusive scan of popc(S) over W+1 words (rbase[W] = number of runs)
  {
    auto it = thrust::make_transform_iterator((const uint32_t*)p.S, PopcOp());
    size_t tb = p.cub_bytes;
    IGN_CUDA(cub::DeviceScan::ExclusiveSum(p.cub_tmp, tb, it, p.rbase, (int)(W + 1), ctx->stream));
    ctx->launches += 2;
  }
  uint32_t hR = 0;
  IGN_TRY(small_d2h(ctx, &hR, p.rbase + W, 4));
  IGN_TRY(small_sync(ctx));
  p.R = hR;
  if ((uint64_t)hR > rcap) {
    *need_rcap = hR;
    return IGN_OK;
  }
  if (hR == 0) return IGN_OK;
  IGN_REQUIRE(hR < 0x7FFFFFF0u, IGN_ERR_OVERFLOW, "CCL: %u runs exceed the 2^31 limit; split the volume into tasks", hR);
  const uint32_t Rn = hR;
  // ---- pass B: tiles, then the rows on tile faces
  uint32_t TY = 8;
  while (TY > 1 && (uint64_t)p.wpr * TY * TY > (uint64_t)TB_WMAX) TY >>= 1;
  TileArgs ta;
  ta.sx = sx; ta.sy = sy; ta.sz = sz; ta.wpr = p.wpr; ta.TY = TY; ta.TZ = TY;
  ta.nty = (sy + TY - 1) / TY;
  ta.ntz = (sz + TY - 1) / TY;
  ta.wpr_shift = ta.ty_shift = 0xFFFFFFFFu;
  if ((p.wpr & (p.wpr - 1)) == 0) {  // TY is a power of two by construction
    ta.wpr_shift = 0;
    while ((1u << ta.wpr_shift) < p.wpr) ta.wpr_shift++;
    ta.ty_shift = 0;
    while ((1u << ta.ty_shift) < TY) ta.ty_shift++;
  }
  ta.S = p.S; ta.Ey = p.Ey; ta.Ez = p.Ez; ta.rbase = p.rbase; ta.parent = p.label;
  {
    ta.wcap = (p.wpr * TY * TY + 3u) & ~3u;
    const size_t smem = (size_t)3 * ta.wcap * 4 + (size_t)TB_RCAP * 4 + (size_t)(TB_THREADS / 32) * TB_QCAP * 4 +
                        (size_t)(ta.wcap + 2) * 2;
    IGN_CUDA(cudaFuncSetAttribute(k_ccl_tiles, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    IGN_REQUIRE((uint64_t)ta.nty * ta.ntz < 0x7FFFFFFFull, IGN_ERR_OVERFLOW, "too many CCL tiles");
    IGN_LAUNCH_PROF(ctx, IGN_PROF_CCL_MERGE, k_ccl_tiles, ta.nty * ta.ntz, TB_THREADS, smem, ta);
  }
  if (ta.nty > 1 || ta.ntz > 1) {
    MergeArgs me;
    me.sx = sx; me.sy = sy; me.sz = sz; me.wpr = p.wpr; me.TY = TY; me.TZ = TY; me.nty = ta.nty; me.ntz = ta.ntz;
    me.words_y = (uint64_t)(ta.nty - 1) * sz * p.wpr;
    me.words_z = (uint64_t)(ta.ntz - 1) * sy * p.wpr;
    me.S = p.S; me.Ey = p.Ey; me.Ez = p.Ez; me.rbase = p.rbase; me.parent = p.label;
    const uint64_t mitems = ((uint64_t)(ta.nty - 1) * sz + (uint64_t)(ta.ntz - 1) * sy) * ((p.wpr + MG_W - 1) / MG_W);
    IGN_REQUIRE(mitems / 256 < 0x7FFFFFFFull, IGN_ERR_OVERFLOW, "too many CCL face words");
    IGN_LAUNCH_PROF(ctx, IGN_PROF_CCL_MERGE, k_ccl_merge, blocks_for(mitems, 256), 256, 0, me);
  }
  // ---- roots: flatten, rank = exclusive scan over (parent[r] == r), labels
  IGN_LAUNCH_PROF(ctx, IGN_PROF_CCL_MERGE, k_ccl_flatten, blocks_for(Rn, 256), 256, 0, p.label, Rn);
  IGN_CUDA(cudaMemsetAsync(p.label + Rn, 0xFF, 4, ctx->stream));  // sentinel: not a root
  {
    IsRootOp op;
    op.parent = p.label;
    auto it = thrust::make_transform_iterator(thrust::counting_iterator<uint32_t>(0), op);
    size_t tb = p.cub_bytes;
    IGN_CUDA(cub::DeviceScan::ExclusiveSum(p.cub_tmp, tb, it, p.rank, (int)(Rn + 1), ctx->stream));
    ctx->launches += 2;
  }
  uint32_t hN = 0;
  IGN_TRY(small_d2h(ctx, &hN, p.rank + Rn, 4));
  IGN_LAUNCH_PROF(ctx, IGN_PROF_CCL_MERGE, k_ccl_runlabel, blocks_for(Rn, 256), 256, 0, p.label, p.rank, Rn);
  IGN_TRY(small_sync(ctx));
  p.ncomp = hN;
  return IGN_OK;
}

template <typename T>
static Reader<T, false> plain_reader(const void* in) {
  Reader<T, false> r;
  r.in = (const T*)in;
  r.gte = r.lte = 0;
  r.use_gte = r.use_lte = 0;
  r.rx = r.ry = r.rz = 0xFFFFFFFFu;
  return r;
}

static int launch_expand(ign_ctx* ctx, const CclPlan& p, uint64_t offset, void* out, int out_dtype,
                         uint64_t max_label) {
  const ExpandArgs e = p.expand_args(offset);
  const bool vec = (p.sx % 4 == 0) && ((uintptr_t)out % 16 == 0);
  // vector path: a warp owns EX_G 128-voxel groups of one row; scalar path: EX_G consecutive words
  const uint64_t warps = vec ? e.rows * (((p.wpr + 3) / 4 + EX_G - 1) / EX_G) : (e.rows * p.wpr + EX_G - 1) / EX_G;
  IGN_REQUIRE(warps * 32 / 256 < 0x7FFFFFFFull, IGN_ERR_OVERFLOW, "CCL expand grid too large");
  const unsigned grid = blocks_for(warps * 32, 256);
  switch (out_dtype) {
    case IGN_U16:
      IGN_REQUIRE(max_label + offset <= 0xFFFFull, IGN_ERR_OVERFLOW, "%llu labels do not fit uint16", (unsigned long long)max_label);
      if (vec) IGN_LAUNCH_PROF(ctx, IGN_PROF_CCL_LABEL, (k_ccl_expand4<uint16_t>), grid, 256, 0, e, (uint16_t*)out);
      else IGN_LAUNCH_PROF(ctx, IGN_PROF_CCL_LABEL, (k_ccl_expand1<uint16_t>), grid, 256, 0, e, (uint16_t*)out);
      break;
    case IGN_U32:
      IGN_REQUIRE(max_label + offset <= 0xFFFFFFFFull, IGN_ERR_OVERFLOW, "labels do not fit uint32");
      if (vec) IGN_LAUNCH_PROF(ctx, IGN_PROF_CCL_LABEL, (k_ccl_expand4<uint32_t>), grid, 256, 0, e, (uint32_t*)out);
      else IGN_LAUNCH_PROF(ctx, IGN_PROF_CCL_LABEL, (k_ccl_expand1<uint32_t>), grid, 256, 0, e, (uint32_t*)out);
      break;
    case IGN_U64:
      if (vec) IGN_LAUNCH_PROF(ctx, IGN_PROF_CCL_LABEL, (k_ccl_expand4<uint64_t>), grid, 256, 0, e, (uint64_t*)out);
      else IGN_LAUNCH_PROF(ctx, IGN_PROF_CCL_LABEL, (k_ccl_expand1<uint64_t>), grid, 256, 0, e, (uint64_t*)out);
      break;
    default:
      set_error("CCL out_dtype must be u16/u32/u64 (got %d)", out_dtype);
      return IGN_ERR_UNSUPPORTED;
  }
  return IGN_OK;
}

// dust on the run labels of p: components with fewer than `threshold` voxels get label 0,
// the others are renumbered 1..kept in the same order.
static int dust_runs(ign_ctx* ctx, Scratch& sc, CclPlan& p, uint64_t threshold, uint32_t* kept) {
  const uint32_t N = p.ncomp;
  *kept = N;
  if (N == 0 || p.R == 0) return IGN_OK;
  const size_t bytes = ((size_t)N + 2) * 4;
  uint32_t* counts = sc.take<uint32_t>((size_t)N + 2);
  uint32_t* keep = sc.take<uint32_t>((size_t)N + 2);
  uint32_t* scan = sc.take<uint32_t>((size_t)N + 2);
  uint32_t* lut = sc.take<uint32_t>((size_t)N + 2);
  size_t tb = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, tb, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)(N + 2));
  void* tmp = sc.take(tb + 256);
  IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small for dust maps");
  IGN_CUDA(cudaMemsetAsync(counts, 0, bytes, ctx->stream));
  const ExpandArgs e = p.expand_args(0);
  IGN_LAUNCH(ctx, k_ccl_count, blocks_for(p.W, 256), 256, 0, e, counts);
  IGN_LAUNCH(ctx, k_dust_flags, blocks_for((uint64_t)N + 2, 256), 256, 0, counts, N, threshold, keep);
  IGN_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, keep, scan, (int)(N + 2), ctx->stream));
  ctx->launches += 2;
  IGN_LAUNCH(ctx, k_dust_lut, blocks_for((uint64_t)N + 1, 256), 256, 0, keep, scan, N, lut);
  IGN_LAUNCH(ctx, k_ccl_relabel_runs, blocks_for(p.R, 256), 256, 0, p.label, p.R, lut);
  uint32_t h = 0;
  IGN_TRY(small_d2h(ctx, &h, scan + (N + 1), 4));  // keep[N+1] is 0: scan[N+1] = number kept
  IGN_TRY(small_sync(ctx));
  *kept = h;
  return IGN_OK;
}

// full pipeline for one reader type; out may be null when only dust-in-place is wanted
template <typename R, typename TL>
static int ccl_run(ign_ctx* ctx, const R& rd, uint64_t sx, uint64_t sy, uint64_t sz,
                   uint64_t dust_threshold, uint64_t offset, void* out, int out_dtype,
                   TL* dust_labels_inplace, uint64_t* n_components) {
  IGN_TRY(check_ccl_dims(sx, sy, sz));
  const uint64_t n = sx * sy * sz, W = ((sx + 31) / 32) * sy * sz;
  Scratch sc(ctx);
  uint64_t rcap = default_rcap(n);
  for (int attempt = 0; attempt < 2; attempt++) {
    sc.rewind();
    IGN_TRY(sc.reserve(ccl_scratch_bytes(W, rcap) + 6 * (rcap + 4) * 4 + 65536));
    CclPlan p;
    uint64_t need = 0;
    IGN_TRY(ccl_structure(ctx, sc, rd, (uint32_t)sx, (uint32_t)sy, (uint32_t)sz, rcap, p, &need));
    if (need > rcap) {
      IGN_REQUIRE(attempt == 0, IGN_ERR_NOMEM, "CCL: %llu runs do not fit the scratch arena", (unsigned long long)need);
      rcap = need + 16;
      continue;
    }
    uint32_t kept = p.ncomp;
    if (dust_threshold > 0 && p.ncomp > 0) IGN_TRY(dust_runs(ctx, sc, p, dust_threshold, &kept));
    if (dust_labels_inplace != nullptr && dust_threshold > 0 && p.R > 0) {
      const ExpandArgs e = p.expand_args(0);
      IGN_LAUNCH(ctx, (k_dust_apply<TL>), blocks_for(p.W * 32, 256), 256, 0, e, dust_labels_inplace);
    }
    if (out != nullptr) {
      if (p.R == 0) IGN_CUDA(cudaMemsetAsync(out, 0, n * dtype_size(out_dtype), ctx->stream));
      else IGN_TRY(launch_expand(ctx, p, offset, out, out_dtype, kept));
    }
    if (n_components) *n_components = kept;
    return IGN_OK;
  }
  return IGN_ERR_OVERFLOW;
}

template <typename T>
static int ccl_task_typed(ign_ctx* ctx, const void* in, uint64_t sx, uint64_t sy, uint64_t sz,
                          int use_gte, double gte, int use_lte, double lte, uint64_t rx, uint64_t ry,
                          uint64_t rz, uint64_t dust, uint64_t offset, uint64_t* out, uint64_t* n) {
  auto rail = [](uint64_t r, uint64_t s) { return (r < s) ? (uint32_t)r : 0xFFFFFFFFu; };
  if (use_gte || use_lte) {
    Reader<T, true> r;
    r.in = (const T*)in;
    r.gte = gte;
    r.lte = lte;
    r.use_gte = use_gte;
    r.use_lte = use_lte;
    r.rx = rail(rx, sx);
    r.ry = rail(ry, sy);
    r.rz = rail(rz, sz);
    return ccl_run(ctx, r, sx, sy, sz, dust, offset, out, IGN_U64, (uint8_t*)nullptr, n);
  }
  if constexpr (std::is_same<T, float>::value) {
    set_error("CCL on float input requires a threshold");
    return IGN_ERR_UNSUPPORTED;
  } else {
    Reader<T, false> r = plain_reader<T>(in);
    r.rx = rail(rx, sx);
    r.ry = rail(ry, sy);
    r.rz = rail(rz, sz);
    return ccl_run(ctx, r, sx, sy, sz, dust, offset, out, IGN_U64, (uint8_t*)nullptr, n);
  }
}

}  // namespace ign

using namespace ign;

// ---------------------------------------------------------------- volume CCL
// begin / finish are split so that a multi-GPU run can exchange the outer planes of
// every rank's volume in between (ONE all-gather) and fold the global relabelling into
// the run labels before the single expansion pass.
struct ign_ccl_volume {
  ign_ctx* ctx;
  const void* in;
  int in_dtype;
  CclPlan plan;
  uint64_t n_local;
  size_t base;  // the masks and run labels are held in the arena above this
};

template <typename T>
static int volume_begin_typed(ign_ctx* ctx, Scratch& sc, ign_ccl_volume* v, uint64_t sx, uint64_t sy, uint64_t sz,
                              uint64_t* first_values, uint32_t* first_labels, uint64_t* last_values,
                              uint32_t* last_labels) {
  const uint64_t n = sx * sy * sz, W = ((sx + 31) / 32) * sy * sz;
  uint64_t rcap = default_rcap(n);
  for (int attempt = 0; attempt < 2; attempt++) {
    sc.rewind();
    IGN_TRY(sc.reserve(ccl_scratch_bytes(W, rcap) + (rcap + 64) * 4 + 65536));
    uint64_t need = 0;
    IGN_TRY(ccl_structure(ctx, sc, plain_reader<T>(v->in), (uint32_t)sx, (uint32_t)sy, (uint32_t)sz, rcap, v->plan, &need));
    if (need > rcap) {
      IGN_REQUIRE(attempt == 0, IGN_ERR_NOMEM, "CCL: %llu runs do not fit the scratch arena", (unsigned long long)need);
      rcap = need + 16;
      continue;
    }
    break;
  }
  v->n_local = v->plan.ncomp;
  if (first_values && first_labels && last_values && last_labels) {
    const uint64_t np = sx * sy;
    const ExpandArgs e = v->plan.expand_args(0);
    if (v->plan.R == 0) {
      IGN_CUDA(cudaMemsetAsync(first_labels, 0, np * 4, ctx->stream));
      IGN_CUDA(cudaMemsetAsync(last_labels, 0, np * 4, ctx->stream));
      IGN_CUDA(cudaMemsetAsync(first_values, 0, np * 8, ctx->stream));
      IGN_CUDA(cudaMemsetAsync(last_values, 0, np * 8, ctx->stream));
    } else {
      IGN_LAUNCH(ctx, (k_ccl_plane<T>), blocks_for(np, 256), 256, 0, (const T*)v->in, e, (uint64_t)0, (uint32_t)sy, first_values, first_labels);
      IGN_LAUNCH(ctx, (k_ccl_plane<T>), blocks_for(np, 256), 256, 0, (const T*)v->in, e, (uint64_t)(sz - 1), (uint32_t)sy, last_values, last_labels);
    }
    IGN_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  return IGN_OK;
}

// One rank's share of a CCL over a dataset that is split into z-slabs (rank r above rank r-1).
// Exactly ONE collective: an all-gather of [n_local | first plane | last plane]; linking the
// N-1 boundaries, the replicated union-find and the relabelling all run on the device.
template <typename T>
static int ccl_sharded_typed(ign_group* g, Scratch& sc, ign_ccl_volume* v, uint64_t sx, uint64_t sy, uint64_t sz, void* out,
                             int out_dtype, uint64_t* n_global) {
  ign_ctx* ctx = g->ctx;
  const int N = g->nranks, me = g->rank;
  const uint64_t np = sx * sy;
  const size_t rec = 256 + 2 * np * 8 + 2 * np * 4;
  IGN_TRY(grow_buffer(ctx, &g->d_send, &g->send_bytes, rec, "multi-GPU CCL"));
  IGN_TRY(grow_buffer(ctx, &g->d_recv, &g->recv_bytes, rec * (size_t)N, "multi-GPU CCL"));
  uint64_t* first_v = (uint64_t*)(g->d_send + 256);
  uint64_t* last_v = first_v + np;
  uint32_t* first_l = (uint32_t*)(last_v + np);
  uint32_t* last_l = first_l + np;
  IGN_TRY(volume_begin_typed<T>(ctx, sc, v, sx, sy, sz, first_v, first_l, last_v, last_l));
  CclPlan& p = v->plan;
  uint64_t head[32] = {0};
  head[0] = v->n_local;
  IGN_TRY(small_h2d(ctx, g->d_send, head, 256));
  IGN_TRY(ign_group_allgather(g, g->d_send, rec, g->d_recv));
  std::vector<uint64_t> nloc(N, 0);
  for (int r = 0; r < N; r++) IGN_TRY(small_d2h(ctx, &nloc[r], g->d_recv + (size_t)r * rec, 8));
  IGN_TRY(small_sync(ctx));
  std::vector<uint64_t> off(N + 1, 0);
  for (int r = 0; r < N; r++) off[r + 1] = off[r] + nloc[r];
  const uint64_t total = off[N];
  IGN_REQUIRE(total < 0x7FFFFFF0ull, IGN_ERR_OVERFLOW, "multi-GPU CCL: too many provisional components");
  const uint32_t items = (uint32_t)total + 2;  // ids 0..total and one sentinel
  const size_t cubb = ccl_cub_bytes(items);
  IGN_TRY(grow_buffer(ctx, &g->d_solve, &g->solve_bytes, 2 * align_up((size_t)items * 4, 256) + align_up(cubb, 256),
                      "multi-GPU CCL"));
  uint32_t* parent = (uint32_t*)g->d_solve;
  uint32_t* rank = (uint32_t*)(g->d_solve + align_up((size_t)items * 4, 256));
  void* tmp = g->d_solve + 2 * align_up((size_t)items * 4, 256);
  IGN_LAUNCH(ctx, k_iota_u32, blocks_for(items, 256), 256, 0, parent, items);
  for (int b = 0; b + 1 < N; b++) {
    const char* ra = g->d_recv + (size_t)b * rec;
    const char* rb = g->d_recv + (size_t)(b + 1) * rec;
    const uint64_t* va = (const uint64_t*)(ra + 256) + np;                     // last plane of rank b
    const uint32_t* la = (const uint32_t*)(ra + 256 + 2 * np * 8) + np;
    const uint64_t* vb = (const uint64_t*)(rb + 256);                          // first plane of rank b+1
    const uint32_t* lb = (const uint32_t*)(rb + 256 + 2 * np * 8);
    IGN_LAUNCH_PROF(ctx, IGN_PROF_CCL_MERGE, k_ccl_link_union, blocks_for(np, 256), 256, 0, va, la, (uint32_t)off[b], vb, lb,
                    (uint32_t)off[b + 1], np, parent);
  }
  // roots in ascending id order: the exclusive scan is the dataset-wide cc3d numbering
  IGN_LAUNCH(ctx, k_ccl_flatten, blocks_for(items - 1, 256), 256, 0, parent, items - 1);
  IGN_CUDA(cudaMemsetAsync(parent + (items - 1), 0xFF, 4, ctx->stream));  // sentinel: not a root
  {
    IsRootOp op;
    op.parent = parent;
    auto it = thrust::make_transform_iterator(thrust::counting_iterator<uint32_t>(0), op);
    size_t tb = cubb;
    IGN_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, it, rank, (int)items, ctx->stream));
    ctx->launches += 2;
  }
  uint32_t hN = 0;
  IGN_TRY(small_d2h(ctx, &hN, rank + (items - 1), 4));  // roots incl. id 0
  IGN_LAUNCH(ctx, k_ccl_rank_of_root, blocks_for(items - 1, 256), 256, 0, parent, rank, items - 1);
  const uint64_t nglob_max = total;
  if (p.R > 0) {
    IGN_LAUNCH(ctx, k_ccl_relabel_runs, blocks_for(p.R, 256), 256, 0, p.label, p.R, (const uint32_t*)parent + off[me]);
    IGN_TRY(launch_expand(ctx, p, 0, out, out_dtype, nglob_max));
  } else {
    IGN_CUDA(cudaMemsetAsync(out, 0, sx * sy * sz * dtype_size(out_dtype), ctx->stream));
  }
  IGN_TRY(small_sync(ctx));
  if (n_global) *n_global = hN ? hN - 1 : 0;
  return IGN_OK;
}

extern "C" {

int ign_ccl6_dev(ign_ctx* ctx, const void* in, int in_dtype, uint64_t sx, uint64_t sy, uint64_t sz,
                 void* out, int out_dtype, uint64_t* n_components) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(in && out, IGN_ERR_INVALID, "null buffer");
  switch (in_dtype) {
    case IGN_U8: return ccl_run(ctx, plain_reader<uint8_t>(in), sx, sy, sz, 0, 0, out, out_dtype, (uint8_t*)nullptr, n_components);
    case IGN_U16: return ccl_run(ctx, plain_reader<uint16_t>(in), sx, sy, sz, 0, 0, out, out_dtype, (uint16_t*)nullptr, n_components);
    case IGN_U32: return ccl_run(ctx, plain_reader<uint32_t>(in), sx, sy, sz, 0, 0, out, out_dtype, (uint32_t*)nullptr, n_components);
    case IGN_U64: return ccl_run(ctx, plain_reader<uint64_t>(in), sx, sy, sz, 0, 0, out, out_dtype, (uint64_t*)nullptr, n_components);
  }
  set_error("CCL: unsupported input dtype %d", in_dtype);
  return IGN_ERR_UNSUPPORTED;
}

int ign_dust_dev(ign_ctx* ctx, void* labels, int dtype, uint64_t sx, uint64_t sy, uint64_t sz,
                 uint64_t threshold) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(labels, IGN_ERR_INVALID, "null buffer");
  if (threshold == 0) return IGN_OK;
  switch (dtype) {
    case IGN_U8: return ccl_run(ctx, plain_reader<uint8_t>(labels), sx, sy, sz, threshold, 0, nullptr, IGN_U64, (uint8_t*)labels, nullptr);
    case IGN_U16: return ccl_run(ctx, plain_reader<uint16_t>(labels), sx, sy, sz, threshold, 0, nullptr, IGN_U64, (uint16_t*)labels, nullptr);
    case IGN_U32: return ccl_run(ctx, plain_reader<uint32_t>(labels), sx, sy, sz, threshold, 0, nullptr, IGN_U64, (uint32_t*)labels, nullptr);
    case IGN_U64: return ccl_run(ctx, plain_reader<uint64_t>(labels), sx, sy, sz, threshold, 0, nullptr, IGN_U64, (uint64_t*)labels, nullptr);
  }
  set_error("dust: unsupported dtype %d", dtype);
  return IGN_ERR_UNSUPPORTED;
}

int ign_ccl_task_dev(ign_ctx* ctx, const void* in, int in_dtype, uint64_t sx, uint64_t sy,
                     uint64_t sz, int use_gte, double gte, int use_lte, double lte,
                     uint64_t rail_x, uint64_t rail_y, uint64_t rail_z, uint64_t dust_threshold,
                     uint64_t label_offset, uint64_t* out, uint64_t* n_components) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(in && out, IGN_ERR_INVALID, "null buffer");
  switch (in_dtype) {
    case IGN_U8: return ccl_task_typed<uint8_t>(ctx, in, sx, sy, sz, use_gte, gte, use_lte, lte, rail_x, rail_y, rail_z, dust_threshold, label_offset, out, n_components);
    case IGN_U16: return ccl_task_typed<uint16_t>(ctx, in, sx, sy, sz, use_gte, gte, use_lte, lte, rail_x, rail_y, rail_z, dust_threshold, label_offset, out, n_components);
    case IGN_U32: return ccl_task_typed<uint32_t>(ctx, in, sx, sy, sz, use_gte, gte, use_lte, lte, rail_x, rail_y, rail_z, dust_threshold, label_offset, out, n_components);
    case IGN_U64: return ccl_task_typed<uint64_t>(ctx, in, sx, sy, sz, use_gte, gte, use_lte, lte, rail_x, rail_y, rail_z, dust_threshold, label_offset, out, n_components);
    case IGN_F32: return ccl_task_typed<float>(ctx, in, sx, sy, sz, use_gte, gte, use_lte, lte, rail_x, rail_y, rail_z, dust_threshold, label_offset, out, n_components);
  }
  set_error("CCL task: unsupported input dtype %d", in_dtype);
  return IGN_ERR_UNSUPPORTED;
}

// ---- host-buffer wrappers
int ign_ccl6(ign_ctx* ctx, const void* in, int in_dtype, uint64_t sx, uint64_t sy, uint64_t sz,
             void* out, int out_dtype, uint64_t* n_components) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(in && out, IGN_ERR_INVALID, "null buffer");
  IGN_TRY(check_ccl_dims(sx, sy, sz));
  const int es = dtype_size(in_dtype), os = dtype_size(out_dtype);
  IGN_REQUIRE(es > 0 && os > 0, IGN_ERR_UNSUPPORTED, "unsupported dtype");
  const uint64_t n = sx * sy * sz;
  Staging st(ctx);
  void *d_in, *d_out;
  st.add(&d_in, n * es, in);
  st.add(&d_out, n * os);
  IGN_TRY(st.stage());
  IGN_TRY(ign_ccl6_dev(ctx, d_in, in_dtype, sx, sy, sz, d_out, out_dtype, n_components));
  IGN_TRY(st.back(out, d_out, n * os));
  return st.sync();
}

int ign_dust(ign_ctx* ctx, void* labels, int dtype, uint64_t sx, uint64_t sy, uint64_t sz,
             uint64_t threshold) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(labels, IGN_ERR_INVALID, "null buffer");
  if (threshold == 0) return IGN_OK;
  IGN_TRY(check_ccl_dims(sx, sy, sz));
  const int es = dtype_size(dtype);
  IGN_REQUIRE(es > 0 && dtype != IGN_F32, IGN_ERR_UNSUPPORTED, "unsupported dtype");
  const uint64_t n = sx * sy * sz;
  Staging st(ctx);
  void* d;
  st.add(&d, n * es, labels);
  IGN_TRY(st.stage());
  IGN_TRY(ign_dust_dev(ctx, d, dtype, sx, sy, sz, threshold));
  IGN_TRY(st.back(labels, d, n * es));
  return st.sync();
}

int ign_ccl6_link_dev(ign_ctx* ctx, const uint64_t* values_a, const uint32_t* labels_a,
                      uint64_t offset_a, const uint64_t* values_b, const uint32_t* labels_b,
                      uint64_t offset_b, uint64_t n_plane, uint64_t* pairs_host, uint64_t capacity,
                      uint64_t* n_pairs) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(values_a && labels_a && values_b && labels_b && n_pairs, IGN_ERR_INVALID, "null argument");
  *n_pairs = 0;
  if (n_plane == 0) return IGN_OK;
  Scratch sc(ctx);
  const uint32_t cap = (uint32_t)(n_plane < 0x7FFFFFFFull ? n_plane : 0x7FFFFFFFull);
  IGN_TRY(sc.reserve((size_t)cap * 16 + 8192));
  uint64_t* d_pairs = sc.take<uint64_t>(2 * (size_t)cap);
  uint32_t* counters = sc.take<uint32_t>(64);
  IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small (CCL link)");
  IGN_CUDA(cudaMemsetAsync(counters, 0, 256, ctx->stream));
  IGN_LAUNCH(ctx, k_ccl_link, blocks_for(n_plane, 256), 256, 0, values_a, labels_a, offset_a, values_b,
             labels_b, offset_b, n_plane, d_pairs, cap, counters);
  uint32_t* h = (uint32_t*)ctx->pinned;
  IGN_CUDA(cudaMemcpyAsync(h, counters, 4, cudaMemcpyDeviceToHost, ctx->stream));
  IGN_CUDA(cudaStreamSynchronize(ctx->stream));
  const uint64_t total = h[0];
  *n_pairs = total;
  if (pairs_host && total) {
    const uint64_t m = total < capacity ? total : capacity;
    IGN_CUDA(cudaMemcpy(pairs_host, d_pairs, m * 16, cudaMemcpyDeviceToHost));
  }
  return IGN_OK;
}

// Host-side global union-find over provisional ids 1..total (the B200-native
// stand-in for create_relabeling, igneous/tasks/image/ccl.py:358-420):
// smaller id wins (ccl.py:70-73); final ids are the ranks of the component
// minima, i.e. identical to a whole-volume cc3d numbering.
int ign_ccl6_solve(const uint64_t* pairs, uint64_t n_pairs, uint64_t total, uint32_t* lut,
                   uint64_t* n_global) {
  IGN_REQUIRE(lut && n_global && (n_pairs == 0 || pairs), IGN_ERR_INVALID, "null argument");
  IGN_REQUIRE(total < 0xFFFFFFF0ull, IGN_ERR_OVERFLOW, "too many provisional components");
  std::vector<uint32_t> p(total + 1);
  for (uint64_t i = 0; i <= total; i++) p[i] = (uint32_t)i;
  auto find = [&](uint32_t i) {
    while (p[i] != i) {
      p[i] = p[p[i]];
      i = p[i];
    }
    return i;
  };
  for (uint64_t k = 0; k < n_pairs; k++) {
    const uint64_t a64 = pairs[2 * k], b64 = pairs[2 * k + 1];
    IGN_REQUIRE(a64 >= 1 && a64 <= total && b64 >= 1 && b64 <= total, IGN_ERR_INVALID,
                "equivalence pair (%llu,%llu) out of range", (unsigned long long)a64, (unsigned long long)b64);
    const uint32_t a = find((uint32_t)a64), b = find((uint32_t)b64);
    if (a < b) p[b] = a;
    else if (b < a) p[a] = b;
  }
  uint32_t next = 0;
  lut[0] = 0;
  for (uint64_t i = 1; i <= total; i++) {
    const uint32_t r = find((uint32_t)i);
    if (r == i) lut[i] = ++next;  // roots are minima: met before their members
    else lut[i] = lut[r];
  }
  *n_global = next;
  return IGN_OK;
}

int ign_ccl6_volume_abort(ign_ccl_volume* v) {
  if (!v) return IGN_OK;
  Scratch held(v->ctx, v->base);  // releases the volume's bytes on return
  delete v;
  return IGN_OK;
}

int ign_ccl6_volume_begin_dev(ign_ctx* ctx, const void* in, int in_dtype, uint64_t sx, uint64_t sy,
                              uint64_t sz, uint64_t* first_values, uint32_t* first_labels,
                              uint64_t* last_values, uint32_t* last_labels, ign_ccl_volume** out,
                              uint64_t* n_local) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(in && out && n_local, IGN_ERR_INVALID, "null argument");
  *out = nullptr;
  IGN_TRY(check_ccl_dims(sx, sy, sz));
  Scratch sc(ctx);
  IGN_REQUIRE(sc.owner(), IGN_ERR_INVALID, "volume CCL must own the scratch arena");
  std::unique_ptr<ign_ccl_volume> v(new ign_ccl_volume());
  v->ctx = ctx;
  v->in = in;
  v->in_dtype = in_dtype;
  switch (in_dtype) {
    case IGN_U8: IGN_TRY(volume_begin_typed<uint8_t>(ctx, sc, v.get(), sx, sy, sz, first_values, first_labels, last_values, last_labels)); break;
    case IGN_U16: IGN_TRY(volume_begin_typed<uint16_t>(ctx, sc, v.get(), sx, sy, sz, first_values, first_labels, last_values, last_labels)); break;
    case IGN_U32: IGN_TRY(volume_begin_typed<uint32_t>(ctx, sc, v.get(), sx, sy, sz, first_values, first_labels, last_values, last_labels)); break;
    case IGN_U64: IGN_TRY(volume_begin_typed<uint64_t>(ctx, sc, v.get(), sx, sy, sz, first_values, first_labels, last_values, last_labels)); break;
    default: set_error("volume CCL: unsupported input dtype %d", in_dtype); return IGN_ERR_UNSUPPORTED;
  }
  // the arena stays held (the masks and run labels live in it) until finish / abort
  v->base = sc.keep();
  *n_local = v->n_local;
  *out = v.release();
  return IGN_OK;
}

// global_lut: NULL, or HOST table [n_local+1] volume-local id -> final id (from the caller's
// cross-volume solve).  Expands the labels once and releases the arena.
int ign_ccl6_volume_finish_dev(ign_ccl_volume* v, const uint32_t* global_lut, uint64_t max_label,
                               void* out, int out_dtype) {
  IGN_REQUIRE(v && out, IGN_ERR_INVALID, "null argument");
  ign_ctx* ctx = v->ctx;
  IGN_TRY(activate(ctx));
  std::unique_ptr<ign_ccl_volume> done(v);
  Scratch sc(ctx, v->base);  // releases the volume's bytes on return
  CclPlan& p = v->plan;
  if (!global_lut) max_label = v->n_local;
  if (p.R == 0) {
    IGN_REQUIRE(dtype_size(out_dtype) > 0, IGN_ERR_UNSUPPORTED, "unsupported out dtype");
    IGN_CUDA(cudaMemsetAsync(out, 0, (uint64_t)p.sx * p.sy * p.sz * dtype_size(out_dtype), ctx->stream));
    return IGN_OK;
  }
  if (global_lut) {
    uint32_t* d_lut = sc.take<uint32_t>(v->n_local + 1);
    IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small for the relabel table (%llu components)",
                (unsigned long long)v->n_local);
    IGN_CUDA(cudaMemcpyAsync(d_lut, global_lut, (v->n_local + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
    IGN_LAUNCH(ctx, k_ccl_relabel_runs, blocks_for(p.R, 256), 256, 0, p.label, p.R, d_lut);
    IGN_CUDA(cudaStreamSynchronize(ctx->stream));  // the host table may be a temporary of the caller
  }
  return launch_expand(ctx, p, 0, out, out_dtype, max_label);
}

int ign_ccl6_volume_dev(ign_ctx* ctx, const void* in, int in_dtype, uint64_t sx, uint64_t sy,
                        uint64_t sz, void* out, int out_dtype, uint64_t* n_components) {
  IGN_REQUIRE(in && out, IGN_ERR_INVALID, "null buffer");
  ign_ccl_volume* v = nullptr;
  uint64_t n = 0;
  IGN_TRY(ign_ccl6_volume_begin_dev(ctx, in, in_dtype, sx, sy, sz, nullptr, nullptr, nullptr, nullptr, &v, &n));
  IGN_TRY(ign_ccl6_volume_finish_dev(v, nullptr, n, out, out_dtype));
  if (n_components) *n_components = n;
  return IGN_OK;
}


int ign_ccl6_sharded_dev(ign_group* g, const void* in, int in_dtype, uint64_t sx, uint64_t sy, uint64_t sz,
                         void* out, int out_dtype, uint64_t* n_global) {
  IGN_REQUIRE(g && in && out, IGN_ERR_INVALID, "null argument");
  ign_ctx* ctx = g->ctx;
  IGN_TRY(activate(ctx));
  IGN_TRY(check_ccl_dims(sx, sy, sz));
  IGN_REQUIRE(dtype_size(out_dtype) > 0, IGN_ERR_UNSUPPORTED, "unsupported out dtype");
  Scratch sc(ctx);
  IGN_REQUIRE(sc.owner(), IGN_ERR_INVALID, "sharded CCL must own the scratch arena");
  ign_ccl_volume v;
  v.ctx = ctx;
  v.in = in;
  v.in_dtype = in_dtype;
  switch (in_dtype) {
    case IGN_U8: return ccl_sharded_typed<uint8_t>(g, sc, &v, sx, sy, sz, out, out_dtype, n_global);
    case IGN_U16: return ccl_sharded_typed<uint16_t>(g, sc, &v, sx, sy, sz, out, out_dtype, n_global);
    case IGN_U32: return ccl_sharded_typed<uint32_t>(g, sc, &v, sx, sy, sz, out, out_dtype, n_global);
    case IGN_U64: return ccl_sharded_typed<uint64_t>(g, sc, &v, sx, sy, sz, out, out_dtype, n_global);
  }
  set_error("sharded CCL: unsupported input dtype %d", in_dtype);
  return IGN_ERR_UNSUPPORTED;
}

}  // extern "C"
