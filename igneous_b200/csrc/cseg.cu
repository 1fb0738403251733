// cseg.cu -- Precomputed `compressed_segmentation` chunk codec on the device
//
// SURVEY.md 8(f) row 1: the wire format either side of the hot path.  CloudVolume encodes /
// decodes it on the host around igneous/tasks/image/image.py:57-100 (every mip a
// DownsampleTask uploads) and igneous/tasks/image/ccl.py:346-356 (RelabelCCLTask's output;
// the CLI's default CCL encoding is compresso, `igneous_cli/cli.py:750`, with
// compressed_segmentation as the other segmentation codec).  Encoding where the labels
// already are shrinks the D2H of a label chunk by the compression ratio.
//
// Format (Neuroglancer): per channel [2 x u32 header per 8x8x8 block | per block: packed
// indices, then -- unless an identical table was already emitted by an earlier block of the
// channel -- the sorted lookup table]; header = (table offset : 24 | bits << 24), offset of the
// packed indices; bits in {0,1,2,4,8,16,32}; offsets in u32 words from the channel start.
// The emission order of oracle/igneous_oracle.c::orc_cseg_encode_* (block raster order, a
// table is emitted by the FIRST block that uses it) is reproduced exactly, so the streams are
// byte-identical:
//   1  k_cseg_scan<T, false>  one warp per block: the distinct values are extracted in
//      ascending order (repeated warp minimum) -> n, bits, 64-bit hash of the table
//   2  radix sort of (hash, block): blocks with equal tables are adjacent, in raster order
//   3  k_cseg_owner  one warp per block compares its table with the earlier blocks of its hash
//      group (first the group's head) -> owner = the first block in raster order with an EQUAL
//      table.  The hash only groups; blocks whose tables differ but hash alike never share.
//   4  exclusive scan of the per-block sizes -> offsets; the largest table offset is checked
//      against the format's 24-bit limit with the total, in the one host sync of the encoder
//   5  k_cseg_scan<T, true>   the same extraction again, now writing indices, tables, headers
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <vector>

#include "common.cuh"

namespace ign {

constexpr unsigned CS_FULL = 0xFFFFFFFFu;
constexpr int CS_MAX_BVOX = 1024;  // voxels per block (8x8x8 = 512 is the standard)

struct CsegDims {
  uint32_t sx, sy, sz, bx, by, bz, gx, gy, gz, bvox;
};

__device__ __forceinline__ uint64_t cs_shfl_xor(uint64_t v, int m) {
  return ((uint64_t)__shfl_xor_sync(CS_FULL, (uint32_t)(v >> 32), m) << 32) | __shfl_xor_sync(CS_FULL, (uint32_t)v, m);
}
__device__ __forceinline__ uint32_t cs_bits(uint32_t n) {
  if (n <= 1) return 0;
  uint32_t b = 1;
  while ((1u << b) < n) b *= 2;
  return b;
}

// Loads block b into a warp: lane l holds block positions l, l+32, ... (position
// p = (z*by + y)*bx + x).  Returns the slots inside the volume (bit k: slot k).
template <typename T, int CS_PER_LANE>
__device__ __forceinline__ uint32_t cs_load(const T* __restrict__ in, const CsegDims& d, uint64_t b, uint32_t lane,
                                            uint64_t (&val)[CS_PER_LANE]) {
  const uint32_t gxx = (uint32_t)(b % d.gx), gyy = (uint32_t)((b / d.gx) % d.gy), gzz = (uint32_t)(b / ((uint64_t)d.gx * d.gy));
  const uint32_t x0 = gxx * d.bx, y0 = gyy * d.by, z0 = gzz * d.bz;
  uint32_t have = 0;
#pragma unroll
  for (int k = 0; k < CS_PER_LANE; k++) {
    const uint32_t p = lane + 32 * k;
    val[k] = 0;
    if (p < d.bvox) {
      const uint32_t x = p % d.bx, y = (p / d.bx) % d.by, z = p / (d.bx * d.by);
      if (x0 + x < d.sx && y0 + y < d.sy && z0 + z < d.sz) {
        val[k] = (uint64_t)in[(x0 + x) + (uint64_t)d.sx * ((y0 + y) + (uint64_t)d.sy * (z0 + z))];
        have |= 1u << k;
      }
    }
  }
  return have;
}

// warp minimum of the values in the slots of `todo` (~0ull when no lane has any)
template <int CS_PER_LANE>
__device__ __forceinline__ uint64_t cs_warp_min(const uint64_t (&val)[CS_PER_LANE], uint32_t todo) {
  uint64_t m = ~0ull;
#pragma unroll
  for (int k = 0; k < CS_PER_LANE; k++)
    if ((todo >> k) & 1u) m = val[k] < m ? val[k] : m;
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    const uint64_t o = cs_shfl_xor(m, s);
    m = o < m ? o : m;
  }
  return m;
}

// One warp per block.  WRITE = false: info[b] = {n, bits}, hash[b].  WRITE = true: the stream.
template <typename T, bool WRITE, int CS_PER_LANE>  // CS_PER_LANE * 32 >= voxels per block
__global__ void __launch_bounds__(128)
    k_cseg_scan(const T* __restrict__ in, CsegDims d, uint64_t nblock, uint32_t* __restrict__ info_n,
                unsigned long long* __restrict__ hash, const uint32_t* __restrict__ enc_off,
                const uint32_t* __restrict__ tab_off, const uint32_t* __restrict__ owner, uint32_t* __restrict__ out) {
  constexpr int WORDS = sizeof(T) / 4;
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t b = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
  if (b >= nblock) return;
  uint64_t val[CS_PER_LANE];
  uint32_t idx[CS_PER_LANE];
  const uint32_t have = cs_load<T, CS_PER_LANE>(in, d, b, lane, val);  // bit k: slot k is inside the volume
  uint32_t todo = have;                                                 // bit k: slot k is not classified yet
#pragma unroll
  for (int k = 0; k < CS_PER_LANE; k++) idx[k] = 0;
  uint32_t n = 0;
  uint64_t h = 0x9E3779B97F4A7C15ull;
  const uint32_t toff = WRITE ? tab_off[b] : 0u;
  const bool own = WRITE ? (owner[b] == (uint32_t)b) : false;
  while (__any_sync(CS_FULL, todo != 0)) {
    const uint64_t m = cs_warp_min<CS_PER_LANE>(val, todo);
#pragma unroll
    for (int k = 0; k < CS_PER_LANE; k++)
      if (((todo >> k) & 1u) && val[k] == m) {
        idx[k] = n;
        todo &= ~(1u << k);
      }
    if (WRITE) {
      if (own && lane == 0) {
        out[toff + n * WORDS] = (uint32_t)m;
        if (WORDS == 2) out[toff + n * WORDS + 1] = (uint32_t)(m >> 32);
      }
    } else {
      h ^= m + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2);
    }
    n++;
  }
  const uint32_t bits = cs_bits(n);
  if (!WRITE) {
    if (lane == 0) {
      info_n[b] = n;
      hash[b] = (h ^ n) * 0xBF58476D1CE4E5B9ull;
    }
    return;
  }
  // ---- packed indices: word w of the block holds positions [w*32/bits, (w+1)*32/bits)
  const uint32_t eoff = enc_off[b];
  if (bits) {
    const uint32_t per = 32 / bits;             // values per word
    const uint32_t nwords = (bits * d.bvox + 31) / 32;
    // every lane contributes its values with atomicOr-free packing: values of one word sit in
    // `per` consecutive positions, i.e. in `per` consecutive lanes (or the same lane for per > 32)
#pragma unroll
    for (int k = 0; k < CS_PER_LANE; k++) {
      const uint32_t p = lane + 32 * k;
      if (32 * k >= d.bvox) break;
      const uint32_t v = ((have >> k) & 1u) ? idx[k] : 0u;
      uint32_t word = v << ((p % per) * bits);
      // OR-reduce over the aligned group of `per` lanes (per is a power of two <= 32)
      for (uint32_t s = 1; s < per; s <<= 1) word |= __shfl_xor_sync(CS_FULL, word, s);
      if (p < d.bvox && (p % per) == 0 && p / per < nwords) out[eoff + p / per] = word;
    }
  }
  if (lane == 0) {
    // header: blocks are in raster order at the start of the channel
    out[2 * b] = toff | (bits << 24);
    out[2 * b + 1] = eoff;
  }
}

__global__ void __launch_bounds__(256) k_iota32(uint32_t* p, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = i;
}

// Do blocks a and b have equal tables?  Both must hold the same number of distinct values: their
// ascending values are extracted in lock step (warp minimum) and compared, stopping at the first
// difference.  Warp-uniform: every lane of the warp calls it with the same a, b.
template <typename T, int CS_PER_LANE>
__device__ __forceinline__ bool cs_same_table(const T* __restrict__ in, const CsegDims& d, uint64_t a, uint64_t b,
                                              uint32_t lane) {
  uint64_t va[CS_PER_LANE], vb[CS_PER_LANE];
  uint32_t ta = cs_load<T, CS_PER_LANE>(in, d, a, lane, va);
  uint32_t tb = cs_load<T, CS_PER_LANE>(in, d, b, lane, vb);
  while (__any_sync(CS_FULL, ta != 0)) {
    const uint64_t ma = cs_warp_min<CS_PER_LANE>(va, ta), mb = cs_warp_min<CS_PER_LANE>(vb, tb);
    if (ma != mb) return false;
#pragma unroll
    for (int k = 0; k < CS_PER_LANE; k++) {
      if (((ta >> k) & 1u) && va[k] == ma) ta &= ~(1u << k);
      if (((tb >> k) & 1u) && vb[k] == mb) tb &= ~(1u << k);
    }
  }
  return true;
}

// sorted (hash, block): heads of the runs of equal hashes (the sort is stable and the blocks
// entered it in ascending order, so a run lists its blocks in raster order)
__global__ void __launch_bounds__(256)
    k_cseg_heads(const unsigned long long* __restrict__ shash, uint32_t n, uint32_t* __restrict__ headpos) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) headpos[i] = (i == 0 || shash[i - 1] != shash[i]) ? i : 0u;
}

// One warp per sorted position i (block sblock[i]; headpos: inclusive max-scan of the head
// positions).  Every block with a table equal to it sits in the same run, so the first block of
// the run with an equal table is the first in raster order: it owns the table.  Without a hash
// collision that is the head, one comparison; a run that mixes tables costs one comparison per
// distinct table before the block's own.
template <typename T, int CS_PER_LANE>
__global__ void __launch_bounds__(128)
    k_cseg_owner(const T* __restrict__ in, CsegDims d, const uint32_t* __restrict__ headpos,
                 const uint32_t* __restrict__ sblock, const uint32_t* __restrict__ n, uint32_t nblock,
                 uint32_t* __restrict__ owner) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t i = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
  if (i >= nblock) return;
  const uint32_t b = sblock[i];
  uint32_t o = b;
  for (uint32_t j = headpos[i]; j < i; j++) {
    const uint32_t c = sblock[j];
    if (n[c] == n[b] && cs_same_table<T, CS_PER_LANE>(in, d, c, b, lane)) {
      o = c;
      break;
    }
  }
  if (lane == 0) owner[b] = o;
}

template <int WORDS>
__global__ void __launch_bounds__(256)
    k_cseg_sizes(const uint32_t* __restrict__ n, const uint32_t* __restrict__ owner, uint32_t nblock, uint32_t bvox,
                 uint32_t* __restrict__ size) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nblock) return;
  const uint32_t bits = cs_bits(n[b]);
  size[b] = (bits * bvox + 31) / 32 + (owner[b] == b ? n[b] * WORDS : 0u);
}

// offsets from the channel start: indices at 2*nblock + scan[b]; own tables right after them.
// *max_toff = the largest table offset (the format stores it in 24 bits).
__global__ void __launch_bounds__(256)
    k_cseg_offsets(const uint32_t* __restrict__ n, const uint32_t* __restrict__ owner, const uint32_t* __restrict__ scan,
                   uint32_t nblock, uint32_t bvox, uint32_t* __restrict__ enc_off, uint32_t* __restrict__ tab_off,
                   uint32_t* __restrict__ max_toff) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t t = 0;
  if (b < nblock) {
    enc_off[b] = 2 * nblock + scan[b];
    const uint32_t o = owner[b];
    const uint32_t obits = cs_bits(n[o]);
    t = 2 * nblock + scan[o] + (obits * bvox + 31) / 32;
    tab_off[b] = t;
  }
  t = __reduce_max_sync(CS_FULL, t);
  if ((threadIdx.x & 31u) == 0 && t != 0) atomicMax(max_toff, t);
}

template <typename T>
__global__ void __launch_bounds__(256)
    k_cseg_decode(const uint32_t* __restrict__ in, uint64_t nwords, CsegDims d, T* __restrict__ out, uint32_t* err) {
  constexpr int WORDS = sizeof(T) / 4;
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  const uint64_t n = (uint64_t)d.sx * d.sy * d.sz;
  if (i >= n) return;
  const uint32_t x = (uint32_t)(i % d.sx), y = (uint32_t)((i / d.sx) % d.sy), z = (uint32_t)(i / ((uint64_t)d.sx * d.sy));
  const uint64_t b = (x / d.bx) + (uint64_t)d.gx * ((y / d.by) + (uint64_t)d.gy * (z / d.bz));
  if (2 * b + 1 >= nwords) { *err = 1; return; }
  const uint32_t h0 = in[2 * b], h1 = in[2 * b + 1];
  const uint32_t bits = h0 >> 24;
  const uint64_t toff = h0 & 0xFFFFFFu, voff = h1;
  if (!(bits == 0 || bits == 1 || bits == 2 || bits == 4 || bits == 8 || bits == 16 || bits == 32)) { *err = 1; return; }
  uint64_t idx = 0;
  if (bits) {
    const uint64_t bitpos = (uint64_t)(((z % d.bz) * d.by + (y % d.by)) * d.bx + (x % d.bx)) * bits;
    const uint64_t w = voff + bitpos / 32;
    if (w >= nwords) { *err = 1; return; }
    idx = (in[w] >> (bitpos % 32)) & (bits == 32 ? 0xFFFFFFFFu : ((1u << bits) - 1u));
  }
  const uint64_t tw = toff + idx * WORDS;
  if (tw + WORDS > nwords) { *err = 1; return; }
  uint64_t v = in[tw];
  if (WORDS == 2) v |= (uint64_t)in[tw + 1] << 32;
  out[i] = (T)v;
}

static int cseg_dims(uint64_t sx, uint64_t sy, uint64_t sz, uint32_t bx, uint32_t by, uint32_t bz, CsegDims* d) {
  IGN_REQUIRE(sx && sy && sz && bx && by && bz, IGN_ERR_INVALID, "cseg: empty chunk or block");
  IGN_REQUIRE((uint64_t)bx * by * bz <= CS_MAX_BVOX, IGN_ERR_UNSUPPORTED, "cseg: blocks of more than %d voxels are not supported", CS_MAX_BVOX);
  IGN_REQUIRE(sx < (1u << 20) && sy < (1u << 20) && sz < (1u << 20), IGN_ERR_OVERFLOW, "cseg: chunk extent too large");
  d->sx = (uint32_t)sx; d->sy = (uint32_t)sy; d->sz = (uint32_t)sz;
  d->bx = bx; d->by = by; d->bz = bz;
  d->gx = (uint32_t)((sx + bx - 1) / bx); d->gy = (uint32_t)((sy + by - 1) / by); d->gz = (uint32_t)((sz + bz - 1) / bz);
  d->bvox = bx * by * bz;
  IGN_REQUIRE((uint64_t)d->gx * d->gy * d->gz < (1u << 23), IGN_ERR_OVERFLOW,
              "cseg: %llu blocks exceed the format's 24-bit table offsets; encode Precomputed chunks, not whole volumes",
              (unsigned long long)((uint64_t)d->gx * d->gy * d->gz));
  return IGN_OK;
}

// one channel; out_dev may be NULL (size query).  *n_words = words of the channel stream.
template <typename T>
static int cseg_encode_channel(ign_ctx* ctx, const T* in, const CsegDims& d, uint32_t* out_dev, uint64_t cap_words,
                               uint64_t* n_words) {
  constexpr int WORDS = sizeof(T) / 4;
  const uint32_t nb = d.gx * d.gy * d.gz;
  Scratch sc(ctx);
  size_t sortb = 0, scanb = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sortb, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                  (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)nb);
  cub::DeviceScan::ExclusiveSum(nullptr, scanb, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)nb + 1);
  {
    size_t mb = 0;
    cub::DeviceScan::InclusiveScan(nullptr, mb, (const uint32_t*)nullptr, (uint32_t*)nullptr, cub::Max(), (int)nb);
    if (mb > scanb) scanb = mb;
  }
  const size_t tmpb = (sortb > scanb ? sortb : scanb) + 256;
  IGN_TRY(sc.reserve(2 * align_up((size_t)nb * 8, 256) + 8 * align_up(((size_t)nb + 2) * 4, 256) + tmpb + 4096));
  unsigned long long* hash = sc.take<unsigned long long>(nb);
  unsigned long long* shash = sc.take<unsigned long long>(nb);
  uint32_t* n = sc.take<uint32_t>((size_t)nb + 1);
  uint32_t* blk = sc.take<uint32_t>((size_t)nb + 1);
  uint32_t* sblk = sc.take<uint32_t>((size_t)nb + 1);
  uint32_t* owner = sc.take<uint32_t>((size_t)nb + 1);
  uint32_t* size = sc.take<uint32_t>((size_t)nb + 1);
  uint32_t* scan = sc.take<uint32_t>((size_t)nb + 2);  // [nb]: total, [nb + 1]: largest table offset
  uint32_t* enc_off = sc.take<uint32_t>((size_t)nb + 1);
  uint32_t* tab_off = sc.take<uint32_t>((size_t)nb + 1);
  void* tmp = sc.take(tmpb);
  IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small (cseg encode)");
  const unsigned gw = blocks_for((uint64_t)nb * 32, 128);
  if (d.bvox <= 512)
    IGN_LAUNCH(ctx, (k_cseg_scan<T, false, 16>), gw, 128, 0, in, d, (uint64_t)nb, n, hash, (const uint32_t*)nullptr,
              (const uint32_t*)nullptr, (const uint32_t*)nullptr, (uint32_t*)nullptr);
  else
    IGN_LAUNCH(ctx, (k_cseg_scan<T, false, 32>), gw, 128, 0, in, d, (uint64_t)nb, n, hash, (const uint32_t*)nullptr,
              (const uint32_t*)nullptr, (const uint32_t*)nullptr, (uint32_t*)nullptr);
  IGN_LAUNCH(ctx, k_iota32, blocks_for(nb, 256), 256, 0, blk, nb);
  {
    size_t tb = tmpb;
    IGN_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tb, hash, shash, blk, sblk, (int)nb, 0, 64, ctx->stream));
    ctx->launches += 9;
  }
  IGN_LAUNCH(ctx, k_cseg_heads, blocks_for(nb, 256), 256, 0, shash, nb, enc_off);  // enc_off / tab_off: free until the offsets pass
  {
    size_t tb = tmpb;
    IGN_CUDA(cub::DeviceScan::InclusiveScan(tmp, tb, enc_off, tab_off, cub::Max(), (int)nb, ctx->stream));
    ctx->launches += 2;
  }
  if (d.bvox <= 512)
    IGN_LAUNCH(ctx, (k_cseg_owner<T, 16>), gw, 128, 0, in, d, tab_off, sblk, n, nb, owner);
  else
    IGN_LAUNCH(ctx, (k_cseg_owner<T, 32>), gw, 128, 0, in, d, tab_off, sblk, n, nb, owner);
  IGN_LAUNCH(ctx, (k_cseg_sizes<WORDS>), blocks_for(nb, 256), 256, 0, n, owner, nb, d.bvox, size);
  IGN_CUDA(cudaMemsetAsync(size + nb, 0, 4, ctx->stream));
  {
    size_t tb = tmpb;
    IGN_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, size, scan, (int)nb + 1, ctx->stream));
    ctx->launches += 2;
  }
  IGN_CUDA(cudaMemsetAsync(scan + nb + 1, 0, 4, ctx->stream));
  IGN_LAUNCH(ctx, k_cseg_offsets, blocks_for(nb, 256), 256, 0, n, owner, scan, nb, d.bvox, enc_off, tab_off, scan + nb + 1);
  uint32_t tail[2] = {0, 0};  // words after the headers, largest table offset
  IGN_TRY(small_d2h(ctx, tail, scan + nb, 8));
  IGN_TRY(small_sync(ctx));
  const uint64_t words = 2ull * nb + tail[0];
  *n_words = words;
  IGN_REQUIRE(tail[1] <= 0xFFFFFFu, IGN_ERR_OVERFLOW,
              "cseg: a lookup table of the encoded chunk starts at word %u, beyond the format's 24-bit table offsets",
              tail[1]);
  if (out_dev != nullptr && words <= cap_words) {
    if (d.bvox <= 512)
      IGN_LAUNCH(ctx, (k_cseg_scan<T, true, 16>), gw, 128, 0, in, d, (uint64_t)nb, (uint32_t*)nullptr, (unsigned long long*)nullptr,
                enc_off, tab_off, owner, out_dev);
    else
      IGN_LAUNCH(ctx, (k_cseg_scan<T, true, 32>), gw, 128, 0, in, d, (uint64_t)nb, (uint32_t*)nullptr, (unsigned long long*)nullptr,
                enc_off, tab_off, owner, out_dev);
  }
  return IGN_OK;
}

}  // namespace ign

using namespace ign;

extern "C" {

int ign_cseg_encode_dev(ign_ctx* ctx, const void* labels, int dtype, uint64_t sx, uint64_t sy, uint64_t sz,
                        uint64_t sc, uint32_t bx, uint32_t by, uint32_t bz, uint32_t* out, uint64_t cap_words,
                        uint64_t* n_words) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(labels && n_words && sc >= 1, IGN_ERR_INVALID, "null argument");
  IGN_REQUIRE(dtype == IGN_U32 || dtype == IGN_U64, IGN_ERR_UNSUPPORTED, "compressed_segmentation holds uint32 / uint64 labels");
  CsegDims d;
  IGN_TRY(cseg_dims(sx, sy, sz, bx, by, bz, &d));
  const uint64_t n = sx * sy * sz;
  uint64_t at = sc;  // the channel offset table comes first
  std::vector<uint32_t> chan_off(sc, 0);
  for (uint64_t c = 0; c < sc; c++) {
    chan_off[c] = (uint32_t)at;
    uint64_t w = 0;
    uint32_t* dst = (out && at < cap_words) ? out + at : nullptr;
    const uint64_t room = (out && at < cap_words) ? cap_words - at : 0;
    if (dtype == IGN_U32) IGN_TRY(cseg_encode_channel<uint32_t>(ctx, (const uint32_t*)labels + c * n, d, dst, room, &w));
    else IGN_TRY(cseg_encode_channel<uint64_t>(ctx, (const uint64_t*)labels + c * n, d, dst, room, &w));
    at += w;
  }
  *n_words = at;
  if (out && at <= cap_words) IGN_TRY(small_h2d(ctx, out, chan_off.data(), sc * 4));
  if (out) IGN_CUDA(cudaStreamSynchronize(ctx->stream));
  return IGN_OK;
}

int ign_cseg_decode_dev(ign_ctx* ctx, const uint32_t* in, uint64_t n_words, int dtype, uint64_t sx, uint64_t sy,
                        uint64_t sz, uint64_t sc, uint32_t bx, uint32_t by, uint32_t bz, void* out) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(in && out && sc >= 1 && n_words >= sc, IGN_ERR_INVALID, "bad argument");
  IGN_REQUIRE(dtype == IGN_U32 || dtype == IGN_U64, IGN_ERR_UNSUPPORTED, "compressed_segmentation holds uint32 / uint64 labels");
  CsegDims d;
  IGN_TRY(cseg_dims(sx, sy, sz, bx, by, bz, &d));
  const uint64_t n = sx * sy * sz;
  std::vector<uint32_t> chan_off(sc, 0);
  IGN_CUDA(cudaMemcpyAsync(chan_off.data(), in, sc * 4, cudaMemcpyDeviceToHost, ctx->stream));
  IGN_CUDA(cudaStreamSynchronize(ctx->stream));
  Scratch arena(ctx);  // `sc` is the channel count here
  IGN_TRY(arena.reserve(4096));
  uint32_t* err = arena.take<uint32_t>(64);
  IGN_REQUIRE(arena.ok(), IGN_ERR_NOMEM, "scratch arena too small (cseg decode)");
  IGN_CUDA(cudaMemsetAsync(err, 0, 4, ctx->stream));
  for (uint64_t c = 0; c < sc; c++) {
    const uint64_t base = chan_off[c];
    IGN_REQUIRE(base <= n_words, IGN_ERR_INVALID, "cseg: channel offset outside the stream");
    if (dtype == IGN_U32)
      IGN_LAUNCH(ctx, (k_cseg_decode<uint32_t>), blocks_for(n, 256), 256, 0, in + base, n_words - base, d, (uint32_t*)out + c * n, err);
    else
      IGN_LAUNCH(ctx, (k_cseg_decode<uint64_t>), blocks_for(n, 256), 256, 0, in + base, n_words - base, d, (uint64_t*)out + c * n, err);
  }
  uint32_t herr = 0;
  IGN_CUDA(cudaMemcpyAsync(&herr, err, 4, cudaMemcpyDeviceToHost, ctx->stream));
  IGN_CUDA(cudaStreamSynchronize(ctx->stream));
  IGN_REQUIRE(herr == 0, IGN_ERR_INVALID, "cseg: malformed stream");
  return IGN_OK;
}

// host-buffer wrappers: encode returns the words needed in *n_words (call with out == NULL first, or
// with a capacity of sc + 2*blocks + 3*voxels words, the worst case)
int ign_cseg_encode(ign_ctx* ctx, const void* labels, int dtype, uint64_t sx, uint64_t sy, uint64_t sz, uint64_t sc,
                    uint32_t bx, uint32_t by, uint32_t bz, uint32_t* out, uint64_t cap_words, uint64_t* n_words) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(labels && n_words, IGN_ERR_INVALID, "null argument");
  const int es = dtype_size(dtype);
  IGN_REQUIRE(dtype == IGN_U32 || dtype == IGN_U64, IGN_ERR_UNSUPPORTED, "compressed_segmentation holds uint32 / uint64 labels");
  Staging st(ctx);
  void *d_in, *d_out;
  st.add(&d_in, sx * sy * sz * sc * es, labels);
  st.add(&d_out, out ? cap_words * 4 : 0);
  IGN_TRY(st.stage());
  IGN_TRY(ign_cseg_encode_dev(ctx, d_in, dtype, sx, sy, sz, sc, bx, by, bz, (uint32_t*)d_out, cap_words, n_words));
  if (out && *n_words <= cap_words) IGN_TRY(st.back(out, d_out, *n_words * 4));
  return st.sync();
}

int ign_cseg_decode(ign_ctx* ctx, const uint32_t* in, uint64_t n_words, int dtype, uint64_t sx, uint64_t sy, uint64_t sz,
                    uint64_t sc, uint32_t bx, uint32_t by, uint32_t bz, void* out) {
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(in && out, IGN_ERR_INVALID, "null argument");
  const int es = dtype_size(dtype);
  IGN_REQUIRE(dtype == IGN_U32 || dtype == IGN_U64, IGN_ERR_UNSUPPORTED, "compressed_segmentation holds uint32 / uint64 labels");
  const uint64_t n = sx * sy * sz * sc;
  Staging st(ctx);
  void *d_in, *d_out;
  st.add(&d_in, n_words * 4, in);
  st.add(&d_out, n * es);
  IGN_TRY(st.stage());
  IGN_TRY(ign_cseg_decode_dev(ctx, (const uint32_t*)d_in, n_words, dtype, sx, sy, sz, sc, bx, by, bz, d_out));
  IGN_TRY(st.back(out, d_out, n * es));
  return st.sync();
}

}  // extern "C"
