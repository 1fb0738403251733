"""compressed_segmentation encoder on the inputs where table sharing and the 24-bit table offsets
go wrong: palettes that differ but may hash alike, every small palette at once, chunks at the
24-bit boundary, every bit width and blocks of more than 512 voxels.

Every chunk is checked three ways: the device stream equals the oracle's byte for byte, the
device decoder returns the input, and an independent numpy decoder of the published Neuroglancer
layout (below) returns the input from the device stream."""
import itertools

import numpy as np
import pytest

gpu = pytest.mark.gpu
DTYPES = [np.uint32, np.uint64]


# ------------------------------------------------------------------ independent decoder
def np_cseg_decode(words, shape, dtype, block_size=(8, 8, 8)):
  """Neuroglancer `compressed_segmentation`: [channel offsets | per channel: 2 x u32 header per
  block (table offset : 24 | bits << 24, index offset), packed indices, lookup tables]; blocks in
  x-fastest raster order, indices packed little-endian within u32 words, offsets in u32 words from
  the channel start.  Returns the [x, y, z, c] chunk (Fortran order)."""
  words = np.asarray(words, dtype=np.uint32)
  dtype = np.dtype(dtype)
  shape = tuple(int(s) for s in shape) + ((1,) if len(shape) == 3 else ())
  sx, sy, sz, sc = shape
  bx, by, bz = block_size
  gx, gy = -(-sx // bx), -(-sy // by)
  per = dtype.itemsize // 4
  w64 = words.astype(np.uint64)
  out = np.zeros(shape, dtype=dtype, order="F")
  x = np.arange(sx, dtype=np.uint64)[:, None, None]
  y = np.arange(sy, dtype=np.uint64)[None, :, None]
  for c in range(sc):
    base = int(words[c])
    for z0 in range(0, sz, bz):  # one layer of blocks at a time bounds the temporaries
      z = np.arange(z0, min(z0 + bz, sz), dtype=np.uint64)[None, None, :]
      blk = x // bx + gx * (y // by + gy * (z // bz))
      pos = ((z % bz) * by + y % by) * bx + x % bx
      h0 = w64[base + 2 * blk]
      h1 = w64[base + 2 * blk + 1]
      bits = h0 >> 24
      assert np.isin(bits, [0, 1, 2, 4, 8, 16, 32]).all()
      toff = base + (h0 & 0xFFFFFF)
      bitpos = pos * bits
      word = np.where(bits > 0, base + h1 + bitpos // 32, 0)
      idx = (w64[word] >> (bitpos % 32)) & ((np.uint64(1) << bits) - 1)
      val = w64[toff + idx * per]
      if per == 2:
        val |= w64[toff + idx * per + 1] << np.uint64(32)
      out[:, :, z0:z0 + bz, c] = val.astype(dtype)
  return out


def headers(words, nblock, channel=0):
  base = int(words[channel])
  h = np.asarray(words[base:base + 2 * nblock], dtype=np.uint32).reshape(nblock, 2)
  return h[:, 0] & 0xFFFFFF, h[:, 0] >> 24  # table offsets, bits


# ------------------------------------------------------------------ chunk builders
def palette_block(pal, bvox, rng):
  """One block holding exactly the values of `pal`, in shuffled positions."""
  pal = np.asarray(pal, dtype=np.uint64)
  assert 1 <= len(pal) <= bvox
  return rng.permutation(pal[np.arange(bvox) % len(pal)])


def distinct_values(rng, k, dtype):
  """k distinct values spread over the whole range of dtype."""
  hi = np.iinfo(dtype).max
  v = np.unique(rng.integers(0, hi, size=2 * k + 16, dtype=np.uint64, endpoint=True))
  return rng.permutation(v)[:k]


def chunk_from_blocks(blocks, grid, dtype, block_size=(8, 8, 8)):
  """blocks: [nblock, bvox] values, block b at raster position b of `grid` (x fastest), voxel p of
  a block at p = (z * by + y) * bx + x.  Missing trailing blocks repeat the first block."""
  gx, gy, gz = grid
  bx, by, bz = block_size
  blocks = np.asarray(blocks)
  nb = gx * gy * gz
  assert blocks.shape[0] <= nb and blocks.shape[1] == bx * by * bz
  if blocks.shape[0] < nb:
    blocks = np.concatenate([blocks, np.repeat(blocks[:1], nb - blocks.shape[0], axis=0)])
  v = blocks.astype(dtype).reshape(gz, gy, gx, bz, by, bx).transpose(2, 5, 1, 4, 0, 3)
  return np.asfortranarray(v.reshape(gx * bx, gy * by, gz * bz))


def check(oracle, vol, block_size=(8, 8, 8)):
  """device stream == oracle stream; device and numpy decoders both return the input."""
  from igneous_b200 import codecs
  got = np.frombuffer(codecs.cseg_encode(vol, block_size), dtype=np.uint32)
  want = oracle.cseg_encode(vol, block_size)
  assert len(got) == len(want)
  assert np.array_equal(got, want)
  v4 = vol if vol.ndim == 4 else vol[..., np.newaxis]
  assert np.array_equal(codecs.cseg_decode(got.tobytes(), vol.shape, vol.dtype, block_size), v4)
  assert np.array_equal(np_cseg_decode(got, vol.shape, vol.dtype, block_size), v4)
  return got


# Palette pairs that differ but hash alike under the encoder's 64-bit table hash (k_cseg_scan), the
# key that groups blocks before their tables are compared.  The census below does not rely on it.
COLLIDING = [
  ((0, 1), (1, 64)),
  ((11, 12), (32, 50)),
  ((2, 10, 11), (2, 23, 63)),
]


# ------------------------------------------------------------------ CPU: the decoder itself
@pytest.mark.parametrize("dtype", DTYPES)
def test_numpy_decoder_matches_oracle_decoder(oracle, dtype):
  rng = np.random.default_rng(11)
  hi = (1 << 40) if dtype == np.uint64 else (1 << 31)
  vols = [
    (rng.integers(0, 5, size=(21, 13, 10, 2)).astype(dtype), (8, 8, 8)),
    (rng.integers(0, hi, size=(16, 8, 9), dtype=np.uint64).astype(dtype), (8, 8, 8)),
    ((rng.integers(0, 300, size=(19, 17, 16)) * 7919).astype(dtype), (16, 8, 8)),
    (rng.integers(0, 3, size=(9, 9, 9)).astype(dtype), (4, 2, 8)),
    (np.zeros((8, 8, 8), dtype=dtype), (8, 8, 8)),
  ]
  for vol, bs in vols:
    vol = np.asfortranarray(vol)
    words = oracle.cseg_encode(vol, bs)
    want = oracle.cseg_decode(words, vol.shape, dtype, bs)
    assert np.array_equal(np_cseg_decode(words, vol.shape, dtype, bs), want)
    assert np.array_equal(want[..., 0] if vol.ndim == 3 else want, vol)


# ------------------------------------------------------------------ GPU: table sharing
@gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("pair", COLLIDING, ids=lambda p: "%s_%s" % p)
def test_colliding_palettes_keep_their_own_tables(ctx, oracle, dtype, pair):
  rng = np.random.default_rng(12)
  a, b = pair
  # A then B: two tables
  vol = chunk_from_blocks([palette_block(a, 512, rng), palette_block(b, 512, rng)], (2, 1, 1), dtype)
  got = check(oracle, vol)
  toff, _ = headers(got, 2)
  assert toff[0] != toff[1]
  # A, B, A, B (and B, A, B, A): within one hash group the first block with an equal table owns it
  for first, second in ((a, b), (b, a)):
    blocks = [palette_block(p, 512, rng) for p in (first, second, first, second)]
    got = check(oracle, chunk_from_blocks(blocks, (2, 2, 1), dtype))
    toff, _ = headers(got, 4)
    assert toff[2] == toff[0] and toff[3] == toff[1] and toff[0] != toff[1]


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_colliding_palettes_in_different_channels(ctx, oracle, dtype):
  rng = np.random.default_rng(13)
  (a, b), (c, d) = COLLIDING[0], COLLIDING[2]
  ch0 = chunk_from_blocks([palette_block(p, 512, rng) for p in (a, b, c, a)], (2, 2, 1), dtype)
  ch1 = chunk_from_blocks([palette_block(p, 512, rng) for p in (b, a, d, c)], (2, 2, 1), dtype)
  ch2 = chunk_from_blocks([palette_block(p, 512, rng) for p in (b, b, d, d)], (2, 2, 1), dtype)
  vol = np.asfortranarray(np.stack([ch0, ch1, ch2], axis=3))
  check(oracle, vol)


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_palette_census(ctx, oracle, dtype):
  """One block per palette: every 2-subset of 0..63 and of 0..129, every 3-subset of 0..39, then
  the same palettes again in shuffled order.  Any two palettes a table hash confuses are in here."""
  rng = np.random.default_rng(14)
  sets = [
    list(itertools.combinations(range(64), 2)),
    list(itertools.combinations(range(130), 2)),
    list(itertools.combinations(range(40), 3)),
  ]
  for pals in sets:
    n = len(pals)
    order = np.concatenate([np.arange(n), rng.permutation(n)])
    idx = np.arange(512)
    blocks = np.empty((2 * n, 512), dtype=np.uint64)
    for i, p in enumerate(order):
      pal = np.asarray(pals[p], dtype=np.uint64)
      blocks[i] = pal[rng.permutation(idx) % len(pal)]
    gz = -(-2 * n // 256)
    check(oracle, chunk_from_blocks(blocks, (16, 16, gz), dtype))


# ------------------------------------------------------------------ GPU: 24-bit table offsets
def _distinct_blocks(m):
  """m blocks of 512 distinct values each (16-bit indices + a 512-entry table: 768 u32 words),
  no value shared between blocks and none equal to 0."""
  return 1 + np.arange(m * 512, dtype=np.uint64).reshape(m, 512)[:, ::-1]


def _boundary_chunk(zero_blocks, grid):
  # 2 * nblock header words + 21788 * 768 words of distinct blocks; then the zero blocks (0-bit
  # indices, one shared 1-word table) and a last block holding a new constant (another 1-word table)
  m = 21788
  blocks = np.concatenate([_distinct_blocks(m), np.zeros((zero_blocks, 512), np.uint64),
                           np.full((1, 512), 0xFFFFFFF0, np.uint64)])
  assert blocks.shape[0] == np.prod(grid)
  return chunk_from_blocks(blocks, grid, np.uint32), blocks.shape[0]


@gpu
def test_last_table_at_offset_2_24_minus_1_is_accepted(ctx, oracle):
  vol, nb = _boundary_chunk(226, (35, 17, 37))
  got = check(oracle, vol)
  toff, bits = headers(got, nb)
  assert toff[-1] == (1 << 24) - 1 and bits[-1] == 0 and toff[-2] == (1 << 24) - 2


@gpu
def test_table_offset_beyond_24_bits_is_refused(ctx, oracle):
  from igneous_b200 import _shim, codecs
  # the zero blocks' table starts at word 2^24, the constant's at 2^24 + 1: 2^24 + 2 words in all
  vol, _ = _boundary_chunk(227, (16, 16, 86))
  with pytest.raises(AssertionError):
    oracle.cseg_encode(vol)  # the oracle encoder returns an error status
  with pytest.raises(_shim.IgneousB200Error):
    codecs.cseg_encode(vol)


@gpu
def test_long_stream_with_early_tables_is_accepted(ctx, oracle):
  """One 512-value table first, then 65099 blocks holding permutations of it: every table offset
  is small, but the stream (2^24 + 18k words) is longer than 2^24 words."""
  rng = np.random.default_rng(15)
  nb = 30 * 35 * 62
  pal = _distinct_blocks(1)[0].astype(np.uint32)
  perms = np.argsort(rng.random((509, 512)), axis=1)  # 509 permutations, cycled
  blocks = pal[perms[np.arange(nb) % len(perms)]]
  got = check(oracle, chunk_from_blocks(blocks, (30, 35, 62), np.uint32))
  assert len(got) > (1 << 24) + 1024
  toff, bits = headers(got, nb)
  assert (toff == toff[0]).all() and (bits == 16).all()


# ------------------------------------------------------------------ GPU: bit widths, block shapes
@gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_every_bit_width(ctx, oracle, dtype):
  rng = np.random.default_rng(16)
  sizes = [1, 2, 3, 4, 5, 16, 17, 256, 257, 512]
  blocks = [palette_block(distinct_values(rng, k, dtype), 512, rng) for k in sizes]
  blocks += [palette_block(np.arange(k), 512, rng) for k in sizes]  # small ids, 0 included
  got = check(oracle, chunk_from_blocks(blocks, (5, 2, 2), dtype))
  _, bits = headers(got, 20)
  assert list(bits[:10]) == [0, 1, 2, 2, 4, 4, 8, 8, 16, 16]


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("bs", [(16, 8, 8), (8, 8, 16), (8, 16, 8)])
def test_blocks_of_1024_voxels(ctx, oracle, dtype, bs):
  rng = np.random.default_rng(17)
  sizes = [1, 2, 3, 17, 257, 512, 513, 1000, 1024]
  blocks = [palette_block(distinct_values(rng, k, dtype), 1024, rng) for k in sizes]
  blocks += [palette_block(p, 1024, rng) for pair in COLLIDING for p in pair]
  blocks += [palette_block(p, 1024, rng) for p in COLLIDING[0]]  # repeats share
  got = check(oracle, chunk_from_blocks(blocks, (3, 3, 2), dtype, bs), bs)
  _, bits = headers(got, 18)
  assert list(bits[:9]) == [0, 1, 2, 8, 16, 16, 16, 16, 16]


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("bs", [(8, 8, 8), (16, 8, 8), (4, 4, 4)])
def test_ragged_edge_blocks_with_small_palettes(ctx, oracle, dtype, bs):
  """Every block holds a random 2-subset of 0..129 (checkerboard), in a chunk whose edge blocks
  are cut short along every axis; the cut blocks hold fewer voxels but the same 2 values."""
  rng = np.random.default_rng(18)
  shape = (bs[0] * 7 + 3, bs[1] * 5 + 5, bs[2] * 4 + 1)
  g = [-(-s // b) for s, b in zip(shape, bs)]
  pairs = np.array(list(itertools.combinations(range(130), 2)), dtype=np.uint64)
  pal = pairs[rng.integers(0, len(pairs), size=g)]
  x, y, z = np.meshgrid(*[np.arange(s) for s in shape], indexing="ij")
  vol = pal[x // bs[0], y // bs[1], z // bs[2], (x + y + z) % 2]
  check(oracle, np.asfortranarray(vol.astype(dtype)), bs)
