"""fastremap-equivalent kernels (one open-addressing hash table behind renumber, remap, unique,
mask, mask_except) on the labels where such a table goes wrong: the all-ones label (the table's
empty-slot marker), 0 and the top bit, each dtype's largest value, label counts that make the table
grow, output dtype edges and counting runs that straddle warps.  Every check is against numpy or a
Python dict."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

U64MAX = (1 << 64) - 1
SPECIAL = [0, 1, 1 << 63, U64MAX - 1, U64MAX]


# ------------------------------------------------------------------ plain references
def ref_renumber(arr):
  """fastremap.renumber: 1..K in order of first appearance in memory order, 0 kept; output dtype
  the smallest unsigned type holding K."""
  order = "F" if (arr.flags.f_contiguous and not arr.flags.c_contiguous) else "C"
  flat = arr.ravel(order=order)
  uniq, first = np.unique(flat, return_index=True)
  nz = uniq != 0
  uniq, first = uniq[nz], first[nz]
  by_first = np.argsort(first, kind="stable")
  ids = np.zeros(len(uniq), dtype=np.uint64)
  ids[by_first] = np.arange(1, len(uniq) + 1, dtype=np.uint64)
  mapping = {int(u): int(i) for u, i in zip(uniq, ids)}
  if (flat == 0).any():
    mapping[0] = 0
  k = len(uniq)
  dt = next(np.dtype(d) for d in (np.uint8, np.uint16, np.uint32, np.uint64) if k <= np.iinfo(d).max)
  out = np.zeros(flat.shape, dtype=np.uint64)
  out[flat != 0] = ids[np.searchsorted(uniq, flat[flat != 0])]
  return out.astype(dt).reshape(arr.shape, order=order), mapping


def ref_remap(arr, table, preserve):
  flat = [int(v) for v in arr.ravel(order="K")]
  out = [table.get(v, v) if preserve else table[v] for v in flat]
  return np.array(out, dtype=arr.dtype).reshape(arr.shape, order="F" if arr.flags.f_contiguous else "C")


def ref_mask(arr, labels, except_, value=0):
  hit = np.isin(arr, np.array(list(labels), dtype=arr.dtype))
  out = arr.copy(order="K")
  out[~hit if except_ else hit] = value
  return out


def special_volume(rng, dtype, shape=(37, 21, 11), extra=()):
  top = int(np.iinfo(dtype).max)
  vals = sorted({v & top for v in SPECIAL} | set(extra))
  vals = np.array(vals, dtype=np.uint64).astype(dtype)
  return np.asfortranarray(vals[rng.integers(0, len(vals), size=shape)]), [int(v) for v in vals]


# ------------------------------------------------------------------ special values
def test_all_ones_u64_through_every_function(ctx):
  from igneous_b200 import fastremap
  rng = np.random.default_rng(21)
  arr, vals = special_volume(rng, np.uint64, extra=(7, 1 << 40))
  # renumber: mapping and dtype; 2^64-1 is a label like any other
  got, gmap = fastremap.renumber(arr)
  want, wmap = ref_renumber(arr)
  assert gmap == wmap and got.dtype == want.dtype and np.array_equal(got, want)
  assert U64MAX in gmap
  # unique with counts
  u, c = fastremap.unique(arr, return_counts=True)
  wu, wc = np.unique(arr, return_counts=True)
  assert np.array_equal(u, wu) and np.array_equal(c, wc.astype(np.uint64))
  assert int(u[-1]) == U64MAX
  # remap: every key present, values include 2^64-1 and 0
  table = {v: (U64MAX if v == 7 else (v * 3 + 5) % (1 << 64)) for v in vals}
  assert np.array_equal(fastremap.remap(arr, table), ref_remap(arr, table, False))
  # a table holding 2^64-1 as a key only: the array value 2^64-1 is mapped, not zeroed
  swap = {U64MAX: 12345, 12345: U64MAX}
  for v in vals:
    swap.setdefault(v, v)
  assert np.array_equal(fastremap.remap(arr, swap), ref_remap(arr, swap, False))


@pytest.mark.parametrize("missing", [(U64MAX,), (0, U64MAX), (1 << 63,), (U64MAX - 1, U64MAX)])
def test_remap_missing_labels(ctx, missing):
  from igneous_b200 import fastremap
  rng = np.random.default_rng(22)
  arr, vals = special_volume(rng, np.uint64, extra=(99,))
  table = {v: v + 1000 for v in vals if v not in missing and v < U64MAX - 1000}
  table.update({v: 17 for v in vals if v not in missing and v >= U64MAX - 1000})
  table[(1 << 62) + 3] = 4  # a key the array lacks
  with pytest.raises(KeyError) as e:
    fastremap.remap(arr, table)
  assert int(e.value.args[0]) in missing  # names a label that really is missing
  kept = fastremap.remap(arr, table, preserve_missing_labels=True)
  assert np.array_equal(kept, ref_remap(arr, table, True))
  for v in missing:
    assert (kept == np.uint64(v)).sum() == (arr == np.uint64(v)).sum()


@pytest.mark.parametrize("labels", [[], [U64MAX], [0, U64MAX], [1 << 63, U64MAX - 1], [5, 6], SPECIAL])
def test_mask_and_mask_except_special(ctx, labels):
  from igneous_b200 import fastremap
  rng = np.random.default_rng(23)
  arr, _ = special_volume(rng, np.uint64, extra=(5,))
  assert np.array_equal(fastremap.mask(arr, labels), ref_mask(arr, labels, False))
  assert np.array_equal(fastremap.mask_except(arr, labels), ref_mask(arr, labels, True))
  assert np.array_equal(fastremap.mask(arr, labels, value=U64MAX), ref_mask(arr, labels, False, U64MAX))
  assert np.array_equal(fastremap.mask_except(arr, labels, value=9), ref_mask(arr, labels, True, 9))


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.uint32])
def test_all_ones_of_narrow_dtypes(ctx, dtype):
  from igneous_b200 import fastremap
  rng = np.random.default_rng(24)
  top = int(np.iinfo(dtype).max)
  arr, vals = special_volume(rng, dtype, extra=(3, top - 2))
  got, gmap = fastremap.renumber(arr)
  want, wmap = ref_renumber(arr)
  assert gmap == wmap and got.dtype == want.dtype and np.array_equal(got, want)
  u, c = fastremap.unique(arr, return_counts=True)
  wu, wc = np.unique(arr, return_counts=True)
  assert u.dtype == arr.dtype and np.array_equal(u, wu) and np.array_equal(c, wc.astype(np.uint64))
  table = {v: top - v for v in vals}
  assert np.array_equal(fastremap.remap(arr, table), ref_remap(arr, table, False))
  del table[top]
  with pytest.raises(KeyError) as e:
    fastremap.remap(arr, table)
  assert int(e.value.args[0]) == top
  assert np.array_equal(fastremap.remap(arr, table, preserve_missing_labels=True), ref_remap(arr, table, True))
  for labels in ([top], [0, top], []):
    assert np.array_equal(fastremap.mask(arr, labels), ref_mask(arr, labels, False))
    assert np.array_equal(fastremap.mask_except(arr, labels), ref_mask(arr, labels, True))


def test_mesher_label_all_ones(ctx, oracle):
  from igneous_b200 import zmesh
  data = np.zeros((20, 18, 16), dtype=np.uint64, order="F")
  data[2:12, 3:15, 2:10] = U64MAX
  data[10:18, 5:13, 6:14] = 1 << 63
  data[4:8, 4:8, 11:15] = U64MAX - 1
  m = zmesh.Mesher((4.0, 4.0, 40.0))
  m.mesh(data)
  tl, tv = oracle.marching_cubes(data)
  want_ids = sorted(int(i) for i in np.unique(tl))
  assert U64MAX in want_ids and sorted(m.ids()) == want_ids
  for lab in want_ids:
    got = m.get(lab, reduction_factor=0, voxel_centered=True)
    wv, wf = oracle.mesh_for_label(tl, tv, lab, resolution=(4.0, 4.0, 40.0), voxel_centered=True)
    assert np.array_equal(got.vertices, wv) and np.array_equal(got.faces, wf)


# ------------------------------------------------------------------ table growth
def _growth_volume(rng, distinct, n=1 << 21):
  """n voxels holding exactly `distinct` labels (0 and 2^64-1 among them), every label at least
  once, in shuffled positions (few runs, so nearly every voxel probes the table)."""
  labels = np.unique(rng.integers(1, U64MAX - 1, size=distinct + distinct // 8 + 64, dtype=np.uint64))
  labels = rng.permutation(labels)[:distinct]
  labels[0], labels[1] = 0, U64MAX
  assert len(np.unique(labels)) == distinct
  flat = np.concatenate([labels, labels[rng.integers(0, distinct, size=n - distinct)]])
  return np.asfortranarray(rng.permutation(flat).reshape(128, 128, n // (128 * 128)))


@pytest.mark.parametrize("distinct", [1 << 19, (1 << 19) + 1, 600_000, 1 << 21],
                         ids=["2^19", "2^19+1", "600k", "all_distinct"])
def test_renumber_and_unique_table_growth(ctx, distinct):
  from igneous_b200 import fastremap
  rng = np.random.default_rng(25)
  arr = _growth_volume(rng, distinct)
  flat = arr.ravel(order="F")
  wu, wfirst, wc = np.unique(flat, return_index=True, return_counts=True)
  assert len(wu) == distinct
  u, c = fastremap.unique(arr, return_counts=True)
  assert np.array_equal(u, wu) and np.array_equal(c, wc.astype(np.uint64))
  got, gmap = fastremap.renumber(arr)
  assert got.dtype == np.uint32 and len(gmap) == distinct
  # ids follow first appearance; 0 stays 0
  nz = wu != 0
  rank = np.empty(nz.sum(), dtype=np.int64)
  rank[np.argsort(wfirst[nz], kind="stable")] = np.arange(1, nz.sum() + 1)
  want_ids = np.zeros(len(wu), dtype=np.int64)
  want_ids[nz] = rank
  assert gmap == {int(k): int(v) for k, v in zip(wu, want_ids)}
  assert np.array_equal(got.ravel(order="F"), want_ids[np.searchsorted(wu, flat)].astype(np.uint32))


@pytest.mark.parametrize("k,dtype", [(255, np.uint8), (256, np.uint16), (65535, np.uint16), (65536, np.uint32)])
def test_renumber_output_dtype_edges(ctx, k, dtype):
  from igneous_b200 import fastremap
  rng = np.random.default_rng(26)
  labels = rng.permutation(np.unique(rng.integers(1, U64MAX, size=k + 64, dtype=np.uint64, endpoint=True)))[:k]
  labels[-1] = U64MAX
  flat = np.concatenate([labels, np.zeros(k // 3 + 5, np.uint64), labels[rng.integers(0, k, size=k)]])
  arr = np.asfortranarray(rng.permutation(flat))
  got, gmap = fastremap.renumber(arr)
  want, wmap = ref_renumber(arr)
  assert got.dtype == np.dtype(dtype) == want.dtype
  assert gmap == wmap and np.array_equal(got, want)


# ------------------------------------------------------------------ unique counts
@pytest.mark.parametrize("dtype", [np.uint8, np.uint32, np.uint64])
def test_unique_runs_across_warp_boundaries(ctx, dtype):
  from igneous_b200 import fastremap
  rng = np.random.default_rng(27)
  top = int(np.iinfo(dtype).max)
  vals = np.array([0, 1, 2, top - 1, top], dtype=np.uint64).astype(dtype)
  lengths = rng.choice([1, 2, 31, 32, 33, 63, 64, 65, 255, 256, 257], size=4000)
  lengths[:6] = [31, 32, 33, 32, 31, 33]  # head runs end just before, at and after a warp edge
  seq = vals[rng.integers(0, len(vals), size=len(lengths))]
  arr = np.repeat(seq, lengths)
  for a in (arr, arr[7:], arr[:-13]):  # shift the runs against the warps
    u, c = fastremap.unique(a, return_counts=True)
    wu, wc = np.unique(a, return_counts=True)
    assert np.array_equal(u, wu) and np.array_equal(c, wc.astype(np.uint64))


@pytest.mark.parametrize("dtype", [np.uint32, np.uint64])
def test_unique_single_value_over_2_24_voxels(ctx, dtype):
  from igneous_b200 import fastremap
  top = np.iinfo(dtype).max
  n = (1 << 24) + 77
  arr = np.full(n, top, dtype=dtype)
  arr[5] = 0
  arr[-40:-20] = 3
  u, c = fastremap.unique(arr, return_counts=True)
  assert list(u) == [0, 3, top] and list(c) == [1, 20, n - 21]
