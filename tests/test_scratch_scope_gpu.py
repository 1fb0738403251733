"""The scratch arena of one context across failed calls and an open CCL volume.

Every entry point gives back the arena bytes it took on every return path, errors included, so a
failed call leaves the context fully usable.  Host-buffer calls stage their arrays outside the
arena, so one made while a CCL volume holds the arena does not touch the volume's masks and runs."""
import ctypes as c

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RES = (16, 16, 40)


def _blobs(shape, seed):
  rng = np.random.default_rng(seed)
  small = rng.integers(0, 4, size=tuple((s + 3) // 4 for s in shape))
  big = np.repeat(np.repeat(np.repeat(small, 4, 0), 4, 1), 4, 2)[:shape[0], :shape[1], :shape[2]]
  return np.asfortranarray(np.where(rng.random(shape) < 0.2, 0, big).astype(np.uint32))


def _u64(*v):
  return [c.c_uint64(int(x)) for x in v]


# ------------------------------------------------------------------ argument-triggered failures
def _remap_missing_key(ctx):
  from igneous_b200 import _shim
  arr = np.array([1, 2, 3, 2], dtype=np.uint32)
  keys, vals = np.array([1, 2], np.uint64), np.array([5, 6], np.uint64)
  d = ctx.to_device(arr)
  try:
    with pytest.raises(KeyError):
      _shim.check(ctx.lib.ign_remap_dev(ctx.handle, _shim.ptr(d), c.c_int(_shim.IGN_U32), c.c_uint64(arr.size),
                                        _shim.ptr(keys), _shim.ptr(vals), c.c_uint64(keys.size), c.c_int(0)))
  finally:
    d.free()


def _ccl_u16_overflow(ctx):
  from igneous_b200 import _shim
  shape = (128, 64, 64)
  vol = np.zeros(shape, dtype=np.uint8, order="F")
  vol[::2, ::2, ::2] = 1  # 64 * 32 * 32 = 65536 isolated voxels: one more component than uint16 holds
  d_in, d_out = ctx.to_device(vol), ctx.alloc(vol.size * 2)
  n = c.c_uint64(0)
  try:
    with pytest.raises(_shim.IgneousB200Error):
      _shim.check(ctx.lib.ign_ccl6_dev(ctx.handle, _shim.ptr(d_in), c.c_int(_shim.IGN_U8), *_u64(*shape),
                                       _shim.ptr(d_out), c.c_int(_shim.IGN_U16), c.byref(n)))
  finally:
    d_in.free()
    d_out.free()


def _cseg_offset_beyond_24_bits(ctx):
  from igneous_b200 import _shim, codecs
  from test_cseg_edges_gpu import _boundary_chunk
  vol, _ = _boundary_chunk(227, (16, 16, 86))
  with pytest.raises(_shim.IgneousB200Error):
    codecs.cseg_encode(vol)


def _mesh_get_other_factor(ctx):
  from igneous_b200 import _shim, zmesh
  m = zmesh.Mesher(RES)
  m.mesh(_blobs((24, 20, 18), 3))
  label = m.ids()[0]
  m.get(label, reduction_factor=4, max_error=40)
  res = (c.c_float * 3)(*[float(r) for r in RES])
  nv, nf = c.c_uint64(0), c.c_uint64(0)
  with pytest.raises(_shim.IgneousB200Error):
    _shim.check(ctx.lib.ign_mesh_get(m._handle, c.c_uint64(label), res, c.c_int(5), c.c_float(40.0), c.c_int(0),
                                     None, None, c.byref(nv), c.byref(nf)))


FAILURES = {
  "remap_dev_missing_key": _remap_missing_key,
  "ccl6_dev_u16_overflow": _ccl_u16_overflow,
  "cseg_encode_offset_beyond_24_bits": _cseg_offset_beyond_24_bits,
  "mesh_get_other_reduction_factor": _mesh_get_other_factor,
}


# ------------------------------------------------------------------ the context still works
def _volume_ccl(ctx, labels):
  from igneous_b200 import _shim
  d_in, d_out = ctx.to_device(labels), ctx.alloc(labels.size * 4)
  n = c.c_uint64(0)
  try:
    _shim.check(ctx.lib.ign_ccl6_volume_dev(ctx.handle, _shim.ptr(d_in), c.c_int(_shim.dtype_code(labels.dtype)),
                                            *_u64(*labels.shape), _shim.ptr(d_out), c.c_int(_shim.IGN_U32),
                                            c.byref(n)))
    return ctx.to_host(d_out, labels.shape, np.uint32), n.value
  finally:
    d_in.free()
    d_out.free()


@pytest.fixture(scope="module")
def mesh_case(oracle):
  seg = oracle.synth_seg((41, 37, 33), pitch=16, num_ids=1 << 20)
  tl, tv = oracle.marching_cubes(seg)
  want, _ = oracle.simplify_welded(oracle.WeldedMeshes(tl, tv), RES, 4, 40.0, True)
  return seg, want


def _check_usable(ctx, oracle, mesh_case):
  from igneous_b200 import zmesh
  labels = _blobs((70, 65, 9), 21)
  want, n_want = oracle.connected_components(labels, return_N=True)
  got, n = _volume_ccl(ctx, labels)
  assert n == n_want and np.array_equal(got, want.astype(np.uint32))
  seg, meshes = mesh_case
  m = zmesh.Mesher(RES)
  m.mesh(seg)
  assert sorted(m.ids()) == sorted(meshes.keys())
  for lab in m.ids():
    g = m.get(lab, reduction_factor=4, max_error=40.0, voxel_centered=True)  # ign_mesh_simplify
    wv, wf = meshes[lab]
    assert np.array_equal(g.vertices, wv) and np.array_equal(g.faces, wf), lab


@pytest.mark.parametrize("failure", list(FAILURES))
def test_failed_call_leaves_the_context_usable(ctx, oracle, mesh_case, failure):
  FAILURES[failure](ctx)
  _check_usable(ctx, oracle, mesh_case)


def test_open_volume_survives_a_host_buffer_call(ctx, oracle):
  from igneous_b200 import _shim, fastremap
  labels = _blobs((64, 48, 40), 7)
  want, n_want = oracle.connected_components(labels, return_N=True)
  d_in, d_out = ctx.to_device(labels), ctx.alloc(labels.size * 4)
  v, n_local = c.c_void_p(), c.c_uint64(0)
  try:
    _shim.check(ctx.lib.ign_ccl6_volume_begin_dev(ctx.handle, _shim.ptr(d_in), c.c_int(_shim.IGN_U32),
                                                  *_u64(*labels.shape), None, None, None, None, c.byref(v),
                                                  c.byref(n_local)))
    small = np.array([[7, 7, 0], [3, 9, 3]], dtype=np.uint64)
    try:
      got, table = fastremap.renumber(small)
      assert np.array_equal(got, oracle.renumber(small)[0])
    except (_shim.IgneousB200Error, MemoryError):
      pass  # the volume holds the arena: refusing is allowed, touching the volume is not
    _shim.check(ctx.lib.ign_ccl6_volume_finish_dev(v, None, c.c_uint64(n_local.value), _shim.ptr(d_out),
                                                   c.c_int(_shim.IGN_U32)))
    v = None
    got = ctx.to_host(d_out, labels.shape, np.uint32)
    assert n_local.value == n_want and np.array_equal(got, want.astype(np.uint32))
  finally:
    if v:
      ctx.lib.ign_ccl6_volume_abort(v)
    d_in.free()
    d_out.free()
