#!/usr/bin/env python3
"""Headline benchmark: Mvoxels/s of the igneous hot path (downsample 2 mode mips
-> 6-connected CCL -> marching-cubes meshing at mip 2) on a synthetic 2048^3
uint32 segmentation resident in HBM, one z-slab of the dataset per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--size S] [--impl reference] [--dump-outputs DIR]

Contract (see the task brief): W untimed warm-up steps, exactly K timed steps
bracketed by barrier + device synchronisation, CUDA-event timing on the stream
the kernels are launched on, max over ranks, ONE JSON line from rank 0.
"""
import argparse
import ctypes as c
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

def _baseline_metric():
  """The metric string of BASELINE.json (the bench line must name exactly that metric)."""
  fallback = "Mvoxels/s on 2048\u00b3 uint32 seg (downsample+CCL+mesh) @1/2/4/8 B200; % HBM roofline"
  try:
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "BASELINE.json")) as f:
      return json.load(f).get("metric", fallback)
  except (OSError, ValueError):
    return fallback


METRIC = _baseline_metric()
RESOLUTION = (16, 16, 40)
PITCH, NUM_IDS = 64, 1 << 20


def measured_peaks():
  path = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(path):
    try:
      return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
      pass
  return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
  """nvidia-smi clocks / throttle reasons during the timed region."""

  def __init__(self, index):
    super().__init__(daemon=True)
    self.index, self.samples, self.stop_flag = index, [], False
    self.proc = None

  def run(self):
    q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    try:
      self.proc = subprocess.Popen(
        ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
         "-lms", "500"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      for line in self.proc.stdout:
        if self.stop_flag:
          break
        self.samples.append([v.strip() for v in line.split(",")])
    except Exception:
      pass

  def finish(self):
    self.stop_flag = True
    if self.proc is not None:
      try:
        self.proc.kill()
      except Exception:
        pass
    sm, mx, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for s in self.samples:
      try:
        sm.append(float(s[0]))
        mx.append(float(s[1]))
        for n, v in zip(names, s[3:7]):
          if v.lower().startswith("active"):
            reasons.add(n)
      except Exception:
        continue
    return {"sm_mhz": float(np.median(sm)) if sm else None,
            "sm_max_mhz": float(max(mx)) if mx else None,
            "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------- CPU legs
def oracle_pipeline(seg, simplify=100):
  """The CPU restatement of one step on a host array: returns voxels processed."""
  from oracle import oracle as O
  mips = O.downsample_segmentation(seg, (2, 2, 1), num_mips=2)
  O.connected_components(seg, out_dtype=np.uint32)
  m2 = mips[1]
  for z0 in range(0, m2.shape[2], 256):
    for y0 in range(0, m2.shape[1], 256):
      for x0 in range(0, m2.shape[0], 256):
        tl, tv = O.marching_cubes(m2[x0:x0 + 257, y0:y0 + 257, z0:z0 + 257])
        W = O.WeldedMeshes(tl, tv)
        if simplify:
          O.simplify_welded(W, RESOLUTION, simplify, 40.0, True)
  return seg.size


_WORKER = {}
REF_CHUNK = (256, 256, 64)


def host_cores():
  """Cores this process may actually use: the affinity mask clipped by the cgroup CPU quota
  (os.cpu_count() reports the whole node even inside a small lease)."""
  try:
    n = len(os.sched_getaffinity(0))
  except (AttributeError, OSError):
    n = os.cpu_count() or 1
  quota = None
  try:
    with open("/sys/fs/cgroup/cpu.max") as f:  # cgroup v2
      q, per = f.read().split()[:2]
      if q != "max":
        quota = float(q) / float(per)
  except (OSError, ValueError):
    try:
      with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f1, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f2:
        q, per = float(f1.read()), float(f2.read())
        if q > 0:
          quota = q / per
    except (OSError, ValueError):
      pass
  if quota is not None:
    n = max(1, min(n, int(quota + 0.5)))
  return n


def ref_chunk_offset(index, size):
  """Chunk `index` of the REF_CHUNK grid over the size^3 bench volume (x fastest, as
  FinelyDividedTaskIterator enumerates tasks, igneous/task_creation/common.py:91-98)."""
  gx, gy, gz = (max(1, size // c) for c in REF_CHUNK)
  index %= gx * gy * gz
  return ((index % gx) * REF_CHUNK[0], ((index // gx) % gy) * REF_CHUNK[1], (index // (gx * gy)) * REF_CHUNK[2])


def _oracle_worker_init(counter, size):
  """Each pool worker synthesises its own chunk of the bench volume ONCE (outside any timed region)."""
  from oracle import oracle as O
  with counter.get_lock():
    wid = counter.value
    counter.value += 1
  # spread the workers' chunks over the volume (stride 37 is coprime with the chunk grid)
  _WORKER["seg"] = O.synth_seg(REF_CHUNK, pitch=PITCH, num_ids=NUM_IDS, seed=0,
                               offset=ref_chunk_offset(wid * 37, size))
  O.lib()


def _oracle_worker(_):
  t = time.perf_counter()
  n = oracle_pipeline(_WORKER["seg"])
  return n, time.perf_counter() - t


def run_reference_arm(args):
  """--impl reference: the reference's CPU implementation of the path.  The
  reference's own kernels (tinybrain / cc3d / zmesh wheels) are absent from
  this image, so this times the C oracle port on the host cores this process may
  use (one chunk worker per core, spawn, as igneous_cli/cli.py:915-933 does).  Every
  worker holds one 256x256x64 chunk cut from the SAME synthetic volume the GPU arm
  processes; a step = every worker runs the pipeline once on its chunk."""
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  import multiprocessing as mp
  from oracle import oracle as O
  O.build()
  cores = host_cores()
  ctx = mp.get_context("spawn")
  # one chunk alone on an otherwise idle host: the reference's real per-worker speed
  _oracle_worker_init(ctx.Value("i", 0), args.size)
  _oracle_worker(0)
  alone = min(_oracle_worker(0)[1] for _ in range(2))
  counter = ctx.Value("i", 0)
  times, per_chunk = [], []
  with ctx.Pool(cores, initializer=_oracle_worker_init, initargs=(counter, args.size)) as pool:
    pool.map(_oracle_worker, range(cores), chunksize=1)  # untimed: all workers initialised and warm
    for it in range(args.warmup + args.steps):
      t = time.perf_counter()
      res = pool.map(_oracle_worker, range(cores), chunksize=1)
      dt = time.perf_counter() - t
      if it >= args.warmup:
        times.append((sum(r[0] for r in res), dt))
        per_chunk.extend(r[1] for r in res)
  vox = sum(t[0] for t in times)
  sec = sum(t[1] for t in times)
  value = vox / sec / 1e6
  shape = REF_CHUNK
  line = {
    "impl": "reference", "metric": METRIC, "value": value, "unit": "Mvoxels/s", "n_gpus": args.gpus,
    "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sec / max(len(times), 1),
    "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32",
    "data": "synthetic", "gpu_launches": 0,
    "config": {"workload": "oracle port of the igneous CPU path on %dx%dx%d uint32 chunks cut from the %d^3 "
                           "jittered-Voronoi bench volume (pitch 64), one chunk per usable host core (%d) per step: "
                           "mode pool 2 mips + 6-connected CCL + marching cubes / weld / quadric simplification "
                           "x100 at mip 2" % (shape + (args.size, cores)),
               "chunk": list(shape), "simplification_factor": 100, "cores_used": cores,
               "os_cpu_count": os.cpu_count(),
               "seconds_per_chunk_alone": alone,
               "seconds_per_chunk_contended_median": float(np.median(per_chunk)) if per_chunk else None},
    "cpu_baseline": {"value": value, "unit": "Mvoxels/s", "cores": cores, "kind": "port",
                     "sample": "%d x %dx%dx%d chunks per step, %d steps" % ((cores,) + shape + (args.steps,))},
    "e2e": {"value": value, "unit": "Mvoxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
  }
  print(json.dumps(line))


def cpu_baseline_sample(pipe, ctx, budget_s=20.0):
  """Oracle timed on ONE host core on a bounded sample of the same volume."""
  from oracle import oracle as O
  O.build()
  sx, sy, sz = pipe.shape
  bz = min(sz, 256)
  bx, by = min(sx, 256), min(sy, 256)
  from igneous_b200 import _shim
  d_box = ctx.alloc(bx * by * bz * 4)
  _shim.check(ctx.lib.ign_copy_box_dev(ctx.handle, _shim.ptr(pipe.d_in), c.c_int(pipe.code),
                                       c.c_uint64(sx), c.c_uint64(sy), c.c_uint64(sz), c.c_uint64(0),
                                       c.c_uint64(0), c.c_uint64(0), c.c_uint64(bx), c.c_uint64(by),
                                       c.c_uint64(bz), _shim.ptr(d_box)))
  seg = ctx.to_host(d_box, (bx, by, bz), np.uint32)
  d_box.free()
  t = time.perf_counter()
  vox, reps = 0, 0
  while True:
    vox += oracle_pipeline(seg, pipe.simplification_factor)
    reps += 1
    if time.perf_counter() - t > budget_s / 2 or reps >= 8:
      break
  dt = time.perf_counter() - t
  return {"value": vox / dt / 1e6, "unit": "Mvoxels/s", "cores": 1, "kind": "port",
          "sample": "%dx%dx%d corner of the bench volume, %d repetitions, %.1f s" % (bx, by, bz, reps, dt)}


# ------------------------------------------------------------ parity self-check
def read_box(ctx, dptr, shape, size, dtype, origin=(0, 0, 0)):
  """Host copy of the `size` box at `origin` of a Fortran-order device volume of `shape`."""
  from igneous_b200 import _shim
  d = ctx.alloc(int(np.prod(size)) * np.dtype(dtype).itemsize)
  _shim.check(ctx.lib.ign_copy_box_dev(ctx.handle, _shim.ptr(dptr), c.c_int(_shim.dtype_code(dtype)),
                                       c.c_uint64(shape[0]), c.c_uint64(shape[1]), c.c_uint64(shape[2]),
                                       c.c_uint64(origin[0]), c.c_uint64(origin[1]), c.c_uint64(origin[2]),
                                       c.c_uint64(size[0]), c.c_uint64(size[1]), c.c_uint64(size[2]), _shim.ptr(d)))
  h = ctx.to_host(d, size, dtype)
  d.free()
  return h


def parity_check(ctx, pipe):
  """Untimed check of the benchmark's own products against the CPU oracle (run once after the
  timed loop, at the benchmark's full size): a 256x256x64 sub-box of the mips (bit-exact), the
  CCL labels of the same sub-box (every oracle component carries exactly one label, two
  components share a label only when they hold the same input id, 0 <-> 0) and every fragment
  of one MeshTask body on a 129x129x65 cutout of the mesh mip (bit-exact vertices and faces)."""
  from igneous_b200 import zmesh
  from oracle import oracle as O
  O.build()
  sx, sy, sz = pipe.shape
  bx, by, bz = min(sx, 256), min(sy, 256), min(sz, 64)

  def box(dptr, shape, size, dtype):
    return read_box(ctx, dptr, shape, size, dtype)

  out = {}
  seg = box(pipe.d_in, pipe.shape, (bx, by, bz), np.uint32)
  want = O.downsample_segmentation(seg, (2, 2, 1), num_mips=pipe.num_mips)
  ok = True
  for k, w in enumerate(want):
    got = box(pipe.d_mips[k], pipe.mip_shapes[k], w.shape, np.uint32)
    ok = ok and np.array_equal(got, w)
  out["mips"] = "ok" if ok else "MISMATCH"
  cc = box(pipe.d_cc, pipe.shape, (bx, by, bz), pipe.ccl_out_dtype).astype(np.uint64)
  loc = O.connected_components(seg).astype(np.uint64)
  ok = np.array_equal(cc == 0, seg == 0)
  pairs = np.unique(np.stack([loc.ravel(), cc.ravel(), seg.ravel().astype(np.uint64)], axis=1), axis=0)
  pairs = pairs[pairs[:, 0] != 0]
  ok = ok and len(np.unique(pairs[:, 0])) == len(pairs)           # one label per oracle component
  by_label = np.unique(pairs[:, 1:], axis=0)
  ok = ok and len(np.unique(by_label[:, 0])) == len(by_label)     # one input id per label
  out["ccl"] = "ok" if ok else "MISMATCH"
  msrc = pipe.d_mips[-1] if pipe.num_mips else pipe.d_in
  mshape = pipe.mip_shapes[-1] if pipe.num_mips else pipe.shape
  cut = box(msrc, mshape, (min(mshape[0], 129), min(mshape[1], 129), min(mshape[2], 65)), np.uint32)
  m = zmesh.Mesher(pipe.resolution)
  m.mesh(cut)
  tl, tv = O.marching_cubes(cut)
  W = O.WeldedMeshes(tl, tv)
  f = pipe.simplification_factor or 0
  ok = sorted(m.ids()) == W.ids()
  if f:
    ref, _ = O.simplify_welded(W, pipe.resolution, f, float(pipe.max_simplification_error), True)
  n_lab = 0
  for lab in (W.ids() if ok else []):
    g = m.get(lab, reduction_factor=f, max_error=pipe.max_simplification_error, voxel_centered=True)
    wv, wf = ref[lab] if f else W.get(lab, pipe.resolution, True)
    ok = ok and np.array_equal(g.vertices, wv) and np.array_equal(g.faces, wf)
    n_lab += 1
  out["mesh"] = ("ok (%d fragments bit-exact)" % n_lab) if ok else "MISMATCH"
  out["status"] = "ok" if all(v.startswith("ok") for v in out.values()) else "FAILED"
  return out


DUMP_BOXES, DUMP_BOX = 32, (64, 64, 16)
MESH_COUNTS = ("tasks", "triangles_in", "vertices_in", "triangles", "vertices", "label_fragments")


def dump_outputs(ctx, pipe, out_dir):
  """--dump-outputs: what the last timed step left behind, as float64 .npy files (exact for every
  uint32 value), so that two builds can be compared output for output on the same inputs.

    mip<k>.npy          [DUMP_BOXES, *DUMP_BOX] sample of mode-pooled mip k
    ccl_labels.npy      [DUMP_BOXES, *DUMP_BOX] sample of the 6-connected CCL labels at mip 0
    ccl_components.npy  [1] number of components
    mesh_counts.npy     the MESH_COUNTS totals of the MeshTask bodies (the step keeps no fragments)

  The volumes are far larger than a dump should be, so each is sampled as DUMP_BOXES boxes (clamped
  to the volume) whose origins come from numpy's default_rng(0): the same boxes on every run with
  the same --size.  At most 48 MiB in all."""
  os.makedirs(out_dir, exist_ok=True)
  u = np.random.default_rng(0).random((DUMP_BOXES, 3))

  def sample(dptr, shape, dtype):
    size = tuple(min(b, s) for b, s in zip(DUMP_BOX, shape))
    origins = (u * (np.asarray(shape) - np.asarray(size) + 1)).astype(np.int64)
    return np.stack([read_box(ctx, dptr, shape, size, dtype, o) for o in origins]).astype(np.float64)

  for k, (dptr, shape) in enumerate(zip(pipe.d_mips, pipe.mip_shapes)):
    np.save(os.path.join(out_dir, "mip%d.npy" % (k + 1)), sample(dptr, shape, pipe.dtype))
  np.save(os.path.join(out_dir, "ccl_labels.npy"), sample(pipe.d_cc, pipe.shape, pipe.ccl_out_dtype))
  np.save(os.path.join(out_dir, "ccl_components.npy"), np.array([pipe.n_components], dtype=np.float64))
  np.save(os.path.join(out_dir, "mesh_counts.npy"),
          np.array([pipe.mesh_stats[k] for k in MESH_COUNTS], dtype=np.float64))


def multigpu_check(ctx, group, rank, world, dist):
  """N-rank parity of the sharded CCL (NCCL all-gather of the boundary planes) against a
  whole-volume oracle CCL of the stacked dataset (tools/check_multigpu.py inside the bench)."""
  import torch
  from igneous_b200 import pipeline
  from oracle import oracle as O
  O.build()
  shape = (96, 80, 40)
  pipe = pipeline.VolumePipeline(ctx, shape, np.uint32, pitch=32, num_ids=6, offset=(0, 0, rank * shape[2]),
                                 group=group, simplification_factor=0, mesh_shape=(32, 32, 32), mesh_streams=1)
  pipe.synth()
  pipe.ccl()
  got = ctx.to_host(pipe.d_cc, shape, np.uint32)
  whole = O.synth_seg((shape[0], shape[1], shape[2] * world), pitch=32, num_ids=6)
  want, n_want = O.connected_components(whole, return_N=True)
  ok = (pipe.n_components == n_want) and np.array_equal(
    got, want[:, :, rank * shape[2]:(rank + 1) * shape[2]].astype(np.uint32))
  pipe.free()
  flag = torch.tensor([1 if ok else 0], device="cuda")
  dist.all_reduce(flag, op=dist.ReduceOp.MIN)
  return "ok (%d ranks, %d components)" % (world, n_want) if int(flag.item()) == 1 else "MISMATCH"


# ------------------------------------------------- per-config lines (BASELINE.json configs)
def run_config(args, ctx, rank, world, dist):
  """--config c1|c2|c3: one JSON line for a BASELINE.json config other than the headline."""
  from igneous_b200 import _shim
  peak, peak_src = measured_peaks()
  lib = ctx.lib
  line = {"metric": METRIC, "unit": "Mvoxels/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic"}
  if args.config == "c2":
    # DownsampleTask 5-level average pyramid on a 2048x2048x512 uint8 image, one 512^3 chunk per launch
    S = 512
    n = S ** 3
    d_in = ctx.alloc(n)
    _shim.check(lib.ign_synth_image_dev(ctx.handle, _shim.ptr(d_in), c.c_uint64(S), c.c_uint64(S), c.c_uint64(S),
                                        c.c_int64(0), c.c_int64(0), c.c_int64(rank * S), c.c_uint64(0)))
    shapes, x = [], S
    for _ in range(5):
      x = (x + 1) // 2
      shapes.append((x, x, S))
    outs = [ctx.alloc(int(np.prod(sh))) for sh in shapes]
    call = lambda: _shim.check(lib.ign_pool_avg_2x2x1_dev(
      ctx.handle, _shim.ptr(d_in), c.c_int(_shim.IGN_U8), c.c_uint64(S), c.c_uint64(S), c.c_uint64(S), c.c_int(5),
      c.c_int(_shim.ROUND_FLOOR), _shim.void_pp([o.ptr for o in outs])))
    chunks = 16  # 2048x2048x512 = 4x4x1 chunks of 512^3: 16 launches per step
    for _ in range(args.warmup):
      for _ in range(chunks):
        call()
    ctx.sync()
    ctx.timer_start(0)
    for _ in range(args.steps * chunks):
      call()
    ctx.timer_stop(0)
    ms = ctx.timer_ms(0) / args.steps
    vox = n * chunks
    bytes_alg = vox * (1 + sum(0.25 ** k for k in range(1, 6)))
    line.update({"value": vox * world / (ms * 1e-3) / 1e6, "ms_per_step": ms, "dtype": "u8",
                 "gpu_launches": 2 * chunks * args.steps,
                 "config": {"workload": "C2: 5-level 2x2x1 average pyramid of a 2048x2048x512 uint8 image, one 512^3 chunk "
                                        "per call (16 calls per step; the 128 MiB chunk is re-read from L2/HBM every call)",
                            "l2": "one 512^3 u8 chunk (134 MB) + outputs exceed the 126 MB L2"},
                 "roofline": {"bound": "hbm", "kernel": "k_avg_fused<u8>", "achieved": bytes_alg / 1e9 / (ms * 1e-3),
                              "peak": peak, "unit": "GB/s", "frac": bytes_alg / 1e9 / (ms * 1e-3) / peak,
                              "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_voxel": 1.333}})
  elif args.config == "c3":
    # CCLFacesTask family on 1024^3 uint64 (~4000 objects): one volume per GPU (z-slab of the dataset)
    from igneous_b200 import pipeline, multigpu
    S = args.size if args.size != 2048 else 1024
    group = multigpu.Group(ctx, rank, world, dist) if world > 1 else None
    pipe = pipeline.VolumePipeline(ctx, (S, S, S), np.uint64, num_mips=0, pitch=64, num_ids=4096, seed=0,
                                   offset=(0, 0, rank * S), simplification_factor=0, group=group, mesh_streams=1,
                                   ccl_out_dtype=np.uint64, id_base=1 << 32)
    pipe.synth()
    for _ in range(args.warmup):
      pipe.ccl()
    ctx.sync()
    if dist is not None:
      dist.barrier()
    pipe.prof_enable(True)
    ctx.timer_start(0)
    for _ in range(args.steps):
      pipe.ccl()
    ctx.timer_stop(0)
    ms = ctx.timer_ms(0) / args.steps
    prof = pipe.prof_read()
    pipe.prof_enable(False)
    if dist is not None:
      import torch
      t = torch.tensor([ms], dtype=torch.float64, device="cuda")
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
      ms = float(t.item())
    n = S ** 3
    alg = n * 16
    kern = {k: v[0] / args.steps for k, v in prof.items() if v[1]}
    line.update({"value": n * world / (ms * 1e-3) / 1e6, "ms_per_step": ms, "dtype": "u64",
                 "gpu_launches": int(sum(v[1] for v in prof.values())),
                 "config": {"workload": "C3: 6-connected CCL of a %d^3 uint64 segmentation per GPU (ids >= 2^32, pitch 64), "
                                        "uint64 labels out%s" % (S, ", one NCCL all-gather of the boundary planes" if world > 1 else ""),
                            "components": pipe.n_components, "kernel_ms_per_step": kern},
                 "roofline": {"bound": "hbm", "kernel": "CCL stage (k_ccl_masks + k_ccl_tiles/merge + k_ccl_expand)",
                              "achieved": alg / 1e9 / (ms * 1e-3), "peak": peak, "unit": "GB/s",
                              "frac": alg / 1e9 / (ms * 1e-3) / peak, "traffic": None, "peak_source": peak_src,
                              "algorithmic_bytes_per_voxel": 16}})
  elif args.config == "c1":
    # DownsampleTask mip0 -> mip1 (2x2x1 mode) on 128x128x64 uint32 through LocalTaskQueue(parallel=1), file:// layer
    import shutil, tempfile
    from igneous_b200 import task_creation as tc
    from igneous_b200._compat import CloudVolume, LocalTaskQueue
    from oracle import oracle as O
    O.build()
    seg = O.synth_seg((128, 128, 64), pitch=16, num_ids=64)
    root = tempfile.mkdtemp(prefix="ign_c1_")
    times = []
    try:
      for it in range(args.warmup + args.steps):
        path = "file://" + os.path.join(root, "layer%d" % it)
        CloudVolume.from_numpy(seg[..., None], vol_path=path, resolution=(16, 16, 40), chunk_size=(64, 64, 64),
                               layer_type="segmentation", max_mip=0)
        t0 = time.perf_counter()
        tq = LocalTaskQueue(parallel=1)
        tq.insert_all(tc.create_downsampling_tasks(path, mip=0, num_mips=1, compress="gzip"))
        dt = time.perf_counter() - t0
        if it >= args.warmup:
          times.append(dt)
      cv = CloudVolume(path)
      cv.mip = 1
      got = np.asarray(cv[cv.meta.bounds(1)])
      want = O.downsample_segmentation(seg[..., None], (2, 2, 1, 1), num_mips=1)[0]
      ok = np.array_equal(got, want)
    finally:
      shutil.rmtree(root, ignore_errors=True)
    ms = 1e3 * float(np.median(times))
    line.update({"value": seg.size / (ms * 1e-3) / 1e6, "ms_per_step": ms, "dtype": "u32", "gpu_launches": None,
                 "config": {"workload": "C1: DownsampleTask mip0->mip1 (2x2x1 mode) on 128x128x64 uint32 through "
                                        "create_downsampling_tasks + LocalTaskQueue(parallel=1) on a file:// layer "
                                        "(task wall time: download, H2D, kernel, D2H, encode, upload)",
                            "parity_vs_oracle": "ok" if ok else "MISMATCH"},
                 "roofline": None})
  if rank == 0:
    print(json.dumps(line))


# -------------------------------------------------------------------- main
def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=5)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--size", type=int, default=2048, help="cube edge of the per-GPU volume (weak scaling) / of the whole volume (strong)")
  ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
  ap.add_argument("--config", default="headline", choices=["headline", "c1", "c2", "c3"],
                  help="BASELINE.json config: headline = the metric's 2048^3 pipeline; c1 / c2 / c3 print their own line")
  ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                  help="weak: one size^3 volume per GPU; strong: ONE size^3 volume split into N z-slabs")
  ap.add_argument("--check", action="store_true", help="N>1: also run the N-rank CCL parity check against the oracle")
  ap.add_argument("--no-parity-check", action="store_true")
  ap.add_argument("--no-e2e", action="store_true")
  ap.add_argument("--no-cpu", action="store_true")
  ap.add_argument("--e2e-steps", type=int, default=2)
  ap.add_argument("--e2e-shared-buffers", action="store_true",
                  help="download the labels into the input host buffer (forced automatically when host RAM is tight)")
  ap.add_argument("--simplify", type=int, default=None, help="simplification factor (default 100)")
  ap.add_argument("--mesh-streams", type=int, default=8, help="concurrent MeshTask bodies per GPU")
  ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                  help="after the timed steps, write a fixed sample of the last step's products to DIR/<name>.npy")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  if args.dump_outputs and (args.impl != "b200" or args.config != "headline"):
    ap.error("--dump-outputs applies to the headline pipeline (--impl b200 --config headline)")
  if args.warmup < 3 and args.impl == "b200":
    args.warmup = 3

  if args.impl == "reference":
    return run_reference_arm(args)

  rank = int(os.environ.get("RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  local_rank = int(os.environ.get("LOCAL_RANK", "0"))
  bind_numa(local_rank)
  dist = None
  if world > 1:
    import torch
    import torch.distributed as dist_mod
    torch.cuda.set_device(local_rank)
    dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dist = dist_mod

  from igneous_b200 import _shim, pipeline
  ctx = _shim.Context(local_rank)
  if args.config != "headline":
    run_config(args, ctx, rank, world, dist)
    if dist is not None:
      dist.barrier()
      dist.destroy_process_group()
    return
  S = args.size
  strong = args.scaling == "strong" and world > 1
  sz_local = S // world if strong else S
  shape = (S, S, sz_local)
  simplify = 100 if args.simplify is None else args.simplify
  group = None
  if world > 1:
    from igneous_b200 import multigpu
    group = multigpu.Group(ctx, rank, world, dist)
  pipe = pipeline.VolumePipeline(ctx, shape, np.uint32, num_mips=2, mesh_shape=(256, 256, 256),
                                 resolution=RESOLUTION, pitch=PITCH, num_ids=NUM_IDS, seed=0,
                                 offset=(0, 0, rank * sz_local), simplification_factor=simplify, group=group,
                                 mesh_streams=args.mesh_streams)
  pipe.synth()
  ctx.sync()

  def barrier():
    ctx.sync()
    if dist is not None:
      dist.barrier()

  for _ in range(args.warmup):
    pipe.step(timers=False)
  barrier()

  sampler = ClockSampler(local_rank) if rank == 0 else None
  if sampler:
    sampler.start()
    time.sleep(0.3)
  launches0 = pipe.launch_count()
  pipe.prof_enable(True)
  stage = {"pool_ms": 0.0, "ccl_ms": 0.0, "mesh_ms": 0.0}
  barrier()
  ctx.timer_start(0)
  for _ in range(args.steps):
    pipe.step(timers=True)
    for k, v in pipe.stage_ms().items():
      stage[k] += v
  ctx.timer_stop(0)
  total_ms = ctx.timer_ms(0)
  barrier()
  prof = pipe.prof_read()
  pipe.prof_enable(False)
  launches = pipe.launch_count() - launches0
  clocks = sampler.finish() if sampler else None

  if dist is not None:
    import torch
    t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
  ms_per_step = total_ms / args.steps
  voxels = pipe.n * world
  value = voxels / (ms_per_step * 1e-3) / 1e6

  # ---- roofline (SURVEY.md 8(d)): the kernel class with the largest summed launch time per
  # step, algorithmic bytes per launch / its average launch duration (CUDA events recorded by
  # the library around those launches, on the stream they run on)
  peak, peak_src = measured_peaks()
  in_b, out_b = 4, pipe.ccl_out_dtype.itemsize
  ms_in = pipe.mesh_stats
  mip2_vox = int(np.prod(pipe.mip_shapes[-1]))
  alg_step = {  # algorithmic bytes of one STEP per kernel class
    "pool": pipe.n * 4 * (1 + 0.25 + 0.0625),
    "ccl_local": pipe.n * in_b,          # k_ccl_masks: every voxel read once
    "ccl_merge": pipe.n * 0.625,         # k_ccl_tiles / merge / roots: the masks (0.625 B/voxel)
    "ccl_label": pipe.n * out_b,         # k_ccl_expand: every label written once
    "mc": mip2_vox * 4,
    "simp_labels": 12.0 * (ms_in.get("triangles_in", 0) + ms_in.get("vertices_in", 0) +
                           ms_in.get("triangles", 0) + ms_in.get("vertices", 0)),
  }
  knames = {"pool": "k_mode_fused<u32,2>", "ccl_local": "k_ccl_masks<u32> (TMA)", "ccl_merge": "k_ccl_tiles + k_ccl_merge + run passes",
            "ccl_label": "k_ccl_expand4<u32>", "mc": "k_mc", "simp_labels": "k_simp_labels"}
  kern = {k: {"ms_per_step": prof[k][0] / args.steps, "launches_per_step": prof[k][1] / args.steps,
              "algorithmic_GBps": (alg_step[k] / 1e9) / (prof[k][0] / args.steps * 1e-3) if prof[k][0] > 0 else None}
          for k in prof}
  for k in kern:
    if kern[k]["algorithmic_GBps"] is not None:
      kern[k]["frac_of_hbm_peak"] = kern[k]["algorithmic_GBps"] / peak
  dominant = max(prof, key=lambda k: prof[k][0])
  dom_ms = prof[dominant][0] / args.steps
  dom_launches = max(prof[dominant][1] / args.steps, 1)
  achieved = (alg_step[dominant] / dom_launches / 1e9) / (dom_ms / dom_launches * 1e-3) if dom_ms > 0 else 0.0
  ccl_ms = sum(prof[k][0] for k in ("ccl_local", "ccl_merge", "ccl_label")) / args.steps
  roofline = {
    "bound": "hbm", "kernel": knames[dominant], "achieved": achieved, "peak": peak, "unit": "GB/s",
    "frac": achieved / peak, "traffic": NCU_TRAFFIC.get(dominant, {}).get("bytes_per_launch"),
    "traffic_source": NCU_TRAFFIC.get(dominant, {}).get("source"),
    "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_step[dominant] / dom_launches,
    "avg_launch_ms": dom_ms / dom_launches, "launches_per_step": dom_launches,
    "share_of_step_kernel_time": prof[dominant][0] / max(sum(v[0] for v in prof.values()), 1e-9),
    "stage_ccl": {"algorithmic_bytes_per_voxel": in_b + out_b, "kernel_ms_per_step": ccl_ms,
                  "wall_ms_per_step": stage["ccl_ms"] / args.steps,
                  "achieved": pipe.n * (in_b + out_b) / 1e9 / (stage["ccl_ms"] / args.steps * 1e-3) if stage["ccl_ms"] > 0 else 0.0},
    "stage_pool": {"algorithmic_bytes_per_voxel": 5.3125, "wall_ms_per_step": stage["pool_ms"] / args.steps,
                   "achieved": pipe.n * 5.3125 / 1e9 / (stage["pool_ms"] / args.steps * 1e-3) if stage["pool_ms"] > 0 else 0.0},
    "kernels": kern,
    "note": "kernel = the class with the largest summed launch time per step (MeshTask bodies run on %d concurrent "
            "streams, so class sums can exceed the stage wall time); stage_* use the stage wall time between CUDA "
            "events on the main stream" % pipe.mesh_streams,
  }
  roofline["stage_ccl"]["frac"] = roofline["stage_ccl"]["achieved"] / peak
  roofline["stage_pool"]["frac"] = roofline["stage_pool"]["achieved"] / peak

  line = {
    "metric": METRIC, "value": value, "unit": "Mvoxels/s", "n_gpus": world, "steps": args.steps,
    "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
    "scaling": "strong" if strong else "weak",
    "vs_baseline": None, "dtype": "u32", "data": "synthetic", "gpu_launches": int(launches),
    "config": {
      "workload": "%dx%dx%d uint32 jittered-Voronoi segmentation per GPU (pitch %d)%s: mode-pool 2 mips, "
                  "6-connected CCL at mip 0 (u32 ids), marching cubes + weld%s at mip 2 in 256^3 tasks"
                  % (S, S, sz_local, PITCH, (" = one %d^3 volume split into %d z-slabs" % (S, world)) if strong else "",
                     (" + quadric simplification x%d" % simplify) if simplify else ""),
      "volume_per_gpu": list(shape), "parallelism": "z-slab per GPU, %d rank(s)" % world,
      "l2": "inputs larger than L2 (%.1f GB volume vs 126 MB L2)" % (pipe.n * 4 / 1e9),
      "simplification_factor": simplify, "components": pipe.n_components, "mesh": pipe.mesh_stats, "mesh_streams": pipe.mesh_streams,
      "stage_ms_per_step": {k: v / args.steps for k, v in stage.items()},
    },
    "roofline": roofline, "clocks": clocks,
  }

  if args.dump_outputs and rank == 0:  # before the e2e leg, which recomputes into the same buffers
    dump_outputs(ctx, pipe, args.dump_outputs)
  if not args.no_parity_check:
    line["parity_check"] = parity_check(ctx, pipe) if rank == 0 else None
  if args.check and world > 1:
    line["multi_gpu_parity"] = multigpu_check(ctx, group, rank, world, dist)
  if rank == 0 and not args.no_cpu:
    line["cpu_baseline"] = cpu_baseline_sample(pipe, ctx)
  if not args.no_e2e:
    line["e2e"] = run_e2e(ctx, pipe, args, dist, world)
  if rank == 0:
    print(json.dumps(line))
  if dist is not None:
    dist.barrier()
    dist.destroy_process_group()


# dram__bytes_read.sum + dram__bytes_write.sum per launch from `ncu --set full` captures (profiles/)
NCU_TRAFFIC = {
  # dram__bytes_read.sum + dram__bytes_write.sum per launch from ncu --set full captures (profiles/)
  "simp_labels": {"bytes_per_launch": 3.926e9, "source": "profiles/r02_simp_labels_v8_full_summary.txt (one 257^3 MeshTask at mip 2)"},
  "ccl_local": {"bytes_per_launch": 6.517e10, "source": "profiles/r02_ccl2048_metrics.csv (2048^3 u32, two CTAs per SM; 1024^3: 5.27e9)"},
  "ccl_label": {"bytes_per_launch": 3.826e10, "source": "profiles/r02_ccl2048_metrics.csv (2048^3 u32)"},
}


def bind_numa(local_rank):
  """Keep this rank's host threads (and therefore its first-touched pinned buffers) on the
  NUMA node of its GPU: the e2e leg moves ~80 GB per step through host DRAM per rank."""
  try:
    import pynvml
    pynvml.nvmlInit()
    h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
    n = (os.cpu_count() + 63) // 64
    mask = pynvml.nvmlDeviceGetCpuAffinity(h, n)
    cpus = [64 * i + b for i, w in enumerate(mask) for b in range(64) if (w >> b) & 1]
    allowed = set(os.sched_getaffinity(0))
    cpus = [x for x in cpus if x in allowed]
    if cpus:
      os.sched_setaffinity(0, cpus)
      return len(cpus)
  except Exception:
    pass
  return None


def _mem_available():
  try:
    with open("/proc/meminfo") as f:
      for line in f:
        if line.startswith("MemAvailable:"):
          return int(line.split()[1]) * 1024
  except OSError:
    pass
  return None


def run_e2e(ctx, pipe, args, dist, world):
  """Same metric through host buffers: every step copies the volume H2D from
  pinned memory, runs the pipeline and copies every product (mips, CCL labels,
  all mesh fragments) back D2H."""
  from igneous_b200 import _shim
  n = pipe.n
  host_kind = "pinned (cudaHostAlloc)"
  # host RAM guard: all local ranks keep input + products resident on the host.  When that
  # does not fit comfortably, the label volume is downloaded into the input buffer (what
  # in_place=True does in the reference) and the input is restored between steps, untimed.
  out_bytes = sum(int(np.prod(s)) * 4 for s in pipe.mip_shapes) + n * pipe.ccl_out_dtype.itemsize
  local_ranks = int(os.environ.get("LOCAL_WORLD_SIZE", world))
  avail = _mem_available()
  if dist is not None:  # every rank must take the same decisions below: agree on the smallest reading
    import torch
    t = torch.tensor([float(avail) if avail is not None else -1.0], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    avail = int(t.item()) if t.item() >= 0 else None
  shared = (avail is not None and (n * 4 + out_bytes) * local_ranks > 0.6 * avail
            and pipe.ccl_out_dtype.itemsize == 4)
  if args.e2e_shared_buffers:
    shared = pipe.ccl_out_dtype.itemsize == 4
  need = (n * 4 + (out_bytes - n * pipe.ccl_out_dtype.itemsize if shared else out_bytes)) * local_ranks
  if avail is not None and need > 0.85 * avail:
    # never drive the host out of memory: report the leg as not measurable on this box
    return {"value": None, "unit": "Mvoxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
            "skipped": "host buffers for %d local rank(s) need %.0f GB, %.0f GB of host RAM available"
                       % (local_ranks, need / 1e9, avail / 1e9)}
  try:
    host_in = ctx.pinned_empty(pipe.shape, np.uint32)
    host = {"mips": [ctx.pinned_empty(s, np.uint32) for s in pipe.mip_shapes],
            "cc": (host_in.view(pipe.ccl_out_dtype) if shared
                   else ctx.pinned_empty(pipe.shape, pipe.ccl_out_dtype))}
  except (MemoryError, _shim.IgneousB200Error):
    # the host could not page-lock the buffers for this rank: fall back to pageable memory
    host_kind = "pageable (pinned allocation failed)"
    host_in = np.empty(pipe.shape, dtype=np.uint32, order="F")
    host = {"mips": [np.empty(s, dtype=np.uint32, order="F") for s in pipe.mip_shapes],
            "cc": (host_in.view(pipe.ccl_out_dtype) if shared
                   else np.empty(pipe.shape, dtype=pipe.ccl_out_dtype, order="F"))}
  ctx.d2h(host_in, pipe.d_in)
  cap_v, cap_f = 1 << 22, 1 << 23
  ctx.sync()
  mesh_bytes = [0]
  res = (c.c_float * 3)(*[float(r) for r in RESOLUTION])

  lock = threading.Lock()
  host_bufs = {}

  def export(task, h, nv, nf, nl, wctx):
    if nv == 0:
      return
    if id(wctx) not in host_bufs:  # one pinned staging pair per mesh stream
      host_bufs[id(wctx)] = (wctx.pinned_empty((cap_v, 3), np.float32, order="C"),
                             wctx.pinned_empty((cap_f, 3), np.uint32, order="C"))
    bv, bf = host_bufs[id(wctx)]
    voff = np.zeros(nl + 1, dtype=np.uint64)
    foff = np.zeros(nl + 1, dtype=np.uint64)
    v = bv if nv <= cap_v else np.empty((nv, 3), np.float32)
    f = bf if nf <= cap_f else np.empty((nf, 3), np.uint32)
    _shim.check(wctx.lib.ign_mesh_export(h, res, c.c_int(1), _shim.ptr(v), _shim.ptr(f),
                                         _shim.ptr(voff), _shim.ptr(foff)))
    with lock:
      mesh_bytes[0] += nv * 12 + nf * 12

  steps = max(1, min(args.e2e_steps, args.steps))

  def one():
    mesh_bytes[0] = 0
    # upload in z-layers; pooling, meshing, CCL and the D2H of the products overlap
    pipe.step_streamed(host_in, host, export)

  one()  # warm-up (pinned pages touched, arena sized)
  ctx.sync()
  ms = 0.0
  for _ in range(steps):
    if shared:  # the label download overwrote the input: restore it outside the timed region
      ctx.d2h(host_in, pipe.d_in)
      ctx.sync()
    if dist is not None:
      dist.barrier()
    t0 = time.perf_counter()
    ctx.timer_start(4)
    one()
    ctx.timer_stop(4)
    ev = ctx.timer_ms(4)
    ms += max(ev, (time.perf_counter() - t0) * 1e3)  # host-side export work counts too
  if dist is not None:
    import torch
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
  h2d = n * 4
  d2h = sum(int(np.prod(s)) * 4 for s in pipe.mip_shapes) + n * pipe.ccl_out_dtype.itemsize + mesh_bytes[0]
  return {"value": n * world / (ms / steps * 1e-3) / 1e6, "unit": "Mvoxels/s",
          "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": steps,
          "ms_per_step": ms / steps, "host_memory": host_kind,
          "host_buffers": ("input buffer reused for the label download, restored between steps outside "
                           "the timed region" if shared else "separate input and output buffers")}


if __name__ == "__main__":
  main()
