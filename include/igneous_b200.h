/*
 * igneous_b200.h -- C ABI of libigneous_b200.so
 *
 * B200 (sm_100a) implementation of the igneous per-chunk hot path.  Every
 * entry point replaces one call the reference (seung-lab/igneous @ 3b6e5b6)
 * makes into a third-party CPU library; the reference call site is cited
 * beside each declaration (paths relative to the igneous repo root).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / numpy types.
 *   - all volumes are Fortran order: index = x + sx*(y + sy*z); a 4-D
 *     (x,y,z,c) array is passed as sz*sc slices.
 *   - every function returns IGN_OK (0) or a negative ign_status; the message
 *     is available from ign_last_error() (thread local).
 *   - functions without suffix take HOST buffers (pageable or pinned) and do
 *     H2D / D2H themselves; *_dev variants take DEVICE pointers obtained from
 *     ign_dev_alloc and run asynchronously on the context's stream.
 *   - one ign_ctx per process per GPU; a ctx is not thread safe.
 *   - there is no CPU fallback: without a usable CUDA device ign_init fails.
 */
#ifndef IGNEOUS_B200_H
#define IGNEOUS_B200_H

#include <stdint.h>

#if defined(__GNUC__)
#define IGN_API __attribute__((visibility("default")))
#else
#define IGN_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ign_ctx ign_ctx;
typedef struct ign_mesher ign_mesher;
typedef struct ign_group ign_group;

typedef enum {
  IGN_OK = 0,
  IGN_ERR_CUDA = -1,        /* CUDA runtime error (sticky errors kill the ctx) */
  IGN_ERR_INVALID = -2,     /* bad argument */
  IGN_ERR_UNSUPPORTED = -3, /* dtype / factor / option not implemented */
  IGN_ERR_NOMEM = -4,
  IGN_ERR_KEY = -5,         /* remap: label missing from the table (KeyError) */
  IGN_ERR_OVERFLOW = -6,    /* capacity exceeded (e.g. > 2^31-2 voxels per CCL call) */
  IGN_ERR_NCCL = -7
} ign_status;

typedef enum {
  IGN_U8 = 1,
  IGN_U16 = 2,
  IGN_U32 = 3,
  IGN_U64 = 4,
  IGN_F32 = 5
} ign_dtype;

/* averaging render rule (tinybrain parity is unpinned offline: SURVEY 8(c)) */
typedef enum { IGN_ROUND_FLOOR = 0, IGN_ROUND_HALF_UP = 1, IGN_ROUND_HALF_EVEN = 2 } ign_rounding;

/* ------------------------------------------------------------------ context */
IGN_API int ign_version(void);
IGN_API const char* ign_last_error(void);
IGN_API int ign_device_count(int* n);
IGN_API int ign_init(int device, ign_ctx** out);
IGN_API int ign_destroy(ign_ctx* ctx);
IGN_API int ign_sync(ign_ctx* ctx);
/* number of kernels this library launched on ctx since ign_init */
IGN_API int ign_launch_count(ign_ctx* ctx, uint64_t* n);
/* raw cudaStream_t of the context (for interop: events, NCCL, torch external stream) */
IGN_API int ign_stream(ign_ctx* ctx, void** stream);

/* device / pinned-host memory */
IGN_API int ign_dev_alloc(ign_ctx* ctx, uint64_t bytes, void** dptr);
IGN_API int ign_dev_free(ign_ctx* ctx, void* dptr);
IGN_API int ign_host_alloc(ign_ctx* ctx, uint64_t bytes, void** hptr); /* pinned */
IGN_API int ign_host_free(ign_ctx* ctx, void* hptr);
IGN_API int ign_h2d(ign_ctx* ctx, void* dst, const void* src, uint64_t bytes);  /* async on ctx stream */
IGN_API int ign_d2h(ign_ctx* ctx, void* dst, const void* src, uint64_t bytes);  /* async on ctx stream */
IGN_API int ign_d2d(ign_ctx* ctx, void* dst, const void* src, uint64_t bytes);
IGN_API int ign_memset(ign_ctx* ctx, void* dst, int byte, uint64_t bytes);

/* CUDA-event timers on the ctx stream: slot in [0,64) */
IGN_API int ign_timer_start(ign_ctx* ctx, int slot);
IGN_API int ign_timer_stop(ign_ctx* ctx, int slot);
IGN_API int ign_timer_ms(ign_ctx* ctx, int slot, float* ms); /* synchronises on the stop event */
/* cross-context ordering on one device: waiter's stream waits for the point where
 * producer last called ign_timer_start(producer, slot); no host synchronisation */
IGN_API int ign_stream_wait_mark(ign_ctx* waiter, ign_ctx* producer, int slot);
/* Re-creates the ctx stream (after synchronising it) with the device's greatest (high != 0) or least
 * stream priority.  Thread blocks of a higher-priority stream are dispatched first whenever an SM
 * frees up: a worker that runs short whole-volume passes (CCL: igneous/tasks/image/ccl.py:173) next to
 * long MeshTask streams (tasks/mesh/mesh.py:371-383) asks for high priority on the former. */
IGN_API int ign_stream_priority(ign_ctx* ctx, int high);

/* per-kernel-class CUDA-event profiling on the ctx stream (bench.py roofline):
 * classes 0 ccl_local, 1 ccl_merge, 2 ccl_label, 3 pool, 4 marching cubes */
IGN_API int ign_prof_enable(ign_ctx* ctx, int on);
IGN_API int ign_prof_read(ign_ctx* ctx, int cls, float* total_ms, uint64_t* launches);

/* strided 3-D sub-box copy between device volumes (task cutouts, +1 overlap) */
IGN_API int ign_copy_box_dev(ign_ctx* ctx, const void* src, int dtype, uint64_t sx, uint64_t sy,
                             uint64_t sz, uint64_t x0, uint64_t y0, uint64_t z0, uint64_t bx,
                             uint64_t by, uint64_t bz, void* dst);

/* ------------------------------------------------------------------ pooling
 * tinybrain.downsample_segmentation(img, factor=(2,2,1), num_mips, sparse)
 *   igneous/tasks/image/image.py:52-53 (bound) and :91 (called)
 * tinybrain.downsample_with_averaging(img, factor=(2,2,1), num_mips, sparse)
 *   igneous/tasks/image/image.py:50-51 and :91
 * outs[m] receives mip m+1, shape (ceil(sx/2^(m+1)), ceil(sy/2^(m+1)), sz).
 * Mode pooling is recursive per mip (COUNTLESS 2-D rule); averaging keeps
 * exact sums inside groups of four mips and renders with `rounding`.
 */
IGN_API int ign_pool_mode_2x2x1(ign_ctx* ctx, const void* in, int dtype, uint64_t sx, uint64_t sy,
                        uint64_t sz, int num_mips, int sparse, void* const* outs);
IGN_API int ign_pool_avg_2x2x1(ign_ctx* ctx, const void* in, int dtype, uint64_t sx, uint64_t sy,
                       uint64_t sz, int num_mips, int rounding, void* const* outs);
IGN_API int ign_pool_mode_2x2x1_dev(ign_ctx* ctx, const void* in, int dtype, uint64_t sx, uint64_t sy,
                            uint64_t sz, int num_mips, int sparse, void* const* outs);
IGN_API int ign_pool_avg_2x2x1_dev(ign_ctx* ctx, const void* in, int dtype, uint64_t sx, uint64_t sy,
                           uint64_t sz, int num_mips, int rounding, void* const* outs);

/* Block pooling with factors 1 or 2 per axis -- every tinybrain.downsample_* call other than
 * the (2,2,1) mode / average pyramids above:
 *   igneous/tasks/image/image.py:46-55 (downsample_method_to_fn: min / max / striding, and
 *   mode / average with a non-(2,2,1) factor such as (2,2,2) for --volumetric)
 * op: 0 min, 1 max, 2 striding (partial edge blocks reduce over the samples that exist);
 *     3 mode, 4 sparse mode (zeros ignored): a planar factor with four samples left uses the
 *       COUNTLESS 2-D pick, otherwise the highest count wins with ties to the earliest sample
 *       (x fastest); 5 / 6 / 7 average rendered with IGN_ROUND_FLOOR / HALF_UP / HALF_EVEN
 *       (the lone row / column / slice of an odd extent counts twice; u8, u16, u32, f32);
 *     8 / 9 / 10 sparse average = mean of the non-zero samples (0 if there are none), same
 *       roundings (tinybrain.downsample_with_averaging(sparse=True)).
 * Every mip is computed from the previous one.  Generic one-thread-per-output kernels.
 * [SURVEY 8(f) row 3, not on the headline path] */
IGN_API int ign_pool_select(ign_ctx* ctx, const void* in, int dtype, uint64_t sx, uint64_t sy,
                            uint64_t sz, uint32_t fx, uint32_t fy, uint32_t fz, int num_mips, int op,
                            void* const* outs);
IGN_API int ign_pool_select_dev(ign_ctx* ctx, const void* in, int dtype, uint64_t sx, uint64_t sy,
                                uint64_t sz, uint32_t fx, uint32_t fy, uint32_t fz, int num_mips,
                                int op, void* const* outs);

/* ---------------------------------------------------------------------- CCL
 * cc3d.connected_components(labels, connectivity=6, out_dtype=np.uint64, return_N)
 *   igneous/tasks/image/ccl.py:173, :235-238, :339-342
 * 6-connected, multi-label (equal non-zero values connect), 0 = background.
 * Output ids 1..N in order of each component's first voxel in Fortran raster
 * order.  in_dtype U8 also serves bool input (threshold_image output).
 * out_dtype: IGN_U16 / IGN_U32 / IGN_U64 (overflow -> IGN_ERR_OVERFLOW).
 */
IGN_API int ign_ccl6(ign_ctx* ctx, const void* in, int in_dtype, uint64_t sx, uint64_t sy, uint64_t sz,
             void* out, int out_dtype, uint64_t* n_components);
IGN_API int ign_ccl6_dev(ign_ctx* ctx, const void* in, int in_dtype, uint64_t sx, uint64_t sy,
                 uint64_t sz, void* out, int out_dtype, uint64_t* n_components);

/* Volumes that span several GPUs (one z-slab per rank).  This replaces the four
 * file-based passes of igneous/tasks/image/ccl.py (CCLFacesTask :126-194,
 * CCLEquivalancesTask :196-294, create_relabeling :358-420, RelabelCCLTask
 * :296-356) for data that is resident in HBM: every rank resolves its own volume
 * (begin), the outer z-planes are exchanged and compared (ign_ccl6_link_dev),
 * the equivalences are solved (ign_ccl6_solve, smaller id wins as ccl.py:70-73)
 * and every rank expands its labels once through the composed table (finish).
 * The result is bit-identical to one whole-volume ign_ccl6 call.
 *
 * ign_ccl6_volume_dev: one volume of up to 2^36 voxels in one call (no slabs: the
 * union-find runs over x-runs, not voxels). */
IGN_API int ign_ccl6_link_dev(ign_ctx* ctx, const uint64_t* values_a, const uint32_t* labels_a,
                              uint64_t offset_a, const uint64_t* values_b, const uint32_t* labels_b,
                              uint64_t offset_b, uint64_t n_plane, uint64_t* pairs_host,
                              uint64_t capacity, uint64_t* n_pairs);
IGN_API int ign_ccl6_solve(const uint64_t* pairs, uint64_t n_pairs, uint64_t total, uint32_t* lut,
                           uint64_t* n_global);
IGN_API int ign_ccl6_volume_dev(ign_ctx* ctx, const void* in, int in_dtype, uint64_t sx, uint64_t sy,
                                uint64_t sz, void* out, int out_dtype, uint64_t* n_components);
/* The same in two halves, so that several volumes (one per GPU) can be linked in
 * between: begin resolves the volume and fills its outer z-planes (voxel values
 * widened to u64 and volume-local ids 1..n_local; device buffers of sx*sy
 * entries, may be NULL); finish takes the caller's HOST table [n_local+1] from
 * volume-local to final ids (NULL = identity) and writes the labels. */
typedef struct ign_ccl_volume ign_ccl_volume;
IGN_API int ign_ccl6_volume_begin_dev(ign_ctx* ctx, const void* in, int in_dtype, uint64_t sx,
                                      uint64_t sy, uint64_t sz,
                                      uint64_t* first_values, uint32_t* first_labels,
                                      uint64_t* last_values, uint32_t* last_labels,
                                      ign_ccl_volume** out, uint64_t* n_local);
IGN_API int ign_ccl6_volume_finish_dev(ign_ccl_volume* v, const uint32_t* global_lut,
                                       uint64_t max_label, void* out, int out_dtype);
IGN_API int ign_ccl6_volume_abort(ign_ccl_volume* v);

/* cc3d.dust(labels, threshold, connectivity=6, in_place=True)
 *   igneous/tasks/image/ccl.py:169-172, :231-234, :335-338
 * zeroes (in place) every 6-connected component with < threshold voxels. */
IGN_API int ign_dust(ign_ctx* ctx, void* labels, int dtype, uint64_t sx, uint64_t sy, uint64_t sz,
             uint64_t threshold);
IGN_API int ign_dust_dev(ign_ctx* ctx, void* labels, int dtype, uint64_t sx, uint64_t sy, uint64_t sz,
                 uint64_t threshold);

/* Fused CCLFacesTask body (igneous/tasks/image/ccl.py:166-175): optional
 * threshold (use_lte/use_gte), blackout_non_face_rails(shape), CCL,
 * += label_offset, background re-zeroed; out is u64. */
IGN_API int ign_ccl_task_dev(ign_ctx* ctx, const void* in, int in_dtype, uint64_t sx, uint64_t sy,
                     uint64_t sz, int use_gte, double gte, int use_lte, double lte,
                     uint64_t rail_x, uint64_t rail_y, uint64_t rail_z, uint64_t dust_threshold,
                     uint64_t label_offset, uint64_t* out, uint64_t* n_components);

/* ---------------------------------------------------------------- fastremap
 * fastremap.renumber(data, in_place=True)            igneous/tasks/mesh/mesh.py:206
 *   ids 1..K by first appearance in memory order, 0 kept.  out is u32;
 *   uniq[0..K) receives the original label of new id i+1.
 * fastremap.remap(arr, table, in_place=True)         igneous/tasks/image/ccl.py:346,
 *                                                    igneous/tasks/mesh/mesh.py:369
 *   preserve_missing=0 -> IGN_ERR_KEY when a label is not in keys[].
 * fastremap.unique(arr, return_counts=True)          igneous/tasks/mesh/mesh.py:318
 *   sorted ascending; call with uniq==NULL to get K only.
 * fastremap.mask / mask_except(arr, labels, in_place) igneous/tasks/mesh/mesh.py:201-204,320,368
 * fastremap.inverse_component_map(parents, components) igneous/tasks/image/ccl.py:280
 *   unique (parent, component) pairs sorted ascending; capacity in *n_pairs.
 */
IGN_API int ign_renumber(ign_ctx* ctx, const void* in, int dtype, uint64_t n, uint32_t* out,
                 uint64_t* uniq, uint64_t uniq_capacity, uint64_t* k);
IGN_API int ign_renumber_dev(ign_ctx* ctx, const void* in, int dtype, uint64_t n, uint32_t* out,
                     uint64_t* uniq_dev, uint64_t uniq_capacity, uint64_t* k);
IGN_API int ign_remap(ign_ctx* ctx, void* arr, int dtype, uint64_t n, const uint64_t* keys,
              const uint64_t* vals, uint64_t n_keys, int preserve_missing);
IGN_API int ign_remap_dev(ign_ctx* ctx, void* arr, int dtype, uint64_t n, const uint64_t* keys_host,
                  const uint64_t* vals_host, uint64_t n_keys, int preserve_missing);
IGN_API int ign_unique(ign_ctx* ctx, const void* in, int dtype, uint64_t n, uint64_t* uniq,
               uint64_t* counts, uint64_t capacity, uint64_t* k);
IGN_API int ign_mask(ign_ctx* ctx, void* arr, int dtype, uint64_t n, const uint64_t* labels,
             uint64_t n_labels, int except, uint64_t value);
IGN_API int ign_inverse_component_map(ign_ctx* ctx, const void* parents, const void* components,
                              int dtype, uint64_t n, uint64_t* pairs, uint64_t* n_pairs);
/* widen/narrow unsigned integer arrays on the device */
IGN_API int ign_cast_dev(ign_ctx* ctx, const void* in, int in_dtype, void* out, int out_dtype, uint64_t n);

/* --------------------------------------------------------------------- mesh
 * zmesh.Mesher(resolution).mesh(data, preserve_order=False)  igneous/tasks/mesh/mesh.py:151,245
 * Mesher.ids()                                                igneous/tasks/mesh/mesh.py:374
 * Mesher.get(id, reduction_factor, max_error, voxel_centered) igneous/tasks/mesh/mesh.py:376-381
 * Multi-label marching cubes over every 2x2x2 cube; per label a welded
 * (vertices f32 [nv,3], faces u32 [nf,3]) mesh in physical units:
 *   position = (half_voxel_coord/2 + (voxel_centered ? 0.5 : 0)) * resolution.
 * Vertices are ordered by (z,y,x), faces by cube raster order.
 * reduction_factor > 0 runs the quadric edge-collapse simplifier towards
 * nf/reduction_factor faces with error bound max_error (physical units).
 */
IGN_API int ign_mesh_begin(ign_ctx* ctx, const void* labels, int dtype, uint64_t sx, uint64_t sy,
                   uint64_t sz, ign_mesher** out);
IGN_API int ign_mesh_begin_dev(ign_ctx* ctx, const void* labels, int dtype, uint64_t sx, uint64_t sy,
                       uint64_t sz, ign_mesher** out);
IGN_API int ign_mesh_num_ids(ign_mesher* m, uint64_t* n);
IGN_API int ign_mesh_ids(ign_mesher* m, uint64_t* ids, uint64_t capacity);
IGN_API int ign_mesh_counts(ign_mesher* m, uint64_t id, uint64_t* nv, uint64_t* nf);
IGN_API int ign_mesh_totals(ign_mesher* m, uint64_t* nv, uint64_t* nf);
IGN_API int ign_mesh_get(ign_mesher* m, uint64_t id, const float resolution[3], int reduction_factor,
                 float max_error, int voxel_centered, float* vertices, uint32_t* faces,
                 uint64_t* nv, uint64_t* nf);
/* Simplify every label of the mesher in place (round-based quadric edge collapse
 * towards nf/reduction_factor faces per label, collapse cost <= max_error^2 in
 * physical units, boundary vertices locked).  ign_mesh_get(reduction_factor>0)
 * calls it on first use; ign_mesh_export then returns the simplified meshes. */
IGN_API int ign_mesh_simplify(ign_mesher* m, const float resolution[3], int reduction_factor,
                              float max_error);
/* bulk export of every label's mesh (simplified if ign_mesh_simplify ran) in ign_mesh_ids order:
 * vertices f32 [U,3], faces u32 [T,3] (label-local indices), offsets [n_ids+1] */
IGN_API int ign_mesh_export(ign_mesher* m, const float resolution[3], int voxel_centered,
                            float* vertices, uint32_t* faces, uint64_t* vert_offsets,
                            uint64_t* face_offsets);
IGN_API int ign_mesh_free(ign_mesher* m);

/* ------------------------------------------------- compressed_segmentation codec
 * The Precomputed `compressed_segmentation` chunk encoding that CloudVolume applies on the host
 * before uploading / after downloading a segmentation chunk around the hot path
 * (igneous/tasks/image/image.py:95-100 `vol[new_bounds] = mipped`, ccl.py:346-356 RelabelCCLTask's
 * output, igneous/task_creation/common.py:215-236 set_encoding).  labels: Fortran order [x,y,z,c],
 * uint32 / uint64; block (bx,by,bz) is (8,8,8) in every Precomputed layer.  The stream is the
 * uint32 word sequence of the file.  encode: *n_words = words needed; nothing is written when
 * out is NULL or cap_words is too small.  One call = one chunk: IGN_ERR_OVERFLOW when a lookup table
 * of a channel would start at word 2^24 or later (the header stores table offsets in 24 bits). */
IGN_API int ign_cseg_encode(ign_ctx* ctx, const void* labels, int dtype, uint64_t sx, uint64_t sy, uint64_t sz,
                            uint64_t sc, uint32_t bx, uint32_t by, uint32_t bz, uint32_t* out,
                            uint64_t cap_words, uint64_t* n_words);
IGN_API int ign_cseg_encode_dev(ign_ctx* ctx, const void* labels, int dtype, uint64_t sx, uint64_t sy,
                                uint64_t sz, uint64_t sc, uint32_t bx, uint32_t by, uint32_t bz,
                                uint32_t* out, uint64_t cap_words, uint64_t* n_words);
IGN_API int ign_cseg_decode(ign_ctx* ctx, const uint32_t* in, uint64_t n_words, int dtype, uint64_t sx,
                            uint64_t sy, uint64_t sz, uint64_t sc, uint32_t bx, uint32_t by, uint32_t bz,
                            void* out);
IGN_API int ign_cseg_decode_dev(ign_ctx* ctx, const uint32_t* in, uint64_t n_words, int dtype, uint64_t sx,
                                uint64_t sy, uint64_t sz, uint64_t sc, uint32_t bx, uint32_t by,
                                uint32_t bz, void* out);

/* --------------------------------------------------- synthetic volumes (bench)
 * SURVEY.md 8(d): jittered-grid Voronoi segmentation / hash-byte image,
 * bit-identical to oracle.synth_seg / oracle.synth_image. */
IGN_API int ign_synth_seg_dev(ign_ctx* ctx, void* out, int dtype, uint64_t sx, uint64_t sy, uint64_t sz,
                      int64_t ox, int64_t oy, int64_t oz, uint32_t pitch, uint64_t num_ids,
                      uint64_t seed, uint64_t id_base);
IGN_API int ign_synth_image_dev(ign_ctx* ctx, uint8_t* out, uint64_t sx, uint64_t sy, uint64_t sz,
                        int64_t ox, int64_t oy, int64_t oz, uint64_t seed);

/* ------------------------------------------------------- multi-GPU CCL merge
 * Replaces the file exchange of igneous/tasks/image/ccl.py:177-194 (faces),
 * :245-294 (equivalences) and :358-420 (create_relabeling) with one NCCL
 * all-gather of compacted (label_a,label_b) face-equivalence pairs.
 * One process per GPU; unique_id is ncclUniqueId bytes (128) created on rank 0
 * by ign_group_unique_id and broadcast by the host-side launcher.  NCCL is
 * dlopen()ed on first use (libnccl.so.2), so the library itself has no link-time
 * dependency on it.  Host orchestration: igneous_b200/multigpu.py. */
IGN_API int ign_group_unique_id(void* id128);
IGN_API int ign_group_init(ign_ctx* ctx, int rank, int nranks, const void* id128, ign_group** out);
IGN_API int ign_group_destroy(ign_group* g);
/* the single collective of the path: every rank contributes `bytes` bytes (its
 * component count + outer planes), everyone receives nranks*bytes */
IGN_API int ign_group_allgather(ign_group* g, const void* send_dev, uint64_t bytes, void* recv_dev);
/* SURVEY.md 8(b) `ign_ccl6_sharded`: this rank's z-slab of a dataset split over the group's ranks
 * (rank r above rank r-1).  Local CCL, ONE all-gather of [n_local | first plane | last plane],
 * then -- on the device, identically on every rank -- the N-1 boundaries are linked, the small
 * dataset-wide union-find is solved (smaller id wins, ccl.py:70-73) and the slab's labels are
 * expanded once with dataset-wide ids.  Bit-identical to one whole-volume ign_ccl6 call on the
 * stacked dataset.  Replaces ccl.py:177-194, :245-294, :358-420, :296-356. */
IGN_API int ign_ccl6_sharded_dev(ign_group* g, const void* in, int in_dtype, uint64_t sx, uint64_t sy,
                                 uint64_t sz, void* out, int out_dtype, uint64_t* n_global);

#ifdef __cplusplus
}
#endif
#endif /* IGNEOUS_B200_H */
