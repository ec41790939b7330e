/*
 * bodyslam_b200.h -- C ABI of the B200-native BodySLAM depth->3D hot path.
 *
 * The reference (GuidoManni/BodySLAM) is pure Python and has no FFI of its own: the
 * drop-in boundary is the Python signatures of MDEM (`colorize`, `DepthEstimator`) and 3DM
 * (`TSDF`, `RGBD`, `update_map_after_pg`), which `bodyslam_b200/*.py` mirror.  This header is
 * what those mirrors bind (ctypes, see INTEGRATION.md); each entry point cites the reference
 * interface it replaces (paths relative to /root/reference, R/ = BodySLAM_Refactored/,
 * N/ = BodySLAM_not_refactored/).
 *
 * Conventions
 *   - every function returns 0 on success, a negative BSLAM_E_* code on failure;
 *     bslam_last_error() returns the message of the calling thread's last failure;
 *   - pointers named d_* are DEVICE pointers owned by the caller (e.g. torch tensors),
 *     pointers named h_* are HOST pointers; nothing is allocated behind the caller's back
 *     except what bslam_tsdf_create is asked to allocate;
 *   - all work is enqueued on `stream` (a cudaStream_t); no entry point synchronises
 *     unless its comment says it returns a host value;
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails
 *     with BSLAM_E_CUDA.
 */
#ifndef BODYSLAM_B200_H
#define BODYSLAM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BSLAM_API __attribute__((visibility("default")))

typedef void *bslam_stream_t;           /* cudaStream_t */
typedef struct bslam_volume bslam_volume; /* opaque dense TSDF box (brick-ordered in HBM) */

enum {
    BSLAM_OK = 0,
    BSLAM_E_ARG = -1,     /* bad argument / shape / unsupported format (Open3D: "Unsupported image format.") */
    BSLAM_E_CUDA = -2,    /* CUDA runtime error, incl. "no device" */
    BSLAM_E_CAPACITY = -3 /* caller-provided output buffer too small */
};

/* brick edge in voxels, frames per integrate launch */
#define BSLAM_BRICK 8
#define BSLAM_MAX_BATCH 256

/* z-march modes of bslam_tsdf_integrate (see DESIGN.md "float32 recurrence") */
#define BSLAM_ZMARCH_BRICK 8   /* camera-space point re-evaluated at every brick base (oracle z_restart=8); in unit-activation
                                  mode at every UNIT base instead = Open3D's literal per-unit recurrence (oracle z_restart=0) */
#define BSLAM_ZMARCH_LITERAL 0 /* Open3D's literal per-column float32 recurrence from z=0 (validation kernel) */

BSLAM_API const char *bslam_last_error(void);
BSLAM_API int bslam_version(void);
/* number of CUDA devices visible (0 when none / no driver); never fails */
BSLAM_API int bslam_device_count(void);

/* ------------------------------------------------------------------ MDEM (K1)
 * Replaces the ZoeDepth `infer_pil(output_type="pil")` tail reached from
 * R/src/depth_estimation/interface.py:61 and N/MDEM/mdem_interface.py:68:
 *     u16 = (metres_f32 * scale_mul).astype(uint16)       (scale_mul = 256)
 * Values are truncated toward zero; out-of-range values saturate to [0, 65535]. */
BSLAM_API int bslam_scale_u16(const float *d_depth, int64_t n, float scale_mul, uint16_t *d_out,
                              bslam_stream_t stream);

/* bytes of device workspace bslam_colorize needs for a batch of B images */
BSLAM_API size_t bslam_colorize_workspace_bytes(int B);

/*
 * Fused metric scaling + colorization of a batch of B images of H*W pixels.
 * Replaces `colorize(value, vmin, vmax, cmap, invalid_val, ..., background_color)`
 * R/examples/depth_estimation/depth_map_scaling.py:12-45 (== batch_processing.py:12-45) for
 * 16-bit integer-valued input, per image:
 *   valid = value != invalid_val;  vmin/vmax = numpy percentile(valid, p_lo / p_hi) (linear);
 *   x = (value - vmin) / (vmax - vmin) in f64 (0 when vmin == vmax);
 *   index = matplotlib Colormap.__call__: trunc(x*256), <0 -> 0, ==256 -> 255, >255 -> 255;
 *   rgba = lut[index]; invalid pixels -> bg_rgba.
 * Input is EITHER d_depth_m (f32 metres; scaled to u16 with scale_mul first and, if
 * d_u16_out != NULL, written there) OR d_u16_in.  d_lut is 256*4 bytes (gamma already folded
 * in by the host).  has_invalid == 0 disables the invalid test (invalid_val outside u16).
 * h_vmin_vmax: optional HOST [B][2] f64 overrides (NaN = compute by percentile).
 * d_vmin_vmax_out: optional DEVICE [B][2] f64, the values used.
 * d_table_override: optional DEVICE [B][65536] u8 index table (value_transform support):
 *   when given, index = d_table_override[b][value] and percentiles are skipped.
 */
BSLAM_API int bslam_colorize(const float *d_depth_m, const uint16_t *d_u16_in, int B, int H, int W,
                             float scale_mul, uint16_t *d_u16_out, uint8_t *d_rgba,
                             const uint8_t *d_lut, double p_lo, double p_hi, int has_invalid,
                             uint16_t invalid_val, uint32_t bg_rgba, const double *h_vmin_vmax,
                             double *d_vmin_vmax_out, const uint8_t *d_table_override,
                             void *d_workspace, bslam_stream_t stream);

/*
 * `colorize` for a FLOAT32 image (metres as ZoeDepth predicts them, numpy or torch -- the reference accepts
 * both, depth_map_scaling.py:14-15): same steps as bslam_colorize, in NumPy's float32 arithmetic
 * (percentile virtual index, lerp, normalisation all float32, as NumPy 2.x evaluates them for a float32 array);
 * the order statistics come from an exact two-level radix select on the floats' order-preserving keys.
 * invalid_val is compared as float (`value == invalid_val`); NaN pixels get the colormap's "bad" colour (0,0,0,0).
 * d_workspace: bslam_colorize_f32_workspace_bytes(B).  h_vmin_vmax / d_vmin_vmax_out as in bslam_colorize.
 */
BSLAM_API size_t bslam_colorize_f32_workspace_bytes(int B);
BSLAM_API int bslam_colorize_f32(const float *d_value, int B, int H, int W, uint8_t *d_rgba, const uint8_t *d_lut,
                                 double p_lo, double p_hi, int has_invalid, float invalid_val, uint32_t bg_rgba,
                                 const double *h_vmin_vmax, double *d_vmin_vmax_out, void *d_workspace,
                                 bslam_stream_t stream);

/* min/max-normalised 8-bit depth, `np.uint8(255*(d-min)/(max-min))`, of
 * N/3DM/slam_utils.py:250-264 (then coloured through d_lut if d_rgb != NULL: 256*3 bytes,
 * e.g. cv2.COLORMAP_JET in BGR order). d_workspace: bslam_colorize_workspace_bytes(B). */
BSLAM_API int bslam_minmax_u8(const uint16_t *d_u16, int B, int H, int W, uint8_t *d_gray,
                              uint8_t *d_rgb, const uint8_t *d_lut3, void *d_workspace,
                              bslam_stream_t stream);

/* median of a u16 image set through the same histogram machinery; used for
 * compute_median_scale_factor (N/EVALUATION/MDEM_eval.py:114-127). d_out: DEVICE [B] f64. */
BSLAM_API int bslam_median_u16(const uint16_t *d_u16, int B, int64_t n_per_image, int has_invalid,
                               uint16_t invalid_val, double *d_out, void *d_workspace,
                               bslam_stream_t stream);

/* ------------------------------------------------------------------ 3DM depth scaling (a4)
 * Replaces Open3D RGBDImage.create_from_color_and_depth(depth_scale, depth_trunc) as called at
 * N/3DM/slam_utils.py:212-220:  d = (float)u16 / (float)depth_scale;  d >= depth_trunc -> 0.
 * depth_trunc <= 0 disables truncation (the cv2 variant, slam_utils.py:231-233). */
BSLAM_API int bslam_depth_from_u16(const uint16_t *d_in, int64_t n, float depth_scale,
                                   float depth_trunc, float *d_out, bslam_stream_t stream);

/* Host helper: n row-major 4x4 float64 matrices inverted by the cofactor (adjugate / determinant) formula, the one
 * Eigen's Matrix4d::inverse() evaluates for Open3D's `extrinsic.inverse()` -- the camera pose of back-projection and
 * unit activation.  No device work. */
BSLAM_API int bslam_invert4x4(const double *h_in, double *h_out, int n);

/* ------------------------------------------------------------------ back-projection (K2)
 * Replaces `pixel_to_3d` N/3DM/scaling_system.py:72-77 applied densely, i.e. Open3D
 * PointCloud.create_from_depth_image / create_from_rgbd_image(depth, intrinsic, extrinsic)
 * as called at N/3DM/mapping_module.py:37,41,42,173:
 *   z = d; x = (u-cx)*z/fx; y = (v-cy)*z/fy; p = cam_to_world * [x,y,z,1]  for d > 0,
 * rows visited with step `stride`, output compacted in row-major order per image.
 * h_K = {fx,fy,cx,cy} (f32, HOST); h_cam_to_world = [B][12] f32 row-major 3x4 (HOST;
 * inverse(extrinsic), computed by the caller in f64).  valid_only == 0 writes one row per
 * visited pixel (NaN for d <= 0) and no compaction happens.
 * d_xyz [capacity][3] f32; d_rgb optional [capacity][3] f32 = u8/255 (needs d_rgb_u8 [B][H][W][3]);
 * d_counts DEVICE [B+1] i64: rows per image and, last, the total.  Images are concatenated.
 * Rows beyond `capacity` are counted but not written (BSLAM_E_CAPACITY is NOT raised; compare). */
BSLAM_API size_t bslam_backproject_workspace_bytes(int B, int H, int W, int stride);
BSLAM_API int bslam_backproject(const float *d_depth, const uint8_t *d_rgb_u8, int B, int H, int W,
                                int stride, const float *h_K, const float *h_cam_to_world,
                                int valid_only, float *d_xyz, float *d_rgb, int64_t capacity,
                                int64_t *d_counts, void *d_workspace, bslam_stream_t stream);

/* ------------------------------------------------------------------ TSDF volume (K3)
 * Replaces `TSDF.__init__` N/3DM/tsdf.py:6-12 for the dense N^3 equivalent of the volume it
 * builds (Open3D UniformTSDFVolume semantics; box of nx*ny*nz voxels whose local z = 0 is
 * global plane gz0 of a larger grid -- z-slab sharding).  World centre of global voxel
 * (X,Y,Z) = origin + (X+.5, Y+.5, Z+.5)*voxel_length.  Storage is brick-ordered
 * (8x8x8 bricks, {tsdf,weight} float2 per voxel, optional f32 rgb planes).
 * d_storage: optional caller-owned device buffer of bslam_tsdf_storage_bytes(); NULL lets the
 * library cudaMalloc on `device`. */
BSLAM_API size_t bslam_tsdf_storage_bytes(int nx, int ny, int nz, int with_color);
BSLAM_API int bslam_tsdf_create(bslam_volume **out, int nx, int ny, int nz, int gz0,
                                double voxel_length, double sdf_trunc, const double *h_origin,
                                int with_color, int device, void *d_storage, bslam_stream_t stream);
BSLAM_API int bslam_tsdf_destroy(bslam_volume *vol);
BSLAM_API int bslam_tsdf_reset(bslam_volume *vol, bslam_stream_t stream);
/* deepcopy of N/3DM/tsdf.py:24 (build_copy_3D_map): dst must have identical geometry */
BSLAM_API int bslam_tsdf_copy(const bslam_volume *src, bslam_volume *dst, bslam_stream_t stream);

/*
 * Replaces `TSDF.build_3D_map(rgbd, intrinsic, extrinsic)` N/3DM/tsdf.py:14-22 (Open3D
 * integrate) for F frames in order (F = 1: the per-frame SLAM loop N/3DM/slam.py:117,179;
 * F > 1: the replay of `update_map_after_pg` N/3DM/slam_utils.py:124-135).
 * d_depth [F][H][W] f32 metres (0 = invalid); d_rgb optional [F][H][W][3] u8 (colour volumes; read
 * through the aligned 32-bit words that hold a pixel's bytes, so up to 3 bytes either side of the
 * buffer are touched -- inside the allocation granule of any CUDA allocator);
 * h_K = {fx,fy,cx,cy} f64 HOST; h_extrinsics [F][16] f64 HOST row-major world->camera.
 * zmarch: BSLAM_ZMARCH_BRICK (fast path) or BSLAM_ZMARCH_LITERAL (validation kernel).
 * d_update_counts: optional DEVICE [F] u64, += number of voxels updated per frame.
 * dry_run != 0 only counts (volume untouched).
 */
BSLAM_API int bslam_tsdf_integrate(bslam_volume *vol, const float *d_depth, const uint8_t *d_rgb,
                                   int F, int H, int W, const double *h_K,
                                   const double *h_extrinsics, int zmarch,
                                   unsigned long long *d_update_counts, int dry_run,
                                   bslam_stream_t stream);

/*
 * The replay shape of `update_map_after_pg` (N/3DM/slam_utils.py:124-135) with the frames as they
 * come off the PNG decoder: uint16 depth in 3DM units.  Fuses `RGBD._read_rgbd_for_tsdf`'s depth
 * conversion (N/3DM/slam_utils.py:212-220: f32(u16) / depth_scale, >= depth_trunc -> 0) into the
 * first pass of the integration; d_depth_scratch [F][H][W] f32 receives the converted frames
 * (what bslam_depth_from_u16 would have produced) and must stay valid until the call's work is done.
 */
BSLAM_API int bslam_tsdf_integrate_u16(bslam_volume *vol, const uint16_t *d_depth_u16, float depth_scale,
                                       float depth_trunc, float *d_depth_scratch, const uint8_t *d_rgb,
                                       int F, int H, int W, const double *h_K, const double *h_extrinsics,
                                       unsigned long long *d_update_counts, bslam_stream_t stream);

/*
 * The same launch in two halves, for callers that stream chunk after chunk (update_map_after_pg-style replays):
 * bslam_tsdf_prepare_u16 enqueues everything that does not touch the volume -- depth conversion + tile statistics,
 * unit marks, culling, claim order -- for F <= BSLAM_MAX_BATCH frames on `prep_stream`;
 * bslam_tsdf_integrate_prepared enqueues the integration of the OLDEST prepared launch on `stream` (it waits for
 * the preparation through an event; no host synchronisation).  Up to two launches may be prepared ahead, so that the
 * preparation of chunk k+1 runs in the SM slots the tail of chunk k's integration leaves idle.  Frame order =
 * preparation order.  The buffers handed to prepare must stay valid until the matching integration is done.
 */
BSLAM_API int bslam_tsdf_prepare_u16(bslam_volume *vol, const uint16_t *d_depth_u16, float depth_scale, float depth_trunc,
                                     float *d_depth_scratch, int F, int H, int W, const double *h_K, const double *h_extrinsics,
                                     bslam_stream_t prep_stream);
BSLAM_API int bslam_tsdf_integrate_prepared(bslam_volume *vol, const uint8_t *d_rgb, unsigned long long *d_update_counts,
                                            bslam_stream_t stream);

/* Round-robin z-sharding: this box holds every `stride_bricks`-th 8-voxel brick layer of the
 * grid, starting at global plane gz0 (= 8 * rank): local plane z is global plane
 * gz0 + (z / 8) * 8 * stride_bricks + z % 8.  Balances integration across ranks whatever the
 * camera looks at; extraction needs contiguous slabs again (re-shard brick layers first, see
 * bodyslam_b200/sharding.py).  stride_bricks = 1 (default) is a contiguous slab. */
BSLAM_API int bslam_tsdf_set_z_interleave(bslam_volume *vol, int stride_bricks);
/* byte offsets {voxels, colour, brick flags, total} inside the storage buffer; a brick layer
 * (all bricks of one bz) is contiguous in each region, which is what re-sharding moves */
BSLAM_API int bslam_tsdf_layout(const bslam_volume *vol, size_t *h_offsets /* [4] */);

/* frames per integrate launch (1..BSLAM_MAX_BATCH, 0 = library default).  Larger batches keep a
 * voxel in registers across more frames; smaller ones keep the batch's depth images L2-resident. */
BSLAM_API int bslam_tsdf_set_batch(bslam_volume *vol, int frames_per_launch);

/*
 * ScalableTSDFVolume semantics -- the volume `TSDF.__init__` literally constructs (N/3DM/tsdf.py:7-12:
 * volume_unit_resolution = 32, depth_sampling_stride = 8).  With unit_resolution > 0 a frame only
 * integrates the unit_resolution^3-voxel units activated by its stride-sampled, back-projected
 * depth points (+- sdf_trunc), and voxel centres are evaluated per unit like Open3D's per-unit
 * UniformTSDFVolume; everything else stays weight 0 exactly like the sparse reference.  The grid
 * must consist of whole units on the world unit grid (origin = k * unit_resolution * voxel_length);
 * z_total: plane count of the whole grid when this volume is a z-shard (0 = nz).  0 switches back
 * to the dense UniformTSDFVolume semantics (default).
 * depth_sampling_stride = -1: "dense with the reference's arithmetic" -- EVERY unit of the box is integrated by every
 * frame (no activation mask), with the per-unit voxel centres and the per-unit float32 z recurrence; on the voxels of
 * the units ScalableTSDFVolume would have activated the result equals the reference's bit for bit.
 */
BSLAM_API int bslam_tsdf_set_unit_activation(bslam_volume *vol, int unit_resolution, int depth_sampling_stride, int z_total);

/* The reference's ScalableTSDFVolume is unbounded; this box is not.  Every integrated frame's
 * stride-sampled depth points (the same sampling ScalableTSDFVolume::Integrate uses) are
 * back-projected and counted: h_stat3 = {points seen, points whose +-sdf_trunc neighbourhood lies
 * entirely outside the box, points partly outside}.  Always on in unit-activation mode; in dense
 * mode bslam_tsdf_set_clip_check(vol, stride > 0, z_total) turns it on (one extra small kernel per
 * launch; z_total = planes of the whole grid when this box is a z-shard, 0 = gz0 + nz).
 * bslam_tsdf_clip_stats synchronises the stream. */
BSLAM_API int bslam_tsdf_set_clip_check(bslam_volume *vol, int sampling_stride, int z_total);
BSLAM_API int bslam_tsdf_clip_stats(bslam_volume *vol, unsigned long long *h_stat3, int reset, bslam_stream_t stream);

/* Chain-length histogram of the last integrate launch: h_hist32[k] = active bricks with 8k+1 .. 8k+8
 * active frames (measurement aid; synchronises). */
BSLAM_API int bslam_tsdf_chain_histogram(bslam_volume *vol, unsigned int *h_hist32, bslam_stream_t stream);

/* z layers per integrate warp: a brick's 8 layers are shared by 2 * 8 / n warps.  8 is the most
 * instruction-efficient; 4 / 2 shorten the serial frame chain of a brick, which bounds the launch
 * time on small shards (8 GPUs).  0 (default) = chosen from the shard's brick count. */
BSLAM_API int bslam_tsdf_set_z_split(bslam_volume *vol, int z_layers_per_warp);

/* Culling statistics accumulated by dry runs (bslam_tsdf_integrate with dry_run = 1) since the last
 * reset: h_stat5 = {(warp, frame) pairs tested, pairs with a voxel projecting into the image, pairs
 * with an updated voxel, voxels tested, free pairs (the cull proved every update has t == 1)}.
 * Measurement aid for DESIGN.md / bench.py; synchronises. */
BSLAM_API int bslam_tsdf_dry_stats(bslam_volume *vol, unsigned long long *h_stat5, int reset, bslam_stream_t stream);

/* Device self-test: n random operand triples through the kernels' shared-reciprocal division and
 * magic-number floor, compared with IEEE `/` and (int) casts; returns the number of mismatches
 * (must be 0).  Synchronises the stream. */
BSLAM_API int bslam_selftest(unsigned long long n, unsigned int seed, unsigned long long *h_mismatches,
                             bslam_stream_t stream);

/* Measurement hook (bench.py roofline): when enabled, the dominant kernel of every integrate
 * launch (brick_integrate_kernel) is bracketed by CUDA events on the launch stream.  Up to 1024
 * launches are buffered between reads; bslam_tsdf_profile_read synchronises on them and returns
 * the accumulated kernel milliseconds and launch count since bslam_tsdf_profile(vol, 1). */
BSLAM_API int bslam_tsdf_profile(bslam_volume *vol, int enable);
BSLAM_API int bslam_tsdf_profile_read(bslam_volume *vol, double *h_ms_total, long long *h_launches);
/* the same events, per stage of a launch: h_ms_stage3 = {depth statistics (+ fused a4), unit marks + culls + claim
 * order, brick_integrate_kernel} accumulated milliseconds (the timeline of one integrate launch) */
BSLAM_API int bslam_tsdf_profile_read_stages(bslam_volume *vol, double *h_ms_stage3, long long *h_launches);

/* brick order <-> Open3D order idx = (x*ny + y)*nz + z (parity / interchange).
 * d_color: [nx*ny*nz*3] f32 or NULL. */
BSLAM_API int bslam_tsdf_export(const bslam_volume *vol, float *d_tsdf, float *d_weight,
                                float *d_color, bslam_stream_t stream);
BSLAM_API int bslam_tsdf_import(bslam_volume *vol, const float *d_tsdf, const float *d_weight,
                                const float *d_color, bslam_stream_t stream);
/* {tsdf,weight} of local plane z as [nx][ny] float2 (halo exchange between z-slabs) */
BSLAM_API int bslam_tsdf_export_plane(const bslam_volume *vol, int z, float *d_plane_f2,
                                      bslam_stream_t stream);
/* colour of local plane z as [nx][ny][3] f32 in [0,255] (colour volumes): the d_halo_hi_color of the slab below */
BSLAM_API int bslam_tsdf_export_plane_color(const bslam_volume *vol, int z, float *d_plane_rgb,
                                            bslam_stream_t stream);

/* ------------------------------------------------------------------ surface extraction (K4)
 * Replaces `TSDF.extract_mesh()` N/3DM/tsdf.py:42-43 (Open3D extract_triangle_mesh):
 * cubes with any zero-weight corner skipped, Bourke tables, vertices shared per edge
 * (x,y,z,axis), triangles (e0,e2,e1).  Two-phase: count (returns HOST counts; synchronises
 * the stream), then emit into caller buffers.
 * d_halo_lo / d_halo_hi: optional [nx][ny] float2 planes z = -1 / z = nz of the neighbouring
 * slabs (NULL = outside the grid = weight 0).  With d_halo_hi the cubes based at local
 * z = nz-1 are emitted here; vertices on edges owned by plane z = nz are NOT (the upper slab,
 * which receives this slab's top plane as its d_halo_lo, emits them).
 * Vertex numbering is deterministic (brick order, 32-voxel chunk, axis, voxel) but differs
 * from Open3D's serial first-seen order; d_keys (optional, [V][4] i32: x,y,z local,axis) lets
 * callers canonicalise.  Vertex ids in d_tri are local to this box unless the edge is owned
 * by plane z = nz, in which case the id is -(1 + (x*ny + y)*4 + axis) (resolved on gather).
 * d_vertices [cap_v][3] f32 world; d_colors optional [cap_v][3] f32 in [0,1] (colour volumes);
 * d_tri [cap_t][3] i32.  Rows beyond capacity are not written.
 * d_halo_hi_color: [nx][ny][3] f32 colour of the d_halo_hi plane (bslam_tsdf_export_plane_color of the slab above).
 * A vertex on a z-edge from this slab's top plane interpolates its colour with it, as the single-box mesh does.
 * Required when d_halo_hi, d_colors and a colour volume are given; ignored otherwise (NULL). */
BSLAM_API int bslam_mc_count(bslam_volume *vol, const float *d_halo_lo, const float *d_halo_hi,
                             int64_t *h_counts /* [2]: V, T */, bslam_stream_t stream);
BSLAM_API int bslam_mc_emit(bslam_volume *vol, const float *d_halo_lo, const float *d_halo_hi,
                            const float *d_halo_hi_color, float *d_vertices, int32_t *d_keys, float *d_colors, int64_t cap_v,
                            int32_t *d_tri, int64_t cap_t, bslam_stream_t stream);

/* Gather side of the z-slab meshes ("per-slab meshes concatenated on gather", north_star): the slabs' d_keys [V][4]
 * and d_tris [T][3] are concatenated bottom slab first (h_nv / h_nt rows each).  In place: key z becomes global
 * (+ h_z_offsets[s]); triangle corners become global ids (+ the slab's vertex base), and the negative ids
 * -(1 + (x*ny + y)*4 + axis) bslam_mc_emit wrote for vertices owned by the next slab's plane 0 are resolved.
 * d_workspace: bslam_mesh_merge_workspace_bytes().  h_unresolved (optional; synchronises): number of
 * references that found no vertex (must be 0). */
BSLAM_API size_t bslam_mesh_merge_workspace_bytes(int n_slabs, int nx, int ny);
BSLAM_API int bslam_mesh_merge(int n_slabs, const int64_t *h_nv, const int64_t *h_nt, const int32_t *h_z_offsets, int nx, int ny,
                               int32_t *d_keys, int32_t *d_tris, void *d_workspace, int64_t *h_unresolved, bslam_stream_t stream);

/* ------------------------------------------------------------------ tensor-pipeline integrator (row f4)
 * Replaces `MAP.integrate(curr_rgbd, i, curr_global_pose)` N/3DM/tsdf.py:71-83, i.e. Open3D
 * `t.pipelines.slam.Model.integrate(frame, depth_scale, depth_max, trunc_voxel_multiplier)` on a VoxelBlockGrid of
 * 16^3 blocks (`MAP.__init__` N/3DM/tsdf.py:57-69), for F frames in order, on the bounded dense box `vol`
 * (origin on the world block grid: origin = k * 16 * voxel_size; created without unit activation):
 * blocks are activated per frame by the depth-touch rule (every 4th pixel, 4 points along the ray over
 * [d - trunc, d + trunc], trunc = trunc_voxel_multiplier * voxel_size), activated voxels get the PROJECTIVE update
 * sdf = depth - z with the depth_max cut (see csrc/bslam_vbg.cu).  d_depth_u16 [F][H][W] raw depth (divided by
 * depth_scale in the kernel, like Open3D), d_rgb optional [F][H][W][3] u8 (colour volumes), h_poses [F][16] f64
 * camera->world (T_frame_to_model), h_depth_max [F] f64 (`curr_rgbd.depth_max`).  d_workspace:
 * bslam_vbg_workspace_bytes() bytes, ZEROED by the caller once; its first 16 bytes accumulate {ray points
 * seen, ray points outside the box} (bslam_vbg_stats; the reference's hash map is unbounded).
 * The workspace also keeps, across calls, the blocks activated by any frame so far (the VoxelBlockGrid's allocated
 * blocks) and the blocks the last integrated frame activated; bslam_vbg_raycast reads both. */
BSLAM_API size_t bslam_vbg_workspace_bytes(int nx, int ny, int nz);
BSLAM_API int bslam_vbg_integrate(bslam_volume *vol, const uint16_t *d_depth_u16, const uint8_t *d_rgb, int F, int H, int W,
                                  const double *h_K, const double *h_poses, const double *h_depth_max, float depth_scale,
                                  float trunc_voxel_multiplier, void *d_workspace, unsigned long long *d_update_counts,
                                  bslam_stream_t stream);
BSLAM_API int bslam_vbg_stats(const void *d_workspace, unsigned long long *h_stat2, bslam_stream_t stream);
/* ------------------------------------------------------------------ ray casting (row f4)
 * Rendered depth, vertex, normal and colour maps of the volume from a pose: Open3D's tensor RayCast (the semantics,
 * and where they deliberately differ from Open3D, are written down in its CPU reference, tests/raycast_ref.c).  One ray
 * per integer pixel; a ray that finds no zero crossing of valid voxels (weight >= weight_threshold, or != 0 when it
 * is 0) writes zeros.  depth = z in the camera frame * depth_scale; vertex and normal are in the camera frame; colour
 * in [0, 1].  Outputs: d_depth [F][H][W] f32 (required), d_vertex, d_normal, d_color [F][H][W][3] f32 (each optional,
 * NULL = not produced; a colour map needs a colour volume).  The volume is read only.
 *
 * bslam_tsdf_raycast: legacy flavour on a DenseTSDFVolume box (dense, unit-activation or unit-arithmetic mode; dims
 * multiples of 8; not z-sharded or z-interleaved): 8^3 bricks relative to the box origin, brick flag bit 0 as the
 * allocation, voxel-centre trilinear interpolation, sdf_trunc of the volume, ray range [depth_min, depth_max].
 * h_extrinsics [F][16] f64 world -> camera; any F (launched 64 frames at a time). */
BSLAM_API int bslam_tsdf_raycast(bslam_volume *vol, int F, int H, int W, const double *h_K, const double *h_extrinsics, float depth_scale,
                                 float depth_min, float depth_max, float weight_threshold, float *d_depth, float *d_vertex, float *d_normal,
                                 float *d_color, bslam_stream_t stream);
/* The same legacy ray cast over a grid cut into contiguous z-slabs [h_slab_z[k], h_slab_z[k+1]) that live on different
 * devices (ShardedTSDF.raycast); the result equals bslam_tsdf_raycast of the whole grid bit for bit.  h_slab_z: n_slabs + 1
 * increasing global planes, multiples of 8, from 0 to the grid's z (1 <= n_slabs <= 64); vol: one of these slabs
 * (not z-interleaved).  Rays are marched in rounds: a ray's state lives in d_state [F][H][W] int32x4 {t or the hit
 * distance, t_prev, last tsdf, owner slab << 2 | status (1 marching, 2 hit, 3 miss)} followed by one int32, the count of
 * rays handed to another slab in the round.
 * bslam_tsdf_raycast_segment: one round on this slab.  first != 0: d_state is not read (every slab computes each ray's
 * first owner itself).  Writes the state of the rays this slab owned and 0 for all others, so the element-wise int32 sum
 * of every slab's d_state is the next round's input; a sample is marched by the slab holding its brick layer.  Stop
 * when the summed hand-over count is 0; at most n_slabs rounds are needed.
 * bslam_tsdf_raycast_shade: the outputs (as bslam_tsdf_raycast) of the finished rays whose trilinear base plane lies in
 * this slab, 0 for every other pixel, from the summed final state: the int32 sum over the slabs is the full map.
 * d_halo_lo / d_halo_hi: the neighbours' planes, packed as bslam_tsdf_raycast_halo_bytes(neighbour, planes) bytes:
 * `planes` [nx][ny] float2 {tsdf, weight} planes, then (colour volumes) `planes` [nx][ny][3] f32 colour planes, then the
 * [nby][nbx] brick flags of the brick layer that holds them.  d_halo_lo: 1 plane (z0 - 1) of the slab below, d_halo_hi:
 * 2 planes (z1, z1 + 1) of the slab above; each is required exactly when that neighbour exists.  F = 0: NULL buffers are
 * accepted and nothing is launched; any F (64 frames per launch). */
BSLAM_API size_t bslam_tsdf_raycast_halo_bytes(const bslam_volume *vol, int planes);
BSLAM_API int bslam_tsdf_raycast_segment(bslam_volume *vol, int n_slabs, const int *h_slab_z, int first, int F, int H, int W, const double *h_K,
                                         const double *h_extrinsics, float depth_min, float depth_max, float weight_threshold, int32_t *d_state,
                                         bslam_stream_t stream);
BSLAM_API int bslam_tsdf_raycast_shade(bslam_volume *vol, int n_slabs, const int *h_slab_z, const void *d_halo_lo, const void *d_halo_hi, int F,
                                       int H, int W, const double *h_K, const double *h_extrinsics, float depth_scale, const int32_t *d_state,
                                       float *d_depth, float *d_vertex, float *d_normal, float *d_color, bslam_stream_t stream);
/* bslam_vbg_raycast: tensor flavour (`MAP.synthesize_model_frame`) on a volume integrated by bslam_vbg_integrate with
 * the workspace d_vbg_workspace: 16^3 blocks on the world block grid, allocated = activated by any frame so far,
 * voxel-corner trilinear interpolation, sdf_trunc = trunc_voxel_multiplier * voxel_size, ray range from Open3D's
 * EstimateRange (down factor 8) over the blocks the last integrated frame activated.  h_pose [16] f64 camera -> world;
 * H, W >= 8.  d_range_workspace: bslam_vbg_raycast_workspace_bytes(H, W) bytes of device scratch (the range map). */
BSLAM_API size_t bslam_vbg_raycast_workspace_bytes(int H, int W);
BSLAM_API int bslam_vbg_raycast(bslam_volume *vol, const void *d_vbg_workspace, int H, int W, const double *h_K, const double *h_pose,
                                float depth_scale, float depth_min, float depth_max, float weight_threshold, float trunc_voxel_multiplier,
                                float *d_depth, float *d_vertex, float *d_normal, float *d_color, void *d_range_workspace,
                                bslam_stream_t stream);

/* ------------------------------------------------------------------ multi-scale RGB-D odometry (row f4)
 * Open3D's tensor `t.pipelines.odometry.rgbd_odometry_multi_scale` (the reference's `_compute_vo_o3d`,
 * N/3DM/visual_odometry.py:97-120) and `t.pipelines.slam.Model.track_frame_to_model` (the same with the ray-cast model
 * frame as the target): point-to-plane (method 0), intensity (1) and hybrid (2) Gauss-Newton over an image pyramid.
 * The semantics are written down in the CPU reference tests/odometry_ref.c; they are restated from knowledge of Open3D,
 * so parity with Open3D itself is UNPINNED (DESIGN.md section 7 lists the recalled details the reference fixes).
 * Sums are float64 and reduced in a fixed order: the result is bit-reproducible (Open3D uses float32 atomics).
 *
 * Levels: level l is (H >> l) x (W >> l) with intrinsics K / 2^l; every level must be at least 1 x 1 (levels <= 16).
 * h_K: fx, fy, cx, cy (f64) of level 0.
 *
 * bslam_odom_prepare: F frames -> d_frames (F * bslam_odom_frame_bytes(H, W, levels), caller-owned).  d_depth [F][H][W]
 * uint16 (depth_dtype 0) or float32 (1), depth = raw / depth_scale, NaN (invalid) when <= 0 or >= depth_max;
 * d_color NULL or [F][H][W][3] uint8 (color_dtype 0, intensity = (0.299 R + 0.587 G + 0.114 B) / 255) or float32 in
 * [0, 1] (1, no division).  Without colour the intensity is NaN: such frames serve PointToPlane only (the intensity
 * methods find no inlier on them and end singular).  Depth pyramid: PyrDownDepth(2 * depth_outlier_trunc); intensity:
 * 5x5 Gaussian, replicated borders.  Per frame and level (coarser after finer) 12 planes of (H >> l) * (W >> l) f32:
 * depth, intensity, vertex x, y, z, normal x, y, z, Sobel x / y of depth, Sobel x / y of intensity (unscaled 3x3).
 *
 * bslam_odom_track: P pairs {source, target} (h_pairs [P][2], frame indices of d_frames), each from h_init [P][16]
 * (row-major f64, source -> target).  Levels run coarsest first; criteria entry c (h_max_iter / h_rel_fitness /
 * h_rel_rmse [levels]) belongs to level levels - 1 - c.  Outputs: d_T [P][16] f64, d_rmse_fitness [P][2] f64 of the last
 * evaluation, d_iters [P][levels] i32 evaluations per criteria entry, d_status [P] i32 (0 = ok, 1 = a singular 6x6
 * system ended the pair; T is the pose before it).  d_workspace: bslam_odom_workspace_bytes(P, H, W, levels).
 * Enqueues 2 * sum(h_max_iter) launches (+ 1 per 128 pairs); no host synchronisation, no copies.  F <= 65535 frames per
 * bslam_odom_prepare call and P <= 65535 pairs per bslam_odom_track / bslam_odom_linearize call (E_ARG beyond).  P == 0 or F == 0
 * (then P must be 0) launches nothing and accepts NULL outputs.
 *
 * bslam_odom_linearize: the 29 float64 sums of every pair at `level` under h_T [P][16]: d_sums [P][29] = upper
 * triangle of J^T J (row-major, 21), J^T huber'(r) (6), sum of huber(r), inlier count. */
BSLAM_API size_t bslam_odom_frame_bytes(int H, int W, int levels);
BSLAM_API int bslam_odom_prepare(const void *d_depth, int depth_dtype, const void *d_color, int color_dtype, int F, int H, int W, int levels,
                                 const double *h_K, float depth_scale, float depth_max, float depth_outlier_trunc, float *d_frames,
                                 bslam_stream_t stream);
BSLAM_API size_t bslam_odom_workspace_bytes(int P, int H, int W, int levels);
BSLAM_API int bslam_odom_track(const float *d_frames, int F, const int *h_pairs, int P, int H, int W, int levels, const double *h_K, int method,
                               const int *h_max_iter, const double *h_rel_fitness, const double *h_rel_rmse, float depth_outlier_trunc,
                               float depth_huber_delta, float intensity_huber_delta, const double *h_init, double *d_T, double *d_rmse_fitness,
                               int *d_iters, int *d_status, void *d_workspace, bslam_stream_t stream);
BSLAM_API int bslam_odom_linearize(const float *d_frames, int F, const int *h_pairs, int P, int H, int W, int levels, int level, const double *h_K,
                                   int method, float depth_outlier_trunc, float depth_huber_delta, float intensity_huber_delta, const double *h_T,
                                   double *d_sums, void *d_workspace, bslam_stream_t stream);

/* ------------------------------------------------------------------ mesh ray casting
 * Open3D's `t.geometry.RaycastingScene` (`cast_rays(...)["t_hit"]` as a synthetic depth map, N/3DM/
 * synthetic_depth_generator.py:74-97): closest hits of rays against triangle meshes through an LBVH built on the device.
 * The semantics are written down in the brute-force CPU reference tests/mesh_raycast_ref.c, which the GPU equals bit for
 * bit; parity with Open3D / Embree is UNPINNED (DESIGN.md section 7, "Mesh ray cast exactness").
 *
 * bslam_mesh_build: d_verts [n_verts][3] f32 and d_tris [n_tris][3] i32 of every geometry, concatenated; h_geom
 * [n_geoms + 1][2] i64 = {first triangle, first vertex} of each geometry, then {n_tris, n_verts}.  Triangle indices are
 * local to their geometry.  d_bvh: bslam_mesh_bvh_bytes(n_tris) bytes, d_workspace: bslam_mesh_build_workspace_bytes(n_tris,
 * n_geoms) bytes, both caller-owned; the workspace may be freed after the call's work has run.  Indices are validated on
 * the device: the call synchronises the stream once to read the result and returns BSLAM_E_ARG with the geometry and
 * triangle of the first index out of range.  Triangles with a non-finite coordinate or a zero float32 normal are left
 * out of the scene.
 *
 * bslam_mesh_cast_rays: d_rays [n][6] f32 {origin, direction}; outputs [n]: t_hit (+inf on a miss), geometry and
 * primitive ids (0xFFFFFFFF on a miss), optional d_uvs [n][2] (Embree's u, v) and d_normals [n][3] (unit, world frame),
 * 0 on a miss.  bslam_mesh_rays_pinhole: the rays of F pinhole frames (h_K 3x3 row-major f64, h_extrinsics [F][16] f64
 * world -> camera) into d_rays [F][H][W][6]; bslam_mesh_cast_pinhole: the same rays cast without storing them, outputs
 * [F][H][W](...).  n == 0 or F * H * W == 0 launches nothing and accepts NULL buffers. */
BSLAM_API size_t bslam_mesh_bvh_bytes(int64_t n_tris);
BSLAM_API size_t bslam_mesh_build_workspace_bytes(int64_t n_tris, int n_geoms);
BSLAM_API int bslam_mesh_build(const float *d_verts, int64_t n_verts, const int32_t *d_tris, int64_t n_tris, const int64_t *h_geom, int n_geoms,
                               void *d_bvh, void *d_workspace, bslam_stream_t stream);
BSLAM_API int bslam_mesh_cast_rays(const void *d_bvh, const float *d_rays, int64_t n, float *d_t_hit, uint32_t *d_geom_ids, uint32_t *d_prim_ids,
                                   float *d_uvs, float *d_normals, bslam_stream_t stream);
BSLAM_API int bslam_mesh_rays_pinhole(int F, int H, int W, const double *h_K, const double *h_extrinsics, float *d_rays, bslam_stream_t stream);
BSLAM_API int bslam_mesh_cast_pinhole(const void *d_bvh, int F, int H, int W, const double *h_K, const double *h_extrinsics, float *d_t_hit,
                                      uint32_t *d_geom_ids, uint32_t *d_prim_ids, float *d_uvs, float *d_normals, bslam_stream_t stream);

/* Surface-extraction flavour of bslam_mc_* / bslam_points_*: a voxel is valid when weight >= weight_threshold
 * (0 = weight > 0, Open3D's legacy `weight != 0` for every weight an integrator writes: they differ only for negative
 * or NaN weights, which count as invalid here; the tensor pipeline's extract_triangle_mesh / extract_point_cloud default
 * is 3) and vertices sit at (index + vertex_offset) * voxel_length (legacy 0.5 = voxel centres; tensor pipeline 0). */
BSLAM_API int bslam_tsdf_set_extract_flavour(bslam_volume *vol, float weight_threshold, double vertex_offset);

/* Replaces `TSDF.extract_pcd()` N/3DM/tsdf.py:39-40 (Open3D extract_point_cloud): interior
 * voxels with w != 0 and -0.98 <= f < 0.98, sign change towards +x/+y/+z neighbour, linear
 * zero crossing; normals from the 0.99-voxel central difference of the trilinear TSDF.
 * Single-box volumes only (gz0 = 0 and no halos). */
/* Incremental mode for the reference's per-frame cadence (extract_pcd after every build_3D_map, N/3DM/slam.py:126,195):
 * the integration kernels flag the bricks they change; a count / emit pair then re-extracts only the bricks whose 3x3x3
 * brick neighbourhood changed since the previous pair and copies every other brick's points from a per-brick cache
 * (<= 128 points per brick; larger bricks are always recomputed).  Same output, same order as the full extraction.
 * with_normals fixes whether normals are produced (bslam_points_emit must then be given / not given d_normals); colour
 * volumes need d_colors; every bslam_points_emit needs its own bslam_points_count first and room for all points. */
BSLAM_API int bslam_points_set_incremental(bslam_volume *vol, int enable, int with_normals);
/* {surface-candidate bricks, bricks recomputed} of the last bslam_points_count (host values, no synchronisation) */
BSLAM_API int bslam_points_last_stats(const bslam_volume *vol, long long *h_stat2);
BSLAM_API int bslam_points_count(bslam_volume *vol, int64_t *h_count, bslam_stream_t stream);
BSLAM_API int bslam_points_emit(bslam_volume *vol, float *d_points, float *d_normals,
                                float *d_colors, int32_t *d_keys, int64_t cap,
                                bslam_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* BODYSLAM_B200_H */
