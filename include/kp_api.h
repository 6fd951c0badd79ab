/*
 * kp_api.h -- C ABI of libkinectpy_b200.so (sm_100a).
 *
 * Drop-in boundary for the per-frame point-cloud path of tiborcamargo/KinectPy.
 * The reference has no FFI of its own: the path sits behind Python free
 * functions that call Open3D methods (SURVEY.md section 8b).  Each entry point
 * below replaces one such Open3D / k4a routine *at the reference's call site*
 * (cited per function, paths relative to the reference root).  The Python
 * mirror of the reference call surface (kinectpy_b200/preprocessing/*.py,
 * kinectpy_b200/floor_removal.py, kinectpy_b200/utils/io.py) binds these with
 * ctypes; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++ types, no exceptions.
 *   - every function returns 0 (KP_OK) or a negative KP_E_* code;
 *     kp_last_error(ctx) gives the message.
 *   - one kp_ctx per host thread / GPU: it owns one CUDA stream and a
 *     grow-only workspace.  Calls on one ctx are serialised by the caller.
 *   - pointer arguments named d_* are DEVICE pointers, h_* are HOST pointers.
 *     Arrays are caller-owned; outputs are caller-allocated at the documented
 *     upper bound, actual counts come back through int64_t* (host).
 *   - points are float32 [n][3] (x,y,z packed); a point whose x is NaN is
 *     "absent" and is skipped by every operation.
 *   - all decisions (voxel index, neighbour order, inlier tests, masks) are
 *     taken in IEEE double on the float32-stored values, without FMA
 *     contraction, in the operation order documented in DESIGN.md; the CPU
 *     oracle (oracle/kp_oracle.c) uses the same contract.
 *   - there is no CPU fallback: without a CUDA device kp_ctx_create fails.
 */
#ifndef KP_API_H
#define KP_API_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define KP_EXPORT __attribute__((visibility("default")))
#else
#define KP_EXPORT
#endif

typedef struct kp_ctx kp_ctx;

enum {
    KP_OK = 0,
    KP_E_ARG = -1,     /* invalid argument (Open3D raises RuntimeError for the same inputs) */
    KP_E_CUDA = -2,    /* CUDA runtime error; see kp_last_error */
    KP_E_RANGE = -3,   /* grid would overflow the packed key (voxel_size too small for the extent) */
    KP_E_NOMEM = -4,
    KP_E_NODEVICE = -5 /* no CUDA device: there is no CPU path */
};

/* flags for kp_unproject_transform */
enum {
    KP_UNPROJECT_INT16 = 1,        /* k4a rounding: x = (int16)floorf(xt*z + 0.5f) ... (SURVEY.md A.1) */
    KP_UNPROJECT_DROP_ANY_ZERO = 2 /* utils/io.py:36 -- a point with x==0 or y==0 or z==0 is invalid */
};

/* ------------------------------------------------------------- context -- */
KP_EXPORT const char *kp_version(void);
KP_EXPORT int kp_device_count(void);
KP_EXPORT int kp_ctx_create(int device, kp_ctx **out);
KP_EXPORT int kp_ctx_destroy(kp_ctx *ctx);
KP_EXPORT const char *kp_last_error(kp_ctx *ctx);
KP_EXPORT void *kp_ctx_stream(kp_ctx *ctx);            /* cudaStream_t */
KP_EXPORT int kp_sync(kp_ctx *ctx);
KP_EXPORT int kp_malloc(kp_ctx *ctx, size_t bytes, void **d_ptr);
KP_EXPORT int kp_free(kp_ctx *ctx, void *d_ptr);
KP_EXPORT int kp_host_alloc(size_t bytes, void **h_ptr); /* pinned */
KP_EXPORT int kp_host_free(void *h_ptr);
KP_EXPORT int kp_memcpy_h2d(kp_ctx *ctx, void *d_dst, const void *h_src, size_t bytes); /* async on ctx stream */
KP_EXPORT int kp_memcpy_d2h(kp_ctx *ctx, void *h_dst, const void *d_src, size_t bytes); /* returns after completion */
KP_EXPORT int kp_memcpy_d2d(kp_ctx *ctx, void *d_dst, const void *d_src, size_t bytes);
KP_EXPORT int kp_memset(kp_ctx *ctx, void *d_dst, int value, size_t bytes);
KP_EXPORT int kp_timer_start(kp_ctx *ctx);               /* CUDA event on the ctx stream */
KP_EXPORT int kp_timer_stop(kp_ctx *ctx, float *h_ms);   /* records, synchronises, returns elapsed ms */
KP_EXPORT int64_t kp_launch_count(kp_ctx *ctx);          /* kernels launched by this ctx so far */
KP_EXPORT int kp_flush_l2(kp_ctx *ctx);                  /* writes a 256 MiB scratch buffer (bench hygiene) */
/* per-kernel-family device time accumulated since the last reset (needs kp_profile_enable(ctx,1);
 * adds an event pair per launch group, so keep it off in throughput runs) */
KP_EXPORT int kp_profile_enable(kp_ctx *ctx, int on);
KP_EXPORT int kp_profile_read(kp_ctx *ctx, int max_entries, const char **h_names, double *h_ms, int64_t *h_calls,
                              double *h_bytes /* algorithmic bytes, nullable */, int *h_n);
KP_EXPORT int kp_profile_reset(kp_ctx *ctx);

/* -------------------------------------------- K1 unproject + transform -- */
/* Replaces: the k4a depth->XYZ step inside offline_processor.exe whose output
 * utils/io.py:15-20 reads (int16 XYZ mm), the validity rule of
 * utils/io.py:36, PointCloud.transform at preprocessing/data.py:46-48 and the
 * np.vstack fusion at preprocessing/data.py:55-58 (sensor-major order).
 *   d_depth  uint16 [B][S][P]   depth in mm, 0 = no return
 *   d_xytab  float32 [S][P][2]  calibration table, NaN = outside FOV
 *   h_T      float64 [S][16]    row-major 4x4 T_master<-sensor, NULL = identity
 *   scale    output unit per mm (1e-3 -> metres, 1.0 -> millimetres)
 *   d_xyz    float32 [B][S*P][3] out; invalid pixels -> NaN,NaN,NaN
 *   d_valid  uint8 [B][S*P] out, nullable
 *   d_xyz16  int16 [B][S*P][3] out, nullable: the `_depth.dat` layout (needs KP_UNPROJECT_INT16)
 *   d_bounds float32 [B][6] out, nullable: min xyz, max xyz over valid points
 *   d_nvalid int32 [B] out, nullable */
KP_EXPORT int kp_unproject_transform(kp_ctx *ctx, const uint16_t *d_depth, const float *d_xytab,
                                     const double *h_T, int B, int S, int64_t P, int flags,
                                     double scale, float *d_xyz, uint8_t *d_valid, int16_t *d_xyz16,
                                     float *d_bounds, int32_t *d_nvalid);

/* Replaces utils/io.py:29-41 (rgbd_to_pointcloud on an int16 `_depth.dat`
 * buffer): int16 [n][3] -> float32 points (value * scale), the any-zero rule
 * (flags & KP_UNPROJECT_DROP_ANY_ZERO), optional extrinsic.  d_keep uint8 [n]
 * nullable: extra per-pixel keep mask AND-ed in (the human crop of
 * preprocessing/data.py:169-175). */
KP_EXPORT int kp_points_from_xyz16(kp_ctx *ctx, const int16_t *d_xyz16, int64_t n, const double *h_T,
                                   int flags, double scale, const uint8_t *d_keep, float *d_xyz,
                                   uint8_t *d_valid);

/* preprocessing/data.py:165-178 human crop mask: pixel non-black in all three
 * channels AND z <= median(z) + gate (median over ALL n int16 z values incl.
 * zeros, numpy semantics: mean of the two middle values for even n).
 * d_rgb uint8 [n][3]; d_keep uint8 [n] out; h_median out nullable. */
KP_EXPORT int kp_crop_mask(kp_ctx *ctx, const uint8_t *d_rgb, const int16_t *d_xyz16, int64_t n,
                           double gate, uint8_t *d_keep, double *h_median);

/* PointCloud.transform (preprocessing/data.py:46-48; SURVEY.md A.8), in place.
 * rotate_only != 0 applies only the 3x3 block (normals). */
KP_EXPORT int kp_transform_points(kp_ctx *ctx, float *d_xyz, int64_t n, const double *h_T16, int rotate_only);

/* min/max over non-NaN points: h_bounds float32[6], h_nvalid nullable */
KP_EXPORT int kp_bounds(kp_ctx *ctx, const float *d_xyz, int64_t n, float *h_bounds, int64_t *h_nvalid);

/* Ordered stream compaction = SelectByIndex on a mask (SURVEY.md A.9;
 * floor_removal.py:50,69,71,72; utils/io.py:37-38).  Keeps row i iff
 * (d_mask ? d_mask[i] != invert : !isnan(x_i)).  Up to three float32 [n][3]
 * attribute arrays ride along (points, colours, normals; any may be NULL).
 * d_index_out int32 [n] nullable receives the kept original indices. */
KP_EXPORT int kp_compact(kp_ctx *ctx, int64_t n, const uint8_t *d_mask, int invert,
                         const float *d_a0, float *d_a0_out, const float *d_a1, float *d_a1_out,
                         const float *d_a2, float *d_a2_out, int32_t *d_index_out, int64_t *h_count);

/* ------------------------------------------------ K2 voxel downsample -- */
/* Replaces PointCloud.voxel_down_sample at preprocessing/filtering.py:23,
 * preprocessing/registration.py:8,100-101, utils/processing.py:308
 * (SURVEY.md A.2).  Radix sort on packed (ix,iy,iz) keys + segmented mean.
 * Output voxels are ordered by (ix,iy,iz); inside a voxel points are summed in
 * input order in double.  Outputs sized for n rows.
 *   d_colors/d_normals nullable; normals are averaged then normalised
 *   d_ijk   int32 [n][3] nullable: voxel index of each OUTPUT row
 *   d_point_voxel int32 [n] nullable: output row of each INPUT point (-1 for NaN)
 *   h_min_bound double[3] nullable: the grid origin used (min - voxel/2) */
KP_EXPORT int kp_voxel_downsample(kp_ctx *ctx, const float *d_xyz, const float *d_colors,
                                  const float *d_normals, int64_t n, double voxel_size,
                                  float *d_xyz_out, float *d_colors_out, float *d_normals_out,
                                  int32_t *d_ijk, int32_t *d_point_voxel, double *h_min_bound,
                                  int64_t *h_m);

/* --------------------------------------------- K3 neighbour search ----- */
/* Uniform-grid spatial hash; exact; canonical (d^2, index) order.
 * Replaces the nanoflann KD-tree queries under remove_statistical_outlier,
 * estimate_normals and registration_icp.
 *   d_queries NULL -> the cloud queries itself (self is then its own first neighbour)
 *   radius > 0 -> hybrid search: at most k neighbours with d^2 < radius^2 (strict)
 *   cell_hint  > 0 -> grid cell edge to use (0 = choose from the data)
 *   d_idx int32 [nq][k] (-1 padded), d_d2 float64 [nq][k] nullable (+inf padded),
 *   d_count int32 [nq] nullable */
KP_EXPORT int kp_knn(kp_ctx *ctx, const float *d_xyz, int64_t n, const float *d_queries, int64_t nq,
                     int k, double radius, double cell_hint, int32_t *d_idx, double *d_d2,
                     int32_t *d_count);

/* PointCloud.remove_statistical_outlier at preprocessing/filtering.py:24,
 * floor_removal.py:73, utils/processing.py:309 (SURVEY.md A.3).
 *   d_keep uint8 [n] out; d_mean float64 [n] nullable out;
 *   h_stats double[3] nullable = {mu, std, threshold}; h_kept = #kept */
KP_EXPORT int kp_sor_mask(kp_ctx *ctx, const float *d_xyz, int64_t n, int nb_neighbors,
                          double std_ratio, double cell_hint, uint8_t *d_keep, double *d_mean,
                          double *h_stats, int64_t *h_kept);

/* PointCloud.remove_radius_outlier (north-star scope; no reference call site;
 * SURVEY.md A.4): keep iff #{j: d^2 < r^2, incl. self} > nb_points. */
KP_EXPORT int kp_radius_mask(kp_ctx *ctx, const float *d_xyz, int64_t n, int nb_points, double radius,
                             uint8_t *d_keep, int32_t *d_counts, int64_t *h_kept);

/* PointCloud.estimate_normals(KDTreeSearchParamHybrid(radius, max_nn)) at
 * preprocessing/registration.py:11-13,103-106 (SURVEY.md A.6).  radius <= 0
 * -> pure kNN(max_nn).  Normals are unoriented (sign arbitrary). */
KP_EXPORT int kp_estimate_normals(kp_ctx *ctx, const float *d_xyz, int64_t n, double radius, int max_nn,
                                  float *d_normals);

/* ------------------------------------------------------- K4 RANSAC ----- */
/* PointCloud.segment_plane at floor_removal.py:70 (SURVEY.md A.5).
 * Hypothesis h draws ransac_n distinct indices kp_rng(seed,h,j) % n (j=0,1,..,
 * repeats rejected); all hypotheses are scored in one batch, then the
 * sequential best / early-exit rule is replayed.
 *   h_plane double[4]: refit plane; d_inlier_mask uint8 [n]: inliers of the
 *   best (pre-refit) plane; h_best_iter nullable; d_counts int64 [iters] nullable */
KP_EXPORT int kp_ransac_plane(kp_ctx *ctx, const float *d_xyz, int64_t n, double distance_threshold,
                              int ransac_n, int num_iterations, double probability, uint64_t seed,
                              double *h_plane, uint8_t *d_inlier_mask, int64_t *h_ninliers,
                              int32_t *h_best_iter, int64_t *d_counts);

/* pcd_above_plane (floor_removal.py:39-51): mask[i] = a*x+b*y+c*z+d < 0 */
KP_EXPORT int kp_plane_side_mask(kp_ctx *ctx, const float *d_xyz, int64_t n, double a, double b,
                                 double c, double d, uint8_t *d_mask, int64_t *h_kept);

/* floor band (floor_removal.py:64-66): lower[i] = coord[axis] >= max(coord[axis]) - band */
KP_EXPORT int kp_band_mask(kp_ctx *ctx, const float *d_xyz, int64_t n, int axis, double band,
                           uint8_t *d_lower, double *h_axis_max, int64_t *h_nlower);

/* ---------------------------------------------------------- K5 ICP ----- */
/* registration_icp(source, target, max_corr, init,
 * TransformationEstimationPointToPlane()) at preprocessing/registration.py:78-84
 * (SURVEY.md A.7).  All iterations run on the device (no host round trip per
 * iteration).  h_T_out double[16] row-major. */
KP_EXPORT int kp_icp_point_to_plane(kp_ctx *ctx, const float *d_src, int64_t n_src, const float *d_tgt,
                                    const float *d_tgt_normals, int64_t n_tgt, double max_corr,
                                    const double *h_init16, int max_iter, double rel_fitness,
                                    double rel_rmse, double *h_T_out, double *h_fitness,
                                    double *h_rmse, int *h_iters, int64_t *h_ncorr);

/* registration_icp(..., TransformationEstimationPointToPoint()) at
 * manual_pointcloud_registration.py:90-98: same loop, the update is Eigen::umeyama (no scaling) over
 * the correspondences. */
KP_EXPORT int kp_icp_point_to_point(kp_ctx *ctx, const float *d_src, int64_t n_src, const float *d_tgt,
                                    int64_t n_tgt, double max_corr, const double *h_init16, int max_iter,
                                    double rel_fitness, double rel_rmse, double *h_T_out, double *h_fitness,
                                    double *h_rmse, int *h_iters, int64_t *h_ncorr);
/* registration_colored_icp(source, target, max_corr, init, TransformationEstimationForColoredICP(),
 * criteria) at preprocessing/registration.py:108-113: the target's tangent-plane colour gradients
 * (hybrid search, radius 2 * max_corr, 30 nn), then the ICP loop with one geometric and one
 * photometric row per correspondence, weights sqrt(lambda) / sqrt(1 - lambda) (Open3D default 0.968).
 * Colours are float32 [n][3] in [0, 1]. */
KP_EXPORT int kp_icp_colored(kp_ctx *ctx, const float *d_src, const float *d_src_colors, int64_t n_src,
                             const float *d_tgt, const float *d_tgt_colors, const float *d_tgt_normals,
                             int64_t n_tgt, double max_corr, double lambda_geometric, const double *h_init16,
                             int max_iter, double rel_fitness, double rel_rmse, double *h_T_out,
                             double *h_fitness, double *h_rmse, int *h_iters, int64_t *h_ncorr);
/* the colour gradients alone (d_grad float32 [n][3]); exported for the parity tests */
KP_EXPORT int kp_color_gradient(kp_ctx *ctx, const float *d_xyz, const float *d_colors, const float *d_normals,
                                int64_t n, double radius, int max_nn, float *d_grad);

/* ---------------------------------------------- global registration ----- */
/* compute_fpfh_feature(pcd, KDTreeSearchParamHybrid(radius, max_nn)) at
 * preprocessing/registration.py:17-20: 33-bin FPFH per point (SPFH of the Darboux angles over the hybrid
 * neighbourhood, then the 1/d^2-weighted blend of the neighbours' SPFHs plus the point's own).
 * d_feat float64 [n][33] (Open3D stores the transpose, 33 x n). */
KP_EXPORT int kp_fpfh(kp_ctx *ctx, const float *d_xyz, const float *d_normals, int64_t n, double radius,
                      int max_nn, double *d_feat);
/* Exact nearest neighbour of every feature a_i among the features b (squared L2 in double, summed in
 * dimension order; ties to the lower index): the two KD-tree searches inside
 * registration_ransac_based_on_feature_matching (preprocessing/registration.py:50).  dim must be 33.
 * d_nn int32 [na]; d_nn_d2 float64 [na] nullable. */
KP_EXPORT int kp_feature_match(kp_ctx *ctx, const double *d_feat_a, int64_t na, const double *d_feat_b,
                               int64_t nb, int dim, int32_t *d_nn, double *d_nn_d2);
/* RegistrationRANSACBasedOnCorrespondence, the second half of
 * registration_ransac_based_on_feature_matching (preprocessing/registration.py:50-57) with
 * TransformationEstimationPointToPoint(False), CorrespondenceCheckerBasedOnEdgeLength(edge_similarity),
 * CorrespondenceCheckerBasedOnDistance(distance_threshold) and RANSACConvergenceCriteria(max_iteration,
 * confidence).  Hypothesis h samples correspondence kp_rng(seed, h, j) % m for j < ransac_n (with
 * replacement).  d_corres int32 [m][2] = (source index, target index).  h_T16 row-major 4x4 (identity
 * when nothing validates); h_best_iter = hypothesis that won (-1 if none); h_validated = hypotheses that
 * passed the checkers. */
KP_EXPORT int kp_ransac_correspondence(kp_ctx *ctx, const float *d_src, int64_t n_src, const float *d_tgt,
                                       int64_t n_tgt, const int32_t *d_corres, int64_t m, double max_corr,
                                       int ransac_n, double edge_similarity, double distance_threshold,
                                       int max_iteration, double confidence, uint64_t seed, double *h_T16,
                                       double *h_fitness, double *h_rmse, int32_t *h_best_iter,
                                       int64_t *h_validated);

/* ----------------------------------------------------- K6 resample ----- */
/* Fixed-N resampling feeding PointNet (BASELINE config C5).
 *   KP_RESAMPLE_RANDOM: select_points_randomly (utils/processing.py:259-275,
 *     np.random.choice(n, N, replace=False); call site datasets/kinect_dataset.py:103-104).
 *     The subset is the N points with the smallest (key, index), key =
 *     min(kp_rng(seed, stream, i) >> 32, 2^32-2), in that order.  N > #valid points
 *     -> KP_E_ARG (numpy raises ValueError).
 *   KP_RESAMPLE_PREFIX: points[:N] (datasets/kinect_dataset_npz.py:96-97); h_count = min(n, N).
 *   d_out float32 [N][3]; d_index_out int32 [N] nullable (RANDOM only). */
enum { KP_RESAMPLE_RANDOM = 0, KP_RESAMPLE_PREFIX = 1 };
KP_EXPORT int kp_resample_fixed_n(kp_ctx *ctx, const float *d_xyz, int64_t n, int64_t N, int mode,
                                  uint64_t seed, uint64_t stream, float *d_out, int32_t *d_index_out,
                                  int64_t *h_count);
/* CSR batch: cloud b = rows h_offsets[b] .. h_offsets[b+1] of d_xyz, sample stream first_stream + b;
 * d_out float32 [B][N][3] (the tensor models/pointnet.py:65 consumes); short PREFIX clouds are
 * zero-padded; h_counts int64 [B] nullable. */
KP_EXPORT int kp_resample_batch(kp_ctx *ctx, const float *d_xyz, const int64_t *h_offsets, int B, int64_t N,
                                int mode, uint64_t seed, uint64_t first_stream, float *d_out,
                                int64_t *h_counts);

/* ------------------------------------------------ whole-frame driver --- */
/* Batched, device-driven driver for BASELINE config C4: per frame unproject ->
 * transform -> fuse -> voxel -> SOR [-> radius outlier removal] -> floor removal (band + RANSAC + merge +
 * SOR) -> ICP refinement of every sub extrinsic (the per-frame body of
 * preprocessing/data.py:35-69 followed by floor_removal.py:57-73 and
 * preprocessing/registration.py:65-86).  Frames are processed in batches of B
 * frames per kernel launch; every intermediate count stays on the device, so a
 * batch is one static launch sequence (a CUDA graph) issued by ONE host thread
 * with no host round trip; W batch slots are in flight at a time. */
typedef struct kp_pipeline kp_pipeline;
typedef struct {
    int32_t S;              /* sensors, sensor 0 = master */
    int64_t P;              /* pixels per sensor */
    int32_t unproject_flags;
    double scale;           /* output unit per mm */
    double voxel_size;      /* fused-cloud voxel (filter_outliers) */
    int32_t sor_k;          double sor_ratio;
    int32_t do_floor;       double floor_band; double ransac_thr; int32_t ransac_n; int32_t ransac_iters;
    int32_t floor_sor_k;    double floor_sor_ratio;
    int32_t do_icp;         double icp_voxel; double icp_max_corr; int32_t icp_max_iter;
    int32_t normals_max_nn; double normals_radius;
    uint64_t seed;
    int32_t n_streams;      /* frames in flight = B frames per launch x W batch slots (no worker threads) */
    /* human crop (preprocessing/data.py:165-178), fused cloud only: a pixel is kept iff its segmentation colour is
     * non-black in all three channels and z16 <= median(z16) + crop_gate, z16 = the int16 z of `_depth.dat` (0 outside
     * the table), median over all P pixels of the (frame, sensor), crop_gate in millimetres whatever `scale` is.
     * The ICP inputs are not cropped. */
    int32_t do_crop;        double crop_gate;
    /* fixed-N output (kp_resample_batch on each frame's final cloud, stream = frame id): 0 = off, else 1..16384 */
    int32_t resample_n;     int32_t resample_mode;   /* KP_RESAMPLE_RANDOM / KP_RESAMPLE_PREFIX */
    /* radius outlier removal (remove_radius_outlier) of the fused cloud after its SOR (after the voxel downsample when
     * sor_k = 0), before floor removal: a point is kept iff more than ror_nb_points points (itself included) lie at
     * d^2 < ror_radius^2, d^2 in double on the float32 coordinates; survivors keep their order.  Its output replaces the
     * SOR output downstream; n_sor still counts the SOR survivors.  ror_nb_points = 0: off; else ror_radius > 0, in the
     * cloud's unit (it follows `scale`, like voxel_size).  The ICP inputs are not filtered. */
    int32_t ror_nb_points;  double ror_radius;
} kp_pipeline_cfg;
typedef struct {
    int64_t n_fused, n_voxel, n_sor, n_floor_inliers, n_out;
    double icp_T[5][16];    /* refined T_master<-sub_i, i = 1..S-1 */
    double icp_fitness[5], icp_rmse[5];
    int32_t icp_iters[5];
    int32_t status;
} kp_frame_result;
KP_EXPORT int kp_pipeline_create(int device, const kp_pipeline_cfg *cfg, const float *h_xytab,
                                 const double *h_T, kp_pipeline **out);
KP_EXPORT int kp_pipeline_destroy(kp_pipeline *p);
KP_EXPORT const char *kp_pipeline_last_error(kp_pipeline *p);
/* depth uint16 [F][S][P]; depth_on_device != 0 -> device pointer (value leg),
 * else host pointer (e2e leg: H2D inside).  h_results [F].  d_out_xyz nullable
 * float32 [F][out_stride][3] device buffer receiving each frame's final cloud
 * (rows beyond n_out are left untouched).  A frame whose final cloud has more
 * than out_stride rows is copied up to out_stride rows, its status and the
 * call's return value are KP_E_RANGE. */
KP_EXPORT int kp_pipeline_run(kp_pipeline *p, const uint16_t *depth, int depth_on_device, int64_t F,
                              kp_frame_result *h_results, float *d_out_xyz, int64_t out_stride);
/* e2e form: as kp_pipeline_run with host depth, and each frame's final cloud is written to the
 * PINNED host buffer (kp_host_alloc) h_out_xyz float32 [F][out_stride][3] (first n_out rows of each
 * frame) by a device kernel: the row counts never visit the host before the copy. */
KP_EXPORT int kp_pipeline_run_host(kp_pipeline *p, const uint16_t *h_depth, int64_t F, kp_frame_result *h_results,
                                   float *h_out_xyz, int64_t out_stride);
/* the general form.  rgb uint8 [F][S][P][3] segmentation images in the same memory space as depth: required when
 * the pipeline crops, refused otherwise (KP_E_ARG).  h_frame_ids int64 [F] nullable (default f): the sample stream of
 * frame f's fixed-N slot, so that a frame gives the same slot whichever call or rank it runs in.  d_fixed nullable
 * float32 [F][resample_n][3] device: frame f's slot = kp_resample_batch on its final cloud with seed cfg.seed and
 * stream h_frame_ids[f]; PREFIX pads a short cloud with zeros; a RANDOM frame with fewer than resample_n points gets
 * status KP_E_ARG and a zero slot (the other frames are unaffected), one whose candidate list overflows KP_E_RANGE.
 * As for every frame status, the call returns it after every frame's record is written. */
KP_EXPORT int kp_pipeline_run_ex(kp_pipeline *p, const uint16_t *depth, const uint8_t *rgb, int inputs_on_device, int64_t F,
                                 const int64_t *h_frame_ids, kp_frame_result *h_results, float *d_out_xyz,
                                 int64_t out_stride, float *d_fixed);
KP_EXPORT int64_t kp_pipeline_launch_count(kp_pipeline *p);
/* frames per launch (B) and batch slots in flight (W) the pipeline was built with */
KP_EXPORT int kp_pipeline_frames_in_flight(kp_pipeline *p, int *batch, int *slots);
/* diagnostics: the device-side counts of the first frame of the last batch on slot 0, h_counts[n], n >= 26 =
 * n_fused, n_voxel, n_sor, n_band, n_band_kept, n_merged, n_floor_sor, n_out, level-0 leftovers of the three
 * neighbour searches [3], level-1 leftovers [3], valid rows of the ICP inputs [6], their voxel counts [6];
 * with n >= 29 also the mid-level leftovers of the three searches [3] (entries 26-28); with n >= 35 also twice
 * the crop median of each sensor [6] (entries 29-34; 0 without the crop); with n >= 36 also the survivors of the
 * radius outlier removal (entry 35; 0 when it is off) */
KP_EXPORT int kp_pipeline_frame_counts(kp_pipeline *p, int64_t *h_counts, int n);
KP_EXPORT int kp_pipeline_profile(kp_pipeline *p, int enable_or_read, int max_entries,
                                  const char **h_names, double *h_ms, int64_t *h_calls, double *h_bytes, int *h_n);

#ifdef __cplusplus
}
#endif
#endif /* KP_API_H */
