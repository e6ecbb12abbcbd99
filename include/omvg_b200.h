/*
 * omvg_b200.h — C ABI of libomvg_b200.so: the two openMVG hot paths on NVIDIA B200 (sm_100a).
 *
 * Plain pointers and sizes only; no C++ / torch types cross this boundary.  Every function returns
 * OMVG_OK (0) or a negative OMVG_E_* code; omvg_last_error() gives the text.  There is NO CPU
 * fallback behind these entry points: without a CUDA device they fail with OMVG_E_CUDA.
 *
 * What each group replaces in the reference (paths relative to /root/reference/src/openMVG):
 *
 *  MATCH  = matching_image_collection/Matcher_Regions.cpp:32-107 (Matcher_Regions::Match with
 *           BRUTE_FORCE_L2), i.e. per pair: matching/regions_matcher.hpp:162-207
 *           (RegionsMatcherT::MatchDistanceRatio) -> matching/matcher_brute_force.hpp:100-200
 *           (2-NN scan, L2<uint8_t> matching/metric.hpp:55-93) -> matching/matching_filters.hpp:38-60
 *           (NNdistanceRatio).  Host shim: openmvg_b200/host/Matcher_Regions_B200.hpp
 *           (implements matching_image_collection/Matcher.hpp:34-48).
 *
 *  BA     = sfm/sfm_data_BA_ceres.cpp:165-608 (Bundle_Adjustment_Ceres::Adjust) from the point
 *           where the Ceres problem is built to the point where parameters are written back, i.e.
 *           ceres::Solve with SPARSE_SCHUR / Levenberg-Marquardt / HuberLoss(16)
 *           (third_party/ceres-solver/internal/ceres/{trust_region_minimizer,
 *           levenberg_marquardt_strategy,schur_eliminator_impl,program_evaluator}.*).
 *           Host shim: openmvg_b200/host/Bundle_Adjustment_B200.hpp
 *           (implements sfm/sfm_data_BA.hpp:91-105).
 */
#ifndef OMVG_B200_H_
#define OMVG_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OMVG_OK            0
#define OMVG_E_ARG        -1   /* invalid argument */
#define OMVG_E_CUDA       -2   /* CUDA runtime / driver error, or no sm_100 device */
#define OMVG_E_STATE      -3   /* call order violated (e.g. run before upload) */
#define OMVG_E_UNSUPPORTED -4  /* feature outside the GPU path (the host shim routes it to the reference) */
#define OMVG_E_NUMERIC    -5   /* BA: solver failure (Ceres FAILURE: not "usable") */

#define OMVG_DESC_LEN 128      /* SIFT descriptor length, bytes (features/descriptor.hpp:30-36) */

int         omvg_version(void);            /* 100 = round 1 */
const char *omvg_last_error(void);         /* thread-local message of the last failing call */
int         omvg_device_count(void);       /* >0 only if sm_100 devices are visible */
void        omvg_trim_cache(void);         /* return cached device work buffers to the driver */

/* ===================================================================== MATCH ============== */
typedef struct omvg_match_ctx omvg_match_ctx;

/* One context = one GPU + one image collection.  device = CUDA ordinal. */
int omvg_match_create(omvg_match_ctx **ctx, int device);
int omvg_match_destroy(omvg_match_ctx *ctx);

/* Declare the collection: counts[k] = number of descriptors of image k (RegionCount()).
 * Allocates the device arena: every image's rows start at a multiple of 256 rows, zero padded. */
int omvg_match_set_images(omvg_match_ctx *ctx, uint32_t n_images, const uint32_t *counts);

/* Descriptor upload: desc = counts[image] rows of 128 bytes, row-major contiguous — exactly
 * Regions::DescriptorRawData() (features/scalar_regions.hpp:39,93).  _host copies H2D from
 * pageable or pinned memory; _device copies D2D from a device pointer (e.g. an NCCL all-gather
 * buffer).  Both are asynchronous on the context's stream. */
int omvg_match_upload_host(omvg_match_ctx *ctx, uint32_t image, const uint8_t *desc);
int omvg_match_upload_device(omvg_match_ctx *ctx, uint32_t image, const void *desc_dev);
/* Whole arena at once from ONE device buffer holding the images back to back (unpadded). */
int omvg_match_upload_device_packed(omvg_match_ctx *ctx, const void *desc_dev);

/* Squared norms + packed database keys for every row (one kernel).  Call after uploads. */
int omvg_match_prepare(omvg_match_ctx *ctx);

/* Match image pairs: for pair p the DATABASE is image pair_i[p], the QUERIES are image pair_j[p]
 * (Matcher_Regions.cpp:73,93).  dist_ratio is Lowe's ratio (squared internally, in float,
 * regions_matcher.hpp:196).  Asynchronous: results stay on the device until omvg_match_fetch. */
int omvg_match_run(omvg_match_ctx *ctx, const uint32_t *pair_i, const uint32_t *pair_j,
                   uint64_t n_pairs, float dist_ratio);

/* Wait for the device (no copy).  Used to time the resident-data path. */
int omvg_match_sync(omvg_match_ctx *ctx);

/* Copy the result of the last omvg_match_run to host memory owned by the context (valid until
 * the next run/destroy): CSR over the pairs in the order given.  Row p holds the kept matches of
 * pair p as (i_, j_) = (row in image pair_i[p], row in image pair_j[p]) in ascending j_
 * (regions_matcher.hpp:198-204); an empty row means the reference would not insert the pair
 * (Matcher_Regions.cpp:99-102). */
int omvg_match_fetch(omvg_match_ctx *ctx, const uint64_t **offsets /* n_pairs+1 */,
                     const uint32_t **ij /* 2*offsets[n_pairs] */, uint64_t *n_matches);

/* Kernel launches issued by this context so far (bench.py's gpu_launches). */
uint64_t omvg_match_launch_count(const omvg_match_ctx *ctx);
/* Device time (ms, CUDA events on the context's stream) and launch count of the dominant
 * kernel (the tcgen05 distance/top-2 kernel) accumulated since the last call with reset!=0. */
int omvg_match_kernel_time(omvg_match_ctx *ctx, double *ms, uint64_t *launches, int reset);
/* Which distance/top-2 kernel omvg_match_run will use for the prepared collection: 5 = fifth-K-slice kernel (the
 * per-column constant rides in the MMA; needs max|b|^2 - min|b|^2 <= 3.9e6 inside every image), 4 = the kernel with
 * the per-accumulator key arithmetic (any uint8 descriptors; also forced by OMVG_MATCH_TC4=1), 0 = not prepared.
 * Both give bit-identical matches. */
int omvg_match_kernel_variant(const omvg_match_ctx *ctx);

/* ---- cascade hashing: openMVG's default matcher for scalar descriptors ("FASTCASCADEHASHINGL2",
 * matching/cascade_hasher.hpp, matching_image_collection/Cascade_Hashing_Matcher_Regions.cpp:38-226).
 * primary[128][128] / secondary[6][10][128]: the Gaussian projections CascadeHasher::Init draws
 * (cascade_hasher.hpp:142-162) — generated by the caller with the same std::mt19937 / std::normal_distribution
 * so that they are the reference's (host/Cascade_Hashing_Matcher_Regions_B200.hpp does it).
 * used[n_images] (or NULL = all): the images the pair list names; the zero-mean descriptor is the mean of their
 * per-image means (:78-105).  Call after omvg_match_prepare. */
int omvg_match_cascade_prepare(omvg_match_ctx *ctx, const float *primary, const float *secondary, const uint8_t *used);
/* Pairs (I = database, J = queries) as in omvg_match_run; fetch with omvg_match_fetch.  Rows hold (i, j) in
 * ascending j; the reference then sorts by (i, j) (IndMatch::getDeduplicated) and drops matches with equal
 * coordinates (IndMatchDecorator) — host-side steps the shim performs with openMVG's own functions. */
int omvg_match_cascade_run(omvg_match_ctx *ctx, const uint32_t *pair_i, const uint32_t *pair_j, uint64_t n_pairs, float dist_ratio);
/* Validation aid (tests only): hash codes [count][4] (bit j = bit j&31 of word j>>5), bucket ids [count][6],
 * zero-mean vector [128]; any pointer may be NULL. */
int omvg_match_cascade_debug_hash(omvg_match_ctx *ctx, uint32_t image, uint32_t *codes, uint16_t *bucket_ids, float *zero_mean);

/* Validation aid (tests only): exact 2-NN of every row of image q_image in image db_image by a
 * plain SIMT dp4a kernel.  d1/i1/d2: host arrays of counts[q_image] entries. */
int omvg_match_debug_top2_simt(omvg_match_ctx *ctx, uint32_t db_image, uint32_t q_image,
                               int32_t *d1, uint32_t *i1, int32_t *d2);
/* Validation aid (tests only): the tensor-core kernel's raw per-query result for ONE pair before
 * the re-scan: best packed key and runner-up key decoded to (d1, group of i1, upper bound of d2). */
int omvg_match_debug_top2_tc(omvg_match_ctx *ctx, uint32_t db_image, uint32_t q_image,
                             int32_t *d1, uint32_t *group1, int32_t *d2_upper);

/* ---- descriptor / match file IO feeding the matcher (SURVEY §8f N3) ----------------------------------
 * omvg_match_load_desc_files = omvg_match_set_images + uploads + omvg_match_prepare from openMVG ".desc" files
 * (features/descriptor.hpp:182-203: size_t count, then count x 128 bytes), read by a pool of host threads into
 * one page-locked buffer and uploaded as each read completes — what Regions_Provider::load
 * (sfm/pipelines/sfm_regions_provider.hpp:88-138) does one std::vector at a time.  counts_out may be NULL. */
int omvg_match_load_desc_files(omvg_match_ctx *ctx, uint32_t n_images, const char *const *desc_paths, uint32_t *counts_out);
/* Writes a CSR result (omvg_match_fetch layout; pair_I / pair_J = the view ids to record) as openMVG's
 * "matches.*.txt" or "matches.*.bin" (matching::Save, matching/indMatch_utils.cpp:80-131; the extension picks the
 * format).  Pairs are written in std::map<Pair,...> order, pairs without matches are skipped. */
int omvg_matches_save(const char *path, uint64_t n_pairs, const uint32_t *pair_I, const uint32_t *pair_J,
                      const uint64_t *offsets, const uint32_t *ij);

/* ===================================================================== GEOMETRIC FILTER ==== */
/* Per-pair a-contrario RANSAC with the fundamental-matrix model: what GeometricFilter_FMatrix_AC::Robust_estimation
 * (matching_image_collection/F_ACRobust.hpp:45-106) runs for every pair of ImageCollectionGeometricFilter::
 * Robust_model_estimation (GeometricFilter.hpp:66-128) — ACKernelAdaptor<SevenPointSolver, EpipolarDistanceError,
 * UnnormalizerT> + ACRANSAC (robust_estimation/robust_estimator_ACRansac.hpp:303-490) with std::mt19937(default_seed).
 * One CTA per pair; same sample sequence, same NFA scoring, same inlier lists as the reference.
 *   offsets[n_pairs+1]        CSR over the putative matches of the pairs (omvg_match_fetch layout)
 *   xI, xJ [n_matches][2]     pixel positions of the matched features in image I / J (MatchesPairToMat)
 *   image_size[n_pairs][4]    wI hI wJ hJ (View::ui_width / ui_height)
 *   precision                 upper bound in pixels (main_GeometricFilter.cpp:304 passes 4.0); must be finite
 *   max_iterations            2048 in main_GeometricFilter.cpp:82
 * out: inliers[n_matches] (pair p: the first n_inliers[p] entries of its segment, ascending match index; the reference
 * keeps the pair iff n_inliers[p] > 2.5 * 7), F[n_pairs][9] row-major un-normalised, stats[n_pairs][2] = {errorMax
 * (pixels), minNFA}. */
int omvg_geom_fundamental_acransac(int device, uint64_t n_pairs, const uint64_t *offsets, const double *xI, const double *xJ,
                                   const int32_t *image_size, double precision, uint32_t max_iterations,
                                   uint32_t *inliers, uint32_t *n_inliers, double *F, double *stats);
/* The same with the model as an argument: OMVG_GEOM_FUNDAMENTAL (above) or OMVG_GEOM_HOMOGRAPHY =
 * GeometricFilter_HMatrix_AC (matching_image_collection/H_ACRobust.hpp:46-112: ACKernelAdaptor<FourPointSolver,
 * AsymmetricError, UnnormalizerI>, point-to-point error model, one model per 4-point sample; the reference keeps the
 * pair iff n_inliers > 2.5 * 4).  F then holds the homography. */
#define OMVG_GEOM_FUNDAMENTAL 0
#define OMVG_GEOM_HOMOGRAPHY  1
int omvg_geom_acransac(int device, int32_t model, uint64_t n_pairs, const uint64_t *offsets, const double *xI, const double *xJ,
                       const int32_t *image_size, double precision, uint32_t max_iterations,
                       uint32_t *inliers, uint32_t *n_inliers, double *F, double *stats);

/* ===================================================================== BA ================= */
#define OMVG_BA_INTR_STRIDE 8   /* doubles reserved per intrinsic block */

/* cameras::EINTRINSIC (cameras/Camera_Common.hpp:39-49); parameter order = getParams() */
#define OMVG_PINHOLE_CAMERA          1   /* f, ppx, ppy                      (Camera_Pinhole.hpp:215-218) */
#define OMVG_PINHOLE_CAMERA_RADIAL1  2   /* + k1                             (Camera_Pinhole_Radial.hpp) */
#define OMVG_PINHOLE_CAMERA_RADIAL3  3   /* + k1 k2 k3 */
#define OMVG_PINHOLE_CAMERA_BROWN    4   /* + k1 k2 k3 t1 t2                 (Camera_Pinhole_Brown.hpp) */
#define OMVG_PINHOLE_CAMERA_FISHEYE  5   /* + k1 k2 k3 k4                    (Camera_Pinhole_Fisheye.hpp) */
#define OMVG_CAMERA_SPHERICAL        7   /* no parameter block (getParams() is empty, Camera_Spherical.hpp); the two
                                            leading doubles of the intrinsic slot carry the image size {w, h}, constants
                                            of ResidualErrorFunctor_Intrinsic_Spherical (functor.hpp:662-760) */

/* Flat scene.  Mirrors what Adjust builds at sfm_data_BA_ceres.cpp:260-396:
 *   poses[n_poses][6]            angle-axis (3) then t = -R*C (3)                  (in/out)
 *   intrinsics[n_intr][8]        getParams() order, unused tail ignored            (in/out)
 *   points[n_points][3]          landmark X                                        (in/out)
 *   view_pose/view_intr[n_views] View::id_pose / View::id_intrinsic as dense indices
 *   obs_view/obs_point[n_obs]    one entry per (landmark, view) observation
 *   obs_xy[n_obs][2]             Observation::x (pixels)
 */
typedef struct {
  int32_t n_poses, n_intrinsics, n_points, n_views;
  int64_t n_obs;
  double *poses;
  double *intrinsics;
  const int32_t *intr_model;
  double *points;
  const int32_t *view_pose;
  const int32_t *view_intr;
  const int32_t *obs_view;
  const int32_t *obs_point;
  const double *obs_xy;
  /* ---- optional extensions (NULL / 0 = absent) -------------------------------------------------
   * Ground control points (sfm_data_BA_ceres.cpp:398-452): extra landmarks with point_fixed = 1
   * (SetParameterBlockConstant, :447) whose observations carry obs_weight = Control_Point_Parameter
   * ::weight (WeightedCostFunction multiplies the residual before the loss,
   * sfm_data_BA_ceres_camera_functor.hpp:35-90) and obs_no_loss = 1 (loss nullptr, :424/:432).
   * obs_weight = 0 removes an observation exactly (see omvg_ba_set_obs_weights). */
  const double  *obs_weight;     /* [n_obs] */
  const uint8_t *obs_no_loss;    /* [n_obs] */
  const uint8_t *point_fixed;    /* [n_points] */
  /* Pose-centre priors (PoseCenterConstraintCostFunction, sfm_data_BA_ceres.cpp:44-80, added at
   * :455-472): residual prior_weight .* (C(pose) - prior_center) under HuberLoss(prior_huber_a),
   * prior_huber_a = Square(pose_center_robust_fitting_error).  The similarity registration of the
   * scene to the priors (:183-236) is host-side geometry done by the caller before this call
   * (Bundle_Adjustment_B200.hpp does it with openMVG's own LeastMedianOfSquares/ApplySimilarity). */
  int32_t n_priors, reserved_;
  const int32_t *prior_pose;     /* [n_priors] pose index */
  const double  *prior_center;   /* [n_priors][3] */
  const double  *prior_weight;   /* [n_priors][3] */
  double prior_huber_a;
} omvg_ba_problem;

/* Optimize_Options (sfm/sfm_data_BA.hpp:66-89) + BA_Ceres_options (sfm_data_BA_ceres.hpp:34-49)
 * + the Ceres Solver::Options the reference ends up with (sfm_data_BA_ceres.cpp:477-493 over
 * ceres/solver.h:62-138).  omvg_ba_default_options() fills the reference's values. */
typedef struct {
  int32_t intrinsics_opt;      /* cameras::Intrinsic_Parameter_Type bit mask (NONE=1,F=2,PP=4,DIST=8) */
  int32_t extrinsics_opt;      /* sfm::Extrinsic_Parameter_Type (NONE=1,ROT=2,TRANS=4,ALL=6) */
  int32_t structure_opt;       /* 0 = NONE, 1 = ADJUST_ALL */
  int32_t use_loss;            /* bUse_loss_function_ */
  double  huber_a;             /* Square(4.0) = 16 */
  int32_t max_num_iterations;  /* 50 */
  int32_t max_consecutive_invalid_steps; /* 5 */
  double  function_tolerance;  /* 1e-6 */
  double  gradient_tolerance;  /* 1e-10 */
  double  parameter_tolerance; /* 1e-8 */
  double  initial_radius, max_radius, min_radius;      /* 1e4, 1e16, 1e-32 */
  double  min_relative_decrease;                        /* 1e-3 */
  double  min_lm_diagonal, max_lm_diagonal;             /* 1e-6, 1e32 */
  /* reduced-camera-system solve (block-Jacobi PCG standing in for SimplicialLDLT) */
  double  pcg_tolerance;       /* relative residual |S z - b| / |b| <= tol ; default 1e-8 (final cost within ~3e-9 of the exact solve) */
  int32_t pcg_max_iterations;  /* default 2000 */
  int32_t verbose;
  int32_t device;              /* CUDA ordinal used by omvg_ba_solve (omvg_ba_create takes its own) ; default 0 */
  int32_t reserved_;
} omvg_ba_options;

typedef struct {
  double  initial_cost, final_cost;   /* 1/2 sum rho(|r|^2), as Ceres' Summary reports */
  int32_t iterations;                 /* Ceres "Minimizer iterations" (recorded iterations incl. #0) */
  int32_t successful_steps, unsuccessful_steps;
  int32_t lm_steps;                   /* linear systems solved (incl. the terminating iteration) */
  int32_t termination;                /* 0 fn-tol, 1 param-tol, 2 grad-tol, 3 max-iters, 4 min-radius, -1 failure */
  int32_t usable;                     /* Summary::IsSolutionUsable() */
  int64_t pcg_iterations;             /* total over all LM steps */
  int64_t kernel_launches;
  double  device_ms;                  /* solve time on the device (CUDA events), upload/download excluded */
  double  jacobian_ms;                /* time in the residual+Jacobian kernel (sum) and its launch count */
  int64_t jacobian_launches;
} omvg_ba_summary;

void omvg_ba_default_options(omvg_ba_options *o);

/* One-shot: upload, solve, write poses/intrinsics/points back into the problem's arrays iff the
 * solution is usable (solver.cc:445-448 semantics).  Returns OMVG_OK, or OMVG_E_NUMERIC when not
 * usable (Adjust() would return false), or OMVG_E_UNSUPPORTED for a camera model / option the GPU
 * path does not implement. */
int omvg_ba_solve(omvg_ba_problem *problem, const omvg_ba_options *options, omvg_ba_summary *summary);

/* Device-resident variant: the scene stays in HBM between solves (bench "value", BA/reject/BA loop). */
typedef struct omvg_ba_ctx omvg_ba_ctx;
int omvg_ba_create(omvg_ba_ctx **ctx, int device, const omvg_ba_problem *problem);   /* uploads */
int omvg_ba_reset(omvg_ba_ctx *ctx);      /* restore the parameters uploaded at create (device copy) */
int omvg_ba_run(omvg_ba_ctx *ctx, const omvg_ba_options *options, omvg_ba_summary *summary);
int omvg_ba_download(omvg_ba_ctx *ctx, double *poses, double *intrinsics, double *points);
int omvg_ba_destroy(omvg_ba_ctx *ctx);
/* Adjust's write-back rules (sfm_data_BA_ceres.cpp:528-568) from the device state into the caller's arrays (which hold
 * the caller's previous values on entry): poses only if extrinsics were refined, ADJUST_ROTATION keeps the pose
 * centre, intrinsics only if intrinsics were refined.  Any pointer may be NULL (that block is skipped). */
int omvg_ba_writeback(omvg_ba_ctx *ctx, const omvg_ba_options *options, double *poses, double *intrinsics, double *points);
/* |reprojection residual| (pixels, no loss) of every observation at the current device parameters, in the
 * caller's observation order: the quantity RemoveOutliers_PixelResidualError (sfm/sfm_data_filters.cpp:40-73)
 * thresholds after each Adjust of the BA / outlier-rejection loop (sequential_SfM.cpp:205-211). */
int omvg_ba_residual_norms(omvg_ba_ctx *ctx, double *norms /* [n_obs] */);
/* Replace the per-observation weights of the resident problem (caller's observation order; weight 0 =
 * observation removed, exactly) — the rejection half of the loop above without rebuilding the scene. */
int omvg_ba_set_obs_weights(omvg_ba_ctx *ctx, const double *weights /* [n_obs] */);
/* The rejection half of `do { BundleAdjustment(); } while (badTrackRejector(4.0, 50))` (sequential_SfM.cpp:205-211,
 * 1237-1243) on the resident scene.  omvg_ba_reject_outliers = RemoveOutliers_PixelResidualError(threshold_px,
 * min_track_length) (sfm/sfm_data_filters.cpp:40-73) at the current device parameters: live observations with
 * |residual| > threshold_px are removed and counted (*n_outliers), then tracks left with fewer than
 * min_track_length observations are removed whole (*n_tracks; their observations are not counted, as in the
 * reference).  Removal = weight 0 (exact) and the track becomes a constant block; control points are left alone.
 * obs_removed_bits[(n_obs+31)/32]: bit o set = observation o (CALLER's order) was removed by THIS call;
 * point_removed[n_points]: 1 = track removed by this call.  Either may be NULL.  Only a bit mask and two counters
 * cross the bus.  omvg_ba_remove_points removes the tracks the caller names (point_mask[n_points] != 0): the
 * angle test RemoveOutliers_AngleError stays host geometry in the shim. */
int omvg_ba_reject_outliers(omvg_ba_ctx *ctx, double threshold_px, int32_t min_track_length,
                            uint32_t *obs_removed_bits, uint8_t *point_removed, int64_t *n_outliers, int64_t *n_tracks);
int omvg_ba_remove_points(omvg_ba_ctx *ctx, const uint8_t *point_mask, uint32_t *obs_removed_bits, int64_t *n_tracks);
/* Make the current (refined) parameters the state omvg_ba_reset() restores. */
int omvg_ba_commit(omvg_ba_ctx *ctx);

/* Validation aids (tests only): one evaluation at the uploaded parameters.
 * r[n_obs][2], J_intr[n_obs][2][8], J_pose[n_obs][2][6], J_point[n_obs][2][3] (row-major blocks,
 * Huber-corrected, NOT Jacobi-scaled), in the caller's observation order; cost returned. */
int omvg_ba_debug_eval(omvg_ba_ctx *ctx, const omvg_ba_options *options, double *cost, double *r,
                       double *J_intr, double *J_pose, double *J_point);

#ifdef __cplusplus
}
#endif
#endif  /* OMVG_B200_H_ */
