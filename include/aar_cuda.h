/*
 * aar_cuda.h — C ABI of the B200 (sm_100a) joint-optimisation path of automatic-ar.
 *
 * The reference (HSarham/automatic-ar) has no FFI layer: the seam of its hot path is the C++
 * call `MultiCamMapper::solve()` / `track()` (libs/multicam_mapper.cpp:419-443) which binds
 * `error_function` / `jacobian_function` into `ucoslam::SparseLevMarq<double>::solve`
 * (libs/sparselevmarq.h:80, 118).  This header is what a binding of that seam looks like:
 * plain pointers and sizes, opaque handle, int status codes, no exceptions, no C++ / torch types.
 * Every entry point cites the reference interface it replaces.  INTEGRATION.md shows the
 * reference-side stub.  Entry points marked "Not in the reference" extend the solve: held poses
 * (aar_set_fixed), held intrinsics (aar_set_fixed_intrinsics), soft pose priors (aar_set_prior) and
 * soft relative-pose priors between two cameras or two markers (aar_set_pair_prior); so does the lens
 * model of aar_problem_desc::lens_model.
 *
 * Conventions
 *   - all matrices are row-major 4x4 doubles (cv::Mat CV_64F as the reference holds them);
 *   - ids are the reference's ids (camera folder number, ArUco marker id, frame ordinal);
 *     indices are ranks of ids in ascending order (MatArray::operator=, multicam_mapper.h:95-105);
 *   - host buffers are caller-owned; one handle = one CUDA device + one stream; not re-entrant;
 *   - there is NO CPU fallback: every function that computes returns AAR_ERR_CUDA when the
 *     device path is unavailable.
 */
#ifndef AAR_CUDA_H
#define AAR_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct aar_problem aar_problem;

enum {
    AAR_OK = 0,
    AAR_ERR_INVALID = 1,      /* bad argument / inconsistent description */
    AAR_ERR_CUDA = 2,         /* CUDA runtime error (no device, launch failure, out of memory) */
    AAR_ERR_UNSUPPORTED = 3,  /* e.g. a non-pinhole camera matrix, more than 4095 cameras */
    AAR_ERR_COMM = 4,         /* NCCL error */
    AAR_ERR_NUMERIC = 5       /* non-finite cost or non-positive Cholesky pivot */
};

/* What MultiCamMapper::init (8 arguments, multicam_mapper.cpp:281-335) receives from the Initializer,
 * flattened.  Detections are in aruco.detections file order: frame, camera, detection order. */
typedef struct {
    int32_t num_cams, num_markers, num_frames;
    const int32_t *cam_ids, *marker_ids, *frame_ids;  /* strictly ascending */
    int32_t root_cam, root_marker;                    /* ids (Initializer::get_root_cam/_marker) */
    float marker_size;                                /* narrowed to float like the reference ctor (multicam_mapper.h:17) */
    const double *cam_T;                              /* [num_cams][16]    camera -> root camera     */
    const double *marker_T;                           /* [num_markers][16] marker -> root marker     */
    const double *frame_T;                            /* [num_frames][16]  root marker -> root camera */
    const double *cam_K;                              /* [num_cams][9] camera matrices (CamConfig::getCamMat) */
    const double *cam_dist;                           /* [num_cams][5] k1 k2 p1 p2 k3 (CamConfig::getDistCoeffs) */
    int64_t num_detections;
    const int32_t *det_frame, *det_cam, *det_marker;  /* ids */
    const float *det_xy;                              /* [num_detections][8] x0 y0 .. x3 y3, raw pixels */
    /* MultiCamMapper::Config (multicam_mapper.h:75-81) + set_with_huber (:40) */
    uint8_t optimize_cam_poses, optimize_marker_poses, optimize_object_poses, optimize_cam_intrinsics;
    uint8_t with_huber;
    uint8_t corners_undistorted;                      /* detections come from a .solution file (already undistorted, multicam_mapper.cpp:1085-1088):
                                                       * no remove_distortions pass, and the Jacobian's "raw" corners are these corners too */
    uint8_t analytic_jacobian;                        /* 0: the reference's central differences on float32-rounded projections (parity path).
                                                       * 1: analytic Jacobian, residuals kept in double (include/aar_analytic.h) — NOT the reference's
                                                       *    arithmetic; with lens_model 0, pose blocks only (with optimize_cam_intrinsics:
                                                       *    AAR_ERR_UNSUPPORTED); track ignores it */
    uint8_t lens_model;                               /* Not in the reference.  0: the corners undistorted once at create with cam_dist (above).
                                                       * 1: residual raw - projectPoints(Xc; K, k1 k2 p1 p2 k3) on the detected corners, no undistortion
                                                       *    in the residual (aar_an_observation_lens, include/aar_analytic.h); K and dist from the
                                                       *    iterate when optimize_cam_intrinsics (all nine columns live), else from cam_K / cam_dist.
                                                       *    Needs analytic_jacobian = 1 and corners_undistorted = 0; other values: AAR_ERR_UNSUPPORTED.
                                                       *    aar_eval_residual, aar_error_report and aar_eval_jacobian follow it; aar_track_* ignore it. */
    double J_delta;                                   /* multicam_mapper.h:189, 0 -> 1e-3 */
    /* placement */
    int32_t device;                                   /* CUDA device ordinal */
    void *stream;                                     /* cudaStream_t to launch on; NULL -> the handle creates its own */
    int32_t rank, world_size;                         /* frame shard of this handle (world_size <= 1: everything) */
} aar_problem_desc;

/* ucoslam::SparseLevMarq<double>::Params (sparselevmarq.h:30-50) as MultiCamMapper sets them
 * (multicam_mapper.cpp:326-330) */
typedef struct {
    int32_t max_iters;                 /* 10000 */
    double min_error;                  /* 1e-5  */
    double min_step_error_diff;        /* 0     */
    double min_average_step_error_diff;/* 1e-4  */
    double tau;                        /* 1     */
    double der_epsilon;                /* 1e-3 (track: FD step of calcDerivates) */
    int32_t ignore_stop_rules;         /* benchmark aid: run exactly max_iters iterations */
    int32_t verbose;                   /* print the reference's per-iteration line (sparselevmarq.h:421) */
} aar_lm_params;

typedef struct { double cost, mu, gain; int32_t tries, accepted; float huber_delta; int32_t pad; } aar_lm_trace;

typedef struct {
    double initial_cost, final_cost;
    int32_t iterations;        /* LM iterations executed */
    int32_t exit_code;         /* mustExit of sparselevmarq.h:453-465: 0 max iters, 1 minError, 2 small step / rejected, 3 error grew */
    int64_t total_tries;
    aar_lm_trace *trace;       /* optional caller buffer */
    int32_t trace_capacity, trace_len;
} aar_lm_report;

void aar_lm_default_params(aar_lm_params *p);

/* MultiCamMapper ctor / init (multicam_mapper.cpp:252-259, 281-335): builds the row map
 * (fill_iteration_arrays :345-377), uploads the observations packed SoA, undistorts them on the
 * device (remove_distortions :554-578). */
int aar_problem_create(const aar_problem_desc *desc, aar_problem **out);
void aar_problem_destroy(aar_problem *p);
const char *aar_last_error(void);

/* sizes: get_num_vars (multicam_mapper.cpp:239-250), num_point_xys/8, structural nnz of J */
int64_t aar_num_vars(const aar_problem *p);
int64_t aar_num_observations(const aar_problem *p);       /* global, after the erasures of :353-367 */
int64_t aar_num_local_observations(const aar_problem *p); /* this rank's shard */
int64_t aar_jacobian_nnz(const aar_problem *p);

/* Bit-exact index contract (SURVEY Appendix C).  Any pointer may be NULL.
 * obs_*: per global observation, in row order (row0 = 8*ordinal).  col_*: first column of each
 * block in io_vec, -1 for the root / a non-optimised group. */
int aar_index_maps(const aar_problem *p, int32_t *obs_frame_idx, int32_t *obs_cam_idx, int32_t *obs_marker_idx,
                   int32_t *obs_has_jacobian, int64_t *col_cam, int64_t *col_marker, int64_t *col_frame,
                   int32_t *shard_frame_begin, int32_t *shard_frame_end);

/* undistorted (device pass) and raw corners of this rank's observations, [n_local][8] floats */
int aar_get_observations(aar_problem *p, float *und_xy, float *raw_xy);

/* mats2eVec (multicam_mapper.cpp:445-461): host side, R -> r like cv::Rodrigues(3x3 -> 3x1) */
int aar_mats2evec(const aar_problem *p, double *z);
/* eVec2Mats (multicam_mapper.cpp:595-606): device expansion read back; 4x4 per camera/marker/frame
 * (frames: this rank's shard only when sharded; others are left untouched) */
int aar_evec2mats(aar_problem *p, const double *z, double *cam_T, double *marker_T, double *frame_T);

/* MultiCamMapper::error_function (multicam_mapper.cpp:731-737): r has 8*n_local entries */
int aar_eval_residual(aar_problem *p, const double *z, float huber_delta, double *r, double *sum_sq);
/* Reprojection-error report at z (not in the reference).  The residual of an observation is r[0..7] of the handle's own residual
 * evaluation (the one aar_eval_residual runs) with the Huber weights OFF; its error is e = sqrt(s / 4), s = r0^2 + ... + r7^2 summed
 * left to right without FMA: the RMS corner distance in pixels.  Every pointer may be NULL except q / q_value when num_q > 0.
 * Entity arrays are indexed by rank of the id (ascending ids); an entity without observations has count 0, sum_sq 0, max 0.
 * Duplicates erased by "last duplicate wins" still have residual rows, so they count like any other observation. */
typedef struct {
    double *det_err;                                  /* [desc num_detections], indexed like desc->det_*: e, NaN for a detection not in
                                                       * the problem (unknown camera / marker id, frame without a pose) */
    int64_t *cam_count, *marker_count, *frame_count;  /* observations */
    double *cam_sum_sq, *marker_sum_sq, *frame_sum_sq;/* sum of s; RMS = sqrt(sum_sq / (4 count)) */
    double *cam_max, *marker_max, *frame_max;         /* max e */
    int32_t num_q;                                    /* in: number of percentiles, <= 256 */
    int32_t reserved;
    const double *q;                                  /* in: [num_q] in [0, 1] */
    double *q_value;                                  /* out: [num_q] exact order statistic sorted(e)[floor(q (n - 1))]; NaN when n = 0 */
    int64_t num_observations;                         /* out: n */
    int64_t num_not_in_problem;                       /* out: detections of the description that are not observations */
    double sum_sq;                                    /* out: Huber-off cost (sum of s over all observations) */
} aar_error_report_out;
#ifdef __cplusplus
static_assert(sizeof(aar_error_report_out) == 128, "aar_error_report_out layout");
#else
_Static_assert(sizeof(aar_error_report_out) == 128, "aar_error_report_out layout");
#endif
/* Single-rank handles only, and not between aar_lm_begin and aar_lm_end (AAR_ERR_INVALID). */
int aar_error_report(aar_problem *p, const double *z, aar_error_report_out *out);
/* MultiCamMapper::jacobian_function (multicam_mapper.cpp:739-801) in the compressed-column form
 * Eigen's setFromTriplets produces: colptr[num_vars+1], rowidx[nnz], vals[nnz].  Single-rank handles only. */
int aar_eval_jacobian(aar_problem *p, const double *z, int64_t *colptr, int32_t *rowidx, double *vals);
/* frame-eliminated normal equations of this rank's shard at z for damping mu (parity hook of the
 * Schur stage): S [n_r*n_r] row-major, UPPER block triangle valid, WITHOUT mu on its diagonal;
 * b [n_r]; cost = sum of squared residuals of the shard.  With priors (aar_set_prior, aar_set_pair_prior) S, b and cost are those of
 * the augmented problem: the camera / marker and pair terms on rank 0, the frame terms on the rank that holds the frame.  n_r = 6 (cameras - 1) + 6 (markers - 1) of the optimised groups; with
 * optimize_cam_intrinsics 12 more per camera, in the internal order [fx cx fy cy k1 k2 | p1 p2 k3 . . .] (csrc/aar_intrinsics.cuh). */
int aar_reduced_system(aar_problem *p, const double *z, double mu, double *S, double *b, double *cost);

/* Not in the reference.  Hold poses fixed in every later solve / aar_reduced_system of this handle: their Jacobian columns are
 * treated as explicit zeros (step exactly 0, excluded from mu0).  Arrays indexed by rank of id: [num_cams], [num_markers],
 * [num_frames] of the description (global frames; every rank passes the same arrays); nonzero = fixed; NULL = none of that kind;
 * all NULL clears.  The root camera / marker and entities of a group that is not optimised may be flagged (no effect).
 * Residuals and cost are unchanged; aar_eval_jacobian, aar_error_report and aar_track_* ignore the mask.  AAR_ERR_INVALID between
 * aar_lm_begin and aar_lm_end, and for a mask that leaves no free column. */
int aar_set_fixed(aar_problem *p, const uint8_t *cam_fixed, const uint8_t *marker_fixed, const uint8_t *frame_fixed);

/* Not in the reference.  Hold intrinsics of chosen cameras fixed in every later solve / aar_reduced_system of a handle with
 * optimize_cam_intrinsics, like aar_set_fixed holds poses: cam_flags [num_cams] indexed by rank of id, bit 0 holds
 * [fx cx fy cy k1 k2], bit 1 holds [p1 p2 k3]; NULL clears.  Combines with the aar_set_fixed mask.  AAR_ERR_INVALID between
 * aar_lm_begin and aar_lm_end, without optimize_cam_intrinsics, for a flag with bits above 1, and for a combined mask that leaves no
 * free column (without lens_model, [p1 p2 k3] is never a free column: the reference's distortion columns are explicit zeros). */
int aar_set_fixed_intrinsics(aar_problem *p, const uint8_t *cam_flags);

/* Not in the reference.  Soft priors: six residual rows sqrt(w) (z_e - zbar_e) per entity in every later solve / aar_reduced_system of
 * this handle; zbar_e from the 4x4 target by the R -> r of aar_mats2evec.  T: [n][16] row-major like desc->cam_T; w: [n][6] information
 * weights (1/sigma^2) of [r0 r1 r2 t0 t1 t2], >= 0 and finite, 0 = none; w == NULL: no prior of that kind; all NULL clears.  Indexed by
 * rank of id; frames global like aar_set_fixed.  Root / non-optimised entities are ignored.  AAR_ERR_INVALID between aar_lm_begin and
 * aar_lm_end, for a negative or non-finite weight, and for a non-finite target of an entity with a nonzero weight.
 * The cost the solver reports and compares (aar_lm_report, the trace, aar_reduced_system) includes sum w (z - zbar)^2; the stop rule
 * still divides by the 8 N reprojection rows.  mu0 = tau max diag(J^T J) is taken over the augmented diagonal, so a weight far above
 * the reprojection diagonal slows the first iterations: for a hard constraint use aar_set_fixed, which also wins over a prior on the
 * same entity (its prior residual stays in the cost as a constant).  The rotation difference is taken component by component in
 * rotation-vector space (to first order the geodesic error near the target; no wrap near |r| = pi).  aar_eval_residual,
 * aar_eval_jacobian, aar_error_report and aar_track_* ignore priors. */
int aar_set_prior(aar_problem *p, const double *cam_T, const double *cam_w, const double *marker_T, const double *marker_w,
                  const double *frame_T, const double *frame_w);

/* Not in the reference.  Soft relative-pose priors between two cameras or two markers (e.g. a stereo pair calibrated on its own, two
 * markers on one rigid board): 12 residual rows per pair in every later solve / aar_reduced_system of this handle.  With T_x the
 * pose the solve optimises (camera -> root camera, marker -> root marker) the pair (a, b) measures T_ab = T_a^-1 T_b (b's coordinates
 * into a's, the direction of desc->cam_T), R_ab = R_a^T R_b, t_ab = R_a^T (t_b - t_a); the rows are sqrt(w_rot / 2) vec(R_ab - Rbar)
 * and sqrt(w_t) (t_ab - tbar), their squared sum w_rot (2 - 2 cos theta) + w_t |t_ab - tbar|^2 (theta: the angle of Rbar^T R_ab;
 * w_rot = 1 / sigma_rot^2 with sigma_rot in radians, w_t = 1 / sigma_t^2).  *_pairs: [n][2] indices (ranks of ids); *_T: [n][16]
 * row-major targets T_ab; *_w: [n][2] w_rot, w_t.  Both counts 0 clears; every call replaces the earlier pairs.  A pair listed twice
 * counts twice.  A side without columns (the root) is a constant identity pose; a pair with no columns on either side, or with both
 * weights 0, is ignored.  AAR_ERR_INVALID between aar_lm_begin and aar_lm_end, for an index out of range, for a == b, for a negative
 * or non-finite weight, and, for a pair with a nonzero weight, for a non-finite target or a target rotation with |Rbar^T Rbar - I| >
 * 1e-9 or det Rbar <= 0.  Adds to aar_set_prior, with the same rules: the cost the solver reports and compares includes the pair
 * terms, mu0 is taken over the augmented diagonal, the stop rule still divides by the 8 N reprojection rows, pair rows are never
 * Huber-weighted, aar_set_fixed wins over a pair on a held entity, and aar_eval_residual, aar_eval_jacobian, aar_error_report and
 * aar_track_* ignore pairs.  Changing the number of stored pairs captures the graph-resident loop again; new values alone keep it. */
int aar_set_pair_prior(aar_problem *p,
                       int32_t num_cam_pairs, const int32_t *cam_pairs, const double *cam_T, const double *cam_w,
                       int32_t num_marker_pairs, const int32_t *marker_pairs, const double *marker_T, const double *marker_w);

/* MultiCamMapper::solve() = SparseLevMarq::solve(z, f, J) (multicam_mapper.cpp:419-428,
 * sparselevmarq.h:439-472): z is in/out like io_vec; the loop is device resident. */
int aar_lm_solve(aar_problem *p, double *z_inout, const aar_lm_params *params, aar_lm_report *report);
/* the same in three steps, z staying on the device in between (bench / step-by-step mode,
 * SparseLevMarq::init + step, sparselevmarq.h:88-96).  aar_lm_begin(p, NULL, params) restarts from the z0 of
 * the previous aar_lm_begin, which is still resident on the device (no host->device copy). */
int aar_lm_begin(aar_problem *p, const double *z0, const aar_lm_params *params);
int aar_lm_iterate(aar_problem *p, int32_t max_iters, aar_lm_report *report);
int aar_lm_end(aar_problem *p, double *z_out);

/* MultiCamMapper::track() (multicam_mapper.cpp:430-443) for every frame of the handle at once:
 * per-frame 6-dof LM against the fixed rig, Jacobian by central differences on z
 * (calcDerivates, sparselevmarq.h:164-220).  z6 [num_frames_local][6] in/out. */
int aar_track_batch(aar_problem *p, double *z6_inout, const aar_lm_params *params, double *final_cost, int32_t *iterations);
/* the same in three steps — start poses to the device / all per-frame solves from the uploaded poses (repeatable) / results back —
 * so that a caller can keep the poses resident; aar_track_ms: device time of the solves since aar_set_profiling(p, 1) */
int aar_track_upload(aar_problem *p, const double *z6);
int aar_track_run(aar_problem *p, const aar_lm_params *params);
int aar_track_download(aar_problem *p, double *z6, double *final_cost, int32_t *iterations);
int aar_track_ms(const aar_problem *p, double *ms, int64_t *runs);

/* The frame shard a handle created from `desc` (rank, world_size) would own, computed on the host without touching a
 * device: contiguous frame-index range [frame_begin, frame_end) balanced by observation count, and its observation
 * (row / 8) range.  Any output pointer may be NULL. */
int aar_shard_plan(const aar_problem_desc *desc, int32_t *frame_begin, int32_t *frame_end, int64_t *obs_begin, int64_t *obs_end, int64_t *num_observations);

/* The observation -> residual-row map of fill_iteration_arrays (multicam_mapper.cpp:345-377) computed on the host
 * without touching a device: per kept observation, in row order (row0 = 8 * ordinal), the frame / camera / marker
 * INDEX and whether it owns Jacobian rows.  Arrays may be NULL (count only); capacity = their length. */
int aar_row_map(const aar_problem_desc *desc, int64_t capacity, int32_t *obs_frame_idx, int32_t *obs_cam_idx, int32_t *obs_marker_idx,
                int32_t *obs_has_jacobian, int64_t *num_observations);

/* multi-GPU (one process per GPU of one box): one handle per rank; id is the 128-byte ncclUniqueId created on rank 0.  Per LM try the
 * reduced system and three scalars are all-reduced with NCCL. */
int aar_comm_unique_id(void *id128);
int aar_comm_init(aar_problem *p, const void *id128);

/* instrumentation for bench.py: kernels launched by this handle so far, and device time (ms, CUDA events on
 * the handle's stream) accumulated per phase since aar_set_profiling(p, 1):
 *   [0] expansion + Jacobian/normal-equation assembly  [1] Schur + all-reduce + reduced solve  [2] back-substitution
 *   [3] trial residual  [4] cost all-reduce + decision  [5] k_jac_project alone  [6] number of launches in [5]
 *   [7] the assembly kernels (k_asm_pairs + k_asm_mruns) alone  [8] k_schur_syrk alone  [9] number of launches in [8]
 *   [10] k_asm_pairs alone  [11] k_asm_mruns alone */
#define AAR_NUM_PHASES 12
int64_t aar_kernel_launches(const aar_problem *p);
/* sizes of this rank's shard: [0] W slots  [1] (frame, camera) pairs  [2] (frame, marker) runs  [3] fused multiply-adds of the upper
 * triangle of the Schur update S -= E E^T per try  [4] bit 0: always 0, bit 1: graph-resident loop built, bit 2: the last reduced solve
 * ran the cluster Cholesky (else the cooperative-grid one), bit 3: the last assembly kept its camera / marker accumulators in shared
 * memory (else it added them into global memory), bit 4: the last assembly used the camera x marker replicas, bits 8..: LM iterations
 * run inside the graph  [5] most blocks seen by one frame  [6] [7] frame index range */
int aar_problem_stats(const aar_problem *p, int64_t *out /* [8] */);
int aar_set_profiling(aar_problem *p, int32_t on);
int aar_get_phase_ms(const aar_problem *p, double *ms /* [AAR_NUM_PHASES] */);

#ifdef __cplusplus
}
#endif
#endif /* AAR_CUDA_H */
