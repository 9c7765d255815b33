// multicam_mapper.h — host-side mirror of the reference's MultiCamMapper (/root/reference/libs/multicam_mapper.h:14-83)
// for the joint-optimisation path: same method names, argument meaning and file formats, cv::Mat replaced by
// aar::Mat44, the optimisation itself forwarded to the CUDA path through the C ABI of include/aar_cuda.h.
// What is NOT here: overlays / visualisation (GUI).
#pragma once
#include <cmath>
#include <map>
#include <set>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/aar_cuda.h"
#include "aar_host_types.h"

namespace ucoslam {
// the solver parameters MultiCamMapper sets (libs/sparselevmarq.h:30-50); the solver itself lives on the device
template <typename T> struct SparseLevMarq {
    typedef std::vector<T> eVector;
    struct Params {
        int maxIters = 10000; T minError = 1e-5, min_step_error_diff = 0, min_average_step_error_diff = 1e-4, tau = 1, der_epsilon = 1e-3;
        bool verbose = false;
    };
};
} // namespace ucoslam

namespace aar {

class Initializer;

class MultiCamMapper {
public:
    struct Config {            // multicam_mapper.h:75-81
        bool optimize_cam_poses = true, optimize_object_poses = true, optimize_marker_poses = true, optimize_cam_intrinsics = true;
    };
    MultiCamMapper();
    explicit MultiCamMapper(Initializer &initializer);                     // multicam_mapper.cpp:252-254
    MultiCamMapper(size_t root_c, const std::map<int, Mat44> &T_to_root_cam, size_t root_m, const std::map<int, Mat44> &T_to_root_marker,
                   const std::map<int, Mat44> &obj_transforms, const FrameCamMarkers &fcm, float m_size, const std::vector<CamConfig> &cam_confs);
    ~MultiCamMapper();
    MultiCamMapper(const MultiCamMapper &) = delete;
    MultiCamMapper &operator=(const MultiCamMapper &) = delete;

    // multicam_mapper.cpp:281-335 — the Initializer's output; detections are RAW pixels, undistorted here (on the device)
    void init(size_t root_c, const std::map<int, Mat44> &T_to_root_cam, size_t root_m, const std::map<int, Mat44> &T_to_root_marker,
              const std::map<int, Mat44> &object_poses, const FrameCamMarkers &fcm, float m_size, const std::vector<CamConfig> &cam_confs);
    // multicam_mapper.cpp:272-279 — new frames against the same rig (tracking)
    void init(const std::map<int, Mat44> &object_poses, const FrameCamMarkers &fcm);

    void set_optmize_flag_cam_poses(bool v) { config.optimize_cam_poses = v; drop_handle(); }
    void set_optmize_flag_marker_poses(bool v) { config.optimize_marker_poses = v; drop_handle(); }
    void set_optmize_flag_object_poses(bool v) { config.optimize_object_poses = v; drop_handle(); }
    void set_optmize_flag_cam_intrinsics(bool v) { config.optimize_cam_intrinsics = v; drop_handle(); }
    void set_with_huber(bool v) { with_huber = v; drop_handle(); }
    // not in the reference: analytic Jacobian + residuals kept in double (include/aar_analytic.h, SURVEY 8(f) row 4); pose blocks only
    void set_analytic_jacobian(bool v) { analytic_jacobian = v; drop_handle(); }
    // not in the reference: the lens model of the analytic mode (aar_problem_desc::lens_model, DESIGN.md §6g): residuals on the raw
    // corners through OpenCV's five-coefficient projection, so that solve() with optimize_cam_intrinsics refines K and the distortion.
    // Implies the analytic Jacobian.  Needs the raw corners of init(): after read_solution_file (undistorted corners only) it throws
    // std::logic_error.  After a solve that refined the intrinsics, frame_cam_markers holds the raw corners undistorted with the
    // refined coefficients, so that a written .solution is self-consistent.
    void set_lens_model(bool v);
    // not in the reference: hold the intrinsics of these cameras (ids) in solve() when optimize_cam_intrinsics: bit 0 holds
    // fx cx fy cy k1 k2, bit 1 holds p1 p2 k3 (aar_set_fixed_intrinsics, include/aar_cuda.h); held values stay the caller's bytes.
    // Replaces the earlier map; an id the mapper does not hold or a flag above 3 throws std::invalid_argument.
    void set_fixed_intrinsics(const std::map<int, uint8_t> &flags);
    void set_config(const Config &c) { config = c; drop_handle(); }
    size_t get_num_vars(const Config &conf) const;

    void solve();     // multicam_mapper.cpp:419-428: device-resident SparseLevMarq::solve(io_vec, error_function, jacobian_function)

    // not in the reference: reprojection errors of the current state (aar_error_report, include/aar_cuda.h), Huber weights off
    struct EntityError { long long observations = 0; double sum_sq = 0, max = 0; double rms() const { return std::sqrt(sum_sq / (4.0 * (double)observations)); } };
    struct ErrorReport {
        long long observations = 0, not_in_problem = 0; double sum_sq = 0;
        std::map<int, EntityError> cams, markers, frames;       // by id
        std::vector<double> q, q_value;                          // exact percentiles of the observation errors
        std::vector<double> det_err;                             // per detection of the handle (raw_frame_cam_markers when present, else frame_cam_markers,
                                                                 // frame / camera / detection order); NaN when not in the problem
    };
    // at io_vec when it belongs to the current Config (after solve()), else at the current transforms
    ErrorReport error_report(const std::vector<double> &q = {0.5, 0.9, 0.99});
    // removes every detection whose error is above max_px and the frames left without an observation; cameras and markers that lose
    // all their observations stay (listed in `out`).  The handle is dropped: the next solve() creates it anew.  Returns the number removed.
    struct Rejection { long long removed = 0, observations = 0; std::vector<int> dropped_frames, unobserved_cams, unobserved_markers; };
    long long remove_outliers(double max_px, Rejection *out = nullptr);
    // not in the reference: hold these cameras / markers / frames (ids) fixed in solve().  Their Jacobian columns are explicit zeros
    // (aar_set_fixed, include/aar_cuda.h) and their Mat44 stay the caller's matrices byte for byte.  The sets persist across handles
    // (remove_outliers drops the frames it removes); track() ignores them.  An id the mapper does not hold throws std::invalid_argument.
    void set_fixed_cams(const std::set<int> &ids);
    void set_fixed_markers(const std::set<int> &ids);
    void set_fixed_frames(const std::set<int> &ids);
    // not in the reference: soft pose priors in solve() (aar_set_prior, include/aar_cuda.h): the pose T is known to sigma_rot (radians,
    // per rotation-vector component) and sigma_t (the solution's translation units); weights 1 / sigma^2, sigma = inf: no prior on that
    // part.  The maps replace the earlier ones and persist across handles (remove_outliers drops the frames it removes); track() ignores
    // them.  An id the mapper does not hold, or a sigma that is not > 0, throws std::invalid_argument.
    struct PosePrior { Mat44 T; double sigma_rot, sigma_t; };
    void set_cam_priors(const std::map<int, PosePrior> &priors);
    void set_marker_priors(const std::map<int, PosePrior> &priors);
    void set_frame_priors(const std::map<int, PosePrior> &priors);
    // not in the reference: soft relative-pose priors between two cameras or two markers in solve() (aar_set_pair_prior,
    // include/aar_cuda.h), keyed by the ids (a, b): T is T_ab = T_a^-1 T_b (b's coordinates into a's, e.g. a stereo pair's
    // calibration), known to sigma_rot (radians of relative rotation) and sigma_t (translation units); weights 1 / sigma^2,
    // sigma = inf: no prior on that part.  The maps replace the earlier ones and persist across handles; every solve() passes them to
    // its handle; track() ignores them.  An id the mapper does not hold, a == b, or a sigma that is not > 0 throws std::invalid_argument.
    struct PairPrior { Mat44 T; double sigma_rot, sigma_t; };
    void set_cam_pair_priors(const std::map<std::pair<int, int>, PairPrior> &priors);
    void set_marker_pair_priors(const std::map<std::pair<int, int>, PairPrior> &priors);
    void track();     // multicam_mapper.cpp:430-443: per-frame 6-dof solve against the fixed rig, every frame of the object at once

    bool write_solution_file(const std::string &path);         // byte-exact .solution (multicam_mapper.cpp:1053-1099)
    bool read_solution_file(const std::string &path);          // multicam_mapper.cpp:1124-1205
    void write_text_solution_file(const std::string &path);    // OpenCV FileStorage YAML (multicam_mapper.cpp:1233-1268)
    static void write_detections_file(const std::string &path, const std::vector<std::vector<std::vector<Marker>>> &seq);      // :216-237
    static std::vector<std::vector<std::vector<Marker>>> read_detections_file(const std::string &path, const std::vector<int> &subseqs = std::vector<int>());   // initializer.cpp:316-362
    static std::vector<int> read_subseqs(const std::string &path);                                                            // :46-55
    // pairwise camera transforms and per-frame ground-truth poses as (rotation vector, translation) records (:86-184)
    static int read_stereo_calib(const std::string &path, std::map<int, std::map<int, Mat44>> &transforms);                    // returns the root camera id
    static void write_stereo_calib(const std::string &path, const std::map<int, std::map<int, Mat44>> &transforms, int root_cam_id);
    static void read_ground_truth(const std::string &path, std::map<size_t, Mat44> &poses);
    static void write_ground_truth(const std::string &path, const std::map<size_t, Mat44> &poses);

    size_t get_root_cam() const { return root_cam; }
    size_t get_root_marker() const { return root_marker; }
    double get_marker_size() const { return marker_size; }

    std::vector<double> io_vec;                                 // the reference's public parameter vector (multicam_mapper.h:47)
    ucoslam::SparseLevMarq<double>::Params solver_params;       // multicam_mapper.cpp:326-330
    // solve()/track() report (the reference prints these, sparselevmarq.h:421)
    double initial_error = 0, final_error = 0; int iterations = 0;

    // id-ordered state (MatArrays, multicam_mapper.h:86-179)
    std::map<int, Mat44> transforms_to_root_cam, transforms_to_root_marker, object_to_global;
    std::map<int, CamConfig> cam_configs;
    FrameCamMarkers frame_cam_markers;                          // undistorted after init(), like the reference
    FrameCamMarkers raw_frame_cam_markers;                      // what init() received (empty after read_solution_file): the Jacobian's corners

private:
    void mats2eVec(const Config &conf, std::vector<double> &out) const;       // :445-461, R -> r like cv::Rodrigues
    void eVec2Mats_full(const std::vector<double> &in);                        // :595-606 for the full Config (solution files)
    void make_handle(bool corners_undistorted);
    void drop_handle();
    void pull_undistorted();
    void check(int rc, const char *what) const;

    Config config;
    std::set<int> fixed_cams, fixed_markers, fixed_frames;
    std::map<int, PosePrior> cam_priors, marker_priors, frame_priors;
    std::map<std::pair<int, int>, PairPrior> cam_pair_priors, marker_pair_priors;
    std::map<int, uint8_t> fixed_intrinsics;
    bool with_huber = false, corners_undistorted = false, analytic_jacobian = false, lens_model = false;
    size_t root_cam = 0, root_marker = 0;
    double marker_size = 0;
    aar_problem *handle = nullptr;
};

} // namespace aar
