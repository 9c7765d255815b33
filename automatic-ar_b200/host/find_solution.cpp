// find_solution — the reference's app (/root/reference/apps/find_solution.cpp:28-181) on the CUDA path, OpenCV-free:
//   find_solution <path_to_data_folder> <marker_size> [-subseqs] [-exclude-cams <cam_id> ...] [-with-huber] [-thresh <t>]
//                 [-consensus-max <k>] [-init <initial.solution>] [-analytic] [-reject-outliers <px>]
//                 [-fix-cams <cam_id> ...] [-fix-markers <marker_id> ...] [-fix-frames <frame_id> ...]
//                 [-prior-cams <file.solution> <sigma_rot_rad> <sigma_t>] [-prior-markers <file.solution> <sigma_rot_rad> <sigma_t>]
//                 [-stereo-prior <stereo_calib_file> <sigma_rot_rad> <sigma_t>] [-refine-intrinsics] [-fix-intrinsics <cam_id> ...] [-fix-p1p2k3]
// Reads <folder>/<cam>/calib.yml and <folder>/aruco.detections, builds the starting point with the Initializer (device: IPPE per
// detection + consensus; include/aar_init.h), writes initial<suffix>.solution(.yaml), solves on the GPU (include/aar_cuda.h) and
// writes final<suffix>.solution(.yaml) — the file names of find_solution.cpp:76-100.  Two additions: -consensus-max (SURVEY 8(f) row 3,
// the reference's exhaustive consensus is O(n^2) in the number of co-observations) and -init (start from an existing .solution
// instead of the detections) and -analytic (analytic Jacobian, residuals in double: include/aar_analytic.h; not the reference's arithmetic),
// -reject-outliers <px> (after the solve, remove the detections whose reprojection error is above px and solve again with the same settings;
// the final file holds the second solve), -fix-cams / -fix-markers / -fix-frames (hold those poses as they are in both solves, e.g. the
// calibrated cameras of a rig that gains one: MultiCamMapper::set_fixed_*), -prior-cams / -prior-markers (the soft form: the camera
// (marker) poses of an earlier calibration are priors with standard deviations sigma_rot in radians and sigma_t in translation units,
// for the ids both problems hold, in both solves: MultiCamMapper::set_*_priors; the file's root camera (marker) must be the problem's,
// since the poses are relative to it), -stereo-prior (the relative poses of a stereo-calibration file, MultiCamMapper::read_stereo_calib,
// are relative-pose priors: for every pair of camera ids i < j that the file and the problem both hold, transforms[i][j] is taken as
// T_ij = T_i^-1 T_j (j's coordinates into i's) with standard deviations sigma_rot in radians of relative rotation and sigma_t, in both
// solves: MultiCamMapper::set_cam_pair_priors; the file's root camera is ignored, relative poses do not depend on it; combines with
// -prior-cams), -refine-intrinsics (refine K and the five distortion coefficients of every camera on the raw corners in both solves:
// MultiCamMapper::set_lens_model, the lens model of the analytic mode; calib.yml's values are the start, and the written corners are
// undistorted with the refined coefficients; needs the detections, so -init is refused), -fix-intrinsics (with -refine-intrinsics:
// those cameras keep calib.yml's K and distortion) and -fix-p1p2k3 (with -refine-intrinsics: p1 p2 k3 of every camera stay calib.yml's,
// for corners that cover too little of the image to observe them).  Unlike the reference (whose option loop starts at argv[4]) options are read from argv[3] on.
#include <chrono>
#include <cmath>
#include <cstdio>
#include <iostream>
#include <set>

#include "initializer.h"
#include "multicam_mapper.h"

int main(int argc, char **argv) {
    if (argc < 3) {
        std::cout << "Usage: find_solution <path_to_data_folder> <marker_size> [-subseqs] [-exclude-cams <cam_id> ...] [-with-huber] [-thresh <t>] [-consensus-max <k>] [-init <file>] [-analytic] [-reject-outliers <px>] [-fix-cams <cam_id> ...] [-fix-markers <marker_id> ...] [-fix-frames <frame_id> ...] [-prior-cams <file.solution> <sigma_rot_rad> <sigma_t>] [-prior-markers <file.solution> <sigma_rot_rad> <sigma_t>] [-stereo-prior <stereo_calib_file> <sigma_rot_rad> <sigma_t>] [-refine-intrinsics] [-fix-intrinsics <cam_id> ...] [-fix-p1p2k3]" << std::endl;
        return -1;
    }
    const std::string folder = argv[1];
    const double marker_size = std::stod(argv[2]);
    bool use_subseqs = false, with_huber = false, set_threshold = false, analytic = false, refine_intrinsics = false, fix_p1p2k3 = false; double threshold = 2.0; int consensus_max = 0; double reject_px = -1;
    std::set<int> excluded_cams, fix_cams, fix_markers, fix_frames, fix_intrinsics; std::string init_path;
    struct PriorFile { std::string path; double sigma_rot = 0, sigma_t = 0; } prior_cams, prior_markers, stereo_prior;
    PriorFile *prior = nullptr; int prior_arg = 0;             // the -prior-* / -stereo-prior option being read and how many of its 3 arguments were read
    enum { NONE, EXCLUDE, THRESH, CMAX, INIT, REJECT, FIXC, FIXM, FIXF, FIXI, PRIOR } flag = NONE;
    for (int i = 3; i < argc; i++) {
        const std::string a = argv[i];
        if (a == "-subseqs") { use_subseqs = true; flag = NONE; }
        else if (a == "-exclude-cams") flag = EXCLUDE;
        else if (a == "-with-huber") { with_huber = true; flag = NONE; }
        else if (a == "-analytic") { analytic = true; flag = NONE; }
        else if (a == "-thresh") { set_threshold = true; flag = THRESH; }
        else if (a == "-consensus-max") flag = CMAX;
        else if (a == "-init") flag = INIT;
        else if (a == "-reject-outliers") flag = REJECT;
        else if (a == "-fix-cams") flag = FIXC;
        else if (a == "-fix-markers") flag = FIXM;
        else if (a == "-fix-frames") flag = FIXF;
        else if (a == "-refine-intrinsics") { refine_intrinsics = true; flag = NONE; }
        else if (a == "-fix-intrinsics") flag = FIXI;
        else if (a == "-fix-p1p2k3") { fix_p1p2k3 = true; flag = NONE; }
        else if (a == "-prior-cams" || a == "-prior-markers") { flag = PRIOR; prior = a == "-prior-cams" ? &prior_cams : &prior_markers; prior_arg = 0; }
        else if (a == "-stereo-prior") { flag = PRIOR; prior = &stereo_prior; prior_arg = 0; }
        else if (flag == PRIOR) {
            if (prior_arg == 0) prior->path = a; else if (prior_arg == 1) prior->sigma_rot = std::stod(a); else prior->sigma_t = std::stod(a);
            if (++prior_arg == 3) flag = NONE;
        }
        else if (flag == EXCLUDE) excluded_cams.insert(std::stoi(a));
        else if (flag == FIXC) fix_cams.insert(std::stoi(a));
        else if (flag == FIXM) fix_markers.insert(std::stoi(a));
        else if (flag == FIXF) fix_frames.insert(std::stoi(a));
        else if (flag == FIXI) fix_intrinsics.insert(std::stoi(a));
        else if (flag == THRESH) { threshold = std::stod(a); flag = NONE; }
        else if (flag == CMAX) { consensus_max = std::stoi(a); flag = NONE; }
        else if (flag == INIT) { init_path = a; flag = NONE; }
        else if (flag == REJECT) { reject_px = std::stod(a); flag = NONE; }
    }
    if (refine_intrinsics && !init_path.empty()) {
        std::cerr << "find_solution: -refine-intrinsics needs the raw detections; a .solution file (-init) holds undistorted corners only" << std::endl;
        return 1;
    }
    std::string suffix;                                         // find_solution.cpp:76-100
    if (use_subseqs) suffix += "_subseqs";
    if (with_huber) suffix += "_with_huber";
    if (!excluded_cams.empty()) { suffix += "_excluded_cams"; for (int c : excluded_cams) suffix += "_" + std::to_string(c); }
    if (set_threshold) { char d[16]; std::snprintf(d, sizeof d, "%.1f", threshold); suffix += "_thresh_" + std::string(d); }
    suffix += ".solution";
    const std::string initial_path = folder + "/initial" + suffix, final_path = folder + "/final" + suffix;
    try {
        std::chrono::duration<double> d(0);
        aar::MultiCamMapper mcm;
        if (!init_path.empty()) {
            if (!mcm.read_solution_file(init_path)) return 1;
            if (std::fabs(marker_size - mcm.get_marker_size()) > 1e-6) std::cout << "note: marker size of the solution file is " << mcm.get_marker_size() << std::endl;
        } else {
            std::vector<aar::CamConfig> cam_configs = aar::CamConfig::read_cam_configs(folder);
            if (cam_configs.empty()) { std::cerr << "find_solution: no <cam>/calib.yml under " << folder << std::endl; return 1; }
            std::vector<int> subseqs;
            if (use_subseqs) subseqs = aar::MultiCamMapper::read_subseqs(folder + "/subseqs.txt");
            aar::Initializer::Detections detections = aar::Initializer::read_detections_file(folder + "/aruco.detections", subseqs);
            auto start = std::chrono::system_clock::now();
            aar::Initializer initializer(marker_size, cam_configs, excluded_cams);
            initializer.threshold = threshold; initializer.consensus_max = consensus_max;
            initializer.set_detections(detections);
            initializer.obtain_pose_estimations();
            initializer.init_transforms();
            mcm.init((size_t)initializer.get_root_cam(), initializer.get_transforms_to_root_cam(), (size_t)initializer.get_root_marker(), initializer.get_transforms_to_root_marker(),
                     initializer.get_object_transforms(), initializer.get_frame_cam_markers(), (float)initializer.get_marker_size(), initializer.get_cam_configs());
            d += std::chrono::system_clock::now() - start;
            std::cout << "initialised " << initializer.get_transforms_to_root_cam().size() << " cameras, " << initializer.get_transforms_to_root_marker().size()
                      << " markers, " << initializer.get_object_transforms().size() << " frames" << std::endl;
            mcm.write_solution_file(initial_path);
            mcm.write_text_solution_file(initial_path + ".yaml");
        }
        mcm.set_optmize_flag_cam_poses(true); mcm.set_optmize_flag_marker_poses(true); mcm.set_optmize_flag_object_poses(true);
        mcm.set_optmize_flag_cam_intrinsics(false);              // find_solution.cpp:140
        if (with_huber) mcm.set_with_huber(true);
        if (analytic) mcm.set_analytic_jacobian(true);
        if (refine_intrinsics) {
            mcm.set_optmize_flag_cam_intrinsics(true);
            mcm.set_lens_model(true);
            std::map<int, uint8_t> held;
            if (fix_p1p2k3) for (auto &p : mcm.transforms_to_root_cam) held[p.first] = 2;
            for (int c : fix_intrinsics) held[c] = 3;
            mcm.set_fixed_intrinsics(held);
        }
        mcm.set_fixed_cams(fix_cams); mcm.set_fixed_markers(fix_markers); mcm.set_fixed_frames(fix_frames);
        for (int k = 0; k < 2; k++) {                             // -prior-cams, -prior-markers
            const PriorFile &pf = k ? prior_markers : prior_cams;
            if (pf.path.empty()) continue;
            aar::MultiCamMapper ref;
            if (!ref.read_solution_file(pf.path)) return 1;
            const size_t root = k ? ref.get_root_marker() : ref.get_root_cam(), want = k ? mcm.get_root_marker() : mcm.get_root_cam();
            if (root != want) {
                std::cerr << "find_solution: the root " << (k ? "marker" : "camera") << " of " << pf.path << " is " << root << ", the problem's is " << want
                          << ": its poses are relative to another root" << std::endl;
                return 1;
            }
            const std::map<int, aar::Mat44> &from = k ? ref.transforms_to_root_marker : ref.transforms_to_root_cam, &held = k ? mcm.transforms_to_root_marker : mcm.transforms_to_root_cam;
            std::map<int, aar::MultiCamMapper::PosePrior> priors;
            for (auto &e : from) if (held.count(e.first)) priors[e.first] = aar::MultiCamMapper::PosePrior{e.second, pf.sigma_rot, pf.sigma_t};
            if (k) mcm.set_marker_priors(priors); else mcm.set_cam_priors(priors);
            std::cout << "priors on " << priors.size() << (k ? " markers" : " cameras") << std::endl;
        }
        if (!stereo_prior.path.empty()) {                         // -stereo-prior
            std::map<int, std::map<int, aar::Mat44>> tr;
            aar::MultiCamMapper::read_stereo_calib(stereo_prior.path, tr);
            std::map<std::pair<int, int>, aar::MultiCamMapper::PairPrior> pairs;
            for (auto &a : tr) {
                if (!mcm.transforms_to_root_cam.count(a.first)) continue;
                for (auto &b : a.second)
                    if (a.first < b.first && mcm.transforms_to_root_cam.count(b.first))
                        pairs[{a.first, b.first}] = aar::MultiCamMapper::PairPrior{b.second, stereo_prior.sigma_rot, stereo_prior.sigma_t};
            }
            mcm.set_cam_pair_priors(pairs);
            std::cout << "pair priors on " << pairs.size() << " camera pairs" << std::endl;
        }
        auto start = std::chrono::system_clock::now();
        mcm.solve();
        d += std::chrono::system_clock::now() - start;
        std::cout.precision(17); std::cout << "final_error: " << mcm.final_error << " iterations: " << mcm.iterations << std::endl;
        if (reject_px >= 0) {
            start = std::chrono::system_clock::now();
            aar::MultiCamMapper::Rejection rj;
            mcm.remove_outliers(reject_px, &rj);
            std::printf("removed %lld of %lld detections above %.17g px\n", rj.removed, rj.observations, reject_px); std::fflush(stdout);
            mcm.solve();
            d += std::chrono::system_clock::now() - start;
            std::cout << "final_error: " << mcm.final_error << " iterations: " << mcm.iterations << std::endl;
        }
        mcm.write_solution_file(final_path);
        mcm.write_text_solution_file(final_path + ".yaml");
        const int minutes = (int)(d.count() / 60); const long seconds = std::lround(d.count() - minutes * 60);
        std::cout << "The algorithm took: " << minutes << " minutes " << seconds << " seconds" << std::endl;
    } catch (const std::exception &e) { std::cerr << "find_solution: " << e.what() << std::endl; return 2; }
    return 0;
}
