// multicam_mapper.cpp — see multicam_mapper.h.  Reference line numbers are into /root/reference/libs/multicam_mapper.cpp.
#include "multicam_mapper.h"
#include "initializer.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <dirent.h>
#include <fstream>
#include <iostream>
#include <sstream>

#include "../../include/aar_crsincos.h"
#include "../csrc/aar_host_math.h"

namespace aar {

namespace {
template <typename T> void wr(std::ofstream &f, const T &v) { f.write(reinterpret_cast<const char *>(&v), sizeof v); }
template <typename T> bool rd(std::ifstream &f, T &v) { f.read(reinterpret_cast<char *>(&v), sizeof v); return (size_t)f.gcount() == sizeof v; }
void write_marker(std::ofstream &f, const Marker &m) { wr(f, m.id); for (int i = 0; i < 8; i++) wr(f, m.xy[i]); }     // aruco_serdes.cpp:9-15
bool read_marker(std::ifstream &f, Marker &m) { if (!rd(f, m.id)) return false; for (int i = 0; i < 8; i++) if (!rd(f, m.xy[i])) return false; return true; }

// cv::Rodrigues(vector -> matrix), same operation order as the device (aar_device_math.cuh)
void vec2rot(const double *r, double *R) {
    double rx = r[0], ry = r[1], rz = r[2];
    const double theta = std::sqrt(rx * rx + ry * ry + rz * rz);
    if (theta < 2.2204460492503131e-16) { for (int i = 0; i < 9; i++) R[i] = (i % 4 == 0) ? 1.0 : 0.0; return; }
    double s, c; aar_sincos(theta, &s, &c);
    const double c1 = 1. - c, it = 1. / theta;
    rx *= it; ry *= it; rz *= it;
    R[0] = c + c1 * (rx * rx); R[1] = c1 * (rx * ry) + s * (-rz); R[2] = c1 * (rx * rz) + s * ry;
    R[3] = c1 * (rx * ry) + s * rz; R[4] = c + c1 * (ry * ry); R[5] = c1 * (ry * rz) + s * (-rx);
    R[6] = c1 * (rx * rz) + s * (-ry); R[7] = c1 * (ry * rz) + s * rx; R[8] = c + c1 * (rz * rz);
}
void mat2vec6(const Mat44 &T, double *v) {     // transformation_mat2vec :475-486
    double R[9];
    for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) R[i * 3 + j] = T.at(i, j);
    aar_host::rotation_to_vector(R, v);
    for (int i = 0; i < 3; i++) v[3 + i] = T.at(i, 3);
}
Mat44 vec62mat(const double *v) {               // vec2transformation_mat :463-473
    Mat44 T; double R[9]; vec2rot(v, R);
    for (int i = 0; i < 3; i++) { for (int j = 0; j < 3; j++) T.at(i, j) = R[i * 3 + j]; T.at(i, 3) = v[3 + i]; }
    return T;
}
std::string num(double v) {                     // shortest round-trip style, a trailing '.' marks integers like cv::FileStorage
    char buf[40]; std::snprintf(buf, sizeof buf, "%.17g", v);
    std::string s(buf);
    if (s.find_first_of(".enai") == std::string::npos) s += ".";
    return s;
}
} // namespace

// ------------------------------------------------------------------------------- CamConfig
bool CamConfig::read_from_file(const std::string &path) {
    std::ifstream f(path);
    if (!f.is_open()) return false;
    std::stringstream ss; ss << f.rdbuf();
    const std::string txt = ss.str();
    auto scalar = [&](const std::string &key, int &out) {
        size_t p = txt.find(key + ":"); if (p == std::string::npos) return false;
        out = std::atoi(txt.c_str() + p + key.size() + 1); return true;
    };
    auto matrix = [&](const std::string &key, double *out, int n) {
        size_t p = txt.find(key + ":"); if (p == std::string::npos) return false;
        size_t a = txt.find("data:", p); if (a == std::string::npos) return false;
        a = txt.find('[', a); size_t b = txt.find(']', a); if (a == std::string::npos || b == std::string::npos) return false;
        std::string body = txt.substr(a + 1, b - a - 1);
        std::replace(body.begin(), body.end(), ',', ' ');
        std::stringstream vs(body); int k = 0; double v;
        while (k < n && (vs >> v)) out[k++] = v;
        for (; k < n; k++) out[k] = 0;      // distortion vectors shorter than 5 are zero padded (setDistCoeffs)
        return true;
    };
    if (!scalar("image_height", height) || !scalar("image_width", width)) return false;
    if (!matrix("camera_matrix", K, 9) || !matrix("distortion_coefficients", dist, 5)) return false;
    return true;
}
std::vector<CamConfig> CamConfig::read_cam_configs(const std::string &folder) {
    // The reference lists the folder in readdir order (libs/filesystem.cpp:5-17) while everything else indexes
    // cam_configs[cam_id]; sorting numerically is the documented deviation (SURVEY Appendix A.2).
    std::vector<int> ids;
    if (DIR *d = opendir(folder.c_str())) {
        while (dirent *e = readdir(d)) { char *end = nullptr; long v = std::strtol(e->d_name, &end, 10); if (end != e->d_name && *end == 0) ids.push_back((int)v); }
        closedir(d);
    }
    std::sort(ids.begin(), ids.end());
    std::vector<CamConfig> out;
    for (int id : ids)
        for (const char *ext : {"yml", "yaml"}) {
            CamConfig cc;
            if (cc.read_from_file(folder + "/" + std::to_string(id) + "/calib." + ext)) { out.push_back(cc); break; }
        }
    return out;
}

// ------------------------------------------------------------------------------- MultiCamMapper
MultiCamMapper::MultiCamMapper() {}
MultiCamMapper::MultiCamMapper(Initializer &in) {                            // :252-254
    init((size_t)in.get_root_cam(), in.get_transforms_to_root_cam(), (size_t)in.get_root_marker(), in.get_transforms_to_root_marker(), in.get_object_transforms(),
         in.get_frame_cam_markers(), (float)in.get_marker_size(), in.get_cam_configs());
}
MultiCamMapper::MultiCamMapper(size_t root_c, const std::map<int, Mat44> &Tc, size_t root_m, const std::map<int, Mat44> &Tm, const std::map<int, Mat44> &To,
                               const FrameCamMarkers &fcm, float m_size, const std::vector<CamConfig> &cc) { init(root_c, Tc, root_m, Tm, To, fcm, m_size, cc); }
MultiCamMapper::~MultiCamMapper() { drop_handle(); }

void MultiCamMapper::check(int rc, const char *what) const {
    if (rc != AAR_OK) throw std::runtime_error(std::string(what) + ": " + aar_last_error());
}
void MultiCamMapper::drop_handle() { if (handle) { aar_problem_destroy(handle); handle = nullptr; } }

size_t MultiCamMapper::get_num_vars(const Config &c) const {     // :239-250
    size_t n = 0;
    if (c.optimize_cam_poses) n += (transforms_to_root_cam.size() - 1) * 6;
    if (c.optimize_marker_poses) n += (transforms_to_root_marker.size() - 1) * 6;
    if (c.optimize_object_poses) n += object_to_global.size() * 6;
    if (c.optimize_cam_intrinsics) n += transforms_to_root_cam.size() * 9;
    return n;
}

void MultiCamMapper::init(size_t root_c, const std::map<int, Mat44> &Tc, size_t root_m, const std::map<int, Mat44> &Tm, const std::map<int, Mat44> &To,
                          const FrameCamMarkers &fcm, float m_size, const std::vector<CamConfig> &cc) {
    drop_handle();
    root_cam = root_c; root_marker = root_m; marker_size = m_size;
    transforms_to_root_cam = Tc; transforms_to_root_marker = Tm; object_to_global = To; frame_cam_markers = fcm; raw_frame_cam_markers = fcm;
    cam_configs.clear();
    for (auto &p : transforms_to_root_cam) {                     // cam_mats[i] = cam_confs[cam_id] (:314-316)
        if (p.first < 0 || (size_t)p.first >= cc.size()) throw std::runtime_error("no CamConfig for camera " + std::to_string(p.first));
        cam_configs[p.first] = cc[(size_t)p.first];
    }
    corners_undistorted = false;
    make_handle(false);
    pull_undistorted();                                          // remove_distortions (:554-578) ran on the device
}

void MultiCamMapper::init(const std::map<int, Mat44> &object_poses, const FrameCamMarkers &fcm) {
    drop_handle();
    object_to_global = object_poses; frame_cam_markers = fcm; raw_frame_cam_markers = fcm;
    corners_undistorted = false;
    make_handle(false);
    pull_undistorted();
}

void MultiCamMapper::make_handle(bool undist) {
    drop_handle();
    std::vector<int> cam_ids, marker_ids, frame_ids, df, dc, dm;
    std::vector<double> Tc, Tm, To, K, D;
    std::vector<float> xy;
    for (auto &p : transforms_to_root_cam) { cam_ids.push_back(p.first); Tc.insert(Tc.end(), p.second.m, p.second.m + 16); const CamConfig &c = cam_configs.at(p.first); K.insert(K.end(), c.K, c.K + 9); D.insert(D.end(), c.dist, c.dist + 5); }
    for (auto &p : transforms_to_root_marker) { marker_ids.push_back(p.first); Tm.insert(Tm.end(), p.second.m, p.second.m + 16); }
    for (auto &p : object_to_global) { frame_ids.push_back(p.first); To.insert(To.end(), p.second.m, p.second.m + 16); }
    // The reference's inverted indices keep the RAW corners (fill_iteration_arrays :304 runs before remove_distortions :322) and its
    // Jacobian differences them (obtain_marker_derivs :981-989): whenever this object was initialised from raw detections the handle
    // is rebuilt from them (the device undistorts again, deterministically); only a .solution file has nothing but undistorted corners.
    const bool from_raw = !raw_frame_cam_markers.empty();
    if (from_raw) undist = false;
    for (auto &f : (from_raw ? raw_frame_cam_markers : frame_cam_markers))
        for (auto &c : f.second)
            for (auto &mk : c.second) { df.push_back(f.first); dc.push_back(c.first); dm.push_back(mk.id); xy.insert(xy.end(), mk.xy, mk.xy + 8); }
    aar_problem_desc d; std::memset(&d, 0, sizeof d);
    d.num_cams = (int)cam_ids.size(); d.num_markers = (int)marker_ids.size(); d.num_frames = (int)frame_ids.size();
    d.cam_ids = cam_ids.data(); d.marker_ids = marker_ids.data(); d.frame_ids = frame_ids.data();
    d.root_cam = (int)root_cam; d.root_marker = (int)root_marker; d.marker_size = (float)marker_size;
    d.cam_T = Tc.data(); d.marker_T = Tm.data(); d.frame_T = To.data(); d.cam_K = K.data(); d.cam_dist = D.data();
    d.num_detections = (int64_t)df.size(); d.det_frame = df.data(); d.det_cam = dc.data(); d.det_marker = dm.data(); d.det_xy = xy.data();
    d.optimize_cam_poses = config.optimize_cam_poses; d.optimize_marker_poses = config.optimize_marker_poses; d.optimize_object_poses = config.optimize_object_poses;
    d.optimize_cam_intrinsics = config.optimize_cam_intrinsics; d.with_huber = with_huber; d.corners_undistorted = undist; d.analytic_jacobian = analytic_jacobian || lens_model;
    d.lens_model = lens_model ? 1 : 0;
    d.J_delta = 1e-3; d.device = 0; d.world_size = 1;
    check(aar_problem_create(&d, &handle), "aar_problem_create");
}

void MultiCamMapper::pull_undistorted() {
    // fill_iteration_arrays (:345-377) erases detections of unknown cameras / markers; the device row order is the
    // order of what remains
    for (auto f = frame_cam_markers.begin(); f != frame_cam_markers.end();) {
        if (!object_to_global.count(f->first)) { f = frame_cam_markers.erase(f); continue; }
        for (auto c = f->second.begin(); c != f->second.end();) {
            if (!transforms_to_root_cam.count(c->first)) { c = f->second.erase(c); continue; }
            auto &v = c->second;
            v.erase(std::remove_if(v.begin(), v.end(), [&](const Marker &m) { return !transforms_to_root_marker.count(m.id); }), v.end());
            ++c;
        }
        ++f;
    }
    const size_t n = (size_t)aar_num_local_observations(handle);
    std::vector<float> und(8 * n);
    check(aar_get_observations(handle, und.data(), nullptr), "aar_get_observations");
    size_t o = 0;
    for (auto &f : frame_cam_markers) for (auto &c : f.second) for (auto &mk : c.second) { if (o >= n) throw std::runtime_error("row map mismatch"); std::memcpy(mk.xy, &und[8 * o], 8 * sizeof(float)); o++; }
    if (o != n) throw std::runtime_error("row map mismatch");
    corners_undistorted = true;      // from now on the host copy holds undistorted corners; the live handle still has the raw ones
}

void MultiCamMapper::mats2eVec(const Config &c, std::vector<double> &out) const {    // :445-461, :488-522
    out.assign(get_num_vars(c), 0.0);
    size_t vi = 0;
    if (c.optimize_cam_poses) for (auto &p : transforms_to_root_cam) if ((size_t)p.first != root_cam) { mat2vec6(p.second, &out[vi]); vi += 6; }
    if (c.optimize_marker_poses) for (auto &p : transforms_to_root_marker) if ((size_t)p.first != root_marker) { mat2vec6(p.second, &out[vi]); vi += 6; }
    if (c.optimize_object_poses) for (auto &p : object_to_global) { mat2vec6(p.second, &out[vi]); vi += 6; }
    if (c.optimize_cam_intrinsics)
        for (auto &p : transforms_to_root_cam) {                 // [fx cx fy cy k1 k2 p1 p2 k3] (:510-522)
            const CamConfig &cc = cam_configs.at(p.first);
            out[vi] = cc.K[0]; out[vi + 1] = cc.K[2]; out[vi + 2] = cc.K[4]; out[vi + 3] = cc.K[5];
            for (int k = 0; k < 5; k++) out[vi + 4 + k] = cc.dist[k];
            vi += 9;
        }
}

void MultiCamMapper::eVec2Mats_full(const std::vector<double> &in) {
    size_t vi = 0;
    for (auto &p : transforms_to_root_cam) { if ((size_t)p.first == root_cam) { p.second = Mat44(); continue; } p.second = vec62mat(&in[vi]); vi += 6; }
    for (auto &p : transforms_to_root_marker) { if ((size_t)p.first == root_marker) { p.second = Mat44(); continue; } p.second = vec62mat(&in[vi]); vi += 6; }
    for (auto &p : object_to_global) { p.second = vec62mat(&in[vi]); vi += 6; }
    for (auto &p : transforms_to_root_cam) {
        CamConfig &cc = cam_configs[p.first];
        std::memset(cc.K, 0, sizeof cc.K); cc.K[8] = 1;
        cc.K[0] = in[vi]; cc.K[2] = in[vi + 1]; cc.K[4] = in[vi + 2]; cc.K[5] = in[vi + 3];
        for (int k = 0; k < 5; k++) cc.dist[k] = in[vi + 4 + k];
        vi += 9;
    }
}

static void check_ids(const std::set<int> &ids, const std::map<int, Mat44> &held, const char *what) {
    for (int id : ids) if (!held.count(id)) throw std::invalid_argument(std::string("set_fixed_") + what + ": no " + what + " with id " + std::to_string(id));
}
void MultiCamMapper::set_fixed_cams(const std::set<int> &ids) { check_ids(ids, transforms_to_root_cam, "cams"); fixed_cams = ids; }
void MultiCamMapper::set_fixed_markers(const std::set<int> &ids) { check_ids(ids, transforms_to_root_marker, "markers"); fixed_markers = ids; }
void MultiCamMapper::set_fixed_frames(const std::set<int> &ids) { check_ids(ids, object_to_global, "frames"); fixed_frames = ids; }

static void check_priors(const std::map<int, MultiCamMapper::PosePrior> &priors, const std::map<int, Mat44> &held, const char *what) {
    for (auto &p : priors) {
        const std::string name = std::string("set_") + what + "_priors: ";
        if (!held.count(p.first)) throw std::invalid_argument(name + "no " + what + " with id " + std::to_string(p.first));
        if (!(p.second.sigma_rot > 0) || !(p.second.sigma_t > 0)) throw std::invalid_argument(name + "sigma of id " + std::to_string(p.first) + " is not > 0");
    }
}
void MultiCamMapper::set_lens_model(bool v) {
    if (v && raw_frame_cam_markers.empty()) throw std::logic_error("set_lens_model: the mapper holds no raw corners (a .solution file stores undistorted ones)");
    lens_model = v; drop_handle();
}
void MultiCamMapper::set_fixed_intrinsics(const std::map<int, uint8_t> &flags) {
    for (auto &p : flags) {
        if (!transforms_to_root_cam.count(p.first)) throw std::invalid_argument("set_fixed_intrinsics: no cams with id " + std::to_string(p.first));
        if (p.second > 3) throw std::invalid_argument("set_fixed_intrinsics: flags " + std::to_string((int)p.second) + " of camera " + std::to_string(p.first) + " (bit 0: fx cx fy cy k1 k2, bit 1: p1 p2 k3)");
    }
    fixed_intrinsics = flags;
}

void MultiCamMapper::set_cam_priors(const std::map<int, PosePrior> &priors) { check_priors(priors, transforms_to_root_cam, "cam"); cam_priors = priors; }
void MultiCamMapper::set_marker_priors(const std::map<int, PosePrior> &priors) { check_priors(priors, transforms_to_root_marker, "marker"); marker_priors = priors; }
void MultiCamMapper::set_frame_priors(const std::map<int, PosePrior> &priors) { check_priors(priors, object_to_global, "frame"); frame_priors = priors; }

static void check_pair_priors(const std::map<std::pair<int, int>, MultiCamMapper::PairPrior> &priors, const std::map<int, Mat44> &held, const char *what) {
    for (auto &p : priors) {
        const std::string name = std::string("set_") + what + "_pair_priors: ", ids = "(" + std::to_string(p.first.first) + ", " + std::to_string(p.first.second) + ")";
        for (int id : {p.first.first, p.first.second})
            if (!held.count(id)) throw std::invalid_argument(name + "no " + what + " with id " + std::to_string(id));
        if (p.first.first == p.first.second) throw std::invalid_argument(name + "pair " + ids + " joins a " + what + " with itself");
        if (!(p.second.sigma_rot > 0) || !(p.second.sigma_t > 0)) throw std::invalid_argument(name + "sigma of pair " + ids + " is not > 0");
    }
}
void MultiCamMapper::set_cam_pair_priors(const std::map<std::pair<int, int>, PairPrior> &priors) { check_pair_priors(priors, transforms_to_root_cam, "cam"); cam_pair_priors = priors; }
void MultiCamMapper::set_marker_pair_priors(const std::map<std::pair<int, int>, PairPrior> &priors) { check_pair_priors(priors, transforms_to_root_marker, "marker"); marker_pair_priors = priors; }

void MultiCamMapper::solve() {
    if (!handle) make_handle(corners_undistorted);
    {   // aar_set_fixed: one byte per camera / marker / frame in id order; NULL for an empty set, all NULL clears
        auto mask = [](const std::set<int> &ids, const std::map<int, Mat44> &held) {
            std::vector<uint8_t> m; if (ids.empty()) return m;
            for (auto &p : held) m.push_back(ids.count(p.first) ? 1 : 0);
            return m;
        };
        const std::vector<uint8_t> c = mask(fixed_cams, transforms_to_root_cam), m = mask(fixed_markers, transforms_to_root_marker), f = mask(fixed_frames, object_to_global);
        check(aar_set_fixed(handle, c.empty() ? nullptr : c.data(), m.empty() ? nullptr : m.data(), f.empty() ? nullptr : f.data()), "aar_set_fixed");
        if (config.optimize_cam_intrinsics) {                   // aar_set_fixed_intrinsics: flags per camera in id order, NULL for none
            std::vector<uint8_t> fi;
            if (!fixed_intrinsics.empty()) for (auto &p : transforms_to_root_cam) { auto it = fixed_intrinsics.find(p.first); fi.push_back(it == fixed_intrinsics.end() ? 0 : it->second); }
            check(aar_set_fixed_intrinsics(handle, fi.empty() ? nullptr : fi.data()), "aar_set_fixed_intrinsics");
        }
    }
    {   // aar_set_prior: targets [n][16] and weights 1 / sigma^2 [n][6] in id order (0 where an entity has no prior); NULL for an empty map
        struct Arrays { std::vector<double> T, w; const double *t() const { return w.empty() ? nullptr : T.data(); } const double *wp() const { return w.empty() ? nullptr : w.data(); } };
        auto arrays = [](const std::map<int, PosePrior> &priors, const std::map<int, Mat44> &held) {
            Arrays a; if (priors.empty()) return a;
            a.T.assign(16 * held.size(), 0.0); a.w.assign(6 * held.size(), 0.0);
            size_t i = 0;
            for (auto &p : held) {
                auto it = priors.find(p.first);
                if (it != priors.end()) {
                    std::memcpy(&a.T[16 * i], it->second.T.m, sizeof it->second.T.m);
                    const double wr = 1.0 / (it->second.sigma_rot * it->second.sigma_rot), wt = 1.0 / (it->second.sigma_t * it->second.sigma_t);
                    for (int k = 0; k < 3; k++) { a.w[6 * i + k] = wr; a.w[6 * i + 3 + k] = wt; }
                }
                i++;
            }
            return a;
        };
        const Arrays c = arrays(cam_priors, transforms_to_root_cam), m = arrays(marker_priors, transforms_to_root_marker), f = arrays(frame_priors, object_to_global);
        check(aar_set_prior(handle, c.t(), c.wp(), m.t(), m.wp(), f.t(), f.wp()), "aar_set_prior");
    }
    {   // aar_set_pair_prior: index pairs [n][2] (ranks of the ids), targets [n][16], weights 1 / sigma^2 [n][2] in map order
        struct Arrays { std::vector<int32_t> ab; std::vector<double> T, w; };
        auto arrays = [](const std::map<std::pair<int, int>, PairPrior> &priors, const std::map<int, Mat44> &held) {
            Arrays a;
            auto rank = [&](int id) { return (int32_t)std::distance(held.begin(), held.find(id)); };
            for (auto &p : priors) {
                a.ab.push_back(rank(p.first.first)); a.ab.push_back(rank(p.first.second));
                a.T.insert(a.T.end(), p.second.T.m, p.second.T.m + 16);
                a.w.push_back(1.0 / (p.second.sigma_rot * p.second.sigma_rot)); a.w.push_back(1.0 / (p.second.sigma_t * p.second.sigma_t));
            }
            return a;
        };
        const Arrays c = arrays(cam_pair_priors, transforms_to_root_cam), m = arrays(marker_pair_priors, transforms_to_root_marker);
        check(aar_set_pair_prior(handle, (int32_t)cam_pair_priors.size(), c.ab.data(), c.T.data(), c.w.data(),
                                 (int32_t)marker_pair_priors.size(), m.ab.data(), m.T.data(), m.w.data()), "aar_set_pair_prior");
    }
    io_vec.assign((size_t)aar_num_vars(handle), 0.0);
    check(aar_mats2evec(handle, io_vec.data()), "aar_mats2evec");
    aar_lm_params prm; aar_lm_default_params(&prm);
    prm.max_iters = solver_params.maxIters; prm.min_error = solver_params.minError; prm.min_step_error_diff = solver_params.min_step_error_diff;
    prm.min_average_step_error_diff = solver_params.min_average_step_error_diff; prm.tau = solver_params.tau; prm.der_epsilon = solver_params.der_epsilon;
    prm.verbose = solver_params.verbose;
    aar_lm_report rep; std::memset(&rep, 0, sizeof rep);
    check(aar_lm_solve(handle, io_vec.data(), &prm, &rep), "aar_lm_solve");
    initial_error = rep.initial_cost; final_error = rep.final_cost; iterations = rep.iterations;
    std::cout << "initial_error: " << initial_error << " error size: " << 8 * aar_num_observations(handle) << std::endl;   // :424
    // eVec2Mats (:427)
    const size_t C = transforms_to_root_cam.size(), M = transforms_to_root_marker.size(), F = object_to_global.size();
    std::vector<double> Tc(16 * C), Tm(16 * M), To(16 * F);
    check(aar_evec2mats(handle, io_vec.data(), Tc.data(), Tm.data(), To.data()), "aar_evec2mats");
    // fixed entities keep the caller's matrices: r -> R of the device expansion does not give back the R the vector was taken from
    size_t i = 0;
    if (config.optimize_cam_poses) for (auto &p : transforms_to_root_cam) { if (!fixed_cams.count(p.first)) std::memcpy(p.second.m, &Tc[16 * i], sizeof p.second.m); i++; }
    i = 0;
    if (config.optimize_marker_poses) for (auto &p : transforms_to_root_marker) { if (!fixed_markers.count(p.first)) std::memcpy(p.second.m, &Tm[16 * i], sizeof p.second.m); i++; }
    i = 0;
    if (config.optimize_object_poses) for (auto &p : object_to_global) { if (!fixed_frames.count(p.first)) std::memcpy(p.second.m, &To[16 * i], sizeof p.second.m); i++; }
    if (config.optimize_cam_intrinsics) {                        // intrinsics_vec2mats (:580-593): the last 9 entries per camera
        size_t vi = io_vec.size() - 9 * C;
        for (auto &p : transforms_to_root_cam) {
            CamConfig &cc = cam_configs[p.first];
            auto it = fixed_intrinsics.find(p.first);
            const int held = it == fixed_intrinsics.end() ? 0 : it->second;     // held parts keep the caller's bytes
            if (!(held & 1)) { cc.K[0] = io_vec[vi]; cc.K[2] = io_vec[vi + 1]; cc.K[4] = io_vec[vi + 2]; cc.K[5] = io_vec[vi + 3]; cc.dist[0] = io_vec[vi + 4]; cc.dist[1] = io_vec[vi + 5]; }
            if (!(held & 2)) { cc.dist[2] = io_vec[vi + 6]; cc.dist[3] = io_vec[vi + 7]; cc.dist[4] = io_vec[vi + 8]; }
            vi += 9;
        }
        if (lens_model) {
            // the undistorted copy of the corners follows the refined coefficients: a handle built from the raw corners with them
            // runs remove_distortions again (it also serves the next solve, which starts from the refined intrinsics)
            const std::vector<double> z = io_vec;
            frame_cam_markers = raw_frame_cam_markers;
            make_handle(false);
            pull_undistorted();
            io_vec = z;
        }
    }
}

MultiCamMapper::ErrorReport MultiCamMapper::error_report(const std::vector<double> &q) {
    if (!handle) make_handle(corners_undistorted);
    if (io_vec.size() != (size_t)aar_num_vars(handle)) mats2eVec(config, io_vec);
    ErrorReport r;
    const size_t C = transforms_to_root_cam.size(), M = transforms_to_root_marker.size(), F = object_to_global.size();
    size_t nd = 0;
    for (auto &f : (raw_frame_cam_markers.empty() ? frame_cam_markers : raw_frame_cam_markers)) for (auto &c : f.second) nd += c.second.size();
    r.det_err.assign(nd, 0.0); r.q = q; r.q_value.assign(q.size(), 0.0);
    std::vector<int64_t> cnt(C + M + F); std::vector<double> sum(C + M + F), mx(C + M + F);
    aar_error_report_out o; std::memset(&o, 0, sizeof o);
    o.det_err = r.det_err.data();
    o.cam_count = cnt.data(); o.marker_count = cnt.data() + C; o.frame_count = cnt.data() + C + M;
    o.cam_sum_sq = sum.data(); o.marker_sum_sq = sum.data() + C; o.frame_sum_sq = sum.data() + C + M;
    o.cam_max = mx.data(); o.marker_max = mx.data() + C; o.frame_max = mx.data() + C + M;
    o.num_q = (int32_t)q.size(); o.q = r.q.data(); o.q_value = r.q_value.data();
    check(aar_error_report(handle, io_vec.data(), &o), "aar_error_report");
    r.observations = o.num_observations; r.not_in_problem = o.num_not_in_problem; r.sum_sq = o.sum_sq;
    size_t i = 0;
    auto fill = [&](const std::map<int, Mat44> &ids, std::map<int, EntityError> &dst) {
        for (auto &p : ids) { EntityError &e = dst[p.first]; e.observations = cnt[i]; e.sum_sq = sum[i]; e.max = mx[i]; i++; }
    };
    fill(transforms_to_root_cam, r.cams); fill(transforms_to_root_marker, r.markers); fill(object_to_global, r.frames);
    return r;
}

long long MultiCamMapper::remove_outliers(double max_px, Rejection *out) {
    const ErrorReport rep = error_report({});
    // det_err follows make_handle's flatten order: the raw detections when present (frame_cam_markers then holds the undistorted copy of
    // exactly those that are in the problem, in the same order), else frame_cam_markers
    const bool from_raw = !raw_frame_cam_markers.empty();
    auto in_problem = [&](int f, int c, int id) { return object_to_global.count(f) && transforms_to_root_cam.count(c) && transforms_to_root_marker.count(id); };
    Rejection rj; rj.observations = rep.observations;
    std::map<int, long long> left;                               // frame -> observations kept
    std::map<int, long long> cam_left, marker_left;
    size_t i = 0;
    for (auto &f : (from_raw ? raw_frame_cam_markers : frame_cam_markers)) {
        for (auto &c : f.second) {
            std::vector<Marker> &v = c.second;
            std::vector<Marker> *u = nullptr;
            if (from_raw) { auto fi = frame_cam_markers.find(f.first); if (fi != frame_cam_markers.end()) { auto ci = fi->second.find(c.first); if (ci != fi->second.end()) u = &ci->second; } }
            size_t w = 0, ui = 0, uw = 0;
            for (size_t k = 0; k < v.size(); k++) {
                const bool inp = in_problem(f.first, c.first, v[k].id);
                const bool drop = rep.det_err[i++] > max_px;         // NaN (not in the problem) is never above
                if (!drop) v[w++] = v[k];
                if (from_raw && inp && u) { if (!drop) (*u)[uw++] = (*u)[ui]; ui++; }
                if (drop) rj.removed++;
                else if (inp) { left[f.first]++; cam_left[c.first]++; marker_left[v[k].id]++; }
            }
            v.resize(w);
            if (u) u->resize(uw);
        }
    }
    auto prune = [](FrameCamMarkers &fcm) {                      // no empty camera lists, no empty frames
        for (auto f = fcm.begin(); f != fcm.end();) {
            for (auto c = f->second.begin(); c != f->second.end();) c = c->second.empty() ? f->second.erase(c) : std::next(c);
            f = f->second.empty() ? fcm.erase(f) : std::next(f);
        }
    };
    for (auto f = object_to_global.begin(); f != object_to_global.end();) {
        if (left.count(f->first)) { ++f; continue; }
        rj.dropped_frames.push_back(f->first);
        fixed_frames.erase(f->first); frame_priors.erase(f->first);
        frame_cam_markers.erase(f->first); raw_frame_cam_markers.erase(f->first);
        f = object_to_global.erase(f);
    }
    prune(frame_cam_markers); prune(raw_frame_cam_markers);
    for (auto &p : transforms_to_root_cam) if (!cam_left.count(p.first)) rj.unobserved_cams.push_back(p.first);
    for (auto &p : transforms_to_root_marker) if (!marker_left.count(p.first)) rj.unobserved_markers.push_back(p.first);
    drop_handle(); io_vec.clear();
    if (out) *out = rj;
    return rj.removed;
}

void MultiCamMapper::track() {
    // track() optimises the object pose only (apps/track.cpp:95-97 sets the flags; forced here like the 6-variable io_vec of :272-279)
    Config keep = config;
    config.optimize_cam_poses = false; config.optimize_marker_poses = false; config.optimize_object_poses = true; config.optimize_cam_intrinsics = false;
    drop_handle(); make_handle(corners_undistorted);
    const size_t F = object_to_global.size();
    io_vec.assign(6 * F, 0.0);
    check(aar_mats2evec(handle, io_vec.data()), "aar_mats2evec");
    aar_lm_params prm; aar_lm_default_params(&prm);
    prm.max_iters = solver_params.maxIters; prm.min_average_step_error_diff = solver_params.min_average_step_error_diff; prm.der_epsilon = solver_params.der_epsilon;
    std::vector<double> cost(F); std::vector<int32_t> its(F);
    check(aar_track_batch(handle, io_vec.data(), &prm, cost.data(), its.data()), "aar_track_batch");
    final_error = 0; iterations = 0;
    size_t i = 0;
    for (auto &p : object_to_global) { p.second = vec62mat(&io_vec[6 * i]); final_error += cost[i]; iterations = std::max(iterations, (int)its[i]); i++; }
    config = keep; drop_handle();
}

// ------------------------------------------------------------------------------- files
bool MultiCamMapper::write_solution_file(const std::string &path) {
    std::ofstream f(path, std::ios_base::binary);
    if (!f.is_open()) { std::cout << "Could not open a file in: " << path << " for writing." << std::endl; return false; }
    const size_t C = transforms_to_root_cam.size(), M = transforms_to_root_marker.size(), F = object_to_global.size();
    wr(f, C); for (auto &p : transforms_to_root_cam) wr(f, p.first);
    wr(f, root_cam);
    for (auto &p : transforms_to_root_cam) { const CamConfig &cc = cam_configs.at(p.first); wr(f, cc.width); wr(f, cc.height); }
    wr(f, M); for (auto &p : transforms_to_root_marker) wr(f, p.first);
    wr(f, root_marker);
    wr(f, marker_size);
    wr(f, F); for (auto &p : object_to_global) wr(f, p.first);
    std::vector<double> full; mats2eVec(Config(), full);        // ALWAYS the full Config (:1085-1086)
    for (double v : full) wr(f, v);
    const size_t nf = frame_cam_markers.size(); wr(f, nf);       // serialize_frame_cam_markers (:1030-1051), undistorted corners
    for (auto &fr : frame_cam_markers) {
        wr(f, fr.first); const size_t nc = fr.second.size(); wr(f, nc);
        for (auto &c : fr.second) { wr(f, c.first); const size_t nm = c.second.size(); wr(f, nm); for (auto &mk : c.second) write_marker(f, mk); }
    }
    wr(f, config.optimize_cam_poses); wr(f, config.optimize_marker_poses); wr(f, config.optimize_object_poses); wr(f, config.optimize_cam_intrinsics);
    return true;
}

bool MultiCamMapper::read_solution_file(const std::string &path) {
    std::ifstream f(path, std::ios_base::binary);
    if (!f.is_open()) { std::cout << "Could not open a file in: " << path << " for reading." << std::endl; return false; }
    drop_handle();
    transforms_to_root_cam.clear(); transforms_to_root_marker.clear(); object_to_global.clear(); cam_configs.clear(); frame_cam_markers.clear(); raw_frame_cam_markers.clear();
    size_t C = 0, M = 0, F = 0;
    if (!rd(f, C)) return false;
    std::vector<int> cid(C); for (auto &v : cid) rd(f, v);
    rd(f, root_cam);
    for (size_t i = 0; i < C; i++) { CamConfig cc; rd(f, cc.width); rd(f, cc.height); cam_configs[cid[i]] = cc; transforms_to_root_cam[cid[i]] = Mat44(); }
    rd(f, M); std::vector<int> mid(M); for (auto &v : mid) rd(f, v);
    rd(f, root_marker);
    for (int id : mid) transforms_to_root_marker[id] = Mat44();
    rd(f, marker_size);
    rd(f, F); std::vector<int> fid(F); for (auto &v : fid) rd(f, v);
    for (int id : fid) object_to_global[id] = Mat44();
    // NOTE the vector is written in MatArray index order = ascending id order for files written by the reference
    // (ids sorted by std::map); files with unsorted id tables are not produced by it.
    std::vector<double> full(get_num_vars(Config()));
    for (auto &v : full) if (!rd(f, v)) return false;
    eVec2Mats_full(full);
    size_t nf = 0; rd(f, nf);                                    // deserialize_frame_cam_markers (:1101-1122); stored under the ids read
    for (size_t a = 0; a < nf; a++) {
        int frame_id = 0; size_t nc = 0; rd(f, frame_id); rd(f, nc);
        for (size_t b = 0; b < nc; b++) {
            int cam_id = 0; size_t nm = 0; rd(f, cam_id); rd(f, nm);
            std::vector<Marker> &v = frame_cam_markers[frame_id][cam_id]; v.resize(nm);
            for (auto &mk : v) if (!read_marker(f, mk)) return false;
        }
    }
    Config c;
    rd(f, c.optimize_cam_poses); rd(f, c.optimize_marker_poses); rd(f, c.optimize_object_poses); rd(f, c.optimize_cam_intrinsics);
    config = c;
    corners_undistorted = true;
    return true;
}

void MultiCamMapper::write_text_solution_file(const std::string &path) {
    std::ofstream f(path);
    f << "%YAML:1.0\n---\n";
    f << "marker_size: " << num(marker_size) << "\n";
    auto seq = [&](const char *name, const char *idname, const std::map<int, Mat44> &mats) {
        f << name << ":\n";
        for (auto &p : mats) {
            f << "   - { " << idname << ":" << p.first << ", transform:!!opencv-matrix\n       rows: 4\n       cols: 4\n       dt: d\n       data: [ ";
            for (int i = 0; i < 16; i++) { f << num(p.second.m[i]); if (i < 15) f << (i % 4 == 3 ? ",\n           " : ", "); }
            f << " ] }\n";
        }
    };
    seq("transforms_to_root_cam", "cam_id", transforms_to_root_cam);
    seq("transforms_to_root_marker", "marker_id", transforms_to_root_marker);
    seq("root_marker_to_root_cam", "frame_id", object_to_global);
}

void MultiCamMapper::write_detections_file(const std::string &path, const std::vector<std::vector<std::vector<Marker>>> &seqv) {
    std::ofstream f(path, std::ios_base::binary);
    if (!f.is_open()) throw std::runtime_error("Could not open to write the detection file at: " + path);
    const size_t nc = seqv.empty() ? 0 : seqv[0].size(); wr(f, nc);
    for (auto &frame : seqv) for (auto &cam : frame) { const size_t n = cam.size(); wr(f, n); for (auto &mk : cam) write_marker(f, mk); }
}

std::vector<std::vector<std::vector<Marker>>> MultiCamMapper::read_detections_file(const std::string &path, const std::vector<int> &subseqs) {
    std::ifstream f(path, std::ios_base::binary);
    if (!f.is_open()) throw std::runtime_error("Could not open to read the detection file at: " + path);
    std::vector<std::vector<std::vector<Marker>>> all;
    size_t nc = 0;
    if (rd(f, nc))
        for (;;) {
            std::vector<std::vector<Marker>> frame(nc);
            bool eof = false;
            for (size_t c = 0; c < nc && !eof; c++) {
                size_t n = 0;
                if (!rd(f, n)) { eof = true; break; }           // EOF inside a frame discards the partial frame (initializer.cpp:335-347)
                frame[c].resize(n);
                for (auto &mk : frame[c]) if (!read_marker(f, mk)) { eof = true; break; }
            }
            if (eof) break;
            all.push_back(frame);
        }
    if (!subseqs.empty()) {                                       // initializer.cpp:350-359
        int prev_last = -1;
        for (size_t i = 0; i + 1 < subseqs.size(); i += 2) {
            for (int fr = prev_last + 1; fr < subseqs[i] && fr < (int)all.size(); fr++) for (auto &c : all[(size_t)fr]) c.clear();
            prev_last = subseqs[i + 1];
        }
    }
    return all;
}

std::vector<int> MultiCamMapper::read_subseqs(const std::string &path) {
    std::ifstream f(path);
    if (!f.is_open()) throw std::runtime_error("Could not open a file at: " + path);
    std::vector<int> v; int x;
    while (f >> x) v.push_back(x);
    return v;
}

// cv::Mat::inv() of a 4x4 (DECOMP_LU: Gaussian elimination with partial pivoting on [A | I], OpenCV's hal::LU operation order)
static Mat44 inv44_lu(const Mat44 &in) {
    double A[16], b[16];
    std::memcpy(A, in.m, sizeof A);
    for (int i = 0; i < 16; i++) b[i] = (i % 5 == 0) ? 1.0 : 0.0;
    for (int i = 0; i < 4; i++) {
        int k = i;
        for (int j = i + 1; j < 4; j++) if (std::fabs(A[j * 4 + i]) > std::fabs(A[k * 4 + i])) k = j;
        if (std::fabs(A[k * 4 + i]) < 2.2204460492503131e-16 * 100) { Mat44 z; std::memset(z.m, 0, sizeof z.m); return z; }      // singular: cv::Mat::inv() returns zeros
        if (k != i) { for (int j = i; j < 4; j++) std::swap(A[i * 4 + j], A[k * 4 + j]); for (int j = 0; j < 4; j++) std::swap(b[i * 4 + j], b[k * 4 + j]); }
        const double d = -1 / A[i * 4 + i];
        for (int j = i + 1; j < 4; j++) {
            const double alpha = A[j * 4 + i] * d;
            for (int kk = i + 1; kk < 4; kk++) A[j * 4 + kk] += alpha * A[i * 4 + kk];
            for (int kk = 0; kk < 4; kk++) b[j * 4 + kk] += alpha * b[i * 4 + kk];
        }
    }
    for (int i = 3; i >= 0; i--)
        for (int j = 0; j < 4; j++) {
            double sum = b[i * 4 + j];
            for (int k = i + 1; k < 4; k++) sum -= A[i * 4 + k] * b[k * 4 + j];
            b[i * 4 + j] = sum / A[i * 4 + i];
        }
    Mat44 R; std::memcpy(R.m, b, sizeof b); return R;
}

// multicam_mapper.cpp:86-117: size_t n1, n1 x { int node1, size_t n2, n2 x { int node2, double r[3], double t[3] } }, int root_cam_id.
// Every stored edge also yields its inverse (transforms[node2][node1] = T.inv(), :111).
int MultiCamMapper::read_stereo_calib(const std::string &path, std::map<int, std::map<int, Mat44>> &transforms) {
    std::ifstream f(path, std::ios_base::binary);
    if (!f.is_open()) throw std::runtime_error("Could not open stereo calib file to read at: " + path);
    size_t n1 = 0; rd(f, n1);
    for (size_t i = 0; i < n1; i++) {
        int node1 = 0; size_t n2 = 0; rd(f, node1); rd(f, n2);
        for (size_t j = 0; j < n2; j++) {
            int node2 = 0; double v[6] = {0, 0, 0, 0, 0, 0};
            rd(f, node2);
            for (int k = 0; k < 6; k++) rd(f, v[k]);
            const Mat44 T = vec62mat(v);
            transforms[node1][node2] = T;
            transforms[node2][node1] = inv44_lu(T);
        }
    }
    int root_cam_id = 0; rd(f, root_cam_id);
    return root_cam_id;
}

void MultiCamMapper::write_stereo_calib(const std::string &path, const std::map<int, std::map<int, Mat44>> &transforms, int root_cam_id) {      // :119-143
    std::ofstream f(path, std::ios_base::binary);
    if (!f.is_open()) throw std::runtime_error("Could not open stereo calib file to write at: " + path);
    const size_t n1 = transforms.size(); wr(f, n1);
    for (auto &a : transforms) {
        wr(f, a.first);
        const size_t n2 = a.second.size(); wr(f, n2);
        for (auto &b : a.second) {
            wr(f, b.first);
            double v[6]; mat2vec6(b.second, v);
            for (int k = 0; k < 6; k++) wr(f, v[k]);
        }
    }
    wr(f, root_cam_id);
}

// multicam_mapper.cpp:145-168: repeated { size_t frame_num, double r[3], double t[3] } until EOF; a record cut short throws
void MultiCamMapper::read_ground_truth(const std::string &path, std::map<size_t, Mat44> &poses) {
    std::ifstream f(path, std::ios_base::binary);
    if (!f.is_open()) throw std::runtime_error("Could not open ground truth file to read at: " + path);
    size_t frame_num = 0;
    while (rd(f, frame_num)) {
        double v[6];
        for (int k = 0; k < 6; k++) if (!rd(f, v[k])) throw std::runtime_error("Unexpected end of input ground truth file : " + path);
        poses[frame_num] = vec62mat(v);
    }
}

void MultiCamMapper::write_ground_truth(const std::string &path, const std::map<size_t, Mat44> &poses) {      // :170-184
    std::ofstream f(path, std::ios_base::binary);
    if (!f.is_open()) throw std::runtime_error("Could not open ground truth file to write at: " + path);
    for (auto &p : poses) {
        const size_t frame_num = p.first; wr(f, frame_num);
        double v[6]; mat2vec6(p.second, v);
        for (int k = 0; k < 6; k++) wr(f, v[k]);
    }
}

} // namespace aar
