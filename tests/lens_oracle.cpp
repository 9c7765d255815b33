/* lens_oracle.cpp — TEST INFRASTRUCTURE: the CPU oracle (oracle/mcm_oracle.cpp, included unchanged) in the lens model of the analytic
 * mode (aar_problem_desc::lens_model = 1, include/aar_analytic.h: aar_an_observation_lens).  The residual of a corner is the RAW
 * detection minus OpenCV's five-coefficient projection, K and dist taken from io_vec when the intrinsics are optimised (all nine
 * columns live), else from the description.  The Huber rule, the erasure of duplicates and the column order are the analytic mode's.
 *
 * aar_lens_oracle_solve_port is aar_oracle_lm_port (track = 0) copied with two changes: it calls the lens residual and Jacobian, and its
 * arrow system keeps the 9 intrinsics columns of every camera beside the pose blocks (io_vec puts them after the frames), so the frame
 * blocks are still eliminated one by one.  Built by the tests into a temporary directory with the flags of oracle/Makefile. */
#include "../oracle/mcm_oracle.cpp"

namespace {

std::map<const OracleHandle *, std::vector<float>> g_raw;     // raw corners per residual row group (8 floats per observation)

void lens_params(const Mcm &m, const MatArrays &ma, int cam_id, double *l) {
    const bool opt = m.config.optimize_cam_intrinsics;
    const M4 &K = opt ? ma.cam_mats.at_id(cam_id) : m.mat_arrays.cam_mats.at_id(cam_id);
    const M4 &d = opt ? ma.dist_coeffs.at_id(cam_id) : m.mat_arrays.dist_coeffs.at_id(cam_id);
    l[0] = K.a[0]; l[1] = K.a[2]; l[2] = K.a[5]; l[3] = K.a[6];
    for (int k = 0; k < 5; k++) l[4 + k] = d.a[k];
}

void lens_error(const Mcm &m, const std::vector<float> &raw, const eVec &input, eVec &error) {
    MatArrays ma; m.ma_init(ma); m.eVec2Mats(input, ma);
    error.assign(m.num_point_xys, 0.0);
    size_t row0 = 0;
    for (auto &f : m.frame_cam_markers) for (auto &c : f.second) for (auto &mk : c.second) {
        Mcm::AnObs q; m.an_gather(ma, nullptr, f.first, c.first, mk.id, q);
        double l[9], e8[8]; lens_params(m, ma, c.first, l);
        aar_an_null_sink ns; aar_an_null_intr_sink is;
        aar_an_observation_lens(q.Ri, q.ti, q.dRc, q.tc, q.Ro, q.to, q.dRo, q.Rm, q.tm, q.dRm, l, q.h, &raw[row0], false, false, false, e8, ns, is);
        for (int i = 0; i < 4; i++) {
            double ex = e8[2 * i], ey = e8[2 * i + 1];
            if (m.with_huber) { const double w = Mcm::getHubberMonoWeight(ex * ex + ey * ey, m.hubberDelta); ex = w * ex; ey = w * ey; }
            error[row0 + 2 * i] = ex; error[row0 + 2 * i + 1] = ey;
        }
        row0 += 8;
    }
}

struct LensTripletSink {
    std::vector<Triplet> *out; size_t row0; long col0;
    void put(int corner, const double *jx, const double *jy) {
        for (int k = 0; k < 9; k++) { out->push_back({(int)(row0 + 2 * corner), (int)(col0 + k), jx[k]}); out->push_back({(int)(row0 + 2 * corner + 1), (int)(col0 + k), jy[k]}); }
    }
};

void lens_jacobian(const Mcm &m, const std::vector<float> &raw, const eVec &input, std::vector<Triplet> &all) {
    MatArrays ma; m.ma_init(ma); m.eVec2Mats(input, ma);
    all.clear();
    const bool opt_i = m.config.optimize_cam_intrinsics;
    const long intr0 = (long)m.num_vars - (opt_i ? 9 * (long)m.num_cameras : 0);
    size_t row0 = 0;
    for (auto &f : m.frame_cam_markers) for (auto &c : f.second) for (auto &mk : c.second) {
        if (m.frame_cam_marker.at(f.first).at(c.first).at(mk.id).second == row0) {
            Mcm::AnObs q; m.an_gather(ma, &input, f.first, c.first, mk.id, q);
            double l[9], e8[8]; lens_params(m, ma, c.first, l);
            Mcm::AnTripletSink sink{&all, row0, q.col_c, q.col_m, q.col_f};
            if (opt_i) {
                LensTripletSink is{&all, row0, intr0 + 9L * m.mat_arrays.cam_mats.m.at(c.first)};
                aar_an_observation_lens(q.Ri, q.ti, q.dRc, q.tc, q.Ro, q.to, q.dRo, q.Rm, q.tm, q.dRm, l, q.h, &raw[row0], q.act_c, q.act_m, q.act_f, e8, sink, is);
            } else {
                aar_an_null_intr_sink is;
                aar_an_observation_lens(q.Ri, q.ti, q.dRc, q.tc, q.Ro, q.to, q.dRo, q.Rm, q.tm, q.dRm, l, q.h, &raw[row0], q.act_c, q.act_m, q.act_f, e8, sink, is);
            }
        }
        row0 += 8;
    }
}

} // namespace

extern "C" {

/* the raw corners of every observation, in row order: the detections of aar_oracle_create (same arguments) grouped like
 * fill_iteration_arrays (frame id, camera id ascending, file order inside), unknown cameras and markers dropped */
void aar_lens_oracle_attach(OracleHandle *h, int64_t ndet, const int *det_frame, const int *det_cam, const int *det_marker, const float *det_xy) {
    const Mcm &m = h->mcm;
    std::map<int, std::map<int, std::vector<int64_t>>> fc;
    for (int64_t i = 0; i < ndet; i++) fc[det_frame[i]][det_cam[i]].push_back(i);
    std::vector<float> &raw = g_raw[h];
    raw.clear();
    for (auto &f : fc) {
        if (!m.frame_cam_markers.count(f.first)) continue;
        for (auto &c : f.second) {
            if (!m.mat_arrays.transforms_to_root_cam.m.count(c.first)) continue;
            for (int64_t i : c.second) {
                if (!m.mat_arrays.transforms_to_root_marker.m.count(det_marker[i])) continue;
                raw.insert(raw.end(), det_xy + 8 * i, det_xy + 8 * i + 8);
            }
        }
    }
}
void aar_lens_oracle_detach(OracleHandle *h) { g_raw.erase(h); }
int64_t aar_lens_oracle_num_raw(OracleHandle *h) { return (int64_t)g_raw[h].size(); }

void aar_lens_oracle_error(OracleHandle *h, const double *z, double *r) {
    eVec e(z, z + h->mcm.num_vars), err; lens_error(h->mcm, g_raw.at(h), e, err);
    std::memcpy(r, err.data(), err.size() * sizeof(double));
}
/* compressed columns (fetch with aar_oracle_get_jacobian); returns nnz */
int64_t aar_lens_oracle_jacobian(OracleHandle *h, const double *z) {
    eVec e(z, z + h->mcm.num_vars);
    std::vector<Triplet> t; lens_jacobian(h->mcm, g_raw.at(h), e, t);
    triplets_to_csc(t, (int)h->mcm.num_point_xys, (int)h->mcm.num_vars, h->colptr, h->rowidx, h->vals);
    return (int64_t)h->vals.size();
}

/* one observation through aar_an_observation_lens with every block active: e[8], pose columns P[18][8] (col-major over rows, as the
 * device's staged row), intrinsics columns I[9][8] */
void aar_lens_oracle_observation(const double *Ri, const double *ti, const double *r_c, const double *Ro, const double *to, const double *r_o,
                                 const double *Rm, const double *tm, const double *r_m, const double *lens, double h, const float *raw,
                                 double *e, double *P, double *I) {
    double dRc[27], dRo[27], dRm[27], Rc[9], tc[3];
    for (int i = 0; i < 3; i++) { for (int j = 0; j < 3; j++) Rc[i * 3 + j] = Ri[j * 3 + i]; }
    for (int i = 0; i < 3; i++) tc[i] = -((Rc[i * 3 + 0] * ti[0] + Rc[i * 3 + 1] * ti[1]) + Rc[i * 3 + 2] * ti[2]);
    aar_an_rodrigues_derivs(r_c, Rc, dRc);
    aar_an_rodrigues_derivs(r_o, Ro, dRo);
    aar_an_rodrigues_derivs(r_m, Rm, dRm);
    struct PS { double *P; void put(int col, int corner, double jx, double jy) { P[col * 8 + 2 * corner] = jx; P[col * 8 + 2 * corner + 1] = jy; } } ps{P};
    struct IS { double *I; void put(int corner, const double *jx, const double *jy) { for (int k = 0; k < 9; k++) { I[k * 8 + 2 * corner] = jx[k]; I[k * 8 + 2 * corner + 1] = jy[k]; } } } is{I};
    aar_an_observation_lens(Ri, ti, dRc, tc, Ro, to, dRo, Rm, tm, dRm, lens, h, raw, true, true, true, e, ps, is);
}
/* the pinhole function on the same inputs (with und = raw): e[8], P[18][8] */
void aar_lens_oracle_pinhole_observation(const double *Ri, const double *ti, const double *r_c, const double *Ro, const double *to, const double *r_o,
                                         const double *Rm, const double *tm, const double *r_m, const double *K4, double h, const float *und,
                                         double *e, double *P) {
    double dRc[27], dRo[27], dRm[27], Rc[9], tc[3];
    for (int i = 0; i < 3; i++) { for (int j = 0; j < 3; j++) Rc[i * 3 + j] = Ri[j * 3 + i]; }
    for (int i = 0; i < 3; i++) tc[i] = -((Rc[i * 3 + 0] * ti[0] + Rc[i * 3 + 1] * ti[1]) + Rc[i * 3 + 2] * ti[2]);
    aar_an_rodrigues_derivs(r_c, Rc, dRc); aar_an_rodrigues_derivs(r_o, Ro, dRo); aar_an_rodrigues_derivs(r_m, Rm, dRm);
    struct PS { double *P; void put(int col, int corner, double jx, double jy) { P[col * 8 + 2 * corner] = jx; P[col * 8 + 2 * corner + 1] = jy; } } ps{P};
    aar_an_observation(Ri, ti, dRc, tc, Ro, to, dRo, Rm, tm, dRm, K4[0], K4[1], K4[2], K4[3], h, und, true, true, true, e, ps);
}

/* aar_oracle_solve_port in the lens model (see the header comment) */
int aar_lens_oracle_solve_port(OracleHandle *h, double *z_io, int max_trace, double *trace, double *final_cost) {
    Mcm &m = h->mcm;
    m.hubberDelta = 10;                                   /* aar_oracle_solve_port */
    const std::vector<float> &raw = g_raw.at(h);
    const int n = (int)m.num_vars;
    auto f = [&](const eVec &z, eVec &x) { lens_error(m, raw, z, x); };
    eVec curr_z(z_io, z_io + n), x64;
    f(curr_z, x64);
    double currErr = 0; for (double v : x64) currErr += v * v;
    double prevErr = currErr, mu = -1, v = 2;
    const int rows = (int)x64.size();
    int it = 0, mustExit = 0;
    /* layout of the arrow system: [pose blocks | 9 intrinsics per camera | frames]; io_vec is [pose blocks | frames | intrinsics] */
    const int n_p = (int)((m.config.optimize_cam_poses ? (m.num_cameras - 1) * 6 : 0) + (m.config.optimize_marker_poses ? (m.num_markers - 1) * 6 : 0));
    const int n_i = m.config.optimize_cam_intrinsics ? 9 * (int)m.num_cameras : 0;
    const bool arrow = m.config.optimize_object_poses;
    const int F = arrow ? (int)m.num_frames : 0, n_f = 6 * (m.config.optimize_object_poses ? (int)m.num_frames : 0);
    const int n_r = n_p + n_i;
    const int n_dense = arrow ? n_r : n;
    std::vector<int> perm((size_t)n);        /* io_vec column -> arrow column */
    for (int i = 0; i < n; i++) perm[(size_t)i] = i < n_p ? i : i < n_p + n_f ? i + n_i : i - n_f;
    for (it = 0; it < m.maxIters && !mustExit; it++) {
        std::vector<Triplet> t;
        lens_jacobian(m, raw, curr_z, t);
        for (auto &q : t) q.col = perm[(size_t)q.col];
        std::vector<int64_t> colptr; std::vector<int> rowidx; std::vector<double> vals;
        triplets_to_csc(t, rows, n, colptr, rowidx, vals);
        std::vector<std::vector<std::pair<int, double>>> rws((size_t)rows);
        for (int c = 0; c < n; c++) for (int64_t k = colptr[(size_t)c]; k < colptr[(size_t)c + 1]; k++) rws[(size_t)rowidx[(size_t)k]].push_back({c, vals[(size_t)k]});
        /* A = JtJ in arrow blocks, B = -Jt x */
        std::vector<double> Hd((size_t)n_dense * n_dense, 0.0), Hff((size_t)F * 36, 0.0), W((size_t)F * n_r * 6, 0.0), B((size_t)n, 0.0);
        for (int r = 0; r < rows; r++) {
            const auto &R = rws[(size_t)r];
            for (auto &a : R) {
                B[(size_t)a.first] -= a.second * x64[(size_t)r];
                for (auto &c : R) {
                    if (a.first < n_dense && c.first < n_dense) Hd[(size_t)a.first * n_dense + c.first] += a.second * c.second;
                    else if (a.first < n_dense && c.first >= n_dense) { int fi = (c.first - n_dense) / 6; W[((size_t)fi * n_r + a.first) * 6 + (c.first - n_dense) % 6] += a.second * c.second; }
                    else if (a.first >= n_dense && c.first >= n_dense) { int fi = (a.first - n_dense) / 6; Hff[(size_t)fi * 36 + ((a.first - n_dense) % 6) * 6 + (c.first - n_dense) % 6] += a.second * c.second; }
                }
            }
        }
        if (mu < 0) {
            double maxv = std::numeric_limits<double>::lowest();
            for (int i = 0; i < n_dense; i++) maxv = std::max(maxv, Hd[(size_t)i * n_dense + i]);
            for (int fi = 0; fi < F; fi++) for (int i = 0; i < 6; i++) maxv = std::max(maxv, Hff[(size_t)fi * 36 + i * 7]);
            mu = maxv * m.tau;
        }
        double gain = 0; int ntries = 0; bool isStepAccepted = false;
        do {
            /* solve (A + mu I) delta = B */
            std::vector<double> S = Hd, bb(B.begin(), B.begin() + n_dense), delta((size_t)n, 0.0);
            for (int i = 0; i < n_dense; i++) S[(size_t)i * n_dense + i] += mu;
            std::vector<std::vector<double>> Lf((size_t)F);
            for (int fi = 0; fi < F; fi++) {
                std::vector<double> L(Hff.begin() + (size_t)fi * 36, Hff.begin() + (size_t)fi * 36 + 36);
                for (int i = 0; i < 6; i++) L[(size_t)i * 7] += mu;
                chol_inplace(L, 6); Lf[(size_t)fi] = L;
                std::vector<double> yb(B.begin() + n_dense + 6 * fi, B.begin() + n_dense + 6 * fi + 6); chol_solve(L, 6, yb.data());
                const double *Wf = &W[(size_t)fi * n_r * 6];
                std::vector<int> nzrows; for (int i = 0; i < n_r; i++) { bool nz = false; for (int k = 0; k < 6; k++) nz |= Wf[(size_t)i * 6 + k] != 0; if (nz) nzrows.push_back(i); }
                std::vector<double> Yw(nzrows.size() * 6);
                for (size_t a = 0; a < nzrows.size(); a++) { double col[6]; for (int k = 0; k < 6; k++) col[k] = Wf[(size_t)nzrows[a] * 6 + k]; chol_solve(L, 6, col); for (int k = 0; k < 6; k++) Yw[a * 6 + k] = col[k]; }
                for (size_t a = 0; a < nzrows.size(); a++) {
                    int i = nzrows[a];
                    for (size_t c = 0; c < nzrows.size(); c++) { double s = 0; for (int k = 0; k < 6; k++) s += Wf[(size_t)i * 6 + k] * Yw[c * 6 + k]; S[(size_t)i * n_dense + nzrows[c]] -= s; }
                    double s = 0; for (int k = 0; k < 6; k++) s += Wf[(size_t)i * 6 + k] * yb[(size_t)k]; bb[(size_t)i] -= s;
                }
            }
            if (n_dense > 0) { chol_inplace(S, n_dense); chol_solve(S, n_dense, bb.data()); }
            for (int i = 0; i < n_dense; i++) delta[(size_t)i] = bb[(size_t)i];
            for (int fi = 0; fi < F; fi++) {
                double rhs[6];
                const double *Wf = &W[(size_t)fi * n_r * 6];
                for (int k = 0; k < 6; k++) { double s = B[(size_t)n_dense + 6 * fi + k]; for (int i = 0; i < n_r; i++) s -= Wf[(size_t)i * 6 + k] * delta[(size_t)i]; rhs[k] = s; }
                chol_solve(Lf[(size_t)fi], 6, rhs);
                for (int k = 0; k < 6; k++) delta[(size_t)n_dense + 6 * fi + k] = rhs[k];
            }
            eVec estimated_z(curr_z);
            for (int i = 0; i < n; i++) estimated_z[(size_t)i] += delta[(size_t)perm[(size_t)i]];
            f(estimated_z, x64);
            double err = 0; for (double q : x64) err += q * q;
            double L = 0; for (int i = 0; i < n; i++) L += delta[(size_t)i] * (mu * delta[(size_t)i] - B[(size_t)i]);
            L *= 0.5;
            gain = (err - prevErr) / L;
            if (gain > 0 && ((err - prevErr) < 0)) {
                mu = mu * std::max(double(0.33), double(1. - std::pow(2 * gain - 1, 3)));
                v = 2.f; currErr = err; curr_z = estimated_z; isStepAccepted = true;
            } else { mu = mu * v; v = v * 5; }
        } while (gain <= 0 && ntries++ < 5 && !isStepAccepted);
        if (currErr < m.minError) mustExit = 1;
        if (std::fabs(prevErr - currErr) <= m.min_step_error_diff || std::fabs((prevErr - currErr) / rows) <= m.min_average_step_error_diff || !isStepAccepted) mustExit = 2;
        if (currErr > prevErr) mustExit = 3;
        if (trace && it < max_trace) { double *tr = trace + 6 * (size_t)it; tr[0] = currErr; tr[1] = mu; tr[2] = gain; tr[3] = ntries + (isStepAccepted ? 1 : 0); tr[4] = isStepAccepted; tr[5] = m.hubberDelta; }
        m.optCallBack();
        prevErr = currErr;
    }
    std::memcpy(z_io, curr_z.data(), (size_t)n * sizeof(double));
    *final_cost = currErr;
    return it;
}

} /* extern "C" */
