/* pair_prior_oracle.cpp — TEST INFRASTRUCTURE: the CPU oracle's reduced system and restated LM run on the least-squares problem
 * augmented by soft relative-pose priors between two cameras or two markers (aar_set_pair_prior, include/aar_cuda.h), on top of the
 * absolute priors and held columns of tests/prior_oracle.cpp (included unchanged).  tests/test_gpu_pair_prior.py compares the device
 * with these functions.
 *
 * A pair (a, b) with target [Rbar | tbar] and weights w_rot, w_t appends 12 rows at z: sqrt(w_rot / 2) vec(R_a^T R_b - Rbar) (row-major)
 * and sqrt(w_t) (R_a^T (t_b - t_a) - tbar), with R_x, t_x from z by the oracle's own r -> R (rodrigues_vec2mat, the one its
 * vec2transformation_mat uses) and their exact Jacobian from aar_an_rodrigues_derivs.  A side without columns (col -1: the root) is
 * the identity.  Pairs are given as cols [n][2] (first io_vec column of each side's block, -1 for none) and rec [n][14]
 * (Rbar row-major 9 | tbar 3 | w_rot | w_t).
 *
 * Both functions are aar_prior_oracle_reduced_system and aar_prior_oracle_solve_port copied except for the pair rows: they follow the
 * absolute-prior rows and come before the held columns are zeroed; in the reduced system they are rig rows (counted when f_lo == 0).
 * With n = 0 they are the functions of prior_oracle.cpp bit for bit (tests/test_pair_prior_cpu.py checks it).  Built by the tests into a
 * temporary directory with the flags of oracle/Makefile. */
#include "prior_oracle.cpp"

namespace {
/* residual rows e[12] and dense Jacobian J[12][12] (columns [r_a t_a | r_b t_b]) of one pair at z; the device's arithmetic
 * (csrc/aar_pair_prior.cuh) */
void pair_block(const int32_t *cols, const double *rec, const eVec &z, double *e, double *J) {
    double R[2][9], t[2][3], dR[2][27];
    for (int s = 0; s < 2; s++) {
        const int col = cols[s];
        if (col < 0) {
            for (int i = 0; i < 9; i++) R[s][i] = (i % 4 == 0) ? 1.0 : 0.0;
            for (int i = 0; i < 3; i++) t[s][i] = 0.0;
            for (int i = 0; i < 27; i++) dR[s][i] = 0.0;
            continue;
        }
        const double *z6 = &z[(size_t)col];
        rodrigues_vec2mat(z6, R[s]);
        for (int i = 0; i < 3; i++) t[s][i] = z6[3 + i];
        aar_an_rodrigues_derivs(z6, R[s], dR[s]);
    }
    const double *Ra = R[0], *Rb = R[1], *ta = t[0], *tb = t[1], *dRa = dR[0], *dRb = dR[1];
    const double *Rbar = rec, *tbar = rec + 9, w_rot = rec[12], w_t = rec[13];
    const double d0 = tb[0] - ta[0], d1 = tb[1] - ta[1], d2 = tb[2] - ta[2];
    for (int r = 0; r < 12; r++) {
        double *Jr = J + 12 * r;
        if (r < 9) {
            const int i = r / 3, j = r - 3 * i;
            const double s = std::sqrt(0.5 * w_rot);
            const double rab = (Ra[i] * Rb[j] + Ra[3 + i] * Rb[3 + j]) + Ra[6 + i] * Rb[6 + j];
            e[r] = s * (rab - Rbar[r]);
            for (int c = 0; c < 3; c++) {
                const double *Da = dRa + 9 * c, *Db = dRb + 9 * c;
                Jr[c] = cols[0] < 0 ? 0.0 : s * ((Da[i] * Rb[j] + Da[3 + i] * Rb[3 + j]) + Da[6 + i] * Rb[6 + j]);
                Jr[3 + c] = 0.0;
                Jr[6 + c] = cols[1] < 0 ? 0.0 : s * ((Ra[i] * Db[j] + Ra[3 + i] * Db[3 + j]) + Ra[6 + i] * Db[6 + j]);
                Jr[9 + c] = 0.0;
            }
        } else {
            const int i = r - 9;
            const double s = std::sqrt(w_t);
            const double tab = (Ra[i] * d0 + Ra[3 + i] * d1) + Ra[6 + i] * d2;
            e[r] = s * (tab - tbar[i]);
            for (int c = 0; c < 3; c++) {
                const double *Da = dRa + 9 * c;
                Jr[c] = cols[0] < 0 ? 0.0 : s * ((Da[i] * d0 + Da[3 + i] * d1) + Da[6 + i] * d2);
                Jr[3 + c] = -(s * Ra[3 * c + i]);
                Jr[6 + c] = 0.0;
                Jr[9 + c] = s * Ra[3 * c + i];
            }
        }
    }
}

/* the pair rows at z: residuals appended to x, Jacobian entries (rows x.size() on) to t when given; a pair without columns on either
 * side adds nothing (aar_set_pair_prior ignores it) */
void pair_rows(int n, const int32_t *cols, const double *rec, const eVec &z, eVec &x, std::vector<Triplet> *t) {
    for (int k = 0; k < n; k++) {
        const int32_t *ck = cols + 2 * (size_t)k;
        if (ck[0] < 0 && ck[1] < 0) continue;
        double e[12], J[144];
        pair_block(ck, rec + 14 * (size_t)k, z, e, J);
        for (int r = 0; r < 12; r++) {
            if (t)
                for (int c = 0; c < 12; c++) {
                    const int col = ck[c / 6];
                    if (col >= 0 && J[12 * r + c] != 0.0) t->push_back({(int)x.size(), col + c % 6, J[12 * r + c]});
                }
            x.push_back(e[r]);
        }
    }
}
} // namespace

extern "C" {

/* the rows of n pairs at z: e [12 n] and J [n][12][12] (columns [r_a t_a | r_b t_b]), every pair as given */
void aar_pair_oracle_rows(int n, const int32_t *cols, const double *rec, const double *z, int num_vars, double *e, double *J) {
    eVec zz(z, z + num_vars);
    for (int k = 0; k < n; k++) pair_block(cols + 2 * (size_t)k, rec + 14 * (size_t)k, zz, e + 12 * (size_t)k, J + 144 * (size_t)k);
}

/* aar_prior_oracle_reduced_system on the problem augmented by n pairs */
int aar_pair_oracle_reduced_system(OracleHandle *h, const uint8_t *col_fixed, const double *zbar, const double *w, int n, const int32_t *cols, const double *rec,
                                   const double *z, double mu, int f_lo, int f_hi, double *S, double *b, double *cost) {
    Mcm &m = h->mcm;
    if (!m.config.optimize_object_poses || m.config.optimize_cam_intrinsics) return -1;
    const int n_r = (int)((m.config.optimize_cam_poses ? (m.num_cameras - 1) * 6 : 0) + (m.config.optimize_marker_poses ? (m.num_markers - 1) * 6 : 0));
    eVec e(z, z + m.num_vars), r; m.error_function(e, r);
    std::vector<Triplet> t; m.jacobian_triplets(e, t);
    std::vector<int> prior_frame;
    prior_rows(zbar, w, (int)m.num_vars, n_r, e, r, &t, &prior_frame);
    const size_t pair_row0 = r.size();
    pair_rows(n, cols, rec, e, r, &t);
    for (size_t k = pair_row0; k < r.size(); k++) prior_frame.push_back(-1);      /* rig rows */
    held(col_fixed, t);
    const size_t num_rows = r.size();
    /* rows grouped by frame: row -> frame index */
    std::vector<int> row_frame(m.num_point_xys / 8);
    { size_t o = 0; int fi = 0; for (auto &f : m.frame_cam_markers) { fi = m.mat_arrays.object_to_global.m.at(f.first); for (auto &c : f.second) for (size_t k = 0; k < c.second.size(); k++) row_frame[o++] = fi; } }
    std::vector<int64_t> colptr; std::vector<int> rowidx; std::vector<double> vals;
    triplets_to_csc(t, (int)num_rows, (int)m.num_vars, colptr, rowidx, vals);
    /* per-row sparse lists */
    std::vector<std::vector<std::pair<int, double>>> rows(num_rows);
    for (int c = 0; c < (int)m.num_vars; c++) for (int64_t k = colptr[c]; k < colptr[c + 1]; k++) rows[(size_t)rowidx[k]].push_back({c, vals[k]});
    std::fill(S, S + (size_t)n_r * n_r, 0.0); std::fill(b, b + n_r, 0.0); *cost = 0;
    const int F = (int)m.num_frames;
    std::vector<double> Hff((size_t)36), W((size_t)n_r * 6), Bf(6);
    /* bucket rows per frame; the camera / marker prior rows and the pair rows go in with the first frame range */
    std::vector<std::vector<int>> frame_rows((size_t)F);
    std::vector<int> rig_rows;
    for (size_t row = 0; row < m.num_point_xys; row++) frame_rows[(size_t)row_frame[row / 8]].push_back((int)row);
    for (size_t k = 0; k < prior_frame.size(); k++) {
        const int row = (int)(m.num_point_xys + k);
        if (prior_frame[k] < 0) rig_rows.push_back(row); else frame_rows[(size_t)prior_frame[k]].push_back(row);
    }
    if (f_lo == 0)
        for (int row : rig_rows) {
            const auto &R = rows[(size_t)row];
            double rv = r[(size_t)row]; *cost += rv * rv;
            for (auto &a : R) {
                b[a.first] -= a.second * rv;
                for (auto &c : R) S[(size_t)a.first * n_r + c.first] += a.second * c.second;
            }
        }
    for (int f = f_lo; f < f_hi && f < F; f++) {
        std::fill(Hff.begin(), Hff.end(), 0.0); std::fill(W.begin(), W.end(), 0.0); std::fill(Bf.begin(), Bf.end(), 0.0);
        const int fcol = n_r + 6 * f;
        for (int row : frame_rows[(size_t)f]) {
            const auto &R = rows[(size_t)row];
            double rv = r[(size_t)row]; *cost += rv * rv;
            for (auto &a : R) {
                if (a.first < n_r) b[a.first] -= a.second * rv; else Bf[(size_t)(a.first - fcol)] -= a.second * rv;
                for (auto &c : R) {
                    if (a.first < n_r && c.first < n_r) S[(size_t)a.first * n_r + c.first] += a.second * c.second;
                    else if (a.first < n_r && c.first >= n_r) W[(size_t)a.first * 6 + (c.first - fcol)] += a.second * c.second;
                    else if (a.first >= n_r && c.first >= n_r) Hff[(size_t)(a.first - fcol) * 6 + (c.first - fcol)] += a.second * c.second;
                }
            }
        }
        for (int i = 0; i < 6; i++) Hff[(size_t)i * 6 + i] += mu;
        std::vector<double> L = Hff;
        if (!chol_inplace(L, 6)) return -2;
        /* Y = Hff^-1 [W^T | Bf] */
        std::vector<double> col(6);
        std::vector<double> Yw((size_t)n_r * 6);
        for (int i = 0; i < n_r; i++) { for (int k = 0; k < 6; k++) col[(size_t)k] = W[(size_t)i * 6 + k]; chol_solve(L, 6, col.data()); for (int k = 0; k < 6; k++) Yw[(size_t)i * 6 + k] = col[(size_t)k]; }
        std::vector<double> yb = Bf; chol_solve(L, 6, yb.data());
        for (int i = 0; i < n_r; i++) {
            bool nz = false; for (int k = 0; k < 6; k++) nz |= W[(size_t)i * 6 + k] != 0;
            if (!nz) continue;
            for (int j = 0; j < n_r; j++) { double s = 0; for (int k = 0; k < 6; k++) s += W[(size_t)i * 6 + k] * Yw[(size_t)j * 6 + k]; S[(size_t)i * n_r + j] -= s; }
            double s = 0; for (int k = 0; k < 6; k++) s += W[(size_t)i * 6 + k] * yb[(size_t)k]; b[i] -= s;
        }
    }
    return 0;
}

/* aar_prior_oracle_solve_port on the problem augmented by n pairs */
int aar_pair_oracle_solve_port(OracleHandle *h, const uint8_t *col_fixed, const double *zbar, const double *w, int n, const int32_t *cols, const double *rec,
                               double *z_io, int max_trace, double *trace, double *final_cost) {
    const int track = 0;
    Mcm &m = h->mcm;
    m.hubberDelta = 10;                                   /* aar_oracle_solve_port */
    const int n_vars = track ? 6 : (int)m.num_vars;
    /* the columns before the first frame (the prior rows of a frame are told apart only in the reduced system) */
    const int n_poses = (int)((m.config.optimize_cam_poses ? (m.num_cameras - 1) * 6 : 0) + (m.config.optimize_marker_poses ? (m.num_markers - 1) * 6 : 0));
    auto f = [&](const eVec &z, eVec &x) { if (track) m.error_function_tracking(z, x); else m.error_function(z, x); prior_rows(zbar, w, n_vars, n_poses, z, x, nullptr, nullptr); pair_rows(n, cols, rec, z, x, nullptr); };
    eVec curr_z(z_io, z_io + n_vars), x64;
    f(curr_z, x64);
    double currErr = 0; for (double v : x64) currErr += v * v;
    double prevErr = currErr, mu = -1, v = 2;
    const int rows_all = (int)x64.size();                 /* the rows of the augmented Jacobian */
    const int rows = (int)m.num_point_xys;                /* the stop rule's divisor: the reprojection rows */
    int it = 0, mustExit = 0;
    /* layout of the arrow system */
    const int n_r = track ? 0 : (int)((m.config.optimize_cam_poses ? (m.num_cameras - 1) * 6 : 0) + (m.config.optimize_marker_poses ? (m.num_markers - 1) * 6 : 0));
    const bool arrow = !track && m.config.optimize_object_poses && !m.config.optimize_cam_intrinsics;
    const int F = arrow ? (int)m.num_frames : 0;
    const int n_dense = arrow ? n_r : n_vars;
    for (it = 0; it < m.maxIters && !mustExit; it++) {
        std::vector<Triplet> t;
        if (track) fd_tracking_jacobian(m, curr_z, t);
        else { m.jacobian_triplets(curr_z, t); eVec xp((size_t)m.num_point_xys); prior_rows(zbar, w, n_vars, n_poses, curr_z, xp, &t, nullptr); pair_rows(n, cols, rec, curr_z, xp, &t); held(col_fixed, t); }
        std::vector<int64_t> colptr; std::vector<int> rowidx; std::vector<double> vals;
        triplets_to_csc(t, rows_all, n_vars, colptr, rowidx, vals);
        std::vector<std::vector<std::pair<int, double>>> rws((size_t)rows_all);
        for (int c = 0; c < n_vars; c++) for (int64_t k = colptr[(size_t)c]; k < colptr[(size_t)c + 1]; k++) rws[(size_t)rowidx[(size_t)k]].push_back({c, vals[(size_t)k]});
        /* A = JtJ in arrow blocks, B = -Jt x */
        std::vector<double> Hd((size_t)n_dense * n_dense, 0.0), Hff((size_t)F * 36, 0.0), W((size_t)F * n_r * 6, 0.0), B((size_t)n_vars, 0.0);
        for (int r = 0; r < rows_all; r++) {
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
            std::vector<double> S = Hd, bb(B.begin(), B.begin() + n_dense), delta((size_t)n_vars, 0.0);
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
            for (int i = 0; i < n_vars; i++) estimated_z[(size_t)i] += delta[(size_t)i];
            f(estimated_z, x64);
            double err = 0; for (double q : x64) err += q * q;
            double L = 0; for (int i = 0; i < n_vars; i++) L += delta[(size_t)i] * (mu * delta[(size_t)i] - B[(size_t)i]);
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
        if (!track) m.optCallBack();   /* the callback is installed by solve() only (mcm.cpp:422); apps/track.cpp goes init -> track() */
        prevErr = currErr;
    }
    std::memcpy(z_io, curr_z.data(), (size_t)n_vars * sizeof(double));
    *final_cost = currErr;
    return it;
}

} /* extern "C" */
