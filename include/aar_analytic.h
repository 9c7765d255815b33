/*
 * aar_analytic.h — the analytic-Jacobian / full-FP64 variant of the joint optimisation (SURVEY.md 8(f) row 4), one
 * implementation for host and device.
 *
 * The reference differentiates project_marker by central differences on float32-rounded projections
 * (libs/multicam_mapper.cpp:803-994: delta = 1e-3 on the Rodrigues vector / translation of one transform, entry =
 * (float(m - p+) - float(m - p-)) / (2 delta)).  This header is the limit delta -> 0 of that scheme evaluated in double
 * precision with no float32 rounding anywhere: same parametrisation (rx ry rz tx ty tz per camera / marker / frame,
 * the camera parameters being those of the camera -> root-camera transform whose INVERSE enters the projection,
 * multicam_mapper.cpp:617-621), same residual convention e = m - p (:1011-1013), same column order.  It is NOT a
 * parity mode: results differ from the reference's at the size of its finite-difference and float32 quantisation
 * errors (1e-6 relative on J).  It is selected by aar_problem_desc::analytic_jacobian and checked against
 *   - central differences of an independently written FP64 projection chain (tests/test_analytic_cpu.py), and
 *   - this very code run on the CPU by the oracle (tests/test_gpu_analytic.py): host and device execute the same
 *     sequence of IEEE operations (both translation units are built without FMA contraction).
 *
 * Chain (X = corner of the marker square, z = 0):
 *     Xm = Rm X + tm            marker -> root marker        (identity for the root marker)
 *     Xo = Ro Xm + to           root marker -> root camera   (frame / object pose)
 *     Xc = Ri Xo + ti           root camera -> camera, [Ri | ti] = inv([Rc | tc])   (identity for the root camera)
 *     p  = (fx Xc.x / Xc.z + cx, fy Xc.y / Xc.z + cy)
 */
#ifndef AAR_ANALYTIC_H
#define AAR_ANALYTIC_H

#include "aar_crsincos.h" /* AAR_HD */

/* dR/dr_k, k = 0, 1, 2, of R = Rodrigues(r): three row-major 3x3 matrices in dR[27].
 * Gallego & Yezzi, "A compact formula for the derivative of a 3-D rotation in exponential coordinates" (2015):
 *     dR/dr_k = ( r_k [r]x + [ r x ((I - R) e_k) ]x ) R / |r|^2
 * and, for |r| < 1e-5, the derivative of the second-order expansion R = I + [r]x + (r r^T - |r|^2 I) / 2. */
AAR_HD void aar_an_rodrigues_derivs(const double *r, const double *R, double *dR) {
    const double th2 = (r[0] * r[0] + r[1] * r[1]) + r[2] * r[2];
    for (int k = 0; k < 3; k++) {
        double *D = dR + 9 * k;
        if (th2 < 1e-10) {
            for (int i = 0; i < 3; i++)
                for (int j = 0; j < 3; j++) D[i * 3 + j] = 0.5 * ((i == k ? r[j] : 0.0) + (j == k ? r[i] : 0.0)) - (i == j ? r[k] : 0.0);
            /* + [e_k]x */
            const int a = (k + 1) % 3, b = (k + 2) % 3;
            D[b * 3 + a] += 1.0; D[a * 3 + b] -= 1.0;
            continue;
        }
        /* a = (I - R) e_k, b = r x a, M = r_k [r]x + [b]x */
        const double a0 = (k == 0 ? 1.0 : 0.0) - R[0 * 3 + k], a1 = (k == 1 ? 1.0 : 0.0) - R[1 * 3 + k], a2 = (k == 2 ? 1.0 : 0.0) - R[2 * 3 + k];
        const double b0 = r[1] * a2 - r[2] * a1, b1 = r[2] * a0 - r[0] * a2, b2 = r[0] * a1 - r[1] * a0;
        const double v0 = r[k] * r[0] + b0, v1 = r[k] * r[1] + b1, v2 = r[k] * r[2] + b2;     /* M = [v]x */
        const double M[9] = {0.0, -v2, v1, v2, 0.0, -v0, -v1, v0, 0.0};
        const double s = 1.0 / th2;
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 3; j++) D[i * 3 + j] = ((M[i * 3 + 0] * R[0 * 3 + j] + M[i * 3 + 1] * R[1 * 3 + j]) + M[i * 3 + 2] * R[2 * 3 + j]) * s;
    }
}

/* sink of aar_an_observation that keeps nothing (residual only) */
struct aar_an_null_sink {
    AAR_HD void put(int, int, double, double) {}
};

/* Residual and analytic Jacobian rows of ONE marker observation.
 *   Ri, ti          inverse camera pose (identity / zero for the root camera)
 *   dRc, tc         dRc/dr_k (27) and translation of the camera pose itself      — read only when act_c
 *   Ro, to, dRo     frame pose and its rotation derivatives (27)                  — dRo read only when act_f
 *   Rm, tm, dRm     marker pose (identity / zero for the root marker), derivatives — dRm read only when act_m
 *   fx cx fy cy h   pinhole intrinsics, half marker size
 *   und             observed (undistorted) corners x0 y0 .. x3 y3, corner order (-h, h) (h, h) (h, -h) (-h, -h)
 *                   (aruco::Marker::get3DPoints, 3rdparty/aruco/aruco/marker.cpp:358-369)
 *   e               [8] residual m - p before any Huber weight
 *   sink.put(col, corner, jx, jy): d e_x / d theta_col and d e_y / d theta_col of that corner, col = 6 * block + dof,
 *                   block 0 camera, 1 marker, 2 frame; dof 0..2 rotation vector, 3..5 translation (multicam_mapper.cpp:898-916) */
template <class Sink>
AAR_HD void aar_an_observation(const double *Ri, const double *ti, const double *dRc, const double *tc,
                               const double *Ro, const double *to, const double *dRo,
                               const double *Rm, const double *tm, const double *dRm,
                               double fx, double cx, double fy, double cy, double h, const float *und,
                               bool act_c, bool act_m, bool act_f, double *e, Sink &sink) {
    double R1[9];                                           /* Ri Ro: maps marker-frame displacements to the camera */
    if (act_m)
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 3; j++) R1[i * 3 + j] = (Ri[i * 3 + 0] * Ro[0 * 3 + j] + Ri[i * 3 + 1] * Ro[1 * 3 + j]) + Ri[i * 3 + 2] * Ro[2 * 3 + j];
    for (int i = 0; i < 4; i++) {
        const double x = (i == 1 || i == 2) ? h : -h, y = (i < 2) ? h : -h;
        double Xm[3], Xo[3], Xc[3];
        for (int j = 0; j < 3; j++) Xm[j] = (Rm[j * 3 + 0] * x + Rm[j * 3 + 1] * y) + tm[j];
        for (int j = 0; j < 3; j++) Xo[j] = ((Ro[j * 3 + 0] * Xm[0] + Ro[j * 3 + 1] * Xm[1]) + Ro[j * 3 + 2] * Xm[2]) + to[j];
        for (int j = 0; j < 3; j++) Xc[j] = ((Ri[j * 3 + 0] * Xo[0] + Ri[j * 3 + 1] * Xo[1]) + Ri[j * 3 + 2] * Xo[2]) + ti[j];
        const double iz = 1.0 / Xc[2], ux = Xc[0] * iz, uy = Xc[1] * iz;
        e[2 * i] = (double)und[2 * i] - (fx * ux + cx);
        e[2 * i + 1] = (double)und[2 * i + 1] - (fy * uy + cy);
        const double a = fx * iz, b = fy * iz;
        /* a displacement g of Xc moves the projection by (a (g0 - ux g2), b (g1 - uy g2)); the residual by minus that */
#define AAR_AN_PUT(col, g0, g1, g2) sink.put((col), i, -(a * ((g0) - ux * (g2))), -(b * ((g1) - uy * (g2))))
        if (act_c) {
            const double d0 = Xo[0] - tc[0], d1 = Xo[1] - tc[1], d2 = Xo[2] - tc[2];     /* Xc = Rc^T (Xo - tc) */
            for (int k = 0; k < 3; k++) {
                const double *D = dRc + 9 * k;                                            /* (dRc/dr_k)^T d */
                const double g0 = (D[0] * d0 + D[3] * d1) + D[6] * d2, g1 = (D[1] * d0 + D[4] * d1) + D[7] * d2, g2 = (D[2] * d0 + D[5] * d1) + D[8] * d2;
                AAR_AN_PUT(k, g0, g1, g2);
            }
            for (int k = 0; k < 3; k++) AAR_AN_PUT(3 + k, -Ri[0 * 3 + k], -Ri[1 * 3 + k], -Ri[2 * 3 + k]);   /* d Xc / d tc = -Rc^T */
        }
        if (act_m) {
            for (int k = 0; k < 3; k++) {
                const double *D = dRm + 9 * k;
                const double w0 = D[0] * x + D[1] * y, w1 = D[3] * x + D[4] * y, w2 = D[6] * x + D[7] * y;   /* (dRm/dr_k) X, X.z = 0 */
                const double g0 = (R1[0] * w0 + R1[1] * w1) + R1[2] * w2, g1 = (R1[3] * w0 + R1[4] * w1) + R1[5] * w2, g2 = (R1[6] * w0 + R1[7] * w1) + R1[8] * w2;
                AAR_AN_PUT(6 + k, g0, g1, g2);
            }
            for (int k = 0; k < 3; k++) AAR_AN_PUT(9 + k, R1[0 * 3 + k], R1[1 * 3 + k], R1[2 * 3 + k]);
        }
        if (act_f) {
            for (int k = 0; k < 3; k++) {
                const double *D = dRo + 9 * k;
                const double w0 = (D[0] * Xm[0] + D[1] * Xm[1]) + D[2] * Xm[2], w1 = (D[3] * Xm[0] + D[4] * Xm[1]) + D[5] * Xm[2], w2 = (D[6] * Xm[0] + D[7] * Xm[1]) + D[8] * Xm[2];
                const double g0 = (Ri[0] * w0 + Ri[1] * w1) + Ri[2] * w2, g1 = (Ri[3] * w0 + Ri[4] * w1) + Ri[5] * w2, g2 = (Ri[6] * w0 + Ri[7] * w1) + Ri[8] * w2;
                AAR_AN_PUT(12 + k, g0, g1, g2);
            }
            for (int k = 0; k < 3; k++) AAR_AN_PUT(15 + k, Ri[0 * 3 + k], Ri[1 * 3 + k], Ri[2 * 3 + k]);
        }
#undef AAR_AN_PUT
    }
}

/* sink of aar_an_observation_lens that keeps no intrinsics columns */
struct aar_an_null_intr_sink {
    AAR_HD void put(int, const double *, const double *) {}
};

/* The lens-model variant (aar_problem_desc::lens_model = 1): the same chain and pose columns, but the residual is taken on the RAW
 * corner against OpenCV's projectPoints with five distortion coefficients:
 *     x' = Xc.x / Xc.z, y' = Xc.y / Xc.z, r2 = x'^2 + y'^2, rad = 1 + ((k3 r2 + k2) r2 + k1) r2
 *     x'' = x' rad + 2 p1 x'y' + p2 (r2 + 2 x'^2),  y'' = y' rad + p1 (r2 + 2 y'^2) + 2 p2 x'y'
 *     p = (fx x'' + cx, fy y'' + cy)
 *   lens            [fx cx fy cy k1 k2 p1 p2 k3] (the io_vec order of one camera's intrinsics)
 *   raw             detected corners x0 y0 .. x3 y3, corner order as in aar_an_observation
 *   sink.put(col, corner, jx, jy)      the 18 pose columns, as in aar_an_observation (through the 2x2 distortion Jacobian)
 *   isink.put(corner, jx, jy)          jx[9], jy[9]: d e_x / d lens_k and d e_y / d lens_k of that corner, k in the order of `lens`
 * With all five coefficients 0 the residual and the pose columns are those of aar_an_observation with und = raw. */
template <class Sink, class ISink>
AAR_HD void aar_an_observation_lens(const double *Ri, const double *ti, const double *dRc, const double *tc,
                                    const double *Ro, const double *to, const double *dRo,
                                    const double *Rm, const double *tm, const double *dRm,
                                    const double *lens, double h, const float *raw,
                                    bool act_c, bool act_m, bool act_f, double *e, Sink &sink, ISink &isink) {
    const double fx = lens[0], cx = lens[1], fy = lens[2], cy = lens[3], k1 = lens[4], k2 = lens[5], p1 = lens[6], p2 = lens[7], k3 = lens[8];
    double R1[9];
    if (act_m)
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 3; j++) R1[i * 3 + j] = (Ri[i * 3 + 0] * Ro[0 * 3 + j] + Ri[i * 3 + 1] * Ro[1 * 3 + j]) + Ri[i * 3 + 2] * Ro[2 * 3 + j];
    for (int i = 0; i < 4; i++) {
        const double x = (i == 1 || i == 2) ? h : -h, y = (i < 2) ? h : -h;
        double Xm[3], Xo[3], Xc[3];
        for (int j = 0; j < 3; j++) Xm[j] = (Rm[j * 3 + 0] * x + Rm[j * 3 + 1] * y) + tm[j];
        for (int j = 0; j < 3; j++) Xo[j] = ((Ro[j * 3 + 0] * Xm[0] + Ro[j * 3 + 1] * Xm[1]) + Ro[j * 3 + 2] * Xm[2]) + to[j];
        for (int j = 0; j < 3; j++) Xc[j] = ((Ri[j * 3 + 0] * Xo[0] + Ri[j * 3 + 1] * Xo[1]) + Ri[j * 3 + 2] * Xo[2]) + ti[j];
        const double iz = 1.0 / Xc[2], ux = Xc[0] * iz, uy = Xc[1] * iz;
        const double r2 = ux * ux + uy * uy, xy2 = 2.0 * (ux * uy), tx = r2 + 2.0 * (ux * ux), ty = r2 + 2.0 * (uy * uy);
        const double rad = 1.0 + ((k3 * r2 + k2) * r2 + k1) * r2;
        const double xd = (ux * rad + p1 * xy2) + p2 * tx, yd = (uy * rad + p1 * ty) + p2 * xy2;
        e[2 * i] = (double)raw[2 * i] - (fx * xd + cx);
        e[2 * i + 1] = (double)raw[2 * i + 1] - (fy * yd + cy);
        /* D = d(x'', y'') / d(x', y'), scaled by the focal lengths and 1 / Z: a displacement g of Xc moves (x', y') by
         * iz (g0 - x' g2, g1 - y' g2) and the projection by A (g0 - x' g2, g1 - y' g2), A = diag(fx, fy) D iz */
        const double drad = 2.0 * ((3.0 * k3 * r2 + 2.0 * k2) * r2 + k1);          /* d rad / d(r2) times 2 */
        const double D00 = (rad + ux * ux * drad) + (2.0 * p1 * uy + 6.0 * p2 * ux);
        const double D01 = ux * uy * drad + (2.0 * p1 * ux + 2.0 * p2 * uy);
        const double D11 = (rad + uy * uy * drad) + (6.0 * p1 * uy + 2.0 * p2 * ux);
        const double a = fx * iz, b = fy * iz;
        const double A00 = a * D00, A01 = a * D01, A10 = b * D01, A11 = b * D11;
#define AAR_AN_PUT(col, g0, g1, g2)                                                                      \
        do { const double q0 = (g0) - ux * (g2), q1 = (g1) - uy * (g2);                                  \
             sink.put((col), i, -(A00 * q0 + A01 * q1), -(A11 * q1 + A10 * q0)); } while (0)
        if (act_c) {
            const double d0 = Xo[0] - tc[0], d1 = Xo[1] - tc[1], d2 = Xo[2] - tc[2];
            for (int k = 0; k < 3; k++) {
                const double *D = dRc + 9 * k;
                const double g0 = (D[0] * d0 + D[3] * d1) + D[6] * d2, g1 = (D[1] * d0 + D[4] * d1) + D[7] * d2, g2 = (D[2] * d0 + D[5] * d1) + D[8] * d2;
                AAR_AN_PUT(k, g0, g1, g2);
            }
            for (int k = 0; k < 3; k++) AAR_AN_PUT(3 + k, -Ri[0 * 3 + k], -Ri[1 * 3 + k], -Ri[2 * 3 + k]);
        }
        if (act_m) {
            for (int k = 0; k < 3; k++) {
                const double *D = dRm + 9 * k;
                const double w0 = D[0] * x + D[1] * y, w1 = D[3] * x + D[4] * y, w2 = D[6] * x + D[7] * y;
                const double g0 = (R1[0] * w0 + R1[1] * w1) + R1[2] * w2, g1 = (R1[3] * w0 + R1[4] * w1) + R1[5] * w2, g2 = (R1[6] * w0 + R1[7] * w1) + R1[8] * w2;
                AAR_AN_PUT(6 + k, g0, g1, g2);
            }
            for (int k = 0; k < 3; k++) AAR_AN_PUT(9 + k, R1[0 * 3 + k], R1[1 * 3 + k], R1[2 * 3 + k]);
        }
        if (act_f) {
            for (int k = 0; k < 3; k++) {
                const double *D = dRo + 9 * k;
                const double w0 = (D[0] * Xm[0] + D[1] * Xm[1]) + D[2] * Xm[2], w1 = (D[3] * Xm[0] + D[4] * Xm[1]) + D[5] * Xm[2], w2 = (D[6] * Xm[0] + D[7] * Xm[1]) + D[8] * Xm[2];
                const double g0 = (Ri[0] * w0 + Ri[1] * w1) + Ri[2] * w2, g1 = (Ri[3] * w0 + Ri[4] * w1) + Ri[5] * w2, g2 = (Ri[6] * w0 + Ri[7] * w1) + Ri[8] * w2;
                AAR_AN_PUT(12 + k, g0, g1, g2);
            }
            for (int k = 0; k < 3; k++) AAR_AN_PUT(15 + k, Ri[0 * 3 + k], Ri[1 * 3 + k], Ri[2 * 3 + k]);
        }
#undef AAR_AN_PUT
        /* intrinsics columns of e = raw - p: minus the derivatives of p */
        const double r4 = r2 * r2, r6 = r4 * r2;
        const double jx[9] = {-xd, -1.0, 0.0, 0.0, -(fx * (ux * r2)), -(fx * (ux * r4)), -(fx * xy2), -(fx * tx), -(fx * (ux * r6))};
        const double jy[9] = {0.0, 0.0, -yd, -1.0, -(fy * (uy * r2)), -(fy * (uy * r4)), -(fy * ty), -(fy * xy2), -(fy * (uy * r6))};
        isink.put(i, jx, jy);
    }
}

#endif /* AAR_ANALYTIC_H */
