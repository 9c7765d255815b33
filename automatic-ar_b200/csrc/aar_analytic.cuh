// aar_analytic.cuh — device side of the analytic-Jacobian / full-FP64 variant (SURVEY.md 8(f) row 4; aar_problem_desc::analytic_jacobian).
//
// The arithmetic is include/aar_analytic.h, shared with the CPU oracle: residual e = m - p in double with no float32 rounding, Jacobian
// by differentiation of the chain of MultiCamMapper::project_marker (/root/reference/libs/multicam_mapper.cpp:608-649) instead of the
// central differences of obtain_transformation_derivs (:803-994).  Everything downstream of the Jacobian rows — the tensor-core assembly,
// the Schur elimination, the reduced Cholesky, the LM loop — is the faithful path's: k_jac_analytic writes the same staged rows as
// k_jac_project<double, true> ([Jc (48) | Jm (48) | Jf (48) | e (8) | marker index | pad], aar_jacobian.cuh), holding derivatives instead
// of central-difference numerators (the assembly's 1 / (2 delta) scale factors are 1 in this mode).
// Not a parity mode and not tuned: one thread per observation, tables read through the L1.
#pragma once
#include "../../include/aar_analytic.h"

namespace aar {

constexpr int CAM_AN = 30;    // per camera: dRc/dr_k (27) | tc (3) of the camera -> root-camera transform itself (the pose tables hold its inverse)
constexpr int RT_AN = 28;     // per marker / frame: dR/dr_k (27) | pad

// Rotation derivatives of every optimised camera / marker / frame at z.  One thread per entity.
__global__ void k_expand_analytic(DevProblem p, const double *__restrict__ z) {
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const double *r; double *dst;
    if (t < p.C) {
        const int c = (int)t;
        if (!p.opt_c || c == p.root_cam) return;
        r = z + col_of_cam(p, c); dst = p.cam_an + (size_t)c * CAM_AN;
        dst[27] = r[3]; dst[28] = r[4]; dst[29] = r[5];
    } else if ((t -= p.C) < p.M) {
        const int m = (int)t;
        if (!p.opt_m || m == p.root_marker) return;
        r = z + col_of_marker(p, m); dst = p.mk_an + (size_t)m * RT_AN;
    } else if ((t -= p.M) < p.F) {
        if (!p.opt_f) return;
        r = z + p.col_frame0 + 6 * (size_t)t; dst = p.fr_an + (size_t)t * RT_AN;
    } else return;
    double R[9], dR[27];
    rodrigues(r[0], r[1], r[2], R);          // the rotation k_expand_jac stores as the base pose of this entity
    aar_an_rodrigues_derivs(r, R, dR);
    for (int i = 0; i < 27; i++) dst[i] = dR[i];
}

// receives the derivative pairs of aar_an_observation into the [18][8] block at the head of a staged row
struct AnBlockSink {
    double *dst;
    AAR_HD void put(int col, int corner, double jx, double jy) { *reinterpret_cast<double2 *>(dst + col * 8 + 2 * corner) = make_double2(jx, jy); }
};

struct AnObsDev { const double *ct, *ca, *ft, *fa, *mt, *ma; double fx, cx, fy, cy; float und[8]; bool act_c, act_m, act_f; };
__device__ __forceinline__ void an_load_obs(const DevProblem &p, long long o, int cm, AnObsDev &q) {
    const int c = obs_cam(cm), m = obs_marker(cm), f = p.obs_f[o];
    q.ct = p.cam_tab + (size_t)c * CAM_TAB; q.ca = p.cam_an + (size_t)c * CAM_AN;       // base entry of the pose tables: [R (9) | t (3)]
    q.ft = p.fr_tab + (size_t)f * FR_TAB; q.fa = p.fr_an + (size_t)f * RT_AN;
    q.mt = p.mk_tab + (size_t)m * MK_TAB; q.ma = p.mk_an + (size_t)m * RT_AN;
    q.fx = p.intr[4 * c]; q.cx = p.intr[4 * c + 1]; q.fy = p.intr[4 * c + 2]; q.cy = p.intr[4 * c + 3];
    q.act_c = p.opt_c && c != p.root_cam; q.act_m = p.opt_m && m != p.root_marker; q.act_f = p.opt_f != 0;
    load8(p.und_a, p.und_b, o, q.und);
}
template <class Sink>
__device__ __forceinline__ void an_eval(const DevProblem &p, const AnObsDev &q, double *e, Sink &sink) {
    aar_an_observation(q.ct, q.ct + 9, q.ca, q.ca + 27, q.ft, q.ft + 9, q.fa, q.mt, q.mt + 9, q.ma, q.fx, q.cx, q.fy, q.cy, p.h, q.und, q.act_c, q.act_m, q.act_f, e, sink);
}

// One staged row per observation (see the header comment); Huber weights of the four corners to Rv = [N][4] (mcm.cpp:1014-1019).
__global__ void __launch_bounds__(128) k_jac_analytic(DevProblem p, float huber_delta, double *__restrict__ Jn, double *__restrict__ Rv) {
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= p.N) return;
    const int cm = p.obs_cm[o];
    AnObsDev q; an_load_obs(p, o, cm, q);
    double *row = Jn + (size_t)o * JROW;
    const bool nj = obs_nojac(cm);           // an erased duplicate (mcm.cpp:368-370): residual rows, no Jacobian rows — the row contributes nothing
    if (nj || !q.act_c) zero48(row);
    if (nj || !q.act_m) zero48(row + 48);
    if (nj || !q.act_f) zero48(row + 96);
    if (nj) { zero16(row + 144); return; }
    double e[8];
    AnBlockSink sink{row};
    an_eval(p, q, e, sink);
    double2 *tail = reinterpret_cast<double2 *>(row + 144);
#pragma unroll
    for (int i = 0; i < 4; i++) tail[i] = make_double2(e[2 * i], e[2 * i + 1]);
    tail[4] = make_double2(__hiloint2double(0, obs_marker(cm)), 0.0); tail[5] = make_double2(0.0, 0.0); tail[6] = make_double2(0.0, 0.0); tail[7] = make_double2(0.0, 0.0);
    if (p.huber) {
        double w[4];
#pragma unroll
        for (int i = 0; i < 4; i++) w[i] = huber_weight(e[2 * i] * e[2 * i] + e[2 * i + 1] * e[2 * i + 1], huber_delta);
        double2 *dst = reinterpret_cast<double2 *>(Rv + (size_t)o * 4); dst[0] = make_double2(w[0], w[1]); dst[1] = make_double2(w[2], w[3]);
    }
}

// eval_curr_solution (mcm.cpp:996-1028) of the full-FP64 variant: e = m - p in double, Huber weight, sum of squares.  Same interface as
// k_residual (aar_kernels.cuh), which stays untouched for the faithful path.
__global__ void __launch_bounds__(256) k_residual_an(DevProblem p, const double *__restrict__ cam, int cam_stride, const double *__restrict__ mk, int mk_stride,
                                                     const double *__restrict__ fr, int fr_stride, float huber_delta, double *__restrict__ r_out, double *__restrict__ cost) {
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    double acc = 0;
    if (o < p.N) {
        const int cm = p.obs_cm[o], f = p.obs_f[o], c = obs_cam(cm), m = obs_marker(cm);
        // the base poses: inverse camera pose (identity for the root camera), frame pose, marker pose (identity for the root marker)
        double Ri[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, ti[3] = {0, 0, 0}, Rm[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, tm[3] = {0, 0, 0}, Ro[9], to[3];
        if (c != p.root_cam) { const double *s = cam + (size_t)c * cam_stride; for (int i = 0; i < 9; i++) Ri[i] = s[i]; for (int i = 0; i < 3; i++) ti[i] = s[9 + i]; }
        if (m != p.root_marker) { const double *s = mk + (size_t)m * mk_stride; for (int i = 0; i < 9; i++) Rm[i] = s[i]; for (int i = 0; i < 3; i++) tm[i] = s[9 + i]; }
        { const double *s = fr + (size_t)f * fr_stride; for (int i = 0; i < 9; i++) Ro[i] = s[i]; for (int i = 0; i < 3; i++) to[i] = s[9 + i]; }
        float und[8]; load8(p.und_a, p.und_b, o, und);
        double e[8]; aar_an_null_sink ns;
        aar_an_observation(Ri, ti, nullptr, nullptr, Ro, to, nullptr, Rm, tm, nullptr, p.intr_tr[4 * c], p.intr_tr[4 * c + 1], p.intr_tr[4 * c + 2], p.intr_tr[4 * c + 3],
                           p.h, und, false, false, false, e, ns);
#pragma unroll
        for (int i = 0; i < 4; i++) {
            double ex = e[2 * i], ey = e[2 * i + 1];
            if (p.huber) { const double w = huber_weight(ex * ex + ey * ey, huber_delta); ex = w * ex; ey = w * ey; }
            if (r_out) { r_out[8 * o + 2 * i] = ex; r_out[8 * o + 2 * i + 1] = ey; }
            acc = fma(ex, ex, acc); acc = fma(ey, ey, acc);
        }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    __shared__ double wsum[8];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) wsum[w] = acc;
    __syncthreads();
    if (w == 0) {
        acc = lane < 8 ? wsum[lane] : 0.0;
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
        if (lane == 0) atomicAdd(cost, acc);
    }
}

} // namespace aar
