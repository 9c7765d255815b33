// aar_kernels.cuh — sm_100a kernels of the MultiCamMapper / SparseLevMarq hot path.
// Included once by aar_cuda.cu (single translation unit, compiled with -fmad=false; see
// aar_device_math.cuh for why).  Reference line numbers are into /root/reference/libs/.
#pragma once
#include <cstdint>
#include "aar_device_math.cuh"

namespace aar {

constexpr int NVAR_CAM = 13;   // inverse camera transform: base + 6 dof x (+,-)
constexpr int NVAR_RT = 7;     // marker / frame: base + 3 rotation dof x (+,-); translations are perturbed on the fly
constexpr int POSE_STRIDE = 12;
constexpr int FC_STRIDE_K = 28;  // per frame: packed lower Cholesky factor of Hff + mu I (21) | y = L^-1 Bf (6) | pad  (aar_schur.cuh: FC_STRIDE)

// Everything the kernels need, by value.
// ---------------------------------------------------------------------------------------------
struct LmTraceDev { double cost, mu, gain; int tries, accepted; float huber_delta; int pad; };   // == aar_lm_trace (include/aar_cuda.h)
constexpr int LM_TRACE_DEV_CAP = 4096;   // records of one launch of the graph-resident loop
// LM state, device resident (sparselevmarq.h:130-135, 237-249): the only copy of the solver's state (the host's h_st is its last
// read-back).  The solve, residual and Jacobian kernels read mu, maxdiag, huber_delta, huber_eval and accepted at these offsets.
struct LmState {
    double cost, prev_cost, trial_cost, mu, v, gain, L;
    double maxdiag;          // local max diagonal of JtJ (first iteration)
    float huber_delta, huber_eval;   // hubberDelta of the next evaluation / the one the accepted iterate was evaluated with (multicam_mapper.cpp:412-417)
    int accepted, tries;
    int iter;                // iterations completed since aar_lm_begin
    int more_tries;          // the do-while of step() (sparselevmarq.h:384-419) runs another try
    int must_exit;           // 0 run | 1..3 stop rules | -1 numeric | -2 inexact float32 staging: redo the iteration with FP64 staging
    int ignore_stop, max_iters /* the graph-resident loop stops at this iteration count */, trace_len /* records in its trace */;
    double min_error, min_step, min_avg, rows;
    long long total_tries;   // tries since aar_lm_begin
    LmTraceDev last;         // record of the last completed iteration
};

struct DevProblem {
    int C, M, F;                 // cameras, markers, LOCAL frames (this rank's shard)
    long long N;                 // local observations
    int root_cam, root_marker;   // indices
    int opt_c, opt_m, opt_f, huber;
    int nrc, nrm, n_r;           // optimised camera / marker blocks, reduced system size 6*(nrc+nrm)
    int col_frame0;              // column of this rank's first frame in z
    double h;                    // half marker size, (float)size/2.f widened
    double J_delta;
    // observations, a1 order (frame, cam, detection order)
    const int *obs_f;            // local frame index
    const int *obs_cm;           // cam | marker<<12 | nojac<<31
    const int *obs_slot_c, *obs_slot_m; // W slot of the camera / marker block in this frame, -1 if none
    const int *obs_pair;         // index of the observation's (frame, camera) pair (runs of consecutive observations in row order)
    const int2 *pair_fc;         // [npairs] local frame, camera
    int npairs;
    double *pair_tab;            // [npairs][PAIR_TAB]: inv(Tc) * To and its perturbed variants (aar_jacobian.cuh: k_pair_tab)
    const float4 *und_a, *und_b, *raw_a, *raw_b; // x0 y0 x1 y1 | x2 y2 x3 y3
    double *intr;                // [C][4] fx cx fy cy at z (constant unless the intrinsics are optimised: then written by k_expand_intr)
    double *intr_tr;             // the same at the trial point (k_residual); == intr when the intrinsics are fixed
    const LmState *st_dev;       // inside aar_lm_iterate: the Huber delta comes from the device state instead of the launch parameter (null otherwise)
    int opt_i, nri, col_intr0;   // intrinsics optimised; 2 C pseudo-blocks behind the pose blocks; their first column in the internal z (aar_intrinsics.cuh)
    // frame CSR of W slots: per frame the camera blocks seen (in order of first appearance), then the marker blocks
    const int *frame_slot_ptr;   // [F+1]
    const int *frame_cs_cum;     // [F+1] camera slots before frame f (so the marker slots of f start at slot_ptr[f] + cs_cum[f+1] - cs_cum[f])
    const int *slot_block;       // [nslots] reduced block index
    // pose tables of the Jacobian kernel (aar_jacobian.cuh: CAM_TAB / MK_TAB / FR_TAB doubles per entity)
    double *cam_tab, *mk_tab, *fr_tab;
    double *cam_tr, *mk_tr, *fr_tr; // trial (z + delta) tables, base only: [.][12]
    const double *cam_fixed, *mk_fixed, *fr_fixed; // host matrices [.][12] for non-optimised groups
    // analytic-Jacobian / full-FP64 variant (aar_analytic.cuh): rotation derivatives of every optimised camera / marker / frame at z
    int analytic;
    double *cam_an, *mk_an, *fr_an;
};

__device__ __forceinline__ int obs_cam(int cm) { return cm & 0xfff; }
__device__ __forceinline__ int obs_marker(int cm) { return (cm >> 12) & 0x7ffff; }
__device__ __forceinline__ bool obs_nojac(int cm) { return cm < 0; }

__device__ __forceinline__ int col_of_cam(const DevProblem &p, int c) { return 6 * (c - (c > p.root_cam ? 1 : 0)); }
__device__ __forceinline__ int col_of_marker(const DevProblem &p, int m) { return 6 * p.nrc + 6 * (m - (m > p.root_marker ? 1 : 0)); }

__device__ __forceinline__ void store_pose(double *dst, const Pose &p) {
#pragma unroll
    for (int i = 0; i < 9; i++) dst[i] = p.r[i];
#pragma unroll
    for (int i = 0; i < 3; i++) dst[9 + i] = p.t[i];
}

// vec2transformation_mat (mcm.cpp:463-473) with one component of the rotation vector or of the
// translation moved by +-delta (obtain_transformation_derivs, mcm.cpp:903-916): variant 0 = base,
// 1+2d+s = dof d, sign s (0:+, 1:-).
__device__ __forceinline__ void expand_variant(const double *z6, int variant, double delta, Pose &T) {
    double rv[3] = {z6[0], z6[1], z6[2]};
    T.t[0] = z6[3]; T.t[1] = z6[4]; T.t[2] = z6[5];
    if (variant > 0) {
        int d = (variant - 1) >> 1;
        double sg = ((variant - 1) & 1) ? -delta : delta;
        if (d < 3) rv[d] = rv[d] + sg;
        else { rodrigues(rv[0], rv[1], rv[2], T.r); T.t[d - 3] = T.t[d - 3] + sg; return; }
    }
    rodrigues(rv[0], rv[1], rv[2], T.r);
}

// cams_vec2mats / markers_vec2mats / object_poses_vec2mats (mcm.cpp:524-552) of a trial point z + delta:
// base poses only, into the *_tr tables read by k_residual.  One thread per entity.
__global__ void k_expand_trial(DevProblem p, const double *__restrict__ z) {
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    Pose T, Ti;
    if (t < p.C) {
        const int c = (int)t;
        double *dst = p.cam_tr + (size_t)c * POSE_STRIDE;
        if (c == p.root_cam) { for (int i = 0; i < 12; i++) dst[i] = (i == 0 || i == 4 || i == 8) ? 1.0 : 0.0; return; }
        if (p.opt_c) expand_variant(z + col_of_cam(p, c), 0, p.J_delta, T); else load_pose(T, p.cam_fixed + (size_t)c * POSE_STRIDE);
        inv_rigid_lu(T, Ti);
        store_pose(dst, Ti);
        return;
    }
    t -= p.C;
    if (t < p.M) {
        const int m = (int)t;
        double *dst = p.mk_tr + (size_t)m * POSE_STRIDE;
        if (m == p.root_marker) { for (int i = 0; i < 12; i++) dst[i] = (i == 0 || i == 4 || i == 8) ? 1.0 : 0.0; return; }
        if (p.opt_m) expand_variant(z + col_of_marker(p, m), 0, p.J_delta, T); else load_pose(T, p.mk_fixed + (size_t)m * POSE_STRIDE);
        store_pose(dst, T);
        return;
    }
    t -= p.M;
    if (t >= p.F) return;
    if (p.opt_f) expand_variant(z + p.col_frame0 + 6 * (size_t)t, 0, p.J_delta, T); else load_pose(T, p.fr_fixed + (size_t)t * POSE_STRIDE);
    store_pose(p.fr_tr + (size_t)t * POSE_STRIDE, T);
}

// T1 = inv(Tc) * To (skipped for the root camera, mcm.cpp:617-621)
__device__ __forceinline__ void make_T1(bool cam_root, const Pose &ci, const Pose &To, Pose &T1) {
    if (cam_root) { T1 = To; return; }
    compose_R(ci.r, To.r, T1.r);
    compose_t(ci.r, ci.t, To.t, T1.t);
}
// project T1 * Tm (Tm skipped for the root marker, mcm.cpp:624-628)
__device__ __forceinline__ void project_T1_Tm(const Pose &T1, bool mk_root, const Pose &Tm, const Intr &k, double h, float *out) {
    double c0[3], c1[3], t[3];
    if (mk_root) {
        c0[0] = T1.r[0]; c0[1] = T1.r[3]; c0[2] = T1.r[6];
        c1[0] = T1.r[1]; c1[1] = T1.r[4]; c1[2] = T1.r[7];
        t[0] = T1.t[0]; t[1] = T1.t[1]; t[2] = T1.t[2];
    } else {
        compose_R01(T1.r, Tm.r, c0, c1);
        compose_t(T1.r, T1.t, Tm.t, t);
    }
    project(c0, c1, t, k, h, out);
}

__device__ __forceinline__ void load8(const float4 *a, const float4 *b, long long o, float *x) {
    float4 u = a[o], v = b[o];
    x[0] = u.x; x[1] = u.y; x[2] = u.z; x[3] = u.w; x[4] = v.x; x[5] = v.y; x[6] = v.z; x[7] = v.w;
}

} // namespace aar

#include "aar_jacobian.cuh"
#include "aar_assemble.cuh"
#include "aar_intrinsics.cuh"
#include "aar_analytic.cuh"

namespace aar {

// eval_curr_solution (mcm.cpp:996-1028): residuals of every observation + sum of squares.
// cam/mk/fr: base pose tables with the given strides (trial tables or variant-0 of the Jacobian tables).
#ifndef AAR_RES_MINBLOCKS
#define AAR_RES_MINBLOCKS 3         // measured at cfg 4 (20 k frames): 231 us at 94 registers / 2 CTAs per SM, 184 us at 3 CTAs (a few spilled bytes), 191 us at 4
#endif
__global__ void __launch_bounds__(256, AAR_RES_MINBLOCKS) k_residual(DevProblem p, const double *__restrict__ cam, int cam_stride, const double *__restrict__ mk, int mk_stride,
                           const double *__restrict__ fr, int fr_stride, float huber_delta, double *__restrict__ r_out, double *__restrict__ cost) {
    long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    double acc = 0;
    if (p.st_dev) huber_delta = p.st_dev->huber_delta;
    if (o < p.N) {
        int cm = p.obs_cm[o], f = p.obs_f[o], c = obs_cam(cm), m = obs_marker(cm);
        Intr k; k.fx = p.intr_tr[4 * c]; k.cx = p.intr_tr[4 * c + 1]; k.fy = p.intr_tr[4 * c + 2]; k.cy = p.intr_tr[4 * c + 3];
        Pose ci, To, Tm, T1;
        load_pose(To, fr + (size_t)f * fr_stride);
        bool cam_root = c == p.root_cam, mk_root = m == p.root_marker;
        if (!cam_root) load_pose(ci, cam + (size_t)c * cam_stride);
        if (!mk_root) load_pose(Tm, mk + (size_t)m * mk_stride);
        make_T1(cam_root, ci, To, T1);
        float pr[8], und[8];
        {   // same expressions as project() of aar_device_math.cuh, with the quotients of a corner sharing one reciprocal
            double c0[3], c1[3], t[3];
            if (mk_root) { c0[0] = T1.r[0]; c0[1] = T1.r[3]; c0[2] = T1.r[6]; c1[0] = T1.r[1]; c1[1] = T1.r[4]; c1[2] = T1.r[7]; t[0] = T1.t[0]; t[1] = T1.t[1]; t[2] = T1.t[2]; }
            else { compose_R01(T1.r, Tm.r, c0, c1); compose_t(T1.r, T1.t, Tm.t, t); }
            Offs of; make_offsets(c0, c1, k, p.h, of); project_offs(of, t, k, pr);
        }
        load8(p.und_a, p.und_b, o, und);
#pragma unroll
        for (int i = 0; i < 4; i++) {
            double ex = (double)(und[2 * i] - pr[2 * i]);       // float - float, widened afterwards (mcm.cpp:1012-1013)
            double ey = (double)(und[2 * i + 1] - pr[2 * i + 1]);
            if (p.huber) { double w = huber_weight(ex * ex + ey * ey, huber_delta); ex = w * ex; ey = w * ey; }
            if (r_out) { r_out[8 * o + 2 * i] = ex; r_out[8 * o + 2 * i + 1] = ey; }
            acc = fma(ex, ex, acc); acc = fma(ey, ey, acc);
        }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    __shared__ double wsum[32];
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) wsum[w] = acc;
    __syncthreads();
    if (w == 0) {
        acc = lane < (blockDim.x >> 5) ? wsum[lane] : 0.0;
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
        if (lane == 0) atomicAdd(cost, acc);
    }
}



// 6x6 Cholesky of packed-upper H + mu I, lower factor L (row-major 6x6, only i>=j used). Returns false on a non-positive pivot.
__device__ __forceinline__ bool chol6(const double *hf, double mu, double *L) {
    double A[36];
    int idx = 0;
#pragma unroll
    for (int i = 0; i < 6; i++)
#pragma unroll
        for (int j = i; j < 6; j++) { double v = hf[idx++]; A[i * 6 + j] = v; A[j * 6 + i] = v; }
#pragma unroll
    for (int i = 0; i < 6; i++) A[i * 6 + i] += mu;
    bool ok = true;
#pragma unroll
    for (int j = 0; j < 6; j++) {
        double d = A[j * 6 + j];
#pragma unroll
        for (int k = 0; k < j; k++) d = fma(-L[j * 6 + k], L[j * 6 + k], d);
        if (!(d > 0)) { ok = false; d = 1; }
        d = sqrt(d);
        L[j * 6 + j] = d;
        double inv = 1.0 / d;
#pragma unroll
        for (int i = j + 1; i < 6; i++) {
            double s = A[i * 6 + j];
#pragma unroll
            for (int k = 0; k < j; k++) s = fma(-L[i * 6 + k], L[j * 6 + k], s);
            L[i * 6 + j] = s * inv;
        }
    }
    return ok;
}
// x <- L^-1 x
__device__ __forceinline__ void fwd6(const double *L, double *x) {
#pragma unroll
    for (int i = 0; i < 6; i++) {
        double s = x[i];
#pragma unroll
        for (int k = 0; k < i; k++) s = fma(-L[i * 6 + k], x[k], s);
        x[i] = s / L[i * 6 + i];
    }
}
// x <- L^-T x
__device__ __forceinline__ void bwd6(const double *L, double *x) {
#pragma unroll
    for (int i = 5; i >= 0; i--) {
        double s = x[i];
#pragma unroll
        for (int k = i + 1; k < 6; k++) s = fma(-L[k * 6 + i], x[k], s);
        x[i] = s / L[i * 6 + i];
    }
}

// Back-substitution delta_f = D^-1 (Bf - W_f^T delta_r), trial point z + delta, and the frame part of the two dot products
// needed by L = 1/2 delta^T (mu delta - B) (sparselevmarq.h:406).  One warp per frame (persistent grid): lanes stride over
// the frame's W slots (consecutive 288-byte blocks -> coalesced), the 6 partial sums meet by shuffles, lane 0 finishes with
// the factor L and y = L^-1 B that k_frame_chol left in `fc`:  delta_f = L^-T (y - L^-1 sum_s W_s^T delta_r[s]).
constexpr int BS_WARPS = 8;
#ifndef AAR_BS_MINBLOCKS
#define AAR_BS_MINBLOCKS 4          // measured at cfg 4 (20 k frames): 139 us with 2 CTAs per SM, 130 us with 4
#endif
__global__ void __launch_bounds__(BS_WARPS * 32, AAR_BS_MINBLOCKS) k_backsub(DevProblem p, const double *__restrict__ fc, const double *__restrict__ Hf, const double *__restrict__ W,
                                                           const double *__restrict__ dr, const double *__restrict__ z, double *__restrict__ zt, double *__restrict__ red3) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double dd = 0, dB = 0;
    for (int f = blockIdx.x * BS_WARPS + warp; f < p.F; f += gridDim.x * BS_WARPS) {
        double acc[6] = {0, 0, 0, 0, 0, 0};
        const int s0 = p.frame_slot_ptr[f], s1 = p.frame_slot_ptr[f + 1];
        // the W blocks of a frame are (s1 - s0) * 36 consecutive doubles: lanes walk them as double2 (coalesced 16-byte loads; a lane per
        // slot left half of every sector unused per instruction).  Pair e2 of the range = slot e2 / 18, row i = (e2 % 18) / 3 of W_s,
        // columns 2 (e2 % 3) and + 1: acc[k] += W_s[i][k] * delta_r[blk(s)][i]
        const double2 *w2 = reinterpret_cast<const double2 *>(W + (size_t)s0 * 36);
        const int npair = (s1 - s0) * 18;
        for (int e2 = lane; e2 < npair; e2 += 32) {
            const int sl = e2 / 18, r = e2 - 18 * sl, i = r / 3, c = r - 3 * i;
            const double2 w = w2[e2];
            const double di = dr[6 * p.slot_block[s0 + sl] + i];
            const double m0 = c == 0 ? di : 0.0, m1 = c == 1 ? di : 0.0, m2 = c == 2 ? di : 0.0;
            acc[0] = fma(w.x, m0, acc[0]); acc[1] = fma(w.y, m0, acc[1]);
            acc[2] = fma(w.x, m1, acc[2]); acc[3] = fma(w.y, m1, acc[3]);
            acc[4] = fma(w.x, m2, acc[4]); acc[5] = fma(w.y, m2, acc[5]);
        }
#pragma unroll
        for (int k = 0; k < 6; k++)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
        if (lane == 0) {
            const double *l = fc + (size_t)f * FC_STRIDE_K;
            double v[6];
            int idx = 0;
#pragma unroll
            for (int r = 0; r < 6; r++) {               // v = y - L^-1 acc  (forward substitution on acc, packed lower factor)
                double t = acc[r];
#pragma unroll
                for (int k = 0; k < r; k++) t = fma(-l[idx + k], acc[k], t);
                acc[r] = t / l[idx + r];
                idx += r + 1;
                v[r] = l[21 + r] - acc[r];
            }
#pragma unroll
            for (int r = 5; r >= 0; r--) {              // delta = L^-T v
                double t = v[r];
#pragma unroll
                for (int k = r + 1; k < 6; k++) t = fma(-l[k * (k + 1) / 2 + r], v[k], t);
                v[r] = t / l[r * (r + 1) / 2 + r];
            }
            const size_t col = (size_t)p.col_frame0 + 6 * (size_t)f;
#pragma unroll
            for (int i = 0; i < 6; i++) {
                const double B = -Hf[(size_t)f * HF_STRIDE + 21 + i];
                zt[col + i] = z[col + i] + v[i]; dd = fma(v[i], v[i], dd); dB = fma(v[i], B, dB);
            }
        }
    }
    // one pair of atomics per CTA
    __shared__ double sdd[BS_WARPS], sdB[BS_WARPS];
    if (lane == 0) { sdd[warp] = dd; sdB[warp] = dB; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0, b = 0;
        for (int w = 0; w < BS_WARPS; w++) { a += sdd[w]; b += sdB[w]; }
        atomicAdd(red3 + 1, a); atomicAdd(red3 + 2, b);
    }
}

// z_trial (reduced part) = z + delta_r
__global__ void k_apply_reduced(int n_r, const double *__restrict__ z, const double *__restrict__ dr, double *__restrict__ zt) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_r) zt[i] = z[i] + dr[i];
}

// max diagonal of JtJ (sparselevmarq.h:369-377): frames part, local
__global__ void k_maxdiag_frames(DevProblem p, const double *__restrict__ Hf, LmState *st) {
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    double m = -DBL_MAX;
    if (f < p.F) { const int di[6] = {0, 6, 11, 15, 18, 20}; for (int i = 0; i < 6; i++) m = fmax(m, Hf[(size_t)f * HF_STRIDE + di[i]]); }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, s));
    if ((threadIdx.x & 31) == 0) {
        // atomic max on a double via CAS
        unsigned long long *addr = (unsigned long long *)&st->maxdiag;
        unsigned long long old = *addr;
        while (__longlong_as_double((long long)old) < m) {
            unsigned long long assumed = old;
            old = atomicCAS(addr, assumed, (unsigned long long)__double_as_longlong(m));
            if (old == assumed) break;
        }
    }
}

// One-thread control kernels of SparseLevMarq::solve (sparselevmarq.h:439-472), launched by both LM loops of aar_lm_iterate;
// inside the CUDA graph (`graph` != 0) they also set the conditions of its WHILE nodes.
// Start of an iteration, after the (all-reduced) normal equations: mu0 (first iteration only, sparselevmarq.h:369-377), reset.
// An inexact float32 staging of this Jacobian (flags[1]) leaves the iteration undecided (must_exit = -2): no try is decided.
__global__ void k_lm_begin_iter(LmState *st, int n_r, const double *__restrict__ Hrr_diag_src, int ld, double tau, double frames_maxdiag_global,
                                const int *__restrict__ flags, int graph, cudaGraphConditionalHandle inner) {
    if (threadIdx.x || blockIdx.x) return;
    if (st->mu < 0) {
        double m = frames_maxdiag_global;
        for (int i = 0; i < n_r; i++) m = fmax(m, Hrr_diag_src[(size_t)i * ld + i]);
        st->mu = m * tau;
    }
    st->tries = 0; st->accepted = 0; st->gain = 0;
    st->must_exit = flags[1] ? -2 : 0;
    if (graph) cudaGraphSetConditional(inner, st->must_exit == 0 ? 1u : 0u);
}
// gain / accept / reject of one try (sparselevmarq.h:402-419). red = [trial_cost, dd_f, dB_f] (all-reduced);
// delta_r.delta_r and delta_r.Br are added here (identical on every rank).  Returns whether the trial point was accepted.
__device__ __forceinline__ bool lm_decide_try(LmState *st, const double *__restrict__ red, int n_r, const double *__restrict__ dr, const double *__restrict__ Br) {
    double dd = red[1], dB = red[2];
    for (int i = 0; i < n_r; i++) { dd = fma(dr[i], dr[i], dd); dB = fma(dr[i], Br[i], dB); }
    const double err = red[0], mu = st->mu;
    const double L = 0.5 * (mu * dd - dB);
    const double gain = (err - st->prev_cost) / L;
    st->L = L; st->gain = gain; st->trial_cost = err;
    const bool accept = gain > 0 && ((err - st->prev_cost) < 0);
    if (accept) {
        double t = 2 * gain - 1;
        st->mu = mu * fmax(0.33, 1. - t * t * t);
        st->v = 2.;
        st->cost = err;
        st->accepted = 1;
    } else { st->mu = mu * st->v; st->v = st->v * 5; }
    st->tries += 1;
    return accept;
}
// end of an iteration (sparselevmarq.h:453-465): a non-finite cost, a non-positive pivot (flags[0]) or a broken camera table
// assumption (flags[2]) stop with must_exit = -1 and no record; otherwise stop rules, record, step callback (multicam_mapper.cpp:412-417)
__device__ __forceinline__ void lm_end_iter(LmState *st, const int *__restrict__ flags) {
    if (!(st->trial_cost - st->trial_cost == 0.0) || flags[0] || flags[2]) { st->must_exit = -1; return; }
    const double currErr = st->cost, prevErr = st->prev_cost;
    int mustExit = 0;
    if (!st->ignore_stop) {
        if (currErr < st->min_error) mustExit = 1;
        if (fabs(prevErr - currErr) <= st->min_step || fabs((prevErr - currErr) / st->rows) <= st->min_avg || !st->accepted) mustExit = 2;
        if (currErr > prevErr) mustExit = 3;
    }
    LmTraceDev &t = st->last;
    t.cost = currErr; t.mu = st->mu; t.gain = st->gain; t.tries = st->tries; t.accepted = st->accepted; t.huber_delta = st->huber_delta; t.pad = 0;
    if (st->huber_delta > 2.5f) st->huber_delta = (float)((double)st->huber_delta - 7.5 / 500);
    st->prev_cost = currErr; st->cost = currErr;
    st->iter += 1;
    st->must_exit = mustExit;
}

// after a try: its decision, the do-while condition of step() (sparselevmarq.h:384-419) and, when no try follows, the end of the
// iteration.  A try after an inexact staging (must_exit = -2, host-driven loop only) is not decided.
__global__ void k_lm_decide(LmState *st, const double *__restrict__ red, int n_r, const double *__restrict__ dr, const double *__restrict__ Br, const int *__restrict__ flags,
                            int graph, cudaGraphConditionalHandle inner) {
    if (threadIdx.x || blockIdx.x) return;
    st->more_tries = 0;
    if (st->must_exit != -2) {
        if (lm_decide_try(st, red, n_r, dr, Br)) st->huber_eval = st->huber_delta;
        st->total_tries += 1;
        st->more_tries = st->gain <= 0 && st->tries <= 5 && !st->accepted;
        if (!st->more_tries) lm_end_iter(st, flags);
    }
    if (graph) cudaGraphSetConditional(inner, st->more_tries ? 1u : 0u);
}
// accepted trial point becomes the iterate (a pointer swap would invalidate the captured graph of the resident loop)
__global__ void k_lm_commit(const LmState *__restrict__ st, long long n, const double *__restrict__ zt, double *__restrict__ z) {
    if (!st->accepted) return;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) z[i] = zt[i];
}
// graph-resident loop only, after the inner WHILE node: the record of a completed iteration into the trace, the outer condition
__global__ void k_lm_next_iter_g(LmState *st, LmTraceDev *__restrict__ trace, cudaGraphConditionalHandle outer) {
    if (threadIdx.x || blockIdx.x) return;
    if (st->must_exit >= 0 && st->trace_len < LM_TRACE_DEV_CAP) trace[st->trace_len++] = st->last;
    cudaGraphSetConditional(outer, (st->must_exit == 0 && st->iter < st->max_iters) ? 1u : 0u);
}

// one-off device undistortion pass — cv::undistortPoints(..., K, dist, noArray, K) as called by
// remove_distortions (mcm.cpp:554-578): 5 fixed-point iterations in double, float32 in/out.
__global__ void k_undistort(long long n4, int obs_shift /* point i belongs to observation i >> obs_shift */, const float2 *__restrict__ in, const int *__restrict__ obs_cm, const double *__restrict__ K9, const double *__restrict__ dist5, float2 *__restrict__ out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    const int c = obs_cam(obs_cm[i >> obs_shift]);
    const double *K = K9 + 9 * (size_t)c, *k = dist5 + 5 * (size_t)c;
    const double fx = K[0], fy = K[4], ifx = 1. / fx, ify = 1. / fy, cx = K[2], cy = K[5];
    float2 uv = in[i];
    double x = uv.x, y = uv.y;
    x = (x - cx) * ifx;
    y = (y - cy) * ify;
    const double x0 = x, y0 = y;
    for (int j = 0; j < 5; j++) {
        double r2 = x * x + y * y;
        double icdist = 1 / (1 + ((k[4] * r2 + k[1]) * r2 + k[0]) * r2);
        if (icdist < 0) { x = ((double)uv.x - cx) * ifx; y = ((double)uv.y - cy) * ify; break; }
        double deltaX = 2 * k[2] * x * y + k[3] * (r2 + 2 * x * x);
        double deltaY = k[2] * (r2 + 2 * y * y) + 2 * k[3] * x * y;
        x = (x0 - deltaX) * icdist;
        y = (y0 - deltaY) * icdist;
    }
    // RR = K * I : the products with the zeros of K and I vanish exactly; ww = 1/(0*x + 0*y + 1) = 1
    double xx = K[0] * x + K[1] * y + K[2];
    double yy = K[3] * x + K[4] * y + K[5];
    double ww = 1. / (K[6] * x + K[7] * y + K[8]);
    out[i] = make_float2((float)(xx * ww), (float)(yy * ww));
}

} // namespace aar

#include "aar_schur.cuh"
#include "aar_dense.cuh"
#include "aar_track.cuh"
