// aar_lens.cuh — the lens model of the analytic variant (aar_problem_desc::lens_model = 1, DESIGN.md §6g).
//
// The residual of a corner is raw - projectPoints(Xc; K, k1 k2 p1 p2 k3): detected pixels, no undistortion pass.  The arithmetic is
// aar_an_observation_lens of include/aar_analytic.h, shared with the CPU oracle.  The kernels here stand beside the pinhole analytic
// ones (aar_analytic.cuh) and write the same staged FP64 rows, so the tensor-core assembly, the Schur elimination, the reduced Cholesky
// and the LM loop run unchanged.  The nine lens parameters of camera c are lens[9 c + k] in io_vec order [fx cx fy cy k1 k2 p1 p2 k3]:
// the description's, or, when the intrinsics are optimised, k_expand_lens's copy of the iterate.
//
// With the intrinsics optimised all nine columns of a camera are live: pseudo-block A = [fx cx fy cy k1 k2] and B = [p1 p2 k3 . . .]
// (aar_intrinsics.cuh), so column k of the camera is column k of A's first column.  B owns a W slot per (frame, camera) pair, the one
// after A's.  Not a tuned path.
#pragma once

namespace aar {

// internal reduced vector -> the nine lens parameters per camera
__global__ void k_expand_lens(DevProblem p, const double *__restrict__ z, double *__restrict__ dst) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 9 * p.C) return;
    const int c = t / 9, k = t - 9 * c;
    dst[t] = z[p.col_intr0 + 12 * (size_t)c + k];
}

// keeps the intrinsics columns of one observation: J[k][row], row = 2 corner + (0: x, 1: y)
struct LensColSink {
    double (*J)[8];
    AAR_HD void put(int corner, const double *jx, const double *jy) {
        for (int k = 0; k < 9; k++) { J[k][2 * corner] = jx[k]; J[k][2 * corner + 1] = jy[k]; }
    }
};

__device__ __forceinline__ void lens_load_obs(const DevProblem &p, long long o, int cm, AnObsDev &q) {
    an_load_obs(p, o, cm, q);
    load8(p.raw_a, p.raw_b, o, q.und);        // the lens model reads the detected corners
}

template <class Sink, class ISink>
__device__ __forceinline__ void lens_eval(const DevProblem &p, const AnObsDev &q, const double *lens, double *e, Sink &sink, ISink &isink) {
    aar_an_observation_lens(q.ct, q.ct + 9, q.ca, q.ca + 27, q.ft, q.ft + 9, q.fa, q.mt, q.mt + 9, q.ma, lens, p.h, q.und, q.act_c, q.act_m, q.act_f, e, sink, isink);
}

// k_jac_analytic of the lens model: one staged row per observation, Huber weights to Rv
__global__ void __launch_bounds__(128) k_jac_lens(DevProblem p, const double *__restrict__ lens, float huber_delta, double *__restrict__ Jn, double *__restrict__ Rv) {
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= p.N) return;
    const int cm = p.obs_cm[o];
    AnObsDev q; lens_load_obs(p, o, cm, q);
    double *row = Jn + (size_t)o * JROW;
    const bool nj = obs_nojac(cm);
    if (nj || !q.act_c) zero48(row);
    if (nj || !q.act_m) zero48(row + 48);
    if (nj || !q.act_f) zero48(row + 96);
    if (nj) { zero16(row + 144); return; }
    double e[8];
    AnBlockSink sink{row}; aar_an_null_intr_sink is;
    lens_eval(p, q, lens + 9 * (size_t)obs_cam(cm), e, sink, is);
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

// k_residual_an of the lens model: e = raw - p, Huber weight, sum of squares into *cost
__global__ void __launch_bounds__(256) k_residual_lens(DevProblem p, const double *__restrict__ lens, const double *__restrict__ cam, const double *__restrict__ mk,
                                                       const double *__restrict__ fr, float huber_delta, double *__restrict__ r_out, double *__restrict__ cost) {
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    double acc = 0;
    if (o < p.N) {
        const int cm = p.obs_cm[o], f = p.obs_f[o], c = obs_cam(cm), m = obs_marker(cm);
        double Ri[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, ti[3] = {0, 0, 0}, Rm[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, tm[3] = {0, 0, 0}, Ro[9], to[3];
        if (c != p.root_cam) { const double *s = cam + (size_t)c * POSE_STRIDE; for (int i = 0; i < 9; i++) Ri[i] = s[i]; for (int i = 0; i < 3; i++) ti[i] = s[9 + i]; }
        if (m != p.root_marker) { const double *s = mk + (size_t)m * POSE_STRIDE; for (int i = 0; i < 9; i++) Rm[i] = s[i]; for (int i = 0; i < 3; i++) tm[i] = s[9 + i]; }
        { const double *s = fr + (size_t)f * POSE_STRIDE; for (int i = 0; i < 9; i++) Ro[i] = s[i]; for (int i = 0; i < 3; i++) to[i] = s[9 + i]; }
        float raw[8]; load8(p.raw_a, p.raw_b, o, raw);
        double e[8]; aar_an_null_sink ns; aar_an_null_intr_sink is;
        aar_an_observation_lens(Ri, ti, nullptr, nullptr, Ro, to, nullptr, Rm, tm, nullptr, lens + 9 * (size_t)c, p.h, raw, false, false, false, e, ns, is);
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

// the nine intrinsics columns of every observation at the expanded z: Ji[o][k][row] (aar_eval_jacobian); zeros for an erased duplicate
__global__ void __launch_bounds__(128) k_lens_dump(DevProblem p, const double *__restrict__ lens, double *__restrict__ Ji) {
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= p.N) return;
    const int cm = p.obs_cm[o];
    double J[9][8];
    if (obs_nojac(cm)) { for (int i = 0; i < 72; i++) Ji[72 * o + i] = 0.0; return; }
    AnObsDev q; lens_load_obs(p, o, cm, q);
    q.act_c = q.act_m = q.act_f = false;
    double e[8]; aar_an_null_sink ns; LensColSink is{J};
    lens_eval(p, q, lens + 9 * (size_t)obs_cam(cm), e, ns, is);
    for (int k = 0; k < 9; k++) for (int r = 0; r < 8; r++) Ji[72 * o + 8 * k + r] = J[k][r];
}

// J^T J blocks and J^T r of the nine intrinsics columns: one warp per (frame, camera) pair, like k_intr_assemble.  Its lanes first
// evaluate the columns of up to LENS_BATCH observations into shared memory (one lane per observation, from the shared header), then
// each lane owns a fixed set of the pair's 162 sums and reads the staged pose rows of the batch:
//   [0, 45)    H_ii = Ji^T Ji, upper triangle of the 9x9 (H_AA, H_AB, H_BB)   -> reduced system, both triangles of A and B's own blocks
//   [45, 54)   g_i = Ji^T r                                                  -> reduced system
//   [54, 108)  W_i = Ji^T Jf, 9 x 6                                         -> the pair's W slots: A's, then B's (padding rows 0)
//   [108, 162) H_ci = Jc^T Ji, 6 x 9 (camera pose x intrinsics of the same camera) -> reduced system
// H_mi = Jm^T Ji (6 x 9 per observation, marker pose x intrinsics) is added to the reduced system with atomics, as in k_intr_assemble.
constexpr int LENS_WARPS = 4, LENS_BATCH = 8, LENS_SUMS = 162;
__global__ void __launch_bounds__(32 * LENS_WARPS) k_intr_assemble_lens(DevProblem p, const double *__restrict__ lens, const int4 *__restrict__ pair_info,
                                                                        const int *__restrict__ pair_cam, const int *__restrict__ pair_slot_i,
                                                                        const double *__restrict__ Jn /* [N][JROW] */, const double *__restrict__ Hw,
                                                                        double *__restrict__ W, double *__restrict__ Hrr, double *__restrict__ gr) {
    __shared__ double sJ[LENS_WARPS][LENS_BATCH][9][8], sR[LENS_WARPS][LENS_BATCH][8];
    __shared__ long long sO[LENS_WARPS][LENS_BATCH];
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const long long pr = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (pr >= p.npairs) return;
    const int4 pi = pair_info[pr];
    const int cam = pair_cam[pr], n_r = p.n_r;
    const int bi = 6 * (p.nrc + p.nrm + 2 * cam);                 // column of fx; lens parameter k is column bi + k
    const bool act_c = p.opt_c && cam != p.root_cam;
    const int cb = 6 * (cam - (cam > p.root_cam ? 1 : 0));
    // the sums this lane owns: t = lane + 32 j
    double acc[6];
#pragma unroll
    for (int j = 0; j < 6; j++) acc[j] = 0.0;
    for (int k0 = 0; k0 < pi.y; k0 += LENS_BATCH) {
        const int nb = min(LENS_BATCH, pi.y - k0);
        if (lane < nb) {
            const long long o = pi.x + k0 + lane;
            const int cm = p.obs_cm[o];
            double (*J)[8] = sJ[wp][lane];
            if (obs_nojac(cm)) {
                for (int k = 0; k < 9; k++) for (int r = 0; r < 8; r++) J[k][r] = 0.0;
                for (int r = 0; r < 8; r++) sR[wp][lane][r] = 0.0;
                sO[wp][lane] = -1;
            } else {
                AnObsDev q; lens_load_obs(p, o, cm, q);
                q.act_c = q.act_m = q.act_f = false;
                double e[8]; aar_an_null_sink ns; LensColSink is{J};
                lens_eval(p, q, lens + 9 * (size_t)cam, e, ns, is);
                const double *row = Jn + (size_t)o * JROW;
                for (int r = 0; r < 8; r++) sR[wp][lane][r] = row[144 + r] * (Hw ? Hw[4 * o + (r >> 1)] : 1.0);
                sO[wp][lane] = o;
            }
        }
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 6; j++) {
            const int t = lane + 32 * j;
            if (t >= LENS_SUMS) break;
            for (int b = 0; b < nb; b++) {
                const long long o = sO[wp][b];
                if (o < 0) continue;
                const double *row = Jn + (size_t)o * JROW;
                double s = 0;
                if (t < 45) {                       // (i, k), i <= k, row-major upper triangle
                    int i = 0, u = t;
                    while (u >= 9 - i) { u -= 9 - i; i++; }
                    const int k = i + u;
                    for (int r = 0; r < 8; r++) s = fma(sJ[wp][b][i][r], sJ[wp][b][k][r], s);
                } else if (t < 54) {
                    const int i = t - 45;
                    for (int r = 0; r < 8; r++) s = fma(sJ[wp][b][i][r], sR[wp][b][r], s);
                } else if (t < 108) {
                    const int i = (t - 54) / 6, d = (t - 54) - 6 * i;
                    for (int r = 0; r < 8; r++) s = fma(sJ[wp][b][i][r], row[96 + 8 * d + r], s);
                } else {
                    const int d = (t - 108) / 9, i = (t - 108) - 9 * d;
                    for (int r = 0; r < 8; r++) s = fma(row[8 * d + r], sJ[wp][b][i][r], s);
                }
                acc[j] += s;
            }
        }
        // marker pose x intrinsics, per observation
        for (int b = 0; b < nb; b++) {
            const long long o = sO[wp][b];
            if (o < 0) continue;
            const int m = obs_marker(p.obs_cm[o]);
            if (!p.opt_m || m == p.root_marker) continue;
            const double *row = Jn + (size_t)o * JROW;
            double *dst = Hrr + (size_t)(6 * (p.nrc + m - (m > p.root_marker ? 1 : 0))) * n_r + bi;
            for (int t = lane; t < 54; t += 32) {
                const int d = t / 9, i = t - 9 * d;
                double s = 0;
                for (int r = 0; r < 8; r++) s = fma(row[48 + 8 * d + r], sJ[wp][b][i][r], s);
                atomicAdd(dst + (size_t)d * n_r + i, s);
            }
        }
        __syncwarp();
    }
    const int slot = pair_slot_i[pr];
#pragma unroll
    for (int j = 0; j < 6; j++) {
        const int t = lane + 32 * j;
        if (t >= LENS_SUMS) break;
        const double v = acc[j];
        if (t < 45) {
            int i = 0, u = t;
            while (u >= 9 - i) { u -= 9 - i; i++; }
            const int k = i + u;
            atomicAdd(Hrr + (size_t)(bi + i) * n_r + bi + k, v);
            if (k != i && (k < 6) == (i < 6)) atomicAdd(Hrr + (size_t)(bi + k) * n_r + bi + i, v);   // diagonal blocks A and B: both triangles
        } else if (t < 54) {
            atomicAdd(gr + bi + (t - 45), v);
        } else if (t < 108) {
            const int i = (t - 54) / 6, d = (t - 54) - 6 * i;
            if (p.opt_f && slot >= 0) W[(size_t)(slot + (i >= 6)) * 36 + (i % 6) * 6 + d] = v;
        } else if (act_c) {
            const int d = (t - 108) / 9, i = (t - 108) - 9 * d;
            atomicAdd(Hrr + (size_t)(cb + d) * n_r + bi + i, v);
        }
    }
    if (p.opt_f && slot >= 0 && lane < 18) W[(size_t)(slot + 1) * 36 + 18 + lane] = 0.0;    // B's padding rows
}

} // namespace aar
