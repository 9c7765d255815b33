// aar_pair_prior.cuh — soft relative-pose priors between two cameras or two markers in the joint solve (aar_set_pair_prior,
// DESIGN.md §6f).
//
// For a pair (a, b) of the same kind the relative pose is T_ab = T_a^-1 T_b (b's coordinates into a's): R_ab = R_a^T R_b,
// t_ab = R_a^T (t_b - t_a), where T_x is the pose the solve optimises (from z by the r -> R of expand_variant(.., 0, ..)).  A pair with
// target [Rbar | tbar] and weights w_rot, w_t appends 12 residual rows
//     sqrt(w_rot / 2) vec(R_ab - Rbar)   (row-major, 9 rows),     sqrt(w_t) (t_ab - tbar)   (3 rows)
// whose squared sum is w_rot (2 - 2 cos theta) + w_t |t_ab - tbar|^2 (the chordal rotation distance: smooth everywhere, its exact
// Jacobian comes from aar_an_rodrigues_derivs).  The reference's SparseLevMarq on that augmented problem needs J_p^T J_p on blocks
// (a, a), (b, b), (a, b) of the reduced matrix and J_p^T e_p in its gradient (k_pair_prior_add, after k_prior_add and before
// k_hold_fixed), and the rows' squared sum in the cost wherever the solver forms one (k_pair_prior_cost).  Every later kernel reads
// the changed equations unchanged: the off-diagonal block lives in the upper block triangle, which the Schur step, both Cholesky
// kernels and the back substitution already read.
#pragma once

namespace aar {

// one pair: the first column of each side's pose block in z (-1: no columns, a constant identity pose — the root), the target
// T_ab = [R | t] (R row-major), the weights.  Only pairs with a column and a nonzero weight are stored (aar_set_pair_prior).
struct PairPriorRec { int col_a, col_b; double R[9], t[3], w_rot, w_t; };

constexpr int PP_WARPS = 4;                  // k_pair_prior_add: one warp per pair, 4 warps per CTA
constexpr int PP_SMEM = 78 + 12 + 144;       // per warp: Ra ta dRa Rb tb dRb (78) | e (12) | J (12 x 12)

// a side's pose at z and, when dR is given, dR/dr_k (three row-major 3x3); the identity without columns
__device__ __forceinline__ void pair_side(const double *__restrict__ z, int col, double *R, double *t, double *dR) {
    if (col < 0) {
        for (int i = 0; i < 9; i++) R[i] = (i % 4 == 0) ? 1.0 : 0.0;
        for (int i = 0; i < 3; i++) t[i] = 0.0;
        return;
    }
    const double *z6 = z + col;
    rodrigues(z6[0], z6[1], z6[2], R);
    for (int i = 0; i < 3; i++) t[i] = z6[3 + i];
    if (dR) aar_an_rodrigues_derivs(z6, R, dR);
}

// residual row r (0..11) of a pair at the side poses; (A^T B)_ij = sum_m A_mi B_mj in the order ((m0 + m1) + m2), the oracle's
// (tests/pair_prior_oracle.cpp)
__device__ __forceinline__ double pair_residual_row(const PairPriorRec &q, int r, const double *Ra, const double *ta, const double *Rb, const double *tb) {
    if (r < 9) {
        const int i = r / 3, j = r - 3 * i;
        const double rab = (Ra[i] * Rb[j] + Ra[3 + i] * Rb[3 + j]) + Ra[6 + i] * Rb[6 + j];
        return sqrt(0.5 * q.w_rot) * (rab - q.R[r]);
    }
    const int i = r - 9;
    const double d0 = tb[0] - ta[0], d1 = tb[1] - ta[1], d2 = tb[2] - ta[2];
    const double tab = (Ra[i] * d0 + Ra[3 + i] * d1) + Ra[6 + i] * d2;
    return sqrt(q.w_t) * (tab - q.t[i]);
}

// J^T J of the pair rows into Hrr (diagonal blocks: both triangles, as the assembly writes them; the (a, b) block: the upper block
// triangle, transposed when b's block comes first) and J^T e into gr, at z.  Lanes 0 / 1 expand the two sides, lanes 0..11 form one
// row of J (columns [r_a t_a | r_b t_b]) and its residual each, then every lane takes entries of J^T [J | e].
__global__ void __launch_bounds__(PP_WARPS * 32) k_pair_prior_add(int n, const PairPriorRec *__restrict__ pr, int n_r, const double *__restrict__ z,
                                                                 double *__restrict__ Hrr, double *__restrict__ gr) {
    __shared__ double sm[PP_WARPS][PP_SMEM];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int k = blockIdx.x * PP_WARPS + w;
    if (k >= n) return;                          // warp-uniform
    const PairPriorRec &q = pr[k];
    double *Ra = sm[w], *ta = Ra + 9, *dRa = Ra + 12, *Rb = Ra + 39, *tb = Ra + 48, *dRb = Ra + 51, *e = Ra + 78, *J = Ra + 90;
    if (lane < 2) pair_side(z, lane ? q.col_b : q.col_a, lane ? Rb : Ra, lane ? tb : ta, lane ? dRb : dRa);
    __syncwarp();
    if (lane < 12) {
        const int r = lane;
        double *Jr = J + 12 * r;
        e[r] = pair_residual_row(q, r, Ra, ta, Rb, tb);
        if (r < 9) {                             // d(R_a^T R_b)_ij: (dR_a/dr_k)^T R_b and R_a^T dR_b/dr_k; no translation columns
            const int i = r / 3, j = r - 3 * i;
            const double s = sqrt(0.5 * q.w_rot);
            for (int c = 0; c < 3; c++) {
                const double *Da = dRa + 9 * c, *Db = dRb + 9 * c;
                Jr[c] = q.col_a < 0 ? 0.0 : s * ((Da[i] * Rb[j] + Da[3 + i] * Rb[3 + j]) + Da[6 + i] * Rb[6 + j]);
                Jr[3 + c] = 0.0;
                Jr[6 + c] = q.col_b < 0 ? 0.0 : s * ((Ra[i] * Db[j] + Ra[3 + i] * Db[3 + j]) + Ra[6 + i] * Db[6 + j]);
                Jr[9 + c] = 0.0;
            }
        } else {                                 // d(R_a^T (t_b - t_a))_i: (dR_a/dr_k)^T d, -R_a^T, 0, R_a^T
            const int i = r - 9;
            const double s = sqrt(q.w_t);
            const double d0 = tb[0] - ta[0], d1 = tb[1] - ta[1], d2 = tb[2] - ta[2];
            for (int c = 0; c < 3; c++) {
                const double *Da = dRa + 9 * c;
                Jr[c] = q.col_a < 0 ? 0.0 : s * ((Da[i] * d0 + Da[3 + i] * d1) + Da[6 + i] * d2);
                Jr[3 + c] = -(s * Ra[3 * c + i]);
                Jr[6 + c] = 0.0;
                Jr[9 + c] = s * Ra[3 * c + i];
            }
        }
    }
    __syncwarp();
    for (int x = lane; x < 144 + 12; x += 32) {
        const int i = x < 144 ? x / 12 : x - 144, j = x < 144 ? x - 12 * i : -1;
        const int ci = i < 6 ? q.col_a : q.col_b;
        if (ci < 0) continue;
        if (j < 0) {                             // gradient entry
            double g = 0.0;
            for (int r = 0; r < 12; r++) g += J[12 * r + i] * e[r];
            if (g != 0.0) atomicAdd(gr + ci + i % 6, g);
            continue;
        }
        const int cj = j < 6 ? q.col_a : q.col_b;
        if (cj < 0 || ci > cj) continue;         // a missing side, or the lower block triangle
        double h = 0.0;
        for (int r = 0; r < 12; r++) h += J[12 * r + i] * J[12 * r + j];
        if (h != 0.0) atomicAdd(Hrr + (size_t)(ci + i % 6) * n_r + cj + j % 6, h);
    }
}

// cost += the pairs' squared residual sum at z (the trial point inside a try): one thread per pair, a block reduction, one atomic
// per CTA into cost (d_red3[0], where k_residual adds the reprojection sum).
__global__ void __launch_bounds__(256) k_pair_prior_cost(int n, const PairPriorRec *__restrict__ pr, const double *__restrict__ z, double *__restrict__ cost) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    double acc = 0.0;
    if (k < n) {
        const PairPriorRec &q = pr[k];
        double Ra[9], ta[3], Rb[9], tb[3];
        pair_side(z, q.col_a, Ra, ta, nullptr);
        pair_side(z, q.col_b, Rb, tb, nullptr);
        for (int r = 0; r < 12; r++) { const double v = pair_residual_row(q, r, Ra, ta, Rb, tb); acc += v * v; }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    __shared__ double wsum[8];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) wsum[w] = acc;
    __syncthreads();
    if (w == 0) {
        acc = lane < (int)(blockDim.x >> 5) ? wsum[lane] : 0.0;
#pragma unroll
        for (int s = 4; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
        if (lane == 0 && acc != 0.0) atomicAdd(cost, acc);
    }
}

} // namespace aar
