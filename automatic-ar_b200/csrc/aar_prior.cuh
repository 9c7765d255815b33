// aar_prior.cuh — soft pose priors on cameras, markers and frames in the joint solve (aar_set_prior, DESIGN.md §6e).
//
// A prior on an entity appends six rows sqrt(w) (z_e - zbar_e) to the residual vector, with the Jacobian rows diag(sqrt(w)) on the
// entity's six columns [r0 r1 r2 t0 t1 t2].  The reference's SparseLevMarq on that augmented problem needs three changes, all made
// here: J^T J gains w on the entity's diagonal and J^T r gains w (z - zbar) (k_prior_add, after the assembly and before anything reads
// the normal equations), and the cost gains sum w (z - zbar)^2 wherever the solver forms one (k_prior_cost, next to k_residual).
// Every later kernel (mu0, Schur step, both Cholesky kernels, back substitution, gain) reads the changed equations unchanged.
#pragma once

namespace aar {

constexpr int PRIOR_STRIDE = 12;   // per entity: zbar [6] | w [6]

// One thread per (entity, component): the first 6 nb threads take the reduced pose blocks (cameras, then markers; block b is
// columns 6 b .. 6 b + 5 of z), the next 6 F this rank's frames (columns col_frame0 + 6 f ..).  nb = 0 on every rank but rank 0:
// the all-reduce of the reduced system and of the cost adds the block terms once.
__device__ __forceinline__ bool prior_entry(long long t, int nb, const double *blk, const uint8_t *blk_has, int F, const double *fr,
                                            const uint8_t *fr_has, int col_frame0, int &ent, int &i, const double *&pr, long long &col) {
    const long long nbt = 6LL * nb;
    if (t < nbt) {
        ent = (int)(t / 6); i = (int)(t - 6LL * ent);
        if (!blk_has[ent]) return false;
        pr = blk + (size_t)ent * PRIOR_STRIDE; col = 6LL * ent + i;
        return true;
    }
    t -= nbt;
    if (t >= 6LL * F) return false;
    ent = (int)(t / 6); i = (int)(t - 6LL * ent);
    if (!fr_has[ent]) return false;
    pr = fr + (size_t)ent * PRIOR_STRIDE; col = (long long)col_frame0 + 6LL * ent + i;
    ent = -1 - ent;                 // a frame
    return true;
}

// J^T J += diag(w), J^T r += w (z - zbar) at z: the diagonal of Hrr and gr for blocks, the diagonal entries {0, 6, 11, 15, 18, 20} of
// the packed Hff and the gradient entries 21..26 of Hf for frames.  Only entities with a prior are written.
__global__ void __launch_bounds__(256) k_prior_add(int nb, const double *__restrict__ blk, const uint8_t *__restrict__ blk_has, int F,
                                                   const double *__restrict__ fr, const uint8_t *__restrict__ fr_has, int col_frame0, int n_r,
                                                   const double *__restrict__ z, double *__restrict__ Hrr, double *__restrict__ gr, double *__restrict__ Hf) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int ent, i; const double *pr; long long col;
    if (!prior_entry(t, nb, blk, blk_has, F, fr, fr_has, col_frame0, ent, i, pr, col)) return;
    const double w = pr[6 + i];
    if (w == 0.0) return;
    const double g = w * (z[col] - pr[i]);
    if (ent >= 0) {
        Hrr[(size_t)col * n_r + col] += w;
        gr[col] += g;
    } else {
        double *h = Hf + (size_t)(-1 - ent) * HF_STRIDE;
        h[6 * i - i * (i - 1) / 2] += w;            // diagonal entry i of the packed upper triangle: 0, 6, 11, 15, 18, 20
        h[21 + i] += g;
    }
}

// cost += sum w (z - zbar)^2 at z (the trial point inside a try): a block reduction, one atomic per CTA into cost (d_red3[0], where
// k_residual adds the reprojection sum).
__global__ void __launch_bounds__(256) k_prior_cost(int nb, const double *__restrict__ blk, const uint8_t *__restrict__ blk_has, int F,
                                                    const double *__restrict__ fr, const uint8_t *__restrict__ fr_has, int col_frame0,
                                                    const double *__restrict__ z, double *__restrict__ cost) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int ent, i; const double *pr; long long col;
    double acc = 0.0;
    if (prior_entry(t, nb, blk, blk_has, F, fr, fr_has, col_frame0, ent, i, pr, col)) {
        const double d = z[col] - pr[i];
        acc = pr[6 + i] * (d * d);
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
