// aar_fixed.cuh — cameras, markers and frames held fixed in the joint solve (aar_set_fixed, DESIGN.md §6d).
//
// Holding an entity fixed means running the reference's SparseLevMarq on the Jacobian whose columns of that entity are explicit
// zeros: their rows and columns of J^T J and their entries of J^T r are zero.  k_hold_fixed writes those zeros into this rank's
// normal equations after the assembly (and k_cm_reduce / k_intr_assemble), before anything reads them.  Every later kernel turns
// zero inputs into exact zeros: a fixed reduced block keeps mu alone on its diagonal and solves to a step of 0, a fixed frame's
// 6x6 block factors to sqrt(mu) I with a zero right-hand side, and zero W slots add nothing to S or b (k_schur_prepare,
// k_schur_syrk and k_backsub multiply them; the Cholesky kernels add mu before they take a root or divide).
#pragma once

namespace aar {

// blk_fixed: one byte per reduced block (cameras, markers, intrinsics pseudo-blocks), frame_fixed: one byte per local frame.  Only
// entries of held entities are written.
//  - W (nslots x 36 doubles, 2.2 GB at cfg 4): a warp takes 32 consecutive slots, reads their two slot maps coalesced and, when one of
//    them is held, writes the 32 x 18 double2 of the group with coalesced stores masked by the ballot of the held slots;
//  - Hrr (n_r^2), gr (n_r), Hf (F x HF_STRIDE): a grid-stride pass, one thread per entry.
__global__ void __launch_bounds__(256) k_hold_fixed(int n_r, const uint8_t *__restrict__ blk_fixed, int F, const uint8_t *__restrict__ frame_fixed,
                                                    long long nslots, const int *__restrict__ slot_block, const int *__restrict__ slot_frame,
                                                    double *__restrict__ Hrr, double *__restrict__ gr, double *__restrict__ Hf, double *__restrict__ W) {
    const int lane = threadIdx.x & 31;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, nthreads = (long long)gridDim.x * blockDim.x;
    for (long long s0 = (tid >> 5) * 32; s0 < nslots; s0 += (nthreads >> 5) * 32) {        // warp-uniform trip count
        const long long s = s0 + lane;
        const bool held = s < nslots && (blk_fixed[slot_block[s]] | frame_fixed[slot_frame[s]]);
        const unsigned ballot = __ballot_sync(0xffffffffu, held);
        if (!ballot) continue;
        double2 *w = reinterpret_cast<double2 *>(W + (size_t)s0 * 36);
        const int n2 = 18 * (int)min(32LL, nslots - s0);
        for (int e = lane; e < n2; e += 32)
            if ((ballot >> (e / 18)) & 1u) w[e] = make_double2(0.0, 0.0);
    }
    const long long nH = (long long)n_r * n_r, nG = nH + n_r, nF = nG + (long long)F * HF_STRIDE;
    for (long long e = tid; e < nF; e += nthreads) {
        if (e < nH) {
            const int i = (int)(e / n_r), j = (int)(e - (long long)i * n_r);
            if (blk_fixed[i / 6] | blk_fixed[j / 6]) Hrr[e] = 0.0;
        } else if (e < nG) {
            const int i = (int)(e - nH);
            if (blk_fixed[i / 6]) gr[i] = 0.0;
        } else {
            const long long k = e - nG;
            if (frame_fixed[k / HF_STRIDE]) Hf[k] = 0.0;
        }
    }
}

} // namespace aar
