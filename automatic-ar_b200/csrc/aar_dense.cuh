// aar_dense.cuh — dense Cholesky solve of the reduced camera+marker system (S + mu I) x = b, the part of
// sparselevmarq.h:394-400 that is left after the frames are eliminated.  n_r = 6(C-1) + 6(M-1) is a few hundred at
// most (468 at BASELINE cfg 4): far too small for tensor cores to matter, far too large for one thread block's
// shared memory, and on the critical path of every LM try.  Left-looking blocked factorisation, one CTA per block
// row of 32, two grid-wide synchronisations per block column (cooperative launch):
//   step k:  every CTA i >= k:  A_ik -= sum_{j<k} L_ij L_kj^T          (32x32x32 tile products from L2)
//            CTA k:             L_kk = chol(A_kk), X_k = L_kk^-1 in shared memory -> grid sync
//            every CTA i > k:   L_ik = A_ik X_k^T   (a tile product, not a row-serial solve) -> grid sync
// then forward / backward substitution by CTA 0.  S: row-major n x n, UPPER triangle valid on entry (the Schur
// kernels only write the upper block triangle); the lower triangle holds L on exit.
#pragma once
#include <cooperative_groups.h>

namespace aar {

constexpr int CH_NB = 32;
constexpr int CH_THREADS = 256;
constexpr int CH_LD = CH_NB + 1;

__global__ void __launch_bounds__(CH_THREADS) k_reduced_solve(int n, double *__restrict__ S, const double *__restrict__ b, double *__restrict__ x, const LmState *__restrict__ st,
                                                              int *__restrict__ chol_fail, double *__restrict__ Xinv /* [nblk][32][32] inverses of the diagonal factors */) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ double sA[CH_NB * CH_LD], sB[CH_NB * CH_LD], sC[CH_NB * CH_LD];
    __shared__ double sv[CH_NB];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int nblk = (n + CH_NB - 1) / CH_NB;
    const double mu = st->mu;
    // lower <- upper, diagonal += mu
    for (long long e = (long long)blockIdx.x * CH_THREADS + tid; e < (long long)n * n; e += (long long)gridDim.x * CH_THREADS) {
        const int i = (int)(e / n), j = (int)(e % n);
        if (i > j) S[e] = S[(size_t)j * n + i];
        else if (i == j) S[e] += mu;
    }
    grid.sync();
    auto load_tile = [&](double *dst, int bi, int bj) {       // rows of block bi, columns of block bj, zero padded
        for (int e = tid; e < CH_NB * CH_NB; e += CH_THREADS) {
            const int r = e / CH_NB, c = e % CH_NB, gr = bi * CH_NB + r, gc = bj * CH_NB + c;
            dst[r * CH_LD + c] = (gr < n && gc < n) ? S[(size_t)gr * n + gc] : 0.0;
        }
    };
    for (int k = 0; k < nblk; k++) {
        for (int i = k + blockIdx.x; i < nblk; i += gridDim.x) {
            // ---- A_ik -= sum_{j<k} L_ij L_kj^T ; each thread owns 2x2 entries of the tile
            double c00 = 0, c01 = 0, c10 = 0, c11 = 0;
            for (int j = 0; j < k; j++) {
                __syncthreads();
                load_tile(sA, i, j); load_tile(sB, k, j);
                __syncthreads();
#pragma unroll 8
                for (int q = 0; q < CH_NB; q++) {
                    const double a0 = sA[ty * CH_LD + q], a1 = sA[(ty + 16) * CH_LD + q], b0 = sB[tx * CH_LD + q], b1 = sB[(tx + 16) * CH_LD + q];
                    c00 = fma(a0, b0, c00); c01 = fma(a0, b1, c01); c10 = fma(a1, b0, c10); c11 = fma(a1, b1, c11);
                }
            }
            __syncthreads();
            load_tile(sC, i, k);
            __syncthreads();
            sC[ty * CH_LD + tx] -= c00; sC[ty * CH_LD + tx + 16] -= c01; sC[(ty + 16) * CH_LD + tx] -= c10; sC[(ty + 16) * CH_LD + tx + 16] -= c11;
            __syncthreads();
            if (i == k) {
                // ---- L_kk = chol(A_kk) in shared memory (padding rows/cols beyond n get a unit diagonal)
                for (int e = tid; e < CH_NB; e += CH_THREADS) if (k * CH_NB + e >= n) sC[e * CH_LD + e] = 1.0;
                __syncthreads();
                for (int j = 0; j < CH_NB; j++) {
                    if (tid == 0) { double d = sC[j * CH_LD + j]; if (!(d > 0)) { atomicExch(chol_fail, 1); d = 1; } sv[0] = sqrt(d); }
                    __syncthreads();
                    const double dj = sv[0];
                    if (tid > j && tid < CH_NB) sC[tid * CH_LD + j] /= dj;
                    if (tid == j) sC[j * CH_LD + j] = dj;
                    __syncthreads();
                    // trailing update of the lower triangle: rows r > j, columns j < c <= r
                    for (int e = tid; e < CH_NB * CH_NB; e += CH_THREADS) {
                        const int r = e / CH_NB, c = e % CH_NB;
                        if (c > j && r >= c) sC[r * CH_LD + c] = fma(-sC[r * CH_LD + j], sC[c * CH_LD + j], sC[r * CH_LD + c]);
                    }
                    __syncthreads();
                }
                // X = L_kk^-1 (lower triangular): thread c < 32 solves L X[:, c] = e_c by forward substitution
                if (tid < CH_NB) {
                    const int c = tid;
                    for (int r = 0; r < CH_NB; r++) {
                        double v = r == c ? 1.0 : 0.0;
                        for (int q = c; q < r; q++) v = fma(-sC[r * CH_LD + q], sB[q * CH_LD + c], v);
                        sB[r * CH_LD + c] = r < c ? 0.0 : v / sC[r * CH_LD + r];
                    }
                }
                __syncthreads();
                for (int e = tid; e < CH_NB * CH_NB; e += CH_THREADS) Xinv[(size_t)k * CH_NB * CH_NB + e] = sB[(e / CH_NB) * CH_LD + e % CH_NB];
            }
            // write the tile back (A_ik updated, or L_kk: lower triangle only)
            for (int e = tid; e < CH_NB * CH_NB; e += CH_THREADS) {
                const int r = e / CH_NB, c = e % CH_NB, gr = i * CH_NB + r, gc = k * CH_NB + c;
                if (gr < n && gc < n && (i != k || c <= r)) S[(size_t)gr * n + gc] = sC[r * CH_LD + c];
            }
        }
        grid.sync();
        // ---- L_ik = A_ik X_k^T for i > k (X_k = L_kk^-1): L_ik[r][c] = sum_q A_ik[r][q] X_k[c][q]
        {
            bool loaded = false;
            for (int i = k + 1 + blockIdx.x; i < nblk; i += gridDim.x) {
                __syncthreads();
                if (!loaded) { for (int e = tid; e < CH_NB * CH_NB; e += CH_THREADS) sB[(e / CH_NB) * CH_LD + e % CH_NB] = Xinv[(size_t)k * CH_NB * CH_NB + e]; loaded = true; }
                load_tile(sC, i, k);
                __syncthreads();
                double c00 = 0, c01 = 0, c10 = 0, c11 = 0;
#pragma unroll 8
                for (int q = 0; q < CH_NB; q++) {
                    const double a0 = sC[ty * CH_LD + q], a1 = sC[(ty + 16) * CH_LD + q], b0 = sB[tx * CH_LD + q], b1 = sB[(tx + 16) * CH_LD + q];
                    c00 = fma(a0, b0, c00); c01 = fma(a0, b1, c01); c10 = fma(a1, b0, c10); c11 = fma(a1, b1, c11);
                }
                const int gr0 = i * CH_NB + ty, gr1 = gr0 + 16, gc0 = k * CH_NB + tx, gc1 = gc0 + 16;
                if (gr0 < n && gc0 < n) S[(size_t)gr0 * n + gc0] = c00;
                if (gr0 < n && gc1 < n) S[(size_t)gr0 * n + gc1] = c01;
                if (gr1 < n && gc0 < n) S[(size_t)gr1 * n + gc0] = c10;
                if (gr1 < n && gc1 < n) S[(size_t)gr1 * n + gc1] = c11;
            }
        }
        grid.sync();
    }
    // ---- L y = b, L^T x = y (CTA 0; dot products spread over the block, one warp per 4 rows)
    if (blockIdx.x != 0) return;
    for (int i = tid; i < n; i += CH_THREADS) x[i] = b[i];
    __syncthreads();
    const int lane = tid & 31, warp = tid >> 5;
    for (int kb = 0; kb < nblk; kb++) {
        const int r0 = kb * CH_NB, nr = min(CH_NB, n - r0);
        // rows of this block minus the contribution of the solved part
        for (int r = warp; r < nr; r += CH_THREADS / 32) {
            double s = 0;
            for (int c = lane; c < r0; c += 32) s = fma(S[(size_t)(r0 + r) * n + c], x[c], s);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) sv[r] = x[r0 + r] - s;
        }
        __syncthreads();
        load_tile(sC, kb, kb);          // the diagonal factor, staged once (the solve below is latency bound)
        __syncthreads();
        if (warp == 0) {   // 32x32 triangular solve, lane r owns row r
            double v = lane < nr ? sv[lane] : 0.0;
            for (int c = 0; c < nr; c++) {
                const double xc = __shfl_sync(0xffffffffu, v, c) / sC[c * CH_LD + c];
                if (lane == c) v = xc;
                else if (lane > c && lane < nr) v = fma(-sC[lane * CH_LD + c], xc, v);
            }
            if (lane < nr) x[r0 + lane] = v;
        }
        __syncthreads();
    }
    for (int kb = nblk - 1; kb >= 0; kb--) {
        const int r0 = kb * CH_NB, nr = min(CH_NB, n - r0), c0 = r0 + nr;
        for (int r = warp; r < nr; r += CH_THREADS / 32) {
            double s = 0;
            for (int c = c0 + lane; c < n; c += 32) s = fma(S[(size_t)c * n + r0 + r], x[c], s);     // L^T: column r0+r below the block
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) sv[r] = x[r0 + r] - s;
        }
        __syncthreads();
        load_tile(sC, kb, kb);
        __syncthreads();
        if (warp == 0) {
            double v = lane < nr ? sv[lane] : 0.0;
            for (int c = nr - 1; c >= 0; c--) {
                const double xc = __shfl_sync(0xffffffffu, v, c) / sC[c * CH_LD + c];
                if (lane == c) v = xc;
                else if (lane < c) v = fma(-sC[c * CH_LD + lane], xc, v);
            }
            if (lane < nr) x[r0 + lane] = v;
        }
        __syncthreads();
    }
}


// ------------------------------------------------------------------------------------------------
// Cluster variant for n <= 512 (every BASELINE configuration: n_r = 468 at cfg 4): ONE thread-block cluster of nblk <= 16 CTAs,
// CTA i owns block row i of the matrix in its shared memory for the whole solve and the synchronisations per block column are
// hardware cluster barriers instead of grid-wide barriers through global memory.
namespace cg = cooperative_groups;

// Round 2: re-built around what clock64 timers inside the round-1 kernel (same algorithm, tiles of other CTAs read through
// distributed shared memory, CUDA-core tile products, a 32 x 32 diagonal factorisation with three CTA barriers per column) showed at n = 468 (0.61 ms for 34 Mflop; cycles of the last block row's CTA: 703 k waiting for the diagonal CTA of each
// step, 241 k in its own tile products, 46 k in the back substitution):
//   * the 32 x 32 diagonal factorisation took ~50 k cycles per block (96 CTA-wide barriers; a register version whose row array
//     the compiler had put in local memory was no faster): now ONE warp, lane = row, the row in registers with unconditional
//     updates only (no local memory), the pivot column by shuffles, 1 / sqrt by rsqrt — no barrier, no division;
//   * tile products were shared-memory-load bound (2.3 k cycles per 32 x 32 x 32 product: 4 LDS per 4 DFMA): now on the FP64
//     tensor cores (mma.sync.m8n8k4.f64), two 8 x 8 output tiles per warp, 3 LDS per 2 DMMA;
//   * remote panels came through distributed shared memory one 8-byte load at a time: finished tiles are now MIRRORED into the
//     lower triangle of S in global memory (L2-resident) and panels are read from there with coalesced ld.global.cg, at most 8
//     tiles per copy; DSMEM only carries the 32-double vectors of the substitutions;
//   * forward substitution ran as 15 more barrier-separated steps: now y_k = L_kk^-1 (b_k - L(k, <k) y) rides on step k;
//   * back substitution pulled a remote tile through one thread per column: now the owner of block row i pushes L(i, k)^T x_i
//     into the partial sums of every CTA k < i (it holds those tiles), one barrier per step;
//   * the block row is loaded from the upper triangle with lanes along the contiguous direction.
#ifdef AAR_SOLVE_TIMING
#define SOLVE_T(slot) do { if (tid == 0 && me == AAR_SOLVE_TIMING) { tt[slot] += clock64() - t_last; } if (tid == 0) t_last = clock64(); } while (0)
#else
#define SOLVE_T(slot) do { } while (0)
#endif
constexpr int CH_PT = 8;                                   // tiles of a remote panel staged at once
constexpr int CH_PLD = CH_PT * CH_NB + 2;
constexpr int CH_XLD = CH_NB + 2;                          // even stride: 16-byte aligned rows, conflict-free column access by lane = row
__host__ __device__ inline size_t cluster2_smem_bytes(int nblk) {
    return ((size_t)CH_NB * (nblk * CH_NB + 2) + (size_t)CH_NB * CH_PLD + 2 * CH_NB * CH_XLD + (size_t)nblk * CH_NB + 3 * CH_NB) * sizeof(double);
}
__device__ __forceinline__ void dmma_k4(double (&c)[2], double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}
// acc0 / acc1 += A[8 rb .. +8][0 .. 32) * B[8 cb .. +8][0 .. 32)^T and the same for column block cb + 1 (A, B row-major in shared memory)
__device__ __forceinline__ void tile_mma(const double *A, int lda, const double *B, int ldb, int g, int q, int rb, int cb, double (&acc0)[2], double (&acc1)[2]) {
    const double *pa = A + (rb * 8 + g) * lda + q, *pb0 = B + (cb * 8 + g) * ldb + q, *pb1 = pb0 + 8 * ldb;
#pragma unroll
    for (int k0 = 0; k0 < CH_NB; k0 += 4) { const double a = pa[k0], b0 = pb0[k0], b1 = pb1[k0]; dmma_k4(acc0, a, b0); dmma_k4(acc1, a, b1); }
}

// 32 x 32 tile (row stride ld, 16-byte aligned rows, even ld) from global memory into shared memory with 16-byte loads, all in flight
__device__ __forceinline__ void stage_tiles(double *dst, int ldd, const double *src, int lds, int nt, int tid) {
    const int r = tid >> 4, c2 = tid & 15;                 // 256 threads: rows r and r + 16, double2 column c2 of every tile
    double2 v0[CH_PT], v1[CH_PT];
#pragma unroll
    for (int t = 0; t < CH_PT; t++)
        if (t < nt) {
            v0[t] = __ldcg(reinterpret_cast<const double2 *>(src + (size_t)r * lds + t * CH_NB) + c2);
            v1[t] = __ldcg(reinterpret_cast<const double2 *>(src + (size_t)(r + 16) * lds + t * CH_NB) + c2);
        }
#pragma unroll
    for (int t = 0; t < CH_PT; t++)
        if (t < nt) {
            *reinterpret_cast<double2 *>(dst + r * ldd + t * CH_NB + 2 * c2) = v0[t];
            *reinterpret_cast<double2 *>(dst + (r + 16) * ldd + t * CH_NB + 2 * c2) = v1[t];
        }
}

__global__ void __launch_bounds__(CH_THREADS) k_reduced_solve_cluster2(int n /* even */, double *__restrict__ S, const double *__restrict__ b, double *__restrict__ x, const LmState *__restrict__ st,
                                                                       int *__restrict__ chol_fail, double *__restrict__ Xinv /* [nblk][32][32] */) {
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(16) double sm[];
    const int nblk = (n + CH_NB - 1) / CH_NB, LD = nblk * CH_NB + 2;
    double *sRow = sm;                                   // [32][LD]    block row `me` of the matrix / of L
    double *sP = sRow + CH_NB * LD;                      // [32][CH_PLD] staged part of a panel L(k + 1, j0 .. j1)
    double *sX = sP + CH_NB * CH_PLD;                    // [32][34]    inverse of this CTA's diagonal factor
    double *sXr = sX + CH_NB * CH_XLD;                   // [32][34]    staged tile of another CTA / work copy of the diagonal tile
    double *sy = sXr + CH_NB * CH_XLD;                   // [nblk*32]   b, then y — replicated in every CTA
    double *ss = sy + nblk * CH_NB;                      // [32]        partial sums of the back substitution (pushed by the CTAs above)
    double *sv = ss + CH_NB;                             // [32]        scratch (pivot column / right-hand side)
    double *sd = sv + CH_NB;                             // [32]        reciprocals of the diagonal of L_kk
    const int me = (int)cluster.block_rank(), tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, q = lane & 3, rb = warp & 3, cb = (warp >> 2) * 2;      // this warp's output tiles: rows 8 rb, columns 8 cb and 8 (cb + 1)
    const double mu = st->mu;
#ifdef AAR_SOLVE_TIMING
    long long t_last = clock64(), tt[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#endif
    for (int e = tid; e < CH_NB * nblk * CH_NB; e += CH_THREADS) {
        const int r = e % CH_NB, c = e / CH_NB, gr = me * CH_NB + r;
        double v = 0.0;
        if (gr < n && c <= gr) v = S[(size_t)c * n + gr] + (c == gr ? mu : 0.0);
        else if (gr >= n && c == gr) v = 1.0;
        sRow[r * LD + c] = v;
    }
    for (int e = tid; e < nblk * CH_NB; e += CH_THREADS) sy[e] = e < n ? b[e] : 0.0;
    if (tid < CH_NB) ss[tid] = 0.0;
    SOLVE_T(0);
    cluster.sync();
    SOLVE_T(1);
    double acc0[2] = {0, 0}, acc1[2] = {0, 0};           // this warp's share of the update of tile (me, k + 1), carried across the barriers of step k
    for (int k = 0; k < nblk; k++) {
        // ================= phase A: CTA k factorises its (fully updated) diagonal tile; the CTAs below start on column k + 1 with the
        // columns j < k that are already final — their products hide behind the serial factorisation
        if (me == k) {
            double *C = sRow + k * CH_NB;
            if (warp == 0) {
                // ---- L_kk = chol(C): lane = row, the row in registers (unconditional updates only: a predicated update sent the
                // array to local memory), pivot column through shared memory (one STS + 16 LDS.128 instead of 62 SHFL per column).
                // Compact loops over shared memory were tried instead of this straight-line code: 37 k cycles per block against 16 k.
                double a[CH_NB];
#pragma unroll
                for (int c = 0; c < CH_NB; c++) a[c] = C[lane * LD + c];
                bool bad = false;
#pragma unroll
                for (int j = 0; j < CH_NB; j++) {
                    double d = __shfl_sync(0xffffffffu, a[j], j);
                    const bool ok = d > 0;
                    bad |= !ok; d = ok ? d : 1.0;
                    const double rs = rsqrt(d);
                    const double l = lane > j ? a[j] * rs : (lane == j ? d * rs : 0.0);
                    a[j] = l;
                    if (j + 1 < CH_NB) {
                        sv[lane] = l;
                        __syncwarp();
#pragma unroll
                        for (int c = (j + 1) & ~1; c < CH_NB; c += 2) {
                            const double2 lc = *reinterpret_cast<const double2 *>(sv + c);
                            if (c > j) a[c] = fma(-l, c <= lane ? lc.x : 0.0, a[c]);
                            a[c + 1] = fma(-l, c + 1 <= lane ? lc.y : 0.0, a[c + 1]);
                        }
                        __syncwarp();
                    }
                    if (lane == j) sd[j] = rs;
                }
                if (bad && lane == 0) atomicExch(chol_fail, 1);
#pragma unroll
                for (int c = 0; c < CH_NB; c++) { const double v = c <= lane ? a[c] : 0.0; C[lane * LD + c] = v; sXr[lane * CH_XLD + c] = v; }
                __syncwarp();
                SOLVE_T(3);
                // ---- X = L_kk^-1: lane = column of X in registers, rows in turn (two partial sums per row), L from the padded copy
                double xc[CH_NB];
#pragma unroll
                for (int r = 0; r < CH_NB; r++) {
                    double v0 = r == lane ? 1.0 : 0.0, v1 = 0.0;
#pragma unroll
                    for (int qq = 0; qq + 1 < r; qq += 2) {
                        const double2 lr = *reinterpret_cast<const double2 *>(sXr + r * CH_XLD + qq);
                        v0 = fma(-lr.x, xc[qq], v0); v1 = fma(-lr.y, xc[qq + 1], v1);
                    }
                    if (r & 1) v0 = fma(-sXr[r * CH_XLD + r - 1], xc[r - 1], v0);
                    const double v = (v0 + v1) * sd[r];
                    xc[r] = r < lane ? 0.0 : v;
                }
#pragma unroll
                for (int r = 0; r < CH_NB; r++) sX[r * CH_XLD + lane] = xc[r];
                SOLVE_T(4);
            }
            // ---- forward substitution rides along: t = b_k - L(k, < k) y (warps 1..7), y_k = X t
            for (int r = warp - 1; r < CH_NB && warp > 0; r += CH_THREADS / 32 - 1) {
                double s = 0;
                for (int c = lane; c < k * CH_NB; c += 32) s = fma(sRow[r * LD + c], sy[c], s);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                if (lane == 0) ss[r] = sy[k * CH_NB + r] - s;                 // ss is free here: pushes into it only start with the back substitution
            }
            __syncthreads();
            if (tid < CH_NB) {
                double s = 0;
                for (int qq = 0; qq <= tid; qq++) s = fma(sX[tid * CH_XLD + qq], ss[qq], s);
                for (int rk = 0; rk < nblk; rk++) cluster.map_shared_rank(sy, rk)[k * CH_NB + tid] = s;
            }
            __syncthreads();
            if (tid < CH_NB) ss[tid] = 0.0;
            for (int e = tid; e < CH_NB * CH_NB; e += CH_THREADS) __stcg(Xinv + (size_t)k * CH_NB * CH_NB + e, sX[(e / CH_NB) * CH_XLD + e % CH_NB]);
        } else if (me > k) {
            // partial update of tile (me, k + 1): sum over j < k of L(me, j) L(k + 1, j)^T
            if (me == k + 1) {
                for (int j = 0; j < k; j++) tile_mma(sRow + j * CH_NB, LD, sRow + j * CH_NB, LD, g, q, rb, cb, acc0, acc1);
            } else {
                const double *rowk = S + (size_t)(k + 1) * CH_NB * n;           // rows of block k + 1, mirrored by CTA k + 1 (columns < 32 k are final)
                for (int j0 = 0; j0 < k; j0 += CH_PT) {
                    const int nt = min(CH_PT, k - j0);
                    __syncthreads();
                    stage_tiles(sP, CH_PLD, rowk + j0 * CH_NB, n, nt, tid);
                    __syncthreads();
                    for (int j = 0; j < nt; j++) tile_mma(sRow + (j0 + j) * CH_NB, LD, sP + j * CH_NB, CH_PLD, g, q, rb, cb, acc0, acc1);
                }
            }
        }
        SOLVE_T(5);
        cluster.sync();                                  // X_k (global) and y_k are visible to the cluster
        SOLVE_T(6);
        // ================= phase B: L(me, k) = C X_k^T for the CTAs below, mirrored into global memory
        if (me > k) {
            double *C = sRow + k * CH_NB;
            stage_tiles(sXr, CH_XLD, Xinv + (size_t)k * CH_NB * CH_NB, CH_NB, 1, tid);
            __syncthreads();
            double d0[2] = {0, 0}, d1[2] = {0, 0};
            tile_mma(C, LD, sXr, CH_XLD, g, q, rb, cb, d0, d1);
            __syncthreads();
            double *c0 = C + (rb * 8 + g) * LD + cb * 8 + 2 * q;
            c0[0] = d0[0]; c0[1] = d0[1]; c0[8] = d1[0]; c0[9] = d1[1];
            const int gr = me * CH_NB + rb * 8 + g, gc = k * CH_NB + cb * 8 + 2 * q;
            if (gr < n) { __stcg(reinterpret_cast<double2 *>(S + (size_t)gr * n + gc), make_double2(d0[0], d0[1])); __stcg(reinterpret_cast<double2 *>(S + (size_t)gr * n + gc + 8), make_double2(d1[0], d1[1])); }
        }
        SOLVE_T(7);
        cluster.sync();                                  // block column k of L is final (shared memory of its owners + global mirror)
        SOLVE_T(8);
        // ================= phase C: the last term (j = k) of the update of column k + 1, then the tile is ready
        if (me > k) {
            if (me == k + 1) { __syncthreads(); tile_mma(sRow + k * CH_NB, LD, sRow + k * CH_NB, LD, g, q, rb, cb, acc0, acc1); }
            else {
                __syncthreads();
                stage_tiles(sXr, CH_XLD, S + (size_t)(k + 1) * CH_NB * n + k * CH_NB, n, 1, tid);
                __syncthreads();
                tile_mma(sRow + k * CH_NB, LD, sXr, CH_XLD, g, q, rb, cb, acc0, acc1);
            }
            double *c0 = sRow + (k + 1) * CH_NB + (rb * 8 + g) * LD + cb * 8 + 2 * q;
            c0[0] -= acc0[0]; c0[1] -= acc0[1]; c0[8] -= acc1[0]; c0[9] -= acc1[1];
            acc0[0] = acc0[1] = acc1[0] = acc1[1] = 0.0;
            __syncthreads();
        }
        SOLVE_T(2);
    }
    SOLVE_T(9);
    // ---- back substitution  L^T x = y : the owner of block row i solves x_i and pushes L(i, k)^T x_i to every CTA k < i
    for (int i = nblk - 1; i >= 0; i--) {
        if (i == me) {
            if (tid < CH_NB) sv[tid] = sy[i * CH_NB + tid] - ss[tid];
            __syncthreads();
            if (tid < CH_NB) {
                double s = 0;
                for (int qq = tid; qq < CH_NB; qq++) s = fma(sX[qq * CH_XLD + tid], sv[qq], s);
                ss[tid] = s;                                                                 // ss now holds x_i for the pushes below
                if (i * CH_NB + tid < n) x[i * CH_NB + tid] = s;
            }
            __syncthreads();
            for (int c = tid; c < i * CH_NB; c += CH_THREADS) {                              // column c of block row i: tile k = c / 32
                double s = 0;
#pragma unroll 8
                for (int qq = 0; qq < CH_NB; qq++) s = fma(sRow[qq * LD + c], ss[qq], s);
                double *dst = cluster.map_shared_rank(ss, c / CH_NB);
                dst[c % CH_NB] += s;                                                         // only CTA i writes during step i
            }
        }
        cluster.sync();
    }
    SOLVE_T(10);
    cluster.sync();
#ifdef AAR_SOLVE_TIMING
    if (tid == 0 && me == AAR_SOLVE_TIMING)
        printf("solve timing CTA %d (cycles): load %lld sync0 %lld | phaseC %lld chol %lld inv %lld phaseA %lld syncA %lld panel %lld syncB %lld | tail %lld backsub %lld\n",
               me, tt[0], tt[1], tt[2], tt[3], tt[4], tt[5], tt[6], tt[7], tt[8], tt[9], tt[10]);
#endif
}

} // namespace aar
