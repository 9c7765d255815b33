// aar_schur.cuh — elimination of the per-frame 6x6 blocks (replaces the sparse LDLT of
// /root/reference/libs/sparselevmarq.h:394-400 on the arrow-shaped JtJ + mu I):
//
//   D_f = Hff_f + mu I = L_f L_f^T          y_f = L_f^-1 B_f            (k_frame_chol, one thread per frame)
//   E_s = W_s L_f^-T   for every W slot s    b[blk(s)] -= E_s y_f         (k_schur_prepare, one thread per slot row)
//   S[blk(s), blk(t)] -= E_s E_t^T  over all slot pairs of every frame    (k_schur_syrk, output-stationary tiles)
//
// The last step is a block-sparse SYRK of an n_r x 6F matrix.  S does not fit shared memory (468^2 doubles at
// BASELINE cfg 4), so the output is tiled: a CTA owns a 96x96 tile of S (16x16 blocks of 6x6, one block pair —
// 36 FP64 accumulators — per thread) and streams over a chunk of frames, staging the E blocks of its 16 row
// blocks and 16 column blocks through shared memory; the partial tiles of the frame chunks leave with one RED
// per entry.  DESIGN.md ("k_schur_syrk") has the roofline.
#pragma once

namespace aar {

constexpr int FC_STRIDE = FC_STRIDE_K;   // per frame: L (lower, packed by rows, 21) | y (6) | pad
constexpr int SY_TB = 16;          // 6x6 blocks per tile side
constexpr int SY_LD = 38;          // padded block stride in shared memory: 16-byte aligned blocks, conflict-free 128-bit loads across blocks
constexpr int SY_FB = 4;           // frames per pipeline stage
constexpr int SY_THREADS = 256;
constexpr size_t SY_SMEM = 2 * (sizeof(double) * 2 * SY_FB * SY_TB * SY_LD + sizeof(int) * 2 * SY_FB * SY_TB);   // two stages

// D = Hff + mu I = L L^T, y = L^-1 (-gf).  Non-positive pivot -> chol_fail (the reference does not check its LDLT,
// sparselevmarq.h:394-400; the host treats it as a rejected step).
__global__ void k_frame_chol(DevProblem p, const LmState *__restrict__ st, const double *__restrict__ Hf, double *__restrict__ fc, int *__restrict__ chol_fail) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= p.F) return;
    double L[36], y[6];
    if (!chol6(Hf + (size_t)f * HF_STRIDE, st->mu, L)) atomicExch(chol_fail, 1);
#pragma unroll
    for (int i = 0; i < 6; i++) y[i] = -Hf[(size_t)f * HF_STRIDE + 21 + i];
    fwd6(L, y);
    double *dst = fc + (size_t)f * FC_STRIDE;
    int idx = 0;
#pragma unroll
    for (int i = 0; i < 6; i++)
#pragma unroll
        for (int j = 0; j <= i; j++) dst[idx++] = L[i * 6 + j];
#pragma unroll
    for (int i = 0; i < 6; i++) dst[21 + i] = y[i];
}

// One thread per W slot: E_s[i][:] = L^-1 W_s[i][:]^T for its six rows, and b[blk(s)] -= E_s y.  The 32 slots of a warp are 9216
// consecutive bytes: they come in and go out through a per-warp shared-memory tile with coalesced 16-byte accesses (one thread
// walking its own 288-byte slot left half of every 32-byte sector unused per instruction: 3.4 TB/s at cfg 4); the 27 doubles of
// the frame's factor are read once per slot (neighbouring lanes share frames: L1 hits).
constexpr int SP_LD = 38;                                  // padded slot stride in shared memory (16-byte aligned, conflict-free for lane = slot)
constexpr size_t SP_TILE_BYTES = 32 * SP_LD * sizeof(double);
#ifndef AAR_SP_MINBLOCKS
#define AAR_SP_MINBLOCKS 2
#endif
__global__ void __launch_bounds__(256, AAR_SP_MINBLOCKS) k_schur_prepare(DevProblem p, long long nslots, const int *__restrict__ slot_frame, const double *__restrict__ fc,
                                                                         const double *__restrict__ W, double *__restrict__ E, double *__restrict__ b) {
    extern __shared__ __align__(16) double sp_smem[];   // [8 warps][32][SP_LD] tiles | [n_r] partial b of this CTA
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *tile = sp_smem + (size_t)warp * 32 * SP_LD;
    double *sb = sp_smem + (size_t)8 * 32 * SP_LD;
    for (int i = threadIdx.x; i < p.n_r; i += blockDim.x) sb[i] = 0.0;
    __syncthreads();
    const long long nwarps = (long long)gridDim.x * 8;
    for (long long s0 = ((long long)blockIdx.x * 8 + warp) * 32; s0 < nslots; s0 += nwarps * 32) {
        const int ns = (int)min(32LL, nslots - s0);
        // ---- 32 slots in: lane l takes double2 number l, l + 32, ... of the 18 * ns of the tile
        const double2 *src = reinterpret_cast<const double2 *>(W + (size_t)s0 * 36);
#pragma unroll
        for (int k = 0; k < 18; k++) {
            const int e = lane + 32 * k;
            if (e < 18 * ns) { const double2 v = src[e]; *reinterpret_cast<double2 *>(tile + (e / 18) * SP_LD + 2 * (e % 18)) = v; }
        }
        __syncwarp();
        if (lane < ns) {
            const long long s = s0 + lane;
            const double *lf = fc + (size_t)slot_frame[s] * FC_STRIDE;
            double l[27];
#pragma unroll
            for (int i = 0; i < 27; i++) l[i] = lf[i];
            double *w = tile + lane * SP_LD;
            double *bs = sb + 6 * p.slot_block[s];
#pragma unroll
            for (int i = 0; i < 6; i++) {
                double x[6];
#pragma unroll
                for (int k = 0; k < 3; k++) { const double2 v = *reinterpret_cast<const double2 *>(w + i * 6 + 2 * k); x[2 * k] = v.x; x[2 * k + 1] = v.y; }
                int idx = 0; double acc = 0.0;
#pragma unroll
                for (int r = 0; r < 6; r++) {            // forward substitution with the packed lower factor
                    double v = x[r];
#pragma unroll
                    for (int k = 0; k < r; k++) v = fma(-l[idx + k], x[k], v);
                    x[r] = v / l[idx + r];
                    idx += r + 1;
                    acc = fma(x[r], l[21 + r], acc);
                }
#pragma unroll
                for (int k = 0; k < 3; k++) *reinterpret_cast<double2 *>(w + i * 6 + 2 * k) = make_double2(x[2 * k], x[2 * k + 1]);
                atomicAdd(bs + i, -acc);
            }
        }
        __syncwarp();
        // ---- 32 slots out
        double2 *dst = reinterpret_cast<double2 *>(E + (size_t)s0 * 36);
#pragma unroll
        for (int k = 0; k < 18; k++) {
            const int e = lane + 32 * k;
            if (e < 18 * ns) dst[e] = *reinterpret_cast<const double2 *>(tile + (e / 18) * SP_LD + 2 * (e % 18));
        }
        __syncwarp();
    }
    __syncthreads();
    for (int i = threadIdx.x; i < p.n_r; i += blockDim.x) if (sb[i] != 0.0) atomicAdd(b + i, sb[i]);
}

// S[tile] -= sum over the frames of this chunk of E_I E_J^T.  frame_block_slot[f*nb + blk] is the W slot of
// reduced block blk in frame f, or -1.  gridDim.x = ntiles * nchunks (tile fastest).
// Software pipeline over batches of SY_FB frames: slot indices are fetched two batches ahead (registers), the E
// blocks one batch ahead (cp.async into the other shared-memory buffer, zero-filled for absent blocks), so the
// FP64 tensor-core products of batch b overlap the global-memory latency of batches b+1 and b+2.
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc, bool valid) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    const int sz = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(sz) : "memory");
}
#ifndef AAR_SY_MINBLOCKS
#define AAR_SY_MINBLOCKS 2
#endif
__global__ void __launch_bounds__(SY_THREADS, AAR_SY_MINBLOCKS) k_schur_syrk(DevProblem p, int nb, int tiles_side, int nchunks, const int *__restrict__ frame_block_slot,
                                                              const double *__restrict__ E, double *__restrict__ S) {
    extern __shared__ __align__(16) unsigned char sy_raw[];
    typedef double EBuf[2][SY_FB][SY_TB * SY_LD];          // [I|J][frame in batch][block][36 (+1)]
    typedef int PBuf[2][SY_FB][SY_TB];
    EBuf *sE = reinterpret_cast<EBuf *>(sy_raw);             // two pipeline stages
    PBuf *sPresent = reinterpret_cast<PBuf *>(sy_raw + 2 * sizeof(EBuf));
    const int ntiles = tiles_side * (tiles_side + 1) / 2;
    int tile = blockIdx.x % ntiles; const int chunk = blockIdx.x / ntiles;
    int ti = 0;
    while (tile >= tiles_side - ti) { tile -= tiles_side - ti; ti++; }
    const int tj = ti + tile;
    const int tid = threadIdx.x;
    const int f0 = (int)((long long)p.F * chunk / nchunks), f1 = (int)((long long)p.F * (chunk + 1) / nchunks);
    const int nbatch = (f1 - f0 + SY_FB - 1) / SY_FB;
    // slot-index prefetch: thread e < 2*SY_FB*SY_TB owns entry (side, ff, blk) of every batch
    const bool idx_thread = tid < 2 * SY_FB * SY_TB;
    const int i_side = tid / (SY_FB * SY_TB), i_ff = (tid / SY_TB) % SY_FB, i_blk = tid % SY_TB;
    const int i_g = (i_side ? tj : ti) * SY_TB + i_blk;
    auto fetch_slot = [&](int batch) -> int {
        const int f = f0 + batch * SY_FB + i_ff;
        return (idx_thread && batch < nbatch && f < f1 && i_g < nb) ? frame_block_slot[(size_t)f * nb + i_g] : -1;
    };
    auto issue_copy = [&](int stage) {      // E blocks of the batch whose slots are in sPresent[stage]
        double *dst0 = &sE[stage][0][0][0]; const int *pres = &sPresent[stage][0][0][0];
        for (int e = tid; e < 2 * SY_FB * SY_TB * 18; e += SY_THREADS) {
            const int k = e % 18, blkid = e / 18;            // blkid = (side*SY_FB + ff)*SY_TB + blk ; 18 x 16 bytes per block
            const int slot = pres[blkid];
            cp_async16(dst0 + (size_t)blkid * SY_LD + 2 * k, E + (size_t)(slot >= 0 ? slot : 0) * 36 + 2 * k, slot >= 0);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // FP64 tensor cores: the CTA tile is a 96 x 96 x (6 * SY_FB) GEMM per batch, A[m][k] = E_I[i][r] with m = (block, i) of the
    // row side and k = (frame in batch, r), B[k][n] the same of the column side; absent blocks were zero-filled by cp.async.
    // 2 x 4 warps, 48 x 24 outputs each = 6 x 3 mma.m8n8k4 tiles (36 accumulators per lane), 6 k-steps per batch:
    // 9 shared-memory loads per 18 DMMA instead of 36 vector loads per 216 FMAs.
    const int lane = tid & 31, wm = (tid >> 5) >> 2, wn = (tid >> 5) & 3, g = lane >> 2, q = lane & 3;
    int offA[6], offB[3], koff[6 * SY_FB / 4];
#pragma unroll
    for (int t = 0; t < 6; t++) { const int m = wm * 48 + t * 8 + g; offA[t] = (m / 6) * SY_LD + (m % 6) * 6; }
#pragma unroll
    for (int u = 0; u < 3; u++) { const int n = wn * 24 + u * 8 + g; offB[u] = (n / 6) * SY_LD + (n % 6) * 6; }
#pragma unroll
    for (int st = 0; st < 6 * SY_FB / 4; st++) { const int k = 4 * st + q; koff[st] = (k / 6) * (SY_TB * SY_LD) + (k % 6); }
    double cacc[6][3][2];
#pragma unroll
    for (int t = 0; t < 6; t++)
#pragma unroll
        for (int u = 0; u < 3; u++) { cacc[t][u][0] = 0.0; cacc[t][u][1] = 0.0; }
    // prologue: slots of batch 0 -> shared, copy of batch 0 in flight, slots of batch 1 in registers
    int slot_next = fetch_slot(0);
    if (idx_thread) (&sPresent[0][0][0][0])[tid] = slot_next;
    slot_next = fetch_slot(1);
    __syncthreads();
    issue_copy(0);
    for (int b = 0; b < nbatch; b++) {
        const int cur = b & 1, nxt = cur ^ 1;
        if (idx_thread) (&sPresent[nxt][0][0][0])[tid] = slot_next;        // slots of batch b+1
        slot_next = fetch_slot(b + 2);
        __syncthreads();
        if (b + 1 < nbatch) { issue_copy(nxt); asm volatile("cp.async.wait_group 1;" ::: "memory"); }
        else asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        {
            const double *A0 = &sE[cur][0][0][0], *B0 = &sE[cur][1][0][0];
#pragma unroll
            for (int st = 0; st < 6 * SY_FB / 4; st++) {
                double a[6], bb[3];
#pragma unroll
                for (int t = 0; t < 6; t++) a[t] = A0[offA[t] + koff[st]];
#pragma unroll
                for (int u = 0; u < 3; u++) bb[u] = B0[offB[u] + koff[st]];
#pragma unroll
                for (int t = 0; t < 6; t++)
#pragma unroll
                    for (int u = 0; u < 3; u++)
                        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                                     : "+d"(cacc[t][u][0]), "+d"(cacc[t][u][1]) : "d"(a[t]), "d"(bb[u]));
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int t = 0; t < 6; t++)
#pragma unroll
        for (int u = 0; u < 3; u++)
#pragma unroll
            for (int e = 0; e < 2; e++) {
                const int m = wm * 48 + t * 8 + g, n = wn * 24 + u * 8 + 2 * q + e;
                const int bim = m / 6, bjn = n / 6, gim = ti * SY_TB + bim, gjn = tj * SY_TB + bjn;
                const double v = cacc[t][u][e];
                if (gim < nb && gjn < nb && (ti != tj || bim <= bjn) && v != 0.0)
                    atomicAdd(S + (size_t)(6 * gim + m % 6) * p.n_r + 6 * gjn + n % 6, -v);
            }
}

} // namespace aar
