// aar_report.cuh — reprojection-error report of a solved rig (aar_error_report, include/aar_cuda.h).
// Input: the 8 unweighted residuals of every observation, as k_residual / k_residual_an write them.
//   k_report_obs: observation error e = sqrt(s / 4), s = r0^2 + ... + r7^2 summed left to right without FMA, and the per-camera /
//                 per-marker / per-frame count, sum of s and max of e.
//   k_sel_hist + k_sel_pick: exact order statistics of e by an MSD radix select over the IEEE bits (non-negative doubles order like
//                 their bit patterns), SEL_PASSES digit passes shared by every requested rank.
#pragma once
#include <cstdint>

namespace aar {

constexpr int REP_THREADS = 256;
constexpr int SEL_BITS = 13, SEL_BINS = 1 << SEL_BITS, SEL_PASSES = 5;   // digits of 13, 13, 13, 13 and 12 bits, most significant first
constexpr int SEL_MAX_Q = 256;
constexpr unsigned long long REP_NAN_BITS = 0x7ff8000000000000ull;     // one NaN pattern: above +inf in bit order, so NaN errors sort last

__host__ __device__ __forceinline__ int sel_shift(int pass) { const int s = 64 - SEL_BITS * (pass + 1); return s < 0 ? 0 : s; }
__host__ __device__ __forceinline__ int sel_width(int pass) { return 64 - SEL_BITS * pass - sel_shift(pass); }

// Per warp: lanes holding the same key in consecutive lanes form a run; the first lane of each run adds the run's count, sum
// and max to the entity with one atomic each.  Frames are contiguous in row order and cameras are runs inside a frame, so a
// warp of 32 rows touches one or two entities.  key < 0: the lane holds no observation.
__device__ __forceinline__ void rep_run_add(int lane, int key, double s, unsigned long long eb, unsigned long long *__restrict__ cnt,
                                            double *__restrict__ sum, unsigned long long *__restrict__ mx) {
    const int prev = __shfl_up_sync(0xffffffffu, key, 1);
    const unsigned heads = __ballot_sync(0xffffffffu, lane == 0 || key != prev);
    const unsigned later = heads & ~((2u << lane) - 1u);
    const int end = later ? __ffs(later) - 1 : 32;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {           // suffix reduction inside the run: lane i ends with [i, end)
        const double so = __shfl_down_sync(0xffffffffu, s, d);
        const unsigned long long mo = __shfl_down_sync(0xffffffffu, eb, d);
        if (lane + d < end) { s += so; eb = mo > eb ? mo : eb; }
    }
    if (key >= 0 && ((heads >> lane) & 1u)) {
        atomicAdd(&cnt[key], (unsigned long long)(end - lane));
        atomicAdd(&sum[key], s);
        atomicMax(&mx[key], eb);
    }
}

// Entity index space of cnt / sum / mx: cameras [0, C), markers [C, C + M), frames [C + M, C + M + F).
// Markers have no locality in row order: per-block shared accumulators when marker_smem (flushed once per block), else global atomics.
__global__ void __launch_bounds__(REP_THREADS) k_report_obs(long long N, const double *__restrict__ r, const int *__restrict__ obs_f, const int *__restrict__ obs_cm,
                                                            int C, int M, int frame0, int marker_smem, double *__restrict__ err,
                                                            unsigned long long *__restrict__ cnt, double *__restrict__ sum, unsigned long long *__restrict__ mx) {
    extern __shared__ unsigned long long rep_smem[];                // [M] sums | [M] max bits | [M] counts
    double *s_sum = reinterpret_cast<double *>(rep_smem);
    unsigned long long *s_max = rep_smem + M;
    unsigned *s_cnt = reinterpret_cast<unsigned *>(rep_smem + 2 * (size_t)M);
    if (marker_smem) {
        for (int m = threadIdx.x; m < M; m += blockDim.x) { s_sum[m] = 0; s_max[m] = 0; s_cnt[m] = 0; }
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const int frame_key0 = C + M + frame0;
    for (long long base = (long long)blockIdx.x * blockDim.x; base < N; base += (long long)gridDim.x * blockDim.x) {   // uniform per block
        const long long o = base + threadIdx.x;
        double s = 0, e = 0; int c = -1, m = -1, f = -1;
        if (o < N) {
            const double2 *q = reinterpret_cast<const double2 *>(r + 8 * o);
            const double2 a = q[0], b = q[1], g = q[2], h = q[3];
            const double v[8] = {a.x, a.y, b.x, b.y, g.x, g.y, h.x, h.y};
            s = __dmul_rn(v[0], v[0]);
#pragma unroll
            for (int i = 1; i < 8; i++) s = __dadd_rn(s, __dmul_rn(v[i], v[i]));
            e = sqrt(s / 4.0);
            if (e != e) e = __longlong_as_double((long long)REP_NAN_BITS);
            err[o] = e;
            const int cm = obs_cm[o];
            c = obs_cam(cm); m = obs_marker(cm); f = frame_key0 + obs_f[o];
        }
        const unsigned long long eb = (unsigned long long)__double_as_longlong(e);
        rep_run_add(lane, c, s, eb, cnt, sum, mx);
        rep_run_add(lane, f, s, eb, cnt, sum, mx);
        if (m >= 0) {
            if (marker_smem) { atomicAdd(&s_cnt[m], 1u); atomicAdd(&s_sum[m], s); atomicMax(&s_max[m], eb); }
            else { atomicAdd(&cnt[C + m], 1ull); atomicAdd(&sum[C + m], s); atomicMax(&mx[C + m], eb); }
        }
    }
    if (marker_smem) {
        __syncthreads();
        for (int m = threadIdx.x; m < M; m += blockDim.x)
            if (s_cnt[m]) { atomicAdd(&cnt[C + m], (unsigned long long)s_cnt[m]); atomicAdd(&sum[C + m], s_sum[m]); atomicMax(&mx[C + m], s_max[m]); }
    }
}

// One digit pass of the select.  prefix[nq]: the bits every target has fixed so far, ascending (targets are sorted by rank).
// An element belongs to the first target with its prefix, and counts into that target's histogram [nq][SEL_BINS]; equal bins
// of a warp are merged before the atomic (ties).  smem_hist: pass 0 only (one prefix, one histogram), privatised per block.
__global__ void __launch_bounds__(REP_THREADS) k_sel_hist(long long N, const unsigned long long *__restrict__ keys, int pass, int nq,
                                                          const unsigned long long *__restrict__ prefix, int smem_hist, unsigned *__restrict__ hist) {
    __shared__ unsigned long long s_pre[SEL_MAX_Q];
    extern __shared__ unsigned s_hist[];
    for (int t = threadIdx.x; t < nq; t += blockDim.x) s_pre[t] = prefix[t];
    if (smem_hist) for (int b = threadIdx.x; b < SEL_BINS; b += blockDim.x) s_hist[b] = 0;
    __syncthreads();
    const int shift = sel_shift(pass), width = sel_width(pass);
    const unsigned long long hi = shift + width >= 64 ? 0ull : ~0ull << (shift + width);
    const unsigned dmask = (1u << width) - 1u;
    const int lane = threadIdx.x & 31;
    for (long long base = (long long)blockIdx.x * blockDim.x; base < N; base += (long long)gridDim.x * blockDim.x) {
        const long long o = base + threadIdx.x;
        unsigned bin = 0xffffffffu;
        if (o < N) {
            const unsigned long long k = keys[o], kp = k & hi;
            int lo = 0, n = nq;                 // first target whose prefix is >= kp
            while (n > 0) { const int h = n >> 1; if (s_pre[lo + h] < kp) { lo += h + 1; n -= h + 1; } else n = h; }
            if (lo < nq && s_pre[lo] == kp) bin = (unsigned)lo * SEL_BINS + (unsigned)((k >> shift) & dmask);
        }
        const unsigned peers = __match_any_sync(0xffffffffu, bin);
        if (bin != 0xffffffffu && lane == __ffs(peers) - 1) {
            if (smem_hist) atomicAdd(&s_hist[bin], (unsigned)__popc(peers));
            else atomicAdd(&hist[bin], (unsigned)__popc(peers));
        }
    }
    if (smem_hist) {
        __syncthreads();
        for (int b = threadIdx.x; b < SEL_BINS; b += blockDim.x) if (s_hist[b]) atomicAdd(&hist[b], s_hist[b]);
    }
}

// One block: for every target in turn, the bucket of the current digit that holds its rank; prefix |= digit, rank -= elements below.
__global__ void __launch_bounds__(REP_THREADS) k_sel_pick(int pass, int nq, unsigned long long *__restrict__ prefix, unsigned long long *__restrict__ rank,
                                                          const unsigned *__restrict__ hist) {
    __shared__ unsigned long long s_old[SEL_MAX_Q], s_warp[REP_THREADS / 32];
    for (int t = threadIdx.x; t < nq; t += blockDim.x) s_old[t] = prefix[t];
    __syncthreads();
    const int shift = sel_shift(pass), per = (1 << sel_width(pass)) / REP_THREADS;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int t = 0; t < nq; t++) {
        int owner = t;
        while (owner > 0 && s_old[owner - 1] == s_old[t]) owner--;
        const unsigned *h = hist + (size_t)owner * SEL_BINS + (size_t)threadIdx.x * per;
        unsigned long long mine = 0;
        for (int b = 0; b < per; b++) mine += h[b];
        unsigned long long incl = mine;             // block-wide inclusive scan of the per-thread sums
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const unsigned long long x = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += x; }
        if (lane == 31) s_warp[w] = incl;
        const unsigned long long k = rank[t];       // read by every thread before the one that owns the bucket rewrites it
        __syncthreads();
        unsigned long long before = incl - mine;
        for (int i = 0; i < w; i++) before += s_warp[i];
        if (k >= before && k < before + mine) {
            unsigned long long acc = before;
            for (int b = 0; b < per; b++) {
                if (k < acc + h[b]) { prefix[t] = s_old[t] | ((unsigned long long)(threadIdx.x * per + b) << shift); rank[t] = k - acc; break; }
                acc += h[b];
            }
        }
        __syncthreads();
    }
}

} // namespace aar
