// aar_cuda.cu — C-ABI layer (include/aar_cuda.h) over the sm_100a kernels of aar_kernels.cuh.
// Host side of the drop-in: problem description -> row/column maps (bit-exact contract), SoA upload,
// device-resident Levenberg-Marquardt loop, NCCL all-reduce of the reduced system for frame shards.
// There is no CPU fallback anywhere in this file: without a CUDA device every entry point fails.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <dlfcn.h>
#include <limits>
#include <unistd.h>
#include <map>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <vector>
#include <sched.h>

#include <cuda_runtime.h>
#include <nccl.h> // types only; the library is dlopen'ed so single-GPU use needs no NCCL

#include "../../include/aar_cuda.h"
#include "aar_host_math.h"
#include "aar_kernels.cuh"
#include "aar_lens.cuh"
#include "aar_report.cuh"
#include "aar_fixed.cuh"
#include "aar_prior.cuh"
#include "aar_pair_prior.cuh"

using namespace aar;

namespace {

thread_local std::string g_err;
void set_err(const char *fmt, ...) {
    char buf[1024];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    g_err = buf;
}
#define CU(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess) { set_err("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); return AAR_ERR_CUDA; } \
    } while (0)

// ------------------------------------------------------------------------------ NCCL (dlopen)
struct Nccl {
    void *lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool load() {
        if (lib) return true;
        const char *names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char *n : names) { lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (lib) break; }
        if (!lib) { set_err("NCCL: cannot dlopen libnccl.so.2: %s", dlerror()); return false; }
        GetUniqueId = (decltype(GetUniqueId))dlsym(lib, "ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))dlsym(lib, "ncclCommInitRank");
        AllReduce = (decltype(AllReduce))dlsym(lib, "ncclAllReduce");
        CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
        GetErrorString = (decltype(GetErrorString))dlsym(lib, "ncclGetErrorString");
        if (!GetUniqueId || !CommInitRank || !AllReduce || !CommDestroy) { set_err("NCCL: missing symbols"); return false; }
        return true;
    }
} g_nccl;

template <typename T> struct DevBuf {
    T *p = nullptr; size_t n = 0;
    cudaError_t alloc(size_t count) { free(); n = count; if (!count) return cudaSuccess; return cudaMalloc((void **)&p, count * sizeof(T)); }
    void free() { if (p) cudaFree(p); p = nullptr; n = 0; }
    ~DevBuf() { free(); }
};

} // namespace

struct aar_problem {
    // ---- description (host)
    int C = 0, M = 0, F = 0;                      // global counts
    std::vector<int> cam_ids, marker_ids, frame_ids;
    int root_cam_id = 0, root_marker_id = 0, root_cam = 0, root_marker = 0;
    float marker_size = 0;
    std::vector<double> cam_T, marker_T, frame_T, cam_K, cam_dist;
    bool opt_c = true, opt_m = true, opt_f = true, huber = false;
    double J_delta = 1e-3;
    int device = 0, rank = 0, world = 1;
    // ---- row map (global, a1 order) and shard
    long long N = 0;                               // global observations
    std::vector<int> g_frame, g_cam, g_marker, g_hasjac; // indices per global observation
    long long num_det = 0; std::vector<long long> g_det;  // desc->num_detections; index into desc->det_* of every global observation (aar_error_report)
    int f_begin = 0, f_end = 0;                    // this rank's frame index range
    long long o_begin = 0, o_end = 0;              // this rank's observation range
    int nrc = 0, nrm = 0, nri = 0, n_r = 0; bool opt_i = false;   // nri: 2 C intrinsics pseudo-blocks (aar_intrinsics.cuh)
    long long n_vars = 0;        // INTERNAL length of z: reduced part (pose blocks, then 12 per camera when the intrinsics are optimised), then frames
    long long n_vars_ext = 0;    // length of the reference's io_vec (get_num_vars, multicam_mapper.cpp:239-250): ... frames, then 9 per camera
    std::vector<double> z_stage; // host staging of the io_vec <-> internal conversion
    long long nslots = 0; int max_slots = 0;
    long long schur_fma = 0;                       // sum over local frames of 6 * n_f (n_f + 1) / 2, n_f = 6 * (blocks seen): the upper triangle of S -= E E^T
    // ---- device
    cudaStream_t stream = nullptr; bool own_stream = false;
    DevBuf<int> d_obs_f, d_obs_cm, d_slot_c, d_slot_m, d_frame_slot_ptr, d_slot_block;
    DevBuf<float4> d_und_a, d_und_b, d_raw_a, d_raw_b;
    DevBuf<int> d_frame_cs_cum, d_slot_frame, d_frame_block_slot, d_frame_obs_ptr, d_trk_iters, d_obs_pair;
    DevBuf<int2> d_pair_fc; DevBuf<double> d_pair_tab; int npairs = 0;
    DevBuf<int4> d_pair_info, d_mrun_info; DevBuf<int> d_perm_fm, d_pair_cam; DevBuf<double> d_cm_rep; int nmruns = 0;     // visiting orders of the tensor-core assembly (aar_assemble.cuh)
    bool analytic = false; DevBuf<double> d_cam_an, d_mk_an, d_fr_an;                 // analytic-Jacobian / full-FP64 variant (aar_analytic.cuh)
    bool lens = false; DevBuf<double> d_lens, d_lens_tr;                               // lens model (aar_lens.cuh): [C][9] at z / at the trial point
    DevBuf<double> d_trk_cam_inv, d_trk_Y, d_trk_z, d_trk_z0, d_trk_cost; bool trk_have_z0 = false; double track_ms = 0; long long track_runs = 0;
    DevBuf<double> d_fc, d_E, d_xinv;
    DevBuf<int> d_pair_slot_i; DevBuf<double> d_intr_tr, d_Ji;
    DevBuf<double> d_intr, d_K9, d_dist5, d_cam_tab, d_mk_tab, d_fr_tab, d_cam_tr, d_mk_tr, d_fr_tr, d_cam_fixed, d_mk_fixed, d_fr_fixed;
    DevBuf<double> d_z, d_zt, d_z0, d_Hf, d_W, d_Hrr, d_gr, d_red, d_dr, d_red3, d_tmp, d_r;
    DevBuf<LmState> d_st;
    DevBuf<int> d_flag;
    LmState *h_st = nullptr; double *h_red3 = nullptr; int *h_flags = nullptr; // pinned; h_st: LM state as last read back or pushed
    // ---- staged rows of central-difference numerators ([N][JROW] float32, or float64 in the exact fallback) and Huber weights ([N][4])
    DevBuf<float> d_Jn32; DevBuf<double> d_Jn64, d_Rv;
    int max_ms = 0, num_sms = 148; size_t smem_optin = 227 * 1024;
    bool use_cluster_solve = true;
    bool last_cluster_solve = false, last_smem_acc = false, last_cm_rep = false;   // paths of the last reduced solve and assembly (aar_problem_stats)
    int force_exact_staging = 0; long long exact_reruns = 0;
    DevProblem dp{};
    // ---- LM
    aar_lm_params params{};
    bool lm_active = false, have_z0 = false;
    double initial_cost = 0;
    // ---- comm
    ncclComm_t comm = nullptr;
    // ---- instrumentation
    long long launches = 0; bool profiling = false; bool exact_next = false;   // exact_next: redo this Jacobian with FP64 staging
    // graph-resident LM loop (aar_lm_iterate): two nested WHILE nodes, conditions set by k_lm_begin_iter / k_lm_decide / k_lm_next_iter_g
    cudaGraph_t lm_graph = nullptr; cudaGraphExec_t lm_exec = nullptr; cudaGraphConditionalHandle lm_outer = 0, lm_inner = 0; cudaStream_t lm_side = nullptr;
    bool lm_graph_tried = false, lm_graph_ok = false; long long lm_graph_launches = 0, lm_graph_iters = 0; int lm_body_launches = 0, lm_try_launches = 0;
    DevBuf<LmTraceDev> d_trace;
    // aar_error_report (aar_report.cuh): observation errors, entity statistics [C + M + F], select state [2 nq], digit histograms [nq][SEL_BINS]
    DevBuf<double> d_rep_err, d_rep_sum; DevBuf<unsigned long long> d_rep_cnt, d_rep_max, d_sel; DevBuf<unsigned> d_sel_hist;
    // aar_set_fixed (aar_fixed.cuh): one byte per reduced block and per local frame; without a mask nothing is launched
    bool has_fixed = false; DevBuf<uint8_t> d_blk_fixed, d_frame_fixed;
    std::vector<uint8_t> fixed_pose_blk, fixed_frame, fixed_intr;   // the masks of aar_set_fixed and aar_set_fixed_intrinsics (empty: none)
    // aar_set_prior (aar_prior.cuh): [zbar 6 | w 6] and a has-prior byte per reduced pose block and per local frame; without priors
    // nothing is launched
    bool has_prior = false; DevBuf<double> d_blk_prior, d_frame_prior; DevBuf<uint8_t> d_blk_has_prior, d_frame_has_prior;
    // aar_set_pair_prior (aar_pair_prior.cuh): one record per stored camera or marker pair; without pairs nothing is launched
    int n_pair = 0; DevBuf<PairPriorRec> d_pair_prior;
    cudaEvent_t ev[16] = {}; double phase_ms[AAR_NUM_PHASES] = {};
};

namespace {

#define LAUNCH(p, kernel, grid, block, smem, ...)                                    \
    do { kernel<<<(grid), (block), (smem), (p)->stream>>>(__VA_ARGS__); (p)->launches++; } while (0)

inline unsigned cdiv(long long a, long long b) { return (unsigned)((a + b - 1) / b); }

void pose12_from_T16(const double *T, double *out) {
    for (int i = 0; i < 3; i++) { for (int j = 0; j < 3; j++) out[i * 3 + j] = T[i * 4 + j]; out[9 + i] = T[i * 4 + 3]; }
}

bool strictly_ascending(const std::vector<int> &v) { for (size_t i = 1; i < v.size(); i++) if (v[i] <= v[i - 1]) return false; return true; }

int rank_of(const std::vector<int> &ids, int id) {
    auto it = std::lower_bound(ids.begin(), ids.end(), id);
    if (it == ids.end() || *it != id) return -1;
    return (int)(it - ids.begin());
}

// ---- host-side parallel loops of aar_problem_create (plain std::thread: the library links nothing but the CUDA runtime)
thread_local int g_ranks_on_host = 1;     // ranks of a sharded run that map their shards at the same time on this host (set by aar_problem_create)
int host_threads(long long work) {
    if (work < (1LL << 16)) return 1;
    static int n = [] {
        const char *e = getenv("AAR_HOST_THREADS");
        if (e && atoi(e) > 0) return atoi(e);
        cpu_set_t set; CPU_ZERO(&set);
        int c = sched_getaffinity(0, sizeof set, &set) == 0 ? CPU_COUNT(&set) : (int)std::thread::hardware_concurrency();
        return std::max(1, std::min(c, 64));
    }();
    return std::max(std::min(n, 8), n / std::max(1, g_ranks_on_host));     // one process per GPU: the ranks share the cores
}
template <class F> void parallel_for(long long n, int T, F fn) {      // fn(begin, end, thread index) over T contiguous chunks of [0, n)
    if (T <= 1 || n <= 0) { fn(0, std::max<long long>(n, 0), 0); return; }
    std::vector<std::thread> th; th.reserve((size_t)T - 1);
    for (int t = 1; t < T; t++) th.emplace_back([&, t] { fn(n * t / T, n * (t + 1) / T, t); });
    fn(0, n / T, 0);
    for (auto &x : th) x.join();
}
// id -> index of a strictly ascending id list: arithmetic when the ids are consecutive, a dense table when their range is small
struct IdMap {
    const std::vector<int> &ids; int lo = 0; bool consecutive = true; std::vector<int> table;
    explicit IdMap(const std::vector<int> &v) : ids(v) {
        if (ids.empty()) return;
        lo = ids.front();
        for (size_t i = 0; i < ids.size(); i++) if (ids[i] != lo + (int)i) { consecutive = false; break; }
        const long long range = (long long)ids.back() - lo + 1;
        if (!consecutive && range <= (long long)(4 * ids.size() + (1 << 20))) { table.assign((size_t)range, -1); for (size_t i = 0; i < ids.size(); i++) table[(size_t)(ids[i] - lo)] = (int)i; }
    }
    int operator()(int id) const {
        if (ids.empty()) return -1;
        if (consecutive) { const long long k = (long long)id - lo; return k >= 0 && k < (long long)ids.size() ? (int)k : -1; }
        if (!table.empty()) { const long long k = (long long)id - lo; return k >= 0 && k < (long long)table.size() ? table[(size_t)k] : -1; }
        return rank_of(ids, id);
    }
};

// column of a block in io_vec (SURVEY Appendix C; multicam_mapper.cpp:815-817, 824-826, 833)
long long col_cam(const aar_problem *p, int i) { if (!p->opt_c || i == p->root_cam) return -1; return 6LL * (i - (i > p->root_cam ? 1 : 0)); }
long long col_marker(const aar_problem *p, int j) { if (!p->opt_m || j == p->root_marker) return -1; return 6LL * p->nrc + 6LL * (j - (j > p->root_marker ? 1 : 0)); }
long long col_frame(const aar_problem *p, int k) { if (!p->opt_f) return -1; return 6LL * (p->nrc + p->nrm) + 6LL * k; }

int allreduce(aar_problem *p, double *buf, size_t n, ncclRedOp_t op) {
    if (!p->comm) return AAR_OK;
    ncclResult_t r = g_nccl.AllReduce(buf, buf, n, ncclFloat64, op, p->comm, p->stream);
    if (r != ncclSuccess) { set_err("ncclAllReduce: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "error"); return AAR_ERR_COMM; }
    return AAR_OK;
}

// residual sum of squares at dz into d_red3[0] (must be zeroed by the caller); optional residual vector.
// unweighted: without the Huber weights whatever the handle's setting (aar_error_report)
int residual(aar_problem *p, const double *dz, float huber_delta, double *d_r_out, bool unweighted = false) {
    DevProblem dq = p->dp;
    if (unweighted) { dq.huber = 0; dq.st_dev = nullptr; }
    LAUNCH(p, k_expand_trial, cdiv((long long)p->C + p->M + p->dp.F, 128), 128, 0, p->dp, dz);
    if (p->lens) {
        if (p->opt_i) LAUNCH(p, k_expand_lens, cdiv(9LL * p->C, 64), 64, 0, p->dp, dz, p->d_lens_tr.p);
        if (p->dp.N > 0)
            LAUNCH(p, k_residual_lens, cdiv(p->dp.N, 256), 256, 0, dq, p->opt_i ? p->d_lens_tr.p : p->d_lens.p, p->d_cam_tr.p, p->d_mk_tr.p, p->d_fr_tr.p, huber_delta,
                   d_r_out, p->d_red3.p);
        return AAR_OK;
    }
    if (p->opt_i) LAUNCH(p, k_expand_intr, cdiv(p->C, 64), 64, 0, p->dp, dz, p->d_intr_tr.p);
    if (p->dp.N > 0 && p->analytic)
        LAUNCH(p, k_residual_an, cdiv(p->dp.N, 256), 256, 0, dq, p->d_cam_tr.p, POSE_STRIDE, p->d_mk_tr.p, POSE_STRIDE, p->d_fr_tr.p, POSE_STRIDE, huber_delta, d_r_out, p->d_red3.p);
    else if (p->dp.N > 0)
        LAUNCH(p, k_residual, cdiv(p->dp.N, 256), 256, 0, dq, p->d_cam_tr.p, POSE_STRIDE, p->d_mk_tr.p, POSE_STRIDE, p->d_fr_tr.p, POSE_STRIDE, huber_delta, d_r_out, p->d_red3.p);
    return AAR_OK;
}

// Soft priors (aar_prior.cuh): rank 0 alone adds the terms of the camera and marker blocks, every rank those of its frames, so the
// all-reduces of the reduced system and of the cost count each once.  One thread per (entity, component) in CTAs of 256.
int prior_blocks(const aar_problem *p) { return p->rank == 0 ? p->nrc + p->nrm : 0; }
unsigned prior_grid(const aar_problem *p) { return cdiv(6LL * (prior_blocks(p) + p->dp.F), 256); }

// J^T J += diag(w), J^T r += w (z - zbar) at d_z into Hrr / gr / Hf; nothing without priors
void prior_add(aar_problem *p) {
    if (!p->has_prior || !prior_grid(p)) return;
    LAUNCH(p, k_prior_add, prior_grid(p), 256, 0, prior_blocks(p), p->d_blk_prior.p, p->d_blk_has_prior.p, p->dp.F, p->d_frame_prior.p,
           p->d_frame_has_prior.p, p->dp.col_frame0, p->n_r, p->d_z.p, p->d_Hrr.p, p->d_gr.p, p->d_Hf.p);
}

// Relative-pose priors (aar_pair_prior.cuh): pairs of cameras or markers only, so rank 0 alone adds them, like the camera and marker
// priors; the all-reduces count them once.
int pair_count(const aar_problem *p) { return p->rank == 0 ? p->n_pair : 0; }

// J^T J and J^T r of the pair rows at d_z into Hrr / gr; nothing without pairs
void pair_prior_add(aar_problem *p) {
    if (!pair_count(p)) return;
    LAUNCH(p, k_pair_prior_add, cdiv(pair_count(p), PP_WARPS), PP_WARPS * 32, 0, pair_count(p), p->d_pair_prior.p, p->n_r, p->d_z.p, p->d_Hrr.p, p->d_gr.p);
}

// the cost the solver compares at dz into d_red3[0] (zeroed by the caller): the reprojection sum of residual(), then the priors'
// sum w (z - zbar)^2 and the pair rows' squared sum.  The reprojection hooks (aar_eval_residual, aar_error_report) call residual() alone.
int solver_cost(aar_problem *p, const double *dz, float huber_delta) {
    if (int rc = residual(p, dz, huber_delta, nullptr)) return rc;
    if (p->has_prior && prior_grid(p))
        LAUNCH(p, k_prior_cost, prior_grid(p), 256, 0, prior_blocks(p), p->d_blk_prior.p, p->d_blk_has_prior.p, p->dp.F, p->d_frame_prior.p,
               p->d_frame_has_prior.p, p->dp.col_frame0, dz, p->d_red3.p);
    if (pair_count(p)) LAUNCH(p, k_pair_prior_cost, cdiv(pair_count(p), 256), 256, 0, pair_count(p), p->d_pair_prior.p, dz, p->d_red3.p);
    return AAR_OK;
}

void prof_mark(aar_problem *p, int i) { if (p->profiling) cudaEventRecord(p->ev[i], p->stream); }

// Dynamic shared-memory caps, set once per device for every kernel launched with more than 48 KB.  A function attribute holds for
// the whole process on a device: a cap sized for one handle would make the larger launches of another, earlier handle fail.  So
// every cap is the most the device allows next to the kernel's static shared memory.  The cap reserves nothing: occupancy follows
// the size a launch asks for.  *cluster_ok: the cluster Cholesky may run on this device.
template <typename K> cudaError_t cap_dynamic_smem(K *kernel, size_t smem_optin) {
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, kernel);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem_optin - a.sharedSizeBytes));
}
int set_smem_caps(aar_problem *p, bool *cluster_ok) {
    static std::mutex mu;
    static std::map<int, bool> done;          // device -> the cluster kernel's attributes were accepted
    std::lock_guard<std::mutex> lock(mu);
    auto it = done.find(p->device);
    if (it == done.end()) {
        const size_t o = p->smem_optin;
        CU(cap_dynamic_smem(k_jac_project<float>, o)); CU(cap_dynamic_smem(k_jac_project<double>, o));
        CU(cap_dynamic_smem(k_asm_pairs<float>, o)); CU(cap_dynamic_smem(k_asm_pairs<double>, o));
        CU(cap_dynamic_smem(k_asm_mruns<float>, o)); CU(cap_dynamic_smem(k_asm_mruns<double>, o));
        CU(cap_dynamic_smem(k_schur_prepare, o)); CU(cap_dynamic_smem(k_schur_syrk, o));
        CU(cap_dynamic_smem(k_report_obs, o)); CU(cap_dynamic_smem(k_sel_hist, o)); CU(cap_dynamic_smem(k_track_cta, o));
        // cluster Cholesky: up to 16 CTAs per cluster (non-portable size)
        const bool ok = cap_dynamic_smem(k_reduced_solve_cluster2, o) == cudaSuccess &&
                        cudaFuncSetAttribute(k_reduced_solve_cluster2, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess;
        if (!ok) cudaGetLastError();
        it = done.emplace(p->device, ok).first;
    }
    *cluster_ok = it->second;
    return AAR_OK;
}

// Launches the Jacobian kernels: k_jac_project (numerators + residual at z, one row per observation) and the tensor-core assembly
// k_asm_pairs + k_asm_mruns (aar_assemble.cuh).
template <typename JT>
int launch_jacobian(aar_problem *p, float huber_eval, JT *Jn) {
    const size_t tab_bytes = (size_t)((p->M * MK_TAB_S + 1) & ~1) * sizeof(double);
    const int tabs_smem = tab_bytes <= 48 * 1024;          // marker tables of the whole rig next to the per-warp pair buffers
    const size_t smem1 = (tabs_smem ? tab_bytes : 0) + PROJ_PAIR_SMEM_BYTES;
    const long long N = p->dp.N;
    // the staged rows hold central-difference numerators (scaled by 1 / (2 delta) once per sum) or, in the analytic variant, derivatives
    const double s1 = p->analytic ? 1.0 : 1.0 / (2 * p->J_delta), s2 = s1 * s1;
    const int grid1 = (int)std::max<long long>(1, std::min<long long>((long long)AAR_PROJ_MINBLOCKS * p->num_sms, (N + PROJ_THREADS - 1) / PROJ_THREADS));
    prof_mark(p, 7);
    auto k1 = k_jac_project<JT>; auto k2 = k_asm_pairs<JT>; auto k3 = k_asm_mruns<JT>;
    AsmPlan pl; pl.pair_info = p->d_pair_info.p; pl.pair_cam = p->d_pair_cam.p; pl.npairs = p->npairs; pl.mrun_info = p->d_mrun_info.p; pl.perm_fm = p->d_perm_fm.p;
    pl.nmruns = p->nmruns; pl.nperm = (int)p->d_perm_fm.n;
    pl.s1 = s1; pl.s2 = s2;
    // dynamic shared memory (aar_assemble.cuh): [camera / marker accumulators] | mbarriers | per-warp rings
    pl.ring_pairs = sizeof(JT) == 4 ? 3 : 2;      // 3 CTAs of 8 warps per SM with float staging
    const size_t ring2 = ASM_BAR_BYTES + (size_t)ASM_WARPS * pl.ring_pairs * asm_stage_bytes<JT>(JROW), ring3 = ASM_BAR_BYTES + asm_ring_bytes<JT>(ASM_MROW);
    pl.smem_acc = std::max(asm_acc_bytes(p->nrc) + ring2, asm_acc_bytes(p->nrm) + ring3) <= p->smem_optin;
    const size_t smem2 = ring2 + (pl.smem_acc ? asm_acc_bytes(p->nrc) : 0), smem3 = ring3 + (pl.smem_acc ? asm_acc_bytes(p->nrm) : 0);
    // camera x marker blocks: ASM_CM_REPLICAS copies of a [nrc][nrm][36] table (up to 256 MB; larger rigs add straight into the reduced matrix)
    const size_t cm_n = (size_t)p->nrc * p->nrm * 36;
    const bool use_rep = p->opt_c && p->opt_m && cm_n > 0 && cm_n * ASM_CM_REPLICAS * sizeof(double) <= (256u << 20);
    p->last_smem_acc = pl.smem_acc; p->last_cm_rep = use_rep;
    if (use_rep) {
        if (p->d_cm_rep.n < cm_n * ASM_CM_REPLICAS) CU(p->d_cm_rep.alloc(cm_n * ASM_CM_REPLICAS));
        CU(cudaMemsetAsync(p->d_cm_rep.p, 0, cm_n * ASM_CM_REPLICAS * sizeof(double), p->stream));
    }
    if (p->lens) {
        if constexpr (std::is_same<JT, double>::value) LAUNCH(p, k_jac_lens, cdiv(N, 128), 128, 0, p->dp, p->d_lens.p, huber_eval, Jn, p->d_Rv.p);
        else { set_err("the analytic variant stages its rows in double"); return AAR_ERR_INVALID; }
    } else if (p->analytic) {
        if constexpr (std::is_same<JT, double>::value) LAUNCH(p, k_jac_analytic, cdiv(N, 128), 128, 0, p->dp, huber_eval, Jn, p->d_Rv.p);
        else { set_err("the analytic variant stages its rows in double"); return AAR_ERR_INVALID; }
    } else
        LAUNCH(p, k1, grid1, PROJ_THREADS, smem1, p->dp, huber_eval, Jn, p->d_Rv.p, tabs_smem, p->d_flag.p, 0LL, N);
    prof_mark(p, 9);
    // every warp takes an equal share of the row stream: at least ~64 rows per warp, at most the resident CTAs of the device
    const long long want = std::max<long long>(1, (N + 64LL * ASM_WARPS - 1) / (64LL * ASM_WARPS));
    if (p->npairs > 0) {
        int per_sm = 1; CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k2, ASM_THREADS, smem2));
        const int grid2 = (int)std::min<long long>((long long)std::max(per_sm, 1) * p->num_sms, want);
        LAUNCH(p, k2, grid2, ASM_THREADS, smem2, p->dp, pl, Jn, p->huber ? p->d_Rv.p : nullptr, p->d_Hf.p, p->d_W.p, p->d_Hrr.p, p->d_gr.p, use_rep ? p->d_cm_rep.p : nullptr);
        if (use_rep) LAUNCH(p, k_cm_reduce, cdiv((long long)cm_n, 256), 256, 0, p->nrc, p->nrm, p->n_r, s2, p->d_cm_rep.p, p->d_Hrr.p);
    }
    prof_mark(p, 12);
    if (p->nmruns > 0) {
        int per_sm = 1; CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k3, ASM_THREADS, smem3));
        const int grid3 = (int)std::min<long long>((long long)std::max(per_sm, 1) * p->num_sms, want);
        LAUNCH(p, k3, grid3, ASM_THREADS, smem3, p->dp, pl, Jn, p->huber ? p->d_Rv.p : nullptr, p->d_W.p, p->d_Hrr.p, p->d_gr.p);
    }
    if (p->lens && p->opt_i && p->npairs > 0) {   // the nine lens columns (aar_lens.cuh): one warp per (frame, camera) pair
        if constexpr (std::is_same<JT, double>::value)
            LAUNCH(p, k_intr_assemble_lens, cdiv(p->npairs, LENS_WARPS), 32 * LENS_WARPS, 0, p->dp, p->d_lens.p, p->d_pair_info.p, p->d_pair_cam.p, p->d_pair_slot_i.p, Jn,
                   p->huber ? p->d_Rv.p : nullptr, p->d_W.p, p->d_Hrr.p, p->d_gr.p);
    } else if (p->opt_i && p->npairs > 0) {   // intrinsics columns (aar_intrinsics.cuh): one warp per (frame, camera) pair, from the same staged rows
        auto k4 = k_intr_assemble<JT>;
        LAUNCH(p, k4, cdiv((long long)p->npairs * 32, 128), 128, 0, p->dp, p->d_pair_info.p, p->d_pair_cam.p, p->d_pair_slot_i.p, Jn, p->huber ? p->d_Rv.p : nullptr, s1, s2,
               p->d_W.p, p->d_Hrr.p, p->d_gr.p);
    }
    prof_mark(p, 8);
    return AAR_OK;
}

// the columns of fixed entities become explicit zeros of J: their rows / columns of J^T J and entries of J^T r (aar_fixed.cuh)
void hold_fixed(aar_problem *p) {
    if (!p->has_fixed) return;
    // a warp per 32 W slots, a thread per entry of Hrr / gr / Hf; at most 8 CTAs of 256 threads per SM, grid-stride beyond
    const long long work = std::max<long long>(p->nslots, (long long)p->n_r * p->n_r + p->n_r + (long long)p->dp.F * HF_STRIDE);
    const unsigned grid = (unsigned)std::max<long long>(1, std::min<long long>(cdiv(work, 256), 8LL * p->num_sms));
    LAUNCH(p, k_hold_fixed, grid, 256, 0, p->n_r, p->d_blk_fixed.p, p->dp.F, p->d_frame_fixed.p, p->nslots, p->d_slot_block.p, p->d_slot_frame.p,
           p->d_Hrr.p, p->d_gr.p, p->d_Hf.p, p->d_W.p);
}

// J^T J blocks and J^T r at d_z (sparselevmarq.h:353-367) into Hf / W / Hrr / gr.  *rows64: the staged rows of this evaluation
// are d_Jn64 (FP64 staging), not d_Jn32.
int jacobian_accumulate(aar_problem *p, float huber_eval, bool defer_check = false, bool *rows64 = nullptr) {
    const long long jobs = (long long)p->C * NVAR_CAM + (long long)p->M * NVAR_RT + (long long)p->dp.F * NVAR_RT;
    LAUNCH(p, k_expand_jac, cdiv(jobs, 128), 128, 0, p->dp, p->d_z.p, p->d_flag.p);
    if (p->lens) { if (p->opt_i) LAUNCH(p, k_expand_lens, cdiv(9LL * p->C, 64), 64, 0, p->dp, p->d_z.p, p->d_lens.p); }
    else if (p->opt_i) LAUNCH(p, k_expand_intr, cdiv(p->C, 64), 64, 0, p->dp, p->d_z.p, p->d_intr.p);
    if (p->analytic) LAUNCH(p, k_expand_analytic, cdiv((long long)p->C + p->M + p->dp.F, 128), 128, 0, p->dp, p->d_z.p);
    else if (p->npairs > 0) LAUNCH(p, k_pair_tab, std::max(1, std::min(p->npairs, 10 * p->num_sms)), PAIR_TAB, 0, p->dp);      // 10 CTAs of 192 threads per SM: one full wave
    const size_t N = (size_t)p->dp.N;
    for (int attempt = 0; attempt < 2; attempt++) {
        const bool exact = p->force_exact_staging || attempt == 1 || p->exact_next || p->analytic;      // the analytic variant has no float32 staging
        if (rows64) *rows64 = exact;
        if (p->d_Hrr.n) CU(cudaMemsetAsync(p->d_Hrr.p, 0, p->d_Hrr.n * sizeof(double), p->stream));
        if (p->d_gr.n) CU(cudaMemsetAsync(p->d_gr.p, 0, p->d_gr.n * sizeof(double), p->stream));
        if (p->d_Hf.n) CU(cudaMemsetAsync(p->d_Hf.p, 0, p->d_Hf.n * sizeof(double), p->stream));
        if (N == 0) return AAR_OK;
        const size_t Np = (N + 31) / 32 * 32;      // rounded up to a multiple of 32 observations
        if (p->d_Rv.n < 4 * Np) CU(p->d_Rv.alloc(4 * Np));          // Huber weights [N][4]
        int rc;
        if (exact) { if (p->d_Jn64.n < JROW * Np) CU(p->d_Jn64.alloc(JROW * Np)); rc = launch_jacobian<double>(p, huber_eval, p->d_Jn64.p); }
        else { if (p->d_Jn32.n < JROW * Np) CU(p->d_Jn32.alloc(JROW * Np)); rc = launch_jacobian<float>(p, huber_eval, p->d_Jn32.p); }
        if (rc) return rc;
        if (exact) { p->exact_next = false; break; }
        // LM loops: k_lm_begin_iter looks at the flag on the device and leaves the iteration undecided (no synchronisation of its own)
        if (defer_check) break;
        // the float32 staging of the numerators is exact unless the kernel says otherwise (never seen on real data)
        CU(cudaMemcpyAsync(p->h_flags, p->d_flag.p, 4 * sizeof(int), cudaMemcpyDeviceToHost, p->stream));
        CU(cudaStreamSynchronize(p->stream));
        if (!p->h_flags[1]) break;
        p->exact_reruns++;
        CU(cudaMemsetAsync(p->d_flag.p + 1, 0, sizeof(int), p->stream));
    }
    prior_add(p);
    pair_prior_add(p);
    hold_fixed(p);      // after the priors: a held entity's columns are zero in the whole augmented Jacobian
    return AAR_OK;
}

__global__ void k_prepare_reduced(int n_r, const double *__restrict__ Hrr, const double *__restrict__ gr, double *__restrict__ red) {
    // red = [S (n_r*n_r) | b (n_r) | Br (n_r)]
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nn = (long long)n_r * n_r;
    if (e < nn) red[e] = Hrr[e];
    else if (e < nn + n_r) { double v = -gr[e - nn]; red[e] = v; red[e + n_r] = v; }
}

// Schur elimination of the frame blocks of this rank into S (must hold Hrr) and b (must hold -gr)
int schur_eliminate(aar_problem *p, double *S, double *b) {
    const int n_r = p->n_r, nb = p->nrc + p->nrm + p->nri, F = p->dp.F;
    if (!p->opt_f || F <= 0) return AAR_OK;
    LAUNCH(p, k_frame_chol, cdiv(F, 128), 128, 0, p->dp, p->d_st.p, p->d_Hf.p, p->d_fc.p, p->d_flag.p);      // also feeds k_backsub
    if (n_r > 0 && p->nslots > 0) {
        const int g1 = (int)std::max<long long>(1, std::min<long long>(4LL * p->num_sms, (p->nslots + 255) / 256));
        LAUNCH(p, k_schur_prepare, g1, 256, 8 * SP_TILE_BYTES + (size_t)n_r * sizeof(double), p->dp, p->nslots, p->d_slot_frame.p, p->d_fc.p, p->d_W.p, p->d_E.p, b);
        const int tiles_side = (nb + SY_TB - 1) / SY_TB, ntiles = tiles_side * (tiles_side + 1) / 2;
        // two CTAs per SM, at most two full waves (no tail wave), at least a few pipeline stages per CTA
        const int nchunks = std::max(1, std::min((2 * AAR_SY_MINBLOCKS * p->num_sms) / ntiles, (F + 4 * SY_FB - 1) / (4 * SY_FB)));
        prof_mark(p, 10);
        LAUNCH(p, k_schur_syrk, ntiles * nchunks, SY_THREADS, SY_SMEM, p->dp, nb, tiles_side, nchunks, p->d_frame_block_slot.p, p->d_E.p, S);
        prof_mark(p, 11);
    }
    return AAR_OK;
}

// one try of the do-while of SparseLevMarq::step (sparselevmarq.h:384-419) up to (not including) the decision
int build_and_solve_reduced(aar_problem *p) {
    const int n_r = p->n_r;
    double *S = p->d_red.p, *b = S + (size_t)n_r * n_r;     // [S | b | Br]: Br = -gr is kept for the gain denominator
    if (n_r > 0) LAUNCH(p, k_prepare_reduced, cdiv((long long)n_r * n_r + n_r, 256), 256, 0, n_r, p->d_Hrr.p, p->d_gr.p, S);
    { int rc = schur_eliminate(p, S, b); if (rc) return rc; }
    if (n_r > 0) {
        { int rc = allreduce(p, S, (size_t)n_r * n_r + 2 * n_r, ncclSum); if (rc) return rc; }
        const int nblk = (n_r + CH_NB - 1) / CH_NB;
        bool done = false;
        if (nblk <= 16 && p->use_cluster_solve) {
            // one thread-block cluster, the factor lives in distributed shared memory (aar_dense.cuh)
            const size_t smem = cluster2_smem_bytes(nblk);
            cudaLaunchConfig_t cfg = {}; cfg.gridDim = dim3(nblk); cfg.blockDim = dim3(CH_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = p->stream;
            cudaLaunchAttribute at[1]; at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = nblk; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            cfg.attrs = at; cfg.numAttrs = 1;
            const double *bc = b; const LmState *stp = p->d_st.p;
            cudaError_t e = cudaLaunchKernelEx(&cfg, k_reduced_solve_cluster2, n_r, S, bc, p->d_dr.p, stp, p->d_flag.p, p->d_xinv.p);
            if (e == cudaSuccess) { done = true; p->launches++; }
            else { cudaGetLastError(); p->use_cluster_solve = false; }      // e.g. the cluster cannot be scheduled: fall back for good
        }
        if (!done) {   // cooperative launch: one CTA per block row of 32 (all co-resident: n_r / 32 <= number of SMs)
            int n = n_r; double *xs = p->d_dr.p; const LmState *stp = p->d_st.p; int *fl = p->d_flag.p; const double *bb = b;
            double *xinv = p->d_xinv.p;
            void *args[] = {&n, &S, &bb, &xs, &stp, &fl, &xinv};
            const int gridc = std::max(1, std::min(nblk, p->num_sms));
            CU(cudaLaunchCooperativeKernel((const void *)k_reduced_solve, dim3(gridc), dim3(CH_THREADS), args, 0, p->stream));
            p->launches++;
        }
        p->last_cluster_solve = done;
        LAUNCH(p, k_apply_reduced, cdiv(n_r, 128), 128, 0, n_r, p->d_z.p, p->d_dr.p, p->d_zt.p);
    }
    return AAR_OK;
}

int fetch_state(aar_problem *p) {
    CU(cudaMemcpyAsync(p->h_st, p->d_st.p, sizeof(LmState), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaMemcpyAsync(p->h_flags, p->d_flag.p, 4 * sizeof(int), cudaMemcpyDeviceToHost, p->stream));   // rides on the same synchronisation
    CU(cudaStreamSynchronize(p->stream));
    return AAR_OK;
}
int push_state(aar_problem *p) {
    CU(cudaMemcpyAsync(p->d_st.p, p->h_st, sizeof(LmState), cudaMemcpyHostToDevice, p->stream));
    return AAR_OK;
}

// ---- the two halves of an LM iteration, launched by the host-driven loop and captured into the graph-resident one (`graph`).
// The residual and Jacobian kernels take hubberDelta from the device state (dp.st_dev); the Huber arguments below only reach
// the analytic variant, which runs on the host-driven loop, where h_st is current.

// J^T J blocks and J^T r at z (sparselevmarq.h:353-367), then k_lm_begin_iter.  The first iteration of a solve (never inside
// the graph) computes mu0 = tau * max diag(JtJ) (sparselevmarq.h:369-377).
int lm_jacobian_phase(aar_problem *p, bool graph) {
    const int n_r = p->n_r;
    int rc;
    prof_mark(p, 0);
    if ((rc = jacobian_accumulate(p, p->h_st->huber_eval, true))) return rc;
    prof_mark(p, 1);
    const double *diag = p->d_Hrr.p; int ld = n_r; double frames_maxdiag = 0.0;
    if (p->h_st->mu < 0) {
        p->h_st->maxdiag = -1e300; push_state(p);
        if (p->opt_f && p->dp.F > 0) LAUNCH(p, k_maxdiag_frames, cdiv(p->dp.F, 128), 128, 0, p->dp, p->d_Hf.p, p->d_st.p);
        if (p->comm) {
            // global diagonal of Hrr (sum) into d_tmp and global frame maximum
            double *tmp = p->d_tmp.p;
            if (n_r) CU(cudaMemcpy2DAsync(tmp, sizeof(double), p->d_Hrr.p, (size_t)(n_r + 1) * sizeof(double), sizeof(double), (size_t)n_r, cudaMemcpyDeviceToDevice, p->stream));
            if ((rc = allreduce(p, tmp, (size_t)n_r, ncclSum))) return rc;
            if ((rc = allreduce(p, &p->d_st.p->maxdiag, 1, ncclMax))) return rc;
            diag = tmp; ld = 0;
        }
        if ((rc = fetch_state(p))) return rc;
        frames_maxdiag = p->h_st->maxdiag;
    }
    LAUNCH(p, k_lm_begin_iter, 1, 1, 0, p->d_st.p, n_r, diag, ld, p->params.tau, frames_maxdiag, p->d_flag.p, (int)graph, p->lm_inner);
    return AAR_OK;
}

// one try of the do-while of SparseLevMarq::step (sparselevmarq.h:384-419): damped solve, back substitution, cost at the trial
// point, the decision and the commit of an accepted trial point
int lm_try(aar_problem *p, bool graph) {
    const int n_r = p->n_r;
    const double *Br = p->d_red.p + (size_t)n_r * n_r + n_r;
    int rc;
    CU(cudaMemsetAsync(p->d_red3.p, 0, 8 * sizeof(double), p->stream));
    prof_mark(p, 2);
    if ((rc = build_and_solve_reduced(p))) return rc;
    prof_mark(p, 3);
    if (p->opt_f && p->dp.F > 0)
        LAUNCH(p, k_backsub, std::max(1, std::min(4 * p->num_sms, (int)cdiv(p->dp.F, BS_WARPS))), BS_WARPS * 32, 0, p->dp, p->d_fc.p, p->d_Hf.p, p->d_W.p, p->d_dr.p, p->d_z.p, p->d_zt.p, p->d_red3.p);
    prof_mark(p, 4);
    if ((rc = solver_cost(p, p->d_zt.p, p->h_st->huber_delta))) return rc;
    prof_mark(p, 5);
    if ((rc = allreduce(p, p->d_red3.p, 3, ncclSum))) return rc;
    LAUNCH(p, k_lm_decide, 1, 1, 0, p->d_st.p, p->d_red3.p, n_r, p->d_dr.p, Br, p->d_flag.p, (int)graph, p->lm_inner);
    LAUNCH(p, k_lm_commit, std::max(1, std::min(2 * p->num_sms, (int)cdiv(p->n_vars, 256))), 256, 0, p->d_st.p, p->n_vars, p->d_zt.p, p->d_z.p);
    return AAR_OK;
}

} // namespace

// ================================================================================ C ABI =====
extern "C" {

const char *aar_last_error(void) { return g_err.c_str(); }
/* other translation units of the library (aar_init.cu) report through the same thread-local message */
void aar_internal_set_error(const char *msg) { g_err = msg ? msg : ""; }

void aar_lm_default_params(aar_lm_params *q) {
    q->max_iters = 10000; q->min_error = 1e-5; q->min_step_error_diff = 0; q->min_average_step_error_diff = 1e-4;
    q->tau = 1; q->der_epsilon = 1e-3; q->ignore_stop_rules = 0; q->verbose = 0;
}

static int create_impl(const aar_problem_desc *d, aar_problem **out, bool host_only) {
    // AAR_CREATE_TIMING=1: wall-clock of the stages of this function to stderr (development aid)
    const bool ctime = getenv("AAR_CREATE_TIMING") != nullptr; auto ct0 = std::chrono::steady_clock::now();
    auto cmark = [&](const char *what) { if (!ctime) return; auto t = std::chrono::steady_clock::now(); fprintf(stderr, "aar_problem_create: %-28s %.3f s\n", what, std::chrono::duration<double>(t - ct0).count()); ct0 = t; };
    if (!d || !out) { set_err("null argument"); return AAR_ERR_INVALID; }
    *out = nullptr;
    if (d->num_cams < 1 || d->num_markers < 1 || d->num_frames < 0 || d->num_cams > 4095 || d->num_markers > 500000) { set_err("bad counts"); return AAR_ERR_INVALID; }
    aar_problem *p = new aar_problem();
    std::unique_ptr<aar_problem, void (*)(aar_problem *)> guard(p, aar_problem_destroy);
    p->C = d->num_cams; p->M = d->num_markers; p->F = d->num_frames;
    p->cam_ids.assign(d->cam_ids, d->cam_ids + p->C);
    p->marker_ids.assign(d->marker_ids, d->marker_ids + p->M);
    p->frame_ids.assign(d->frame_ids, d->frame_ids + p->F);
    if (!strictly_ascending(p->cam_ids) || !strictly_ascending(p->marker_ids) || !strictly_ascending(p->frame_ids)) { set_err("ids must be strictly ascending"); return AAR_ERR_INVALID; }
    p->root_cam_id = d->root_cam; p->root_marker_id = d->root_marker;
    p->root_cam = rank_of(p->cam_ids, d->root_cam); p->root_marker = rank_of(p->marker_ids, d->root_marker);
    if (p->root_cam < 0 || p->root_marker < 0) { set_err("root camera/marker id not among the ids"); return AAR_ERR_INVALID; }
    p->marker_size = d->marker_size;
    p->cam_T.assign(d->cam_T, d->cam_T + 16 * (size_t)p->C);
    p->marker_T.assign(d->marker_T, d->marker_T + 16 * (size_t)p->M);
    p->frame_T.assign(d->frame_T, d->frame_T + 16 * (size_t)p->F);
    p->cam_K.assign(d->cam_K, d->cam_K + 9 * (size_t)p->C);
    p->cam_dist.assign(d->cam_dist, d->cam_dist + 5 * (size_t)p->C);
    for (int c = 0; c < p->C; c++) {
        const double *K = &p->cam_K[9 * (size_t)c];
        if (K[1] != 0 || K[3] != 0 || K[6] != 0 || K[7] != 0 || K[8] != 1) { set_err("camera %d: only [fx 0 cx; 0 fy cy; 0 0 1] camera matrices are supported", p->cam_ids[c]); return AAR_ERR_UNSUPPORTED; }
    }
    auto rigid_last_row = [](const std::vector<double> &T) { for (size_t i = 0; i * 16 < T.size(); i++) { const double *r = &T[i * 16 + 12]; if (r[0] != 0 || r[1] != 0 || r[2] != 0 || r[3] != 1) return false; } return true; };
    if (!rigid_last_row(p->cam_T) || !rigid_last_row(p->marker_T) || !rigid_last_row(p->frame_T)) { set_err("transforms must have last row [0 0 0 1]"); return AAR_ERR_UNSUPPORTED; }
    p->opt_c = d->optimize_cam_poses; p->opt_m = d->optimize_marker_poses; p->opt_f = d->optimize_object_poses; p->huber = d->with_huber;
    p->J_delta = d->J_delta > 0 ? d->J_delta : 1e-3;
    p->device = d->device; p->rank = d->world_size > 1 ? d->rank : 0; p->world = d->world_size > 1 ? d->world_size : 1;
    if (p->rank < 0 || p->rank >= p->world) { set_err("bad rank"); return AAR_ERR_INVALID; }
    g_ranks_on_host = std::max(1, d->world_size);
    p->opt_i = d->optimize_cam_intrinsics != 0;
    p->analytic = d->analytic_jacobian != 0;
    if (d->lens_model > 1) { set_err("lens_model %d: only 0 (undistorted corners, pinhole) and 1 (OpenCV's five-coefficient model on raw corners) exist", (int)d->lens_model); return AAR_ERR_UNSUPPORTED; }
    p->lens = d->lens_model == 1;
    if (p->lens && !p->analytic) { set_err("lens_model 1 needs analytic_jacobian = 1: the central-difference path is the reference's pinhole residual"); return AAR_ERR_UNSUPPORTED; }
    if (p->lens && d->corners_undistorted) { set_err("lens_model 1 needs the raw corners: corners_undistorted = 1 (a .solution file) holds none"); return AAR_ERR_UNSUPPORTED; }
    if (p->analytic && p->opt_i && !p->lens) { set_err("analytic_jacobian with optimize_cam_intrinsics: the pinhole intrinsics block is built for the central-difference path only (lens_model 1 refines intrinsics in the analytic mode)"); return AAR_ERR_UNSUPPORTED; }
    p->nrc = p->opt_c ? p->C - 1 : 0; p->nrm = p->opt_m ? p->M - 1 : 0; p->nri = p->opt_i ? 2 * p->C : 0; p->n_r = 6 * (p->nrc + p->nrm + p->nri);
    p->n_vars = p->n_r + (p->opt_f ? 6LL * p->F : 0);
    p->n_vars_ext = 6LL * (p->nrc + p->nrm) + (p->opt_f ? 6LL * p->F : 0) + (p->opt_i ? 9LL * p->C : 0);

    // ---- fill_iteration_arrays (multicam_mapper.cpp:345-377): frame id ^, cam id ^, detection order;
    // detections of unknown cameras / markers are erased.  (Detections of a frame without an object pose make
    // the reference throw std::out_of_range in project_marker; they are dropped here.)
    // The host passes below run on all the cores the process may use (25.6 M detections at BASELINE cfg 4).
    const long long nd = d->num_detections;
    const IdMap fmap(p->frame_ids), cmap(p->cam_ids), mmap(p->marker_ids);
    std::vector<int> kf((size_t)nd), kc((size_t)nd), km((size_t)nd);
    cmark("copies, id maps");
    std::vector<long long> keep;
    {
        const int T = host_threads(nd);
        std::vector<long long> cnt((size_t)T + 1, 0);
        parallel_for(nd, T, [&](long long b0, long long b1, int t) {
            long long n = 0;
            for (long long i = b0; i < b1; i++) {
                const int fi = fmap(d->det_frame[i]), ci = cmap(d->det_cam[i]), mi = mmap(d->det_marker[i]);
                const bool ok = fi >= 0 && ci >= 0 && mi >= 0;
                kf[(size_t)i] = ok ? fi : -1; kc[(size_t)i] = ci; km[(size_t)i] = mi; n += ok;
            }
            cnt[(size_t)t + 1] = n;
        });
        for (int t = 0; t < T; t++) cnt[(size_t)t + 1] += cnt[(size_t)t];
        keep.resize((size_t)cnt[(size_t)T]);
        parallel_for(nd, T, [&](long long b0, long long b1, int t) {
            long long w = cnt[(size_t)t];
            for (long long i = b0; i < b1; i++) if (kf[(size_t)i] >= 0) keep[(size_t)w++] = i;
        });
    }
    auto before = [&](long long a, long long b) { return kf[(size_t)a] != kf[(size_t)b] ? kf[(size_t)a] < kf[(size_t)b] : kc[(size_t)a] < kc[(size_t)b]; };
    if (!std::is_sorted(keep.begin(), keep.end(), before)) // aruco.detections order is already (frame, cam)
        std::stable_sort(keep.begin(), keep.end(), before);
    p->N = (long long)keep.size();
    p->g_frame.resize((size_t)p->N); p->g_cam.resize((size_t)p->N); p->g_marker.resize((size_t)p->N); p->g_hasjac.assign((size_t)p->N, 1);
    parallel_for(p->N, host_threads(p->N), [&](long long b0, long long b1, int) {
        for (long long o = b0; o < b1; o++) { const long long i = keep[(size_t)o]; p->g_frame[(size_t)o] = kf[(size_t)i]; p->g_cam[(size_t)o] = kc[(size_t)i]; p->g_marker[(size_t)o] = km[(size_t)i]; }
    });
    { std::vector<int>().swap(kf); std::vector<int>().swap(kc); std::vector<int>().swap(km); }
    std::vector<long long> frame_ptr((size_t)p->F + 1, 0);
    for (long long o = 0; o < p->N; o++) frame_ptr[(size_t)p->g_frame[(size_t)o] + 1]++;
    for (int f = 0; f < p->F; f++) frame_ptr[(size_t)f + 1] += frame_ptr[(size_t)f];
    // a repeated (frame, cam, marker) overwrites the earlier entry of the inverted indices (:368-370):
    // only the LAST occurrence contributes Jacobian rows
    parallel_for(p->F, host_threads(p->N), [&](long long f0, long long f1, int) {
        std::vector<long long> stamp((size_t)p->M, -1), lastidx((size_t)p->M, 0);
        for (long long o = frame_ptr[(size_t)f0]; o < frame_ptr[(size_t)f1];) {
            long long e = o;
            while (e < frame_ptr[(size_t)f1] && p->g_frame[(size_t)e] == p->g_frame[(size_t)o] && p->g_cam[(size_t)e] == p->g_cam[(size_t)o]) e++;
            for (long long q = o; q < e; q++) {
                const size_t m = (size_t)p->g_marker[(size_t)q];
                if (stamp[m] == o) p->g_hasjac[(size_t)lastidx[m]] = 0;
                stamp[m] = o; lastidx[m] = q;
            }
            o = e;
        }
    });
    // ---- frame shard: contiguous frame ranges balanced by observation count (SURVEY 8e)
    auto boundary = [&](int r) -> int {
        if (r <= 0) return 0; if (r >= p->world) return p->F;
        long long target = p->N * r / p->world;
        int f = (int)(std::lower_bound(frame_ptr.begin(), frame_ptr.end(), target) - frame_ptr.begin());
        return std::min(f, p->F);
    };
    p->f_begin = boundary(p->rank); p->f_end = boundary(p->rank + 1);
    p->o_begin = frame_ptr[(size_t)p->f_begin]; p->o_end = frame_ptr[(size_t)p->f_end];
    const int Fl = p->f_end - p->f_begin; const long long Nl = p->o_end - p->o_begin;

    cmark("row map, shard");
    // ---- W slots: per local frame, the distinct active camera blocks seen (order of first appearance), then the
    // distinct active marker blocks; cs_cum / ms_cum are the running numbers of camera / marker slots.
    // Two passes over the local frames (count, prefix sum, fill), both parallel.
    if (Nl >= (1LL << 31) - 1) { set_err("more than 2^31 observations on one rank"); return AAR_ERR_UNSUPPORTED; }
    const int nblk_r = p->nrc + p->nrm + p->nri;
    std::vector<int> slot_ptr((size_t)Fl + 1, 0), cs_cum((size_t)Fl + 1, 0), ms_cum((size_t)Fl + 1, 0), is_cnt((size_t)Fl + 1, 0), slot_c((size_t)Nl, -1), slot_m((size_t)Nl, -1), slot_i((size_t)Nl, -1);
    const bool slots_c = p->opt_f && p->opt_c, slots_m = p->opt_f && p->opt_m, slots_i = p->opt_f && p->opt_i;   // intrinsics: pseudo-block A of every camera seen, root included
    const bool slots_ib = slots_i && p->lens;      // the lens model's block B has columns too: its slot follows A's
    const int Tf = host_threads(Nl);
    parallel_for(Fl, Tf, [&](long long f0, long long f1, int) {
        std::vector<long long> stamp((size_t)std::max(nblk_r, 1), -1);
        for (long long f = f0; f < f1; f++) {
            const long long o0 = frame_ptr[(size_t)(p->f_begin + f)], o1 = frame_ptr[(size_t)(p->f_begin + f) + 1];
            int ncs = 0, nms = 0, nis = 0;
            for (long long o = o0; o < o1; o++) {
                const int c = p->g_cam[(size_t)o], m = p->g_marker[(size_t)o];
                if (slots_c && c != p->root_cam) { const size_t bk = (size_t)(c - (c > p->root_cam ? 1 : 0)); if (stamp[bk] != f) { stamp[bk] = f; ncs++; } }
                if (slots_m && m != p->root_marker) { const size_t bk = (size_t)(p->nrc + m - (m > p->root_marker ? 1 : 0)); if (stamp[bk] != f) { stamp[bk] = f; nms++; } }
                if (slots_i) { const size_t bk = (size_t)(p->nrc + p->nrm + 2 * c); if (stamp[bk] != f) { stamp[bk] = f; nis += slots_ib ? 2 : 1; } }
            }
            cs_cum[(size_t)f + 1] = ncs; ms_cum[(size_t)f + 1] = nms; is_cnt[(size_t)f + 1] = nis;
        }
    });
    p->max_slots = 0; p->max_ms = 0; p->schur_fma = 0;
    for (int f = 0; f < Fl; f++) {
        const int ncs = cs_cum[(size_t)f + 1], nms = ms_cum[(size_t)f + 1], nis = is_cnt[(size_t)f + 1];
        slot_ptr[(size_t)f + 1] = slot_ptr[(size_t)f] + ncs + nms + nis;
        cs_cum[(size_t)f + 1] += cs_cum[(size_t)f]; ms_cum[(size_t)f + 1] += ms_cum[(size_t)f];
        p->max_slots = std::max(p->max_slots, ncs + nms + nis); p->max_ms = std::max(p->max_ms, nms);
        const long long nf = 6LL * (ncs + nms + nis); p->schur_fma += 6 * nf * (nf + 1) / 2;
    }
    p->nslots = (long long)slot_ptr[(size_t)Fl];
    std::vector<int> slot_block((size_t)p->nslots), slot_frame((size_t)p->nslots), frame_block_slot((size_t)std::max(Fl, 1) * std::max(nblk_r, 1));
    parallel_for(Fl, Tf, [&](long long f0, long long f1, int) {
        std::vector<int> seen((size_t)std::max(nblk_r, 1), -1);
        std::fill(frame_block_slot.begin() + (size_t)f0 * std::max(nblk_r, 1), frame_block_slot.begin() + (size_t)f1 * std::max(nblk_r, 1), -1);
        for (long long f = f0; f < f1; f++) {
            const long long o0 = frame_ptr[(size_t)(p->f_begin + f)], o1 = frame_ptr[(size_t)(p->f_begin + f) + 1];
            int next = slot_ptr[(size_t)f];
            const int first = next;
            if (slots_c)
                for (long long o = o0; o < o1; o++) {
                    const int c = p->g_cam[(size_t)o];
                    if (c == p->root_cam) continue;
                    const int bk = c - (c > p->root_cam ? 1 : 0);
                    if (seen[(size_t)bk] < first) { seen[(size_t)bk] = next; slot_block[(size_t)next++] = bk; }
                    slot_c[(size_t)(o - p->o_begin)] = seen[(size_t)bk];
                }
            if (slots_m)
                for (long long o = o0; o < o1; o++) {
                    const int m = p->g_marker[(size_t)o];
                    if (m == p->root_marker) continue;
                    const int bk = p->nrc + m - (m > p->root_marker ? 1 : 0);
                    if (seen[(size_t)bk] < first) { seen[(size_t)bk] = next; slot_block[(size_t)next++] = bk; }
                    slot_m[(size_t)(o - p->o_begin)] = seen[(size_t)bk];
                }
            if (slots_i)
                for (long long o = o0; o < o1; o++) {
                    const int bk = p->nrc + p->nrm + 2 * p->g_cam[(size_t)o];
                    if (seen[(size_t)bk] < first) {
                        seen[(size_t)bk] = next; slot_block[(size_t)next++] = bk;
                        if (slots_ib) { seen[(size_t)bk + 1] = next; slot_block[(size_t)next++] = bk + 1; }
                    }
                    slot_i[(size_t)(o - p->o_begin)] = seen[(size_t)bk];
                }
            for (int sl = first; sl < next; sl++) { slot_frame[(size_t)sl] = (int)f; frame_block_slot[(size_t)f * nblk_r + slot_block[(size_t)sl]] = sl; }
        }
    });

    if (host_only) { guard.release(); *out = p; return AAR_OK; }   // aar_shard_plan: row map and shard only
    // ---- device
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { set_err("no CUDA device: the B200 path has no CPU fallback"); return AAR_ERR_CUDA; }
    CU(cudaSetDevice(p->device));
    if (d->stream) p->stream = (cudaStream_t)d->stream; else { CU(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking)); p->own_stream = true; }
    for (auto &e : p->ev) CU(cudaEventCreate(&e));
    CU(cudaMallocHost((void **)&p->h_st, sizeof(LmState)));
    std::memset(p->h_st, 0, sizeof(LmState));
    p->h_st->huber_eval = 2.5f;      // the parity hooks evaluate with the Huber delta of the last accepted evaluation: 2.5 before any solve
    CU(cudaMallocHost((void **)&p->h_red3, 8 * sizeof(double)));
    CU(cudaMallocHost((void **)&p->h_flags, 4 * sizeof(int)));
    {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, p->device) == cudaSuccess && v > 0) p->num_sms = v;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, p->device) == cudaSuccess && v > 0) p->smem_optin = (size_t)v;
    }

    cmark("W slots, device set-up");
    std::vector<int> obs_f((size_t)Nl), obs_cm((size_t)Nl);
    std::vector<float4> raw_a((size_t)Nl), raw_b((size_t)Nl);
    parallel_for(Nl, host_threads(Nl), [&](long long b0, long long b1, int) {
        for (long long o = b0; o < b1; o++) {
            const long long g = p->o_begin + o, i = keep[(size_t)g];
            obs_f[(size_t)o] = p->g_frame[(size_t)g] - p->f_begin;
            obs_cm[(size_t)o] = p->g_cam[(size_t)g] | (p->g_marker[(size_t)g] << 12) | (p->g_hasjac[(size_t)g] ? 0 : (int)0x80000000u);
            const float *xy = d->det_xy + 8 * i;
            raw_a[(size_t)o] = make_float4(xy[0], xy[1], xy[2], xy[3]); raw_b[(size_t)o] = make_float4(xy[4], xy[5], xy[6], xy[7]);
        }
    });
    // (frame, camera) pairs: runs of consecutive observations in row order; every perturbation of inv(Tc) * To is
    // evaluated once per pair (k_pair_tab) instead of once per observation
    std::vector<int> obs_pair((size_t)Nl); std::vector<int2> pair_fc;
    for (long long o = 0; o < Nl; o++) {
        const int f = obs_f[(size_t)o], c = obs_cm[(size_t)o] & 0xfff;
        if (pair_fc.empty() || pair_fc.back().x != f || pair_fc.back().y != c) pair_fc.push_back(make_int2(f, c));
        obs_pair[(size_t)o] = (int)pair_fc.size() - 1;
    }
    p->npairs = (int)pair_fc.size();
    std::vector<double> intr(4 * (size_t)p->C), fixed_c(12 * (size_t)p->C), fixed_m(12 * (size_t)p->M), fixed_f(12 * (size_t)std::max(Fl, 1));
    for (int c = 0; c < p->C; c++) { const double *K = &p->cam_K[9 * (size_t)c]; intr[4 * (size_t)c] = K[0]; intr[4 * (size_t)c + 1] = K[2]; intr[4 * (size_t)c + 2] = K[4]; intr[4 * (size_t)c + 3] = K[5]; pose12_from_T16(&p->cam_T[16 * (size_t)c], &fixed_c[12 * (size_t)c]); }
    for (int m = 0; m < p->M; m++) pose12_from_T16(&p->marker_T[16 * (size_t)m], &fixed_m[12 * (size_t)m]);
    for (int f = 0; f < Fl; f++) pose12_from_T16(&p->frame_T[16 * (size_t)(p->f_begin + f)], &fixed_f[12 * (size_t)f]);

    cmark("observation arrays, pairs");
#define UP(buf, vec)                                                                                             \
    do { CU((buf).alloc((vec).size())); if ((vec).size()) CU(cudaMemcpyAsync((buf).p, (vec).data(), (vec).size() * sizeof((vec)[0]), cudaMemcpyHostToDevice, p->stream)); } while (0)
    UP(p->d_obs_f, obs_f); UP(p->d_obs_cm, obs_cm); UP(p->d_slot_c, slot_c); UP(p->d_slot_m, slot_m);
    UP(p->d_frame_slot_ptr, slot_ptr); UP(p->d_slot_block, slot_block); UP(p->d_frame_cs_cum, cs_cum);
    UP(p->d_slot_frame, slot_frame); UP(p->d_frame_block_slot, frame_block_slot);
    {
        std::vector<int> fop((size_t)Fl + 1); for (int f = 0; f <= Fl; f++) fop[(size_t)f] = (int)(frame_ptr[(size_t)(p->f_begin + f)] - p->o_begin); UP(p->d_frame_obs_ptr, fop);
        // visiting orders of the tensor-core assembly (aar_assemble.cuh): the (frame, camera) pairs with their row ranges, and the
        // rows of each frame by (marker, camera) cut into (frame, marker) runs.  Root-marker rows have no marker block: not listed.
        std::vector<int4> pair_info((size_t)p->npairs);
        for (long long o = 0; o < Nl; o++) {
            const int pr = obs_pair[(size_t)o];
            if (o == 0 || obs_pair[(size_t)o - 1] != pr) pair_info[(size_t)pr] = make_int4((int)o, 0, pair_fc[(size_t)pr].x, pair_fc[(size_t)pr].y);
            pair_info[(size_t)pr].y++;
        }
        {   // descriptors of k_asm_pairs: (first row, rows, frame, W slot) and the camera of every pair
            std::vector<int> pair_cam((size_t)p->npairs);
            for (int pr = 0; pr < p->npairs; pr++) { int4 &pi = pair_info[(size_t)pr]; pair_cam[(size_t)pr] = pi.w; pi.w = slot_c[(size_t)pi.x]; }
            std::vector<int> pair_slot_i((size_t)p->npairs, -1);
            for (int pr = 0; pr < p->npairs; pr++) pair_slot_i[(size_t)pr] = slot_i[(size_t)pair_info[(size_t)pr].x];
            UP(p->d_pair_info, pair_info); UP(p->d_pair_cam, pair_cam); UP(p->d_pair_slot_i, pair_slot_i);
        }
        std::vector<int> perm_fm; std::vector<int4> mrun_info;
        if (p->opt_m) {
            perm_fm.reserve((size_t)Nl); mrun_info.reserve((size_t)(ms_cum.empty() ? 0 : ms_cum.back()) + 16);
            std::vector<int> cnt((size_t)p->M + 1);
            for (int f = 0; f < Fl; f++) {
                const int o0 = fop[(size_t)f], o1 = fop[(size_t)f + 1];
                std::fill(cnt.begin(), cnt.end(), 0);
                for (int o = o0; o < o1; o++) cnt[(size_t)((obs_cm[(size_t)o] >> 12) & 0x7ffff) + 1]++;
                const int base = (int)perm_fm.size();
                int run = 0;
                for (int m = 0; m < p->M; m++) {            // counting sort by marker, stable: cameras ascend inside a run
                    const int n = cnt[(size_t)m + 1];
                    cnt[(size_t)m + 1] = (m == p->root_marker) ? -1 : base + run;
                    if (n > 0 && m != p->root_marker) { mrun_info.push_back(make_int4(base + run, n, -1, m - (m > p->root_marker ? 1 : 0))); run += n; }
                }
                perm_fm.resize((size_t)base + run);
                for (int o = o0; o < o1; o++) {
                    const int m = (obs_cm[(size_t)o] >> 12) & 0x7ffff;
                    if (m == p->root_marker) continue;
                    perm_fm[(size_t)cnt[(size_t)m + 1]++] = o;
                }
            }
            for (auto &r : mrun_info) r.z = slot_m[(size_t)perm_fm[(size_t)r.x]];
            if ((long long)mrun_info.size() >= (1LL << 31) - 1) { set_err("too many (frame, marker) runs on one rank"); return AAR_ERR_UNSUPPORTED; }
        }
        p->nmruns = (int)mrun_info.size();
        UP(p->d_perm_fm, perm_fm); UP(p->d_mrun_info, mrun_info);
    }

    UP(p->d_raw_a, raw_a); UP(p->d_raw_b, raw_b); UP(p->d_obs_pair, obs_pair); UP(p->d_pair_fc, pair_fc);
    CU(p->d_pair_tab.alloc((size_t)std::max(p->npairs, 1) * PAIR_TAB));
    UP(p->d_intr, intr); UP(p->d_intr_tr, intr); UP(p->d_K9, p->cam_K); UP(p->d_dist5, p->cam_dist);
    UP(p->d_cam_fixed, fixed_c); UP(p->d_mk_fixed, fixed_m); UP(p->d_fr_fixed, fixed_f);
#undef UP
    CU(p->d_und_a.alloc((size_t)Nl)); CU(p->d_und_b.alloc((size_t)Nl));
    CU(p->d_cam_tab.alloc((size_t)p->C * CAM_TAB)); CU(p->d_mk_tab.alloc((size_t)p->M * MK_TAB)); CU(p->d_fr_tab.alloc((size_t)std::max(Fl, 1) * FR_TAB));
    if (p->lens) {
        std::vector<double> lens(9 * (size_t)p->C);
        for (int c = 0; c < p->C; c++) {
            const double *K = &p->cam_K[9 * (size_t)c], *dd = &p->cam_dist[5 * (size_t)c]; double *l = &lens[9 * (size_t)c];
            l[0] = K[0]; l[1] = K[2]; l[2] = K[4]; l[3] = K[5]; for (int k = 0; k < 5; k++) l[4 + k] = dd[k];
        }
        CU(p->d_lens.alloc(lens.size())); CU(p->d_lens_tr.alloc(lens.size()));
        CU(cudaMemcpyAsync(p->d_lens.p, lens.data(), lens.size() * sizeof(double), cudaMemcpyHostToDevice, p->stream));
        CU(cudaMemcpyAsync(p->d_lens_tr.p, lens.data(), lens.size() * sizeof(double), cudaMemcpyHostToDevice, p->stream));
        CU(cudaStreamSynchronize(p->stream));     // `lens` leaves scope
    }
    if (p->analytic) { CU(p->d_cam_an.alloc((size_t)p->C * CAM_AN)); CU(p->d_mk_an.alloc((size_t)p->M * RT_AN)); CU(p->d_fr_an.alloc((size_t)std::max(Fl, 1) * RT_AN)); }
    CU(p->d_cam_tr.alloc((size_t)p->C * POSE_STRIDE)); CU(p->d_mk_tr.alloc((size_t)p->M * POSE_STRIDE)); CU(p->d_fr_tr.alloc((size_t)std::max(Fl, 1) * POSE_STRIDE));
    const size_t nz = (size_t)std::max<long long>(p->n_vars, 1);
    CU(p->d_z.alloc(nz)); CU(p->d_zt.alloc(nz)); CU(p->d_z0.alloc(nz));
    CU(p->d_fc.alloc((size_t)std::max(Fl, 1) * FC_STRIDE)); CU(p->d_E.alloc((size_t)std::max<long long>(p->nslots, 1) * 36));
    CU(p->d_Hf.alloc((size_t)std::max(Fl, 1) * HF_STRIDE)); CU(p->d_W.alloc((size_t)std::max<long long>(p->nslots, 1) * 36));
    CU(p->d_Hrr.alloc((size_t)std::max(p->n_r, 1) * std::max(p->n_r, 1))); CU(p->d_gr.alloc((size_t)std::max(p->n_r, 1)));
    CU(p->d_red.alloc((size_t)p->n_r * p->n_r + 2 * (size_t)p->n_r + 8)); CU(p->d_dr.alloc((size_t)std::max(p->n_r, 1)));
    CU(p->d_xinv.alloc((size_t)((p->n_r + CH_NB - 1) / CH_NB + 1) * CH_NB * CH_NB));
    CU(p->d_red3.alloc(8)); CU(p->d_tmp.alloc((size_t)std::max(p->n_r, 1) + 8)); CU(p->d_st.alloc(1)); CU(p->d_flag.alloc(4));
    CU(cudaMemsetAsync(p->d_flag.p, 0, 4 * sizeof(int), p->stream));
    CU(cudaMemsetAsync(p->d_st.p, 0, sizeof(LmState), p->stream));

    cmark("visiting orders, uploads, allocations");
    DevProblem &dp = p->dp;
    dp.C = p->C; dp.M = p->M; dp.F = Fl; dp.N = Nl; dp.root_cam = p->root_cam; dp.root_marker = p->root_marker;
    dp.opt_c = p->opt_c; dp.opt_m = p->opt_m; dp.opt_f = p->opt_f; dp.huber = p->huber;
    dp.nrc = p->nrc; dp.nrm = p->nrm; dp.n_r = p->n_r; dp.col_frame0 = p->n_r + 6 * p->f_begin;
    dp.opt_i = p->opt_i; dp.nri = p->nri; dp.col_intr0 = 6 * (p->nrc + p->nrm); dp.st_dev = nullptr;
    dp.h = (double)(p->marker_size / 2.f); // aruco::Marker::get3DPoints: half size in float (marker.cpp:358-369)
    dp.J_delta = p->J_delta;
    dp.obs_f = p->d_obs_f.p; dp.obs_cm = p->d_obs_cm.p; dp.obs_slot_c = p->d_slot_c.p; dp.obs_slot_m = p->d_slot_m.p;
    dp.obs_pair = p->d_obs_pair.p; dp.pair_fc = p->d_pair_fc.p; dp.npairs = p->npairs; dp.pair_tab = p->d_pair_tab.p;
    dp.und_a = p->d_und_a.p; dp.und_b = p->d_und_b.p; dp.raw_a = p->d_raw_a.p; dp.raw_b = p->d_raw_b.p;
    dp.intr = p->d_intr.p; dp.intr_tr = p->opt_i ? p->d_intr_tr.p : p->d_intr.p; dp.frame_slot_ptr = p->d_frame_slot_ptr.p; dp.slot_block = p->d_slot_block.p;
    dp.frame_cs_cum = p->d_frame_cs_cum.p;
    dp.cam_tab = p->d_cam_tab.p; dp.mk_tab = p->d_mk_tab.p; dp.fr_tab = p->d_fr_tab.p; dp.cam_tr = p->d_cam_tr.p; dp.mk_tr = p->d_mk_tr.p; dp.fr_tr = p->d_fr_tr.p;
    dp.cam_fixed = p->d_cam_fixed.p; dp.mk_fixed = p->d_mk_fixed.p; dp.fr_fixed = p->d_fr_fixed.p;
    dp.analytic = p->analytic ? 1 : 0; dp.cam_an = p->d_cam_an.p; dp.mk_an = p->d_mk_an.p; dp.fr_an = p->d_fr_an.p;

    // ---- remove_distortions (multicam_mapper.cpp:554-578) on the device: raw -> und.
    // raw_a/raw_b hold corners (0,1) / (2,3); run the point kernel on each half.
    if (Nl > 0 && d->corners_undistorted) {
        CU(cudaMemcpyAsync(p->d_und_a.p, p->d_raw_a.p, (size_t)Nl * sizeof(float4), cudaMemcpyDeviceToDevice, p->stream));
        CU(cudaMemcpyAsync(p->d_und_b.p, p->d_raw_b.p, (size_t)Nl * sizeof(float4), cudaMemcpyDeviceToDevice, p->stream));
    } else if (Nl > 0) {
        // raw_a / raw_b viewed as 2 Nl float2 points each: point i belongs to observation i >> 1
        LAUNCH(p, k_undistort, cdiv(2 * Nl, 256), 256, 0, 2 * Nl, 1, reinterpret_cast<const float2 *>(p->d_raw_a.p), p->d_obs_cm.p, p->d_K9.p, p->d_dist5.p, reinterpret_cast<float2 *>(p->d_und_a.p));
        LAUNCH(p, k_undistort, cdiv(2 * Nl, 256), 256, 0, 2 * Nl, 1, reinterpret_cast<const float2 *>(p->d_raw_b.p), p->d_obs_cm.p, p->d_K9.p, p->d_dist5.p, reinterpret_cast<float2 *>(p->d_und_b.p));
    }
    { const char *e = getenv("AAR_FORCE_EXACT_STAGING"); p->force_exact_staging = e && *e == '1'; }   // test hook: FP64 staging of the Jacobian block
    {   // cluster Cholesky: up to 16 CTAs per cluster, block row + staging in shared memory
        bool cluster_ok = false;
        if (int rc = set_smem_caps(p, &cluster_ok)) return rc;
        const int nblk = (p->n_r + CH_NB - 1) / CH_NB;
        const size_t smem = cluster2_smem_bytes(nblk);
        const char *e = getenv("AAR_NO_CLUSTER_SOLVE");                       // development aid: force the cooperative-grid kernel
        if (!cluster_ok || nblk > 16 || smem > p->smem_optin - 1024 || (p->n_r & 1) || (e && *e == '1')) p->use_cluster_solve = false;
    }
    CU(cudaStreamSynchronize(p->stream));
    cmark("undistortion, attributes, sync");
    aar_lm_default_params(&p->params);
    p->num_det = nd; p->g_det = std::move(keep);
    guard.release();
    *out = p;
    return AAR_OK;
}

int aar_problem_create(const aar_problem_desc *d, aar_problem **out) { return create_impl(d, out, false); }

int aar_shard_plan(const aar_problem_desc *d, int32_t *frame_begin, int32_t *frame_end, int64_t *obs_begin, int64_t *obs_end, int64_t *num_observations) {
    aar_problem *p = nullptr;
    int rc = create_impl(d, &p, true);
    if (rc) return rc;
    if (frame_begin) *frame_begin = p->f_begin; if (frame_end) *frame_end = p->f_end;
    if (obs_begin) *obs_begin = p->o_begin; if (obs_end) *obs_end = p->o_end; if (num_observations) *num_observations = p->N;
    delete p;
    return AAR_OK;
}

int aar_row_map(const aar_problem_desc *d, int64_t capacity, int32_t *of, int32_t *oc, int32_t *om, int32_t *oj, int64_t *num_observations) {
    aar_problem *p = nullptr;
    int rc = create_impl(d, &p, true);
    if (rc) return rc;
    if (num_observations) *num_observations = p->N;
    if (p->N > capacity && (of || oc || om || oj)) { delete p; set_err("aar_row_map: capacity too small"); return AAR_ERR_INVALID; }
    rc = aar_index_maps(p, of, oc, om, oj, nullptr, nullptr, nullptr, nullptr, nullptr);
    delete p;
    return rc;
}

void aar_problem_destroy(aar_problem *p) {
    if (!p) return;
    if (!p->stream && !p->h_st) { delete p; return; }   // host-only handle
    cudaSetDevice(p->device);
    if (p->stream) cudaStreamSynchronize(p->stream);
    if (p->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(p->comm);
    for (auto &e : p->ev) if (e) cudaEventDestroy(e);
    if (p->h_st) cudaFreeHost(p->h_st);
    if (p->h_red3) cudaFreeHost(p->h_red3);
    if (p->h_flags) cudaFreeHost(p->h_flags);
    if (p->lm_exec) cudaGraphExecDestroy(p->lm_exec);
    if (p->lm_graph) cudaGraphDestroy(p->lm_graph);
    if (p->lm_side) cudaStreamDestroy(p->lm_side);
    if (p->own_stream && p->stream) cudaStreamDestroy(p->stream);
    delete p;
}

int64_t aar_num_vars(const aar_problem *p) { return p ? p->n_vars_ext : 0; }
int64_t aar_num_observations(const aar_problem *p) { return p ? p->N : 0; }
int64_t aar_num_local_observations(const aar_problem *p) { return p ? p->o_end - p->o_begin : 0; }
int64_t aar_jacobian_nnz(const aar_problem *p) {
    if (!p) return 0;
    long long nnz = 0;
    for (long long o = 0; o < p->N; o++) {
        if (!p->g_hasjac[(size_t)o]) continue;
        nnz += 48LL * ((col_cam(p, p->g_cam[(size_t)o]) >= 0) + (col_marker(p, p->g_marker[(size_t)o]) >= 0) + (p->opt_f ? 1 : 0)) + (p->opt_i ? 72 : 0);
    }
    return nnz;
}

int aar_index_maps(const aar_problem *p, int32_t *of, int32_t *oc, int32_t *om, int32_t *oj, int64_t *cc, int64_t *cmk, int64_t *cf, int32_t *fb, int32_t *fe) {
    if (!p) return AAR_ERR_INVALID;
    for (long long o = 0; o < p->N; o++) {
        if (of) of[o] = p->g_frame[(size_t)o];
        if (oc) oc[o] = p->g_cam[(size_t)o];
        if (om) om[o] = p->g_marker[(size_t)o];
        if (oj) oj[o] = p->g_hasjac[(size_t)o];
    }
    if (cc) for (int i = 0; i < p->C; i++) cc[i] = col_cam(p, i);
    if (cmk) for (int j = 0; j < p->M; j++) cmk[j] = col_marker(p, j);
    if (cf) for (int k = 0; k < p->F; k++) cf[k] = col_frame(p, k);
    if (fb) *fb = p->f_begin;
    if (fe) *fe = p->f_end;
    return AAR_OK;
}

int aar_get_observations(aar_problem *p, float *und_xy, float *raw_xy) {
    if (!p) return AAR_ERR_INVALID;
    CU(cudaSetDevice(p->device));
    const size_t Nl = (size_t)p->dp.N;
    std::vector<float4> a(Nl), b(Nl);
    for (int pass = 0; pass < 2; pass++) {
        float *dst = pass ? raw_xy : und_xy;
        if (!dst || !Nl) continue;
        CU(cudaMemcpyAsync(a.data(), pass ? p->d_raw_a.p : p->d_und_a.p, Nl * sizeof(float4), cudaMemcpyDeviceToHost, p->stream));
        CU(cudaMemcpyAsync(b.data(), pass ? p->d_raw_b.p : p->d_und_b.p, Nl * sizeof(float4), cudaMemcpyDeviceToHost, p->stream));
        CU(cudaStreamSynchronize(p->stream));
        for (size_t o = 0; o < Nl; o++) { float *q = dst + 8 * o; q[0] = a[o].x; q[1] = a[o].y; q[2] = a[o].z; q[3] = a[o].w; q[4] = b[o].x; q[5] = b[o].y; q[6] = b[o].z; q[7] = b[o].w; }
    }
    return AAR_OK;
}

int aar_mats2evec(const aar_problem *p, double *z) {
    if (!p || !z) return AAR_ERR_INVALID;
    size_t vi = 0;
    auto put = [&](const double *T) {
        double R[9], rv[3];
        for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) R[i * 3 + j] = T[i * 4 + j];
        aar_host::rotation_to_vector(R, rv);
        for (int i = 0; i < 3; i++) { z[vi + i] = rv[i]; z[vi + 3 + i] = T[i * 4 + 3]; }
        vi += 6;
    };
    if (p->opt_c) for (int i = 0; i < p->C; i++) if (i != p->root_cam) put(&p->cam_T[16 * (size_t)i]);
    if (p->opt_m) for (int i = 0; i < p->M; i++) if (i != p->root_marker) put(&p->marker_T[16 * (size_t)i]);
    if (p->opt_f) for (int i = 0; i < p->F; i++) put(&p->frame_T[16 * (size_t)i]);
    if (p->opt_i)                                            // fill_io_vec_cam_intrinsics (multicam_mapper.cpp:488-498)
        for (int c = 0; c < p->C; c++) {
            const double *K = &p->cam_K[9 * (size_t)c];
            z[vi] = K[0]; z[vi + 1] = K[2]; z[vi + 2] = K[4]; z[vi + 3] = K[5];
            for (int k = 0; k < 5; k++) z[vi + 4 + k] = p->cam_dist[5 * (size_t)c + k];
            vi += 9;
        }
    return AAR_OK;
}

// io_vec of the reference [cameras | markers | frames | 9 per camera: fx cx fy cy k1 k2 p1 p2 k3] (multicam_mapper.cpp:445-461,
// 488-522) <-> internal z [cameras | markers | 12 per camera: fx cx fy cy k1 k2 | p1 p2 k3 . . . | frames] (aar_intrinsics.cuh).
// Identity unless the intrinsics are optimised.
static void z_ext2int(const aar_problem *p, const double *ze, double *zi) {
    const size_t np = 6 * (size_t)(p->nrc + p->nrm), nf = p->opt_f ? 6 * (size_t)p->F : 0;
    std::memcpy(zi, ze, np * sizeof(double));
    for (int c = 0; c < p->C; c++) { double *d = zi + np + 12 * (size_t)c; std::memcpy(d, ze + np + nf + 9 * (size_t)c, 9 * sizeof(double)); d[9] = d[10] = d[11] = 0.0; }
    std::memcpy(zi + (size_t)p->n_r, ze + np, nf * sizeof(double));
}
static void z_int2ext(const aar_problem *p, const double *zi, double *ze) {
    const size_t np = 6 * (size_t)(p->nrc + p->nrm), nf = p->opt_f ? 6 * (size_t)p->F : 0;
    std::memcpy(ze, zi, np * sizeof(double));
    std::memcpy(ze + np, zi + (size_t)p->n_r, nf * sizeof(double));
    for (int c = 0; c < p->C; c++) std::memcpy(ze + np + nf + 9 * (size_t)c, zi + np + 12 * (size_t)c, 9 * sizeof(double));
}
static int upload_z(aar_problem *p, const double *z, double *dst) {
    if (p->n_vars <= 0) return AAR_OK;
    if (p->opt_i) {
        CU(cudaStreamSynchronize(p->stream));               // the staging vector may still feed an earlier copy
        p->z_stage.resize((size_t)p->n_vars);
        z_ext2int(p, z, p->z_stage.data());
        z = p->z_stage.data();
    }
    CU(cudaMemcpyAsync(dst, z, (size_t)p->n_vars * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    return AAR_OK;
}
// device z (internal order) -> caller's io_vec; the stream is synchronised on return when the intrinsics are optimised
static int download_z(aar_problem *p, const double *src, double *z_out) {
    if (p->n_vars <= 0) return AAR_OK;
    if (!p->opt_i) { CU(cudaMemcpyAsync(z_out, src, (size_t)p->n_vars * sizeof(double), cudaMemcpyDeviceToHost, p->stream)); return AAR_OK; }
    CU(cudaStreamSynchronize(p->stream));
    p->z_stage.resize((size_t)p->n_vars);
    CU(cudaMemcpyAsync(p->z_stage.data(), src, (size_t)p->n_vars * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaStreamSynchronize(p->stream));
    z_int2ext(p, p->z_stage.data(), z_out);
    return AAR_OK;
}

int aar_evec2mats(aar_problem *p, const double *z, double *cam_T, double *marker_T, double *frame_T) {
    if (!p || !z) return AAR_ERR_INVALID;
    CU(cudaSetDevice(p->device));
    int rc = upload_z(p, z, p->d_zt.p); if (rc) return rc;
    // trial tables hold the INVERSE camera transform; expand the cameras into a scratch via the marker path instead:
    // cameras are read back from the Jacobian tables' construction is inverse-only, so re-expand on the fly here.
    LAUNCH(p, k_expand_trial, cdiv((long long)p->C + p->M + p->dp.F, 128), 128, 0, p->dp, p->d_zt.p);
    std::vector<double> mk(12 * (size_t)p->M), fr(12 * (size_t)std::max(p->dp.F, 1)), ci(12 * (size_t)p->C);
    CU(cudaMemcpyAsync(mk.data(), p->d_mk_tr.p, mk.size() * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaMemcpyAsync(fr.data(), p->d_fr_tr.p, fr.size() * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaMemcpyAsync(ci.data(), p->d_cam_tr.p, ci.size() * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaStreamSynchronize(p->stream));
    auto to16 = [](const double *q, double *T) { for (int i = 0; i < 3; i++) { for (int j = 0; j < 3; j++) T[i * 4 + j] = q[i * 3 + j]; T[i * 4 + 3] = q[9 + i]; } T[12] = 0; T[13] = 0; T[14] = 0; T[15] = 1; };
    if (marker_T) for (int m = 0; m < p->M; m++) to16(&mk[12 * (size_t)m], marker_T + 16 * (size_t)m);
    if (frame_T) for (int f = 0; f < p->dp.F; f++) to16(&fr[12 * (size_t)f], frame_T + 16 * (size_t)(p->f_begin + f));
    if (cam_T) {
        // camera -> root camera = closed-form rigid inverse of the stored inverse ([R^T | -R^T t]); output-only convenience
        for (int c = 0; c < p->C; c++) {
            const double *q = &ci[12 * (size_t)c]; double *T = cam_T + 16 * (size_t)c;
            for (int i = 0; i < 3; i++) { for (int j = 0; j < 3; j++) T[i * 4 + j] = q[j * 3 + i]; T[i * 4 + 3] = -(q[0 * 3 + i] * q[9] + q[1 * 3 + i] * q[10] + q[2 * 3 + i] * q[11]); }
            T[12] = 0; T[13] = 0; T[14] = 0; T[15] = 1;
        }
    }
    return AAR_OK;
}

int aar_eval_residual(aar_problem *p, const double *z, float huber_delta, double *r, double *sum_sq) {
    if (!p || !z) return AAR_ERR_INVALID;
    CU(cudaSetDevice(p->device));
    int rc = upload_z(p, z, p->d_zt.p); if (rc) return rc;
    const size_t nr = 8 * (size_t)p->dp.N;
    if (r && p->d_r.n < nr) CU(p->d_r.alloc(std::max<size_t>(nr, 8)));
    CU(cudaMemsetAsync(p->d_red3.p, 0, 8 * sizeof(double), p->stream));
    residual(p, p->d_zt.p, huber_delta, r ? p->d_r.p : nullptr);
    if (r && nr) CU(cudaMemcpyAsync(r, p->d_r.p, nr * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaMemcpyAsync(p->h_red3, p->d_red3.p, 8 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaStreamSynchronize(p->stream));
    CU(cudaGetLastError());
    if (sum_sq) *sum_sq = p->h_red3[0];
    return AAR_OK;
}

int aar_error_report(aar_problem *p, const double *z, aar_error_report_out *out) {
    if (!p || !z || !out) return AAR_ERR_INVALID;
    if (p->world != 1) { set_err("aar_error_report: single-rank handles only"); return AAR_ERR_INVALID; }
    if (p->lm_active) { set_err("aar_error_report between aar_lm_begin and aar_lm_end would overwrite the trial buffers of the resident loop"); return AAR_ERR_INVALID; }
    const int nq = out->num_q;
    if (nq < 0 || nq > SEL_MAX_Q || (nq > 0 && (!out->q || !out->q_value))) { set_err("aar_error_report: num_q must be in [0, %d] with q and q_value given", SEL_MAX_Q); return AAR_ERR_INVALID; }
    for (int t = 0; t < nq; t++) if (!(out->q[t] >= 0.0 && out->q[t] <= 1.0)) { set_err("aar_error_report: q[%d] = %g is not in [0, 1]", t, out->q[t]); return AAR_ERR_INVALID; }
    CU(cudaSetDevice(p->device));
    const long long N = p->dp.N;
    const size_t ne = (size_t)p->C + p->M + p->F;
    int rc = upload_z(p, z, p->d_zt.p); if (rc) return rc;
    if (p->d_r.n < 8 * (size_t)N) CU(p->d_r.alloc(std::max<size_t>(8 * (size_t)N, 8)));
    if (p->d_rep_err.n < (size_t)N) CU(p->d_rep_err.alloc(std::max<size_t>((size_t)N, 1)));
    if (p->d_rep_cnt.n < ne) { CU(p->d_rep_cnt.alloc(ne)); CU(p->d_rep_sum.alloc(ne)); CU(p->d_rep_max.alloc(ne)); }
    CU(cudaMemsetAsync(p->d_red3.p, 0, 8 * sizeof(double), p->stream));
    CU(cudaMemsetAsync(p->d_rep_cnt.p, 0, ne * sizeof(unsigned long long), p->stream));
    CU(cudaMemsetAsync(p->d_rep_sum.p, 0, ne * sizeof(double), p->stream));
    CU(cudaMemsetAsync(p->d_rep_max.p, 0, ne * sizeof(unsigned long long), p->stream));
    if ((rc = residual(p, p->d_zt.p, 0.f, p->d_r.p, true))) return rc;
    if (N > 0) {
        const size_t msm = (size_t)p->M * 20;
        const int marker_smem = msm + 4096 <= p->smem_optin;
        int per_sm = 1; CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_report_obs, REP_THREADS, marker_smem ? msm : 0));
        const int grid = (int)std::min<long long>((long long)std::max(per_sm, 1) * p->num_sms, cdiv(N, REP_THREADS));
        LAUNCH(p, k_report_obs, grid, REP_THREADS, marker_smem ? msm : 0, N, p->d_r.p, p->dp.obs_f, p->dp.obs_cm, p->C, p->M, p->f_begin, marker_smem,
               p->d_rep_err.p, p->d_rep_cnt.p, p->d_rep_sum.p, p->d_rep_max.p);
    }
    // exact order statistics: ranks floor(q (n - 1)), ascending, share the digit passes
    std::vector<int> order((size_t)nq);
    std::vector<unsigned long long> sel(2 * (size_t)nq, 0);      // [prefix | rank] in rank order
    if (nq > 0 && N > 0) {
        std::iota(order.begin(), order.end(), 0);
        auto rank_of_q = [&](int t) { return (unsigned long long)std::floor(out->q[t] * (double)(N - 1)); };
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return rank_of_q(a) < rank_of_q(b); });
        for (int t = 0; t < nq; t++) sel[(size_t)nq + t] = rank_of_q(order[(size_t)t]);
        if (p->d_sel.n < 2 * (size_t)nq) CU(p->d_sel.alloc(2 * (size_t)nq));
        if (p->d_sel_hist.n < (size_t)nq * SEL_BINS) CU(p->d_sel_hist.alloc((size_t)nq * SEL_BINS));
        CU(cudaMemcpyAsync(p->d_sel.p, sel.data(), sel.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, p->stream));
        const auto *keys = reinterpret_cast<const unsigned long long *>(p->d_rep_err.p);
        for (int pass = 0; pass < SEL_PASSES; pass++) {
            const int smem_hist = pass == 0;                       // one histogram, most contended digit (sign, exponent)
            CU(cudaMemsetAsync(p->d_sel_hist.p, 0, (size_t)(smem_hist ? 1 : nq) * SEL_BINS * sizeof(unsigned), p->stream));
            int per_sm = 1; CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_sel_hist, REP_THREADS, smem_hist ? SEL_BINS * sizeof(unsigned) : 0));
            const int grid = (int)std::min<long long>((long long)std::max(per_sm, 1) * p->num_sms, cdiv(N, REP_THREADS));
            LAUNCH(p, k_sel_hist, grid, REP_THREADS, smem_hist ? SEL_BINS * sizeof(unsigned) : 0, N, keys, pass, nq, p->d_sel.p, smem_hist, p->d_sel_hist.p);
            LAUNCH(p, k_sel_pick, 1, REP_THREADS, 0, pass, nq, p->d_sel.p, p->d_sel.p + nq, p->d_sel_hist.p);
        }
        CU(cudaMemcpyAsync(sel.data(), p->d_sel.p, (size_t)nq * sizeof(unsigned long long), cudaMemcpyDeviceToHost, p->stream));
    }
    std::vector<unsigned long long> cnt(ne), mx(ne); std::vector<double> sum(ne), err(out->det_err ? (size_t)N : 0);
    CU(cudaMemcpyAsync(cnt.data(), p->d_rep_cnt.p, ne * sizeof(unsigned long long), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaMemcpyAsync(sum.data(), p->d_rep_sum.p, ne * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaMemcpyAsync(mx.data(), p->d_rep_max.p, ne * sizeof(unsigned long long), cudaMemcpyDeviceToHost, p->stream));
    if (!err.empty()) CU(cudaMemcpyAsync(err.data(), p->d_rep_err.p, err.size() * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaMemcpyAsync(p->h_red3, p->d_red3.p, 8 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaStreamSynchronize(p->stream));
    CU(cudaGetLastError());
    for (int t = 0; t < nq; t++) {
        double v = std::numeric_limits<double>::quiet_NaN();
        if (N > 0) std::memcpy(&v, &sel[(size_t)t], sizeof v);
        out->q_value[order.empty() ? t : order[(size_t)t]] = v;
    }
    auto put = [&](size_t e0, size_t n, int64_t *c, double *s, double *m) {
        for (size_t i = 0; i < n; i++) {
            if (c) c[i] = (int64_t)cnt[e0 + i];
            if (s) s[i] = sum[e0 + i];
            if (m) std::memcpy(&m[i], &mx[e0 + i], sizeof(double));
        }
    };
    put(0, (size_t)p->C, out->cam_count, out->cam_sum_sq, out->cam_max);
    put((size_t)p->C, (size_t)p->M, out->marker_count, out->marker_sum_sq, out->marker_max);
    put((size_t)p->C + p->M, (size_t)p->F, out->frame_count, out->frame_sum_sq, out->frame_max);
    if (out->det_err) {
        std::fill(out->det_err, out->det_err + p->num_det, std::numeric_limits<double>::quiet_NaN());
        for (long long o = 0; o < N; o++) out->det_err[p->g_det[(size_t)o]] = err[(size_t)o];
    }
    out->num_observations = N; out->num_not_in_problem = p->num_det - N; out->sum_sq = p->h_red3[0];
    return AAR_OK;
}

int aar_eval_jacobian(aar_problem *p, const double *z, int64_t *colptr, int32_t *rowidx, double *vals) {
    if (!p || !z || !colptr || !rowidx || !vals) return AAR_ERR_INVALID;
    if (p->world != 1) { set_err("aar_eval_jacobian: single-rank handles only"); return AAR_ERR_INVALID; }
    if (p->lm_active) { set_err("aar_eval_jacobian between aar_lm_begin and aar_lm_end would replace the resident iterate"); return AAR_ERR_INVALID; }
    CU(cudaSetDevice(p->device));
    int rc = upload_z(p, z, p->d_z.p); if (rc) return rc;
    // the staged rows the solver assembles from: float32 when every numerator fits one, else re-staged in FP64 before this returns
    bool rows64 = false;
    if ((rc = jacobian_accumulate(p, p->h_st->huber_eval, false, &rows64))) return rc;
    const size_t N = (size_t)p->N;
    const int ni = p->lens ? 9 : 4;          // intrinsics columns with values: all nine in the lens model, fx cx fy cy in the reference's
    std::vector<double> J64(rows64 ? JROW * N : 0), Ji(p->opt_i ? (size_t)(8 * ni) * N : 0);
    std::vector<float> J32(rows64 ? 0 : JROW * N);
    if (N > 0) {
        if (rows64) CU(cudaMemcpyAsync(J64.data(), p->d_Jn64.p, JROW * N * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        else CU(cudaMemcpyAsync(J32.data(), p->d_Jn32.p, JROW * N * sizeof(float), cudaMemcpyDeviceToHost, p->stream));
        if (p->opt_i) {     // intrinsics columns: no staged rows, recomputed from the pose and pair tables just expanded
            if (p->d_Ji.n < Ji.size()) CU(p->d_Ji.alloc(Ji.size()));
            if (p->lens) LAUNCH(p, k_lens_dump, cdiv(p->dp.N, 128), 128, 0, p->dp, p->d_lens.p, p->d_Ji.p);
            else LAUNCH(p, k_intr_dump, cdiv(p->dp.N, 128), 128, 0, p->dp, p->d_Ji.p);
            CU(cudaMemcpyAsync(Ji.data(), p->d_Ji.p, Ji.size() * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        }
    }
    CU(cudaStreamSynchronize(p->stream));
    CU(cudaGetLastError());
    // entry (o, col, q) of the dense 8x18 block, col = 6 * block + dof: a derivative in the analytic variant, else the
    // central-difference numerator divided by 2 delta as obtain_marker_derivs does (mcm.cpp:976-994; a product with the
    // reciprocal would not round the same)
    auto Jv = [&](long long o, int col, int q) {
        const size_t i = (size_t)o * JROW + (size_t)col * 8 + q;
        const double v = rows64 ? J64[i] : (double)J32[i];
        return p->analytic ? v : v / (2 * p->J_delta);
    };
    // compressed columns in the order setFromTriplets leaves them: columns ascending, rows ascending
    std::vector<std::vector<long long>> by_cam((size_t)p->C), by_marker((size_t)p->M), by_frame((size_t)p->F);
    for (long long o = 0; o < p->N; o++) {
        if (!p->g_hasjac[(size_t)o]) continue;
        by_cam[(size_t)p->g_cam[(size_t)o]].push_back(o); by_marker[(size_t)p->g_marker[(size_t)o]].push_back(o); by_frame[(size_t)p->g_frame[(size_t)o]].push_back(o);
    }
    long long nnz = 0, col = 0;
    colptr[0] = 0;
    auto emit = [&](const std::vector<long long> &obs, int local_col0) {
        for (int d = 0; d < 6; d++) {
            for (long long o : obs)
                for (int q = 0; q < 8; q++) { rowidx[nnz] = (int32_t)(8 * o + q); vals[nnz] = Jv(o, local_col0 + d, q); nnz++; }
            colptr[++col] = nnz;
        }
    };
    if (p->opt_c) for (int i = 0; i < p->C; i++) if (i != p->root_cam) emit(by_cam[(size_t)i], 0);
    if (p->opt_m) for (int i = 0; i < p->M; i++) if (i != p->root_marker) emit(by_marker[(size_t)i], 6);
    if (p->opt_f) for (int i = 0; i < p->F; i++) emit(by_frame[(size_t)i], 12);
    if (p->opt_i)                                            // 9 columns per camera, root included; without the lens model the distortion columns are explicit zeros (mcm.cpp:835-893)
        for (int i = 0; i < p->C; i++)
            for (int d = 0; d < 9; d++) {
                for (long long o : by_cam[(size_t)i])
                    for (int q = 0; q < 8; q++) { rowidx[nnz] = (int32_t)(8 * o + q); vals[nnz] = d < ni ? Ji[(size_t)o * 8 * ni + (size_t)d * 8 + q] : 0.0; nnz++; }
                colptr[++col] = nnz;
            }
    return AAR_OK;
}

int aar_reduced_system(aar_problem *p, const double *z, double mu, double *S, double *b, double *cost) {
    if (!p || !z) return AAR_ERR_INVALID;
    if (p->lm_active) { set_err("aar_reduced_system between aar_lm_begin and aar_lm_end would replace the resident iterate and LM state"); return AAR_ERR_INVALID; }
    CU(cudaSetDevice(p->device));
    int rc = upload_z(p, z, p->d_z.p); if (rc) return rc;
    CU(cudaMemsetAsync(p->d_red3.p, 0, 8 * sizeof(double), p->stream));
    if ((rc = solver_cost(p, p->d_z.p, p->h_st->huber_eval))) return rc;
    if ((rc = jacobian_accumulate(p, p->h_st->huber_eval))) return rc;
    p->h_st->mu = mu; push_state(p);
    const int n_r = p->n_r;
    double *dS = p->d_red.p;
    if (n_r > 0) LAUNCH(p, k_prepare_reduced, cdiv((long long)n_r * n_r + n_r, 256), 256, 0, n_r, p->d_Hrr.p, p->d_gr.p, dS);
    if ((rc = schur_eliminate(p, dS, dS + (size_t)n_r * n_r))) return rc;
    if (S && n_r) CU(cudaMemcpyAsync(S, dS, (size_t)n_r * n_r * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    if (b && n_r) CU(cudaMemcpyAsync(b, dS + (size_t)n_r * n_r, (size_t)n_r * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaMemcpyAsync(p->h_red3, p->d_red3.p, 8 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaStreamSynchronize(p->stream));
    CU(cudaGetLastError());
    if (cost) *cost = p->h_red3[0];
    return AAR_OK;
}

// ------------------------------------------------------------------------------- LM loop ----
int aar_lm_begin(aar_problem *p, const double *z0, const aar_lm_params *params) {
    if (!p) return AAR_ERR_INVALID;
    if (!z0 && !p->have_z0) { set_err("aar_lm_begin(z0 = NULL) restarts from the previous z0, but there is none"); return AAR_ERR_INVALID; }
    CU(cudaSetDevice(p->device));
    if (params) p->params = *params; else aar_lm_default_params(&p->params);
    int rc = AAR_OK;
    if (z0) {
        if ((rc = upload_z(p, z0, p->d_z.p))) return rc;
        if (p->n_vars > 0) CU(cudaMemcpyAsync(p->d_z0.p, p->d_z.p, (size_t)p->n_vars * sizeof(double), cudaMemcpyDeviceToDevice, p->stream));
        p->have_z0 = true;
    } else if (p->n_vars > 0) // restart from the starting point that is already resident on the device
        CU(cudaMemcpyAsync(p->d_z.p, p->d_z0.p, (size_t)p->n_vars * sizeof(double), cudaMemcpyDeviceToDevice, p->stream));
    // MultiCamMapper::solve: hubberDelta = 10 before the solver starts (multicam_mapper.cpp:425)
    const float huber0 = 10.f;
    CU(cudaMemsetAsync(p->d_flag.p, 0, 4 * sizeof(int), p->stream));
    // SparseLevMarq::init (sparselevmarq.h:237-249)
    CU(cudaMemsetAsync(p->d_red3.p, 0, 8 * sizeof(double), p->stream));
    if ((rc = solver_cost(p, p->d_z.p, huber0))) return rc;
    if ((rc = allreduce(p, p->d_red3.p, 1, ncclSum))) return rc;
    CU(cudaMemcpyAsync(p->h_red3, p->d_red3.p, 8 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    CU(cudaStreamSynchronize(p->stream));
    CU(cudaGetLastError());
    const aar_lm_params &P = p->params;
    LmState &h = *p->h_st;
    std::memset(&h, 0, sizeof(LmState));
    h.cost = h.prev_cost = p->initial_cost = p->h_red3[0];
    h.mu = -1; h.v = 2;       // v: uninitialised in the reference (sparselevmarq.h:133)
    h.huber_delta = h.huber_eval = huber0;
    h.ignore_stop = P.ignore_stop_rules; h.min_error = P.min_error; h.min_step = P.min_step_error_diff; h.min_avg = P.min_average_step_error_diff;
    h.rows = (double)(8 * p->N);
    if ((rc = push_state(p))) return rc;
    p->lm_active = true;
    if (!std::isfinite(h.cost)) { set_err("initial cost is not finite"); return AAR_ERR_NUMERIC; }
    return AAR_OK;
}


// ------------------------------------------------------------------------------- LM loops ----
// aar_lm_iterate runs SparseLevMarq::solve (sparselevmarq.h:439-472) in one of two ways.  Both launch the same kernels in the same
// order: lm_jacobian_phase, then lm_try until k_lm_decide says that no try follows (the do-while of step(), :384-419).  Every
// decision (accept / reject, damping, stop rules, hubberDelta annealing, the record of an iteration) is made on the device, in LmState.
//  - Graph-resident: two nested CUDA-graph WHILE nodes whose conditions the control kernels set,
//      WHILE outer { lm_jacobian_phase; WHILE inner { lm_try }; k_lm_next_iter_g }
//    Nothing returns to the host between the launch of the graph and its end.
//  - Host-driven: the same two functions launched from the host, with one read-back of LmState per try.  It runs the first
//    iteration of a solve (it sizes the scratch buffers and computes mu0, which needs a MAX all-reduce when sharded), the FP64 redo
//    of an iteration whose float32 staging was inexact, sharded handles (NCCL inside a conditional body), the analytic variant,
//    profiling, verbose mode, AAR_FORCE_EXACT_STAGING=1 and AAR_NO_GRAPH=1.
#define GR(call)                                                                                          \
    do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { set_err("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); ok = false; goto done; } } while (0)

static bool lm_graph_build(aar_problem *p) {
    p->lm_graph_tried = true;
    bool ok = true;
    cudaStream_t main_stream = p->stream;
    const long long launches_before = p->launches;
    cudaGraph_t body_outer = nullptr, body_inner = nullptr, tmp = nullptr;
    cudaGraphNode_t node_outer, node_inner;
    bool cap_outer = false, cap_inner = false;
    cudaGraphNodeParams np = {}, ni = {};
    cudaStreamCaptureStatus cs; const cudaGraphNode_t *deps = nullptr; size_t ndeps = 0; cudaGraph_t cg = nullptr;
    long long l0 = 0;
    if (cudaStreamCreateWithFlags(&p->lm_side, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); return false; }
    if (p->d_trace.alloc(LM_TRACE_DEV_CAP) != cudaSuccess) { cudaGetLastError(); return false; }
    GR(cudaGraphCreate(&p->lm_graph, 0));
    GR(cudaGraphConditionalHandleCreate(&p->lm_outer, p->lm_graph, 1, cudaGraphCondAssignDefault));
    GR(cudaGraphConditionalHandleCreate(&p->lm_inner, p->lm_graph, 0, 0));
    std::memset(&np, 0, sizeof np);
    np.type = cudaGraphNodeTypeConditional; np.conditional.handle = p->lm_outer; np.conditional.type = cudaGraphCondTypeWhile; np.conditional.size = 1;
    GR(cudaGraphAddNode(&node_outer, p->lm_graph, nullptr, 0, &np));
    body_outer = np.conditional.phGraph_out[0];
    GR(cudaStreamBeginCaptureToGraph(main_stream, body_outer, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed)); cap_outer = true;
    if (lm_jacobian_phase(p, true)) { ok = false; goto done; }
    // the inner WHILE node goes in by hand, behind everything captured so far; the capture continues behind it
    GR(cudaStreamGetCaptureInfo_v2(main_stream, &cs, nullptr, &cg, &deps, &ndeps));
    std::memset(&ni, 0, sizeof ni);
    ni.type = cudaGraphNodeTypeConditional; ni.conditional.handle = p->lm_inner; ni.conditional.type = cudaGraphCondTypeWhile; ni.conditional.size = 1;
    GR(cudaGraphAddNode(&node_inner, body_outer, deps, ndeps, &ni));
    body_inner = ni.conditional.phGraph_out[0];
    GR(cudaStreamUpdateCaptureDependencies(main_stream, &node_inner, 1, cudaStreamSetCaptureDependencies));
    p->lm_body_launches = (int)(p->launches - launches_before);
    // one try of the do-while, captured on a side stream into the inner body
    l0 = p->launches;
    p->stream = p->lm_side;
    GR(cudaStreamBeginCaptureToGraph(p->lm_side, body_inner, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed)); cap_inner = true;
    if (lm_try(p, true)) { ok = false; goto done; }
    GR(cudaStreamEndCapture(p->lm_side, &tmp)); cap_inner = false;
    p->stream = main_stream;
    p->lm_try_launches = (int)(p->launches - l0);
    LAUNCH(p, k_lm_next_iter_g, 1, 1, 0, p->d_st.p, p->d_trace.p, p->lm_outer);
    p->lm_body_launches += 1;
    GR(cudaStreamEndCapture(main_stream, &tmp)); cap_outer = false;
    GR(cudaGraphInstantiate(&p->lm_exec, p->lm_graph, 0));
done:
    p->stream = main_stream;
    if (cap_inner) { cudaStreamEndCapture(p->lm_side, &tmp); }
    if (cap_outer) { cudaStreamEndCapture(main_stream, &tmp); }
    p->launches = launches_before;                       // capture is not execution
    if (!ok) { cudaGetLastError(); if (p->lm_exec) { cudaGraphExecDestroy(p->lm_exec); p->lm_exec = nullptr; } }
    p->lm_graph_ok = ok;
    return ok;
}
#undef GR

// the kernels of an LM iteration changed (aar_set_fixed, aar_set_prior): the next aar_lm_iterate captures the graph again
static void drop_lm_graph(aar_problem *p) {
    if (p->lm_exec) cudaGraphExecDestroy(p->lm_exec);
    if (p->lm_graph) cudaGraphDestroy(p->lm_graph);
    if (p->lm_side) cudaStreamDestroy(p->lm_side);
    p->lm_exec = nullptr; p->lm_graph = nullptr; p->lm_side = nullptr;
    p->lm_graph_tried = p->lm_graph_ok = false;
}

// up to `iters` LM iterations inside the graph; one host synchronisation at the end
static int lm_graph_run(aar_problem *p, int iters, aar_lm_report *rep) {
    LmState &h = *p->h_st;
    const int iter0 = h.iter; const long long tries0 = h.total_tries;
    h.max_iters = h.iter + iters; h.trace_len = 0;
    int rc;
    if ((rc = push_state(p))) return rc;
    CU(cudaGraphLaunch(p->lm_exec, p->stream));
    if ((rc = fetch_state(p))) return rc;                    // the one synchronisation of the call
    CU(cudaGetLastError());
    p->lm_graph_launches++; p->lm_graph_iters += h.iter - iter0;
    p->launches += (long long)(h.iter - iter0) * p->lm_body_launches + (h.total_tries - tries0) * p->lm_try_launches + (h.must_exit == -2 ? p->lm_body_launches : 0);
    if (rep && rep->trace && h.trace_len > 0 && rep->trace_len < rep->trace_capacity) {
        const int n = std::min(h.trace_len, rep->trace_capacity - rep->trace_len);
        CU(cudaMemcpyAsync(rep->trace + rep->trace_len, p->d_trace.p, (size_t)n * sizeof(aar_lm_trace), cudaMemcpyDeviceToHost, p->stream));
        CU(cudaStreamSynchronize(p->stream));
        rep->trace_len += n;
    }
    return AAR_OK;
}

// one LM iteration with the host in the loop: one read-back of the state per try
static int lm_host_iteration(aar_problem *p, aar_lm_report *rep) {
    static_assert(sizeof(LmTraceDev) == sizeof(aar_lm_trace), "trace layouts differ");
    LmState &h = *p->h_st;
    const double prev_cost = h.prev_cost;
    int rc;
    if ((rc = lm_jacobian_phase(p, false))) return rc;
    for (int ntries = 0;; ntries++) {
        if ((rc = lm_try(p, false))) return rc;
        if ((rc = fetch_state(p))) return rc;
        prof_mark(p, 6);
        CU(cudaGetLastError());
        if (p->profiling) {
            cudaEventSynchronize(p->ev[6]);
            float ms;
            if (ntries == 0) {
                cudaEventElapsedTime(&ms, p->ev[0], p->ev[1]); p->phase_ms[0] += ms;
                cudaEventElapsedTime(&ms, p->ev[7], p->ev[9]); p->phase_ms[5] += ms; p->phase_ms[6] += 1;
                cudaEventElapsedTime(&ms, p->ev[9], p->ev[8]); p->phase_ms[7] += ms;
                if (p->npairs > 0) { cudaEventElapsedTime(&ms, p->ev[9], p->ev[12]); p->phase_ms[10] += ms; cudaEventElapsedTime(&ms, p->ev[12], p->ev[8]); p->phase_ms[11] += ms; }
            }
            if (p->opt_f && p->dp.F > 0 && p->n_r > 0 && p->nslots > 0) { cudaEventElapsedTime(&ms, p->ev[10], p->ev[11]); p->phase_ms[8] += ms; p->phase_ms[9] += 1; }
            cudaEventElapsedTime(&ms, p->ev[2], p->ev[3]); p->phase_ms[1] += ms;
            cudaEventElapsedTime(&ms, p->ev[3], p->ev[4]); p->phase_ms[2] += ms;
            cudaEventElapsedTime(&ms, p->ev[4], p->ev[5]); p->phase_ms[3] += ms;
            cudaEventElapsedTime(&ms, p->ev[5], p->ev[6]); p->phase_ms[4] += ms;
        }
        if (!h.more_tries) break;
    }
    if (h.must_exit >= 0) {                              // the iteration completed: h.last is its record
        const LmTraceDev &t = h.last;
        if (p->params.verbose)
            printf("Curr Error=%.5g AErr(prev-curr)=%.5g gain=%.5g dumping factor=%.5g\n", t.cost, (prev_cost - t.cost) / h.rows, t.gain, t.mu);
        if (rep && rep->trace && rep->trace_len < rep->trace_capacity) std::memcpy(&rep->trace[rep->trace_len++], &t, sizeof(aar_lm_trace));
    }
    return AAR_OK;
}

// the error of a numeric stop (must_exit = -1), from the flags read back with the state
static int lm_numeric_error(aar_problem *p) {
    // flags[0]: a non-positive pivot in a frame block or in the reduced system (the kernels substituted 1 to keep going):
    //   the step that was just taken is not the solution of the damped normal equations.  The reference does not check
    //   its LDLT (sparselevmarq.h:394-400) and would continue on garbage; this path stops and says so.
    // flags[2]: the rotation of a translation-perturbed inverse camera pose differed from the unperturbed one, so the
    //   translation-only camera variants of k_expand_jac do not reproduce cv::Mat::inv() bit for bit.
    const int *flags = p->h_flags;
    set_err(flags[0] ? "non-positive Cholesky pivot at iteration %d (damped normal equations not positive definite)"
                     : flags[2] ? "camera inverse of a translation-perturbed pose changed its rotation at iteration %d (bit-exact table assumption violated)"
                                : "non-finite cost at iteration %d", p->h_st->iter);
    CU(cudaMemsetAsync(p->d_flag.p, 0, 4 * sizeof(int), p->stream));
    return AAR_ERR_NUMERIC;
}

static int lm_iterate(aar_problem *p, int max_iters, aar_lm_report *rep) {
    LmState &h = *p->h_st;
    const int iter0 = h.iter;
    const char *no_graph = getenv("AAR_NO_GRAPH");           // development aid: host-driven loop only
    const bool graph_eligible = !p->comm && !p->profiling && !p->params.verbose && !p->force_exact_staging && !p->analytic && !(no_graph && *no_graph == '1') && p->dp.N > 0;
    h.must_exit = 0;
    while (h.must_exit == 0 && h.iter - iter0 < max_iters) {
        int rc;
        if (graph_eligible && h.mu >= 0 && !p->exact_next && (p->lm_graph_ok || (!p->lm_graph_tried && lm_graph_build(p))))
            rc = lm_graph_run(p, std::min(max_iters - (h.iter - iter0), LM_TRACE_DEV_CAP), rep);
        else
            rc = lm_host_iteration(p, rep);
        if (rc) return rc;
        if (h.must_exit == -1) return lm_numeric_error(p);
        if (h.must_exit == -2) {     // inexact float32 staging: nothing was decided; redo the iteration with FP64 staging (never seen on real data)
            p->exact_reruns++; p->exact_next = true; h.must_exit = 0;
            CU(cudaMemsetAsync(p->d_flag.p + 1, 0, sizeof(int), p->stream));
        }
    }
    if (rep) { rep->final_cost = h.cost; rep->iterations = h.iter - iter0; rep->exit_code = h.must_exit; rep->total_tries = h.total_tries; }
    return AAR_OK;
}

int aar_lm_iterate(aar_problem *p, int32_t max_iters, aar_lm_report *rep) {
    if (!p || !p->lm_active) { set_err("aar_lm_iterate without aar_lm_begin"); return AAR_ERR_INVALID; }
    CU(cudaSetDevice(p->device));
    if (rep) { rep->trace_len = 0; rep->initial_cost = p->initial_cost; }
    p->dp.st_dev = p->d_st.p;
    const int rc = lm_iterate(p, max_iters, rep);
    p->dp.st_dev = nullptr;                              // the evaluation hooks obey their Huber argument
    if (rc) p->lm_active = false;
    return rc;
}
int aar_lm_end(aar_problem *p, double *z_out) {
    if (!p || !p->lm_active) return AAR_ERR_INVALID;
    CU(cudaSetDevice(p->device));
    if (z_out && p->n_vars > 0) {
        if (p->comm && p->opt_f) {
            // every rank owns its frame columns; the reduced part is identical everywhere: zero foreign frames, all-reduce(sum), rank>0 zero their reduced part
            const size_t fb = (size_t)p->dp.col_frame0, fe = fb + 6 * (size_t)p->dp.F, n = (size_t)p->n_vars;
            CU(cudaMemcpyAsync(p->d_zt.p, p->d_z.p, n * sizeof(double), cudaMemcpyDeviceToDevice, p->stream));
            if (p->rank != 0 && p->n_r) CU(cudaMemsetAsync(p->d_zt.p, 0, (size_t)p->n_r * sizeof(double), p->stream));
            if (fb > (size_t)p->n_r) CU(cudaMemsetAsync(p->d_zt.p + p->n_r, 0, (fb - (size_t)p->n_r) * sizeof(double), p->stream));
            if (fe < n) CU(cudaMemsetAsync(p->d_zt.p + fe, 0, (n - fe) * sizeof(double), p->stream));
            int rc = allreduce(p, p->d_zt.p, n, ncclSum); if (rc) return rc;
            if ((rc = download_z(p, p->d_zt.p, z_out))) return rc;
        } else { int rc = download_z(p, p->d_z.p, z_out); if (rc) return rc; }
    }
    CU(cudaStreamSynchronize(p->stream));
    p->lm_active = false;
    return AAR_OK;
}

int aar_lm_solve(aar_problem *p, double *z, const aar_lm_params *params, aar_lm_report *rep) {
    int rc = aar_lm_begin(p, z, params); if (rc) return rc;
    rc = aar_lm_iterate(p, p->params.max_iters, rep); if (rc) return rc;
    return aar_lm_end(p, z);
}

// MultiCamMapper::track() for all local frames: upload the start poses / run the per-frame solves / read the results back.
// The three steps are separate entry points so that a caller whose poses already live on the device (bench.py: `value`) can
// time the solves alone; aar_track_batch is the host-buffer call of the reference boundary (mcm.cpp:430-443).
static int track_alloc(aar_problem *p) {
    const int F = p->dp.F;
    if (!p->d_trk_z.n) {
        CU(p->d_trk_cam_inv.alloc((size_t)p->C * POSE_STRIDE)); CU(p->d_trk_Y.alloc((size_t)p->M * 12));
        CU(p->d_trk_z.alloc((size_t)F * 6)); CU(p->d_trk_z0.alloc((size_t)F * 6)); CU(p->d_trk_cost.alloc((size_t)F)); CU(p->d_trk_iters.alloc((size_t)F));
    }
    return AAR_OK;
}
int aar_track_upload(aar_problem *p, const double *z6) {
    if (!p || !z6) return AAR_ERR_INVALID;
    CU(cudaSetDevice(p->device));
    if (p->dp.F == 0) return AAR_OK;
    int rc = track_alloc(p); if (rc) return rc;
    CU(cudaMemcpyAsync(p->d_trk_z0.p, z6, (size_t)p->dp.F * 6 * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    p->trk_have_z0 = true;
    return AAR_OK;
}
int aar_track_run(aar_problem *p, const aar_lm_params *params) {
    if (!p) return AAR_ERR_INVALID;
    CU(cudaSetDevice(p->device));
    const int F = p->dp.F;
    if (F == 0) return AAR_OK;
    if (!p->trk_have_z0) { set_err("aar_track_run without aar_track_upload"); return AAR_ERR_INVALID; }
    aar_lm_params P; if (params) P = *params; else aar_lm_default_params(&P);
    // the rig is the one the handle was created with (camera / marker transforms are not optimised by track())
    LAUNCH(p, k_track_prepare, cdiv((long long)p->C + p->M, 128), 128, 0, p->dp, p->d_trk_cam_inv.p, p->d_trk_Y.p);
    CU(cudaMemcpyAsync(p->d_trk_z.p, p->d_trk_z0.p, (size_t)F * 6 * sizeof(double), cudaMemcpyDeviceToDevice, p->stream));
    TrackParams tp; tp.max_iters = P.max_iters; tp.min_error = P.min_error; tp.min_step_error_diff = P.min_step_error_diff;
    tp.min_average_step_error_diff = P.min_average_step_error_diff; tp.tau = P.tau; tp.der_epsilon = P.der_epsilon; tp.huber = p->huber;
    const size_t smem = track_cta_smem(p->C);
    const char *e = getenv("AAR_TRACK");
    prof_mark(p, 13);
    if (smem <= p->smem_optin && !(e && !strcmp(e, "warp"))) {      // one CTA per frame, T1 = inv(Tc) * To once per camera and pose variant
        LAUNCH(p, k_track_cta, F, TRKB_THREADS, smem, p->dp, tp, p->d_frame_obs_ptr.p, p->d_trk_cam_inv.p, p->d_trk_Y.p, p->d_trk_z.p, p->d_trk_cost.p, p->d_trk_iters.p);
    } else
        LAUNCH(p, k_track, cdiv(F, TRK_WARPS), TRK_WARPS * 32, 0, p->dp, tp, p->d_frame_obs_ptr.p, p->d_trk_cam_inv.p, p->d_trk_Y.p, p->d_trk_z.p, p->d_trk_cost.p, p->d_trk_iters.p);
    prof_mark(p, 14);
    CU(cudaGetLastError());
    if (p->profiling) { CU(cudaEventSynchronize(p->ev[14])); float ms; cudaEventElapsedTime(&ms, p->ev[13], p->ev[14]); p->track_ms += ms; p->track_runs++; }
    return AAR_OK;
}
int aar_track_download(aar_problem *p, double *z6, double *final_cost, int32_t *iterations) {
    if (!p) return AAR_ERR_INVALID;
    CU(cudaSetDevice(p->device));
    const int F = p->dp.F;
    if (F > 0) {
        if (z6) CU(cudaMemcpyAsync(z6, p->d_trk_z.p, (size_t)F * 6 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        if (final_cost) CU(cudaMemcpyAsync(final_cost, p->d_trk_cost.p, (size_t)F * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        if (iterations) CU(cudaMemcpyAsync(iterations, p->d_trk_iters.p, (size_t)F * sizeof(int), cudaMemcpyDeviceToHost, p->stream));
    }
    CU(cudaStreamSynchronize(p->stream));
    CU(cudaGetLastError());
    return AAR_OK;
}
int aar_track_batch(aar_problem *p, double *z6, const aar_lm_params *params, double *final_cost, int32_t *iterations) {
    if (!p || !z6) return AAR_ERR_INVALID;
    int rc;
    if ((rc = aar_track_upload(p, z6))) return rc;
    if ((rc = aar_track_run(p, params))) return rc;
    return aar_track_download(p, z6, final_cost, iterations);
}
int aar_track_ms(const aar_problem *p, double *ms, int64_t *runs) {
    if (!p) return AAR_ERR_INVALID;
    if (ms) *ms = p->track_ms; if (runs) *runs = p->track_runs;
    return AAR_OK;
}

int aar_comm_unique_id(void *id128) {
    if (!id128) return AAR_ERR_INVALID;
    if (!g_nccl.load()) return AAR_ERR_COMM;
    ncclUniqueId id;
    if (g_nccl.GetUniqueId(&id) != ncclSuccess) { set_err("ncclGetUniqueId failed"); return AAR_ERR_COMM; }
    std::memcpy(id128, &id, sizeof id);
    return AAR_OK;
}
int aar_comm_init(aar_problem *p, const void *id128) {
    if (!p || !id128) return AAR_ERR_INVALID;
    if (p->world <= 1) return AAR_OK;
    if (!g_nccl.load()) return AAR_ERR_COMM;
    CU(cudaSetDevice(p->device));
    ncclUniqueId id; std::memcpy(&id, id128, sizeof id);
    ncclResult_t r = g_nccl.CommInitRank(&p->comm, p->world, id, p->rank);
    if (r != ncclSuccess) { set_err("ncclCommInitRank: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "error"); p->comm = nullptr; return AAR_ERR_COMM; }
    return AAR_OK;
}

int64_t aar_kernel_launches(const aar_problem *p) { return p ? p->launches : 0; }
int aar_problem_stats(const aar_problem *p, int64_t *out) {
    if (!p || !out) return AAR_ERR_INVALID;
    out[0] = p->nslots; out[1] = p->npairs; out[2] = p->nmruns; out[3] = p->schur_fma;
    out[4] = (p->lm_graph_ok ? 2 : 0) | (p->last_cluster_solve ? 4 : 0) | (p->last_smem_acc ? 8 : 0) | (p->last_cm_rep ? 16 : 0) | ((long long)p->lm_graph_iters << 8); out[5] = p->max_slots; out[6] = p->f_begin; out[7] = p->f_end;
    return AAR_OK;
}
// uploads the union of the pose mask (aar_set_fixed) and the intrinsics flags (aar_set_fixed_intrinsics) for k_hold_fixed
static int apply_fixed(aar_problem *p, std::vector<uint8_t> pose_blk, std::vector<uint8_t> frame, std::vector<uint8_t> intr) {
    const int nb = p->nrc + p->nrm + p->nri, Fl = p->dp.F;
    std::vector<uint8_t> blk((size_t)std::max(nb, 1), 0), fr((size_t)std::max(Fl, 1), 0);
    bool any = false; long long free_blocks = 0;
    for (int i = 0; i < p->nrc + p->nrm; i++) { const bool f = !pose_blk.empty() && pose_blk[(size_t)i]; blk[(size_t)i] = f; any |= f; free_blocks += !f; }
    for (int c = 0; c < p->nri / 2; c++)
        for (int k = 0; k < 2; k++) {
            const bool f = !intr.empty() && ((intr[(size_t)c] >> k) & 1);
            blk[(size_t)(p->nrc + p->nrm + 2 * c + k)] = f; any |= f;
            free_blocks += !f && (k == 0 || p->lens);        // the reference's block B (distortion, padding) has no live column
        }
    if (p->opt_f)
        for (int k = 0; k < p->F; k++) {
            const bool f = !frame.empty() && frame[(size_t)k];
            if (k >= p->f_begin && k < p->f_end) fr[(size_t)(k - p->f_begin)] = f;
            any |= f; free_blocks += !f;
        }
    // with every column fixed the step is 0 and the gain 0 / 0
    if (any && free_blocks == 0) { set_err("the fixed masks leave no free column to solve for"); return AAR_ERR_INVALID; }
    CU(cudaSetDevice(p->device));
    if (any) {
        if (!p->d_blk_fixed.p) { CU(p->d_blk_fixed.alloc(blk.size())); CU(p->d_frame_fixed.alloc(fr.size())); }   // allocated once: the captured graph keeps the pointers
        CU(cudaMemcpyAsync(p->d_blk_fixed.p, blk.data(), blk.size(), cudaMemcpyHostToDevice, p->stream));
        CU(cudaMemcpyAsync(p->d_frame_fixed.p, fr.data(), fr.size(), cudaMemcpyHostToDevice, p->stream));
        CU(cudaStreamSynchronize(p->stream));
    }
    if (any != p->has_fixed) drop_lm_graph(p);   // the body of the graph-resident loop gains or loses k_hold_fixed
    p->has_fixed = any;
    p->fixed_pose_blk = std::move(pose_blk); p->fixed_frame = std::move(frame); p->fixed_intr = std::move(intr);
    return AAR_OK;
}
int aar_set_fixed(aar_problem *p, const uint8_t *cam_fixed, const uint8_t *marker_fixed, const uint8_t *frame_fixed) {
    if (!p) return AAR_ERR_INVALID;
    if (p->lm_active) { set_err("aar_set_fixed between aar_lm_begin and aar_lm_end"); return AAR_ERR_INVALID; }
    // only flags on optimised, non-root entities count
    std::vector<uint8_t> blk((size_t)(p->nrc + p->nrm), 0), fr;
    if (p->opt_c && cam_fixed)
        for (int i = 0; i < p->C; i++) if (i != p->root_cam) blk[(size_t)(i - (i > p->root_cam ? 1 : 0))] = cam_fixed[i] != 0;
    if (p->opt_m && marker_fixed)
        for (int j = 0; j < p->M; j++) if (j != p->root_marker) blk[(size_t)(p->nrc + j - (j > p->root_marker ? 1 : 0))] = marker_fixed[j] != 0;
    if (p->opt_f && frame_fixed) fr.assign(frame_fixed, frame_fixed + p->F);
    if (std::none_of(blk.begin(), blk.end(), [](uint8_t v) { return v != 0; })) blk.clear();
    return apply_fixed(p, std::move(blk), std::move(fr), p->fixed_intr);
}
int aar_set_fixed_intrinsics(aar_problem *p, const uint8_t *cam_flags) {
    if (!p) return AAR_ERR_INVALID;
    if (p->lm_active) { set_err("aar_set_fixed_intrinsics between aar_lm_begin and aar_lm_end"); return AAR_ERR_INVALID; }
    if (!p->opt_i) { set_err("aar_set_fixed_intrinsics: the handle does not optimise the intrinsics"); return AAR_ERR_INVALID; }
    std::vector<uint8_t> intr;
    if (cam_flags) {
        for (int c = 0; c < p->C; c++) if (cam_flags[c] > 3) { set_err("aar_set_fixed_intrinsics: camera %d: flags %d (bit 0 holds fx cx fy cy k1 k2, bit 1 p1 p2 k3)", p->cam_ids[(size_t)c], (int)cam_flags[c]); return AAR_ERR_INVALID; }
        intr.assign(cam_flags, cam_flags + p->C);
    }
    return apply_fixed(p, p->fixed_pose_blk, p->fixed_frame, std::move(intr));
}
int aar_set_prior(aar_problem *p, const double *cam_T, const double *cam_w, const double *marker_T, const double *marker_w,
                  const double *frame_T, const double *frame_w) {
    if (!p) return AAR_ERR_INVALID;
    if (p->lm_active) { set_err("aar_set_prior between aar_lm_begin and aar_lm_end"); return AAR_ERR_INVALID; }
    const int nb = p->nrc + p->nrm, Fl = p->dp.F;
    std::vector<double> blk((size_t)std::max(nb, 1) * PRIOR_STRIDE, 0.0), fr((size_t)std::max(Fl, 1) * PRIOR_STRIDE, 0.0);
    std::vector<uint8_t> blk_has((size_t)std::max(nb, 1), 0), fr_has((size_t)std::max(Fl, 1), 0);
    bool any = false;
    // every weight is checked, and the target of every entity with a nonzero weight; then only optimised, non-root entities (and this
    // rank's frames) are kept.  zbar is the R -> r of aar_mats2evec, so a target equal to the start matrix gives z - zbar = 0 exactly.
    auto take = [&](const char *what, int n, const double *T, const double *w, auto slot) -> int {
        if (!w) return AAR_OK;
        for (int e = 0; e < n; e++) {
            const double *we = w + 6 * (size_t)e;
            bool nonzero = false;
            for (int i = 0; i < 6; i++) {
                if (!(std::isfinite(we[i]) && we[i] >= 0)) { set_err("aar_set_prior: %s %d: weight %d is %g (must be finite and >= 0)", what, e, i, we[i]); return AAR_ERR_INVALID; }
                nonzero |= we[i] != 0;
            }
            if (!nonzero) continue;
            const double *Te = T ? T + 16 * (size_t)e : nullptr;
            bool finite = Te != nullptr;
            for (int k = 0; k < 12 && finite; k++) finite = std::isfinite(Te[k]);
            if (!finite) { set_err("aar_set_prior: %s %d has a nonzero weight and a %s target", what, e, Te ? "non-finite" : "missing"); return AAR_ERR_INVALID; }
            double *dst; uint8_t *has;
            if (!slot(e, dst, has)) continue;
            double R[9];
            for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) R[i * 3 + j] = Te[i * 4 + j];
            aar_host::rotation_to_vector(R, dst);
            for (int i = 0; i < 3; i++) dst[3 + i] = Te[i * 4 + 3];
            for (int i = 0; i < 6; i++) dst[6 + i] = we[i];
            *has = 1; any = true;
        }
        return AAR_OK;
    };
    int rc;
    if ((rc = take("camera", p->C, cam_T, cam_w, [&](int i, double *&d, uint8_t *&h) {
        if (!p->opt_c || i == p->root_cam) return false;
        const int b = i - (i > p->root_cam ? 1 : 0); d = &blk[(size_t)b * PRIOR_STRIDE]; h = &blk_has[(size_t)b]; return true; }))) return rc;
    if ((rc = take("marker", p->M, marker_T, marker_w, [&](int j, double *&d, uint8_t *&h) {
        if (!p->opt_m || j == p->root_marker) return false;
        const int b = p->nrc + j - (j > p->root_marker ? 1 : 0); d = &blk[(size_t)b * PRIOR_STRIDE]; h = &blk_has[(size_t)b]; return true; }))) return rc;
    bool any_frame = false;      // on any rank: every rank of a sharded handle launches the same kernels
    if ((rc = take("frame", p->F, frame_T, frame_w, [&](int k, double *&d, uint8_t *&h) {
        if (!p->opt_f) return false;
        any_frame = true;
        if (k < p->f_begin || k >= p->f_end) return false;
        d = &fr[(size_t)(k - p->f_begin) * PRIOR_STRIDE]; h = &fr_has[(size_t)(k - p->f_begin)]; return true; }))) return rc;
    any |= any_frame;
    CU(cudaSetDevice(p->device));
    if (any) {
        if (!p->d_blk_prior.p) {     // allocated once: the captured graph keeps the pointers
            CU(p->d_blk_prior.alloc(blk.size())); CU(p->d_frame_prior.alloc(fr.size()));
            CU(p->d_blk_has_prior.alloc(blk_has.size())); CU(p->d_frame_has_prior.alloc(fr_has.size()));
        }
        CU(cudaMemcpyAsync(p->d_blk_prior.p, blk.data(), blk.size() * sizeof(double), cudaMemcpyHostToDevice, p->stream));
        CU(cudaMemcpyAsync(p->d_frame_prior.p, fr.data(), fr.size() * sizeof(double), cudaMemcpyHostToDevice, p->stream));
        CU(cudaMemcpyAsync(p->d_blk_has_prior.p, blk_has.data(), blk_has.size(), cudaMemcpyHostToDevice, p->stream));
        CU(cudaMemcpyAsync(p->d_frame_has_prior.p, fr_has.data(), fr_has.size(), cudaMemcpyHostToDevice, p->stream));
        CU(cudaStreamSynchronize(p->stream));
    }
    if (any != p->has_prior) drop_lm_graph(p);   // the graph-resident loop gains or loses k_prior_add / k_prior_cost
    p->has_prior = any;
    return AAR_OK;
}
int aar_set_pair_prior(aar_problem *p, int32_t num_cam_pairs, const int32_t *cam_pairs, const double *cam_T, const double *cam_w,
                       int32_t num_marker_pairs, const int32_t *marker_pairs, const double *marker_T, const double *marker_w) {
    if (!p) return AAR_ERR_INVALID;
    if (p->lm_active) { set_err("aar_set_pair_prior between aar_lm_begin and aar_lm_end"); return AAR_ERR_INVALID; }
    std::vector<PairPriorRec> recs;
    // every pair is checked; then a pair is kept when a side has columns and a weight is nonzero (the others add nothing)
    auto take = [&](const char *what, int count, int n, const int32_t *pairs, const double *T, const double *w, auto col) -> int {
        if (n < 0) { set_err("aar_set_pair_prior: %d %s pairs", n, what); return AAR_ERR_INVALID; }
        if (n > 0 && (!pairs || !T || !w)) { set_err("aar_set_pair_prior: %d %s pairs and a NULL array", n, what); return AAR_ERR_INVALID; }
        for (int k = 0; k < n; k++) {
            const int a = pairs[2 * (size_t)k], b = pairs[2 * (size_t)k + 1];
            if (a < 0 || a >= count || b < 0 || b >= count) { set_err("aar_set_pair_prior: %s pair %d (%d, %d): index out of range [0, %d)", what, k, a, b, count); return AAR_ERR_INVALID; }
            if (a == b) { set_err("aar_set_pair_prior: %s pair %d joins %s %d with itself", what, k, what, a); return AAR_ERR_INVALID; }
            const double *we = w + 2 * (size_t)k, *Te = T + 16 * (size_t)k;
            for (int i = 0; i < 2; i++)
                if (!(std::isfinite(we[i]) && we[i] >= 0)) { set_err("aar_set_pair_prior: %s pair %d: weight %d is %g (must be finite and >= 0)", what, k, i, we[i]); return AAR_ERR_INVALID; }
            if (we[0] == 0 && we[1] == 0) continue;
            for (int i = 0; i < 12; i++)
                if (!std::isfinite(Te[i])) { set_err("aar_set_pair_prior: %s pair %d has a nonzero weight and a non-finite target", what, k); return AAR_ERR_INVALID; }
            double R[9], orth = 0;
            for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) R[i * 3 + j] = Te[i * 4 + j];
            for (int i = 0; i < 3; i++)
                for (int j = 0; j < 3; j++) orth = std::max(orth, std::fabs(R[i] * R[j] + R[3 + i] * R[3 + j] + R[6 + i] * R[6 + j] - (i == j ? 1.0 : 0.0)));
            const double det = R[0] * (R[4] * R[8] - R[5] * R[7]) - R[1] * (R[3] * R[8] - R[5] * R[6]) + R[2] * (R[3] * R[7] - R[4] * R[6]);
            if (!(orth <= 1e-9) || !(det > 0)) { set_err("aar_set_pair_prior: %s pair %d: the target rotation is not a rotation (|R^T R - I| = %g, det R = %g)", what, k, orth, det); return AAR_ERR_INVALID; }
            PairPriorRec r;
            r.col_a = (int)col(a); r.col_b = (int)col(b);
            if (r.col_a < 0 && r.col_b < 0) continue;
            std::memcpy(r.R, R, sizeof R);
            for (int i = 0; i < 3; i++) r.t[i] = Te[i * 4 + 3];
            r.w_rot = we[0]; r.w_t = we[1];
            recs.push_back(r);
        }
        return AAR_OK;
    };
    int rc;
    if ((rc = take("camera", p->C, num_cam_pairs, cam_pairs, cam_T, cam_w, [&](int i) { return col_cam(p, i); }))) return rc;
    if ((rc = take("marker", p->M, num_marker_pairs, marker_pairs, marker_T, marker_w, [&](int j) { return col_marker(p, j); }))) return rc;
    CU(cudaSetDevice(p->device));
    const int n = (int)recs.size();
    if (n != p->n_pair) {        // the graph-resident loop gains or loses the pair kernels, or their grids change: capture it again
        drop_lm_graph(p);
        CU(p->d_pair_prior.alloc(recs.size()));
        p->n_pair = n;
    }
    if (n) {                     // same count: the captured graph keeps the pointer and reads the new values
        CU(cudaMemcpyAsync(p->d_pair_prior.p, recs.data(), recs.size() * sizeof(PairPriorRec), cudaMemcpyHostToDevice, p->stream));
        CU(cudaStreamSynchronize(p->stream));
    }
    return AAR_OK;
}

int aar_set_profiling(aar_problem *p, int32_t on) { if (!p) return AAR_ERR_INVALID; p->profiling = on != 0; for (double &m : p->phase_ms) m = 0; p->track_ms = 0; p->track_runs = 0; return AAR_OK; }
int aar_get_phase_ms(const aar_problem *p, double *ms) {
    if (!p || !ms) return AAR_ERR_INVALID;
    for (int i = 0; i < AAR_NUM_PHASES; i++) ms[i] = p->phase_ms[i];
    return AAR_OK;
}

} // extern "C"
