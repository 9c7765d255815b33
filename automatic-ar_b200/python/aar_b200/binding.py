"""ctypes binding of the C ABI in include/aar_cuda.h (libaar_cuda.so).

This is the thin Python driver used by tests/, bench.py and __graft_entry__.py; the product is the
shared library.  Nothing here computes: every call goes to the CUDA path and raises AarError when
the library or the device is missing (there is no CPU fallback).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

PKG_ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))  # automatic-ar_b200/
REPO_ROOT = os.path.dirname(PKG_ROOT)
LIB_PATH = os.environ.get("AAR_LIB", os.path.join(PKG_ROOT, "libaar_cuda.so"))   # AAR_LIB: development aid (kernel variants)
CSRC = os.path.join(PKG_ROOT, "csrc")

NVCC_FLAGS = ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-fmad=false",  # parity: a*b+c stays two IEEE operations; FMAs are explicit fma() calls
              "-Xcompiler", "-fPIC", "-shared"]

# declared by include/aar_cuda.h — tests check that the library exports every one of them
EXPORTS = ["aar_lm_default_params", "aar_problem_create", "aar_problem_destroy", "aar_last_error", "aar_num_vars",
           "aar_num_observations", "aar_num_local_observations", "aar_jacobian_nnz", "aar_index_maps", "aar_get_observations",
           "aar_mats2evec", "aar_evec2mats", "aar_eval_residual", "aar_error_report", "aar_eval_jacobian", "aar_reduced_system", "aar_set_fixed", "aar_set_fixed_intrinsics", "aar_set_prior", "aar_set_pair_prior", "aar_lm_solve",
           "aar_lm_begin", "aar_lm_iterate", "aar_lm_end", "aar_track_batch", "aar_track_upload", "aar_track_run", "aar_track_download", "aar_track_ms", "aar_shard_plan", "aar_row_map", "aar_comm_unique_id", "aar_comm_init",
           "aar_kernel_launches", "aar_set_profiling", "aar_get_phase_ms", "aar_problem_stats"]


class AarError(RuntimeError):
    pass


def build(force=False, verbose=False):
    """nvcc cross-compiles for sm_100a without a GPU; the .so stays in-tree."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(REPO_ROOT, "include", f) for f in os.listdir(os.path.join(REPO_ROOT, "include"))]
    if not force and os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(s) for s in srcs):
        return LIB_PATH
    cmd = ["nvcc"] + NVCC_FLAGS + ["-o", LIB_PATH, os.path.join(CSRC, "aar_cuda.cu"), os.path.join(CSRC, "aar_init.cu")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode:
        print(" ".join(cmd)); print(r.stdout); print(r.stderr)
    if r.returncode:
        raise AarError("nvcc failed")
    return LIB_PATH


class Desc(C.Structure):
    _fields_ = [("num_cams", C.c_int32), ("num_markers", C.c_int32), ("num_frames", C.c_int32),
                ("cam_ids", C.c_void_p), ("marker_ids", C.c_void_p), ("frame_ids", C.c_void_p),
                ("root_cam", C.c_int32), ("root_marker", C.c_int32), ("marker_size", C.c_float),
                ("cam_T", C.c_void_p), ("marker_T", C.c_void_p), ("frame_T", C.c_void_p), ("cam_K", C.c_void_p), ("cam_dist", C.c_void_p),
                ("num_detections", C.c_int64), ("det_frame", C.c_void_p), ("det_cam", C.c_void_p), ("det_marker", C.c_void_p), ("det_xy", C.c_void_p),
                ("optimize_cam_poses", C.c_uint8), ("optimize_marker_poses", C.c_uint8), ("optimize_object_poses", C.c_uint8),
                ("optimize_cam_intrinsics", C.c_uint8), ("with_huber", C.c_uint8), ("corners_undistorted", C.c_uint8), ("analytic_jacobian", C.c_uint8), ("lens_model", C.c_uint8),
                ("J_delta", C.c_double), ("device", C.c_int32), ("stream", C.c_void_p), ("rank", C.c_int32), ("world_size", C.c_int32)]


class LmParams(C.Structure):
    _fields_ = [("max_iters", C.c_int32), ("min_error", C.c_double), ("min_step_error_diff", C.c_double),
                ("min_average_step_error_diff", C.c_double), ("tau", C.c_double), ("der_epsilon", C.c_double),
                ("ignore_stop_rules", C.c_int32), ("verbose", C.c_int32)]


class LmTrace(C.Structure):
    _fields_ = [("cost", C.c_double), ("mu", C.c_double), ("gain", C.c_double), ("tries", C.c_int32), ("accepted", C.c_int32),
                ("huber_delta", C.c_float), ("pad", C.c_int32)]


class LmReport(C.Structure):
    _fields_ = [("initial_cost", C.c_double), ("final_cost", C.c_double), ("iterations", C.c_int32), ("exit_code", C.c_int32),
                ("total_tries", C.c_int64), ("trace", C.POINTER(LmTrace)), ("trace_capacity", C.c_int32), ("trace_len", C.c_int32)]


class ErrorReportOut(C.Structure):
    _fields_ = [("det_err", C.c_void_p), ("cam_count", C.c_void_p), ("marker_count", C.c_void_p), ("frame_count", C.c_void_p),
                ("cam_sum_sq", C.c_void_p), ("marker_sum_sq", C.c_void_p), ("frame_sum_sq", C.c_void_p),
                ("cam_max", C.c_void_p), ("marker_max", C.c_void_p), ("frame_max", C.c_void_p),
                ("num_q", C.c_int32), ("reserved", C.c_int32), ("q", C.c_void_p), ("q_value", C.c_void_p),
                ("num_observations", C.c_int64), ("num_not_in_problem", C.c_int64), ("sum_sq", C.c_double)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise AarError(f"{LIB_PATH} is missing: build it with __graft_entry__.build() (no CPU fallback exists)")
        L = C.CDLL(LIB_PATH)
        L.aar_last_error.restype = C.c_char_p
        for f in ("aar_num_vars", "aar_num_observations", "aar_num_local_observations", "aar_jacobian_nnz", "aar_kernel_launches"):
            getattr(L, f).restype = C.c_int64
            getattr(L, f).argtypes = [C.c_void_p]
        _lib = L
    return _lib


def _chk(rc, what):
    if rc != 0:
        raise AarError(f"{what} failed (status {rc}): {lib().aar_last_error().decode()}")


def _vp(a):
    return a.ctypes.data_as(C.c_void_p)


class Problem:
    """MultiCamMapper-shaped handle on one GPU (one rank's frame shard when world_size > 1)."""

    @staticmethod
    def shard_plan(rig, rank, world_size):
        """aar_shard_plan: (frame_begin, frame_end, obs_begin, obs_end, num_observations) of a rank, host only."""
        d, keep = Problem._desc(rig, True, True, True, True, False, 0, None, rank, world_size, 0.0)
        fb = C.c_int32(0); fe = C.c_int32(0); ob = C.c_int64(0); oe = C.c_int64(0); n = C.c_int64(0)
        _chk(lib().aar_shard_plan(C.byref(d), C.byref(fb), C.byref(fe), C.byref(ob), C.byref(oe), C.byref(n)), "aar_shard_plan")
        return fb.value, fe.value, ob.value, oe.value, n.value

    @staticmethod
    def row_map(rig):
        """aar_row_map: the bit-exact observation -> row map (frame / camera / marker indices, has_jacobian), host only."""
        d, keep = Problem._desc(rig, True, True, True, True, False, 0, None, 0, 1, 0.0)
        n = C.c_int64(0)
        _chk(lib().aar_row_map(C.byref(d), C.c_int64(0), None, None, None, None, C.byref(n)), "aar_row_map")
        of = np.zeros(n.value, np.int32); oc = np.zeros(n.value, np.int32); om = np.zeros(n.value, np.int32); oj = np.zeros(n.value, np.int32)
        _chk(lib().aar_row_map(C.byref(d), n, _vp(of), _vp(oc), _vp(om), _vp(oj), C.byref(n)), "aar_row_map")
        return dict(frame_idx=of, cam_idx=oc, marker_idx=om, has_jac=oj)

    @staticmethod
    def _desc(rig, use_init, cams, markers, objects, with_huber, device, stream, rank, world_size, J_delta, intrinsics=False, analytic=False, lens=False,
              corners_undistorted=False):
        k = {}
        k["cam_ids"] = np.ascontiguousarray(rig.cam_ids, np.int32); k["marker_ids"] = np.ascontiguousarray(rig.marker_ids, np.int32)
        k["frame_ids"] = np.ascontiguousarray(rig.frame_ids, np.int32)
        k["cam_T"] = np.ascontiguousarray(rig.T_cam_init if use_init else rig.T_cam_true, np.float64)
        k["marker_T"] = np.ascontiguousarray(rig.T_marker_init if use_init else rig.T_marker_true, np.float64)
        k["frame_T"] = np.ascontiguousarray(rig.T_frame_init if use_init else rig.T_frame_true, np.float64)
        k["K"] = np.ascontiguousarray(rig.K, np.float64); k["dist"] = np.ascontiguousarray(rig.dist, np.float64)
        k["det_frame"] = np.ascontiguousarray(rig.det_frame, np.int32); k["det_cam"] = np.ascontiguousarray(rig.det_cam, np.int32)
        k["det_marker"] = np.ascontiguousarray(rig.det_marker, np.int32); k["det_xy"] = np.ascontiguousarray(rig.det_xy, np.float32)
        d = Desc()
        d.num_cams, d.num_markers, d.num_frames = len(k["cam_ids"]), len(k["marker_ids"]), len(k["frame_ids"])
        d.cam_ids, d.marker_ids, d.frame_ids = _vp(k["cam_ids"]), _vp(k["marker_ids"]), _vp(k["frame_ids"])
        d.root_cam, d.root_marker, d.marker_size = int(rig.root_cam), int(rig.root_marker), float(rig.marker_size)
        d.cam_T, d.marker_T, d.frame_T, d.cam_K, d.cam_dist = _vp(k["cam_T"]), _vp(k["marker_T"]), _vp(k["frame_T"]), _vp(k["K"]), _vp(k["dist"])
        d.num_detections = len(k["det_frame"])
        d.det_frame, d.det_cam, d.det_marker, d.det_xy = _vp(k["det_frame"]), _vp(k["det_cam"]), _vp(k["det_marker"]), _vp(k["det_xy"])
        d.optimize_cam_poses, d.optimize_marker_poses, d.optimize_object_poses, d.optimize_cam_intrinsics = int(cams), int(markers), int(objects), int(intrinsics)
        d.with_huber = int(with_huber); d.J_delta = J_delta; d.device = device
        d.analytic_jacobian = int(analytic); d.lens_model = int(lens); d.corners_undistorted = int(corners_undistorted)
        d.stream = C.c_void_p(stream) if stream else None
        d.rank, d.world_size = rank, world_size
        return d, k

    def __init__(self, rig, use_init=True, cams=True, markers=True, objects=True, with_huber=False, device=0, stream=None,
                 rank=0, world_size=1, J_delta=0.0, intrinsics=False, analytic=False, lens=False, corners_undistorted=False):
        """lens=True: the lens model of the analytic mode (aar_problem_desc::lens_model = 1): residuals on the raw corners against OpenCV's
        five-coefficient projection; implies analytic=True.  With intrinsics=True it refines K and the distortion of every camera."""
        L = lib()
        analytic = analytic or lens
        d, self._keep = self._desc(rig, use_init, cams, markers, objects, with_huber, device, stream, rank, world_size, J_delta, intrinsics, analytic, lens,
                                   corners_undistorted)
        self.h = C.c_void_p()
        _chk(L.aar_problem_create(C.byref(d), C.byref(self.h)), "aar_problem_create")
        self.nC, self.nM, self.nF = d.num_cams, d.num_markers, d.num_frames
        # reduced system: pose blocks, then two 6-wide pseudo-blocks per camera when the intrinsics are optimised (csrc/aar_intrinsics.cuh)
        self.n_r = 6 * ((self.nC - 1 if cams else 0) + (self.nM - 1 if markers else 0) + (2 * self.nC if intrinsics else 0))

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            lib().aar_problem_destroy(self.h); self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    num_vars = property(lambda s: int(lib().aar_num_vars(s.h)))
    num_obs = property(lambda s: int(lib().aar_num_observations(s.h)))
    num_local_obs = property(lambda s: int(lib().aar_num_local_observations(s.h)))
    jacobian_nnz = property(lambda s: int(lib().aar_jacobian_nnz(s.h)))
    kernel_launches = property(lambda s: int(lib().aar_kernel_launches(s.h)))

    def index_maps(self):
        N = self.num_obs
        of = np.zeros(N, np.int32); oc = np.zeros(N, np.int32); om = np.zeros(N, np.int32); oj = np.zeros(N, np.int32)
        cc = np.zeros(self.nC, np.int64); cm = np.zeros(self.nM, np.int64); cf = np.zeros(self.nF, np.int64)
        fb = C.c_int32(0); fe = C.c_int32(0)
        _chk(lib().aar_index_maps(self.h, _vp(of), _vp(oc), _vp(om), _vp(oj), _vp(cc), _vp(cm), _vp(cf), C.byref(fb), C.byref(fe)), "aar_index_maps")
        return dict(frame_idx=of, cam_idx=oc, marker_idx=om, has_jac=oj, col_cam=cc, col_marker=cm, col_frame=cf, frame_begin=fb.value, frame_end=fe.value)

    def observations(self):
        n = self.num_local_obs
        und = np.zeros((n, 8), np.float32); raw = np.zeros((n, 8), np.float32)
        _chk(lib().aar_get_observations(self.h, _vp(und), _vp(raw)), "aar_get_observations")
        return und, raw

    def mats2evec(self):
        z = np.zeros(self.num_vars); _chk(lib().aar_mats2evec(self.h, _vp(z)), "aar_mats2evec"); return z

    def evec2mats(self, z):
        z = np.ascontiguousarray(z, np.float64)
        Tc = np.zeros((self.nC, 4, 4)); Tm = np.zeros((self.nM, 4, 4)); Tf = np.zeros((self.nF, 4, 4))
        _chk(lib().aar_evec2mats(self.h, _vp(z), _vp(Tc), _vp(Tm), _vp(Tf)), "aar_evec2mats")
        return Tc, Tm, Tf

    def residual(self, z, huber_delta=2.5, want_vector=True):
        z = np.ascontiguousarray(z, np.float64)
        r = np.zeros(8 * self.num_local_obs) if want_vector else None
        ss = C.c_double(0)
        _chk(lib().aar_eval_residual(self.h, _vp(z), C.c_float(huber_delta), _vp(r) if want_vector else None, C.byref(ss)), "aar_eval_residual")
        return r, ss.value

    def error_report(self, z, q=(0.5, 0.9, 0.99)):
        """aar_error_report: reprojection error per detection (indexed like the rig's det_* arrays, NaN when not in the problem), count /
        sum of squares / max error per camera, marker and frame, exact percentiles q -> q_value, totals."""
        z = np.ascontiguousarray(z, np.float64)
        qa = np.ascontiguousarray(q, np.float64).reshape(-1)
        n_det = len(self._keep["det_frame"])
        r = dict(det_err=np.zeros(n_det), q=qa, q_value=np.zeros(len(qa)))
        out = ErrorReportOut()
        out.det_err = _vp(r["det_err"])
        for ent, n in (("cam", self.nC), ("marker", self.nM), ("frame", self.nF)):
            r[ent + "_count"] = np.zeros(n, np.int64); r[ent + "_sum_sq"] = np.zeros(n); r[ent + "_max"] = np.zeros(n)
            for k in ("count", "sum_sq", "max"):
                setattr(out, f"{ent}_{k}", _vp(r[f"{ent}_{k}"]))
        out.num_q = len(qa); out.q = _vp(qa); out.q_value = _vp(r["q_value"])
        _chk(lib().aar_error_report(self.h, _vp(z), C.byref(out)), "aar_error_report")
        r.update(observations=out.num_observations, not_in_problem=out.num_not_in_problem, sum_sq=out.sum_sq)
        return r

    def jacobian(self, z):
        z = np.ascontiguousarray(z, np.float64)
        nnz = self.jacobian_nnz
        colptr = np.zeros(self.num_vars + 1, np.int64); rowidx = np.zeros(nnz, np.int32); vals = np.zeros(nnz)
        _chk(lib().aar_eval_jacobian(self.h, _vp(z), _vp(colptr), _vp(rowidx), _vp(vals)), "aar_eval_jacobian")
        return colptr, rowidx, vals

    def reduced_system(self, z, mu):
        z = np.ascontiguousarray(z, np.float64)
        S = np.zeros((self.n_r, self.n_r)); b = np.zeros(self.n_r); cost = C.c_double(0)
        _chk(lib().aar_reduced_system(self.h, _vp(z), C.c_double(mu), _vp(S), _vp(b), C.byref(cost)), "aar_reduced_system")
        return S, b, cost.value

    def set_fixed(self, cams=None, markers=None, frames=None):
        """aar_set_fixed: hold cameras / markers / frames fixed in the later solves and reduced systems of this handle.  Boolean arrays by
        index ([num_cams], [num_markers], [num_frames] of the description); None = none of that kind; all None clears."""
        keep = []

        def mask(m, n, what):
            if m is None:
                return None
            a = np.asarray(m).reshape(-1)
            if len(a) != n:
                raise ValueError(f"set_fixed: {what} has {len(a)} entries, the description {n}")
            keep.append(np.ascontiguousarray(a != 0, dtype=np.uint8))
            return _vp(keep[-1])
        _chk(lib().aar_set_fixed(self.h, mask(cams, self.nC, "cams"), mask(markers, self.nM, "markers"), mask(frames, self.nF, "frames")), "aar_set_fixed")

    def set_fixed_intrinsics(self, flags=None):
        """aar_set_fixed_intrinsics: per camera index, bit 0 holds [fx cx fy cy k1 k2], bit 1 holds [p1 p2 k3]; None clears."""
        if flags is None:
            _chk(lib().aar_set_fixed_intrinsics(self.h, None), "aar_set_fixed_intrinsics")
            return
        a = np.ascontiguousarray(np.asarray(flags).reshape(-1), dtype=np.uint8)
        if len(a) != self.nC:
            raise ValueError(f"set_fixed_intrinsics: {len(a)} entries, the description has {self.nC} cameras")
        _chk(lib().aar_set_fixed_intrinsics(self.h, _vp(a)), "aar_set_fixed_intrinsics")

    def set_prior(self, cams=None, markers=None, frames=None):
        """aar_set_prior: soft pose priors in the later solves and reduced systems of this handle.  Each argument is a pair (T [n, 4, 4]
        targets, w [n, 6] information weights 1/sigma^2 of [r0 r1 r2 t0 t1 t2], 0 = none) by index of the description; None = no prior
        of that kind; all None clears."""
        keep = []

        def pair(tw, n, what):
            if tw is None:
                return None, None
            T, w = tw
            T = np.ascontiguousarray(T, dtype=np.float64); w = np.ascontiguousarray(w, dtype=np.float64)
            if T.shape != (n, 4, 4) or w.shape != (n, 6):
                raise ValueError(f"set_prior: {what} needs T [{n}, 4, 4] and w [{n}, 6], got {T.shape} and {w.shape}")
            keep.extend((T, w))
            return _vp(T), _vp(w)
        args = [*pair(cams, self.nC, "cams"), *pair(markers, self.nM, "markers"), *pair(frames, self.nF, "frames")]
        _chk(lib().aar_set_prior(self.h, *args), "aar_set_prior")

    def set_pair_prior(self, cams=None, markers=None):
        """aar_set_pair_prior: soft relative-pose priors between two cameras or two markers in the later solves and reduced systems of
        this handle.  Each argument is a triple (pairs [n, 2] indices (a, b) of the description, T [n, 4, 4] targets of
        T_ab = T_a^-1 T_b, w [n, 2] weights w_rot = 1/sigma_rot^2, w_t = 1/sigma_t^2); None = no pairs of that kind; both None clears."""
        keep = []

        def triple(ptw, what):
            if ptw is None:
                return 0, None, None, None
            P, T, w = ptw
            P = np.ascontiguousarray(P, dtype=np.int32); T = np.ascontiguousarray(T, dtype=np.float64); w = np.ascontiguousarray(w, dtype=np.float64)
            n = len(P)
            if P.shape != (n, 2) or T.shape != (n, 4, 4) or w.shape != (n, 2):
                raise ValueError(f"set_pair_prior: {what} needs pairs [n, 2], T [n, 4, 4] and w [n, 2], got {P.shape}, {T.shape} and {w.shape}")
            keep.extend((P, T, w))
            return n, _vp(P), _vp(T), _vp(w)
        args = [*triple(cams, "cams"), *triple(markers, "markers")]
        _chk(lib().aar_set_pair_prior(self.h, *args), "aar_set_pair_prior")

    @staticmethod
    def default_params(**kw):
        p = LmParams(); lib().aar_lm_default_params(C.byref(p))
        for k, v in kw.items():
            setattr(p, k, v)
        return p

    def _report(self, cap):
        rep = LmReport(); tr = (LmTrace * cap)()
        rep.trace = C.cast(tr, C.POINTER(LmTrace)); rep.trace_capacity = cap
        return rep, tr

    @staticmethod
    def _trace_array(rep, tr):
        return np.array([[t.cost, t.mu, t.gain, t.tries, t.accepted, t.huber_delta] for t in tr[:rep.trace_len]]).reshape(-1, 6)

    def solve(self, z0, params=None, trace_capacity=256):
        """MultiCamMapper::solve(): returns z, final cost, iterations, trace [cost, mu, gain, tries, accepted, huber]."""
        z = np.array(z0, np.float64, copy=True)
        rep, tr = self._report(trace_capacity)
        p = params if params is not None else self.default_params()
        _chk(lib().aar_lm_solve(self.h, _vp(z), C.byref(p), C.byref(rep)), "aar_lm_solve")
        self.last_report = rep
        return z, rep.final_cost, rep.iterations, self._trace_array(rep, tr)

    def solve_inplace(self, z, params=None):
        """aar_lm_solve on a caller-owned (e.g. pinned) float64 array, in place; returns the report."""
        assert z.dtype == np.float64 and z.flags["C_CONTIGUOUS"]
        rep, _ = self._report(1)
        p = params if params is not None else self.default_params()
        _chk(lib().aar_lm_solve(self.h, _vp(z), C.byref(p), C.byref(rep)), "aar_lm_solve")
        return rep

    def track_batch(self, z6, params=None):
        """MultiCamMapper::track() for every frame of the handle: z6 [F_local, 6] -> (z6, final cost [F], iterations [F])."""
        z = np.array(z6, np.float64, copy=True).reshape(-1, 6)
        cost = np.zeros(len(z)); iters = np.zeros(len(z), np.int32)
        p = params if params is not None else self.default_params()
        _chk(lib().aar_track_batch(self.h, _vp(z), C.byref(p), _vp(cost), _vp(iters)), "aar_track_batch")
        return z, cost, iters

    def track_upload(self, z6):
        z = np.ascontiguousarray(z6, np.float64).reshape(-1, 6)
        _chk(lib().aar_track_upload(self.h, _vp(z)), "aar_track_upload")

    def track_run(self, params=None):
        p = params if params is not None else self.default_params()
        _chk(lib().aar_track_run(self.h, C.byref(p)), "aar_track_run")

    def track_download(self, n_frames):
        z = np.zeros((n_frames, 6)); cost = np.zeros(n_frames); iters = np.zeros(n_frames, np.int32)
        _chk(lib().aar_track_download(self.h, _vp(z), _vp(cost), _vp(iters)), "aar_track_download")
        return z, cost, iters

    def track_ms(self):
        ms = C.c_double(0); runs = C.c_int64(0)
        _chk(lib().aar_track_ms(self.h, C.byref(ms), C.byref(runs)), "aar_track_ms")
        return ms.value, runs.value

    def lm_begin(self, z0=None, params=None):
        """z0 = None restarts from the z0 of the previous lm_begin (device resident, no copy)."""
        z = None if z0 is None else np.ascontiguousarray(z0, np.float64)
        p = params if params is not None else self.default_params()
        _chk(lib().aar_lm_begin(self.h, None if z is None else _vp(z), C.byref(p)), "aar_lm_begin")

    def lm_iterate(self, n, trace_capacity=0):
        rep, tr = self._report(max(trace_capacity, 1))
        _chk(lib().aar_lm_iterate(self.h, C.c_int32(n), C.byref(rep)), "aar_lm_iterate")
        return rep, self._trace_array(rep, tr)

    def lm_end(self):
        z = np.zeros(self.num_vars); _chk(lib().aar_lm_end(self.h, _vp(z)), "aar_lm_end"); return z

    def comm_init(self, id_bytes: bytes):
        buf = C.create_string_buffer(id_bytes, 128)
        _chk(lib().aar_comm_init(self.h, buf), "aar_comm_init")

    def stats(self):
        v = (C.c_int64 * 8)()
        _chk(lib().aar_problem_stats(self.h, v), "aar_problem_stats")
        d = dict(zip(["slots", "pairs", "mruns", "schur_fma", "mode_bits", "max_slots_per_frame", "frame_begin", "frame_end"], [int(x) for x in v]))
        d["peer_reduction"] = bool(d["mode_bits"] & 1); d["graph_loop"] = bool(d["mode_bits"] & 2); d["graph_iterations"] = d["mode_bits"] >> 8
        # paths of the last reduced solve and the last assembly
        d["cluster_solve"] = bool(d["mode_bits"] & 4); d["smem_accumulators"] = bool(d["mode_bits"] & 8); d["cm_replicas"] = bool(d["mode_bits"] & 16)
        return d

    def set_profiling(self, on=True):
        _chk(lib().aar_set_profiling(self.h, C.c_int32(int(on))), "aar_set_profiling")

    def phase_ms(self):
        v = (C.c_double * 12)()
        _chk(lib().aar_get_phase_ms(self.h, v), "aar_get_phase_ms")
        return dict(zip(["jacobian", "schur_solve", "backsub", "residual", "decide_comm", "jacobian_kernel", "jacobian_launches", "accumulate_kernel", "syrk_kernel", "syrk_launches", "asm_pairs_kernel", "asm_mruns_kernel"], list(v)))


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    _chk(lib().aar_comm_unique_id(buf), "aar_comm_unique_id")
    return buf.raw


# ------------------------------------------------------------------ include/aar_init.h
INIT_EXPORTS = ["aar_init_create", "aar_init_destroy", "aar_init_get_estimations", "aar_init_transforms", "aar_init_set_rig", "aar_init_object_transforms",
                "aar_init_counts", "aar_init_get_ids", "aar_init_get_rig", "aar_init_get_object_transforms", "aar_init_edges", "aar_init_consensus", "aar_init_timings"]


class InitDesc(C.Structure):
    _fields_ = [("num_cams", C.c_int32), ("cam_K", C.c_void_p), ("cam_dist", C.c_void_p), ("marker_size", C.c_double), ("num_frames", C.c_int32),
                ("num_detections", C.c_int64), ("det_frame", C.c_void_p), ("det_cam", C.c_void_p), ("det_marker", C.c_void_p), ("det_xy", C.c_void_p),
                ("excluded_cams", C.c_void_p), ("threshold", C.c_double), ("min_detections", C.c_int32), ("consensus_max", C.c_int32),
                ("device", C.c_int32), ("stream", C.c_void_p)]


class Initializer:
    """Initializer-shaped handle (include/aar_init.h): IPPE per detection, rig and object-pose initialisation on the device."""

    def __init__(self, num_cams, K, dist, marker_size, num_frames, det_frame, det_cam, det_marker, det_xy, excluded=None, threshold=2.0,
                 consensus_max=0, device=0, stream=None):
        self.L = lib(); self.h = C.c_void_p()
        self.N = len(det_frame)
        self._keep = [np.ascontiguousarray(K, dtype=np.float64).reshape(num_cams, 9), np.ascontiguousarray(dist, dtype=np.float64).reshape(num_cams, 5),
                      np.ascontiguousarray(det_frame, dtype=np.int32), np.ascontiguousarray(det_cam, dtype=np.int32),
                      np.ascontiguousarray(det_marker, dtype=np.int32), np.ascontiguousarray(det_xy, dtype=np.float32).reshape(-1, 8)]
        ex = np.zeros(num_cams, dtype=np.uint8)
        if excluded is not None:
            ex[list(excluded)] = 1
        self._keep.append(ex)
        k = self._keep
        d = InitDesc(num_cams, _vp(k[0]), _vp(k[1]), float(marker_size), int(num_frames), self.N, _vp(k[2]), _vp(k[3]), _vp(k[4]), _vp(k[5]), _vp(ex),
                     float(threshold), 2, int(consensus_max), int(device), stream)
        _chk(self.L.aar_init_create(C.byref(d), C.byref(self.h)), "aar_init_create")

    @classmethod
    def from_rig(cls, rig, **kw):
        nF = int(rig.frame_ids.max()) + 1 if rig.F else 0
        return cls(rig.C, rig.K, rig.dist, float(rig.marker_size), nF, rig.det_frame, rig.det_cam, rig.det_marker, rig.det_xy, **kw)

    def close(self):
        if self.h:
            self.L.aar_init_destroy(self.h); self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def estimations(self):
        T = np.zeros((self.N, 2, 4, 4)); err = np.zeros((self.N, 2)); nc = np.zeros(self.N, dtype=np.uint8)
        _chk(self.L.aar_init_get_estimations(self.h, _vp(T), _vp(err), _vp(nc)), "aar_init_get_estimations")
        return T, err, nc

    def init_transforms(self):
        _chk(self.L.aar_init_transforms(self.h), "aar_init_transforms")

    def set_rig(self, cam_ids, cam_T, marker_ids, marker_T):
        ci = np.ascontiguousarray(cam_ids, dtype=np.int32); mi = np.ascontiguousarray(marker_ids, dtype=np.int32)
        cT = np.ascontiguousarray(cam_T, dtype=np.float64); mT = np.ascontiguousarray(marker_T, dtype=np.float64)
        _chk(self.L.aar_init_set_rig(self.h, len(ci), _vp(ci), _vp(cT), len(mi), _vp(mi), _vp(mT)), "aar_init_set_rig")

    def init_object_transforms(self):
        _chk(self.L.aar_init_object_transforms(self.h), "aar_init_object_transforms")

    def counts(self):
        c = np.zeros(7, dtype=np.int32)
        _chk(self.L.aar_init_counts(self.h, _vp(c)), "aar_init_counts")
        return c

    def results(self):
        c = self.counts()
        cam_ids = np.zeros(c[0], dtype=np.int32); marker_ids = np.zeros(c[1], dtype=np.int32)
        _chk(self.L.aar_init_get_ids(self.h, _vp(cam_ids), _vp(marker_ids)), "aar_init_get_ids")
        ci = np.zeros(c[2], dtype=np.int32); cT = np.zeros((c[2], 4, 4)); mi = np.zeros(c[3], dtype=np.int32); mT = np.zeros((c[3], 4, 4))
        _chk(self.L.aar_init_get_rig(self.h, _vp(ci), _vp(cT), _vp(mi), _vp(mT)), "aar_init_get_rig")
        fi = np.zeros(c[4], dtype=np.int32); fT = np.zeros((c[4], 4, 4))
        _chk(self.L.aar_init_get_object_transforms(self.h, _vp(fi), _vp(fT)), "aar_init_get_object_transforms")
        return dict(cam_ids=cam_ids, marker_ids=marker_ids, root_cam=int(c[5]), root_marker=int(c[6]), cams=(ci, cT), markers=(mi, mT), objects=(fi, fT))

    def edges(self, cams=True):
        n = C.c_int32(0)
        _chk(self.L.aar_init_edges(self.h, int(cams), 0, None, None, None, None, C.byref(n)), "aar_init_edges")
        a = np.zeros(n.value, dtype=np.int32); b = np.zeros(n.value, dtype=np.int32); ln = np.zeros(n.value, dtype=np.int64); w = np.zeros(n.value)
        _chk(self.L.aar_init_edges(self.h, int(cams), n.value, _vp(a), _vp(b), _vp(ln), _vp(w), C.byref(n)), "aar_init_edges")
        return a, b, ln, w

    def timings(self):
        ms = np.zeros(3); n = C.c_int64(0)
        _chk(self.L.aar_init_timings(self.h, _vp(ms), C.byref(n)), "aar_init_timings")
        return dict(ippe_ms=ms[0], rig_ms=ms[1], objects_ms=ms[2], launches=n.value)


def init_consensus(marker_size, T, T1inv, T2inv, device=0):
    """aar_init_consensus: (index of the winner, its consensus error)."""
    T = np.ascontiguousarray(T, dtype=np.float64); A = np.ascontiguousarray(T1inv, dtype=np.float64); B = np.ascontiguousarray(T2inv, dtype=np.float64)
    best = C.c_int32(-1); w = C.c_double(0)
    _chk(lib().aar_init_consensus(int(device), C.c_double(marker_size), C.c_int64(len(T)), _vp(T), _vp(A), _vp(B), C.byref(best), C.byref(w)), "aar_init_consensus")
    return best.value, w.value
