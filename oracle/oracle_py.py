"""ctypes wrapper of the CPU oracle (TEST INFRASTRUCTURE ONLY).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import
this module.  `load(prefer_ref=True)` returns oracle/_ref/libaar_oracle_ref.so (restated
MultiCamMapper + the UNMODIFIED reference sparselevmarq.h) when it has been built, otherwise the
pure port oracle/libaar_oracle.so.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_libs = {}

_dp = C.POINTER(C.c_double)
_fp = C.POINTER(C.c_float)
_ip = C.POINTER(C.c_int)
_lp = C.POINTER(C.c_int64)


def _ptr(a, t):
    return a.ctypes.data_as(t)


def lib_path(ref: bool) -> str:
    return os.path.join(_HERE, "_ref", "libaar_oracle_ref.so") if ref else os.path.join(_HERE, "libaar_oracle.so")


def build(quiet=True):
    import subprocess
    subprocess.run(["make", "-C", _HERE, "all"], check=True,
                   stdout=subprocess.DEVNULL if quiet else None)


def load(prefer_ref=True):
    for ref in ([True, False] if prefer_ref else [False]):
        p = lib_path(ref)
        if os.path.exists(p):
            if p not in _libs:
                L = C.CDLL(p)
                L.aar_oracle_create.restype = C.c_void_p
                L.aar_oracle_num_vars.restype = C.c_int64
                L.aar_oracle_num_rows.restype = C.c_int64
                L.aar_oracle_jacobian.restype = C.c_int64
                if ref:
                    L.aar_oracle_time_ref_steps.restype = C.c_double
                _libs[p] = L
            return _libs[p], ref
    raise FileNotFoundError("oracle library not built: run `make -C oracle`")


class Oracle:
    """One restated MultiCamMapper instance built from a synth.Rig-like object."""

    def __init__(self, rig, prefer_ref=True, use_init=True, sincos_mode=1):
        self.L, self.is_ref = load(prefer_ref)
        self.L.aar_oracle_set_sincos_mode(C.c_int(sincos_mode))
        Tc = np.ascontiguousarray(rig.T_cam_init if use_init else rig.T_cam_true, dtype=np.float64)
        Tm = np.ascontiguousarray(rig.T_marker_init if use_init else rig.T_marker_true, dtype=np.float64)
        Tf = np.ascontiguousarray(rig.T_frame_init if use_init else rig.T_frame_true, dtype=np.float64)
        K = np.ascontiguousarray(rig.K, dtype=np.float64); d = np.ascontiguousarray(rig.dist, dtype=np.float64)
        ci = np.ascontiguousarray(rig.cam_ids, dtype=np.int32); mi = np.ascontiguousarray(rig.marker_ids, dtype=np.int32)
        fi = np.ascontiguousarray(rig.frame_ids, dtype=np.int32)
        df = np.ascontiguousarray(rig.det_frame, dtype=np.int32); dc = np.ascontiguousarray(rig.det_cam, dtype=np.int32)
        dm = np.ascontiguousarray(rig.det_marker, dtype=np.int32); dxy = np.ascontiguousarray(rig.det_xy, dtype=np.float32)
        self.h = C.c_void_p(self.L.aar_oracle_create(
            C.c_int(len(ci)), _ptr(ci, _ip), _ptr(Tc, _dp), _ptr(K, _dp), _ptr(d, _dp),
            C.c_int(len(mi)), _ptr(mi, _ip), _ptr(Tm, _dp),
            C.c_int(len(fi)), _ptr(fi, _ip), _ptr(Tf, _dp),
            C.c_int(int(rig.root_cam)), C.c_int(int(rig.root_marker)), C.c_float(float(rig.marker_size)),
            C.c_int64(len(df)), _ptr(df, _ip), _ptr(dc, _ip), _ptr(dm, _ip), _ptr(dxy, _fp)))
        self.nC, self.nM, self.nF = len(ci), len(mi), len(fi)
        self.set_config()

    def __del__(self):
        try:
            self.L.aar_oracle_destroy(self.h)
        except Exception:
            pass

    def set_sincos_mode(self, mode):
        self.L.aar_oracle_set_sincos_mode(C.c_int(mode))

    def set_config(self, cams=True, markers=True, objects=True, intrinsics=False, with_huber=False, huber_delta=2.5):
        self.cams, self.markers = bool(cams), bool(markers)
        self.L.aar_oracle_set_config(self.h, C.c_int(cams), C.c_int(markers), C.c_int(objects), C.c_int(intrinsics),
                                     C.c_int(with_huber), C.c_float(huber_delta))

    def set_max_iters(self, n):
        self.L.aar_oracle_set_max_iters(self.h, C.c_int(int(n)))

    def set_analytic(self, on=True):
        """analytic-Jacobian / full-FP64 variant (include/aar_analytic.h): error(), jacobian(), reduced_system() and the solves follow it."""
        self.L.aar_oracle_set_analytic(self.h, C.c_int(int(on)))

    def error_fp64_chain(self, z):
        """m - p of the restated OpenCV chain kept in double: independent of include/aar_analytic.h (no Huber)."""
        z = np.ascontiguousarray(z, dtype=np.float64); r = np.zeros(self.num_rows)
        self.L.aar_oracle_error_fp64_chain(self.h, _ptr(z, _dp), _ptr(r, _dp)); return r

    @property
    def num_vars(self): return int(self.L.aar_oracle_num_vars(self.h))
    @property
    def num_rows(self): return int(self.L.aar_oracle_num_rows(self.h))

    def observations(self):
        n = self.num_rows // 8
        f = np.zeros(n, np.int32); c = np.zeros(n, np.int32); m = np.zeros(n, np.int32)
        und = np.zeros((n, 8), np.float32); raw = np.zeros((n, 8), np.float32); hj = np.zeros(n, np.int32)
        self.L.aar_oracle_get_observations(self.h, _ptr(f, _ip), _ptr(c, _ip), _ptr(m, _ip), _ptr(und, _fp), _ptr(raw, _fp), _ptr(hj, _ip))
        return dict(frame_id=f, cam_id=c, marker_id=m, und=und, raw=raw, has_jac=hj)

    def mats2evec(self):
        z = np.zeros(self.num_vars); self.L.aar_oracle_mats2evec(self.h, _ptr(z, _dp)); return z

    def evec2mats(self, z):
        z = np.ascontiguousarray(z, dtype=np.float64)
        Tc = np.zeros((self.nC, 4, 4)); Tm = np.zeros((self.nM, 4, 4)); Tf = np.zeros((self.nF, 4, 4))
        self.L.aar_oracle_evec2mats(self.h, _ptr(z, _dp), _ptr(Tc, _dp), _ptr(Tm, _dp), _ptr(Tf, _dp))
        return Tc, Tm, Tf

    def error(self, z):
        z = np.ascontiguousarray(z, dtype=np.float64); r = np.zeros(self.num_rows)
        self.L.aar_oracle_error(self.h, _ptr(z, _dp), _ptr(r, _dp)); return r

    def jacobian(self, z):
        """CSC (colptr int64, rowidx int32, vals float64) exactly as setFromTriplets leaves it."""
        z = np.ascontiguousarray(z, dtype=np.float64)
        nnz = int(self.L.aar_oracle_jacobian(self.h, _ptr(z, _dp)))
        colptr = np.zeros(self.num_vars + 1, np.int64); rowidx = np.zeros(nnz, np.int32); vals = np.zeros(nnz)
        self.L.aar_oracle_get_jacobian(self.h, _ptr(colptr, _lp), _ptr(rowidx, _ip), _ptr(vals, _dp))
        return colptr, rowidx, vals

    def reduced_system(self, z, mu, f_lo=0, f_hi=None):
        z = np.ascontiguousarray(z, dtype=np.float64)
        n_r = 6 * (self.nC - 1 if self.cams else 0) + 6 * (self.nM - 1 if self.markers else 0)      # the hook sizes S from the Config
        S = np.zeros((n_r, n_r)); b = np.zeros(n_r); cost = C.c_double(0)
        rc = self.L.aar_oracle_reduced_system(self.h, _ptr(z, _dp), C.c_double(mu), C.c_int(f_lo), C.c_int(self.nF if f_hi is None else f_hi),
                                              _ptr(S, _dp), _ptr(b, _dp), C.byref(cost))
        if rc != 0:
            raise RuntimeError(f"oracle reduced_system failed rc={rc}")
        return S, b, cost.value

    def _solve(self, fn, z0, max_trace, *extra):
        z = np.array(z0, dtype=np.float64, copy=True); tr = np.zeros((max_trace, 6)); fc = C.c_double(0)
        it = fn(self.h, _ptr(z, _dp), C.c_int(max_trace), _ptr(tr, _dp), C.byref(fc), *extra)
        return z, fc.value, int(it), tr[:min(it, max_trace)]

    def solve_port(self, z0, max_trace=256):
        """MultiCamMapper::solve() with the restated LM loop.  trace rows: cost, mu, gain, tries, accepted, huber."""
        return self._solve(self.L.aar_oracle_solve_port, z0, max_trace)

    def solve_ref(self, z0, max_trace=256, verbose=False):
        """MultiCamMapper::solve() driving the unmodified reference sparselevmarq.h (ref build only)."""
        if not self.is_ref:
            raise RuntimeError("reference SLM build (oracle/_ref) not available")
        return self._solve(self.L.aar_oracle_solve_ref, z0, max_trace, C.c_int(int(verbose)))

    def solve(self, z0, max_trace=256):
        return self.solve_ref(z0, max_trace) if self.is_ref else self.solve_port(z0, max_trace)

    # ---- track mode (one frame against the fixed rig)
    def track_init(self, frame_id, T, det_cam, det_marker, det_xy):
        T = np.ascontiguousarray(T, dtype=np.float64)
        dc = np.ascontiguousarray(det_cam, dtype=np.int32); dm = np.ascontiguousarray(det_marker, dtype=np.int32)
        dxy = np.ascontiguousarray(det_xy, dtype=np.float32)
        rows = self.L.aar_oracle_track_init(self.h, C.c_int(int(frame_id)), _ptr(T, _dp), C.c_int64(len(dc)), _ptr(dc, _ip), _ptr(dm, _ip), _ptr(dxy, _fp))
        z = np.zeros(6); self.L.aar_oracle_track_get_z(self.h, _ptr(z, _dp))
        return int(rows), z

    def track_error(self, z, rows):
        z = np.ascontiguousarray(z, dtype=np.float64); r = np.zeros(rows)
        self.L.aar_oracle_track_error(self.h, _ptr(z, _dp), _ptr(r, _dp)); return r

    def track_port(self, z0, max_trace=64):
        return self._solve(self.L.aar_oracle_track_port, z0, max_trace)

    def track_ref(self, z0, max_trace=64):
        """MultiCamMapper::track() driving the unmodified reference sparselevmarq.h (ref build only)."""
        if not self.is_ref:
            raise RuntimeError("reference SLM build (oracle/_ref) not available")
        return self._solve(self.L.aar_oracle_track_ref, z0, max_trace)

    def track(self, z0, max_trace=64):
        return self.track_ref(z0, max_trace) if self.is_ref else self.track_port(z0, max_trace)

    def time_ref_steps(self, z0, iters):
        z = np.ascontiguousarray(z0, dtype=np.float64)
        return float(self.L.aar_oracle_time_ref_steps(self.h, _ptr(z, _dp), C.c_int(iters)))


# ---- free functions for the cv2 pin tests
def rodrigues(r, sincos_mode=0):
    L, _ = load(); L.aar_oracle_set_sincos_mode(C.c_int(sincos_mode))
    r = np.ascontiguousarray(r, dtype=np.float64); R = np.zeros(9)
    L.aar_oracle_rodrigues(_ptr(r, _dp), _ptr(R, _dp)); return R.reshape(3, 3)


def rodrigues_derivs(r, sincos_mode=1):
    """dR/dr_k (3, 3, 3) of include/aar_analytic.h at the rotation vector r."""
    L, _ = load(); L.aar_oracle_set_sincos_mode(C.c_int(sincos_mode))
    r = np.ascontiguousarray(r, dtype=np.float64); dR = np.zeros(27)
    L.aar_oracle_rodrigues_derivs(_ptr(r, _dp), _ptr(dR, _dp)); return dR.reshape(3, 3, 3)


def rodrigues_inv(R):
    L, _ = load(); R = np.ascontiguousarray(R, dtype=np.float64); r = np.zeros(3)
    L.aar_oracle_rodrigues_inv(_ptr(R, _dp), _ptr(r, _dp)); return r


def inv44(A):
    L, _ = load(); A = np.ascontiguousarray(A, dtype=np.float64); B = np.zeros((4, 4))
    L.aar_oracle_inv44(_ptr(A, _dp), _ptr(B, _dp)); return B


def mul44(A, B):
    L, _ = load(); A = np.ascontiguousarray(A, dtype=np.float64); B = np.ascontiguousarray(B, dtype=np.float64); Cc = np.zeros((4, 4))
    L.aar_oracle_mul44(_ptr(A, _dp), _ptr(B, _dp), _ptr(Cc, _dp)); return Cc


def undistort(xy, K, dist):
    L, _ = load(); xy = np.ascontiguousarray(xy, dtype=np.float32).reshape(-1, 2); out = np.zeros_like(xy)
    K = np.ascontiguousarray(K, dtype=np.float64); dist = np.ascontiguousarray(dist, dtype=np.float64)
    L.aar_oracle_undistort(C.c_int64(len(xy)), _ptr(xy, _fp), _ptr(K, _dp), _ptr(dist, _dp), _ptr(out, _fp)); return out


def sincos(x):
    L, _ = load(); s = C.c_double(0); c = C.c_double(0)
    L.aar_oracle_sincos(C.c_double(x), C.byref(s), C.byref(c)); return s.value, c.value


class InitOracle:
    """The restated Initializer (oracle/init_oracle.cpp) on flat detections in aruco.detections order."""

    def __init__(self, num_cams, K, dist, marker_size, num_frames, det_frame, det_cam, det_marker, det_xy, excluded=None,
                 threshold=2.0, consensus_max=0, sincos_mode=1, prefer_ref=True):
        self.L, _ = load(prefer_ref)
        self.L.aar_oracle_set_sincos_mode(C.c_int(sincos_mode))
        self.L.aar_init_oracle_create.restype = C.c_void_p
        self.N = len(det_frame); self.num_cams = num_cams; self.num_frames = num_frames
        K = np.ascontiguousarray(K, dtype=np.float64).reshape(num_cams, 9); dist = np.ascontiguousarray(dist, dtype=np.float64).reshape(num_cams, 5)
        df = np.ascontiguousarray(det_frame, dtype=np.int32); dc = np.ascontiguousarray(det_cam, dtype=np.int32)
        dm = np.ascontiguousarray(det_marker, dtype=np.int32); xy = np.ascontiguousarray(det_xy, dtype=np.float32).reshape(-1, 8)
        ex = np.zeros(num_cams, dtype=np.uint8)
        if excluded is not None:
            ex[list(excluded)] = 1
        self.h = C.c_void_p(self.L.aar_init_oracle_create(C.c_int(num_cams), _ptr(K, _dp), _ptr(dist, _dp), C.c_double(marker_size), C.c_int(num_frames),
                                                          C.c_int64(self.N), _ptr(df, _ip), _ptr(dc, _ip), _ptr(dm, _ip), _ptr(xy, _fp),
                                                          ex.ctypes.data_as(C.c_void_p), C.c_double(threshold), C.c_int(consensus_max)))

    def __del__(self):
        if getattr(self, "h", None):
            self.L.aar_init_oracle_destroy(self.h); self.h = None

    def obtain_pose_estimations(self):
        self.L.aar_init_oracle_obtain_pose_estimations(self.h)
        T = np.zeros((self.N, 2, 4, 4)); err = np.zeros((self.N, 2)); nc = np.zeros(self.N, dtype=np.uint8)
        self.L.aar_init_oracle_get_estimations(self.h, _ptr(T, _dp), _ptr(err, _dp), nc.ctypes.data_as(C.c_void_p))
        return T, err, nc

    def init_transforms(self):
        self.L.aar_init_oracle_init_transforms(self.h)

    def init_object_transforms(self):
        self.L.aar_init_oracle_init_object_transforms(self.h)

    def set_rig(self, cam_ids, cam_T, marker_ids, marker_T):
        ci = np.ascontiguousarray(cam_ids, dtype=np.int32); mi = np.ascontiguousarray(marker_ids, dtype=np.int32)
        cT = np.ascontiguousarray(cam_T, dtype=np.float64); mT = np.ascontiguousarray(marker_T, dtype=np.float64)
        self.L.aar_init_oracle_set_rig(self.h, C.c_int(len(ci)), _ptr(ci, _ip), _ptr(cT, _dp), C.c_int(len(mi)), _ptr(mi, _ip), _ptr(mT, _dp))

    def _map(self, fn):
        n = fn(self.h, C.c_int(0), None, None)
        ids = np.zeros(n, dtype=np.int32); T = np.zeros((n, 4, 4))
        fn(self.h, C.c_int(n), _ptr(ids, _ip), _ptr(T, _dp))
        return ids, T

    def _set(self, fn):
        n = fn(self.h, C.c_int(0), None)
        ids = np.zeros(n, dtype=np.int32)
        fn(self.h, C.c_int(n), _ptr(ids, _ip))
        return ids

    def results(self):
        L = self.L
        return dict(cam_ids=self._set(L.aar_init_oracle_cam_ids), marker_ids=self._set(L.aar_init_oracle_marker_ids),
                    root_cam=int(L.aar_init_oracle_root_cam(self.h)), root_marker=int(L.aar_init_oracle_root_marker(self.h)),
                    cams=self._map(L.aar_init_oracle_transforms_to_root_cam), markers=self._map(L.aar_init_oracle_transforms_to_root_marker),
                    objects=self._map(L.aar_init_oracle_object_transforms))

    def edges(self, cams=True):
        n = self.L.aar_init_oracle_edges(self.h, C.c_int(int(cams)), C.c_int(0), None, None, None, None)
        a = np.zeros(n, dtype=np.int32); b = np.zeros(n, dtype=np.int32); ln = np.zeros(n, dtype=np.int64); w = np.zeros(n)
        self.L.aar_init_oracle_edges(self.h, C.c_int(int(cams)), C.c_int(n), _ptr(a, _ip), _ptr(b, _ip), _ptr(ln, _lp), _ptr(w, _dp))
        return a, b, ln, w


def init_solve_pnp(size, raw8, K, dist, sincos_mode=1):
    """aruco::solvePnP_ of one detection: (T [2,4,4] float32-valued, err [2])."""
    L, _ = load()
    L.aar_oracle_set_sincos_mode(C.c_int(sincos_mode))
    raw = np.ascontiguousarray(raw8, dtype=np.float32); K = np.ascontiguousarray(K, dtype=np.float64); d = np.ascontiguousarray(dist, dtype=np.float64)
    T = np.zeros((2, 4, 4)); e = np.zeros(2)
    L.aar_init_oracle_solve_pnp(C.c_float(size), _ptr(raw, _fp), _ptr(K, _dp), _ptr(d, _dp), _ptr(T, _dp), _ptr(e, _dp))
    return T, e


def init_ippe_raw(size, raw8, K, dist):
    """intermediate values of solvePoseOfCentredSquare: normalised points, H, (Ra, ta), (Rb, tb), float errors."""
    L, _ = load()
    raw = np.ascontiguousarray(raw8, dtype=np.float32); K = np.ascontiguousarray(K, dtype=np.float64); d = np.ascontiguousarray(dist, dtype=np.float64)
    q = np.zeros(8, dtype=np.float32); H = np.zeros(9); Ra = np.zeros(9); ta = np.zeros(3); Rb = np.zeros(9); tb = np.zeros(3); er = np.zeros(2, dtype=np.float32)
    L.aar_init_oracle_ippe_raw(C.c_float(size), _ptr(raw, _fp), _ptr(K, _dp), _ptr(d, _dp), _ptr(q, _fp), _ptr(H, _dp), _ptr(Ra, _dp), _ptr(ta, _dp), _ptr(Rb, _dp), _ptr(tb, _dp), _ptr(er, _fp))
    return q, H.reshape(3, 3), Ra.reshape(3, 3), ta, Rb.reshape(3, 3), tb, er


def init_consensus(marker_size, T, T1inv, T2inv, consensus_max=0):
    L, _ = load()
    T = np.ascontiguousarray(T, dtype=np.float64); A = np.ascontiguousarray(T1inv, dtype=np.float64); B = np.ascontiguousarray(T2inv, dtype=np.float64)
    w = C.c_double(0)
    i = L.aar_init_oracle_consensus(C.c_double(marker_size), C.c_int64(len(T)), _ptr(T, _dp), _ptr(A, _dp), _ptr(B, _dp), C.c_int(consensus_max), C.byref(w))
    return int(i), w.value


def acos_shared(x):
    L, _ = load()
    L.aar_init_oracle_acos.restype = C.c_double
    return L.aar_init_oracle_acos(C.c_double(x))
