"""The lens model of the analytic mode (aar_problem_desc::lens_model = 1, DESIGN.md §6g) on the CPU.

aar_an_observation_lens (include/aar_analytic.h) is pinned against OpenCV's projectPoints (projection, intrinsics columns, dp/dXc) and
its pose columns against central differences of an independent chain built from cv2.Rodrigues and cv2.projectPoints.  With all five
coefficients 0 it is the pinhole function of the analytic mode.  tests/lens_oracle.cpp runs the unchanged oracle in this model; the
GPU tests (tests/test_gpu_lens.py) hold the device against it."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import oracle_py
from aar_b200 import synth
from conftest import ROOT, parity_record

cv2 = pytest.importorskip("cv2")

ORACLE_FLAGS = ["-std=gnu++14", "-O2", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off", "-mfma", "-fno-fast-math", "-w"]   # oracle/Makefile
_dp = ctypes.POINTER(ctypes.c_double)
_fp = ctypes.POINTER(ctypes.c_float)


def _p(a, t=_dp):
    return a.ctypes.data_as(t)


def build_lens_oracle(out_dir):
    """tests/lens_oracle.cpp (it includes oracle/mcm_oracle.cpp) -> <out_dir>/libaar_lens_oracle.so, loaded."""
    so = os.path.join(str(out_dir), "libaar_lens_oracle.so")
    subprocess.run(["/usr/bin/g++", *ORACLE_FLAGS, "-o", so, os.path.join(ROOT, "tests", "lens_oracle.cpp")], check=True)
    L = ctypes.CDLL(so)
    L.aar_oracle_create.restype = ctypes.c_void_p
    for f in ("aar_oracle_num_vars", "aar_oracle_num_rows", "aar_oracle_jacobian", "aar_lens_oracle_jacobian", "aar_lens_oracle_num_raw"):
        getattr(L, f).restype = ctypes.c_int64
    return L


class LensOracle(oracle_py.Oracle):
    """oracle_py.Oracle in the lens model: error(), jacobian() and solve_port() / solve() are those of tests/lens_oracle.cpp, the rest
    is the oracle's own code.  The intrinsics (Config) flag selects K and dist from io_vec."""

    def __init__(self, lib, rig, **kw):
        load = oracle_py.load
        oracle_py.load = lambda prefer_ref=True: (lib, False)
        try:
            super().__init__(rig, prefer_ref=False, **kw)
        finally:
            oracle_py.load = load
        df, dc, dm = (np.ascontiguousarray(a, np.int32) for a in (rig.det_frame, rig.det_cam, rig.det_marker))
        dxy = np.ascontiguousarray(rig.det_xy, np.float32)
        self._det = (df, dc, dm, dxy)
        self.L.aar_lens_oracle_attach(self.h, ctypes.c_int64(len(df)), _p(df, ctypes.POINTER(ctypes.c_int)), _p(dc, ctypes.POINTER(ctypes.c_int)),
                                      _p(dm, ctypes.POINTER(ctypes.c_int)), _p(dxy, _fp))
        assert self.L.aar_lens_oracle_num_raw(self.h) == self.num_rows

    def __del__(self):
        try:
            self.L.aar_lens_oracle_detach(self.h)
        except Exception:
            pass
        super().__del__()

    def error(self, z):
        z = np.ascontiguousarray(z, dtype=np.float64); r = np.zeros(self.num_rows)
        self.L.aar_lens_oracle_error(self.h, _p(z), _p(r)); return r

    def jacobian(self, z):
        z = np.ascontiguousarray(z, dtype=np.float64)
        nnz = int(self.L.aar_lens_oracle_jacobian(self.h, _p(z)))
        colptr = np.zeros(self.num_vars + 1, np.int64); rowidx = np.zeros(nnz, np.int32); vals = np.zeros(nnz)
        self.L.aar_oracle_get_jacobian(self.h, colptr.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), rowidx.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), _p(vals))
        return colptr, rowidx, vals

    def solve_port(self, z0, max_trace=256):
        return self._solve(self.L.aar_lens_oracle_solve_port, z0, max_trace)

    def solve(self, z0, max_trace=256):
        return self.solve_port(z0, max_trace)


@pytest.fixture(scope="module")
def lens_lib(oracle_mod, tmp_path_factory):
    return build_lens_oracle(tmp_path_factory.mktemp("lens_oracle"))


def csc_to_dense(colptr, rowidx, vals, rows):
    J = np.zeros((rows, len(colptr) - 1))
    for c in range(len(colptr) - 1):
        J[rowidx[colptr[c]:colptr[c + 1]], c] = vals[colptr[c]:colptr[c + 1]]
    return J


def _pose(rng, rot, trans):
    r = rng.normal(0, rot, 3)
    return r, cv2.Rodrigues(r)[0], np.asarray(trans, float) + rng.normal(0, 0.05, 3)


def _observation(lib, Ri, ti, r_c, Ro, to, r_o, Rm, tm, r_m, lens, h, raw):
    e = np.zeros(8); P = np.zeros(18 * 8); I = np.zeros(9 * 8)
    args = [np.ascontiguousarray(a, np.float64) for a in (Ri, ti, r_c, Ro, to, r_o, Rm, tm, r_m, lens)]
    lib.aar_lens_oracle_observation(*[_p(a) for a in args], ctypes.c_double(h), _p(np.ascontiguousarray(raw, np.float32), _fp), _p(e), _p(P), _p(I))
    return e, P.reshape(18, 8), I.reshape(9, 8)


def _corners(h):
    return np.array([[-h, h, 0], [h, h, 0], [h, -h, 0], [-h, -h, 0]], float)


def _random_case(rng, zero_dist=False):
    r_c, Rc, tc = _pose(rng, 0.3, [0.2, -0.1, 0.05])
    r_o, Ro, to = _pose(rng, 0.8, [0.0, 0.0, 1.2])
    r_m, Rm, tm = _pose(rng, 0.5, [0.05, 0.02, 0.0])
    Ri, ti = Rc.T, -Rc.T @ tc
    K = [900 + 200 * rng.random(), 600 + 80 * rng.random(), 900 + 200 * rng.random(), 340 + 40 * rng.random()]
    d = [0.0] * 5 if zero_dist else [rng.normal(0, 0.2), rng.normal(0, 0.1), rng.normal(0, 3e-3), rng.normal(0, 3e-3), rng.normal(0, 0.05)]
    raw = (np.array([640, 360] * 4) + rng.normal(0, 50, 8)).astype(np.float32)
    return dict(r_c=r_c, Rc=Rc, tc=tc, Ri=Ri, ti=ti, r_o=r_o, Ro=Ro, to=to, r_m=r_m, Rm=Rm, tm=tm, lens=np.array(K + d), raw=raw, h=0.025)


def _chain(c, h):
    """Xc of the four corners from the poses, written independently of the header (cv2.Rodrigues, 4x4 products)."""
    def T(R, t):
        M = np.eye(4); M[:3, :3] = R; M[:3, 3] = t; return M
    Tc = T(cv2.Rodrigues(c["r_c"])[0], c["tc"]); To = T(cv2.Rodrigues(c["r_o"])[0], c["to"]); Tm = T(cv2.Rodrigues(c["r_m"])[0], c["tm"])
    X = np.c_[_corners(h), np.ones(4)].T
    return (np.linalg.inv(Tc) @ To @ Tm @ X)[:3].T


def _cv2_project(Xc, lens):
    fx, cx, fy, cy = lens[:4]
    K = np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1.0]])
    p, J = cv2.projectPoints(Xc.reshape(-1, 1, 3), np.zeros(3), np.zeros(3), K, np.asarray(lens[4:], float))
    return p.reshape(-1), J


def test_lens_function_against_cv2_project_points(lens_lib):
    rng = np.random.default_rng(7)
    worst = dict(projection_px=0.0, intrinsics_rel=0.0, dp_dXc_rel=0.0)
    for _ in range(200):
        c = _random_case(rng)
        # Ri = I, ti = 0: the frame translation columns are -dp/dXc
        e, P, I = _observation(lens_lib, np.eye(3), np.zeros(3), np.zeros(3), c["Ro"], c["to"], c["r_o"], c["Rm"], c["tm"], c["r_m"], c["lens"], c["h"], c["raw"])
        c2 = dict(c); c2.update(r_c=np.zeros(3), tc=np.zeros(3))
        p, J = _cv2_project(_chain(c2, c["h"]), c["lens"])
        worst["projection_px"] = max(worst["projection_px"], np.abs((c["raw"].astype(np.float64) - e) - p).max())
        Jint = -J[:, [6, 8, 7, 9, 10, 11, 12, 13, 14]].T          # cv2: rvec tvec | fx fy | cx cy | k1 k2 p1 p2 k3
        worst["intrinsics_rel"] = max(worst["intrinsics_rel"], max(np.abs(I[k] - Jint[k]).max() / np.abs(Jint[k]).max() for k in range(9)))
        dXc = -J[:, 3:6].T
        worst["dp_dXc_rel"] = max(worst["dp_dXc_rel"], max(np.abs(P[15 + k] - dXc[k]).max() / np.abs(dXc[k]).max() for k in range(3)))
    parity_record("lens_function_vs_cv2_projectPoints", bar_px=1e-9, bar_rel=1e-9, **worst)
    assert worst["projection_px"] <= 1e-9 and worst["intrinsics_rel"] <= 1e-9 and worst["dp_dXc_rel"] <= 1e-9, worst


def test_lens_pose_columns_against_central_differences(lens_lib):
    rng = np.random.default_rng(8)
    worst = 0.0
    keys = [("r_c", 0), ("tc", 3), ("r_m", 6), ("tm", 9), ("r_o", 12), ("to", 15)]
    for _ in range(20):
        c = _random_case(rng)
        e, P, _ = _observation(lens_lib, c["Ri"], c["ti"], c["r_c"], c["Ro"], c["to"], c["r_o"], c["Rm"], c["tm"], c["r_m"], c["lens"], c["h"], c["raw"])
        Pfd = np.zeros((18, 8)); hh = 1e-6
        for key, col0 in keys:
            for k in range(3):
                cp, cm = dict(c), dict(c)
                cp[key] = c[key].copy(); cp[key][k] += hh; cm[key] = c[key].copy(); cm[key][k] -= hh
                pp, _ = _cv2_project(_chain(cp, c["h"]), c["lens"]); pm, _ = _cv2_project(_chain(cm, c["h"]), c["lens"])
                Pfd[col0 + k] = -(pp - pm) / (2 * hh)
        worst = max(worst, np.abs(P - Pfd).max() / np.abs(Pfd).max())
    parity_record("lens_pose_columns_vs_central_differences", max_rel_dev=worst, bar=5e-8)
    assert worst < 5e-8, worst                                # the bar of tests/test_analytic_cpu.py


def test_zero_coefficients_are_the_pinhole_function(lens_lib):
    rng = np.random.default_rng(9)
    for _ in range(100):
        c = _random_case(rng, zero_dist=True)
        e, P, _ = _observation(lens_lib, c["Ri"], c["ti"], c["r_c"], c["Ro"], c["to"], c["r_o"], c["Rm"], c["tm"], c["r_m"], c["lens"], c["h"], c["raw"])
        e0 = np.zeros(8); P0 = np.zeros(18 * 8)
        args = [np.ascontiguousarray(a, np.float64) for a in (c["Ri"], c["ti"], c["r_c"], c["Ro"], c["to"], c["r_o"], c["Rm"], c["tm"], c["r_m"], c["lens"][:4])]
        lens_lib.aar_lens_oracle_pinhole_observation(*[_p(a) for a in args], ctypes.c_double(c["h"]), _p(c["raw"], _fp), _p(e0), _p(P0))
        assert e.tobytes() == e0.tobytes()
        assert np.array_equal(P, P0.reshape(18, 8))           # == (a product with an exact zero may flip the sign of a zero)


@pytest.mark.parametrize("flags", [(True, True, True), (False, True, True), (True, False, True), (True, True, False)])
def test_zero_coefficients_rig_equals_the_analytic_oracle(oracle_mod, lens_lib, flags):
    """An undistorted rig (calib dist 0: the undistortion pass is the identity, so the analytic mode's corners are the raw ones): the
    lens oracle's residual and Jacobian are the analytic oracle's, including an erased duplicate."""
    rig = synth.make_rig(3, 5, 12, 6, seed=21)
    rig.det_frame = np.concatenate([rig.det_frame, rig.det_frame[[3]]]); rig.det_cam = np.concatenate([rig.det_cam, rig.det_cam[[3]]])
    rig.det_marker = np.concatenate([rig.det_marker, rig.det_marker[[3]]]); rig.det_xy = np.concatenate([rig.det_xy, rig.det_xy[[3]] + 0.25])
    a = oracle_mod.Oracle(rig, prefer_ref=False); a.set_config(cams=flags[0], markers=flags[1], objects=flags[2]); a.set_analytic(True)
    o = LensOracle(lens_lib, rig); o.set_config(cams=flags[0], markers=flags[1], objects=flags[2])
    z = a.mats2evec()
    assert o.error(z).tobytes() == a.error(z).tobytes()
    cp, ri, v = o.jacobian(z); cpa, ria, va = a.jacobian(z)
    assert np.array_equal(cp, cpa) and np.array_equal(ri, ria) and np.array_equal(v, va)


def test_lens_oracle_intrinsics_jacobian_and_solve(lens_lib):
    """The oracle's nine intrinsics columns against central differences of its own residual, and its solve lowers the cost of a
    distorted rig started from zero distortion."""
    rig = synth.make_rig(3, 6, 20, 6, seed=5, distorted=True)
    true_dist = rig.dist.copy()
    rig.dist = np.zeros_like(rig.dist)
    o = LensOracle(lens_lib, rig); o.set_config(intrinsics=True)
    z = o.mats2evec(); n = o.num_vars
    J = csc_to_dense(*o.jacobian(z), o.num_rows)
    for c in range(n - 9 * rig.C, n):
        d = np.zeros(n); hh = 1e-6 * max(1.0, abs(z[c]))
        d[c] = hh
        fd = (o.error(z + d) - o.error(z - d)) / (2 * hh)
        assert np.abs(J[:, c] - fd).max() <= 1e-6 * max(1.0, np.abs(fd).max()), c
    c0 = float(np.sum(o.error(z) ** 2))
    z_s, cost, it, tr = o.solve(z)
    assert it > 2 and cost < 0.2 * c0, (it, cost, c0)
    assert np.abs(z_s[n - 9 * rig.C:].reshape(rig.C, 9)[:, 4] - true_dist[:, 0]).max() < 0.05


@pytest.mark.parametrize("name", ["cfg1"])
def test_copied_lm_equals_the_oracle_solver(oracle_mod, lens_lib, name):
    """The LM of tests/lens_oracle.cpp (a copy of the oracle's restated loop with the intrinsics kept in its arrow system) against the
    oracle's own solver (the unmodified reference sparselevmarq.h when oracle/_ref is built, else the restated loop) on the same
    function: an undistorted rig, where the lens residual and Jacobian are the analytic mode's bit for bit."""
    rig = synth.make_config(name)
    a = oracle_mod.Oracle(rig); a.set_analytic(True)
    o = LensOracle(lens_lib, rig)
    z0 = a.mats2evec()
    rec = dict(reference_solver=bool(a.is_ref))
    for k in (1, 3, 10000):
        a.set_max_iters(k); o.set_max_iters(k)
        z_a, c_a, it_a, tr_a = a.solve(z0)
        z_o, c_o, it_o, tr_o = o.solve(z0)
        dc = abs(c_o - c_a) / c_a; dz = np.abs(z_o - z_a).max() / max(1.0, np.abs(z_a).max())
        rec[str(k)] = dict(iterations=(it_a, it_o), rel_dev_cost=dc, rel_dev_z=dz)
        assert it_a == it_o and dc <= 1e-10 and dz <= 1e-10, (k, rec[str(k)])
    parity_record("lens_oracle_lm_vs_oracle_solver", workload=name, **rec)
