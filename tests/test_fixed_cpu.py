"""Cameras, markers and frames held fixed (aar_set_fixed, DESIGN.md §6d), on the CPU oracle.  Holding an entity fixed is the reference's
SparseLevMarq run on the Jacobian whose columns of that entity are explicit zeros; the oracle's hook feeds its solvers that Jacobian.

- every non-root camera (marker) held through the hook is the reference's own group flag optimize_cam_poses = 0
  (optimize_marker_poses = 0) on the same poses: the zeroed rows and columns only ever add or subtract exact zeros, so the free entries
  agree to the last bits, over three LM iterations and over a full solve;
- the hook leaves the residuals alone, and a cleared mask gives the oracle of a handle that never had one, bit for bit;
- the find_solution app refuses an id it does not hold before it touches a device.

The hook is tests/fixed_oracle.cpp: the oracle's reduced system and restated LM, copied with the held columns zeroed in their
Jacobian, built here next to the unchanged oracle."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import oracle_py
from aar_b200 import synth
from conftest import ROOT, parity_record

ORACLE_FLAGS = ["-std=gnu++14", "-O2", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off", "-mfma", "-fno-fast-math", "-w"]   # oracle/Makefile


def build_fixed_oracle(out_dir):
    """tests/fixed_oracle.cpp (it includes oracle/mcm_oracle.cpp) -> <out_dir>/libaar_fixed_oracle.so, loaded."""
    so = os.path.join(str(out_dir), "libaar_fixed_oracle.so")
    subprocess.run(["/usr/bin/g++", *ORACLE_FLAGS, "-o", so, os.path.join(ROOT, "tests", "fixed_oracle.cpp")], check=True)
    L = ctypes.CDLL(so)
    L.aar_oracle_create.restype = ctypes.c_void_p
    for f in ("aar_oracle_num_vars", "aar_oracle_num_rows", "aar_oracle_jacobian"):
        getattr(L, f).restype = ctypes.c_int64
    return L


class FixedOracle(oracle_py.Oracle):
    """oracle_py.Oracle whose handle lives in the library of tests/fixed_oracle.cpp: set_fixed_columns() holds columns of io_vec in
    reduced_system() and in the restated LM (solve_port, solve); everything else is the oracle's own code."""

    def __init__(self, lib, rig, **kw):
        load = oracle_py.load
        oracle_py.load = lambda prefer_ref=True: (lib, False)
        try:
            super().__init__(rig, **kw)
        finally:
            oracle_py.load = load
        self._col = None

    def set_fixed_columns(self, col_fixed=None):
        """boolean [num_vars] (True = held), or None for none"""
        if col_fixed is None:
            self._col = None
            return
        m = np.ascontiguousarray(col_fixed, dtype=np.uint8).reshape(-1)
        if len(m) != self.num_vars:
            raise ValueError(f"col_fixed has {len(m)} entries, io_vec {self.num_vars}")
        self._col = m

    def _held(self):
        return None if self._col is None else self._col.ctypes.data_as(ctypes.c_void_p)

    def reduced_system(self, z, mu, f_lo=0, f_hi=None):
        z = np.ascontiguousarray(z, dtype=np.float64)
        n_r = 6 * (self.nC - 1 if self.cams else 0) + 6 * (self.nM - 1 if self.markers else 0)
        S = np.zeros((n_r, n_r)); b = np.zeros(n_r); cost = ctypes.c_double(0)
        rc = self.L.aar_fixed_oracle_reduced_system(self.h, self._held(), oracle_py._ptr(z, oracle_py._dp), ctypes.c_double(mu), ctypes.c_int(f_lo),
                                                    ctypes.c_int(self.nF if f_hi is None else f_hi), oracle_py._ptr(S, oracle_py._dp),
                                                    oracle_py._ptr(b, oracle_py._dp), ctypes.byref(cost))
        if rc != 0:
            raise RuntimeError(f"oracle reduced_system failed rc={rc}")
        return S, b, cost.value

    def solve_port(self, z0, max_trace=256):
        return self._solve(lambda h, *a: self.L.aar_fixed_oracle_solve_port(h, self._held(), *a), z0, max_trace)

    def solve(self, z0, max_trace=256):
        return self.solve_port(z0, max_trace)


@pytest.fixture(scope="module")
def fixed_lib(oracle_mod, tmp_path_factory):
    return build_fixed_oracle(tmp_path_factory.mktemp("fixed_oracle"))


def _port(oracle_mod, rig, **config):
    o = oracle_mod.Oracle(rig, prefer_ref=False)          # the restated SparseLevMarq of the unchanged oracle
    o.set_config(**config)
    return o


def _held_port(lib, rig, **config):
    o = FixedOracle(lib, rig, prefer_ref=False)
    o.set_config(**config)
    return o


def _round_tripped(oracle_mod, rig, group):
    """The rig with the matrices of `group` replaced by their r -> R expansion at z0: a solve that optimises a group reads its matrices
    from z, the group flag keeps the description's, and r -> R -> r -> R is not the identity.  Both sides then hold the same poses."""
    import copy
    o = _port(oracle_mod, rig)                            # evec2mats overwrites the oracle's matrices: a throwaway instance
    Tc, Tm, _ = o.evec2mats(o.mats2evec())
    r = copy.copy(rig)
    if group == "cams":
        r.T_cam_init = Tc
    else:
        r.T_marker_init = Tm
    return r


def _group_columns(rig, group):
    """io_vec columns of every non-root camera or marker (layout [cameras | markers | frames], roots left out)."""
    m = np.zeros(6 * (rig.C - 1 + rig.M - 1 + rig.F), bool)
    if group == "cams":
        m[:6 * (rig.C - 1)] = True
    else:
        m[6 * (rig.C - 1):6 * (rig.C - 1 + rig.M - 1)] = True
    return m


@pytest.mark.parametrize("group", ["cams", "markers"])
def test_hook_equals_reference_group_flag(oracle_mod, fixed_lib, group):
    rig = synth.make_config("cfg1")
    held = _held_port(fixed_lib, rig)
    flag = _port(oracle_mod, _round_tripped(oracle_mod, rig, group), cams=group != "cams", markers=group != "markers")
    z0 = held.mats2evec()
    m = _group_columns(rig, group)
    held.set_fixed_columns(m)
    zf0 = flag.mats2evec()
    assert np.array_equal(z0[~m], zf0)
    rec = {}
    for label, iters in (("3_iterations", 3), ("full_solve", 10000)):
        held.set_max_iters(iters); flag.set_max_iters(iters)
        z_h, c_h, it_h, tr_h = held.solve_port(z0)
        z_f, c_f, it_f, tr_f = flag.solve_port(zf0)
        assert it_h == it_f and (iters == 10000 or it_h == iters), (label, it_h, it_f)
        assert np.array_equal(z_h[m], z0[m]), label                                      # the held entries never move
        dz = float(np.abs(z_h[~m] - z_f).max() / np.abs(z_f).max())
        dc = float((np.abs(tr_h[:, 0] - tr_f[:, 0]) / tr_f[:, 0]).max())
        dmu = float((np.abs(tr_h[:, 1] - tr_f[:, 1]) / tr_f[:, 1]).max())
        rec[label] = dict(iterations=it_h, rel_dev_free_z=dz, rel_dev_cost_per_iteration=dc, rel_dev_mu=dmu, rel_dev_final_cost=abs(c_h - c_f) / c_f)
        assert dz <= 1e-12 and dc <= 1e-12 and dmu <= 1e-12 and abs(c_h - c_f) <= 1e-12 * c_f, (label, rec[label])
    parity_record("fixed_hook_vs_reference_group_flag", group=group, workload="cfg1", bar=1e-12, **rec)


def test_hook_leaves_residuals_and_cleared_mask_is_the_plain_oracle(oracle_mod, fixed_lib):
    rig = synth.make_config("cfg1")
    plain = _port(oracle_mod, rig)
    o = _held_port(fixed_lib, rig)
    z0 = plain.mats2evec()
    z1 = z0 + np.random.default_rng(3).normal(0, 1e-3, z0.shape)
    n_r = 6 * (rig.C - 1 + rig.M - 1)
    m = np.zeros(o.num_vars, bool)
    m[6:12] = True                                        # the second non-root camera
    m[6 * (rig.C - 1) + 12:6 * (rig.C - 1) + 18] = True   # a marker
    m[n_r + 6 * 17:n_r + 6 * 19] = True                   # two frames
    with pytest.raises(ValueError):
        o.set_fixed_columns(m[:-1])
    o.set_fixed_columns(m)
    assert o.error(z1).tobytes() == plain.error(z1).tobytes()
    S, b, c = o.reduced_system(z1, 7.0)
    S_p, b_p, c_p = plain.reduced_system(z1, 7.0)
    mr = m[:n_r]
    assert c == c_p and not S[mr].any() and not S[:, mr].any() and not b[mr].any()
    assert np.abs(S_p[mr]).max() > 0 and np.abs(b_p[mr]).max() > 0
    o.set_max_iters(3); plain.set_max_iters(3)
    z_m, _, _, _ = o.solve_port(z0)
    assert np.array_equal(z_m[m], z0[m]) and not np.array_equal(z_m[~m], z0[~m])
    o.set_fixed_columns(None)
    S_c, b_c, c_c = o.reduced_system(z1, 7.0)
    assert S_c.tobytes() == S_p.tobytes() and b_c.tobytes() == b_p.tobytes() and c_c == c_p
    z_c, fc_c, it_c, tr_c = o.solve_port(z0)
    z_p, fc_p, it_p, tr_p = plain.solve_port(z0)
    assert z_c.tobytes() == z_p.tobytes() and fc_c == fc_p and it_c == it_p and tr_c.tobytes() == tr_p.tobytes()


def test_find_solution_refuses_an_id_it_does_not_hold(tmp_path):
    from aar_b200 import binding
    binding.build()
    host = os.path.join(ROOT, "automatic-ar_b200", "host")
    subprocess.run(["make", "-s", "-C", host], check=True)
    rig = synth.make_rig(C=3, M=5, F=12, obs_per_frame=5.0, seed=4)
    a = str(tmp_path / "a.solution")
    synth.write_solution_file(a, rig)
    usage = subprocess.run([os.path.join(host, "find_solution")], capture_output=True, text=True).stdout
    assert all(o in usage for o in ("-fix-cams", "-fix-markers", "-fix-frames"))
    for opt, bad in (("-fix-cams", max(rig.cam_ids) + 1), ("-fix-markers", max(rig.marker_ids) + 7), ("-fix-frames", max(rig.frame_ids) + 1)):
        r = subprocess.run([os.path.join(host, "find_solution"), str(tmp_path), "0.05", "-init", a, opt, str(bad)], capture_output=True, text=True)
        assert r.returncode == 2 and "set_fixed_" in r.stderr and str(bad) in r.stderr, (opt, r.returncode, r.stderr)
    assert not os.path.exists(tmp_path / "final.solution")
