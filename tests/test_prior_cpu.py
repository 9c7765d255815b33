"""Soft pose priors (aar_set_prior, DESIGN.md §6e), on the CPU oracle.  A solve with priors is the reference's SparseLevMarq run on the
augmented least-squares problem: for every column c of io_vec with a weight w > 0 one residual row sqrt(w) (z - zbar) is appended, with
the Jacobian entry sqrt(w) in column c.  tests/prior_oracle.cpp copies the oracle's reduced system and restated LM with exactly that
change, and this file checks the copies:

- without priors they are the copies of tests/fixed_oracle.cpp bit for bit (reduced system and solve, with and without a mask);
- their cost is the oracle's reprojection sum plus the closed form sum w (z - zbar)^2;
- camera and marker priors add diag(w) to S and -w (z - zbar) to b, nothing else;
- their frame rule against an independent construction: the oracle's Jacobian and residuals with the prior rows stacked under them
  in scipy, frames eliminated in numpy."""
import copy
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

import oracle_py
from aar_b200 import synth
from conftest import ROOT, parity_record
from test_fixed_cpu import ORACLE_FLAGS, FixedOracle, build_fixed_oracle


def build_prior_oracle(out_dir):
    """tests/prior_oracle.cpp (it includes oracle/mcm_oracle.cpp) -> <out_dir>/libaar_prior_oracle.so, loaded."""
    so = os.path.join(str(out_dir), "libaar_prior_oracle.so")
    subprocess.run(["/usr/bin/g++", *ORACLE_FLAGS, "-o", so, os.path.join(ROOT, "tests", "prior_oracle.cpp")], check=True)
    L = ctypes.CDLL(so)
    L.aar_oracle_create.restype = ctypes.c_void_p
    for f in ("aar_oracle_num_vars", "aar_oracle_num_rows", "aar_oracle_jacobian"):
        getattr(L, f).restype = ctypes.c_int64
    return L


class PriorOracle(FixedOracle):
    """FixedOracle whose reduced_system() and restated LM (solve_port, solve) run on the problem augmented by the priors of
    set_prior_columns(); held columns (set_fixed_columns) combine with them."""

    def __init__(self, lib, rig, **kw):
        super().__init__(lib, rig, **kw)
        self._zbar = self._w = None

    def set_prior_columns(self, zbar=None, w=None):
        """zbar, w [num_vars] (w = 0: no prior on that column), or None for none"""
        if w is None:
            self._zbar = self._w = None
            return
        self._zbar = np.ascontiguousarray(zbar, dtype=np.float64).reshape(-1)
        self._w = np.ascontiguousarray(w, dtype=np.float64).reshape(-1)
        assert len(self._zbar) == len(self._w) == self.num_vars

    def _prior(self):
        if self._w is None:
            return None, None
        return self._zbar.ctypes.data_as(ctypes.c_void_p), self._w.ctypes.data_as(ctypes.c_void_p)

    def reduced_system(self, z, mu, f_lo=0, f_hi=None):
        z = np.ascontiguousarray(z, dtype=np.float64)
        n_r = 6 * (self.nC - 1 if self.cams else 0) + 6 * (self.nM - 1 if self.markers else 0)
        S = np.zeros((n_r, n_r)); b = np.zeros(n_r); cost = ctypes.c_double(0)
        rc = self.L.aar_prior_oracle_reduced_system(self.h, self._held(), *self._prior(), oracle_py._ptr(z, oracle_py._dp), ctypes.c_double(mu),
                                                    ctypes.c_int(f_lo), ctypes.c_int(self.nF if f_hi is None else f_hi), oracle_py._ptr(S, oracle_py._dp),
                                                    oracle_py._ptr(b, oracle_py._dp), ctypes.byref(cost))
        if rc != 0:
            raise RuntimeError(f"prior oracle reduced_system failed rc={rc}")
        return S, b, cost.value

    def solve_port(self, z0, max_trace=256):
        return self._solve(lambda h, *a: self.L.aar_prior_oracle_solve_port(h, self._held(), *self._prior(), *a), z0, max_trace)


# ------------------------------------------------------------------ priors by entity -> by column of io_vec
def entity_columns(rig):
    """first io_vec column of every camera / marker / frame with every group optimised ([cameras | markers | frames], roots left
    out: -1), as aar_index_maps reports them"""
    nrc, nrm = rig.C - 1, rig.M - 1
    cc = np.full(rig.C, -1); cm = np.full(rig.M, -1)
    cc[[i for i in range(rig.C) if rig.cam_ids[i] != rig.root_cam]] = 6 * np.arange(nrc)
    cm[[j for j in range(rig.M) if rig.marker_ids[j] != rig.root_marker]] = 6 * (nrc + np.arange(nrm))
    return cc, cm, 6 * (nrc + nrm) + 6 * np.arange(rig.F)


def target_rig(rig, Tc, Tm, Tf):
    r = copy.copy(rig)
    r.T_cam_init, r.T_marker_init, r.T_frame_init = Tc, Tm, Tf
    return r


def prior_columns(oracle_mod, rig, cams=None, markers=None, frames=None):
    """(zbar, w) [num_vars] of entity priors given as (T [n, 4, 4], w [n, 6]) pairs (None = none of that kind).  zbar is the oracle's
    R -> r of the targets (an oracle built on the target matrices), the conversion aar_set_prior makes."""
    T = [rig.T_cam_init, rig.T_marker_init, rig.T_frame_init]
    for k, tw in enumerate((cams, markers, frames)):
        if tw is not None:
            T[k] = tw[0]
    zbar = oracle_mod.Oracle(target_rig(rig, *T)).mats2evec()
    w = np.zeros_like(zbar)
    for tw, first in zip((cams, markers, frames), entity_columns(rig)):
        if tw is None:
            continue
        for i, c in enumerate(first):
            if c >= 0:
                w[c:c + 6] = tw[1][i]
    return zbar, w


def moved_targets(oracle_mod, rig, z, scale, seed):
    """target matrices away from z: the expansion of z + N(0, scale) (so that z - zbar and the gradient terms are not zero)"""
    rng = np.random.default_rng(seed)
    return oracle_mod.Oracle(rig).evec2mats(z + rng.normal(0, scale, z.shape))


def weights(n, seed, lo=0.5, hi=2e3):
    """per-entity information weights [n, 6], a few components 0"""
    w = np.random.default_rng(seed).uniform(lo, hi, (n, 6))
    w[::5, 2] = 0.0
    return w


@pytest.fixture(scope="module")
def prior_lib(oracle_mod, tmp_path_factory):
    return build_prior_oracle(tmp_path_factory.mktemp("prior_oracle"))


@pytest.fixture(scope="module")
def fixed_lib(oracle_mod, tmp_path_factory):
    return build_fixed_oracle(tmp_path_factory.mktemp("fixed_oracle"))


def _mask(rig, o):
    m = np.zeros(o.num_vars, bool)
    cc, cm, cf = entity_columns(rig)
    m[cc[cc >= 0][1]:cc[cc >= 0][1] + 6] = True
    m[cm[cm >= 0][2]:cm[cm >= 0][2] + 6] = True
    m[cf[5]:cf[5] + 6] = True
    return m


@pytest.mark.parametrize("masked", [False, True], ids=["no_mask", "mask"])
def test_without_priors_the_copies_are_the_fixed_oracle(oracle_mod, prior_lib, fixed_lib, masked):
    rig = synth.make_config("cfg1")
    po = PriorOracle(prior_lib, rig, prefer_ref=False); fo = FixedOracle(fixed_lib, rig, prefer_ref=False)
    if masked:
        m = _mask(rig, po); po.set_fixed_columns(m); fo.set_fixed_columns(m)
    z0 = po.mats2evec()
    z1 = z0 + np.random.default_rng(3).normal(0, 1e-3, z0.shape)
    for f_lo, f_hi in ((0, None), (7, 20)):
        S_p, b_p, c_p = po.reduced_system(z1, 7.0, f_lo, f_hi)
        S_f, b_f, c_f = fo.reduced_system(z1, 7.0, f_lo, f_hi)
        assert S_p.tobytes() == S_f.tobytes() and b_p.tobytes() == b_f.tobytes() and c_p == c_f
    for iters in (3, 10000):
        po.set_max_iters(iters); fo.set_max_iters(iters)
        z_p, c_p, it_p, tr_p = po.solve_port(z0)
        z_f, c_f, it_f, tr_f = fo.solve_port(z0)
        assert z_p.tobytes() == z_f.tobytes() and c_p == c_f and it_p == it_f and tr_p.tobytes() == tr_f.tobytes(), iters


def test_cost_and_rig_terms_in_closed_form(oracle_mod, prior_lib):
    """cost = reprojection sum + sum w (z - zbar)^2; camera / marker priors add diag(w) to S and -w (z - zbar) to b"""
    rig = synth.make_config("cfg1")
    o = PriorOracle(prior_lib, rig, prefer_ref=False)
    z0 = o.mats2evec()
    z1 = z0 + np.random.default_rng(5).normal(0, 1e-3, z0.shape)
    Tc, Tm, Tf = moved_targets(oracle_mod, rig, z0, 2e-3, 6)
    n_r = 6 * (rig.C - 1 + rig.M - 1)
    S0, b0, c0 = o.reduced_system(z1, 11.0)
    rec = {}
    for label, kw in (("rig", dict(cams=(Tc, weights(rig.C, 1)), markers=(Tm, weights(rig.M, 2)))),
                      ("all", dict(cams=(Tc, weights(rig.C, 1)), markers=(Tm, weights(rig.M, 2)), frames=(Tf, weights(rig.F, 3, 1.0, 50.0))))):
        zbar, w = prior_columns(oracle_mod, rig, **kw)
        o.set_prior_columns(zbar, w)
        S, b, c = o.reduced_system(z1, 11.0)
        r = o.error(z1)
        c_x = math.fsum((r * r).tolist()) + math.fsum((w * (z1 - zbar) ** 2).tolist())
        dc = abs(c - c_x) / c_x
        assert dc <= 1e-12, (label, dc)
        rec[label] = dict(rel_dev_cost=dc)
        if label == "rig":
            assert not w[n_r:].any() and w[:n_r].any()
            dS = np.abs(S - (S0 + np.diag(w[:n_r]))).max() / np.abs(S0).max()
            db = np.abs(b - (b0 - w[:n_r] * (z1[:n_r] - zbar[:n_r]))).max() / np.abs(b0).max()
            rec[label].update(rel_dev_S=float(dS), rel_dev_b=float(db))
            assert dS <= 1e-15 and db <= 1e-15, rec
    # a target equal to the start matrix: z - zbar = 0 exactly at z0
    zbar, w = prior_columns(oracle_mod, rig, cams=(rig.T_cam_init, weights(rig.C, 1)))
    assert np.array_equal(zbar, z0)
    parity_record("prior_oracle_closed_form", workload="cfg1", bar_cost=1e-12, bar_rig_S_b=1e-15, **rec)


def test_frame_rule_against_stacked_jacobian(oracle_mod, prior_lib):
    """priors on cameras, markers and every frame of a small rig: the copy's S and b against the frame elimination of the oracle's
    Jacobian with the prior rows stacked under it (scipy), formed in numpy"""
    import scipy.sparse as sp
    rig = synth.make_rig(C=3, M=5, F=12, obs_per_frame=5.0, seed=4)
    o = PriorOracle(prior_lib, rig, prefer_ref=False)
    z0 = o.mats2evec()
    z = z0 + np.random.default_rng(8).normal(0, 1e-3, z0.shape)
    Tc, Tm, Tf = moved_targets(oracle_mod, rig, z0, 2e-3, 9)
    zbar, w = prior_columns(oracle_mod, rig, cams=(Tc, weights(rig.C, 1)), markers=(Tm, weights(rig.M, 2)), frames=(Tf, weights(rig.F, 3, 1.0, 50.0)))
    o.set_prior_columns(zbar, w)
    mu = 3.0
    colptr, rowidx, vals = o.jacobian(z)
    n = o.num_vars
    J = sp.csc_matrix((vals, rowidx, colptr), shape=(o.num_rows, n))
    cols = np.flatnonzero(w > 0)
    P = sp.csr_matrix((np.sqrt(w[cols]), (np.arange(len(cols)), cols)), shape=(len(cols), n))
    Ja = sp.vstack([J, P]).toarray()
    x = np.concatenate([o.error(z), np.sqrt(w[cols]) * (z[cols] - zbar[cols])])
    A, B = Ja.T @ Ja, -Ja.T @ x
    n_r = 6 * (rig.C - 1 + rig.M - 1)
    S, b = A[:n_r, :n_r].copy(), B[:n_r].copy()
    for f in range(rig.F):
        s = slice(n_r + 6 * f, n_r + 6 * f + 6)
        D = A[s, s] + mu * np.eye(6)
        S -= A[:n_r, s] @ np.linalg.solve(D, A[s, :n_r])
        b -= A[:n_r, s] @ np.linalg.solve(D, B[s])
    S_o, b_o, c_o = o.reduced_system(z, mu)
    dS = np.abs(S_o - S).max() / np.abs(S).max()
    db = np.abs(b_o - b).max() / np.abs(b).max()
    dc = abs(c_o - x @ x) / (x @ x)
    parity_record("prior_oracle_frame_rule_vs_stacked_jacobian", rig="C3_M5_F12", rel_dev_S=float(dS), rel_dev_b=float(db), rel_dev_cost=float(dc), bar=1e-12)
    assert dS <= 1e-12 and db <= 1e-12 and dc <= 1e-12, (dS, db, dc)
    # shards: the frame ranges [0, 5) and [5, F) add up to the whole, the rig terms counted once (f_lo == 0)
    S1, b1, c1 = o.reduced_system(z, mu, 0, 5)
    S2, b2, c2 = o.reduced_system(z, mu, 5, rig.F)
    assert np.abs(S1 + S2 - S_o).max() <= 1e-13 * np.abs(S_o).max() and np.abs(b1 + b2 - b_o).max() <= 1e-13 * np.abs(b_o).max()
    assert abs(c1 + c2 - c_o) <= 1e-13 * c_o
