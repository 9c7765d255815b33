"""Soft relative-pose priors between two cameras or two markers (aar_set_pair_prior, DESIGN.md §6f), on the CPU oracle.  A solve with
pair priors is the reference's SparseLevMarq run on the least-squares problem augmented by 12 rows per pair (a, b):
sqrt(w_rot / 2) vec(R_a^T R_b - Rbar) and sqrt(w_t) (R_a^T (t_b - t_a) - tbar).  tests/pair_prior_oracle.cpp copies the prior oracle's
reduced system and restated LM with exactly that change, and this file checks it:

- its pair rows and Jacobian against an independent numpy formulation (Rodrigues written out, central differences of the residual),
  including rotation vectors below the small-angle switch of aar_an_rodrigues_derivs;
- the rows' squared sum against the closed form w_rot (2 - 2 cos theta) + w_t |t_ab - tbar|^2;
- without pairs the copies are those of tests/prior_oracle.cpp bit for bit (with and without absolute priors and a mask);
- a translation-only pair with the root is an absolute translation prior."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

import oracle_py
from aar_b200 import synth
from conftest import ROOT, parity_record
from test_fixed_cpu import ORACLE_FLAGS
from test_prior_cpu import PriorOracle, _mask, build_prior_oracle, entity_columns, moved_targets, prior_columns, weights


def build_pair_oracle(out_dir):
    """tests/pair_prior_oracle.cpp (it includes tests/prior_oracle.cpp) -> <out_dir>/libaar_pair_oracle.so, loaded."""
    so = os.path.join(str(out_dir), "libaar_pair_oracle.so")
    subprocess.run(["/usr/bin/g++", *ORACLE_FLAGS, "-o", so, os.path.join(ROOT, "tests", "pair_prior_oracle.cpp")], check=True)
    L = ctypes.CDLL(so)
    L.aar_oracle_create.restype = ctypes.c_void_p
    for f in ("aar_oracle_num_vars", "aar_oracle_num_rows", "aar_oracle_jacobian"):
        getattr(L, f).restype = ctypes.c_int64
    return L


def pair_cols(rig, kind, pairs):
    """[n, 2] first io_vec column of each side (every group optimised; -1 for the root) of index pairs of `kind` (cams / markers)"""
    cc, cm, _ = entity_columns(rig)
    first = cc if kind == "cams" else cm
    return np.ascontiguousarray(first[np.asarray(pairs, dtype=np.int64)], dtype=np.int32).reshape(-1, 2)


def pair_records(T, w):
    """[n, 14] records (Rbar 9 | tbar 3 | w_rot w_t) of targets T [n, 4, 4] and weights w [n, 2]"""
    T = np.asarray(T, dtype=np.float64); w = np.asarray(w, dtype=np.float64)
    return np.ascontiguousarray(np.concatenate([T[:, :3, :3].reshape(-1, 9), T[:, :3, 3], w], axis=1))


class PairPriorOracle(PriorOracle):
    """PriorOracle whose reduced_system() and restated LM (solve_port, solve) also carry the pair rows of set_pairs()."""

    def __init__(self, lib, rig, **kw):
        super().__init__(lib, rig, **kw)
        self.set_pairs()

    def set_pairs(self, cols=None, rec=None):
        """cols [n, 2] io_vec columns (-1: none), rec [n, 14]; None for none"""
        if cols is None:
            self._pc = np.zeros((0, 2), np.int32); self._pr = np.zeros((0, 14))
            return
        self._pc = np.ascontiguousarray(cols, dtype=np.int32).reshape(-1, 2)
        self._pr = np.ascontiguousarray(rec, dtype=np.float64).reshape(-1, 14)
        assert len(self._pc) == len(self._pr)

    def _pairs(self):
        return ctypes.c_int(len(self._pc)), self._pc.ctypes.data_as(ctypes.c_void_p), self._pr.ctypes.data_as(ctypes.c_void_p)

    def reduced_system(self, z, mu, f_lo=0, f_hi=None):
        z = np.ascontiguousarray(z, dtype=np.float64)
        n_r = 6 * (self.nC - 1 if self.cams else 0) + 6 * (self.nM - 1 if self.markers else 0)
        S = np.zeros((n_r, n_r)); b = np.zeros(n_r); cost = ctypes.c_double(0)
        rc = self.L.aar_pair_oracle_reduced_system(self.h, self._held(), *self._prior(), *self._pairs(), oracle_py._ptr(z, oracle_py._dp), ctypes.c_double(mu),
                                                   ctypes.c_int(f_lo), ctypes.c_int(self.nF if f_hi is None else f_hi), oracle_py._ptr(S, oracle_py._dp),
                                                   oracle_py._ptr(b, oracle_py._dp), ctypes.byref(cost))
        if rc != 0:
            raise RuntimeError(f"pair oracle reduced_system failed rc={rc}")
        return S, b, cost.value

    def solve_port(self, z0, max_trace=256):
        return self._solve(lambda h, *a: self.L.aar_pair_oracle_solve_port(h, self._held(), *self._prior(), *self._pairs(), *a), z0, max_trace)

    def pair_cost(self, z):
        """the pairs' squared residual sum at z (pairs without columns left out, as the solve does)"""
        e, _ = pair_rows(self.L, self._pc, self._pr, z)
        keep = (self._pc >= 0).any(axis=1)
        return math.fsum((e[keep] ** 2).ravel().tolist())


def pair_rows(lib, cols, rec, z):
    """aar_pair_oracle_rows: e [n, 12] and J [n, 12, 12] (columns [r_a t_a | r_b t_b])"""
    cols = np.ascontiguousarray(cols, dtype=np.int32); rec = np.ascontiguousarray(rec, dtype=np.float64); z = np.ascontiguousarray(z, dtype=np.float64)
    n = len(cols)
    e = np.zeros((n, 12)); J = np.zeros((n, 12, 12))
    lib.aar_pair_oracle_rows(ctypes.c_int(n), cols.ctypes.data_as(ctypes.c_void_p), rec.ctypes.data_as(ctypes.c_void_p), oracle_py._ptr(z, oracle_py._dp),
                             ctypes.c_int(len(z)), oracle_py._ptr(e, oracle_py._dp), oracle_py._ptr(J, oracle_py._dp))
    return e, J


def relative(T, pairs):
    """T_ab = T_a^-1 T_b of index pairs over poses T [n, 4, 4]"""
    return np.stack([np.linalg.inv(T[a]) @ T[b] for a, b in pairs])


def moved_relative(T, pairs, seed, rot=0.02, trans=0.02):
    """targets away from the relative poses of T: R_ab Rodrigues(N(0, rot)), t_ab + N(0, trans)"""
    rng = np.random.default_rng(seed)
    out = relative(T, pairs)
    for k in range(len(out)):
        out[k, :3, :3] = out[k, :3, :3] @ np_rodrigues(rng.normal(0, rot, 3))
        out[k, :3, 3] += rng.normal(0, trans, 3)
    return out


# ------------------------------------------------------------------ the independent numpy formulation
def np_rodrigues(r):
    """R = I + sin(th)/th K + (1 - cos(th))/th^2 K^2, K = [r]x, with 1 - cos(th) = 2 sin^2(th/2) (no cancellation near 0)"""
    r = np.asarray(r, dtype=np.float64)
    th = math.sqrt(float(r @ r))
    K = np.array([[0, -r[2], r[1]], [r[2], 0, -r[0]], [-r[1], r[0], 0]])
    if th == 0.0:
        return np.eye(3) + K
    a = math.sin(th) / th
    b = 2.0 * math.sin(th / 2) ** 2 / (th * th)
    return np.eye(3) + a * K + b * (K @ K)


def np_pair_residual(x, rec):
    """12 residual rows of one pair from x = [r_a t_a | r_b t_b] (numpy)"""
    Ra, ta, Rb, tb = np_rodrigues(x[0:3]), x[3:6], np_rodrigues(x[6:9]), x[9:12]
    Rbar, tbar, w_rot, w_t = rec[:9].reshape(3, 3), rec[9:12], rec[12], rec[13]
    return np.concatenate([math.sqrt(w_rot / 2) * (Ra.T @ Rb - Rbar).ravel(), math.sqrt(w_t) * (Ra.T @ (tb - ta) - tbar)])


@pytest.fixture(scope="module")
def pair_lib(oracle_mod, tmp_path_factory):
    return build_pair_oracle(tmp_path_factory.mktemp("pair_oracle"))


@pytest.fixture(scope="module")
def prior_lib(oracle_mod, tmp_path_factory):
    return build_prior_oracle(tmp_path_factory.mktemp("prior_oracle"))


def test_pair_rows_against_numpy(pair_lib):
    """oracle rows and Jacobian against numpy: residual to 1e-13, J against central differences (h = 1e-6) to 1e-7 relative; rotation
    vectors of ordinary size, below the small-angle switch (|r| < 1e-5) and exactly zero"""
    rng = np.random.default_rng(21)
    cases = [("ordinary", rng.normal(0, 0.8, 12)), ("small_angle", np.concatenate([rng.normal(0, 3e-6, 3), rng.normal(0, 1, 3), rng.normal(0, 3e-6, 3), rng.normal(0, 1, 3)])),
             ("zero_rotation", np.concatenate([np.zeros(3), rng.normal(0, 1, 3), np.zeros(3), rng.normal(0, 1, 3)]))]
    rec = {}
    for label, x in cases:
        T = np.eye(4); T[:3, :3] = np_rodrigues(rng.normal(0, 0.5, 3)); T[:3, 3] = rng.normal(0, 1, 3)
        r = pair_records(T[None], [[rng.uniform(1, 1e4), rng.uniform(1, 1e4)]])[0]
        z = np.concatenate([rng.normal(0, 1, 6), x[:6], rng.normal(0, 1, 6), x[6:]])
        e, J = pair_rows(pair_lib, [[6, 18]], r[None], z)
        e_np = np_pair_residual(x, r)
        de = float(np.abs(e[0] - e_np).max())
        h = 1e-6
        Jn = np.stack([(np_pair_residual(x + h * np.eye(12)[c], r) - np_pair_residual(x - h * np.eye(12)[c], r)) / (2 * h) for c in range(12)], axis=1)
        dJ = float(np.abs(J[0] - Jn).max() / np.abs(Jn).max())
        rec[label] = dict(abs_dev_residual=de, rel_dev_jacobian=dJ)
        assert de <= 1e-13 * max(1.0, float(np.abs(e_np).max())) and dJ <= 1e-7, (label, de, dJ)
        # the structure: no translation columns in the rotation rows, none of r_b in the translation rows, +-sqrt(w_t) R_a^T
        assert not J[0, :9, 3:6].any() and not J[0, :9, 9:12].any() and not J[0, 9:, 6:9].any()
        assert np.array_equal(J[0, 9:, 3:6], -J[0, 9:, 9:12])
        # a side without columns is the identity pose (its Jacobian columns are never read; its rotation columns are zero)
        e1, J1 = pair_rows(pair_lib, [[-1, 18]], r[None], z)
        x1 = np.concatenate([np.zeros(6), x[6:]])
        assert np.abs(e1[0] - np_pair_residual(x1, r)).max() <= 1e-13 * max(1.0, float(np.abs(e1).max())) and not J1[0][:, :3].any()
    parity_record("pair_oracle_rows_vs_numpy", bar_residual=1e-13, bar_jacobian=1e-7, **rec)


def test_cost_in_closed_form(oracle_mod, pair_lib):
    """the rows' squared sum is w_rot (2 - 2 cos theta) + w_t |t_ab - tbar|^2, and the reduced system's cost grows by exactly it"""
    rig = synth.make_config("cfg1")
    o = PairPriorOracle(pair_lib, rig, prefer_ref=False)
    z0 = o.mats2evec()
    z1 = z0 + np.random.default_rng(5).normal(0, 1e-3, z0.shape)
    Tc, Tm, _ = oracle_mod.Oracle(rig).evec2mats(z1)
    cp = [(a, b) for a in range(rig.C) for b in range(rig.C) if a != b][:7]
    mp = [(0, 3), (5, 2), (1, 4)]
    Tcb, Tmb = moved_relative(Tc, cp, 1), moved_relative(Tm, mp, 2)
    wc = np.random.default_rng(3).uniform(1, 1e4, (len(cp), 2)); wm = np.random.default_rng(4).uniform(1, 1e4, (len(mp), 2))
    cols = np.concatenate([pair_cols(rig, "cams", cp), pair_cols(rig, "markers", mp)])
    recs = np.concatenate([pair_records(Tcb, wc), pair_records(Tmb, wm)])
    e, _ = pair_rows(pair_lib, cols, recs, z1)
    Tall = np.concatenate([relative(Tc, cp), relative(Tm, mp)]); Tbar = np.concatenate([Tcb, Tmb]); w = np.concatenate([wc, wm])
    closed = []
    for k in range(len(cols)):
        c = (np.trace(Tbar[k, :3, :3].T @ Tall[k, :3, :3]) - 1) / 2
        closed.append(w[k, 0] * (2 - 2 * c) + w[k, 1] * float(np.sum((Tall[k, :3, 3] - Tbar[k, :3, 3]) ** 2)))
    rows = (e ** 2).sum(axis=1)
    dk = float(np.abs(rows - closed).max() / max(closed))
    S0, b0, c0 = o.reduced_system(z1, 11.0)
    o.set_pairs(cols, recs)
    S1, b1, c1 = o.reduced_system(z1, 11.0)
    dc = abs((c1 - c0) - math.fsum(closed)) / c1
    parity_record("pair_oracle_closed_form", workload="cfg1", pairs=len(cols), rel_dev_rows=dk, rel_dev_reduced_cost=dc, bar=1e-12)
    assert dk <= 1e-12 and dc <= 1e-13, (dk, dc)
    assert not np.array_equal(S0, S1) and not np.array_equal(b0, b1)


@pytest.mark.parametrize("kind", ["plain", "priors", "priors_mask"])
def test_without_pairs_the_copies_are_the_prior_oracle(oracle_mod, pair_lib, prior_lib, kind):
    rig = synth.make_config("cfg1")
    po = PairPriorOracle(pair_lib, rig, prefer_ref=False); qo = PriorOracle(prior_lib, rig, prefer_ref=False)
    z0 = po.mats2evec()
    if kind != "plain":
        Tc, Tm, Tf = moved_targets(oracle_mod, rig, z0, 2e-3, 6)
        zbar, w = prior_columns(oracle_mod, rig, cams=(Tc, weights(rig.C, 1)), markers=(Tm, weights(rig.M, 2)), frames=(Tf, weights(rig.F, 3, 1.0, 50.0)))
        po.set_prior_columns(zbar, w); qo.set_prior_columns(zbar, w)
    if kind == "priors_mask":
        m = _mask(rig, po); po.set_fixed_columns(m); qo.set_fixed_columns(m)
    z1 = z0 + np.random.default_rng(3).normal(0, 1e-3, z0.shape)
    for f_lo, f_hi in ((0, None), (7, 20)):
        S_p, b_p, c_p = po.reduced_system(z1, 7.0, f_lo, f_hi)
        S_q, b_q, c_q = qo.reduced_system(z1, 7.0, f_lo, f_hi)
        assert S_p.tobytes() == S_q.tobytes() and b_p.tobytes() == b_q.tobytes() and c_p == c_q
    for iters in (3, 10000):
        po.set_max_iters(iters); qo.set_max_iters(iters)
        z_p, c_p, it_p, tr_p = po.solve_port(z0)
        z_q, c_q, it_q, tr_q = qo.solve_port(z0)
        assert z_p.tobytes() == z_q.tobytes() and c_p == c_q and it_p == it_q and tr_p.tobytes() == tr_q.tobytes(), iters


def test_translation_only_pair_with_root_is_absolute_prior(oracle_mod, pair_lib):
    """pair (root, b) with w_rot = 0: its rows are sqrt(w_t) (t_b - tbar), the absolute prior with rotation weights 0 and translation
    weights w_t on b"""
    rig = synth.make_config("cfg1")
    o = PairPriorOracle(pair_lib, rig, prefer_ref=False)
    z0 = o.mats2evec()
    z1 = z0 + np.random.default_rng(9).normal(0, 1e-3, z0.shape)
    root = [i for i in range(rig.C) if rig.cam_ids[i] == rig.root_cam][0]
    b = [i for i in range(rig.C) if i != root][1]
    Tc = oracle_mod.Oracle(rig).evec2mats(z0 + np.random.default_rng(10).normal(0, 2e-3, z0.shape))[0]
    wt = 3.7e3
    o.set_pairs(pair_cols(rig, "cams", [(root, b)]), pair_records(Tc[b][None], [[0.0, wt]]))
    S_p, b_p, c_p = o.reduced_system(z1, 5.0)
    o.set_pairs()
    w = np.zeros((rig.C, 6)); w[b, 3:] = wt
    o.set_prior_columns(*prior_columns(oracle_mod, rig, cams=(Tc, w)))
    S_a, b_a, c_a = o.reduced_system(z1, 5.0)
    dS = float(np.abs(S_p - S_a).max() / np.abs(S_a).max()); db = float(np.abs(b_p - b_a).max() / np.abs(b_a).max()); dc = abs(c_p - c_a) / c_a
    parity_record("pair_oracle_translation_pair_vs_absolute_prior", workload="cfg1", rel_dev_S=dS, rel_dev_b=db, rel_dev_cost=dc, bar=1e-15)
    assert dS <= 1e-15 and db <= 1e-15 and dc <= 1e-15, (dS, db, dc)
