"""Soft relative-pose priors between two cameras or two markers (aar_set_pair_prior, csrc/aar_pair_prior.cuh, DESIGN.md §6f); run on
the B200 with -m gpu.

The contract: a solve with pair priors is the reference's SparseLevMarq on the problem augmented by 12 rows per pair (and by the rows
of absolute priors, aar_set_prior).  The oracle's reduced system and restated LM on exactly that problem (tests/pair_prior_oracle.cpp,
PairPriorOracle of test_pair_prior_cpu.py) are the reference: the checks below are the device against the oracle with the same pairs
(and priors and mask), with the bars of test_gpu_prior.py."""
import copy
import math
import os
import re
import struct
import subprocess

import numpy as np
import pytest

from aar_b200 import synth
from conftest import ROOT, parity_record
from test_gpu_fixed import _columns, _mixed
from test_gpu_parity import _end_point_bar, _oracle_envelope, _same, _same_cost
from test_gpu_prior import _priors
from test_gpu_reduced_system import _rig
from test_pair_prior_cpu import PairPriorOracle, build_pair_oracle, moved_relative, np_rodrigues, pair_cols, pair_records, relative
from test_prior_cpu import prior_columns

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def binding():
    from aar_b200 import binding as b
    b.lib()
    return b


@pytest.fixture(scope="module")
def pair_lib(oracle_mod, tmp_path_factory):
    return build_pair_oracle(tmp_path_factory.mktemp("pair_oracle"))


def _root(rig, kind):
    ids, root = (rig.cam_ids, rig.root_cam) if kind == "cams" else (rig.marker_ids, rig.root_marker)
    return int(np.flatnonzero(np.asarray(ids) == root)[0])


def _index_pairs(rig, kind, which, seed=0):
    """index pairs of `kind`: 'all' = every unordered pair a < b; 'mixed' = pairs with the root on either side, in both index orders,
    a repeated pair and random others"""
    n = rig.C if kind == "cams" else rig.M
    if which == "all":
        return [(a, b) for a in range(n) for b in range(a + 1, n)]
    root = _root(rig, kind)
    others = [i for i in range(n) if i != root]
    lo, hi = min(others), max(others)
    out = [(root, lo), (hi, root), (lo, hi), (hi, lo), (lo, hi)]
    rng = np.random.default_rng(seed)
    for _ in range(min(12, n * (n - 1) // 2)):
        a, b = rng.choice(n, 2, replace=False)
        out.append((int(a), int(b)))
    return out


def _pairs(oracle_mod, rig, kind, which, z=None, seed=31, lo=1e2, hi=1e6):
    """(pairs, T, w) of `kind` with targets away from the relative poses at z (default z0)"""
    o = oracle_mod.Oracle(rig)
    Tc, Tm, _ = o.evec2mats(o.mats2evec() if z is None else z)
    P = _index_pairs(rig, kind, which, seed)
    T = moved_relative(Tc if kind == "cams" else Tm, P, seed)
    w = np.random.default_rng(seed + 1).uniform(lo, hi, (len(P), 2))
    return np.array(P, np.int32), T, w


def _setup(binding, oracle_mod, pair_lib, rig, cams=None, markers=None, priors=None, masks=None, with_huber=False, analytic=False):
    """device handle and oracle with the same pairs (and priors, mask)"""
    o = PairPriorOracle(pair_lib, rig)
    o.set_config(with_huber=with_huber, huber_delta=2.5)
    if analytic:
        o.set_analytic(True)
    p = binding.Problem(rig, with_huber=with_huber, analytic=analytic)
    if priors:
        p.set_prior(**priors)
        o.set_prior_columns(*prior_columns(oracle_mod, rig, **priors))
    p.set_pair_prior(cams=cams, markers=markers)
    cols, recs = [], []
    for kind, ptw in (("cams", cams), ("markers", markers)):
        if ptw is not None:
            cols.append(pair_cols(rig, kind, ptw[0])); recs.append(pair_records(ptw[1], ptw[2]))
    if cols:
        o.set_pairs(np.concatenate(cols), np.concatenate(recs))
    col = np.zeros(p.num_vars, bool)
    if masks is not None:
        p.set_fixed(*masks)
        col = _columns(p, *masks)
        o.set_fixed_columns(col)
    return p, o, col


def _compare(p, o, z, mu):
    S_g, b_g, c_g = p.reduced_system(z, mu)
    S_o, b_o, _ = o.reduced_system(z, mu)
    r = o.error(z)
    c_x = math.fsum((r * r).tolist()) + o.pair_cost(z)
    if o._w is not None:
        c_x += math.fsum((o._w * (z - o._zbar) ** 2).tolist())
    iu = np.triu_indices(p.n_r)
    dS = np.abs(S_g[iu] - S_o[iu]).max() / np.abs(S_o).max()
    db = np.abs(b_g - b_o).max() / np.abs(b_o).max()
    dc = abs(c_g - c_x) / c_x
    return dict(rel_dev_S=float(dS), rel_dev_b=float(db), rel_dev_cost=float(dc), ok=bool(dS <= 1e-12 and db <= 1e-12 and dc <= 1e-12))


# ------------------------------------------------------------------ the reduced system against the oracle with the same pairs
CASES_RS = [("C5_M29", "cams"), ("C5_M29", "markers"), ("C5_M29", "both_priors_fixed"), ("C16_M64", "cams_all"), ("C16_M64", "cams_all_huber")]


@pytest.mark.parametrize("name,kind", CASES_RS, ids=[f"{n}-{k}" for n, k in CASES_RS])
def test_reduced_system_with_pairs_matches_oracle(binding, oracle_mod, pair_lib, name, kind):
    rig = _rig(name)
    huber = kind.endswith("huber")
    if huber:                                                     # outliers, so that the Huber weights differ from 1
        rig = copy.copy(rig); rig.det_xy = rig.det_xy.copy(); rig.det_xy[::37] += 25.0
    which = "all" if "all" in kind else "mixed"
    cams = _pairs(oracle_mod, rig, "cams", which) if kind.startswith(("cams", "both")) else None
    markers = _pairs(oracle_mod, rig, "markers", which, seed=47) if kind.startswith(("markers", "both")) else None
    fixed = kind.endswith("fixed")
    p, o, col = _setup(binding, oracle_mod, pair_lib, rig, cams=cams, markers=markers, priors=_priors(oracle_mod, rig, "all") if fixed else None,
                       masks=_mixed(rig) if fixed else None, with_huber=huber)
    z0 = o.mats2evec()
    z1 = z0 + np.random.default_rng(5).normal(0, 1e-3, z0.shape)
    devs = [_compare(p, o, z, mu) for z, mu in ((z0, 5.0), (z1, 321.0))]
    parity_record("pair_prior_reduced_system_vs_oracle", rig=name, kind=kind, n_r=p.n_r, camera_pairs=0 if cams is None else len(cams[0]),
                  marker_pairs=0 if markers is None else len(markers[0]), held_columns=int(col.sum()), at_z0=devs[0], at_perturbed_z=devs[1], bar=1e-12)
    assert all(d["ok"] for d in devs), devs
    if name == "C16_M64":
        assert p.n_r == 468 and len(cams[0]) == 120


# ------------------------------------------------------------------ one and three LM iterations against the oracle's solver
CASES_LM = [("cfg1", ""), ("cfg2_distorted", ""), ("C6_M82", ""), ("cfg1", "analytic")]


def _workload(name):
    if name == "cfg2_distorted":
        return synth.make_config("cfg2", distorted=True)
    return synth.make_config(name) if name.startswith("cfg") else _rig(name)


def _both(oracle_mod, rig):
    return dict(cams=_pairs(oracle_mod, rig, "cams", "mixed"), markers=_pairs(oracle_mod, rig, "markers", "mixed", seed=47))


@pytest.mark.parametrize("name,variant", CASES_LM, ids=[n + ("-" + v if v else "") for n, v in CASES_LM])
def test_lm_iterations_with_pairs_match_oracle(binding, oracle_mod, pair_lib, name, variant):
    """C6_M82: n_r = 516, the cooperative-grid Cholesky."""
    rig = _workload(name)
    p, o, _ = _setup(binding, oracle_mod, pair_lib, rig, **_both(oracle_mod, rig), analytic=variant == "analytic")
    z0 = o.mats2evec()
    worst = 0.0
    for k in (1, 3):
        z_g, fc_g, it_g, tr_g = p.solve(z0, binding.Problem.default_params(max_iters=k, ignore_stop_rules=1))
        o.set_max_iters(k)
        z_o, fc_o, it_o, tr_o = o.solve(z0)
        dz, dc = np.abs(z_g - z_o).max() / np.abs(z_o).max(), abs(fc_g - fc_o) / fc_o
        worst = max(worst, dz, dc)
        assert it_g == it_o == k and dz <= 1e-10 and dc <= 1e-10, (k, dz, dc)
        assert abs(p.last_report.initial_cost - o.reduced_system(z0, 1.0)[2]) <= 1e-12 * p.last_report.initial_cost
    st = p.stats()
    parity_record("pair_prior_lm_iterations_vs_oracle", workload=name, variant=variant or "faithful", n_r=p.n_r, cluster_solve=st["cluster_solve"],
                  worst_rel_dev=worst, bar=1e-10)
    if name == "C6_M82":
        assert not st["cluster_solve"]


# ------------------------------------------------------------------ full solves
@pytest.mark.parametrize("name", ["cfg1", "cfg2_distorted"])
def test_full_solve_with_pairs(binding, oracle_mod, pair_lib, name):
    rig = _workload(name)
    p, o, _ = _setup(binding, oracle_mod, pair_lib, rig, **_both(oracle_mod, rig))
    z0 = o.mats2evec()
    z_g, fc_g, it_g, _ = p.solve(z0)
    z_o, fc_o, it_o, _ = o.solve(z0)
    env_c, _ = _oracle_envelope(o, z0, fc_o, z_o)
    d_cost = abs(fc_g - fc_o) / fc_o
    passes = _end_point_bar(d_cost, env_c, 2e-5)
    parity_record("pair_prior_full_solve_vs_oracle", workload=name, iterations_gpu=it_g, iterations_oracle=it_o, rel_dev_final_cost=d_cost,
                  ref_envelope_cost=env_c, passes_by=passes)
    assert abs(it_g - it_o) <= 1


# ------------------------------------------------------------------ behaviour
def test_zero_weights_held_side_and_translation_pair(binding, oracle_mod):
    rig = synth.make_config("cfg1")
    p, plain = binding.Problem(rig), binding.Problem(rig)
    z0 = p.mats2evec()
    prm = binding.Problem.default_params(max_iters=5, ignore_stop_rules=1)
    both = _both(oracle_mod, rig)
    # all weights 0: the solve without pairs
    p.set_pair_prior(**{k: (P, T, np.zeros_like(w)) for k, (P, T, w) in both.items()})
    z_p, c_p, _, _ = p.solve(z0, prm)
    z_n, c_n, _, _ = plain.solve(z0, prm)
    dz = float(np.abs(z_p - z_n).max() / np.abs(z_n).max())
    assert dz <= 3e-13 and abs(c_p - c_n) <= 1e-12 * c_n, (dz, c_p, c_n)
    # a held side stays where it is: the mask wins
    p.set_pair_prior(**both)
    P = both["cams"][0]
    held = int([i for i in P.ravel() if i != _root(rig, "cams")][0])
    masks = (np.eye(rig.C, dtype=bool)[held], None, None)
    p.set_fixed(*masks)
    col = _columns(p, *masks)
    z_h, _, _, _ = p.solve(z0, prm)
    assert col.any() and np.array_equal(z_h[col], z0[col]) and not np.array_equal(z_h[~col], z0[~col])
    p.set_fixed()
    # a translation-only pair (root, b) is the absolute translation prior on b, device against device
    root = _root(rig, "cams"); b = [i for i in range(rig.C) if i != root][1]
    Tc = p.evec2mats(z0 + np.random.default_rng(10).normal(0, 2e-3, z0.shape))[0]
    wt = 3.7e3
    q, a = binding.Problem(rig), binding.Problem(rig)
    q.set_pair_prior(cams=(np.array([[root, b]]), Tc[b][None], np.array([[0.0, wt]])))
    w = np.zeros((rig.C, 6)); w[b, 3:] = wt
    a.set_prior(cams=(Tc, w))
    S_q, b_q, c_q = q.reduced_system(z0, 5.0)
    S_a, b_a, c_a = a.reduced_system(z0, 5.0)
    iu = np.triu_indices(q.n_r)
    dS = float(np.abs(S_q[iu] - S_a[iu]).max() / np.abs(S_a).max()); db = float(np.abs(b_q - b_a).max() / np.abs(b_a).max()); dc = abs(c_q - c_a) / c_a
    z_q, f_q, _, _ = q.solve(z0, prm)
    z_a, f_a, _, _ = a.solve(z0, prm)
    dzt = float(np.abs(z_q - z_a).max() / np.abs(z_a).max())
    parity_record("pair_prior_limits", workload="cfg1", zero_weights_rel_dev_z=dz, held_side_unchanged=True, translation_pair_vs_prior=dict(
        rel_dev_S=dS, rel_dev_b=db, rel_dev_cost=dc, five_iterations_rel_dev_z=dzt), bar_zero_weights=3e-13, bar_reduced=1e-12, bar_lm=1e-10)
    assert dS <= 1e-12 and db <= 1e-12 and dc <= 1e-12 and dzt <= 1e-10 and abs(f_q - f_a) <= 1e-10 * f_a, (dS, db, dc, dzt)


def test_graph_loop_equals_host_loop_and_reads_new_targets(binding, oracle_mod, monkeypatch):
    rig = synth.make_config("cfg1")
    p, plain = binding.Problem(rig), binding.Problem(rig)
    z0 = p.mats2evec()
    prm = binding.Problem.default_params(max_iters=7, ignore_stop_rules=1)
    rec = {}
    launches = {}
    for label, seed in (("first_targets", 31), ("new_targets", 59)):
        pr = {"cams": _pairs(oracle_mod, rig, "cams", "mixed", seed=31), "markers": _pairs(oracle_mod, rig, "markers", "mixed", seed=47)}
        if label == "new_targets":                                # same pairs and count, new target values: the graph is kept and must read them
            pr = {k: (P, moved_relative(p.evec2mats(z0)[0 if k == "cams" else 1], P, seed), w) for k, (P, _, w) in pr.items()}
        p.set_pair_prior(**pr)
        monkeypatch.setenv("AAR_NO_GRAPH", "1")
        z_h, c_h, it_h, tr_h = p.solve(z0, prm)
        monkeypatch.delenv("AAR_NO_GRAPH")
        g0 = p.stats()["graph_iterations"]
        l0 = p.kernel_launches
        z_g, c_g, it_g, tr_g = p.solve(z0, prm)
        launches[label] = p.kernel_launches - l0
        st = p.stats()
        assert st["graph_loop"] and st["graph_iterations"] - g0 == 6, st
        assert it_g == it_h == 7 and _same(z_g, z_h) and abs(c_g - c_h) <= 1e-9 * c_h and np.array_equal(tr_g[:, 3:6], tr_h[:, 3:6]), (label, c_g, c_h)
        rec[label] = dict(rel_dev_z=float(np.abs(z_g - z_h).max() / np.abs(z_h).max()), rel_dev_cost=abs(c_g - c_h) / c_h, final_cost=c_g)
    assert rec["first_targets"]["final_cost"] != rec["new_targets"]["final_cost"]
    with_pairs = launches["new_targets"]
    p.set_pair_prior()                                             # cleared: the graph is captured again, without the pair kernels
    l0 = p.kernel_launches
    z_c, c_c, _, _ = p.solve(z0, prm)
    cleared = p.kernel_launches - l0
    l0 = plain.kernel_launches
    z_n, c_n, _, _ = plain.solve(z0, prm)
    never = plain.kernel_launches - l0
    cost_ok, flips = _same_cost(plain, z_c, c_c, z_n, c_n)
    parity_record("pair_prior_graph_vs_host_loop_and_clear", workload="cfg1", iterations=7, launches_with_pairs=launches, launches_after_clear=cleared,
                  launches_never_with_pairs=never, **rec)
    assert launches["first_targets"] == launches["new_targets"]
    assert cleared == never < with_pairs and p.stats()["graph_loop"], (with_pairs, cleared, never)
    assert _same(z_c, z_n) and cost_ok, flips


# ------------------------------------------------------------------ refusals and argument handling
def test_refusals(binding, oracle_mod):
    rig = synth.make_config("cfg1")
    p = binding.Problem(rig)
    z0 = p.mats2evec()
    P, T, w = _pairs(oracle_mod, rig, "cams", "mixed")
    with pytest.raises(ValueError):
        p.set_pair_prior(cams=(P[:-1], T, w))
    with pytest.raises(ValueError):
        p.set_pair_prior(markers=(P, T, np.ones((len(P), 3))))
    p.lm_begin(z0)
    with pytest.raises(binding.AarError, match="aar_lm_begin"):
        p.set_pair_prior(cams=(P, T, w))
    p.lm_end()
    for bad in ((0, rig.C), (-1, 0)):
        Q = P.copy(); Q[1] = bad
        with pytest.raises(binding.AarError, match="out of range"):
            p.set_pair_prior(cams=(Q, T, w))
    Q = P.copy(); Q[2] = (1, 1)
    with pytest.raises(binding.AarError, match="itself"):
        p.set_pair_prior(cams=(Q, T, w))
    for bad in (-1.0, np.nan, np.inf):
        v = w.copy(); v[1, 1] = bad
        with pytest.raises(binding.AarError, match="weight"):
            p.set_pair_prior(cams=(P, T, v))
    U = T.copy(); U[0, 1, 3] = np.nan
    with pytest.raises(binding.AarError, match="non-finite"):
        p.set_pair_prior(cams=(P, U, w))
    v = w.copy(); v[0] = 0.0                                       # no weight: the target is not read
    p.set_pair_prior(cams=(P, U, v))
    for label, R in (("scaled", 1.001 * T[0, :3, :3]), ("reflection", T[0, :3, :3] @ np.diag([1.0, 1.0, -1.0])), ("skewed", T[0, :3, :3] @ np_rodrigues([0, 0, 0.1]) + 1e-6)):
        U = T.copy(); U[0, :3, :3] = R
        with pytest.raises(binding.AarError, match="not a rotation"):
            p.set_pair_prior(cams=(P, U, w))
    p.set_pair_prior(cams=(P, T, w))
    # a pair whose sides have no columns (the camera group not optimised) adds nothing and launches nothing
    q = binding.Problem(rig, cams=False)
    l0 = q.kernel_launches
    S0, b0, c0 = q.reduced_system(z0[6 * (rig.C - 1):], 5.0)
    n0 = q.kernel_launches - l0
    q.set_pair_prior(cams=(P, T, w))
    l0 = q.kernel_launches
    S1, b1, c1 = q.reduced_system(z0[6 * (rig.C - 1):], 5.0)
    assert q.kernel_launches - l0 == n0 and np.abs(S1 - S0).max() <= 1e-13 * np.abs(S0).max() and abs(c1 - c0) <= 1e-13 * c0


# ------------------------------------------------------------------ the find_solution app
@pytest.fixture(scope="module")
def host_bins():
    from aar_b200 import binding
    binding.build()
    host = os.path.join(ROOT, "automatic-ar_b200", "host")
    subprocess.run(["make", "-s", "-C", host], check=True)
    return host


def _run(host_bins, folder, start, *opts):
    r = subprocess.run([os.path.join(host_bins, "find_solution"), str(folder), "0.05", "-init", start, *opts], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    return r.stdout


def _write_stereo(host_bins, path, cam_ids, Tc, root_id):
    """the reference's stereo-calibration records of T_ij = T_i^-1 T_j for every i < j, written by write_stereo_calib (read back and
    written again by solution_tool stereo)"""
    import oracle_py
    raw = path + ".in"
    with open(raw, "wb") as fh:
        fh.write(struct.pack("<Q", len(cam_ids) - 1))
        for i in range(len(cam_ids) - 1):
            fh.write(struct.pack("<iQ", int(cam_ids[i]), len(cam_ids) - 1 - i))
            for j in range(i + 1, len(cam_ids)):
                T = np.linalg.inv(Tc[i]) @ Tc[j]
                fh.write(struct.pack("<i6d", int(cam_ids[j]), *oracle_py.rodrigues_inv(np.ascontiguousarray(T[:3, :3])), *T[:3, 3]))
        fh.write(struct.pack("<i", int(root_id)))
    subprocess.run([os.path.join(host_bins, "solution_tool"), "stereo", raw, path], check=True, capture_output=True)


def _pair_dist(oracle_mod, rig, vec, Tc_ref):
    """largest distance over every camera pair i < j between the relative poses of the solution and those of Tc_ref"""
    Tc = oracle_mod.Oracle(rig).evec2mats(vec[:oracle_mod.Oracle(rig).num_vars])[0]
    P = [(i, j) for i in range(rig.C) for j in range(i + 1, rig.C)]
    return float(np.abs(relative(Tc, P) - relative(Tc_ref, P)).max())


@pytest.mark.parametrize("reject", [False, True], ids=["plain", "reject_outliers"])
def test_find_solution_stereo_prior(host_bins, oracle_mod, tmp_path, reject):
    rig = synth.make_config("cfg1")
    if reject:
        rig = copy.copy(rig); rig.det_xy = rig.det_xy.copy(); rig.det_xy[::41] += 30.0
    extra = ["-reject-outliers", "5"] if reject else []
    d0 = tmp_path / "solve"; d0.mkdir()
    init = str(d0 / "init.solution"); synth.write_solution_file(init, rig)
    _run(host_bins, d0, init)
    vec = synth.read_solution_file(str(d0 / "final.solution"))["vec"]
    o = oracle_mod.Oracle(rig)
    Tc, Tm, Tf = o.evec2mats(vec[:o.num_vars])
    solved = copy.copy(rig); solved.T_cam_init, solved.T_marker_init, solved.T_frame_init = Tc, Tm, Tf
    stereo = str(tmp_path / "stereo.calib"); _write_stereo(host_bins, stereo, rig.cam_ids, Tc, rig.root_cam)
    # the same relative poses from a solve expressed with another root camera
    other = int([i for i in range(rig.C) if rig.cam_ids[i] != rig.root_cam][0])
    Tc_other = np.stack([np.linalg.inv(Tc[other]) @ Tc[i] for i in range(rig.C)])
    stereo_other = str(tmp_path / "stereo_other_root.calib"); _write_stereo(host_bins, stereo_other, rig.cam_ids, Tc_other, rig.cam_ids[other])
    # the start: the solved rig with every non-root camera moved
    start = copy.copy(solved); start.T_cam_init = Tc.copy()
    rng = np.random.default_rng(17)
    for i in range(rig.C):
        if rig.cam_ids[i] != rig.root_cam:
            start.T_cam_init[i, :3, :3] = start.T_cam_init[i, :3, :3] @ np_rodrigues(rng.normal(0, 0.01, 3))
            start.T_cam_init[i, :3, 3] += rng.normal(0, 0.01, 3)
    start_file = str(tmp_path / "start.solution"); synth.write_solution_file(start_file, start)
    res = {}
    for label, opts in (("none", []), ("sigma_1e-3", ["-stereo-prior", stereo, "1e-3", "1e-3"]), ("sigma_1e6", ["-stereo-prior", stereo, "1e6", "1e6"]),
                        ("other_root_sigma_1e-3", ["-stereo-prior", stereo_other, "1e-3", "1e-3"])):
        d = tmp_path / label; d.mkdir()
        out = _run(host_bins, d, start_file, *opts, *extra)
        if opts:
            assert f"pair priors on {rig.C * (rig.C - 1) // 2} camera pairs" in out, out
        if reject:
            assert int(out.split("removed ")[1].split()[0]) > 0
        v = synth.read_solution_file(str(d / "final.solution"))["vec"]
        res[label] = dict(pair_dist=_pair_dist(oracle_mod, rig, v, Tc), final_cost=float(re.findall(r"final_error: (\S+)", out)[-1]))
    assert res["sigma_1e-3"]["pair_dist"] < res["none"]["pair_dist"], res
    assert res["other_root_sigma_1e-3"]["pair_dist"] < res["none"]["pair_dist"], res
    assert abs(res["sigma_1e6"]["final_cost"] - res["none"]["final_cost"]) <= 1e-6 * res["none"]["final_cost"], res
    parity_record("pair_prior_find_solution_app", reject_outliers=reject, **res)


# ------------------------------------------------------------------ sharded handles: world 2 against one GPU
def _worker(rank, world, port, out_dir):
    import sys
    sys.path.insert(0, os.path.join(ROOT, "automatic-ar_b200", "python")); sys.path.insert(0, os.path.join(ROOT, "oracle")); sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch
    import torch.distributed as dist
    import oracle_py
    from aar_b200 import binding
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    rig = synth.make_config("cfg2")
    pr = _both(oracle_py, rig)
    p = binding.Problem(rig, device=rank, rank=rank, world_size=world)
    p.set_pair_prior(**pr)
    idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        idt.copy_(torch.frombuffer(bytearray(binding.comm_unique_id()), dtype=torch.uint8))
    dist.broadcast(idt, 0)
    p.comm_init(bytes(idt.cpu().numpy().tobytes()))
    z0 = p.mats2evec()
    mu = 1234.5
    S, b, c = p.reduced_system(z0, mu)
    buf = torch.from_numpy(np.concatenate([S.ravel(), b, [c]])).cuda()
    dist.all_reduce(buf)
    buf = buf.cpu().numpy()
    z, fc, it, _ = p.solve(z0, binding.Problem.default_params(max_iters=3, ignore_stop_rules=1))
    if rank == 0:
        single = binding.Problem(rig, device=0)
        single.set_pair_prior(**pr)
        S1, b1, c1 = single.reduced_system(z0, mu)
        n = p.n_r; iu = np.triu_indices(n)
        rec = dict(reduced_system_rel_dev=np.abs(buf[:n * n].reshape(n, n)[iu] - S1[iu]).max() / np.abs(S1).max(),
                   reduced_rhs_rel_dev=np.abs(buf[n * n:n * n + n] - b1).max() / np.abs(b1).max(), cost_rel_dev=abs(buf[-1] - c1) / c1)
        z1, fc1, it1, _ = single.solve(z0, binding.Problem.default_params(max_iters=3, ignore_stop_rules=1))
        rec.update(three_iterations_rel_dev_z=np.abs(z - z1).max() / np.abs(z1).max(), three_iterations_rel_dev_cost=abs(fc - fc1) / fc1)
        parity_record("pair_prior_world2_cfg2_vs_single_gpu", **rec)
        assert rec["reduced_system_rel_dev"] <= 1e-12 and rec["reduced_rhs_rel_dev"] <= 1e-12 and rec["cost_rel_dev"] <= 1e-12, rec
        assert it == it1 == 3 and rec["three_iterations_rel_dev_z"] <= 1e-10 and rec["three_iterations_rel_dev_cost"] <= 1e-10, rec
        open(os.path.join(out_dir, "ok"), "w").write("ok")
    p.close()
    dist.destroy_process_group()


def test_sharded_pairs_match_single_gpu(oracle_mod, tmp_path):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    port = 29500 + os.getpid() % 200
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert os.path.exists(os.path.join(tmp_path, "ok"))
