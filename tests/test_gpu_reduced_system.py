"""The reduced system and its dense solve at the sizes the benchmark runs (run on the B200 with -m gpu).

Every LM try ends in the frame elimination (k_schur_prepare + k_schur_syrk, output tiles of 16 x 16 blocks) and a dense Cholesky of
the reduced system: k_reduced_solve_cluster2 for up to 16 block rows of 32, the cooperative-grid k_reduced_solve beyond.  The rigs
below sit on the boundaries of those kernels (one tile, a partial tile, several full tiles, the largest cluster, the first
cooperative size, more block rows than SMs) and of the assembly (accumulators past the shared-memory limit, no camera x marker
replicas).  The stats bits of aar_problem_stats say which path ran, so a rig that lands on the wrong side of a threshold fails.

- S, b and the cost against the oracle's frame elimination;
- the step of one LM try against a high-precision solve of the same S + mu I (backward and forward error), on both Cholesky kernels;
- one and three LM iterations against the oracle's solver, the intrinsics block beyond one tile, the graph-resident loop with the
  16-CTA cluster and the cooperative launch inside;
- several live handles of different sizes in one process: the shared-memory caps of the kernels are process-wide for a device, so
  a second handle must not break the launches of the first, nor the graph the first one captured."""
import copy
import functools
import math

import numpy as np
import pytest

from aar_b200 import synth
from conftest import parity_record
from test_gpu_parity import _same, _same_cost

pytestmark = pytest.mark.gpu

U = 2.0 ** -53                  # unit roundoff of float64
SY_TB, SY_FB, CH_NB = 16, 4, 32  # blocks per SYRK tile side, frames per SYRK pipeline stage, rows per Cholesky block row (csrc/)


@pytest.fixture(scope="module")
def binding():
    from aar_b200 import binding as b
    b.lib()
    return b


@functools.lru_cache(maxsize=None)
def _num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _big_M(C=4):
    """Markers of the rig whose reduced system has more block rows of 32 than the device has SMs: 6 (C - 1 + M - 1) > 32 SMs
    (M = 788 on 148 SMs).  Its marker accumulators (224 B per block) no longer fit next to the float32 staging ring of k_asm_mruns."""
    nb = 32 * _num_sms() // 6 + 1
    return max(nb - (C - 1) + 1, 770)


# name -> make_rig arguments.  F is not a multiple of SY_FB (the last SYRK pipeline batch is partial); obs_per_frame is high
# enough that most markers are seen.
RIGS = {
    "C2_M16": dict(C=2, M=16, F=15, obs_per_frame=16.0),        # nb 16, n_r 96: one full tile; F <= 16: one SYRK chunk
    "C3_M16": dict(C=3, M=16, F=61, obs_per_frame=24.0),        # nb 17, n_r 102: a second tile of one block; last Cholesky block of 6 rows
    "C5_M29": dict(C=5, M=29, F=61, obs_per_frame=40.0),        # nb 32, n_r 192: two full tiles
    "C6_M29": dict(C=6, M=29, F=61, obs_per_frame=40.0),        # nb 33, n_r 198: three tiles
    "C20_M12": dict(C=20, M=12, F=41, obs_per_frame=60.0),      # markers=False: nb 19, two camera tiles
    "C16_M64": dict(C=16, M=64, F=61, obs_per_frame=128.0),     # nb 78, n_r 468: the benchmark's (cfg4) shape
    "C16_M66": dict(C=16, M=66, F=61, obs_per_frame=128.0),     # nb 80, n_r 480: five full tiles, 15 full Cholesky blocks
    "C6_M81": dict(C=6, M=81, F=61, obs_per_frame=60.0),        # nb 85, n_r 510: 16 block rows, the largest cluster
    "C6_M82": dict(C=6, M=82, F=61, obs_per_frame=60.0),        # nb 86, n_r 516: the first size on the cooperative kernel
    "C4_Mbig": dict(C=4, M=None, F=49, obs_per_frame=160.0),    # nb > 32 SMs / 6: cooperative grid loop, global-RED assembly
    "C100_M300": dict(C=100, M=300, F=22, obs_per_frame=500.0),  # nb 398: nrc nrm 36 x 32 replicas > 256 MB, no replicas
}


@functools.lru_cache(maxsize=None)
def _rig(name):
    kw = dict(RIGS[name])
    if kw["M"] is None:
        kw["M"] = _big_M(kw["C"])
    F = kw.pop("F")
    for f in range(F, F + 8):              # frames with fewer than two detections are dropped: keep the count off a multiple of 4
        rig = synth.make_rig(F=f, seed=41, **kw)
        if rig.F % SY_FB:
            return rig
    raise AssertionError(name)


def _oracle(oracle_mod, rig, cams=True, markers=True, with_huber=False, intrinsics=False):
    o = oracle_mod.Oracle(rig)
    o.set_config(cams=cams, markers=markers, with_huber=with_huber, huber_delta=2.5, intrinsics=intrinsics)
    return o


def _problem(binding, monkeypatch, rig, env=(), **kw):
    """A handle created with the switches `env` set (aar_problem_create reads them)."""
    for k in env:
        monkeypatch.setenv(k, "1")
    try:
        return binding.Problem(rig, **kw)
    finally:
        for k in env:
            monkeypatch.delenv(k)


def _expect_replicas(rig, cams, markers):
    nrc, nrm = (rig.C - 1) * cams, (rig.M - 1) * markers
    return bool(cams and markers and 0 < nrc * nrm * 36 * 32 * 8 <= 256 << 20)


def _syrk_shape(n_blocks, F):
    """Tiles per side and frame chunks of k_schur_syrk (schur_eliminate in aar_cuda.cu)."""
    ts = (n_blocks + SY_TB - 1) // SY_TB
    return ts, max(1, min((2 * 2 * _num_sms()) // (ts * (ts + 1) // 2), (F + 4 * SY_FB - 1) // (4 * SY_FB)))


def _compare_reduced_system(p, o, z, mu):
    """Problem.reduced_system against the oracle's frame elimination: the bars of test_tensor_core_assembly_matches_oracle.  The cost
    is compared with the exactly rounded sum of the squares of the oracle's residuals (bit-exact with the device's): the oracle's own
    running sum drifts from it by up to 4e-13 relative over the ~60 k residual rows of these rigs."""
    S_g, b_g, c_g = p.reduced_system(z, mu)
    S_o, b_o, c_o = o.reduced_system(z, mu)
    assert S_g.shape == S_o.shape and len(b_g) == p.n_r > 0
    r = o.error(z)
    c_x = math.fsum((r * r).tolist())
    iu = np.triu_indices(p.n_r)
    dS = np.abs(S_g[iu] - S_o[iu]).max() / np.abs(S_o).max()
    db = np.abs(b_g - b_o).max() / np.abs(b_o).max()
    dc = abs(c_g - c_x) / c_x
    return dict(rel_dev_S=float(dS), rel_dev_b=float(db), rel_dev_cost=float(dc), oracle_running_sum_rel_dev_cost=float(abs(c_o - c_x) / c_x),
                ok=bool(dS <= 1e-12 and db <= 1e-12 and dc <= 1e-13))


# ------------------------------------------------------------------ a. assembly and Schur complement against the oracle
CASES_A = [("C2_M16", ""), ("C3_M16", ""), ("C5_M29", ""), ("C6_M29", ""), ("C6_M29", "no_cams"), ("C20_M12", "no_markers"),
           ("C16_M64", ""), ("C16_M64", "huber"), ("C16_M66", ""), ("C6_M81", ""), ("C6_M82", ""), ("C4_Mbig", ""), ("C4_Mbig", "exact"),
           ("C100_M300", "")]


@pytest.mark.parametrize("name,flags", CASES_A, ids=[n + ("-" + f if f else "") for n, f in CASES_A])
def test_reduced_system_matches_oracle_multi_tile(binding, oracle_mod, monkeypatch, name, flags):
    rig = _rig(name)
    cams, markers, huber = flags != "no_cams", flags != "no_markers", flags == "huber"
    if huber:                                                     # outliers, so that the Huber weights differ from 1
        rig = copy.copy(rig); rig.det_xy = rig.det_xy.copy(); rig.det_xy[::37] += 25.0
    o = _oracle(oracle_mod, rig, cams=cams, markers=markers, with_huber=huber)
    p = _problem(binding, monkeypatch, rig, env=("AAR_FORCE_EXACT_STAGING",) if flags == "exact" else (), cams=cams, markers=markers, with_huber=huber)
    nb = p.n_r // 6
    z0 = o.mats2evec()
    z1 = z0 + np.random.default_rng(5).normal(0, 1e-3, z0.shape)
    devs = [_compare_reduced_system(p, o, z, mu) for z, mu in ((z0, 5.0), (z1, 321.0))]
    st = p.stats()
    # paths of the assembly: shared-memory accumulators unless the marker accumulators outgrow the staging ring's neighbour
    expect_smem = name != "C4_Mbig"
    expect_rep = _expect_replicas(rig, cams, markers)
    tiles, chunks = _syrk_shape(nb, rig.F)
    parity_record("reduced_system_multi_tile_vs_oracle", rig=name, flags=flags, C=rig.C, M=rig.M, F=rig.F, observations=p.num_obs, n_r=p.n_r,
                  syrk_tiles_per_side=tiles, syrk_chunks=chunks, smem_accumulators=st["smem_accumulators"], cm_replicas=st["cm_replicas"],
                  at_z0=devs[0], at_perturbed_z=devs[1], bar_S_b=1e-12, bar_cost=1e-13)
    assert st["smem_accumulators"] == expect_smem and st["cm_replicas"] == expect_rep, (st, expect_smem, expect_rep)
    if name == "C2_M16":
        assert tiles == 1 and chunks == 1
    assert all(d["ok"] for d in devs), devs


# ------------------------------------------------------------------ b. the dense solve, checked on its own
def _mu0(o, z0, tau=1.0):
    """mu0 = tau max diag(J^T J) (sparselevmarq.h:369-377) from the oracle's bit-exact Jacobian: column sums of squares."""
    colptr, _, vals = o.jacobian(z0)
    cols = np.repeat(np.arange(len(colptr) - 1), np.diff(colptr))
    return tau * np.bincount(cols, weights=vals * vals, minlength=len(colptr) - 1).max()


def _ld_residual(A, x, b, rows=1024):
    """b - A x accumulated in long double, by row blocks."""
    xl = x.astype(np.longdouble); r = np.empty(len(b), np.longdouble)
    for i in range(0, len(b), rows):
        r[i:i + rows] = b[i:i + rows].astype(np.longdouble) - A[i:i + rows].astype(np.longdouble) @ xl
    return r


def _check_one_step(binding, p, o, expect_cluster):
    """One LM try: the reduced step delta_r = z1[:n_r] - z0[:n_r] against S + mu0 I of the same handle.  The step is recovered from
    z1 = fl(z0 + delta), which rounds it to the ulp of z (|error_i| <= u max|z1|): both bars add what that rounding can account for."""
    import scipy.linalg
    z0 = o.mats2evec()
    z1, _, it, tr = p.solve(z0, binding.Problem.default_params(max_iters=1, ignore_stop_rules=1))
    assert it == 1 and tr[0, 3] == 1 and tr[0, 4] == 1, tr               # one try, accepted: z1 carries the step of mu0
    st = p.stats()
    assert st["cluster_solve"] == expect_cluster, (st, expect_cluster)
    n_r = p.n_r
    d = z1[:n_r] - z0[:n_r]
    mu0 = _mu0(o, z0)
    S, b, _ = p.reduced_system(z0, mu0)                                  # mu on the frame blocks only: the solve adds it to the reduced diagonal
    A = np.triu(S) + np.triu(S, 1).T + mu0 * np.eye(n_r)
    nA, nd, nb_ = np.abs(A).sum(axis=1).max(), np.abs(d).max(), np.abs(b).max()
    rounding = U * np.abs(z1[:n_r]).max()                                # bound of the componentwise error of d
    back = float(np.abs(_ld_residual(A, d, b)).max() / (nA * nd + nb_))
    back_bar = float(1e-12 + nA * rounding / (nA * nd + nb_))
    cf = scipy.linalg.cho_factor(A)
    x = scipy.linalg.cho_solve(cf, b)
    x = x + scipy.linalg.cho_solve(cf, _ld_residual(A, x, b).astype(np.float64))
    ev = np.linalg.eigvalsh(A)
    kappa = float(ev[-1] / ev[0])
    fwd = float(np.abs(d - x).max() / np.abs(x).max())
    fwd_bar = float(max(1e-10, 100 * kappa * U) + rounding / np.abs(x).max())
    return dict(n_r=n_r, mu0=float(mu0), cluster_solve=st["cluster_solve"], backward_error=back, backward_bar=back_bar, forward_error=fwd,
                forward_bar=fwd_bar, kappa2=kappa, step_rel_to_z=float(nd / np.abs(z1[:n_r]).max())), back <= back_bar and fwd <= fwd_bar


# every rig of (a) with both poses optimised; the cooperative kernel again on every rig the cluster kernel takes (n_r <= 510)
_CLUSTER_RIGS = ("C2_M16", "C3_M16", "C5_M29", "C6_M29", "C16_M64", "C16_M66", "C6_M81")
CASES_B = [(n, "default") for n in _CLUSTER_RIGS + ("C6_M82", "C4_Mbig", "C100_M300")] + [(n, "no_cluster") for n in _CLUSTER_RIGS]


@pytest.mark.parametrize("name,solver", CASES_B, ids=[n + "-" + s for n, s in CASES_B])
def test_reduced_solve_backward_and_forward_error(binding, oracle_mod, monkeypatch, name, solver):
    """The step of k_reduced_solve_cluster2 (n_r <= 510) and of k_reduced_solve (n_r > 510, and every size with
    AAR_NO_CLUSTER_SOLVE=1) against an iteratively refined Cholesky solve of the same system.  The backward error does not depend
    on the conditioning: a wrong tile gives O(1).  Up to n_r = 516 also one and three LM iterations against the oracle's solver."""
    rig = _rig(name)
    o = _oracle(oracle_mod, rig)
    p = _problem(binding, monkeypatch, rig, env=("AAR_NO_CLUSTER_SOLVE",) if solver == "no_cluster" else ())
    expect_cluster = solver == "default" and p.n_r <= 16 * CH_NB
    rec, ok = _check_one_step(binding, p, o, expect_cluster)
    if p.n_r <= 516 and solver == "default":
        z0 = o.mats2evec()
        worst = 0.0
        for k in (1, 3):                                              # the bars of test_lm_first_iterations_match_reference_solver
            o.set_max_iters(k)
            z_o, fc_o, it_o, tr_o = o.solve(z0)
            z_g, fc_g, it_g, tr_g = p.solve(z0, binding.Problem.default_params(max_iters=k))
            dc, dz = abs(fc_g - fc_o) / fc_o, np.abs(z_g - z_o).max() / np.abs(z_o).max()
            worst = max(worst, dc, dz)
            assert it_o == it_g == k and dc <= 1e-10 and dz <= 1e-10, (k, it_o, it_g, dc, dz)
            assert np.allclose(tr_g[:, 1], tr_o[:, 1], rtol=1e-9, atol=0)
        o.set_max_iters(10000)
        rec["lm_1_and_3_iterations_vs_oracle_worst_rel_dev"] = worst
    parity_record("reduced_solve_step_backward_forward_error", rig=name, solver=solver, **rec)
    assert ok, rec


# ------------------------------------------------------------------ c. the intrinsics block beyond one tile
def test_intrinsics_block_multi_tile_lm_steps(binding, oracle_mod):
    """C = 4, M = 12 with the intrinsics: nb = 3 + 11 + 8 = 22 blocks, two SYRK tiles.  The oracle's reduced_system refuses the
    intrinsics, so the comparison is the LM step (the bars of test_intrinsics_block_lm_steps_and_solve)."""
    rig = synth.make_rig(C=4, M=12, F=41, obs_per_frame=16.0, seed=43)
    o = _oracle(oracle_mod, rig, intrinsics=True)
    p = binding.Problem(rig, intrinsics=True)
    assert p.n_r == 6 * 22
    z0 = o.mats2evec()
    worst = 0.0
    for steps in (1, 3):
        o.set_max_iters(steps)
        z_o, c_o, it_o, _ = o.solve(z0)
        z_g, c_g, it_g, _ = p.solve(z0, binding.Problem.default_params(max_iters=steps, ignore_stop_rules=1))
        dz = np.abs(z_g - z_o).max() / max(np.abs(z_o).max(), 1.0); dc = abs(c_g - c_o) / c_o
        worst = max(worst, dz, dc)
        assert it_g == it_o == steps and dz <= 1e-10 and dc <= 1e-10, (steps, it_g, it_o, dz, dc)
    assert p.stats()["cluster_solve"]
    parity_record("intrinsics_block_multi_tile_lm_vs_reference_solver", n_r=p.n_r, F=rig.F, worst_rel_dev=worst, bar=1e-10)


# ------------------------------------------------------------------ d. graph-resident loop against host-driven loop
@pytest.mark.parametrize("name", ["C6_M81", "C6_M82"])
def test_graph_loop_equals_host_loop_at_cluster_limit(binding, monkeypatch, name):
    """7 iterations with the stop rules off: n_r = 510 puts the 16-CTA cluster launch inside the graph, n_r = 516 the cooperative
    launch.  The assertions of test_graph_resident_loop_equals_host_driven_loop, and the graph must have run."""
    rig = _rig(name)
    p = binding.Problem(rig)
    z0 = p.mats2evec()
    prm = binding.Problem.default_params(max_iters=7, ignore_stop_rules=1)
    monkeypatch.setenv("AAR_NO_GRAPH", "1")
    z_h, c_h, it_h, tr_h = p.solve(z0, prm)
    monkeypatch.delenv("AAR_NO_GRAPH")
    g0 = p.stats()["graph_iterations"]
    z_g, c_g, it_g, tr_g = p.solve(z0, prm)
    st = p.stats()
    cost_ok, flips = _same_cost(p, z_g, c_g, z_h, c_h)
    parity_record("graph_loop_vs_host_loop_cluster_limit", rig=name, n_r=p.n_r, cluster_solve=st["cluster_solve"], graph_loop=st["graph_loop"],
                  graph_iterations=st["graph_iterations"] - g0, rel_dev_z=float(np.abs(z_g - z_h).max() / np.abs(z_h).max()),
                  rel_dev_cost=abs(c_g - c_h) / c_h, rows_rounding_differently=flips, rel_tol_z=1e-9)
    assert st["graph_loop"] and st["graph_iterations"] - g0 == 6, st          # every iteration but the first runs inside the graph
    assert st["cluster_solve"] == (p.n_r <= 16 * CH_NB)
    assert it_g == it_h == 7 and cost_ok and _same(z_g, z_h) and np.array_equal(tr_g[:, 3:6], tr_h[:, 3:6]), (c_g, c_h, flips)
    assert _same(tr_g[:, 0], tr_h[:, 0]) and _same(tr_g[:, 1], tr_h[:, 1], 1e-7)


# ------------------------------------------------------------------ e. several live handles
def _second_handle(binding, kind):
    """Handle B: cfg1 (n_r = 42), or a track-only handle of the same rig (n_r = 0)."""
    rig = synth.make_config("cfg1")
    return binding.Problem(rig) if kind == "cfg1" else binding.Problem(rig, cams=False, markers=False)


@pytest.mark.parametrize("kind", ["cfg1", "track_only"])
def test_second_handle_keeps_first_handle_paths(binding, oracle_mod, kind):
    """Handle A (the cfg4 shape, n_r = 468) checked against the oracle, a smaller handle B created and run, then A again at another mu
    (a stale E cannot pass): the same bars, and A still runs the cluster Cholesky."""
    rig = _rig("C16_M64")
    o = _oracle(oracle_mod, rig)
    pA = binding.Problem(rig)
    z0 = o.mats2evec()
    dev1 = _compare_reduced_system(pA, o, z0, 5.0)
    step1, ok1 = _check_one_step(binding, pA, o, True)
    pB = _second_handle(binding, kind)
    zB = pB.mats2evec()
    SB, bB, cB = pB.reduced_system(zB, 3.0)
    assert len(bB) == pB.n_r and np.isfinite(cB)
    _, fcB, itB, _ = pB.solve(zB)
    assert itB > 0 and fcB < cB
    dev2 = _compare_reduced_system(pA, o, z0, 77.0)
    step2, ok2 = _check_one_step(binding, pA, o, True)
    parity_record("several_live_handles_first_handle_after_second", handle_b=kind, n_r_a=pA.n_r, n_r_b=pB.n_r, before=dict(dev1, step=step1),
                  after=dict(dev2, step=step2), bar_S_b=1e-12, bar_cost=1e-13)
    assert dev1["ok"] and ok1 and dev2["ok"] and ok2, (dev1, step1, dev2, step2)
    assert pA.stats()["cluster_solve"]


@pytest.mark.parametrize("kind", ["cfg1", "track_only"])
def test_solve_split_around_another_handle(binding, kind):
    """A's solve split around the creation and the solve of B: lm_begin, lm_iterate(3) (the graph is built and used), B, lm_iterate(3).
    The same 6 iterations as A alone (the bars of test_split_solve_equals_one_solve)."""
    rig = _rig("C16_M64")
    pA = binding.Problem(rig)
    z0 = pA.mats2evec()
    prm = binding.Problem.default_params(max_iters=6, ignore_stop_rules=1)
    z_1, c_1, it_1, tr_1 = pA.solve(z0, prm)
    tries_1 = pA.last_report.total_tries
    g0 = pA.stats()["graph_iterations"]
    pA.lm_begin(z0, prm)
    rep_a, tr_a = pA.lm_iterate(3, trace_capacity=3)
    pB = _second_handle(binding, kind)
    _, fcB, itB, _ = pB.solve(pB.mats2evec())
    rep_b, tr_b = pA.lm_iterate(3, trace_capacity=3)
    z_s = pA.lm_end()
    tr_s = np.concatenate([tr_a, tr_b])
    st = pA.stats()
    cost_ok, flips = _same_cost(pA, z_s, rep_b.final_cost, z_1, c_1)
    parity_record("several_live_handles_split_solve", handle_b=kind, iterations=[rep_a.iterations, rep_b.iterations], graph_iterations=st["graph_iterations"] - g0,
                  cluster_solve=st["cluster_solve"], rel_dev_z=float(np.abs(z_s - z_1).max() / np.abs(z_1).max()), rows_rounding_differently=flips)
    assert rep_a.iterations == rep_b.iterations == 3 and it_1 == 6 and itB > 0
    assert st["graph_iterations"] - g0 == 5 and st["cluster_solve"], st      # the first iteration of a solve runs on the host
    assert rep_b.total_tries == tries_1 == tr_1[:, 3].sum()
    assert np.array_equal(tr_s[:, 3:6], tr_1[:, 3:6])
    assert _same(tr_s[:, 0], tr_1[:, 0]) and _same(tr_s[:, 1], tr_1[:, 1], 1e-7)
    assert cost_ok and _same(z_s, z_1), (rep_b.final_cost, c_1, flips)
