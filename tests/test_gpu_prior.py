"""Soft pose priors in the joint solve (aar_set_prior, csrc/aar_prior.cuh, DESIGN.md §6e); run on the B200 with -m gpu.

The contract: a solve with priors is the reference's SparseLevMarq on the augmented least-squares problem (six rows sqrt(w) (z - zbar)
per entity with a prior).  The oracle's reduced system and restated LM run on exactly that problem (tests/prior_oracle.cpp, PriorOracle
of test_prior_cpu.py) are the reference: every check below is the device against the oracle with the same priors (and mask), with the
bars of test_gpu_fixed.py."""
import copy
import math
import os
import re
import subprocess

import numpy as np
import pytest

from aar_b200 import synth
from conftest import ROOT, parity_record
from test_gpu_fixed import _columns, _mixed
from test_gpu_parity import _end_point_bar, _oracle_envelope, _same, _same_cost
from test_gpu_reduced_system import _rig
from test_prior_cpu import PriorOracle, build_prior_oracle, moved_targets, prior_columns, weights

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def binding():
    from aar_b200 import binding as b
    b.lib()
    return b


@pytest.fixture(scope="module")
def prior_lib(oracle_mod, tmp_path_factory):
    return build_prior_oracle(tmp_path_factory.mktemp("prior_oracle"))


def _priors(oracle_mod, rig, kind, seed=11, scale=2e-3):
    """entity priors of `kind` (cams / markers / frames / all) with targets away from z0 and weights comparable to the reprojection
    diagonal; every 3rd camera and marker and every 2nd frame has one"""
    z0 = oracle_mod.Oracle(rig).mats2evec()
    Tc, Tm, Tf = moved_targets(oracle_mod, rig, z0, scale, seed)
    wc, wm, wf = weights(rig.C, seed + 1, 1e2, 1e6), weights(rig.M, seed + 2, 1e2, 1e6), weights(rig.F, seed + 3, 1e1, 1e5)
    wc[1::3] = 0; wc[2::3] = 0; wm[1::3] = 0; wm[2::3] = 0; wf[1::2] = 0
    out = {}
    if kind in ("cams", "all"):
        out["cams"] = (Tc, wc)
    if kind in ("markers", "all"):
        out["markers"] = (Tm, wm)
    if kind in ("frames", "all"):
        out["frames"] = (Tf, wf)
    return out


def _pair(binding, oracle_mod, prior_lib, rig, priors, masks=None, with_huber=False, analytic=False):
    """device handle and oracle with the same priors (and mask)"""
    o = PriorOracle(prior_lib, rig)
    o.set_config(with_huber=with_huber, huber_delta=2.5)
    if analytic:
        o.set_analytic(True)
    p = binding.Problem(rig, with_huber=with_huber, analytic=analytic)
    p.set_prior(**priors)
    o.set_prior_columns(*prior_columns(oracle_mod, rig, **priors))
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
    c_x = math.fsum((r * r).tolist()) + math.fsum((o._w * (z - o._zbar) ** 2).tolist())
    iu = np.triu_indices(p.n_r)
    dS = np.abs(S_g[iu] - S_o[iu]).max() / np.abs(S_o).max()
    db = np.abs(b_g - b_o).max() / np.abs(b_o).max()
    dc = abs(c_g - c_x) / c_x
    return dict(rel_dev_S=float(dS), rel_dev_b=float(db), rel_dev_cost=float(dc), ok=bool(dS <= 1e-12 and db <= 1e-12 and dc <= 1e-12))


# ------------------------------------------------------------------ the reduced system against the oracle with the same priors
CASES_RS = [("C5_M29", "cams"), ("C5_M29", "markers"), ("C5_M29", "frames"), ("C5_M29", "all"), ("C5_M29", "all_fixed"), ("C16_M64", "all"),
            ("C16_M64", "all_huber")]


@pytest.mark.parametrize("name,kind", CASES_RS, ids=[f"{n}-{k}" for n, k in CASES_RS])
def test_reduced_system_with_priors_matches_oracle(binding, oracle_mod, prior_lib, name, kind):
    rig = _rig(name)
    huber = kind.endswith("huber")
    if huber:                                                     # outliers, so that the Huber weights differ from 1
        rig = copy.copy(rig); rig.det_xy = rig.det_xy.copy(); rig.det_xy[::37] += 25.0
    p, o, col = _pair(binding, oracle_mod, prior_lib, rig, _priors(oracle_mod, rig, kind.split("_")[0]),
                      masks=_mixed(rig) if kind.endswith("fixed") else None, with_huber=huber)
    z0 = o.mats2evec()
    z1 = z0 + np.random.default_rng(5).normal(0, 1e-3, z0.shape)
    devs = [_compare(p, o, z, mu) for z, mu in ((z0, 5.0), (z1, 321.0))]
    parity_record("prior_reduced_system_vs_oracle", rig=name, kind=kind, n_r=p.n_r, prior_columns=int((o._w > 0).sum()), held_columns=int(col.sum()),
                  at_z0=devs[0], at_perturbed_z=devs[1], bar=1e-12)
    assert all(d["ok"] for d in devs), devs


# ------------------------------------------------------------------ one and three LM iterations against the oracle's solver
CASES_LM = [("cfg1", ""), ("cfg2_distorted", ""), ("C6_M82", ""), ("cfg1", "analytic")]


def _workload(name):
    if name == "cfg2_distorted":
        return synth.make_config("cfg2", distorted=True)
    return synth.make_config(name) if name.startswith("cfg") else _rig(name)


@pytest.mark.parametrize("name,variant", CASES_LM, ids=[n + ("-" + v if v else "") for n, v in CASES_LM])
def test_lm_iterations_with_priors_match_oracle(binding, oracle_mod, prior_lib, name, variant):
    """C6_M82: n_r = 516, the cooperative-grid Cholesky."""
    rig = _workload(name)
    p, o, _ = _pair(binding, oracle_mod, prior_lib, rig, _priors(oracle_mod, rig, "all"), analytic=variant == "analytic")
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
    parity_record("prior_lm_iterations_vs_oracle", workload=name, variant=variant or "faithful", n_r=p.n_r, cluster_solve=st["cluster_solve"],
                  worst_rel_dev=worst, bar=1e-10)
    if name == "C6_M82":
        assert not st["cluster_solve"]


# ------------------------------------------------------------------ full solves
@pytest.mark.parametrize("name", ["cfg1", "cfg2_distorted"])
def test_full_solve_with_priors(binding, oracle_mod, prior_lib, name):
    rig = _workload(name)
    p, o, _ = _pair(binding, oracle_mod, prior_lib, rig, _priors(oracle_mod, rig, "all"))
    z0 = o.mats2evec()
    z_g, fc_g, it_g, _ = p.solve(z0)
    z_o, fc_o, it_o, _ = o.solve(z0)
    env_c, _ = _oracle_envelope(o, z0, fc_o, z_o)
    d_cost = abs(fc_g - fc_o) / fc_o
    passes = _end_point_bar(d_cost, env_c, 2e-5)
    parity_record("prior_full_solve_vs_oracle", workload=name, iterations_gpu=it_g, iterations_oracle=it_o, rel_dev_final_cost=d_cost,
                  ref_envelope_cost=env_c, passes_by=passes)
    assert abs(it_g - it_o) <= 1


# ------------------------------------------------------------------ limits
def test_zero_weights_and_held_entity_with_prior(binding, oracle_mod):
    rig = synth.make_config("cfg1")
    p, plain = binding.Problem(rig), binding.Problem(rig)
    z0 = p.mats2evec()
    prm = binding.Problem.default_params(max_iters=5, ignore_stop_rules=1)
    pr = _priors(oracle_mod, rig, "all")
    p.set_prior(**{k: (T, np.zeros_like(w)) for k, (T, w) in pr.items()})
    z_p, c_p, _, _ = p.solve(z0, prm)
    z_n, c_n, _, _ = plain.solve(z0, prm)
    dz = float(np.abs(z_p - z_n).max() / np.abs(z_n).max())
    assert dz <= 3e-13 and abs(c_p - c_n) <= 1e-12 * c_n, (dz, c_p, c_n)
    # a held entity with a prior: the mask wins, its entries stay == z0; its prior residual is a constant of the cost
    masks = _mixed(rig)
    p.set_prior(**pr)
    p.set_fixed(*masks)
    col = _columns(p, *masks)
    z_h, c_h, _, _ = p.solve(z0, prm)
    assert np.array_equal(z_h[col], z0[col]) and not np.array_equal(z_h[~col], z0[~col])
    parity_record("prior_limits", workload="cfg1", zero_weights_rel_dev_z=dz, held_with_prior_unchanged=True, bar_zero_weights=3e-13)


# ------------------------------------------------------------------ the two loops, new target values, and clearing the priors
def test_graph_loop_equals_host_loop_and_reads_new_targets(binding, oracle_mod, monkeypatch):
    rig = synth.make_config("cfg1")
    p, plain = binding.Problem(rig), binding.Problem(rig)
    z0 = p.mats2evec()
    prm = binding.Problem.default_params(max_iters=7, ignore_stop_rules=1)
    rec = {}
    for label, seed in (("first_targets", 11), ("new_targets", 29)):
        pr = _priors(oracle_mod, rig, "all", seed=seed)
        if label == "new_targets":                                # only the values change: the graph is kept and must read them
            pr = {k: (T, old[k][1]) for k, (T, _) in pr.items()}
        old = pr
        p.set_prior(**pr)
        monkeypatch.setenv("AAR_NO_GRAPH", "1")
        z_h, c_h, it_h, tr_h = p.solve(z0, prm)
        monkeypatch.delenv("AAR_NO_GRAPH")
        g0 = p.stats()["graph_iterations"]
        z_g, c_g, it_g, tr_g = p.solve(z0, prm)
        st = p.stats()
        assert st["graph_loop"] and st["graph_iterations"] - g0 == 6, st
        assert it_g == it_h == 7 and _same(z_g, z_h) and abs(c_g - c_h) <= 1e-9 * c_h and np.array_equal(tr_g[:, 3:6], tr_h[:, 3:6]), (label, c_g, c_h)
        rec[label] = dict(rel_dev_z=float(np.abs(z_g - z_h).max() / np.abs(z_h).max()), rel_dev_cost=abs(c_g - c_h) / c_h, final_cost=c_g)
    assert rec["first_targets"]["final_cost"] != rec["new_targets"]["final_cost"]
    l0 = p.kernel_launches
    p.solve(z0, prm)
    with_priors = p.kernel_launches - l0
    p.set_prior()                                                  # cleared: the graph is captured again, without the prior kernels
    l0 = p.kernel_launches
    z_c, c_c, _, _ = p.solve(z0, prm)
    cleared = p.kernel_launches - l0
    l0 = plain.kernel_launches
    z_n, c_n, _, _ = plain.solve(z0, prm)
    never = plain.kernel_launches - l0
    cost_ok, flips = _same_cost(plain, z_c, c_c, z_n, c_n)
    parity_record("prior_graph_vs_host_loop_and_clear", workload="cfg1", iterations=7, launches_with_priors=with_priors, launches_after_clear=cleared,
                  launches_never_with_priors=never, **rec)
    assert cleared == never < with_priors and p.stats()["graph_loop"], (with_priors, cleared, never)
    assert _same(z_c, z_n) and cost_ok, flips


# ------------------------------------------------------------------ refusals and argument handling
def test_refusals(binding, oracle_mod):
    rig = synth.make_config("cfg1")
    p = binding.Problem(rig)
    z0 = p.mats2evec()
    pr = _priors(oracle_mod, rig, "all")
    Tc, wc = pr["cams"]
    with pytest.raises(ValueError):
        p.set_prior(cams=(Tc[:-1], wc[:-1]))
    with pytest.raises(ValueError):
        p.set_prior(frames=(pr["frames"][0], np.ones((rig.F, 3))))
    p.lm_begin(z0)
    with pytest.raises(binding.AarError, match="aar_lm_begin"):
        p.set_prior(**pr)
    p.lm_end()
    for bad in (-1.0, np.nan, np.inf):
        w = wc.copy(); w[1, 4] = bad
        with pytest.raises(binding.AarError, match="weight"):
            p.set_prior(cams=(Tc, w))
    T = Tc.copy(); T[np.flatnonzero(wc.any(axis=1))[0], 0, 3] = np.nan
    with pytest.raises(binding.AarError, match="non-finite"):
        p.set_prior(cams=(T, wc))
    T = Tc.copy(); T[np.flatnonzero(~wc.any(axis=1))[0], 0, 3] = np.nan       # no weight: the target is not read
    p.set_prior(cams=(T, wc))
    # a prior on the root camera alone has no columns: nothing is added, nothing is launched
    root = np.array([cid == rig.root_cam for cid in rig.cam_ids])
    w = np.zeros((rig.C, 6)); w[root] = 1e6
    p.set_prior(cams=(Tc, w))
    l0 = p.kernel_launches
    S0, b0, c0 = p.reduced_system(z0, 5.0)                         # the order of the FP64 atomic sums varies: bars, not bits
    root_only = p.kernel_launches - l0
    p.set_prior()
    l0 = p.kernel_launches
    p.reduced_system(z0, 5.0)
    assert root_only == p.kernel_launches - l0
    # a target equal to the start matrix: z - zbar = 0 exactly, so b and the cost are those without the prior, S gains diag(w)
    w = np.zeros((rig.C, 6)); w[~root] = 1e4
    p.set_prior(cams=(rig.T_cam_init, w))
    S, b, c = p.reduced_system(z0, 5.0)
    d = np.zeros(p.n_r); d[:6 * (rig.C - 1)] = 1e4
    assert np.abs(b - b0).max() <= 1e-13 * np.abs(b0).max() and abs(c - c0) <= 1e-13 * c0
    assert np.abs(S - S0 - np.diag(d)).max() <= 1e-13 * np.abs(S0).max()


# ------------------------------------------------------------------ the find_solution app
@pytest.fixture(scope="module")
def host_bins():
    from aar_b200 import binding
    binding.build()
    host = os.path.join(ROOT, "automatic-ar_b200", "host")
    subprocess.run(["make", "-s", "-C", host], check=True)
    return host


def _run(host_bins, folder, start, *opts, check=True):
    r = subprocess.run([os.path.join(host_bins, "find_solution"), str(folder), "0.05", "-init", start, *opts], capture_output=True, text=True)
    if check:
        assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    return r


def _final(folder, out):
    return synth.read_solution_file(str(folder / "final.solution"))["vec"], float(re.findall(r"final_error: (\S+)", out)[-1])


@pytest.mark.parametrize("reject", [False, True], ids=["plain", "reject_outliers"])
def test_find_solution_prior_cams(host_bins, oracle_mod, tmp_path, reject):
    rig = synth.make_config("cfg1")
    if reject:
        rig = copy.copy(rig); rig.det_xy = rig.det_xy.copy(); rig.det_xy[::41] += 30.0
    extra = ["-reject-outliers", "5"] if reject else []
    # the solved rig, written back as the prior file
    d0 = tmp_path / "solve"; d0.mkdir()
    init = str(d0 / "init.solution"); synth.write_solution_file(init, rig)
    _run(host_bins, d0, init)
    vec = synth.read_solution_file(str(d0 / "final.solution"))["vec"]
    o = oracle_mod.Oracle(rig)
    Tc, Tm, Tf = o.evec2mats(vec[:o.num_vars])
    solved = copy.copy(rig); solved.T_cam_init, solved.T_marker_init, solved.T_frame_init = Tc, Tm, Tf
    prior_file = str(tmp_path / "prior.solution"); synth.write_solution_file(prior_file, solved)
    # the start: the solved rig with every non-root camera moved
    from oracle_py import rodrigues
    start = copy.copy(solved); start.T_cam_init = Tc.copy()
    rng = np.random.default_rng(17)
    for i in range(rig.C):
        if rig.cam_ids[i] != rig.root_cam:
            start.T_cam_init[i, :3, :3] = start.T_cam_init[i, :3, :3] @ rodrigues(rng.normal(0, 0.01, 3))
            start.T_cam_init[i, :3, 3] += rng.normal(0, 0.01, 3)
    start_file = str(tmp_path / "start.solution"); synth.write_solution_file(start_file, start)
    ref = synth.read_solution_file(prior_file)["vec"]
    nrc = 6 * (rig.C - 1)
    res = {}
    for label, opts in (("none", []), ("sigma_1e-3", ["-prior-cams", prior_file, "1e-3", "1e-3"]), ("sigma_1e6", ["-prior-cams", prior_file, "1e6", "1e6"])):
        d = tmp_path / label; d.mkdir()
        out = _run(host_bins, d, start_file, *opts, *extra).stdout
        if opts:
            assert f"priors on {rig.C} cameras" in out, out
        if reject:
            assert int(out.split("removed ")[1].split()[0]) > 0
        v, cost = _final(d, out)
        res[label] = dict(cam_dist=float(np.abs(v[:nrc] - ref[:nrc]).max()), final_cost=cost)
    assert res["sigma_1e-3"]["cam_dist"] < res["none"]["cam_dist"], res
    assert abs(res["sigma_1e6"]["final_cost"] - res["none"]["final_cost"]) <= 1e-6 * res["none"]["final_cost"], res
    # a prior file with another root camera: its poses are relative to that root
    other = copy.copy(solved); other.root_cam = int([c for c in rig.cam_ids if c != rig.root_cam][0])
    other_file = str(tmp_path / "other_root.solution"); synth.write_solution_file(other_file, other)
    d = tmp_path / "mismatch"; d.mkdir()
    r = _run(host_bins, d, start_file, "-prior-cams", other_file, "1e-3", "1e-3", check=False)
    assert r.returncode == 1 and "root camera" in r.stderr, (r.returncode, r.stderr)
    parity_record("prior_find_solution_app", reject_outliers=reject, **res)


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
    pr = _priors(oracle_py, rig, "all")
    p = binding.Problem(rig, device=rank, rank=rank, world_size=world)
    p.set_prior(**pr)
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
        single.set_prior(**pr)
        S1, b1, c1 = single.reduced_system(z0, mu)
        n = p.n_r; iu = np.triu_indices(n)
        rec = dict(reduced_system_rel_dev=np.abs(buf[:n * n].reshape(n, n)[iu] - S1[iu]).max() / np.abs(S1).max(),
                   reduced_rhs_rel_dev=np.abs(buf[n * n:n * n + n] - b1).max() / np.abs(b1).max(), cost_rel_dev=abs(buf[-1] - c1) / c1)
        z1, fc1, it1, _ = single.solve(z0, binding.Problem.default_params(max_iters=3, ignore_stop_rules=1))
        rec.update(three_iterations_rel_dev_z=np.abs(z - z1).max() / np.abs(z1).max(), three_iterations_rel_dev_cost=abs(fc - fc1) / fc1)
        parity_record("prior_world2_cfg2_vs_single_gpu", **rec)
        assert rec["reduced_system_rel_dev"] <= 1e-12 and rec["reduced_rhs_rel_dev"] <= 1e-12 and rec["cost_rel_dev"] <= 1e-12, rec
        assert it == it1 == 3 and rec["three_iterations_rel_dev_z"] <= 1e-10 and rec["three_iterations_rel_dev_cost"] <= 1e-10, rec
        open(os.path.join(out_dir, "ok"), "w").write("ok")
    p.close()
    dist.destroy_process_group()


def test_sharded_priors_match_single_gpu(oracle_mod, tmp_path):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    port = 29500 + os.getpid() % 200
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert os.path.exists(os.path.join(tmp_path, "ok"))
