"""Cameras, markers and frames held fixed in the joint solve (aar_set_fixed, csrc/aar_fixed.cuh, DESIGN.md §6d); run on the B200 with -m gpu.

The contract: the solve is the reference's SparseLevMarq on the Jacobian whose columns of the held entities are explicit zeros.  The
oracle's reduced system and restated LM fed exactly that Jacobian (tests/fixed_oracle.cpp, FixedOracle of test_fixed_cpu.py) is the reference, so every check below is the device against the
oracle with the same mask, plus the property the contract implies: a held entry of z compares == to z0 after any number of iterations."""
import copy
import os
import re
import subprocess

import numpy as np
import pytest

from aar_b200 import synth
from conftest import ROOT, parity_record
from test_fixed_cpu import FixedOracle, build_fixed_oracle
from test_gpu_parity import _end_point_bar, _oracle_envelope, _same, _same_cost
from test_gpu_reduced_system import _compare_reduced_system, _rig

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def binding():
    from aar_b200 import binding as b
    b.lib()
    return b


@pytest.fixture(scope="module")
def fixed_lib(oracle_mod, tmp_path_factory):
    return build_fixed_oracle(tmp_path_factory.mktemp("fixed_oracle"))


def _entity_masks(rig, cams=(), markers=(), frames=()):
    c = np.zeros(rig.C, bool); m = np.zeros(rig.M, bool); f = np.zeros(rig.F, bool)
    c[list(cams)] = True; m[list(markers)] = True; f[list(frames)] = True
    return c, m, f


def _columns(p, c, m, f):
    """io_vec columns of the held entities (the block columns of aar_index_maps; -1 = root / group not optimised)."""
    im = p.index_maps()
    col = np.zeros(p.num_vars, bool)
    for flags, first in ((c, im["col_cam"]), (m, im["col_marker"]), (f, im["col_frame"])):
        for i in np.flatnonzero(flags):
            if first[i] >= 0:
                col[first[i]:first[i] + 6] = True
    return col


def _mixed(rig):
    """a few non-root cameras and markers, every 7th frame"""
    non_root_c = [i for i in range(rig.C) if rig.cam_ids[i] != rig.root_cam]
    non_root_m = [j for j in range(rig.M) if rig.marker_ids[j] != rig.root_marker]
    return _entity_masks(rig, non_root_c[:max(1, len(non_root_c) // 3)], non_root_m[1::4], range(0, rig.F, 7))


def _pair(binding, fixed_lib, rig, masks, with_huber=False, analytic=False, **kw):
    """device handle and oracle with the same mask"""
    o = FixedOracle(fixed_lib, rig)
    o.set_config(with_huber=with_huber, huber_delta=2.5)
    if analytic:
        o.set_analytic(True)
    p = binding.Problem(rig, with_huber=with_huber, analytic=analytic, **kw)
    p.set_fixed(*masks)
    col = _columns(p, *masks)
    o.set_fixed_columns(col)
    return p, o, col


# ------------------------------------------------------------------ 3. the reduced system against the oracle with the same mask
CASES_RS = [("C5_M29", "cams"), ("C5_M29", "markers"), ("C5_M29", "frames"), ("C5_M29", "all"), ("C16_M64", "all"), ("C16_M64", "all_huber")]


@pytest.mark.parametrize("name,kind", CASES_RS, ids=[f"{n}-{k}" for n, k in CASES_RS])
def test_reduced_system_with_mask_matches_oracle(binding, fixed_lib, name, kind):
    rig = _rig(name)
    huber = kind.endswith("huber")
    if huber:                                                     # outliers, so that the Huber weights differ from 1
        rig = copy.copy(rig); rig.det_xy = rig.det_xy.copy(); rig.det_xy[::37] += 25.0
    c, m, f = _mixed(rig)
    if kind == "cams":
        m[:] = False; f[:] = False
    elif kind == "markers":
        c[:] = False; f[:] = False
    elif kind == "frames":
        c[:] = False; m[:] = False
    p, o, col = _pair(binding, fixed_lib, rig, (c, m, f), with_huber=huber)
    held = col[:p.n_r]
    z0 = o.mats2evec()
    z1 = z0 + np.random.default_rng(5).normal(0, 1e-3, z0.shape)
    devs = []
    for z, mu in ((z0, 5.0), (z1, 321.0)):
        devs.append(_compare_reduced_system(p, o, z, mu))
        S, b, _ = p.reduced_system(z, mu)
        U = np.triu(S)
        devs[-1]["held_rows_cols_b_exactly_zero"] = bool(not U[held].any() and not U[:, held].any() and not b[held].any())
    parity_record("fixed_reduced_system_vs_oracle", rig=name, kind=kind, n_r=p.n_r, held_reduced_columns=int(held.sum()), held_frames=int(f.sum()),
                  at_z0=devs[0], at_perturbed_z=devs[1], bar_S_b=1e-12)
    assert kind == "frames" or held.any()
    assert all(d["ok"] and d["held_rows_cols_b_exactly_zero"] for d in devs), devs


# ------------------------------------------------------------------ 4. / 8. one and three LM iterations against the oracle's solver
CASES_LM = [("cfg1", ""), ("cfg2_distorted", ""), ("C6_M82", ""), ("cfg1", "analytic")]


def _workload(name):
    if name == "cfg2_distorted":
        return synth.make_config("cfg2", distorted=True)
    return synth.make_config(name) if name.startswith("cfg") else _rig(name)


@pytest.mark.parametrize("name,variant", CASES_LM, ids=[n + ("-" + v if v else "") for n, v in CASES_LM])
def test_lm_iterations_with_mask_match_oracle(binding, fixed_lib, name, variant):
    """C6_M82: n_r = 516, the cooperative-grid Cholesky."""
    rig = _workload(name)
    masks = _mixed(rig)
    p, o, col = _pair(binding, fixed_lib, rig, masks, analytic=variant == "analytic")
    z0 = o.mats2evec()
    worst = 0.0
    for k in (1, 2, 3):
        z_g, fc_g, it_g, tr_g = p.solve(z0, binding.Problem.default_params(max_iters=k, ignore_stop_rules=1))
        assert it_g == k and np.array_equal(z_g[col], z0[col]), k            # held entries == z0 after every iteration
        if k == 2:
            continue
        o.set_max_iters(k)
        z_o, fc_o, it_o, tr_o = o.solve(z0)
        dz, dc = np.abs(z_g - z_o).max() / np.abs(z_o).max(), abs(fc_g - fc_o) / fc_o
        worst = max(worst, dz, dc)
        assert it_o == k and dz <= 1e-10 and dc <= 1e-10, (k, dz, dc)
    st = p.stats()
    parity_record("fixed_lm_iterations_vs_oracle", workload=name, variant=variant or "faithful", n_r=p.n_r, held_columns=int(col.sum()),
                  cluster_solve=st["cluster_solve"], worst_rel_dev=worst, bar=1e-10)
    if name == "C6_M82":
        assert not st["cluster_solve"]


# ------------------------------------------------------------------ 5. full solves
@pytest.mark.parametrize("name", ["cfg1", "cfg2_distorted"])
def test_full_solve_with_mask(binding, fixed_lib, name):
    rig = _workload(name)
    p, o, col = _pair(binding, fixed_lib, rig, _mixed(rig))
    z0 = o.mats2evec()
    z_g, fc_g, it_g, _ = p.solve(z0)
    z_o, fc_o, it_o, _ = o.solve(z0)
    assert np.array_equal(z_g[col], z0[col]) and np.array_equal(z_o[col], z0[col])
    env_c, _ = _oracle_envelope(o, z0, fc_o, z_o)
    d_cost = abs(fc_g - fc_o) / fc_o
    passes = _end_point_bar(d_cost, env_c, 2e-5)
    parity_record("fixed_full_solve_vs_oracle", workload=name, held_columns=int(col.sum()), iterations_gpu=it_g, iterations_oracle=it_o,
                  rel_dev_final_cost=d_cost, ref_envelope_cost=env_c, passes_by=passes)
    assert abs(it_g - it_o) <= 1


# ------------------------------------------------------------------ 6. the device against its own group flags
def _round_tripped(oracle_mod, rig, group):
    """the rig whose matrices of `group` are their r -> R expansion at z0, as the solve that optimises the group reads them (the
    oracle's expansion is the device's bit for bit; a throwaway instance, evec2mats overwrites its matrices)"""
    o = oracle_mod.Oracle(rig)
    Tc, _, Tf = o.evec2mats(o.mats2evec())
    r = copy.copy(rig)
    if group == "cams":
        r.T_cam_init = Tc
    else:
        r.T_frame_init = Tf
    return r


@pytest.mark.parametrize("group", ["cams", "frames"])
def test_every_entity_held_equals_group_flag(binding, oracle_mod, group):
    rig = synth.make_config("cfg2")
    p = binding.Problem(rig)
    non_root = np.array([cid != rig.root_cam for cid in rig.cam_ids])
    masks = (non_root, None, None) if group == "cams" else (None, None, np.ones(rig.F, bool))
    q = binding.Problem(_round_tripped(oracle_mod, rig, group), cams=group != "cams", objects=group != "frames")
    p.set_fixed(*masks)
    col = _columns(p, *[np.zeros(n, bool) if a is None else a for a, n in zip(masks, (rig.C, rig.M, rig.F))])
    z0 = p.mats2evec(); zq0 = q.mats2evec()
    free = ~col if group == "cams" else np.arange(p.num_vars) < p.n_r
    assert np.array_equal(z0[free], zq0)
    prm = binding.Problem.default_params(max_iters=3, ignore_stop_rules=1)
    z_p, c_p, _, tr_p = p.solve(z0, prm)
    z_q, c_q, _, tr_q = q.solve(zq0, prm)
    dz = float(np.abs(z_p[free] - z_q).max() / np.abs(z_q).max())
    parity_record("fixed_every_entity_vs_group_flag", group=group, workload="cfg2", iterations=3, rel_dev_free_z=dz, rel_dev_cost=abs(c_p - c_q) / c_q, bar=1e-10)
    assert np.array_equal(z_p[col], z0[col]) and dz <= 1e-10 and abs(c_p - c_q) <= 1e-10 * c_q, (dz, c_p, c_q)
    assert np.array_equal(tr_p[:, 3:5], tr_q[:, 3:5])


# ------------------------------------------------------------------ 7. the two loops, and clearing the mask
def test_graph_loop_equals_host_loop_and_clearing_restores_launches(binding, monkeypatch):
    rig = synth.make_config("cfg1")
    p = binding.Problem(rig)
    plain = binding.Problem(rig)
    masks = _mixed(rig); col = _columns(p, *masks)
    p.set_fixed(*masks)
    z0 = p.mats2evec()
    prm = binding.Problem.default_params(max_iters=7, ignore_stop_rules=1)
    monkeypatch.setenv("AAR_NO_GRAPH", "1")
    z_h, c_h, it_h, tr_h = p.solve(z0, prm)
    monkeypatch.delenv("AAR_NO_GRAPH")
    g0 = p.stats()["graph_iterations"]
    z_g, c_g, it_g, tr_g = p.solve(z0, prm)
    st = p.stats()
    cost_ok, flips = _same_cost(plain, z_g, c_g, z_h, c_h)
    assert st["graph_loop"] and st["graph_iterations"] - g0 == 6, st
    assert it_g == it_h == 7 and cost_ok and _same(z_g, z_h) and np.array_equal(tr_g[:, 3:6], tr_h[:, 3:6]), (c_g, c_h, flips)
    assert np.array_equal(z_g[col], z0[col]) and np.array_equal(z_h[col], z0[col])
    l0 = p.kernel_launches
    p.solve(z0, prm)
    masked = p.kernel_launches - l0
    p.set_fixed()                                                  # cleared: the graph is captured again, without k_hold_fixed
    l0 = p.kernel_launches
    z_c, _, _, _ = p.solve(z0, prm)
    cleared = p.kernel_launches - l0
    l0 = plain.kernel_launches
    z_n, _, _, _ = plain.solve(z0, prm)
    never = plain.kernel_launches - l0
    parity_record("fixed_graph_vs_host_loop_and_clear", workload="cfg1", iterations=7, rel_dev_z=float(np.abs(z_g - z_h).max() / np.abs(z_h).max()),
                  launches_with_mask=masked, launches_after_clear=cleared, launches_never_masked=never, rows_rounding_differently=flips)
    assert cleared == never < masked and p.stats()["graph_loop"], (masked, cleared, never)
    assert _same(z_c, z_n) and not np.array_equal(z_c[col], z0[col])
    # a flag on the root camera alone has no effect: nothing is held, nothing is launched
    root = np.array([cid == rig.root_cam for cid in rig.cam_ids])
    p.set_fixed(cams=root)
    l0 = p.kernel_launches
    p.solve(z0, prm)
    assert p.kernel_launches - l0 == never


# ------------------------------------------------------------------ 9. refusals and argument handling
def test_refusals(binding):
    rig = synth.make_config("cfg1")
    p = binding.Problem(rig)
    z0 = p.mats2evec()
    c, m, f = _mixed(rig)
    with pytest.raises(ValueError):
        p.set_fixed(cams=c[:-1])
    with pytest.raises(ValueError):
        p.set_fixed(frames=np.ones(rig.F + 1, bool))
    p.lm_begin(z0)
    with pytest.raises(binding.AarError, match="aar_lm_begin"):
        p.set_fixed(c, m, f)
    p.lm_end()
    with pytest.raises(binding.AarError, match="no free column"):
        p.set_fixed(np.ones(rig.C, bool), np.ones(rig.M, bool), np.ones(rig.F, bool))
    # frames only: every pose but the frames is free, so holding all frames is accepted; a handle that optimises frames alone is not
    p.set_fixed(frames=np.ones(rig.F, bool))
    objects_only = binding.Problem(rig, cams=False, markers=False)
    with pytest.raises(binding.AarError, match="no free column"):
        objects_only.set_fixed(frames=np.ones(rig.F, bool))
    objects_only.set_fixed(cams=np.ones(rig.C, bool), markers=np.ones(rig.M, bool))     # groups that are not optimised: no effect
    # None = none of that kind: cameras held, markers free
    p.set_fixed(cams=c, markers=None)
    S, b, _ = p.reduced_system(z0, 5.0)
    col = _columns(p, c, np.zeros(rig.M, bool), np.zeros(rig.F, bool))[:p.n_r]
    assert not b[col].any() and b[~col].any()


# ------------------------------------------------------------------ 10. the find_solution app
@pytest.fixture(scope="module")
def host_bins():
    from aar_b200 import binding
    binding.build()
    host = os.path.join(ROOT, "automatic-ar_b200", "host")
    subprocess.run(["make", "-s", "-C", host], check=True)
    return host


def _yaml_records(path, section, idname):
    txt = open(path).read()
    names = ["transforms_to_root_cam:", "transforms_to_root_marker:", "root_marker_to_root_cam:"]
    i = names.index(section)
    sec = txt.split(section)[1]
    if i + 1 < len(names):
        sec = sec.split(names[i + 1])[0]
    return dict(zip((int(v) for v in re.findall(idname + r":(-?\d+)", sec)), re.findall(r"data: \[([^\]]*)\]", sec)))


@pytest.mark.parametrize("reject", [False, True], ids=["plain", "reject_outliers"])
def test_find_solution_fix_options(host_bins, tmp_path, reject):
    rig = synth.make_config("cfg1")
    if reject:                                                    # detections the rejection removes before the second solve
        rig = copy.copy(rig); rig.det_xy = rig.det_xy.copy(); rig.det_xy[::41] += 30.0
    init = str(tmp_path / "initial.solution")
    synth.write_solution_file(init, rig)
    # the matrices the mapper holds after reading initial.solution, written back unchanged
    rt, rty = str(tmp_path / "rt.solution"), str(tmp_path / "rt.solution.yaml")
    subprocess.run([os.path.join(host_bins, "solution_tool"), "roundtrip", init, rt, rty], check=True)
    cams = [int(i) for i in rig.cam_ids if i != rig.root_cam][:1]
    markers = [int(i) for i in rig.marker_ids if i != rig.root_marker][1:3]
    frames = [int(i) for i in rig.frame_ids[::9]]
    cmd = [os.path.join(host_bins, "find_solution"), str(tmp_path), "0.05", "-init", init, "-fix-cams", *map(str, cams),
           "-fix-markers", *map(str, markers), "-fix-frames", *map(str, frames)]
    if reject:
        cmd += ["-reject-outliers", "5"]
    out = subprocess.run(cmd, check=True, capture_output=True, text=True).stdout
    if reject:
        assert int(out.split("removed ")[1].split()[0]) > 0
    fin, ref = synth.read_solution_file(str(tmp_path / "final.solution")), synth.read_solution_file(rt)
    moved = 0
    for sec, idname, ids, held in (("transforms_to_root_cam:", "cam_id", rig.cam_ids, cams), ("transforms_to_root_marker:", "marker_id", rig.marker_ids, markers),
                                   ("root_marker_to_root_cam:", "frame_id", rig.frame_ids, frames)):
        a, b = _yaml_records(str(tmp_path / "final.solution.yaml"), sec, idname), _yaml_records(rty, sec, idname)
        for i in held:
            if i in a:                                           # a frame the rejection removed is no longer in the file
                assert a[i] == b[i], (sec, i)                    # the 4x4 record, byte for byte
        moved += sum(a[i] != b[i] for i in a if i not in held)
    assert moved > 0
    # the records of the binary file: rotation vector and translation of every held camera / marker
    def vec_index(ids, root, i):
        return [j for j in ids if j != root].index(i)
    nrc = len(rig.cam_ids) - 1
    for i in cams:
        k = 6 * vec_index(list(rig.cam_ids), rig.root_cam, i)
        assert fin["vec"][k:k + 6].tobytes() == ref["vec"][k:k + 6].tobytes(), i
    for i in markers:
        k = 6 * (nrc + vec_index(list(rig.marker_ids), rig.root_marker, i))
        assert fin["vec"][k:k + 6].tobytes() == ref["vec"][k:k + 6].tobytes(), i
    parity_record("fixed_find_solution_app", reject_outliers=reject, held_cams=cams, held_markers=markers, held_frames=len(frames), free_records_moved=int(moved),
                  held_records_byte_identical=True)
