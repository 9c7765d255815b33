"""GPU parity tests (run on the B200 with -m gpu): the CUDA path behind the C ABI (include/aar_cuda.h)
against the CPU oracle on the same seeded inputs.  Index maps, undistorted corners, residuals and
Jacobians must be BIT-EXACT (the float32 projection rounding of multicam_mapper.cpp:644-648 leaves no
room for a tolerance); sums of products (reduced system, costs, LM trajectory) are compared with the
tolerances of BASELINE.json's north star written at each assert."""
import copy
import os

import numpy as np
import pytest

from aar_b200 import synth
from conftest import ROOT, parity_record

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def binding():
    from aar_b200 import binding as b
    b.lib()
    return b


def small_rig(seed=3, **kw):
    args = dict(C=3, M=6, F=40, obs_per_frame=6.0, seed=seed)
    args.update(kw)
    return synth.make_rig(**args)


def test_index_maps_bit_exact(binding, oracle_mod):
    rig = small_rig()
    # detections of an unknown camera / marker / frame and a duplicated (frame, cam, marker) exercise the erasures
    extra_f = np.array([rig.frame_ids[0], rig.frame_ids[1], 10 ** 6, rig.det_frame[5]], np.int32)
    extra_c = np.array([99, rig.cam_ids[1], rig.cam_ids[0], rig.det_cam[5]], np.int32)
    extra_m = np.array([rig.marker_ids[0], 12345, rig.marker_ids[0], rig.det_marker[5]], np.int32)
    rig.det_frame = np.concatenate([rig.det_frame, extra_f]); rig.det_cam = np.concatenate([rig.det_cam, extra_c])
    rig.det_marker = np.concatenate([rig.det_marker, extra_m])
    rig.det_xy = np.concatenate([rig.det_xy, rig.det_xy[:4] + 1.0])
    # the oracle cannot hold a frame without a pose (the reference would throw): drop that one for it
    keep = rig.det_frame != 10 ** 6
    rig_o = copy.copy(rig)
    rig_o.det_frame, rig_o.det_cam, rig_o.det_marker, rig_o.det_xy = rig.det_frame[keep], rig.det_cam[keep], rig.det_marker[keep], rig.det_xy[keep]
    o = oracle_mod.Oracle(rig_o)
    p = binding.Problem(rig)
    obs = o.observations(); maps = p.index_maps()
    assert p.num_obs == len(obs["frame_id"])
    assert np.array_equal(rig.frame_ids[maps["frame_idx"]], obs["frame_id"])
    assert np.array_equal(rig.cam_ids[maps["cam_idx"]], obs["cam_id"])
    assert np.array_equal(rig.marker_ids[maps["marker_idx"]], obs["marker_id"])
    assert np.array_equal(maps["has_jac"], obs["has_jac"]) and (obs["has_jac"] == 0).sum() == 1
    assert p.num_vars == o.num_vars
    und, raw = p.observations()
    assert np.array_equal(und, obs["und"]) and np.array_equal(raw[obs["has_jac"] == 1], obs["raw"][obs["has_jac"] == 1])
    # Jacobian sparsity pattern bit-exact (explicit zeros kept), values bit-exact
    z = o.mats2evec()
    cp_o, ri_o, v_o = o.jacobian(z)
    cp_g, ri_g, v_g = p.jacobian(z)
    assert np.array_equal(cp_o, cp_g) and np.array_equal(ri_o, ri_g)
    assert np.array_equal(v_o, v_g)
    r_g, _ = p.residual(z)
    assert np.array_equal(r_g, o.error(z))
    parity_record("index_maps_sparsity_pattern_jacobian_residual_with_erasures_and_duplicates", observations=int(p.num_obs), jacobian_nnz=int(len(v_g)),
                  erased_or_duplicate_detections=4, bit_exact=True)


@pytest.mark.parametrize("distorted,staging", [(False, "float32"), (True, "float32"), (True, "fp64")], ids=["False", "True", "fp64_staging"])
def test_residual_and_jacobian_bit_exact(binding, oracle_mod, monkeypatch, distorted, staging):
    rig = small_rig(seed=5, distorted=distorted, F=60)
    o = oracle_mod.Oracle(rig, sincos_mode=1)
    if staging == "fp64":       # read when the handle is created: every evaluation stages its Jacobian rows in FP64
        monkeypatch.setenv("AAR_FORCE_EXACT_STAGING", "1")
    p = binding.Problem(rig)
    und, raw = p.observations()
    obs = o.observations()
    assert np.array_equal(und, obs["und"])                      # device undistortion == cv::undistortPoints restatement
    if distorted:
        assert not np.array_equal(und, raw)
    rng = np.random.default_rng(0)
    z0 = o.mats2evec()
    assert np.abs(p.mats2evec() - z0).max() < 1e-12
    for z in (z0, z0 + rng.normal(0, 1e-2, z0.shape)):
        r_o = o.error(z)
        r_g, ss = p.residual(z)
        assert np.array_equal(r_g, r_o)                             # bit-exact residuals
        assert abs(ss - r_o @ r_o) <= 1e-12 * (r_o @ r_o)           # summation order only
        cp_o, ri_o, v_o = o.jacobian(z)
        cp_g, ri_g, v_g = p.jacobian(z)
        assert np.array_equal(cp_o, cp_g) and np.array_equal(ri_o, ri_g)
        assert np.array_equal(v_o, v_g)                             # bit-exact quantised central differences
    # against the libm-sincos oracle (what cv::Rodrigues computes) count float flips: expected 0 at this size
    o.set_sincos_mode(0)
    flips = (o.error(z0) != p.residual(z0)[0]).sum()
    o.set_sincos_mode(1)
    assert flips <= 2
    parity_record("undistortion_residual_jacobian_vs_oracle", distorted=bool(distorted), staging=staging, residual_rows=int(len(r_o)), jacobian_nnz=int(len(v_o)), bit_exact=True,
                  float32_flips_against_libm_sincos_oracle=int(flips))


def test_config_flags_and_huber(binding, oracle_mod):
    rig = small_rig(seed=7)
    for cams, markers, objects in [(False, True, True), (True, False, True), (True, True, False), (False, False, True)]:
        o = oracle_mod.Oracle(rig); o.set_config(cams=cams, markers=markers, objects=objects)
        p = binding.Problem(rig, cams=cams, markers=markers, objects=objects)
        z = o.mats2evec()
        assert p.num_vars == o.num_vars == len(z)
        assert np.array_equal(p.residual(z)[0], o.error(z))
        cp_o, ri_o, v_o = o.jacobian(z); cp_g, ri_g, v_g = p.jacobian(z)
        assert np.array_equal(cp_o, cp_g) and np.array_equal(ri_o, ri_g) and np.array_equal(v_o, v_g)
    o = oracle_mod.Oracle(rig); o.set_config(with_huber=True, huber_delta=1.5)
    p = binding.Problem(rig, with_huber=True)
    z = o.mats2evec()
    assert np.array_equal(p.residual(z, huber_delta=1.5)[0], o.error(z))


def test_jacobian_bit_exact_with_marker_tables_in_global_memory(binding, oracle_mod):
    """130 markers: their pose tables (130 x 49 doubles) outgrow the 48 KB of shared memory k_jac_project stages them in
    (launch_jacobian), so the kernel reads them from global memory.  Residuals and Jacobian bit-exact against the oracle."""
    rig = small_rig(seed=29, M=130, F=100, obs_per_frame=12.0)
    assert rig.M * 49 * 8 > 48 * 1024
    o = oracle_mod.Oracle(rig); p = binding.Problem(rig)
    z0 = o.mats2evec()
    for z in (z0, z0 + np.random.default_rng(1).normal(0, 1e-3, z0.shape)):
        assert np.array_equal(p.residual(z)[0], o.error(z))
        cp_o, ri_o, v_o = o.jacobian(z); cp_g, ri_g, v_g = p.jacobian(z)
        assert np.array_equal(cp_o, cp_g) and np.array_equal(ri_o, ri_g) and np.array_equal(v_o, v_g)
    parity_record("jacobian_vs_oracle_marker_tables_in_global_memory", markers=int(rig.M), observations=int(p.num_obs), jacobian_nnz=int(len(v_g)), bit_exact=True)


def test_reduced_system_matches_oracle(binding, oracle_mod):
    rig = small_rig(seed=9, F=50)
    o = oracle_mod.Oracle(rig); p = binding.Problem(rig)
    z = o.mats2evec(); mu = 1234.5
    S_o, b_o, c_o = o.reduced_system(z, mu)
    S_g, b_g, c_g = p.reduced_system(z, mu)
    iu = np.triu_indices(p.n_r)
    scale = np.abs(S_o).max()
    assert np.abs(S_g[iu] - S_o[iu]).max() <= 1e-10 * scale        # sums of products in a different order
    assert np.abs(b_g - b_o).max() <= 1e-10 * np.abs(b_o).max()
    assert abs(c_g - c_o) <= 1e-12 * c_o
    parity_record("reduced_schur_system_vs_oracle", n_r=int(p.n_r), rel_dev_S=float(np.abs(S_g[iu] - S_o[iu]).max() / scale),
                  rel_dev_b=float(np.abs(b_g - b_o).max() / np.abs(b_o).max()), rel_dev_cost=float(abs(c_g - c_o) / c_o), bar=1e-10)


def _oracle_envelope(o, z0, fc_o, z_o, n=3, eps=1e-13):
    """How far the REFERENCE solver's own result moves when z0 is perturbed by eps (relative): the quantised
    central-difference Jacobian (float32 projections, multicam_mapper.cpp:644-648, 976-994) makes the LM trajectory
    jump whenever one projection crosses a float32 rounding boundary, so results are only reproducible to this envelope."""
    rng = np.random.default_rng(123)
    dc, dz = 0.0, 0.0
    for _ in range(n):
        z_p, fc_p, _, _ = o.solve(z0 * (1 + eps * rng.standard_normal(z0.shape)))
        dc = max(dc, abs(fc_p - fc_o) / fc_o); dz = max(dz, np.abs(z_p - z_o).max())
    return dc, dz


@pytest.mark.parametrize("name", ["cfg1", "cfg2"])
def test_lm_first_iterations_match_reference_solver(binding, oracle_mod, name):
    """Teacher-forced parity of SparseLevMarq::step: k iterations from the same z0 (before any float32 flip can
    separate the trajectories) give the same z, cost and damping."""
    rig = synth.make_config(name)
    o = oracle_mod.Oracle(rig); p = binding.Problem(rig)
    z0 = o.mats2evec()
    for k in (1, 3):
        o.set_max_iters(k)
        z_o, fc_o, it_o, tr_o = o.solve(z0)
        z_g, fc_g, it_g, tr_g = p.solve(z0, binding.Problem.default_params(max_iters=k))
        assert it_o == it_g == k
        assert abs(fc_g - fc_o) <= 1e-10 * fc_o                              # north star: per-iteration 1e-10 relative
        assert np.abs(z_g - z_o).max() <= 1e-10 * np.abs(z_o).max()
        assert np.allclose(tr_g[:, 1], tr_o[:, 1], rtol=1e-9, atol=0)         # damping factor after each iteration


def _end_point_bar(dev, envelope, cap):
    """North star: 1e-6 relative on the end point.  The reference's quantised central-difference Jacobian makes ITS OWN end point
    move by `envelope` under a 1e-13 perturbation of z0 (measured in the same test), so a deviation above 1e-6 is accepted only
    while it is inside 4 x that measured envelope (and never beyond `cap`); an envelope that was not observed (0) accepts nothing."""
    if dev <= 1e-6:
        return "1e-6"
    assert envelope > 0 and dev <= min(4 * envelope, cap), (dev, envelope, cap)
    return "envelope"


@pytest.mark.parametrize("name", ["cfg1", "cfg2"])
def test_lm_solve_matches_reference_solver(binding, oracle_mod, name):
    """MultiCamMapper::solve(): device-resident LM vs the oracle driving the reference sparselevmarq.h."""
    rig = synth.make_config(name)
    o = oracle_mod.Oracle(rig); p = binding.Problem(rig)
    z0 = o.mats2evec()
    z_o, fc_o, it_o, tr_o = o.solve(z0)
    z_g, fc_g, it_g, tr_g = p.solve(z0)
    n = min(it_o, it_g)
    assert abs(it_o - it_g) <= 1                                      # stop rule may fire one iteration apart (SURVEY 7)
    d_trace = np.abs(tr_g[:n, 0] - tr_o[:n, 0]) / tr_o[:n, 0]
    assert np.abs(tr_g[:n, 0] - tr_o[:n, 0]).max() <= 1e-8 * tr_o[0, 0]   # per-iteration cost
    assert np.allclose(tr_g[:n, 1], tr_o[:n, 1], rtol=1e-6)               # damping
    # North star: final cost and poses within 1e-6 relative.  The reference itself is only reproducible to a few
    # 1e-6 (see _oracle_envelope: a 1e-13 relative change of z0 moves ITS final cost by 1-4e-6 and z by ~1e-5): _end_point_bar.
    env_c, env_z = _oracle_envelope(o, z0, fc_o, z_o)
    d_cost = abs(fc_g - fc_o) / fc_o
    Tc_o, Tm_o, Tf_o = o.evec2mats(z_o); Tc_g, Tm_g, Tf_g = p.evec2mats(z_g)
    d_pose = max(np.abs(A - B).max() for A, B in ((Tc_o, Tc_g), (Tm_o, Tm_g), (Tf_o, Tf_g)))
    # the device result is as good a solution as the reference's: the oracle evaluates the same cost at z_g
    r_fin = o.error(z_g)
    d_self = abs(r_fin @ r_fin - fc_g) / fc_g
    # how long the two trajectories stay together to 1e-10 (before the first float32 flip of a projection separates them)
    together = int(np.argmax(d_trace > 1e-10)) if (d_trace > 1e-10).any() else n
    rec = parity_record("lm_solve_" + name, iterations_ref=it_o, iterations_gpu=it_g, final_cost_ref=fc_o, final_cost_gpu=fc_g,
                        rel_dev_final_cost=d_cost, max_abs_dev_pose_entries=d_pose, ref_envelope_cost=env_c, ref_envelope_z=env_z,
                        per_iteration_cost_rel_dev=d_trace, iterations_identical_to_1e10=together,
                        oracle_cost_at_gpu_z_rel_dev=d_self, north_star=1e-6)
    rec_c = _end_point_bar(d_cost, env_c, 2e-5); rec_z = _end_point_bar(d_pose, env_z, 5e-5)
    parity_record("lm_solve_" + name + "_bar", cost_passes_by=rec_c, poses_pass_by=rec_z)
    assert d_self <= 1e-12
    # and the solve actually recovers the synthetic ground truth (markers to a few mm)
    assert np.abs(Tm_g[:, :3, 3] - rig.T_marker_true[:, :3, 3]).max() < 5e-3


@pytest.mark.parametrize("name", ["cfg1", "cfg2"])
def test_lm_step_parity_along_the_reference_trajectory(binding, oracle_mod, name):
    """SparseLevMarq::step at EVERY iterate of the reference's own trajectory (not only from z0): start both solvers at the
    reference's k-th iterate and take one step — z, cost and damping agree to 1e-10 wherever the trajectory is, including next
    to the end point.  Together with the envelope measurement this is the whole of the end-point argument: every step is the
    reference's step to 1e-10; the end points differ only through the float32 flips of the reference's quantised Jacobian."""
    rig = synth.make_config(name)
    o = oracle_mod.Oracle(rig); p = binding.Problem(rig)
    z0 = o.mats2evec()
    _, _, it_full, _ = o.solve(z0)
    worst_c = worst_z = 0.0
    zk = z0
    for k in range(it_full):
        o.set_max_iters(1)
        z_o, fc_o, it_o, tr_o = o.solve(zk)
        z_g, fc_g, it_g, tr_g = p.solve(zk, binding.Problem.default_params(max_iters=1))
        assert it_o == it_g == 1
        dc = abs(fc_g - fc_o) / fc_o; dz = np.abs(z_g - z_o).max() / np.abs(z_o).max()
        worst_c = max(worst_c, dc); worst_z = max(worst_z, dz)
        assert dc <= 1e-10 and dz <= 1e-10, (k, dc, dz)
        assert np.allclose(tr_g[:, 1], tr_o[:, 1], rtol=1e-9, atol=0)
        zk = z_o                                                         # teacher forcing: continue from the REFERENCE's iterate
    o.set_max_iters(10000)
    parity_record("lm_step_along_reference_trajectory_" + name, steps=it_full, worst_rel_dev_cost=worst_c, worst_rel_dev_z=worst_z, bar=1e-10)


def test_lm_with_huber_matches_oracle(binding, oracle_mod):
    rig = synth.make_config("cfg1", seed=21)
    rig.det_xy[::37] += 25.0                                            # outliers
    o = oracle_mod.Oracle(rig); o.set_config(with_huber=True)
    p = binding.Problem(rig, with_huber=True)
    z0 = o.mats2evec()
    z_o, fc_o, it_o, tr_o = o.solve(z0)
    z_g, fc_g, it_g, tr_g = p.solve(z0)
    # with outliers the solve runs for dozens of iterations; the trajectories are bit-identical until the first
    # float32 flip, so the tight trace comparison covers the first iterations and the end point is compared
    # against the reference's own reproducibility envelope
    n = min(it_o, it_g, 8)
    assert np.abs(tr_g[:n, 0] - tr_o[:n, 0]).max() <= 1e-8 * tr_o[0, 0]
    assert np.array_equal(tr_g[:n, 5], tr_o[:n, 5])                     # huber delta schedule (optCallBack)
    env_c, env_z = _oracle_envelope(o, z0, fc_o, z_o)
    d_cost = abs(fc_g - fc_o) / fc_o; d_z = np.abs(z_g - z_o).max() / max(1.0, np.abs(z_o).max())
    nn = min(it_o, it_g)
    parity_record("lm_solve_huber_cfg1_outliers", iterations_ref=it_o, iterations_gpu=it_g, rel_dev_final_cost=d_cost, rel_dev_z=d_z,
                  ref_envelope_cost=env_c, ref_envelope_z=env_z, per_iteration_cost_rel_dev=np.abs(tr_g[:nn, 0] - tr_o[:nn, 0]) / tr_o[:nn, 0], north_star=1e-6)
    by_c = _end_point_bar(d_cost, env_c, 1e-3); by_z = _end_point_bar(d_z, env_z, 5e-4)
    parity_record("lm_solve_huber_cfg1_outliers_bar", cost_passes_by=by_c, z_passes_by=by_z)


def test_full_size_properties_cfg3(binding, oracle_mod):
    """cfg 3 (8 cams, 24 markers, 10k frames, ~0.5M observations): residuals bit-exact against the oracle;
    the cost decreases monotonically to the noise floor and the oracle confirms the final cost."""
    rig = synth.make_config("cfg3")
    o = oracle_mod.Oracle(rig); p = binding.Problem(rig)
    z0 = o.mats2evec()
    r_o = o.error(z0); r_g, ss = p.residual(z0)
    assert np.array_equal(r_g, r_o)
    z_g, fc, it, tr = p.solve(z0)
    assert np.all(np.diff(tr[:, 0]) < 0)
    rms = np.sqrt(fc / (8 * p.num_obs))
    assert 0.25 < rms < 0.35                                             # 0.3 px corner noise
    r_fin = o.error(z_g)
    assert abs(r_fin @ r_fin - fc) <= 1e-9 * fc
    o.set_sincos_mode(0)
    flips = int((o.error(z0) != r_g).sum())                               # the same residuals against the libm-sincos oracle (what cv::Rodrigues calls)
    o.set_sincos_mode(1)
    parity_record("cfg3_full_size_residual_and_solve", observations=int(p.num_obs), residual_rows=int(len(r_o)), residual_bit_exact=True,
                  float32_flips_against_libm_sincos_oracle=flips, iterations=int(it), rms_px=float(rms), oracle_cost_at_device_z_rel_dev=float(abs(r_fin @ r_fin - fc) / fc))
    assert flips <= 1e-5 * len(r_o)


def _track_check(label, z_g, cost_g, it_g, z_o, cost_o, it_o, tol):
    """GPU track results against a baseline, frame by frame: iteration counts within one, final cost and pose within `tol` relative."""
    dit = np.abs(it_g.astype(np.int64) - it_o.astype(np.int64))
    dc = np.abs(cost_g - cost_o) / np.maximum(cost_o, 1e-12)
    dz = np.abs(z_g - z_o).max(axis=1) / np.maximum(1.0, np.abs(z_o).max(axis=1))
    assert dit.max() <= 1, (label, np.argmax(dit), it_g[np.argmax(dit)], it_o[np.argmax(dit)])
    assert dc.max() <= tol, (label, np.argmax(dc), dc.max())
    assert dz.max() <= tol, (label, np.argmax(dz), dz.max())
    return dict(worst_rel_dev_cost=dc.max(), worst_rel_dev_z=dz.max(), worst_iteration_count_diff=int(dit.max()))


def _track_against_reference(binding, oracle_mod, case, tol, label):
    """MultiCamMapper::track() batched on the device against (1) the per-frame results stored in tests/golden/track_golden.npz
    (tests/golden/make_golden_track.py; its `baseline` says which solver produced them) and (2) the oracle run now, which drives
    the unmodified reference sparselevmarq.h when oracle/_ref is built and the oracle's restatement of its LM loop otherwise."""
    from golden.make_golden_track import oracle_track, track_rig
    rig = track_rig(case)
    with_huber = case.endswith("huber")
    p = binding.Problem(rig, cams=False, markers=False, objects=True, with_huber=with_huber)
    z0 = p.mats2evec().reshape(-1, 6)
    z_g, cost_g, it_g = p.track_batch(z0)
    g = np.load(os.path.join(ROOT, "tests", "golden", "track_golden.npz"))
    assert np.abs(g[case + "_z_init"] - z0).max() < 1e-12                              # the same rig as when the file was written
    rec_golden = _track_check(label + " vs golden", z_g, cost_g, it_g, g[case + "_z"], g[case + "_cost"], g[case + "_iterations"], tol)
    (z_init, z_o, cost_o, it_o), is_ref = oracle_track(oracle_mod, rig, with_huber)
    assert np.abs(z_init - z0).max() < 1e-12
    rec_live = _track_check(label + " vs oracle", z_g, cost_g, it_g, z_o, cost_o, it_o, tol)
    parity_record(label, frames_checked=int(rig.F), observations=int(p.num_obs), bar=tol,
                  golden=dict(rec_golden, baseline=str(g["baseline"])),
                  oracle=dict(rec_live, baseline="reference sparselevmarq.h" if is_ref else "restated LM loop (aar_oracle_lm_port)"))
    return z_g, cost_g, it_g, p


@pytest.mark.parametrize("with_huber", [False, True])
def test_track_batch_matches_reference_per_frame(binding, oracle_mod, with_huber):
    """MultiCamMapper::track() (mcm.cpp:430-443) batched over frames vs SparseLevMarq::solve(z, f) (2-argument overload: calcDerivates
    Jacobian) frame by frame, stored and run by the oracle (_track_against_reference)."""
    # north star: final cost and poses within 1e-6 relative.  With outliers + Huber the |d| <= 1e-4 pruning of
    # calcDerivates (a discontinuity) and the early stop rule leave the reference itself reproducible to ~1e-5 only.
    _track_against_reference(binding, oracle_mod, "small_rig_huber" if with_huber else "small_rig", 1e-5 if with_huber else 1e-6,
                             "track_small_rig_huber" if with_huber else "track_small_rig")


def test_track_batch_at_cfg5_density(binding, oracle_mod, monkeypatch):
    """BASELINE config 5 density (16 cameras, 64 markers, ~256 marker observations = 2 048 residual rows per frame), 240 frames:
    every frame against the 2-argument SparseLevMarq::solve (_track_against_reference), and the CTA-per-frame kernel against the
    warp-per-frame kernel of round 1 (same arithmetic per residual, different summation order)."""
    z_g, cost_g, it_g, p = _track_against_reference(binding, oracle_mod, "cfg5_240", 1e-6, "track_cfg5_density_240_frames")
    monkeypatch.setenv("AAR_TRACK", "warp")
    z_w, cost_w, it_w = p.track_batch(p.mats2evec().reshape(-1, 6))
    monkeypatch.delenv("AAR_TRACK")
    assert np.array_equal(it_w, it_g)
    dz = np.abs(z_w - z_g).max(); dc = (np.abs(cost_w - cost_g) / cost_g).max()
    parity_record("track_cta_kernel_vs_warp_kernel_cfg5_density", max_abs_dev_z=dz, max_rel_dev_cost=dc)
    assert dz <= 1e-9 and dc <= 1e-9


def test_edge_cases_ragged_inputs(binding, oracle_mod):
    """Ragged / degenerate inputs the reference handles: one camera only (no camera block), one marker only (no marker
    block), frames whose detections were all erased, duplicated detections, and an exact-staging re-run of the Jacobian."""
    # one camera: n_r = 6 (M - 1); one marker: n_r = 6 (C - 1)
    for kw in (dict(C=1, M=5), dict(C=3, M=1)):
        rig = synth.make_rig(F=30, obs_per_frame=4.0 if kw["M"] > 1 else 2.5, seed=17, **kw)
        o = oracle_mod.Oracle(rig); p = binding.Problem(rig)
        z0 = o.mats2evec()
        assert p.num_vars == o.num_vars
        assert np.array_equal(p.residual(z0)[0], o.error(z0))
        cp_o, ri_o, v_o = o.jacobian(z0); cp_g, ri_g, v_g = p.jacobian(z0)
        assert np.array_equal(cp_o, cp_g) and np.array_equal(ri_o, ri_g) and np.array_equal(v_o, v_g)
        for k in (1, 3):
            o.set_max_iters(k)
            z_o, fc_o, it_o, _ = o.solve(z0)
            z_g, fc_g, it_g, _ = p.solve(z0, binding.Problem.default_params(max_iters=k))
            assert it_o == it_g and abs(fc_g - fc_o) <= 1e-10 * fc_o and np.abs(z_g - z_o).max() <= 1e-9 * max(1.0, np.abs(z_o).max())
    # a frame whose only detections belong to an unknown marker: it keeps its pose variables but contributes no rows
    rig = small_rig(seed=19, F=12)
    f_kill = rig.frame_ids[4]
    sel = rig.det_frame == f_kill
    rig.det_marker = rig.det_marker.copy(); rig.det_marker[sel] = 99999
    o = oracle_mod.Oracle(rig); p = binding.Problem(rig)
    z0 = o.mats2evec()
    assert p.num_obs == o.num_rows // 8 == (~sel).sum()
    assert np.array_equal(p.residual(z0)[0], o.error(z0))
    S_o, b_o, c_o = o.reduced_system(z0, 10.0); S_g, b_g, c_g = p.reduced_system(z0, 10.0)
    iu = np.triu_indices(p.n_r)
    assert np.abs(S_g[iu] - S_o[iu]).max() <= 1e-10 * np.abs(S_o).max() and np.abs(b_g - b_o).max() <= 1e-10 * np.abs(b_o).max()
    z_g, fc_g, it_g, tr_g = p.solve(z0, binding.Problem.default_params(max_iters=2))
    col = p.index_maps()["col_frame"][4]
    assert np.array_equal(z_g[col:col + 6], z0[col:col + 6])        # (H + mu I) delta = 0 for a frame without rows: the pose stays put


def test_exact_staging_fallback_matches(binding, oracle_mod, monkeypatch):
    """The FP64-staging instantiation of the Jacobian kernels (taken when a central-difference numerator does not fit a
    float) must give the same normal equations as the float32 staging."""
    rig = small_rig(seed=23, F=30)
    o = oracle_mod.Oracle(rig); z0 = o.mats2evec()
    S32, b32, _ = binding.Problem(rig).reduced_system(z0, 77.0)
    monkeypatch.setenv("AAR_FORCE_EXACT_STAGING", "1")
    S64, b64, _ = binding.Problem(rig).reduced_system(z0, 77.0)
    iu = np.triu_indices(len(b32))
    assert np.abs(S32[iu] - S64[iu]).max() <= 1e-13 * np.abs(S64).max() and np.abs(b32 - b64).max() <= 1e-13 * np.abs(b64).max()


def _normal_equations(o, z):
    """S = J^T J and b = -J^T r with nothing eliminated (objects=False: every column is a camera or marker column), from the
    oracle's bit-exact Jacobian and residuals; the cost is r^T r."""
    import scipy.sparse
    colptr, rowidx, vals = o.jacobian(z)
    r = o.error(z)
    J = scipy.sparse.csc_matrix((vals, rowidx, colptr), shape=(len(r), o.num_vars))
    return (J.T @ J).toarray(), -(J.T @ r), float(r @ r)


def test_tensor_core_assembly_matches_oracle(binding, oracle_mod):
    """k_asm_pairs + k_asm_mruns (FP64 tensor cores, one warp per (frame, camera) pair / (frame, marker) run, aar_assemble.cuh)
    against the oracle's normal equations, which sum the same products in another order: on a rig with duplicated detections,
    an emptied frame, root camera / marker observations, with and without Huber weights, and for every Config flag combination.
    With the frames optimised the oracle eliminates them itself; without, S and b are J^T J and -J^T r of its Jacobian."""
    rig = small_rig(seed=31, F=120)
    # duplicated (frame, cam, marker) detections (only the last one has Jacobian rows) and a frame that loses all its rows
    dup = np.array([5, 40, 41], np.int64)
    rig.det_frame = np.concatenate([rig.det_frame, rig.det_frame[dup]]); rig.det_cam = np.concatenate([rig.det_cam, rig.det_cam[dup]])
    rig.det_marker = np.concatenate([rig.det_marker, rig.det_marker[dup]]); rig.det_xy = np.concatenate([rig.det_xy, rig.det_xy[dup] + 0.5])
    rig.det_marker = rig.det_marker.copy(); rig.det_marker[rig.det_frame == rig.frame_ids[7]] = 99999
    rig.det_xy = rig.det_xy.copy(); rig.det_xy[::29] += 9.0          # outliers, so that the Huber weights differ from 1
    for huber in (False, True):
        for cams, markers, objects in [(True, True, True), (False, True, True), (True, False, True), (True, True, False)]:
            o = oracle_mod.Oracle(rig); o.set_config(cams=cams, markers=markers, objects=objects, with_huber=huber, huber_delta=2.5)
            z0 = o.mats2evec()
            S_g, b_g, c_g = binding.Problem(rig, cams=cams, markers=markers, objects=objects, with_huber=huber).reduced_system(z0, 5.0)
            S_o, b_o, c_o = o.reduced_system(z0, 5.0) if objects else _normal_equations(o, z0)
            assert S_g.shape == S_o.shape and len(b_g) > 0
            iu = np.triu_indices(len(b_g))
            dS = np.abs(S_g[iu] - S_o[iu]).max() / np.abs(S_o).max()
            db = np.abs(b_g - b_o).max() / np.abs(b_o).max()
            dc = abs(c_g - c_o) / c_o
            parity_record("tensor_core_assembly_vs_oracle", huber=huber, cams=cams, markers=markers, objects=objects, n_r=len(b_g),
                          rel_dev_S=dS, rel_dev_b=db, rel_dev_cost=dc, bar_S_b=1e-12, bar_cost=1e-13)
            assert dS <= 1e-12 and db <= 1e-12 and dc <= 1e-13, (huber, cams, markers, objects, dS, db, dc)


# ------------------------------------------------------------------ camera-intrinsics block (SURVEY 8(f) row 4)
def _with_intrinsics(rig):
    """Columns of io_vec with optimize_cam_intrinsics on: [cams | markers | frames | 9 per camera] (multicam_mapper.cpp:445-461)."""
    z_intr = np.concatenate([np.concatenate([[rig.K[c, 0, 0], rig.K[c, 0, 2], rig.K[c, 1, 1], rig.K[c, 1, 2]], rig.dist[c]]) for c in range(rig.C)])
    return z_intr


@pytest.mark.parametrize("distorted", [False, True])
def test_intrinsics_block_jacobian_and_residual_bit_exact(binding, oracle_mod, distorted):
    """MultiCamMapper's default Config optimises the camera intrinsics too (multicam_mapper.h:75-81; find_solution switches it off):
    9 columns per camera — fx, cx, fy, cy by central differences, the five distortion columns structurally present and zero
    (multicam_mapper.cpp:835-893) — and projections that read K from io_vec."""
    rig = small_rig(seed=13, C=3, M=5, F=30, distorted=distorted)
    o = oracle_mod.Oracle(rig); o.set_config(intrinsics=True)
    p = binding.Problem(rig, intrinsics=True)
    z = o.mats2evec()
    assert p.num_vars == o.num_vars == 6 * (rig.C - 1 + rig.M - 1 + rig.F) + 9 * rig.C
    assert np.array_equal(p.mats2evec()[-9 * rig.C:], _with_intrinsics(rig)) and np.array_equal(z[-9 * rig.C:], _with_intrinsics(rig))
    rng = np.random.default_rng(2)
    for trial in range(2):
        zz = z.copy()
        if trial:      # move every parameter, the intrinsics included: the projections must follow io_vec, not the camera files
            zz += rng.normal(0, 1e-3, len(zz)); zz[-9 * rig.C:] += rng.normal(0, 0.5, 9 * rig.C)
        r_g, _ = p.residual(zz)
        assert np.array_equal(r_g, o.error(zz))
        cp_o, ri_o, v_o = o.jacobian(zz)
        cp_g, ri_g, v_g = p.jacobian(zz)
        assert p.jacobian_nnz == len(v_o)
        assert np.array_equal(cp_o, cp_g) and np.array_equal(ri_o, ri_g)
        assert np.array_equal(v_o, v_g), np.abs(v_o - v_g).max()
    n0 = 6 * (rig.C - 1 + rig.M - 1 + rig.F)
    nz_cols = [np.any(v_g[cp_g[n0 + 9 * c + k]:cp_g[n0 + 9 * c + k + 1]] != 0) for c in range(rig.C) for k in range(9)]
    assert nz_cols == [True] * 4 + [False] * 5 + [True] * 4 + [False] * 5 + [True] * 4 + [False] * 5
    parity_record("intrinsics_block_jacobian_vs_oracle", distorted=bool(distorted), nnz=int(len(v_g)), bit_exact=True)


def test_intrinsics_block_lm_steps_and_solve(binding, oracle_mod):
    """SparseLevMarq::step with the intrinsics columns in the system: per-iteration cost / z against the reference solver driving the
    restated MultiCamMapper; end point against its reproducibility envelope."""
    rig = small_rig(seed=14, C=3, M=6, F=40)
    o = oracle_mod.Oracle(rig); o.set_config(intrinsics=True)
    p = binding.Problem(rig, intrinsics=True)
    z0 = o.mats2evec()
    worst = 0.0
    for steps in (1, 2, 3):
        o.set_max_iters(steps)
        z_o, c_o, it_o, tr_o = o.solve(z0)
        prm = binding.Problem.default_params(max_iters=steps, ignore_stop_rules=1)
        z_g, c_g, it_g, tr_g = p.solve(z0, prm)
        dz = np.abs(z_g - z_o).max() / max(np.abs(z_o).max(), 1.0); dc = abs(c_g - c_o) / c_o
        worst = max(worst, dz, dc)
        assert dz <= 1e-10 and dc <= 1e-10, (steps, dz, dc)
        assert np.array_equal(z_g[-9 * rig.C:].reshape(-1, 9)[:, 4:], z0[-9 * rig.C:].reshape(-1, 9)[:, 4:])     # zero columns: the distortion coefficients never move
    o.set_max_iters(10000)
    z_o, c_o, it_o, tr_o = o.solve(z0)
    z_g, c_g, it_g, tr_g = p.solve(z0)
    env_c, env_z = _oracle_envelope(o, z0, c_o, z_o)
    d_cost = abs(c_g - c_o) / c_o
    parity_record("intrinsics_block_lm_vs_reference_solver", first_steps_worst_rel_dev=worst, iterations=[int(it_g), int(it_o)], final_cost=[float(c_g), float(c_o)],
                  rel_dev_final_cost=d_cost, ref_envelope_cost=env_c, north_star=1e-6)
    _end_point_bar(d_cost, env_c, 2e-5)


# bars of a comparison of two LM runs that take the same decisions (also used by test_gpu_lm_loop.py)
def _same(a, b, tol=1e-9):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and np.abs(a - b).max() <= tol * max(np.abs(b).max(), 1e-300)


def _same_cost(plain, z_g, c_g, z_h, c_h):
    """The cost sums squares of residuals of float32-rounded projections (multicam_mapper.cpp:644-648): where the two iterates
    differ in the last bits, a projection may round to the neighbouring float and move its row's square by a float32 step.  The
    costs agree to 1e-12 beyond what the rows that round differently at the two iterates account for (Huber weights are <= 1)."""
    r_g, _ = plain.residual(z_g); r_h, _ = plain.residual(z_h)
    flips = r_g != r_h
    return abs(c_g - c_h) <= 1e-12 * c_h + np.abs(r_g[flips] ** 2 - r_h[flips] ** 2).sum(), int(flips.sum())


def _end_point_dev(p, z0, z_g, z_h):
    """Relative distance of the two end points of a full solve, and the bar it passed.  1e-9 unless a quantised Jacobian entry
    rounded differently on the way: two runs of the SAME loop then also land on end points 7e-9 apart at cfg2 (measured on the
    B200: identical iterations, tries, damping and Huber schedule; the order of the FP64 atomic sums decides which end point), so a
    larger distance must lie within 4 x how far the end point moves under a 1e-13 relative change of z0 (_oracle_envelope), and 1e-6."""
    dz = np.abs(z_g - z_h).max() / np.abs(z_h).max()
    if dz <= 1e-9:
        return dz, "1e-9"
    rng = np.random.default_rng(123)
    env = max(np.abs(p.solve(z0 * (1 + 1e-13 * rng.standard_normal(z0.shape)))[0] - z_h).max() / np.abs(z_h).max() for _ in range(3))
    assert 0 < env and dz <= min(4 * env, 1e-6), (dz, env)
    return dz, "envelope %.2e" % env


def test_graph_resident_loop_equals_host_driven_loop(binding, oracle_mod, monkeypatch):
    """aar_lm_iterate runs SparseLevMarq::solve as nested CUDA-graph WHILE nodes (decisions on the device); AAR_NO_GRAPH=1 keeps the
    host-driven loop (one read-back per try).  Same kernels in the same order: iteration and try counts must be identical and
    iterates, costs and damping equal up to the order of the atomic sums of the assembly (two runs of the SAME loop differ in the last
    bits too), with and without Huber (the hubberDelta annealing lives in the device state)."""
    flips_seen = 0; end_points = {}
    for name, huber in (("cfg1", False), ("cfg2", False), ("cfg1", True)):
        rig = synth.make_config(name)
        p = binding.Problem(rig, with_huber=huber)
        plain = binding.Problem(rig)
        z0 = p.mats2evec()
        monkeypatch.setenv("AAR_NO_GRAPH", "1")
        z_h, c_h, it_h, tr_h = p.solve(z0)
        monkeypatch.delenv("AAR_NO_GRAPH")
        l0 = p.kernel_launches
        z_g, c_g, it_g, tr_g = p.solve(z0)
        cost_ok, flips = _same_cost(plain, z_g, c_g, z_h, c_h); flips_seen += flips
        assert it_g == it_h and cost_ok, (name, huber, it_g, it_h, c_g, c_h, flips)
        end_points[name + ("_huber" if huber else "")] = _end_point_dev(p, z0, z_g, z_h)
        assert np.array_equal(tr_g[:, 3:5], tr_h[:, 3:5]) and _same(tr_g[:, 0], tr_h[:, 0]) and _same(tr_g[:, 1], tr_h[:, 1], 1e-7) and np.array_equal(tr_g[:, 5], tr_h[:, 5])
        assert p.kernel_launches > l0
        # a capped number of iterations and the stop rules switched off (the bench's mode)
        prm = binding.Problem.default_params(max_iters=7, ignore_stop_rules=1)
        monkeypatch.setenv("AAR_NO_GRAPH", "1")
        z_h, c_h, it_h, tr_h = p.solve(z0, prm)
        monkeypatch.delenv("AAR_NO_GRAPH")
        z_g, c_g, it_g, tr_g = p.solve(z0, prm)
        cost_ok, flips = _same_cost(plain, z_g, c_g, z_h, c_h); flips_seen += flips
        assert it_g == it_h == 7 and cost_ok and _same(z_g, z_h) and np.array_equal(tr_g[:, 3:6], tr_h[:, 3:6]), (name, huber, c_g, c_h, flips)
        plain.close()
    parity_record("graph_resident_loop_vs_host_driven_loop", same_iterations_tries_huber=True, rel_tol_z=1e-9, rel_tol_cost=1e-12,
                  rows_rounding_differently=flips_seen, full_solve_end_point_rel_dev=end_points, workloads=["cfg1", "cfg2", "cfg1 + Huber"])
