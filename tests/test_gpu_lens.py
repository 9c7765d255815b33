"""GPU tests of the lens model of the analytic mode (aar_problem_desc::lens_model = 1, DESIGN.md §6g): the CUDA path against the CPU
oracle in the same model (tests/lens_oracle.cpp).  The arithmetic of one observation is the shared header's on both sides, so residuals
and Jacobian entries are held to 1e-12 relative and the record says whether they were bit-identical; sums of products carry the
tolerances written at each assert."""
import ctypes

import numpy as np
import pytest

from aar_b200 import synth
from conftest import parity_record
from test_lens_cpu import LensOracle, build_lens_oracle, csc_to_dense

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def binding():
    from aar_b200 import binding as b
    b.lib()
    return b


@pytest.fixture(scope="module")
def lens_lib(oracle_mod, tmp_path_factory):
    return build_lens_oracle(tmp_path_factory.mktemp("lens_oracle_gpu"))


def _rig_with_erasures(seed=3, **kw):
    args = dict(C=3, M=6, F=40, obs_per_frame=6.0, seed=seed, distorted=True); args.update(kw)
    rig = synth.make_rig(**args)
    extra_f = np.array([rig.det_frame[5], rig.det_frame[9], rig.det_frame[12]], np.int32)
    extra_c = np.array([77, rig.det_cam[9], rig.det_cam[12]], np.int32)
    extra_m = np.array([rig.det_marker[5], 9999, rig.det_marker[12]], np.int32)
    rig.det_frame = np.concatenate([rig.det_frame, extra_f]); rig.det_cam = np.concatenate([rig.det_cam, extra_c])
    rig.det_marker = np.concatenate([rig.det_marker, extra_m]); rig.det_xy = np.concatenate([rig.det_xy, rig.det_xy[[5, 9, 12]] + 0.5])
    return rig


def _to_internal(o, n_r_dev, A):
    """io_vec-ordered reduced quantity [poses | 9 per camera] -> the device's internal order [poses | 12 per camera] (padding zero)."""
    n_p = n_r_dev - 12 * o.nC
    idx = list(range(n_p)) + [n_p + 12 * c + k for c in range(o.nC) for k in range(9)]
    if A.ndim == 1:
        out = np.zeros(n_r_dev); out[idx] = A
    else:
        out = np.zeros((n_r_dev, n_r_dev)); out[np.ix_(idx, idx)] = A
    return out


def _oracle_reduced(o, z, mu, intrinsics):
    """Frame-eliminated normal equations of the oracle's J and r (dense numpy), reduced columns [poses | intrinsics] in io order."""
    r = o.error(z); J = csc_to_dense(*o.jacobian(z), o.num_rows)
    n = o.num_vars; n_i = 9 * o.nC if intrinsics else 0
    n_p = 6 * ((o.nC - 1) + (o.nM - 1)); nf = n - n_p - n_i
    red = np.r_[np.arange(n_p), np.arange(n_p + nf, n)]
    Jr, Jf = J[:, red], J[:, n_p:n_p + nf]
    S = Jr.T @ Jr; b = -Jr.T @ r
    for f in range(nf // 6):
        Jff = Jf[:, 6 * f:6 * f + 6]
        rows = np.nonzero(np.abs(Jff).sum(1))[0]
        Hff = Jff[rows].T @ Jff[rows] + mu * np.eye(6)
        Wt = Jr[rows].T @ Jff[rows]
        S -= Wt @ np.linalg.solve(Hff, Wt.T)
        b -= Wt @ np.linalg.solve(Hff, -Jff[rows].T @ r[rows])
    return S, b, float(r @ r)


def _upper_blocks(n):
    blk = np.arange(n) // 6
    return blk[:, None] <= blk[None, :]


CONFIGS = [(True, True, True, False), (False, True, True, False), (True, False, True, False), (True, True, False, False), (False, False, True, False),
           (True, True, True, True), (False, True, True, True), (True, False, True, True), (True, True, False, True)]


@pytest.mark.parametrize("huber", [False, True])
def test_lens_residual_and_jacobian_match_the_oracle(binding, lens_lib, huber):
    rig = _rig_with_erasures(seed=4)
    if huber:
        rig.det_xy[::11] += 12.0
    worst_r = worst_j = 0.0; identical = True
    for cams, markers, objects, intr in CONFIGS:
        o = LensOracle(lens_lib, rig); o.set_config(cams=cams, markers=markers, objects=objects, intrinsics=intr, with_huber=huber, huber_delta=1.5)
        p = binding.Problem(rig, cams=cams, markers=markers, objects=objects, intrinsics=intr, with_huber=huber, lens=True)
        z = o.mats2evec()
        z = z + np.random.default_rng(1).normal(0, 1e-4, z.shape) * np.maximum(1.0, np.abs(z)) * (np.arange(len(z)) < len(z) - 9 * rig.C * intr)
        assert p.num_vars == o.num_vars == len(z)
        r_o = o.error(z); r_g, ss = p.residual(z, huber_delta=1.5)
        dr = np.abs(r_g - r_o).max()
        assert dr <= 1e-12 * max(1.0, np.abs(r_o).max())
        assert abs(ss - r_o @ r_o) <= 1e-12 * (r_o @ r_o)
        cp_o, ri_o, v_o = o.jacobian(z); cp_g, ri_g, v_g = p.jacobian(z)
        assert np.array_equal(cp_o, cp_g) and np.array_equal(ri_o, ri_g)
        q = binding.Problem(rig, cams=cams, markers=markers, objects=objects, intrinsics=intr)        # the parity path's pattern
        cp_q, ri_q, _ = q.jacobian(z)
        assert np.array_equal(cp_q, cp_g) and np.array_equal(ri_q, ri_g)
        dj = np.abs(v_g - v_o).max() / np.abs(v_o).max()
        assert dj <= 1e-12
        worst_r = max(worst_r, dr); worst_j = max(worst_j, dj)
        identical = identical and np.array_equal(r_g, r_o) and np.array_equal(v_g, v_o)
        p.close(); q.close()
    parity_record("lens_residual_and_jacobian_vs_oracle" + ("_huber" if huber else ""), max_abs_dev_residual_px=worst_r, max_rel_dev_jacobian=worst_j,
                  bit_identical=bool(identical), bar=1e-12)


@pytest.mark.parametrize("shape", [dict(C=3, M=6, F=50), dict(C=6, M=30, F=60)])
def test_lens_reduced_system_matches_the_oracle(binding, lens_lib, shape):
    """Intrinsics on, at z0 and at a perturbed z; the larger rig has 46 blocks (3 SYRK tile rows) with B blocks in the last two."""
    rig = _rig_with_erasures(seed=9, obs_per_frame=min(6.0, shape["M"] / 2), **shape)
    o = LensOracle(lens_lib, rig); o.set_config(intrinsics=True)
    p = binding.Problem(rig, intrinsics=True, lens=True)
    z0 = o.mats2evec(); mu = 1234.5
    z1 = z0 + np.random.default_rng(2).normal(0, 1e-3, z0.shape) * np.maximum(1.0, np.abs(z0) * 1e-2)
    rec = {}
    up = _upper_blocks(p.n_r)
    for label, z in (("z0", z0), ("perturbed", z1)):
        S_o, b_o, c_o = _oracle_reduced(o, z, mu, True)
        S_o, b_o = _to_internal(o, p.n_r, S_o), _to_internal(o, p.n_r, b_o)
        S_g, b_g, c_g = p.reduced_system(z, mu)
        dS = np.abs(np.where(up, S_g - S_o, 0)).max() / np.abs(S_o).max(); db = np.abs(b_g - b_o).max() / np.abs(b_o).max(); dc = abs(c_g - c_o) / c_o
        rec[label] = dict(rel_dev_S=dS, rel_dev_b=db, rel_dev_cost=dc)
        assert dS <= 1e-10 and db <= 1e-10 and dc <= 1e-12, (label, rec[label])
        pad = np.zeros(p.n_r, bool); pad[[p.n_r - 12 * rig.C + 12 * c + k for c in range(rig.C) for k in (9, 10, 11)]] = True
        assert not S_g[pad].any() and not S_g[:, pad].any() and not b_g[pad].any()      # B's padding columns: mu alone
    parity_record("lens_reduced_system_vs_oracle", n_r=int(p.n_r), blocks=int(p.n_r // 6), bar_S_b=1e-10, bar_cost=1e-12, **rec)


@pytest.mark.parametrize("name,intr", [("cfg1", True), ("cfg1", False), ("cfg2", True)])
def test_lens_lm_matches_the_oracle(binding, lens_lib, name, intr):
    rig = synth.make_config(name, distorted=name == "cfg2")
    o = LensOracle(lens_lib, rig); o.set_config(intrinsics=intr)
    p = binding.Problem(rig, intrinsics=intr, lens=True)
    z0 = o.mats2evec()
    worst = {}
    for k in (1, 3):
        o.set_max_iters(k)
        z_o, fc_o, it_o, tr_o = o.solve(z0)
        z_g, fc_g, it_g, tr_g = p.solve(z0, binding.Problem.default_params(max_iters=k))
        assert it_o == it_g == k
        dc = abs(fc_g - fc_o) / fc_o; dz = np.abs(z_g - z_o).max() / np.abs(z_o).max()
        worst[k] = (dc, dz)
        assert dc <= 1e-10 and dz <= 1e-10, (k, dc, dz)
    o.set_max_iters(10000)
    z_o, fc_o, it_o, tr_o = o.solve(z0)
    z_g, fc_g, it_g, tr_g = p.solve(z0, binding.Problem.default_params(max_iters=10000))
    d_cost = abs(fc_g - fc_o) / fc_o; d_z = np.abs(z_g - z_o).max() / max(1.0, np.abs(z_o).max())
    parity_record("lens_lm_solve_" + name + ("_intrinsics" if intr else "_poses"), iterations_ref=it_o, iterations_gpu=it_g, final_cost_ref=fc_o,
                  final_cost_gpu=fc_g, rel_dev_final_cost=d_cost, rel_dev_z=d_z, one_step_rel_dev_cost_z=worst[1], three_steps_rel_dev_cost_z=worst[3], bar=1e-6)
    assert abs(it_o - it_g) <= 1
    assert d_cost <= 1e-6 and d_z <= 1e-6


def _redistorted_rig(seed=12, C=3, M=8, F=150, model=(-0.35, 0.12, 1e-3, -1.5e-3, 0.02)):
    """A pinhole rig whose detections are re-distorted with `model` (strong by default); calib holds a perturbed K and zero distortion."""
    rig = synth.make_rig(C=C, M=M, F=F, obs_per_frame=6.0, seed=seed)
    true = np.tile(np.array(model), (C, 1))
    xy = rig.det_xy.astype(np.float64).reshape(-1, 4, 2)
    K = rig.K[rig.det_cam]
    xn = (xy[..., 0] - K[:, None, 0, 2]) / K[:, None, 0, 0]; yn = (xy[..., 1] - K[:, None, 1, 2]) / K[:, None, 1, 1]
    xd, yd = synth._distort(xn, yn, true[0])
    rig.det_xy = np.stack([xd * K[:, None, 0, 0] + K[:, None, 0, 2], yd * K[:, None, 1, 1] + K[:, None, 1, 2]], -1).reshape(-1, 8).astype(np.float32)
    K_true = rig.K.copy()
    rig.K = rig.K.copy(); rig.K[:, 0, 0] *= 1.02; rig.K[:, 1, 1] *= 0.985; rig.K[:, 0, 2] *= 1.01; rig.K[:, 1, 2] *= 0.99
    r2max = float(np.max(xn ** 2 + yn ** 2))
    return rig, K_true, true, r2max


def _rms(cost, n_obs):
    return float(np.sqrt(cost / (4 * n_obs)))


def test_lens_recovers_a_strong_distortion(binding, lens_lib):
    import copy
    rig, K_true, d_true, r2max = _redistorted_rig()
    truth = copy.copy(rig); truth.K = K_true; truth.dist = d_true
    p_t = binding.Problem(truth, lens=True)                                    # poses only, the true lens model
    z_t, c_t, _, _ = p_t.solve(p_t.mats2evec())
    p_l = binding.Problem(rig, intrinsics=True, lens=True)                     # lens model, intrinsics on, from K off and dist 0
    z_l, c_l, _, _ = p_l.solve(p_l.mats2evec())
    p_r = binding.Problem(rig, intrinsics=True)                                # the reference's intrinsics block from the same start
    z_r, c_r, _, _ = p_r.solve(p_r.mats2evec())
    n = p_l.num_obs
    o_t = LensOracle(lens_lib, truth); o_l = LensOracle(lens_lib, rig); o_l.set_config(intrinsics=True)
    _, co_t, _, _ = o_t.solve(o_t.mats2evec()); _, co_l, _, _ = o_l.solve(o_l.mats2evec())
    bar = _rms(co_l, n) / _rms(co_t, n) + 0.01                                 # what the oracle's CPU solve reaches on this rig, plus 1 %
    rms_t, rms_l, rms_r = _rms(c_t, n), _rms(c_l, n), _rms(c_r, n)
    # the recovered distortion as a displacement field (pixels, fx of the truth) over the covered r^2, not coefficient by coefficient
    lens = z_l[-9 * rig.C:].reshape(rig.C, 9)
    rr = np.linspace(0, np.sqrt(r2max), 40); ang = np.linspace(0, 2 * np.pi, 36, endpoint=False)
    xn = (rr[:, None] * np.cos(ang)).ravel(); yn = (rr[:, None] * np.sin(ang)).ravel()
    worst_field = 0.0
    for c in range(rig.C):
        dx_t, dy_t = synth._distort(xn, yn, d_true[c]); dx_l, dy_l = synth._distort(xn, yn, lens[c, 4:])
        worst_field = max(worst_field, float(np.max(np.hypot(dx_l - dx_t, dy_l - dy_t)) * K_true[c, 0, 0]))
    parity_record("lens_recovery_strong_distortion", rms_true_model=rms_t, rms_lens_refined=rms_l, rms_reference_intrinsics_block=rms_r,
                  ratio_bar_from_oracle=bar, oracle_rms_true=_rms(co_t, n), oracle_rms_refined=_rms(co_l, n), r2_covered=r2max,
                  displacement_field_max_dev_px=worst_field)
    assert rms_l <= bar * rms_t, (rms_l, rms_t, bar)
    assert rms_r > 1.5 * rms_t, (rms_r, rms_t)
    assert worst_field < 0.5, worst_field


def test_held_intrinsics(binding, lens_lib):
    rig = _rig_with_erasures(seed=6, F=50)
    p = binding.Problem(rig, intrinsics=True, lens=True)
    q = binding.Problem(rig, intrinsics=True, lens=True)
    z0 = p.mats2evec(); mu = 77.0
    flags = np.array([1, 2, 3], np.uint8)                       # camera 0 holds A, camera 1 holds B, camera 2 both
    p.set_fixed_intrinsics(flags)
    S, b, c = p.reduced_system(z0, mu); S_q, b_q, c_q = q.reduced_system(z0, mu)
    held = np.zeros(p.n_r, bool); n_p = p.n_r - 12 * rig.C
    for cam, f in enumerate(flags):
        if f & 1: held[n_p + 12 * cam:n_p + 12 * cam + 6] = True
        if f & 2: held[n_p + 12 * cam + 6:n_p + 12 * cam + 12] = True
    up = _upper_blocks(p.n_r)
    S_ref = np.where(held[:, None] | held[None, :], 0.0, S_q); b_ref = np.where(held, 0.0, b_q)
    assert not S[held].any() and not S[:, held].any() and not b[held].any() and c == c_q
    dS = np.abs(np.where(up, S - S_ref, 0)).max() / np.abs(S_q).max(); db = np.abs(b - b_ref).max() / np.abs(b_q).max()
    assert dS <= 1e-13 and db <= 1e-13, (dS, db)
    z, cost, it, _ = p.solve(z0, binding.Problem.default_params(max_iters=20))
    io = np.zeros(len(z0), bool); ni = len(z0) - 9 * rig.C
    for cam, f in enumerate(flags):
        if f & 1: io[ni + 9 * cam:ni + 9 * cam + 6] = True
        if f & 2: io[ni + 9 * cam + 6:ni + 9 * cam + 9] = True
    assert np.array_equal(z[io], z0[io]) and not np.array_equal(z[~io], z0[~io])
    parity_record("lens_held_intrinsics", rel_dev_S=dS, rel_dev_b=db, iterations=it)
    # the no-free-column check sees the intrinsics flags
    p.set_fixed(cams=np.ones(rig.C), markers=np.ones(rig.M), frames=np.ones(rig.F))          # intrinsics of camera 0 still free
    with pytest.raises(binding.AarError, match="no free column"):
        p.set_fixed_intrinsics(np.full(rig.C, 3, np.uint8))
    p.set_fixed(); p.set_fixed_intrinsics(None)
    with pytest.raises(binding.AarError):
        p.set_fixed_intrinsics(np.array([4, 0, 0], np.uint8))
    with pytest.raises(ValueError):
        p.set_fixed_intrinsics(np.zeros(rig.C + 1, np.uint8))
    r = binding.Problem(rig, lens=True)
    with pytest.raises(binding.AarError):
        r.set_fixed_intrinsics(np.zeros(rig.C, np.uint8))      # no intrinsics to hold


def test_lens_refusals(binding):
    rig = _rig_with_erasures(seed=2)
    L = binding.lib()
    for kw, want in ((dict(lens=True, analytic=False), 3), (dict(lens=True, analytic=True, corners_undistorted=True), 3)):
        d, keep = binding.Problem._desc(rig, True, True, True, True, False, 0, None, 0, 1, 0.0, False, **kw)
        h = ctypes.c_void_p()
        assert L.aar_problem_create(ctypes.byref(d), ctypes.byref(h)) == want, kw
    d, keep = binding.Problem._desc(rig, True, True, True, True, False, 0, None, 0, 1, 0.0, False, True)
    d.lens_model = 2
    h = ctypes.c_void_p()
    assert L.aar_problem_create(ctypes.byref(d), ctypes.byref(h)) == 3
    with pytest.raises(binding.AarError):                      # the pinhole analytic mode still has no intrinsics block
        binding.Problem(rig, intrinsics=True, analytic=True)


def test_lens_error_report(binding, lens_lib):
    rig = _rig_with_erasures(seed=5)
    rig.det_xy[::13] += 9.0
    p = binding.Problem(rig, with_huber=True, intrinsics=True, lens=True)
    o = LensOracle(lens_lib, rig); o.set_config(intrinsics=True)                           # Huber off
    z = p.mats2evec()
    rep = p.error_report(z)
    r = o.error(z).reshape(-1, 8)
    s = np.sum(r * r, 1); e = np.sqrt(s / 4)
    det = rep["det_err"]; ok = ~np.isnan(det)
    assert ok.sum() == len(e) == rep["observations"]
    dev = np.abs(np.sort(det[ok]) - np.sort(e)).max()
    assert dev <= 1e-12 * e.max()
    assert abs(rep["sum_sq"] - s.sum()) <= 1e-12 * s.sum()
    parity_record("lens_error_report_vs_numpy", max_abs_dev_px=dev, rel_dev_sum=abs(rep["sum_sq"] - s.sum()) / s.sum())


def test_fixed_intrinsics_on_the_reference_intrinsics_block(binding):
    """aar_set_fixed_intrinsics on a handle of the parity path (central differences, no lens model): a held block A zeroes its rows and
    columns of S and b, and its entries of io_vec stay z0 after a solve; block B has no live column there, so a mask that leaves only
    B free is refused."""
    rig = _rig_with_erasures(seed=7, F=40, distorted=False)
    p = binding.Problem(rig, intrinsics=True); q = binding.Problem(rig, intrinsics=True)
    z0 = p.mats2evec(); mu = 55.0
    flags = np.array([1, 0, 3], np.uint8)
    p.set_fixed_intrinsics(flags)
    S, b, c = p.reduced_system(z0, mu); S_q, b_q, c_q = q.reduced_system(z0, mu)
    n_p = p.n_r - 12 * rig.C
    held = np.zeros(p.n_r, bool)
    held[n_p:n_p + 6] = True; held[n_p + 24:n_p + 36] = True
    up = _upper_blocks(p.n_r)
    assert not S[held].any() and not S[:, held].any() and not b[held].any() and c == c_q
    assert np.abs(S_q[held][:, held]).max() > 0
    dS = np.abs(np.where(up, S - np.where(held[:, None] | held[None, :], 0.0, S_q), 0)).max() / np.abs(S_q).max()
    db = np.abs(b - np.where(held, 0.0, b_q)).max() / np.abs(b_q).max()
    assert dS <= 1e-13 and db <= 1e-13, (dS, db)
    z, _, it, _ = p.solve(z0, binding.Problem.default_params(max_iters=5))
    ni = len(z0) - 9 * rig.C
    io = np.zeros(len(z0), bool); io[ni:ni + 6] = True; io[ni + 18:ni + 27] = True
    assert np.array_equal(z[io], z0[io]) and not np.array_equal(z[ni + 9:ni + 13], z0[ni + 9:ni + 13])
    parity_record("parity_path_held_intrinsics", rel_dev_S=dS, rel_dev_b=db, iterations=it)
    p.set_fixed(cams=np.ones(rig.C), markers=np.ones(rig.M), frames=np.ones(rig.F))
    with pytest.raises(binding.AarError, match="no free column"):      # only the B blocks, explicit zero columns, would be left
        p.set_fixed_intrinsics(np.ones(rig.C, np.uint8))
    p.set_fixed_intrinsics(np.array([1, 1, 0], np.uint8))              # camera 2's fx cx fy cy are free


# ------------------------------------------------------------------ the find_solution app
@pytest.fixture(scope="module")
def host_bins():
    import os
    import subprocess
    from conftest import ROOT
    binding_mod = __import__("aar_b200.binding", fromlist=["build"])
    binding_mod.build()
    host = os.path.join(ROOT, "automatic-ar_b200", "host")
    subprocess.run(["make", "-s", "-C", host], check=True)
    return host


def _run_app(host, folder, *opts, check=True):
    import os
    import subprocess
    r = subprocess.run([os.path.join(host, "find_solution"), str(folder), "0.05", *opts], capture_output=True, text=True)
    if check:
        assert r.returncode == 0, (opts, r.returncode, r.stdout[-2000:], r.stderr[-2000:])
    return r


def _final_rms(stdout):
    """sqrt(final_error / (4 observations)) of the last solve an app run printed"""
    cost = float(stdout.rsplit("final_error: ", 1)[1].split()[0])
    n_obs = int(stdout.rsplit("error size: ", 1)[1].split()[0]) // 8
    return float(np.sqrt(cost / (4 * n_obs)))


@pytest.mark.parametrize("reject", [False, True], ids=["plain", "reject_outliers"])
def test_find_solution_refine_intrinsics(host_bins, tmp_path, reject):
    """A synthetic dataset whose calib.yml holds a perturbed K and zero distortion, detections through a strong lens:
    find_solution -refine-intrinsics writes K and dist close to the truth and corners undistorted with them, so that re-reading the
    file and solving the poses alone on the parity path reaches the refined solve's RMS."""
    import shutil
    # seed 3: the Initializer, fed calib.yml's wrong model, starts the solve in the basin of the truth (on some rigs it does not, and
    # only -reject-outliers recovers; that is the Initializer's start, not the solve: the oracle ends at the same point)
    rig, K_true, d_true, r2max = _redistorted_rig(seed=3)
    if reject:
        rig.det_xy = rig.det_xy.copy(); rig.det_xy[::53] += 25.0
    folders = {k: tmp_path / k for k in ("plain", "refine", "held", "reread")}
    for k in ("plain", "refine", "held"):
        synth.write_dataset(str(folders[k]), rig)
    extra = ["-reject-outliers", "3"] if reject else []
    out_plain = _run_app(host_bins, folders["plain"], *extra).stdout
    out_ref = _run_app(host_bins, folders["refine"], "-refine-intrinsics", *extra).stdout
    if reject:
        assert int(out_ref.split("removed ")[1].split()[0]) > 0
    sol = synth.read_solution_file(str(folders["refine"] / "final.solution"))
    lens = sol["vec"][-9 * rig.C:].reshape(rig.C, 9)
    f_dev = max(abs(lens[c, k] - K_true[c, i, i]) / K_true[c, i, i] for c in range(rig.C) for k, i in ((0, 0), (2, 1)))
    pp_dev = max(abs(lens[c, k] - K_true[c, i, 2]) for c in range(rig.C) for k, i in ((1, 0), (3, 1)))
    rr = np.linspace(0, np.sqrt(r2max), 40); ang = np.linspace(0, 2 * np.pi, 36, endpoint=False)
    xn = (rr[:, None] * np.cos(ang)).ravel(); yn = (rr[:, None] * np.sin(ang)).ravel()
    field = max(float(np.max(np.hypot(*(np.subtract(synth._distort(xn, yn, lens[c, 4:]), synth._distort(xn, yn, d_true[c])))))) * K_true[c, 0, 0]
                for c in range(rig.C))
    # the written corners: re-read the file, poses only on the parity path (the find_solution default)
    folders["reread"].mkdir()
    shutil.copy(folders["refine"] / "final.solution", folders["reread"] / "refined.solution")
    out_re = _run_app(host_bins, folders["reread"], "-init", str(folders["reread"] / "refined.solution")).stdout
    rms_plain, rms_ref, rms_re = _final_rms(out_plain), _final_rms(out_ref), _final_rms(out_re)
    # held: camera 1 keeps calib.yml's K and dist byte for byte, and p1 p2 k3 of every camera stay calib.yml's
    _run_app(host_bins, folders["held"], "-refine-intrinsics", "-fix-intrinsics", "1", "-fix-p1p2k3", *extra)
    ini = synth.read_solution_file(str(folders["held"] / "initial.solution"))["vec"][-9 * rig.C:].reshape(rig.C, 9)
    held = synth.read_solution_file(str(folders["held"] / "final.solution"))["vec"][-9 * rig.C:].reshape(rig.C, 9)
    assert held[1].tobytes() == ini[1].tobytes()
    assert held[:, 6:].tobytes() == ini[:, 6:].tobytes()
    assert not np.array_equal(held[0, :6], ini[0, :6]) and not np.array_equal(held[2, :6], ini[2, :6])
    # -init with -refine-intrinsics: a .solution file holds no raw corners
    r = _run_app(host_bins, folders["reread"], "-init", str(folders["reread"] / "refined.solution"), "-refine-intrinsics", check=False)
    assert r.returncode == 1 and "-refine-intrinsics" in r.stderr
    parity_record("lens_find_solution_refine_intrinsics", reject_outliers=reject, focal_rel_dev=f_dev, principal_point_dev_px=pp_dev,
                  displacement_field_max_dev_px=field, rms_unrefined=rms_plain, rms_refined=rms_ref, rms_reread_pose_only_parity=rms_re)
    assert f_dev < 5e-3 and pp_dev < 8.0 and field < 1.0, (f_dev, pp_dev, field)
    assert rms_ref < 0.45 and rms_re <= 1.02 * rms_ref, (rms_ref, rms_re)     # noise 0.3 px per coordinate: about 0.39 px
    if not reject:                                                            # (the unrefined run's rejection removes good detections too)
        assert rms_plain > 1.5 * rms_ref, (rms_plain, rms_ref)
