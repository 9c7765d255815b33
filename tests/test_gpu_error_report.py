"""Reprojection-error report (aar_error_report, include/aar_cuda.h) and reject-and-resolve in the facade and apps.
Per-detection errors are pinned bit for bit against numpy applied to aar_eval_residual with the Huber weights off; entity statistics
against bincounts; percentiles against np.partition; the facade's re-solve after rejection against a control solve of the same
detections deleted by hand."""
import copy
import ctypes as C
import os
import re
import struct
import subprocess

import numpy as np
import pytest

from conftest import ROOT, parity_record
from aar_b200 import synth

HOST = os.path.join(ROOT, "automatic-ar_b200", "host")
Q = (0.0, 0.5, 0.9, 0.99, 1.0)


@pytest.fixture(scope="module")
def binding():
    from aar_b200 import binding as b
    b.build()
    return b


@pytest.fixture(scope="module")
def host_bins(binding):
    subprocess.run(["make", "-s", "-C", HOST], check=True)
    return HOST


def test_report_struct_layout_matches_header(binding):
    hdr = open(os.path.join(ROOT, "include", "aar_cuda.h")).read()
    m = re.search(r"static_assert\(sizeof\(aar_error_report_out\) == (\d+)", hdr)
    assert m and C.sizeof(binding.ErrorReportOut) == int(m.group(1)) == 128
    assert "aar_error_report" in binding.EXPORTS


# ------------------------------------------------------------------ helpers
def obs_errors(r):
    """e = sqrt(s / 4), s summed column by column (one product and one add at a time)."""
    r = r.reshape(-1, 8)
    s = r[:, 0] * r[:, 0]
    for j in range(1, 8):
        s = s + r[:, j] * r[:, j]
    return np.sqrt(s / 4), s


def row_order(rig):
    """desc index of every observation in row order: known ids only, frame then camera ascending, detection order."""
    fi = np.searchsorted(rig.frame_ids, rig.det_frame); ci = np.searchsorted(rig.cam_ids, rig.det_cam); mi = np.searchsorted(rig.marker_ids, rig.det_marker)
    ok = (fi < rig.F) & (ci < rig.C) & (mi < rig.M)
    ok[ok] &= (rig.frame_ids[fi[ok]] == rig.det_frame[ok]) & (rig.cam_ids[ci[ok]] == rig.det_cam[ok]) & (rig.marker_ids[mi[ok]] == rig.det_marker[ok])
    idx = np.nonzero(ok)[0]
    return idx[np.lexsort((np.arange(len(idx)), ci[idx], fi[idx]))]


def with_extras(rig):
    """appends a duplicate of detection 0 (same frame / camera / marker, other corners) and a detection of an unknown marker id"""
    rig = copy.copy(rig)
    dup_xy = rig.det_xy[0] + np.float32(0.75)
    rig.det_frame = np.concatenate([rig.det_frame, rig.det_frame[:1], rig.det_frame[:1]])
    rig.det_cam = np.concatenate([rig.det_cam, rig.det_cam[:1], rig.det_cam[:1]])
    rig.det_marker = np.concatenate([rig.det_marker, rig.det_marker[:1], np.array([rig.marker_ids.max() + 1000], np.int32)])
    rig.det_xy = np.concatenate([rig.det_xy, dup_xy[None], rig.det_xy[:1]]).astype(np.float32)
    return rig


def kth(e, q):
    k = int(np.floor(q * (len(e) - 1)))
    return np.partition(e, k)[k]


# ------------------------------------------------------------------ the report against numpy
@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["cfg1", "cfg2_distorted"])
@pytest.mark.parametrize("analytic", [False, True])
def test_report_matches_numpy_on_eval_residual(binding, workload, analytic):
    rig = synth.make_config("cfg1") if workload == "cfg1" else synth.make_config("cfg2", distorted=True)
    rig = with_extras(rig)
    p = binding.Problem(rig, analytic=analytic)
    z = p.mats2evec()
    z = z + np.random.default_rng(3).normal(0, 1e-3, z.shape)          # away from the starting point: errors of a few pixels
    rep = p.error_report(z, Q)
    r, cost = p.residual(z, huber_delta=2.5)                          # non-Huber handle: unweighted residuals
    e, s = obs_errors(r)
    order = row_order(rig)
    assert len(order) == p.num_obs == rep["observations"] and rep["not_in_problem"] == rig.N - p.num_obs == 1
    want = np.full(rig.N, np.nan); want[order] = e
    assert np.array_equal(rep["det_err"], want, equal_nan=True)        # bit-identical; NaN exactly where not in the problem
    assert np.isnan(rep["det_err"][-1]) and np.isfinite(rep["det_err"][-2])   # the unknown marker / the appended duplicate
    # entity statistics
    im = p.index_maps()
    for ent, idx, n in (("cam", im["cam_idx"], rig.C), ("marker", im["marker_idx"], rig.M), ("frame", im["frame_idx"], rig.F)):
        assert np.array_equal(rep[ent + "_count"], np.bincount(idx, minlength=n)), ent
        mx = np.zeros(n); np.maximum.at(mx, idx, e)
        assert np.array_equal(rep[ent + "_max"], mx), ent
        ss = np.bincount(idx, weights=s, minlength=n)
        assert np.all(np.abs(rep[ent + "_sum_sq"] - ss) <= 1e-12 * np.abs(ss)), ent
    assert abs(rep["cam_sum_sq"].sum() - cost) <= 1e-12 * cost and abs(rep["sum_sq"] - cost) <= 1e-12 * cost
    # exact percentiles
    assert np.array_equal(rep["q_value"], [kth(e, q) for q in Q])
    # a Huber handle reports the unweighted errors
    ph = binding.Problem(rig, with_huber=True, analytic=analytic)
    reph = ph.error_report(z, Q)
    for k in ("det_err", "cam_count", "cam_max", "marker_max", "frame_max", "q_value"):
        assert np.array_equal(reph[k], rep[k], equal_nan=True), k
    parity_record("error_report_vs_numpy_" + workload + ("_analytic" if analytic else ""), observations=int(p.num_obs),
                  q=list(Q), q_value=rep["q_value"], rel_dev_total_sum_sq=abs(rep["sum_sq"] - cost) / cost, bar="bit-identical errors, 1e-12 sums")


@pytest.mark.gpu
def test_percentiles_one_observation_and_ties(binding):
    base = synth.make_config("cfg1")
    one = copy.copy(base)
    for k in ("det_frame", "det_cam", "det_marker", "det_xy"):
        setattr(one, k, getattr(base, k)[:1].copy())
    p = binding.Problem(one)
    rep = p.error_report(p.mats2evec(), Q)
    e, _ = obs_errors(p.residual(p.mats2evec())[0])
    assert rep["observations"] == 1 and np.array_equal(rep["q_value"], np.full(len(Q), e[0]))
    # many ties: one detection repeated 3000 times next to the rig's own
    tie = copy.copy(base)
    rep_n = 3000
    tie.det_frame = np.concatenate([np.repeat(base.det_frame[:1], rep_n), base.det_frame])
    tie.det_cam = np.concatenate([np.repeat(base.det_cam[:1], rep_n), base.det_cam])
    tie.det_marker = np.concatenate([np.repeat(base.det_marker[:1], rep_n), base.det_marker])
    tie.det_xy = np.concatenate([np.repeat(base.det_xy[:1], rep_n, axis=0), base.det_xy])
    p = binding.Problem(tie)
    z = p.mats2evec()
    qs = (0.0, 0.1, 0.25, 0.5, 0.6, 0.9, 0.99, 1.0)
    rep = p.error_report(z, qs)
    e, _ = obs_errors(p.residual(z)[0])
    assert len(np.unique(e)) < len(e) // 2
    assert np.array_equal(rep["q_value"], [kth(e, q) for q in qs])


@pytest.mark.gpu
def test_sharded_handle_and_bad_q_are_refused(binding):
    rig = synth.make_config("cfg1")
    try:
        p = binding.Problem(rig, rank=0, world_size=2)       # a frame shard; no communicator is needed to create it
    except binding.AarError as e:
        pytest.skip(f"a world-2 handle cannot be created on one GPU without a communicator: {e}")
    with pytest.raises(binding.AarError, match=r"status 1\).*single-rank"):
        p.error_report(p.mats2evec())
    p1 = binding.Problem(rig)
    with pytest.raises(binding.AarError, match="status 1"):
        p1.error_report(p1.mats2evec(), q=(0.5, 1.5))


# ------------------------------------------------------------------ reject and re-solve through the facade
def write_solution_dict(path, d, keep=None):
    """.solution from read_solution_file's dict (same vector bits), keeping only the detections where keep is true and the frames
    that still have one"""
    keep = np.ones(len(d["det_frame"]), bool) if keep is None else keep
    df, dc, dm, xy = d["det_frame"][keep], d["det_cam"][keep], d["det_marker"][keep], d["det_xy"][keep]
    fk = np.isin(d["frame_ids"], df)
    p0 = 6 * (len(d["cam_ids"]) - 1 + len(d["marker_ids"]) - 1); nf = len(d["frame_ids"])
    vec = np.concatenate([d["vec"][:p0], d["vec"][p0:p0 + 6 * nf].reshape(-1, 6)[fk].reshape(-1), d["vec"][p0 + 6 * nf:]])
    frame_ids = d["frame_ids"][fk]
    with open(path, "wb") as fh:
        fh.write(struct.pack("<Q", len(d["cam_ids"]))); fh.write(d["cam_ids"].astype("<i4").tobytes())
        fh.write(struct.pack("<Q", d["root_cam"]))
        for w, h in d["image_sizes"]:
            fh.write(struct.pack("<ii", w, h))
        fh.write(struct.pack("<Q", len(d["marker_ids"]))); fh.write(d["marker_ids"].astype("<i4").tobytes())
        fh.write(struct.pack("<Q", d["root_marker"])); fh.write(struct.pack("<d", d["marker_size"]))
        fh.write(struct.pack("<Q", len(frame_ids))); fh.write(frame_ids.astype("<i4").tobytes())
        fh.write(vec.astype("<f8").tobytes())
        frames = list(frame_ids)
        fh.write(struct.pack("<Q", len(frames)))
        for f in frames:
            cams = [c for c in np.unique(dc[df == f])]
            fh.write(struct.pack("<iQ", int(f), len(cams)))
            for c in cams:
                sel = (df == f) & (dc == c)
                fh.write(struct.pack("<iQ", int(c), int(sel.sum())))
                rec = np.zeros(int(sel.sum()), dtype=[("id", "<i4"), ("xy", "<f4", 8)]); rec["id"] = dm[sel]; rec["xy"] = xy[sel]
                fh.write(rec.tobytes())
        fh.write(struct.pack("<4?", *d["flags"]))


def pose_distance(d, rig):
    """max rotation (Frobenius of R - R_true) and translation deviation of the camera and marker poses of a .solution"""
    nc, nm = rig.C - 1, rig.M - 1
    v = d["vec"][:6 * (nc + nm)].reshape(-1, 6)
    T_true = np.concatenate([rig.T_cam_true[1:], rig.T_marker_true[1:]])
    dr = np.linalg.norm(synth.rodrigues(v[:, :3]) - T_true[:, :3, :3], axis=(1, 2)).max()
    dt = np.abs(v[:, 3:] - T_true[:, :3, 3]).max()
    return float(dr), float(dt)


def run(args):
    return subprocess.run(args, check=True, capture_output=True, text=True).stdout


@pytest.mark.gpu
def test_reject_and_resolve_matches_control_solve(binding, host_bins, tmp_path):
    rig = copy.copy(synth.make_config("cfg1"))
    rig.det_xy = rig.det_xy.copy()
    bad = np.arange(0, rig.N, 37)
    rig.det_xy[bad] += 25.0
    synth.write_solution_file(str(tmp_path / "initial.solution"), rig)
    out = run([os.path.join(host_bins, "find_solution"), str(tmp_path), "0.05", "-init", str(tmp_path / "initial.solution"), "-with-huber"])
    assert "removed" not in out and "report" not in out                    # without the option: no report lines
    first_path = str(tmp_path / "final_with_huber.solution")
    first = synth.read_solution_file(first_path)
    # at 5 px the report flags the injected detections.  cfg 1 has about 6 detections per frame: Huber bounds an outlier's pull but does
    # not remove it, so a frame pose it drags can bring an outlier under 5 px and put co-observed detections above (recorded below)
    p = binding.Problem(rig)
    n = p.num_vars
    rep = p.error_report(first["vec"][:n], Q)
    flagged = np.nonzero(rep["det_err"] > 5.0)[0]
    injected = np.zeros(rig.N, bool); injected[bad] = True
    assert np.mean(rep["det_err"][bad] > 5.0) >= 0.9
    # the facade: solution_report -reject
    rep_out = run([os.path.join(host_bins, "solution_report"), first_path, "-reject", "5", str(tmp_path / "rejected.solution")])
    m = re.search(r"removed (\d+) of (\d+) detections above 5 px", rep_out)
    assert m and int(m.group(1)) == len(flagged) and int(m.group(2)) == rig.N
    got = synth.read_solution_file(str(tmp_path / "rejected.solution"))
    # the control: the same detections deleted here, the first solve's poses, solved through find_solution -init
    ctrl_dir = tmp_path / "control"; os.makedirs(ctrl_dir)
    keep = np.ones(rig.N, bool); keep[flagged] = False
    write_solution_dict(str(ctrl_dir / "control.solution"), first, keep)
    ctrl_out = run([os.path.join(host_bins, "find_solution"), str(ctrl_dir), "0.05", "-init", str(ctrl_dir / "control.solution")])
    ctrl = synth.read_solution_file(str(ctrl_dir / "final.solution"))
    for k in ("frame_ids", "det_frame", "det_cam", "det_marker", "det_xy"):
        assert np.array_equal(got[k], ctrl[k]), k
    # the same solve: same detections, same start, same settings.  Not asserted bit for bit: the device LM is not bit-reproducible run to
    # run (atomic accumulation of the normal equations; 3e-13 on the poses of two solves of one input) and 15 iterations amplify that
    c_got = float(rep_out.split("final_error:")[1].split()[0]); c_ctrl = float(ctrl_out.split("final_error:")[1].split()[0])
    it_got = int(rep_out.split("iterations:")[1].split()[0]); it_ctrl = int(ctrl_out.split("iterations:")[1].split()[0])
    n_pose = 6 * (rig.C - 1 + rig.M - 1)
    d_vec = float(np.abs(got["vec"] - ctrl["vec"]).max())
    assert got["flags"] == ctrl["flags"] and abs(it_got - it_ctrl) <= 1
    assert abs(c_got - c_ctrl) <= 1e-9 * c_ctrl and d_vec <= 5e-5, (c_got, c_ctrl, d_vec)
    d_huber, d_reject = pose_distance(first, rig), pose_distance(got, rig)
    parity_record("reject_and_resolve_cfg1_outliers", flagged=int(len(flagged)), injected=int(len(bad)), injected_flagged=int(injected[flagged].sum()), min_error_injected=float(rep["det_err"][bad].min()),
                  max_error_not_injected=float(np.delete(rep["det_err"], bad).max()), huber_kept_rot_trans=d_huber,
                  rejected_resolved_rot_trans=d_reject, q_value_before=rep["q_value"], cost_facade_control=[c_got, c_ctrl], iterations_facade_control=[it_got, it_ctrl],
                  max_abs_dev_vec_facade_control=d_vec, max_abs_dev_pose_part=float(np.abs(got["vec"][:n_pose] - ctrl["vec"][:n_pose]).max()))
    assert d_reject[0] < d_huber[0] and d_reject[1] < d_huber[1], (d_reject, d_huber)
    # and reports again on what is left
    after = rep_out.split("report after")[1]
    assert int(re.search(r"total observations (\d+)", after).group(1)) == rig.N - len(flagged)


@pytest.mark.gpu
def test_reject_drops_a_frame_whose_detections_are_all_outliers(host_bins, tmp_path):
    rig = copy.copy(synth.make_config("cfg1"))
    rig.det_xy = rig.det_xy.copy()
    f_bad = int(rig.frame_ids[len(rig.frame_ids) // 2])
    sel = rig.det_frame == f_bad
    rig.det_xy[sel] += np.random.default_rng(5).normal(0, 40.0, rig.det_xy[sel].shape).astype(np.float32)
    a = str(tmp_path / "initial.solution")
    synth.write_solution_file(a, rig)
    out = run([os.path.join(host_bins, "find_solution"), str(tmp_path), "0.05", "-init", a, "-reject-outliers", "5"])
    m = re.search(r"removed (\d+) of (\d+) detections above 5 px", out)
    assert m and int(m.group(1)) >= int(sel.sum()) and int(m.group(2)) == rig.N
    assert out.count("final_error:") == 2
    fin = synth.read_solution_file(str(tmp_path / "final.solution"))
    assert f_bad not in set(fin["frame_ids"].tolist()) and f_bad not in set(fin["det_frame"].tolist())
    assert len(fin["frame_ids"]) == rig.F - 1


# ------------------------------------------------------------------ solution_report against the binding
def yaml_mats(path):
    txt = open(path).read()
    secs = {}
    for name, nxt in (("transforms_to_root_cam", "transforms_to_root_marker"), ("transforms_to_root_marker", "root_marker_to_root_cam"), ("root_marker_to_root_cam", None)):
        sec = txt.split(name + ":")[1]
        if nxt:
            sec = sec.split(nxt + ":")[0]
        secs[name] = np.array([[float(v) for v in m.replace("\n", " ").split(",")] for m in re.findall(r"data: \[([^\]]*)\]", sec)]).reshape(-1, 4, 4)
    return secs


@pytest.mark.gpu
def test_solution_report_prints_the_binding_values(binding, host_bins, tmp_path):
    rig = copy.copy(synth.make_config("cfg1"))
    a, b, y = str(tmp_path / "a.solution"), str(tmp_path / "b.solution"), str(tmp_path / "b.yaml")
    synth.write_solution_file(a, rig)
    run([os.path.join(host_bins, "solution_tool"), "roundtrip", a, b, y])
    m = yaml_mats(y)                           # the matrices the facade holds after reading the file, exactly (%.17g)
    rig.T_cam_init, rig.T_marker_init, rig.T_frame_init = m["transforms_to_root_cam"], m["transforms_to_root_marker"], m["root_marker_to_root_cam"]
    qs = (0.0, 0.25, 0.5, 0.95, 1.0)
    p = binding.Problem(rig)
    rep = p.error_report(p.mats2evec(), qs)
    out = run([os.path.join(host_bins, "solution_report"), a, "-frames", "-q", ",".join(repr(q) for q in qs)])
    lines = out.strip().splitlines()
    assert lines[0] == "report before"
    tot = lines[1].split()
    # sums are accumulated with atomics (their order is not fixed): equal to 1e-12; counts, maxima and percentiles are exact
    close = lambda a, b: np.all(np.abs(np.asarray(a, float) - np.asarray(b, float)) <= 1e-12 * np.abs(np.asarray(b, float)))
    assert tot[0] == "total" and int(tot[2]) == rep["observations"] and int(tot[4]) == rep["not_in_problem"] and close(float(tot[6]), rep["sum_sq"])
    pct = [l.split() for l in lines if l.startswith("percentile ")]
    assert [float(l[1]) for l in pct] == list(qs) and [float(l[3]) for l in pct] == list(rep["q_value"])
    for ent, key, ids in (("camera", "cam", rig.cam_ids), ("marker", "marker", rig.marker_ids), ("frame", "frame", rig.frame_ids)):
        rows = [l.split() for l in lines if l.startswith(ent + " ")]
        assert [int(r[1]) for r in rows] == list(ids)
        assert [int(r[3]) for r in rows] == list(rep[key + "_count"])
        assert close([float(r[5]) for r in rows], rep[key + "_sum_sq"])
        assert close([float(r[7]) for r in rows], np.sqrt(rep[key + "_sum_sq"] / (4.0 * rep[key + "_count"])))
        assert [float(r[9]) for r in rows] == list(rep[key + "_max"])
