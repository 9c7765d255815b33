"""Generates tests/golden/track_golden.npz — MultiCamMapper::track() (libs/multicam_mapper.cpp:430-443: the 2-argument
SparseLevMarq::solve, calcDerivates Jacobian) frame by frame on the three rigs of the track parity tests in tests/test_gpu_parity.py:
per frame the start pose z_init, the solved pose z, the final cost and the iteration count.

The CPU oracle runs the solve: with oracle/_ref built (`make -C oracle ref REFERENCE=<checkout of the original project>`) the
unmodified reference sparselevmarq.h, otherwise the oracle's restatement of its LM loop (oracle/mcm_oracle.cpp, aar_oracle_lm_port).
The file records which one in `baseline`.  Run:  python tests/golden/make_golden_track.py"""
import copy
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (os.path.join(ROOT, "automatic-ar_b200", "python"), os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)
from aar_b200 import synth  # noqa: E402

CASES = ("small_rig", "small_rig_huber", "cfg5_240")


def track_rig(case):
    """The rig of a track parity test: the solved rig (cameras, markers) is fixed while tracking."""
    if case == "cfg5_240":
        rig = copy.copy(synth.make_config("cfg5", frames=240))
    else:
        rig = copy.copy(synth.make_rig(C=3, M=6, F=25, obs_per_frame=6.0, seed=13, distorted=True))
    rig.T_cam_init, rig.T_marker_init = rig.T_cam_true, rig.T_marker_true
    if case == "small_rig_huber":
        rig.det_xy = rig.det_xy.copy(); rig.det_xy[::23] += 12.0                   # outliers
    return rig


def oracle_track(oracle_py, rig, with_huber):
    """Per frame of the rig: (z_init [F, 6], z [F, 6], cost [F], iterations [F]) of the oracle's track(), and whether it ran the reference."""
    o = oracle_py.Oracle(rig); o.set_config(cams=False, markers=False, objects=True, with_huber=with_huber)
    out = [], [], [], []
    for k in range(rig.F):
        fid = rig.frame_ids[k]
        sel = rig.det_frame == fid
        _, z_init = o.track_init(fid, rig.T_frame_init[k], rig.det_cam[sel], rig.det_marker[sel], rig.det_xy[sel])
        z, cost, it, _ = o.track(z_init)
        for lst, v in zip(out, (z_init, z, cost, it)):
            lst.append(v)
    return tuple(np.array(v) for v in out), o.is_ref


def main():
    import oracle_py
    if not os.path.exists(oracle_py.lib_path(False)):
        oracle_py.build()
    g = {}
    kinds = set()
    for case in CASES:
        (z_init, z, cost, it), is_ref = oracle_track(oracle_py, track_rig(case), case.endswith("huber"))
        kinds.add(is_ref)
        g.update({f"{case}_z_init": z_init, f"{case}_z": z, f"{case}_cost": cost, f"{case}_iterations": it.astype(np.int32)})
    assert len(kinds) == 1
    g["baseline"] = np.array("reference sparselevmarq.h" if kinds.pop() else "restated LM loop (aar_oracle_lm_port)")
    np.savez_compressed(os.path.join(HERE, "track_golden.npz"), **g)
    print("wrote track_golden.npz:", str(g["baseline"]), {c: len(g[c + "_cost"]) for c in CASES})


if __name__ == "__main__":
    main()
