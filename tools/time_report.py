"""Cost of the reprojection-error report and of reject-and-resolve at BASELINE config 4 (one GPU).

1. solves the rig with every 37th detection moved by 25 px (plain LM, the outliers kept);
2. aar_error_report at the solution, CUDA events on the handle's stream after warm-up: entity statistics + 3 percentiles, and the same
   with the per-detection output (adds the copy of the errors to the host and their scatter to detection order);
3. what -reject-outliers costs after that: aar_problem_create of the kept detections and the re-solve from the first solve's poses.
Prints one JSON line; the GPU name and power limit are read in the same run."""
import argparse, copy, json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "automatic-ar_b200", "python"))
import numpy as np
import torch
from aar_b200 import binding, synth

ap = argparse.ArgumentParser(); ap.add_argument("--workload", default="cfg4"); ap.add_argument("--frames", type=int, default=None)
ap.add_argument("--reps", type=int, default=20); ap.add_argument("--threshold", type=float, default=5.0)
a = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("time_report.py: no CUDA device")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()[0]
t0 = time.time(); rig = copy.copy(synth.make_config(a.workload, frames=a.frames)); t_gen = time.time() - t0
rig.det_xy = rig.det_xy.copy(); bad = np.arange(0, rig.N, 37); rig.det_xy[bad] += 25.0
stream = torch.cuda.Stream()
p = binding.Problem(rig, stream=stream.cuda_stream)
t0 = time.time(); z, cost, iters, _ = p.solve(p.mats2evec()); t_solve1 = time.time() - t0

Q = (0.5, 0.9, 0.99)
ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def timed(fn):
    for _ in range(2):
        fn()                                      # warm-up: allocations of the handle's report buffers, module load
    ms = []
    for _ in range(a.reps):
        ev0.record(stream); t = time.time(); r = fn(); w = time.time() - t; ev1.record(stream); ev1.synchronize()
        ms.append((ev0.elapsed_time(ev1), 1e3 * w))
    return r, float(np.median([m[0] for m in ms])), float(np.median([m[1] for m in ms]))


out = binding.ErrorReportOut(); qa = np.array(Q); qv = np.zeros(len(Q))
out.num_q = len(Q); out.q = binding._vp(qa); out.q_value = binding._vp(qv)
zc = np.ascontiguousarray(z)
_, ms_stats, wall_stats = timed(lambda: binding._chk(binding.lib().aar_error_report(p.h, binding._vp(zc), binding.C.byref(out)), "aar_error_report"))
rep, ms_full, wall_full = timed(lambda: p.error_report(z, Q))
flag = rep["det_err"] > a.threshold
# reject-and-resolve: a new handle of the kept detections, started from the first solve's poses
Tc, Tm, Tf = p.evec2mats(z)
kept = copy.copy(rig)
for k in ("det_frame", "det_cam", "det_marker", "det_xy"):
    setattr(kept, k, np.ascontiguousarray(getattr(rig, k)[~flag]))
kept.T_cam_init, kept.T_marker_init, kept.T_frame_init = Tc, Tm, Tf
del p; torch.cuda.synchronize()
t0 = time.time(); p2 = binding.Problem(kept, stream=stream.cuda_stream); torch.cuda.synchronize(); t_create = time.time() - t0
t0 = time.time(); z2, cost2, iters2, _ = p2.solve(p2.mats2evec()); t_solve2 = time.time() - t0
print(json.dumps(dict(workload=a.workload, gpu=gpu, observations=int(rep["observations"]), injected=int(len(bad)), flagged=int(flag.sum()),
                      flagged_are_injected=bool(np.array_equal(np.nonzero(flag)[0], bad)), rig_generation_s=round(t_gen, 1),
                      first_solve=dict(seconds=round(t_solve1, 3), iterations=int(iters), cost=cost),
                      report_stats_and_3_percentiles=dict(device_ms=ms_stats, wall_ms=wall_stats),
                      report_with_per_detection_output=dict(device_ms=ms_full, wall_ms=wall_full),
                      q=list(Q), q_value=[float(v) for v in rep["q_value"]],
                      reject=dict(create_s=round(t_create, 3), resolve_s=round(t_solve2, 3), iterations=int(iters2), cost=cost2))))
