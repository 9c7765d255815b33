"""Cost of holding entities fixed (aar_set_fixed, csrc/aar_fixed.cuh) at BASELINE config 4 (one GPU).

One handle alternates between no mask and a mask (8 of the 16 cameras, every 10th frame) between aar_lm_begin calls; each round runs
`--iters` LM iterations with the stop rules off from the same z0.  The first two are not timed (the host-driven first iteration, and
the capture of the graph, which every change between mask and no mask invalidates); the rest run in the graph-resident loop.
Reported: the median ms per LM iteration of each arm over the rounds after warm-up (host clock around aar_lm_iterate, which ends in a
device synchronisation) with the LM tries they took, and the device time of k_hold_fixed per launch from torch.profiler (CUDA activities)
in a separate host-driven masked solve.
Prints one JSON line; the GPU name and power limit are read in the same run."""
import argparse, json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "automatic-ar_b200", "python"))
import numpy as np
import torch
from aar_b200 import binding, synth

ap = argparse.ArgumentParser(); ap.add_argument("--workload", default="cfg4"); ap.add_argument("--frames", type=int, default=None)
ap.add_argument("--iters", type=int, default=6); ap.add_argument("--rounds", type=int, default=6); ap.add_argument("--warmup", type=int, default=1)
a = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("time_fixed.py: no CUDA device")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()[0]
t0 = time.time(); rig = synth.make_config(a.workload, frames=a.frames); t_gen = time.time() - t0
p = binding.Problem(rig)
z0 = p.mats2evec()
cams = np.zeros(rig.C, bool); cams[np.arange(1, rig.C, 2)] = True          # 8 of 16; the root (index 0) is free
frames = np.zeros(rig.F, bool); frames[::10] = True
prm = binding.Problem.default_params(max_iters=a.iters, ignore_stop_rules=1)


def run(masked):
    if masked:
        p.set_fixed(cams=cams, frames=frames)
    else:
        p.set_fixed()
    p.lm_begin(z0, prm)
    rep0, _ = p.lm_iterate(2)    # the first iteration runs host-driven (mu0); the second captures the graph again (the mask changed) and runs in it
    t = time.time(); rep, _ = p.lm_iterate(a.iters - 2); dt = time.time() - t
    z = p.lm_end()
    assert rep.iterations == a.iters - 2
    tries[masked] = int(rep.total_tries - rep0.total_tries)     # LM tries of the timed iterations (each try is a Schur + solve + residual)
    return 1e3 * dt / (a.iters - 2), z


tries = {}


ms = {False: [], True: []}
for r in range(a.warmup + a.rounds):
    for masked in (False, True):
        m, z = run(masked)
        if r >= a.warmup:
            ms[masked].append(m)
        if masked:
            col = np.zeros(p.num_vars, bool)
            im = p.index_maps()
            for i in np.flatnonzero(cams): col[im["col_cam"][i]:im["col_cam"][i] + 6] = True
            for k in np.flatnonzero(frames): col[im["col_frame"][k]:im["col_frame"][k] + 6] = True
            assert np.array_equal(z[col], z0[col])

# device time of k_hold_fixed: one masked solve of a few iterations under the profiler
from torch.profiler import ProfilerActivity, profile
p.set_fixed(cams=cams, frames=frames)
os.environ["AAR_NO_GRAPH"] = "1"                 # host-driven loop: every launch is a kernel record of the profiler
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    p.solve(z0, binding.Problem.default_params(max_iters=a.iters, ignore_stop_rules=1))
    torch.cuda.synchronize()
del os.environ["AAR_NO_GRAPH"]
hold = [e for e in prof.events() if "k_hold_fixed" in e.name and e.device_type == torch.autograd.DeviceType.CUDA]
hold_us = [getattr(e, "device_time", None) or e.cuda_time for e in hold]
st = p.stats()
print(json.dumps(dict(workload=a.workload, gpu=gpu, frames=rig.F, observations=p.num_obs, w_slots=st["slots"], iterations_per_round=a.iters,
                      rounds=a.rounds, timed_iterations_per_arm=a.rounds * (a.iters - 2), rig_generation_s=round(t_gen, 1),
                      held=dict(cameras=int(cams.sum()), frames=int(frames.sum())),
                      ms_per_lm_iteration=dict(no_mask_median=float(np.median(ms[False])), mask_median=float(np.median(ms[True])),
                                               no_mask_all=[round(v, 3) for v in ms[False]], mask_all=[round(v, 3) for v in ms[True]]),
                      tries_per_round_of_timed_iterations=dict(no_mask=tries[False], mask=tries[True]),
                      k_hold_fixed=dict(launches_profiled=len(hold), us_per_launch_median=float(np.median(hold_us)) if hold_us else None))))
