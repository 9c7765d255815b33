"""Cost of the lens model of the analytic mode (aar_problem_desc::lens_model = 1, csrc/aar_lens.cuh) on one GPU.

For each workload (default cfg3 and cfg4, distorted detections) three handles run `--iters` LM iterations with the stop rules off from
the same z0: the pinhole analytic mode with pose blocks only, the lens model with pose blocks only, and the lens model with the
intrinsics of every camera refined.  All three run the host-driven loop (the analytic mode has no graph-resident loop).  Reported: ms
per LM iteration after the first (host clock around aar_lm_iterate, which ends in a device synchronisation), and the device time per
launch of k_jac_analytic, k_jac_lens and k_intr_assemble_lens from torch.profiler (CUDA activities) in separate short solves.
Prints one JSON line per workload; the GPU name and power limit are read in the same run."""
import argparse, json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "automatic-ar_b200", "python"))
import numpy as np
import torch
from aar_b200 import binding, synth

ap = argparse.ArgumentParser(); ap.add_argument("--workloads", default="cfg3,cfg4"); ap.add_argument("--frames", type=int, default=None)
ap.add_argument("--iters", type=int, default=6)
a = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("time_lens.py: no CUDA device")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()[0]
from torch.profiler import ProfilerActivity, profile


def kernel_us(prof, name):
    ev = [e for e in prof.events() if e.name.split("(")[0].endswith(name) and e.device_type == torch.autograd.DeviceType.CUDA]
    us = [getattr(e, "device_time", None) or e.cuda_time for e in ev]
    return dict(launches_profiled=len(us), us_per_launch_median=float(np.median(us)) if us else None)


for wl in a.workloads.split(","):
    t0 = time.time(); rig = synth.make_config(wl, frames=a.frames, distorted=True); t_gen = time.time() - t0
    modes = dict(analytic_poses=dict(analytic=True), lens_poses=dict(lens=True), lens_intrinsics=dict(lens=True, intrinsics=True))
    prm = binding.Problem.default_params(max_iters=a.iters, ignore_stop_rules=1)
    out = dict(workload=wl, gpu=gpu, frames=rig.F, rig_generation_s=round(t_gen, 1), iterations=a.iters)
    for name, kw in modes.items():
        p = binding.Problem(rig, **kw)
        z0 = p.mats2evec()
        p.lm_begin(z0, prm)
        p.lm_iterate(1)
        t = time.time(); rep, _ = p.lm_iterate(a.iters - 1); dt = time.time() - t
        p.lm_end()
        out[name] = dict(ms_per_lm_iteration=round(1e3 * dt / (a.iters - 1), 3), tries=int(rep.total_tries), observations=p.num_obs)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            p.solve(z0, binding.Problem.default_params(max_iters=2, ignore_stop_rules=1))
            torch.cuda.synchronize()
        for k in ("k_jac_analytic", "k_jac_lens", "k_intr_assemble_lens"):
            r = kernel_us(prof, k)
            if r["launches_profiled"]:
                out[name][k] = r
        p.close()
    print(json.dumps(out), flush=True)
