"""Cost of soft relative-pose priors (aar_set_pair_prior, csrc/aar_pair_prior.cuh) at BASELINE config 4 (one GPU).

One handle alternates between no pair priors and priors on every camera pair (a < b) plus the marker pairs (j, j + 1) (targets: the
relative poses at the start moved by N(0, 1e-3), sigma 1e-2 rad / 1e-2 translation units) between aar_lm_begin calls; each round runs
`--iters` LM iterations with the stop rules off from the same z0.  The first two are not timed (the host-driven first iteration, and
the capture of the graph, which every change between pairs and none invalidates); the rest run in the graph-resident loop.
Reported: the median ms per LM iteration of each arm over the rounds after warm-up (host clock around aar_lm_iterate, which ends in a
device synchronisation) with the LM tries they took, and the device time of k_pair_prior_add / k_pair_prior_cost per launch from
torch.profiler (CUDA activities) in a separate host-driven solve with the pairs.
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
    raise SystemExit("time_pair_prior.py: no CUDA device")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()[0]
t0 = time.time(); rig = synth.make_config(a.workload, frames=a.frames); t_gen = time.time() - t0
p = binding.Problem(rig)
z0 = p.mats2evec()
Tc, Tm, _ = p.evec2mats(z0 + np.random.default_rng(7).normal(0, 1e-3, z0.shape))


def pairs(T, P):
    return np.array(P, np.int32), np.stack([np.linalg.inv(T[i]) @ T[j] for i, j in P]), np.full((len(P), 2), 1e4)


cam_pairs = [(i, j) for i in range(rig.C) for j in range(i + 1, rig.C)]
marker_pairs = [(j, j + 1) for j in range(rig.M - 1)]
priors = dict(cams=pairs(Tc, cam_pairs), markers=pairs(Tm, marker_pairs))
prm = binding.Problem.default_params(max_iters=a.iters, ignore_stop_rules=1)


def run(with_pairs):
    if with_pairs:
        p.set_pair_prior(**priors)
    else:
        p.set_pair_prior()
    p.lm_begin(z0, prm)
    rep0, _ = p.lm_iterate(2)    # the first iteration runs host-driven (mu0); the second captures the graph again and runs in it
    t = time.time(); rep, _ = p.lm_iterate(a.iters - 2); dt = time.time() - t
    p.lm_end()
    assert rep.iterations == a.iters - 2
    tries[with_pairs] = int(rep.total_tries - rep0.total_tries)     # LM tries of the timed iterations
    return 1e3 * dt / (a.iters - 2)


tries = {}
ms = {False: [], True: []}
for r in range(a.warmup + a.rounds):
    for with_pairs in (False, True):
        m = run(with_pairs)
        if r >= a.warmup:
            ms[with_pairs].append(m)

# device time of the two kernels: one solve with the pairs of a few iterations under the profiler
from torch.profiler import ProfilerActivity, profile
p.set_pair_prior(**priors)
os.environ["AAR_NO_GRAPH"] = "1"                 # host-driven loop: every launch is a kernel record of the profiler
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    p.solve(z0, binding.Problem.default_params(max_iters=a.iters, ignore_stop_rules=1))
    torch.cuda.synchronize()
del os.environ["AAR_NO_GRAPH"]


def kernel_us(name):
    ev = [e for e in prof.events() if name in e.name and e.device_type == torch.autograd.DeviceType.CUDA]
    us = [getattr(e, "device_time", None) or e.cuda_time for e in ev]
    return dict(launches_profiled=len(us), us_per_launch_median=float(np.median(us)) if us else None)


print(json.dumps(dict(workload=a.workload, gpu=gpu, frames=rig.F, observations=p.num_obs, iterations_per_round=a.iters, rounds=a.rounds,
                      timed_iterations_per_arm=a.rounds * (a.iters - 2), rig_generation_s=round(t_gen, 1),
                      pairs=dict(camera_pairs=len(cam_pairs), marker_pairs=len(marker_pairs)),
                      ms_per_lm_iteration=dict(no_pairs_median=float(np.median(ms[False])), pairs_median=float(np.median(ms[True])),
                                               no_pairs_all=[round(v, 3) for v in ms[False]], pairs_all=[round(v, 3) for v in ms[True]]),
                      tries_per_round_of_timed_iterations=dict(no_pairs=tries[False], pairs=tries[True]),
                      k_pair_prior_add=kernel_us("k_pair_prior_add"), k_pair_prior_cost=kernel_us("k_pair_prior_cost"))))
