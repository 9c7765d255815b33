"""Cost of soft pose priors (aar_set_prior, csrc/aar_prior.cuh) at BASELINE config 4 (one GPU).

One handle alternates between no priors and priors on every non-root camera, every non-root marker and every frame (targets at the
start poses moved by N(0, 1e-3), sigma 1e-2 rad / 1e-2 translation units) between aar_lm_begin calls; each round runs `--iters` LM
iterations with the stop rules off from the same z0.  The first two are not timed (the host-driven first iteration, and the capture of
the graph, which every change between priors and none invalidates); the rest run in the graph-resident loop.
Reported: the median ms per LM iteration of each arm over the rounds after warm-up (host clock around aar_lm_iterate, which ends in a
device synchronisation) with the LM tries they took, and the device time of k_prior_add / k_prior_cost per launch from torch.profiler
(CUDA activities) in a separate host-driven solve with priors.
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
    raise SystemExit("time_prior.py: no CUDA device")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()[0]
t0 = time.time(); rig = synth.make_config(a.workload, frames=a.frames); t_gen = time.time() - t0
p = binding.Problem(rig)
z0 = p.mats2evec()
Tc, Tm, Tf = p.evec2mats(z0 + np.random.default_rng(7).normal(0, 1e-3, z0.shape))
priors = dict(cams=(Tc, np.full((rig.C, 6), 1e4)), markers=(Tm, np.full((rig.M, 6), 1e4)), frames=(Tf, np.full((rig.F, 6), 1e4)))
prm = binding.Problem.default_params(max_iters=a.iters, ignore_stop_rules=1)


def run(with_priors):
    if with_priors:
        p.set_prior(**priors)
    else:
        p.set_prior()
    p.lm_begin(z0, prm)
    rep0, _ = p.lm_iterate(2)    # the first iteration runs host-driven (mu0); the second captures the graph again and runs in it
    t = time.time(); rep, _ = p.lm_iterate(a.iters - 2); dt = time.time() - t
    p.lm_end()
    assert rep.iterations == a.iters - 2
    tries[with_priors] = int(rep.total_tries - rep0.total_tries)     # LM tries of the timed iterations
    return 1e3 * dt / (a.iters - 2)


tries = {}
ms = {False: [], True: []}
for r in range(a.warmup + a.rounds):
    for with_priors in (False, True):
        m = run(with_priors)
        if r >= a.warmup:
            ms[with_priors].append(m)

# device time of the two kernels: one solve with priors of a few iterations under the profiler
from torch.profiler import ProfilerActivity, profile
p.set_prior(**priors)
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
                      priors=dict(cameras=rig.C - 1, markers=rig.M - 1, frames=rig.F),
                      ms_per_lm_iteration=dict(no_priors_median=float(np.median(ms[False])), priors_median=float(np.median(ms[True])),
                                               no_priors_all=[round(v, 3) for v in ms[False]], priors_all=[round(v, 3) for v in ms[True]]),
                      tries_per_round_of_timed_iterations=dict(no_priors=tries[False], priors=tries[True]),
                      k_prior_add=kernel_us("k_prior_add"), k_prior_cost=kernel_us("k_prior_cost"))))
