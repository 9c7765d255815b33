#!/usr/bin/env python
"""bench.py — LM iterations/s and corner-observations/s of the MultiCamMapper joint optimisation.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg4] [--frames F] [--dump-outputs DIR]

One *step* is one Levenberg-Marquardt iteration of MultiCamMapper::solve() (quantised finite-difference
Jacobian + normal equations + per-frame Schur elimination + reduced solve + trial residual + accept/reject,
libs/sparselevmarq.h:348-430 of the reference) over every marker observation of the workload.  The default
workload is BASELINE.json configs[3] (16 cameras, 64 markers, 100 000 frames, ~25.6 M marker observations
= ~102 M corner observations), the configuration the north star's target is quoted on; it fits one B200.
With N > 1 (launched by torch.distributed.run, one rank per GPU) the same problem is frame-sharded and the
reduced system + cost are NCCL-all-reduced every try  ->  "scaling": "strong".

value   device-resident throughput: observations, poses and z are in HBM before the timed region.
e2e     the same iterations through the C-ABI call a reference user would make (aar_lm_solve with HOST
        io_vec, pinned): host->device copy of z, K iterations, device->host copy of z and of the LM state.
--impl reference   times the reference's own CPU path (oracle/_ref: restated MultiCamMapper residual/Jacobian
        driving the UNMODIFIED libs/sparselevmarq.h) on the host cores, on a bounded frame sample of the
        same workload.  It runs exactly --steps steps; with --workload cfg5 a step is a full pass of per-frame
        track() solves over the sample, so the default --steps 20 takes 20 times as long as one pass.
--dump-outputs DIR writes what the timed path computed in its last step as DIR/<name>.npy (float64, at most
        64 MB in all): z and final_cost of the LM solve; z, cost and iterations per frame of track (cfg5).

The LM trajectory is restarted from z0 every RESTART iterations (device-side copy, inside the timed
region) so that every timed step is a productive LM iteration and not a converged one.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p_ in (os.path.join(ROOT, "automatic-ar_b200", "python"),):
    if p_ not in sys.path:
        sys.path.insert(0, p_)

RESTART = 10            # LM iterations between restarts from z0
W_J_FLOP = 9.0e3        # algorithmic FP64 flop per marker observation per Jacobian evaluation (SURVEY 8d, DESIGN.md)
W_PROJ_FLOP = 5912.0    # ... of which in k_jac_project: 37 projections x 152 + 288 for the central differences
W_ASM_FLOP = 3040.0     # ... and in the assembly kernels: 2 736 (upper J^T J blocks) + 304 (J^T r, cost)
W_AN_FLOP = 1700.0      # the analytic variant's k_jac_analytic (--analytic): 3 chained rigid transforms, one division, 18 directional derivatives per corner
OBS_BYTES = 76          # HBM bytes per marker observation read by k_jac_project (2 x 8 float corners + 12 B indices; the pair table adds 1536 B per (frame, camera) pair)
STAGE_BYTES = 640       # HBM bytes per marker observation written by k_jac_project (144 float numerators + 8 double residuals)
CPU_SAMPLE_FRAMES = 300
CPU_SAMPLE_ITERS = 3


def load_peaks():
    peaks = {"hbm_gbs": 6650.0, "hbm_src": "fallback", "fp64_tflops": 36.7, "fp64_src": "r1 DFMA microbenchmark (profiles/r1_fp64_peak.json)"}
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peaks["hbm_gbs"] = float(mp["hbm_gbs"]); peaks["hbm_src"] = "measured (MEASURED_PEAKS.json)"
    except Exception:
        pass
    try:
        fp = json.load(open(os.path.join(ROOT, "profiles", "r1_fp64_peak.json")))
        peaks["fp64_tflops"] = float(fp["dfma_tflops"])
    except Exception:
        pass
    return peaks


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu = gpu_index; self.rows = []; self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True); self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        window = [r for r in self.rows if t0 - 0.15 <= r[0] <= t1 + 0.15] or self.rows[-2:]     # very short timed regions: nearest samples (under load: warm-up precedes)
        for ts, line in window:
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); pw.append(float(f[3]))
            except Exception:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


DUMP_BYTES = 64_000_000         # --dump-outputs: at most this many bytes of array data in all


def dump_outputs(out_dir, **arrays):
    """--dump-outputs: every array as out_dir/<name>.npy in float64, so that two builds can be compared output for output.  When they
    exceed DUMP_BYTES together, the arrays of the longest leading dimension (one row per frame, say) keep the same fixed, seeded
    sample of rows, whose indices go to out_dir/rows.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    if sum(a.nbytes for a in arrays.values()) > DUMP_BYTES:
        n = max(len(a) for a in arrays.values())
        big = [k for k, a in arrays.items() if len(a) == n]
        rest = sum(a.nbytes for k, a in arrays.items() if k not in big)
        keep = np.sort(np.random.default_rng(0).choice(n, (DUMP_BYTES - rest) * n // (sum(arrays[k].nbytes for k in big) + 8 * n), replace=False))
        arrays.update({k: arrays[k][keep] for k in big}, rows=keep)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def cpu_reference_run(workload, frames, iters, warmup=0):
    """The reference's CPU implementation of the path on the host cores (test infrastructure: oracle/)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py
    from aar_b200 import synth
    rig = synth.make_config(workload, frames=frames)
    o = oracle_py.Oracle(rig)
    try:        # torch.distributed.run exports OMP_NUM_THREADS=1: the CPU arm uses every host core it may run on
        o.L.aar_oracle_set_omp_threads(len(os.sched_getaffinity(0)))
    except Exception:
        pass
    z0 = o.mats2evec()
    kind = "reference" if o.is_ref else "port"
    cores = int(o.L.aar_oracle_omp_threads())
    if o.is_ref:
        if warmup:
            o.time_ref_steps(z0, warmup)
        secs = o.time_ref_steps(z0, iters)
    else:
        if warmup:
            o.set_max_iters(warmup); o.solve_port(z0)
        t = time.time(); done = 0
        while done < iters:             # restarted from z0 when the stop rules end a solve early, so that exactly `iters` steps run
            o.set_max_iters(iters - done); _, _, it, _ = o.solve_port(z0); done += int(it)
        secs = time.time() - t
        o.set_max_iters(10000)
    n_obs = o.num_rows // 8
    return dict(seconds=secs, iters=iters, n_obs=n_obs, kind=kind, cores=cores, rig=rig, oracle=o, z0=z0,
                sample=f"{workload} restricted to its first {rig.F} frames ({n_obs} marker observations), {iters} SparseLevMarq::step calls from the initial estimate"
                       + ("" if o.is_ref else " [restated LM loop]"))


def parity_check(r, device):
    """The CUDA path against the CPU reference arm on the SAME rig the cpu_baseline leg just timed (the benchmarked workload
    restricted to its first frames): residual ==, reduced Schur system <= 1e-10, cost after 1..3 SparseLevMarq::step <= 1e-10."""
    import numpy as np
    from aar_b200 import binding
    o, rig, z0 = r["oracle"], r["rig"], r["z0"]
    p = binding.Problem(rig, device=device)
    out = {"sample": r["sample"].split(",")[0]}
    r_o = o.error(z0); r_g, _ = p.residual(z0)
    out["residual_bit_exact"] = bool(np.array_equal(r_g, r_o)); out["residual_rows"] = int(len(r_o))
    mu = 1.0e3
    S_o, b_o, c_o = o.reduced_system(z0, mu); S_g, b_g, c_g = p.reduced_system(z0, mu)
    iu = np.triu_indices(p.n_r)
    out["reduced_system_rel_dev"] = float(np.abs(S_g[iu] - S_o[iu]).max() / np.abs(S_o).max())
    out["reduced_rhs_rel_dev"] = float(np.abs(b_g - b_o).max() / np.abs(b_o).max())
    devs = []
    for k in (1, 2, 3):
        o.set_max_iters(k)
        z_o, fc_o, it_o, _ = o.solve(z0)
        z_g, fc_g, it_g, _ = p.solve(z0, binding.Problem.default_params(max_iters=k))
        devs.append({"steps": k, "cost_ref": float(fc_o), "cost_gpu": float(fc_g), "rel_dev_cost": float(abs(fc_g - fc_o) / fc_o),
                     "rel_dev_z": float(np.abs(z_g - z_o).max() / np.abs(z_o).max())})
    o.set_max_iters(10000)
    out["lm_steps"] = devs
    out["ok"] = bool(out["residual_bit_exact"] and out["reduced_system_rel_dev"] <= 1e-10 and out["reduced_rhs_rel_dev"] <= 1e-10
                     and all(d["rel_dev_cost"] <= 1e-10 and d["rel_dev_z"] <= 1e-10 for d in devs))
    p.close()
    return out


def run_reference(args, rank):
    if rank != 0:
        return
    r = cpu_reference_run(args.workload, args.frames or CPU_SAMPLE_FRAMES, max(args.steps, 1), warmup=min(args.warmup, 1))
    v = 4.0 * r["n_obs"] * r["iters"] / r["seconds"]
    line = {"impl": "reference", "metric": "corner_obs_per_s", "value": v, "unit": "corner-observations/s", "n_gpus": args.gpus,
            "steps": r["iters"], "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * r["seconds"] / r["iters"],
            "lm_iters_per_s": r["iters"] / r["seconds"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": args.workload, "sampled_frames": args.frames or CPU_SAMPLE_FRAMES, "marker_observations": r["n_obs"]},
            "cpu_baseline": {"value": v, "unit": "corner-observations/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
            "e2e": {"value": v, "unit": "corner-observations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


W_TRACK_FLOP = 13 * 152.0 + 48.0 + 432.0     # per marker observation and LM iteration of track(): 13 projections (base + 2 x 6 dofs), central differences, 6x6 J^T J + J^T r
TRACK_CPU_FRAMES = 240


def track_rig(frames):
    import copy
    from aar_b200 import synth
    rig = copy.copy(synth.make_config("cfg5", frames=frames))
    rig.T_cam_init, rig.T_marker_init = rig.T_cam_true, rig.T_marker_true        # the solved rig is fixed while tracking
    return rig


def track_cpu_run(frames, check_device=None, passes=1):
    """MultiCamMapper::track() on the host cores: the oracle running the reference's 2-argument SparseLevMarq::solve frame by frame
    (calcDerivates is OpenMP-parallel inside a frame, sparselevmarq.h:164-220) over the first `frames` frames of config 5, `passes` times."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py
    rig = track_rig(frames)
    o = oracle_py.Oracle(rig); o.set_config(cams=False, markers=False, objects=True)
    try:
        o.L.aar_oracle_set_omp_threads(len(os.sched_getaffinity(0)))
    except Exception:
        pass
    order = np.argsort(rig.det_frame, kind="stable"); starts = np.searchsorted(rig.det_frame[order], rig.frame_ids); ends = np.searchsorted(rig.det_frame[order], rig.frame_ids, side="right")
    t = time.time()
    for _ in range(passes):
        zs, costs, its, n_obs = [], [], [], 0
        for k in range(rig.F):
            sel = order[starts[k]:ends[k]]
            rows, zi = o.track_init(int(rig.frame_ids[k]), rig.T_frame_init[k], rig.det_cam[sel], rig.det_marker[sel], rig.det_xy[sel])
            z, fc, it, _ = o.track(zi)
            zs.append(z); costs.append(fc); its.append(it); n_obs += len(sel)
    secs = time.time() - t
    work = passes * float(sum(4.0 * (ends[k] - starts[k]) * its[k] for k in range(rig.F)))
    out = dict(seconds=secs, frames=rig.F, n_obs=n_obs, work=work, kind="reference" if o.is_ref else "port", cores=int(o.L.aar_oracle_omp_threads()),
               sample=f"cfg5 restricted to its first {rig.F} frames ({n_obs} marker observations), full per-frame solves (mean {np.mean(its):.1f} LM iterations)")
    if check_device is not None:
        from aar_b200 import binding
        p = binding.Problem(rig, cams=False, markers=False, objects=True, device=check_device)
        zg, cg, ig = p.track_batch(p.mats2evec().reshape(-1, 6))
        zo = np.array(zs); co = np.array(costs)
        out["parity_check"] = {"frames": rig.F, "worst_rel_dev_cost": float((np.abs(cg - co) / np.maximum(co, 1e-12)).max()),
                               "worst_rel_dev_z": float((np.abs(zg - zo).max(axis=1) / np.maximum(1.0, np.abs(zo).max(axis=1))).max()),
                               "iteration_counts_equal": bool(np.array_equal(ig, np.array(its))), "bar": 1e-6}
        out["parity_check"]["ok"] = bool(out["parity_check"]["worst_rel_dev_cost"] <= 1e-6 and out["parity_check"]["worst_rel_dev_z"] <= 1e-6)
        p.close()
    return out


def run_track_reference(args, rank):
    if rank != 0:
        return
    K = max(args.steps, 1)
    r = track_cpu_run(args.frames or TRACK_CPU_FRAMES, passes=K)
    v = r["work"] / r["seconds"]
    print(json.dumps({"impl": "reference", "metric": "corner_obs_per_s", "value": v, "unit": "corner-observations/s", "n_gpus": args.gpus, "steps": K, "warmup": 0,
                      "ms_per_step": 1e3 * r["seconds"] / K, "frames_per_s": K * r["frames"] / r["seconds"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                      "config": {"workload": "cfg5", "sampled_frames": r["frames"], "marker_observations": r["n_obs"]},
                      "cpu_baseline": {"value": v, "unit": "corner-observations/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
                      "e2e": {"value": v, "unit": "corner-observations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}), flush=True)


def run_track(args, rank, world, local_rank):
    """BASELINE config 5: MultiCamMapper::track() as ONE batched call — 100 000 independent per-frame 6-dof LM solves against the
    fixed rig, frames sharded over the ranks (no collective).  A step = one pass of full per-frame solves over all frames."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from aar_b200 import binding
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG") and not os.environ.get("NCCL_DEBUG_FILE"):
            os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    binding.lib()
    t0 = time.time(); rig = track_rig(args.frames); t_gen = time.time() - t0
    stream = torch.cuda.Stream()
    t0 = time.time()
    p = binding.Problem(rig, cams=False, markers=False, objects=True, device=local_rank, stream=stream.cuda_stream, rank=rank, world_size=world)
    torch.cuda.synchronize(); t_create = time.time() - t0
    st = p.stats(); fb, fe = st["frame_begin"], st["frame_end"]
    z0 = p.mats2evec().reshape(-1, 6)[fb:fe].copy()
    nobs_f = np.bincount(np.searchsorted(rig.frame_ids, rig.det_frame), minlength=rig.F)[fb:fe]
    K, W = args.steps, args.warmup

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        clocks = ClockSampler(local_rank); clocks.start()
        p.track_upload(z0)
        for _ in range(W):
            p.track_run()
        p.set_profiling(True); launches0 = p.kernel_launches
        barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        tw0 = time.time(); e0.record(stream)
        for _ in range(K):
            p.track_run()
        e1.record(stream); barrier(); tw1 = time.time()
        ms = e0.elapsed_time(e1); launches = p.kernel_launches - launches0
        k_ms, k_runs = p.track_ms(); p.set_profiling(False)
        clk = clocks.stop(tw0, tw1)
        z, cost, its = p.track_download(fe - fb)
        # end to end: host poses in, host poses / costs / iteration counts out, every step
        p.track_batch(z0); barrier()
        tw2 = time.time()
        for _ in range(K):
            ze, ce, ie = p.track_batch(z0)
        barrier(); ms_e2e = 1e3 * (time.time() - tw2)
    work = float((4.0 * nobs_f * its).sum())              # corner observations x LM iterations of one pass, this rank
    t = torch.tensor([ms, ms_e2e, -work, -float(nobs_f.sum()), -float(its.sum()), -float(cost.sum()), -float(fe - fb), k_ms / max(k_runs, 1)], dtype=torch.float64, device="cuda")
    if world > 1:
        tm = t.clone(); dist.all_reduce(tm, op=dist.ReduceOp.MAX); ts = t.clone(); dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        t = torch.cat([tm[:2], ts[2:7], tm[7:]])
    ms, ms_e2e, work_all, n_obs, its_sum, cost_sum, frames_all, kern_ms = float(t[0]), float(t[1]), -float(t[2]), -float(t[3]), -float(t[4]), -float(t[5]), -float(t[6]), float(t[7])
    if args.dump_outputs:               # the last timed pass: poses, costs and iteration counts of every frame, shards in frame order
        shards = [(z, cost, its)]
        if world > 1:
            shards = [None] * world; dist.all_gather_object(shards, (z, cost, its))
        if rank == 0:
            dump_outputs(args.dump_outputs, z=np.concatenate([s[0] for s in shards]), cost=np.concatenate([s[1] for s in shards]),
                         iterations=np.concatenate([s[2] for s in shards]))
    if rank == 0:
        peaks = load_peaks()
        value = work_all * K / (ms * 1e-3)
        flop = W_TRACK_FLOP * work / 4.0 + 152.0 * work / 4.0          # this rank's pass: Jacobian iterations + (at least) one trial residual per iteration
        ach = flop / (kern_ms * 1e-3) / 1e12 if kern_ms > 0 else 0.0
        bytes_alg = 40.0 * float(nobs_f.sum())
        line = {"metric": "corner_obs_per_s", "value": value, "unit": "corner-observations/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
                "frames_per_s": frames_all * K / (ms * 1e-3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "value_note": "corner observations x LM iterations executed per second (every per-frame LM iteration evaluates residual + central-difference Jacobian + 6x6 solve over the frame's observations)",
                "config": {"workload": "cfg5", "cameras": rig.C, "markers": rig.M, "frames": rig.F, "marker_observations": int(n_obs), "parallelism": f"frame-shard x{world}, no collective",
                           "lm_iterations_mean": its_sum / frames_all, "rms_px": float(np.sqrt(cost_sum / (8 * n_obs))),
                           "l2": "observations of a rank (%.0f MB) are re-read every LM iteration; %s the 126 MB L2" % (40e-6 * float(nobs_f.sum()), "exceed" if 40 * float(nobs_f.sum()) > 126e6 else "fit"),
                           "step": "one pass of MultiCamMapper::track() over all frames (full per-frame solves)"},
                "e2e": {"value": work_all * K / (ms_e2e * 1e-3), "unit": "corner-observations/s", "ms_per_step": ms_e2e / K, "frames_per_s": frames_all * K / (ms_e2e * 1e-3),
                        "h2d_bytes_per_step": int(48 * frames_all), "d2h_bytes_per_step": int(60 * frames_all), "call": "aar_track_batch(host z6 in/out, cost, iterations)",
                        "create_s": t_create},
                "gpu_launches": int(launches), "clocks": clk,
                "roofline": {"kernel": "k_track_cta", "bound": "fp64", "achieved": ach, "peak": peaks["fp64_tflops"], "unit": "TFLOP/s", "frac": ach / peaks["fp64_tflops"], "peak_source": peaks["fp64_src"],
                             "ms_per_launch": kern_ms, "algorithmic_flop_per_launch": flop, "flop_per_marker_obs_and_iteration": W_TRACK_FLOP + 152.0,
                             "note": "rank 0's shard; the reference arithmetic is non-FMA (two IEEE operations per a*b+c) and every quotient is an IEEE division",
                             "hbm": {"achieved": bytes_alg * (its_sum / frames_all) / (kern_ms * 1e-3) / 1e9 if kern_ms > 0 else 0.0, "peak": peaks["hbm_gbs"], "unit": "GB/s", "algorithmic_bytes_per_iteration": bytes_alg},
                             "traffic": None},
                "setup_s": {"generate": t_gen, "create_upload_undistort": t_create}}
        line["roofline"]["hbm"]["frac"] = line["roofline"]["hbm"]["achieved"] / peaks["hbm_gbs"]
        if world == 1 and not args.no_cpu_baseline and not args.analytic:
            r = track_cpu_run(TRACK_CPU_FRAMES, check_device=local_rank)
            line["cpu_baseline"] = {"value": r["work"] / r["seconds"], "unit": "corner-observations/s", "frames_per_s": r["frames"] / r["seconds"], "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}
            line["parity_check"] = r["parity_check"]
        print(json.dumps(line), flush=True)
    p.close()
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


def run_ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist
    from aar_b200 import binding, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG") and not os.environ.get("NCCL_DEBUG_FILE"):
            os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"      # NCCL logs to STDOUT by default; stdout carries the one JSON line only
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    binding.lib()
    t0 = time.time()
    rig = synth.make_config(args.workload, frames=args.frames)
    t_gen = time.time() - t0
    stream = torch.cuda.Stream()
    t0 = time.time()
    p = binding.Problem(rig, device=local_rank, stream=stream.cuda_stream, rank=rank, world_size=world, analytic=args.analytic)
    if world > 1:
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(binding.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        p.comm_init(bytes(idt.cpu().numpy().tobytes()))
    torch.cuda.synchronize()
    t_create = time.time() - t0
    n_obs, n_local, n_vars = p.num_obs, p.num_local_obs, p.num_vars
    z0 = p.mats2evec()
    zpin = torch.empty(n_vars, dtype=torch.float64).pin_memory()
    zpin_np = zpin.numpy()

    prm = binding.Problem.default_params(ignore_stop_rules=1)
    K, W = args.steps, args.warmup

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    seg_tries = [0]          # total_tries of the report is cumulative since the last lm_begin
    last_rep = [None]

    def iterate(n, done):
        """n LM iterations, restarting from the device-resident z0 every RESTART iterations; returns tries executed."""
        tries = 0
        while n > 0:
            if done % RESTART == 0 and done > 0:
                p.lm_begin(None, prm); seg_tries[0] = 0
            m = min(n, RESTART - done % RESTART)
            rep, _ = p.lm_iterate(m)
            last_rep[0] = rep
            tries += rep.total_tries - seg_tries[0]; seg_tries[0] = rep.total_tries
            n -= m; done += m
        return done, tries

    # ---------------------------------------------------------------- device-resident arm
    with torch.cuda.stream(stream):
        clocks = ClockSampler(local_rank); clocks.start()      # started before the warm-up so that samples exist even for a short timed region
        p.lm_begin(z0, prm)
        done, _ = iterate(W, 0)
        launches0 = p.kernel_launches
        barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        tw0 = time.time()
        e0.record(stream)
        done, tries_total = iterate(K, done)                   # single GPU: the graph-resident loop (no host in it); sharded: host-driven tries
        e1.record(stream)
        final_cost = last_rep[0].final_cost
        barrier()
        tw1 = time.time()
        ms = e0.elapsed_time(e1)
        launches = p.kernel_launches - launches0
        clk = clocks.stop(tw0, tw1)
        if args.dump_outputs:           # the iterate after the last timed step, read before the pass below restarts from z0
            z_last = p.lm_end()
        # the same K iterations once more with per-phase CUDA events on the launching stream (host-driven loop: events cannot sit
        # inside the graph): kernel durations for the roofline entries, not part of `value`
        p.lm_begin(None, prm); seg_tries[0] = 0
        iterate(W, 0)
        p.set_profiling(True)
        barrier()
        g0 = torch.cuda.Event(enable_timing=True); g1 = torch.cuda.Event(enable_timing=True)
        g0.record(stream)
        iterate(K, W)
        g1.record(stream)
        barrier()
        ms_profiled = g0.elapsed_time(g1)
        ph = p.phase_ms()
        p.set_profiling(False)
        p.lm_end()

        # ------------------------------------------------------------ end-to-end arm (host io_vec through aar_lm_solve)
        chunk = min(K, RESTART)
        prm_e = binding.Problem.default_params(ignore_stop_rules=1, max_iters=chunk)
        zpin_np[:] = z0
        p.solve_inplace(zpin_np, prm_e)                     # warm-up
        barrier()
        f0 = torch.cuda.Event(enable_timing=True); f1 = torch.cuda.Event(enable_timing=True)
        tw2 = time.time()
        f0.record(stream)
        left = K; e2e_tries = 0; calls = 0
        while left > 0:
            m = min(left, chunk)
            prm_e.max_iters = m
            zpin_np[:] = z0
            rep = p.solve_inplace(zpin_np, prm_e)
            e2e_tries += rep.total_tries; left -= m; calls += 1
        f1.record(stream)
        barrier()
        tw3 = time.time()
        ms_e2e = max(f0.elapsed_time(f1), 1e3 * (tw3 - tw2))     # host wall clock includes the copies' sync points

    t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])

    st = p.stats()
    fin = torch.tensor([float(final_cost)], dtype=torch.float64, device="cuda")      # identical on every rank by construction; checked here
    if world > 1:
        lo = fin.clone(); dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(fin, op=dist.ReduceOp.MAX)
        assert float(lo) == float(fin), "ranks disagree on the cost"
    fma = torch.tensor([float(st["schur_fma"])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(fma)

    if rank == 0:
        peaks = load_peaks()
        corner = 4.0 * n_obs
        value = corner * K / (ms * 1e-3)
        nl = max(ph["jacobian_launches"], 1.0)
        jac_ms = ph["jacobian_kernel"] / nl                 # k_jac_project, CUDA events on the launching stream, inside the timed region
        acc_ms = ph["accumulate_kernel"] / nl               # k_asm_pairs + k_asm_mruns
        syrk_ms = ph["syrk_kernel"] / max(ph["syrk_launches"], 1.0)
        syrk_flop = 2.0 * st["schur_fma"]                   # this rank's frames
        traffic = {}
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "jacobian_traffic.json")))
        except Exception:
            pass

        def entry(kernel, ms_launch, flop, bytes_alg, note, traffic_key):
            ach = flop / (ms_launch * 1e-3) / 1e12 if ms_launch > 0 else 0.0
            hbm = bytes_alg / (ms_launch * 1e-3) / 1e9 if ms_launch > 0 else 0.0
            t = traffic.get(traffic_key) if world == 1 and args.workload == "cfg4" and args.frames is None else None
            return {"kernel": kernel, "bound": "fp64", "achieved": ach, "peak": peaks["fp64_tflops"], "unit": "TFLOP/s", "frac": ach / peaks["fp64_tflops"],
                    "peak_source": peaks["fp64_src"], "ms_per_launch": ms_launch, "share_of_step": ms_launch * (1 if "syrk" not in kernel else ph["syrk_launches"] / nl) / (ms / K),
                    "algorithmic_flop_per_launch": flop, "note": note,
                    "hbm": {"achieved": hbm, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": hbm / peaks["hbm_gbs"], "algorithmic_bytes_per_launch": bytes_alg, "peak_source": peaks["hbm_src"]},
                    "traffic": t, "traffic_over_algorithmic": (t / bytes_alg if (t and bytes_alg) else None),
                    "dram_gbs_at_traffic": (t / (ms_launch * 1e-3) / 1e9 if (t and ms_launch > 0) else None),
                    "dram_frac_of_peak_at_traffic": (t / (ms_launch * 1e-3) / 1e9 / peaks["hbm_gbs"] if (t and ms_launch > 0) else None)}
        if args.analytic:        # not the headline: the analytic-Jacobian / full-FP64 variant (include/aar_analytic.h), rows staged in double
            kernels_an = entry("k_jac_analytic", jac_ms, W_AN_FLOP * n_local, OBS_BYTES * n_local,
                               "analytic 8 x 18 Jacobian block + residual of every marker observation in double (about 1.7 kflop: 3 chained rigid transforms, one division and 18 "
                               "directional derivatives per corner); writes 1280-byte rows — bound by the HBM writes, not by FP64", None)
        kernels = [
            kernels_an if args.analytic else
            entry("k_jac_project", jac_ms, W_PROJ_FLOP * n_local, OBS_BYTES * n_local,
                  "37 pinhole projections per marker observation (residual + quantised central-difference numerators); the reference's a*b+c are two IEEE operations "
                  "(-fmad=false, bit-exact parity), so the attainable peak of this kernel is the non-FMA issue rate = half the DFMA peak", "k_jac_project"),
            entry("k_asm_pairs+k_asm_mruns", acc_ms, W_ASM_FLOP * n_local, 0.0,
                  "J^T J / J^T r block products on the FP64 tensor cores (12 m8n8k4 DMMA per observation, 44 % of their lanes algorithmic); input is the staged numerator rows, "
                  "not algorithmic bytes", "k_asm"),
            entry("k_schur_syrk", syrk_ms, syrk_flop, 0.0, "S -= E E^T over the frames of this rank (upper triangle), FP64 tensor cores; launched once per LM try", "k_schur_syrk"),
        ]
        dom = max(kernels, key=lambda e: e["share_of_step"])
        flop_step = ((W_AN_FLOP + W_ASM_FLOP if args.analytic else W_J_FLOP) * n_local + 152.0 * n_local * tries_total / K + syrk_flop * tries_total / K)
        step_ach = flop_step / (ms / K * 1e-3) / 1e12
        line = {
            "metric": "corner_obs_per_s", "value": value, "unit": "corner-observations/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "lm_iters_per_s": K / (ms * 1e-3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": args.workload, "cameras": rig.C, "markers": rig.M, "frames": rig.F, "marker_observations": n_obs,
                       "corner_observations": int(corner), "num_vars": n_vars, "reduced_system": p.n_r, "parallelism": f"frame-shard x{world}",
                       "lm_loop": ("graph-resident (%d of the timed + warm-up iterations inside the CUDA graph)" % st["graph_iterations"]) if st["graph_loop"] else "host-driven",
                       "collective": ("reduced system and decision scalars summed by their consumers over NVLink peer memory (cudaIpc); NCCL for set-up only" if st["peer_reduction"]
                                      else ("ncclAllReduce per LM try" if world > 1 else "none")),
                       "l2": ("per-step working set %.0f MB per rank (observations + staged Jacobian block, streamed once per step) %s the 126 MB L2; no explicit flush"
                              % ((OBS_BYTES + 2 * STAGE_BYTES) * n_local / 1e6, "exceeds" if (OBS_BYTES + 2 * STAGE_BYTES) * n_local > 2 * 126e6 else "does NOT exceed")),
                       "jacobian": ("analytic, residuals in double (aar_problem_desc::analytic_jacobian = 1; NOT the reference's arithmetic)" if args.analytic
                                    else "the reference's central differences on float32-rounded projections (bit-exact parity path)"),
                       "restart_every": RESTART, "step": "one SparseLevMarq::step (J + JtJ + Schur + solve + trial residual)"},
            "e2e": {"value": corner * K / (ms_e2e * 1e-3), "unit": "corner-observations/s", "ms_per_step": ms_e2e / K,
                    "h2d_bytes_per_step": int(8 * n_vars * calls / K), "d2h_bytes_per_step": int((8 * n_vars * calls + 96 * e2e_tries) / K),
                    "call": f"aar_lm_solve(host io_vec) x{calls}, {chunk} iterations each",
                    "create_s": t_create, "create_note": "aar_problem_create (row map, upload, undistortion) is the MultiCamMapper constructor, outside solve(); reported, not in value"},
            "gpu_launches": int(launches),
            "clocks": clk,
            "roofline": dict(dom, kernels=kernels,
                             whole_step={"achieved": step_ach, "peak": peaks["fp64_tflops"], "unit": "TFLOP/s", "frac": step_ach / peaks["fp64_tflops"],
                                         "algorithmic_flop_per_step": flop_step, "rank": 0}),
            "phases_ms_per_step": {k: v / K for k, v in ph.items() if not k.endswith("_launches")}, "total_tries": int(tries_total),
            "phases_note": "per-phase / per-kernel CUDA-event times of a second pass over the same K iterations with the host-driven loop (%.3f ms per step); "
                           "`value` is the pass without events%s" % (ms_profiled / K, " (graph-resident loop)" if world == 1 else ""),
            "final_cost": float(fin), "final_cost_note": "cost after the last timed LM iteration (RESTART-periodic trajectory): equal across --gpus N to summation order",
            "setup_s": {"generate": t_gen, "create_upload_undistort": t_create},
        }
        if world == 1 and not args.no_cpu_baseline:
            r = cpu_reference_run(args.workload, CPU_SAMPLE_FRAMES, CPU_SAMPLE_ITERS)
            line["cpu_baseline"] = {"value": 4.0 * r["n_obs"] * r["iters"] / r["seconds"], "unit": "corner-observations/s", "cores": r["cores"],
                                    "kind": r["kind"], "sample": r["sample"], "ms_per_step_on_sample": 1e3 * r["seconds"] / r["iters"]}
            try:
                line["parity_check"] = parity_check(r, local_rank)
            except Exception as e:
                line["parity_check"] = {"error": str(e)[:300]}
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, z=z_last, final_cost=[float(fin)])
    p.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg4")
    ap.add_argument("--frames", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-track", action="store_true")
    ap.add_argument("--analytic", action="store_true", help="analytic-Jacobian / full-FP64 variant instead of the parity path (no cpu_baseline / parity_check legs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step as DIR/<name>.npy (float64): z and final_cost of the LM solve, "
                         "or z, cost and iterations per frame of track (cfg5)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        (run_track_reference if args.workload == "cfg5" else run_reference)(args, rank)
        return
    if world == 1 and args.gpus > 1:
        # launched without torchrun: re-launch one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", str(29500 + os.getpid() % 1000), os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    args.warmup = max(args.warmup, 3)
    (run_track if args.workload == "cfg5" else run_ours)(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
