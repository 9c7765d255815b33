"""Frame-sharded solve on N GPUs (NCCL all-reduce of the reduced Schur system and the cost, SURVEY 8e) against the
single-GPU solve of the same problem: world 2 on BASELINE config 2 and world 8 on config 3.  Needs that many CUDA devices
(gpurun --gpus N); skipped otherwise.  The deviations achieved are kept in gpurun_out/parity_achieved.jsonl."""
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, parity_record

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, out_dir, cfg):
    for p in (os.path.join(ROOT, "automatic-ar_b200", "python"),):
        sys.path.insert(0, p)
    import torch
    import torch.distributed as dist
    from aar_b200 import binding, synth
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    rig = synth.make_config(cfg)
    p = binding.Problem(rig, device=rank, rank=rank, world_size=world)
    idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        idt.copy_(torch.frombuffer(bytearray(binding.comm_unique_id()), dtype=torch.uint8))
    dist.broadcast(idt, 0)
    p.comm_init(bytes(idt.cpu().numpy().tobytes()))
    z0 = p.mats2evec()
    # reduced Schur system of the shards, summed over the ranks (SURVEY 8e: 1e-12 relative across GPU counts)
    mu = 1234.5
    S, b, c = p.reduced_system(z0, mu)
    buf = torch.from_numpy(np.concatenate([S.ravel(), b, [c]])).cuda()
    dist.all_reduce(buf)
    buf = buf.cpu().numpy()
    out = {}
    for k in (3, 10000):
        z, fc, it, tr = p.solve(z0, binding.Problem.default_params(max_iters=k))
        out[k] = (z, fc, it, tr)
    if rank == 0:
        single = binding.Problem(rig, device=0)
        S1, b1, c1 = single.reduced_system(z0, mu)
        n = p.n_r; iu = np.triu_indices(n)
        dS = np.abs(buf[:n * n].reshape(n, n)[iu] - S1[iu]).max() / np.abs(S1).max()
        db = np.abs(buf[n * n:n * n + n] - b1).max() / np.abs(b1).max(); dc = abs(buf[-1] - c1) / c1
        rec = {"world": world, "workload": cfg, "reduced_system_rel_dev": dS, "reduced_rhs_rel_dev": db, "cost_rel_dev": dc}
        assert dS <= 1e-12 and db <= 1e-12 and dc <= 1e-12, rec
        for k in (3, 10000):
            z1, fc1, it1, tr1 = single.solve(z0, binding.Problem.default_params(max_iters=k))
            z, fc, it, tr = out[k]
            if k == 3:      # before any float32 flip can separate the trajectories: summation order only
                assert it == it1 == 3
                rec["three_iterations_rel_dev_cost"] = abs(fc - fc1) / fc1; rec["three_iterations_rel_dev_z"] = np.abs(z - z1).max() / np.abs(z1).max()
                assert abs(fc - fc1) <= 1e-10 * fc1 and np.abs(z - z1).max() <= 1e-10 * np.abs(z1).max()
            else:           # full solve: inside the reproducibility envelope of the quantised Jacobian (DESIGN.md)
                rec["full_solve_iterations"] = [int(it1), int(it)]; rec["full_solve_rel_dev_cost"] = abs(fc - fc1) / fc1
                assert abs(it - it1) <= 1 and abs(fc - fc1) <= 2e-5 * fc1
        rec["collective"] = "ncclAllReduce per try, host-driven loop"
        parity_record(f"multi_gpu_world{world}_{cfg}_vs_single_gpu", **rec)
        open(os.path.join(out_dir, "ok"), "w").write("ok")
    # every rank returns the full z: the shards' frame poses are exchanged at the end
    zs = [torch.zeros(len(z0), dtype=torch.float64, device="cuda") for _ in range(world)]
    dist.all_gather(zs, torch.from_numpy(out[3][0]).cuda())
    assert all(torch.equal(zs[0], zs[r]) for r in range(1, world))
    p.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,cfg", [(2, "cfg2"), (8, "cfg3")])
def test_sharded_solve_matches_single_gpu(tmp_path, world, cfg):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    port = 29700 + os.getpid() % 200 + world
    mp.spawn(_worker, args=(world, port, str(tmp_path), cfg), nprocs=world, join=True)
    assert os.path.exists(os.path.join(tmp_path, "ok"))
