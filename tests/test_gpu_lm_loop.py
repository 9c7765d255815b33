"""aar_lm_iterate across calls: the LM state (LmState) stays on the device between calls, and both loops (graph-resident and
host-driven) decide with it.  A solve split into several calls must take the decisions of one call, and the verbose log of the
host-driven loop must print the records of the trace."""
import ctypes

import numpy as np
import pytest

from aar_b200 import synth
from conftest import parity_record
from test_gpu_parity import _end_point_dev, _same, _same_cost

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def binding():
    from aar_b200 import binding as b
    b.lib()
    return b


def _split_solve(p, z0, prm, step=3):
    """lm_begin, lm_iterate(step) until the stop rules end the solve or max_iters are done, lm_end: how bench.py drives the loop."""
    p.lm_begin(z0, prm)
    traces, iters = [], 0
    while iters < prm.max_iters:
        want = min(step, prm.max_iters - iters)
        rep, tr = p.lm_iterate(want, trace_capacity=step)
        assert rep.iterations == want or rep.exit_code != 0, (rep.iterations, want, rep.exit_code)
        traces.append(tr); iters += rep.iterations
        if rep.exit_code:
            break
    return p.lm_end(), rep.final_cost, iters, np.concatenate(traces), rep.total_tries, rep.initial_cost


@pytest.mark.parametrize("loop", ["graph", "host"])
def test_split_solve_equals_one_solve(binding, monkeypatch, loop):
    rig = synth.make_config("cfg1")
    p = binding.Problem(rig, with_huber=True)
    plain = binding.Problem(rig)
    z0 = p.mats2evec()
    if loop == "host":
        monkeypatch.setenv("AAR_NO_GRAPH", "1")
    records, iters = {}, {}
    for mode, prm in (("solve", binding.Problem.default_params()), ("capped", binding.Problem.default_params(max_iters=10, ignore_stop_rules=1))):
        g0 = p.stats()["graph_iterations"]
        z_1, c_1, it_1, tr_1 = p.solve(z0, prm, trace_capacity=16384)
        tries_1 = p.last_report.total_tries
        z_s, c_s, it_s, tr_s, tries_s, _ = _split_solve(p, z0, prm)
        graph_iters = p.stats()["graph_iterations"] - g0; iters[mode] = int(it_1)
        # every iteration but the first of each solve runs inside the graph, none with AAR_NO_GRAPH=1
        assert graph_iters == (it_1 - 1 + it_s - 1 if loop == "graph" else 0), (loop, graph_iters, it_1, it_s)
        assert it_s == it_1 == len(tr_1) and tries_s == tries_1 == tr_1[:, 3].sum(), (mode, it_s, it_1, tries_s, tries_1)
        assert np.array_equal(tr_s[:, 3:6], tr_1[:, 3:6]), mode             # tries, accepted, Huber schedule
        assert _same(tr_s[:, 0], tr_1[:, 0]) and _same(tr_s[:, 1], tr_1[:, 1], 1e-7), mode
        cost_ok, flips = _same_cost(plain, z_s, c_s, z_1, c_1)
        assert cost_ok, (mode, c_s, c_1, flips)
        if mode == "solve":
            records[mode] = _end_point_dev(p, z0, z_s, z_1)
        else:
            assert it_1 == 10 and _same(z_s, z_1), mode
            records[mode] = float(np.abs(z_s - z_1).max() / np.abs(z_1).max())
    plain.close()
    parity_record("lm_split_solve_vs_one_solve", loop=loop, workload="cfg1 + Huber", iterate_step=3, iterations=iters, z_rel_dev=records)


def test_verbose_lines_are_the_trace(binding, capfd):
    """verbose = 1 prints the reference's line per iteration (sparselevmarq.h:421) from the record of the iteration, across calls."""
    rig = synth.make_config("cfg1")
    p = binding.Problem(rig, with_huber=True)
    capfd.readouterr()
    _, _, iters, tr, _, initial = _split_solve(p, p.mats2evec(), binding.Problem.default_params(verbose=1))
    ctypes.CDLL(None).fflush(None)                                  # the library's printf goes through the C stdio buffer
    out = [line for line in capfd.readouterr().out.splitlines() if line.startswith("Curr Error=")]
    rows = 8 * p.num_obs
    prev = np.concatenate([[initial], tr[:-1, 0]])
    want = ["Curr Error=%.5g AErr(prev-curr)=%.5g gain=%.5g dumping factor=%.5g" % (c, (pc - c) / rows, g, mu)
            for (c, mu, g), pc in zip(tr[:, :3], prev)]
    assert len(want) == iters > 0 and out == want, (iters, out[:3], want[:3])
