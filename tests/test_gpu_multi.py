"""The library's own multi-GPU layer (include/psulvsb.h "multi-GPU"): NCCL communicator per handle, hypothesis-sharded
scoring with the 8-byte max-allreduce, and ONE registration with its consistency rows sharded over the ranks
(psulvsb_solve_sharded; the reference loop registration.cc:682-767 cannot be split, being one thread).

world = 1 runs on any GPU box; world = 2 needs two GPUs and is skipped otherwise."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_world(world, tmp_path, n=3000):
    idf = str(tmp_path / "nccl_id.bin")
    outs = [str(tmp_path / f"rank{r}.npz") for r in range(world)]
    procs = [subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "tools", "sharded_worker.py"), str(r),
                               str(world), idf, outs[r], str(n)], cwd=ROOT, stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(world)]
    logs = []
    for p in procs:
        try:
            o, _ = p.communicate(timeout=600)
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise
        logs.append(o)
    for r, p in enumerate(procs):
        assert p.returncode == 0, f"rank {r} failed:\n{logs[r][-3000:]}"
    return [dict(np.load(o)) for o in outs]


def check_ranks(res, world):
    from psulvsb_b200 import sharding

    for r in res:
        assert r["sharded_ints"][4] == 0 and r["alone_ints"][4] == 0
        # the sharded registration is the single-GPU registration, bit for bit, on every rank
        assert np.array_equal(r["sharded_ints"], r["alone_ints"]), (r["sharded_ints"], r["alone_ints"])
        assert np.array_equal(r["sharded_R"], r["alone_R"]) and np.array_equal(r["sharded_t"], r["alone_t"])
        assert r["alone_ints"][1] >= 250  # 300 true inliers
        cnt, hid = sharding.unpack_best(int(r["best"][0]))
        assert hid == 4096 // 3 and cnt >= 250
        assert np.array_equal(r["rows"], np.arange(1000) + 1)
    assert len({int(r["best"][0]) for r in res}) == 1  # the same global best on every rank
    assert max(int(r["local_best"][0]) for r in res) == sharding.unpack_best(int(res[0]["best"][0]))[0]


def test_world_of_one_through_nccl(tmp_path):
    check_ranks(run_world(1, tmp_path), 1)


def test_world_of_two_shards_rows_and_hypotheses(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    check_ranks(run_world(2, tmp_path), 2)


def test_sharded_entry_points_without_communicator():
    import psulvsb_b200  # noqa: F401
    from psulvsb_b200 import capi, synth

    h = capi.Handle(0)
    pair = synth.make_pair(800, 0.9, 9)
    params = capi.default_params(noise_bound=0.05, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005,
                                 wallclock_cap_s=0.0, seed=3)
    prob = capi.HostProblem(pair["src"], pair["dst"])
    a = h.solve_sharded(params, prob)  # no communicator: psulvsb_solve
    b, _ = h.solve(params, prob)
    assert np.array_equal(np.array(a.rotation[:]), np.array(b.rotation[:])) and a.final_inlier_count == b.final_inlier_count
    assert h.comm_world == 1
    with pytest.raises(ValueError):
        h.comm_create(0, 1, b"short")
