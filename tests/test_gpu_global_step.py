"""Global-step mode (SURVEY.md §8e): one line-search step size for the whole batch, agreed across ranks with one NCCL collective.

Not a reference semantic (the reference searches per instance), so the checks are consistency properties against the per-instance mode:
  * every instance takes the same step; it is a ladder candidate that the per-instance filter accepts for every instance
    (so it cannot exceed any instance's own first accepted candidate when acceptance is monotone down to it);
  * with a single instance the two modes coincide bit for bit.
The 2-rank NCCL path runs under torchrun when >= 2 GPUs are visible (tests/mgpu_global_step.py)."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from wb_humanoid_mpc_b200 import abi, model_loader
from test_gpu_wb import make_instances

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]


def lg(res, name):
    from wb_humanoid_mpc_b200.solver import LOG_FIELDS

    return res["log"][:, :, LOG_FIELDS.index(name)]


@pytest.fixture(scope="module")
def model():
    return model_loader.load_packaged_model()


def test_single_instance_matches_per_instance_mode(model):
    from wb_humanoid_mpc_b200.solver import B200SqpSolver

    insts = make_instances(model, np.random.default_rng(5), [("walk", 1.1, [0.5, 0.1, 0.7925, 0.2])])
    res = {}
    for mode in (0, 1):
        s = B200SqpSolver(model, abi.default_settings(model, sqp_iteration=3, global_step=mode))
        if mode:
            s.enable_global_step()
        res[mode] = s.run(insts)
        s.close()
    assert np.array_equal(lg(res[0], "step_size"), lg(res[1], "step_size"))
    assert np.array_equal(res[0]["x"], res[1]["x"]) and np.array_equal(res[0]["u"], res[1]["u"])


def test_batch_takes_one_admissible_step(model):
    from wb_humanoid_mpc_b200.solver import B200SqpSolver

    rng = np.random.default_rng(11)
    specs = [("walk", 1.1, [rng.uniform(-0.5, 1.0), rng.uniform(-0.3, 0.3), 0.7925, rng.uniform(-0.5, 0.5)]) for _ in range(6)]
    insts = make_instances(model, rng, specs)
    per = B200SqpSolver(model, abi.default_settings(model, sqp_iteration=1, global_step=0))
    r0 = per.run(insts)
    glob = B200SqpSolver(model, abi.default_settings(model, sqp_iteration=1, global_step=1))
    glob.enable_global_step()   # single process: no communicator, the local statistics decide
    r1 = glob.run(insts)
    ladder = glob.global_ladder()
    assert ladder[0] == 1.0 and np.allclose(ladder[1:] / ladder[:-1], 0.5) and ladder[-1] >= 1e-4
    a = lg(r1, "step_size")[:, 0]
    assert np.all(a == a[0]), "all instances must take the same step"
    assert a[0] == 0.0 or np.any(np.isclose(ladder, a[0]))
    # the linearisation is identical in both modes: same baseline merit, same Armijo slope, same QP step norms
    for key in ("base_merit", "armijo"):
        assert np.allclose(lg(r0, key)[:, 0], lg(r1, key)[:, 0], rtol=1e-12, atol=0)
    # instances whose own search stopped at the global candidate end at the same iterate
    same = np.isclose(lg(r0, "step_size")[:, 0], a[0])
    assert np.allclose(r0["x"][same], r1["x"][same], rtol=0, atol=1e-12)
    g, idx = glob.global_stats()
    if a[0] > 0:
        assert len(g) == idx + 1, "the ladder is walked lazily: nothing beyond the applied candidate is rolled out"
        assert ladder[idx] == a[0] and g[idx, 0] == g[idx, 3] == len(insts)
        assert np.all(g[:idx, 0] < g[:idx, 3]), "a larger candidate accepted by everybody would have been chosen"


def test_centroidal_handle_global_step():
    """the global-step mode on a centroidal handle: two instances take one common admissible step"""
    from test_gpu_cen_ocp import make_instance
    from wb_humanoid_mpc_b200.solver import B200SqpSolver

    cmodel = model_loader.load_packaged_model("g1_centroidal")
    rng = np.random.default_rng(4)
    insts = [make_instance(cmodel, rng, "walk", 0.2, [0.3, 0.0, 0.7925, 0.0]), make_instance(cmodel, rng, "stance", 0.2, [0.0, 0.1, 0.7925, 0.1])]
    if len(insts[0]["t_nodes"]) != len(insts[1]["t_nodes"]):
        insts[1] = make_instance(cmodel, rng, "walk", 0.2, [0.0, 0.1, 0.7925, 0.1])
    s = B200SqpSolver(cmodel, abi.default_settings(cmodel, sqp_iteration=1, global_step=1))
    r = s.run(insts)
    a = lg(r, "step_size")[:, 0]
    assert a[0] == a[1] and (a[0] == 0.0 or np.any(np.isclose(s.global_ladder(), a[0])))
    g, idx = s.global_stats()
    assert idx == len(g) - 1 if a[0] > 0 else idx == -1


def test_two_rank_nccl(model):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (python -m pytest tests/test_gpu_global_step.py -m gpu on a machine with two)")
    env = dict(os.environ, PYTHONPATH=f"{ROOT}:{ROOT / 'tests'}")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                          "--master-port", "29533", str(ROOT / "tests" / "mgpu_global_step.py")], capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "GLOBAL_STEP_OK" in out.stdout
