"""The closed-loop path pinned to THE REFERENCE'S OWN CODE: tests/golden/ref_simulate_{hammer,uniform_gearbox}.npz hold what the
reference's core/simulate.py::simulate returned (controllers/lqr.py, the planner, sensors and pose registers executed unmodified on the
functional MuJoCo stand-in of oracle/mujoco_standin.py, full 1500-step runs written by oracle/gen_golden_simulate.py).

  * oracle/replay_oracle.py reproduces those runs, i.e. the restated loop (LQR gain, frame schedule, lagged qacc / sensordata, control
    law, sensor-frame twists, noise model) is the reference's;
  * the kernels' rollout algorithm (host build of csrc/rbm_dynamics.cuh here, the CUDA kernel in tests/test_gpu_replay.py) reproduces
    them too.
What the stand-in restates of MuJoCo (plant step, F/T sensor) is listed in its header; that part stays unpinned against MuJoCo itself."""
import os

import numpy as np
import pytest

from conftest import load_golden
from oracle import replay_oracle as ro
from oracle import rnea_vec as rv
from rigid_body_manipulation_b200 import engine, identification as idn, planner

os.environ.setdefault("TQDM_DISABLE", "1")


def _consts(g):
    return dict(hposes_Rt=g["hposes_Rt"], simats=g["simats"], uscrews=g["uscrews"], twist_0=g["twist_0"], dtwist_0=g["dtwist_0"])


def test_reference_simulate_equals_the_restated_loop():
    for target in ("hammer", "uniform_gearbox"):
        g = load_golden(f"ref_simulate_{target}.npz")
        Kr = ro.lqr_gain(_consts(g), g["key_qpos"], np.zeros(6), [10.0, 10.0, 10.0, 1e4, 1e4, 1e4])
        assert np.abs(g["gain_matrix"] - Kr).max() < 1e-12 * np.abs(Kr).max()    # the reference's controller on the stand-in == the restatement
        pl = planner.QuinticPlan(g["displacements"], g["key_qpos"], float(g["timestep"]), int(g["n_steps"]))
        out = ro.closed_loop_replay(_consts(g), g["pose_sen_llj"], g["G_sensed"], pl.trajectory(), Kr, g["key_qpos"])
        assert len(out["step"]) == g["twist_sen"].shape[0] == 150
        for key, mine in (("twist_sen", out["twist_sen"]), ("dtwist_sen", out["dtwist_sen"]), ("ft_sen", idn.perturb_wrench(out["wrench"], 0.05, 0))):
            assert np.abs(g[key] - mine).max() < 1e-12 * np.abs(mine).max(), (target, key)
        assert np.abs(g["regressors"] - out["regressor"]).max() < 1e-12 * np.abs(out["regressor"]).max(), target


@pytest.mark.parametrize("target", ["hammer", "uniform_gearbox"])
def test_rollout_algorithm_reproduces_the_reference_run(target):
    host_harness = pytest.importorskip("host_harness")
    if host_harness.nvcc_path() is None:  # pragma: no cover
        pytest.skip("nvcc is needed to build the host harness")
    g = load_golden(f"ref_simulate_{target}.npz")
    an = engine.analyze_model(g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"], pose_sen_llj=g["pose_sen_llj"])
    assert an[0] == "seq_iso"
    pl = planner.QuinticPlan(g["displacements"], g["key_qpos"], float(g["timestep"]), int(g["n_steps"]))
    phi = ro.inertia_to_phi(g["G_sensed"])
    out = host_harness.closed_loop(an, pl, g["gain_matrix"], phi, g["key_qpos"][None])
    fr = out["frames"][..., 0]
    assert fr.shape[0] == g["twist_sen"].shape[0] == 150
    assert np.abs(fr[:, 18:24] - g["twist_sen"]).max() < 1e-9 * np.abs(g["twist_sen"]).max()
    assert np.abs(fr[:, 24:30] - g["dtwist_sen"]).max() < 1e-9 * np.abs(g["dtwist_sen"]).max()
    noisy = idn.perturb_wrench(fr[:, 30:36], 0.05, 0)                                    # simulate.py:279-290
    assert np.abs(noisy - g["ft_sen"]).max() < 1e-9 * np.abs(g["ft_sen"]).max()
    Y = rv.regressor_batched(fr[:, 18:24], fr[:, 24:30])
    assert np.abs(Y - g["regressors"]).max() < 1e-9 * np.abs(g["regressors"]).max()
    # and the identification the reference's logger would run on its own data (loggers.py:127-129) == ours on ours
    phi_ref = np.linalg.lstsq(g["regressors"].reshape(-1, 10), g["ft_sen"].reshape(-1), rcond=None)[0]
    phi_own = np.linalg.lstsq(Y.reshape(-1, 10), noisy.reshape(-1), rcond=None)[0]
    assert np.abs(phi_ref - phi_own).max() < 1e-7 * np.abs(phi_ref).max()
