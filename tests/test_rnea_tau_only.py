"""tau does not depend on the gantry velocities qd[0..2] of the sequential structure (a Galilean boost: no rotation precedes those
joints), so the fast inverse-dynamics kernels that return tau alone treat them as structural zeros and never load them
(fast_rnea_core<..., TWIST = false>, csrc/rbm_rnea.cuh).  The -m "not gpu" part checks that evaluation on the host harness against
the goldens and the full evaluation; the -m gpu part checks what the kernels load and that asking for the twist still reads the
gantry velocities."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import load_golden
from rigid_body_manipulation_b200 import engine

TARGETS = ["hammer", "uniform_gearbox", "kill_la_kill"]


def rel_err(a, b, floor=1e-6):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    ax = tuple(range(1, a.ndim))
    return np.max(np.abs(a - b), axis=ax) / np.maximum(np.max(np.abs(b), axis=ax), floor)


def _harness():
    hh = pytest.importorskip("host_harness")
    if hh.nvcc_path() is None:  # pragma: no cover
        pytest.skip("nvcc is needed to build the host harness")
    return hh


@pytest.fixture(scope="module")
def tau_only(tmp_path_factory):
    """tests/host_harness/tau_only.cu built for the host: (path, fast params, traj (n, 3, 6), dtype) -> tau (n, 6) of the tau-only
    recursion."""
    hh = _harness()
    src = os.path.join(hh.HERE, "tau_only.cu")
    lib = str(tmp_path_factory.mktemp("tau_only") / "libtau_only.so")
    subprocess.run([hh.nvcc_path(), "-O2", "-std=c++17", "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets", "-gencode",
                    "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC", "-I", hh.CSRC, "-I", os.path.join(hh.ROOT, "include"),
                    "-o", lib, src], check=True)
    dll = C.CDLL(lib)

    def run(path, fast_params, traj, dtype=np.float64):
        traj = np.ascontiguousarray(traj, dtype=dtype)
        tau = np.empty((traj.shape[0], 6), dtype)
        fn = dll.h_fast_rnea_tau_only_f64 if dtype == np.float64 else dll.h_fast_rnea_tau_only_f32
        fp = np.ascontiguousarray(fast_params, dtype=np.float64)
        ptr = lambda a: a.ctypes.data_as(C.c_void_p)
        assert fn(C.c_int(hh.PATH_ID[path]), ptr(fp), ptr(traj), ptr(tau), C.c_int64(traj.shape[0])) == 0
        return tau

    return run


def _analyze(g):
    return engine.analyze_model(g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"], pose_sen_llj=g["pose_sen_llj"])


# ---- host harness (no GPU) ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("t", TARGETS)
def test_tau_only_recursion_matches_golden_and_full_evaluation(t, tau_only):
    hh = _harness()
    g = load_golden(f"ref_inverse_{t}.npz")
    path, fast, _ = _analyze(g)
    tau = tau_only(path, fast, g["traj"])
    assert rel_err(tau, g["tau"]).max() < 1e-12
    full, _, _ = hh.fast_rnea(path, fast, g["traj"], mode=0)
    assert rel_err(tau, full).max() < 1e-13
    tau_r = tau_only("seq_rigid", fast, g["traj"])
    assert rel_err(tau_r, g["tau"]).max() < 1e-12


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_tau_only_recursion_never_reads_the_gantry_velocities(dtype, tau_only):
    hh = _harness()
    g = load_golden("ref_inverse_hammer.npz")
    path, fast, _ = _analyze(g)
    traj = g["traj"].astype(dtype)
    nan, zero = traj.copy(), traj.copy()
    nan[:, 1, :3] = np.nan
    zero[:, 1, :3] = 0.0
    t_nan = tau_only(path, fast, nan, dtype)
    t_zero = tau_only(path, fast, zero, dtype)
    assert np.isfinite(t_nan).all() and np.array_equal(t_nan, t_zero)
    # the full evaluation (what the twist-returning kernels run their forward sweep with) does read them
    assert np.isnan(hh.fast_rnea(path, fast, nan, mode=0, dtype=dtype)[1]).any()


# ---- device kernels ---------------------------------------------------------------------------------------------------------------
TOLS = {"f64": 1e-9, "f32": 1e-4}


def _gpu():
    import torch

    from gpu_util import model_from_golden, sample_states, soa
    from oracle import rnea_vec as rv

    return torch, model_from_golden, sample_states, soa, rv


def _oracle(rv, g, traj):
    return rv.inverse_batched(traj, g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"])


@pytest.mark.gpu
@pytest.mark.parametrize("dt", ["f64", "f32"])
@pytest.mark.parametrize("n", [4096, 4096 + 77])  # even / odd row pitch: both fp32 kernels
def test_device_tau_ignores_the_gantry_velocities(dt, n):
    torch, model_from_golden, sample_states, soa, rv = _gpu()
    tdt = torch.float64 if dt == "f64" else torch.float32
    g = load_golden("ref_inverse_hammer.npz")
    m = model_from_golden(g)
    traj = sample_states(np.random.default_rng(n), n)
    ref = _oracle(rv, g, traj)
    q, qd, qdd = soa(traj, tdt)
    qd_nan, qd_other = qd.clone(), qd.clone()
    qd_nan[:3] = float("nan")
    qd_other[:3] = qd_other[:3] * -3.0 + 1.0
    tau = m.rnea(q, qd_nan, qdd)
    assert rel_err(tau.t().cpu().numpy(), ref["tau"]).max() < TOLS[dt]
    assert torch.equal(tau, m.rnea(q, qd_other, qdd)) and torch.equal(tau, m.rnea(q, qd, qdd))
    # the AoS kernels load every value but evaluate the same tau-only recursion
    traj_nan = traj.copy()
    traj_nan[:, 1, :3] = np.nan
    tau_aos = m.rnea_aos(torch.as_tensor(traj_nan, dtype=tdt, device="cuda")).cpu().numpy()
    assert rel_err(tau_aos, ref["tau"]).max() < TOLS[dt]
    # asking for the twist reads them again: V_6 moves with the gantry velocities, tau does not
    tau_tw, V, dV = m.rnea(q, qd, qdd, want_twists=True)
    assert torch.equal(tau_tw, tau)
    assert rel_err(V.t().cpu().numpy(), ref["twists"][:, 6]).max() < TOLS[dt]
    assert rel_err(dV.t().cpu().numpy(), ref["dtwists"][:, 6]).max() < TOLS[dt]
    tau_o, V_o, _ = m.rnea(q, qd_other, qdd, want_twists=True)
    assert torch.equal(tau_o, tau) and not torch.equal(V_o, V)
    assert torch.isnan(m.rnea(q, qd_nan, qdd, want_twists=True)[1]).any()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-9), (np.float32, 1e-4)])
def test_host_soa_entry_with_unset_gantry_rows(dtype, tol):
    _, model_from_golden, sample_states, _, rv = _gpu()
    g = load_golden("ref_inverse_hammer.npz")
    m = model_from_golden(g)
    n = 131_072 * 2 + 17
    traj = sample_states(np.random.default_rng(3), n)
    ref = _oracle(rv, g, traj)["tau"]
    q, qd, qdd = (np.ascontiguousarray(traj[:, k, :].T).astype(dtype) for k in range(3))
    q[:3] = np.nan
    qd[:3] = np.nan
    tau = m.rnea_host_soa(q, qd, qdd, chunk=131_072)
    assert rel_err(tau.T, ref).max() < tol


@pytest.mark.gpu
def test_generic_path_still_reads_every_velocity():
    torch, model_from_golden, sample_states, soa, _ = _gpu()
    g = load_golden("ref_inverse_hammer.npz")
    m = model_from_golden(g, force_generic=True)
    q, qd, qdd = soa(sample_states(np.random.default_rng(4), 1000))
    qd[:3] = float("nan")
    assert torch.isnan(m.rnea(q, qd, qdd)).any()
