"""`not gpu`: the generic per-sample algorithms at every joint count of tests/chains.py (1 to 16), with and without a tip wrench, compiled
for the host from the headers the kernels use (tests/host_harness), against the oracles.  The -m gpu twin, tests/test_gpu_joint_counts.py,
runs the same chains through the kernels; a failure here that is absent there (or the reverse) places a bug on the host or the device
side of the shared headers."""
import numpy as np
import pytest

import chains
from oracle import lqr_oracle as lo
from oracle import replay_oracle as ro
from oracle import rnea_vec as rv
from rigid_body_manipulation_b200 import planner
from test_payload_identification import harness, oracle_payload, phi_to_inertia  # noqa: F401  (harness is a fixture)

host_harness = pytest.importorskip("host_harness")
if host_harness.nvcc_path() is None:  # pragma: no cover
    pytest.skip("nvcc is needed to build the host harness", allow_module_level=True)

CASES = [pytest.param(nj, tip, id=f"nj{nj}-{'tip' if tip else 'notip'}") for nj in chains.NJ_ALL for tip in (True, False)]


def _chain(nj, tip):
    ch = chains.random_chain(nj, seed=100 + nj, tip=tip)
    return ch, ch.analyze()


def _rel(a, b):
    return np.abs(np.asarray(a, np.float64) - b).max() / max(np.abs(b).max(), 1e-6)


def _controls(nj, n, seed):
    return np.random.default_rng(seed).standard_normal((n, nj)) * 20


def test_model_validation_accepts_1_to_16_joints_only():
    """rbm_model_analyze and rbm_model_create validate the joint count before they touch a device: 1 and 16 are accepted, 17 is
    unsupported and 0 invalid (the constants of a 17-joint chain are well formed, so only the count can be refused)."""
    import ctypes as C

    from rigid_body_manipulation_b200 import _lib
    from rigid_body_manipulation_b200.engine import _ptr

    lib = _lib.load()
    ch = chains.random_chain(17, 0, tip=False)
    c = {k: np.ascontiguousarray(v, np.float64) for k, v in ch.consts.items()}
    ptrs = [_ptr(c[k]) for k in ("hposes_Rt", "simats", "uscrews", "twist_0", "dtwist_0")]
    path = C.c_int(-1)
    for nj, want in ((1, _lib.RBM_OK), (16, _lib.RBM_OK), (17, _lib.RBM_ERR_UNSUPPORTED), (0, _lib.RBM_ERR_INVALID)):
        assert lib.rbm_model_analyze(nj, *ptrs, None, None, None, 0, C.byref(path), None, None) == want, nj
        assert (lib.rbm_generic_param_count(nj) > 0) == (want == _lib.RBM_OK)
        if want != _lib.RBM_OK:
            h = C.c_void_p()
            assert lib.rbm_model_create(nj, *ptrs, None, None, None, 0, 0, C.byref(h)) == want and not h.value
    assert chains.random_chain(16, 0).analyze()[0] == "generic"


@pytest.mark.parametrize("nj,tip", CASES)
def test_generic_rnea(nj, tip):
    ch, an = _chain(nj, tip)
    traj = ch.sample(200, nj)
    ref = rv.inverse_batched(traj, **_vec(ch))
    out = host_harness.generic_rnea(an[2], nj, traj, full=True)
    assert _rel(out["tau"], ref["tau"]) < 1e-9
    assert _rel(out["poses"], ref["poses"]) < 1e-9
    assert _rel(out["twists"], ref["twists"]) < 1e-9 and _rel(out["dtwists"], ref["dtwists"]) < 1e-9
    if nj == 6:
        unrolled = host_harness.generic_rnea(an[2], nj, traj, unrolled=True)
        assert _rel(unrolled["tau"], ref["tau"]) < 1e-9
    # fp32: the 2e5 edge row loses ~1e-2 of its angle to float rounding, which the oracle (fed the same float inputs) sees too
    t32 = traj.astype(np.float32)
    ref32 = rv.inverse_batched(t32.astype(np.float64), **_vec(ch))["tau"]
    assert _rel(host_harness.generic_rnea_f32(an[2], nj, t32), ref32) < 1e-4


def _vec(ch):
    c = ch.consts
    return dict(hposes_Rt=c["hposes_Rt"], simats=c["simats"], uscrews=c["uscrews"], twist_0=c["twist_0"], dtwist_0=c["dtwist_0"], **lo.tip_kw(c))


@pytest.mark.parametrize("nj,tip", CASES)
def test_forward_dynamics_step_and_linearisation(nj, tip):
    ch, an = _chain(nj, tip)
    n = 12
    traj = ch.sample(n, 200 + nj)
    q, qd, u = traj[:, 0], traj[:, 1], _controls(nj, n, nj)
    c = ch.consts
    ref = lo.forward_dynamics(c, q, qd, u)
    assert _rel(host_harness.forward_dynamics(an, q, qd, u), ref) < 1e-9
    _, qn, qdn = host_harness.forward_dynamics(an, q, qd, u, dt=0.002)
    y = lo.step(c, q, qd, u, 0.002)
    assert _rel(np.concatenate([qn, qdn], 1), y) < 1e-11
    # the three settings and bounds of tests/test_kernel_dynamics_host.py.  Not at q = 2e5: there q +- eps itself is rounded by
    # ulp(2e5) = 3e-11, a 3e-6 relative error of the finite-difference step on both sides that no bound of 2e-8 can absorb
    lin = np.where(np.abs(q) > 1e3, 1.0, q)
    ref = lo.forward_dynamics(c, lin, qd, u)
    for centered, eps, tol_a, tol_b in ((True, 1e-5, 2e-8, 2e-8), (True, 1e-8, 5e-6, 5e-6), (False, 1e-6, 1e-4, 2e-7)):
        A, B, qdd = host_harness.linearize(an, lin, qd, u, dt=0.002, eps=eps, centered=centered)
        Ar, Br = lo.transition_fd(c, lin, qd, u, dt=0.002, eps=eps, centered=centered)
        assert np.abs(A - Ar).max() < tol_a and np.abs(B - Br).max() < tol_b, (centered, eps, np.abs(A - Ar).max(), np.abs(B - Br).max())
        assert _rel(qdd, ref) < 1e-9


@pytest.mark.parametrize("nj,tip", CASES)
def test_closed_loop(nj, tip):
    ch, an = _chain(nj, tip)
    rng = np.random.default_rng(300 + nj)
    key = rng.uniform(-1, 1, nj)
    n_steps = 100
    plan = planner.QuinticPlan(rng.uniform(-0.5, 0.5, nj), key, 0.002, n_steps)
    K = -np.hstack([50.0 * np.eye(nj), 5.0 * np.eye(nj)])
    phi = chains.phi_sensed(nj)
    G_s = phi_to_inertia(phi)
    q0 = np.stack([key, key + rng.uniform(-0.05, 0.05, nj)])
    qd0 = np.stack([np.zeros(nj), rng.uniform(-0.1, 0.1, nj)])
    out = host_harness.closed_loop(an, plan, K, phi, q0, qd0)   # divisor = nj, the engine's default
    for e in range(2):
        ref = ro.closed_loop_replay(ch.consts, ch.pose_sen_Rt, G_s, plan.trajectory(), K, q0[e], qd0[e], nu=float(nj))
        assert np.array_equal(out["frame_steps"], ref["step"])
        fr = out["frames"][..., e]
        for sl, key_ in ((slice(0, 3 * nj), "act"), (slice(3 * nj, 3 * nj + 6), "twist_sen"), (slice(3 * nj + 6, 3 * nj + 12), "dtwist_sen"),
                         (slice(3 * nj + 12, 3 * nj + 18), "wrench")):
            want = ref[key_].reshape(len(ref["step"]), -1)
            assert _rel(fr[:, sl], want) < 1e-9, (e, key_)
        fin = out["final"][:, e]
        assert np.abs(fin[:nj] - ref["q_final"]).max() < 1e-11 and np.abs(fin[nj:2 * nj] - ref["qd_final"]).max() < 1e-11


@pytest.mark.parametrize("nj,tip", CASES)
def test_gram_pack_and_payload_rows(nj, tip, harness):  # noqa: F811
    ch, an = _chain(nj, tip)
    n = 300
    traj = ch.sample(n, 400 + nj)
    rng = np.random.default_rng(nj)
    out = rv.inverse_batched(traj, **_vec(ch))
    Vs, dVs = rv.sensor_frame_twists_batched(ch.pose_sen_Rt, out["twists"][:, -1], out["dtwists"][:, -1])
    f = rv.regressor_batched(Vs, dVs) @ chains.phi_sensed(nj) + 0.01 * rng.standard_normal((n, 6))
    ref = rv.gram_pack(rv.regressor_batched(Vs, dVs), f)
    got = host_harness.regressor_gram(an, traj[:, 0], traj[:, 1], traj[:, 2], f)
    assert got[111] == n and np.abs(got - ref).max() < 1e-10 * np.abs(ref).max()
    c = ch.consts
    ref_phi, ref_tau0 = oracle_payload(c, ch.pose_sen_Rt, traj, **lo.tip_kw(c))
    Phi, tau0 = harness["payload"](an, traj)
    scale = np.abs(ref_tau0).max()
    assert np.abs(tau0 - ref_tau0).max() < 1e-9 * scale and np.abs(Phi - ref_phi).max() < 1e-9 * scale
