"""`not gpu`: the per-state algorithms of csrc/rbm_dynamics.cuh (LQR linearisation, forward dynamics / step, closed-loop rollout),
compiled for the host from the same header the kernels use (tests/host_harness), against the CPU restatements -- the same checks
tests/test_gpu_linearize.py and tests/test_gpu_replay.py make through the C ABI on a GPU."""
import numpy as np
import pytest

import model_classes
from conftest import load_golden
from oracle import lqr_oracle as lo
from oracle import replay_oracle as ro
from rigid_body_manipulation_b200 import engine
from rigid_body_manipulation_b200 import model as pm
from rigid_body_manipulation_b200 import planner

host_harness = pytest.importorskip("host_harness")
if host_harness.nvcc_path() is None:  # pragma: no cover
    pytest.skip("nvcc is needed to build the host harness", allow_module_level=True)


def _states(rng, n):
    q = np.concatenate([rng.uniform(-1.5, 2.5, (n, 3)), rng.uniform(-6 * np.pi, 6 * np.pi, (n, 3))], axis=1)
    qd = rng.standard_normal((n, 6)) * [1, 1, 1, 3, 3, 3]
    return q, qd


def _consts(c):
    return dict(hposes_Rt=c.hposes_Rt, simats=c.simats, uscrews=c.uscrews, twist_0=c.twist_0, dtwist_0=c.dtwist_0)


def _model(target, force_generic):
    """(consts, analysis, sensor pose, sensed spatial inertia, keyframe) of a packaged target or of a tests/model_classes.py class;
    asserts the kernel path the model selects."""
    if target in model_classes.CLASSES:
        mc = model_classes.build(target)
        an = model_classes.analyze(mc, force_generic=force_generic)
        if force_generic:
            assert an[0] == "generic"
        return mc.consts, an, mc.pose_sen_Rt, mc.G_sensed, mc.key_qpos
    c = pm.load_packaged("sequential", target)
    an = engine.analyze_model(c.hposes_Rt, c.simats, c.uscrews, c.twist_0, c.dtwist_0, pose_sen_llj=c.pose_sen_Rt, force_generic=force_generic)
    assert an[0] == ("generic" if force_generic else "seq_iso")
    return _consts(c), an, c.pose_sen_Rt, ro.sensor_inertia(c.simat_object_llj, c.pose_sen_Rt), c.key_qpos


@pytest.mark.parametrize("target", ["hammer", "kill_la_kill", *model_classes.CLASSES])
@pytest.mark.parametrize("force_generic", [False, True])
def test_linearisation_and_step_match_the_transition_fd_restatement(target, force_generic):
    consts, an, _, _, _ = _model(target, force_generic)
    rng = np.random.default_rng(3)
    n = 12
    q, qd = _states(rng, n)
    u = rng.standard_normal((n, 6)) * [100, 100, 400, 1, 1, 1.0]
    qdd = host_harness.forward_dynamics(an, q, qd, u)
    ref = lo.forward_dynamics(consts, q, qd, u)
    assert np.abs(qdd - ref).max() < 1e-9 * np.abs(ref).max()
    _, qn, qdn = host_harness.forward_dynamics(an, q, qd, u, dt=0.002)
    y = lo.step(consts, q, qd, u, 0.002)
    assert np.abs(np.concatenate([qn, qdn], 1) - y).max() < 1e-11 * np.abs(y).max()
    A, B, qdd2 = host_harness.linearize(an, q, qd, u, dt=0.002, eps=1e-5, centered=True)
    Ar, Br = lo.transition_fd(consts, q, qd, u, dt=0.002, eps=1e-5, centered=True)
    assert np.abs(qdd2 - ref).max() < 1e-9 * np.abs(ref).max()
    assert np.abs(A - Ar).max() < 2e-8 and np.abs(B - Br).max() < 2e-8
    A, B, _ = host_harness.linearize(an, q, qd, u, dt=0.002, eps=1e-8, centered=True)   # the reference's StateSpaceConfig defaults
    Ar, Br = lo.transition_fd(consts, q, qd, u, dt=0.002, eps=1e-8, centered=True)
    assert np.abs(A - Ar).max() < 5e-6 and np.abs(B - Br).max() < 5e-6
    A, B, _ = host_harness.linearize(an, q, qd, u, dt=0.002, eps=1e-6, centered=False)
    Ar, Br = lo.transition_fd(consts, q, qd, u, dt=0.002, eps=1e-6, centered=False)
    assert np.abs(A - Ar).max() < 1e-4 and np.abs(B - Br).max() < 2e-7


@pytest.mark.parametrize("target", ["hammer", *model_classes.CLASSES])
@pytest.mark.parametrize("force_generic", [False, True])
def test_closed_loop_rollout_matches_the_literal_loop(target, force_generic):
    consts, an, pose_sen, G_s, key_qpos = _model(target, force_generic)
    phi = ro.inertia_to_phi(G_s)
    n_steps = 130
    plan = planner.QuinticPlan([0.2, 1.4, 0.6, np.pi, 0.0, 18.8495559215], key_qpos, 0.002, 1500)
    plan.n_steps = n_steps                       # the first 130 steps of the 1500-step base.yaml profile
    K = ro.lqr_gain(consts, key_qpos, np.zeros(6), [10, 10, 10, 1e4, 1e4, 1e4])
    q0 = np.stack([key_qpos, key_qpos + [0.01, -0.02, 0.015, 0.05, -0.04, 0.03]])
    qd0 = np.stack([np.zeros(6), [0.02, 0.01, -0.03, 0.1, -0.2, 0.05]])
    out = host_harness.closed_loop(an, plan, K, phi, q0, qd0)
    traj = planner.QuinticPlan([0.2, 1.4, 0.6, np.pi, 0.0, 18.8495559215], key_qpos, 0.002, 1500).trajectory()[:n_steps]
    for e in range(2):
        ref = ro.closed_loop_replay(consts, pose_sen, G_s, traj, K, q0[e], qd0[e])
        assert np.array_equal(out["frame_steps"], ref["step"])
        fr = out["frames"][..., e]
        for sl, key in ((slice(0, 18), "act"), (slice(18, 24), "twist_sen"), (slice(24, 30), "dtwist_sen"), (slice(30, 36), "wrench")):
            want = ref[key].reshape(len(ref["step"]), -1)
            assert np.abs(fr[:, sl] - want).max() < 1e-9 * np.abs(want).max(), (e, key)
        assert np.abs(out["final"][:6, e] - ref["q_final"]).max() < 1e-11 and np.abs(out["final"][6:12, e] - ref["qd_final"]).max() < 1e-11


@pytest.mark.parametrize("target", ["uniform_gearbox", *model_classes.CLASSES])
@pytest.mark.parametrize("force_generic", [False, True])
def test_fused_regressor_gram_matches_the_materialised_normal_equations(target, force_generic):
    from oracle import rnea_vec as rv

    c, an, pose_sen, G_s, _ = _model(target, force_generic)
    rng = np.random.default_rng(11)
    n = 300
    q, qd = _states(rng, n)
    qdd = rng.standard_normal((n, 6)) * [3, 3, 3, 10, 10, 10]
    out = rv.inverse_batched(np.stack([q, qd, qdd], axis=1), c["hposes_Rt"], c["simats"], c["uscrews"], c["twist_0"], c["dtwist_0"])
    Vs, dVs = rv.sensor_frame_twists_batched(pose_sen, out["twists"][:, -1], out["dtwists"][:, -1])
    Y = rv.regressor_batched(Vs, dVs)
    phi = ro.inertia_to_phi(G_s)
    f = Y @ phi + 0.01 * rng.standard_normal((n, 6))
    ref = rv.gram_pack(Y, f)
    got = host_harness.regressor_gram(an, q, qd, qdd, f)
    assert got[111] == n
    assert np.abs(got - ref).max() < 1e-10 * np.abs(ref).max()


def test_generic_linearisation_keeps_the_base_twist_in_the_velocity_columns():
    """ADVICE r1 (csrc/rbm_dynamics.cuh GenericEval::id_velocity): a model with twist_0 != 0 has V_0 x (S qd) coupling terms in
    d tau / d qd.  Host build of the same header, against the literal transition FD with the same moving base."""
    c = pm.load_packaged("sequential", "hammer")
    tw0 = np.array([0.3, -0.2, 0.1, 0.4, -0.5, 0.6])
    an = engine.analyze_model(c.hposes_Rt, c.simats, c.uscrews, tw0, c.dtwist_0, pose_sen_llj=c.pose_sen_Rt)
    assert an[0] == "generic"  # a moving base leaves the structure-specialised path
    consts = dict(_consts(c), twist_0=tw0)
    rng = np.random.default_rng(11)
    n = 8
    q, qd = _states(rng, n)
    u = rng.standard_normal((n, 6)) * [100, 100, 400, 1, 1, 1.0]
    for centered, eps, tol in ((True, 1e-5, 2e-8), (False, 1e-6, 1e-4)):
        A, B, _ = host_harness.linearize(an, q, qd, u, dt=0.002, eps=eps, centered=centered)
        Ar, Br = lo.transition_fd(consts, q, qd, u, dt=0.002, eps=eps, centered=centered)
        assert np.abs(A - Ar).max() < tol and np.abs(B - Br).max() < 2e-7
    A0, _ = lo.transition_fd(dict(consts, twist_0=np.zeros(6)), q, qd, u, dt=0.002, eps=1e-5, centered=True)
    Ar, _ = lo.transition_fd(consts, q, qd, u, dt=0.002, eps=1e-5, centered=True)
    assert np.abs(A0 - Ar).max() > 1e-5  # the coupling the old code dropped is far above the tolerance
