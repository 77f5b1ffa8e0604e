"""`not gpu`: the kernels' per-sample arithmetic, instantiated for the host from the same __host__ __device__ headers the CUDA
kernels are built from (tests/host_harness), against the golden vectors produced by the reference's own files -- plus the
device-free model analysis (rbm_model_analyze: which kernel path a model selects, and with which constants).
Launch / memory / TMA behaviour is covered by the -m gpu suite through the real C ABI."""
import numpy as np
import pytest

import model_classes
from conftest import load_golden
from rigid_body_manipulation_b200 import engine

host_harness = pytest.importorskip("host_harness")
if host_harness.nvcc_path() is None:  # pragma: no cover
    pytest.skip("nvcc is needed to build the host harness", allow_module_level=True)

TARGETS = ["hammer", "uniform_gearbox", "kill_la_kill"]
GENERIC = ["nj6", "nj4", "nj9"]


def rel_err(a, b, floor=1e-6):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    ax = tuple(range(1, a.ndim))
    return np.max(np.abs(a - b), axis=ax) / np.maximum(np.max(np.abs(b), axis=ax), floor)


def analyze(g, **kw):
    extra = dict(wrench_tip=g["wrench_tip"], pose_tip_ee=g["pose_tip"]) if "wrench_tip" in g.files else {}
    return engine.analyze_model(g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"], pose_sen_llj=g["pose_sen_llj"], **extra, **kw)


@pytest.mark.parametrize("t", TARGETS)
def test_model_analysis_selects_the_specialised_path_for_the_reference_robot(t):
    g = load_golden(f"ref_inverse_{t}.npz")
    path, fast, generic = analyze(g)
    assert path == "seq_iso"
    # FastParams layout (csrc/rbm_model.cuh): g[3] | mass[6] | h[6][3] | I[6][6] | tm[6][3] | senR[9] | sent[3] | sen_diag
    assert np.array_equal(fast[:3], g["dtwist_0"][:3])
    assert np.allclose(fast[3:8], 8.0) and abs(fast[8] - (8.0 + float(g["gt_mass"]))) < 1e-12
    h6 = fast[9 + 15 : 9 + 18]
    assert np.allclose(h6, float(g["gt_mass"]) * g["gt_com"], atol=1e-12)  # first moment of link 6 = the object's (link CoM is at the origin)
    assert np.allclose(fast[27:27 + 30].reshape(5, 6)[:, :3], 0.05333333) and not fast[27:27 + 30].reshape(5, 6)[:, 3:].any()
    assert fast[-1] == 1.0 and np.array_equal(fast[-13:-4].reshape(3, 3), np.diag([-1.0, -1.0, 1.0]))  # Rz(180 deg) sensor site, snapped
    assert analyze(g, force_generic=True)[0] == "generic"
    assert len(generic) == 42 + 83 * 6 and np.array_equal(generic[6:12], g["dtwist_0"])  # GP_HEAD + GJ_STRIDE * nj (csrc/rbm_model.cuh)


def test_model_analysis_fallbacks():
    g = load_golden("ref_inverse_hammer.npz")
    for name in GENERIC:
        assert analyze(load_golden(f"ref_inverse_generic_{name}.npz"))[0] == "generic"
    sim = g["simats"].copy()
    sim[2, 3, 3] *= 1.5  # anisotropic link 2: still a rigid body -> SEQ_RIGID
    assert engine.analyze_model(g["hposes_Rt"], sim, g["uscrews"], g["twist_0"], g["dtwist_0"])[0] == "seq_rigid"
    sim[2, 0, 4] += 0.3  # breaks the rigid-body form (asymmetric coupling) -> generic
    assert engine.analyze_model(g["hposes_Rt"], sim, g["uscrews"], g["twist_0"], g["dtwist_0"])[0] == "generic"
    tw0 = g["twist_0"].copy()
    tw0[3] = 0.1  # moving base
    assert engine.analyze_model(g["hposes_Rt"], g["simats"], g["uscrews"], tw0, g["dtwist_0"])[0] == "generic"
    us = g["uscrews"].copy()
    us[3] = [0, 0, 0, 0, 1, 0]  # wrist joint about y
    assert engine.analyze_model(g["hposes_Rt"], g["simats"], us, g["twist_0"], g["dtwist_0"])[0] == "generic"
    with pytest.raises(ValueError):
        engine.analyze_model(g["hposes_Rt"][:-1], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"])


def _classes_reference(name):
    """A tests/model_classes.py class in the form of a golden: sampled states and the vectorised oracle's answers."""
    from oracle import rnea_vec as rv

    mc = model_classes.build(name)
    rng = np.random.default_rng(13)
    n = 500
    traj = model_classes.sample_states(rng, n)
    out = rv.inverse_batched(traj, mc.hposes_Rt, mc.simats, mc.uscrews, mc.twist_0, mc.dtwist_0)
    return dict(traj=traj, tau=out["tau"], twists=out["twists"], dtwists=out["dtwists"]), model_classes.analyze(mc)


@pytest.mark.parametrize("t", TARGETS + list(model_classes.CLASSES))
def test_fast_recursion_matches_reference_golden(t):
    if t in model_classes.CLASSES:
        g, (path, fast, _) = _classes_reference(t)
    else:
        g = load_golden(f"ref_inverse_{t}.npz")
        path, fast, _ = analyze(g)
    tau, V, dV = host_harness.fast_rnea(path, fast, g["traj"])
    assert rel_err(tau, g["tau"]).max() < 1e-12
    assert rel_err(V, g["twists"][:, 6]).max() < 1e-12 and rel_err(dV, g["dtwists"][:, 6]).max() < 1e-12
    tau32, V32, dV32 = host_harness.fast_rnea(path, fast, g["traj"], dtype=np.float32)
    assert rel_err(tau32, g["tau"]).max() < 1e-4
    assert rel_err(V32, g["twists"][:, 6]).max() < 1e-4 and rel_err(dV32, g["dtwists"][:, 6]).max() < 1e-4
    # the all-rigid descriptor evaluates the same model
    tau_r, _, _ = host_harness.fast_rnea("seq_rigid", fast, g["traj"])
    assert rel_err(tau_r, g["tau"]).max() < 1e-12


def test_reduced_evaluations_decompose_the_inverse_dynamics():
    """tau(q, qd, qdd) = M(q) qdd + C(q, qd) + g(q): the inertia-only and velocity-only instantiations used by the linearisation
    kernel add up to the full evaluation."""
    g = load_golden("ref_inverse_kill_la_kill.npz")
    path, fast, _ = analyze(g)
    traj = g["traj"]
    full, _, _ = host_harness.fast_rnea(path, fast, traj, mode=0)
    inertia, _, _ = host_harness.fast_rnea(path, fast, traj, mode=1)
    velocity, _, _ = host_harness.fast_rnea(path, fast, traj, mode=2)
    rest = traj.copy()
    rest[:, 1:] = 0.0
    gravity, _, _ = host_harness.fast_rnea(path, fast, rest, mode=0)
    assert rel_err(inertia + velocity + gravity, full).max() < 1e-12
    # the inertia-only part is linear in qdd, the velocity part quadratic in qd
    t2 = traj.copy()
    t2[:, 2] *= 2.0
    t2[:, 1] *= 3.0
    assert rel_err(host_harness.fast_rnea(path, fast, t2, mode=1)[0], 2.0 * inertia).max() < 1e-12
    assert rel_err(host_harness.fast_rnea(path, fast, t2, mode=2)[0], 9.0 * velocity, 1e-3).max() < 1e-11


@pytest.mark.parametrize("fname", [f"ref_inverse_{t}.npz" for t in TARGETS] + [f"ref_inverse_generic_{n}.npz" for n in GENERIC])
def test_generic_recursion_matches_reference_golden(fname):
    g = load_golden(fname)
    _, _, gp = analyze(g, force_generic=True)
    nj = g["uscrews"].shape[0]
    out = host_harness.generic_rnea(gp, nj, g["traj"], full=True)
    assert rel_err(out["tau"], g["tau"]).max() < 1e-12
    assert np.abs(out["poses"] - g["poses"]).max() < 1e-13
    assert rel_err(out["twists"], g["twists"]).max() < 1e-12 and rel_err(out["dtwists"], g["dtwists"]).max() < 1e-12
    assert rel_err(out["V"], g["twists"][:, nj]).max() < 1e-12
    if nj == 6:
        assert np.array_equal(host_harness.generic_rnea(gp, nj, g["traj"], unrolled=True)["tau"], out["tau"])
    assert rel_err(host_harness.generic_rnea_f32(gp, nj, g["traj"]), g["tau"]).max() < 1e-4
    Vs, dVs, Y = host_harness.sensor_regressor(g["pose_sen_llj"], out["V"], out["dV"])
    assert rel_err(Vs, g["twist_sen"]).max() < 1e-12 and rel_err(dVs, g["dtwist_sen"]).max() < 1e-12
    assert rel_err(Y, g["regressor"]).max() < 1e-12


def test_folded_joint_transform_with_non_unit_screws_and_tiny_angles():
    """The generic kernel folds SE3.exp(-S q) . M at model creation into R = c RA + s RB + RC, p = c PA + s PB + q PC + PD
    (csrc/rbm_model.cuh) and has no small-angle branch.  Screws the goldens do not contain -- rotation parts of norm 0.7, 1.9 and 1e-3
    (nearly prismatic), a rescaled pitch -- and states on both sides of liegroups' isclose(angle, 0) switch (|q| = 1e-9, 2e-8) and far
    outside the trigonometric fast range (q = 50) must still agree with the vectorised restatement of the reference
    (dynamics.py:109-157 on liegroups' exp / left Jacobian)."""
    from oracle import rnea_vec as rv

    g = load_golden("ref_inverse_generic_nj6.npz")
    us = g["uscrews"].copy()
    us[0, 3:] *= 0.7
    us[2, 3:] *= 1.9
    us[2, :3] *= 0.4
    us[3, 3:] *= 1e-3
    traj = g["traj"].copy()
    traj[2, 0, :] = 1e-9
    traj[3, 0, :] = -2e-8
    traj[4, 0, :] = 50.0
    _, _, gp = engine.analyze_model(g["hposes_Rt"], g["simats"], us, g["twist_0"], g["dtwist_0"], wrench_tip=g["wrench_tip"], pose_tip_ee=g["pose_tip"],
                                    force_generic=True)
    out = host_harness.generic_rnea(gp, 6, traj, full=True)
    ref = rv.inverse_batched(traj, g["hposes_Rt"], g["simats"], us, g["twist_0"], g["dtwist_0"], wrench_tip=g["wrench_tip"], pose_tip_Rt=g["pose_tip"])
    assert rel_err(out["tau"], ref["tau"]).max() < 1e-12
    assert np.abs(out["poses"] - ref["poses"]).max() < 1e-12
    assert rel_err(out["twists"], ref["twists"]).max() < 1e-12 and rel_err(out["dtwists"], ref["dtwists"]).max() < 1e-12
