"""Pins the CPU oracles (oracle/rnea_oracle.py per-sample, oracle/rnea_vec.py vectorised,
oracle/model_oracle.py constants) against the golden vectors that were produced by executing the
reference's own files (oracle/gen_golden.py) and -- when the checkout is present -- against the
reference files directly."""
import os

import numpy as np
import pytest

from conftest import load_golden
from oracle import reference_loader as rl
from oracle import rnea_oracle as ro
from oracle import rnea_vec as rv

TARGETS = ["hammer", "uniform_gearbox", "kill_la_kill"]
GENERIC = ["nj6", "nj4", "nj9"]


def se3_from_Rt(Rt):
    return ro.SE3(ro.SO3(np.array(Rt[:9]).reshape(3, 3)), np.array(Rt[9:]))


def rel_err(a, b, floor=1e-300):
    """norm-wise relative error per sample: max|a-b| / max(max|b|, floor)."""
    a, b = np.asarray(a), np.asarray(b)
    ax = tuple(range(1, a.ndim))
    return np.max(np.abs(a - b), axis=ax) / np.maximum(np.max(np.abs(b), axis=ax), floor)


def golden_cases():
    return [f"ref_inverse_{t}.npz" for t in TARGETS] + [f"ref_inverse_generic_{g}.npz" for g in GENERIC]


@pytest.mark.parametrize("fname", golden_cases())
def test_per_sample_oracle_matches_reference_golden(fname):
    g = load_golden(fname)
    hposes = [se3_from_Rt(r) for r in g["hposes_Rt"]]
    kw = {}
    if "wrench_tip" in g.files:
        kw = dict(wrench_tip=g["wrench_tip"], pose_tip_ee=se3_from_Rt(g["pose_tip"]))
    n = min(48, len(g["traj"]))
    for s in range(n):
        tau, poses, tw, dtw = ro.inverse(g["traj"][s], hposes, g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"], **kw)
        # identical op order => agreement to round-off
        assert np.allclose(tau, g["tau"][s], rtol=1e-13, atol=1e-12)
        assert np.allclose(np.array(tw), g["twists"][s], rtol=1e-13, atol=1e-13)
        assert np.allclose(np.array(dtw), g["dtwists"][s], rtol=1e-13, atol=1e-12)
        for i in range(len(g["uscrews"])):
            assert np.allclose(poses[i].rot.as_matrix().reshape(9), g["poses"][s, i, :9], atol=1e-14)
            assert np.allclose(poses[i].trans, g["poses"][s, i, 9:], atol=1e-14)
        Vs, dVs = ro.sensor_frame_twists(se3_from_Rt(g["pose_sen_llj"]), tw[-1], dtw[-1])
        assert np.allclose(Vs, g["twist_sen"][s], atol=1e-13)
        assert np.allclose(dVs, g["dtwist_sen"][s], rtol=1e-13, atol=1e-12)
        assert np.allclose(ro.regressor(Vs, dVs), g["regressor"][s], rtol=1e-13, atol=1e-12)


@pytest.mark.parametrize("fname", golden_cases())
def test_vectorised_oracle_matches_reference_golden(fname):
    g = load_golden(fname)
    kw = {}
    if "wrench_tip" in g.files:
        kw = dict(wrench_tip=g["wrench_tip"], pose_tip_Rt=g["pose_tip"])
    out = rv.inverse_batched(g["traj"], g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"], **kw)
    assert rel_err(out["tau"], g["tau"], 1e-6).max() < 1e-12
    assert rel_err(out["twists"], g["twists"], 1e-6).max() < 1e-12
    assert rel_err(out["dtwists"], g["dtwists"], 1e-6).max() < 1e-12
    assert np.abs(out["poses"] - g["poses"]).max() < 1e-13
    nj = g["uscrews"].shape[0]
    Vs, dVs = rv.sensor_frame_twists_batched(g["pose_sen_llj"], out["twists"][:, nj], out["dtwists"][:, nj])
    assert rel_err(Vs, g["twist_sen"], 1e-6).max() < 1e-12
    assert rel_err(dVs, g["dtwist_sen"], 1e-6).max() < 1e-12
    Y = rv.regressor_batched(Vs, dVs)
    assert rel_err(Y, g["regressor"], 1e-6).max() < 1e-12


def test_setup_functions_match_reference_golden():
    g = load_golden("ref_setup_functions.npz")
    poses = [se3_from_Rt(r) for r in g["poses_Rt"]]
    assert np.array_equal(ro.spatial_inertia_stack(g["mass"], g["diag"]), g["simats_diag"])
    assert np.allclose(ro.transfer_simat(poses, g["simats_diag"]), g["transferred"], rtol=1e-14, atol=1e-14)
    assert np.allclose(ro.transfer_simat(poses[3], g["simats_diag"][3]), g["transferred_single"], rtol=1e-14, atol=1e-14)
    assert np.allclose(ro.transfer_simat(poses, g["dense"]), g["transferred_dense"], rtol=1e-13, atol=1e-13)
    for k, p in enumerate(poses):
        assert np.allclose(ro.parallel_axis_imat(p, g["imats"][k], g["mass"][k]), g["ct_imat"][k], rtol=1e-13, atol=1e-13)
        assert np.allclose(ro.transfer_simat_adjoint_form(p, g["dense"][k]), g["ct_simat"][k], rtol=1e-13, atol=1e-13)
        assert np.allclose(ro.linvel_of_point(g["twists"][k], p), g["linvel"][k], atol=1e-14)
        assert np.allclose(ro.linvel_of_point(g["twists"][k], p, True), g["linvel_h"][k], atol=1e-14)
        assert np.allclose(ro.linacc_of_point(g["twists"][k], g["dtwists"][k], p), g["linacc"][k], atol=1e-13)
        assert np.allclose(ro.linacc_of_point(g["twists"][k], g["dtwists"][k], p, True), g["linacc_h"][k], atol=1e-13)
        assert np.allclose(ro.regressor(g["twists"][k], g["dtwists"][k]), g["regressor"][k], atol=1e-13)

    def Rt(p):
        return np.concatenate([np.asarray(p.rot.as_matrix()).reshape(9), p.trans])

    assert np.allclose([Rt(p) for p in ro.compose(g["trans"], g["quats"])], g["comp_q"], atol=1e-15)
    assert np.allclose([Rt(p) for p in ro.compose(g["trans"], g["poses_Rt"][:, :9].copy())], g["comp_m"], atol=1e-15)
    assert np.allclose([Rt(p) for p in ro.compose(g["trans"])], g["comp_none"], atol=1e-15)
    assert np.allclose(Rt(ro.compose(g["trans"][0], g["quats"][0])), g["comp_single"], atol=1e-15)
    assert np.array_equal(ro.homogenize(g["trans"][0]), g["hom"])
    assert np.array_equal(ro.homogenize(g["trans"][1], 0), g["hom0"])
    # the reference's scratch check (test_adjoint_inv_transpose.py) as executed by gen_golden
    assert not bool(g["adj_T_close_inv"]) and bool(g["adj_inv_close_pinv"])


def test_static_gravity_known_answer():
    # SURVEY.md 8(a): at the keyframe, at rest, tau = [0, 0, (32 + m_obj) g, 0, 0, 0] up to the object's CoM torque
    for t in TARGETS:
        g = load_golden(f"ref_inverse_{t}.npz")
        assert np.array_equal(g["traj"][1, 0], g["key_qpos"]) and not g["traj"][1, 1:].any()
        tau = g["tau"][1]
        assert abs(tau[2] - (32.0 + float(g["gt_mass"])) * 9.81) < 1e-9
        assert abs(tau[0]) < 1e-9 and abs(tau[1]) < 1e-9


def test_regressor_reproduces_body_wrench():
    # Y(V, dV) phi == G dV - ad(V)^T G V for a rigid body with parameters phi (SURVEY.md 8(a) a11)
    rng = np.random.default_rng(0)
    m, c = 1.7, np.array([0.1, -0.2, 0.3])
    A = rng.standard_normal((3, 3))
    Ic = A @ A.T + np.eye(3)
    I0 = Ic + m * (c @ c * np.eye(3) - np.outer(c, c))
    cx = rv.skew(c)
    G = np.block([[m * np.eye(3), -m * cx], [m * cx, I0]])
    phi = np.array([m, *(m * c), I0[0, 0], I0[1, 1], I0[2, 2], I0[0, 1], I0[1, 2], I0[2, 0]])
    for _ in range(5):
        V, dV = rng.standard_normal(6), rng.standard_normal(6)
        lhs = ro.regressor(V, dV) @ phi
        rhs = G @ dV - ro.SE3.curlywedge(V).T @ G @ V
        assert np.allclose(lhs, rhs, atol=1e-12)


def test_tau_is_affine_in_qdd():
    g = load_golden("ref_inverse_hammer.npz")
    tr = g["traj"][10:14].copy()
    args = (g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"])
    t0 = rv.inverse_batched(tr, *args)["tau"]
    tr2 = tr.copy()
    tr2[:, 2] *= 2.0
    tr3 = tr.copy()
    tr3[:, 2] *= 3.0
    t2 = rv.inverse_batched(tr2, *args)["tau"]
    t3 = rv.inverse_batched(tr3, *args)["tau"]
    assert np.allclose(t3 - t2, t2 - t0, atol=1e-10)


def test_oracle_matches_reference_files_live():
    """Every stored sample of the reference's own dynamics.inverse (oracle/gen_golden.py) against the per-sample oracle, at the
    tolerances of a side-by-side run of the two."""
    for t in TARGETS:
        g = load_golden(f"ref_inverse_{t}.npz")
        hp = [se3_from_Rt(r) for r in g["hposes_Rt"]]
        pose_sen = se3_from_Rt(g["pose_sen_llj"])
        for s, traj in enumerate(g["traj"]):
            tau, _, tw, dtw = ro.inverse(traj, hp, g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"])
            assert np.allclose(tau, g["tau"][s], rtol=1e-14, atol=1e-13)
            assert np.allclose(np.array(tw), g["twists"][s], atol=1e-14)
            assert np.allclose(np.array(dtw), g["dtwists"][s], rtol=1e-14, atol=1e-13)
            assert np.allclose(ro.regressor(*ro.sensor_frame_twists(pose_sen, tw[-1], dtw[-1])), g["regressor"][s], atol=1e-13)


@pytest.mark.reference
@pytest.mark.skipif(not rl.available(), reason="reference checkout absent (GPU box)")
def test_golden_model_constants_are_reproducible():
    from oracle import model_oracle as mo

    xml = os.path.join(rl.REFERENCE_ROOT, "xml_models")
    for t in TARGETS:
        c = mo.build_constants(os.path.join(xml, "manipulators", "sequential.xml"), os.path.join(xml, "targets", t, "object_cad_gt.csv"))
        g = load_golden(f"ref_inverse_{t}.npz")
        assert np.array_equal(c.hposes_Rt(), g["hposes_Rt"])
        assert np.array_equal(c.simats, g["simats"])
        assert np.array_equal(c.uscrews, g["uscrews"])
