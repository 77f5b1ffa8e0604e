"""Payload identification from joint torques: tau = tau0 + Phi phi with phi the payload's 10 parameters in the sensor frame
(csrc/rbm_payload.cuh, k_payload_regressor / k_payload_gram, Model.payload_regressor / payload_gram).

The reference for Phi uses the oracle alone: RNEA is linear in the link inertias, so column k of Phi is
tau(simats_6 + G_6(e_k)) - tau(simats_6), where G_6(phi) is the sensor-frame spatial inertia of phi moved to the last link's frame.
The -m "not gpu" part checks the per-sample arithmetic on the host harness (tests/host_harness/payload.cu); the -m gpu part checks the
kernels, the Gram pack and the identification it feeds."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import model_classes as mcs
from conftest import load_golden
from oracle import replay_oracle as ro
from oracle import rnea_vec as rv
from rigid_body_manipulation_b200 import engine
from rigid_body_manipulation_b200 import model as pm

FAST_GOLDENS = ["ref_inverse_hammer.npz", "ref_inverse_uniform_gearbox.npz", "ref_inverse_kill_la_kill.npz"]
GENERIC_GOLDENS = ["ref_inverse_generic_nj4.npz", "ref_inverse_generic_nj6.npz", "ref_inverse_generic_nj9.npz"]
SCALE = np.array([1, 1e-2, 1e-2, 1e-2, 1e-3, 1e-3, 1e-3, 1e-3, 1e-3, 1e-3])


# ---- oracle-only reference -------------------------------------------------------------------------------------------------------
def phi_to_inertia(phi):
    """Inverse of replay_oracle.inertia_to_phi: [[m 1, -[h]x], [[h]x, Ibar]]."""
    m, h, I = phi[0], phi[1:4], phi[4:]
    H = rv.skew(np.asarray(h, float))
    Ib = np.array([[I[0], I[3], I[5]], [I[3], I[1], I[4]], [I[5], I[4], I[2]]])
    return np.block([[m * np.eye(3), -H], [H, Ib]])


def sensor_to_link(pose_sen_Rt, G_s):
    """Spatial inertia given in the sensor frame, expressed in the last link's frame: Ad(T_sen)^T G_s Ad(T_sen)."""
    p = np.asarray(pose_sen_Rt, float)
    Ad = rv.adjoint(p[:9].reshape(3, 3)[None], p[9:][None])[0]
    return Ad.T @ G_s @ Ad


def oracle_payload(consts, pose_sen_Rt, traj, **kw):
    """-> Phi (n, nj, 10), tau0 (n, nj)."""
    args = lambda sim: (traj, consts["hposes_Rt"], sim, consts["uscrews"], consts["twist_0"], consts["dtwist_0"])
    tau0 = rv.inverse_batched(*args(consts["simats"]), **kw)["tau"]
    cols = []
    for k in range(10):
        sim = np.array(consts["simats"], float, copy=True)
        sim[-1] += sensor_to_link(pose_sen_Rt, phi_to_inertia(np.eye(10)[k]))
        cols.append(rv.inverse_batched(*args(sim), **kw)["tau"] - tau0)
    return np.stack(cols, axis=-1), tau0


def golden_consts(g):
    consts = dict(hposes_Rt=g["hposes_Rt"], simats=g["simats"], uscrews=g["uscrews"], twist_0=g["twist_0"], dtwist_0=g["dtwist_0"])
    kw = dict(wrench_tip=g["wrench_tip"], pose_tip_Rt=g["pose_tip"]) if "wrench_tip" in g.files else {}
    return consts, kw


def analyze_golden(g, force_generic=False):
    consts, kw = golden_consts(g)
    extra = dict(wrench_tip=kw["wrench_tip"], pose_tip_ee=kw["pose_tip_Rt"]) if kw else {}
    return engine.analyze_model(consts["hposes_Rt"], consts["simats"], consts["uscrews"], consts["twist_0"], consts["dtwist_0"],
                                pose_sen_llj=g["pose_sen_llj"], force_generic=force_generic, **extra)


def object_free():
    return pm.load_packaged("sequential", None)


def object_phi(c):
    """The packaged object's parameters in the sensor frame: the inertia the model folded into link 6, seen from the sensor."""
    return ro.inertia_to_phi(ro.sensor_inertia(c.simat_object_llj, c.pose_sen_Rt))


def states(nj, n, seed):
    rng = np.random.default_rng(seed)
    if nj == 6:
        return mcs.sample_states(rng, n)
    return np.stack([rng.uniform(-3, 3, (n, nj)), rng.standard_normal((n, nj)), rng.standard_normal((n, nj)) * 3], 1)


def tau_err(got, ref, tau_scale):
    return np.abs(np.asarray(got, np.float64) - ref).max() / tau_scale


# ---- host harness ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    """tests/host_harness/payload.cu built for the host: payload(analysis, traj, dtype) -> (Phi (n, nj, 10), tau0 (n, nj)) and
    gram(analysis, traj, tau (n, nj)) -> pack."""
    hh = pytest.importorskip("host_harness")
    if hh.nvcc_path() is None:  # pragma: no cover
        pytest.skip("nvcc is needed to build the host harness")
    lib = str(tmp_path_factory.mktemp("payload") / "libpayload.so")
    subprocess.run([hh.nvcc_path(), "-O2", "-std=c++17", "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets", "-gencode",
                    "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC", "-I", hh.CSRC, "-I", os.path.join(hh.ROOT, "include"),
                    "-o", lib, os.path.join(hh.HERE, "payload.cu")], check=True)
    dll = C.CDLL(lib)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)

    def args(analysis, traj, dtype):
        path, fast, generic = analysis
        nj = traj.shape[2]
        soa = [np.ascontiguousarray(traj[:, k, :].T, dtype=dtype) for k in range(3)]
        return [C.c_int(hh.PATH_ID[path]), ptr(np.ascontiguousarray(fast, np.float64)), ptr(np.ascontiguousarray(generic, np.float64)), C.c_int(nj)], soa

    def payload(analysis, traj, dtype=np.float64):
        n, _, nj = traj.shape
        head, soa = args(analysis, traj, dtype)
        Phi, tau0 = np.empty((n, nj, 10), dtype), np.empty((nj, n), dtype)
        fn = dll.h_payload_f64 if dtype == np.float64 else dll.h_payload_f32
        assert fn(*head, *[ptr(a) for a in soa], ptr(Phi), ptr(tau0), C.c_int64(n)) == 0
        return Phi, tau0.T

    def gram(analysis, traj, tau):
        n = traj.shape[0]
        head, soa = args(analysis, traj, np.float64)
        pack = np.empty(112)
        assert dll.h_payload_gram_f64(*head, *[ptr(a) for a in soa], ptr(np.ascontiguousarray(tau.T, np.float64)), ptr(pack), C.c_int64(n)) == 0
        return pack

    return dict(payload=payload, gram=gram)


def _case(name, force_generic=False):
    """(constants, sensor pose, oracle keyword arguments, analysis) of a golden file or a model class of tests/model_classes.py."""
    if name.endswith(".npz"):
        g = load_golden(name)
        consts, kw = golden_consts(g)
        return consts, g["pose_sen_llj"], kw, analyze_golden(g, force_generic)
    mc = mcs.build(name)
    return mc.consts, mc.pose_sen_Rt, {}, mcs.analyze(mc, force_generic=force_generic)


@pytest.mark.parametrize("name", FAST_GOLDENS + GENERIC_GOLDENS + list(mcs.CLASSES))
@pytest.mark.parametrize("force_generic", [False, True])
def test_host_payload_rows_match_the_oracle(name, force_generic, harness):
    consts, pose_sen, kw, an = _case(name, force_generic)
    if name in GENERIC_GOLDENS and not force_generic:
        assert an[0] == "generic"
    traj = states(consts["uscrews"].shape[0], 300, 11)
    ref_phi, ref_tau0 = oracle_payload(consts, pose_sen, traj, **kw)
    scale = np.abs(ref_tau0).max()
    Phi, tau0 = harness["payload"](an, traj)
    assert tau_err(tau0, ref_tau0, scale) < 1e-9
    assert tau_err(Phi, ref_phi, scale) < 1e-9
    if an[0] != "generic":
        # the gantry rows see the payload's force only: structurally zero in the kernels, numerically zero in the oracle
        assert np.all(Phi[:, :3, 4:] == 0.0) and np.abs(ref_phi[:, :3, 4:]).max() < 1e-12 * scale
        Phi32, tau32 = harness["payload"](an, traj, np.float32)
        assert tau_err(tau32, ref_tau0, scale) < 1e-4 and tau_err(Phi32, ref_phi, scale) < 1e-4


def test_host_generic_path_matches_the_fast_path(harness):
    c = object_free()
    args = (c.hposes_Rt, c.simats, c.uscrews, c.twist_0, c.dtwist_0)
    fast = engine.analyze_model(*args, pose_sen_llj=c.pose_sen_Rt)
    gen = engine.analyze_model(*args, pose_sen_llj=c.pose_sen_Rt, force_generic=True)
    traj = states(6, 500, 12)
    Pf, tf = harness["payload"](fast, traj)
    Pg, tg = harness["payload"](gen, traj)
    scale = np.abs(tf).max()
    assert tau_err(Pg, Pf, scale) < 1e-11 and tau_err(tg, tf, scale) < 1e-11


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_host_fast_path_ignores_the_gantry_positions_and_velocities(dtype, harness):
    c = object_free()
    args = (c.hposes_Rt, c.simats, c.uscrews, c.twist_0, c.dtwist_0)
    traj = states(6, 300, 15)
    nan = traj.copy()
    nan[:, :2, :3] = np.nan
    for fg in (False, True):
        an = engine.analyze_model(*args, pose_sen_llj=c.pose_sen_Rt, force_generic=fg)
        Pa, ta = harness["payload"](an, traj, dtype)
        Pb, tb = harness["payload"](an, nan, dtype)
        if not fg:
            assert np.array_equal(Pa, Pb) and np.array_equal(ta, tb)
        else:  # the generic recursion reads every input
            assert np.isnan(Pb).any() and np.isnan(tb).any()


def test_object_free_packaged_model_selects_the_fast_path():
    c = object_free()
    path, fast, _ = engine.analyze_model(c.hposes_Rt, c.simats, c.uscrews, c.twist_0, c.dtwist_0, pose_sen_llj=c.pose_sen_Rt)
    assert path == "seq_iso" and fast[-1] == 1  # the reference's Rz(180 deg) sensor site: the diagonal adjoint


def test_host_torques_with_the_object_for_every_packaged_target(harness):
    """tau of the model WITH the object = tau0 + Phi phi_true of the object-free model, for all 23 packaged targets."""
    c0 = object_free()
    an = engine.analyze_model(c0.hposes_Rt, c0.simats, c0.uscrews, c0.twist_0, c0.dtwist_0, pose_sen_llj=c0.pose_sen_Rt)
    traj = states(6, 400, 13)
    Phi, tau0 = harness["payload"](an, traj)
    names = sorted(pm.packaged_targets())
    assert len(names) == 23
    for name in names:
        c = pm.load_packaged("sequential", name)
        assert np.array_equal(c.pose_sen_Rt, c0.pose_sen_Rt)
        tau = rv.inverse_batched(traj, c.hposes_Rt, c.simats, c.uscrews, c.twist_0, c.dtwist_0)["tau"]
        assert tau_err(tau0 + Phi @ object_phi(c), tau, np.abs(tau).max()) < 1e-9, name


@pytest.mark.parametrize("name", ["ref_inverse_hammer.npz", "offset_sensor", "ref_inverse_generic_nj9.npz"])
def test_host_gram_pack_is_the_normal_equations(name, harness):
    consts, pose_sen, kw, an = _case(name)
    nj = consts["uscrews"].shape[0]
    traj = states(nj, 700, 14)
    Phi, tau0 = harness["payload"](an, traj)
    tau = tau0 + np.random.default_rng(1).standard_normal(tau0.shape)
    pack = harness["gram"](an, traj, tau)
    A, r = Phi.reshape(-1, 10), (tau - tau0).reshape(-1)
    ref = np.concatenate([(A.T @ A).reshape(100), A.T @ r, [r @ r], [len(traj)]])
    assert np.abs(pack - ref).max() < 1e-12 * np.abs(ref).max()
    assert np.array_equal(pack[:100].reshape(10, 10), pack[:100].reshape(10, 10).T)


# ---- device kernels ---------------------------------------------------------------------------------------------------------------
TOLS = {"f64": 1e-9, "f32": 1e-4}


def _torch():
    import torch

    return torch


def _model(name, force_generic=False):
    from rigid_body_manipulation_b200.engine import Model

    if name == "object_free":
        c = object_free()
        return Model(c.hposes_Rt, c.simats, c.uscrews, c.twist_0, c.dtwist_0, pose_sen_llj=c.pose_sen_Rt, force_generic=force_generic)
    if name.endswith(".npz"):
        from gpu_util import model_from_golden

        return model_from_golden(load_golden(name), force_generic=force_generic)
    args, kw = mcs.build(name).model_args()
    return Model(*args, **kw, force_generic=force_generic)


def _soa(traj, dtype):
    torch = _torch()
    t = torch.as_tensor(np.ascontiguousarray(traj), dtype=dtype, device="cuda")
    return tuple(t[:, k, :].t().contiguous() for k in range(3))


@pytest.mark.gpu
@pytest.mark.parametrize("name,force_generic", [(f, False) for f in FAST_GOLDENS[:1] + GENERIC_GOLDENS] + [(c, False) for c in mcs.CLASSES] +
                         [("ref_inverse_hammer.npz", True), ("offset_sensor", True)])
@pytest.mark.parametrize("dt", ["f64", "f32"])
def test_device_payload_rows_match_the_oracle(name, force_generic, dt):
    torch = _torch()
    consts, pose_sen, kw, _ = _case(name)
    m = _model(name, force_generic)
    nj = m.nj
    traj = states(nj, 1000, 21)
    ref_phi, ref_tau0 = oracle_payload(consts, pose_sen, traj, **kw)
    scale = np.abs(ref_tau0).max()
    q, qd, qdd = _soa(traj, torch.float64 if dt == "f64" else torch.float32)
    out = m.payload_regressor(q, qd, qdd, want_rows=True, want_tau0=True)
    assert out["Phi"].shape == (1000, nj, 10) and out["tau0"].shape == (nj, 1000)
    assert tau_err(out["Phi"].cpu().numpy(), ref_phi, scale) < TOLS[dt]
    assert tau_err(out["tau0"].t().cpu().numpy(), ref_tau0, scale) < TOLS[dt]
    only = m.payload_regressor(q, qd, qdd, want_rows=False, want_tau0=True)
    assert only["Phi"] is None and torch.equal(only["tau0"], out["tau0"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["object_free", "rigid", "offset_sensor", "rigid_offset_sensor"])
@pytest.mark.parametrize("dt", ["f64", "f32"])
def test_device_tau0_is_model_rnea_bit_for_bit(name, dt):
    torch = _torch()
    m = _model(name)
    assert m.kernel_path != "generic"
    q, qd, qdd = _soa(states(6, 4096 + 77, 22), torch.float64 if dt == "f64" else torch.float32)
    assert torch.equal(m.payload_regressor(q, qd, qdd, want_rows=False, want_tau0=True)["tau0"], m.rnea(q, qd, qdd))


def _gram_ws(m, n):
    torch = _torch()
    return torch.empty(max(1, int(m._lib.rbm_gram_workspace_bytes(m._h, n)) // 8), dtype=torch.float64, device="cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("dt", ["f64", "f32"])
def test_fast_path_never_reads_the_gantry_positions_and_velocities(dt):
    torch = _torch()
    tdt = torch.float64 if dt == "f64" else torch.float32
    for fg in (False, True):
        m = _model("object_free", force_generic=fg)
        n = 5000
        q, qd, qdd = _soa(states(6, n, 23), tdt)
        tau = torch.randn((6, n), dtype=tdt, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
        q_nan, qd_nan = q.clone(), qd.clone()
        q_nan[:3] = float("nan")
        qd_nan[:3] = float("nan")
        a = m.payload_regressor(q, qd, qdd, want_tau0=True)
        b = m.payload_regressor(q_nan, qd_nan, qdd, want_tau0=True)
        pa, pb = m.payload_gram(q, qd, qdd, tau).clone(), m.payload_gram(q_nan, qd_nan, qdd, tau).clone()
        if not fg:
            assert torch.equal(a["Phi"], b["Phi"]) and torch.equal(a["tau0"], b["tau0"]) and torch.equal(pa, pb)
        else:  # the generic path reads every row
            assert torch.isnan(b["Phi"]).any() and torch.isnan(b["tau0"]).any() and torch.isnan(pb).any()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["object_free", "offset_sensor", "rigid", "ref_inverse_generic_nj9.npz"])
@pytest.mark.parametrize("n", [0, 1, 255, 256, 257, 100_000, 1 << 21])
@pytest.mark.parametrize("dt", ["f64", "f32"])
def test_gram_matches_materialised_normal_equations(name, n, dt):
    torch = _torch()
    if name.endswith(".npz") and n == 1 << 21:
        pytest.skip("the 2^21 size is covered by the fast-path models")
    tdt = torch.float64 if dt == "f64" else torch.float32
    m = _model(name)
    nj = m.nj
    q, qd, qdd = _soa(states(nj, n, n + 5), tdt)
    gen = torch.Generator(device="cuda").manual_seed(n)
    tau = torch.randn((nj, n), dtype=tdt, device="cuda", generator=gen) * 5
    pack = m.payload_gram(q, qd, qdd, tau).cpu().numpy()
    assert pack[111] == n
    if n == 0:
        assert not pack.any()
        return
    # the materialised reference in fp64 from the fp64 kernel's rows (the rows themselves are checked against the oracle above)
    q64, qd64, qdd64 = (t.double() for t in (q, qd, qdd))
    out = m.payload_regressor(q64, qd64, qdd64, want_tau0=True)
    A = out["Phi"].reshape(-1, 10)
    r = (tau.double() - out["tau0"]).t().reshape(-1)
    ref = torch.cat([(A.t() @ A).reshape(100), A.t() @ r, (r @ r).reshape(1)]).cpu().numpy()
    scale = np.abs(ref[:100]).max()
    tol = TOLS[dt]
    assert np.abs(pack[:100] - ref[:100]).max() < tol * scale
    assert np.abs(pack[100:110] - ref[100:110]).max() < tol * max(np.abs(ref[100:110]).max(), np.sqrt(scale * ref[110]))
    assert abs(pack[110] - ref[110]) < tol * ref[110]
    G = pack[:100].reshape(10, 10)
    assert np.array_equal(G, G.T)
    assert np.array_equal(pack, m.payload_gram(q, qd, qdd, tau).cpu().numpy())  # fixed reduction order, no atomics


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,tol", [("f64", 1e-12), ("f32", 2e-6)])
def test_gram_is_additive_at_the_configs2_size(dtype, tol):
    torch = _torch()
    tdt = torch.float64 if dtype == "f64" else torch.float32
    m = _model("object_free")
    n = 12_500_000
    gen = torch.Generator(device="cuda").manual_seed(8)
    q = (torch.rand((6, n), generator=gen, device="cuda", dtype=tdt) * 2 - 1) * 6
    qd = torch.randn((6, n), generator=gen, device="cuda", dtype=tdt)
    qdd = torch.randn((6, n), generator=gen, device="cuda", dtype=tdt) * 3
    tau = torch.randn((6, n), generator=gen, device="cuda", dtype=tdt) * 20
    whole = m.payload_gram(q, qd, qdd, tau).cpu().numpy()
    cut = 5_000_011
    parts = sum(m.payload_gram(*(t[:, a:b].contiguous() for t in (q, qd, qdd, tau))).cpu().numpy() for a, b in ((0, cut), (cut, n)))
    assert whole[111] == n and parts[111] == n
    assert np.abs(whole[:111] - parts[:111]).max() < tol * np.abs(whole[:100]).max()


def _identify_setup(n, seed):
    torch = _torch()
    from rigid_body_manipulation_b200.engine import Model

    traj = states(6, n, seed)
    q, qd, qdd = _soa(traj, torch.float64)
    return traj, q, qd, qdd, Model


@pytest.mark.gpu
def test_identification_recovers_every_packaged_target():
    """tau_meas from Model.rnea on the model WITH the object; the object-free model's payload Gram identifies the object's
    sensor-frame parameters, noise-free, for all 23 targets (one pack per object, the grouped solve)."""
    torch = _torch()
    from rigid_body_manipulation_b200 import identification

    traj, q, qd, qdd, Model = _identify_setup(20_000, 31)
    m0 = _model("object_free")
    names = sorted(pm.packaged_targets())
    packs = torch.empty((len(names), 112), dtype=torch.float64, device="cuda")
    truths = []
    for k, name in enumerate(names):
        c = pm.load_packaged("sequential", name)
        mo = Model(c.hposes_Rt, c.simats, c.uscrews, c.twist_0, c.dtwist_0, pose_sen_llj=c.pose_sen_Rt)
        m0.payload_gram(q, qd, qdd, mo.rnea(q, qd, qdd), pack=packs[k])
        truths.append(object_phi(c))
    for name, r, phi in zip(names, identification.solve_many(packs), truths):
        assert r.rank == 10 and r.n_samples == 20_000, name
        scale = np.array([phi[0]] * 4 + [max(np.abs(phi[4:]).max(), 1e-12)] * 6)
        assert (np.abs(r.phi - phi) / scale).max() < 1e-7, (name, r.phi, phi)


@pytest.mark.gpu
def test_identification_with_noise_matches_lstsq_and_the_ft_route():
    torch = _torch()
    from rigid_body_manipulation_b200 import identification

    n = 20_000
    traj, q, qd, qdd, Model = _identify_setup(n, 32)
    c = pm.load_packaged("sequential", "hammer")
    mo = Model(c.hposes_Rt, c.simats, c.uscrews, c.twist_0, c.dtwist_0, pose_sen_llj=c.pose_sen_Rt)
    m0 = _model("object_free")
    phi_true = object_phi(c)
    tau = mo.rnea(q, qd, qdd)
    noise = torch.as_tensor(np.random.default_rng(0).standard_normal((6, n)) * 0.5, device="cuda")
    got = identification.solve(m0.payload_gram(q, qd, qdd, tau + noise))
    out = m0.payload_regressor(q, qd, qdd, want_tau0=True)
    A = out["Phi"].reshape(-1, 10).cpu().numpy()
    r = (tau + noise - out["tau0"]).t().reshape(-1).cpu().numpy()
    ref, *_ = np.linalg.lstsq(A, r, rcond=None)
    assert np.abs(got.phi - ref).max() < 1e-9 * max(1.0, got.cond ** 0.5) * max(1.0, np.abs(ref).max())
    # the F/T route on the same trajectory: wrench = Y phi_true, the same object
    f = mo.regressor_from_traj(q, qd, qdd, want_rows=False, phi=phi_true)["wrench"]
    ft = identification.solve(mo.regressor_gram(q, qd, qdd, f))
    clean = identification.solve(m0.payload_gram(q, qd, qdd, tau))
    assert (np.abs(clean.phi - ft.phi) / SCALE).max() < 1e-7, (clean.phi, ft.phi)
    # a model that already contains the object sees no payload
    none = identification.solve(mo.payload_gram(q, qd, qdd, tau))
    assert (np.abs(none.phi) / SCALE).max() < 1e-7, none.phi


@pytest.mark.gpu
def test_argument_checks_and_canaries():
    torch = _torch()
    from rigid_body_manipulation_b200 import _lib

    m = _model("object_free")
    n = 300
    q, qd, qdd = _soa(states(6, n, 33), torch.float64)
    tau = torch.zeros((6, n), dtype=torch.float64, device="cuda")
    for bad in (q[:5], q.float(), q.cpu()):
        with pytest.raises(ValueError):
            m.payload_regressor(bad, qd, qdd)
        with pytest.raises(ValueError):
            m.payload_gram(q, qd, qdd, bad)
    with pytest.raises(ValueError):
        m.payload_gram(q, qd, qdd, tau, pack=torch.empty(111, dtype=torch.float64, device="cuda"))
    # undersized workspace
    ws = _gram_ws(m, n)
    pack = torch.empty(112, dtype=torch.float64, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = m._lib.rbm_payload_gram_f64(m._h, p(q), p(qd), p(qdd), p(tau), p(pack), p(ws), ws.numel() * 8 - 8, n, n, st)
    assert rc == _lib.RBM_ERR_INVALID
    # canary-padded outputs: nothing written past n samples
    canary, ld = 12345.0, n + 64
    pad = lambda t: torch.cat([t, torch.zeros((6, ld - n), dtype=t.dtype, device="cuda")], 1).contiguous()
    qp, qdp, qddp = pad(q), pad(qd), pad(qdd)
    Phi = torch.full((ld * 6 * 10,), canary, dtype=torch.float64, device="cuda")
    tau0 = torch.full((6, ld), canary, dtype=torch.float64, device="cuda")
    rc = m._lib.rbm_payload_regressor_f64(m._h, p(qp), p(qdp), p(qddp), p(Phi), p(tau0), n, ld, st)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.all(Phi[n * 60:] == canary) and torch.all(tau0[:, n:] == canary)
    ref = m.payload_regressor(q, qd, qdd, want_tau0=True)
    assert torch.equal(Phi[:n * 60].reshape(n, 6, 10), ref["Phi"]) and torch.equal(tau0[:, :n], ref["tau0"])
