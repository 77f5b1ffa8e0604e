"""-m gpu: every generic entry point at every joint count of tests/chains.py (1 to 16, and 6 for the constant-bank SoA instance), through
engine.Model, against the oracles.  The chains carry a tip wrench through a tip pose, a moving base and tilted gravity, so the split of
the tip wrench (in the bias h, never in M) is checked on the device as well.  tests/test_joint_counts_host.py runs the same chains
(same seeds) through the host build of the per-sample code.  Tolerances: 1e-9 norm-wise per sample in fp64, 1e-4 in fp32, and the
linearisation and Gram bounds of tests/test_gpu_linearize.py and tests/test_gpu_regressor.py."""
import numpy as np
import pytest
import torch

import chains
from gpu_util import rel_err
from oracle import lqr_oracle as lo
from oracle import replay_oracle as ro
from oracle import rnea_vec as rv
from rigid_body_manipulation_b200 import planner
from test_payload_identification import oracle_payload, phi_to_inertia

pytestmark = pytest.mark.gpu
TOL64, TOL32 = 1e-9, 1e-4
NJ = [pytest.param(nj, id=f"nj{nj}") for nj in chains.NJ_ALL]


def _model(nj):
    from rigid_body_manipulation_b200.engine import Model

    ch = chains.random_chain(nj, seed=100 + nj)
    ch.analyze()
    args, kw = ch.model_args()
    m = Model(*args, **kw)
    assert m.kernel_path == "generic" and m.nj == nj
    return ch, m


def _vec(ch):
    c = ch.consts
    return dict(hposes_Rt=c["hposes_Rt"], simats=c["simats"], uscrews=c["uscrews"], twist_0=c["twist_0"], dtwist_0=c["dtwist_0"], **lo.tip_kw(c))


def _soa(traj, dtype=torch.float64):
    t = torch.as_tensor(np.ascontiguousarray(traj), dtype=dtype, device="cuda")
    return tuple(t[:, k, :].t().contiguous() for k in range(3))


def _host(t):
    return t.double().cpu().numpy()


def _err32(got, want, nj):
    """fp32 error of torques: norm-wise per sample, except with one joint, where the per-sample norm is a single torque that crosses
    zero within a batch (measured on a B200: 3.3e-4 and 5.2e-4 relative at isolated near-zero samples, ~1e-7 elsewhere); there the
    norm is taken over the batch."""
    return rel_err(got, want).max() if nj > 1 else np.abs(got - want).max() / np.abs(want).max()


def _oracle(ch, traj):
    """The oracle on exactly the inputs the kernel saw (fp32 inputs are rounded before they reach the oracle)."""
    return rv.inverse_batched(np.asarray(traj, np.float64), **_vec(ch))


def test_joint_count_limits_on_the_device():
    from rigid_body_manipulation_b200.engine import Model

    ch = chains.random_chain(17, 0, tip=False)
    args, kw = ch.model_args()
    with pytest.raises(NotImplementedError, match="RBM_MAX_JOINTS"):
        Model(*args, **kw)
    with pytest.raises(ValueError, match="nj must be >= 1"):
        Model(args[0][:1], args[1][:1], args[2][:0], *args[3:], **kw)


@pytest.mark.parametrize("nj", NJ)
@pytest.mark.parametrize("n", [1, 255, 4099])
def test_rnea_soa_aos_and_full_state(nj, n):
    ch, m = _model(nj)
    traj = ch.sample(n, 10 + nj)
    ref = _oracle(ch, traj)
    tau, V, dV = m.rnea(*_soa(traj), want_twists=True)
    assert rel_err(_host(tau).T, ref["tau"]).max() < TOL64
    assert rel_err(_host(V).T, ref["twists"][:, nj]).max() < TOL64 and rel_err(_host(dV).T, ref["dtwists"][:, nj]).max() < TOL64
    assert torch.equal(m.rnea(*_soa(traj)), tau)  # tau-only launch: same bits
    aos = m.rnea_aos(torch.as_tensor(traj, device="cuda"))
    assert rel_err(_host(aos), ref["tau"]).max() < TOL64
    t_full, poses, tw, dtw = m.rnea_full(torch.as_tensor(traj, device="cuda"))
    assert rel_err(_host(t_full), ref["tau"]).max() < TOL64 and rel_err(_host(poses), ref["poses"]).max() < TOL64
    assert rel_err(_host(tw), ref["twists"]).max() < TOL64 and rel_err(_host(dtw), ref["dtwists"]).max() < TOL64
    t32 = traj.astype(np.float32)
    ref32 = _oracle(ch, t32)
    tau32, V32, dV32 = m.rnea(*_soa(t32, torch.float32), want_twists=True)
    err32 = max(_err32(_host(tau32).T, ref32["tau"], nj), rel_err(_host(V32).T, ref32["twists"][:, nj]).max(),
                rel_err(_host(dV32).T, ref32["dtwists"][:, nj]).max())
    print(f"fp32 rnea nj={nj} n={n}: max norm-wise error {err32:.3g}")
    assert err32 < TOL32
    assert _err32(_host(m.rnea_aos(torch.as_tensor(t32, device="cuda"))), ref32["tau"], nj) < TOL32


@pytest.mark.parametrize("nj", NJ)
def test_regressor_from_traj_and_gram(nj):
    ch, m = _model(nj)
    n = 4099
    traj = ch.sample(n, 20 + nj)
    rng = np.random.default_rng(nj)
    phi = chains.phi_sensed(nj)
    f = rng.standard_normal((n, 6)) * np.array([5, 5, 5, 1, 1, 1.0])
    for dtype, tol in ((torch.float64, TOL64), (torch.float32, TOL32)):
        tr = traj.astype(np.float32) if dtype == torch.float32 else traj
        ref = _oracle(ch, tr)
        Vs, dVs = rv.sensor_frame_twists_batched(ch.pose_sen_Rt, ref["twists"][:, nj], ref["dtwists"][:, nj])
        Y = rv.regressor_batched(Vs, dVs)
        out = m.regressor_from_traj(*_soa(tr, dtype), want_rows=True, want_twists=True, phi=phi)
        assert rel_err(_host(out["Y"]), Y).max() < tol
        assert rel_err(_host(out["twist_sen"]).T, Vs).max() < tol and rel_err(_host(out["dtwist_sen"]).T, dVs).max() < tol
        assert rel_err(_host(out["wrench"]).T, Y @ phi).max() < tol
        fr = f.astype(np.float32).astype(np.float64) if dtype == torch.float32 else f
        want = rv.gram_pack(Y, fr)
        pack = m.regressor_gram(*_soa(tr, dtype), torch.as_tensor(fr.T.copy(), dtype=dtype, device="cuda")).cpu().numpy()
        scale = np.abs(want[:100]).max()
        assert pack[111] == n
        assert np.abs(pack[:100] - want[:100]).max() < tol * scale
        assert np.abs(pack[100:110] - want[100:110]).max() < tol * max(np.abs(want[100:110]).max(), 1.0)
        assert abs(pack[110] - want[110]) < tol * want[110]


@pytest.mark.parametrize("nj", NJ)
def test_payload_regressor_and_gram(nj):
    ch, m = _model(nj)
    n = 1000
    traj = ch.sample(n, 30 + nj)
    c = ch.consts
    for dtype, tol in ((torch.float64, TOL64), (torch.float32, TOL32)):
        tr = traj.astype(np.float32).astype(np.float64) if dtype == torch.float32 else traj
        ref_phi, ref_tau0 = oracle_payload(c, ch.pose_sen_Rt, tr, **lo.tip_kw(c))
        scale = np.abs(ref_tau0).max()
        q, qd, qdd = _soa(tr, dtype)
        out = m.payload_regressor(q, qd, qdd, want_rows=True, want_tau0=True)
        assert np.abs(_host(out["tau0"]).T - ref_tau0).max() < tol * scale
        assert np.abs(_host(out["Phi"]) - ref_phi).max() < tol * scale
        tau = torch.as_tensor(ref_tau0.T + np.random.default_rng(nj).standard_normal((nj, n)), dtype=dtype, device="cuda")
        pack = m.payload_gram(q, qd, qdd, tau).cpu().numpy()
        A, r = ref_phi.reshape(-1, 10), (_host(tau).T - ref_tau0).reshape(-1)
        want = np.concatenate([(A.T @ A).reshape(100), A.T @ r, [r @ r], [n]])
        gs = np.abs(want[:100]).max()
        assert pack[111] == n and np.abs(pack[:100] - want[:100]).max() < tol * gs
        assert np.abs(pack[100:110] - want[100:110]).max() < tol * max(np.abs(want[100:110]).max(), np.sqrt(gs * want[110]))


@pytest.mark.parametrize("nj", NJ)
def test_linearize_forward_dynamics_and_step(nj):
    ch, m = _model(nj)
    c = ch.consts
    n = 255
    traj = ch.sample(n, 40 + nj)
    q, qd = traj[:, 0], traj[:, 1]
    u = np.random.default_rng(nj).standard_normal((n, nj)) * 20
    to = lambda a: torch.as_tensor(np.ascontiguousarray(a.T), device="cuda")
    ref = lo.forward_dynamics(c, q, qd, u)
    assert np.abs(_host(m.forward_dynamics(to(q), to(qd), to(u))).T - ref).max() < TOL64 * np.abs(ref).max()
    qn, qdn = m.step(to(q), to(qd), to(u), dt=0.002)
    y = lo.step(c, q, qd, u, 0.002)
    assert np.abs(np.concatenate([_host(qn).T, _host(qdn).T], 1) - y).max() < 1e-11 * np.abs(y).max()
    # finite differences at q = 2e5 carry the rounding of q +- eps (tests/test_joint_counts_host.py): linearise off that row
    lin = np.where(np.abs(q) > 1e3, 1.0, q)[:64]
    qdl, ul = qd[:64], u[:64]
    ref_l = lo.forward_dynamics(c, lin, qdl, ul)
    for centered, eps, tol_a, tol_b in ((True, 1e-5, 2e-8, 2e-8), (True, 1e-8, 5e-6, 5e-6), (False, 1e-6, 1e-4, 2e-7)):
        A, B, qdd = m.linearize(to(lin), to(qdl), to(ul), dt=0.002, eps=eps, centered=centered, want_qdd=True)
        Ar, Br = lo.transition_fd(c, lin, qdl, ul, dt=0.002, eps=eps, centered=centered)
        assert np.abs(_host(A) - Ar).max() < tol_a and np.abs(_host(B) - Br).max() < tol_b, (centered, eps)
        assert np.abs(_host(qdd).T - ref_l).max() < TOL64 * np.abs(ref_l).max()


@pytest.mark.parametrize("nj", NJ)
def test_closed_loop(nj):
    ch, m = _model(nj)
    rng = np.random.default_rng(300 + nj)
    key = rng.uniform(-1, 1, nj)
    plan = planner.QuinticPlan(rng.uniform(-0.5, 0.5, nj), key, 0.002, 100)
    K = -np.hstack([50.0 * np.eye(nj), 5.0 * np.eye(nj)])
    phi = chains.phi_sensed(nj)
    q0 = np.stack([key, key + rng.uniform(-0.05, 0.05, nj), key - 0.02], axis=1)
    qd0 = np.stack([np.zeros(nj), rng.uniform(-0.1, 0.1, nj), np.full(nj, 0.05)], axis=1)
    out = m.closed_loop(plan, K, phi, torch.as_tensor(q0, device="cuda"), torch.as_tensor(qd0, device="cuda"))  # divisor = nj
    steps = out["frame_steps"].cpu().numpy()
    frames, final = _host(out["frames"]), _host(out["final"])
    for e in range(q0.shape[1]):
        ref = ro.closed_loop_replay(ch.consts, ch.pose_sen_Rt, phi_to_inertia(phi), plan.trajectory(), K, q0[:, e], qd0[:, e], nu=float(nj))
        assert np.array_equal(steps, ref["step"])
        for sl, key_ in ((slice(0, 3 * nj), "act"), (slice(3 * nj, 3 * nj + 6), "twist_sen"), (slice(3 * nj + 6, 3 * nj + 12), "dtwist_sen"),
                         (slice(3 * nj + 12, 3 * nj + 18), "wrench")):
            want = ref[key_].reshape(len(steps), -1)
            assert np.abs(frames[:, sl, e] - want).max() < TOL64 * np.abs(want).max(), (e, key_)
        assert np.abs(final[:nj, e] - ref["q_final"]).max() < 1e-11 and np.abs(final[nj:2 * nj, e] - ref["qd_final"]).max() < 1e-11


@pytest.mark.parametrize("nj", NJ)
def test_rnea_planned(nj):
    ch, m = _model(nj)
    rng = np.random.default_rng(500 + nj)
    plan = planner.QuinticPlan(rng.uniform(-1, 1, nj), rng.uniform(-1, 1, nj), 0.002, 1500)
    for dtype, tol, kw in ((torch.float64, TOL64, {}), (torch.float32, TOL32, {}), (torch.float64, TOL64, dict(n=4099, step0=3.0, stride=0.37))):
        tau, traj = m.rnea_planned(plan, dtype=dtype, want_traj=True, **kw)
        t = _host(traj).transpose(2, 0, 1)
        if not kw:
            assert np.abs(t - plan.trajectory()).max() < (1e-11 if dtype == torch.float64 else 1e-5) * np.abs(t).max()
        ref = _oracle(ch, t)["tau"]
        assert (rel_err(_host(tau).T, ref).max() if dtype == torch.float64 else _err32(_host(tau).T, ref, nj)) < tol


@pytest.mark.parametrize("nj", NJ)
def test_regressor_gram_grouped(nj):
    ch, m = _model(nj)
    F, G = 20, 37
    traj = ch.sample(F * G, 60 + nj).reshape(F, G, 3, nj)
    f = np.random.default_rng(nj).standard_normal((F, G, 6))
    log_q = torch.as_tensor(np.ascontiguousarray(traj.transpose(0, 2, 3, 1)), device="cuda")   # (F, 3, nj, G)
    packs = m.regressor_gram_grouped(log_q[:, 0], log_q[:, 1], log_q[:, 2], torch.as_tensor(np.ascontiguousarray(f.transpose(0, 2, 1)), device="cuda"))
    packs = packs.cpu().numpy()
    for g in (0, 17, G - 1):
        ref = _oracle(ch, traj[:, g])
        Vs, dVs = rv.sensor_frame_twists_batched(ch.pose_sen_Rt, ref["twists"][:, nj], ref["dtwists"][:, nj])
        want = rv.gram_pack(rv.regressor_batched(Vs, dVs), f[:, g])
        assert np.abs(packs[g] - want).max() < TOL64 * np.abs(want).max()


def test_nj16_rnea_at_scale():
    """2^20 samples of the 16-joint chain in one launch: 4096 random samples and the last 300 against the oracle."""
    ch, m = _model(16)
    n = 1 << 20
    traj = ch.sample(n, 7)
    tau = _host(m.rnea(*_soa(traj))).T
    idx = np.concatenate([np.random.default_rng(1).choice(n, 4096, replace=False), np.arange(n - 300, n)])
    assert rel_err(tau[idx], _oracle(ch, traj[idx])["tau"]).max() < TOL64
    assert np.isfinite(tau).all()


def test_nj16_linearize_at_scale():
    """2^18 states of the 16-joint chain (A: 1024 rows, B: 512 rows of 2^18 doubles): 64 states against the transition FD."""
    ch, m = _model(16)
    n = 1 << 18
    traj = ch.sample(n, 8)
    q = np.where(np.abs(traj[:, 0]) > 1e3, 1.0, traj[:, 0])
    to = lambda a: torch.as_tensor(np.ascontiguousarray(a.T), device="cuda")
    A, B = m.linearize(to(q), to(traj[:, 1]), None, dt=0.002, eps=1e-5)
    idx = np.concatenate([np.random.default_rng(2).choice(n, 62, replace=False), [0, n - 1]])
    it = torch.as_tensor(idx, device="cuda")
    Ar, Br = lo.transition_fd(ch.consts, q[idx], traj[idx, 1], None, dt=0.002, eps=1e-5)
    assert np.abs(_host(A[it]) - Ar).max() < 2e-8 and np.abs(_host(B[it]) - Br).max() < 2e-8
    assert bool(torch.isfinite(A).all()) and bool(torch.isfinite(B).all())
