"""-m gpu: every fast entry point on the model classes of tests/model_classes.py, against the fp64 oracles in oracle/.

The packaged robot selects SEQ_ISO with a sign-pattern sensor adjoint (SEN_DIAG) and gravity along z; these classes select the SEQ_RIGID
instantiations, the SEN_DIAG = false ones and a tilted base acceleration.  Sizes are chosen per entry point to reach each dispatch
branch (paired / unpaired / one-sample fp32 SoA, plain / TMA AoS, direct / TMA / tensor-core Gram with whole tiles and both half-tile
tails).  The packaged hammer model runs between the classes' calls of the AoS and Gram launchers; the Gram launcher raises the shared
memory limit of each kernel variant in its own cached slot, so this also switches between those slots.  Tolerances are the suite's
bars: 1e-9 in fp64, 1e-4 in fp32, norm-wise per sample (gpu_util.rel_err)."""
import ctypes as C
from dataclasses import dataclass

import numpy as np
import pytest
import torch

import model_classes
from gpu_util import rel_err, sample_states, soa
from oracle import lqr_oracle as lo
from oracle import replay_oracle as ro
from oracle import rnea_vec as rv
from rigid_body_manipulation_b200 import _lib, identification, planner
from rigid_body_manipulation_b200.engine import Model

pytestmark = pytest.mark.gpu

TOL64 = 1e-9
TOL32 = 1e-4
N_GRAM = 300_004        # 585 whole 512-sample TMA tiles + a 484-sample tail that reaches both half-tiles; a multiple of 4, so that the
                        # fp32 row pitch (n * 4 bytes) is 16-byte aligned too and fp32 takes the TMA and tensor-core kernels as well
N_RNEA = 4096 + 77      # 32 AoS tiles of 128 + a ragged 77; odd, so fp32 SoA with ld = n takes the one-sample kernel
INPUT_GAIN = [10.0, 10.0, 10.0, 1e4, 1e4, 1e4]             # configurations/base.yaml controller.input_gain
DISP = [0.2, 1.4, 0.6, np.pi, 0.0, 18.8495559215]          # configurations/base.yaml planner.displacements


@dataclass
class Case:
    mc: model_classes.ModelClass
    traj: np.ndarray    # (N_GRAM, 3, 6) sampled states
    f: np.ndarray       # (N_GRAM, 6) wrenches for the Gram
    tau: np.ndarray     # oracle answers for the first N_RNEA states
    V: np.ndarray
    dV: np.ndarray
    Vs: np.ndarray      # sensor-frame twists and regressor rows for all N_GRAM states
    dVs: np.ndarray
    Y: np.ndarray


@pytest.fixture(scope="module", params=model_classes.CLASSES)
def case(request):
    """One class and its oracle results (computed once per class)."""
    mc = model_classes.build(request.param)
    model_classes.analyze(mc)  # the class selects the path and sen_diag it was built for
    rng = np.random.default_rng(100 + model_classes.CLASSES.index(request.param))
    traj = sample_states(rng, N_GRAM)
    f = rng.standard_normal((N_GRAM, 6)) * np.array([5, 5, 5, 1, 1, 1.0])
    out = rv.inverse_batched(traj, mc.hposes_Rt, mc.simats, mc.uscrews, mc.twist_0, mc.dtwist_0)
    Vs, dVs = rv.sensor_frame_twists_batched(mc.pose_sen_Rt, out["twists"][:, 6], out["dtwists"][:, 6])
    return Case(mc=mc, traj=traj, f=f, tau=out["tau"][:N_RNEA], V=out["twists"][:N_RNEA, 6], dV=out["dtwists"][:N_RNEA, 6], Vs=Vs, dVs=dVs,
                Y=rv.regressor_batched(Vs, dVs))


def make_model(mc, **flags):
    args, kw = mc.model_args()
    m = Model(*args, **kw, **flags)
    assert m.kernel_path == mc.path, (mc.name, m.kernel_path)
    return m


def hammer_model(**flags):
    return make_model(model_classes.build("hammer"), **flags)


def host(t):
    """(rows, n) device tensor -> (n, rows) float64 array."""
    return t.t().double().cpu().numpy()


def vp(t):
    return C.c_void_p(t.data_ptr())


# ---- inverse dynamics ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 129, N_RNEA])
def test_rnea_fp64_tau_and_twists(case, n):
    m = make_model(case.mc)
    q, qd, qdd = soa(case.traj[:n])
    tau, V, dV = m.rnea(q, qd, qdd, want_twists=True)
    assert rel_err(host(tau), case.tau[:n]).max() < TOL64
    assert rel_err(host(V), case.V[:n]).max() < TOL64
    assert rel_err(host(dV), case.dV[:n]).max() < TOL64
    assert torch.equal(m.rnea(q, qd, qdd), tau)  # the tau-only kernel: same recursion, same bits


def _check_f32(case, n, tau, V, dV):
    assert rel_err(host(tau[:, :n]), case.tau[:n]).max() < TOL32
    assert rel_err(host(V[:, :n]), case.V[:n]).max() < TOL32
    assert rel_err(host(dV[:, :n]), case.dV[:n]).max() < TOL32


def test_rnea_fp32_tau_and_twists(case):
    m = make_model(case.mc)
    lib = _lib.load()
    # contiguous, even n: two samples per thread (f32x2), every thread paired
    n = 4096
    q, qd, qdd = soa(case.traj[:n], torch.float32)
    tau, V, dV = m.rnea(q, qd, qdd, want_twists=True)
    _check_f32(case, n, tau, V, dV)
    assert torch.equal(m.rnea(q, qd, qdd), tau)
    # contiguous, odd n (odd row pitch): one sample per thread
    n = N_RNEA
    q, qd, qdd = soa(case.traj[:n], torch.float32)
    tau, V, dV = m.rnea(q, qd, qdd, want_twists=True)
    _check_f32(case, n, tau, V, dV)
    assert torch.equal(m.rnea(q, qd, qdd), tau)

    def raw(n, ld, offset, twists):
        """The raw ABI on (6, ld) buffers that start `offset` floats into their allocation; the padding must stay untouched."""
        bufs = []
        for k in range(3):
            b = torch.full((6 * ld + offset,), float("nan"), dtype=torch.float32, device="cuda")
            b[offset:].view(6, ld)[:, :n] = torch.as_tensor(case.traj[:n, k, :].T, dtype=torch.float32, device="cuda")
            bufs.append(b[offset:].view(6, ld))
        outs = [torch.full((6 * ld + offset,), -7.0, dtype=torch.float32, device="cuda")[offset:].view(6, ld) for _ in range(3 if twists else 1)]
        ptrs = [vp(o) for o in outs] + ([None, None] if not twists else [])
        rc = lib.rbm_rnea_f32(m._h, *(vp(b) for b in bufs), *ptrs, n, ld, C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, _lib.last_error()
        torch.cuda.synchronize()
        for o in outs:
            assert (o[:, n:] == -7.0).all()
        return outs

    # even row pitch, odd n: f32x2 with the last thread's pair cut short (unpaired tail)
    tau, V, dV = raw(N_RNEA, N_RNEA + 1, 0, True)
    _check_f32(case, N_RNEA, tau, V, dV)
    assert torch.equal(raw(N_RNEA, N_RNEA + 1, 0, False)[0], tau)
    # base pointers one float off an 8-byte boundary: one sample per thread
    tau, V, dV = raw(4096, 4098, 1, True)
    _check_f32(case, 4096, tau, V, dV)
    assert torch.equal(raw(4096, 4098, 1, False)[0], tau)


@pytest.mark.parametrize("dtype,tol", [(torch.float64, TOL64), (torch.float32, TOL32)])
def test_rnea_aos(case, dtype, tol):
    m, plain = make_model(case.mc), make_model(case.mc, no_tma=True)
    ham = hammer_model()
    for n in (100, N_RNEA):  # below one 128-sample tile: plain kernel; above: TMA tiles + ragged tail
        traj = torch.as_tensor(case.traj[:n], dtype=dtype, device="cuda")
        tau = m.rnea_aos(traj)
        assert rel_err(tau.double().cpu().numpy(), case.tau[:n]).max() < tol
        ham.rnea_aos(traj)
        assert torch.equal(m.rnea_aos(traj), tau)
        assert rel_err(plain.rnea_aos(traj).double().cpu().numpy(), case.tau[:n]).max() < tol


def test_rnea_planned(case):
    mc = case.mc
    m = make_model(mc)
    plan = planner.QuinticPlan(DISP, mc.key_qpos, 0.002, 1500)

    def oracle(traj):
        t = traj.permute(2, 0, 1).double().cpu().numpy()
        return t, rv.inverse_batched(t, mc.hposes_Rt, mc.simats, mc.uscrews, mc.twist_0, mc.dtwist_0)["tau"]

    tau, traj = m.rnea_planned(plan, want_traj=True)
    t, ref = oracle(traj)
    assert np.abs(t - plan.trajectory()).max() < 1e-11 * np.abs(t).max()
    assert rel_err(host(tau), ref).max() < TOL64
    tau, traj = m.rnea_planned(plan, n=300, step0=3.0, stride=4.5, want_traj=True)  # fractional stride: between planned steps
    assert rel_err(host(tau), oracle(traj)[1]).max() < TOL64
    tau32, traj32 = m.rnea_planned(plan, dtype=torch.float32, want_traj=True)
    assert rel_err(host(tau32), oracle(traj32)[1]).max() < TOL32


def test_host_entries(case):
    """rbm_rnea_host / _host_soa / _planned_host, chunked: bit-identical to the device entries, and the oracle."""
    mc = case.mc
    m = make_model(mc)
    n, chunk = N_RNEA, 1024
    traj = case.traj[:n]
    dev = m.rnea_aos(torch.as_tensor(traj, device="cuda")).cpu().numpy()
    assert np.array_equal(m.rnea_host(traj, chunk=chunk), dev)
    assert rel_err(dev, case.tau[:n]).max() < TOL64
    q, qd, qdd = (np.ascontiguousarray(traj[:, k, :].T) for k in range(3))
    want = m.rnea(*soa(traj)).cpu().numpy()
    q[:3] = np.nan   # rows the tau-only kernel does not read: the gantry positions and velocities
    qd[:3] = np.nan
    got = m.rnea_host_soa(q, qd, qdd, chunk=chunk)
    assert np.array_equal(got, want)
    assert rel_err(got.T, case.tau[:n]).max() < TOL64
    plan = planner.QuinticPlan(DISP, mc.key_qpos, 0.002, 1500)
    tau_p, traj_p = m.rnea_planned(plan, want_traj=True)
    assert np.array_equal(m.rnea_planned_host(plan, chunk=chunk).numpy(), tau_p.cpu().numpy())
    t = traj_p.permute(2, 0, 1).cpu().numpy()
    assert rel_err(host(tau_p), rv.inverse_batched(t, mc.hposes_Rt, mc.simats, mc.uscrews, mc.twist_0, mc.dtwist_0)["tau"]).max() < TOL64


# ---- sensor-frame regressor, Gram, identification ---------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,tol", [(torch.float64, TOL64), (torch.float32, TOL32)])
def test_regressor_from_traj(case, dtype, tol):
    m = make_model(case.mc)
    n = N_RNEA
    q, qd, qdd = soa(case.traj[:n], dtype)
    out = m.regressor_from_traj(q, qd, qdd, want_rows=True, want_twists=True, phi=case.mc.phi)
    assert rel_err(out["Y"].double().cpu().numpy(), case.Y[:n]).max() < tol
    assert rel_err(host(out["twist_sen"]), case.Vs[:n]).max() < tol
    assert rel_err(host(out["dtwist_sen"]), case.dVs[:n]).max() < tol
    assert rel_err(host(out["wrench"]), case.Y[:n] @ case.mc.phi).max() < tol


GRAM_MODES = {"fp64": (torch.float64, {}, TOL64), "fp32": (torch.float32, {}, TOL32),
              "fp32_tc": (torch.float32, dict(gram_tensor_cores=True), TOL32)}


@pytest.mark.parametrize("mode", list(GRAM_MODES))
@pytest.mark.parametrize("n,no_tma", [(511, False), (4096, False), (4097, False), (N_GRAM, False), (N_GRAM, True)])
def test_regressor_gram(case, mode, n, no_tma):
    """511 and odd 4097 take the direct-load kernel; 4096 whole TMA (or, with gram_tensor_cores, tensor-core) tiles; N_GRAM whole tiles
    + a tail over both half-tiles, in fp64 and fp32 alike (16-byte aligned rows); no_tma=True the direct-load kernel at N_GRAM."""
    dtype, flags, tol = GRAM_MODES[mode]
    m = make_model(case.mc, no_tma=no_tma, **flags)
    ham = hammer_model(no_tma=no_tma, **flags)
    q, qd, qdd = soa(case.traj[:n], dtype)
    fd = torch.as_tensor(case.f[:n], dtype=dtype, device="cuda").t().contiguous()
    ref = rv.gram_pack(case.Y[:n], case.f[:n])
    pack = m.regressor_gram(q, qd, qdd, fd).cpu().numpy()
    scale = np.abs(ref[:100]).max()
    assert np.abs(pack[:100] - ref[:100]).max() < tol * scale
    assert np.abs(pack[100:110] - ref[100:110]).max() < tol * (scale if dtype == torch.float32 else max(np.abs(ref[100:110]).max(), 1.0))
    assert abs(pack[110] - ref[110]) < tol * ref[110]
    assert pack[111] == n
    G = pack[:100].reshape(10, 10)
    assert np.array_equal(G, G.T)
    ham.regressor_gram(q, qd, qdd, fd)                                        # another variant of the same launcher in between
    assert np.array_equal(m.regressor_gram(q, qd, qdd, fd).cpu().numpy(), pack)  # fixed reduction order: bit-reproducible


def test_identification_recovers_the_class_parameters(case):
    """f = Y phi synthesised on the device over 2^20 samples, fp64 Gram, 10x10 solve on the host -> the class's phi."""
    m = make_model(case.mc)
    n = 1 << 20
    q, qd, qdd = soa(sample_states(np.random.default_rng(42), n))
    phi = case.mc.phi
    f = m.regressor_from_traj(q, qd, qdd, want_rows=False, phi=phi)["wrench"]
    ident = identification.solve(m.regressor_gram(q, qd, qdd, f))
    assert ident.n_samples == n and ident.rank == 10
    assert np.abs(ident.phi - phi).max() < 1e-8 * np.abs(phi).max(), (ident.phi, phi)


def test_regressor_gram_grouped(case):
    """Frame-major (F, rows, groups) log: one pack per group against the oracle's pack of that group's samples."""
    m = make_model(case.mc)
    F, G = 60, 7
    sub = case.traj[:F * G].reshape(F, G, 3, 6)
    dev = lambda a: torch.as_tensor(np.ascontiguousarray(a.transpose(0, 2, 1)), device="cuda")  # (F, G, k) -> (F, k, G)
    f = case.f[:F * G].reshape(F, G, 6)
    packs = m.regressor_gram_grouped(dev(sub[:, :, 0]), dev(sub[:, :, 1]), dev(sub[:, :, 2]), dev(f)).cpu().numpy()
    Y = case.Y[:F * G].reshape(F, G, 6, 10)
    for g in range(G):
        ref = rv.gram_pack(Y[:, g], f[:, g])
        assert np.abs(packs[g] - ref).max() < TOL64 * np.abs(ref).max(), g


# ---- linearisation, forward dynamics, closed loop -------------------------------------------------------------------------------
def _dev(a):
    return None if a is None else torch.as_tensor(np.ascontiguousarray(a.T), device="cuda")


def test_linearize(case):
    c = case.mc.consts
    m = make_model(case.mc)
    n = 48
    tr = sample_states(np.random.default_rng(3), n)
    q, qd = tr[:, 0], tr[:, 1]
    u = np.random.default_rng(4).standard_normal((n, 6)) * np.array([100, 100, 400, 1, 1, 1.0])

    def run(**kw):
        A, B, qdd = m.linearize(_dev(q), _dev(qd), _dev(u), dt=0.002, want_qdd=True, **kw)
        return A.cpu().numpy(), B.cpu().numpy(), qdd.t().cpu().numpy()

    A, B, qdd = run(eps=1e-5, centered=True)
    Ar, Br = lo.transition_fd(c, q, qd, u, dt=0.002, eps=1e-5, centered=True)
    assert np.abs(qdd - lo.forward_dynamics(c, q, qd, u)).max() < 1e-9 * np.abs(qdd).max()
    assert np.abs(A - Ar).max() < 2e-8 and np.abs(B - Br).max() < 2e-8
    # the kernel skips the gantry columns (SequentialDesc::q_matters / qd_matters): the literal transition FD confirms they are the
    # identity's, here with links off the isotropic form and gravity off the z axis as well
    assert np.abs(Ar[:, 6:, :3]).max() < 1e-8 and np.abs(Ar[:, 6:, 6:9] - np.eye(6)[None, :, :3]).max() < 1e-8
    assert np.abs(A[:, 6:, :3]).max() < 1e-8 and np.abs(A[:, 6:, 6:9] - np.eye(6)[None, :, :3]).max() < 1e-8
    A, B, _ = run(eps=1e-8, centered=True)
    Ar, Br = lo.transition_fd(c, q, qd, u, dt=0.002, eps=1e-8, centered=True)
    assert np.abs(A - Ar).max() < 5e-6 and np.abs(B - Br).max() < 5e-6
    A, B, _ = run(eps=1e-6, centered=False)
    Ar, Br = lo.transition_fd(c, q, qd, u, dt=0.002, eps=1e-6, centered=False)
    assert np.abs(A - Ar).max() < 1e-4 and np.abs(B - Br).max() < 2e-7


def test_forward_dynamics_and_step(case):
    c = case.mc.consts
    m = make_model(case.mc)
    n, dt = 64, 0.002
    tr = sample_states(np.random.default_rng(21), n)
    q, qd = tr[:, 0], tr[:, 1]
    u = np.random.default_rng(22).standard_normal((n, 6)) * np.array([100, 100, 400, 1, 1, 1.0])
    ref = lo.forward_dynamics(c, q, qd, u)
    assert np.abs(m.forward_dynamics(_dev(q), _dev(qd), _dev(u)).t().cpu().numpy() - ref).max() < 1e-9 * np.abs(ref).max()
    qn, qdn = m.step(_dev(q), _dev(qd), _dev(u), dt=dt)
    y = lo.step(c, q, qd, u, dt)
    assert np.abs(np.concatenate([qn.t().cpu().numpy(), qdn.t().cpu().numpy()], 1) - y).max() < 1e-11 * np.abs(y).max()
    qi, qdi = _dev(q), _dev(qd)
    m.step(qi, qdi, _dev(u), dt=dt, inplace=True)
    assert torch.equal(qi, qn) and torch.equal(qdi, qdn)


def test_closed_loop(case):
    mc = case.mc
    c = mc.consts
    m = make_model(mc)
    plan = planner.QuinticPlan(DISP, mc.key_qpos, 0.002, 400)
    K = ro.lqr_gain(c, mc.key_qpos, np.zeros(6), INPUT_GAIN)
    q0 = np.stack([mc.key_qpos, mc.key_qpos + [0.01, -0.02, 0.015, 0.05, -0.04, 0.03]])   # keyframe start, perturbed start
    qd0 = np.stack([np.zeros(6), [0.02, 0.01, -0.03, 0.1, -0.2, 0.05]])
    out = m.closed_loop(plan, K, mc.phi, _dev(q0), _dev(qd0))
    frames, steps, final = out["frames"].cpu().numpy(), out["frame_steps"].cpu().numpy(), out["final"].cpu().numpy()
    traj = plan.trajectory()
    for e in range(2):
        ref = ro.closed_loop_replay(c, mc.pose_sen_Rt, mc.G_sensed, traj, K, q0[e], qd0[e])
        assert np.array_equal(steps, ref["step"])
        for sl, key in ((slice(0, 18), "act"), (slice(18, 24), "twist_sen"), (slice(24, 30), "dtwist_sen"), (slice(30, 36), "wrench")):
            want = ref[key].reshape(len(ref["step"]), -1)
            assert np.abs(frames[:, sl, e] - want).max() < TOL64 * np.abs(want).max(), (e, key)
        assert np.abs(final[:6, e] - ref["q_final"]).max() < 1e-10 and np.abs(final[6:12, e] - ref["qd_final"]).max() < 1e-10
