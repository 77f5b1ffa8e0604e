"""-m gpu parity tests of the batched inverse dynamics (C ABI rbm_rnea_*) against
 (a) golden vectors produced by executing the reference's own dynamics.py (tests/golden, oracle/gen_golden.py)
 (b) the vectorised CPU oracle (oracle/rnea_vec.py) at BASELINE.json config 2 size (2^20 samples).
Tolerances (BASELINE.json north_star): 1e-9 relative in fp64, 1e-4 relative in fp32, norm-wise per sample."""
import numpy as np
import pytest
import torch

from gpu_util import load_golden, model_from_golden, rel_err, sample_states, soa
from oracle import rnea_vec as rv

pytestmark = pytest.mark.gpu

TOL64 = 1e-9
TOL32 = 1e-4
TARGETS = ["hammer", "uniform_gearbox", "kill_la_kill"]
GENERIC = ["nj6", "nj4", "nj9"]
ALL = [f"ref_inverse_{t}.npz" for t in TARGETS] + [f"ref_inverse_generic_{g}.npz" for g in GENERIC]


@pytest.mark.parametrize("fname", ALL)
@pytest.mark.parametrize("force_generic", [False, True])
def test_fp64_soa_matches_reference_golden(fname, force_generic):
    g = load_golden(fname)
    m = model_from_golden(g, force_generic=force_generic)
    is_target = "generic" not in fname
    assert m.kernel_path == ("seq_iso" if (is_target and not force_generic) else "generic")
    q, qd, qdd = soa(g["traj"])
    tau, V, dV = m.rnea(q, qd, qdd, want_twists=True)
    torch.cuda.synchronize()
    nj = m.nj
    assert rel_err(tau.t().cpu().numpy(), g["tau"]).max() < TOL64
    assert rel_err(V.t().cpu().numpy(), g["twists"][:, nj]).max() < TOL64
    assert rel_err(dV.t().cpu().numpy(), g["dtwists"][:, nj]).max() < TOL64
    tau2 = m.rnea(q, qd, qdd)
    assert torch.equal(tau, tau2)  # with / without the twist outputs: same arithmetic


@pytest.mark.parametrize("fname", ALL)
def test_fp64_aos_and_full_state(fname):
    g = load_golden(fname)
    m = model_from_golden(g)
    traj = torch.as_tensor(g["traj"], device="cuda")
    tau = m.rnea_aos(traj)
    assert rel_err(tau.cpu().numpy(), g["tau"]).max() < TOL64
    tau_f, poses, tw, dtw = m.rnea_full(traj)
    assert rel_err(tau_f.cpu().numpy(), g["tau"]).max() < TOL64
    assert np.abs(poses.cpu().numpy() - g["poses"]).max() < 1e-12
    assert rel_err(tw.cpu().numpy(), g["twists"]).max() < TOL64
    assert rel_err(dtw.cpu().numpy(), g["dtwists"]).max() < TOL64


@pytest.mark.parametrize("fname", ALL)
@pytest.mark.parametrize("force_generic", [False, True])
def test_fp32_mode(fname, force_generic):
    g = load_golden(fname)
    m = model_from_golden(g, force_generic=force_generic)
    q, qd, qdd = soa(g["traj"], torch.float32)
    tau = m.rnea(q, qd, qdd)
    assert tau.dtype == torch.float32
    assert rel_err(tau.t().cpu().numpy(), g["tau"]).max() < TOL32
    tau_aos = m.rnea_aos(torch.as_tensor(g["traj"], dtype=torch.float32, device="cuda"))
    assert rel_err(tau_aos.cpu().numpy(), g["tau"]).max() < TOL32


def test_static_gravity_known_answer():
    g = load_golden("ref_inverse_hammer.npz")
    m = model_from_golden(g)
    traj = np.zeros((1, 3, 6))
    traj[0, 0] = g["key_qpos"]
    tau = m.rnea_aos(torch.as_tensor(traj, device="cuda")).cpu().numpy()[0]
    assert abs(tau[2] - (32.0 + float(g["gt_mass"])) * 9.81) < 1e-9
    assert np.abs(tau[[0, 1]]).max() < 1e-9


def test_config1_planned_trajectory():
    """BASELINE.json config 1 (open-loop part): tau for all 1500 planned steps of base.yaml, V6/dV6 included."""
    g = load_golden("ref_inverse_hammer.npz")
    c1 = load_golden("ref_config1_hammer.npz")
    m = model_from_golden(g)
    q, qd, qdd = soa(c1["traj"])
    tau, V, dV = m.rnea(q, qd, qdd, want_twists=True)
    assert rel_err(tau.t().cpu().numpy(), c1["tau"]).max() < TOL64
    assert rel_err(V.t().cpu().numpy(), c1["twist6"], 1e-3).max() < TOL64
    assert rel_err(dV.t().cpu().numpy(), c1["dtwist6"], 1e-3).max() < TOL64


@pytest.mark.parametrize("n", [0, 1, 31, 127, 128, 129, 1000])
def test_ragged_sizes(n):
    g = load_golden("ref_inverse_uniform_gearbox.npz")
    m = model_from_golden(g)
    rng = np.random.default_rng(n)
    traj = sample_states(rng, n)
    ref = rv.inverse_batched(traj, g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"])["tau"] if n else np.zeros((0, 6))
    q, qd, qdd = soa(traj) if n else tuple(torch.empty((6, 0), dtype=torch.float64, device="cuda") for _ in range(3))
    tau = m.rnea(q, qd, qdd).t().cpu().numpy()
    tau_aos = m.rnea_aos(torch.as_tensor(traj, device="cuda").reshape(n, 3, 6)).cpu().numpy()
    if n:
        assert rel_err(tau, ref).max() < TOL64
        assert rel_err(tau_aos, ref).max() < TOL64
    else:
        assert tau.shape == (0, 6) and tau_aos.shape == (0, 6)


def test_config2_one_million_samples_fp64():
    """BASELINE.json config 2: 2^20 synthetic samples, fp64, every sample checked against the vectorised oracle."""
    g = load_golden("ref_inverse_hammer.npz")
    m = model_from_golden(g)
    n = 1 << 20
    traj = sample_states(np.random.default_rng(0), n)
    q, qd, qdd = soa(traj)
    tau = m.rnea(q, qd, qdd).t().cpu().numpy()
    worst = 0.0
    for s0 in range(0, n, 1 << 16):
        sl = slice(s0, s0 + (1 << 16))
        ref = rv.inverse_batched(traj[sl], g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"])["tau"]
        worst = max(worst, rel_err(tau[sl], ref).max())
    assert worst < TOL64, worst
    # size-independent property at full size: tau is affine in qdd  (tau(q,qd,2a) - tau(q,qd,a) == tau(q,qd,a) - tau(q,qd,0))
    t0 = m.rnea(q, qd, torch.zeros_like(qdd))
    t1 = m.rnea(q, qd, qdd)
    t2 = m.rnea(q, qd, 2 * qdd)
    lin = ((t2 - t1) - (t1 - t0)).abs().max().item()
    assert lin < 1e-9 * t1.abs().max().item()


def test_host_end_to_end_path():
    g = load_golden("ref_inverse_hammer.npz")
    m = model_from_golden(g)
    n = 300_000
    traj = sample_states(np.random.default_rng(5), n)
    tau_dev = m.rnea_aos(torch.as_tensor(traj, device="cuda")).cpu().numpy()
    tau_host = m.rnea_host(traj, chunk=65536)
    assert np.array_equal(tau_host, tau_dev)
    pinned = torch.as_tensor(traj).pin_memory()
    tau_p = m.rnea_host(pinned)
    assert np.array_equal(tau_p.numpy(), tau_dev)
    t32 = m.rnea_host(traj.astype(np.float32))
    assert rel_err(t32, tau_dev).max() < TOL32


def test_invalid_arguments_raise():
    g = load_golden("ref_inverse_hammer.npz")
    m = model_from_golden(g)
    q = torch.zeros((6, 4), dtype=torch.float64, device="cuda")
    with pytest.raises(ValueError):
        m.rnea(q, q, torch.zeros((6, 5), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        m.rnea(q.cpu(), q.cpu(), q.cpu())  # no CPU path
    with pytest.raises(ValueError):
        m.rnea(q.half(), q.half(), q.half())
    from rigid_body_manipulation_b200.engine import Model

    with pytest.raises(ValueError):
        Model(g["hposes_Rt"][:-1], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"])
    bad = g["simats"].copy()
    bad[3, 2, 2] = np.nan
    with pytest.raises(ValueError):
        Model(g["hposes_Rt"], bad, g["uscrews"], g["twist_0"], g["dtwist_0"])


@pytest.mark.parametrize("force_generic", [False, True])
def test_planned_trajectory_kernel_matches_config1(force_generic):
    """SURVEY.md 8(f) rank 1: the quintic planner evaluated in-kernel (no input traffic) reproduces the reference's planned
    trajectory (planners/joint_position_planner.py:86-131) and its feed-forward tau for all 1500 steps of base.yaml."""
    from rigid_body_manipulation_b200.planner import traj_5th_spline

    g = load_golden("ref_inverse_hammer.npz")
    c1 = load_golden("ref_config1_hammer.npz")
    pg = load_golden("ref_planner.npz")
    m = model_from_golden(g, force_generic=force_generic)
    plan = traj_5th_spline(pg["base_disp"], [1, 1, 1, 0, 0, 0], 0.002, int(pg["base_n_steps"]))
    tau, traj = m.rnea_planned(plan, want_traj=True)
    traj = traj.permute(2, 0, 1).cpu().numpy()  # (n, 3, 6)
    assert np.abs(traj - c1["traj"]).max() < 1e-11 * np.abs(c1["traj"]).max()
    assert rel_err(tau.t().cpu().numpy(), c1["tau"]).max() < TOL64
    # sub-sampled (every 10th step = the 50 fps frame grid of core/simulate.py:196) and fp32
    tau10 = m.rnea_planned(plan, n=150, step0=0, stride=10.0)
    assert rel_err(tau10.t().cpu().numpy(), c1["tau"][::10]).max() < TOL64
    tau32 = m.rnea_planned(plan, dtype=torch.float32)
    assert rel_err(tau32.t().cpu().numpy(), c1["tau"]).max() < TOL32  # the profile itself is evaluated in double in both modes


def test_fast_and_generic_kernels_agree_at_scale():
    """The structure-specialised kernel (snapped 0 / +-1 pattern, rigid-body inertia parameters) and the generic kernel (dense
    constants exactly as given) are two independent evaluations of the same model: 2^20 samples, agreement to round-off."""
    g = load_golden("ref_inverse_kill_la_kill.npz")  # strongly off-axis object
    fast, generic = model_from_golden(g), model_from_golden(g, force_generic=True)
    assert fast.kernel_path == "seq_iso" and generic.kernel_path == "generic"
    q, qd, qdd = soa(sample_states(np.random.default_rng(8), 1 << 20))
    a, b = fast.rnea(q, qd, qdd), generic.rnea(q, qd, qdd)
    scale = b.abs().amax(dim=0).clamp_min(1e-6)
    assert ((a - b).abs().amax(dim=0) / scale).max().item() < 1e-12


def test_rigid_variant_of_the_fast_path():
    """Same kinematic structure with non-isotropic link inertias selects the SEQ_RIGID kernel; checked against the C oracle."""
    from model_classes import rigid_link_simats
    from oracle import build_c
    from rigid_body_manipulation_b200.engine import Model

    g = load_golden("ref_inverse_hammer.npz")
    rng = np.random.default_rng(5)
    sim = rigid_link_simats(g["simats"], rng)  # links 1-5: offset centre of mass and a full inertia tensor (still physical rigid bodies)
    mdl = Model(g["hposes_Rt"], sim, g["uscrews"], g["twist_0"], g["dtwist_0"])
    assert mdl.kernel_path == "seq_rigid"
    traj = sample_states(rng, 5000)
    ref = build_c.inverse_batched_c(traj, g["hposes_Rt"], sim, g["uscrews"], g["twist_0"], g["dtwist_0"])
    q, qd, qdd = soa(traj)
    assert rel_err(mdl.rnea(q, qd, qdd).t().cpu().numpy(), ref).max() < TOL64
    # a model that breaks the structure (tilted home rotation) must fall back to the generic kernel, not be snapped
    h = g["hposes_Rt"].copy()
    th = 1e-6
    Rz = np.array([[np.cos(th), -np.sin(th), 0], [np.sin(th), np.cos(th), 0], [0, 0, 1]])
    h[2, :9] = (Rz @ h[2, :9].reshape(3, 3)).reshape(9)
    tilted = Model(h, g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"])
    assert tilted.kernel_path == "generic"
    ref = build_c.inverse_batched_c(traj, h, g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"])
    assert rel_err(tilted.rnea(q, qd, qdd).t().cpu().numpy(), ref).max() < TOL64


def test_extreme_inputs():
    """Huge joint angles exercise the slow (Payne-Hanek) path of the device sincos; non-finite inputs must propagate, not crash."""
    from oracle import build_c

    g = load_golden("ref_inverse_hammer.npz")
    m = model_from_golden(g)
    rng = np.random.default_rng(2)
    traj = sample_states(rng, 4096)
    traj[:, 0, 3:] = rng.uniform(-1, 1, (4096, 3)) * 10.0 ** rng.uniform(3, 9, (4096, 3))
    ref = build_c.inverse_batched_c(traj, g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"])
    q, qd, qdd = soa(traj)
    assert rel_err(m.rnea(q, qd, qdd).t().cpu().numpy(), ref).max() < TOL64
    traj[7, 0, 4] = np.inf
    traj[9, 2, 1] = np.nan
    q, qd, qdd = soa(traj)
    tau = m.rnea(q, qd, qdd).t().cpu().numpy()
    assert np.isnan(tau[7]).any() and np.isnan(tau[9]).any()
    keep = np.ones(4096, bool)
    keep[[7, 9]] = False
    assert rel_err(tau[keep], ref[keep]).max() < TOL64


def test_maximum_size_property_fp32():
    """Largest single-launch batch used in the configs[4] sweep that fits beside its outputs (2^28 fp32 samples = 25.8 GB of
    inputs): size-independent property -- tau is affine in qdd -- checked on the device, plus a spot parity check."""
    from oracle import build_c

    g = load_golden("ref_inverse_hammer.npz")
    m = model_from_golden(g)
    n = 1 << 28
    if torch.cuda.mem_get_info()[0] < 60e9:
        pytest.skip("not enough free HBM")
    gen = torch.Generator(device="cuda").manual_seed(7)
    q = torch.empty((6, n), dtype=torch.float32, device="cuda")
    q[:3] = torch.rand((3, n), generator=gen, device="cuda") * 4 - 1.5
    q[3:] = (torch.rand((3, n), generator=gen, device="cuda") * 2 - 1) * 6 * np.pi
    qd = torch.randn((6, n), generator=gen, device="cuda")
    qdd = torch.randn((6, n), generator=gen, device="cuda") * 3
    t1 = m.rnea(q, qd, qdd)
    idx = torch.randint(0, n, (4096,), device="cuda")
    traj = torch.stack([q[:, idx].t(), qd[:, idx].t(), qdd[:, idx].t()], dim=1).double().cpu().numpy()
    ref = build_c.inverse_batched_c(traj, g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"])
    assert rel_err(t1[:, idx].t().cpu().numpy(), ref).max() < TOL32
    last = torch.arange(n - 300, n, device="cuda")  # the ragged end of the grid
    trajl = torch.stack([q[:, last].t(), qd[:, last].t(), qdd[:, last].t()], dim=1).double().cpu().numpy()
    refl = build_c.inverse_batched_c(trajl, g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"])
    assert rel_err(t1[:, last].t().cpu().numpy(), refl).max() < TOL32
    qdd.mul_(2.0)
    t2 = m.rnea(q, qd, qdd)
    qdd.zero_()
    t0 = m.rnea(q, qd, qdd)
    lin = (t2 - t1).sub_(t1).add_(t0).abs_().amax().item()
    assert lin < 2e-4 * t1.abs().amax().item()


@pytest.mark.parametrize("n", [1024, 4096 + 77, 300_004, 1 << 20])
@pytest.mark.parametrize("no_tma", [False, True])
def test_fp32_soa_sizes_and_flags(n, no_tma):
    """fp32 SoA batches of several sizes / alignments (with and without RBM_FLAG_NO_TMA, which only affects the AoS and Gram
    kernels) against the fp64 C oracle at 1e-4; and the AoS entry point on the same data (TMA in / out when aligned)."""
    from oracle import build_c

    g = load_golden("ref_inverse_hammer.npz")
    m = model_from_golden(g, no_tma=no_tma)
    traj = sample_states(np.random.default_rng(n), n)
    ref = build_c.inverse_batched_c(traj, g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"])
    q, qd, qdd = soa(traj, torch.float32)
    tau = m.rnea(q, qd, qdd)
    assert rel_err(tau.t().cpu().numpy(), ref).max() < TOL32
    tau_tw, V, dV = m.rnea(q, qd, qdd, want_twists=True)
    assert torch.equal(tau, tau_tw)
    tw = rv.inverse_batched(traj, g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"])
    assert rel_err(V.t().cpu().numpy(), tw["twists"][:, 6]).max() < TOL32
    assert rel_err(dV.t().cpu().numpy(), tw["dtwists"][:, 6]).max() < TOL32
    tau_aos = m.rnea_aos(torch.as_tensor(traj, dtype=torch.float32, device="cuda"))
    assert rel_err(tau_aos.cpu().numpy(), ref).max() < TOL32
    tau_aos64 = m.rnea_aos(torch.as_tensor(traj, device="cuda"))
    assert rel_err(tau_aos64.cpu().numpy(), ref).max() < TOL64


def test_full_size_properties_of_configs1():
    """BASELINE configs[1] at its full size (2^20 samples, fp64) through properties that need no oracle run: tau is affine in qdd at
    fixed (q, qd) -- tau(qdd1 + qdd2) - tau(qdd1) - tau(qdd2) + tau(0) = 0 --, independent of the gantry positions (the rows the kernel
    never loads), and the SoA, AoS and host entry points agree on every sample."""
    g = load_golden("ref_inverse_hammer.npz")
    m = model_from_golden(g)
    n = 1 << 20
    traj = sample_states(np.random.default_rng(21), n)
    q, qd, qdd = soa(traj)
    z = torch.zeros_like(qdd)
    qdd2 = torch.roll(qdd, 1, dims=1)
    t12, t1, t2, t0 = m.rnea(q, qd, qdd + qdd2), m.rnea(q, qd, qdd), m.rnea(q, qd, qdd2), m.rnea(q, qd, z)
    resid = (t12 - t1 - t2 + t0).abs().max().item()
    assert resid < 1e-10 * t12.abs().max().item()
    moved = q.clone()
    moved[:3] += 7.25
    assert torch.equal(m.rnea(moved, qd, qdd), t1)                      # bit-identical: those rows are not read
    dev = torch.as_tensor(traj, device="cuda")
    assert rel_err(m.rnea_aos(dev).cpu().numpy(), t1.t().cpu().numpy()).max() < 1e-13
    host = m.rnea_host_soa(*(np.ascontiguousarray(traj[:, k, :].T) for k in range(3)))
    assert np.array_equal(host, t1.cpu().numpy())                       # same kernel behind the host entry


def test_generic_kernel_with_non_unit_screws_and_tiny_angles():
    """The generic kernels fold SE3.exp(-S q) . M into affine forms of (cos, sin, q) at model creation and carry no small-angle branch
    (csrc/rbm_model.cuh).  Screws outside the goldens -- rotation parts of norm 0.7, 1.9 and 1e-3, a rescaled pitch -- and states on both
    sides of liegroups' isclose(angle, 0) switch and far outside the trigonometric fast range, through the unrolled constant-bank kernel
    (SoA, nj = 6) and the run-time-loop kernel (AoS / full state), against the vectorised restatement of dynamics.py:109-157."""
    from rigid_body_manipulation_b200.engine import Model

    g = load_golden("ref_inverse_generic_nj6.npz")
    us = g["uscrews"].copy()
    us[0, 3:] *= 0.7
    us[2, 3:] *= 1.9
    us[2, :3] *= 0.4
    us[3, 3:] *= 1e-3
    rng = np.random.default_rng(11)
    n = 1000
    traj = np.stack([rng.uniform(-3, 3, (n, 6)), rng.standard_normal((n, 6)), rng.standard_normal((n, 6)) * 3], axis=1)
    traj[0] = 0.0
    traj[1, 0, :] = 1e-9
    traj[2, 0, :] = -2e-8
    traj[3, 0, :] = 50.0
    traj[4, 0, :] = -2.0e5  # beyond the fast range of the trigonometry
    m = Model(g["hposes_Rt"], g["simats"], us, g["twist_0"], g["dtwist_0"], wrench_tip=g["wrench_tip"], pose_tip_ee=g["pose_tip"], device=0)
    assert m.kernel_path == "generic"
    ref = rv.inverse_batched(traj, g["hposes_Rt"], g["simats"], us, g["twist_0"], g["dtwist_0"], wrench_tip=g["wrench_tip"], pose_tip_Rt=g["pose_tip"])
    q, qd, qdd = soa(traj)
    tau, V, dV = m.rnea(q, qd, qdd, want_twists=True)
    assert rel_err(tau.t().cpu().numpy(), ref["tau"]).max() < TOL64
    assert rel_err(V.t().cpu().numpy(), ref["twists"][:, 6]).max() < TOL64 and rel_err(dV.t().cpu().numpy(), ref["dtwists"][:, 6]).max() < TOL64
    full = m.rnea_full(torch.as_tensor(traj, device="cuda"))
    assert rel_err(full[0].cpu().numpy(), ref["tau"]).max() < TOL64
    assert np.abs(full[1].cpu().numpy() - ref["poses"]).max() < 1e-9
    assert rel_err(m.rnea(q.float(), qd.float(), qdd.float()).t().cpu().numpy()[:4], ref["tau"][:4]).max() < 1e-3
