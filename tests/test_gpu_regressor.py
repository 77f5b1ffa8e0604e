"""-m gpu parity of the sensor-frame regressor, the fused Gram accumulation and the identification they feed
(reference core/simulate.py:202-224, dynamics/dynamics.py:215-249, loggers/loggers.py:127-129)."""
import numpy as np
import pytest
import torch

from gpu_util import load_golden, model_from_golden, rel_err, sample_states, soa
from oracle import rnea_vec as rv
from rigid_body_manipulation_b200 import engine, identification

pytestmark = pytest.mark.gpu
ALL = ["ref_inverse_hammer.npz", "ref_inverse_uniform_gearbox.npz", "ref_inverse_kill_la_kill.npz", "ref_inverse_generic_nj6.npz",
       "ref_inverse_generic_nj4.npz", "ref_inverse_generic_nj9.npz"]


@pytest.mark.parametrize("fname", ALL)
def test_regressor_rows_and_sensor_twists_from_given_twists(fname):
    g = load_golden(fname)
    nj = g["uscrews"].shape[0]
    Vs, dVs = engine.sensor_twists(g["pose_sen_llj"], g["twists"][:, nj], g["dtwists"][:, nj])
    assert rel_err(Vs.cpu().numpy(), g["twist_sen"]).max() < 1e-12
    assert rel_err(dVs.cpu().numpy(), g["dtwist_sen"]).max() < 1e-12
    Y = engine.regressor_rows(g["twist_sen"], g["dtwist_sen"])
    assert rel_err(Y.cpu().numpy(), g["regressor"]).max() < 1e-13


@pytest.mark.parametrize("fname", ALL)
@pytest.mark.parametrize("force_generic", [False, True])
def test_fused_regressor_from_trajectory(fname, force_generic):
    g = load_golden(fname)
    m = model_from_golden(g, force_generic=force_generic)
    q, qd, qdd = soa(g["traj"])
    phi = np.array([1.3, 0.1, -0.2, 0.3, 0.02, 0.03, 0.04, 0.001, -0.002, 0.003])
    out = m.regressor_from_traj(q, qd, qdd, want_rows=True, want_twists=True, phi=phi)
    assert rel_err(out["twist_sen"].t().cpu().numpy(), g["twist_sen"]).max() < 1e-9
    assert rel_err(out["dtwist_sen"].t().cpu().numpy(), g["dtwist_sen"]).max() < 1e-9
    assert rel_err(out["Y"].cpu().numpy(), g["regressor"]).max() < 1e-9
    assert rel_err(out["wrench"].t().cpu().numpy(), g["regressor"] @ phi).max() < 1e-9
    # fp32 mode
    q32, qd32, qdd32 = soa(g["traj"], torch.float32)
    o32 = m.regressor_from_traj(q32, qd32, qdd32, want_rows=True, want_twists=True, phi=phi)
    assert rel_err(o32["Y"].cpu().numpy(), g["regressor"]).max() < 1e-4
    assert rel_err(o32["twist_sen"].t().cpu().numpy(), g["twist_sen"]).max() < 1e-4
    assert rel_err(o32["dtwist_sen"].t().cpu().numpy(), g["dtwist_sen"]).max() < 1e-4
    assert rel_err(o32["wrench"].t().cpu().numpy(), g["regressor"] @ phi).max() < 1e-4


@pytest.mark.parametrize("n", [4096, 262_144 + 256 * 5 + 100])
def test_gram_fp32_mode(n):
    """The fast model (TMA and direct-load fp32 kernels) and a generic six-joint model (k_regressor_gram<float, PATH_GENERIC>)."""
    rng = np.random.default_rng(n)
    traj = sample_states(rng, n)
    f = rng.standard_normal((n, 6)) * np.array([5, 5, 5, 1, 1, 1.0])
    q, qd, qdd = soa(traj, torch.float32)
    fd = torch.as_tensor(f, dtype=torch.float32, device="cuda").t().contiguous()
    for fname, path in (("ref_inverse_hammer.npz", "seq_iso"), ("ref_inverse_generic_nj6.npz", "generic")):
        g = load_golden(fname)
        _, ref = _gram_reference(g, traj, f)
        for no_tma in (False, True):
            m = model_from_golden(g, no_tma=no_tma)
            assert m.kernel_path == path
            pack = m.regressor_gram(q, qd, qdd, fd).cpu().numpy()
            assert np.abs(pack[:100] - ref[:100]).max() < 1e-4 * np.abs(ref[:100]).max()
            assert np.abs(pack[100:110] - ref[100:110]).max() < 1e-4 * np.abs(ref[:100]).max()
            assert pack[111] == n


def _gram_reference(g, traj, f):
    nj = g["uscrews"].shape[0]
    kw = dict(wrench_tip=g["wrench_tip"], pose_tip_Rt=g["pose_tip"]) if "wrench_tip" in g.files else {}
    out = rv.inverse_batched(traj, g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"], **kw)
    Vs, dVs = rv.sensor_frame_twists_batched(g["pose_sen_llj"], out["twists"][:, nj], out["dtwists"][:, nj])
    Y = rv.regressor_batched(Vs, dVs)
    return Y, rv.gram_pack(Y, f)


@pytest.mark.parametrize("fname", ["ref_inverse_hammer.npz", "ref_inverse_generic_nj6.npz", "ref_inverse_generic_nj9.npz"])
@pytest.mark.parametrize("n", [1, 255, 766, 1_026, 4096, 100_003, 100_352, 300_002])
@pytest.mark.parametrize("no_tma", [False, True])
def test_gram_matches_materialised_normal_equations(fname, n, no_tma):
    """Aligned batches of >= 512 samples on the fast path take the TMA-pipelined kernel (512-sample tiles, two samples per thread:
    4096 and 100_352 are whole tiles; 766 has one tile + a 254-sample tail (first half-tile only), 1_026 two tiles + 2 samples,
    300_002 a 482-sample tail (both half-tiles)); odd n (row pitch not 16-byte aligned), tiny n, generic models and no_tma=True take
    the direct-load kernel.  Both must agree with the materialised normal equations."""
    g = load_golden(fname)
    m = model_from_golden(g, no_tma=no_tma)
    nj = m.nj
    rng = np.random.default_rng(n)
    traj = sample_states(rng, n) if nj == 6 else np.stack([rng.uniform(-3, 3, (n, nj)), rng.standard_normal((n, nj)), rng.standard_normal((n, nj))], 1)
    f = rng.standard_normal((n, 6)) * np.array([5, 5, 5, 1, 1, 1.0])
    Y, ref = _gram_reference(g, traj, f)
    q, qd, qdd = soa(traj)
    fd = torch.as_tensor(f, device="cuda").t().contiguous()
    pack = m.regressor_gram(q, qd, qdd, fd).cpu().numpy()
    scale = np.abs(ref[:100]).max()
    assert np.abs(pack[:100] - ref[:100]).max() < 1e-9 * scale
    assert np.abs(pack[100:110] - ref[100:110]).max() < 1e-9 * max(np.abs(ref[100:110]).max(), 1.0)
    assert abs(pack[110] - ref[110]) < 1e-9 * ref[110]
    assert pack[111] == n
    # bit-reproducible (fixed reduction order, no atomics)
    assert np.array_equal(pack, m.regressor_gram(q, qd, qdd, fd).cpu().numpy())
    # symmetric by construction
    G = pack[:100].reshape(10, 10)
    assert np.array_equal(G, G.T)


def test_gram_empty_batch():
    g = load_golden("ref_inverse_hammer.npz")
    m = model_from_golden(g)
    e = torch.empty((6, 0), dtype=torch.float64, device="cuda")
    pack = m.regressor_gram(e, e, e, e).cpu().numpy()
    assert not pack.any()


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-8), (torch.float32, 2e-3)])
def test_identification_recovers_object_parameters(dtype, tol):
    """Exact-recovery property at scale (config-3 shaped, one shard): f = Y phi_true synthesised on the device, Gram
    accumulated over 2^21 samples, 10x10 solve on the host -> phi_true; and agreement with np.linalg.lstsq on a subset."""
    g = load_golden("ref_inverse_uniform_gearbox.npz")
    m = model_from_golden(g)
    n = 1 << 21
    rng = np.random.default_rng(42)
    traj = sample_states(rng, n)
    q, qd, qdd = soa(traj, dtype)
    phi_true = np.array([0.585, -0.0032, 1.9e-5, -8e-6, 3.85e-4, 2.9e-4, 3.0e-4, 1e-6, 2e-6, -1e-6]) * np.array([1, 1, 1, 1, 10, 10, 10, 10, 10, 10])
    f = m.regressor_from_traj(q, qd, qdd, want_rows=False, phi=phi_true)["wrench"]
    ident = identification.solve(m.regressor_gram(q, qd, qdd, f))
    assert ident.n_samples == n and ident.rank == 10
    err = np.abs(ident.phi - phi_true) / np.array([1, 1e-2, 1e-2, 1e-2, 1e-3, 1e-3, 1e-3, 1e-3, 1e-3, 1e-3])
    assert err.max() < tol, (ident.phi, phi_true)
    if dtype == torch.float64:
        assert ident.residual_ss < 1e-12 * ident.f_ss
        sub = 20000
        out = rv.inverse_batched(traj[:sub], g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"])
        Vs, dVs = rv.sensor_frame_twists_batched(g["pose_sen_llj"], out["twists"][:, 6], out["dtwists"][:, 6])
        Y = rv.regressor_batched(Vs, dVs)
        noise = np.random.default_rng(0).standard_normal((sub, 6)) * 0.05
        fn = Y @ phi_true + noise
        ref = rv.identify_lstsq(Y, fn)  # the reference's solver (loggers.py:129)
        fd = torch.as_tensor(fn, device="cuda").t().contiguous()
        got = identification.solve(m.regressor_gram(q[:, :sub].contiguous(), qd[:, :sub].contiguous(), qdd[:, :sub].contiguous(), fd))
        assert np.abs(got.phi - ref).max() < 1e-9 * max(1.0, got.cond ** 0.5)


def test_gram_linearity_checksum_at_full_size():
    """Size-independent property at config-3 per-rank size (1.25e7 samples): the pack is additive over a split of the batch."""
    g = load_golden("ref_inverse_hammer.npz")
    m = model_from_golden(g)
    n = 12_500_000
    gen = torch.Generator(device="cuda").manual_seed(1234)
    q = torch.empty((6, n), dtype=torch.float64, device="cuda")
    q[:3] = torch.rand((3, n), generator=gen, device="cuda", dtype=torch.float64) * 4 - 1.5
    q[3:] = (torch.rand((3, n), generator=gen, device="cuda", dtype=torch.float64) * 2 - 1) * 6 * np.pi
    qd = torch.randn((6, n), generator=gen, device="cuda", dtype=torch.float64)
    qdd = torch.randn((6, n), generator=gen, device="cuda", dtype=torch.float64) * 3
    f = torch.randn((6, n), generator=gen, device="cuda", dtype=torch.float64)
    whole = m.regressor_gram(q, qd, qdd, f).clone()
    cut = 5_000_011
    a = m.regressor_gram(q[:, :cut].contiguous(), qd[:, :cut].contiguous(), qdd[:, :cut].contiguous(), f[:, :cut].contiguous()).clone()
    b = m.regressor_gram(q[:, cut:].contiguous(), qd[:, cut:].contiguous(), qdd[:, cut:].contiguous(), f[:, cut:].contiguous()).clone()
    diff = (whole - (a + b)).abs().max().item()
    assert diff < 1e-10 * whole.abs().max().item()
    assert whole[111].item() == n


def test_config1_identification_pipeline():
    """The reference's end-of-run identification (loggers.py:110-156) on the open-loop config-1 data: regressors at the 151 frame
    steps of the base.yaml trajectory, wrench = Y phi + the reference's 5 % noise, lstsq on all / train / valid / test."""
    g = load_golden("ref_inverse_hammer.npz")
    c1 = load_golden("ref_config1_hammer.npz")
    m = model_from_golden(g)
    steps = c1["frame_steps"]
    traj = c1["traj"][steps]
    Y = c1["regressor_frames"]
    # ground truth of the object in the sensor frame from the folded inertia
    from rigid_body_manipulation_b200 import model as rbm_model

    c = rbm_model.load_packaged("sequential", "hammer")
    phi_true = identification.sensor_frame_params(c.target, c.pose_sen_obj_Rt)
    f_clean = Y @ phi_true
    f_noisy = identification.perturb_wrench(f_clean)
    q, qd, qdd = soa(traj)
    fd = torch.as_tensor(f_noisy, device="cuda").t().contiguous()
    res = identification.identify_splits(m, q, qd, qdd, fd)
    tr, va, te = identification.split_indices(len(steps))
    for name, idx in (("all", np.arange(len(steps))), ("train", tr), ("valid", va), ("test", te)):
        ref = rv.identify_lstsq(Y[idx], f_noisy[idx])  # np.linalg.lstsq on the stacked regressor (loggers.py:127-129)
        got = res[name]
        assert got.n_samples == len(idx)
        # normal equations square the condition number: agreement scales with cond * eps
        assert np.abs(got.phi - ref).max() < 1e-8 * max(1.0, np.abs(ref).max()) * max(1.0, got.cond * 1e-6), (name, got.cond)
    assert np.array_equal(res["valid"].phi, res["test"].phi)
    # noise-free: exact recovery of the CAD parameters expressed in the sensor frame
    clean = identification.solve(m.regressor_gram(q, qd, qdd, torch.as_tensor(f_clean, device="cuda").t().contiguous()))
    assert np.abs(clean.phi - phi_true).max() < 1e-6 * max(1.0, clean.cond * 1e-6)


def test_per_object_grams_for_all_packaged_targets():
    """SURVEY.md 8(f) rank 2 / north star "10x10 per object": one model per target object (all 23 CAD rows), one Gram pack per
    object stacked as (23, 112), identified in one go; every object's sensor-frame parameters are recovered from noise-free data."""
    from rigid_body_manipulation_b200 import model as rbm_model
    from rigid_body_manipulation_b200.engine import Model

    names = sorted(rbm_model.packaged_targets())
    assert len(names) == 23
    n = 20_000
    q, qd, qdd = soa(sample_states(np.random.default_rng(77), n))
    packs = torch.empty((len(names), 112), dtype=torch.float64, device="cuda")
    truths = []
    for k, name in enumerate(names):
        c = rbm_model.load_packaged("sequential", name)
        m = Model(c.hposes_Rt, c.simats, c.uscrews, c.twist_0, c.dtwist_0, pose_sen_llj=c.pose_sen_Rt)
        assert m.kernel_path == "seq_iso"
        # the wrench the object loads the sensor with: its own inertia (the reference's diag-inertia recipe) seen from the sensor frame
        T = np.eye(4)
        T[:3, :3], T[:3, 3] = c.pose_sen_Rt[:9].reshape(3, 3), c.pose_sen_Rt[9:]
        G = rbm_model.move_inertia(T, c.simat_object_llj)
        phi = np.array([G[0, 0], G[5, 1], G[3, 2], G[4, 0], G[3, 3], G[4, 4], G[5, 5], G[3, 4], G[4, 5], G[5, 3]])
        truths.append(phi)
        f = m.regressor_from_traj(q, qd, qdd, want_rows=False, phi=phi)["wrench"]
        m.regressor_gram(q, qd, qdd, f, pack=packs[k])
    from rigid_body_manipulation_b200 import distributed

    distributed.allreduce_gram(packs)  # grouped form; a no-op on one rank
    res = identification.solve_many(packs)
    for name, r, phi in zip(names, res, truths):
        assert r.rank == 10 and r.n_samples == n, name
        scale = np.array([phi[0]] * 4 + [max(np.abs(phi[4:]).max(), 1e-12)] * 6)
        assert (np.abs(r.phi - phi) / scale).max() < 1e-7, (name, r.phi, phi)


@pytest.mark.parametrize("n", [100, 256, 4096, 262_144 + 256 * 5 + 100, 2_100_000])
def test_gram_fp32_on_the_tensor_cores(n):
    """RBM_FLAG_GRAM_TENSOR_CORES (csrc/rbm_gram_tc.cu): second moments of the 18 regressor features through tcgen05.mma kind::tf32
    with an exact hi/lo operand split, accumulator in TMEM, flushed to fp64 every 2048 samples.  Same bar as the register fp32 kernel
    (1e-4 of the largest entry, north_star's fp32 tolerance); ragged tails, sub-tile batches and multi-tile-per-CTA sizes."""
    g = load_golden("ref_inverse_hammer.npz")
    rng = np.random.default_rng(n)
    traj = sample_states(rng, n)
    f = rng.standard_normal((n, 6)) * np.array([5, 5, 5, 1, 1, 1.0])
    _, ref = _gram_reference(g, traj, f)
    q, qd, qdd = soa(traj, torch.float32)
    fd = torch.as_tensor(f, dtype=torch.float32, device="cuda").t().contiguous()
    m = model_from_golden(g, gram_tensor_cores=True)
    pack = m.regressor_gram(q, qd, qdd, fd).cpu().numpy()
    scale = np.abs(ref[:100]).max()
    assert np.abs(pack[:100] - ref[:100]).max() < 1e-4 * scale
    assert np.abs(pack[100:110] - ref[100:110]).max() < 1e-4 * scale
    assert abs(pack[110] - ref[110]) < 1e-4 * ref[110]
    assert pack[111] == n
    G = pack[:100].reshape(10, 10)
    assert np.array_equal(G, G.T)
    assert np.array_equal(pack, m.regressor_gram(q, qd, qdd, fd).cpu().numpy())  # fixed reduction order here too
    # the register fp32 kernel on the same data: the two fp32 modes agree to well inside the bar
    reg = model_from_golden(g).regressor_gram(q, qd, qdd, fd).cpu().numpy()
    assert np.abs(pack[:111] - reg[:111]).max() < 5e-5 * scale


def test_tensor_core_gram_identifies_like_the_register_kernel():
    """TF32 characterisation on phi-hat (VERDICT r1 item 4c): exact-recovery data, 2^21 samples; the estimate from the tensor-core
    Gram against the one from the register fp32 Gram and against the truth."""
    g = load_golden("ref_inverse_uniform_gearbox.npz")
    n = 1 << 21
    traj = sample_states(np.random.default_rng(42), n)
    q, qd, qdd = soa(traj, torch.float32)
    phi_true = np.array([0.585, -0.0032, 1.9e-5, -8e-6, 3.85e-3, 2.9e-3, 3.0e-3, 1e-5, 2e-5, -1e-5])
    scale = np.array([1, 1e-2, 1e-2, 1e-2, 1e-3, 1e-3, 1e-3, 1e-3, 1e-3, 1e-3])
    est = {}
    for name, kw in (("tc", dict(gram_tensor_cores=True)), ("reg", {})):
        m = model_from_golden(g, **kw)
        f = m.regressor_from_traj(q, qd, qdd, want_rows=False, phi=phi_true)["wrench"]
        est[name] = identification.solve(m.regressor_gram(q, qd, qdd, f))
        assert est[name].rank == 10
        assert (np.abs(est[name].phi - phi_true) / scale).max() < 2e-3
    assert (np.abs(est["tc"].phi - est["reg"].phi) / scale).max() < 2e-3


@pytest.mark.parametrize("dtype,tc,tol", [(torch.float64, False, 1e-12), (torch.float32, False, 2e-6), (torch.float32, True, 5e-5)])
def test_gram_is_additive_at_the_configs2_size(dtype, tc, tol):
    """BASELINE configs[2] per-GPU share (12.5 M samples), size-independent properties: the pack of the whole batch equals the sum of the
    packs of its two halves (what the multi-GPU all-reduce relies on), the sample count is exact, and a batch that is the same 4096
    samples repeated gives 3052 x the pack of one copy (+ the ragged remainder), so every tile of the persistent grid is accounted for."""
    g = load_golden("ref_inverse_uniform_gearbox.npz")
    m = model_from_golden(g, gram_tensor_cores=tc)
    n = 12_500_000
    gen = torch.Generator(device="cuda").manual_seed(7)
    q = (torch.rand((6, n), generator=gen, device="cuda", dtype=dtype) * 2 - 1) * 6
    qd = torch.randn((6, n), generator=gen, device="cuda", dtype=dtype)
    qdd = torch.randn((6, n), generator=gen, device="cuda", dtype=dtype) * 3
    f = torch.randn((6, n), generator=gen, device="cuda", dtype=dtype) * 2
    whole = m.regressor_gram(q, qd, qdd, f).cpu().numpy()
    h = 6_250_240  # a multiple of 256 so that both halves stay on the TMA path (16-byte aligned row starts)
    halves = sum(m.regressor_gram(*(t[:, a:b].contiguous() for t in (q, qd, qdd, f))).cpu().numpy() for a, b in ((0, h), (h, n)))
    scale = np.abs(whole[:100]).max()
    assert whole[111] == n and halves[111] == n
    assert np.abs(whole[:111] - halves[:111]).max() < tol * scale
    # periodic batch: 4096 distinct samples tiled over the whole 12.5 M
    reps, rem = divmod(n, 4096)
    tile = lambda t: t[:, :4096].repeat(1, reps + 1)[:, :n].contiguous()
    per = m.regressor_gram(tile(q), tile(qd), tile(qdd), tile(f)).cpu().numpy()
    one = m.regressor_gram(*(t[:, :4096].contiguous() for t in (q, qd, qdd, f))).cpu().numpy()
    tail = m.regressor_gram(*(t[:, :rem].contiguous() for t in (q, qd, qdd, f))).cpu().numpy() if rem else 0.0
    expect = reps * one + tail
    assert np.abs(per[:111] - expect[:111]).max() < max(tol, 1e-11) * np.abs(expect[:100]).max() * (50 if dtype == torch.float32 else 1)
