"""-m gpu: every SoA entry point of the C ABI at a padded row pitch ld > n, called through raw pointers as in test_gpu_abi_raw.py.

engine.Model always passes ld = n, so a kernel that indexed a row by n instead of ld would pass the rest of the suite.  Here the input
padding holds NaN and the output padding a canary, for ld = n + 1 and ld = n + 64, on the fast model (hammer), the rigid-link /
off-axis-sensor class, and generic chains of 6 and 9 joints.  Three things hold for every case:
  * every padding element of every output still holds the canary;
  * the first n columns are bit-identical to the ld = n call when the same kernel runs; where the pitch changes the kernel
    (`_kernel` records which: the fp32 two-samples-per-thread RNEA needs an even pitch, the fp64 TMA Gram a 16-byte one) they agree
    with the oracle (1e-4 in fp32) or the materialised normal equations (1e-9), and the no-TMA model gives the ld = n bits again;
  * ld = n - 1 returns RBM_ERR_INVALID.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import chains
import model_classes
from gpu_util import load_golden, rel_err
from oracle import rnea_vec as rv
from rigid_body_manipulation_b200 import _lib, planner

pytestmark = pytest.mark.gpu
CANARY = -7.25
N = 1037               # odd: ld = n + 1 is even, ld = n + 64 odd
N_GRAM = 100_352 + 77  # 196 whole TMA tiles and a ragged tail
MODELS = ["hammer", "rigid_offset_sensor", "chain6", "chain9"]
DTYPES = {"f64": torch.float64, "f32": torch.float32}


def _model(name, no_tma=False):
    from rigid_body_manipulation_b200.engine import Model

    if name == "hammer":
        g = load_golden("ref_inverse_hammer.npz")
        args, kw, path = (g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"]), dict(pose_sen_llj=g["pose_sen_llj"]), "seq_iso"
    elif name in model_classes.CLASSES:
        mc = model_classes.build(name)
        (args, kw), path = mc.model_args(), mc.path
    else:
        (args, kw), path = chains.random_chain(int(name[5:]), seed=700).model_args(), "generic"
    m = Model(*args, **kw, no_tma=no_tma)
    assert m.kernel_path == path
    return m


def _traj(m, n, seed=0):
    if m.nj == 6 and m.kernel_path != "generic":
        return model_classes.sample_states(np.random.default_rng(seed), n)
    return chains.sample_traj(m.nj, n, seed)


def vp(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def pad_in(rows, ld, dtype):
    """(k, n) host rows -> device (k, ld) with NaN beyond column n."""
    rows = np.asarray(rows)
    b = torch.full((rows.shape[0], max(ld, rows.shape[1])), float("nan"), dtype=dtype, device="cuda")  # ld < n: rejected before use
    b[:, : rows.shape[1]] = torch.as_tensor(rows, dtype=dtype, device="cuda")
    return b


def pad_out(shape, dtype, device="cuda"):
    return torch.full(shape, CANARY, dtype=dtype, device=device)


def _kernel(entry, m, no_tma, n, ld, dt):
    """Which kernel the launcher picks, where the pitch takes part in the choice (csrc/rbm_rnea.cu, csrc/rbm_regressor.cu)."""
    fast = m.kernel_path != "generic"
    if entry == "rnea" and dt == "f32" and fast:
        return "f32x2" if ld % 2 == 0 else "scalar"
    if entry == "regressor_gram" and fast and not no_tma:
        return "tma" if (ld * (8 if dt == "f64" else 4)) % 16 == 0 and n >= 512 else "direct"
    return "one"


# ---- entry points: each takes (m, n, ld, dt) and returns (status, {name: output tensor whose last axis is the pitch}) --------------
def _soa_inputs(m, n, ld, dt, seed=0):
    tr = _traj(m, n, seed)
    return [pad_in(tr[:, k, :].T, ld, DTYPES[dt]) for k in range(3)], tr


def e_rnea(m, n, ld, dt):
    (q, qd, qdd), _ = _soa_inputs(m, n, ld, dt)
    o = {k: pad_out((r, ld), DTYPES[dt]) for k, r in (("tau", m.nj), ("V", 6), ("dV", 6))}
    fn = m._lib.rbm_rnea_f64 if dt == "f64" else m._lib.rbm_rnea_f32
    return fn(m._h, vp(q), vp(qd), vp(qdd), vp(o["tau"]), vp(o["V"]), vp(o["dV"]), n, ld, None), o


def _plan(m):
    rng = np.random.default_rng(m.nj)
    return planner.QuinticPlan(rng.uniform(-1, 1, m.nj), rng.uniform(-1, 1, m.nj), 0.002, 1500)


def _plan_args(m):
    p = _plan(m)
    return [np.ascontiguousarray(a, np.float64).ctypes.data_as(C.c_void_p) for a in (p.coeffs, p.displacement, p.pos_offset)], p


def e_rnea_planned(m, n, ld, dt):
    (co, di, of), p = _plan_args(m)
    o = {"tau": pad_out((m.nj, ld), DTYPES[dt]), "traj": pad_out((3 * m.nj, ld), DTYPES[dt])}
    fn = m._lib.rbm_rnea_planned_f64 if dt == "f64" else m._lib.rbm_rnea_planned_f32
    return fn(m._h, co, di, of, p.timestep, 5.0, 1.3, vp(o["tau"]), vp(o["traj"]), n, ld, None), o


def e_regressor_from_traj(m, n, ld, dt):
    (q, qd, qdd), _ = _soa_inputs(m, n, ld, dt)
    phi = torch.as_tensor(chains.phi_sensed(1), dtype=DTYPES[dt], device="cuda")
    o = {k: pad_out((6, ld), DTYPES[dt]) for k in ("Vs", "dVs", "wrench")}
    fn = m._lib.rbm_regressor_from_traj_f64 if dt == "f64" else m._lib.rbm_regressor_from_traj_f32
    return fn(m._h, vp(q), vp(qd), vp(qdd), None, vp(o["Vs"]), vp(o["dVs"]), vp(phi), vp(o["wrench"]), n, ld, None), o


def _ws(m, n):
    return torch.empty(max(1, int(m._lib.rbm_gram_workspace_bytes(m._h, n)) // 8), dtype=torch.float64, device="cuda")


def _gram_inputs(m, n, ld, dt, rows):
    (q, qd, qdd), tr = _soa_inputs(m, n, ld, dt, seed=n)
    y = np.random.default_rng(n).standard_normal((rows, n)) * 3
    return q, qd, qdd, pad_in(y, ld, DTYPES[dt]), tr, y


def e_regressor_gram(m, n, ld, dt):
    q, qd, qdd, f, _, _ = _gram_inputs(m, n, ld, dt, 6)
    o = {"pack": pad_out((112,), torch.float64)}
    ws = _ws(m, n)
    fn = m._lib.rbm_regressor_gram_f64 if dt == "f64" else m._lib.rbm_regressor_gram_f32
    return fn(m._h, vp(q), vp(qd), vp(qdd), vp(f), vp(o["pack"]), vp(ws), ws.numel() * 8, n, ld, None), o


def e_payload_regressor(m, n, ld, dt):
    (q, qd, qdd), _ = _soa_inputs(m, n, ld, dt)
    o = {"tau0": pad_out((m.nj, ld), DTYPES[dt])}
    fn = m._lib.rbm_payload_regressor_f64 if dt == "f64" else m._lib.rbm_payload_regressor_f32
    return fn(m._h, vp(q), vp(qd), vp(qdd), None, vp(o["tau0"]), n, ld, None), o


def e_payload_gram(m, n, ld, dt):
    q, qd, qdd, tau, _, _ = _gram_inputs(m, n, ld, dt, m.nj)
    o = {"pack": pad_out((112,), torch.float64)}
    ws = _ws(m, n)
    fn = m._lib.rbm_payload_gram_f64 if dt == "f64" else m._lib.rbm_payload_gram_f32
    return fn(m._h, vp(q), vp(qd), vp(qdd), vp(tau), vp(o["pack"]), vp(ws), ws.numel() * 8, n, ld, None), o


def e_linearize(m, n, ld, dt):
    (q, qd, _), _ = _soa_inputs(m, n, ld, dt)
    u = pad_in(np.random.default_rng(1).standard_normal((m.nj, n)) * 20, ld, torch.float64)
    nj = m.nj
    o = {"A": pad_out((4 * nj * nj, ld), torch.float64), "B": pad_out((2 * nj * nj, ld), torch.float64), "qdd": pad_out((nj, ld), torch.float64)}
    return m._lib.rbm_linearize_f64(m._h, vp(q), vp(qd), vp(u), 0.002, 1e-6, 1, vp(o["A"]), vp(o["B"]), vp(o["qdd"]), n, ld, None), o


def e_forward_dynamics(m, n, ld, dt):
    (q, qd, _), _ = _soa_inputs(m, n, ld, dt)
    u = pad_in(np.random.default_rng(1).standard_normal((m.nj, n)) * 20, ld, torch.float64)
    o = {k: pad_out((m.nj, ld), torch.float64) for k in ("qdd", "q_next", "qd_next")}
    return m._lib.rbm_forward_dynamics_f64(m._h, vp(q), vp(qd), vp(u), 0.002, vp(o["qdd"]), vp(o["q_next"]), vp(o["qd_next"]), n, ld, None), o


def e_closed_loop(m, n, ld, dt):
    nj = m.nj
    (co, di, of), p = _plan_args(m)
    rng = np.random.default_rng(2)
    q0 = pad_in(p.pos_offset[:, None] + rng.uniform(-0.05, 0.05, (nj, n)), ld, torch.float64)
    qd0 = pad_in(rng.uniform(-0.1, 0.1, (nj, n)), ld, torch.float64)
    K = torch.as_tensor(-np.hstack([50.0 * np.eye(nj), 5.0 * np.eye(nj)]), device="cuda")
    phi = torch.as_tensor(chains.phi_sensed(2), device="cuda")
    n_steps, max_frames = 60, 3
    o = {"frames": pad_out((max_frames, 3 * nj + 18, ld), torch.float64), "final": pad_out((3 * nj, ld), torch.float64)}
    fsteps = torch.full((max_frames,), -1, dtype=torch.int32, device="cuda")
    nfr = torch.zeros(1, dtype=torch.int32, device="cuda")
    rc = m._lib.rbm_closed_loop_f64(m._h, co, di, of, p.timestep, 0.0, n_steps, vp(K), vp(phi), 0.002, 50.0, float(nj), vp(q0), vp(qd0), vp(o["frames"]),
                                    max_frames, vp(fsteps), vp(nfr), vp(o["final"]), n, ld, None)
    return rc, o


def e_rnea_host_soa(m, n, ld, dt):
    npdt = np.float64 if dt == "f64" else np.float32
    tr = _traj(m, n)
    ins = []
    for k in range(3):
        a = np.full((m.nj, max(ld, n)), np.nan, npdt)
        a[:, :n] = tr[:, k, :].T
        ins.append(a)
    tau = np.full((m.nj, ld), CANARY, npdt)
    fn = m._lib.rbm_rnea_host_soa_f64 if dt == "f64" else m._lib.rbm_rnea_host_soa_f32
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    return fn(m._h, p(ins[0]), p(ins[1]), p(ins[2]), p(tau), n, ld, 256), {"tau": torch.as_tensor(tau)}


def e_rnea_planned_host(m, n, ld, dt):
    (co, di, of), p = _plan_args(m)
    tau = np.full((m.nj, ld), CANARY, np.float64 if dt == "f64" else np.float32)
    fn = m._lib.rbm_rnea_planned_host_f64 if dt == "f64" else m._lib.rbm_rnea_planned_host_f32
    return fn(m._h, co, di, of, p.timestep, 5.0, 1.3, tau.ctypes.data_as(C.c_void_p), n, ld, 256), {"tau": torch.as_tensor(tau)}


ENTRIES = {"rnea": (e_rnea, ("f64", "f32")), "rnea_planned": (e_rnea_planned, ("f64", "f32")),
           "regressor_from_traj": (e_regressor_from_traj, ("f64", "f32")), "regressor_gram": (e_regressor_gram, ("f64", "f32")),
           "payload_regressor": (e_payload_regressor, ("f64", "f32")), "payload_gram": (e_payload_gram, ("f64", "f32")),
           "linearize": (e_linearize, ("f64",)), "forward_dynamics": (e_forward_dynamics, ("f64",)), "closed_loop": (e_closed_loop, ("f64",)),
           "rnea_host_soa": (e_rnea_host_soa, ("f64", "f32")), "rnea_planned_host": (e_rnea_planned_host, ("f64", "f32"))}
GRAMS = ("regressor_gram", "payload_gram")


def _padding_intact(outs, n):
    for k, t in outs.items():
        if k != "pack":
            assert bool((t[..., n:] == CANARY).all()), k


def _gram_reference(m, n, dt):
    """The materialised normal equations of e_regressor_gram's inputs, in fp64 from the (rounded) inputs."""
    (_, _, _, _, tr, f) = _gram_inputs(m, n, n, dt, 6)
    if dt == "f32":
        tr, f = tr.astype(np.float32).astype(np.float64), f.astype(np.float32).astype(np.float64)
    out = rv.inverse_batched(tr, m.hposes_Rt, m.simats, m.uscrews, m.twist_0, m.dtwist_0, wrench_tip=m.wrench_tip, pose_tip_Rt=m.pose_tip)
    Vs, dVs = rv.sensor_frame_twists_batched(m.pose_sen, out["twists"][:, -1], out["dtwists"][:, -1])
    return rv.gram_pack(rv.regressor_batched(Vs, dVs), f.T)


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("entry", list(ENTRIES))
def test_padded_pitch(model, entry):
    fn, dts = ENTRIES[entry]
    n = N_GRAM if entry in GRAMS else N
    m, plain = _model(model), _model(model, no_tma=True)
    for dt in dts:
        rc, base = fn(m, n, n, dt)
        assert rc == 0, _lib.last_error()
        rc, base_plain = fn(plain, n, n, dt)
        assert rc == 0, _lib.last_error()
        for ld in (n + 1, n + 64):
            for mm, no_tma, ref in ((m, False, base), (plain, True, base_plain)):
                rc, outs = fn(mm, n, ld, dt)
                assert rc == 0, _lib.last_error()
                torch.cuda.synchronize()
                _padding_intact(outs, n)
                kernel = _kernel(entry, mm, no_tma, n, ld, dt)
                same = kernel == _kernel(entry, mm, no_tma, n, n, dt)
                for k, t in outs.items():
                    got, want = t[..., :n] if k != "pack" else t, ref[k][..., :n] if k != "pack" else ref[k]
                    if same:
                        assert torch.equal(got.cpu(), want.cpu()), (dt, ld, k, kernel)
                    elif entry == "rnea":   # fp32 two-samples-per-thread kernel: against the oracle on the rounded inputs
                        tr = _traj(mm, n).astype(np.float32).astype(np.float64)
                        o = rv.inverse_batched(tr, mm.hposes_Rt, mm.simats, mm.uscrews, mm.twist_0, mm.dtwist_0, wrench_tip=mm.wrench_tip,
                                               pose_tip_Rt=mm.pose_tip)
                        want_np = {"tau": o["tau"], "V": o["twists"][:, -1], "dV": o["dtwists"][:, -1]}[k]
                        assert rel_err(got.double().cpu().numpy().T, want_np).max() < 1e-4, (ld, k)
                    else:                   # TMA Gram at an aligned pitch: the materialised normal equations
                        want_np = _gram_reference(mm, n, dt)
                        g = got.cpu().numpy()
                        scale = np.abs(want_np[:100]).max()
                        tol = 1e-9 if dt == "f64" else 1e-4
                        assert g[111] == n and np.abs(g[:100] - want_np[:100]).max() < tol * scale
                        assert np.abs(g[100:111] - want_np[100:111]).max() < tol * max(np.abs(want_np[100:111]).max(), 1.0)
        rc, _ = fn(m, n, n - 1, dt)
        assert rc == _lib.RBM_ERR_INVALID, (entry, dt)


@pytest.mark.parametrize("model", ["hammer", "chain9"])
@pytest.mark.parametrize("ld,ld_out", [(37, 37), (38, 37), (101, 37), (37, 38), (37, 101), (101, 101)])
def test_padded_pitch_grouped_gram(model, ld, ld_out):
    """rbm_regressor_gram_grouped_f64: group pitch ld of the frame-major log and output pitch ld_out, each > n_groups or not."""
    m = _model(model)
    nj, F, G = m.nj, 12, 37
    tr = _traj(m, F * G, 3).reshape(F, G, 3, nj)
    f = np.random.default_rng(4).standard_normal((F, G, 6))
    x = torch.full((F, 3 * nj + 6, ld), float("nan"), dtype=torch.float64, device="cuda")   # one frame: q, qd, qdd, f rows
    x[:, : 3 * nj, :G] = torch.as_tensor(tr.transpose(0, 2, 3, 1).reshape(F, 3 * nj, G), device="cuda")
    x[:, 3 * nj:, :G] = torch.as_tensor(f.transpose(0, 2, 1), device="cuda")
    packs = pad_out((112, ld_out), torch.float64)
    fs = (3 * nj + 6) * ld
    base = x.data_ptr()
    row = lambda r: C.c_void_p(base + r * ld * 8)
    rc = m._lib.rbm_regressor_gram_grouped_f64(m._h, row(0), row(nj), row(2 * nj), row(3 * nj), fs, fs, F, vp(packs), G, ld, ld_out, None)
    assert rc == 0, _lib.last_error()
    torch.cuda.synchronize()
    assert bool((packs[:, G:] == CANARY).all())
    got = packs[:, :G].t().cpu().numpy()
    for g in (0, 18, G - 1):
        o = rv.inverse_batched(tr[:, g], m.hposes_Rt, m.simats, m.uscrews, m.twist_0, m.dtwist_0)
        Vs, dVs = rv.sensor_frame_twists_batched(m.pose_sen, o["twists"][:, -1], o["dtwists"][:, -1])
        want = rv.gram_pack(rv.regressor_batched(Vs, dVs), f[:, g])
        assert np.abs(got[g] - want).max() < 1e-9 * np.abs(want).max()
    # bit-identical to the unpadded call
    dense = x[:, :, :G].contiguous()
    p2 = pad_out((112, G), torch.float64)
    b2 = dense.data_ptr()
    row2 = lambda r: C.c_void_p(b2 + r * G * 8)
    fs2 = (3 * nj + 6) * G
    assert m._lib.rbm_regressor_gram_grouped_f64(m._h, row2(0), row2(nj), row2(2 * nj), row2(3 * nj), fs2, fs2, F, vp(p2), G, G, G, None) == 0
    assert torch.equal(p2, packs[:, :G])
    bad = (G - 1, ld_out) if ld == G else (ld, G - 1)
    if ld == G or ld_out == G:
        assert m._lib.rbm_regressor_gram_grouped_f64(m._h, row(0), row(nj), row(2 * nj), row(3 * nj), fs, fs, F, vp(packs), G, *bad, None) == _lib.RBM_ERR_INVALID
