"""ORACLE / TEST INFRASTRUCTURE ONLY -- never imported by the product package.

CPU restatement of what the reference's `StateSpace.update_matrices` (reference dynamics/dynamics.py:41-46) asks of
MuJoCo: `mjd_transitionFD(m, d, eps, centered, A, B, C, D)` -- finite differences of the ONE-STEP TRANSITION
x+ = f(x, u) of the simulated plant, literally: perturb one state / control element by +-eps, take a full step,
difference the next states.  MuJoCo 3.3.0 (pinned in the reference's uv.lock:1131-1132) is absent from the image,
so its published algorithm is restated for the reference's plant (sequential.xml: nv = nu = 6, na = 0, unit-gear
motors `sequential.xml:42-49`, no damping / armature / friction / contacts, default semi-implicit Euler integrator,
timestep 0.002):

    qacc = M(q)^-1 (ctrl - qfrc_bias(q, qvel)),   qvel+ = qvel + dt qacc,   qpos+ = qpos + dt qvel+
    A[:, i] = (f(x + eps e_i, u) - f(x - eps e_i, u)) / (2 eps)        (centred; forward differences otherwise)
    B[:, k] = (f(x, u + eps e_k) - f(x, u - eps e_k)) / (2 eps)

with x = [qpos; qvel] (slide / hinge joints: mj_integratePos / mj_differentiatePos are plain + and -).  The forward
dynamics is built from the vectorised inverse-dynamics oracle (oracle/rnea_vec.py): M column by column with the base
acceleration switched off, bias = ID(q, qd, 0).  C and D (sensor Jacobians, dynamics.py:35-36) are not consumed by
any caller (controllers/lqr.py:48-49 uses A and B only) and are not restated.

Parity unpinned against MuJoCo itself (cannot be executed here); the CUDA kernel differentiates the INVERSE dynamics
instead (one factorisation per state), so agreement with this literal restatement is a genuine cross-check.
"""
from __future__ import annotations

import numpy as np

from . import rnea_vec as rv


def tip_kw(consts):
    """The optional tip load of `consts` ("wrench_tip", "pose_tip_Rt", as in rbm_model_create) as keyword arguments of
    rnea_vec.inverse_batched; empty when the model has none."""
    return {k: consts[k] for k in ("wrench_tip", "pose_tip_Rt") if consts.get(k) is not None}


def _id(consts, q, qd, qdd, gravity=True):
    """Inverse dynamics; gravity=False switches off the base motion AND the tip wrench, so that ID(q, 0, e_j) is column j of M.
    The tip wrench is a constant external load: it belongs to the bias h, never to M."""
    traj = np.stack([q, qd, qdd], axis=1)
    dtw0 = consts["dtwist_0"] if gravity else np.zeros(6)
    tw0 = consts["twist_0"] if gravity else np.zeros(6)
    kw = tip_kw(consts) if gravity else {}
    return rv.inverse_batched(traj, consts["hposes_Rt"], consts["simats"], consts["uscrews"], tw0, dtw0, **kw)["tau"]


def mass_matrix(consts, q):
    """(B, nj) -> (B, nj, nj): column j = ID(q, 0, e_j) without gravity."""
    B, nj = q.shape
    M = np.zeros((B, nj, nj))
    z = np.zeros_like(q)
    for j in range(nj):
        e = np.zeros_like(q)
        e[:, j] = 1.0
        M[:, :, j] = _id(consts, q, z, e, gravity=False)
    return M


def forward_dynamics(consts, q, qd, u):
    M = mass_matrix(consts, q)
    h = _id(consts, q, qd, np.zeros_like(q))
    return np.linalg.solve(M, (u - h)[..., None])[..., 0]


def step(consts, q, qd, u, dt):
    qacc = forward_dynamics(consts, q, qd, u)
    qd1 = qd + dt * qacc
    q1 = q + dt * qd1
    return np.concatenate([q1, qd1], axis=1)


def transition_fd(consts, q, qd, u=None, dt=0.002, eps=1e-8, centered=True):
    """Batched mjd_transitionFD: q, qd, u (B, nj) -> A (B, 2nj, 2nj), B (B, 2nj, nj)."""
    q, qd = np.asarray(q, float), np.asarray(qd, float)
    Bn, nj = q.shape
    u = np.zeros_like(q) if u is None else np.asarray(u, float)
    A = np.zeros((Bn, 2 * nj, 2 * nj))
    Bm = np.zeros((Bn, 2 * nj, nj))
    y0 = None if centered else step(consts, q, qd, u, dt)
    for i in range(2 * nj):
        dq = np.zeros_like(q)
        dv = np.zeros_like(q)
        (dq if i < nj else dv)[:, i % nj] = eps
        yp = step(consts, q + dq, qd + dv, u, dt)
        if centered:
            ym = step(consts, q - dq, qd - dv, u, dt)
            A[:, :, i] = (yp - ym) / (2 * eps)
        else:
            A[:, :, i] = (yp - y0) / eps
    for k in range(nj):
        du = np.zeros_like(q)
        du[:, k] = eps
        yp = step(consts, q, qd, u + du, dt)
        if centered:
            ym = step(consts, q, qd, u - du, dt)
            Bm[:, :, k] = (yp - ym) / (2 * eps)
        else:
            Bm[:, :, k] = (yp - y0) / eps
    return A, Bm
