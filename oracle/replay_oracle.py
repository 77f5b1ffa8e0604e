"""ORACLE / TEST INFRASTRUCTURE ONLY -- never imported by the product package.

CPU restatement of the reference's closed-loop main loop, core/simulate.py:185-270, on the plant of oracle/lqr_oracle.py.
PINNED against the reference's own `simulate()` executed unmodified on the functional MuJoCo stand-in (oracle/mujoco_standin.py;
tests/test_reference_simulate.py: agreement to 1e-14 on every logged quantity).  MuJoCo 3.3.0 itself is absent, so the pieces of
MuJoCo's published behaviour that the stand-in and this file share (listed below) remain UNPINNED against MuJoCo.  Line by line:

  :186-188  tgt_traj = planner.plan(step); tgt_ctrl = inverse(tgt_traj)[0]
  :191-194  act_traj = (d.qpos, d.qvel, d.qacc)   -- qacc is what the PREVIOUS mj_step's forward pass left in `d`, i.e. it belongs
            to the previous state; twists / dtwists of the last link from inverse(act_traj)
  :196-226  every frame (`frame_count <= d.time * fps`): sensor-frame twists (:202-209), F/T reading from d.sensordata (:218-221,
            also left by the previous forward pass), regressor (:223)
  :257-268  res_qpos = mj_differentiatePos(m, res, m.nu, qpos, tgt_q) = (tgt_q - qpos) / nu   (the `dt` slot receives m.nu = 6);
            res_state = [res_qpos, tgt_qd - qvel];  ctrl = tgt_ctrl - K res_state
  :270      mj_step: forward pass at (qpos, qvel, ctrl) -> qacc, sensors; semi-implicit Euler; time += timestep

MuJoCo pieces restated: (1) the plant of lqr_oracle.py; (2) force / torque sensors on the site of body "target/"
(core/core.py:241-259): mj_sensorAcc reports cfrc_int of that body -- the Newton-Euler wrench the parent applies to the subtree
(attachment body + object), with gravity entering as the world's fictitious acceleration exactly like dtwist_0 -- expressed in the
site frame:  F = G_s dV_s - ad(V_s)^T G_s V_s  with G_s the subtree's spatial inertia in the sensor frame;  (3) the values left in
`d.qacc` / `d.sensordata` before the first step by the controller's mjd_transitionFD are taken as those of a forward pass at the
keyframe with ctrl = 0 (they differ from MuJoCo's leftovers by the O(eps = 1e-8) state perturbation of its last FD evaluation).
"""
from __future__ import annotations

import numpy as np

from . import lqr_oracle as lo
from . import rnea_vec as rv


def sensor_inertia(simat_object_llj, pose_sen_Rt):
    """Spatial inertia of the sensed subtree in the sensor frame from its inertia in link 6's joint frame."""
    p = np.asarray(pose_sen_Rt, float)  # T_{sen,llj}
    R, t = p[:9].reshape(3, 3), p[9:]
    Ad_inv = rv.adjoint(R.T[None], (-R.T @ t)[None])[0]  # Ad(T_{llj,sen})
    return Ad_inv.T @ np.asarray(simat_object_llj, float) @ Ad_inv


def inertia_to_phi(G):
    """[m, m c, Ixx Iyy Izz Ixy Iyz Izx] of a rigid-body spatial inertia [[m 1, -[h]x], [[h]x, I]]."""
    return np.array([G[0, 0], G[5, 1], G[3, 2], G[4, 0], G[3, 3], G[4, 4], G[5, 5], G[3, 4], G[4, 5], G[5, 3]])


def _sensor_state(consts, pose_sen_Rt, q, qd, qacc):
    out = rv.inverse_batched(np.stack([q, qd, qacc])[None], consts["hposes_Rt"], consts["simats"], consts["uscrews"], consts["twist_0"], consts["dtwist_0"],
                             **lo.tip_kw(consts))
    return rv.sensor_frame_twists_batched(pose_sen_Rt, out["twists"][:, -1], out["dtwists"][:, -1])


def _ft_reading(G_s, Vs, dVs):
    ad = rv.curlywedge(Vs)[0]
    return G_s @ dVs[0] - ad.T @ (G_s @ Vs[0])


def lqr_gain(consts, q, qd, input_gain, dt=0.002, eps=1e-8, centered=True):
    """controllers/lqr.py:38-51."""
    from scipy import linalg

    A, B = lo.transition_fd(consts, q[None], qd[None], None, dt=dt, eps=eps, centered=centered)
    A, B = A[0], B[0]
    Q, R = np.eye(A.shape[0]), np.diag(input_gain)
    P = linalg.solve_discrete_are(A, B, Q, R)
    return linalg.pinv(R + B.T @ P @ B) @ B.T @ P @ A


def closed_loop_replay(consts, pose_sen_Rt, G_s, plan_traj, K, q0, qd0=None, dt=0.002, fps=50.0, nu=6.0):
    n_steps, nj = plan_traj.shape[0], plan_traj.shape[2]
    q, qd = np.array(q0, float), np.zeros(nj) if qd0 is None else np.array(qd0, float)
    time = 0.0
    qacc = lo.forward_dynamics(consts, q[None], qd[None], np.zeros((1, nj)))[0]
    wrench = _ft_reading(G_s, *_sensor_state(consts, pose_sen_Rt, q, qd, qacc))
    tgt_ctrl_all = rv.inverse_batched(plan_traj, consts["hposes_Rt"], consts["simats"], consts["uscrews"], consts["twist_0"], consts["dtwist_0"],
                                      **lo.tip_kw(consts))["tau"]
    log = dict(step=[], time=[], tgt=[], act=[], twist_sen=[], dtwist_sen=[], wrench=[], regressor=[], ctrl=[])
    frame_count = 0
    for step in range(n_steps):
        tgt = plan_traj[step]
        if frame_count <= time * fps:
            Vs, dVs = _sensor_state(consts, pose_sen_Rt, q, qd, qacc)
            log["step"].append(step); log["time"].append(time); log["tgt"].append(tgt.copy()); log["act"].append(np.stack([q, qd, qacc]))
            log["twist_sen"].append(Vs[0]); log["dtwist_sen"].append(dVs[0]); log["wrench"].append(wrench.copy())
            log["regressor"].append(rv.regressor_batched(Vs, dVs)[0])
            frame_count += 1
        res = np.concatenate([(tgt[0] - q) / nu, tgt[1] - qd])
        u = tgt_ctrl_all[step] - K @ res
        log["ctrl"].append(u)
        qacc = lo.forward_dynamics(consts, q[None], qd[None], u[None])[0]
        wrench = _ft_reading(G_s, *_sensor_state(consts, pose_sen_Rt, q, qd, qacc))
        qd = qd + dt * qacc
        q = q + dt * qd
        time += dt
    out = {k: np.array(v) for k, v in log.items()}
    out["q_final"], out["qd_final"], out["qacc_final"] = q, qd, qacc
    return out
