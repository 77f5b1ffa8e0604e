"""Model classes that reach the fast kernels the packaged robot never selects, and the sampled state distribution (shared by the CPU
and the -m gpu suites; no torch).

Every packaged target and golden is SEQ_ISO with the reference's Rz(180 deg) sensor site and gravity along z, so without these models
the SEQ_RIGID instantiations, the SEN_DIAG = false instantiations (full sensor adjoint) and any tilted base acceleration would go
unlaunched.  Each builder starts from the packaged hammer model and states the kernel path and `sen_diag` the model must select; a
test asserts both before it relies on them, so a change in model detection fails loudly instead of moving the test onto another kernel.

  rigid                links 1-5 as general rigid bodies (offset centre of mass, full SPD inertia)      -> seq_rigid, sen_diag 1
  offset_sensor        the hammer's inertias, sensor site rotated about z and offset, gravity tilted     -> seq_iso,   sen_diag 0
  rigid_offset_sensor  both                                                                              -> seq_rigid, sen_diag 0
  hammer               the packaged model unchanged (the class the rest of the suite covers)             -> seq_iso,   sen_diag 1
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from oracle import replay_oracle as ro
from rigid_body_manipulation_b200 import model as pm

CLASSES = ("rigid", "offset_sensor", "rigid_offset_sensor")
TILTED_DTWIST_0 = np.array([2.0, -3.0, 9.0, 0.0, 0.0, 0.0])  # linear base acceleration (gravity) off the z axis


def sample_states(rng, n):
    """SURVEY.md 8(d) config-2 input distribution (same as oracle/gen_golden.py): (n, 3, 6) = (q, qd, qdd) per sample."""
    q = np.concatenate([rng.uniform(-1.5, 2.5, (n, 3)), rng.uniform(-6 * np.pi, 6 * np.pi, (n, 3))], axis=1)
    qd = rng.standard_normal((n, 6)) * np.array([1, 1, 1, 3, 3, 3.0])
    qdd = rng.standard_normal((n, 6)) * np.array([3, 3, 3, 10, 10, 10.0])
    return np.stack([q, qd, qdd], axis=1)


def rigid_link_simats(simats, rng):
    """Links 1-5 get an offset centre of mass (+-0.1 m) and a full SPD rotational inertia: still physical rigid bodies, but no longer
    the isotropic blocks SEQ_ISO needs, so the model selects SEQ_RIGID.  Draws from `rng`; link 0 and link 6 are kept."""
    sim = np.array(simats, dtype=np.float64, copy=True)
    for k in range(1, 6):
        m, c = 8.0 + k, rng.uniform(-0.1, 0.1, 3)
        A = rng.standard_normal((3, 3)) * 0.1
        Ic = A @ A.T + 0.05 * np.eye(3)
        cx = np.array([[0, -c[2], c[1]], [c[2], 0, -c[0]], [-c[1], c[0], 0]])
        sim[k] = np.block([[m * np.eye(3), -m * cx], [m * cx, Ic + m * (c @ c * np.eye(3) - np.outer(c, c))]])
    return sim


def offset_sensor_pose(pose_sen_Rt, angle=0.3, offset=(0.01, -0.02, 0.05)):
    """The sensor site rotated by `angle` about z and moved by `offset`: Ad(T) is no longer a component-wise sign pattern."""
    c, s = np.cos(angle), np.sin(angle)
    Rz = np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])
    R = Rz @ np.asarray(pose_sen_Rt, np.float64)[:9].reshape(3, 3)
    return np.concatenate([R.reshape(9), np.asarray(offset, np.float64)])


@dataclass
class ModelClass:
    name: str
    hposes_Rt: np.ndarray
    simats: np.ndarray
    uscrews: np.ndarray
    twist_0: np.ndarray
    dtwist_0: np.ndarray
    pose_sen_Rt: np.ndarray
    phi: np.ndarray               # the sensed object's 10 inertial parameters in this model's sensor frame
    G_sensed: np.ndarray          # its spatial inertia in that frame
    key_qpos: np.ndarray
    path: str                     # kernel path the model must select
    sen_diag: int                 # whether the fast kernels may treat the sensor adjoint as a sign pattern

    @property
    def consts(self):
        """The constants in the form the oracles take (oracle/lqr_oracle.py, oracle/replay_oracle.py)."""
        return dict(hposes_Rt=self.hposes_Rt, simats=self.simats, uscrews=self.uscrews, twist_0=self.twist_0, dtwist_0=self.dtwist_0)

    def model_args(self):
        """Positional and keyword arguments of engine.Model / engine.analyze_model."""
        return (self.hposes_Rt, self.simats, self.uscrews, self.twist_0, self.dtwist_0), dict(pose_sen_llj=self.pose_sen_Rt)


def build(name):
    c = pm.load_packaged("sequential", "hammer")
    simats, dtwist_0, pose_sen = c.simats, c.dtwist_0, c.pose_sen_Rt
    rigid = name in ("rigid", "rigid_offset_sensor")
    offset = name in ("offset_sensor", "rigid_offset_sensor")
    if name not in CLASSES and name != "hammer":
        raise ValueError(f"unknown model class {name!r}")
    if rigid:
        simats = rigid_link_simats(c.simats, np.random.default_rng(5))
    if offset:
        pose_sen = offset_sensor_pose(c.pose_sen_Rt)
        dtwist_0 = TILTED_DTWIST_0.copy()
    G_s = ro.sensor_inertia(c.simat_object_llj, pose_sen)
    return ModelClass(name=name, hposes_Rt=c.hposes_Rt, simats=simats, uscrews=c.uscrews, twist_0=c.twist_0, dtwist_0=dtwist_0,
                      pose_sen_Rt=pose_sen, phi=ro.inertia_to_phi(G_s), G_sensed=G_s, key_qpos=c.key_qpos,
                      path="seq_rigid" if rigid else "seq_iso", sen_diag=0 if offset else 1)


def analyze(mc, **kw):
    """engine.analyze_model on the class's constants, after asserting it selects the path and sen_diag the class was built for."""
    from rigid_body_manipulation_b200 import engine

    args, kwargs = mc.model_args()
    an = engine.analyze_model(*args, **kwargs, **kw)
    if not kw.get("force_generic"):
        assert an[0] == mc.path, (mc.name, an[0])
        assert an[1][-1] == mc.sen_diag, (mc.name, an[1][-1])
    return an
