"""Random kinematic chains of 1 to 16 joints for the generic kernels, and their state sampler (shared by the CPU and the -m gpu suites;
no torch).

The generic path promises any chain of nj <= 16 joints, but the packaged robot has six and the goldens four, six and nine.  The joint
counts of NJ reach nj = 1, the maximum of 16, and the run-time-count kernels (`k_rnea_generic_soa<T, 0>` and every other generic
kernel) at counts no golden has; 6 is kept apart because the SoA RNEA runs a compile-time instance with the parameters in the
constant bank there.  Each chain is built like oracle/gen_golden.py::golden_generic: random home poses, dense SPD spatial inertias,
screws cycling rotation / translation / pitched screw, a moving base, gravity off the z axis, a sensor pose with an offset and,
optionally, a tip wrench through a tip pose.  `Chain.analyze` asserts the generic path before a test relies on it.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

NJ = (1, 2, 3, 5, 7, 8, 12, 16)
NJ_ALL = NJ + (6,)  # 6: the compile-time-count SoA RNEA instance
EDGE_ANGLES = (0.0, 1e-9, 2e5)  # rest, below liegroups' small-angle threshold, far outside [-pi, pi] (the slow argument reduction)


def random_rotation(rng):
    q = rng.standard_normal(4)
    w, x, y, z = q / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (w * y + x * z)],
                     [2 * (w * z + x * y), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (w * x + y * z), 1 - 2 * (x * x + y * y)]])


@dataclass
class Chain:
    nj: int
    consts: dict          # the oracles' form: hposes_Rt, simats, uscrews, twist_0, dtwist_0 [, wrench_tip, pose_tip_Rt]
    pose_sen_Rt: np.ndarray

    def sample(self, n, seed):
        """sample_traj for this chain: 2e5 only on the pure revolute joints, where it exercises the slow trigonometric path.  On a
        prismatic or pitched joint it would be a displacement of ~1e5 m, whose inertia matrix no finite-precision solve reproduces."""
        return sample_traj(self.nj, n, seed, revolute=~np.any(self.consts["uscrews"][:, :3] != 0, axis=1))

    @property
    def tip(self):
        return "wrench_tip" in self.consts

    def model_args(self):
        """Positional and keyword arguments of engine.Model / engine.analyze_model."""
        c = self.consts
        kw = dict(pose_sen_llj=self.pose_sen_Rt)
        if self.tip:
            kw.update(wrench_tip=c["wrench_tip"], pose_tip_ee=c["pose_tip_Rt"])
        return (c["hposes_Rt"], c["simats"], c["uscrews"], c["twist_0"], c["dtwist_0"]), kw

    def analyze(self):
        """engine.analyze_model on the chain, after asserting it selects the generic path (device-free)."""
        from rigid_body_manipulation_b200 import engine

        args, kw = self.model_args()
        an = engine.analyze_model(*args, **kw)
        assert an[0] == "generic", (self.nj, an[0])
        return an


def random_chain(nj, seed, tip=True):
    rng = np.random.default_rng(seed)
    hRt = np.zeros((nj + 1, 12))
    hRt[0, [0, 4, 8]] = 1.0
    for k in range(1, nj + 1):
        hRt[k, :9] = random_rotation(rng).reshape(9)
        hRt[k, 9:] = rng.uniform(-0.5, 0.5, 3)
    simats = np.zeros((nj + 1, 6, 6))
    for k in range(1, nj + 1):
        A = rng.standard_normal((6, 6))
        simats[k] = A @ A.T + 0.5 * np.eye(6)
    uscrews = np.zeros((nj, 6))
    for k in range(nj):
        a = rng.standard_normal(3)
        a /= np.linalg.norm(a)
        if k % 3 == 0:        # rotation about a random axis through the origin
            uscrews[k, 3:] = a
        elif k % 3 == 1:      # translation along a random axis
            uscrews[k, :3] = a
        else:                 # pitched screw about an axis off the origin
            uscrews[k, 3:] = a
            uscrews[k, :3] = rng.uniform(-0.7, 0.7, 3)
    g = rng.standard_normal(3)
    dtwist_0 = np.concatenate([9.81 * g / np.linalg.norm(g), rng.standard_normal(3) * 0.1])  # tilted gravity, angular base acceleration
    consts = dict(hposes_Rt=hRt, simats=simats, uscrews=uscrews, twist_0=rng.standard_normal(6) * 0.3, dtwist_0=dtwist_0)
    pose_sen = np.concatenate([random_rotation(rng).reshape(9), rng.uniform(-0.2, 0.2, 3)])
    if tip:
        consts["wrench_tip"] = rng.standard_normal(6)
        consts["pose_tip_Rt"] = np.concatenate([random_rotation(rng).reshape(9), rng.uniform(-0.3, 0.3, 3)])
    return Chain(nj=nj, consts=consts, pose_sen_Rt=pose_sen)


def sample_traj(nj, n, seed, revolute=None):
    """(n, 3, nj) = (q, qd, qdd) per sample: positions in +-3, and the leading rows put the joints at EDGE_ANGLES (the 2e5 row only
    the joints of the boolean mask `revolute`, default all)."""
    rng = np.random.default_rng(seed)
    traj = np.stack([rng.uniform(-3, 3, (n, nj)), rng.standard_normal((n, nj)), rng.standard_normal((n, nj)) * 3], axis=1)
    revolute = np.ones(nj, bool) if revolute is None else np.asarray(revolute, bool)
    for r, a in enumerate(EDGE_ANGLES[:n]):
        traj[r, 0, revolute if abs(a) > 1 else slice(None)] = a
    return traj


def phi_sensed(seed):
    """10 inertial parameters of a physical rigid body (mass, offset centre of mass, SPD inertia) in a sensor frame."""
    rng = np.random.default_rng(seed)
    m, c = 1.3, rng.uniform(-0.05, 0.05, 3)
    A = rng.standard_normal((3, 3)) * 0.05
    Ic = A @ A.T + 0.01 * np.eye(3)
    I = Ic + m * (c @ c * np.eye(3) - np.outer(c, c))
    return np.array([m, *(m * c), I[0, 0], I[1, 1], I[2, 2], I[0, 1], I[1, 2], I[2, 0]])
