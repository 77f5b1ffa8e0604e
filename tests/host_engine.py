"""TEST INFRASTRUCTURE ONLY: an `engine`-shaped object whose arithmetic is the kernels' own __host__ __device__ code compiled for the
host (tests/host_harness).  tests/test_dropin_reference_simulate.py swaps it in for `rigid_body_manipulation_b200.engine` inside the
drop-in packages so that the reference's unmodified simulate() can run on top of them in the GPU-less container.  The product
package has no such switch: its engine is the CUDA library or nothing."""
import numpy as np
import torch

import host_harness as hh
from rigid_body_manipulation_b200 import engine as real_engine

pose_to_Rt = real_engine.pose_to_Rt      # pure numpy converters, shared
poses_to_Rt = real_engine.poses_to_Rt


def current_device():
    return 0


def _t(a):
    return None if a is None else torch.as_tensor(np.ascontiguousarray(a))


class Model:
    """Same constructor and the methods the drop-in packages call (rnea_full_host, linearize), evaluated on the host."""

    def __init__(self, hposes_body_parent, simats_body, uscrews_body, twist_0, dtwist_0, wrench_tip=None, pose_tip_ee=None, pose_sen_llj=None,
                 device=None, force_generic=False, no_tma=False):
        self.uscrews = np.ascontiguousarray(uscrews_body, dtype=np.float64)
        self.nj = self.uscrews.shape[0]
        self.analysis = real_engine.analyze_model(hposes_body_parent, simats_body, uscrews_body, twist_0, dtwist_0, wrench_tip, pose_tip_ee, pose_sen_llj,
                                                  force_generic=force_generic)  # rbm_model_analyze: device-free, the product's own code
        self.kernel_path = self.analysis[0]
        self.device = torch.device("cpu")

    def rnea_full_host(self, traj):
        out = hh.generic_rnea(self.analysis[2], self.nj, np.ascontiguousarray(traj, dtype=np.float64), full=True)
        return out["tau"], out["poses"], out["twists"], out["dtwists"]

    def linearize(self, q, qd, u=None, dt=0.002, eps=1e-8, centered=True, want_qdd=False):
        tn = lambda x: None if x is None else x.detach().cpu().numpy().T
        A, B, qdd = hh.linearize(self.analysis, tn(q), tn(qd), tn(u), dt=dt, eps=eps, centered=centered)
        out = (_t(A), _t(B))
        return out + (_t(qdd.T),) if want_qdd else out


def transfer_simat(poses_Rt, simats, adjoint_form=False):
    P, G = np.asarray(poses_Rt, dtype=np.float64), np.asarray(simats, dtype=np.float64)
    if P.shape[0] != G.shape[0]:
        raise ValueError("The numbers of spatial inertia tensors and SE3 instances do not match.")
    return _t(hh.transfer_simat(P, G, adjoint_form))


def coordinate_transfer_imat(poses_Rt, imats, mass):
    return _t(hh.coordinate_transfer_imat(poses_Rt, imats, mass))


def spatial_inertia(mass, diag):
    return _t(hh.spatial_inertia(mass, diag))


def compose_poses(trans, rot):
    out, status = hh.compose_poses(trans, rot)
    return _t(out), _t(status)


def point_motion(twists, dtwists, points, want_acc=True):
    lv, la = hh.point_motion(twists, dtwists, points, want_acc)
    return _t(lv), _t(la)


def regressor_rows(twists, dtwists):
    tn = lambda x: x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else x
    return _t(hh.regressor_rows(tn(twists), tn(dtwists)))


def sensor_twists(pose, twists, dtwists):
    Vs, dVs, _ = hh.sensor_regressor(pose_to_Rt(pose), twists, dtwists)
    return _t(Vs), _t(dVs)
