"""Helpers shared by the -m gpu tests (all compute goes through the C ABI via rigid_body_manipulation_b200.engine)."""
import numpy as np
import torch

from conftest import load_golden
from model_classes import sample_states  # torch-free, shared with the CPU suite


def rel_err(a, b, floor=1e-6):
    """norm-wise relative error per sample: max_j |a - b| / max(max_j |b|, floor)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    ax = tuple(range(1, a.ndim))
    return np.max(np.abs(a - b), axis=ax) / np.maximum(np.max(np.abs(b), axis=ax), floor)


def model_from_golden(g, **kw):
    from rigid_body_manipulation_b200.engine import Model

    extra = {}
    if "wrench_tip" in g.files:
        extra = dict(wrench_tip=g["wrench_tip"], pose_tip_ee=g["pose_tip"])
    return Model(g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"], pose_sen_llj=g["pose_sen_llj"], **extra, **kw)


def soa(traj, dtype=torch.float64):
    """(n, 3, nj) host array -> three contiguous CUDA tensors (nj, n)."""
    t = torch.as_tensor(np.ascontiguousarray(traj), dtype=dtype, device="cuda")
    return tuple(t[:, k, :].t().contiguous() for k in range(3))


__all__ = ["rel_err", "model_from_golden", "soa", "sample_states", "load_golden"]
