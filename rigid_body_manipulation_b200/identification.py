"""Inertial-parameter identification from the fused Gram pack (replaces reference loggers/loggers.py:127-129).

The reference stacks every frame's 6x10 regressor into a (6F, 10) matrix and calls np.linalg.lstsq.  At 1e8 samples
that matrix is 48 GB, so the device accumulates the normal equations instead (rbm_regressor_gram_*), shards all-reduce
the 112-double pack, and the 10x10 system is solved here in float64 on the host (once per solve, O(1e3) flops).

pack layout: [Y^T Y (100, row-major) | Y^T f (10) | f^T f | n_samples].

The same parameters can be identified from joint torques instead of the wrist sensor (Model.payload_gram, rbm_payload_gram_*): on
the model without the payload, tau = tau0 + Phi phi, and the pack [Phi^T Phi | Phi^T r | r^T r | n] of r = tau - tau0 has exactly
this layout.  `solve`, `solve_many` and distributed.allreduce_gram therefore apply unchanged to either route, and the packs of the
two routes may be summed into one estimate.
Parameter order: [m, m cx, m cy, m cz, Ixx, Iyy, Izz, Ixy, Iyz, Izx] about the sensor-frame origin
(reference dynamics.py:225-230, loggers.py:133).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

PARAM_LABELS = ["total_mass", "mx", "my", "mz", "ixx", "iyy", "izz", "ixy", "iyz", "izx"]


@dataclass
class Identification:
    phi: np.ndarray          # (10,)
    n_samples: float
    residual_ss: float       # ||Y phi - f||^2 from the normal equations (cancellation-limited: ~1e-16 * f_ss)
    f_ss: float              # ||f||^2
    rms_residual: float      # per scalar wrench component
    cond: float              # condition number of the column-scaled Gram
    rank: int


def unpack(pack):
    p = np.asarray(pack.detach().cpu().numpy() if hasattr(pack, "detach") else pack, dtype=np.float64)
    if p.shape != (112,):
        raise ValueError("gram pack must have 112 elements")
    return p[:100].reshape(10, 10), p[100:110], float(p[110]), float(p[111])


def solve(pack, rcond: float = 1e-13) -> Identification:
    """Minimum-norm least-squares solution of the normal equations, column-equilibrated (the columns of Y mix m/s^2,
    rad/s^2 and (rad/s)^2 scales) and solved by a symmetric eigen-decomposition with a relative cut-off, so rank-deficient
    excitations (e.g. a trajectory that never rotates) behave like np.linalg.lstsq's minimum-norm answer."""
    G, b, ff, n = unpack(pack)
    G = 0.5 * (G + G.T)
    d = np.sqrt(np.clip(np.diag(G), 0.0, None))
    d[d == 0.0] = 1.0
    Gs = G / np.outer(d, d)
    w, V = np.linalg.eigh(Gs)
    keep = w > rcond * max(w.max(), 0.0)
    z = V[:, keep] @ ((V[:, keep].T @ (b / d)) / w[keep])
    phi = z / d
    rss = max(ff - 2.0 * phi @ b + phi @ G @ phi, 0.0)
    cond = float(w.max() / w[keep].min()) if keep.any() else float("inf")
    return Identification(phi=phi, n_samples=n, residual_ss=rss, f_ss=ff, rms_residual=float(np.sqrt(rss / max(6.0 * n, 1.0))), cond=cond, rank=int(keep.sum()))


def solve_many(packs, rcond: float = 1e-13) -> list:
    """One identification per row of a (k, 112) stack of packs (e.g. one object per row after a grouped all-reduce)."""
    p = np.asarray(packs.detach().cpu().numpy() if hasattr(packs, "detach") else packs, dtype=np.float64)
    if p.ndim != 2 or p.shape[1] != 112:
        raise ValueError("packs must have shape (k, 112)")
    return [solve(row, rcond) for row in p]


def score(estimate, gt_params, aabb_scale: float) -> float:
    """The reference's normalised squared error (main.py:21-38): mass / first moments / inertias made dimensionless with
    m, m*L, m*L^2 (L = aabb_scale), averaged over the 10 parameters."""
    estimate, gt = np.asarray(estimate, dtype=float), np.asarray(gt_params, dtype=float)
    m = gt[0]
    s = ((estimate[0] - gt[0]) ** 2) / (m * aabb_scale**0) ** 2
    s += ((estimate[1:4] - gt[1:4]) ** 2).sum() / (m * aabb_scale**1) ** 2
    s += ((estimate[4:10] - gt[4:10]) ** 2).sum() / (m * aabb_scale**2) ** 2
    return float(s / 10.0)


def sensor_frame_params(target, pose_sen_obj_Rt) -> np.ndarray:
    """Ground-truth phi of a target expressed in the SENSOR frame (what the regressor identifies), from the body-frame CAD
    values: c_s = R c + t, I_s(origin) = R I_com R^T + m (|c_s|^2 1 - c_s c_s^T)."""
    Rt = np.asarray(pose_sen_obj_Rt, dtype=float)
    R, t = Rt[:9].reshape(3, 3), Rt[9:]
    c = R @ target.com + t
    I0 = R @ target.inertia_com @ R.T + target.mass * (c @ c * np.eye(3) - np.outer(c, c))
    return np.array([target.mass, *(target.mass * c), I0[0, 0], I0[1, 1], I0[2, 2], I0[0, 1], I0[1, 2], I0[2, 0]])


# ---------------------------------------------------------------------------------------------------------------
# dataset handling around the solve (reference loggers/loggers.py:82-156, core/simulate.py:281-290)
# ---------------------------------------------------------------------------------------------------------------
def split_indices(n: int, valid_ratio: float = 0.1, test_ratio: float = 0.1, seed: int = 0):
    """Frame indices of the train / valid / test subsets exactly as the reference's `Logger._split` draws them
    (loggers.py:94-106): one `default_rng(seed).shuffle` of range(n); train = the first n - n_test - n_valid, valid = the
    next n_valid -- and `test` is the SAME slice as valid (the reference slices [num_train : num_train + num_valid] twice,
    loggers.py:105-106; reproduced, not fixed)."""
    num_test = int(n * test_ratio)
    num_valid = int(n * valid_ratio)
    num_train = n - num_test - num_valid
    order = list(range(n))
    np.random.default_rng(seed).shuffle(order)
    order = np.asarray(order, dtype=np.int64)
    valid = order[num_train : num_train + num_valid]
    return order[:num_train], valid, valid.copy()


def perturb_wrench(fts, error_rate: float = 0.05, seed: int = 0):
    """The reference's measurement-noise model (core/simulate.py:281-290): zero-mean Gaussian noise on forces and on torques
    with sigma = error_rate * max_frames ||force|| (resp. ||torque||), one generator seeded `seed`, forces drawn first.
    fts: (n, 6) host array [force; torque]; returns a perturbed copy."""
    fts = np.array(fts, dtype=np.float64, copy=True)
    rng = np.random.default_rng(seed)
    fs_std = error_rate * np.linalg.norm(fts[..., :3], axis=1).max()
    ts_std = error_rate * np.linalg.norm(fts[..., 3:], axis=1).max()
    fts[..., :3] += fs_std * rng.standard_normal((len(fts), 3))
    fts[..., 3:] += ts_std * rng.standard_normal((len(fts), 3))
    return fts


def identify_splits(model, q, qd, qdd, f, valid_ratio: float = 0.1, test_ratio: float = 0.1, seed: int = 0, reduce=None) -> dict:
    """`Logger.finish` (loggers.py:147-156) on the device: identification on all frames and on the train / valid / test
    subsets.  q, qd, qdd, f are CUDA tensors (nj, n) / (6, n); `reduce` is an optional callable applied to every Gram pack
    (e.g. distributed.allreduce_gram when the frames are sharded)."""
    import torch

    n = q.shape[1]
    out = {}
    subsets = dict(zip(("train", "valid", "test"), split_indices(n, valid_ratio, test_ratio, seed)))
    for name, idx in [("all", None)] + list(subsets.items()):
        if idx is None:
            args = (q, qd, qdd, f)
        else:
            sel = torch.as_tensor(idx, device=q.device)
            args = tuple(t.index_select(1, sel).contiguous() for t in (q, qd, qdd, f))
        pack = model.regressor_gram(*args).clone()
        if reduce is not None:
            reduce(pack)
        out[name] = solve(pack)
    return out
