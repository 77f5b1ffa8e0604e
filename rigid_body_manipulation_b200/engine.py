"""Batched B200 engine: a model handle plus the batched entry points, on torch CUDA tensors.

PyTorch is plumbing here (device memory, streams); all arithmetic happens in librbm_b200.so through
the C ABI of include/rbm_b200.h.  The constants are exactly the arguments the reference binds onto
`dynamics.inverse` with functools.partial (reference core/simulate.py:150-156).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib


def _f64(a, shape=None):
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
    if shape is not None and a.shape != tuple(shape):
        raise ValueError(f"expected shape {tuple(shape)}, got {a.shape}")
    return a


def pose_to_Rt(pose) -> np.ndarray:
    """SE3-like (anything with .rot.as_matrix() and .trans), a 4x4 / 3x4 matrix, or 12 scalars -> [R row-major | t]."""
    if hasattr(pose, "rot") and hasattr(pose, "trans"):
        R = np.asarray(pose.rot.as_matrix(), dtype=np.float64)
        t = np.asarray(pose.trans, dtype=np.float64)
        return np.concatenate([R.reshape(9), t.reshape(3)])
    a = np.asarray(pose, dtype=np.float64)
    if a.shape == (12,):
        return a.copy()
    if a.shape in ((4, 4), (3, 4)):
        return np.concatenate([a[:3, :3].reshape(9), a[:3, 3]])
    raise ValueError("pose must be an SE3-like object, a 4x4 matrix or 12 scalars [R | t]")


def poses_to_Rt(poses) -> np.ndarray:
    if isinstance(poses, np.ndarray) and poses.ndim == 2 and poses.shape[1] == 12:
        return _f64(poses)
    return np.stack([pose_to_Rt(p) for p in poses])


def current_device() -> int:
    """Index of the CUDA device new models are created on."""
    return torch.cuda.current_device()


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    return C.c_void_p(a.data_ptr())


def analyze_model(hposes_body_parent, simats_body, uscrews_body, twist_0, dtwist_0, wrench_tip=None, pose_tip_ee=None, pose_sen_llj=None,
                  force_generic=False):
    """Device-free model analysis (rbm_model_analyze; works without a GPU): the kernel path the constants select and the parameter
    blocks the kernels would receive.  Returns (path_name, fast_params ndarray, generic_params ndarray)."""
    lib = _lib.load()
    uscrews = _f64(uscrews_body)
    nj = uscrews.shape[0]
    Rt = poses_to_Rt(hposes_body_parent)
    simats = _f64(simats_body)
    if Rt.shape != (nj + 1, 12) or simats.shape != (nj + 1, 6, 6):
        raise ValueError(f"need nj+1 = {nj + 1} home poses and spatial inertias")
    opt = lambda a, conv: None if a is None else conv(a)
    wt, tip, sen = opt(wrench_tip, lambda a: _f64(a, (6,))), opt(pose_tip_ee, pose_to_Rt), opt(pose_sen_llj, pose_to_Rt)
    path = C.c_int(-1)
    fast = np.zeros(lib.rbm_fast_param_count())
    generic = np.zeros(max(lib.rbm_generic_param_count(nj), 0))
    rc = lib.rbm_model_analyze(nj, _ptr(Rt), _ptr(simats), _ptr(uscrews), _ptr(_f64(twist_0, (6,))), _ptr(_f64(dtwist_0, (6,))), _ptr(wt), _ptr(tip),
                               _ptr(sen), _lib.FLAG_FORCE_GENERIC if force_generic else 0, C.byref(path), _ptr(fast), _ptr(generic))
    _lib.check(rc, "rbm_model_analyze")
    return _lib.PATH_NAMES[path.value], fast, generic


class Model:
    """Device-resident model constants (opaque `rbm_model*`) for one CUDA device."""

    def __init__(self, hposes_body_parent, simats_body, uscrews_body, twist_0, dtwist_0, wrench_tip=None,
                 pose_tip_ee=None, pose_sen_llj=None, device=None, force_generic=False, no_tma=False):
        lib = _lib.load()
        self.uscrews = _f64(uscrews_body)
        if self.uscrews.ndim != 2 or self.uscrews.shape[1] != 6:
            raise ValueError("uscrews_body must have shape (nj, 6)")
        self.nj = nj = self.uscrews.shape[0]
        self.hposes_Rt = poses_to_Rt(hposes_body_parent)
        if self.hposes_Rt.shape != (nj + 1, 12):
            raise ValueError(f"hposes_body_parent must hold nj+1 = {nj + 1} poses (entry 0 is the unused world pose)")
        self.simats = _f64(simats_body, (nj + 1, 6, 6))
        self.twist_0 = _f64(twist_0, (6,))
        self.dtwist_0 = _f64(dtwist_0, (6,))
        self.wrench_tip = None if wrench_tip is None else _f64(wrench_tip, (6,))
        self.pose_tip = None if pose_tip_ee is None else pose_to_Rt(pose_tip_ee)
        self.pose_sen = None if pose_sen_llj is None else pose_to_Rt(pose_sen_llj)
        if device is None:
            device = torch.cuda.current_device() if torch.cuda.is_available() else 0
        self.device = torch.device("cuda", int(device) if not isinstance(device, torch.device) else (device.index or 0))
        handle = C.c_void_p()
        rc = lib.rbm_model_create(nj, _ptr(self.hposes_Rt), _ptr(self.simats), _ptr(self.uscrews), _ptr(self.twist_0),
                                  _ptr(self.dtwist_0), _ptr(self.wrench_tip), _ptr(self.pose_tip), _ptr(self.pose_sen),
                                  (_lib.FLAG_FORCE_GENERIC if force_generic else 0) | (_lib.FLAG_NO_TMA if no_tma else 0),
                                  self.device.index, C.byref(handle))
        _lib.check(rc, "rbm_model_create")
        self._h = handle
        self._lib = lib
        self.kernel_path = _lib.PATH_NAMES[lib.rbm_model_kernel_path(handle)]

    def close(self):
        if getattr(self, "_h", None):
            self._lib.rbm_model_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- helpers ----------------------------------------------------------------------------
    def _check_dev(self, *tensors):
        for t in tensors:
            if t is None:
                continue
            if not t.is_cuda or t.device != self.device:
                raise ValueError(f"tensor must live on {self.device} (got {t.device}); there is no CPU path")
            if not t.is_contiguous():
                raise ValueError("tensor must be contiguous")

    @staticmethod
    def _stream():
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    # ---- batched inverse dynamics: SoA [nj][n] ----------------------------------------------
    def rnea(self, q, qd, qdd, tau=None, want_twists=False):
        """q, qd, qdd: CUDA tensors (nj, n) float64 or float32.  Returns tau (nj, n) [, V (6, n), dV (6, n)]."""
        self._check_dev(q, qd, qdd, tau)
        if q.shape != qd.shape or q.shape != qdd.shape or q.dim() != 2 or q.shape[0] != self.nj:
            raise ValueError(f"q, qd, qdd must all have shape ({self.nj}, n)")
        if q.dtype not in (torch.float64, torch.float32) or qd.dtype != q.dtype or qdd.dtype != q.dtype:
            raise ValueError("q, qd, qdd must share dtype float64 or float32")
        n = q.shape[1]
        if tau is None:
            tau = torch.empty_like(q)
        elif tau.shape != q.shape or tau.dtype != q.dtype:
            raise ValueError("tau must match q in shape and dtype")
        V = dV = None
        if want_twists:
            V = torch.empty((6, n), dtype=q.dtype, device=q.device)
            dV = torch.empty((6, n), dtype=q.dtype, device=q.device)
        fn = self._lib.rbm_rnea_f64 if q.dtype == torch.float64 else self._lib.rbm_rnea_f32
        with torch.cuda.device(self.device):
            rc = fn(self._h, _ptr(q), _ptr(qd), _ptr(qdd), _ptr(tau), _ptr(V), _ptr(dV), n, n, self._stream())
        _lib.check(rc, "rbm_rnea")
        return (tau, V, dV) if want_twists else tau

    # ---- batched inverse dynamics: AoS [n][3][nj], the reference's own `traj` layout ------------
    def rnea_aos(self, traj, tau=None):
        self._check_dev(traj, tau)
        if traj.dim() != 3 or traj.shape[1] != 3 or traj.shape[2] != self.nj:
            raise ValueError(f"traj must have shape (n, 3, {self.nj})")
        if traj.dtype not in (torch.float64, torch.float32):
            raise ValueError("traj must be float64 or float32")
        n = traj.shape[0]
        if tau is None:
            tau = torch.empty((n, self.nj), dtype=traj.dtype, device=traj.device)
        elif tuple(tau.shape) != (n, self.nj) or tau.dtype != traj.dtype:
            raise ValueError(f"tau must have shape ({n}, {self.nj}) and the dtype of traj")
        fn = self._lib.rbm_rnea_aos_f64 if traj.dtype == torch.float64 else self._lib.rbm_rnea_aos_f32
        with torch.cuda.device(self.device):
            rc = fn(self._h, _ptr(traj), _ptr(tau), n, self._stream())
        _lib.check(rc, "rbm_rnea_aos")
        return tau

    def rnea_full(self, traj):
        """Everything `dynamics.inverse` returns, per sample: tau (n,nj), poses (n,nj,12), twists, dtwists (n,nj+1,6)."""
        self._check_dev(traj)
        if traj.dim() != 3 or traj.shape[1] != 3 or traj.shape[2] != self.nj or traj.dtype != torch.float64:
            raise ValueError(f"traj must be float64 with shape (n, 3, {self.nj})")
        n, nj = traj.shape[0], self.nj
        kw = dict(dtype=torch.float64, device=traj.device)
        tau = torch.empty((n, nj), **kw)
        poses = torch.empty((n, nj, 12), **kw)
        tw = torch.empty((n, nj + 1, 6), **kw)
        dtw = torch.empty((n, nj + 1, 6), **kw)
        with torch.cuda.device(self.device):
            rc = self._lib.rbm_rnea_full_f64(self._h, _ptr(traj), _ptr(tau), _ptr(poses), _ptr(tw), _ptr(dtw), n, self._stream())
        _lib.check(rc, "rbm_rnea_full")
        return tau, poses, tw, dtw

    def rnea_full_host(self, traj):
        """Host-in / host-out version of `rnea_full` for small batches: traj (n, 3, nj) numpy -> numpy (tau, poses, twists, dtwists)."""
        traj = np.ascontiguousarray(traj, dtype=np.float64)
        if traj.ndim != 3 or traj.shape[1] != 3 or traj.shape[2] != self.nj:
            raise ValueError(f"traj must have shape (n, 3, {self.nj})")
        n, nj = traj.shape[0], self.nj
        tau = np.empty((n, nj))
        poses = np.empty((n, nj, 12))
        tw = np.empty((n, nj + 1, 6))
        dtw = np.empty((n, nj + 1, 6))
        rc = self._lib.rbm_rnea_full_host_f64(self._h, _ptr(traj), _ptr(tau), _ptr(poses), _ptr(tw), _ptr(dtw), n)
        _lib.check(rc, "rbm_rnea_full_host")
        return tau, poses, tw, dtw

    # ---- planner-driven: trajectory generated in the kernel (no input traffic) -------------------------------------
    def rnea_planned(self, plan, n=None, step0=None, stride=1.0, dtype=torch.float64, want_traj=False, tau=None):
        """tau (nj, n) for steps step0 + s*stride of a planner.QuinticPlan (defaults: every planned step).
        With want_traj also returns the generated (q, qd, qdd) as a (3, nj, n) tensor."""
        n = plan.n_steps if n is None else int(n)
        step0 = float(plan.init_step if step0 is None else step0)
        if len(plan.displacement) != self.nj or len(plan.pos_offset) != self.nj:
            raise ValueError(f"plan must have {self.nj} joints")
        if dtype not in (torch.float64, torch.float32):
            raise ValueError("dtype must be float64 or float32")
        if tau is None:
            tau = torch.empty((self.nj, n), dtype=dtype, device=self.device)
        elif tuple(tau.shape) != (self.nj, n) or tau.dtype != dtype:
            raise ValueError(f"tau must have shape ({self.nj}, {n}) and dtype {dtype}")
        self._check_dev(tau)
        traj = torch.empty((3, self.nj, n), dtype=dtype, device=self.device) if want_traj else None
        co = np.ascontiguousarray(plan.coeffs, dtype=np.float64)
        di = np.ascontiguousarray(plan.displacement, dtype=np.float64)
        of = np.ascontiguousarray(plan.pos_offset, dtype=np.float64)
        fn = self._lib.rbm_rnea_planned_f64 if dtype == torch.float64 else self._lib.rbm_rnea_planned_f32
        with torch.cuda.device(self.device):
            rc = fn(self._h, _ptr(co), _ptr(di), _ptr(of), float(plan.timestep), step0, float(stride), _ptr(tau), _ptr(traj), n, n, self._stream())
        _lib.check(rc, "rbm_rnea_planned")
        return (tau, traj) if want_traj else tau

    # ---- host end-to-end ---------------------------------------------------------------------------
    @staticmethod
    def _host_array(a, what):
        """(tensor-or-ndarray, is_tensor, numpy dtype) of a contiguous HOST buffer; raises for CUDA tensors / strided views."""
        if isinstance(a, torch.Tensor):
            if a.is_cuda:
                raise ValueError(f"{what} must live in host memory")
            if not a.is_contiguous():
                raise ValueError(f"{what} must be contiguous")
            if a.dtype not in (torch.float64, torch.float32):
                raise ValueError(f"{what} must be float64 or float32")
            return a, True, np.dtype(np.float64 if a.dtype == torch.float64 else np.float32)
        a = np.asarray(a)
        if a.dtype not in (np.float64, np.float32) or not a.flags.c_contiguous:
            raise ValueError(f"{what} must be a C-contiguous float64 / float32 array")
        return a, False, a.dtype

    def rnea_host(self, traj, tau=None, chunk=0):
        """traj: HOST array / pinned CPU tensor (n, 3, nj); returns tau on the host (same kind).  H2D, kernel and D2H are
        pipelined inside the library (rbm_rnea_host_*)."""
        if not isinstance(traj, torch.Tensor):
            traj = np.ascontiguousarray(traj)
        arr, is_t, dt = self._host_array(traj, "traj")
        shape = tuple(arr.shape)
        if len(shape) != 3 or shape[1] != 3 or shape[2] != self.nj:
            raise ValueError(f"traj must have shape (n, 3, {self.nj})")
        n = shape[0]
        if tau is None:
            tau = torch.empty((n, self.nj), dtype=arr.dtype, pin_memory=True) if is_t else np.empty((n, self.nj), dtype=dt)
        else:
            tau, _, tdt = self._host_array(tau, "tau")
            if tuple(tau.shape) != (n, self.nj) or tdt != dt:
                raise ValueError(f"tau must be a host buffer of shape ({n}, {self.nj}) with the dtype of traj")
        fn = self._lib.rbm_rnea_host_f64 if dt == np.float64 else self._lib.rbm_rnea_host_f32
        rc = fn(self._h, _ptr(arr), _ptr(tau), n, int(chunk))
        _lib.check(rc, "rbm_rnea_host")
        return tau

    def rnea_host_soa(self, q, qd, qdd, tau=None, chunk=0):
        """SoA host entry: q, qd, qdd HOST buffers (nj, n) -> tau (nj, n) on the host.  Only the rows the model's tau-only kernel
        actually reads cross the bus: for the sequential structure neither the three gantry positions (`live_inputs()`) nor the
        three gantry velocities, which tau does not depend on, so 12 of the 18 input rows are uploaded and the caller may leave
        q[:3] and qd[:3] unset.  One strided copy per run of live rows and chunk, pipelined with the kernel and the D2H of tau."""
        bufs = []
        for name, a in (("q", q), ("qd", qd), ("qdd", qdd)):
            arr, is_t, dt = self._host_array(a, name)
            bufs.append((arr, is_t, dt))
        (qa, is_t, dt) = bufs[0]
        if qa.ndim != 2 or qa.shape[0] != self.nj or any(tuple(b[0].shape) != tuple(qa.shape) or b[2] != dt for b in bufs[1:]):
            raise ValueError(f"q, qd, qdd must be host buffers of one dtype with shape ({self.nj}, n)")
        n = qa.shape[1]
        if tau is None:
            tau = torch.empty((self.nj, n), dtype=qa.dtype, pin_memory=True) if is_t else np.empty((self.nj, n), dtype=dt)
        else:
            tau, _, tdt = self._host_array(tau, "tau")
            if tuple(tau.shape) != (self.nj, n) or tdt != dt:
                raise ValueError(f"tau must be a host buffer of shape ({self.nj}, {n}) with the dtype of q")
        fn = self._lib.rbm_rnea_host_soa_f64 if dt == np.float64 else self._lib.rbm_rnea_host_soa_f32
        rc = fn(self._h, _ptr(qa), _ptr(bufs[1][0]), _ptr(bufs[2][0]), _ptr(tau), n, n, int(chunk))
        _lib.check(rc, "rbm_rnea_host_soa")
        return tau

    def rnea_planned_host(self, plan, n=None, step0=None, stride=1.0, dtype=torch.float64, tau=None, chunk=0):
        """Planner-driven end to end: the trajectory is generated in the kernel, so nothing is uploaded and only tau (nj, n) comes
        back to the host (pinned tensor), chunked so that the D2H of one chunk overlaps the kernel of the next."""
        n = plan.n_steps if n is None else int(n)
        step0 = float(plan.init_step if step0 is None else step0)
        if len(plan.displacement) != self.nj or len(plan.pos_offset) != self.nj:
            raise ValueError(f"plan must have {self.nj} joints")
        if dtype not in (torch.float64, torch.float32):
            raise ValueError("dtype must be float64 or float32")
        if tau is None:
            tau = torch.empty((self.nj, n), dtype=dtype, pin_memory=True)
        else:
            tau, _, tdt = self._host_array(tau, "tau")
            if tuple(tau.shape) != (self.nj, n) or tdt != np.dtype(np.float64 if dtype == torch.float64 else np.float32):
                raise ValueError(f"tau must be a host buffer of shape ({self.nj}, {n}) and dtype {dtype}")
        co = np.ascontiguousarray(plan.coeffs, dtype=np.float64)
        di = np.ascontiguousarray(plan.displacement, dtype=np.float64)
        of = np.ascontiguousarray(plan.pos_offset, dtype=np.float64)
        fn = self._lib.rbm_rnea_planned_host_f64 if dtype == torch.float64 else self._lib.rbm_rnea_planned_host_f32
        rc = fn(self._h, _ptr(co), _ptr(di), _ptr(of), float(plan.timestep), step0, float(stride), _ptr(tau), n, n, int(chunk))
        _lib.check(rc, "rbm_rnea_planned_host")
        return tau

    def live_inputs(self):
        """Boolean mask (3, nj): which rows of (q, qd, qdd) the model's inverse-dynamics kernel reads when the twists are asked for
        too (rbm_model_live_inputs).  A tau-only call (`rnea` without want_twists, `rnea_host_soa`) on the sequential structure also
        skips the three gantry velocities qd[:3]."""
        mask = np.zeros(3 * self.nj, dtype=np.int32)
        rc = self._lib.rbm_model_live_inputs(self._h, _ptr(mask))
        _lib.check(rc, "rbm_model_live_inputs")
        return mask.reshape(3, self.nj).astype(bool)

    # ---- sensor-frame regressor / identification --------------------------------------------------
    def _check_soa(self, *ts):
        self._check_dev(*ts)
        q = ts[0]
        if q.dim() != 2 or q.shape[0] != self.nj or q.dtype not in (torch.float64, torch.float32):
            raise ValueError(f"q must be float64 / float32 with shape ({self.nj}, n)")
        for t in ts[1:3]:
            if t.shape != q.shape or t.dtype != q.dtype:
                raise ValueError("q, qd, qdd must share shape and dtype")
        return q.shape[1], q.dtype

    def regressor_from_traj(self, q, qd, qdd, want_rows=True, want_twists=False, phi=None):
        """(q, qd, qdd) (nj, n) -> dict with any of: Y (n, 6, 10), twist_sen / dtwist_sen (6, n), wrench (6, n) = Y phi."""
        n, dt = self._check_soa(q, qd, qdd)
        kw = dict(dtype=dt, device=q.device)
        Y = torch.empty((n, 6, 10), **kw) if want_rows else None
        Vs = torch.empty((6, n), **kw) if want_twists else None
        dVs = torch.empty((6, n), **kw) if want_twists else None
        ph = F = None
        if phi is not None:
            ph = torch.as_tensor(phi, **kw).contiguous()
            if ph.shape != (10,):
                raise ValueError("phi must hold the 10 inertial parameters")
            F = torch.empty((6, n), **kw)
        fn = self._lib.rbm_regressor_from_traj_f64 if dt == torch.float64 else self._lib.rbm_regressor_from_traj_f32
        with torch.cuda.device(self.device):
            rc = fn(self._h, _ptr(q), _ptr(qd), _ptr(qdd), _ptr(Y), _ptr(Vs), _ptr(dVs), _ptr(ph), _ptr(F), n, n, self._stream())
        _lib.check(rc, "rbm_regressor_from_traj")
        return dict(Y=Y, twist_sen=Vs, dtwist_sen=dVs, wrench=F)

    def regressor_gram(self, q, qd, qdd, f, pack=None):
        """Fused regressor + normal equations: returns the 112-double device pack [Y^T Y | Y^T f | f^T f | n]."""
        n, dt = self._check_soa(q, qd, qdd)
        self._check_dev(f, pack)
        if f.shape != (6, n) or f.dtype != dt:
            raise ValueError("f must have shape (6, n) and the dtype of q")
        if pack is None:
            pack = torch.empty(112, dtype=torch.float64, device=q.device)
        elif pack.shape != (112,) or pack.dtype != torch.float64:
            raise ValueError("pack must be a float64 tensor of 112 elements")
        ws = self._gram_workspace(n)
        fn = self._lib.rbm_regressor_gram_f64 if dt == torch.float64 else self._lib.rbm_regressor_gram_f32
        with torch.cuda.device(self.device):
            rc = fn(self._h, _ptr(q), _ptr(qd), _ptr(qdd), _ptr(f), _ptr(pack), _ptr(ws), ws.numel() * 8, n, n, self._stream())
        _lib.check(rc, "rbm_regressor_gram")
        return pack

    def _gram_workspace(self, n):
        """Device scratch of the Gram kernels (rbm_gram_workspace_bytes), cached on the model and grown on demand."""
        ws_bytes = int(self._lib.rbm_gram_workspace_bytes(self._h, n))
        ws = getattr(self, "_gram_ws", None)
        if ws is None or ws.numel() * 8 < ws_bytes:
            ws = self._gram_ws = torch.empty(max(1, ws_bytes // 8), dtype=torch.float64, device=self.device)
        return ws

    # ---- payload identification from joint torques -------------------------------------------------------
    def payload_regressor(self, q, qd, qdd, want_rows=True, want_tau0=False):
        """Joint-torque payload regressor of this model (the robot WITHOUT the payload): tau = tau0 + Phi phi with phi the payload's 10
        parameters in the sensor frame (pose_sen_llj), as in `regressor_from_traj`.  Returns a dict with Phi (n, nj, 10) and tau0
        (nj, n), each None unless asked for."""
        n, dt = self._check_soa(q, qd, qdd)
        kw = dict(dtype=dt, device=q.device)
        Phi = torch.empty((n, self.nj, 10), **kw) if want_rows else None
        tau0 = torch.empty((self.nj, n), **kw) if want_tau0 else None
        fn = self._lib.rbm_payload_regressor_f64 if dt == torch.float64 else self._lib.rbm_payload_regressor_f32
        with torch.cuda.device(self.device):
            rc = fn(self._h, _ptr(q), _ptr(qd), _ptr(qdd), _ptr(Phi), _ptr(tau0), n, n, self._stream())
        _lib.check(rc, "rbm_payload_regressor")
        return dict(Phi=Phi, tau0=tau0)

    def payload_gram(self, q, qd, qdd, tau, pack=None):
        """Normal equations of the joint-torque route from measured torques tau (nj, n): the 112-double device pack
        [Phi^T Phi | Phi^T r | r^T r | n] with r = tau - tau0, solved like an F/T pack by identification.solve."""
        n, dt = self._check_soa(q, qd, qdd)
        self._check_dev(tau, pack)
        if tau.shape != (self.nj, n) or tau.dtype != dt:
            raise ValueError(f"tau must have shape ({self.nj}, n) and the dtype of q")
        if pack is None:
            pack = torch.empty(112, dtype=torch.float64, device=q.device)
        elif pack.shape != (112,) or pack.dtype != torch.float64:
            raise ValueError("pack must be a float64 tensor of 112 elements")
        ws = self._gram_workspace(n)
        fn = self._lib.rbm_payload_gram_f64 if dt == torch.float64 else self._lib.rbm_payload_gram_f32
        with torch.cuda.device(self.device):
            rc = fn(self._h, _ptr(q), _ptr(qd), _ptr(qdd), _ptr(tau), _ptr(pack), _ptr(ws), ws.numel() * 8, n, n, self._stream())
        _lib.check(rc, "rbm_payload_gram")
        return pack

    def regressor_gram_grouped(self, q, qd, qdd, f):
        """One Gram pack per group for frame-major logs: q, qd, qdd (F, nj, n) and f (F, 6, n), float64 CUDA tensors.  Strided VIEWS of
        a log tensor are consumed in place: q, qd, qdd must share their frame stride, all four the row stride, and the group axis must
        be dense.  Returns packs (n, 112) (a transposed view of the kernel's [112][n] output)."""
        F, nj, n = q.shape
        ts = (q, qd, qdd, f)
        if any((not t.is_cuda) or t.device != self.device for t in ts):
            raise ValueError(f"tensors must live on {self.device}; there is no CPU path")
        if nj != self.nj or qd.shape != q.shape or qdd.shape != q.shape or f.shape != (F, 6, n) or any(t.dtype != torch.float64 for t in ts):
            raise ValueError(f"q, qd, qdd must be float64 (F, {self.nj}, n) and f (F, 6, n)")
        st = q.stride()
        if any(t.stride(2) != 1 or t.stride(1) != st[1] for t in ts) or (F > 1 and any(t.stride(0) != st[0] for t in (qd, qdd))):
            raise ValueError("q, qd, qdd must share their frame stride, all four arrays the row stride, with a dense group axis")
        packs = torch.empty((112, n), dtype=torch.float64, device=q.device)
        with torch.cuda.device(self.device):
            rc = self._lib.rbm_regressor_gram_grouped_f64(self._h, _ptr(q), _ptr(qd), _ptr(qdd), _ptr(f), int(st[0]) if F > 1 else 0,
                                                          int(f.stride(0)) if F > 1 else 0, F, _ptr(packs), n, int(st[1]), n, self._stream())
        _lib.check(rc, "rbm_regressor_gram_grouped")
        return packs.t()

    # ---- LQR linearisation -----------------------------------------------------------------------------
    def linearize(self, q, qd, u=None, dt=0.002, eps=1e-8, centered=True, want_qdd=False):
        """States (q, qd) (nj, n) [+ ctrl u (nj, n)] -> A (n, 2nj, 2nj), B (n, 2nj, nj) as element-major VIEWS
        (storage is [(r*cols + c)][n], so `A[s]` is a strided 2-D view; call .contiguous() for a packed copy)."""
        self._check_dev(q, qd, u)
        if q.dtype != torch.float64 or q.dim() != 2 or q.shape[0] != self.nj or qd.shape != q.shape or qd.dtype != q.dtype:
            raise ValueError(f"q, qd must be float64 with shape ({self.nj}, n)")
        if u is not None and (u.shape != q.shape or u.dtype != q.dtype):
            raise ValueError("u must match q")
        n, nj = q.shape[1], self.nj
        A = torch.empty((2 * nj, 2 * nj, n), dtype=q.dtype, device=q.device)
        B = torch.empty((2 * nj, nj, n), dtype=q.dtype, device=q.device)
        qdd = torch.empty_like(q) if want_qdd else None
        with torch.cuda.device(self.device):
            rc = self._lib.rbm_linearize_f64(self._h, _ptr(q), _ptr(qd), _ptr(u), float(dt), float(eps), int(bool(centered)), _ptr(A), _ptr(B),
                                             _ptr(qdd), n, n, self._stream())
        _lib.check(rc, "rbm_linearize")
        out = (A.permute(2, 0, 1), B.permute(2, 0, 1))
        return out + (qdd,) if want_qdd else out


    def forward_dynamics(self, q, qd, u=None):
        """qdd = M(q)^-1 (u - h(q, qd)) for CUDA tensors (nj, n) float64."""
        self._check_dev(q, qd, u)
        if q.dtype != torch.float64 or q.dim() != 2 or q.shape[0] != self.nj or qd.shape != q.shape:
            raise ValueError(f"q, qd must be float64 with shape ({self.nj}, n)")
        qdd = torch.empty_like(q)
        with torch.cuda.device(self.device):
            rc = self._lib.rbm_forward_dynamics_f64(self._h, _ptr(q), _ptr(qd), _ptr(u), 0.0, _ptr(qdd), None, None, q.shape[1], q.shape[1], self._stream())
        _lib.check(rc, "rbm_forward_dynamics")
        return qdd

    def step(self, q, qd, u=None, dt=0.002, inplace=False):
        """One semi-implicit Euler transition (q, qd) -> (q+, qd+) of the plant under joint forces u."""
        self._check_dev(q, qd, u)
        if q.dtype != torch.float64 or q.dim() != 2 or q.shape[0] != self.nj or qd.shape != q.shape:
            raise ValueError(f"q, qd must be float64 with shape ({self.nj}, n)")
        qn, qdn = (q, qd) if inplace else (torch.empty_like(q), torch.empty_like(qd))
        with torch.cuda.device(self.device):
            rc = self._lib.rbm_forward_dynamics_f64(self._h, _ptr(q), _ptr(qd), _ptr(u), float(dt), None, _ptr(qn), _ptr(qdn), q.shape[1], q.shape[1],
                                                    self._stream())
        _lib.check(rc, "rbm_forward_dynamics (step)")
        return qn, qdn


    # ---- closed-loop rollout -----------------------------------------------------------------------------
    def closed_loop(self, plan, gain, phi_sensed, q0, qd0=None, dt=None, fps=50.0, pos_residual_divisor=None, max_frames=None, want_final=True):
        """The reference's main loop (core/simulate.py:185-270) for n environments in ONE launch (one environment per thread).
        plan: planner.QuinticPlan;  gain: (nj, 2 nj);  phi_sensed: the 10 inertial parameters of the body hanging off the F/T sensor, in
        the sensor frame;  q0 [, qd0]: CUDA (nj, n) float64 initial states.  Returns a dict of device tensors:
          frames (F, 3 nj + 18, n) = [act (3 nj) | V_s | dV_s | wrench] per logged frame, frame_steps (F,) int32, final (3 nj, n)."""
        self._check_dev(q0, qd0)
        if q0.dtype != torch.float64 or q0.dim() != 2 or q0.shape[0] != self.nj or (qd0 is not None and (qd0.shape != q0.shape or qd0.dtype != q0.dtype)):
            raise ValueError(f"q0, qd0 must be float64 with shape ({self.nj}, n)")
        if len(plan.displacement) != self.nj or len(plan.pos_offset) != self.nj:
            raise ValueError(f"plan must have {self.nj} joints")
        n, nj = q0.shape[1], self.nj
        dt = float(plan.timestep if dt is None else dt)
        div = float(nj if pos_residual_divisor is None else pos_residual_divisor)  # the reference passes m.nu as mj_differentiatePos' dt
        K = torch.as_tensor(np.ascontiguousarray(gain, dtype=np.float64), device=self.device)
        if K.shape != (nj, 2 * nj):
            raise ValueError(f"gain must have shape ({nj}, {2 * nj})")
        ph = torch.as_tensor(np.ascontiguousarray(phi_sensed, dtype=np.float64), device=self.device)
        if ph.shape != (10,):
            raise ValueError("phi_sensed must hold the 10 inertial parameters")
        if max_frames is None:
            max_frames = int(np.ceil(plan.n_steps * dt * fps)) + 2
        frames = torch.zeros((max_frames, 3 * nj + 18, n), dtype=torch.float64, device=self.device)
        fsteps = torch.full((max_frames,), -1, dtype=torch.int32, device=self.device)
        nfr = torch.zeros(1, dtype=torch.int32, device=self.device)
        final = torch.empty((3 * nj, n), dtype=torch.float64, device=self.device) if want_final else None
        co = np.ascontiguousarray(plan.coeffs, dtype=np.float64)
        di = np.ascontiguousarray(plan.displacement, dtype=np.float64)
        of = np.ascontiguousarray(plan.pos_offset, dtype=np.float64)
        with torch.cuda.device(self.device):
            rc = self._lib.rbm_closed_loop_f64(self._h, _ptr(co), _ptr(di), _ptr(of), float(plan.timestep), float(plan.init_step), int(plan.n_steps),
                                               _ptr(K), _ptr(ph), dt, float(fps), div, _ptr(q0), _ptr(qd0), _ptr(frames), int(max_frames), _ptr(fsteps),
                                               _ptr(nfr), _ptr(final), n, n, self._stream())
        _lib.check(rc, "rbm_closed_loop")
        nf = min(int(nfr.item()), max_frames)
        return dict(frames=frames[:nf], frame_steps=fsteps[:nf], final=final, n_frames_total=int(nfr.item()))


# ---- model-free batched helpers (device tensors in, device tensors out) ------------------------------------
def _dev64(x, shape_tail):
    t = x if isinstance(x, torch.Tensor) else torch.as_tensor(np.asarray(x, dtype=np.float64))
    t = t.to(device="cuda", dtype=torch.float64).contiguous()
    if tuple(t.shape[1:]) != tuple(shape_tail):
        raise ValueError(f"expected trailing shape {tuple(shape_tail)}, got {tuple(t.shape[1:])}")
    return t


def _cur_stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def regressor_rows(twists, dtwists):
    """get_regressor_matrix batched: (n, 6), (n, 6) -> (n, 6, 10) on the device."""
    tw, dtw = _dev64(twists, (6,)), _dev64(dtwists, (6,))
    if tw.shape != dtw.shape:
        raise ValueError("twists and dtwists must have the same shape")
    Y = torch.empty((tw.shape[0], 6, 10), dtype=torch.float64, device=tw.device)
    _lib.check(_lib.load().rbm_regressor_rows_f64(_ptr(tw), _ptr(dtw), _ptr(Y), tw.shape[0], _cur_stream()), "rbm_regressor_rows")
    return Y


def sensor_twists(pose, twists, dtwists):
    """core/simulate.py:202-209 batched: V_s = Ad(T) V, dV_s = Ad(T) dV."""
    Rt = pose_to_Rt(pose)
    tw, dtw = _dev64(twists, (6,)), _dev64(dtwists, (6,))
    o1, o2 = torch.empty_like(tw), torch.empty_like(dtw)
    _lib.check(_lib.load().rbm_sensor_twists_f64(_ptr(Rt), _ptr(tw), _ptr(dtw), _ptr(o1), _ptr(o2), tw.shape[0], _cur_stream()), "rbm_sensor_twists")
    return o1, o2


def transfer_simat(poses_Rt, simats, adjoint_form=False):
    """transfer_simat (default) or coordinate_transfer_simat (adjoint_form=True), batched: (n,12), (n,6,6) -> (n,6,6)."""
    P, G = _dev64(poses_Rt, (12,)), _dev64(simats, (6, 6))
    if P.shape[0] != G.shape[0]:
        raise ValueError("The numbers of spatial inertia tensors and SE3 instances do not match.")
    out = torch.empty_like(G)
    lib = _lib.load()
    fn = lib.rbm_coordinate_transfer_simat_f64 if adjoint_form else lib.rbm_transfer_simat_f64
    _lib.check(fn(_ptr(P), _ptr(G), _ptr(out), P.shape[0], _cur_stream()), "rbm_transfer_simat")
    return out


def coordinate_transfer_imat(poses_Rt, imats, mass):
    P, I = _dev64(poses_Rt, (12,)), _dev64(imats, (3, 3))
    m = _dev64(np.atleast_1d(mass) if not isinstance(mass, torch.Tensor) else mass, ())
    out = torch.empty_like(I)
    _lib.check(_lib.load().rbm_coordinate_transfer_imat_f64(_ptr(P), _ptr(I), _ptr(m), _ptr(out), P.shape[0], _cur_stream()), "rbm_coordinate_transfer_imat")
    return out


def spatial_inertia(mass, diag):
    m = _dev64(np.atleast_1d(mass) if not isinstance(mass, torch.Tensor) else mass, ())
    d = _dev64(diag, (3,))
    if m.shape[0] != d.shape[0]:
        raise ValueError("Lenght of 'mass' of the bodies and that of 'diagonal_inertia' vectors must match.")
    out = torch.empty((m.shape[0], 6, 6), dtype=torch.float64, device=m.device)
    _lib.check(_lib.load().rbm_spatial_inertia_f64(_ptr(m), _ptr(d), _ptr(out), m.shape[0], _cur_stream()), "rbm_spatial_inertia")
    return out


def compose_poses(trans, rot):
    """(n,3) + (n,4) wxyz quaternions or (n,9) rotation matrices -> poses (n,12) and an int32 status vector."""
    rot_t = rot if isinstance(rot, torch.Tensor) else torch.as_tensor(np.asarray(rot, dtype=np.float64))
    rot_len = int(rot_t.shape[1])
    t, r = _dev64(trans, (3,)), _dev64(rot_t, (rot_len,))
    out = torch.empty((t.shape[0], 12), dtype=torch.float64, device=t.device)
    status = torch.empty((t.shape[0],), dtype=torch.int32, device=t.device)
    _lib.check(_lib.load().rbm_compose_f64(_ptr(t), _ptr(r), rot_len, _ptr(out), _ptr(status), t.shape[0], _cur_stream()), "rbm_compose")
    return out, status


def point_motion(twists, dtwists, points, want_acc=True):
    """extract_linvel / extract_linacc_frame_transferred batched -> (linvel (n,3), linacc (n,3) or None)."""
    tw, p = _dev64(twists, (6,)), _dev64(points, (3,))
    dtw = _dev64(dtwists, (6,)) if (want_acc and dtwists is not None) else None
    lv = torch.empty_like(p)
    la = torch.empty_like(p) if dtw is not None else None
    _lib.check(_lib.load().rbm_point_motion_f64(_ptr(tw), _ptr(dtw), _ptr(p), _ptr(lv), _ptr(la), p.shape[0], _cur_stream()), "rbm_point_motion")
    return lv, la
