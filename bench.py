#!/usr/bin/env python
"""Benchmark of the batched inverse-dynamics hot path (BASELINE.json metric: RNEA samples/s, % of HBM roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dtype f64|f32] [--samples B] [--dump-outputs DIR]
    python bench.py --impl reference ...        # the reference's CPU algorithm (oracle port) on the host cores

A "step" is one pass of the fused RNEA kernel over one resident batch of B synthetic (q, qd, qdd) samples
(BASELINE.json configs[1]: B = 2^20, fp64, the base.yaml manipulator + target object).  Under torchrun every rank
owns its own B samples (weak scaling, no data-path collective: samples are independent); the timed region is
bracketed by barrier + synchronize, device time is taken with CUDA events and the max over ranks is reported.
One JSON line is printed by rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "rnea_samples_per_s"
UNIT = "samples/s"
WORKLOAD = "configs[1]: batched inverse dynamics, 2^20 synthetic (q,qd,qdd) samples, base.yaml manipulator (sequential.xml) + hammer target"


def sample_states(rng, n):
    """SURVEY.md 8(d) config-2 distribution."""
    q = np.concatenate([rng.uniform(-1.5, 2.5, (n, 3)), rng.uniform(-6 * np.pi, 6 * np.pi, (n, 3))], axis=1)
    qd = rng.standard_normal((n, 6)) * np.array([1, 1, 1, 3, 3, 3.0])
    qdd = rng.standard_normal((n, 6)) * np.array([3, 3, 3, 10, 10, 10.0])
    return np.stack([q, qd, qdd], axis=1)


def load_constants():
    from rigid_body_manipulation_b200 import model as rbm_model

    return rbm_model.load_packaged("sequential", "hammer")


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi based, as the profiling recipe asks) during the timed region
# --------------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {
                pynvml.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                pynvml.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                pynvml.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                pynvml.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            }
            while not self._stop.is_set():
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.02)
        except Exception as e:  # pragma: no cover - depends on the box
            self.reasons.add(f"sampler_error:{type(e).__name__}")

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=2)

    def summary(self):
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "n_samples": len(self.samples)}


# --------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's per-sample algorithm on all host cores
# --------------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    consts, trajs = args
    from oracle import rnea_oracle as ro

    hposes = [ro.SE3(ro.SO3(np.array(r[:9]).reshape(3, 3)), np.array(r[9:])) for r in consts["hposes_Rt"]]
    t0 = time.perf_counter()
    acc = 0.0
    for tr in trajs:
        tau, _, _, _ = ro.inverse(tr, hposes, consts["simats"], consts["uscrews"], consts["twist_0"], consts["dtwist_0"])
        acc += float(tau[0])
    return time.perf_counter() - t0, acc


def cpu_reference_rate(consts, n_samples, cores=None, pool=None):
    """samples/s of the reference's algorithm (per-sample numpy + liegroups ops, oracle/rnea_oracle.py) on `cores` processes."""
    import multiprocessing as mp

    cores = cores or os.cpu_count() or 1
    trajs = sample_states(np.random.default_rng(123), n_samples)
    parts = [trajs[i::cores] for i in range(cores)]
    own = pool is None
    if own:
        pool = mp.get_context("fork").Pool(cores)
    try:
        t0 = time.perf_counter()
        pool.map(_cpu_worker, [(consts, p) for p in parts])
        wall = time.perf_counter() - t0
    finally:
        if own:
            pool.close()
            pool.join()
    return n_samples / wall, cores, wall


def consts_dict(c):
    return dict(hposes_Rt=c.hposes_Rt, simats=c.simats, uscrews=c.uscrews, twist_0=c.twist_0, dtwist_0=c.dtwist_0)


def run_reference_arm(args):
    """The reference's CPU algorithm for the path (per-sample oracle port; the reference itself is Python + an absent
    third-party dependency and cannot travel to the GPU box) on every host core, same metric / config as the GPU arm.
    Each step is a bounded sample of the workload, sized from a short calibration so the run ends within ~2 minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp

    c = load_constants()
    consts = consts_dict(c)
    cores = os.cpu_count() or 1
    pool = mp.get_context("fork").Pool(cores)
    try:
        rate, _, _ = cpu_reference_rate(consts, cores * 100, cores, pool)  # calibration (also warms the workers)
        budget_s = 90.0
        per_step = args.cpu_samples if args.cpu_samples > 0 else int(max(cores * 20, min(rate * budget_s / max(args.steps + args.warmup, 1), 4000 * cores)))
        for _ in range(args.warmup):
            cpu_reference_rate(consts, per_step, cores, pool)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            cpu_reference_rate(consts, per_step, cores, pool)
        wall = time.perf_counter() - t0
    finally:
        pool.close()
        pool.join()
    value = per_step * args.steps / wall
    sample = f"{per_step} samples/step of the configs[1] distribution, per-sample oracle port (oracle/rnea_oracle.py) over {cores} processes"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": {"workload": WORKLOAD, "batch_per_step": per_step, "layout": "AoS (3,6) per sample"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------------
L2_BYTES = 126e6
BASE_YAML_PLAN = dict(displacement=[0.2, 1.4, 0.6, np.pi, 0.0, 6 * np.pi], pos_offset=[1, 1, 1, 0, 0, 0], timestep=0.002, n_steps=1500)


class RneaWorkload:
    """configs[1] (and, with --dtype f32 / --samples, the configs[4] sweep): tau for B resident samples."""
    metric, unit = METRIC, UNIT
    launches_per_step = 1
    name = "rnea"

    def __init__(self, args, model, rank, torch, dtype=None, samples=None, host_buffers=True):
        dtype = dtype or args.dtype
        self.torch, self.model, self.B = torch, model, samples or args.samples
        self.dtype = dtype
        self.esize = 8 if dtype == "f64" else 4
        self.tdt = torch.float64 if dtype == "f64" else torch.float32
        self.alg_bytes = 24 * self.esize * self.B  # SURVEY.md 8(d): 18 scalars read + 6 written per sample
        live = int(model.live_inputs().sum())
        self.moved_bytes = (live + 6) * self.esize * self.B  # rows the kernel really loads + the 6 rows of tau it stores
        self.live_rows = live
        self.workload = WORKLOAD if (self.B == 1 << 20 and dtype == "f64") else f"batched inverse dynamics, {self.B} synthetic samples, {dtype}, base.yaml manipulator + hammer"
        npdt = np.float64 if dtype == "f64" else np.float32
        host = sample_states(np.random.default_rng(1000 + rank), self.B).astype(npdt)
        # L2 rule: rotate over enough independent buffer sets that the data touched between two uses of one set
        # exceeds 3x the 126 MB L2, so no timed launch can be served from cache
        self.nset = 1 if self.alg_bytes > 16 * L2_BYTES else max(2, int(np.ceil(3 * L2_BYTES / self.alg_bytes)) + 1)
        dev = torch.as_tensor(host, device="cuda")
        self.sets = []
        for i in range(self.nset):
            q, qd, qdd = (dev[:, k, :].t().contiguous() for k in range(3))
            if i:  # distinct values per set, same distribution
                q, qd, qdd = q + 1e-3 * i, qd * (1 + 1e-3 * i), qdd * (1 - 1e-3 * i)
            self.sets.append((q, qd, qdd, torch.empty_like(q)))
        del dev
        self.k = 0
        self.layout = "SoA [3][6][B] resident in HBM"
        if host_buffers:  # pinned host buffers of the end-to-end legs (allocated AFTER the NUMA binding of the process)
            self.traj_pinned = torch.as_tensor(host).pin_memory()                       # AoS (B, 3, 6): the reference's traj layout
            self.soa_pinned = [torch.as_tensor(np.ascontiguousarray(host[:, k, :].T)).pin_memory() for k in range(3)]  # (6, B) each
            self.tau_host = torch.empty((self.B, 6), dtype=self.tdt).pin_memory()
            self.tau_host_soa = torch.empty((6, self.B), dtype=self.tdt).pin_memory()
            from rigid_body_manipulation_b200 import planner

            self.plan = planner.QuinticPlan(**BASE_YAML_PLAN)
        # headline e2e: SoA host buffers, live rows only
        self.h2d, self.d2h = live * self.esize * self.B, 6 * self.esize * self.B
        self.e2e_api = (f"Model.rnea_host_soa -> rbm_rnea_host_soa_* (pinned host SoA q,qd,qdd in, pinned host tau out; the {live} rows the kernel reads are uploaded "
                        "(rbm_model_live_inputs), strided cudaMemcpy2DAsync per chunk, 3-stream pipeline)")

    def step(self):
        q, qd, qdd, tau = self.sets[self.k % self.nset]
        self.k += 1
        self.tau = self.model.rnea(q, qd, qdd, tau=tau)

    def outputs(self):
        """what the last step() returned to its caller: name -> (tensor, axis that runs over the samples)"""
        return {"tau": (self.tau, 1)}

    def e2e_step(self):
        self.model.rnea_host_soa(*self.soa_pinned, tau=self.tau_host_soa)

    # other end-to-end shapes of the same metric, reported beside the headline one
    def e2e_variants(self):
        B, es = self.B, self.esize
        stride = self.plan.n_steps / B  # B samples spread over the planned 1500 steps (fractional steps of the same quintic)
        return {
            "aos_host": (lambda: self.model.rnea_host(self.traj_pinned, tau=self.tau_host), 18 * es * B, 6 * es * B,
                         "Model.rnea_host -> rbm_rnea_host_*: the reference's (B,3,6) traj layout, all 18 values per sample uploaded"),
            "planned_host": (lambda: self.model.rnea_planned_host(self.plan, n=B, step0=0.0, stride=stride, dtype=self.tdt, tau=self.tau_host_soa), 0, 6 * es * B,
                             "Model.rnea_planned_host -> rbm_rnea_planned_host_*: base.yaml quintic evaluated in the kernel, only tau crosses the bus"),
        }


class GramWorkload:
    """configs[2] per-rank share: fused sensor-frame regressor + Gram of B samples (+ one 112-double all-reduce when N > 1)."""
    metric, unit = "regressor_gram_samples_per_s", "samples/s"
    launches_per_step = 2  # accumulate + finalize
    name = "gram"
    graphable = False  # 0.2-0.4 ms steps (and a collective at N > 1): the host is far from the critical path

    def __init__(self, args, model, rank, torch, dtype=None, samples=None, host_buffers=True):
        from rigid_body_manipulation_b200 import distributed

        dtype = dtype or args.dtype
        self.torch, self.model, self.B, self.dist = torch, model, samples or args.samples, distributed
        self.dtype = dtype
        self.esize = 8 if dtype == "f64" else 4
        self.tdt = torch.float64 if dtype == "f64" else torch.float32
        self.alg_bytes = 24 * self.esize * self.B  # q, qd, qdd, f read; nothing written per sample
        live = int(model.live_inputs().sum())
        self.moved_bytes = (live + 6) * self.esize * self.B  # live rows of q, qd, qdd + the 6 rows of f
        self.live_rows = live
        self.workload = f"configs[2] per-GPU share: regressor + Y^T Y / Y^T f Gram over {self.B} synthetic samples, {dtype}"
        gen = torch.Generator(device="cuda").manual_seed(1234 + rank)
        B = self.B
        self.nset = 1 if self.alg_bytes > 16 * L2_BYTES else max(2, int(np.ceil(3 * L2_BYTES / self.alg_bytes)) + 1)
        phi = np.array([0.585, -0.0032, 1.9e-5, -8e-6, 3.85e-3, 2.9e-3, 3.0e-3, 1e-5, 2e-5, -1e-5])
        self.sets = []
        for _ in range(self.nset):
            q = torch.empty((6, B), dtype=self.tdt, device="cuda")
            q[:3] = torch.rand((3, B), generator=gen, device="cuda", dtype=self.tdt) * 4 - 1.5
            q[3:] = (torch.rand((3, B), generator=gen, device="cuda", dtype=self.tdt) * 2 - 1) * (6 * np.pi)
            qd = torch.randn((6, B), generator=gen, device="cuda", dtype=self.tdt)
            qd[3:] *= 3
            qdd = torch.randn((6, B), generator=gen, device="cuda", dtype=self.tdt) * 3
            qdd[3:] *= 3.3333
            f = model.regressor_from_traj(q, qd, qdd, want_rows=False, phi=phi)["wrench"]
            self.sets.append((q, qd, qdd, f))
        self.pack = torch.empty(112, dtype=torch.float64, device="cuda")
        self.k = 0
        self.reducer = distributed.allreduce_gram  # torch.distributed / NCCL; replaced by NcclGramReducer for the second collective
        self.layout = "SoA q,qd,qdd,f [6][B] resident in HBM"
        if host_buffers:
            self.host = [t.cpu().pin_memory() for t in self.sets[0]]
            self.stage = [torch.empty_like(t) for t in self.sets[0]]
        self.h2d, self.d2h = 24 * self.esize * B, 112 * 8
        self.e2e_api = "pinned host q,qd,qdd,f -> cudaMemcpyAsync -> Model.regressor_gram -> pack.cpu()"

    def step(self):
        q, qd, qdd, f = self.sets[self.k % self.nset]
        self.k += 1
        self.model.regressor_gram(q, qd, qdd, f, pack=self.pack)
        self.reducer(self.pack)

    def outputs(self):
        return {"pack": (self.pack, None)}

    def local_step(self):
        """the same without the collective"""
        q, qd, qdd, f = self.sets[self.k % self.nset]
        self.k += 1
        self.model.regressor_gram(q, qd, qdd, f, pack=self.pack)

    def e2e_step(self):
        for h, d in zip(self.host, self.stage):
            d.copy_(h, non_blocking=True)
        self.model.regressor_gram(*self.stage, pack=self.pack)
        self.reducer(self.pack)
        return self.pack.cpu()

    def e2e_variants(self):
        return {}


def planned_states(rng, n, sigma=0.05):
    """configs[3] / SURVEY.md 8(d) config 4: joint states along the planned base.yaml trajectory -- a random (fractional) step of
    the quintic per state -- plus a small N(0, sigma) offset on positions and velocities."""
    from rigid_body_manipulation_b200 import planner

    plan = planner.QuinticPlan(**BASE_YAML_PLAN)
    traj = plan.trajectory(rng.uniform(0.0, plan.n_steps, n))  # (n, 3, 6)
    q = traj[:, 0, :] + sigma * rng.standard_normal((n, 6))
    qd = traj[:, 1, :] + sigma * rng.standard_normal((n, 6))
    return q, qd


class LinearizeWorkload:
    """configs[3]: A (12x12), B (12x6) of the discrete transition at B joint states (RNEA-based finite differences)."""
    metric, unit = "lqr_linearizations_per_s", "states/s"
    launches_per_step = 1
    name = "linearize"
    graphable = False  # 0.35 ms steps

    def __init__(self, args, model, rank, torch, dtype=None, samples=None, host_buffers=True):
        self.torch, self.model, self.B = torch, model, samples or args.samples
        self.dtype = "f64"
        self.esize, self.tdt = 8, torch.float64
        self.alg_bytes = 228 * 8 * self.B  # 12 scalars read, 144 + 72 written per state (SURVEY.md 8(d))
        live_q = int(model.live_inputs()[0].sum())
        self.moved_bytes = (live_q + 6 + 216) * 8 * self.B
        self.live_rows = live_q + 6
        self.workload = (f"configs[3]: LQR linearisation (A 12x12, B 12x6) at {self.B} joint states along the planned base.yaml trajectory "
                         "(random step + N(0, 0.05)), centred FD eps 1e-8, dt 0.002, f64")
        q, qd = planned_states(np.random.default_rng(2000 + rank), self.B)
        self.q = torch.as_tensor(np.ascontiguousarray(q.T), device="cuda")
        self.qd = torch.as_tensor(np.ascontiguousarray(qd.T), device="cuda")
        self.nset = 1
        self.layout = "SoA q,qd [6][B] in; element-major A [144][B], B [72][B] out (output alone is 1.7 KB/state >> L2 for B = 2^20)"
        self.h2d, self.d2h = 12 * 8 * self.B, 216 * 8 * self.B
        self.e2e_api = "pinned host q,qd -> Model.linearize -> A,B copied to pinned host"
        if host_buffers:
            self.qh, self.qdh = self.q.cpu().pin_memory(), self.qd.cpu().pin_memory()
            self.Ah = torch.empty((12, 12, self.B), dtype=self.tdt).pin_memory()
            self.Bh = torch.empty((12, 6, self.B), dtype=self.tdt).pin_memory()

    def step(self):
        self.out = self.model.linearize(self.q, self.qd, None, dt=0.002, eps=1e-8, centered=True)

    def outputs(self):
        return {"A": (self.out[0], 0), "B": (self.out[1], 0)}

    def e2e_step(self):
        q, qd = self.qh.cuda(non_blocking=True), self.qdh.cuda(non_blocking=True)
        A, Bm = self.model.linearize(q, qd, None, dt=0.002, eps=1e-8, centered=True)
        self.Ah.copy_(A.permute(1, 2, 0), non_blocking=True)
        self.Bh.copy_(Bm.permute(1, 2, 0), non_blocking=True)
        self.torch.cuda.synchronize()

    def e2e_variants(self):
        return {}


WORKLOADS = {"rnea": RneaWorkload, "gram": GramWorkload, "linearize": LinearizeWorkload}


class Timer:
    """Device-side timing shared by the primary workload and the extras: barrier + synchronize on both sides, CUDA events on the
    launching stream, max over ranks.  Every count that governs a loop containing a collective is identical on all ranks."""

    def __init__(self, torch, dist, world):
        self.torch, self.dist, self.world = torch, dist, world

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def heat_count(self, step, seconds):
        """how many untimed steps fill `seconds` -- derived from a max-reduced estimate, never from a per-rank wall-clock loop"""
        t0 = time.perf_counter()
        for _ in range(3):
            step()
        self.torch.cuda.synchronize()
        (est,) = self.max_over_ranks([(time.perf_counter() - t0) / 3])
        return int(min(20000, max(10, seconds / max(est, 1e-6))))

    def capture(self, step, steps):
        """CUDA graph of `steps` back-to-back steps (the library launches on torch's current stream, so its launches -- programmatic
        dependent launch attributes included -- are captured as issued), or None when the capture fails.  A 2^20-sample launch lasts
        ~30 us and one call through Python + ctypes costs ~14 us of host time (tools/bench_launch_overhead.py): on a busy host an eager
        loop starves the GPU; replaying a graph takes the host out of the timed region."""
        torch = self.torch
        try:
            g = torch.cuda.CUDAGraph()
            # thread_local: NCCL's watchdog thread polls events while this thread captures (multi-rank runs)
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                for _ in range(steps):
                    step()
            g.replay()  # one untimed replay
            torch.cuda.synchronize()
            return g
        except Exception:  # pragma: no cover - depends on the driver
            try:
                torch.cuda.synchronize()
            except Exception:
                pass
            return None

    def timed(self, step, steps, graph=None):
        """total ms for exactly `steps` back-to-back steps (max over ranks); `graph` = those steps captured by capture()"""
        torch = self.torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        if graph is not None:
            graph.replay()
        else:
            for _ in range(steps):
                step()
        e1.record()
        self.barrier()
        return self.max_over_ranks([e0.elapsed_time(e1)])[0]

    def isolated(self, step, steps):
        """mean of per-launch event pairs (contains the stream bubbles the event records insert)"""
        torch = self.torch
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in evs:
            a.record()
            step()
            b.record()
        self.barrier()
        return self.max_over_ranks([float(np.mean([a.elapsed_time(b) for a, b in evs]))])[0]

    def wall(self, step, steps, warm):
        """host wall-clock seconds for `steps` calls of a synchronous end-to-end step (max over ranks)"""
        for _ in range(warm):
            step()
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        self.barrier()
        return self.max_over_ranks([time.perf_counter() - t0])[0]


def roofline_block(wl, kern_ms_avg, kern_ms_isolated, traffic):
    peak, peak_src = measured_peak_gbs()
    achieved = wl.alg_bytes / (kern_ms_avg * 1e-3) / 1e9
    moved = wl.moved_bytes / (kern_ms_avg * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "peak_source": peak_src, "kernel_ms": kern_ms_avg, "kernel_ms_isolated": kern_ms_isolated,
            "algorithmic_bytes_per_launch": wl.alg_bytes,
            # the kernel does not load rows its result cannot depend on (rbm_model_live_inputs): `frac` is on SURVEY 8(d)'s contract
            # bytes, `frac_moved` on the bytes the launch really moves through DRAM
            "bytes_moved_per_launch": wl.moved_bytes, "achieved_moved": moved, "frac_moved": moved / peak, "live_input_rows": wl.live_rows}


DUMP_BYTES = 64 << 20


def sample_outputs(outputs):
    """Device copies of a step's outputs (name -> (tensor, sample axis or None)), at most DUMP_BYTES in all.  When the outputs are
    larger, every output that runs over the samples keeps the same sorted subset of them, drawn with a fixed seed, so two runs with
    the same arguments keep the same samples.  Returns the copies and the number of samples kept (None = all)."""
    import torch

    nbytes = lambda t: t.numel() * t.element_size()
    total = sum(nbytes(t) for t, _ in outputs.values())
    keep = None
    if total > DUMP_BYTES:
        (n,) = {t.shape[ax] for t, ax in outputs.values() if ax is not None}
        fixed = sum(nbytes(t) for t, ax in outputs.values() if ax is None)
        k = int((DUMP_BYTES - fixed) // ((total - fixed) / n))
        keep = np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    out = {}
    for name, (t, ax) in outputs.items():
        if keep is not None and ax is not None:
            t = t.index_select(ax, torch.as_tensor(keep, device=t.device))
        out[name] = t.clone()
    return out, None if keep is None else len(keep)


def write_outputs(dirname, outputs):
    os.makedirs(dirname, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(dirname, f"{name}.npy"), t.cpu().numpy())


def traffic_entry(key):
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            return json.load(f).get(key)
    return None


def gram_extra(args, model, rank, world, local, torch, dist, tm, dtype):
    """configs[2] share of this rank (12.5 M samples; 100 M at 8 GPUs) with the all-reduce INSIDE the timed step, through both
    collectives, plus the collective timed alone and parity of the reduced pack."""
    from rigid_body_manipulation_b200 import distributed

    wl = GramWorkload(args, model, rank, torch, dtype=dtype, samples=args.gram_samples, host_buffers=False)
    steps = max(5, min(args.steps, 20))
    out = {"samples_per_gpu": wl.B, "samples_total": wl.B * world, "dtype": dtype, "steps": steps}
    for _ in range(3):
        wl.step()
    n_heat = tm.heat_count(wl.step, 0.15)
    for _ in range(n_heat):
        wl.step()
    ms = tm.timed(wl.step, steps)
    out["collective"] = "torch-nccl" if world > 1 else "none (1 rank)"
    out["value"] = world * wl.B * steps / (ms * 1e-3)
    out["ms_per_step"] = ms / steps
    rl = roofline_block(wl, ms / steps, None, traffic_entry(f"gram_{dtype}_{wl.B}"))
    out.update(frac=rl["frac"], frac_moved=rl["frac_moved"], achieved=rl["achieved"], achieved_moved=rl["achieved_moved"])
    ms_local = tm.timed(wl.local_step, steps)
    out["ms_per_step_no_collective"] = ms_local / steps
    # parity of the reduced pack: local packs gathered and summed on the host in rank order vs the all-reduced pack
    wl.k = 0
    wl.local_step()
    local_pack = wl.pack.clone()
    torch.cuda.synchronize()
    if world > 1:
        gathered = [torch.empty_like(local_pack) for _ in range(world)]
        dist.all_gather(gathered, local_pack)
        ref = torch.stack(gathered).cpu().numpy().sum(axis=0)
        p1 = local_pack.clone()
        distributed.allreduce_gram(p1)
        red = distributed.NcclGramReducer(local)  # the C ABI's own collective (rbm_allreduce_gram_n); constructed collectively
        p2 = local_pack.clone()
        red(p2)
        torch.cuda.synchronize()
        a1, a2 = p1.cpu().numpy(), p2.cpu().numpy()
        scale = np.abs(ref[:100]).max()
        out["pack_n_ok"] = bool(a1[111] == world * wl.B and a2[111] == world * wl.B)
        out["pack_matches_allgather_sum"] = bool(np.abs(a1 - ref).max() <= 1e-12 * scale)
        out["pack_vs_allgather_max_rel"] = float(np.abs(a1 - ref).max() / scale)
        out["collectives_bit_identical"] = bool(np.array_equal(a1, a2))
        # the collective alone (both bindings), and the whole step again through the library's own collective
        scratch = local_pack.clone()
        n_ar = 200
        ms_ar = tm.timed(lambda: distributed.allreduce_gram(scratch), n_ar)
        scratch.copy_(local_pack)
        ms_ar2 = tm.timed(lambda: red(scratch), n_ar)
        out["allreduce_us"] = 1e3 * ms_ar / n_ar
        out["allreduce_us_rbm"] = 1e3 * ms_ar2 / n_ar
        wl.reducer = red
        for _ in range(3):
            wl.step()
        ms2 = tm.timed(wl.step, steps)
        # the three legs again in the opposite order, best of two each: the FP64-heavy Gram kernel is clock-sensitive and the SM clock
        # drifts over the first seconds of load, so a single pass would favour whichever leg runs last
        ms2 = min(ms2, tm.timed(wl.step, steps))
        ms_local = min(ms_local, tm.timed(wl.local_step, steps))
        wl.reducer = distributed.allreduce_gram
        ms = min(ms, tm.timed(wl.step, steps))
        out["value"] = world * wl.B * steps / (ms * 1e-3)
        out["ms_per_step"] = ms / steps
        out["ms_per_step_no_collective"] = ms_local / steps
        rl = roofline_block(wl, ms / steps, None, traffic_entry(f"gram_{dtype}_{wl.B}"))
        out.update(frac=rl["frac"], frac_moved=rl["frac_moved"], achieved=rl["achieved"], achieved_moved=rl["achieved_moved"])
        out["rbm_allreduce_gram_n"] = {"value": world * wl.B * steps / (ms2 * 1e-3), "ms_per_step": ms2 / steps,
                                       "frac": wl.alg_bytes / (ms2 / steps * 1e-3) / 1e9 / rl["peak"]}
        red.close()
    else:
        out["pack_n_ok"] = bool(local_pack[111].item() == wl.B)
    del wl
    torch.cuda.empty_cache()
    return out


def small_extra(cls, args, model, rank, world, torch, tm, dtype, samples):
    wl = cls(args, model, rank, torch, dtype=dtype, samples=samples, host_buffers=False)
    steps = max(5, min(args.steps, 20))
    for _ in range(3):
        wl.step()
    for _ in range(tm.heat_count(wl.step, 0.1)):
        wl.step()
    ms = tm.timed(wl.step, steps)
    rl = roofline_block(wl, ms / steps, None, traffic_entry(f"{wl.name}_{wl.dtype}_{wl.B}"))
    out = {"workload": wl.workload, "metric": wl.metric, "unit": wl.unit, "value": world * wl.B * steps / (ms * 1e-3), "ms_per_step": ms / steps, "steps": steps,
           "frac": rl["frac"], "frac_moved": rl["frac_moved"], "achieved": rl["achieved"], "achieved_moved": rl["achieved_moved"], "traffic": rl["traffic"]}
    del wl
    torch.cuda.empty_cache()
    return out


def generic_extra(args, rank, world, local, torch, tm):
    """The any-model kernel on a model with NO structure (tests/golden/ref_inverse_generic_nj6.npz: general screws, dense SPD inertias,
    moving base, tip wrench).  It is bound by the FP64 pipe, not by HBM: 1680 FP64 instructions per sample (ncu,
    profiles/r2_generic_nj6_ncu_full.csv) against 64 FP64 lanes per SM and clock."""
    from rigid_body_manipulation_b200.engine import Model

    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "tests", "golden", "ref_inverse_generic_nj6.npz")
    if not os.path.exists(path):
        return {"skipped": "tests/golden/ref_inverse_generic_nj6.npz not found"}
    g = np.load(path)
    gm = Model(g["hposes_Rt"], g["simats"], g["uscrews"], g["twist_0"], g["dtwist_0"], wrench_tip=g["wrench_tip"], pose_tip_ee=g["pose_tip"], device=local)
    out = {}
    sms = torch.cuda.get_device_properties(local).multi_processor_count
    for dtype in ("f64", "f32"):
        r = small_extra(RneaWorkload, args, gm, rank, world, torch, tm, dtype, 1 << 22)
        r["workload"] = f"batched inverse dynamics, generic kernel, structure-free 6-joint model, {1 << 22} samples, {dtype}"
        r["kernel_path"] = gm.kernel_path
        if dtype == "f64":
            ceiling = sms * 64 * 1.965e9 / 1680.0  # samples/s per GPU at 100 % FP64-pipe utilisation and the maximum SM clock
            r["bound"] = "fp64 pipe"
            r["fp64_instructions_per_sample"] = 1680
            r["fp64_ceiling_samples_per_s"] = world * ceiling
            r["frac_of_fp64_ceiling"] = r["value"] / (world * ceiling)
        out[dtype] = r
    del gm
    return out


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    # NUMA: pin this rank (and therefore the pinned host buffers it allocates below) to the GPU's own socket
    numa = {"bound": False, "why": "disabled (--no-numa)"}
    if not args.no_numa:
        from rigid_body_manipulation_b200 import numa as rbm_numa

        try:
            numa = rbm_numa.bind_to_device(local)
        except Exception as e:  # pragma: no cover - depends on the box
            numa = {"bound": False, "why": f"{type(e).__name__}: {e}"}
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from rigid_body_manipulation_b200.engine import Model

    c = load_constants()
    model = Model(c.hposes_Rt, c.simats, c.uscrews, c.twist_0, c.dtwist_0, pose_sen_llj=c.pose_sen_Rt, device=local)
    wl = WORKLOADS[args.workload](args, model, rank, torch)
    B = wl.B
    tm = Timer(torch, dist, world)

    # ---- device-resident throughput -------------------------------------------------------------------
    for _ in range(args.warmup):
        wl.step()
    tm.barrier()
    n_heat = tm.heat_count(wl.step, 0.3)  # ~0.3 s of untimed steps so that the clock sampler sees loaded clocks
    tm.barrier()
    # the K timed steps as one CUDA graph (workloads whose step contains a collective stay eager); every rank decides alike.  In both
    # launch modes they start at input set 0, so the inputs of the last one depend on the arguments alone (the number of heat steps
    # before an eager pass comes from a timing estimate)
    graph = None
    if not args.eager and getattr(wl, "graphable", True):
        wl.k = 0
        graph = tm.capture(wl.step, args.steps)
        (ok,) = tm.max_over_ranks([0.0 if graph is not None else 1.0])
        if ok != 0.0:
            graph = None
    graph_outputs = wl.outputs() if graph is not None else None  # the buffers the graph's last captured step writes
    dump = None
    with ClockSampler(local) as clk:
        for _ in range(n_heat):
            wl.step()
        wl.k = 0
        # pass 1 -- the reported value: exactly K steps back to back, bracketed by barrier + synchronize
        total_ms = tm.timed(wl.step, args.steps, graph=graph)
        if args.dump_outputs and rank == 0:  # copied before pass 2 runs more steps into the same buffers
            dump = sample_outputs(graph_outputs or wl.outputs())
        # pass 2 -- per-launch durations (an event pair around every launch, same stream)
        kern_ms_isolated = tm.isolated(wl.step, args.steps)
    if dump is not None:
        write_outputs(args.dump_outputs, dump[0])
    # one step == one launch of the dominant kernel (plus, for the Gram workload, a single-CTA finalisation): its average
    # launch duration over the timed region is total / K.  The isolated figure (event pair around every launch) additionally
    # contains the stream bubbles that event records insert between launches and is reported for reference.
    kern_ms_avg = total_ms / args.steps
    value = world * B * args.steps / (total_ms * 1e-3)

    # ---- end to end through the public API (pinned host buffers; H2D + kernel + D2H inside the timed region) ----
    e2e_steps = max(1, min(args.steps, 20))
    e2e_warm = max(1, min(args.warmup, 3))
    e2e_s = tm.wall(wl.e2e_step, e2e_steps, e2e_warm)
    e2e_value = world * B * e2e_steps / e2e_s
    e2e_variants = {}
    for name, (fn, h2d, d2h, api) in wl.e2e_variants().items():
        s_ = tm.wall(fn, e2e_steps, e2e_warm)
        e2e_variants[name] = {"value": world * B * e2e_steps / s_, "unit": wl.unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "api": api}
    numa_all = [None] * world
    if world > 1:
        dist.all_gather_object(numa_all, {k: numa.get(k) for k in ("pci", "numa_node", "bound", "n_cpus", "mempolicy", "why")})
    else:
        numa_all = [{k: numa.get(k) for k in ("pci", "numa_node", "bound", "n_cpus", "mempolicy", "why")}]

    # ---- the other BASELINE configs, attached to the same line (every rank takes part: some contain collectives) ----
    extra = {}
    if args.workload == "rnea" and not args.no_extra:
        del wl.sets
        torch.cuda.empty_cache()
        extra["gram"] = {"f64": gram_extra(args, model, rank, world, local, torch, dist, tm, "f64"),
                         "f32": gram_extra(args, model, rank, world, local, torch, dist, tm, "f32")}
        extra["linearize"] = small_extra(LinearizeWorkload, args, model, rank, world, torch, tm, "f64", 1 << 20)
        extra["rnea_f32"] = small_extra(RneaWorkload, args, model, rank, world, torch, tm, "f32", 1 << 24)
        extra["rnea_generic"] = generic_extra(args, rank, world, local, torch, tm)

    if rank == 0:
        line = {
            "metric": wl.metric, "value": value, "unit": wl.unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": wl.dtype, "data": "synthetic",
            "config": {"workload": wl.workload, "batch_per_gpu": B, "layout": wl.layout, "kernel_path": model.kernel_path,
                       "l2_policy": (f"{wl.nset} rotating buffer set(s) x {wl.alg_bytes / 1e6:.0f} MB algorithmic bytes per step (L2 = 126 MB)" if wl.nset > 1
                                     else f"inputs of one step ({wl.alg_bytes / 1e6:.0f} MB) exceed the 126 MB L2"),
                       "parallelism": (f"samples sharded x{world}, no collective on this workload" if args.workload != "gram" or world == 1
                                       else f"samples sharded x{world}, one 112-double NCCL all-reduce per step")
                       + ("; extra.gram: configs[2] share per rank with the NCCL all-reduce inside the timed step" if extra else ""),
                       "launch_mode": (f"CUDA graph of the {args.steps} timed steps, replayed once inside the timed region" if graph is not None
                                       else "eager: one library call per step from the Python loop"),
                       "numa": numa_all},
            "roofline": roofline_block(wl, kern_ms_avg, kern_ms_isolated, traffic_entry(f"{args.workload}_{wl.dtype}_{B}")),
            "e2e": {"value": e2e_value, "unit": wl.unit, "h2d_bytes_per_step": wl.h2d, "d2h_bytes_per_step": wl.d2h, "api": wl.e2e_api, "steps": e2e_steps,
                    "variants": e2e_variants},
            "gpu_launches": args.steps * wl.launches_per_step,
            "clocks": clk.summary(),
        }
        if extra:
            line["extra"] = extra
        if dump is not None:
            line["outputs"] = {"dir": args.dump_outputs, "arrays": {k: list(t.shape) for k, t in dump[0].items()},
                               "samples_kept": dump[1] if dump[1] is not None else "all"}
        if world == 1 and not args.no_cpu and args.workload == "rnea":
            if numa.get("bound"):  # the CPU leg forks one worker per host core: undo the socket-local CPU binding first
                from rigid_body_manipulation_b200 import numa as rbm_numa

                rbm_numa.restore_affinity(numa)
            consts = consts_dict(c)
            cores = os.cpu_count() or 1
            rate, _, _ = cpu_reference_rate(consts, cores * 100, cores)  # calibration
            n_cpu = args.cpu_samples if args.cpu_samples > 0 else int(max(cores * 100, rate * 15.0))  # ~15 s of CPU work
            v, cores, wall = cpu_reference_rate(consts, n_cpu, cores)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"{n_cpu} samples of the same distribution, per-sample oracle port of reference dynamics.inverse, {wall:.1f} s wall on {cores} processes"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--workload", default="rnea", choices=["rnea", "gram", "linearize"], help="rnea = BASELINE.json configs[1] (the headline)")
    ap.add_argument("--samples", type=int, default=1 << 20, help="samples (states) per GPU per step")
    ap.add_argument("--cpu-samples", type=int, default=0, help="CPU baseline sample count (0 = auto)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--eager", action="store_true", help="time an eager Python loop of library calls instead of replaying a CUDA graph of the K steps")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra.* legs (configs[2] Gram + all-reduce, configs[3] linearisation, fp32 RNEA)")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to the GPU's NUMA node")
    ap.add_argument("--gram-samples", type=int, default=12_500_000, help="samples per GPU of the extra.gram leg (12.5 M x 8 GPUs = configs[2]'s 100 M)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (rank 0's shard; at most 64 MB in all, larger outputs "
                         "keep a fixed seeded subset of the samples), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
