"""Throughput of the joint-torque payload Gram (Model.payload_gram) with the F/T Gram (Model.regressor_gram) as the yardstick.

    python tools/bench_payload_gram.py [--n 12500000] [--rounds 5] [--launches 4] [--warmup 3] [--out FILE]

12.5 M samples per GPU is BASELINE configs[2]'s per-GPU share.  For fp64 and fp32, on the packaged robot (the object-free model for
the payload route, the model with the hammer for the F/T route, both the fast sequential path) and on the same models forced onto the
generic path, the two Grams run on the same seeded device inputs (q, qd, qdd and either tau or the wrench f).  Timing: CUDA events
around `--launches` back-to-back launches, the two routes alternating for `--rounds` rounds after `--warmup` launches of each, so
clock and neighbour drift hit both alike (>= 20 timed launches per route and configuration by default).  The inputs (1.8-3 GB) are
larger than L2, so every pass reads HBM.  Bytes per sample count what the kernels load: the payload fast path 18 rows (q[3..5],
qd[3..5], qdd, tau), the F/T fast path 21 (q[3..5], qd, qdd, f), both generic kernels 24.  Prints one JSON line with G samples/s,
bytes per sample and the fraction of 6550 GB/s, together with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HBM_GBS = 6550.0
ROWS = {("payload", "fast"): 18, ("ft", "fast"): 21, ("payload", "generic"): 24, ("ft", "generic"): 24}


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout
    name, power = [x.strip() for x in out.strip().splitlines()[0].split(",")]
    return dict(name=name, power_limit=power)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=12_500_000)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--launches", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()

    import torch

    from rigid_body_manipulation_b200 import model as pm
    from rigid_body_manipulation_b200.engine import Model

    if not torch.cuda.is_available():
        raise SystemExit("bench_payload_gram needs a CUDA device")
    info = card()
    c0, c1 = pm.load_packaged("sequential", None), pm.load_packaged("sequential", "hammer")
    mk = lambda c, fg: Model(c.hposes_Rt, c.simats, c.uscrews, c.twist_0, c.dtwist_0, pose_sen_llj=c.pose_sen_Rt, force_generic=fg)
    n = a.n
    result = dict(n=n, card=info, hbm_peak_GBs=HBM_GBS, configs={})
    for dname, dt in (("f64", torch.float64), ("f32", torch.float32)):
        gen = torch.Generator(device="cuda").manual_seed(11)
        q = (torch.rand((6, n), generator=gen, device="cuda", dtype=dt) * 2 - 1) * 6
        qd = torch.randn((6, n), generator=gen, device="cuda", dtype=dt)
        qdd = torch.randn((6, n), generator=gen, device="cuda", dtype=dt) * 3
        tau = torch.randn((6, n), generator=gen, device="cuda", dtype=dt) * 20
        f = torch.randn((6, n), generator=gen, device="cuda", dtype=dt) * 2
        for path, fg in (("fast", False), ("generic", True)):
            m0, m1 = mk(c0, fg), mk(c1, fg)
            pack = torch.empty(112, dtype=torch.float64, device="cuda")
            runs = dict(payload=lambda: m0.payload_gram(q, qd, qdd, tau, pack=pack), ft=lambda: m1.regressor_gram(q, qd, qdd, f, pack=pack))
            for fn in runs.values():
                for _ in range(a.warmup):
                    fn()
            torch.cuda.synchronize()
            times = {k: [] for k in runs}
            for _ in range(a.rounds):
                for k, fn in runs.items():
                    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s.record()
                    for _ in range(a.launches):
                        fn()
                    e.record()
                    e.synchronize()
                    times[k].append(s.elapsed_time(e) / 1e3 / a.launches)
            for k, ts in times.items():
                t = float(np.median(ts))
                bps = ROWS[(k, path)] * (8 if dt == torch.float64 else 4)
                result["configs"][f"{k}_{path}_{dname}"] = dict(
                    kernel_path=(m0 if k == "payload" else m1).kernel_path, G_samples_per_s=n / t / 1e9, seconds_median=t,
                    seconds_min=float(min(ts)), seconds_max=float(max(ts)), timed_launches=a.rounds * a.launches, bytes_per_sample=bps,
                    fraction_of_hbm=n * bps / t / (HBM_GBS * 1e9))
            del m0, m1
        del q, qd, qdd, tau, f
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if a.out:
        with open(a.out, "a") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
