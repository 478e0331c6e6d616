"""A/B of the compile-time-shape TMA-input kernel (MTG_OPT_V5_STATIC_SHAPE on = 0, off = -1) in one process.

For each configuration the two arms alternate for --rounds rounds on the same resident inputs (bench.py's generator and
seed); a sample is the mean of 20 launches timed with CUDA events.  Per arm: median / min / max ms, trajectories/s and
the HBM fraction against the peak bench.py uses; per configuration: bitwise equality of coefficients, status and d_free
between the arms.  One JSON line per configuration.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

import bench
import mav_trajectory_generation_b200 as m

ARMS = (("off", -1), ("on", 0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C5,C3,C2,C4")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--launches", type=int, default=20)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    peak, peak_src = bench.measured_peaks()
    s = m.Solver(0)
    for cfg in args.configs.split(","):
        N, r, K, D, B = bench.CONFIGS[cfg]
        prob = m.Problem(N, r, K, D)
        _, times, dfix = bench.synth_batch(torch, N, K, D, B, dev, seed=4321)
        outs, ms = {}, {name: [] for name, _ in ARMS}
        for name, val in ARMS:  # untimed warm-up of both arms, and their outputs
            s.set_option(m.capi.OPT_V5_STATIC_SHAPE, val)
            coeffs = torch.empty((B, K, D, N), dtype=torch.float64, device=dev)
            status = torch.full((B,), -1, dtype=torch.int32, device=dev)
            dfree = torch.empty((B, D, prob.n_free), dtype=torch.float64, device=dev)
            s.solve_linear(prob, times, dfix, coeffs=coeffs, d_free=dfree, status=status)
            torch.cuda.synchronize()
            outs[name] = (coeffs, status, dfree)
        coeffs = torch.empty((B, K, D, N), dtype=torch.float64, device=dev)
        for _ in range(args.rounds):
            for name, val in ARMS:
                s.set_option(m.capi.OPT_V5_STATIC_SHAPE, val)
                for _ in range(3):
                    s.solve_linear(prob, times, dfix, coeffs=coeffs)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.launches):
                    s.solve_linear(prob, times, dfix, coeffs=coeffs)
                e1.record()
                torch.cuda.synchronize()
                ms[name].append(e0.elapsed_time(e1) / args.launches)
        nbytes = prob.bytes_per_trajectory * B
        row = {"config": cfg, "batch": B, "K": K, "N": N, "r": r, "D": D, "rounds": args.rounds,
               "launches_per_sample": args.launches, "hbm_peak_GBps": peak, "peak_source": peak_src}
        for name, _ in ARMS:
            med = statistics.median(ms[name])
            row[name] = {"median_ms": round(med, 4), "min_ms": round(min(ms[name]), 4), "max_ms": round(max(ms[name]), 4),
                         "traj_per_s": round(B / (med * 1e-3)), "frac_of_hbm_peak": round(nbytes / (med * 1e-3) / 1e9 / peak, 4),
                         "samples_ms": [round(x, 4) for x in ms[name]]}
        row["median_gain"] = round(row["off"]["median_ms"] / row["on"]["median_ms"] - 1.0, 4)
        row["on_worst_beats_off_best"] = row["on"]["max_ms"] < row["off"]["min_ms"]
        a, b = outs["off"], outs["on"]
        row["bitwise_equal"] = {"coeffs": bool(torch.equal(a[0], b[0])), "status": bool(torch.equal(a[1], b[1])),
                                "d_free": bool(torch.equal(a[2], b[2]))}
        row["status_all_zero"] = bool((a[1] == 0).all().item())
        print(json.dumps(row), flush=True)
        del outs, coeffs, times, dfix
    s.close()


if __name__ == "__main__":
    main()
