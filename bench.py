#!/usr/bin/env python3
"""bench.py -- min-snap trajectories/sec of the batched solveLinear() hot path on B200.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun)
  python bench.py --impl reference --gpus N --steps K --warmup W

A "step" = one pass of the hot path over one batch of synthetic random-waypoint trajectories.
Default workload = BASELINE.json config C5: 1 048 576 trajectories x 16 segments, 3-D, N=10 min-snap,
fp64, STRONG scaling: the batch is sharded over the job's N GPUs (N=1: the whole batch on one GPU --
the per-trajectory configuration is the headline C3's).  Prints ONE JSON line (rank 0).

  value      whole-job trajectories/s of the compute phase, shards resident in HBM (CUDA events on the
             launching stream, barrier + synchronize on both sides, max over ranks).
  scatter_gather (N>1)  the full BASELINE C5 data path: rank 0 holds the batch; chunked, full-duplex NCCL
             send/recv of the inputs out and the coefficients back, overlapped with the solves
             (mav_trajectory_generation_b200/sharding.py); root NVLink ingest GB/s against the measured
             770 GB/s peer-copy figure of B200_PROFILING.md.  Two NVLink peer-memory forms of the same job
             are timed beside it: `fused_peer_store` (every rank's solve kernel TMA-stores its coefficients
             into the root's output, no gather step) and `peer_dma_pipeline` (copy engines pull the inputs
             and push the coefficients, chunked over three streams); `best_path` names the fastest.
  e2e        same metric through the host-pointer C-ABI call (what
             PolynomialOptimization<N>::solveLinear() / BatchPolynomialOptimization calls):
             pinned HOST buffers (bound to the GPU's NUMA node), H2D + kernels + D2H inside the timed region.
  roofline   HBM: algorithmic bytes/launch (4568 B/trajectory, SURVEY.md 8d) / kernel time,
             against MEASURED_PEAKS.json hbm_gbs.
  configs (N=1)  the other single-GPU configurations with their own roofline fractions: C3 (262 144 x 16,
             the headline batch), C2, C4, K=50 and K=100 (the reference timing program's sizes,
             polynomial_timing_evaluation.cpp:114-129), a generic (non-waypoint) mask, B=1 latency.
  cpu_baseline  the CPU oracle (restatement of the reference's Eigen path, oracle/oracle.cpp)
             on all usable host cores (affinity and cgroup quota respected), bounded sample (rank 0, N=1).

--dump-outputs DIR  after the timed steps, writes what the last one computed -- the coefficients and the per-trajectory
             status of a fixed, seeded sample of the batch (32 MiB of coefficients at most) and the sampled row
             indices -- as DIR/{coeffs,status,rows}.npy (float64; a _rank<r> suffix per rank when N > 1).  The
             inputs depend only on the arguments, so two builds can be compared output for output.

--impl reference times that CPU restatement itself (the reference needs Eigen/glog, absent
from this image, so oracle/_ref cannot exist; see DESIGN.md): kind "port".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CONFIGS = {
    # name: (N, r, K, D, total batch)
    "C5": (10, 4, 16, 3, 1048576),
    "C3": (10, 4, 16, 3, 262144),
    "C2": (10, 4, 8, 3, 65536),
    "C4": (8, 3, 4, 3, 1048576),
    # large K (reference timing program sizes): batches of ~3 GB of coefficients, a multiple of the 18 944 trajectories
    # one pass of the persistent grid covers, so that the line shows the kernel and not the wave quantisation of a
    # small batch (65 536 x K=50: 0.393, 32 768 x K=100: 0.340; tools/k_sweep.py)
    "K50": (10, 4, 50, 3, 246272),
    "K100": (10, 4, 100, 3, 113664),
}
METRIC = "min-snap trajectories/sec (N=10, 16-seg, 3D)"
UNIT = "trajectories/s"
NVLINK_PEER_GBS = 770.0  # measured peer copy per direction, /opt/skills/guides/B200_PROFILING.md


def config_dict(cfg, total):
    """Identical in both arms (ours / --impl reference) so that the driver's same_config check holds."""
    N, r, K, D, _ = CONFIGS[cfg]
    return {"workload": f"{cfg}: batch {total} random-waypoint {K}-segment {D}D N={N} derivative_to_optimize={r} fp64, "
                        f"sharded over the job's GPUs (strong scaling; N=1: whole batch on one GPU)",
            "total_trajectories": int(total), "segments": K, "dimensions": D, "N": N, "derivative_to_optimize": r}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(cfg):
    """dram bytes per launch from the committed ncu --set full capture, or None."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(path) as f:
            return json.load(f).get(cfg)
    except Exception:
        return None


class ClockSampler:
    """Samples SM clock and throttle reasons DURING the timed region.  The region is tens of milliseconds,
    far shorter than nvidia-smi's sampling period, so NVML is polled from a thread (nvidia_ml_py); falls
    back to one nvidia-smi query if NVML is unavailable."""

    REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20),
               ("hw_thermal_slowdown", 0x40), ("hw_power_brake", 0x80))

    def __init__(self, index=0):
        self.index = index
        self.samples = []
        self.reason_bits = 0
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self._nvml = None
        self._handle = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._poll, daemon=True)
            self._thread.start()
        except Exception:
            self._nvml = None

    def _poll(self):
        p = self._nvml
        while not self._stop.is_set():
            try:
                self.samples.append(float(p.nvmlDeviceGetClockInfo(self._handle, p.NVML_CLOCK_SM)))
                self.reason_bits |= int(p.nvmlDeviceGetCurrentClocksEventReasons(self._handle))
            except Exception:
                try:
                    self.reason_bits |= int(p.nvmlDeviceGetCurrentClocksThrottleReasons(self._handle))
                except Exception:
                    pass
            time.sleep(0.002)

    def stop(self):
        if self._nvml is not None:
            self._stop.set()
            self._thread.join(timeout=1.0)
            sm = sorted(self.samples)
            reasons = [name for name, bit in self.REASONS if self.reason_bits & bit]
            if sm:
                return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz, "reasons": reasons,
                        "samples": len(sm), "source": "nvml"}
        try:  # fallback: a single nvidia-smi query right after the region
            out = subprocess.run(["nvidia-smi", "-i", str(self.index),
                                  "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.active",
                                  "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
            a, b, c = [x.strip() for x in out.strip().split(",")[:3]]
            return {"sm_mhz": float(a), "sm_max_mhz": float(b), "reasons": [c], "samples": 1, "source": "nvidia-smi"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}


def synth_batch(torch, N, K, D, B, device, seed):
    """Random-waypoint batch with the distribution of createRandomVertices(box +-10) +
    estimateSegmentTimesNfabian(v=3, a=5) (reference vertex.cpp:27-82, :255-272), generated on the
    device with a counter-based generator (the bit-exact mt19937 fixture is what tests/ use)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    pos = torch.rand((B, K + 1, D), generator=g, device=device, dtype=torch.float64) * 20.0 - 10.0
    dist = (pos[:, 1:] - pos[:, :-1]).norm(dim=2).clamp_min(0.2)
    v, a = 3.0, 5.0
    times = dist / v * 2 * (1.0 + 6.5 * v / a * torch.exp(-dist / v * 2))
    h = N // 2
    nf = 2 * h + K - 1
    dfix = torch.zeros((B, D, nf), device=device, dtype=torch.float64)
    dfix[:, :, 0] = pos[:, 0]
    dfix[:, :, h:h + K - 1] = pos[:, 1:K].transpose(1, 2)
    dfix[:, :, h + K - 1] = pos[:, K]
    return pos, times.contiguous(), dfix.contiguous()


DUMP_BYTES = 32 << 20  # coefficient bytes written by --dump-outputs


def dump_outputs(torch, out_dir, coeffs, status, lo, total, world, rank):
    """Writes the sampled rows of this rank's outputs (coeffs [B][K][D][N], status [B] of global rows lo..lo+B)."""
    import numpy as np
    row_bytes = coeffs[0].numel() * coeffs.element_size()
    n = min(total, max(1, DUMP_BYTES // row_bytes))
    rows = np.sort(np.random.default_rng(0).choice(total, size=n, replace=False))
    rows = rows[(rows >= lo) & (rows < lo + coeffs.shape[0])]
    idx = torch.from_numpy(rows - lo).to(coeffs.device)
    suffix = f"_rank{rank}" if world > 1 else ""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"rows{suffix}.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, f"coeffs{suffix}.npy"), coeffs[idx].cpu().numpy())
    np.save(os.path.join(out_dir, f"status{suffix}.npy"), status[idx].cpu().numpy().astype(np.float64))


def _best_threads(O, N, r, K, D):
    """Probe the oracle with all hardware threads and with half of them (SMT siblings often do not help
    this allocation-heavy code); return (threads, trajectories/s) of the faster setting."""
    hw = O.hardware_threads() or os.cpu_count() or 1
    best = (hw, 0.0)
    for threads in sorted({hw, max(1, hw // 2)}, reverse=True):
        probe = max(8192, 256 * threads)
        pos, times = O.make_waypoint_batch(K, D, probe, base_seed=1000)
        O.solve_waypoint_batch(N, r, pos, times, n_threads=threads, mode=0, want_coeffs=False)  # warm
        _, s = O.solve_waypoint_batch(N, r, pos, times, n_threads=threads, mode=0, want_coeffs=False)
        rate = probe / max(s, 1e-9)
        if rate > best[1]:
            best = (threads, rate)
    return best


def cpu_baseline_sample(N, r, K, D, target_seconds=12.0, max_traj=2000000):
    """Times the CPU oracle (kind 'port') on a bounded sample, best of {all, half} host threads."""
    import oracle_lib as O
    O.build()
    threads, rate = _best_threads(O, N, r, K, D)
    # parallel efficiency actually delivered by the host (shared boxes): rate with `threads` vs one thread
    p1, t1_ = O.make_waypoint_batch(K, D, 2048, base_seed=1000)
    O.solve_waypoint_batch(N, r, p1, t1_, n_threads=1, mode=0, want_coeffs=False)
    _, s_one = O.solve_waypoint_batch(N, r, p1, t1_, n_threads=1, mode=0, want_coeffs=False)
    rate_one = 2048 / max(s_one, 1e-9)
    n = int(min(max_traj, max(4096, rate * target_seconds)))
    pos, times = O.make_waypoint_batch(K, D, n, base_seed=1000)
    _, s = O.solve_waypoint_batch(N, r, pos, times, n_threads=threads, mode=0, want_coeffs=False)
    # the nonlinear optimiser's inner step only (updateSegmentTimes + solveLinear on a set-up object,
    # reference polynomial_optimization_nonlinear_impl.h:569-570): max over threads of the clocked time
    n1 = min(n, 200000)
    _, s1 = O.solve_waypoint_batch(N, r, pos[:n1], times[:n1], n_threads=threads, mode=1, want_coeffs=False)
    return {"value": n / s, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{n} trajectories of the workload (mt19937 fixture seeds 1000+b), construct+setupFromVertices+"
                      f"solveLinear per trajectory, {threads} host threads, {s:.2f} s wall",
            "update_times_plus_solve_only": n1 / s1, "per_core": (n / s) / threads, "one_thread_value": rate_one,
            "effective_parallelism": (n / s) / rate_one, "cpu_info": O.cpu_info()}, n, s


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    N, r, K, D, total = CONFIGS[args.config]
    if args.total:
        total = args.total
    import oracle_lib as O
    O.build()
    threads, rate = _best_threads(O, N, r, K, D)
    # bounded sample per step: the whole --steps/--warmup run is sized to ~60 s of CPU work
    per_step_s = max(0.05, 60.0 / max(1, args.steps + args.warmup))
    per_step = int(max(2048, min(400000, rate * per_step_s)))
    pos, times = O.make_waypoint_batch(K, D, per_step, base_seed=1000)
    for _ in range(args.warmup):
        O.solve_waypoint_batch(N, r, pos, times, n_threads=threads, mode=0, want_coeffs=False)
    t = 0.0
    for _ in range(args.steps):
        _, s = O.solve_waypoint_batch(N, r, pos, times, n_threads=threads, mode=0, want_coeffs=False)
        t += s
    value = per_step * args.steps / t
    p1, t1 = pos[:2048], times[:2048]
    _, s_one = O.solve_waypoint_batch(N, r, p1, t1, n_threads=1, mode=0, want_coeffs=False)
    rate_one = 2048 / max(s_one, 1e-9)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(args.config, total),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{per_step} trajectories per step (bounded sample of the workload), CPU restatement "
                                   f"of the reference Eigen path (Eigen/glog absent: reference itself unbuildable), "
                                   f"{threads} host threads",
                         "per_core": value / threads, "one_thread_value": rate_one,
                         "effective_parallelism": value / rate_one, "cpu_info": O.cpu_info()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def _time_launches(torch, fn, steps, warmup=3):
    """Average device time of fn() (one launch per call) with CUDA events on the current stream."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def measure_config(torch, m, solver, name, N, r, K, D, B, dev, peak, steps=20, mask=None):
    """One single-GPU configuration: trajectories/s with resident inputs and its HBM roofline fraction."""
    try:
        prob = m.Problem(N, r, K, D, fixed_mask=mask)
        if mask is None:
            _, times, dfix = synth_batch(torch, N, K, D, B, dev, seed=4321)
        else:
            g = torch.Generator(device=dev)
            g.manual_seed(77)
            times = torch.rand((B, K), generator=g, device=dev, dtype=torch.float64) * 4.0 + 2.0
            dfix = torch.rand((B, D, prob.n_fixed), generator=g, device=dev, dtype=torch.float64) * 4.0 - 2.0
        coeffs = torch.empty((B, K, D, N), dtype=torch.float64, device=dev)
        status = torch.zeros((B,), dtype=torch.int32, device=dev)
        ms = _time_launches(torch, lambda: solver.solve_linear(prob, times, dfix, coeffs=coeffs, status=status), steps)
        ok = bool((status == 0).all().item()) and bool(torch.isfinite(coeffs).all().item())
        nbytes = prob.bytes_per_trajectory * B
        ach = nbytes / (ms * 1e-3) / 1e9
        return {"workload": f"{name}: batch {B} x {K}-segment {D}D N={N} r={r}" + (" generic mask" if mask is not None else ""),
                "value": B / (ms * 1e-3), "unit": UNIT, "kernel_ms": ms, "bytes_per_trajectory": prob.bytes_per_trajectory,
                "achieved_GBps": ach, "frac_of_hbm_peak": ach / peak, "results_ok": ok,
                "kernel": {1: "waypoint", 2: "generic", 3: "nofree"}[prob.kernel],
                "l2": "%.0f MB per step" % (nbytes / 1e6)}
    except Exception as e:  # extras never fail the bench
        return {"workload": name, "failed": str(e)}


def widened_rows(torch, m, solver, dev, peak):
    """SURVEY.md 8f rows built past the hot path, each with its own throughput: batched Mellinger gradient (fused
    cost-only pass vs the round-1 expand + solve + cost kernels) and batched evaluateRange / sampling."""
    out = {}
    try:
        N, r, K, D, B = 10, 4, 16, 3, 32768
        prob = m.Problem(N, r, K, D)
        _, times, dfix = synth_batch(torch, N, K, D, B, dev, seed=11)
        res = {}
        for name, flag in (("fused_cost_only", 0), ("expand_solve_cost_kernels", 1)):
            solver.set_option(m.capi.OPT_MELLINGER_UNFUSED, flag)
            ms = _time_launches(torch, lambda: solver.cost_gradient_mellinger(prob, times, dfix), 5, warmup=2)
            res[name] = {"gradients_per_s": B / (ms * 1e-3), "solves_per_s": B * (K + 1) / (ms * 1e-3), "ms": ms}
        solver.set_option(m.capi.OPT_MELLINGER_UNFUSED, 0)
        res["workload"] = f"getCostAndGradientMellinger for {B} trajectories, C3 shape ({K + 1} re-solves each)"
        out["mellinger_gradient"] = res
    except Exception as e:
        out["mellinger_gradient"] = {"failed": str(e)}
    try:
        N, r, K, D, B, S = 10, 4, 16, 3, 65536, 128
        prob = m.Problem(N, r, K, D)
        _, times, dfix = synth_batch(torch, N, K, D, B, dev, seed=12)
        coeffs = solver.solve_linear(prob, times, dfix)
        t_end = float(times.sum(dim=1).min().item())
        dt = t_end / (S - 2)
        ms = _time_launches(torch, lambda: solver.evaluate_range(times, coeffs, 0.0, t_end, dt, derivs=(0, 1, 2, 3, 4),
                                                                 max_samples=S), 5, warmup=2)
        nbytes = B * (8 * K + 8 * K * D * N + 8 * S * 5 * D + 4)
        out["evaluate_range"] = {"workload": f"sampleTrajectoryInRange sample set (derivatives 0..4) of {B} C3 trajectories, "
                                             f"{S} samples each", "ms": ms, "samples_per_s": B * (S - 1) / (ms * 1e-3),
                                 "achieved_GBps": nbytes / (ms * 1e-3) / 1e9,
                                 "frac_of_hbm_peak": nbytes / (ms * 1e-3) / 1e9 / peak}
    except Exception as e:
        out["evaluate_range"] = {"failed": str(e)}
    try:  # computeCost() of solved trajectories (SURVEY.md 8a-13) and Trajectory::evaluate on a uniform grid
        N, r, K, D, B, S = 10, 4, 16, 3, 262144, 64
        prob = m.Problem(N, r, K, D)
        _, times, dfix = synth_batch(torch, N, K, D, B, dev, seed=13)
        coeffs = solver.solve_linear(prob, times, dfix)
        cost = torch.empty((B,), dtype=torch.float64, device=dev)
        ms = _time_launches(torch, lambda: solver.compute_cost(prob, times, coeffs, cost=cost), 5, warmup=2)
        nbytes = B * (8 * K + 8 * K * D * N + 8)
        out["compute_cost"] = {"workload": f"computeCost() of {B} solved C3 trajectories", "ms": ms,
                               "trajectories_per_s": B / (ms * 1e-3), "achieved_GBps": nbytes / (ms * 1e-3) / 1e9,
                               "frac_of_hbm_peak": nbytes / (ms * 1e-3) / 1e9 / peak}
        t_end = float(times.sum(dim=1).min().item())
        ms = _time_launches(torch, lambda: solver.evaluate(times, coeffs, 1, 0.0, t_end / S, S), 5, warmup=2)
        nbytes = B * (8 * K + 8 * K * D * N + 8 * S * D)
        out["evaluate_uniform_grid"] = {"workload": f"Trajectory::evaluate (velocity) of {B} C3 trajectories on {S} grid points",
                                        "ms": ms, "samples_per_s": B * S / (ms * 1e-3),
                                        "achieved_GBps": nbytes / (ms * 1e-3) / 1e9,
                                        "frac_of_hbm_peak": nbytes / (ms * 1e-3) / 1e9 / peak}
    except Exception as e:
        out["compute_cost"] = {"failed": str(e)}
    return out


def b1_latency(torch, m, solver, dev):
    """PolynomialOptimization<N>::solveLinear() on ONE object = a B=1 call (C1 shape; every nlopt callback,
    reference nonlinear_impl.h:569-570).  Wall-clock per call including the synchronisation the caller needs."""
    try:
        N, r, K, D = 10, 4, 2, 3
        prob = m.Problem(N, r, K, D)
        _, times, dfix = synth_batch(torch, N, K, D, 1, dev, seed=5)
        coeffs = torch.empty((1, K, D, N), dtype=torch.float64, device=dev)
        reps = 300
        for _ in range(20):
            solver.solve_linear(prob, times, dfix, coeffs=coeffs)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            solver.solve_linear(prob, times, dfix, coeffs=coeffs)
            torch.cuda.synchronize()
        dev_us = (time.perf_counter() - t0) / reps * 1e6
        h_t, h_f = times.cpu().pin_memory(), dfix.cpu().pin_memory()
        h_c = torch.empty((1, K, D, N), dtype=torch.float64).pin_memory()
        for _ in range(20):
            solver.solve_linear_host(prob, h_t, h_f, h_c)
        t0 = time.perf_counter()
        for _ in range(reps):
            solver.solve_linear_host(prob, h_t, h_f, h_c)
        host_us = (time.perf_counter() - t0) / reps * 1e6
        return {"workload": "C1 shape (2 segments, 3D, N=10), B=1", "device_pointer_call_plus_sync_us": dev_us,
                "host_pointer_call_us": host_us, "reps": reps}
    except Exception as e:
        return {"failed": str(e)}


def run_ours(args):
    import torch
    import torch.distributed as dist

    import mav_trajectory_generation_b200 as m
    from mav_trajectory_generation_b200 import sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # the scatter/gather path is point-to-point: let NCCL spread every send/recv over many channels
        # (measured at N = 2: 8 channels 203 GB/s, 32 channels 417 GB/s into the root)
        os.environ.setdefault("NCCL_MIN_P2P_NCHANNELS", "32")
        os.environ.setdefault("NCCL_MAX_P2P_NCHANNELS", "32")
        dist.init_process_group("nccl", device_id=dev)

    N, r, K, D, total = CONFIGS[args.config]
    if args.total:
        total = args.total
    bounds = sharding.shard_bounds(total, world)
    B = bounds[rank + 1] - bounds[rank]           # this rank's shard (strong scaling: total is fixed)
    prob = m.Problem(N, r, K, D)
    solver = m.Solver(local)
    _, times, dfix = synth_batch(torch, N, K, D, B, dev, seed=1234 + rank)
    coeffs = torch.empty((B, K, D, N), dtype=torch.float64, device=dev)
    status = torch.zeros((B,), dtype=torch.int32, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- compute phase, shards resident in HBM ("value")
    warm = max(args.warmup, 3)
    for _ in range(warm):
        solver.solve_linear(prob, times, dfix, coeffs=coeffs, status=status)
    barrier()
    # a GPU that has just left idle may still be ramping its clocks after three 1 ms steps: keep warming (untimed) until
    # 0.25 s of work has run; the count is reported as warmup_effective
    t_warm = time.perf_counter()
    while time.perf_counter() - t_warm < 0.25:
        for _ in range(8):
            solver.solve_linear(prob, times, dfix, coeffs=coeffs, status=status)
        torch.cuda.synchronize()
        warm += 8
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = solver.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.perf_counter()
    ev0.record()   # two events around the K launches: nothing but the solver's kernels between them
    for i in range(args.steps):
        solver.solve_linear(prob, times, dfix, coeffs=coeffs, status=status)
    ev1.record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = solver.launch_count - launches0
    local_ms = ev0.elapsed_time(ev1)
    total_ms = allmax(local_ms)
    kern_ms = local_ms / max(1, launches)  # this rank's average launch duration (launch gaps included)
    clocks = sampler.stop() if rank == 0 else None
    ok = bool((status == 0).all().item()) and bool(torch.isfinite(coeffs).all().item())
    value = total * args.steps / (total_ms * 1e-3)
    if args.dump_outputs:  # before the phases below reuse `coeffs`
        dump_outputs(torch, args.dump_outputs, coeffs, status, bounds[rank], total, world, rank)

    # ---------------- BASELINE C5 data path: root holds the batch, NCCL scatter / solve / gather
    sg = None
    if world > 1 and not args.no_scatter_gather:
        if rank == 0:
            _, t_root, f_root = synth_batch(torch, N, K, D, total, dev, seed=99)
            o_root = torch.empty((total, K, D, N), dtype=torch.float64, device=dev)
        else:
            t_root = f_root = o_root = None
        bufs = {}

        def solve_fn(t, f, c):
            solver.solve_linear(prob, t, f, coeffs=c)

        def sg_step():
            sharding.scatter_solve_gather(solve_fn, t_root, f_root, o_root, total, K, D, N, prob.n_fixed, dev,
                                          chunks=args.chunks, local_buffers=bufs)

        for _ in range(3):
            sg_step()
        barrier()
        sg_steps = max(1, min(args.steps, 10))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(sg_steps):
            sg_step()
        e1.record()
        barrier()
        sg_ms = allmax(e0.elapsed_time(e1)) / sg_steps
        if rank == 0:
            # determinism: rows gathered from rank 1 equal a local solve of the same rows (bitwise)
            lo, hi = bounds[1], min(bounds[1] + 4096, bounds[2])
            chk = solver.solve_linear(prob, t_root[lo:hi].contiguous(), f_root[lo:hi].contiguous())
            torch.cuda.synchronize()
            in_bytes = (total - bounds[1]) * 8 * (K + D * prob.n_fixed)
            out_bytes = (total - bounds[1]) * 8 * K * D * N
            sg = {"ms_per_step": sg_ms, "value": total / (sg_ms * 1e-3), "unit": UNIT, "steps": sg_steps,
                  "chunks": args.chunks, "root_egress_bytes": int(in_bytes), "root_ingress_bytes": int(out_bytes),
                  "root_ingress_GBps": out_bytes / (sg_ms * 1e-3) / 1e9,
                  "frac_of_nvlink_peer_peak": out_bytes / (sg_ms * 1e-3) / 1e9 / NVLINK_PEER_GBS,
                  "nvlink_peer_peak_GBps": NVLINK_PEER_GBS,
                  "gathered_rows_bitwise_equal_local_solve": bool(torch.equal(chk, o_root[lo:hi])),
                  "results_finite": bool(torch.isfinite(o_root).all().item())}
        # ---- the same job with the gather FUSED into the solve: every rank's kernel stores its coefficients through
        # NVLink peer memory straight into the root's output (sharding.peer_solve_into_root); no collective
        try:
            if args.no_peer_paths:
                raise RuntimeError("skipped (--no-peer-paths)")
            if rank == 0:
                o_root.zero_()
            t_pb = sharding.PeerBuffer(solver, t_root, 0)
            f_pb = sharding.PeerBuffer(solver, f_root, 0)
            o_pb = sharding.PeerBuffer(solver, o_root, 0)
            pbufs = {}

            def peer_step():
                sharding.peer_solve_into_root(solver, prob, t_pb, f_pb, o_pb, total, dev, local_buffers=pbufs)

            for _ in range(3):
                peer_step()
            barrier()
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t_w0 = time.perf_counter()
            p0.record()
            for _ in range(sg_steps):
                peer_step()
            p1.record()
            barrier()
            peer_wall_ms = allmax((time.perf_counter() - t_w0) * 1e3) / sg_steps
            peer_ms = allmax(p0.elapsed_time(p1)) / sg_steps
            if rank == 0:
                lo, hi = bounds[1], min(bounds[1] + 4096, bounds[2])
                chk = solver.solve_linear(prob, t_root[lo:hi].contiguous(), f_root[lo:hi].contiguous())
                torch.cuda.synchronize()
                sg["fused_peer_store"] = {
                    "what": "no gather step: every rank's solve kernel TMA-stores its coefficients over NVLink peer "
                            "memory (CUDA IPC mapping of the root's output) into their final place; inputs by one peer "
                            "DMA per rank",
                    "ms_per_step": peer_ms, "ms_per_step_wall_incl_barrier": peer_wall_ms,
                    "value": total / (peer_ms * 1e-3), "unit": UNIT,
                    "root_ingress_GBps": out_bytes / (peer_ms * 1e-3) / 1e9,
                    "frac_of_nvlink_peer_peak": out_bytes / (peer_ms * 1e-3) / 1e9 / NVLINK_PEER_GBS,
                    "rows_bitwise_equal_local_solve": bool(torch.equal(chk, o_root[lo:hi])),
                    "results_finite": bool(torch.isfinite(o_root).all().item())}
            # ---- and with the copy engines doing the exchange: chunked pull / solve / push pipeline on three streams
            # (sharding.peer_dma_solve_gather); full-size NVLink write packets, no SM time spent on the transfer
            barrier()
            if rank == 0:
                o_root.zero_()
            dbufs = {}
            by_chunks = {}
            for n_chunks in (args.chunks, 2 * args.chunks, 4 * args.chunks):
                def dma_step():
                    sharding.peer_dma_solve_gather(solver, prob, t_pb, f_pb, o_pb, total, dev, chunks=n_chunks,
                                                   local_buffers=dbufs)

                for _ in range(3):
                    dma_step()
                barrier()
                d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t_w0 = time.perf_counter()
                d0.record()
                for _ in range(sg_steps):
                    dma_step()
                d1.record()
                barrier()
                wall_ms = allmax((time.perf_counter() - t_w0) * 1e3) / sg_steps
                by_chunks[n_chunks] = (allmax(d0.elapsed_time(d1)) / sg_steps, wall_ms)
            best_chunks = min(by_chunks, key=lambda c: by_chunks[c][0])
            dma_ms, dma_wall_ms = by_chunks[best_chunks]
            if rank == 0:
                sg["peer_dma_pipeline"] = {
                    "what": "copy engines do the exchange: per rank a 3-stream pipeline over `chunks` pieces -- peer DMA "
                            "pull of the inputs, local solve, peer DMA push of the coefficients into their final place "
                            "in the root's output; no collective, no SM time on the transfer",
                    "ms_per_step": dma_ms, "ms_per_step_wall_incl_barrier": dma_wall_ms, "chunks": best_chunks,
                    "ms_per_step_by_chunks": {str(c): v[0] for c, v in by_chunks.items()},
                    "value": total / (dma_ms * 1e-3), "unit": UNIT,
                    "root_ingress_GBps": out_bytes / (dma_ms * 1e-3) / 1e9,
                    "frac_of_nvlink_peer_peak": out_bytes / (dma_ms * 1e-3) / 1e9 / NVLINK_PEER_GBS,
                    "rows_bitwise_equal_local_solve": bool(torch.equal(chk, o_root[lo:hi])),
                    "results_finite": bool(torch.isfinite(o_root).all().item())}
            del dbufs
            barrier()
            for pb in (t_pb, f_pb, o_pb):
                pb.close()
            del pbufs
        except Exception as e:  # reported, never fails the bench
            if rank == 0 and sg is not None:
                sg["peer_dma_pipeline" if "fused_peer_store" in sg else "fused_peer_store"] = {"failed": str(e)[:300]}
        if rank == 0 and sg is not None:
            paths = {"nccl_pipeline": sg["ms_per_step"]}
            for key in ("fused_peer_store", "peer_dma_pipeline"):
                if isinstance(sg.get(key), dict) and "ms_per_step" in sg[key]:
                    paths[key] = sg[key]["ms_per_step"]
            best = min(paths, key=paths.get)
            sg["best_path"] = best
            sg["best_ms_per_step"] = paths[best]
            sg["best_frac_of_nvlink_peer_peak"] = out_bytes / (paths[best] * 1e-3) / 1e9 / NVLINK_PEER_GBS
        if world > 1:
            dist.barrier()
        del t_root, f_root, o_root, bufs
        torch.cuda.empty_cache()

    # ---------------- end-to-end through the host-pointer C-ABI ("e2e"), pinned buffers on the GPU's NUMA node
    numa_node, prev_aff = sharding.bind_to_gpu_numa_node(local)
    h_times = torch.empty((B, K), dtype=torch.float64).pin_memory()
    h_dfix = torch.empty((B, D, prob.n_fixed), dtype=torch.float64).pin_memory()
    h_coeffs = torch.empty((B, K, D, N), dtype=torch.float64).pin_memory()
    h_status = torch.empty((B,), dtype=torch.int32).pin_memory()
    h_times.copy_(times)
    h_dfix.copy_(dfix)
    e2e_steps = max(1, min(args.steps, 5))
    solver.solve_linear_host(prob, h_times, h_dfix, h_coeffs, status=h_status)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        solver.solve_linear_host(prob, h_times, h_dfix, h_coeffs, status=h_status)
    torch.cuda.synchronize()
    t_e2e = allmax(time.perf_counter() - t0)
    e2e_value = total * e2e_steps / t_e2e
    # bitwise check on a slice (the full 4 GB comparison would need a second device copy of the output)
    nchk = min(B, 65536)
    e2e_ok = bool((h_status == 0).all().item()) and bool(torch.equal(h_coeffs[:nchk].to(dev), coeffs[:nchk])) and \
        bool(torch.equal(h_coeffs[B - nchk:].to(dev), coeffs[B - nchk:]))
    del h_times, h_dfix, h_coeffs, h_status
    if prev_aff is not None:
        os.sched_setaffinity(0, prev_aff)  # the CPU baseline below must see every usable core again

    # ---------------- "next" row 8f-1: fused Nfabian time allocation + packing (positions in)
    fused_value = None
    try:
        pos_d = synth_batch(torch, N, K, D, B, dev, seed=1234 + rank)[0].contiguous()
        nf_steps = max(1, min(args.steps, 20))
        ms_f = _time_launches(torch, lambda: solver.solve_waypoints_nfabian(N, r, pos_d, 3.0, 5.0, 6.5, coeffs=coeffs),
                              nf_steps)
        fused_value = B / (ms_f * 1e-3)
        del pos_d
    except Exception as e:  # optional extra, never fails the bench
        fused_value = f"failed: {e}"

    if world > 1:
        dist.barrier()
    if rank == 0:
        peak, peak_src = measured_peaks()
        bytes_per_launch = prob.bytes_per_trajectory * B
        achieved = bytes_per_launch / (kern_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(args.config, total),
            "shard": {"trajectories_per_gpu": B, "parallelism": f"shard{world}" if world > 1 else "single",
                      "data_path_collective": "none in the compute phase (value); scatter_gather times the NCCL path",
                      "l2": "inputs+outputs per GPU per step (%.0f MB) exceed the 126 MB L2; no flush needed" %
                            (bytes_per_launch / 1e6),
                      "kernel": {1: "waypoint", 2: "generic", 3: "nofree"}[prob.kernel]},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic(args.config),
                         "traffic_source": "constant from the committed ncu --set full capture (profiles/ncu_traffic.json), "
                                           "not measured by this run",
                         "peak_source": peak_src,
                         "bytes_per_trajectory": prob.bytes_per_trajectory, "kernel_ms": kern_ms,
                         "trajectories_per_launch": B},
            "e2e": {"value": e2e_value, "unit": UNIT,
                    "h2d_bytes_per_step": int(8 * B * (K + D * prob.n_fixed)),
                    "d2h_bytes_per_step": int(8 * B * K * D * N + 4 * B), "steps": e2e_steps,
                    "bitwise_equal_to_device_path": e2e_ok, "bytes_are": "per GPU",
                    "numa_node_of_pinned_buffers": numa_node},
            "gpu_launches": int(launches), "warmup_effective": int(warm), "clocks": clocks, "results_ok": ok,
            "fused_waypoint_entry_traj_per_s_rank0": fused_value,
            "wall_s_timed_region": t_wall,
        }
        if sg is not None:
            line["scatter_gather"] = sg
        if world == 1:
            del times, dfix, coeffs, status
            torch.cuda.empty_cache()
            if not args.no_extras:
                h = N // 2
                gmask = [[1] * h] + [[1, 1] + [0] * (h - 2) for _ in range(15)] + [[1] * h]  # interior velocity fixed too
                import numpy as np
                extras = {}
                for name in ("C3", "C2", "C4", "K50", "K100"):
                    n_, r_, k_, d_, b_ = CONFIGS[name]
                    extras[name] = measure_config(torch, m, solver, name, n_, r_, k_, d_, b_, dev, peak)
                extras["generic_mask"] = measure_config(torch, m, solver, "C3 shape, velocity fixed at every vertex",
                                                        10, 4, 16, 3, 65536, dev, peak,
                                                        mask=np.array(gmask, dtype=np.uint8), steps=5)
                extras["b1_latency"] = b1_latency(torch, m, solver, dev)
                extras.update(widened_rows(torch, m, solver, dev, peak))
                line["configs"] = extras
            if not args.no_cpu_baseline:
                try:
                    cb, _, _ = cpu_baseline_sample(N, r, K, D)
                    line["cpu_baseline"] = cb
                except Exception as e:  # the baseline is reported, never required for the GPU number
                    line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port",
                                            "sample": f"failed: {e}"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C5", choices=sorted(CONFIGS),
                    help="workload whose TOTAL batch is sharded over the GPUs (default C5 = 1 048 576 x 16 segments)")
    ap.add_argument("--total", type=int, default=0, help="override the total number of trajectories")
    ap.add_argument("--chunks", type=int, default=4, help="pipeline pieces per rank in the scatter/gather path")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the per-configuration lines (N=1)")
    ap.add_argument("--no-scatter-gather", action="store_true")
    ap.add_argument("--peer-store", action="store_true", help="(default now; kept for old command lines)")
    ap.add_argument("--no-peer-paths", action="store_true",
                    help="skip the two NVLink peer-memory variants of the C5 data path (fused solve + gather through TMA "
                         "stores into the root's output; copy-engine pull / solve / push pipeline)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed, seeded sample of the last timed step's outputs to DIR/*.npy")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of the CUDA path; the reference arm does not keep its coefficients")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
