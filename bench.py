#!/usr/bin/env python
"""bench.py -- sliding-window solves/sec on synthetic 10-frame x 150-feature windows (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU); the windows are independent, so the batch is split across ranks
with no data-path collective (weak scaling: 1024 windows per GPU) and NCCL is only used for the barrier and the
max-over-ranks timing.  One "step" = one pass of the hot path (Estimator::optimization() solve half: <= 12
dogleg iterations) over one batch of 1024 windows per GPU.

  value : whole-job solves/s with the batch already resident in HBM (CUDA-event time of the launch sequence
          on the library's stream, summed over the K steps, max over ranks)
  e2e   : the same metric through the reference-facing call cerb_solve_batch with HOST buffers (page-locked once with
          cerb_register_host_buffer, like an estimator would do with its long-lived arrays): H2D of the descriptors as they
          are + device pack + solve + D2H inside the timed region
  --impl reference : the CPU path (oracle port of the reference's Ceres solve; the reference itself cannot be
          compiled here) on all host cores over the same 1024-window batch per step.
Inputs per step (about 340 MB per GPU) are larger than the 126 MB L2, so no explicit L2 flush is needed.
  --dump-outputs DIR : after the timed steps, what each timed path returned in its last step (solved states and solve
          reports, float64; every window, or a fixed seeded sample of them past 64 MB) as DIR/{resident,e2e}_<name>.npy, so
          that two builds can be compared output for output on the same seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WINDOWS_PER_GPU = 1024
FEATURES = 150
PRIOR_FEATURES = 24
CPU_SAMPLE = 256
DUMP_LIMIT = 64 << 20          # bytes of --dump-outputs in all; beyond it a fixed seeded sample of windows


def static_config(NW, F, world):
    """The part of `config` that names the workload: identical on the GPU arm and the reference arm."""
    return {"workload": f"{NW} independent synthetic 10-frame x {F}-feature stereo windows per GPU (BASELINE.json configs[1]): {F * 21} visual factors, 10 IMU-leg factors, dense 86-dim marginalization prior, extrinsics free, <= 12 dogleg iterations (all 12 are used)",
            "windows_per_gpu": NW, "features": F,
            "l2": "inputs per step (~300 MB/GPU) exceed the 126 MB L2; no explicit flush",
            "parallelism": f"batch split x{world}, no data-path collective"}


def b_alg(F):
    """Compulsory fp64 HBM bytes per solve (SURVEY.md section 8(d)): inputs read once + outputs written once."""
    return 114160 + 816 * F


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.05)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "", 1).isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "", 1).isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(self.rows)}


def solve_outputs(batch, rep):
    """What a caller of the solve receives for each window: the solved states and the solve report, as float64."""
    st = batch.state_array()
    out = {k: st[k].astype(np.float64) for k in st.dtype.names}
    out["para_Feature"] = batch.para_Feature.copy()
    for k in rep.dtype.names:
        out["report_" + k] = rep[k].astype(np.float64)
    return out


def dump_outputs(directory, prefix, outputs, limit):
    """directory/<prefix><name>.npy for every output, rows = windows; over `limit` bytes, a fixed seeded sample of the windows
    (their indices in <prefix>window_index.npy either way)."""
    os.makedirs(directory, exist_ok=True)
    n = len(next(iter(outputs.values())))
    per_window = 8 + sum(a.nbytes for a in outputs.values()) / n
    keep = min(n, int(limit // per_window))
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    np.save(os.path.join(directory, prefix + "window_index.npy"), idx.astype(np.float64))
    for k, a in outputs.items():
        np.save(os.path.join(directory, prefix + k + ".npy"), a[idx])


def usable_cpus():
    """CPUs this process may actually burn: the affinity mask clipped by the cgroup CPU quota (the GPU boxes expose
    128 hardware threads but cap the container at 16 CPUs; oversubscribing past ~2x the quota only adds throttling)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, 2 * int(-(-int(quota) // int(period)))))
    except (OSError, ValueError):
        pass
    return n


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank's host threads (and so the first-touch placement of its page-locked batch buffers) to the NUMA node its GPU hangs off,
    so that the H2D DMA of the end-to-end path does not cross the socket interconnect.  Best effort: returns a note for `details`."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True, timeout=10).stdout.strip()
        bus = out.lower()
        if bus.startswith("00000000:"): bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return "numa node unknown"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-"); cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if not allowed:
            return f"numa node {node}: none of its cpus in the affinity mask"
        os.sched_setaffinity(0, allowed)
        return f"numa node {node} ({len(allowed)} cpus)"
    except Exception as e:      # no sysfs / no permission: run unpinned
        return f"unpinned ({type(e).__name__})"


def run_reference(args, rank, world):
    """CPU arm: the oracle port of Estimator::optimization() on all host cores, the same 1024-window batch per step as the GPU arm."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from cerberus_b200 import abi, synth
    from oracle_lib import OracleBackend
    NW, F = args.windows, args.features
    cfg = abi.default_config()
    cfg.max_batch, cfg.max_features, cfg.max_obs = NW, ((F + 7) // 8) * 8 + 8, (((F + 7) // 8) * 8 + 8) * abi.NUM_FRAMES
    ob = OracleBackend(cfg)
    cores = usable_cpus()
    base = synth.generate_batch(min(NW, CPU_SAMPLE if F <= 200 else 32), F, ob, cfg=cfg, prior_features=PRIOR_FEATURES)
    batch = synth.tile_batch(base, NW) if NW > base.n else base       # the preintegration set-up of 1024 windows on the CPU would take minutes; the solve does not care
    saved = batch.copy_states()
    nthreads = min(cores, NW)
    times = []
    for it in range(args.warmup + args.steps):
        batch.restore_states(saved)
        t0 = time.perf_counter()
        ob.solve_batch(batch, nthreads=nthreads)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    total = sum(times)
    value = NW * args.steps / total
    line = {
        "impl": "reference", "metric": "sliding-window solves/sec (10-frame x 150-feature windows)", "value": value, "unit": "solves/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": static_config(NW, F, world),
        "cpu_baseline": {"value": value, "unit": "solves/s", "cores": nthreads, "kind": "port",
                         "sample": f"{NW} windows per step ({base.n} distinct windows tiled), one window per thread on {nthreads} threads, each solve single-threaded like the reference (estimator.cpp:1224)"},
        "e2e": {"value": value, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


_REAL_STDOUT = None


def _quiet_stdout():
    """Everything except the ONE JSON line goes to stderr: libraries (NCCL prints its version banner to stdout under torchrun) write
    to file descriptor 1 directly, so fd 1 is pointed at stderr and the JSON line is written to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + "\n").encode())


def main():
    _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--windows", type=int, default=WINDOWS_PER_GPU)
    ap.add_argument("--features", type=int, default=FEATURES)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--distinct", type=int, default=0, help="distinct synthetic windows to generate (tiled up to --windows); 0: all distinct up to 200 features, else 64")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the outputs of the last timed step of each path to DIR/*.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    from cerberus_b200 import abi, synth, lib, parallel
    dist = None
    device = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        torch.cuda.set_device(local_rank)
        device = torch.device("cuda", local_rank)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist_mod.init_process_group("nccl", device_id=device)
        dist = dist_mod
    numa_note = bind_to_gpu_numa_node(local_rank)
    NW, F = args.windows, args.features
    cfg = abi.default_config()
    cfg.device = local_rank
    cfg.max_batch, cfg.max_features, cfg.max_obs = NW, ((F + 7) // 8) * 8 + 8, (((F + 7) // 8) * 8 + 8) * abi.NUM_FRAMES
    gpu = lib.Backend(cfg)                                     # no CPU fallback: raises without CUDA
    t_setup = time.perf_counter()
    distinct = args.distinct or (NW if F <= 200 else min(NW, 64))
    if distinct >= NW:
        batch = synth.generate_batch(NW, F, gpu, cfg=cfg, window0=rank * NW, prior_features=PRIOR_FEATURES)
    else:       # stress sizes: the numpy set-up of thousands of 2000-feature windows would dominate the run; the solver does not care
        batch = synth.tile_batch(synth.generate_batch(distinct, F, gpu, cfg=cfg, window0=rank * NW, prior_features=PRIOR_FEATURES), NW)
    saved = batch.copy_states()
    t_setup = time.perf_counter() - t_setup

    def barrier():
        if dist is not None:
            dist.barrier()
        gpu.sync()

    # ---- device-resident throughput (value) -----------------------------------------------------------------------
    gpu.upload(batch)
    for _ in range(args.warmup):
        gpu.solve_resident(); gpu.sync()
    barrier()
    ev_ms, launches = 0.0, 0
    with ClockSampler(local_rank) as clk:
        t0 = time.perf_counter()
        for _ in range(args.steps):
            gpu.solve_resident(); gpu.sync()
            ms, nl = gpu.last_solve_stats()
            ev_ms += ms; launches += nl
        wall_resident = time.perf_counter() - t0
        barrier()
        if args.dump_outputs:                            # the resident path's last step, fetched outside the timed region
            resident_out = solve_outputs(batch, gpu.download(batch))
        # ---- end to end through the host-buffer call ---------------------------------------------------------------
        e2e_s = 0.0
        regs = gpu.register_batch(batch)                 # page-lock the caller's arrays once (outside the timed region)
        for it in range(args.warmup + args.steps):
            batch.restore_states(saved)
            barrier()
            t0 = time.perf_counter()
            rep = gpu.solve_batch(batch)
            dt = time.perf_counter() - t0
            if it >= args.warmup:
                e2e_s += dt
        dma_ops, staged_bytes = gpu.last_upload_stats()
        e2e_ms, e2e_launches = gpu.last_solve_stats()
        gpu.unregister(regs)
    clocks = clk.summary()
    if args.dump_outputs:
        tag = f"rank{rank}_" if world > 1 else ""
        dump_outputs(args.dump_outputs, tag + "resident_", resident_out, DUMP_LIMIT // (2 * world))
        dump_outputs(args.dump_outputs, tag + "e2e_", solve_outputs(batch, rep), DUMP_LIMIT // (2 * world))
    if dist is not None:
        ev_ms = parallel.max_over_ranks(ev_ms, dist, device)
        e2e_s = parallel.max_over_ranks(e2e_s, dist, device)
        wall_resident = parallel.max_over_ranks(wall_resident, dist, device)
    total_windows = world * NW * args.steps
    value = total_windows / (ev_ms * 1e-3)
    e2e_value = total_windows / e2e_s
    # bytes that cross PCIe per step, counted from the copies the library issues: descriptors + states as they are, tracks, observations
    # (80 B records), inverse depths, per IMU-leg factor the 33 scalar members + jacobian columns 21..30 + covariance, prior matrix + vector
    import ctypes as C
    nF = np.array([batch.descs[w].n_features for w in range(NW)]); nO = np.array([batch.descs[w].n_obs for w in range(NW)])
    npri = np.array([batch.descs[w].prior.n if batch.descs[w].prior.valid else 0 for w in range(NW)])
    h2d = int(NW * (C.sizeof(abi.WindowDesc) + C.sizeof(abi.WindowState) + 10 * (33 + 310 + 961) * 8) + (nF * (16 + 8) + nO * 80 + npri * npri * 8 + npri * 8).sum())
    d2h = int(NW * (240 * 8 + cfg.max_features * 8 + C.sizeof(abi.SolveReport)))

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        traffic = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "solve_kernel_traffic.json")))
            if tj.get("windows") == NW and tj.get("features") == F:       # the ncu capture is of the default workload only
                traffic = tj.get("dram_bytes_per_launch")
        except Exception:
            pass
        kernel_s = ev_ms * 1e-3 / args.steps
        achieved = b_alg(F) * NW / kernel_s / 1e9
        line = {
            "metric": "sliding-window solves/sec (10-frame x 150-feature windows)", "value": value, "unit": "solves/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": static_config(NW, F, world),
            "details": {"wall_ms_per_step_resident": 1e3 * wall_resident / args.steps, "setup_s": t_setup, "mean_iterations": float(np.mean(rep["iterations"])),
                        "e2e_ms_per_step": 1e3 * e2e_s / args.steps, "e2e_dma_ops_per_step": int(dma_ops), "e2e_staged_bytes_per_step": int(staged_bytes),
                        "e2e_device_ms_last_step": e2e_ms, "e2e_kernel_launches_per_step": int(e2e_launches),
                        "host_affinity": numa_note,
                        "e2e_host_buffers": "page-locked once with cerb_register_host_buffer; descriptors DMA'd as they are, AoS -> HBM layout on the device"},
            "e2e": {"value": e2e_value, "unit": "solves/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "note": "vilo_solve_kernel; algorithmic bytes = (114160 + 816 F) per solve x windows per launch; peak = " + peak_src +
                                 "; the kernel is fp64-latency bound, not HBM bound (arithmetic intensity ~420 flop/B, SURVEY.md 8(d))",
                         "fp64_gflops_algorithmic": 0.1 * (F / 150.0) * value},      # ~0.1 Gflop per 150-feature solve, dominated by the visual factors (proportional to F)
        }
        if world == 1 and not args.no_cpu_baseline:
            try:
                sys.path.insert(0, os.path.join(ROOT, "tests"))
                from oracle_lib import OracleBackend
                ob = OracleBackend(cfg)
                cores = usable_cpus()
                ns = min(CPU_SAMPLE, NW)
                batch.restore_states(saved)
                sub = synth.tile_batch(batch, ns) if ns != NW else batch          # the first ns windows at their initial states
                nthreads = min(cores, ns)
                t0 = time.perf_counter()
                ob.solve_batch(sub, nthreads=nthreads)
                dt = time.perf_counter() - t0
                batch.restore_states(saved)
                one = synth.tile_batch(batch, 4)
                t0 = time.perf_counter()
                ob.solve_batch(one, nthreads=1)
                dt1 = time.perf_counter() - t0
                line["cpu_baseline"] = {"value": ns / dt, "unit": "solves/s", "cores": nthreads, "kind": "port", "per_core_value": 4 / dt1,
                                        "sample": f"all-core: the first {ns} windows of the batch, one window per thread on {nthreads} threads, each solve single-threaded like the reference "
                                                  f"(estimator.cpp:1224), {dt:.2f} s wall; per-core: 4 windows on 1 thread, {dt1:.2f} s wall"}
            except Exception as e:  # the oracle is test infrastructure; its absence must not hide the GPU number
                line["cpu_baseline"] = {"value": None, "unit": "solves/s", "cores": 0, "kind": "port", "sample": f"unavailable: {e}"}
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
