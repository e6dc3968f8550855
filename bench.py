#!/usr/bin/env python
"""bench.py -- MCL filter-steps/s on the BASELINE.json configuration.

    python bench.py --gpus N --steps K --warmup W            # this backend (CUDA, sm_100a)
    python bench.py --impl reference --gpus N ...            # the reference algorithm on the host cores

A "step" is one beluga::Amcl::update (amcl_core.hpp:165-201) on one scan of the synthetic
trajectory: diff-drive propagate -> likelihood-field reweight -> normalize -> systematic resample
-> estimate.  Workload (BASELINE.json configs[1]): 1M particles x 1080 beams, 2000x2000 grid.

Reported (one JSON line on stdout, rank 0):
  value      steps/s from the device time of the step's kernels (CUDA events on the launching
             stream; scan points already in HBM when the first event is recorded)
  e2e        steps/s through the C-ABI call bb200_amcl_update with HOST buffers: per step the scan
             (H2D from pinned staging) goes in and the pose estimate comes back, host clock around it
  roofline   the dominant kernel (reweight_lfm) against the measured HBM copy peak
  cpu_baseline  the CPU oracle (a port of the reference pipeline; the reference itself needs
             Eigen/Sophus/range-v3, absent here) on the host cores, bounded sample, same workload

--dump-outputs DIR writes what the last timed step returned (pose estimate, weight sum) and the particle set it left
behind as DIR/<name>.npy (float64), so that two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: nothing is written into it
# The CPU reference runs OpenMP teams on a CPU quota (cgroup): spinning idle threads burn the quota and get the
# whole process throttled (8 threads on 20k particles: 264 ms/step spinning, 33 ms/step sleeping).  Must be set
# before libgomp initialises.
os.environ.setdefault("OMP_WAIT_POLICY", "passive")

METRIC = "MCL filter-steps/sec at 1M particles x 1080 beams (likelihood field, 2000x2000 grid, systematic resample)"
UNIT = "steps/s"
MOTION = (0.1, 0.05, 0.1, 0.05)  # likelihood_params.yaml:6-12
LFM = dict(max_obstacle_distance=2.0, max_laser_distance=100.0, z_hit=0.5, z_random=0.5, sigma_hit=0.2)  # :55-65
PATH_STEPS = 100
# --dump-outputs: at most this many particles (32 B state + 8 B weight each: 40 MB), a seeded sample beyond it
DUMP_MAX_PARTICLES = 1_000_000
DUMP_SAMPLE_SEED = 0
SCALING = "strong"  # the metric is quoted "at 1M particles": N GPUs shard the SAME filter (--weak: --particles per GPU instead)


def reference_particles(args):
    return args.particles * (args.gpus if args.weak else 1)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--particles", type=int, default=1_000_000, help="particles of the filter (with --weak: per GPU)")
    ap.add_argument("--weak", action="store_true", help="weak scaling: --particles per GPU, one filter of N x particles")
    ap.add_argument("--beams", type=int, default=1080)
    ap.add_argument("--grid", type=int, default=2000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-weak-line", action="store_true", help="N > 1: skip the extra weak-scaling measurement (--particles per GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy (native arm; "
                    "with N > 1 the particles are rank 0's shard)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the outputs of the native arm")
    return args


def dump_outputs(out_dir, outputs, states, weights):
    """outputs: name -> float64 array of the last timed step; states/weights: the particle set after it (a fixed, seeded
    sample of DUMP_MAX_PARTICLES particles, in index order, when the set is larger)."""
    if len(weights) > DUMP_MAX_PARTICLES:
        keep = np.sort(np.random.default_rng(DUMP_SAMPLE_SEED).choice(len(weights), DUMP_MAX_PARTICLES, replace=False))
        states, weights = states[keep], weights[keep]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in {**outputs, "particle_states": states, "particle_weights": weights}.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def make_workload(args):
    from beluga_b200 import synthetic

    return synthetic.make_scenario(grid_size=args.grid, n_beams=args.beams, steps=PATH_STEPS)


def workload_name(args, n_total):
    return f"{n_total} particles x {args.beams}-beam LikelihoodFieldModel, {args.grid}x{args.grid} grid @0.05 m, diff-drive + systematic resample"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.samples = []
        self._stop = threading.Event()
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._nvml = self._open_nvml(device)

    @staticmethod
    def _open_nvml(device: int):
        """(module, handle) for in-process NVML sampling, or None -> one nvidia-smi process per sample (slow: a 60 ms timed
        region then sees a single sample)."""
        try:
            import pynvml
            import torch

            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(device).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            try:
                handle = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                handle = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            pynvml.nvmlDeviceGetClockInfo(handle, pynvml.NVML_CLOCK_SM)  # probe
            return pynvml, handle
        except Exception:
            return None

    def _sample_nvml(self):
        nv, h = self._nvml
        sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        try:
            mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        flag = lambda bit: "Active" if mask & bit else "Not Active"  # noqa: E731
        # same column layout as the nvidia-smi query: index, sm, max sm, power, hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
        return [str(self.device), str(sm), str(mx), "", flag(0x8), flag(0x40), flag(0x20), flag(0x4)]

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nvml is not None:
                    self.samples.append(self._sample_nvml())
                    self._stop.wait(0.01)
                    continue
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-i", str(self.device)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([c.strip() for c in out.split(",")])
            except Exception:
                self._nvml = None  # NVML went away: fall back to nvidia-smi
            self._stop.wait(0.05)

    def __enter__(self):
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thread.join(timeout=5)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        mx = [float(s[2]) for s in self.samples if s[2].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(self.samples), "source": "nvml" if self._nvml is not None else "nvidia-smi"}


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic_bytes():
    """dram__bytes_read.sum + dram__bytes_write.sum of one reweight_lfm launch from the committed ncu capture."""
    path = os.path.join(ROOT, "profiles", "lfm_traffic.json")
    try:
        return json.load(open(path))["dram_bytes_per_launch"]
    except Exception:
        return None


def usable_cpus() -> int:
    """CPUs this process can really use: the affinity mask capped by the cgroup CPU quota (the GPU box
    shows 128 logical CPUs but grants 16; 128 OpenMP threads on 16 CPUs run 16x slower than 32)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, -(-int(quota) // int(period))))
    except Exception:
        pass
    return n


def cpu_reference_steps_per_s(args, scenario, n_full, steps, warmup=1, seq_particles=100_000):
    """The reference algorithm (oracle port, counter-RNG mode, propagate/reweight/normalize threaded like
    std::execution::par) on the FULL particle count for `steps` steps -- no extrapolation.  Thread count: the better of
    1x and 2x the usable CPUs, picked on one probe step each; both are reported.  `seq` is the same port on ONE thread
    (std::execution::seq), timed on a bounded particle sample because a full sequential step costs ~5 s per million."""
    from oracle import pyoracle as orc

    native = orc.use_native_build()  # -O3 -march=native on this host (SURVEY 8d); same results as the portable build
    cpus = usable_cpus()
    affinity = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)

    def make(n, threads):
        o = orc.Amcl(orc.AmclParam(min_particles=n, max_particles=n, scheme=orc.SYSTEMATIC, seed=1, rng_mode=1, threads=threads),
                     orc.MotionParam(*MOTION))
        o.set_map(orc.LFM, orc.LfmParam(**LFM), orc.Grid(scenario.cells, scenario.resolution))
        o.initialize_normal(scenario.initial_mean, scenario.initial_cov)
        return o

    def run(o, first, count):
        t0 = time.perf_counter()
        for k in range(first, first + count):
            r = o.update(orc.se2(*scenario.poses[k % PATH_STEPS]), scenario.scans[k % PATH_STEPS])
            assert r.updated == 1
        return (time.perf_counter() - t0) / count

    probes = {}
    for threads in sorted({cpus, 2 * cpus}):
        o = make(n_full, threads)
        run(o, 0, 1)  # first touch of the buffers
        probes[threads] = min(run(o, 1, 1), run(o, 2, 1))
        del o
    threads = min(probes, key=probes.get)
    o = make(n_full, threads)
    run(o, 0, max(1, warmup))
    dt = run(o, max(1, warmup), steps)
    del o
    n_seq = min(seq_particles, n_full)
    o = make(n_seq, 1)
    run(o, 0, 1)
    dt_seq = run(o, 1, 2)
    del o
    return {
        "value": 1.0 / dt, "unit": UNIT, "cores": threads, "kind": "port", "usable_cpus": cpus, "affinity_cpus": affinity,
        "omp_wait_policy": os.environ.get("OMP_WAIT_POLICY"), "build": "-O3 -march=native" if native else "-O3",
        "par": {"steps_per_s": 1.0 / dt, "ms_per_step": dt * 1e3, "threads": threads, "particles": n_full, "steps": steps, "extrapolated": False,
                "probe_ms_per_step": {str(t): v * 1e3 for t, v in probes.items()}},
        "seq": {"steps_per_s": 1.0 / (dt_seq * (n_full / n_seq)), "ms_per_step_sample": dt_seq * 1e3, "threads": 1, "particles": n_seq,
                "extrapolated": n_seq != n_full, "scale": n_full / n_seq},
        "sample": f"{steps} steps of the full {n_full} particles x {args.beams} beams (no extrapolation), {dt * 1e3:.1f} ms/step with {threads} OpenMP "
                  f"threads ({cpus} usable CPUs of {affinity} in the affinity mask); seq: {dt_seq * 1e3:.1f} ms/step for {n_seq} particles on 1 thread",
    }


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    scenario = make_workload(args)
    n_total = reference_particles(args)
    base = cpu_reference_steps_per_s(args, scenario, n_total, steps=args.steps, warmup=max(1, min(args.warmup, 3)))
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 / base["value"], "higher_is_better": True, "scaling": SCALING, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args, n_total), "particles": n_total, "parallelism": f"cpu-omp{base['cores']}"},
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_native(args):
    import torch

    import beluga_b200 as bb
    from beluga_b200 import build as bb_build

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if rank == 0:
        bb_build.build()
    if world > 1:
        dist.barrier()
    if bb.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device (the backend has no CPU fallback)")
    torch.cuda.set_device(local_rank)

    scenario = make_workload(args)
    lfm = bb.LikelihoodFieldModelParam(**LFM)
    grid = bb.OccupancyGrid(scenario.cells, scenario.resolution)
    n_steps = args.warmup + 2 * args.steps  # K device-timed steps, then K end-to-end steps
    poses = [bb.se2(*scenario.poses[k % PATH_STEPS]) for k in range(n_steps + 1)]
    scans = [np.ascontiguousarray(scenario.scans[k % PATH_STEPS]) for k in range(n_steps + 1)]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > L2 (126 MB)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def measure(n_total, with_clocks, keep_outputs=False):
        """K timed steps of ONE filter of n_total particles over `world` GPUs.  Device time: CUDA events on the filter's
        own stream from the first kernel of the step to the read-back (exchanges and the waits inside them included);
        end to end: host clock around the public update call.  Max over ranks.  keep_outputs: also return what the
        last step returned and the particle set it left."""
        shard = n_total // world
        if shard * world != n_total:
            raise SystemExit(f"bench.py: {n_total} particles do not split into {world} equal shards")
        if world == 1:
            params = bb.AmclParams(min_particles=n_total, max_particles=n_total, resample_scheme=bb.RESAMPLE_SYSTEMATIC, seed=1, device=local_rank)
            amcl = bb.Amcl(bb.DifferentialDriveModelParam(*MOTION), params)
            filt = amcl.filter

            def step(k):
                r = amcl.update(poses[k], scans[k])  # bb200_amcl_update: synchronous, the estimate is read back inside
                assert r.updated == 1 and r.resampled == 1
                return {"estimate_mean": np.array(r.estimate.mean), "estimate_cov": np.array(r.estimate.cov).reshape(3, 3),
                        "weight_sum": np.array([r.weight_sum])}
        else:
            # ONE filter sharded over the ranks.  Each rank calls bb200_amcl_update on its shard; the exchanges (largest
            # weight, fixed-point totals, moments) and the redistribution of resampled states run over NVLink peer memory
            # inside the library's kernels -- no NCCL call inside a step (torch.distributed only carried the IPC handles).
            from beluga_b200.distributed import ShardedAmcl

            params = bb.AmclParams(resample_scheme=bb.RESAMPLE_SYSTEMATIC, seed=1, device=local_rank)
            amcl = ShardedAmcl(bb.DifferentialDriveModelParam(*MOTION), params, shard=shard)
            filt = amcl.filter

            def step(k):
                out = amcl.update(poses[k], scans[k])
                assert out is not None and out[2]["resampled"]
                return {"estimate_mean": np.asarray(out[0]), "estimate_cov": np.asarray(out[1]), "weight_sum": np.array([out[2]["weight_sum"]])}

        amcl.update_map(bb.SENSOR_LIKELIHOOD_FIELD, lfm, grid)
        amcl.initialize(scenario.initial_mean, scenario.initial_cov)
        filt.set_timing(True)
        for k in range(args.warmup):
            step(k)
        launches0 = filt.launch_count()
        device_ms, wall_ms, kernel_ms = [], [], {}
        sync_all()

        def timed_loop():
            """Device time per kernel: CUDA events on the filter's stream around every launch of the step."""
            for k in range(args.warmup, args.warmup + args.steps):
                flush.zero_()  # evict L2 between timed steps
                sync_all()
                filt.clear_timings()
                step(k)
                per_step = {}
                for name, ms in filt.last_timings():
                    per_step[name] = per_step.get(name, 0.0) + ms
                device_ms.append(sum(per_step.values()))
                for name, ms in per_step.items():
                    kernel_ms.setdefault(name, []).append(ms)
            sync_all()

        def e2e_loop():
            """End to end: host clock around the public update call (host scan in, estimate out), the next K steps of the
            path, without the per-kernel event marks of the loop above."""
            outputs = None
            filt.set_timing(False)
            for k in range(args.warmup + args.steps, args.warmup + 2 * args.steps):
                flush.zero_()
                sync_all()
                t0 = time.perf_counter()
                outputs = step(k)
                wall_ms.append((time.perf_counter() - t0) * 1e3)
            sync_all()
            return outputs

        if with_clocks:
            with ClockSampler(local_rank) as clocks:
                timed_loop()
                launches = filt.launch_count() - launches0
                outputs = e2e_loop()
            clock_summary = clocks.summary()
        else:
            timed_loop()
            launches = filt.launch_count() - launches0
            outputs = e2e_loop()
            clock_summary = None
        particles = filt.particles() if keep_outputs else None
        totals = torch.tensor([sum(device_ms), sum(wall_ms)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(totals, op=dist.ReduceOp.MAX)
        dev_total_ms, wall_total_ms = totals.tolist()
        last = (args.warmup + 2 * args.steps - 1) % PATH_STEPS
        mean = outputs["estimate_mean"]
        err = float(np.hypot(mean[2] - scenario.poses[last][0], mean[3] - scenario.poses[last][1]))
        if world > 1:
            amcl.close()
        del amcl
        return {"n_total": n_total, "shard": shard, "dev_ms": dev_total_ms / args.steps, "wall_ms": wall_total_ms / args.steps,
                "kernels_ms": {name: float(np.mean(v)) for name, v in kernel_ms.items()}, "launches": int(launches), "clocks": clock_summary,
                "final_position_error_m": err, "outputs": outputs, "particles": particles}

    n_total = reference_particles(args)
    m = measure(n_total, with_clocks=True, keep_outputs=bool(args.dump_outputs))
    weak = None
    if world > 1 and not args.weak and not args.no_weak_line:
        weak = measure(args.particles * world, with_clocks=False)  # the same run at --particles PER GPU

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        g = args.grid * args.grid
        shard = m["shard"]
        k1 = m["kernels_ms"]["reweight_lfm"]
        # SURVEY 8(d) per-unit figures for the reweight launch: 32 B state read + 8 B weight read + 8 B weight write
        # per particle, one 4-byte field value per beam lookup, the field once.
        k1_bytes = shard * (48 + 4 * args.beams) + 4 * g
        step_bytes = n_total * (216 + 4 * args.beams) + 4 * g * world
        achieved = k1_bytes / (k1 * 1e-3) / 1e9
        value = 1e3 / m["dev_ms"]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": m["dev_ms"], "higher_is_better": True, "scaling": "weak" if args.weak else SCALING, "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": workload_name(args, n_total), "particles": n_total, "particles_per_gpu": shard, "parallelism": f"shard{world}",
                       "l2": "256 MiB device write between timed steps (flushes the 126 MB L2)",
                       "timing": "CUDA events on the filter's stream, first kernel of the step to the read-back (shard exchanges and their waits "
                                 "included), per step, max over ranks",
                       "exchange": "none (one GPU)" if world == 1 else "peer-memory mail blocks + peer stores inside the library's kernels (no NCCL in the step)",
                       "final_position_error_m": m["final_position_error_m"]},
            "e2e": {"value": 1e3 / m["wall_ms"], "unit": UNIT, "h2d_bytes_per_step": int(scans[0].nbytes + 32), "d2h_bytes_per_step": int(9 * 8 + 128),
                    "ms_per_step": m["wall_ms"],
                    "protocol": "host clock around Amcl.update (pinned staging of the scan, estimate read back), the K steps after the "
                                "device-timed ones, L2 flushed between steps, no event marks"},
            "gpu_launches": m["launches"],
            "roofline": {"bound": "hbm", "kernel": "reweight_lfm_fixed_param_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic_bytes(), "peak_source": peak_src, "algorithmic_bytes_per_launch": k1_bytes,
                         "kernel_ms": k1, "kernel_share_of_step": k1 / m["dev_ms"],
                         "step_achieved_gbs": step_bytes / (m["dev_ms"] * 1e-3) / 1e9,
                         "note": "the lookups are served by L1/L2 (the field is L2 resident, DRAM traffic = `traffic`); the kernel is bound by "
                                 "instruction issue, the L1 data pipe and the latency of the gather, see profiles/ and DESIGN.md"},
            "kernels_ms": m["kernels_ms"],
            "clocks": m["clocks"],
        }
        if weak is not None:
            wk1 = weak["kernels_ms"]["reweight_lfm"]
            wbytes = weak["shard"] * (48 + 4 * args.beams) + 4 * g
            line["weak"] = {"particles": weak["n_total"], "particles_per_gpu": weak["shard"], "steps_per_s": 1e3 / weak["dev_ms"],
                            "ms_per_step": weak["dev_ms"], "particle_steps_per_s": weak["n_total"] * 1e3 / weak["dev_ms"],
                            "e2e_ms_per_step": weak["wall_ms"], "kernels_ms": weak["kernels_ms"],
                            "roofline_frac": wbytes / (wk1 * 1e-3) / 1e9 / peak, "final_position_error_m": weak["final_position_error_m"]}
        if not args.no_cpu_baseline and world == 1:  # timed beside the GPU arm on rank 0 at N = 1 only
            line["cpu_baseline"] = cpu_reference_steps_per_s(args, scenario, n_total, steps=5)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, m["outputs"], *m["particles"])
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
