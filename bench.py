#!/usr/bin/env python
# SPDX-License-Identifier: Apache-2.0
"""Benchmark of the vectorised Upkie env-step path (see DESIGN.md "Measurement").

    python bench.py --gpus N --steps K --warmup W [--workload servos|pendulum|mpc]
    python bench.py --impl reference ...      # CPU arm (oracle port on host cores)
    python bench.py --gpus 1 ... --dump-outputs DIR

A "step" is one pass of the hot path over one batch: one 5 ms control tick
(5 x 1 ms physics substeps) of every env of the batch = one kernel launch.
Prints ONE JSON line on rank 0. The inputs are seeded: with the same arguments
every run times the same computation, and ``--dump-outputs DIR`` writes the
outputs of the last timed step as ``DIR/<name>.npy`` so that two builds can be
compared output for output.

Workloads (BASELINE.json configs):
  servos   (default) configs[2]/[4]: 65536 UpkieServos envs per GPU, pure torque
           actions ~ U(-tau_max, tau_max), floor friction ~ U(0.5, 1.2), initial
           pitch ~ U(-0.3, 0.3), link inertias x (1 + U(-0.2, 0.2)), fall/height
           termination with fused next-step auto-reset; env-index sharded across
           GPUs (weak scaling), NCCL all-gather of the [T=32] rollout buffer.
  pendulum configs[1]: 4096 ground-velocity envs, actions ~ U(-3, 3) m/s.
  mpc      configs[3]: 4096 robots x horizon-16 box-QP per tick.
"""

import argparse
import json
import os

# One OpenMP / BLAS thread, as torchrun sets for every rank of a multi-GPU run: the stepping thread of the host path
# is latency-critical (copy, launch, synchronise per step) and idle-spinning OpenMP workers on its cores cost the
# single-GPU run up to half of its end-to-end rate in round 1 (per-GPU e2e at N = 1 was half of N >= 2 on the same
# node). Must happen before numpy / torch are imported. The CPU baseline uses its own std::thread pool.
os.environ.setdefault("OMP_NUM_THREADS", "1")
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# algorithmic bytes per env-step (SURVEY.md section 8d; DESIGN.md "Roofline")
# + 24 B: three IMU-acceleration floats kept in the state row; + 32 B: four friction impulses (get_contact_points)
B_ALG = {"servos": 542 + 284 + 3 * 4 * 2 + 4 * 4 * 2, "pendulum": 346 + 3 * 4 * 2 + 16 + 4 * 4 * 2, "mpc": 157}
# compact rollout records: observation rows 72 B instead of 120 B, no reward (4 B) / truncated (1 B) stores
B_ALG_SERVOS_COMPACT = B_ALG["servos"] - 48 - 5
N_ACTION_BUFFERS = 16
ROLLOUT_T = 32  # steps per rollout gather; shortened to K // 4 when the timed region has fewer than 128 steps
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, arrays):
    """Write ``{name: tensor}`` (outputs of the last timed step, first axis = env) as ``directory/<name>.npy``, float64
    kept, everything else as float32. Above DUMP_LIMIT_BYTES in all, every array keeps the same seeded sample of envs,
    whose indices go to ``env_index.npy``."""
    host = {name: t.detach().cpu().numpy() for name, t in arrays.items()}
    host = {name: a.astype(np.float64 if a.dtype == np.float64 else np.float32) for name, a in host.items()}
    n = next(iter(host.values())).shape[0]
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        keep = DUMP_LIMIT_BYTES * n // (total + 8 * n)
        index = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        host = {name: a[index] for name, a in host.items()}
        host["env_index"] = index.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """SM clock / throttle reasons of one GPU around and DURING the timed region.

    Round 1's sampler initialised NVML inside its thread after the timed region had started; the driver's 20-step
    run lasts ~2 ms, so it never produced a sample. Now NVML is initialised up front, the thread samples from
    before the warm-up on, `mark_begin()` / `mark_end()` bracket the timed region, and `sample_now()` takes one
    reading synchronously right after the timed launches were enqueued (the GPU is still executing them)."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index=0):
        self.index = index
        self.samples = []  # (t, sm_mhz, power_w, reason bits, in_region_sync)
        self._stop = threading.Event()
        self._thread = None
        self._t0 = self._t1 = None
        self._nv = None
        self._h = None
        self.max_mhz = None
        self.source = "unavailable"
        try:
            import pynvml as nv

            nv.nvmlInit()
            self._nv = nv
            self._h = nv.nvmlDeviceGetHandleByIndex(self._physical_index(nv, index))
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM))
            self.source = "nvml"
        except Exception as exc:  # no NVML: nvidia-smi polling (slow, ~50 ms per query)
            self._nv = None
            self.source = f"nvidia-smi ({type(exc).__name__})"

    @staticmethod
    def _physical_index(nv, index):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [x for x in vis.split(",") if x.strip() != ""]
            if index < len(ids) and ids[index].strip().isdigit():
                return int(ids[index])
        return index

    def _read(self):
        nv = self._nv
        if nv is not None:
            sm = float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
            try:
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
            except Exception:
                reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
            try:
                power = nv.nvmlDeviceGetPowerUsage(self._h) / 1000.0
            except Exception:
                power = 0.0
            bits = {
                "hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap,
            }
            return sm, power, [k for k in self.NAMES if reasons & bits[k]]
        out = subprocess.run(
            ["nvidia-smi", f"--id={self.index}",
             "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits"],
            capture_output=True, text=True, timeout=5,
        ).stdout.strip()
        f = [x.strip() for x in out.split(",")]
        self.max_mhz = float(f[1])
        return float(f[0]), float(f[2]), [k for i, k in enumerate(self.NAMES) if f[3 + i] == "Active"]

    def sample_now(self, sync=True):
        try:
            sm, power, reasons = self._read()
            self.samples.append((time.perf_counter(), sm, power, reasons, sync))
        except Exception:
            pass

    def _run(self):
        while not self._stop.is_set():
            self.sample_now(sync=False)
            self._stop.wait(0.002 if self._nv is not None else 0.1)

    def mark_begin(self):
        self._t0 = time.perf_counter()

    def mark_end(self):
        self._t1 = time.perf_counter()

    def __enter__(self):
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thread.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [f"no sample ({self.source})"]}
        t0 = self._t0 if self._t0 is not None else -1e30
        t1 = self._t1 if self._t1 is not None else 1e30
        inside = [x for x in self.samples if t0 <= x[0] <= t1]
        used = inside if inside else self.samples[-3:]
        reasons = sorted({r for x in used for r in x[3]})
        return {
            "sm_mhz": float(np.median([x[1] for x in used])),
            "sm_max_mhz": self.max_mhz,
            "reasons": reasons,
            "power_w": float(np.max([x[2] for x in used])),
            "samples_in_timed_region": len(inside),
            "samples_total": len(self.samples),
            "source": self.source,
        }


# ---- CPU arm ---------------------------------------------------------------------------------

def servos_config():
    from upkie_b200 import _abi

    cfg = _abi.default_sim_config()
    cfg.servos_fall_termination = 1
    cfg.min_base_height = 0.15
    cfg.rand_pitch = 0.3
    if os.environ.get("UPKIE_BENCH_JOINT_LIMITS"):  # developer knob: 0 off, 1 scalar slow path, 2 ten-row, 3 hybrid
        cfg.joint_limits = int(os.environ["UPKIE_BENCH_JOINT_LIMITS"])
    # Torso-floor contact rows: OFF for the headline, ON (the library's default) in the secondary line
    # other_workloads.servos_65536_body_contacts. SURVEY 8(d) defines this workload with "reset when |pitch| > 1 or base
    # z < 0.15 m", i.e. it recycles robots by letting their torso sink through the floor. With the rows on, a crouched
    # robot SITS on the torso box (bottom 0.21 m below the base origin of the stand-in model) at z ~ 0.21 > 0.15 and never
    # terminates: a third of the robots ends up resting on the floor for good (tools/r02/body_gate_stats.cpp), every warp
    # takes the general row solver every substep, and the figure measures a different workload. Both are reported.
    cfg.body_contacts = int(os.environ.get("UPKIE_BENCH_BODY_CONTACTS", "0"))
    if os.environ.get("UPKIE_BENCH_MIN_BASE_HEIGHT"):  # developer knob: reset height of the workload (SURVEY 8d: 0.15 m)
        cfg.min_base_height = float(os.environ["UPKIE_BENCH_MIN_BASE_HEIGHT"])
    if os.environ.get("UPKIE_BENCH_RESIDUAL_THRESHOLD"):  # developer knob: 0 = always 50 sweeps (Bullet's own default; PyBullet sets 1e-7)
        cfg.solver_residual_threshold = float(os.environ["UPKIE_BENCH_RESIDUAL_THRESHOLD"])
    return cfg


class CpuServos:
    """The servos workload on the oracle (CPU restatement, fp64): same envs, randomisation, torque actions and
    fall / height termination with reset as the GPU arm. The simulator and its worker pool are created once
    (round 1 re-created both inside every timed call)."""

    def __init__(self, n_envs, threads, seed=2025, n_action_buffers=4):
        from oracle import oracle
        from upkie_b200.model import Model

        oracle.build()
        model = Model.standard_upkie()
        self.n, self.threads = int(n_envs), int(threads)
        rng = np.random.default_rng(seed)
        self.sim = oracle.OracleSim(model, servos_config(), self.n, threads=self.threads)
        self.sim.set_randomization(friction=rng.uniform(0.5, 1.2, self.n), inertia_eps=rng.uniform(-0.2, 0.2, (self.n, 6)))
        self.init = np.zeros((self.n, 25))
        self.init[:, 2] = 0.6
        pitch = rng.uniform(-0.3, 0.3, self.n)
        self.init[:, 3] = np.cos(pitch / 2)
        self.init[:, 5] = np.sin(pitch / 2)
        self.sim.reset(self.init)
        tau = np.asarray(model.tau_max)
        self.acts = []
        for _ in range(n_action_buffers):  # pre-drawn like the GPU arm's rotating action buffers
            act = np.zeros((self.n, 6, 6))
            act[:, :, 0] = np.nan
            act[:, :, 5] = tau
            act[:, :, 2] = rng.uniform(-1, 1, (self.n, 6)) * tau
            self.acts.append(act)
        self.k = 0

    def tick(self):
        """One env tick of every env + the masked reset of the fallen ones (the GPU arm's fused auto-reset)."""
        _, _, term, _ = self.sim.step_servos(self.acts[self.k % len(self.acts)])
        self.k += 1
        if term.any():
            self.sim.reset(self.init, mask=term)

    def rate(self, min_seconds=2.0, max_ticks=10_000):
        """(env-steps/s, seconds, ticks): whole ticks until `min_seconds` of wall time have passed."""
        self.tick()  # warm-up
        t0 = time.perf_counter()
        ticks = 0
        while ticks < max_ticks:
            self.tick()
            ticks += 1
            dt = time.perf_counter() - t0
            if dt >= min_seconds:
                break
        dt = time.perf_counter() - t0
        return self.n * ticks / dt, dt, ticks


def cpu_baseline_servos(n_envs):
    """`cpu_baseline` of the GPU arm's line: the oracle on all host threads on the SAME config (n_envs envs per tick),
    for >= 2 s of wall time, plus a single-thread figure on a 2 048-env sample."""
    cores = os.cpu_count() or 1
    allc = CpuServos(n_envs, cores)
    rate, dt, ticks = allc.rate(2.0)
    one = CpuServos(2048, 1)
    rate1, dt1, ticks1 = one.rate(1.0)
    return {
        "value": rate, "unit": "env-steps/s", "cores": cores, "kind": "port", "same_config": True,
        "sample": f"{n_envs} envs x {ticks} ticks of the same workload (joint_limits={int(servos_config().joint_limits)}), "
                  f"oracle fp64, persistent pool of {cores} threads, {dt:.1f} s wall",
        "single_thread_value": rate1,
        "single_thread_sample": f"2048 envs x {ticks1} ticks, 1 thread, {dt1:.1f} s wall",
    }


def run_reference_arm(args, rank, world):
    """`--impl reference`: the reference's CPU implementation of the path. The reference itself (pybullet +
    gymnasium + upkie_description) cannot be installed here (DESIGN.md "Reference arm"), so this times the oracle
    port with all host threads, on the GPU arm's config: one step = one tick of all 65 536 envs."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n = args.envs_per_gpu or 65536
    w = CpuServos(n, cores)
    # bounded: the whole --steps K --warmup W run must end within a few minutes whatever the host
    probe0 = time.perf_counter()
    w.tick()
    per_tick = time.perf_counter() - probe0
    budget = 150.0
    if per_tick * (args.steps + args.warmup) > budget:
        n = max(2048, int(n * budget / (per_tick * (args.steps + args.warmup))) // 2048 * 2048)
        w = CpuServos(n, cores)
    for _ in range(max(1, args.warmup)):
        w.tick()
    per_step = []
    t_all = time.perf_counter()
    for _ in range(args.steps):
        t0 = time.perf_counter()
        w.tick()
        per_step.append(time.perf_counter() - t0)
    t_total = time.perf_counter() - t_all
    value = n * args.steps / t_total
    one = CpuServos(2048, 1)
    rate1, dt1, ticks1 = one.rate(1.0)
    line = {
        "impl": "reference",
        "metric": "env-steps/sec",
        "value": value,
        "unit": "env-steps/s",
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": 1e3 * t_total / max(1, args.steps),
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f64",
        "data": "synthetic",
        "config": {
            "workload": "UpkieServos 6-DoF torque actions, domain-randomized, fall/height termination + reset "
                        f"(BASELINE configs[2]/[4]); CPU port, each step = one tick of {n} envs",
            "envs_per_step": n,
            "same_config_as_gpu_arm": n == 65536,
            "joint_limit_rows": int(servos_config().joint_limits),
            "solver_residual_threshold": float(servos_config().solver_residual_threshold),
            "body_contact_rows": int(servos_config().body_contacts) != 0,
        },
        "cpu_baseline": {
            "value": value, "unit": "env-steps/s", "cores": cores, "kind": "port",
            "sample": f"{n} envs x 1 tick per step, {args.steps} steps, oracle fp64, persistent pool of {cores} threads; "
                      f"median step {1e3 * float(np.median(per_step)):.1f} ms",
            "single_thread_value": rate1,
            "single_thread_sample": f"2048 envs x {ticks1} ticks, 1 thread, {dt1:.1f} s wall",
        },
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---- GPU arm -------------------------------------------------------------------------------------

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="servos", choices=["servos", "pendulum", "mpc", "plumbing"])
    ap.add_argument("--envs-per-gpu", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-workloads", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (servos, pendulum, mpc; 1 GPU)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload == "plumbing" or world > 1):
        ap.error("--dump-outputs: the servos, pendulum and mpc workloads of the GPU arm on one GPU")

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    from upkie_b200 import _abi
    from upkie_b200.envs import B200VectorEnv
    from upkie_b200.model import Model
    from upkie_b200.robot_state import RobotState, RobotStateRandomization

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # host buffers and the stepping thread on the GPU's NUMA node (the e2e path is PCIe-bound)
    from upkie_b200.numa import bind_to_gpu_node, gpu_numa_node

    previous_affinity = bind_to_gpu_node(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # The rollout all-gather runs on NCCL's own stream while the next rollout simulates. The step kernel
        # occupies every SM (255 registers x 224 threads leave no room for a second block), so the collective's
        # CTAs only get SMs when a simulation block retires. Measured on 2 GPUs (tools/run_2gpu_variants.sh): a
        # high-priority NCCL stream or fewer CTAs (NCCL_MAX_CTAS) make it worse, the default is best.
        pg_options = None
        if os.environ.get("UPKIE_BENCH_NCCL_PRIORITY", "0") == "1":
            pg_options = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        dist.init_process_group("nccl", device_id=dev, pg_options=pg_options)

    model = Model.standard_upkie()
    peaks, peaks_kind = read_peaks()
    W = max(3, args.warmup)
    K = args.steps

    if args.workload == "plumbing":
        print(json.dumps(bench_plumbing(torch, dev, model)), flush=True)
        return
    if args.workload == "mpc":
        result = bench_mpc(args, torch, dev, rank, world, K, W)
    else:
        result = bench_env(args, torch, dist, dev, rank, world, model, K, W)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    units, t_ms, kernel_ms, e2e, launches, clocks, config, n_per_gpu = result
    if previous_affinity is not None:
        os.sched_setaffinity(0, previous_affinity)  # the CPU baseline below uses every host core
    config["host_numa"] = (f"stepping thread and pinned buffers on NUMA node {gpu_numa_node(local_rank)} of the GPU"
                           if previous_affinity is not None else "no NUMA binding (single node or unknown topology)")
    total_units = units * world
    value = total_units / (t_ms * 1e-3)
    b_alg = B_ALG_SERVOS_COMPACT if config.get("rollout_record", "").startswith("compact") else B_ALG[args.workload]
    achieved = b_alg * n_per_gpu / (kernel_ms * 1e-3) / 1e9  # GB/s per GPU, dominant kernel
    side = ncu_sidecar(args.workload, config, n_per_gpu, "early" if W + K <= 64 else "steady")
    line = {
        "metric": "env-steps/sec" if args.workload != "mpc" else "qp-solves/sec",
        "value": value,
        "unit": "env-steps/s" if args.workload != "mpc" else "qp-solves/s",
        "n_gpus": world,
        "steps": K,
        "warmup": W,
        "ms_per_step": t_ms / K,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": config,
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": launches,
        "roofline": {
            "bound": "hbm",
            "achieved": achieved,
            "peak": peaks["hbm_gbs"],
            "unit": "GB/s",
            "frac": achieved / peaks["hbm_gbs"],
            # dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel from the ncu sidecar of THIS
            # build (profiles/ncu_sidecar.json, written by tools/ncu_summary.py, keyed on the hash of the CUDA
            # sources); null when no capture of this build / workload exists
            "traffic": side.get("dram_bytes"),
            "traffic_source": side.get("source"),
            "peak_kind": f"{peaks_kind} (MEASURED_PEAKS.json hbm_gbs)" if peaks_kind == "measured" else "fallback 6650 GB/s",
            "algorithmic_bytes_per_unit": b_alg,
            "kernel_ms": kernel_ms,
            "kernel_ms_statistic": "median over the timed steps of the CUDA-event interval around each launch",
            "note": "fp32 issue-bound path (DESIGN.md): HBM fraction is reported as asked, the binding bound is the "
                    "fp32 pipe; see fp32_issue",
        },
    }
    if args.workload != "mpc":
        # secondary roofline: non-tensor fp32 issue slots (one warp instruction per scheduler and cycle)
        sm_mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz")
        instr = side.get("instr_per_env_step")
        if sm_mhz and instr:
            sched_cycles = 148 * 4 * sm_mhz * 1e6  # issue slots per second
            ipc = instr * (n_per_gpu / 32.0) / (kernel_ms * 1e-3) / sched_cycles
            line["roofline"]["fp32_issue"] = {
                "ipc_per_scheduler": ipc, "peak_ipc": 1.0, "frac": ipc,
                # tools/micro/ffma2_bench.cu on this pool: three-register scalar FFMA saturates at 0.59 inst/cycle/scheduler
                "measured_scalar_ffma_ceiling_ipc": 0.59,
                "instr_per_env_step": instr,
                "fp_instr_share": side.get("fp_instr_share"),
                "sm_mhz_used": sm_mhz,
                "source": side.get("source"),
            }
        else:
            line["roofline"]["fp32_issue"] = {
                "ipc_per_scheduler": None,
                "reason": "no SM clock sample" if not sm_mhz else f"no ncu sidecar for this build ({side.get('source')})",
            }
    if world == 1 and not args.no_cpu_baseline and args.workload != "mpc":
        line["cpu_baseline"] = cpu_baseline_servos(n_per_gpu if args.workload == "servos" else 65536)
    elif world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_mpc_baseline()
    if world == 1 and args.workload == "servos" and not args.no_other_workloads:
        # BASELINE configs[1] and [3] on the record of the same run (device-timed, secondary lines)
        line["other_workloads"] = other_workloads(torch, dev, model)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def ncu_sidecar(workload, config, n_per_gpu, regime):
    """Per-launch DRAM bytes and warp instructions per env-step of the benchmarked kernel, from the sidecar that
    tools/ncu_summary.py writes from an `ncu --set full` capture, valid only for the build it was captured on.
    `regime`: the work per env-step depends on where the episodes are - "early" (the driver's 25 steps after a reset:
    robots still falling from their initial pitch) or "steady" (falling, tumbling, resetting mix after ~100 steps)."""
    from upkie_b200 import build as b

    path = os.path.join(ROOT, "profiles", "ncu_sidecar.json")
    key = f"{workload}:limits{config.get('joint_limit_solver', 0)}:n{n_per_gpu}:{regime}"
    try:
        with open(path) as f:
            data = json.load(f)
    except Exception:
        return {"source": "profiles/ncu_sidecar.json missing"}
    h = b.source_hash()
    ent = data.get(h, {}).get(key)
    if ent is None:
        have = [k for k in data if key in data[k]]
        return {"source": f"no ncu capture of build {h} for {key}" + (f" (captures exist for builds {have})" if have else "")}
    out = dict(ent)
    out["source"] = f"profiles/ncu_sidecar.json[{h}][{key}] <- {ent.get('report', '?')}"
    return out


def other_workloads(torch, dev, model):
    """Short device-timed runs of BASELINE configs[1] (4 096 ground-velocity envs) and configs[3] (MPC 4 096 x
    horizon 16, and the reference's default horizon 50), so that they are on the driver's record too."""
    out = {}
    try:
        from upkie_b200 import _abi
        from upkie_b200.envs import B200VectorEnv
        from upkie_b200.mpc import BatchedMPCBalancer
        from upkie_b200.robot_state import RobotState, RobotStateRandomization

        def timed(fn, k=200, w=20):
            for i in range(w):
                fn(i)
            torch.cuda.synchronize()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(k + 1)]
            ev[0].record()
            for i in range(k):
                fn(i)
                ev[i + 1].record()
            torch.cuda.synchronize()
            return ev[0].elapsed_time(ev[k]) / k, float(np.median([ev[i].elapsed_time(ev[i + 1]) for i in range(k)]))

        def timed_graph(fn, k=48, reps=8):
            """Device time per call with the launches replayed from a CUDA graph: at 4 096 problems a kernel is as
            short as the Python / ctypes launch cadence (~10-20 us), which the event intervals above then measure
            instead of the kernel. Returns None when the capture is not possible."""
            try:
                s = torch.cuda.Stream(device=dev)
                s.wait_stream(torch.cuda.current_stream(dev))
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=s):
                    for i in range(k):
                        fn(i)
                torch.cuda.synchronize()
                g.replay()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    g.replay()
                e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) / (k * reps)
            except Exception:
                return None

        n = 4096
        gen = torch.Generator(device=dev)
        gen.manual_seed(7)
        env = B200VectorEnv(n, "pendulum", device=dev.index, autoreset_mode="next_step", model=model,
                            init_state=RobotState(randomization=RobotStateRandomization(pitch=0.1)))
        env.sim.set_autoreset(1, 2025, 0)
        env.sim.reset(seed=2025)
        acts = [((torch.rand((n, 1), device=dev, generator=gen) * 2 - 1) * 3.0).contiguous() for _ in range(8)]
        ms, med = timed(lambda i: env.sim.step_pendulum(acts[i % 8]))
        out["pendulum_4096"] = {"metric": "env-steps/sec", "value": n / (ms * 1e-3), "ms_per_step": ms,
                                "kernel_ms_median": med, "workload": "BASELINE configs[1]"}
        gms = timed_graph(lambda i: env.sim.step_pendulum(acts[i % 8]))
        if gms:
            out["pendulum_4096"].update({"graph_replay_ms_per_step": gms, "graph_replay_value": n / (gms * 1e-3)})
        env.close()
        for H in (16, 50):
            cfg = _abi.default_mpc_config()
            cfg.nb_timesteps = H
            mpc = BatchedMPCBalancer(n, config=cfg, device=dev.index)
            U = lambda lo, hi: torch.rand(n, device=dev, generator=gen) * (hi - lo) + lo  # noqa: E731
            xs = [torch.stack([U(-0.5, 0.5), U(-0.2, 0.2), U(-0.5, 0.5), U(-1, 1)], dim=1).contiguous() for _ in range(8)]
            vt, contact = U(-1, 1), torch.ones(n, dtype=torch.uint8, device=dev)
            ms, med = timed(lambda i: mpc.step_tensors(xs[i % 8], vt, contact, 0.005))
            out[f"mpc_4096_h{H}"] = {"metric": "qp-solves/sec", "value": n / (ms * 1e-3), "ms_per_step": ms,
                                     "kernel_ms_median": med,
                                     "workload": "BASELINE configs[3]" + (" at the reference's default horizon" if H == 50 else "")}
            gms = timed_graph(lambda i: mpc.step_tensors(xs[i % 8], vt, contact, 0.005))
            if gms:
                out[f"mpc_4096_h{H}"].update({"graph_replay_ms_per_step": gms, "graph_replay_value": n / (gms * 1e-3)})
    except Exception as exc:  # secondary lines must never take the headline down
        out["error"] = repr(exc)
    out["servos_65536_exact_mode"] = exact_mode_line()
    out["servos_65536_body_contacts"] = body_contacts_line()
    return out


def body_contacts_line():
    """The servos workload with the torso-floor contact rows on (the library's default physics): own process, steady
    state (the robots need ~100 ticks to fold onto their torsos), device buffers."""
    try:
        env = dict(os.environ, UPKIE_BENCH_BODY_CONTACTS="1", UPKIE_BENCH_DEVICE_ONLY="1")
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "60", "--warmup", "150",
                            "--no-cpu-baseline", "--no-other-workloads"], env=env, capture_output=True, text=True, timeout=300)
        j = json.loads(r.stdout.strip().splitlines()[-1])
        return {"metric": "env-steps/sec", "value": j["value"], "ms_per_step": j["ms_per_step"],
                "kernel_ms_median": j["roofline"]["kernel_ms"],
                "workload": "headline workload with body_contacts = 1: ~1/3 of the robots sit on their torso box and never "
                            "reach the 0.15 m reset height; every warp solves its rows in general_contact_solve()"}
    except Exception as exc:
        return {"error": repr(exc)}


def exact_mode_line():
    """The servos workload on the exact-arithmetic companion library (no --use_fast_math, upkie_b200/build.py): what
    the one shortcut of the headline kernel buys. Own process (a second copy of the library cannot be the package's
    singleton), device buffers, full records (the exact library has the TILE=0 kernels only)."""
    try:
        from upkie_b200 import build as b

        if not os.path.exists(b.EXACT_LIB_PATH):
            return {"unavailable": "libupkie_b200_exact.so not built"}
        env = dict(os.environ, UPKIE_B200_LIB=b.EXACT_LIB_PATH, UPKIE_BENCH_ROLLOUT="full",
                   UPKIE_BENCH_DEVICE_ONLY="1")
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "100", "--warmup", "10",
                            "--no-cpu-baseline", "--no-other-workloads"], env=env, capture_output=True, text=True, timeout=300)
        j = json.loads(r.stdout.strip().splitlines()[-1])
        return {"metric": "env-steps/sec", "value": j["value"], "ms_per_step": j["ms_per_step"],
                "kernel_ms_median": j["roofline"]["kernel_ms"],
                "workload": "headline workload, exact arithmetic: no fast-math, full 126 B records"}
    except Exception as exc:
        return {"error": repr(exc)}


def bench_env(args, torch, dist, dev, rank, world, model, K, W):
    from upkie_b200 import _abi
    from upkie_b200.envs import B200VectorEnv
    from upkie_b200.robot_state import RobotState, RobotStateRandomization

    servos = args.workload == "servos"
    n = args.envs_per_gpu or (65536 if servos else 4096)
    gen = torch.Generator(device=dev)
    gen.manual_seed(2025 + rank)
    if servos:
        cfg = servos_config()
        env = B200VectorEnv(n, "servos", config=cfg, device=dev.index, autoreset_mode="next_step",
                            env_offset=rank * n, model=model, copy=False)
        mu = torch.empty(n, device=dev).uniform_(0.5, 1.2, generator=gen)
        eps = torch.empty((n, 6), device=dev).uniform_(-0.2, 0.2, generator=gen)
        env.sim.set_randomization(friction=mu, inertia_eps=eps)
        tau = torch.tensor(model.tau_max, dtype=torch.float32, device=dev)
        acts = []
        for _ in range(N_ACTION_BUFFERS):
            a = torch.zeros((n, 6, 6), device=dev)
            a[:, :, 0] = float("nan")
            a[:, :, 5] = tau
            a[:, :, 2] = (torch.rand((n, 6), device=dev, generator=gen) * 2 - 1) * tau
            acts.append(a.contiguous())
        # rollout records: "compact" = position / velocity / torque rows + terminated (73 B/env/step); the constants
        # of the reference (temperature, voltage, reward, truncated) are not written nor gathered. "full" = 126 B.
        compact_rollout = os.environ.get("UPKIE_BENCH_ROLLOUT", "compact") == "compact"
        if compact_rollout:
            def step(a, obs=None, reward=None, terminated=None, truncated=None):
                return env.sim.step_servos_compact(a, obs=obs, terminated=terminated)
        else:
            step = env.sim.step_servos
        obs_bytes = (18 if compact_rollout else 30) * 4
        act_bytes = 36 * 4
    else:
        init = RobotState(randomization=RobotStateRandomization(pitch=0.1))
        env = B200VectorEnv(n, "pendulum", device=dev.index, autoreset_mode="next_step", env_offset=rank * n,
                            model=model, init_state=init, copy=False)
        acts = [((torch.rand((n, 1), device=dev, generator=gen) * 2 - 1) * 3.0).contiguous()
                for _ in range(N_ACTION_BUFFERS)]
        step = env.sim.step_pendulum
        compact_rollout = False
        obs_bytes = 4 * 4
        act_bytes = 4
    env.sim.set_autoreset(1, 2025, rank * n)
    env.sim.reset(seed=2025, env_offset=rank * n)

    # rollout buffer gathered over NVLink once per T steps (SURVEY 8e). At least four gathers - issued AND waited
    # for - fall inside the timed region whatever K is (the driver runs K = 20: T = 5)
    from upkie_b200.sharding import PeerRolloutBuffer, RolloutBuffer

    T_roll = max(1, min(ROLLOUT_T, K // 4))

    # two buffers: the gather of rollout r (NVLink) overlaps the simulation of r + 1. "peer": symmetric-memory
    # buffers, every rank pushes its slot to the peers with the copy engines (no SM); "nccl": all_gather_into_tensor
    # Measured (tools/run_2gpu_variants.sh, tools/run_8gpu.sh): 2 GPUs peer 96 % vs nccl 84 % weak-scaling efficiency;
    # 8 GPUs nccl 64 %, the first (unstaggered, one-stream) peer push collapsed there -> nccl stays the default
    # beyond 2 GPUs until the staggered push is validated at 8.
    # Transport of the rollout records (UPKIE_BENCH_GATHER overrides): "multicast" - the step kernel's row stores go
    # to the NVSwitch multicast address of a symmetric-memory buffer (multimem.st), one store reaches every GPU, the
    # only collective left is a barrier per rollout; "peerstore" - same kernel storing each row into every peer's
    # buffer over NVLink (no multicast object needed); "peer" - copy-engine pushes per rollout; "nccl" -
    # all_gather_into_tensor. Default: multicast where the symmetric memory supports it, else peerstore, else nccl.
    want = os.environ.get("UPKIE_BENCH_GATHER", "auto") if world > 1 else "none"
    gather_mode = want
    gather_note = ""
    if want in ("auto", "multicast", "peerstore", "peer"):
        try:
            if not (servos and compact_rollout) and want != "peer":
                raise RuntimeError("in-kernel transports carry the compact servos records")
            rollouts = [PeerRolloutBuffer(T_roll, n, obs_bytes // 4, dev, compact=compact_rollout) for _ in range(2)]
            if want == "auto":
                gather_mode = "multicast" if rollouts[0].multicast_supported else "peerstore"
            elif want == "multicast" and not rollouts[0].multicast_supported:
                raise RuntimeError("symmetric memory reports no multicast support")
        except Exception as exc:  # symmetric memory unavailable on this box: fall back to NCCL's collective
            gather_note = f"symmetric-memory rollout buffer unavailable ({exc!r}); NCCL all-gather instead"
            print(f"bench.py: {gather_note}", file=sys.stderr)
            gather_mode = "nccl"
    if gather_mode not in ("peer", "multicast", "peerstore"):
        rollouts = [RolloutBuffer(T_roll, n, obs_bytes // 4, dev, compact=compact_rollout) for _ in range(2)]
    works = [None, None]
    # stalls of the simulation stream waiting for the gather of the buffer it is about to overwrite
    stall_events = []
    counters = {"gathers": 0}
    pending = {"push": None}
    # UPKIE_BENCH_PUSH=now: the immediate in-kernel transports (rows leave at the END of the launch that produced them)
    # Default "now" since the second session of round 2: measured best at 2 and at 4 GPUs with the final kernels
    # (profiles/r02_multigpu.md, last section: 20-step run at N = 4: now 2.15e9, deferred 2.05e9, kernel 1.84e9 env-steps/s)
    push_mode = os.environ.get("UPKIE_BENCH_PUSH", "now")  # now | deferred | kernel
    deferred = push_mode == "deferred"

    def wait_for(cur, record):
        """The gather that last read buffer `cur` must be done before its slots are overwritten."""
        if works[cur] is None:
            return
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        if gather_mode in ("multicast", "peerstore"):
            pass  # stream order: publish() already ran on this stream
        elif gather_mode == "peer":
            rollouts[cur].wait()
        else:
            works[cur].wait()
        ev1.record()
        if record:
            stall_events.append((ev0, ev1))
        works[cur] = None

    def do_step(k, timed):
        """Step k (counted from the first warm-up step): the kernel writes its records straight into the rollout
        slot of this step; every T_roll steps the rollout is handed to the transport."""
        cur = (k // T_roll) % 2
        if k % T_roll == 0:
            wait_for(cur, timed)
        a = acts[k % N_ACTION_BUFFERS]
        if gather_mode in ("multicast", "peerstore") and push_mode == "kernel":
            # the fastest step kernel (TILE=1, local stores) writes the local slot; a 2 us kernel of its own sends the
            # rows to every GPU right behind it on the same stream
            so, sr, ste, stru = rollouts[cur].slot(k)
            step(a, obs=so, reward=sr, terminated=ste, truncated=stru)
            env.sim.push_rows(rollouts[cur].push_descriptor(k, multicast=gather_mode == "multicast"))
        elif gather_mode in ("multicast", "peerstore") and deferred:
            # this step's rows go to the local slot; the PROLOGUE of the same launch sends the previous step's rows to
            # every GPU (NVSwitch multicast store, or stores into the peers' buffers), so that their NVLink latency
            # hides under the simulation; a barrier per rollout replaces the gather
            env.sim.step_servos_push(a, *rollouts[cur].local_slot(k), pending["push"])
            pending["push"] = rollouts[cur].push_descriptor(k, multicast=gather_mode == "multicast")
        elif gather_mode == "multicast":
            # immediate form: the kernel's rows go to the multicast address of this rank's slot at the end of the launch
            env.sim.step_servos_multicast(a, *rollouts[cur].multicast_slot(k))
        elif gather_mode == "peerstore":
            # no multicast object: the kernel stores each row into every peer's buffer over NVLink itself
            env.sim.step_servos_peers(a, *rollouts[cur].peer_slots(k))
        else:
            so, sr, ste, stru = rollouts[cur].slot(k)
            step(a, obs=so, reward=sr, terminated=ste, truncated=stru)
        if world > 1 and (k + 1) % T_roll == 0:
            # one gather of the [T, n, record] buffer per rollout, asynchronous
            if timed:
                counters["gathers"] += 1
            if gather_mode in ("multicast", "peerstore"):
                if deferred and pending["push"] is not None:
                    env.sim.push_rows(pending["push"])  # the rollout's last rows have no later launch to ride on
                    pending["push"] = None
                rollouts[cur].publish()
                works[cur] = True
            elif gather_mode == "peer":
                works[cur] = rollouts[cur].push()
            else:
                _, works[cur] = rollouts[cur].gather_raw(async_op=True)

    clk = ClockSampler(dev.index)
    clk.__enter__()
    # Warm-up THROUGH THE TIMED CODE PATH (same kernel instantiation, same transport, at least one rollout hand-over):
    # the first multicast store / barrier kernel / NCCL collective of a process costs ~1.5 ms once (lazy module load,
    # channel set-up), which the driver's 20-step timed region must not carry. W is rounded up to whole rollouts.
    Wa = ((W + T_roll - 1) // T_roll) * T_roll if world > 1 else W
    for k in range(Wa):
        do_step(k, False)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches0 = env.sim.launches
    events = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    end = torch.cuda.Event(enable_timing=True)
    # ncu --profile-from-start off: "1" brackets the timed device loop, "e2e" the host-buffer loop
    profiling = os.environ.get("UPKIE_BENCH_CUDA_PROFILER", "") not in ("", "e2e")
    profiling_e2e = os.environ.get("UPKIE_BENCH_CUDA_PROFILER", "") == "e2e"
    if True:
        torch.cuda.synchronize()
        if profiling:
            torch.cuda.profiler.start()
        clk.mark_begin()
        events[0].record()
        for k in range(K):
            do_step(Wa + k, True)
            events[k + 1].record()
        for i_ in range(2):
            wait_for(i_, True)
        end.record()  # after the last step AND every gather issued inside the timed region
        clk.sample_now()  # the GPU is still working through the queue: one reading inside the timed region for sure
        torch.cuda.synchronize()
        clk.mark_end()
        if profiling:
            torch.cuda.profiler.stop()
        if world > 1:
            dist.barrier()
    gathers = counters["gathers"]
    clk.__exit__()
    total_ms = events[0].elapsed_time(end)
    per_step = np.array([events[k].elapsed_time(events[k + 1]) for k in range(K)])
    # steps that waited for a gather carry that wait in their event interval: the median is the kernel alone
    kernel_ms = float(np.median(per_step))
    gather_stall_ms = float(sum(a.elapsed_time(b) for a, b in stall_events))
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_ms = float(t.item()) / K
    launches = env.sim.launches - launches0
    if args.dump_outputs:
        last = Wa + K - 1  # the rollout slot the last timed step wrote; nothing writes it after the timed region
        outputs = rollouts[(last // T_roll) % 2].slot(last)
        names = ("obs", "reward", "terminated", "truncated")
        dump_outputs(args.dump_outputs, {name: out for name, out in zip(names, outputs) if out is not None})

    if os.environ.get("UPKIE_BENCH_DEVICE_ONLY") == "1":  # exact-mode companion run: no host-buffer kernels in that library
        config = {"workload": "device-only run", "envs_per_gpu": n, "rollout_record": "full",
                  "joint_limit_solver": int(getattr(env.config, "joint_limits", 0))}
        return n * K, t_ms * K, kernel_ms, {"value": None}, launches, clk.summary(), config, n
    # e2e through the public VectorEnv API with HOST buffers (H2D + kernel + D2H per step)
    # this step's inputs live in pinned host memory (4 rotating buffers), outputs land in pinned memory
    host_acts = [a.cpu().pin_memory().numpy() for a in acts[:4]]
    Ke = max(100, min(K, 400))
    for k in range(12):  # warm-up: first-touch of the handle's pinned staging buffers, streams, events
        env.step(host_acts[k % 4])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    if profiling_e2e:
        torch.cuda.profiler.start()
    step_s = np.empty(Ke)
    t0 = time.perf_counter()
    for k in range(Ke):
        ts = time.perf_counter()
        env.step(host_acts[k % 4])  # returns when the step's results are in host memory
        step_s[k] = time.perf_counter() - ts
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if profiling_e2e:
        torch.cuda.profiler.stop()
    te = torch.tensor([e2e_s, float(np.median(step_s))], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e = {
        "value": n * world * Ke / float(te[0].item()),
        "unit": "env-steps/s",
        "h2d_bytes_per_step": n * act_bytes,
        # servos: position/velocity/torque rows (72 B) + terminated; temperature, voltage, reward and truncated
        # are constants of the reference that the env fills once on the host (DESIGN.md, host path)
        "d2h_bytes_per_step": n * ((72 if servos else obs_bytes) + 1),
        "steps": Ke,
        "warmup": 12,
        "median_ms_per_step": 1e3 * float(te[1].item()),
        "value_from_median_step": n * world / float(te[1].item()),
        "api": "B200VectorEnv(copy=False).step(numpy action) -> numpy obs/reward/terminated/truncated (views of the "
               "handle's pinned result buffers, valid until the next step; the default copy=True adds a host memcpy)",
    }
    transport = {
        "none": "",
        "peer": "; rollout buffer pushed to the peers' symmetric-memory buffers by the copy engines over NVLink",
        "multicast": "; the step kernel sends the previous step's rollout rows to the NVSwitch multicast address of the "
                     "symmetric rollout buffer (multimem.st in the launch's prologue): every GPU receives them, one "
                     "barrier per rollout, no collective kernel",
        "peerstore": "; the step kernel stores the previous step's rollout rows into every peer's symmetric rollout "
                     "buffer over NVLink (in the launch's prologue), one barrier per rollout, no collective kernel",
        "nccl": "; NCCL all_gather_into_tensor of the rollout buffer",
    }[gather_mode]
    config = {
        "workload": (
            "UpkieServos 6-DoF torque actions, 65536 envs/GPU, friction~U(0.5,1.2), init pitch~U(+-0.3), inertia "
            "eps~U(+-0.2), fall/height termination + fused next-step autoreset (BASELINE configs[2], per-GPU shard "
            "of configs[4])"
            if servos else "UpkiePendulum (UpkieGroundVelocity) 4096 envs, actions~U(-3,3) m/s (BASELINE configs[1])"
        ),
        "envs_per_gpu": n,
        "global_envs": n * world,
        "rollout_record": ("compact 73 B/env/step (position, velocity, torque rows + terminated; the reference's constants "
                           "temperature, voltage, reward, truncated are not stored)" if compact_rollout
                           else f"{obs_bytes + 6} B/env/step"),
        "substeps_per_step": 5,
        # Bullet's hip / knee joint-limit constraint rows (pybullet_backend.py:121 loadURDF): 0 off, 1 scalar slow
        # path, 2 packed ten-row solver, 3 ten-row solver for the warps that hold a robot on a bound
        "joint_limit_rows": int(getattr(env.config, "joint_limits", 0)) != 0,
        "joint_limit_solver": int(getattr(env.config, "joint_limits", 0)),
        # Bullet's solver exit rule with PyBullet's default threshold (solverResidualThreshold = 1e-7): a robot's PGS
        # sweeps end once no row changed its relative velocity by more than sqrt(threshold) in a sweep; 0 = 50 sweeps
        "solver_residual_threshold": float(getattr(env.config, "solver_residual_threshold", 0.0)),
        # body-ground contact rows of the model's collision points (the torso box; include/upkie_b200.h: body_contacts;
        # library default ON). Off in the headline workload, whose "base below 0.15 m" reset rule presumes that the
        # torso sinks through the floor (servos_config() above); other_workloads.servos_65536_body_contacts has them on
        "body_contact_rows": int(getattr(env.config, "body_contacts", 0)) != 0,
        "parallelism": f"env-index sharded x{world}" + transport,
        "l2": f"{N_ACTION_BUFFERS} rotating action buffers ({N_ACTION_BUFFERS * n * act_bytes / 1e6:.0f} MB"
              " vs 126 MB L2); robot state stays resident by design",
    }
    if world > 1:
        config["gather"] = {
            "transport": gather_mode + ({"kernel": " (push kernel behind every step)", "deferred": " (deferred push)", "now": " (stores at the end of the step kernel)"}[push_mode] if gather_mode in ("multicast", "peerstore") else ""),
            "rollout_steps": T_roll, "gathers_in_timed_region": gathers,
            "bytes_per_rank_and_gather": int(rollouts[0].nbytes),
            # time the simulation stream spent waiting for a gather before re-using its buffer, inside the timed region
            "sim_stream_stall_ms_total": gather_stall_ms,
            "warmup_steps_run": Wa,  # --warmup rounded up to whole rollouts, through the same transport
            "note": gather_note,
        }
    return n * K, t_ms * K, kernel_ms, e2e, launches, clk.summary(), config, n


def bench_plumbing(torch, dev, model, steps=10_000):
    """BASELINE configs[0]: ONE Upkie-PyBullet-Pendulum-equivalent env at 200 Hz under the README PD policy
    (README.md:62-64), 10 k steps, reset on `terminated`, through the public env API with host arrays; the same
    loop on the CPU oracle beside it (single thread)."""
    from oracle import oracle
    from upkie_b200 import _abi
    from upkie_b200.envs import B200VectorEnv

    gains = np.array([10.0, 1.0, 0.0, 0.1], dtype=np.float32)
    env = B200VectorEnv(1, "pendulum", model=model, device=dev.index)
    obs, _ = env.reset(seed=0)
    for _ in range(50):
        obs, _, term, _, _ = env.step((gains @ obs[0]).reshape(1, 1))
    t0 = time.perf_counter()
    resets = 0
    for _ in range(steps):
        obs, _, term, _, _ = env.step((gains @ obs[0]).reshape(1, 1))
        if term[0]:
            obs, _ = env.reset()
            resets += 1
    gpu_rate = steps / (time.perf_counter() - t0)
    pitch_final = float(obs[0, 0])
    cfg = _abi.default_sim_config()
    osim = oracle.OracleSim(model, cfg, 1)
    init = np.zeros((1, 25))
    init[0, 2], init[0, 3] = 0.6, 1.0
    osim.reset(init)
    o = osim.reset_obs(4)
    t0 = time.perf_counter()
    for _ in range(steps):
        o, _, oterm, _ = osim.step_gyropod((gains.astype(np.float64) @ o[0]).reshape(1, 1), 1)
        if oterm[0]:
            osim.reset(init)
            o = osim.reset_obs(4)
    cpu_rate = steps / (time.perf_counter() - t0)
    return {
        "metric": "env-steps/sec", "value": gpu_rate, "unit": "env-steps/s", "n_gpus": 1, "steps": steps, "warmup": 50,
        "ms_per_step": 1e3 / gpu_rate, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "single UpkiePendulum env, 200 Hz, README PD policy, 10k steps (BASELINE configs[0]); "
                               "latency-bound plumbing case, not the throughput configuration",
                   "resets": resets, "final_pitch": pitch_final},
        "e2e": {"value": gpu_rate, "unit": "env-steps/s", "h2d_bytes_per_step": 4, "d2h_bytes_per_step": 22,
                "api": "B200VectorEnv(1, 'pendulum').step(numpy)"},
        "gpu_launches": steps,
        "cpu_baseline": {"value": cpu_rate, "unit": "env-steps/s", "cores": 1, "kind": "port",
                         "sample": f"{steps} steps of the same closed loop on the fp64 oracle, 1 thread"},
    }


def bench_mpc(args, torch, dev, rank, world, K, W):
    from upkie_b200 import _abi
    from upkie_b200.mpc import BatchedMPCBalancer

    n = args.envs_per_gpu or 4096
    cfg = _abi.default_mpc_config()
    cfg.nb_timesteps = 16
    mpc = BatchedMPCBalancer(n, config=cfg, device=dev.index)
    gen = torch.Generator(device=dev)
    gen.manual_seed(4 + rank)

    def U(lo, hi, *shape):
        return torch.rand(shape, device=dev, generator=gen) * (hi - lo) + lo

    xs = [torch.stack([U(-0.5, 0.5, n), U(-0.2, 0.2, n), U(-0.5, 0.5, n), U(-1, 1, n)], dim=1).contiguous()
          for _ in range(N_ACTION_BUFFERS)]
    vt = U(-1, 1, n)
    contact = torch.ones(n, dtype=torch.uint8, device=dev)
    for k in range(W):
        mpc.step_tensors(xs[k % N_ACTION_BUFFERS], vt, contact, 0.005)
    torch.cuda.synchronize()
    events = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    with ClockSampler(dev.index) as clk:
        clk.mark_begin()
        events[0].record()
        for k in range(K):
            mpc.step_tensors(xs[k % N_ACTION_BUFFERS], vt, contact, 0.005)
            events[k + 1].record()
        clk.sample_now()
        torch.cuda.synchronize()
        clk.mark_end()
    total_ms = events[0].elapsed_time(events[K])
    per_step = np.array([events[k].elapsed_time(events[k + 1]) for k in range(K)])
    if args.dump_outputs:  # before the host-array loop below overwrites it
        dump_outputs(args.dump_outputs, {"commanded_velocity": mpc.commanded_velocity})
    xh = [x.cpu().numpy() for x in xs[:4]]
    vth, ch = vt.cpu().numpy(), contact.cpu().numpy()
    Ke = max(10, min(K, 400))
    t0 = time.perf_counter()
    for k in range(Ke):
        mpc.step(xh[k % 4], vth, ch, 0.005)
    e2e_s = time.perf_counter() - t0
    e2e = {"value": n * Ke / e2e_s, "unit": "qp-solves/s", "h2d_bytes_per_step": n * (16 + 4 + 1),
           "d2h_bytes_per_step": n * 4, "steps": Ke, "api": "BatchedMPCBalancer.step(numpy) -> numpy"}
    config = {"workload": "MPC balancer 4096 robots x horizon-16 box-QP per 5 ms tick (BASELINE configs[3])",
              "robots": n, "horizon": 16, "l2": "working set < L2 by nature (4096 x 157 B)"}
    return n * K, total_ms, float(np.median(per_step)), e2e, K, clk.summary(), config, n


def cpu_mpc_baseline():
    from oracle import oracle
    from upkie_b200 import _abi

    cfg = _abi.default_mpc_config()
    cfg.nb_timesteps = 16
    m = oracle.OracleMpc(cfg)
    rng = np.random.default_rng(0)
    n = 4096
    x0 = np.stack([rng.uniform(-0.5, 0.5, n), rng.uniform(-0.2, 0.2, n), rng.uniform(-0.5, 0.5, n), rng.uniform(-1, 1, n)], 1)
    cores = os.cpu_count() or 1
    t0 = time.perf_counter()
    reps = 4
    for _ in range(reps):
        m.step(x0, rng.uniform(-1, 1, n), np.ones(n, np.uint8), 0.005, np.zeros(n), threads=cores)
    dt = time.perf_counter() - t0
    return {"value": n * reps / dt, "unit": "qp-solves/s", "cores": cores, "kind": "port",
            "sample": f"{reps} x 4096 solves, fp64 dense active-set oracle, {cores} threads"}


if __name__ == "__main__":
    main()
