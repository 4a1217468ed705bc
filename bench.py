#!/usr/bin/env python
"""Benchmark of the accelerated path (driver contract: one JSON line on stdout).

    python bench.py --gpus N --steps K --warmup W            # jiminy_b200 on N B200s of one node
    python bench.py --impl reference --steps K --warmup W    # the CPU restatement of the reference path
    python bench.py ... --dump-outputs DIR                   # also save what the last timed step computed

The inputs are seeded: two runs with the same arguments step the same envs with the same actions, so the dumps
of two builds of the project can be compared array for array.

A "step" is one `Engine::step(0.04)` of every env of the batch -- for the default workload 4096
PD-controlled ANYmal envs per GPU with spring-damper ground contact, RK4 at dtMax = 1 ms (160 full
dynamics evaluations + 8 derivative repairs + 41 stepper iterations per env-step), fp64.
`value` is env-steps/s with actions already resident in HBM; `e2e` goes through the public C ABI
with host buffers (pinned host actions -> H2D, step, sensor matrix D2H) every step.
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

METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons / power during the timed region (B200_PROFILING.md's clocks line), polled through
    NVML every 5 ms (nvidia-smi itself needs ~100 ms per sample, longer than a short timed region); falls back to
    `nvidia-smi -lms` when pynvml is unavailable."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self._stop_evt, self.proc = index, [], threading.Event(), None

    def _run_nvml(self) -> bool:
        try:
            import pynvml as nv
            nv.nvmlInit()
            try:   # the CUDA ordinal is not the NVML index when CUDA_VISIBLE_DEVICES reorders / hides devices
                import torch
                h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + str(torch.cuda.get_device_properties(self.index).uuid)).encode())
            except Exception:
                h = nv.nvmlDeviceGetHandleByIndex(self.index)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception:
            return False
        bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while True:
            try:
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append([str(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), str(mx),
                                     str(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)] +
                                    ["Active" if (r & bits[n]) else "Not Active" for n in
                                     ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")])
            except Exception:
                break
            if self._stop_evt.wait(0.005):
                break
        return True

    def run(self):
        if self._run_nvml():
            return
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self._stop_evt.is_set():
                    break
                self.samples.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        self._stop_evt.set()
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=1.0)
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": len(self.samples)}
        try:
            sm = [float(s[0]) for s in self.samples if len(s) >= 7]
            if sm:
                out["sm_mhz"] = float(np.median(sm))
                out["sm_max_mhz"] = float(self.samples[0][1])
                out["power_w_max"] = max(float(s[2]) for s in self.samples if len(s) >= 7)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                out["reasons"] = [n for k, n in enumerate(names)
                                  if any(len(s) >= 7 and s[3 + k].lower().startswith("active") for s in self.samples)]
        except Exception:
            pass
        return out


def cpu_baseline(sc_name, threads_all=True, budget_s=12.0, contact_model=None, solver=None, dt_max=None, **kw):
    """The oracle (a C++ restatement of the reference's CPU path) on this box's host cores: a bounded
    sample of the same workload.  Returns env-steps/s single-thread and with all OpenMP threads."""
    from jiminy_b200 import scenarios
    from oracle.oracle import OracleBatch
    ncores = OracleBatch.use_all_cores()
    out = {"usable": OracleBatch.usable_cores()}
    for label, n_env, par in (("single_thread", 8, False), ("all_threads", 32 * ncores, True)):
        sc = scenarios.make(sc_name, n_env, contact_model=contact_model, solver=solver, dt_max=dt_max, **kw)
        orc = OracleBatch(sc.robot, sc.options, n_env)
        if sc.kp is not None:
            orc.set_pd_controller(sc.kp, sc.kd)
        orc.set_command(sc.target0)
        assert not orc.start(sc.q0, sc.v0).any()
        orc.set_command(sc.sample_targets(0))
        orc.step(sc.step_dt, parallel=par)          # warm-up
        t0, k = time.perf_counter(), 0
        # (the cartpole's random-force policy would walk the cart into its +-10 m position bound after ~200 steps)
        while time.perf_counter() - t0 < budget_s / 2 and k < (80 if sc_name == "cartpole" else 200):
            orc.set_command(sc.sample_targets(k + 1))
            rc = orc.step(sc.step_dt, parallel=par)
            assert kw.get("action", "pd") == "torque" or not rc.any()     # (raw torques: an explicit stepper may diverge, see tools/stability_sweep.py)
            k += 1
        dt = time.perf_counter() - t0
        out[label] = {"value": n_env * k / dt, "n_env": n_env, "steps": k, "seconds": dt}
    return ncores, out


PORT_NOTE = ("kind=port: a scalar C++ restatement of the reference path (oracle/), not jiminy itself (it cannot be built here); on "
             "the one setting the reference publishes (Atlas, Euler 5 ms, constraint contacts: 3.65 k env-steps/s on one thread, "
             "Python pipeline included) the port does 1.3 k single-thread, i.e. it is >= 2.8x slower than real jiminy")


def workload_name(args, sc):
    """The same string in both arms (the driver compares them)."""
    return f"{args.workload}: {args.n_env} envs per GPU, one Engine::step({sc.step_dt}) per step"


def kernel_source_sha():
    """Identity of the device code of the step kernel (the .cuh files) the profile numbers belong to."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "jiminy_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith(".cuh"):
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def step_outputs(eng):
    """What a caller of `step` reads back after it (BatchedEngine or OracleBatch), one row per env, as float64 arrays."""
    t, q, v, a = eng.get_state()
    return {"t": t, "q": q, "v": v, "a": a, "sensors": eng.get_sensors(),
            "status": eng.get_status().astype(np.float64), "env_index": np.arange(len(t), dtype=np.float64)}


def dump_outputs(directory, outputs):
    """Writes `outputs` as `<directory>/<name>.npy`.  Above DUMP_LIMIT_BYTES in all, a fixed seeded sample of envs
    (the same rows in every array, listed in `env_index`) is written instead, so that two builds compare row for row."""
    n_env = len(outputs["env_index"])
    row_bytes = sum(x[:1].nbytes for x in outputs.values())
    if n_env * row_bytes > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n_env, DUMP_LIMIT_BYTES // row_bytes, replace=False))
        outputs = {name: x[rows] for name, x in outputs.items()}
    os.makedirs(directory, exist_ok=True)
    for name, x in outputs.items():
        np.save(os.path.join(directory, f"{name}.npy"), np.ascontiguousarray(x, dtype=np.float64))


def run_reference(args):
    """`--impl reference`: times the reference's CPU implementation of the path.  The reference itself
    cannot be built in this image (Eigen / Boost / Pinocchio / hpp-fcl absent, no network), so this is
    the oracle port (oracle/), with all host threads, on the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from jiminy_b200 import scenarios
    from oracle.oracle import OracleBatch
    ncores = OracleBatch.use_all_cores()
    n_env = min(args.n_env, 64 * ncores)        # bounded sample of the 4096-env batch
    sc = scenarios.make(args.workload, n_env, contact_model=args.contact_model, solver=args.ode_solver, dt_max=args.dt_max,
                        action=args.action, flagged_fraction=args.flagged_fraction)
    orc = OracleBatch(sc.robot, sc.options, n_env)
    if sc.kp is not None:
        orc.set_pd_controller(sc.kp, sc.kd)
    orc.set_command(sc.target0)
    assert not orc.start(sc.q0, sc.v0).any()
    for k in range(args.warmup):
        orc.set_command(sc.sample_targets(k))
        orc.step(sc.step_dt, parallel=True)
    t0 = time.perf_counter()
    for k in range(args.steps):
        orc.set_command(sc.sample_targets(args.warmup + k))
        rc = orc.step(sc.step_dt, parallel=True)
        assert args.action == "torque" or not rc.any()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, step_outputs(orc))
    value = n_env * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args, sc), "scenario": sc.description, "step_dt": sc.step_dt,
                   "sample": f"{n_env}-env sample of the {args.n_env}-env batch, same scenario as the GPU arm"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": ncores, "kind": "port", "usable_cores": OracleBatch.usable_cores(),
                         "sample": f"{n_env} envs x {args.steps} env-steps, OpenMP over envs",
                         "note": PORT_NOTE},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from jiminy_b200 import core, scenarios

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; jiminy_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n_env = args.n_env                                   # per GPU (weak scaling: envs are independent)
    sc = scenarios.make(args.workload, n_env, seed=rank, contact_model=args.contact_model, solver=args.ode_solver, dt_max=args.dt_max,
                        action=args.action, flagged_fraction=args.flagged_fraction)
    eng = core.BatchedEngine(sc.robot, sc.options, n_env, device=local_rank)
    if sc.kp is not None:
        eng.set_pd_controller(sc.kp, sc.kd)
    eng.set_command(sc.target0)
    eng.start(sc.q0, sc.v0)
    nm, width = max(sc.robot.nmotors, 1), eng.width
    stream = torch.cuda.ExternalStream(eng.stream(), device=local_rank)
    total = args.warmup + args.steps
    # actions of every step: on the device (HBM-resident arm) and in pinned host memory (e2e arm)
    acts_host = torch.empty((2 * total, n_env, nm), dtype=torch.float64).pin_memory()
    for k in range(2 * total):
        acts_host[k].copy_(torch.from_numpy(sc.sample_targets(k)))
    acts_dev = acts_host.to(f"cuda:{local_rank}")
    obs_host = torch.empty((n_env, max(width, 1)), dtype=torch.float64).pin_memory()
    obs_np = obs_host.numpy()
    sens_ptr, _ = eng.device_views()
    # multi-GPU: the only exchange of the path is the end-of-step observation concat (SURVEY.md 8e)
    from jiminy_b200.parallel import ObservationExchange
    xch = ObservationExchange(eng, rank, world, local_rank, prefer_peer=not args.nccl_gather)
    use_p2p = xch.mode == "peer"
    obs_gather = xch.note
    flush = torch.empty(160 * 1024 * 1024 // 8, dtype=torch.float64, device=f"cuda:{local_rank}")  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_obs():
        xch.gather()

    # ---------------- HBM-resident arm: `value`
    for k in range(args.warmup):
        eng.set_command_device(acts_dev[k].data_ptr())
        eng.step(sc.step_dt)
        gather_obs()
    barrier()
    eng.synchronize()       # raises PeerTimeout if a rank's completion signal never arrived during the warm-up
    if use_p2p:
        # the peer-memory exchange against the plain NCCL all-gather of the same step: must be identical
        got = xch.view().clone()
        same = torch.tensor([1 if torch.equal(got, xch.reference_gather()) else 0], device=f"cuda:{local_rank}")
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        if int(same.item()) != 1:
            raise RuntimeError("peer-memory observation exchange differs from the NCCL all-gather (rerun with --nccl-gather)")
        obs_gather += "; verified bit-equal to nccl all_gather"
        barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = eng.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    evk = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin.record(stream)
    for k in range(args.steps):
        flush.add_(1.0)   # evict L2 between timed steps (state of 4096 envs fits L2; inputs are re-read cold)
        sev = torch.cuda.Event()
        sev.record(torch.cuda.current_stream())
        stream.wait_event(sev)
        eng.set_command_device(acts_dev[args.warmup + k].data_ptr())
        ev[k][0].record(stream)
        eng.step(sc.step_dt)
        evk[k].record(stream)
        gather_obs()                       # multi-GPU: the step kernel's stream waits for the all-gather
        ev[k][1].record(stream)
    t_end.record(stream)
    barrier()
    eng.synchronize()       # PeerTimeout here = a signal of the timed region never arrived: no number is printed
    launches = eng.launch_count() - launches0
    # read back before the arms below step the batch further: the dump is the state of the last timed step
    outputs = step_outputs(eng) if args.dump_outputs and rank == 0 else None
    clocks = sampler.stop()
    kernel_ms = [a.elapsed_time(b) for (a, _), b in zip(ev, evk)]      # step kernel alone (roofline)
    step_ms = [a.elapsed_time(b) for a, b in ev]                        # step + observation all-gather
    step_ms_dev = float(np.mean(kernel_ms))
    wall_ms = t_begin.elapsed_time(t_end)
    # [t_begin, t_end] also contains the L2 flush kernels; the cost of the path is the sum of the
    # per-step intervals (kernel + gather), max over ranks
    t_path_ms = float(np.sum(step_ms))
    gather_ms = float(np.mean(step_ms) - np.mean(kernel_ms))
    if world > 1:
        tt = torch.tensor([t_path_ms], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_path_ms = float(tt.item())
    status = eng.get_status()
    n_bad = int(((status & ~8) != 0).sum())            # failed envs (8 = JB_ENV_JOINT_LIMIT is informational)
    n_bounds = int(((status & 8) != 0).sum())          # envs whose joint-bound constraints have been active: stepped by the full body

    # ---------------- end-to-end arm: host buffers through the C ABI every step
    barrier()
    e2e_t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in range(args.steps):
        eng.set_command_pinned(acts_host[total + k].numpy())       # H2D of this step's actions
        eng.step(sc.step_dt)
        eng.get_sensors(obs_np)                                     # D2H of the sensor matrix (synchronises)
        gather_obs()
    e1.record(stream)
    barrier()
    e2e_wall = time.perf_counter() - e2e_t0
    e2e_ms = max(e0.elapsed_time(e1), 1e3 * e2e_wall)
    if world > 1:
        tt = torch.tensor([e2e_ms], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_ms = float(tt.item())
        bad = torch.tensor([n_bad, n_bounds], device=f"cuda:{local_rank}")
        dist.all_reduce(bad)
        n_bad, n_bounds = int(bad[0].item()), int(bad[1].item())
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    total_envs = world * n_env
    value = total_envs * args.steps / (t_path_ms * 1e-3)
    e2e_value = total_envs * args.steps / (e2e_ms * 1e-3)
    peaks, peak_kind = read_peaks()
    bytes_per_launch = sc.algorithmic_bytes_per_env_step() * n_env
    # `traffic` and the FP64-pipe figure come from the committed ncu capture of THIS device code (profiles/ncu_traffic.json is
    # written by tools/ncu_traffic.py with the hash of jiminy_b200/csrc): a stale capture reports null, never an old number
    traffic, fp64_pct, prof_src, stale_capture = None, None, None, None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            default = (args.contact_model in (None, "spring_damper") and args.ode_solver is None and args.dt_max is None and
                       args.action == "pd" and args.flagged_fraction == 0.0)
            rec = json.load(fh).get(args.workload) if default else None
        if rec and rec["n_env"] == n_env and rec.get("kernel_source_sha") == kernel_source_sha():
            traffic, fp64_pct, prof_src = rec["traffic_bytes"], rec["fp64_pipe_active_pct"], rec.get("source")
        elif rec and rec["n_env"] == n_env:
            # the device sources changed since the capture: the figures above stay null; what the last capture of this
            # workload measured is reported apart, labelled with the device code it belongs to
            stale_capture = {"traffic": rec["traffic_bytes"], "fp64_pipe_active_pct": rec["fp64_pipe_active_pct"],
                             "ncu_capture": rec.get("source"), "kernel_source_sha": rec.get("kernel_source_sha"),
                             "note": "taken on an earlier version of the device sources (hash above), not on the code timed here"}
    except Exception:
        pass
    achieved_gbs = bytes_per_launch / (step_ms_dev * 1e-3) / 1e9
    # supplementary (never the reported metric): the same steps back to back WITHOUT the L2 flush -- what a rollout loop
    # that does nothing else between two steps sees; for the small configs the cold misses of the flushed timing are most of it
    warm_ms = None
    if world == 1:
        nw = min(args.steps, 20)
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record(stream)
        for k in range(nw):
            eng.set_command_device(acts_dev[args.warmup + k].data_ptr())
            eng.step(sc.step_dt)
        w1.record(stream)
        eng.synchronize()
        warm_ms = w0.elapsed_time(w1) / nw
    ncores, cpu = (None, None)
    if not args.no_cpu_baseline:
        ncores, cpu = cpu_baseline(args.workload, contact_model=args.contact_model, solver=args.ode_solver, dt_max=args.dt_max,
                                   action=args.action, flagged_fraction=args.flagged_fraction)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t_path_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args, sc), "scenario": sc.description, "envs_total": total_envs, "lane_plan": eng.describe(),
                   "l2": "160 MB buffer rewritten between timed steps (flush)", "ms_per_step_warm_l2_back_to_back": warm_ms, "obs_all_gather_ms": gather_ms, "obs_exchange": obs_gather,
                   "envs_failed": n_bad, "envs_flagged": n_bounds, "timed_region_wall_ms": wall_ms},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(n_env * nm * 8 * world),
                "d2h_bytes_per_step": int(n_env * width * 8 * world), "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": achieved_gbs / peaks["hbm_gbs"], "traffic": traffic, "peak_kind": peak_kind,
                     "fp64_pipe_active_pct_ncu": fp64_pct, "ncu_capture": prof_src, "kernel_source_sha": kernel_source_sha(),
                     "last_capture": stale_capture,
                     "kernel": "env_step_kernel", "kernel_ms": step_ms_dev,
                     "algorithmic_bytes_per_launch": bytes_per_launch,
                     "note": "fp64-pipe / latency bound by construction (state stays on chip for the whole "
                             "env-step): see fp64 figures in DESIGN.md and profiles/"},
    }
    if cpu is not None:
        line["cpu_baseline"] = {"value": cpu["all_threads"]["value"], "unit": UNIT, "cores": ncores, "kind": "port",
                                "sample": f"{cpu['all_threads']['n_env']} envs x {cpu['all_threads']['steps']} env-steps, "
                                          f"OpenMP over envs ({cpu['all_threads']['seconds']:.1f} s)",
                                "single_thread_value": cpu["single_thread"]["value"], "usable_cores": cpu["usable"], "note": PORT_NOTE}
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="jiminy_b200", choices=["jiminy_b200", "reference"])
    ap.add_argument("--workload", default="anymal", choices=["anymal", "atlas", "cartpole", "double_pendulum", "anymal_flexible"])
    ap.add_argument("--ode-solver", default=None, choices=["euler_explicit", "runge_kutta_4", "runge_kutta_dopri"],
                    help="override stepper.odeSolver of the scenario")
    ap.add_argument("--dt-max", type=float, default=None, help="override stepper.dtMax of the scenario")
    ap.add_argument("--nccl-gather", action="store_true",
                    help="multi-GPU: exchange observations with an NCCL all-gather after the step instead of the in-kernel "
                         "stores into peer memory")
    ap.add_argument("--contact-model", default=None, choices=["spring_damper", "constraint"],
                    help="override contacts.model of the scenario (the BASELINE metric is quoted on spring_damper)")
    ap.add_argument("--n-env", type=int, default=4096, help="envs per GPU")
    ap.add_argument("--action", default="pd", choices=["pd", "torque"],
                    help="legged robots: PD position targets around the standing posture (default) or raw torque actions U(-20, 20) Nm")
    ap.add_argument("--flagged-fraction", type=float, default=0.0,
                    help="PD mode: share of the envs driven through their hip joint bounds (stepped by the full body with joint-bound constraints)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the time, state, sensors and status of every env after the last timed step as "
                         "DIR/<name>.npy (float64; a seeded sample of envs above 64 MB in all); multi-GPU: rank 0's envs")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
