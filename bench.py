#!/usr/bin/env python
"""bench.py -- agent-steps/s of the batched swarm step (+obs+reward+done+global_state).

Contract (driver):  python bench.py --gpus N --steps K --warmup W   (torchrun for N > 1)
prints ONE JSON line on rank 0.

Workload = BASELINE.json configs[3] ("C4", the config the metric is quoted on): 32-drone swarm,
8 obstacles, reference-default DroneEnvConfig (world 20, K=3, S=4, max_steps 400), per-env domain
randomisation with the ranges of the reference's configs/domain_randomization_v1.yaml (mass / accel /
speed / dt / obstacle-radius / world scales, thrust and sensor noise; its control_delay_steps block
is off by default because it routes the step to the slower general kernel: --dr-delay),
65536 env instances PER GPU (weak scaling; the whole of C4 fits one GPU), i.i.d. U(-1,1) float32
actions read from device memory, auto-reset on, global_state emitted.  A "step" advances every env
instance once (step launch + the small auto-reset launch enqueued behind it).  The per-step working
set (~0.5 GB) exceeds the 126 MB L2.  The same run also times the path with randomisation off -- the
one that is bit-identical to the reference -- and reports it under "dr_off".

  value     device-resident throughput: actions applied (device counter) / CUDA-event time, max over ranks
  e2e       same metric through the host-buffer C-ABI call (pinned H2D actions + D2H of every output)
  roofline  algorithmic bytes (SURVEY 8d: B = 244 + (34 + 12 M)/N per slot-step) / kernel time vs measured HBM peak
  cpu_baseline  the C oracle (a port of the reference's algorithm) on all host cores, bounded sample

`--impl reference` times the UNMODIFIED Python reference env (staged under oracle/_ref/ by oracle/make_ref.py, one
worker process per host thread, >= 2 s) and reports the C port beside it; where the staged copy is missing it
falls back to the port alone and says so (`reference_kind`).

  --scaling strong   BASELINE config 4 as written: 65536 env instances IN TOTAL, sharded over the N GPUs
  --graph T          time CUDA-graph replays of T captured steps (SwarmEngine.capture_steps) instead of a Python
                     loop over step(): what the launch-bound batch sizes BASELINE names (4096 x 8 drones) need
  named_sizes        the default run also reports C2 / C3 / C4-shard / C5 at BASELINE's own env counts
  --dump-outputs DIR after the timed steps, write what their last step handed its caller (every output field of
                     the step: obs, reward, dist, the flag arrays, __all__ flags, global_state) as DIR/<name>.npy
                     (float32; float64 stays float64) for a seeded sample of env instances (DIR/env_index.npy) that
                     keeps the dump under 64 MB.  Inputs are fixed by the arguments, so two builds run with the
                     same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (kind, config, default envs per GPU)
    "c4": ("swarm", {"num_drones": 32, "num_obstacles": 8}, 65536),
    "c4_w44": ("swarm", {"num_drones": 32, "num_obstacles": 8, "world_size": 44.0}, 65536),
    "c2": ("swarm", {"num_drones": 8, "num_obstacles": 4}, 262144),
    "c3": ("swarm", {"num_drones": 16, "num_obstacles": 8}, 131072),
    "c5": ("swarm", {"num_drones": 128, "num_obstacles": 8}, 8192),
    "c5_w70": ("swarm", {"num_drones": 128, "num_obstacles": 8, "world_size": 70.0}, 8192),
    "c1": ("single", {"num_obstacles": 8}, 1048576),
    # DronePhysicsEnv as a point mass (DESIGN.md 9): 24 sub-steps of 1/240 s per step, reference default 3 drones
    "phys": ("physics", {"num_drones": 3, "num_obstacles": 8}, 524288),
    "phys8": ("physics", {"num_drones": 8, "num_obstacles": 8}, 262144),
}


# configs/domain_randomization_v1.yaml:9-60 of the reference (control_delay_steps: see --dr-delay)
DR_V1 = {"mass_scale": (0.85, 1.15), "max_accel_scale": (0.90, 1.10), "max_speed_scale": (0.90, 1.10),
         "dt_scale": (0.95, 1.05), "obstacle_radius_scale": (0.9, 1.1), "world_size_scale": (0.95, 1.05),
         "thrust_noise_std": 0.03, "position_noise_std": 0.02, "velocity_noise_std": 0.02,
         "obstacle_distance_noise_std": 0.03}


def dr_enabled(args):
    return args.dr == "on" or (args.dr == "auto" and args.workload == "c4")


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.01)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def cpu_port_rate(kind, cfg, n_envs, budget_s, threads, dr=False):
    """Times the C oracle (port of the reference algorithm) on the host cores: bounded sample."""
    import swarm_oracle as so

    o = so.OracleSwarm(n_envs, cfg, kind=kind, dr=DR_V1 if dr else None, dr_seed=2026)
    o.seed(np.arange(n_envs, dtype=np.uint64))
    o.reset()
    rng = np.random.default_rng(1000)
    acts = [rng.uniform(-1, 1, size=(n_envs, o.N, 3)).astype(np.float32) for _ in range(4)]
    o.step(acts[0], auto_reset=True, num_threads=threads)  # warm
    steps, agent_steps = 0, 0
    t0 = time.perf_counter()
    while True:
        agent_steps += int(o.active.sum()) if kind == "swarm" else n_envs * o.N
        o.step(acts[steps % 4], auto_reset=True, num_threads=threads)
        steps += 1
        if time.perf_counter() - t0 >= budget_s:
            break
    dt = time.perf_counter() - t0
    return agent_steps / dt, steps, dt


def python_reference_rate(kind, cfg, min_seconds, min_steps=1):
    """The unmodified reference env on every host thread (oracle/ref_runner.py); None where it is not staged."""
    try:
        import ref_runner
        if ref_runner.reference_src() is None:
            return None
        return ref_runner.time_reference(kind, cfg, min_seconds=min_seconds, min_steps=min_steps)
    except Exception as exc:  # noqa: BLE001  (a baseline leg must never take the bench line down)
        sys.stderr.write(f"python reference leg failed: {exc!r}\n")
        return None


def run_reference_arm(args, kind, cfg, wl_name, default_envs):
    """--impl reference: the reference's own CPU implementation on all host threads, same config / metric / unit.
    Each "step" advances every worker's env instance once; the timed region is at least 2 s long (a 0.1 s region
    measured the thread ramp-up, not the env)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = len(os.sched_getaffinity(0))
    dr = dr_enabled(args)
    port_rate, port_steps, port_dt = cpu_port_rate(kind, cfg, args.cpu_envs, max(2.0, args.cpu_seconds / 4), threads, dr)
    port = {"value": port_rate, "unit": "agent-steps/s", "cores": threads, "kind": "port",
            "sample": f"{args.cpu_envs} env instances x {port_steps} steps in {port_dt:.1f} s (oracle/swarm_oracle.c, "
                      f"scalar C port of the reference algorithm, {threads} threads" + (", randomisation on)" if dr else ")")}
    ref = python_reference_rate(kind, cfg, min_seconds=max(2.0, args.cpu_seconds / 2), min_steps=args.steps)
    if ref is not None:
        val, ref_kind, steps_done, dt = ref["rate"], "python_reference", ref["steps_per_proc"], ref["seconds"]
        base = {"value": val, "unit": "agent-steps/s", "cores": ref["procs"], "kind": "reference",
                "sample": f"the unmodified reference env (oracle/_ref, pure Python + numpy), {ref['procs']} worker processes x "
                          f"{ref['envs_per_proc']} env instance(s) of the {wl_name} config x {steps_done} steps in {dt:.1f} s, "
                          f"randomisation off (no reference code implements it)"}
        note = ("the reference's own env code, unmodified, one process per host thread (it has no vectorisation: "
                "config_builders.py:19-23); `port` = oracle/swarm_oracle.c, a scalar C port of the same algorithm, "
                "multi-threaded -- the stronger CPU baseline")
    else:
        val, ref_kind, steps_done, dt = port_rate, "c_port", port_steps, port_dt
        base = port
        note = ("oracle/_ref is not staged here (the reference is pure Python: oracle/make_ref.py copies it where "
                "/root/reference exists): this is oracle/swarm_oracle.c, a scalar C port of its algorithm pinned "
                "bit-exact to fixtures recorded from it")
    line = {
        "impl": "reference", "reference_kind": ref_kind, "metric": "agent_steps_per_sec", "value": val,
        "unit": "agent-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / max(steps_done, 1) * 1e3,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(wl_name, kind, cfg, default_envs, args.gpus, dr),
        "cpu_baseline": base, "port": port,
        "e2e": {"value": val, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "note": note,
    }
    print(json.dumps(line), flush=True)


DUMP_BYTES = 48 << 20   # --dump-outputs budget (files + headers stay under 64 MB)


def dump_outputs(eng, out_dir):
    """The step's output fields (_abi.HOST_OUT_FIELDS present on this engine) of a fixed sample of env instances,
    as out_dir/<name>.npy; the sampled env indices as out_dir/env_index.npy."""
    import torch
    from swarm_b200 import _abi

    fields = {n: getattr(eng, n) for n in _abi.HOST_OUT_FIELDS if getattr(eng, n, None) is not None}
    per_env = 8 + sum(t[0].numel() * (8 if t.dtype == torch.float64 else 4) for t in fields.values())
    n = min(eng.E, DUMP_BYTES // per_env)
    idx = np.arange(eng.E) if n == eng.E else np.sort(np.random.default_rng(0).choice(eng.E, n, replace=False))
    sel = torch.from_numpy(idx).to(eng.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_index.npy"), idx.astype(np.float64))
    for name, t in fields.items():
        t = t.index_select(0, sel)
        t = t if t.dtype == torch.float64 else t.to(torch.float32)
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def kernel_name(kind, n, envs):
    """The kernel `swarm_step` selects for this shape (swarm_abi.cu: rot_eligible / rotx_eligible / launch)."""
    if kind == "swarm" and n in (8, 16, 32):
        return "swarm_step_rot_kernel"
    if kind == "swarm" and n in (64, 128) and envs >= 4096:
        return "swarm_step_rotx_kernel"
    return "swarm_env_kernel_small" if n <= 32 else "swarm_env_kernel"


def workload_config(name, kind, cfg, envs_per_gpu, n_gpus, dr=False):
    full = {"world_size": 20.0, "max_steps": 400, "neighbor_k": 3, "sensed_obstacles": 4}
    full.update(cfg)
    return {"workload": f"{name}: {kind} env, N={full.get('num_drones', 1)} drones, M={full['num_obstacles']} "
                        f"obstacles, K={full['neighbor_k']}, S={full['sensed_obstacles']}, world {full['world_size']}, "
                        f"{envs_per_gpu} env instances per GPU x {n_gpus} GPU(s), U(-1,1) actions, auto-reset, "
                        f"global_state on, domain randomisation {'on (domain_randomization_v1 ranges, no control delay)' if dr else 'off'}",
            "envs_per_gpu": envs_per_gpu, "num_drones": full.get("num_drones", 1),
            "num_obstacles": full["num_obstacles"], "parallelism": f"env-sharded x{n_gpus}, no data-path collective",
            "l2_policy": "per-step working set larger than L2 (no flush needed)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--envs-per-gpu", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=12)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--cpu-envs", type=int, default=2048)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-global-state", action="store_true")
    ap.add_argument("--no-dr-off", action="store_true", help="skip the secondary DR-off measurement")
    ap.add_argument("--dr-delay", action="store_true",
                    help="also randomise control_delay_steps ({0,1,2} with p {0.7,0.2,0.1}); runs on the general kernel")
    ap.add_argument("--dr", default="auto", choices=["auto", "on", "off"],
                    help="domain randomisation (domain_randomization_v1 ranges); auto = on for c4 (BASELINE configs[3])")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --envs-per-gpu on every GPU; strong: that many env instances IN TOTAL over the GPUs")
    ap.add_argument("--graph", type=int, default=0, metavar="T",
                    help="time CUDA-graph replays of T captured steps instead of a Python loop over step()")
    ap.add_argument("--no-named-sizes", action="store_true", help="skip the block at BASELINE's own env counts")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (rank 0's env instances, a seeded "
                         "sample of them where all would exceed 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.graph and args.steps % args.graph:
        ap.error("--steps must be a multiple of --graph (each replay runs --graph steps)")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm has no device outputs)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    kind, cfg, default_envs = WORKLOADS[args.workload]
    E = args.envs_per_gpu or default_envs
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    if args.scaling == "strong":
        E = max(E // world_env, 1)   # the named batch, sharded (BASELINE config 4: 65536 envs over 8 GPUs)

    if args.impl == "reference":
        run_reference_arm(args, kind, cfg, args.workload, E)
        return

    # stdout carries exactly one JSON line: keep NCCL's "NCCL version ..." banner (NCCL_DEBUG=VERSION) out of it
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    import torch
    import torch.distributed as dist
    import swarm_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def make_engine(dr, kind_=None, cfg_=None, E_=None):
        kind_, cfg_, E_ = kind_ or kind, cfg_ or cfg, E_ or E
        e = swarm_b200.SwarmEngine(E_, cfg_, kind=kind_, device=dev, global_state=not args.no_global_state,
                                   domain_randomization=(dr if isinstance(dr, dict) else DR_V1) if dr else None,
                                   dr_seed=2026, env_index_base=rank * E_)
        # env e of rank r is global env r*E + e: seeds are a function of the GLOBAL env index
        e.seed(np.arange(rank * E_, (rank + 1) * E_, dtype=np.uint64))
        e.reset()
        return e

    if args.dr_delay:
        DR_V1["control_delay_steps"] = ((0, 1, 2), (0.7, 0.2, 0.1))
    eng = make_engine(dr_enabled(args))
    N = eng.N
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    n_act = 4
    actions = [torch.rand((E, N, 3), generator=gen, device=dev) * 2.0 - 1.0 for _ in range(n_act)]

    def timed(e, steps, warmup, sample_clocks, graph_T=None, acts=None):
        """W untimed + K timed steps, CUDA events on the launching stream, max over ranks.  graph_T > 0: the K steps
        are K / T replays of a CUDA graph of T captured steps.  main() only passes a --steps that is a multiple of
        --graph; the secondary legs (pre-warm, DR off, named sizes) have K rounded down to a multiple of T (at least T)."""
        graph_T = args.graph if graph_T is None else graph_T
        acts = actions if acts is None else acts
        E_, N_ = e.E, e.N
        graph, launches_per_replay = None, 0
        if graph_T > 0:
            ring = torch.stack([acts[t % len(acts)] for t in range(graph_T)]).contiguous()
            l_before = e.launch_count
            graph = e.capture_steps(ring, auto_reset=True)
            launches_per_replay = (e.launch_count - l_before) * graph_T // (graph_T + 1)   # capture = 1 warm-up step + T
            steps = max(steps // graph_T, 1) * graph_T
            for w in range(max(warmup // graph_T, 1)):
                graph.replay()
        else:
            for w in range(warmup):
                e.step(acts[w % len(acts)], auto_reset=True)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e.reset_stats()
        sampler = ClockSampler(local_rank) if sample_clocks else None
        if sampler:
            sampler.start()
        l0 = e.launch_count
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record()
        if graph is not None:
            for k in range(steps // graph_T):
                graph.replay()
        else:
            for k in range(steps):
                e.step(acts[k % len(acts)], auto_reset=True)
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        clk = sampler.stop() if sampler else None
        st_ = e.stats()
        n_launch = launches_per_replay * (steps // graph_T) if graph is not None else e.launch_count - l0
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        tot = torch.tensor([st_["agent_steps"], E_ * N_ * steps, st_["episodes"], n_launch, steps], dtype=torch.float64,
                           device=dev)
        if world > 1:
            # the one collective of the path: the episode-statistics reduction (NCCL, tiny)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        tot = [float(x) for x in tot.tolist()]
        tot[4] /= world
        return float(t.item()), tot, clk

    timed(eng, 3, max(args.warmup, 3), False)   # (the first launches on a fresh box run cold: keep them out)
    elapsed_ms, (agent_steps_all, slot_steps_all, episodes_all, launches_all, steps_done), clocks = \
        timed(eng, args.steps, args.warmup, True)
    steps_done = int(steps_done)
    value = agent_steps_all / (elapsed_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(eng, args.dump_outputs)   # before the host-buffer arm steps the same engine again

    dr_off = None
    if dr_enabled(args) and not args.no_dr_off:
        # the reference-identical path (no reference code implements the randomisation): same shape, DR off
        eng0 = make_engine(False)
        ms0, (as0, ss0, ep0, l0, sd0), _ = timed(eng0, max(args.steps // 2, 10), max(args.warmup, 3), False)
        B0 = eng0.algorithmic_bytes_per_agent_step()
        dr_off = {"value": as0 / (ms0 * 1e-3), "unit": "agent-steps/s", "ms_per_step": ms0 / sd0,
                  "roofline_frac": B0 * ss0 / (ms0 * 1e-3) / 1e9 / peaks()[0],
                  "note": "domain randomisation off: bit-identical to the reference's step (tests/)"}
        eng0.close()
        del eng0

    dr_delay = None
    if dr_enabled(args) and not args.no_dr_off and not args.dr_delay:
        # the yaml's whole actuation block: control_delay_steps {0, 1, 2} on top (command ring in HBM, same kernel)
        eng1 = make_engine({**DR_V1, "control_delay_steps": ((0, 1, 2), (0.7, 0.2, 0.1))})
        ms1, (as1, ss1, ep1, l1, sd1), _ = timed(eng1, max(args.steps // 4, 10), max(args.warmup, 3), False)
        B1 = eng1.algorithmic_bytes_per_agent_step()
        dr_delay = {"value": as1 / (ms1 * 1e-3), "unit": "agent-steps/s", "ms_per_step": ms1 / sd1,
                    "roofline_frac": B1 * ss1 / (ms1 * 1e-3) / 1e9 / peaks()[0],
                    "note": "domain randomisation + control_delay_steps (0,1,2)/(0.7,0.2,0.1): command ring read + written"}
        eng1.close()
        del eng1

    # ---- BASELINE's own env counts (launch-bound: a CUDA graph of 20 steps per replay, and the plain loop beside it)
    named = None
    if world == 1 and args.workload == "c4" and not args.envs_per_gpu and not args.no_named_sizes and not args.graph:
        named = {}
        for label, wl, En, dr_on in (("c2_4096_envs", "c2", 4096, False), ("c3_16384_envs", "c3", 16384, False),
                                     ("c4_8192_envs_per_gpu", "c4", 8192, True),
                                     ("c4_8192_envs_per_gpu_dr_off", "c4", 8192, False), ("c5_8192_envs", "c5", 8192, False)):
            k2, c2, _ = WORKLOADS[wl]
            e2 = make_engine(dr_on, k2, c2, En)
            g2 = torch.Generator(device=dev)
            g2.manual_seed(99)
            acts2 = [torch.rand((En, e2.N, 3), generator=g2, device=dev) * 2.0 - 1.0 for _ in range(4)]
            B2 = e2.algorithmic_bytes_per_agent_step()
            msg, (asg, ssg, _, _, sdg), _ = timed(e2, 400, 20, False, graph_T=20, acts=acts2)
            msl, (asl, ssl, _, _, sdl), _ = timed(e2, 200, 10, False, graph_T=0, acts=acts2)
            named[label] = {"value": asg / (msg * 1e-3), "us_per_step": msg / sdg * 1e3,
                            "roofline_frac": B2 * ssg / (msg * 1e-3) / 1e9 / peaks()[0],
                            "mode": "CUDA graph, 20 steps per replay",
                            "python_loop": {"value": asl / (msl * 1e-3), "us_per_step": msl / sdl * 1e3,
                                            "roofline_frac": B2 * ssl / (msl * 1e-3) / 1e9 / peaks()[0]}}
            e2.close()
            del e2, acts2

    # ---- end-to-end through host buffers
    e2e = None
    if not args.no_e2e:
        h = eng.host_buffers()
        host_actions = [a.cpu().pin_memory() for a in actions[:2]]   # the caller's pinned action buffers

        def e2e_run(outputs, n_steps):
            """n_steps of swarm_step_host with the named output set; (ms per step, agent-steps done), max / sum over ranks"""
            for w in range(3):
                eng.step_host(host_actions[w % 2], auto_reset=True, outputs=outputs)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            eng.reset_stats()
            t0 = time.perf_counter()
            ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ee0.record()
            for k in range(n_steps):
                out = eng.step_host(host_actions[k % 2], auto_reset=True, outputs=outputs)
                _ = float(out["reward"][0, 0])               # host reads the result
            ee1.record()
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            ms = max(wall * 1e3, ee0.elapsed_time(ee1))
            te_ = torch.tensor([ms], dtype=torch.float64, device=dev)
            se_ = torch.tensor([eng.stats()["agent_steps"]], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(te_, op=dist.ReduceOp.MAX)
                dist.all_reduce(se_, op=dist.ReduceOp.SUM)
            return te_, se_

        # headline: every output of env.step() -- obs, reward, distance, the five flag arrays (one packed byte per
        # agent, ABI 5), the __all__ flags and global_state; beside it the same with unpacked flag arrays (round 1 / 2a)
        # and the "lean" set (obs, reward, flags: env.step() without the info dicts)
        e2e_set = "packed"
        te, se = e2e_run(e2e_set, args.e2e_steps)
        variants = {}
        for vname, vset in (("unpacked_flag_arrays", None), ("lean_obs_reward_flags", "lean")):
            tv, sv = e2e_run(vset, max(args.e2e_steps // 2, 4))
            vb = eng.host_bytes_per_step(vset)
            variants[vname] = {"value": float(sv.item()) / (float(tv.item()) * 1e-3), "unit": "agent-steps/s",
                               "h2d_bytes_per_step": vb[0], "d2h_bytes_per_step": vb[1]}
        h2d, d2h = eng.host_bytes_per_step(e2e_set)
        # what the link gives a bare pinned device->host copy of the largest output (explains the e2e number)
        # (all ranks at once, behind a barrier: with several GPUs per host this is the ceiling the e2e number lives
        #  under -- the ranks share the host's PCIe root complexes / memory controllers)
        pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h["obs"].copy_(eng.obs, non_blocking=True)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        pe0.record()
        for _ in range(4):
            h["obs"].copy_(eng.obs, non_blocking=True)
        pe1.record()
        torch.cuda.synchronize()
        link_gbs = 4 * eng.obs.numel() * 4 / (pe0.elapsed_time(pe1) * 1e-3) / 1e9
        lk = torch.tensor([link_gbs, -link_gbs, link_gbs], dtype=torch.float64, device=dev)
        if world > 1:
            lmin = lk.clone()
            dist.all_reduce(lmin, op=dist.ReduceOp.MIN)
            dist.all_reduce(lk, op=dist.ReduceOp.SUM)
            link_min, link_max, link_sum = float(lmin[0]), -float(lmin[1]), float(lk[2])
        else:
            link_min = link_max = link_sum = link_gbs
        e2e = {"value": float(se.item()) / (float(te.item()) * 1e-3), "unit": "agent-steps/s",
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": args.e2e_steps,
               "ms_per_step": float(te.item()) / args.e2e_steps,
               "d2h_gbs": d2h / (float(te.item()) / args.e2e_steps * 1e-3) / 1e9, "link_d2h_gbs_measured": link_gbs,
               "link_d2h_concurrent": {"ranks": world, "gbs_per_rank_min": link_min, "gbs_per_rank_max": link_max,
                                       "gbs_total": link_sum,
                                       "note": "bare pinned device->host copy of the obs tensor on every rank at once"},
               "variants": variants,
               "path": "swarm_step_host: pinned host actions -> H2D -> fused step -> D2H of obs, reward, dist, "
                       "the 5 per-agent flag arrays as one packed byte, __all__ flags, global_state "
                       "(4 env-axis chunks on side streams)"}

    if rank == 0:
        peak, peak_src = peaks()
        B = eng.algorithmic_bytes_per_agent_step()
        kernel_ms = elapsed_ms / steps_done
        bytes_per_launch = B * E * N   # per GPU
        achieved = bytes_per_launch / (kernel_ms * 1e-3) / 1e9
        traffic = None
        prof = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(prof):
            try:
                traffic = json.load(open(prof)).get(args.workload, {}).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        line = {
            "metric": "agent_steps_per_sec", "value": value, "unit": "agent-steps/s", "n_gpus": world,
            "steps": steps_done, "warmup": args.warmup, "ms_per_step": elapsed_ms / steps_done,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, kind, cfg, E, world, dr_enabled(args)),
            "slot_steps_per_sec": slot_steps_all / (elapsed_ms * 1e-3),
            "episodes_in_timed_region": episodes_all,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src,
                         "bytes_per_agent_step": B, "bytes_per_launch": bytes_per_launch,
                         "kernel": kernel_name(kind, N, E) + " (step launch) + its auto-reset launch; achieved uses the time of both",
                         "kernel_ms": kernel_ms},
            "e2e": e2e,
            "dr_off": dr_off,
            "dr_delay": dr_delay,
            "named_sizes": named,
            "gpu_launches": int(launches_all),
            "clocks": clocks,
        }
        if not args.no_cpu:
            threads = len(os.sched_getaffinity(0))
            rate, csteps, cdt = cpu_port_rate(kind, cfg, args.cpu_envs, args.cpu_seconds, threads, dr_enabled(args))
            port = {"value": rate, "unit": "agent-steps/s", "cores": threads, "kind": "port",
                    "sample": f"{args.cpu_envs} env instances x {csteps} steps of the same config in {cdt:.1f} s "
                              f"(oracle/swarm_oracle.c, scalar C port of the reference algorithm, {threads} threads)"}
            ref = python_reference_rate(kind, cfg, min_seconds=min(args.cpu_seconds, 8.0))
            if ref is not None:
                # the reference itself (pure Python, staged by oracle/make_ref.py) is the baseline; the port rides along
                line["cpu_baseline"] = {
                    "value": ref["rate"], "unit": "agent-steps/s", "cores": ref["procs"], "kind": "reference",
                    "sample": f"the unmodified reference env (oracle/_ref), {ref['procs']} worker processes x "
                              f"{ref['envs_per_proc']} env instance(s) x {ref['steps_per_proc']} steps of the same config in "
                              f"{ref['seconds']:.1f} s (randomisation off: no reference code implements it)"}
                line["cpu_port"] = port
            else:
                line["cpu_baseline"] = port
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
