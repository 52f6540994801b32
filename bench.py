#!/usr/bin/env python
"""bench.py - env-steps/s of the batched step hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One "step" = one gca_step over one batch of 65,536 environments per GPU (SingleAircraft2Env,
continuous actions, 80 intruders, fast mode, Philox draws, VecEnv auto-reset, observation
written every step): 2 kernels - the main kernel (ownship role + the streaming pass over the
intruders) and the finish (+ spawn phase).  Prints ONE JSON line (rank 0).

  value      whole-job env-steps/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e        the same metric through the host-buffer C-ABI call (gca_step_host): actions come
             from pinned host memory and obs/reward/done/info are copied back every step
  roofline   the dominant kernel (step_intruders_kernel): its algorithmic bytes per launch (40 N per
             env) / its launch duration, measured live with CUDA events between the kernels of the step
             (gca_profile_*), vs the measured HBM peak; `step` gives the same for the whole step
  cpu_baseline  the CPU oracle port on the box's host cores, on a bounded sample (rank 0, N=1), and
             `python_reference`: the unmodified reference's own Python loop as timed in the build
             container (profiles/python_reference_timing.json; the reference cannot travel to the box)

--impl reference times the CPU oracle port alone, with the oracle library only (no libgca.so, no
product package): the reference is Python and cannot travel to the GPU box; the port is pinned
bit-exact to it by tests/test_oracle_golden.py.

--dump-outputs DIR writes what the last timed step returned (rank 0) as DIR/<name>.npy, so that two
builds run with the same arguments (same seeds, same inputs) can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "gym-guidance-collision-avoidance-single_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

ENVS_PER_GPU = 65536
N_INTRUDERS = 80
VARIANT = "SingleAircraft2Env"
METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
GRAPH_STEPS = 50            # steps captured per CUDA graph (actions cycle through this many batches)
DUMP_OBS_ROWS = 16384       # --dump-outputs: observation rows of a seeded sample of envs (21.5 MB of f32 at N = 80)


def workload_name():
    return ("%s continuous [-1,1]^2 actions, %d envs/GPU, %d intruders, fast mode (f32 state+obs, f64 ownship), "
            "Philox draws, auto-reset, vector obs written every step" % (VARIANT, ENVS_PER_GPU, N_INTRUDERS))


def workload_config(**extra):
    """`config` of the JSON line: the same keys in both arms (ours / reference)."""
    cfg = {"workload": workload_name(), "envs_per_gpu": ENVS_PER_GPU, "intruders": N_INTRUDERS, "variant": VARIANT,
           "mode": "fast", "draws": "philox", "auto_reset": True, "sample": None, "l2": None, "launch": None}
    cfg.update(extra)
    return cfg


def algorithmic_bytes_per_env_step(n, continuous=True):
    """DESIGN.md 'Algorithmic bytes': what one env-step must move in fast mode."""
    per_intruder = 8 + 8 + 8 + 16            # read pos, read vel, write pos, write 4 f32 obs entries
    flags = 4 * ((n + 31) // 32)             # conflict-flag words read (written only on a transition)
    fixed = (16 + 32 + 16 + 1 + 16 + 32      # own_pos r/w, heading+speed r/w, own_vel w, vel flag w, goal r, counters r/w
             + (8 if continuous else 4)      # action
             + 4 + 1 + 1                     # reward, done, info
             + 32)                           # ownship + goal tail of the observation
    return per_intruder * n + flags + fixed


def streaming_bytes_per_env_step(n):
    """Algorithmic bytes of the dominant kernel alone (step_intruders_kernel, SURVEY 8(d)): per intruder 8 (pos r) +
    8 (vel r) + 8 (pos w) + 16 (obs entries w) = 40."""
    return 40 * n


def handover_bytes_per_env_step(n):
    """NOT algorithmic: the 16-byte ownship record every 8-intruder work item of the streaming pass re-reads (an
    implementation overhead, served by the L2; reported beside the roofline, never inside it)."""
    return 16 * ((n + 7) // 8)


def python_reference_figures():
    """The unmodified reference's own Python step loop, timed in the BUILD container by
    tools/time_python_reference.py (BASELINE.md section 3 protocol): it cannot run on the GPU box (no gym, the
    reference tree does not travel), so the line carries the committed figures with their provenance."""
    try:
        with open(os.path.join(ROOT, "profiles", "python_reference_timing.json")) as f:
            return json.load(f)
    except Exception:
        return None


def bind_to_gpu_numa_node(index):
    """Pin this rank's host thread to the cores of the NUMA node its GPU hangs off, so that the pinned buffers it
    allocates next (first touch) are local to the GPU's PCIe root.  Returns what to restore, or None."""
    try:
        import torch
        p = torch.cuda.get_device_properties(index)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as f:
            node = int(f.read().strip())
        if node < 0:
            return {"old": None, "note": "GPU %s reports no NUMA node (single-node host)" % bdf}
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        old = os.sched_getaffinity(0)
        use = cpus & old
        if not use:
            return {"old": None, "note": "NUMA node %d has no core this process may use" % node}
        os.sched_setaffinity(0, use)
        return {"old": old, "note": "host thread and pinned buffers on NUMA node %d (%d cores) of GPU %s" % (node, len(use), bdf)}
    except Exception as e:     # no sysfs / no permission: leave the placement to the OS
        return {"old": None, "note": "not bound (%s)" % type(e).__name__}


def dump_outputs(out_dir, env):
    """What step() returned in the last timed step, as float32 (float64 where the output is) .npy files: reward, done
    and info of every env, and obs of a fixed, seeded sample of envs whose ids obs_rows holds."""
    os.makedirs(out_dir, exist_ok=True)
    rows = np.sort(np.random.RandomState(0).choice(env.num_envs, min(DUMP_OBS_ROWS, env.num_envs), replace=False))
    arrays = {"obs": env.obs.cpu().numpy()[rows], "obs_rows": rows.astype(np.float64), "reward": env.reward.cpu().numpy(),
              "done": env.done.cpu().numpy(), "info": env.info.cpu().numpy()}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64 if a.dtype == np.float64 else np.float32))


def restore_affinity(numa):
    if numa and numa.get("old"):
        try:
            os.sched_setaffinity(0, numa["old"])
        except Exception:
            pass


def measure_d2h_ceiling(torch, nbytes, barrier, copies=8):
    """Time `copies` device->host copies of nbytes into pinned memory (what one e2e step downloads), all ranks at once."""
    src = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    dst = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(copies):
        dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    return {"seconds": time.perf_counter() - t0, "copies": copies}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_kernel_us():
    """duration of one launch of the step kernel in the committed ncu capture (cold, serialised), if present."""
    try:
        with open(os.path.join(ROOT, "profiles", "step_kernel_ncu.json")) as f:
            return json.load(f).get("gpu_time_us")
    except Exception:
        return None


def ncu_traffic():
    """dram bytes per launch of the step kernel from the committed ncu summary, if present."""
    path = os.path.join(ROOT, "profiles", "step_kernel_ncu.json")
    try:
        with open(path) as f:
            return json.load(f).get("dram_bytes_per_launch")
    except Exception:
        return None


# ------------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Polls SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index, period=0.01):
        threading.Thread.__init__(self, daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = str(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------- CPU arm
def oracle_shards(cores, envs, seed):
    """(nothing of the product is imported here: the workload's gca_config is written out in oracle/structs.py)"""
    from oracle import oracle as orc
    from oracle import structs
    cfg = structs.bench_workload_config()
    per = envs // cores
    shards = []
    for c in range(cores):
        e = orc.OracleEnv(cfg, per, N_INTRUDERS, draws=1, trig=orc.TRIG_SHARED, seed=seed, env_id0=c * per,
                          f32_positions=True, auto_reset=True)
        shards.append(e)
    return shards


def run_cpu(steps, warmup, sample_envs=None, budget_s=20.0):
    """Time the CPU oracle port: `cores` threads (ctypes releases the GIL), each advancing its own
    shard of a bounded sample of the workload (same variant, N, fast-mode rules, Philox, auto-reset)."""
    from concurrent.futures import ThreadPoolExecutor
    cores = os.cpu_count() or 1
    if sample_envs is None:
        sample_envs = 512 * cores
    shards = oracle_shards(cores, sample_envs, seed=0)
    per = shards[0].B
    rng = np.random.RandomState(1)
    acts = [rng.uniform(-1, 1, (per, 2)).astype(np.float32).astype(np.float64) for _ in range(cores)]
    pool = ThreadPoolExecutor(cores)
    list(pool.map(lambda e: e.reset(), shards))

    def one_step():
        list(pool.map(lambda ea: ea[0].step(ea[1]), zip(shards, acts)))
    for _ in range(max(warmup, 1)):
        one_step()
    t0 = time.perf_counter()
    one_step()
    per_step = time.perf_counter() - t0
    steps = max(1, min(steps, int(budget_s / max(per_step, 1e-6))))
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    dt = time.perf_counter() - t0
    pool.shutdown()
    value = per * cores * steps / dt
    out = {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
           "sample": "%d envs x %d intruders x %d steps (%.1f s), C oracle port (oracle/gca_oracle.c), %d threads"
                     % (per * cores, N_INTRUDERS, steps, dt, cores), "sample_envs": per * cores, "sample_steps": steps}
    py = python_reference_figures()
    if py is not None:
        out["python_reference"] = py
    return out, steps, dt


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import subprocess
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")], stdout=sys.stderr)   # the oracle ONLY
    cb, steps, dt = run_cpu(args.steps, args.warmup, budget_s=60.0)
    assert "gca_b200" not in sys.modules, "the reference arm must not import the product"
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
            "config": workload_config(sample="%d envs x %d steps on %d host threads (bounded sample of the workload)"
                                             % (cb["sample_envs"], cb["sample_steps"], cb["cores"])),
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------- GPU arm
def main_gpu(args):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if rank == 0:
        ge.build()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":      # NCCL would print its banner on stdout,
            os.environ["NCCL_DEBUG"] = "WARN"                           # ahead of the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()

    from gca_b200.batched import BatchedAircraftEnv
    from gym_guidance_collision_avoidance_single.envs.config import Config

    B, N = ENVS_PER_GPU, N_INTRUDERS
    env = BatchedAircraftEnv(VARIANT, B, Config, n_intruders=N, mode="fast", draws="philox", device=local, seed=2024,
                             env_id0=rank * B)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1 + rank)
    actions = [torch.rand((B, 2), device="cuda", generator=gen) * 2 - 1 for _ in range(GRAPH_STEPS)]
    env.reset()
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    K, W = args.steps, max(args.warmup, 3)
    # K steps = full replays of a CUDA graph of G = min(K, GRAPH_STEPS) steps + an eager remainder
    G = max(1, min(K, GRAPH_STEPS))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(W):
            env.step(actions[i % GRAPH_STEPS])
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(G):
            env.step(actions[i])
    graph.replay()                                    # one untimed replay
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    start.record()
    done_steps = 0
    replays = K // G
    for _ in range(replays):
        graph.replay()
        done_steps += G
    eager_steps = K - done_steps
    for i in range(eager_steps):
        env.step(actions[i])
    stop.record()
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:              # before the legs below step the same envs again
        dump_outputs(args.dump_outputs, env)
    ms = start.elapsed_time(stop)
    t = torch.tensor([ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * B * K / (ms * 1e-3)

    # ---- the dominant kernel, timed live: CUDA events between the kernels of each step, same workload, right
    # after the timed region (eager launches; the events sit on the stream the kernels are launched on)
    Kp = max(20, min(K, 200))
    env.profile(True)
    for i in range(Kp):
        env.step(actions[i % GRAPH_STEPS])
    prof = env.read_profile()
    env.profile(False)
    kernels_per_step = env.kernels_per_step

    # ---- end to end through the host-buffer C-ABI call (GCA_BENCH_KERNEL_ONLY=1 skips it for ncu captures)
    kernel_only = os.environ.get("GCA_BENCH_KERNEL_ONLY") == "1"
    host_actions = [a.cpu().numpy() for a in actions[:8]]
    numa = bind_to_gpu_numa_node(local)               # before the pinned buffers are allocated (first touch)
    for i in range(3):
        env.step_host(host_actions[i % 8])
    Ke = 3 if kernel_only else max(3, min(K, 300))

    def wall_max(seconds):
        te = torch.tensor([seconds], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return float(te.item())

    # (a) one step at a time: upload, step, download, synchronise
    barrier()
    t0 = time.perf_counter()
    for i in range(Ke):
        obs, rew, dn, info = env.step_host(host_actions[i % 8])
        _ = float(rew[0])
    torch.cuda.synchronize()
    e2e_serial = world * B * Ke / wall_max(time.perf_counter() - t0)
    # (b) VecEnv step_async / step_wait with two steps in flight: the download of step t runs under the kernels of t + 1
    for i in range(2):
        env.step_host_begin(host_actions[i % 8])
        env.step_host_wait()
    barrier()
    t0 = time.perf_counter()
    env.step_host_begin(host_actions[0])
    for i in range(1, Ke):
        env.step_host_begin(host_actions[i % 8])
        obs, rew, dn, info = env.step_host_wait()
        _ = float(rew[0])
    obs, rew, dn, info = env.step_host_wait()
    _ = float(rew[0])
    torch.cuda.synchronize()
    e2e_value = world * B * Ke / wall_max(time.perf_counter() - t0)
    h2d, d2h = env.host_io_bytes()
    # (c) what the host link gives this rank while every rank downloads at once: the ceiling of (a) and (b)
    link = measure_d2h_ceiling(torch, d2h, barrier)
    link_gbs = d2h * link["copies"] / wall_max(link["seconds"]) / 1e9
    restore_affinity(numa)

    if rank == 0:
        peak, peak_src = measured_peaks()
        bytes_per_step = algorithmic_bytes_per_env_step(N) * B
        step_ms = ms / K
        step_gbs = bytes_per_step / (step_ms * 1e-3) / 1e9
        bytes_per_launch = streaming_bytes_per_env_step(N) * B
        launch_ms = prof["intruders_ms"] / max(prof["steps"], 1)
        achieved = bytes_per_launch / (launch_ms * 1e-3) / 1e9
        prof_step_ms = (prof["own_ms"] + prof["intruders_ms"] + prof["finish_ms"] + prof["spawn_ms"]) / max(prof["steps"], 1)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32+f64", "data": "synthetic",
            "config": workload_config(
                sample="the whole workload: %d envs per GPU x %d steps" % (B, K),
                l2="per-step footprint %.0f MB (state+obs) exceeds the 126 MB L2; no flush between steps" % (bytes_per_step / 1e6),
                launch="%d replay(s) of a CUDA graph of %d steps + %d eager step(s); %d kernels per step"
                       % (replays, G, eager_steps, kernels_per_step)),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": Ke,
                    "api": "BatchedAircraftEnv.step_host_begin / step_host_wait -> gca_step_host_begin / _wait (pinned host "
                           "buffers, two steps in flight: the download of step t under the kernels of step t + 1)",
                    "serial_value": e2e_serial,
                    "serial_api": "BatchedAircraftEnv.step_host -> gca_step_host (one step at a time)",
                    "host_link_gbs": (h2d + d2h) * (e2e_value / world / B) / 1e9,
                    "link_ceiling_gbs": link_gbs,
                    "link_ceiling_note": "per rank: %d device->host copies of %d bytes into pinned memory, every rank at "
                                         "once, max over ranks - what the host memory system gives one rank with %d "
                                         "GPU(s) downloading" % (link["copies"], d2h, world),
                    "numa": numa.get("note") if numa else None,
                    "note": "bound by the device->host copy of the observations over PCIe, not by the kernels"},
            "gpu_launches": K * kernels_per_step,
            "roofline": {"bound": "hbm", "kernel": "step_intruders_kernel", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic(), "peak_source": peak_src,
                         "bytes_per_env_step": streaming_bytes_per_env_step(N), "kernel_ms": launch_ms,
                         "overhead_bytes_per_env_step": handover_bytes_per_env_step(N),
                         "overhead_note": "the 16-byte ownship record each 8-intruder work item re-reads (L2 hits): not algorithmic, not in `achieved`",
                         "share_of_step": launch_ms / prof_step_ms if prof_step_ms else None,
                         "timing": "CUDA events between the kernels of %d eager steps (gca_profile_*); the kernel is the main "
                                   "kernel of the step (its first blocks play the ownship role, the others stream the "
                                   "intruders); an event interval includes the drain / launch gap around the kernel, so "
                                   "achieved is a lower bound (kernel_us_ncu: the committed ncu capture)" % prof["steps"],
                         "kernel_us_ncu": ncu_kernel_us(),
                         "l2_note": "achieved = ALGORITHMIC bytes / live time. In the graph the DRAM traffic is lower than that: "
                                    "the position plane a step writes (plain stores) is largely still in the 126 MB L2 when "
                                    "the next step reads it (tiles walked in alternating directions) and is discarded after "
                                    "the read instead of written back; `traffic` is the cold, serialised ncu capture",
                         "kernels_ms": {"main (ownship role + streaming pass)": launch_ms,
                                        "finish + spawn phase": prof["finish_ms"] / max(prof["steps"], 1)},
                         "step": {"achieved": step_gbs, "frac": step_gbs / peak,
                                  "bytes_per_env_step": algorithmic_bytes_per_env_step(N), "ms": step_ms}},
        }
        if world == 1 and not kernel_only:
            cb, _, _ = run_cpu(10 ** 9, 1, budget_s=12.0)
            line["cpu_baseline"] = cb
    env.check()
    env.close()
    # ---- the other configs / metrics of BASELINE.json.  EVERY rank runs them on its own shard (independent envs /
    # roots: no collective on the data path); a leg's time is the MAX over ranks and its value the whole-job aggregate,
    # like the headline.  At N > 1 only the BASELINE configs (#3 HER, #4 MCTS, #5 stack) run; the rest is N = 1 detail.
    extras = {}
    if not kernel_only:
        legs = [("her", bench_her), ("mcts", lambda d: bench_mcts(d, with_cpu=(world == 1 and rank == 0))), ("stack", bench_stack)]
        if world == 1:
            legs += [("d9her", bench_d9her), ("mctsrnd", bench_mctsrnd), ("her_replay", bench_her_replay), ("n0", bench_n0),
                     ("faithful", bench_faithful)]
        for name, fn in legs:
            if world > 1:
                dist.barrier()
            extras[name] = reduce_leg(fn(local), world, dist if world > 1 else None)
    if rank == 0:
        line.update(extras)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_MS_KEYS = ("ms_per_step", "ms_per_launch")


def reduce_leg(d, world, dist):
    """Whole-job figure of a leg every rank ran on its own shard: time = MAX over ranks, value = world x the units one
    rank processed / that time (nested dicts with a `value` and a ms key are treated alike)."""
    if not isinstance(d, dict):
        return d
    out = {}
    for k, v in d.items():
        out[k] = reduce_leg(v, world, dist) if isinstance(v, dict) else v
    key = next((k for k in _MS_KEYS if k in d), None)
    if dist is not None and key is not None and isinstance(d.get("value"), (int, float)):
        import torch
        t = torch.tensor([float(d[key])], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        out["value"] = world * d["value"] * d[key] / ms
        out[key] = ms
        out["n_gpus"] = world
        out["per_rank"] = {k: d[k] for k in ("envs", "roots", "batch") if k in d}
    return out


def bench_mcts(device, with_cpu):
    """Second metric of BASELINE.json: MCTS rollouts/s = completed random playouts (root -> terminal or
    depth 3, 10 sub-frames per move, N = 80) per second, config #4.  Rank-local (independent roots)."""
    import torch
    from gca_b200 import abi, mcts
    from gca_b200.batched import BatchedAircraftEnv
    from Simulators.config import Config as SimConfig
    from Algorithms.MCTS.config_single import Config as MctsConfig
    R, P, depth = 4096, 100, 3
    env = BatchedAircraftEnv("SingleAircraftMCTSEnv", R, SimConfig, n_intruders=80, mode="faithful", device=device, seed=2)
    roots = env.reset().clone()                      # raw observations after reset = MCTS root states
    cfg = abi.make_mcts_config(MctsConfig)
    for _ in range(20):
        mcts.playouts(roots, P, depth=depth, cfg=cfg, seed=5)
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 100
    start.record()
    for i in range(reps):
        rewards, _, flags = mcts.playouts(roots, P, depth=depth, cfg=cfg, seed=6 + i)
    stop.record()
    torch.cuda.synchronize()
    ms = start.elapsed_time(stop) / reps
    out = {"metric": "mcts_rollouts_per_sec", "value": R * P / (ms * 1e-3), "unit": "rollouts/s", "roots": R,
           "playouts_per_root": P, "depth": depth, "intruders": 80, "ms_per_launch": ms,
           "mean_reward": float(rewards.mean().item()), "terminal_fraction": float((flags != 0).float().mean().item()),
           "dtype": "f64", "bound": "fp64 pipe (no HBM roofline: a 2.6 KB root is read once per CTA of 100 playouts)"}
    # FP64 roofline of the playout kernel: f64 operations per launch counted by ncu (profiles/mcts_kernel_ncu.json,
    # same workload) / the launch time measured here, against the measured non-fused DMUL+DADD peak of this pool's
    # B200 (profiles/fp64_peak.json; the parity contract forbids contracting the reference's mul/add pairs into FMAs)
    rl = fp64_roofline("mcts_kernel_ncu.json", ms)
    if rl:
        out["roofline"] = rl
    # device-resident UCT search (SURVEY 8(f) rank 1): decisions/s = best_action(100 simulations, depth 3) per root
    try:
        R2 = 65536
        env2 = BatchedAircraftEnv("SingleAircraftMCTSEnv", R2, SimConfig, n_intruders=80, mode="faithful", device=device, seed=3)
        roots2 = env2.reset().clone()
        env2.close()
        for _ in range(2):
            mcts.search(roots2, P, depth, cfg=cfg, seed=1)
        torch.cuda.synchronize()
        start.record()
        for i in range(3):
            mcts.search(roots2, P, depth, cfg=cfg, seed=2 + i)
        stop.record()
        torch.cuda.synchronize()
        ms2 = start.elapsed_time(stop) / 3
        out["search"] = {"metric": "mcts_decisions_per_sec", "value": R2 / (ms2 * 1e-3), "unit": "searches/s",
                         "roots": R2, "simulations": P, "depth": depth, "ms_per_launch": ms2,
                         "simulations_per_sec": R2 * P / (ms2 * 1e-3),
                         "api": "gca_mcts_search (UCT tree per root resident on the device, one lane per root)"}
        rl2 = fp64_roofline("mcts_search_ncu.json", ms2)
        if rl2:
            out["search"]["roofline"] = rl2
    except Exception as exc:                                          # pragma: no cover
        out["search"] = {"error": str(exc)}
    env.close()
    if with_cpu:
        # same protocol as the step baseline: the C oracle port on ALL host cores (ctypes releases the GIL), one shard
        # of roots per thread, a bounded sample
        from concurrent.futures import ThreadPoolExecutor
        from oracle import oracle as orc
        cores = os.cpu_count() or 1
        all_roots = roots.cpu().numpy()
        pool = ThreadPoolExecutor(cores)

        def timed(fn, per, budget_s=4.0):
            """grow the sample (roots per thread) until one pass takes about budget_s seconds of wall clock"""
            while True:
                n = per * cores
                host_roots = all_roots[:n] if all_roots.shape[0] >= n else all_roots.repeat((n + R - 1) // R, 0)[:n]
                shards = [host_roots[c * per:(c + 1) * per] for c in range(cores)]
                t0 = time.perf_counter()
                list(pool.map(fn, shards))
                dt = time.perf_counter() - t0
                if dt >= budget_s / 2 or per >= (1 << 16):
                    return per, dt
                per = int(min(1 << 16, max(per * 2, per * budget_s / max(dt, 1e-3))))

        per, dt = timed(lambda sh: orc.mcts_search_philox(cfg, 80, sh, P, depth, seed=2), 4)
        out["search"]["cpu_baseline"] = {"value": per * cores / dt, "unit": "searches/s", "cores": cores, "kind": "port",
                                         "sample": "%d roots x %d simulations (%.1f s), C oracle port, %d threads" % (per * cores, P, dt, cores)}
        per, dt = timed(lambda sh: orc.mcts_playouts(cfg, 80, sh, 50, depth, seed=6), 16)
        pool.shutdown()
        out["cpu_baseline"] = {"value": per * cores * 50 / dt, "unit": "rollouts/s", "cores": cores, "kind": "port",
                               "sample": "%d roots x 50 playouts (%.1f s), C oracle port (oracle/gca_oracle_mcts.c), %d threads"
                                         % (per * cores, dt, cores)}
        py = python_reference_figures()
        if py is not None and "mcts" in py:
            out["cpu_baseline"]["python_reference"] = py["mcts"]
    return out


def fp64_roofline(profile_name, ms):
    """FP64 roofline of a kernel: f64 operations per launch counted by ncu on the same workload (profiles/<name>.json) /
    the launch time measured live, against the measured non-fused DMUL+DADD peak of this pool's B200
    (profiles/fp64_peak.json; the parity contract forbids contracting the reference's mul/add pairs into FMAs)."""
    try:
        with open(os.path.join(ROOT, "profiles", profile_name)) as f:
            prof = json.load(f)
        with open(os.path.join(ROOT, "profiles", "fp64_peak.json")) as f:
            peak = float(json.load(f)["dmul_dadd_tflops"])
        ops = float(prof["f64_ops_per_launch"])
        ach = ops / (ms * 1e-3) / 1e12
        return {"bound": "fp64", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                "peak_source": "measured (tools/fp64_peak.cu, separate DMUL+DADD)", "ops_per_launch": ops,
                "kernel": prof.get("kernel"), "fp64_pipe_pct_ncu": prof.get("fp64_pipe_pct_of_peak_sustained_active")}
    except Exception:
        return None


def bench_her(device):
    """BASELINE.json config #3: SingleAircraftHEREnv (dict observation: observation / achieved_goal / desired_goal)
    stepped on the device, followed by a relabel batch: compute_reward on M = 4*B (achieved, substitute goal) pairs
    (k = 4 future goals per transition, Algorithms/DDPG/DDPG.py:38,308-315)."""
    import torch
    from gca_b200 import abi
    from gca_b200.batched import BatchedAircraftEnv, compute_reward
    from gym_guidance_collision_avoidance_single.envs.config import Config
    B, N, k = ENVS_PER_GPU, N_INTRUDERS, 4
    env = BatchedAircraftEnv("SingleAircraftHEREnv", B, Config, n_intruders=N, mode="fast", draws="philox", device=device, seed=4)
    env.reset()
    acts = [torch.rand((B, 2), device="cuda") * 2 - 1 for _ in range(8)]
    goals = torch.rand((k, B, 2), device="cuda")                       # substitute goals (normalised, like desired_goal)

    def one(i):
        env.step(acts[i % 8])
        return compute_reward(env.achieved, goals, Config.goal_radius, abi.OBS_HER)     # [B, 2] against [k, B, 2]
    for i in range(5):
        one(i)
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 200
    start.record()
    for i in range(reps):
        one(i)
    stop.record()
    torch.cuda.synchronize()
    ms_eager = start.elapsed_time(stop) / reps
    ms = graph_step_ms(one, 8)                                         # the headline's launch mode
    env.close()
    return {"metric": METRIC, "value": B / (ms * 1e-3), "unit": UNIT, "envs": B, "intruders": N,
            "relabel_pairs_per_step": k * B, "ms_per_step": ms, "ms_per_step_eager": ms_eager,
            "note": "step (dict observation, own-first layout) + HER relabel reward on 4*B pairs; CUDA graph of 8 steps "
                    "replayed (ms_per_step_eager: the same launched one call at a time)"}


def graph_step_ms(step_fn, n_batches, reps=6):
    """ms per step of `step_fn(i)` captured as a CUDA graph of n_batches steps and replayed (same launch mode as the
    headline number); warm-up on a side stream as graph capture requires."""
    import torch
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(3):
            step_fn(i % n_batches)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(n_batches):
            step_fn(i)
    graph.replay()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        graph.replay()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / (reps * n_batches)


def bench_d9her(device):
    """SURVEY 8(f) rank 2: Simulators/SingleAircraftDiscrete9HEREnv (random ownship start, observation = ownship + the
    4 nearest intruders, dict goals) - the env the repo's own learners train on.  5 kernels per step (the nearest-n
    pass runs behind the spawn kernel on the final intruder set)."""
    import torch
    from gca_b200.batched import BatchedAircraftEnv
    from Simulators.config import Config as SimConfig
    B, N = ENVS_PER_GPU, N_INTRUDERS
    env = BatchedAircraftEnv("SingleAircraftDiscrete9HEREnv", B, SimConfig, n_intruders=N, mode="fast", draws="philox",
                             device=device, seed=6)
    env.reset()
    acts = [torch.randint(0, 9, (B,), device="cuda", dtype=torch.int32) for _ in range(8)]
    for i in range(5):
        env.step(acts[i % 8])
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 200
    start.record()
    for i in range(reps):
        env.step(acts[i % 8])
    stop.record()
    torch.cuda.synchronize()
    ms_eager = start.elapsed_time(stop) / reps
    acts50 = [torch.randint(0, 9, (B,), device="cuda", dtype=torch.int32) for _ in range(GRAPH_STEPS)]
    ms = graph_step_ms(lambda i: env.step(acts50[i]), GRAPH_STEPS)
    k = env.kernels_per_step
    env.close()
    out = {"metric": METRIC, "value": B / (ms * 1e-3), "unit": UNIT, "envs": B, "intruders": N, "ms_per_step": ms,
           "ms_per_step_eager": ms_eager, "kernels_per_step": k, "obs_dim": 24,
           "note": "nearest-4 observation (24 values + goals); CUDA graph of %d steps replayed" % GRAPH_STEPS}
    # the Discrete(3) sibling: + nearest-intruder reward term measured in the finish kernel
    env3 = BatchedAircraftEnv("SingleAircraftDiscrete3HEREnv", B, SimConfig, n_intruders=N, mode="fast", draws="philox",
                              device=device, seed=7)
    env3.reset()
    acts3 = [torch.randint(0, 3, (B,), device="cuda", dtype=torch.int32) for _ in range(GRAPH_STEPS)]
    ms3 = graph_step_ms(lambda i: env3.step(acts3[i]), GRAPH_STEPS)
    env3.close()
    out["d3her"] = {"value": B / (ms3 * 1e-3), "unit": UNIT, "ms_per_step": ms3}
    return out


def bench_mctsrnd(device):
    """SURVEY 8(f) rank 4: Simulators/SingleAircraftMCTSRandIntruderEnv (intruders that turn at random after every step,
    per-step drift, six raw entries per intruder).  5 kernels per step: the turn / observation pass runs behind the
    spawn kernel on the final intruder set, one lane per (env, intruder).  Algorithmic bytes per env-step: per intruder
    24 (position r/w, velocity r) in the streaming pass + 8 + 8 + 16 (position, velocity, heading / speed read again)
    + 24 (six f32 entries written) = 80, plus the per-env scalars."""
    import torch
    from gca_b200.batched import BatchedAircraftEnv
    from Simulators.config import Config as SimConfig
    B, N = ENVS_PER_GPU, N_INTRUDERS
    env = BatchedAircraftEnv("SingleAircraftMCTSRandIntruderEnv", B, SimConfig, n_intruders=N, mode="fast",
                             draws="philox", device=device, seed=8)
    env.reset()
    acts = [torch.randint(0, 9, (B,), device="cuda", dtype=torch.int32) for _ in range(GRAPH_STEPS)]
    for i in range(5):
        env.step(acts[i])
    ms = graph_step_ms(lambda i: env.step(acts[i]), GRAPH_STEPS)
    k = env.kernels_per_step
    # the planner model of Agent_RandInt.py (nodes_single_randintru.py) on these observations: every playout moves and
    # turns its own intruders, one warp per playout
    from gca_b200 import abi, mcts
    from Algorithms.MCTS.config_single import Config as MctsConfig
    R, P, depth = 2048, 100, 3
    roots = env.obs[:R].double().contiguous()
    mcfg = abi.make_mcts_config(MctsConfig, random_intruders=True)
    mcts.playouts(roots, P, depth=depth, cfg=mcfg, seed=1)
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for rep_i in range(10):
        mcts.playouts(roots, P, depth=depth, cfg=mcfg, seed=2 + rep_i)
    stop.record()
    torch.cuda.synchronize()
    pms = start.elapsed_time(stop) / 10
    env.close()
    peak, _ = measured_peaks()
    bytes_per_env_step = 80 * N + 122
    gbs = bytes_per_env_step * B / (ms * 1e-3) / 1e9
    return {"metric": METRIC, "value": B / (ms * 1e-3), "unit": UNIT, "envs": B, "intruders": N, "ms_per_step": ms,
            "kernels_per_step": k, "obs_dim": 6 * N + 8, "bytes_per_env_step": bytes_per_env_step,
            "hbm_frac": gbs / peak, "note": "CUDA graph of %d steps replayed" % GRAPH_STEPS,
            "model": {"metric": "mcts_rollouts_per_sec", "value": R * P / (pms * 1e-3), "unit": "rollouts/s", "roots": R,
                      "playouts_per_root": P, "depth": depth, "intruders": N, "ms_per_launch": pms,
                      "roofline": fp64_roofline("mctsrnd_model_ncu.json", pms),
                      "kernel": "mcts_playout_rnd_lane_kernel (nodes_single_randintru.py model; one playout per lane, two roots per CTA, "
                                "intruders out of reach culled exactly once per root; bound by instruction issue - one Philox block per "
                                "intruder and sub-frame -, the FP64 fraction is reported for comparison with the other MCTS kernels)"}}


def bench_her_replay(device):
    """SURVEY 8(f) rank 3: HER "future" relabelling sampler (baselines her_sampler.py:19-61) on a device-resident
    episode buffer: gather of six rows per transition + goal substitution + reward.  Pure data movement: algorithmic
    bytes = 2 * (2 dim_o + dim_u + 4 dim_g) * 4 + 16 per transition (rows read once, written once; r + 3 int32 out)."""
    import torch
    from gca_b200 import abi, replay
    E, T, dim_o, dim_u, batch = 4096, 50, 4 * N_INTRUDERS + 6, 2, 262144
    g = torch.Generator(device="cuda").manual_seed(0)
    eb = {"o": torch.rand((E, T + 1, dim_o), device="cuda", generator=g), "u": torch.rand((E, T, dim_u), device="cuda", generator=g),
          "g": torch.rand((E, T, 2), device="cuda", generator=g), "ag": torch.rand((E, T + 1, 2), device="cuda", generator=g)}
    for i in range(5):
        replay.sample_her_transitions(eb, batch, 4, 20.0, abi.OBS_HER, seed=1, call=i)
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 50
    start.record()
    for i in range(reps):
        replay.sample_her_transitions(eb, batch, 4, 20.0, abi.OBS_HER, seed=1, call=10 + i)
    stop.record()
    torch.cuda.synchronize()
    ms = start.elapsed_time(stop) / reps
    bytes_per = 2 * (2 * dim_o + dim_u + 4 * 2) * 4 + 16
    peak, src = measured_peaks()
    gbs = batch * bytes_per / (ms * 1e-3) / 1e9
    return {"metric": "her_transitions_per_sec", "value": batch / (ms * 1e-3), "unit": "transitions/s", "batch": batch,
            "episodes": E, "T": T, "dim_o": dim_o, "ms_per_launch": ms, "bytes_per_transition": bytes_per,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                         "peak_source": src, "note": "includes the torch.empty of the output tensors per call"}}


def bench_n0(device):
    """SURVEY 8(d) input #1 at the package default `Config.intruder_size = 0` (PKG/config.py:9): SingleAircraftEnv,
    discrete actions, no intruders - 2 kernels per step, 155 algorithmic bytes per env-step.  65,536 envs are 10 MB of
    state (L2 resident); 4 Mi envs make it HBM bound."""
    import torch
    from gca_b200.batched import BatchedAircraftEnv
    from gym_guidance_collision_avoidance_single.envs.config import Config
    peak, src = measured_peaks()
    out = {"metric": METRIC, "unit": UNIT, "intruders": 0, "bytes_per_env_step": algorithmic_bytes_per_env_step(0, continuous=False)}
    for B in (ENVS_PER_GPU, 4 * 1024 * 1024):
        env = BatchedAircraftEnv("SingleAircraftEnv", B, Config, n_intruders=0, mode="fast", draws="philox", device=device, seed=8)
        env.reset()
        acts = [torch.randint(0, 9, (B,), device="cuda", dtype=torch.int32) for _ in range(GRAPH_STEPS)]
        ms = graph_step_ms(lambda i: env.step(acts[i]), GRAPH_STEPS)
        k = env.kernels_per_step
        env.close()
        gbs = B * out["bytes_per_env_step"] / (ms * 1e-3) / 1e9
        out["envs_%d" % B] = {"value": B / (ms * 1e-3), "ms_per_step": ms, "kernels_per_step": k, "hbm_gbs": gbs,
                              "hbm_frac": gbs / peak, "note": "L2 resident" if B == ENVS_PER_GPU else "HBM bound"}
    return out


def bench_faithful(device):
    """The headline workload in FAITHFUL mode: the reference's mixed f32 / f64 arithmetic with f64-capable intruder
    positions (16 B each, both planes) and f64 observations (2 624 B per env) - what the 1e-9 parity contract is
    stated on.  Algorithmic bytes per env-step: 16 + 8 + 16 + 32 per intruder + the fixed part of the fast path."""
    import torch
    from gca_b200.batched import BatchedAircraftEnv
    from gym_guidance_collision_avoidance_single.envs.config import Config
    B, N = ENVS_PER_GPU, N_INTRUDERS
    env = BatchedAircraftEnv(VARIANT, B, Config, n_intruders=N, mode="faithful", draws="philox", device=device, seed=9)
    env.reset()
    acts = [torch.rand((B, 2), device="cuda", dtype=torch.float64) * 2 - 1 for _ in range(GRAPH_STEPS)]
    ms = graph_step_ms(lambda i: env.step(acts[i]), GRAPH_STEPS)
    env.close()
    peak, src = measured_peaks()
    bytes_per = (16 + 8 + 16 + 32) * N + algorithmic_bytes_per_env_step(0) + 32
    gbs = B * bytes_per / (ms * 1e-3) / 1e9
    return {"metric": METRIC, "value": B / (ms * 1e-3), "unit": UNIT, "envs": B, "intruders": N, "ms_per_step": ms,
            "dtype": "f64 observations, f32/f64 positions", "bytes_per_env_step": bytes_per, "hbm_gbs": gbs,
            "hbm_frac": gbs / peak}


def bench_stack(device):
    """BASELINE.json config #5: SingleAircraftStackEnv, 4-frame stacked image observation (device rasteriser)."""
    import torch
    from gca_b200.stack import ImageBatch
    from gym_guidance_collision_avoidance_single.envs.config import Config
    B, N, k = ENVS_PER_GPU, N_INTRUDERS, 4
    env = ImageBatch(B, Config, n_intruders=N, frame_stack=k, device=device, seed=3)
    env.reset()
    acts = [torch.randint(0, 9, (B,), device="cuda", dtype=torch.int32) for _ in range(4)]
    for i in range(3):
        env.step(acts[i % 4])
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    start.record()
    for i in range(reps):
        env.step(acts[i % 4])
    stop.record()
    torch.cuda.synchronize()
    ms = start.elapsed_time(stop) / reps
    peak, _ = measured_peaks()
    frame_bytes = env.H * env.W
    out = {"metric": METRIC, "value": B / (ms * 1e-3), "unit": UNIT, "envs": B, "intruders": N, "frame_stack": k,
           "ms_per_step": ms, "kernels_per_step": 2,
           "frame_bytes_per_env_step": frame_bytes,
           "hbm_frac_frames_only": (B * frame_bytes / (ms * 1e-3) / 1e9) / peak,
           "note": "step kernels + rasteriser; bound by the rasteriser's per-sample blending (FP32 issue, "
                   "profiles/r1_raster_ncu_full.txt), not by HBM"}
    env.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path (--impl ours)")
    if args.impl == "reference":
        main_reference(args)
    else:
        main_gpu(args)


if __name__ == "__main__":
    main()
