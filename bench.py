"""Benchmark of the on-policy hot path: env-steps/sec over full cycles (rollout -> GAE -> PPO update).

    python bench.py --gpus N --steps K --warmup W            # this repo's engine, N GPUs of one node
    python bench.py --impl reference --steps K --warmup W    # the reference's own AgentPPO on the host cores (oracle/_ref)
    python bench.py --steps K --warmup W --dump-outputs DIR  # + one step's outputs from the seeded start, as DIR/<name>.npy

Workload (BASELINE.json configs[1], SURVEY.md section 8(d)): AgentPPO on Pendulum-v1, 65 536 envs PER GPU
(env-sharded, weak scaling), horizon 128, 2x64 GELU MLP actor + critic, Config defaults batch_size=128,
repeat_times=8 -> 8 minibatch updates per cycle.  One "step" = explore_env(env, 128) + update_net(buffer).
Prints ONE JSON line on rank 0.  See DESIGN.md "Measurement" for how each field is produced.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

NUM_ENVS = 65536
HORIZON = 128
NET_DIMS = [64, 64]
BATCH_SIZE = 128
REPEAT_TIMES = 8.0
METRIC = "env-steps/sec (rollout+GAE+update) at 65 536 envs"
UNIT = "env-steps/s"
FLOP_PER_ENV_STEP = 17408          # actor fwd 8704 + critic fwd 8704 (SURVEY 8(d))
HBM_BYTES_PER_ENV_STEP = 30        # 26 B trajectory + 4 B value written by the fused rollout kernel
NCU_DRAM_BYTES_PER_LAUNCH = 198.11e6  # measured once with ncu (2.22 MB read + 195.89 MB written), profiles/r02_v2_rollout_ts_metrics.txt
DUMP_ENVS = 4096                   # env columns --dump-outputs keeps of the rollout buffer: 17 MB in all at horizon 128
BUFFER_NAMES = ("states", "actions", "logprobs", "rewards", "undones", "unmasks")


def workload_config(n_gpus, num_envs=None):
    num_envs = NUM_ENVS if num_envs is None else num_envs
    return {"workload": "AgentPPO Pendulum-v1, 65 536 envs per GPU, horizon 128, 2x64 GELU MLP (BASELINE configs[1])"
            if num_envs == NUM_ENVS else f"AgentPPO Pendulum-v1, {num_envs} envs per GPU ({num_envs * n_gpus} in total: strong "
            "scaling of BASELINE configs[1]), horizon 128, 2x64 GELU MLP",
            "num_envs_per_gpu": num_envs, "num_envs_total": num_envs * n_gpus, "horizon_len": HORIZON,
            "net_dims": NET_DIMS, "batch_size": BATCH_SIZE, "repeat_times": REPEAT_TIMES,
            "update_times": int(HORIZON * REPEAT_TIMES / BATCH_SIZE), "parallelism": f"env-shard x{n_gpus}",
            "l2": "each step writes a fresh 252 MB trajectory (> 126 MB L2); no explicit flush needed",
            "rng": "Philox4x32-10 on device (policy noise, env resets, minibatch indices)"}


def measured_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], tflops=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    source="MEASURED_PEAKS.json (hbm copy; cuBLAS bf16 sustained)")
    return dict(hbm_gbs=6650.0, tflops=1590.0, source="fallback of B200_PROFILING.md")


class ClockSampler:
    """SM clock / power / throttle reasons sampled every 4 ms DURING the timed region, in-process through NVML
    (nvidia_ml_py).  An external `nvidia-smi -lms` loop was measured to stall kernel submission for up to 100 ms per
    query on these hosts, which is as long as the whole timed region; the NVML calls below take microseconds."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, gpu_index):
        import threading
        self.samples, self.stop_flag, self.thread, self.handle, self.nv = [], threading.Event(), None, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            uuid = None
            try:
                import torch
                uuid = "GPU-" + str(torch.cuda.get_device_properties(gpu_index).uuid)
            except Exception:
                pass
            self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid) if uuid else pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.nv = pynvml
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception as err:  # noqa: BLE001
            self.error = repr(err)

    def _loop(self):
        nv, h = self.nv, self.handle
        while not self.stop_flag.is_set():
            try:
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except AttributeError:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetPowerUsage(h) / 1000.0, reasons))
            except Exception:  # noqa: BLE001
                pass
            self.stop_flag.wait(0.004)

    def start(self):
        if self.nv is None:
            return
        import threading
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def mark(self):
        """Samples taken from now on belong to the timed region."""
        self.first_timed = len(self.samples)

    def stop(self):
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable: " + getattr(self, "error", "?")]}
        self.stop_flag.set()
        self.thread.join()
        timed = self.samples[getattr(self, "first_timed", 0):] or self.samples
        if not timed:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["no samples"]}
        reasons = sorted({name for _, _, r in timed for name, bit in self.REASONS if r & bit})
        return {"sm_mhz": statistics.median(c for c, _, _ in timed), "sm_max_mhz": self.sm_max, "reasons": reasons,
                "samples": len(timed), "power_w_max": max(p for _, p, _ in timed), "how": "NVML in-process, 4 ms period"}


def cpu_backend():
    """The CPU implementation that is timed as the reference arm / cpu_baseline: the UNMODIFIED reference's own AgentPPO
    from oracle/_ref (placed by oracle/make_ref.py; travels with the snapshot) -> kind "reference"; only if that copy is
    absent, the PyTorch-CPU port of its op sequence (oracle/cpu_port.py) -> kind "port"."""
    from oracle import ref_runner
    if ref_runner.available():
        return "reference", ref_runner.time_ref_cycles, "oracle/_ref elegantrl.agents.AgentPPO (unmodified reference, gpu_id=-1)"
    from oracle.cpu_port import time_cpu_cycles
    return "port", time_cpu_cycles, "oracle/cpu_port.py (oracle/_ref absent)"


def calibrate_threads(time_fn, num_envs=NUM_ENVS, cache=os.path.join("/tmp", "b200rl_cpu_threads.json")):
    """torch's default of one intra-op thread per logical CPU is several times SLOWER than 8-32 threads on these tiny
    ops, so the baseline uses the best count -- chosen on FULL-SIZE cycles (the same workload that is then timed), best
    of 3 per candidate after one warm-up.  The choice is cached on the box (/tmp) for an hour: the driver runs the reference
    arm and the engine arm back to back, and both legs must time the CPU implementation with the SAME thread count (the
    host is shared and noisy: two independent calibrations picked 8 and 32 threads in one round-2 run)."""
    try:
        c = json.load(open(cache))
        if time.time() - c["when"] < 3600 and c["num_envs"] == num_envs and c["ncpu"] == (os.cpu_count() or 8):
            return int(c["threads"]), {int(k): v for k, v in c["scores"].items()}
    except Exception:  # noqa: BLE001
        pass
    ncpu = os.cpu_count() or 8
    candidates = [t for t in (8, 16, 32) if t <= ncpu] or [max(1, ncpu)]
    scores = {}
    for t in candidates:
        r = time_fn(num_envs, HORIZON, NET_DIMS, warmup=1, cycles=3, threads=t, batch_size=BATCH_SIZE, repeat_times=REPEAT_TIMES)
        best_cycle = min(e + u for e, u in zip(r["explore_s"], r["update_s"]))
        scores[t] = num_envs * HORIZON / best_cycle
    best = max(scores, key=scores.get)
    try:
        json.dump({"when": time.time(), "num_envs": num_envs, "ncpu": ncpu, "threads": best, "scores": scores}, open(cache, "w"))
    except Exception:  # noqa: BLE001
        pass
    return best, scores


def dump_outputs(out_dir, buffer, losses, agent):
    """Write what one cycle handed its caller as float32 ``out_dir/<name>.npy``, so that two builds run with the same arguments
    can be compared output for output: the six buffer tensors as the caller holds them after ``update_net_device`` (which
    rewrites rewards / undones in place, as the reference does) and ``last_state``, on a fixed, seeded sample of env columns;
    the three losses; the actor and critic parameters after the update."""
    import numpy as np
    import torch as th
    os.makedirs(out_dir, exist_ok=True)
    n = buffer[0].shape[1]
    cols = np.sort(np.random.default_rng(0).choice(n, min(n, DUMP_ENVS), replace=False))
    idx = th.from_numpy(cols).to(buffer[0].device)
    arrays = {name: t.index_select(1, idx) for name, t in zip(BUFFER_NAMES, buffer)}
    arrays["last_state"] = agent.last_state.index_select(0, idx)
    arrays["losses"] = losses
    for prefix, module in (("act", agent.act), ("cri", agent.cri)):
        arrays.update({f"{prefix}.{k}": v for k, v in module.state_dict().items()})
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def run_reference(args):
    """The reference's own CPU implementation of the path (see cpu_backend) on the host cores, same config / metric;
    rank 0 only.  Each step is a full cycle at 65 536 envs unless K + W such cycles would not fit in ~3 minutes; then
    every step is the same cycle on a power-of-two subset of the envs (said in cpu_baseline.sample)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch as th
    kind, time_fn, what = cpu_backend()
    threads, scores = calibrate_threads(time_fn)
    budget_s, num_envs = 180.0, NUM_ENVS
    est_full = NUM_ENVS * HORIZON / scores[threads]          # seconds per full cycle, from the calibration run
    while num_envs > 4096 and (args.warmup + args.steps) * est_full * num_envs / NUM_ENVS > budget_s:
        num_envs //= 2
    r = time_fn(num_envs, HORIZON, NET_DIMS, warmup=args.warmup, cycles=args.steps, threads=threads,
                batch_size=BATCH_SIZE, repeat_times=REPEAT_TIMES)
    total = sum(r["explore_s"]) + sum(r["update_s"])
    value = num_envs * HORIZON * args.steps / total
    sample = (f"{what}: {args.steps} cycles of {num_envs} envs x {HORIZON} steps + update after {args.warmup} warm-up; {threads} torch "
              f"threads of {os.cpu_count()} logical CPUs, chosen on full-size cycles (best of 3 per candidate: "
              f"{({t: round(v / 1e6, 2) for t, v in scores.items()})} M env-steps/s)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample,
                             "sample_envs": num_envs},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_engine(args):
    import torch as th
    import torch.distributed as dist
    from elegantrl_b200 import Config, _lib
    from elegantrl_b200.agents import AgentPPO
    from elegantrl_b200.envs import PendulumVecEnv

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch N>1 with torch.distributed.run)"
    th.cuda.set_device(local_rank)
    dev = th.device(f"cuda:{local_rank}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    # default: BASELINE configs[1] per GPU (weak scaling).  --total-envs T: T / world envs per GPU (strong scaling study)
    n_envs = NUM_ENVS if args.total_envs is None else args.total_envs // world
    strong = args.total_envs is not None

    env_args = {'env_name': 'Pendulum-v1', 'num_envs': n_envs, 'max_step': 200, 'state_dim': 3, 'action_dim': 1,
                'if_discrete': False}
    cfg = Config(AgentPPO, PendulumVecEnv, env_args)
    cfg.net_dims, cfg.batch_size, cfg.repeat_times, cfg.random_seed = NET_DIMS, BATCH_SIZE, REPEAT_TIMES, 0

    def make_agent_env():
        """Agent and env from fixed seeds: the same inputs on every run with the same arguments."""
        th.manual_seed(0)  # identical initial parameters on every rank
        agent = AgentPPO(NET_DIMS, 3, 1, gpu_id=local_rank, args=cfg)
        if world > 1:
            agent.enable_data_parallel()
            agent.sharded_mode = args.sharded_mode
        env = PendulumVecEnv(num_envs=n_envs, gpu_id=local_rank, max_step=200, seed=rank)
        agent.last_state = env.reset()[0]
        # stagger episode phases like a long-running job (otherwise every env truncates at the same step)
        env.cur_step[:] = th.randint(0, 200, (n_envs,), device=dev, dtype=th.int32)
        return agent, env

    agent, env = make_agent_env()

    def barrier():
        if world > 1:
            dist.barrier()
        th.cuda.synchronize()

    def cycle_device():
        buffer = agent.explore_env(env, HORIZON)
        return agent.update_net_device(list(buffer))

    # pinned host mirrors for the end-to-end arm: the env state block [3, N] in, last_state + env state + 3 scalars out
    host_in = th.empty((3, n_envs), dtype=th.float32).pin_memory()
    host_last_state = th.empty((n_envs, 3), dtype=th.float32).pin_memory()
    host_in.copy_(env.engine_state_block())

    copy_stream = th.cuda.Stream(device=dev)   # the D2H copies ride beside GAE + update instead of in front of them

    def cycle_e2e():
        block = env.engine_state_block()
        block.copy_(host_in, non_blocking=True)              # H2D: the step's inputs from pinned host memory
        buffer = agent.explore_env(env, HORIZON)             # public API
        copy_stream.wait_stream(th.cuda.current_stream())    # ... after the rollout
        with th.cuda.stream(copy_stream):
            host_last_state.copy_(agent.last_state, non_blocking=True)   # D2H: final state of the rollout
            host_in.copy_(block, non_blocking=True)          # D2H: env state for the host-side loop
        result = agent.update_net(list(buffer))              # public API: returns 3 Python floats (D2H + sync)
        copy_stream.synchronize()                            # the host owns host_in / host_last_state from here on
        return result

    for _ in range(max(args.warmup, 3)):
        cycle_device()
    barrier()

    # ---- timed region 1: `value` -- inputs resident in HBM, no host round trips inside
    def timed_region(steps, sampler=None):
        """K back-to-back cycles, no host synchronisation inside; CUDA events around the region and each rollout."""
        ev0, ev1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
        roll_events, out = [], None
        barrier()
        if sampler is not None:
            sampler.mark()
        ev0.record()
        for _ in range(steps):
            a, b = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
            a.record()
            buffer = agent.explore_env(env, HORIZON)
            b.record()
            roll_events.append((a, b))
            out = agent.update_net_device(list(buffer))
        ev1.record()
        barrier()
        return ev0, ev1, roll_events, out

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # Rehearsal of the timed region, same code path and tensor lifetimes: without it the caching allocator meets a new
    # live-set in the first un-synchronised iterations and calls cudaMalloc (a multi-ms, device-synchronising stall).
    timed_region(args.steps)
    launches0 = lib.b200rl_launch_count()
    ev0, ev1, roll_events, out = timed_region(args.steps, sampler)
    elapsed_ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    launches = lib.b200rl_launch_count() - launches0
    rollout_list = [a.elapsed_time(b) for a, b in roll_events]
    rollout_ms = statistics.median(rollout_list)  # median: robust against a straggler launch
    assert th.isfinite(out).all(), "non-finite losses"
    t = th.tensor([elapsed_ms], dtype=th.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())

    # ---- timed region 2: `e2e` -- public API with host buffers, H2D / D2H inside
    for _ in range(2):
        cycle_e2e()
    barrier()
    ev0.record()
    for _ in range(args.steps):
        cycle_e2e()
    ev1.record()
    barrier()
    t = th.tensor([ev0.elapsed_time(ev1)], dtype=th.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())

    if args.dump_outputs:
        # The update's floating-point sums are not bit-reproducible and Pendulum amplifies the last bits over a few cycles, so
        # the state after the timed steps differs from run to run.  The step that is written out is one step of the timed
        # path from the seeded initial state instead: identical inputs on every run, comparable outputs across builds.
        dump_agent, dump_env = make_agent_env()
        buffer = dump_agent.explore_env(dump_env, HORIZON)
        losses = dump_agent.update_net_device(list(buffer))
        barrier()
        if rank == 0:
            dump_outputs(args.dump_outputs, buffer, losses, dump_agent)

    env_steps = n_envs * HORIZON * args.steps * world
    value = env_steps / (elapsed_ms * 1e-3)
    peaks = measured_peaks()
    per_launch_env_steps = n_envs * HORIZON
    flops = FLOP_PER_ENV_STEP * per_launch_env_steps + 8704 * n_envs  # + V(last_state)
    achieved_tflops = flops / (rollout_ms * 1e-3) / 1e12
    hbm_gbs = HBM_BYTES_PER_ENV_STEP * per_launch_env_steps / (rollout_ms * 1e-3) / 1e9
    roofline = {"kernel": "rollout_pendulum_ts_kernel (fused env + actor + critic + trajectory stores; both hidden layers on tcgen05, layer-2 A operand in tensor memory)", "bound": "tensor",
                "achieved": achieved_tflops, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": achieved_tflops / peaks["tflops"],
                "traffic": NCU_DRAM_BYTES_PER_LAUNCH if n_envs == 65536 else None, "traffic_unit": "bytes per launch: dram__bytes_read.sum + dram__bytes_write.sum of "
                "one `ncu --set full` capture (profiles/r02_v2_rollout_ts_metrics.txt); algorithmic 251.9e6 written, the tail "
                "of the trajectory is still in L2 when the kernel ends", "peak_source": peaks["source"], "avg_launch_ms": rollout_ms,
                "launch_ms_min_max": [min(rollout_list), max(rollout_list)],
                "share_of_step": rollout_ms / (elapsed_ms / args.steps),
                "pipe": "algorithmic MLP FLOPs (17 408 per env-step, fp32-equivalent) over the measured bf16 tensor peak; the kernel itself is bound by the CUDA-core side (256 GELUs per env-step), see DESIGN.md",
                "hbm": {"achieved": hbm_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": hbm_gbs / peaks["hbm_gbs"],
                        "bytes_per_env_step": HBM_BYTES_PER_ENV_STEP}}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(world, n_envs),
            # how the env shards exchange what the update needs (outside `config`: both arms describe the same workload)
            "exchange": (getattr(agent, "sharded_mode", None) if world > 1 else None), "clocks": clocks,
            "e2e": {"value": env_steps / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": 3 * n_envs * 4, "d2h_bytes_per_step": 3 * 4 + n_envs * 3 * 4 + 3 * n_envs * 4,
                    "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": int(launches), "roofline": roofline}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle.cpu_port import time_cpu_cycles
        kind, time_fn, what = cpu_backend()
        threads, scores = calibrate_threads(time_fn)
        cb = time_fn(n_envs, HORIZON, NET_DIMS, warmup=1, cycles=args.cpu_cycles, threads=threads,
                     batch_size=BATCH_SIZE, repeat_times=REPEAT_TIMES)
        line["cpu_baseline"] = {"value": cb["env_steps_per_sec"], "unit": UNIT, "cores": cb["threads"], "kind": kind,
                                "sample": f"{what}: {cb['cycles']} full cycles (65 536 envs x 128 steps + update) after 1 warm-up; "
                                          f"{cb['threads']} torch threads of {os.cpu_count()} logical CPUs, chosen on full-size cycles "
                                          f"(best of 3 per candidate: {({t: round(v / 1e6, 2) for t, v in scores.items()})} M env-steps/s); "
                                          f"explore {statistics.mean(cb['explore_s']):.3f}s + update {statistics.mean(cb['update_s']):.3f}s per cycle"}
        # the same pinned op sequence as EAGER PyTorch on this very GPU (SURVEY 8(d) "stronger baseline"): what a user of the
        # reference gets with gpu_id=0 -- ~45 launches per env step, ~250 per minibatch.  Informational; ~2 s.
        gb = time_cpu_cycles(n_envs, HORIZON, NET_DIMS, warmup=2, cycles=5, threads=threads, device=f"cuda:{local_rank}",
                             batch_size=BATCH_SIZE, repeat_times=REPEAT_TIMES)
        line["cpu_baseline"]["eager_pytorch_same_gpu"] = {
            "value": gb["env_steps_per_sec"], "unit": UNIT,
            "sample": f"5 full cycles after 2 warm-ups; explore {1e3 * statistics.mean(gb['explore_s']):.1f} ms + update "
                      f"{1e3 * statistics.mean(gb['update_s']):.1f} ms per cycle"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-cycles", type=int, default=4, help="CPU-baseline sample size (full cycles)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--total-envs", type=int, default=None, help="strong-scaling study: this many envs in total, split over the GPUs")
    ap.add_argument("--sharded-mode", default="auto", choices=["auto", "peer", "peer_allreduce", "gather", "allreduce"],
                    help="N > 1: how the env shards' gradients meet (auto = in-kernel peer-memory exchange when available)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, run one more step of the timed path from the seeded initial state and write what "
                         "it computed (buffer sample, losses, parameters) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_engine(args)


if __name__ == "__main__":
    main()
