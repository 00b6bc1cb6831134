#!/usr/bin/env python
"""bench.py -- env-steps/sec of the MetaGym hot path on N B200s of one node (BASELINE.json metric by default).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload quadrotor|maze3d|mixed] [--impl reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W [--workload ...]

Workloads (one process per GPU, envs sharded by global index, no data-path collective):
  quadrotor (default; BASELINE.json configs[2], the config the metric is quoted on): Quadrotor velocity_control, 65 536
            envs per GPU, dt = 0.005 = 5 Euler substeps of 1 ms (the reference's only integrator; SURVEY.md fact 2),
            nt = 1000, 64 velocity tasks (seeds 0..63), U(0.1, 15) random actions, auto-reset on.  One "step" = one
            env.step() of every env of the batch = ONE launch of the state-update kernel through the C ABI
            (mgb_quad_step).
  maze3d    (configs[3]): MetaMazeDiscrete3D SURVIVAL, 15x15 mazes, 128x128 uint8 frames, 1024 envs per GPU (8192 over
            8 GPUs), 64 reference-sampled tasks; one step = one mgb_maze_step of every env.  Extras: the many-task
            regime (one task per env: the pose cache is over budget and the direct raycaster runs) and the amortised
            set_task cost.
  mixed     (configs[4]): 16 384 quadrotor hovering_control + 16 384 MetaMaze2D ESCAPE envs per GPU, fused T = 32 step
            rollouts with device-drawn actions, every chunk exchanged so that each rank holds all ranks' trajectories
            (kernel-side NVLink peer stores; NCCL arena all-gather reported beside it).  One step = one env-step of
            every env (a chunk is 32 steps).

Timing (every workload): the timed region is exactly K steps.  quadrotor / maze3d: the K-step block is captured in
CUDA graphs of at most 256 launches (any K: no eager launches inside the timed region) after one untimed lead-in
step that keeps the timed steps in steady state, replayed ceil(W / K) times as warm-up and once timed; mixed: max(2, ceil(W / 32)) warm-up chunks, then K / 32 timed chunks (K must be a
multiple of 32).  `ms_per_step` = timed time / K.  CUDA events on the launching stream, barrier + synchronize on both
sides, max over ranks.  How many steps run before and inside the timed region depends on the arguments only, so
with the same arguments every run computes the same outputs.

--dump-outputs DIR: after the timed steps, rank 0 writes what its timed path computed in its last step, the arrays a
caller of env.step() (mixed: of the fused rollouts, last step of the no-exchange chunk loop) receives, as
DIR/<name>.npy in float32 (float64 where the engine returns float64).  Above 64 MB in all, a fixed seeded sample of
envs is written instead, with the sampled env indices in DIR/<name>_env_index.npy.

  value     device-resident inputs/outputs.  quadrotor: actions are read from and observations written to rollout buffers
            [32, n, .] (obs 160 MB > 126 MB L2: never L2-hot; the 6 MB recurrent state stays in L2 between steps).
  roofline  algorithmic bytes (SURVEY.md 8d) x envs / average launch duration, against MEASURED_PEAKS.json.
  e2e       the same step through the host-buffer C-ABI entry point with PINNED HOST buffers: H2D of the actions, kernel,
            D2H of obs/reward/done inside the timed region (wall clock, synchronous call).
  cpu_baseline / --impl reference: the numpy port of the reference loop (oracle/quadrotor_np.py, bit-identical to the
            reference on the golden vectors; maze workloads: the C restatement oracle/maze_oracle.c), one env per usable
            host core.  The reference is pure Python and does not exist on the GPU box; oracle/_ref has nothing to
            compile.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the benchmark writes nothing into the tree it runs from (the CPU arm's spawned workers inherit the variable)
sys.dont_write_bytecode = True
os.environ["PYTHONDONTWRITEBYTECODE"] = "1"

N_ENVS_PER_GPU = 65536
DT, NT, N_TASKS = 0.005, 1000, 64
TASK = "velocity_control"
FLOPS_PER_STEP = 350 * 5 + 60   # dt 0.005 = 5 substeps
BYTES_PER_STEP = 281          # SURVEY.md 8d: read state 88 + ct 4 + action 16; write state 88 + ct 4 + obs 76 + rew 4 + done 1
SLOTS = 32                    # slots of the rollout buffers the step launches cycle through
MIN_TIMED_MS = 50.0
MAZE3D_BYTES = 128 * 128 * 3 + 1630      # SURVEY.md 8d: uint8 frame + per-env maze state
MAZE2D_BYTES = 160
QUAD_HOVER_ROLLOUT_BYTES = 85            # SURVEY.md 8d fused T-step rollout: action 16 + obs 64 + rew 4 + done 1
MIXED_T = 32                             # steps per fused rollout chunk of the mixed workload
DUMP_MAX_BYTES = 64 * 10 ** 6

WORKLOADS = {
    "quadrotor": {
        "metric": "env-steps/sec (quadrotor 6-DoF, 65k envs)",
        "workload": "quadrotor velocity_control, %d envs/GPU, dt=0.005 (5 Euler substeps of 1 ms), nt=1000, "
                    "64 velocity tasks, U(0.1,15) actions, auto-reset" % N_ENVS_PER_GPU,
        "envs_per_gpu": N_ENVS_PER_GPU, "dtype": "f32"},
    "maze3d": {
        "metric": "env-steps/sec (MetaMaze3D 15x15, 128x128 obs, 1024 envs/GPU)",
        "workload": "MetaMazeDiscrete3D SURVIVAL, 15x15 maze, 128x128x3 uint8 obs, 1024 envs/GPU, 64 tasks, "
                    "uniform {0..3} actions, max_steps=200, auto-reset",
        "envs_per_gpu": 1024, "dtype": "f64+u8"},
    "mixed": {
        "metric": "env-steps/sec (mixed quadrotor + MetaMaze2D rollout with trajectory all-gather, 32k envs/GPU)",
        "workload": "16384 quadrotor hovering_control (dt=0.01) + 16384 MetaMaze2D ESCAPE (view_grid=1, 15x15) envs/GPU, "
                    "fused T=32 rollouts, device-drawn actions, every chunk gathered on every rank",
        "envs_per_gpu": 32768, "dtype": "f32"},
}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons of one GPU, sampled every 100 ms while the load runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.rows.append((time.time(), parts))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if (t0 is None or t >= t0) and (t1 is None or t <= t1 + 0.15)]
        if not rows:
            rows = [r for (_, r) in self.rows]
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}

    def close(self):
        """Make sure no nvidia-smi outlives the benchmark, also when a leg raised before stop()."""
        if self.proc is not None and self.proc.poll() is None:
            self.proc.terminate()
            self.proc.wait()


def dump_outputs(path, arrays):
    """arrays: name -> host array with the env axis first.  Writes <path>/<name>.npy in float32 (float64 stays
    float64).  Above DUMP_MAX_BYTES in all, the same fraction of envs of every array is kept, drawn with a fixed seed,
    and the kept env indices go to <name>_env_index.npy."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    out = {k: v.astype(np.float64 if v.dtype == np.float64 else np.float32) for k, v in arrays.items()}
    total = sum(v.nbytes for v in out.values())
    if total > DUMP_MAX_BYTES:
        frac = DUMP_MAX_BYTES / (total + 8.0 * sum(len(v) for v in out.values()))
        for k in list(out):
            n = len(out[k])
            idx = np.sort(np.random.RandomState(0).choice(n, max(1, int(n * frac)), replace=False))
            out[k] = np.ascontiguousarray(out[k][idx])
            out[k + "_env_index"] = idx.astype(np.float64)
    for k, v in out.items():
        np.save(os.path.join(path, k + ".npy"), v)


# ---------------------------------------------------------------------------------------------------------------
# CPU arm
# ---------------------------------------------------------------------------------------------------------------
def usable_cores():
    """Host threads this process may really use: the scheduler affinity, capped by the cgroup CPU quota."""
    aff = len(os.sched_getaffinity(0))
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:          # cgroup v2: "<quota|max> <period>"
            q, p = f.read().split()[:2]
            if q != "max":
                quota = float(q) / float(p)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                p = float(f.read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    n = aff if quota is None else max(1, min(aff, int(math.floor(quota + 1e-9))))
    return n, {"affinity": aff, "cgroup_quota": quota, "os_cpu_count": os.cpu_count()}


_CPU_CACHE = {}


def cpu_arm(workload, seconds, warm=1.0):
    """The reference's CPU implementation of the workload's step on every usable host core.  One run per process
    (cached), so the `cpu_baseline` of the GPU line and a --impl reference line on the same box cannot disagree."""
    key = (workload, seconds)
    if key in _CPU_CACHE:
        return _CPU_CACHE[key]
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[v] = "1"                                  # inherited by the spawned workers: no BLAS thread pools
    cores, how = usable_cores()
    if workload == "quadrotor":
        from oracle.quadrotor_np import measure_throughput_detail
        res = measure_throughput_detail(task=TASK, dt=DT, nt=NT, seconds=seconds, processes=cores, warmup_seconds=warm)
        sample = ("numpy single-env port of the reference loop (oracle/quadrotor_np.py; bit-identical to the reference "
                  "on the golden vectors), one env per process, %d processes x %.0f s, velocity_control dt=0.005, "
                  "U(0.1,15) actions" % (cores, seconds))
    elif workload == "maze3d":
        from oracle.maze_oracle import measure_throughput_detail
        res = measure_throughput_detail(kind="3D", seconds=seconds, processes=cores, warmup_seconds=warm)
        sample = ("C restatement of maze_view + grid rules (oracle/maze_oracle.c, bit-exact vs reference episodes; the "
                  "reference runs the same loops under numba), 15x15 SURVIVAL 128x128, one env per process, %d "
                  "processes x %.0f s" % (cores, seconds))
    else:
        from oracle.maze_oracle import measure_throughput_detail as maze_detail
        from oracle.quadrotor_np import measure_throughput_detail as quad_detail
        half = max(1, cores // 2)
        rq = quad_detail(task="hovering_control", dt=0.01, nt=NT, seconds=seconds, processes=half, warmup_seconds=warm)
        rm = maze_detail(kind="2D", seconds=seconds, processes=max(1, cores - half), warmup_seconds=warm)
        # the mixed batch advances one quadrotor and one maze env together: harmonic combination of the two rates
        # measured with half the cores each
        both = 2.0 / (1.0 / rq["value"] + 1.0 / rm["value"])
        res = {"value": both, "rates": rq["rates"] + rm["rates"], "wall_s": max(rq["wall_s"], rm["wall_s"]),
               "parts": {"quadrotor_hovering": rq["value"], "maze2d": rm["value"]}}
        sample = ("numpy quadrotor port (hovering_control dt=0.01) on %d processes + C maze2d oracle on %d, %.0f s; "
                  "combined as env-steps/s of a half/half batch" % (half, cores - half, seconds))
    rates = sorted(res["rates"])
    out = {"value": res["value"], "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample,
           "per_process_steps_per_s": {"min": rates[0], "median": statistics.median(rates), "max": rates[-1]},
           "wall_s": res["wall_s"], "cores_how": how}
    if "parts" in res:
        out["parts"] = res["parts"]
    _CPU_CACHE[key] = out
    return out


def base_config(workload, world):
    w = WORKLOADS[workload]
    return {"workload": w["workload"], "envs_per_gpu": w["envs_per_gpu"],
            "global_envs": w["envs_per_gpu"] * world, "parallelism": "dp%d" % world}


def run_reference(args, rank, world):
    """--impl reference: the CPU implementation on the host cores (rank 0 only).  The K "steps" are K equal slices of ONE
    bounded run; ms_per_step is the real wall time of a slice."""
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    timed_s = float(args.cpu_seconds) if args.cpu_seconds else 30.0
    t0 = time.time()
    cpu = cpu_arm(args.workload, timed_s, warm=2.0)
    slice_ms = cpu["wall_s"] * 1e3 / max(1, args.steps)
    cfg = base_config(args.workload, args.gpus)
    info = {"launch": "CPU arm: %d processes, one env each; the K steps are K equal slices (%.1f ms each) of one bounded "
                      "%.0f s run after 2 s warm-up" % (cpu["cores"], slice_ms, timed_s)}
    line = {
        "impl": "reference", "metric": w["metric"], "value": cpu["value"], "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": slice_ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": w["dtype"], "data": "synthetic", "config": cfg,
        "run_info": info, "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s_total": None,
    }
    line["wall_s_total"] = time.time() - t0
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# graph-replayed K-step blocks
# ---------------------------------------------------------------------------------------------------------------
class GraphedBlock(object):
    """Exactly K steps of `enqueue(t)` captured in CUDA graphs so that ANY K is replayed from graphs (no eager launch in
    a timed region).  The K steps are cut into pieces of 256 (t = 0..255) and a remainder (t = 0..K % 256 - 1); the
    first piece is a graph that begins with one untimed lead-in step, the last one a graph that ends by recording `end`,
    and the pieces between are replays of one 256-step graph.  `start` is recorded on a branch that waits for the
    lead-in step alone, so the kernels keep their programmatic dependent-launch chain and `elapsed_ms()` of a replay is
    the K steps in steady state: no graph launch, no first-kernel launch latency.  A replay runs `steps` = K + 1 steps;
    `last_t` is the t of the block's last step."""
    UNIT = 256

    def __init__(self, torch, dev, enqueue, K, warm_steps):
        self.torch, self.K = torch, K
        self.start = torch.cuda.Event(enable_timing=True, external=True)     # recorded by a node of the graph
        self.end = torch.cuda.Event(enable_timing=True, external=True)
        self.stream = torch.cuda.Stream(device=dev)
        self.branch = torch.cuda.Stream(device=dev)
        self.steps = K + 1
        self.stream.wait_stream(torch.cuda.current_stream(dev))     # side stream: ordered after the caller's pending work
        with torch.cuda.stream(self.stream):
            for t in range(max(3, warm_steps)):
                enqueue(t)
            self.stream.synchronize()
            sizes = [self.UNIT] * (K // self.UNIT) + ([K % self.UNIT] if K % self.UNIT else [])
            self.plan = [(self._capture(enqueue, sizes[0], start=True, end=len(sizes) == 1), sizes[0], 1)]
            if len(sizes) > 2:                                       # (graph, steps, replays)
                self.plan.append((self._capture(enqueue, self.UNIT), self.UNIT, len(sizes) - 2))
            if len(sizes) > 1:
                self.plan.append((self._capture(enqueue, sizes[-1], end=True), sizes[-1], 1))
        self.last_t = sizes[-1] - 1
        torch.cuda.synchronize(dev)

    def _capture(self, enqueue, steps, start=False, end=False):
        g = self.torch.cuda.CUDAGraph()
        with self.torch.cuda.graph(g, stream=self.stream):
            if start:
                enqueue(0)                                  # lead-in step
                self.branch.wait_stream(self.stream)
                self.start.record(self.branch)
            for t in range(steps):
                enqueue(t)
            if start:
                self.stream.wait_stream(self.branch)        # join the branch before the capture ends
            if end:
                self.end.record()
        return g

    def elapsed_ms(self):
        """Device time of the last completed replay of the block."""
        return self.start.elapsed_time(self.end)

    def replay(self, times=1):
        """`times` x K steps, on the current stream."""
        for _ in range(times):
            for g, _, reps in self.plan:
                for _ in range(reps):
                    g.replay()

    def describe(self, what):
        sizes = " + ".join("%d x %d" % (reps, steps) for _, steps, reps in self.plan)
        return "K=%d %s launches after one lead-in in CUDA graphs (replays x launches: %s), replayed once timed" % (
            self.K, what, sizes)


class Ctx(object):
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: metagym_b200 has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.peak, self.peak_src = measured_peak_gbs()
        self.outputs = None
        self.e0 = torch.cuda.Event(enable_timing=True)
        self.e1 = torch.cuda.Event(enable_timing=True)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t)

    def timed(self, fn):
        """Device time of fn() in ms: barrier + synchronize on both sides, CUDA events, max over ranks."""
        self.barrier()
        self.e0.record()
        fn()
        self.e1.record()
        self.barrier()
        return self.max_over_ranks(self.e0.elapsed_time(self.e1))

    def time_block(self, block, W):
        """ceil(W / K) warm-up replays of the block (every graph of it has run before the timed one), then one timed
        replay: exactly K steps, timed by the events the block's graphs record.  -> dict"""
        K = block.K
        warm = max(1, -(-W // K))
        self.barrier()
        t_wall0 = time.time()
        block.replay(warm + 1)
        self.barrier()
        t_wall1 = time.time()
        ms = self.max_over_ranks(block.elapsed_ms())
        return {"ms": ms, "timed_steps": K, "repeats": 1, "ms_per_step": ms / K, "warmup_steps": warm * block.steps + 1,
                "t_wall0": t_wall0, "t_wall1": t_wall1, "K": K}

    def snapshot(self, arrays):
        """Host copies of the timed path's last-step outputs, kept for --dump-outputs (rank 0)."""
        if self.args.dump_outputs and self.rank == 0:
            self.outputs = {k: v.detach().cpu().numpy() for k, v in arrays.items()}

    def close(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def hold_load_for_clocks(ctx, sampler, block, t_wall0):
    """Keep the same load running long enough for nvidia-smi (100 ms period) to see it; -> clocks dict (rank 0)."""
    t_load0 = time.time()
    while time.time() - t_load0 < 1.5:
        block.replay(8)
        ctx.torch.cuda.synchronize(ctx.dev)
    return sampler.stop(t_wall0, time.time()) if ctx.rank == 0 else None


# ---------------------------------------------------------------------------------------------------------------
# workload: quadrotor (the BASELINE metric)
# ---------------------------------------------------------------------------------------------------------------
def run_quadrotor(ctx, sampler):
    torch, dev, args, world, rank = ctx.torch, ctx.dev, ctx.args, ctx.world, ctx.rank
    from metagym_b200 import BatchedQuadrotor
    from metagym_b200.rollout import RolloutArena
    n = args.envs or N_ENVS_PER_GPU
    K, W = args.steps, args.warmup
    env = BatchedQuadrotor(task=TASK, dt=DT, nt=NT, seed=list(range(N_TASKS)), num_envs=n, device=ctx.local_rank,
                           squeeze=False, auto_reset=True, rng_seed=0, env_index_base=rank * n)
    env.reset()
    D = env.obs_dim
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    G = SLOTS
    acts = torch.rand((G, n, 4), device=dev, generator=gen) * 14.9 + 0.1
    obs = torch.empty((G, n, D), dtype=torch.float32, device=dev)
    rew = torch.empty((G, n), dtype=torch.float32, device=dev)
    done = torch.empty((G, n), dtype=torch.uint8, device=dev)

    def enqueue(t):
        env.step(acts[t % G], out=(obs[t % G], rew[t % G], done[t % G]))

    block = GraphedBlock(torch, dev, enqueue, K, min(W, G))
    tm = ctx.time_block(block, W)
    s = block.last_t % G
    ctx.snapshot({"obs": obs[s], "reward": rew[s], "done": done[s]})
    us_per_launch = tm["ms_per_step"] * 1e3
    value = n * world / (tm["ms_per_step"] * 1e-3)
    achieved = n * BYTES_PER_STEP / (us_per_launch * 1e-6) / 1e9
    clocks = hold_load_for_clocks(ctx, sampler, block, tm["t_wall0"])
    finite = bool(torch.isfinite(obs).all()) and bool(torch.isfinite(rew).all())
    kernel_name = env.step_kernel_name() if hasattr(env, "step_kernel_name") else "quad_step"

    extras, e2e = {}, None
    if not args.no_extras:
        # ---- end to end through the host-buffer C-ABI entry point, pinned buffers, copies inside the timed region
        h_act = torch.empty((n, 4), dtype=torch.float32).pin_memory()
        h_act.copy_(acts[0].cpu())
        h_obs = torch.empty((n, D), dtype=torch.float32).pin_memory()
        h_rew = torch.empty((n,), dtype=torch.float32).pin_memory()
        h_done = torch.empty((n,), dtype=torch.uint8).pin_memory()
        for _ in range(5):
            env.step_host_buffers(h_act, h_obs, h_rew, h_done)
        Ke = max(20, min(K, 200))
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(Ke):
            env.step_host_buffers(h_act, h_obs, h_rew, h_done)
        torch.cuda.synchronize(dev)
        dt_e = ctx.max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": n * world * Ke / dt_e, "unit": "env-steps/s", "h2d_bytes_per_step": n * 16,
               "d2h_bytes_per_step": n * (D * 4 + 4 + 1), "steps": Ke, "timer": "host wall clock around the synchronous "
               "mgb_quad_step_host calls (pinned host buffers), max over ranks",
               "result_checksum": float(h_rew.double().sum())}
        # bytes over PCIe per second per GPU, both directions (the kernel reads actions from / writes results to pinned host memory)
        e2e["pcie_gbs_per_gpu"] = (e2e["h2d_bytes_per_step"] + e2e["d2h_bytes_per_step"]) * Ke / dt_e * 1e-9
        assert bool(torch.isfinite(h_obs).all())

        # ---- fused T-step rollout kernel (state in registers), same buffers
        out = {"obs": obs, "rew": rew, "done": done, "act": None}
        for _ in range(3):
            env.rollout(G, actions=acts, out=out)
        reps = max(8, int(MIN_TIMED_MS / 1.5))
        msf = ctx.timed(lambda: [env.rollout(G, actions=acts, out=out) for _ in range(reps)])
        extras["fused_rollout"] = {"value": n * world * reps * G / (msf * 1e-3), "unit": "env-steps/s",
                                   "T": G, "launches": reps, "us_per_env_step_launch_equiv": msf * 1e3 / (reps * G),
                                   "note": "mgb_quad_rollout: T steps per launch, state held in registers"}
        if world > 1:
            # ---- the one collective of the path: every rank's rollout chunk on every rank, as ONE NCCL all-gather of
            # the arena the rollout kernel wrote (RolloutArena)
            fields = {"obs": ((G, n, D), torch.float32), "act": ((G, n, 4), torch.float32),
                      "rew": ((G, n), torch.float32), "done": ((G, n), torch.uint8)}
            ar = RolloutArena(fields, dev)
            env.rollout(G, actions=None, act_seed=3, out=ar.views)
            for _ in range(3):
                ar.all_gather()
            msg = ctx.timed(lambda: [ar.all_gather() for _ in range(5)]) / 5
            nbytes = ar.payload_bytes()
            extras["rollout_allgather"] = {"ms": msg, "bytes_per_rank": nbytes, "how": "one all_gather_into_tensor of "
                                           "the rollout arena (RolloutArena)",
                                           "busbw_GBps": nbytes * (world - 1) / (msg * 1e-3) / 1e9}
            del ar
            extras["fused_rollout_peer_gather"] = quad_peer_gather(ctx, env, n, D, G)
        env.close()
        del env, obs, rew, done, acts
        torch.cuda.empty_cache()
        # ---- streaming variant: 4 194 304 envs, the state (403 MB) no longer fits L2 and streams from HBM
        if rank == 0:
            ns = 4194304
            big = BatchedQuadrotor(task=TASK, dt=DT, nt=NT, seed=list(range(N_TASKS)), num_envs=ns,
                                   device=ctx.local_rank, squeeze=False, auto_reset=True)
            big.reset()
            a2 = torch.rand((2, ns, 4), device=dev, generator=gen) * 14.9 + 0.1
            for t in range(4):
                big.step(a2[t % 2])
            torch.cuda.synchronize(dev)
            iters = 200
            ctx.e0.record()
            for t in range(iters):
                big.step(a2[t % 2])
            ctx.e1.record()
            torch.cuda.synchronize(dev)
            us = ctx.e0.elapsed_time(ctx.e1) * 1e3 / iters
            extras["streaming"] = {"envs": ns, "us_per_launch": us, "launches": iters, "value": ns / us * 1e6,
                                   "unit": "env-steps/s", "achieved_GBps": ns * BYTES_PER_STEP / us * 1e-3,
                                   "frac": ns * BYTES_PER_STEP / us * 1e-3 / ctx.peak}
            big.close()
            del big, a2
            torch.cuda.empty_cache()
            # ---- the other half of the hot path at its per-GPU shapes (full runs: --workload maze3d / mixed)
            try:
                extras["metamaze"] = maze_step_rates(ctx)
            except Exception as ex:      # the contract metric above must not depend on this leg
                extras["metamaze"] = {"error": repr(ex)[:200]}
    else:
        env.close()

    if rank != 0:
        return None
    cfg = base_config("quadrotor", world)
    info = {}
    info.update({
        "launch": block.describe("mgb_quad_step") + " (programmatic dependent launch between consecutive steps)",
        "timed_region": "K = %d steps in %.2f ms after %d warm-up steps, CUDA events, max over ranks" % (
            tm["timed_steps"], tm["ms"], tm["warmup_steps"]),
        "l2": "rollout buffers obs [32,n,19] f32 = 160 MB > 126 MB L2 (inputs/outputs never L2-hot); "
              "the 6 MB recurrent state is L2-resident by nature of the workload; see extras.streaming "
              "for the 4M-env run whose state streams from HBM",
        "integrator": "semi-implicit Euler substeps (the reference's integrator); BASELINE's 'RK4' has "
                      "no reference counterpart (SURVEY.md fact 2)"})
    traffic, traffic_src = ncu_traffic("quad_step")
    line = {
        "metric": WORKLOADS["quadrotor"]["metric"], "value": value, "unit": "env-steps/s", "n_gpus": world,
        "steps": K, "warmup": W, "ms_per_step": tm["ms_per_step"], "timed_steps": tm["timed_steps"],
        "repeats": tm["repeats"], "timed_ms": tm["ms"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg, "run_info": info,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": ctx.peak, "unit": "GB/s",
                     "frac": achieved / ctx.peak, "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": ctx.peak_src, "kernel": kernel_name,
                     "bytes_per_env_step": BYTES_PER_STEP, "envs_per_launch": n, "us_per_launch": us_per_launch,
                     # secondary figure SURVEY.md 8d asks for: ~350 flop per substep + ~60 per step (hand count)
                     "flops_per_env_step": FLOPS_PER_STEP,
                     "achieved_fp32_tflops": n / (us_per_launch * 1e-6) * FLOPS_PER_STEP / 1e12,
                     "fp32_peak_tflops_nominal": 148 * 128 * 2 * 1.965e9 / 1e12},
        "gpu_launches": tm["timed_steps"], "clocks": clocks, "finite_outputs": finite,
    }
    if e2e is not None:
        line["e2e"] = e2e
    line.update(extras)
    return line


def ncu_traffic(kernel):
    """dram bytes of ONE launch of the dominant kernel from the committed `ncu --set full` capture (profiles/)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)[kernel]
        return t["bytes"], t["source"]
    except Exception:
        return None, "no committed capture"


def quad_peer_gather(ctx, env, n, D, G):
    """The same exchange done by the rollout kernel itself: every output is also stored into the other ranks' receive
    arenas over NVLink (PeerArena); the only cross-rank call left is a one-element rendezvous."""
    torch, dev, world, rank = ctx.torch, ctx.dev, ctx.world, ctx.rank
    arenas = []
    try:
        from metagym_b200.rollout import PeerArena
        fields = {"obs": ((G, n, D), torch.float32), "act": ((G, n, 4), torch.float32),
                  "rew": ((G, n), torch.float32), "done": ((G, n), torch.uint8)}
        arenas = [PeerArena(fields, dev) for _ in range(2)]
        tick = [0]
        views = [None]

        def chunk_peer():
            ar = arenas[tick[0] & 1]
            tick[0] += 1
            ar.attach(env)
            env.rollout(G, actions=None, act_seed=3, out=ar.views)
            views[0] = ar.sync()

        for _ in range(3):
            chunk_peer()
        reps = 24
        msp = ctx.timed(lambda: [chunk_peer() for _ in range(reps)])
        own = bool(torch.equal(views[0]["obs"][rank], arenas[(tick[0] - 1) & 1]["obs"]))
        return {"value": n * world * reps * G / (msp * 1e-3), "unit": "env-steps/s", "T": G,
                "chunk_bytes_per_rank": arenas[0].payload_bytes(),
                "ingress_GBps_per_gpu": arenas[0].payload_bytes() * (world - 1) * reps / (msp * 1e-3) / 1e9,
                "gathered_shape": list(views[0]["obs"].shape), "own_slot_ok": own,
                "note": "quad_rollout_kernel<.,1>: outputs stored into every rank's arena by the kernel (NVLink "
                        "peer stores), rendezvous = 1-element all-reduce; no NCCL on the data"}
    except Exception as ex:            # reported, never fatal for the headline numbers
        return {"error": repr(ex)[:300]}
    finally:
        env.set_mirrors([])
        for ar in arenas:
            try:
                ar.close()
            except Exception:
                pass


# ---------------------------------------------------------------------------------------------------------------
# workload: maze3d (BASELINE configs[3])
# ---------------------------------------------------------------------------------------------------------------
def reference_tasks(k):
    """k tasks from the reference-stream sampler, seeds 0..k-1 (random.seed(s); np.random.seed(s); SURVEY.md 8d)."""
    from metagym_b200 import MazeTaskSampler
    return [MazeTaskSampler(n=15, allow_loops=True, crowd_ratio=0.35, seed=s) for s in range(k)]


def fast_tasks(k, seed=0):
    import numpy as np
    from metagym_b200 import MazeTaskSampler
    rs = np.random.RandomState(seed)
    return [MazeTaskSampler(n=15, allow_loops=True, crowd_ratio=0.35, rng=rs) for _ in range(k)]


def maze_step_rates(ctx):
    """Short single-GPU legs of the quadrotor line: maze3d (config 4 per-GPU shape) and maze2d step rates."""
    torch, dev = ctx.torch, ctx.dev
    from metagym_b200 import BatchedMetaMaze2D, BatchedMetaMazeDiscrete3D
    tasks = fast_tasks(64)
    out = {}
    for name, make, n, nbytes in (
            ("maze3d_15x15_128x128_u8_1024envs",
             lambda: BatchedMetaMazeDiscrete3D(resolution=(128, 128), max_steps=200, task_type="SURVIVAL", num_envs=1024,
                                               device=dev.index, squeeze=False, auto_reset=True, obs_dtype="uint8"),
             1024, MAZE3D_BYTES),
            ("maze2d_15x15_g1_16384envs",
             lambda: BatchedMetaMaze2D(max_steps=200, task_type="ESCAPE", view_grid=1, num_envs=16384, device=dev.index,
                                       squeeze=False, auto_reset=True), 16384, MAZE2D_BYTES)):
        env = make()
        env.set_task(tasks)
        env.reset()
        acts = torch.randint(0, 4, (16, n), device=dev, dtype=torch.int32)
        block = GraphedBlock(torch, dev, lambda t: env.step(acts[t % 16]), 64, 8)
        tm = _time_block_local(ctx, block)
        us = tm["ms_per_step"] * 1e3
        out[name] = {"value": n / us * 1e6, "unit": "env-steps/s", "us_per_step": us, "timed_steps": tm["timed_steps"],
                     "algorithmic_bytes_per_env_step": nbytes, "frac_of_measured_hbm": n * nbytes / us * 1e-3 / ctx.peak,
                     "parity": "bit-exact vs reference golden episodes (tests/test_maze_gpu.py)"}
        del block
        env.close()
    return out


def _time_block_local(ctx, block):
    """Rank-local timing (no collectives): used for legs only rank 0 runs while the other ranks wait at a barrier."""
    torch = ctx.torch
    block.replay(1)
    torch.cuda.synchronize(ctx.dev)
    ctx.e0.record(); block.replay(1); ctx.e1.record()
    torch.cuda.synchronize(ctx.dev)
    R = max(1, int(math.ceil(1.2 * MIN_TIMED_MS / max(ctx.e0.elapsed_time(ctx.e1), 1e-3))))
    ctx.e0.record(); block.replay(R); ctx.e1.record()
    torch.cuda.synchronize(ctx.dev)
    ms = ctx.e0.elapsed_time(ctx.e1)
    steps = R * block.steps
    return {"ms": ms, "timed_steps": steps, "repeats": R, "ms_per_step": ms / steps, "t_wall0": 0, "t_wall1": 0,
            "K": block.K}


def run_maze3d(ctx, sampler):
    torch, dev, args, world, rank = ctx.torch, ctx.dev, ctx.args, ctx.world, ctx.rank
    import numpy as np
    from metagym_b200 import BatchedMetaMazeDiscrete3D
    n = args.envs or 1024
    K, W = args.steps, args.warmup
    tasks = reference_tasks(64)
    env = BatchedMetaMazeDiscrete3D(resolution=(128, 128), max_steps=200, task_type="SURVIVAL", num_envs=n,
                                    device=ctx.local_rank, squeeze=False, auto_reset=True, obs_dtype="uint8",
                                    env_index_base=rank * n)
    t0 = time.perf_counter()
    env.set_task(tasks)
    env.reset()
    g = torch.Generator(device=dev).manual_seed(77 + rank)
    acts = torch.randint(0, 4, (SLOTS, n), device=dev, dtype=torch.int32, generator=g)
    env.step(acts[0])
    torch.cuda.synchronize(dev)
    set_task_s = time.perf_counter() - t0
    last = {}

    def enqueue(t):
        last["out"] = env.step(acts[t % SLOTS])     # the env's own output buffers, the same ones every step

    block = GraphedBlock(torch, dev, enqueue, K, min(W, SLOTS))
    tm = ctx.time_block(block, W)
    ctx.snapshot(dict(zip(("obs", "reward", "done"), last["out"][:3])))
    launch = block.describe("mgb_maze_step")
    us = tm["ms_per_step"] * 1e3
    value = n * world / (tm["ms_per_step"] * 1e-3)
    achieved = n * MAZE3D_BYTES / (us * 1e-6) / 1e9
    clocks = hold_load_for_clocks(ctx, sampler, block, tm["t_wall0"])
    launches_per_step = env.launches_per_step() if hasattr(env, "launches_per_step") else 2
    extras, e2e = {}, None
    if not args.no_extras:
        # ---- e2e: actions from pinned host memory, the frames read back to pinned host memory, every step
        h_act = torch.randint(0, 4, (n,), dtype=torch.int32).pin_memory()
        h_obs = torch.empty((n, 128, 128, 3), dtype=torch.uint8).pin_memory()
        h_rew = torch.empty((n,), dtype=torch.float64).pin_memory()
        d_act = torch.empty((n,), dtype=torch.int32, device=dev)

        def host_step():
            d_act.copy_(h_act, non_blocking=True)
            o, r, d, _ = env.step(d_act)
            h_obs.copy_(o, non_blocking=True)
            h_rew.copy_(r, non_blocking=True)
            torch.cuda.synchronize(dev)

        for _ in range(3):
            host_step()
        Ke = max(20, min(K, 100))
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(Ke):
            host_step()
        dt_e = ctx.max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": n * world * Ke / dt_e, "unit": "env-steps/s", "h2d_bytes_per_step": n * 4,
               "d2h_bytes_per_step": n * (128 * 128 * 3 + 8), "steps": Ke,
               "timer": "host wall clock, pinned buffers, copies + synchronize inside", "result_checksum": float(h_rew.sum())}
        e2e["pcie_gbs_per_gpu"] = (e2e["h2d_bytes_per_step"] + e2e["d2h_bytes_per_step"]) * Ke / dt_e * 1e-9
        del block
        env.close()
        if rank == 0:
            # ---- many-task regime: one task per env (1024 tasks x ~50 MB of cached poses > the cache budget): the direct
            # raycaster renders every frame; and the cost of set_task amortised over an episode of 200 steps
            many = fast_tasks(n, seed=5)
            env2 = BatchedMetaMazeDiscrete3D(resolution=(128, 128), max_steps=200, task_type="SURVIVAL", num_envs=n,
                                             device=ctx.local_rank, squeeze=False, auto_reset=True, obs_dtype="uint8",
                                             cache=False)
            t0 = time.perf_counter()
            env2.set_task(many, env2task=np.arange(n))
            torch.cuda.synchronize(dev)
            st_many = time.perf_counter() - t0
            env2.reset()
            b2 = GraphedBlock(torch, dev, lambda t: env2.step(acts[t % SLOTS]), 32, 4)
            t2 = _time_block_local(ctx, b2)
            us2 = t2["ms_per_step"] * 1e3
            extras["many_tasks"] = {"tasks": n, "us_per_step": us2, "value": n / us2 * 1e6, "unit": "env-steps/s",
                                    "renderer": "direct float64 raycaster (maze3d_kernel<false>), one task per env",
                                    "set_task_s": st_many,
                                    "frac_of_measured_hbm": n * MAZE3D_BYTES / us2 * 1e-3 / ctx.peak}
            del b2
            # ---- per-episode task resampling (SURVEY.md 8f row 3): an env that finishes an episode gets a fresh task.
            # (a) host samplers alone, (b) mgb_maze_update_tasks alone (stream-ordered, no device sync), (c) the loop:
            # step, read `done`, re-task the finished envs with freshly sampled tasks
            import random as _random
            from metagym_b200 import MazeTaskSampler
            rs = np.random.RandomState(11)
            t0 = time.perf_counter()
            fresh = [MazeTaskSampler(n=15, allow_loops=True, crowd_ratio=0.35, rng=rs) for _ in range(256)]
            rate_fast = 256 / (time.perf_counter() - t0)
            t0 = time.perf_counter()
            _ = [MazeTaskSampler(n=15, allow_loops=True, crowd_ratio=0.35, seed=1000 + k) for k in range(32)]
            rate_ref = 32 / (time.perf_counter() - t0)
            ids = np.arange(256)
            env2.update_tasks(ids, fresh)
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            for r in range(8):
                env2.update_tasks((ids + 64 * r) % n, fresh)
            host_s = time.perf_counter() - t0
            torch.cuda.synchronize(dev)
            rate_upd = 8 * 256 / (time.perf_counter() - t0)
            steps_loop, retasked = 300, 0
            pool, pi = fresh, 0
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            for t in range(steps_loop):
                _, _, d, _ = env2.step(acts[t % SLOTS])
                fin = torch.nonzero(d).flatten().cpu().numpy()          # the learner reads `done` anyway
                if fin.size:
                    new = [pool[(pi + k) % len(pool)] for k in range(fin.size)]
                    pi += fin.size
                    env2.update_tasks(fin, new)
                    retasked += int(fin.size)
            torch.cuda.synchronize(dev)
            dt_loop = time.perf_counter() - t0
            # (d) the same loop with the DEVICE sampler: no host round trip at all (mgb_maze_resample_tasks(done))
            for t in range(20):
                _, _, d, _ = env2.step(acts[t % SLOTS])
                env2.resample_tasks(d, seed=5, allow_loops=True, crowd_ratio=0.35)
            torch.cuda.synchronize(dev)
            ndone = torch.zeros((), dtype=torch.int64, device=dev)
            ctx.e0.record()
            for t in range(steps_loop):
                _, _, d, _ = env2.step(acts[t % SLOTS])
                env2.resample_tasks(d, seed=5, allow_loops=True, crowd_ratio=0.35)
                ndone += d.sum()
            ctx.e1.record()
            torch.cuda.synchronize(dev)
            ms_dev = ctx.e0.elapsed_time(ctx.e1)
            # sampler alone: every env resampled at once
            ctx.e0.record()
            for _ in range(10):
                env2.resample_tasks(None, seed=6, allow_loops=True, crowd_ratio=0.35)
            ctx.e1.record()
            torch.cuda.synchronize(dev)
            rate_dev = 10 * n / (ctx.e0.elapsed_time(ctx.e1) * 1e-3)
            extras["task_churn"] = {
                "device_sampler_tasks_per_s": rate_dev,
                "device_loop": {"steps": steps_loop, "envs": n, "retasked": int(ndone), "value": n * steps_loop / (ms_dev * 1e-3),
                                "unit": "env-steps/s", "tasks_per_s": int(ndone) / (ms_dev * 1e-3),
                                "note": "step + mgb_maze_resample_tasks(done): finished envs get a maze drawn on the device "
                                        "(one kernel, stream-ordered, no host synchronisation)"},
                "host_sampler_tasks_per_s": {"reference_streams": rate_ref, "rng_sampler": rate_fast},
                "update_tasks_per_s": rate_upd, "update_tasks_host_s_per_call_of_256": host_s / 8,
                "loop": {"steps": steps_loop, "envs": n, "retasked": retasked, "value": n * steps_loop / dt_loop,
                         "unit": "env-steps/s", "tasks_per_s": retasked / dt_loop,
                         "note": "step + done read-back + mgb_maze_update_tasks of the finished envs (tasks drawn from a "
                                 "pre-sampled pool; sampling cost is the host_sampler line)"}}
            env2.close()
    else:
        env.close()
    if rank != 0:
        return None
    cfg = base_config("maze3d", world)
    info = {}
    info.update({"launch": launch,
                "timed_region": "K = %d steps in %.2f ms after %d warm-up steps" % (tm["timed_steps"], tm["ms"],
                                                                                   tm["warmup_steps"]),
                "renderer": "pose cache (64 tasks): cached static layers + per-step integer compose; see many_tasks for "
                            "the direct raycaster", "set_task_plus_first_step_s": set_task_s,
                "l2": "frames 50 MB/step written to one buffer (L2 126 MB): outputs may stay L2-resident; the cache of "
                      "baked frames (~3 GB) does not"})
    line = {"metric": WORKLOADS["maze3d"]["metric"], "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": tm["ms_per_step"], "timed_steps": tm["timed_steps"], "repeats": tm["repeats"],
            "timed_ms": tm["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64+u8",
            "data": "synthetic", "config": cfg, "run_info": info,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": ctx.peak, "unit": "GB/s",
                         "frac": achieved / ctx.peak, "traffic": ncu_traffic("maze3d_step")[0],
                         "traffic_source": ncu_traffic("maze3d_step")[1], "peak_source": ctx.peak_src,
                         "kernel": "maze3d_step_kernel", "bytes_per_env_step": MAZE3D_BYTES, "envs_per_launch": n,
                         "us_per_launch": us,
                         # the pose-cache design READS a finished 48 KB frame per env as well as writing one: what the kernel
                         # really moves, and the measured floor of just moving it (scripts/microbench/framecopy.cu: 16.4 us
                         # for 1024 frames with a TMA ring, LDG/STG.128 or cudaMemcpy alike = 6.1 TB/s read + write)
                         "moved_bytes_per_env_step": MAZE3D_BYTES + 128 * 128 * 3,
                         "frac_of_moved_bytes": n * (MAZE3D_BYTES + 128 * 128 * 3) / us * 1e-3 / ctx.peak,
                         "frame_move_floor_us_per_1024_envs": 16.4,
                         "floor_source": "profiles/r2_framecopy.txt"},
            "gpu_launches": tm["timed_steps"] * launches_per_step, "clocks": clocks}
    if e2e is not None:
        line["e2e"] = e2e
    line.update(extras)
    return line


# ---------------------------------------------------------------------------------------------------------------
# workload: mixed (BASELINE configs[4])
# ---------------------------------------------------------------------------------------------------------------
def run_mixed(ctx, sampler):
    torch, dev, args, world, rank = ctx.torch, ctx.dev, ctx.args, ctx.world, ctx.rank
    from metagym_b200 import BatchedMetaMaze2D, BatchedQuadrotor
    from metagym_b200.rollout import PeerArena, RolloutArena
    NQ = NM = (args.envs or 32768) // 2
    T = MIXED_T
    K, W = args.steps, args.warmup
    quad = BatchedQuadrotor(task="hovering_control", dt=0.01, nt=1000, num_envs=NQ, device=ctx.local_rank,
                            squeeze=False, auto_reset=True, env_index_base=rank * NQ)
    maze = BatchedMetaMaze2D(max_steps=200, task_type="ESCAPE", view_grid=1, num_envs=NM, device=ctx.local_rank,
                             squeeze=False, auto_reset=True, env_index_base=rank * NM)
    maze.set_task(reference_tasks(64))
    quad.reset()
    maze.reset()
    fields = {
        "q_obs": ((T, NQ, 16), torch.float32), "q_act": ((T, NQ, 4), torch.float32),
        "q_rew": ((T, NQ), torch.float32), "q_done": ((T, NQ), torch.uint8),
        "m_obs": ((T, NM, 3, 3), torch.float32), "m_act": ((T, NM), torch.int32),
        "m_rew": ((T, NM), torch.float64), "m_done": ((T, NM), torch.uint8),
    }

    def collect(v):
        quad.rollout(T, actions=None, act_seed=7, out={"obs": v["q_obs"], "rew": v["q_rew"], "done": v["q_done"],
                                                       "act": v["q_act"]})
        maze.rollout(T, actions=None, act_seed=9, out={"obs": v["m_obs"], "rew": v["m_rew"], "done": v["m_done"],
                                                       "act": v["m_act"]})

    plain = RolloutArena(fields, dev)
    payload = plain.payload_bytes()
    for _ in range(max(2, -(-W // T))):
        collect(plain.views)
    reps = K // T
    ms_none = ctx.timed(lambda: [collect(plain.views) for _ in range(reps)])
    ctx.snapshot({k: v[T - 1] for k, v in plain.views.items()})
    results = {"no_exchange": {"value": (NQ + NM) * world * T * reps / (ms_none * 1e-3), "ms_per_chunk": ms_none / reps}}
    how = "none (1 GPU: the chunk is already where the learner is)"
    ms_best, t_wall0 = ms_none, time.time()
    launches_per_chunk = 2
    if world > 1:
        # (a) NCCL: ONE all-gather of the arena per chunk, double-buffered (gather k overlaps rollout k+1)
        arenas = [RolloutArena(fields, dev), RolloutArena(fields, dev)]
        pend, tick = [None], [0]

        def pipelined():
            ar = arenas[tick[0] & 1]
            tick[0] += 1
            collect(ar.views)
            if pend[0] is not None:
                pend[0].wait()
            _, pend[0] = ar.all_gather(async_op=True)

        for _ in range(4):
            pipelined()
        ms_nccl = ctx.timed(lambda: [pipelined() for _ in range(reps)])
        if pend[0] is not None:
            pend[0].wait()
        ms_ag = ctx.timed(lambda: [arenas[0].all_gather() for _ in range(8)]) / 8
        results["nccl_arena_allgather_pipelined"] = {
            "value": (NQ + NM) * world * T * reps / (ms_nccl * 1e-3), "ms_per_chunk": ms_nccl / reps,
            "allgather_alone_ms": ms_ag, "busbw_GBps": arenas[0].nbytes * (world - 1) / (ms_ag * 1e-3) / 1e9}
        del arenas
        # (b) kernel-side: the rollout kernels store every output into all ranks' arenas (NVLink peer stores); four
        # arenas in rotation, asynchronous one-element rendezvous (ordering argument: scripts/bench_mixed.py)
        peers = [PeerArena(fields, dev) for _ in range(4)]
        works, ptick = [None] * 4, [0]

        def collect_peer():
            i = ptick[0] % 4
            ptick[0] += 1
            ar = peers[i]
            ar.attach(quad, maze)
            collect(ar.views)
            _, works[i] = ar.sync(async_op=True)
            j = (i - 1) % 4
            if works[j] is not None:
                works[j].wait()
                works[j] = None

        for _ in range(6):
            collect_peer()
        t_wall0 = time.time()
        ms_peer = ctx.timed(lambda: [collect_peer() for _ in range(reps)])
        for w_ in works:
            if w_ is not None:
                w_.wait()
        torch.cuda.synchronize(dev)
        # the peer-written arena must equal an NCCL all-gather of the same chunk, byte for byte
        chk_ar = peers[(ptick[0] - 1) % 4]
        check = torch.empty(world * chk_ar.nbytes, dtype=torch.uint8, device=dev)
        ctx.dist.all_gather_into_tensor(check, chk_ar.buf.contiguous())
        same = bool(torch.equal(check, chk_ar._recv))
        results["kernel_side_peer_stores"] = {
            "value": (NQ + NM) * world * T * reps / (ms_peer * 1e-3), "ms_per_chunk": ms_peer / reps,
            "ingress_GBps_per_gpu": payload * (world - 1) * reps / (ms_peer * 1e-3) / 1e9,
            "equals_nccl_allgather": same}
        quad.set_mirrors([])
        maze.set_mirrors([])
        for a_ in peers:
            a_.close()
        ms_best = ms_peer
        how = ("kernel-side all-gather: the fused rollout kernels store every output into all %d ranks' arenas over "
               "NVLink (cp.async.bulk + st to peer mappings), 1-element NCCL rendezvous per chunk" % world)

    # clocks while the reported variant's load runs
    t_l = time.time()
    while time.time() - t_l < 1.5:
        for _ in range(16):
            collect(plain.views)
        torch.cuda.synchronize(dev)
    clocks = sampler.stop(t_wall0, time.time()) if rank == 0 else None
    steps_timed = reps * T
    value = (NQ + NM) * world * steps_timed / (ms_best * 1e-3)
    ms_per_step = ms_best / steps_timed
    # e2e: chunk read back to pinned host memory every chunk (the learner on the host)
    e2e = None
    if not args.no_extras:
        host = torch.empty(plain.nbytes, dtype=torch.uint8).pin_memory()

        def chunk_to_host():
            collect(plain.views)
            host.copy_(plain.buf, non_blocking=True)
            torch.cuda.synchronize(dev)

        for _ in range(2):
            chunk_to_host()
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(8):
            chunk_to_host()
        dt_e = ctx.max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": (NQ + NM) * world * T * 8 / dt_e, "unit": "env-steps/s", "h2d_bytes_per_step": 0,
               "d2h_bytes_per_step": payload / T, "steps": 8 * T,
               "timer": "host wall clock; actions are drawn on the device (random-action rollout), the whole chunk "
                        "{obs, act, rew, done} is copied to pinned host memory every chunk"}
    quad.close()
    maze.close()
    if rank != 0:
        return None
    cfg = base_config("mixed", world)
    info = {}
    info.update({"launch": "per chunk: mgb_quad_rollout + mgb_maze_rollout (T=32 steps each, state in registers / smem)",
                "exchange": how, "chunk_bytes_per_rank": payload,
                "timed_region": "%d chunks = %d steps in %.1f ms" % (reps, steps_timed, ms_best),
                "l2": "chunk outputs 2 x %.0f MB cycle through 4 arenas (> L2 with the gathered copies at N>1)" % (payload / 1e6)})
    bytes_step = NQ * QUAD_HOVER_ROLLOUT_BYTES + NM * (4 + 36 + 8 + 1 + 4)
    achieved = bytes_step / (ms_per_step * 1e-3) / 1e9
    line = {"metric": WORKLOADS["mixed"]["metric"], "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_per_step, "timed_steps": steps_timed, "repeats": reps, "timed_ms": ms_best,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "run_info": info,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": ctx.peak, "unit": "GB/s",
                         "frac": achieved / ctx.peak, "traffic": None, "peak_source": ctx.peak_src,
                         "kernel": "quad_rollout_kernel + maze2d_rollout_kernel (FP32-issue bound, not HBM bound: "
                                   "SURVEY.md 8d)", "bytes_per_step_per_gpu": bytes_step},
            "exchange_variants": results, "gpu_launches": reps * launches_per_chunk, "clocks": clocks}
    if e2e is not None:
        line["e2e"] = e2e
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4096)
    ap.add_argument("--warmup", type=int, default=64)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="quadrotor", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (default: the workload's BASELINE shape)")
    ap.add_argument("--no-extras", action="store_true", help="skip streaming / fused / e2e / cpu legs")
    ap.add_argument("--cpu-seconds", type=float, default=0.0, help="length of the CPU arm (default 10 s; reference arm 30 s)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs to DIR/<name>.npy (float32 / float64, <= 64 MB in all)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert args.warmup >= 3, "W >= 3 warm-up steps are required"
    assert args.steps >= 1
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if args.workload == "mixed" and args.steps % MIXED_T:
        ap.error("--workload mixed times whole rollout chunks: --steps must be a multiple of %d" % MIXED_T)

    ctx = Ctx(args)
    sampler = ClockSampler(ctx.local_rank)
    if ctx.rank == 0:
        sampler.start()
    try:
        line = {"quadrotor": run_quadrotor, "maze3d": run_maze3d, "mixed": run_mixed}[args.workload](ctx, sampler)
    finally:
        sampler.close()
    if ctx.rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, ctx.outputs)
        if not args.no_extras:
            line["cpu_baseline"] = cpu_arm(args.workload, float(args.cpu_seconds) if args.cpu_seconds else 10.0)
        print(json.dumps(line), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
