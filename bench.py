#!/usr/bin/env python
"""Benchmark of the movement-primitive black-box rollout path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch: B = 65,536 episodes per GPU of
fancy_ProMP/HoleReacher-v0 (BASELINE.json configs[1]) = trajectory generation + velocity controller
+ reacher dynamics + collision tests + reward aggregation for up to 200 env steps per episode, on
synthetic random MP parameters (sigma * N(0,1), torch Philox) and random task contexts.

Prints ONE JSON line (see README / DESIGN.md "Measurement" for the keys):
  value            whole-job env-steps/s with inputs resident in HBM (device-timed, max over ranks)
  e2e              the same metric through the public API from pinned HOST buffers, per step reset + H2D of that step's
                   parameters + rollout + D2H of its returns / lengths / flags inside the timed region, four batches in flight
                   (fancy_gym_b200.EpisodePipeline: every batch with its own env state and compute stream, replayed as CUDA
                   graphs; copies and consecutive rollouts overlap); e2e_sync = reset() + step() with one batch at a time
                   (the host waits for each batch before the next H2D)
  roofline         fused rollout kernel: algorithmic ops (SURVEY.md §8d: 4356 per HoleReacher/ProMP env step)
                   / measured kernel time, against the FP32 FFMA peak measured in the same run (fg_ffma_probe)
  roofline_trajgen trajectory-only kernel (fg_trajgen): algorithmic bytes (8 B per (t, dof)) / time vs measured HBM GB/s
  cpu_baseline     the oracle port of the reference's CPU path on this box's host cores (rank 0, N=1, bounded sample):
                   one env per process like the reference; the numpy-vectorised port is reported as an extra
Multi-GPU (torchrun, one rank per GPU): the env batch is sharded, no data-path collective; per-step returns /
lengths / flags reach every rank inside the timed region — stored by the rollout kernel itself into peer-mapped gather buffers
over NVLink (FG_BENCH_EXCHANGE=nccl: an overlapped ncclAllGather instead) ("scaling": "weak").

--dump-outputs DIR writes what the last timed step of `value` returned (rank 0's envs) as DIR/<name>.npy: the arrays step()
hands its caller (obs, return, terminated, truncated, is_success, is_collided, end_effector, trajectory_length).  The inputs
are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ENV_ID = "fancy_ProMP/HoleReacher-v0"
B_PER_GPU = 65536
N_PARAMS = 25
SIGMA = 0.25
CPU_BATCH = 64                   # envs per oracle call in the CPU baseline (numpy-vectorised port)
OPS_PER_ENV_STEP = 4356          # SURVEY.md §8d, HoleReacher/ProMP (FMA = 2, each collision test once per step)
TRAJ_BYTES_PER_ENV = 2 * 200 * 5 * 4 + N_PARAMS * 4   # fg_trajgen: pos + vel out, params in
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, limit_bytes=DUMP_LIMIT_BYTES):
    """Writes `arrays` (numpy, one row per env) as out_dir/<name>.npy: float32 and boolean arrays as float32, all others as
    float64 (exact for the int32 lengths).  If they would take more than `limit_bytes`, the same seeded sample of env rows
    is written from every array, and the chosen rows go to env_index.npy."""
    import numpy as np
    out = {k: np.asarray(v, dtype=np.float32 if v.dtype in (np.float32, np.bool_) else np.float64) for k, v in arrays.items()}
    n = len(next(iter(out.values())))
    row_bytes = sum(v[0].nbytes for v in out.values())
    budget = limit_bytes - 128 * (len(out) + 1)          # room for the .npy headers
    if n * row_bytes > budget:
        idx = np.sort(np.random.default_rng(0).choice(n, budget // (row_bytes + 8), replace=False))
        out = {k: v[idx] for k, v in out.items()}
        out["env_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def ncu_numbers():
    """dram bytes, executed warp instructions and pipe utilisations of the committed `ncu --set full` captures of the same
    kernels at the same sizes: profiles/ncu_numbers.json, written by tools/ncu_to_json.py from profiles/*_ncu_summary.txt (a CPU
    test keeps the two in step) — nothing ncu-derived is hard-coded here"""
    p = os.path.join(ROOT, "profiles", "ncu_numbers.json")
    if not os.path.exists(p):
        return {}
    with open(p) as f:
        return json.load(f)


# ------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference path, one worker process per host core
# ------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    seed0, n_batches, batch, sigma = args
    import numpy as np
    from oracle.blackbox import make_oracle
    orc = make_oracle(ENV_ID, mode="shipped")
    orc.env.compute_margins = False          # time the reference's work only: no oracle-side margin bookkeeping,
    orc.env.double_collision_eval = True     # and both collision tests twice per step as the reference does (Q3)
    steps = 0
    t0 = time.perf_counter()
    for e in range(n_batches):
        s = seed0 + e * batch
        orc.reset(seeds=range(s, s + batch))
        th = (sigma * np.random.default_rng(1234 + s).standard_normal((batch, N_PARAMS))).astype(np.float32)
        _, _, _, _, info = orc.step(th)
        steps += int(info["trajectory_length"].sum())
    return steps, n_batches * batch, time.perf_counter() - t0


class CpuReference:
    """The oracle port of the reference path on ALL host cores: one worker process per core (fork), each running whole
    episodes through oracle/blackbox.py (the BlackBoxWrapper.step loop, black_box_wrapper.py:150-217, on oracle/reacher.py).

    `batch=1` is the reference's own structure — one env per process, one Python-level env step at a time — and is what
    `value` reports (kind "port"); calibration in the build container, which has /root/reference: the reference's own
    BlackBoxWrapper + HoleReacherEnv files run 2.7k env-steps/s per core, this port 2.9k.  `batch=64` lets numpy vectorise over 64 envs per call: several times FASTER per env
    than anything the reference can do; it is reported separately as `vectorised_port_value` ("not the reference")."""

    def __init__(self, sigma=SIGMA):
        import multiprocessing as mp
        self.cores = os.cpu_count() or 1
        self.sigma = sigma
        self.pool = mp.get_context("fork").Pool(self.cores)
        self.pool.map(_cpu_worker, [(10_000_000 + 1000 * w, 1, 2, sigma) for w in range(self.cores)])      # warm-up / imports
        self._next_seed = 0

    def sample(self, n_batches, batch=1):
        """every worker runs `n_batches` oracle calls of `batch` envs -> dict(env_steps, episodes, wall_s)"""
        s0 = self._next_seed
        self._next_seed += self.cores * n_batches * batch
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_worker, [(s0 + w * n_batches * batch, n_batches, batch, self.sigma) for w in range(self.cores)])
        wall = time.perf_counter() - t0
        return dict(env_steps=sum(r[0] for r in res), episodes=sum(r[1] for r in res), wall_s=wall)

    def close(self):
        self.pool.close()
        self.pool.join()

    def baseline(self, scalar_episodes_per_worker=32, vector_batches_per_worker=4):
        """cpu_baseline object of the bench line: ~10-30 s of CPU work in total"""
        sc = self.sample(scalar_episodes_per_worker, batch=1)
        ve = self.sample(vector_batches_per_worker, batch=CPU_BATCH)
        return dict(value=sc["env_steps"] / sc["wall_s"], unit="env-steps/s", cores=self.cores, kind="port",
                    episodes_per_s=sc["episodes"] / sc["wall_s"], wall_s=sc["wall_s"], env_steps=sc["env_steps"],
                    episodes=sc["episodes"],
                    sample=f"{sc['episodes']} episodes ({sc['env_steps']} env steps) of {ENV_ID}, sigma={self.sigma}: {self.cores} worker "
                           f"processes x {scalar_episodes_per_worker} episodes, one env per process stepped one env step at a time through "
                           f"oracle/blackbox.py ('shipped' float32 MP, collision tests twice per step like the reference)",
                    vectorised_port_value=ve["env_steps"] / ve["wall_s"],
                    vectorised_port_note=f"NOT the reference: the same port with numpy vectorised over {CPU_BATCH} envs per call "
                                         f"({ve['episodes']} episodes in {ve['wall_s']:.2f} s)")


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock, power and throttle reasons of one GPU every ~20 ms through NVML (the same counters as the
    `nvidia-smi --query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.*` line of B200_PROFILING.md)."""
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
               "hw_power_brake_slowdown": 0x80}

    def __init__(self, device_index):
        self.idx = device_index
        self.sm, self.power, self.mask = [], [], 0
        self.sm_max = None
        self._stop = threading.Event()
        self._ready = threading.Event()      # set after the first sample: NVML init / imports must not land in a timed region
        self._th = None
        self.err = None

    def _loop(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES re-numbers devices: resolve through the UUID torch reports
            import torch
            uuid = str(torch.cuda.get_device_properties(self.idx).uuid)
            h = None
            for i in range(pynvml.nvmlDeviceGetCount()):
                hi = pynvml.nvmlDeviceGetHandleByIndex(i)
                u = pynvml.nvmlDeviceGetUUID(hi)
                u = u.decode() if isinstance(u, bytes) else u
                if uuid in u or u.replace("GPU-", "") == uuid:
                    h = hi
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            while not self._stop.is_set():
                self.sm.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                self.power.append(pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0)
                self.mask |= int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                self._ready.set()
                self._stop.wait(0.02)
        except Exception as e:      # noqa: BLE001
            self.err = repr(e)
        self._ready.set()

    def __enter__(self):
        self._th = threading.Thread(target=self._loop, daemon=True)
        self._th.start()
        self._ready.wait(timeout=10)
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._th.join(timeout=5)

    def summary(self):
        if not self.sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=[f"NVML unavailable: {self.err}"])
        busy = sorted(s for s, p in zip(self.sm, self.power))
        return dict(sm_mhz=busy[len(busy) // 2], sm_min_mhz=busy[0], sm_max_mhz=self.sm_max,
                    power_w_max=max(self.power), samples=len(self.sm),
                    reasons=sorted(k for k, bit in self.REASONS.items() if self.mask & bit))


# ------------------------------------------------------------------------------------------------
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def run_reference(args, rank, world, emit):
    """`--impl reference`: the reference's CPU path (oracle port: the reference is Python with uninstalled dependencies and
    /root/reference does not travel to the GPU box) on all host cores.  One "step" is a bounded sample of the workload:
    every worker process runs 2 episodes, one env at a time like the reference.  Rank 0 only."""
    if rank != 0:
        return
    cpu = CpuReference(args.sigma)
    per_worker = 2
    for _ in range(min(args.warmup, 2)):
        cpu.sample(1)
    tot_steps = tot_eps = busy = 0.0
    for _ in range(args.steps):
        r = cpu.sample(per_worker)
        tot_steps += r["env_steps"]; tot_eps += r["episodes"]; busy += r["wall_s"]
    value = tot_steps / max(busy, 1e-9)
    vec = cpu.sample(2, batch=CPU_BATCH)
    cpu.close()
    line = dict(metric="env-steps/sec (fancy_ProMP/HoleReacher-v0 MP black-box rollout)", value=value, unit="env-steps/s",
                n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * busy / max(args.steps, 1),
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic", impl="reference",
                config=dict(workload=f"{ENV_ID}, bounded CPU sample per step: {per_worker} episodes x {cpu.cores} worker processes "
                                     f"(one env per process), sigma={args.sigma}"),
                episodes_per_s=tot_eps / max(busy, 1e-9),
                cpu_baseline=dict(value=value, unit="env-steps/s", cores=cpu.cores, kind="port",
                                  sample=f"{args.steps} steps x {per_worker * cpu.cores} episodes; oracle port of the reference's loop, one env "
                                         f"per process stepped one env step at a time",
                                  vectorised_port_value=vec["env_steps"] / vec["wall_s"],
                                  vectorised_port_note=f"NOT the reference: the same port vectorised over {CPU_BATCH} envs per call"),
                e2e=dict(value=value, unit="env-steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=B_PER_GPU)
    ap.add_argument("--sigma", type=float, default=SIGMA)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries the ONE JSON line and nothing else: whatever libraries write to file descriptor 1 on the way (NCCL's
    # "NCCL version ..." banner at communicator set-up) goes to stderr; the descriptor is restored for the final print
    sys.stdout.flush()
    _stdout_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(_stdout_fd, 1)
        print(json.dumps(line), flush=True)

    if args.impl == "reference":
        run_reference(args, rank, world, emit)
        return

    import ctypes as C

    import numpy as np
    import torch
    import torch.distributed as dist

    import fancy_gym_b200 as fancy_gym
    from fancy_gym_b200 import _lib

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    bound_cpus = []
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # one process per GPU: run on the CPUs next to this GPU, so that the pinned parameter buffers allocated below (first
        # touch) and the per-step H2D copies of `e2e` stay on the GPU's side of the socket interconnect
        if os.environ.get("FG_BENCH_BIND", "1") == "1":
            from fancy_gym_b200.dist import bind_to_gpu_cpus
            bound_cpus = bind_to_gpu_cpus(local_rank)
        dist.init_process_group("nccl", device_id=dev)
    B = args.envs_per_gpu
    K, W = args.steps, args.warmup

    # multi-GPU: the exchange of step k has to finish before the rollout of step k + RING re-uses its result block.  RING = 2
    # (the wrapper's default) already hides the all-gather; deeper rings (4, 8: FG_BENCH_RESULT_RING) were measured at N = 4
    # and change nothing (0.3367 ms per step each), i.e. the ranks are not waiting for each other's exchange
    RING = int(os.environ.get("FG_BENCH_RESULT_RING", "2")) if world > 1 else 2
    # end to end: batches in flight.  One GPU: 2 (H2D 0.12 ms, rollout 0.27 ms).  Eight ranks share the host's PCIe / memory
    # bandwidth and the H2D of a batch takes about as long as its rollout (24 GB/s per GPU with all ranks copying,
    # tools/probe_h2d_numa.py): a third batch in flight keeps both busy (tools/probe_e2e_slots.py: 0.336 -> 0.306 ms at N = 8)
    # With the rollouts of consecutive batches overlapping (one compute stream per batch in flight) and every batch replayed as
    # two CUDA graphs, four batches in flight reach the device's two-launches-in-flight rate (tools/probe_e2e_slots.py, one
    # GPU: 2 / 3 / 4 slots 0.233 / 0.202 / 0.182 ms per step; eager submits are host bound at 0.22 ms)
    E2E_SLOTS = int(os.environ.get("FG_BENCH_E2E_SLOTS", "4"))
    E2E_GRAPHS = os.environ.get("FG_BENCH_E2E_GRAPHS", "1") == "1"
    RING = max(RING, E2E_SLOTS)
    env = fancy_gym.make(ENV_ID, num_envs=B, device=dev, context_sampler="device",
                         mp_config_override={"black_box_kwargs": {"result_sets": RING}})
    base = env.unwrapped
    # rotating input sets so that every timed step reads inputs that are cold in the 126 MB L2
    set_bytes = B * (N_PARAMS * 4 + 5 * 8 * 2 + 4 * 8 + 5)
    n_sets = max(2, int(np.ceil(2 * 126e6 / set_bytes)))
    gen = torch.Generator(device=dev).manual_seed(1000 + rank)
    from types import SimpleNamespace
    sets = []
    for s in range(n_sets):
        env.reset(seed=10_000 * (rank + 1) + s)
        # every set carries its own start state (joint angles, contexts, zeroed velocity / step counter / done flag); the
        # rollout runs with keep_state=1, i.e. reads it and leaves it untouched, so a timed step is the launch itself
        sets.append(dict(params=(args.sigma * torch.randn(B, N_PARAMS, generator=gen, device=dev)).contiguous(),
                         state=SimpleNamespace(q=base.q.clone(), v=torch.zeros_like(base.v), steps=torch.zeros_like(base.steps),
                                               done=torch.zeros_like(base.done), ctx=base.ctx.clone())))

    from fancy_gym_b200.dist import PeerResultExchange, all_gather_result_blocks
    gathered = [torch.zeros(world * env._result_block.numel(), dtype=torch.uint8, device=dev) for _ in range(RING)] if world > 1 else None
    in_flight = []
    n_gathers = [0]

    # Multi-GPU exchange.  Default: FUSED into the rollout — every env's result row is stored by the kernel itself into the
    # gather buffer of every rank over NVLink peer memory (fg_rollout_io.peer_bufs, torch symmetric memory), the ranks only
    # order a one-CTA barrier behind the launch on a side stream: no collective kernel shares the SMs with the rollout.
    # FG_BENCH_EXCHANGE=nccl selects the overlapped ncclAllGather of round 1 (also the fallback if peer memory cannot be mapped).
    exchange = {"mode": "none", "peer": None, "note": None}

    def make_exchange(e):
        if world == 1:
            return None
        ok, err, px = 1, None, None
        if os.environ.get("FG_BENCH_EXCHANGE", "peer") == "peer":
            try:
                px = PeerResultExchange(e, ring=4)
            except Exception as ex_:      # noqa: BLE001
                ok, err = 0, repr(ex_)
        else:
            ok = 0
        flag = torch.tensor([ok], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            if px is not None:
                px.detach(e)
            exchange["note"] = err
            return None
        return px

    exchange["peer"] = make_exchange(env)
    exchange["mode"] = "none" if world == 1 else ("peer-stores" if exchange["peer"] is not None else "nccl-allgather")

    def pre_launch():
        """peer stores: launch j overwrites the ring slot of launch j - ring; every rank has read it once the barrier of launch
        j - ring + 1 has passed"""
        px = exchange["peer"]
        if px is not None:
            while len(in_flight) > px.ring - 2:
                in_flight.pop(0).wait()

    def gather_results():
        """returns / lengths / flags of every rank to every rank.  peer-stores: already written by the rollout kernel; publish
        = barrier on the side stream.  nccl-allgather: ONE NCCL all-gather of the step's result block per step,
        no packing kernels (fancy_gym_b200/dist).  The exchange of step k runs on NCCL's stream while the rollouts of the
        next steps (which write the OTHER result sets of the wrapper's ring) run on ours; before step k starts ITS
        exchange the stream waits for that of step k - (RING - 1), so no rollout overwrites a block that is still being sent."""
        if exchange["peer"] is not None:
            in_flight.append(exchange["peer"].publish())
        elif world > 1:
            while len(in_flight) > RING - 2:
                in_flight.pop(0).wait()
            in_flight.append(all_gather_result_blocks(env._result_block, out=gathered[n_gathers[0] % RING], async_op=True)[1])
            n_gathers[0] += 1
            if os.environ.get("FG_BENCH_SYNC_GATHER"):      # (experiment switch: no overlap with the next rollout)
                finish_gathers()

    def finish_gathers():
        while in_flight:
            in_flight.pop(0).wait()

    def step_device(s):
        pre_launch()
        env.launch(s["params"], state=s["state"], keep_state=True)
        gather_results()

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---------------- device-timed value ----------------
    # warm-up runs EXACTLY the body of the timed loop (lazy module loading of every kernel in it, NCCL channel set-up)
    total_steps = torch.zeros((), dtype=torch.int64, device=dev)
    for i in range(W):
        step_device(sets[i % n_sets])
        total_steps += env._len.sum()
    finish_gathers()
    sync_all()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    total_steps.zero_()
    step_sums = torch.zeros(K, dtype=torch.int64, device=dev)
    clk = ClockSampler(local_rank)
    clk.__enter__()            # sampled during the device-timed region (NVML queries of 8 ranks at once are kept out of the
                               # host-timed e2e loops: they take driver locks the launches also need)
    if True:
        sync_all()
        t_start = torch.cuda.Event(enable_timing=True); t_end = torch.cuda.Event(enable_timing=True)
        t_start.record()
        host_t0 = time.perf_counter()
        for i in range(K):
            s = sets[(W + i) % n_sets]
            pre_launch()
            kev[i][0].record()
            env.launch(s["params"], state=s["state"], keep_state=True)
            kev[i][1].record()
            gather_results()
            torch.sum(env._len, dim=0, dtype=torch.int64, out=step_sums[i])      # the env steps of this launch: ONE small kernel
        finish_gathers()       # the last exchange is inside the timed region
        t_end.record()
        host_issue_ms = (time.perf_counter() - host_t0) * 1e3 / K     # host time to ISSUE one step (no sync inside)
        sync_all()
    last_outputs = None
    if args.dump_outputs and rank == 0:
        # the result buffers of the last timed launch, copied before later launches of the ring overwrite them
        te, tr, success, collided = env._flag_bytes
        outs = {"obs": env._obs, "return": env._ret, "terminated": te, "truncated": tr, "is_success": success,
                "is_collided": collided, "end_effector": env._info[:, 0:2], "trajectory_length": env._len}
        last_outputs = {k: x.cpu().numpy() for k, x in outs.items()}
    if world > 1:
        clk.__exit__()
    elapsed_ms = t_start.elapsed_time(t_end)
    kernel_ms = sum(a.elapsed_time(b) for a, b in kev) / K
    env_steps = int(step_sums.sum().item())
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    n = torch.tensor([float(env_steps)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(n, op=dist.ReduceOp.SUM)
    elapsed_ms_max, env_steps_all = float(t.item()), float(n.item())
    value = env_steps_all / (elapsed_ms_max * 1e-3)
    episodes_per_s = world * B * K / (elapsed_ms_max * 1e-3)

    # ---------------- FP32 peak probe + roofline of the rollout kernel ----------------
    sink = torch.zeros(4, dtype=torch.float32, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    flops = C.c_double()
    sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
    best = 0.0
    for rep in range(4):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        _lib.check(_lib.lib.fg_ffma_probe(sm_count * 8, 4000, sink.data_ptr(), C.byref(flops), stream))
        b.record()
        torch.cuda.synchronize(dev)
        if rep:
            best = max(best, flops.value / (a.elapsed_time(b) * 1e-3) / 1e12)
    fp32_peak = best
    steps_per_launch = env_steps / K
    achieved = OPS_PER_ENV_STEP * steps_per_launch / (kernel_ms * 1e-3) / 1e12
    ncu = ncu_numbers()
    ncu_roll, ncu_traj = ncu.get("rollout_config2", {}), ncu.get("trajgen_promp", {})
    roofline = dict(bound="fp32", achieved=achieved, peak=fp32_peak, unit="TFLOP/s", frac=achieved / fp32_peak if fp32_peak else None,
                    traffic=ncu_roll.get("dram_bytes") if B == B_PER_GPU else None, traffic_unit="bytes per launch (ncu dram read + write)",
                    kernel="k_rollout<HOLE_REACHER, PROMP, vel, 5>", kernel_ms=kernel_ms,
                    peak_source="FFMA chain probe measured in this run (fg_ffma_probe); MEASURED_PEAKS.json has no CUDA-core figure",
                    note="achieved counts ALGORITHMIC ops: 4356 per env step incl. the literal 500 wall samples; the kernel uses an "
                         "exact-equivalent interval search, so frac is not a pipe utilisation (see profiles/ for ncu pipe numbers)")

    # ---------------- trajectory-only kernel vs HBM ----------------
    hbm_peak, hbm_src = measured_peaks()
    Bt = 1 << 18
    tp = (args.sigma * torch.randn(Bt, N_PARAMS, generator=gen, device=dev)).contiguous()
    env.traj_gen.set_params(tp); env.traj_gen.set_initial_conditions(0.0, None, None); env.traj_gen.set_duration(2.0, 0.01)
    # two rotating output sets (4.2 GB > L2), allocated once: nothing but the kernel runs in the timed region
    outs = [(torch.empty(Bt, 200, 5, device=dev), torch.empty(Bt, 200, 5, device=dev)) for _ in range(2)]
    for i in range(3):
        env.traj_gen._run_trajgen(out=outs[i % 2])
    torch.cuda.synchronize(dev)
    reps = 20
    tev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for i in range(reps):
        tev[i][0].record()
        env.traj_gen._run_trajgen(out=outs[i % 2])
        tev[i][1].record()
    torch.cuda.synchronize(dev)
    del outs
    traj_ms = sum(a.elapsed_time(b) for a, b in tev) / reps        # average launch duration over the timed launches
    traj_gbs = Bt * TRAJ_BYTES_PER_ENV / (traj_ms * 1e-3) / 1e9
    roofline_traj = dict(bound="hbm", achieved=traj_gbs, peak=hbm_peak, unit="GB/s", frac=traj_gbs / hbm_peak,
                         traffic=ncu_traj.get("dram_bytes"), traffic_unit="bytes per launch (ncu dram read + write; algorithmic: %d)" % (Bt * TRAJ_BYTES_PER_ENV),
                         kernel="k_trajgen_closed<PROMP,5,5>", kernel_ms=traj_ms, peak_source=hbm_src,
                         trajectories_per_s=Bt / (traj_ms * 1e-3), workload=f"{Bt} ProMP trajectories [200,5] pos+vel (2.1 GB output, > L2)")

    # ---------------- end to end through the public API from host buffers ----------------
    host_params = [torch.empty(B, N_PARAMS, dtype=torch.float32).pin_memory() for _ in range(2)]
    for hp, s in zip(host_params, sets):
        hp.copy_(s["params"].cpu())
    host_ret = torch.empty(B, dtype=torch.float64).pin_memory()
    host_len = torch.empty(B, dtype=torch.int32).pin_memory()
    host_flags = torch.empty(B, dtype=torch.bool).pin_memory()

    def step_e2e(i):
        env.reset(seed=None)                                          # fresh contexts (fg_reset, numpy-exact streams)
        p = host_params[i % 2].to(dev, non_blocking=True)             # H2D
        obs, ret, te, tr, info = env.step(p)                          # public API
        host_ret.copy_(ret, non_blocking=True)                        # D2H
        host_len.copy_(info["trajectory_length"], non_blocking=True)
        host_flags.copy_(te, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()                  # the caller reads the returns
        return int(host_len.sum())

    for i in range(W):
        step_e2e(i)
    sync_all()
    t0 = time.perf_counter()
    e2e_steps = 0
    for i in range(K):
        e2e_steps += step_e2e(i)
    sync_all()
    e2e_s = time.perf_counter() - t0

    def e2e_dict(seconds, steps, api):
        t = torch.tensor([seconds], dtype=torch.float64, device=dev)
        n = torch.tensor([float(steps)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(n, op=dist.ReduceOp.SUM)
        return dict(value=float(n.item()) / float(t.item()), unit="env-steps/s", h2d_bytes_per_step=B * N_PARAMS * 4,
                    d2h_bytes_per_step=B * (8 + 4 + 1), episodes_per_s=world * B * K / float(t.item()),
                    ms_per_step=1e3 * float(t.item()) / K, api=api)

    e2e_sync = e2e_dict(e2e_s, e2e_steps, "fancy_gym_b200.make(...).reset() + .step(params from pinned host memory) + D2H of "
                        "return/length/terminated, one batch at a time (the host waits for every batch before the next H2D)")

    # the same calls, two batches in flight (EpisodePipeline: submit / wait, the step_async / step_wait pattern): every step
    # still copies ITS parameters from pinned host memory and ITS results back; the copies overlap the neighbouring rollouts
    def make_pipeline(e):
        if E2E_GRAPHS:
            try:
                return fancy_gym.EpisodePipeline(e, slots=E2E_SLOTS, graphs=True), "two CUDA graphs per batch (reset | H2D + rollout + D2H)"
            except Exception as ex_:      # noqa: BLE001  (capture refused: the eager pipeline measures the same calls)
                return fancy_gym.EpisodePipeline(e, slots=E2E_SLOTS), "eager submits (graph capture failed: %r)" % (ex_,)
        return fancy_gym.EpisodePipeline(e, slots=E2E_SLOTS), "eager submits"

    pipe, pipe_mode = make_pipeline(env)
    for i, hp in enumerate(pipe.host_params):
        hp.copy_(host_params[i % len(host_params)])

    def run_pipelined(n, pipe=pipe):
        steps, first = 0, pipe.next_slot
        for i in range(n):
            slot = (first + i) % pipe.SLOTS
            if i >= pipe.SLOTS:
                steps += int(pipe.wait(slot)[1].sum(dtype=torch.int64))      # the caller reads the lengths (and returns) of batch i - SLOTS
            pipe.submit(slot)
        for i in range(max(0, n - pipe.SLOTS), n):
            steps += int(pipe.wait((first + i) % pipe.SLOTS)[1].sum(dtype=torch.int64))
        return steps

    run_pipelined(max(W, pipe.SLOTS))
    sync_all()
    t0 = time.perf_counter()
    p_steps = run_pipelined(K)
    sync_all()
    p_s = time.perf_counter() - t0
    clk.__exit__()
    e2e = e2e_dict(p_s, p_steps, "fancy_gym_b200.EpisodePipeline(env).submit()/wait(): per batch reset() + H2D of the parameters "
                   "from pinned host memory + rollout + D2H of return/length/terminated; %d batches in flight, each with its own env "
                   "state and compute stream (copies and the rollouts of consecutive batches overlap), %s "
                   "(e2e_sync: reset() + step() with one batch at a time)" % (E2E_SLOTS, pipe_mode))
    if e2e_sync["value"] > e2e["value"]:
        e2e, e2e_sync = e2e_sync, e2e

    # ---------------- the same end-to-end step replayed as ONE CUDA graph (extra; the headline e2e stays the eager API) -----
    e2e_graph = None
    try:
        if world > 1:
            raise RuntimeError("skipped for N > 1 (an extra of the single-GPU line)")
        runner = fancy_gym.GraphedEpisode(env)
        runner.host_params.copy_(host_params[0])
        for _ in range(W):
            runner.run()
        sync_all()
        t0 = time.perf_counter()
        g_steps = 0
        for i in range(K):       # (an optimiser writes its samples straight into runner.host_params; H2D is part of the graph)
            g_steps += int(runner.run()[1].sum())
        sync_all()
        g_s = time.perf_counter() - t0
        tg = torch.tensor([g_s], dtype=torch.float64, device=dev)
        ng = torch.tensor([float(g_steps)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tg, op=dist.ReduceOp.MAX)
            dist.all_reduce(ng, op=dist.ReduceOp.SUM)
        e2e_graph = dict(value=float(ng.item()) / float(tg.item()), unit="env-steps/s", ms_per_step=1e3 * float(tg.item()) / K,
                         api="fancy_gym_b200.GraphedEpisode(env).run(): reset + H2D + rollout + D2H as one cudaGraphLaunch")
    except Exception as e:      # noqa: BLE001  (an extra; never fails the bench)
        e2e_graph = dict(error=repr(e))

    # ---------------- the other BASELINE.json configurations + a sustained run (extras; the headline stays configs[1]) ------
    def make_sets(e, Bc, P, sigma, n_sets_c, seed0):
        e_base = e.unwrapped
        out = []
        for i in range(n_sets_c):
            e.reset(seed=seed0 + i)
            out.append(dict(params=(sigma * torch.randn(Bc, P, generator=gen, device=dev)).contiguous(),
                            state=SimpleNamespace(q=e_base.q.clone(), v=torch.zeros_like(e_base.v), steps=torch.zeros_like(e_base.steps),
                                                  done=torch.zeros_like(e_base.done), ctx=e_base.ctx.clone())))
        return out

    def timed_launches(e, sets_c, reps, n_streams=1, min_seconds=0.0, gather=False):
        """device-timed launches of the fused rollout from rotating input sets (keep_state: the launch itself is the step);
        n_streams = 2 keeps two batches in flight (the wrapper's two result sets make that safe); returns ms per launch and
        env steps per launch"""
        main = torch.cuda.current_stream(dev)
        streams = [torch.cuda.Stream(dev) for _ in range(n_streams)] if n_streams > 1 else [main]
        tot = torch.zeros((), dtype=torch.int64, device=dev)
        parts = [torch.zeros((), dtype=torch.int64, device=dev) for _ in streams]

        def run(n):
            for i in range(n):
                st = streams[i % len(streams)]
                with torch.cuda.stream(st):
                    sc = sets_c[i % len(sets_c)]
                    if gather:
                        pre_launch()
                    e.launch(sc["params"], state=sc["state"], keep_state=True)
                    if gather:
                        gather_results()
                    parts[i % len(streams)] += e._len.sum()
        run(3)
        finish_gathers() if gather else None
        sync_all()
        for p_ in parts:
            p_.zero_()
        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        done_reps = 0
        t_host = time.perf_counter()
        a_.record(main)
        for st in streams:
            st.wait_stream(main)
        while True:
            run(reps)
            done_reps += reps
            if time.perf_counter() - t_host >= min_seconds:
                break
        if gather:
            finish_gathers()
        for st in streams:
            main.wait_stream(st)
        b_.record(main)
        sync_all()
        for p_ in parts:
            tot += p_
        ms = a_.elapsed_time(b_) / done_reps
        return ms, int(tot.item()) / done_reps, done_reps

    def agg(ms, steps_per_launch, Bc):
        t_ = torch.tensor([ms], dtype=torch.float64, device=dev)
        n_ = torch.tensor([steps_per_launch], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_, op=dist.ReduceOp.MAX)
            dist.all_reduce(n_, op=dist.ReduceOp.SUM)
        ms_, st_ = float(t_.item()), float(n_.item())
        return dict(ms_per_launch=ms_, env_steps_per_s=st_ / (ms_ * 1e-3), episodes_per_s=world * Bc / (ms_ * 1e-3),
                    mean_episode_length=st_ / (world * Bc), envs_per_gpu=Bc)

    extras = {}
    try:
        if world == 1:
            # sustained: the headline launch repeated for >= 2 s with clocks and power sampled under load
            with ClockSampler(local_rank) as cs:
                ms, spl, n_done = timed_launches(env, sets, 200, min_seconds=2.0)
            extras["sustained"] = dict(agg(ms, spl, B), launches=n_done, seconds=ms * n_done * 1e-3, clocks=cs.summary(),
                                       workload="BASELINE configs[1], the timed launch of `value` repeated for >= 2 s")
            # the same launches with two batches in flight (two streams): the second batch fills the SMs the sub-wave grid of
            # the first leaves partly empty and covers its tail (what `e2e`'s pipeline also does)
            ms, spl, _ = timed_launches(env, sets, 100, n_streams=2)
            extras["config2_two_batches_in_flight"] = dict(agg(ms, spl, B), workload="BASELINE configs[1], two launches in flight on two streams")
            # sigma = 1.0: most episodes end in a collision at different steps (re-packing of live envs inside the kernel)
            s1 = make_sets(env, B, N_PARAMS, 1.0, 6, 50_000)
            ms, spl, _ = timed_launches(env, s1, 40)
            extras["sigma1"] = dict(agg(ms, spl, B), workload=f"{ENV_ID} x {B}, sigma = 1.0, one launch at a time")
            ms, spl, _ = timed_launches(env, s1, 40, n_streams=2)
            extras["sigma1"]["two_batches_in_flight"] = agg(ms, spl, B)
            del s1
            # (more than two batches in flight add ~2 %: tools/probe_sigma1_streams.py)
            # (one batch of 65 536 at sigma = 1.0 cannot beat its longest episode: 200 dependent steps of ~1 us; the same
            #  workload four times as wide — the tail of one launch is a quarter of the work instead of most of it)
            e1w = fancy_gym.make(ENV_ID, num_envs=4 * B, device=dev, context_sampler="device")
            s1w = make_sets(e1w, 4 * B, N_PARAMS, 1.0, 3, 50_000)
            ms, spl, _ = timed_launches(e1w, s1w, 20)
            extras["sigma1"]["envs_x4_one_launch"] = agg(ms, spl, 4 * B)
            del e1w, s1w
            # config 3: fancy_DMP/ViaPointReacher-v0 x 262 144
            e3 = fancy_gym.make("fancy_DMP/ViaPointReacher-v0", num_envs=1 << 18, device=dev, context_sampler="device")
            s3 = make_sets(e3, 1 << 18, 30, 1.0, 3, 60_000)
            ms, spl, _ = timed_launches(e3, s3, 10)
            extras["config3"] = dict(agg(ms, spl, 1 << 18), workload="fancy_DMP/ViaPointReacher-v0 x 262144, weights N(0,1) (x50 inside)")
            del e3, s3
            # config 4: fancy_ProDMP/SimpleReacher-v0 x 65 536 with replanning t % 25, 4 plans, condition_on_desired:
            # reset + ALL FOUR plans in one launch (step_plans), and the same with one launch per plan
            over4 = {"black_box_kwargs": {"replanning_schedule": lambda p_, v_, o_, a_, t_: t_ % 25 == 0, "max_planning_times": 4,
                                          "condition_on_desired": True}}
            e4 = fancy_gym.make("fancy_ProDMP/SimpleReacher-v0", num_envs=B, device=dev, mp_config_override=over4)
            acts = [torch.randn(B, 4, 12, generator=gen, device=dev) for _ in range(4)]

            def episode4(i, fused):
                e4.reset(seed=None)
                if fused:
                    return e4.step_plans(acts[i % 4])[4]["trajectory_length"].sum()
                tot4 = 0
                for j in range(4):
                    tot4 = tot4 + e4.step(acts[i % 4][:, j])[4]["trajectory_length"].sum()
                return tot4
            c4 = {}
            for fused in (True, False):
                e4.reset(seed=1)
                for i in range(3):
                    episode4(i, fused)
                torch.cuda.synchronize(dev)
                a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a_.record()
                tot4 = 0
                for i in range(20):
                    tot4 = tot4 + episode4(i, fused)
                b_.record()
                torch.cuda.synchronize(dev)
                c4["one_launch" if fused else "launch_per_plan"] = agg(a_.elapsed_time(b_) / 20, int(tot4) / 20, B)
            extras["config4"] = dict(c4["one_launch"], launch_per_plan=c4["launch_per_plan"],
                                     workload="fancy_ProDMP/SimpleReacher-v0 x 65536, replanning t % 25, 4 plans, condition_on_desired; "
                                              "per episode batch: reset + step_plans (one fused launch for all four plans)")
            del e4, acts
        if world == 1:
            # learned tau / delay per env (SURVEY §8f rank 2): the per-env basis evaluated inside the rollout, and the
            # two-kernel path it replaces (fg_trajgen_phase -> [B, T, dof] trajectory in HBM -> FG_MP_TRAJ rollout)
            et = fancy_gym.make(ENV_ID, num_envs=B, device=dev, mp_config_override={
                "phase_generator_kwargs": {"phase_generator_type": "linear", "learn_tau": True, "learn_delay": True}})
            pt = (args.sigma * torch.randn(B, N_PARAMS + 2, generator=gen, device=dev)).contiguous()
            pt[:, 0] = 0.5 + 1.5 * torch.rand(B, generator=gen, device=dev)
            pt[:, 1] = 0.3 * torch.rand(B, generator=gen, device=dev)
            lt = {}
            for mode, flag in (("in_rollout", "1"), ("trajgen_then_rollout", "0")):
                os.environ["FG_PHASE_FUSED"] = flag
                tot_t = 0
                for i in range(3):
                    et.reset(seed=None)
                    et.step(pt)
                torch.cuda.synchronize(dev)
                a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a_.record()
                for i in range(20):
                    et.reset(seed=None)
                    tot_t = tot_t + et.step(pt)[4]["trajectory_length"].sum()
                b_.record()
                torch.cuda.synchronize(dev)
                lt[mode] = agg(a_.elapsed_time(b_) / 20, int(tot_t) / 20, B)
            os.environ.pop("FG_PHASE_FUSED", None)
            extras["learned_tau_delay"] = dict(lt["in_rollout"], trajgen_then_rollout=lt["trajgen_then_rollout"],
                                               workload=f"{ENV_ID} x {B} with a learned tau and delay per env; per step: reset + step()")
            del et, pt
        # config 5: 2^20 envs per GPU (N > 1: with the per-step all-gather of every rank's results)
        B5 = 1 << 20
        e5 = fancy_gym.make(ENV_ID, num_envs=B5, device=dev, context_sampler="device", mp_config_override={"black_box_kwargs": {"result_sets": RING}})
        s5 = make_sets(e5, B5, N_PARAMS, args.sigma, 2, 70_000 + 10 * rank)
        if world > 1:
            env_small, peer_small = env, exchange["peer"]
            env = e5                    # gather_results() exchanges env._result_block
            finish_gathers()
            if peer_small is not None:
                exchange["peer"] = make_exchange(e5)
            gathered = [torch.zeros(world * e5._result_block.numel(), dtype=torch.uint8, device=dev) for _ in range(RING)]
        ms, spl, _ = timed_launches(e5, s5, 6, gather=world > 1)
        extras["config5" if world > 1 else "config5_1gpu"] = dict(
            agg(ms, spl, B5), workload=f"{ENV_ID} x {B5} envs per GPU, sigma = {args.sigma}" +
            (", all_gather(return, length, flags) of every rank per launch" if world > 1 else ""))
        if world > 1:
            finish_gathers()
            env, exchange["peer"] = env_small, peer_small
        # ... and end to end: per batch reset + H2D of 105 MB of parameters from pinned host memory + step() + D2H of the results
        pipe5, _ = make_pipeline(e5)
        for i, hp in enumerate(pipe5.host_params):
            hp.copy_(s5[i % len(s5)]["params"])
        run_pipelined(2 * E2E_SLOTS, pipe5)
        sync_all()
        t0 = time.perf_counter()
        n5 = 12
        st5 = run_pipelined(n5, pipe5)
        sync_all()
        dt5 = time.perf_counter() - t0
        t5 = torch.tensor([dt5], dtype=torch.float64, device=dev)
        c5 = torch.tensor([float(st5)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t5, op=dist.ReduceOp.MAX)
            dist.all_reduce(c5, op=dist.ReduceOp.SUM)
        extras["config5" if world > 1 else "config5_1gpu"]["e2e"] = dict(
            value=float(c5.item()) / float(t5.item()), unit="env-steps/s", ms_per_step=1e3 * float(t5.item()) / n5,
            h2d_bytes_per_step=B5 * N_PARAMS * 4, d2h_bytes_per_step=B5 * 13, batches_in_flight=E2E_SLOTS)
        del pipe5, e5, s5
    except Exception as ex:      # noqa: BLE001  (extras never fail the bench line)
        extras["error"] = repr(ex)
    torch.cuda.empty_cache()

    # ---------------- CPU baseline (rank 0, N = 1 only) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ref = CpuReference(args.sigma)
        cpu = ref.baseline()
        ref.close()

    clocks = clk.summary()
    if B == B_PER_GPU and clocks.get("sm_mhz") and ncu_roll.get("warp_instructions"):
        # what the machine actually executed: warp instructions of the committed ncu capture of this launch / live kernel time
        # against the issue rate (4 schedulers x 1 instruction per clock per SM at the sampled SM clock); pipe shares: the capture's
        roofline["executed"] = dict(warp_instructions_per_launch=ncu_roll["warp_instructions"],
                                    thread_instructions_per_env_step=ncu_roll["warp_instructions"] * ncu_roll.get("threads_per_instruction", 32.0) / steps_per_launch,
                                    issue_slot_frac=ncu_roll["warp_instructions"] / (kernel_ms * 1e-3 * clocks["sm_mhz"] * 1e6 * sm_count * 4),
                                    ncu_pct_of_peak_sustained_active=ncu_roll.get("pipes"),
                                    source=ncu_roll.get("source"))
    if rank == 0:
        line = dict(metric="env-steps/sec (fancy_ProMP/HoleReacher-v0 MP black-box rollout)", value=value, unit="env-steps/s",
                    n_gpus=world, steps=K, warmup=W, ms_per_step=elapsed_ms_max / K, higher_is_better=True, scaling="weak",
                    vs_baseline=None, dtype="f32", data="synthetic",
                    config=dict(workload=f"{ENV_ID}, {B} envs per GPU (BASELINE configs[1]), one fused rollout launch per step",
                                envs_per_gpu=B, n_params=N_PARAMS, sigma=args.sigma, max_episode_steps=200,
                                contexts="device sampler (numpy-exact PCG64 streams, fg_reset)", parallelism=f"env-shard x{world}",
                                l2="inputs rotate over %d sets (%.0f MB > 126 MB L2)" % (n_sets, n_sets * set_bytes / 1e6),
                                collective={"none": "none",
                                            "peer-stores": "fused: the rollout kernel stores (return, length, flags) of every env into every rank's gather "
                                                           "buffer over NVLink peer memory; one barrier per step on a side stream (ring of 4 slots)",
                                            "nccl-allgather": "all_gather(return,length,flags) per step, asynchronous behind the next rollouts "
                                                              "(ring of %d result sets)" % RING}[exchange["mode"]],
                                exchange_note=exchange["note"],
                                cpu_binding=(f"rank 0 bound to the {len(bound_cpus)} CPUs local to its GPU" if bound_cpus else "none")),
                    episodes_per_s=episodes_per_s, mean_episode_length=env_steps / (K * B), host_issue_ms_per_step=host_issue_ms,
                    roofline=roofline, roofline_trajgen=roofline_traj, cpu_baseline=cpu, e2e=e2e, e2e_sync=e2e_sync, e2e_graph=e2e_graph,
                    clocks=clocks, gpu_launches=K, configs=extras)
        if last_outputs is not None:
            dump_outputs(args.dump_outputs, last_outputs)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
