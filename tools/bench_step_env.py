"""Benchmark of the step-based envs (fg_env_step, one control step per call): prints ONE JSON line.

For HoleReacher-5 (float32 and float64 actions), ViaPointReacher-5 and SimpleReacher-2, at B = 2^16 and 2^20 envs (the
second one's working set, ~340 MB per step for HoleReacher-5, is far above the 126 MB L2):
  kernel_us          time per step of 200 back-to-back step() launches captured in one CUDA graph, from CUDA events
  env_steps_per_s    B / kernel time
  algo_bytes         bytes per env-step the algorithm has to move (state in and out, action, context, outputs: computed
                     from the shapes below, not measured), algo_TBps = algo_bytes * env-steps/s, and its share of the
                     7.7 TB/s HBM3e data-sheet figure of one B200
  eager_calls_per_s  env.step() calls per second from a Python loop (launch overhead included)
  graph_calls_per_s  replays per second of a CUDA graph holding one step() call
The GPU's name and power limit are read with `nvidia-smi --query-gpu=name,power.limit` (read-only).

    python tools/bench_step_env.py [--sizes 65536 1048576] [--launches 200]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HBM_TBPS = 7.7          # NVIDIA data sheet, HGX B200, per GPU
CONFIGS = [("HoleReacher-v0", "float32"), ("HoleReacher-v0", "float64"), ("ViaPointReacher-v0", "float32"),
           ("SimpleReacher-v0", "float32")]
OBS_EXTRA = {"HoleReacher-v0": 4, "ViaPointReacher-v0": 5, "SimpleReacher-v0": 3}


def algo_bytes(name, n, dtype):
    """(read, written) bytes of one env-step: q, v float64 [n] each, steps int32, ctx float64 [4] and the action in;
    q, v, steps, done (1 byte), the float32 observation, reward float64, 4 flag bytes and info float64 [2] out"""
    a = (8 if dtype == "float64" else 4) * n
    read = 8 * n + 8 * n + 4 + 32 + a
    written = 8 * n + 8 * n + 4 + 1 + 4 * (3 * n + OBS_EXTRA[name]) + 8 + 4 + 16
    return read, written


def gpu_name_and_power():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, check=True).stdout.splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception:      # noqa: BLE001
        import torch
        return torch.cuda.get_device_name(0), "unknown"


def bench_one(fg, name, dtype, B, launches):
    import torch
    dev = "cuda:0"
    env = fg.make(f"fancy/{name}", num_envs=B, device=dev)
    env.reset(seed=0)
    gen = torch.Generator(device=dev).manual_seed(0)
    a = torch.randn(B, env.n_links, generator=gen, device=dev).to(getattr(torch, dtype))
    for _ in range(20):                                   # warm-up (allocates the output ring)
        env.step(a)
    torch.cuda.synchronize()
    # kernel time: `launches` back-to-back steps in one graph, timed with CUDA events
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(launches):
            env.step(a)
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(3):
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) * 1e3 / launches)
    kernel_us = min(times)
    # step() calls per second: eager Python loop, and a graph of ONE step() replayed
    n_calls = max(launches, 200)
    t0 = time.perf_counter()
    for _ in range(n_calls):
        env.step(a)
    torch.cuda.synchronize()
    eager = n_calls / (time.perf_counter() - t0)
    g1 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g1):
        env.step(a)
    g1.replay()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n_calls):
        g1.replay()
    torch.cuda.synchronize()
    graphed = n_calls / (time.perf_counter() - t0)
    rd, wr = algo_bytes(name, env.n_links, dtype)
    rate = B / (kernel_us * 1e-6)
    tbps = (rd + wr) * rate / 1e12
    del g, g1
    return dict(env=name, n_links=env.n_links, action_dtype=dtype, B=B, kernel_us=round(kernel_us, 2),
                kernel_us_runs=[round(x, 2) for x in times], env_steps_per_s=float(f"{rate:.4g}"),
                algo_bytes_read=rd, algo_bytes_written=wr, algo_TBps=round(tbps, 3),
                share_of_hbm_datasheet=round(tbps / HBM_TBPS, 3), eager_calls_per_s=round(eager), graph_calls_per_s=round(graphed))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--sizes", type=int, nargs="+", default=[1 << 16, 1 << 20])
    ap.add_argument("--launches", type=int, default=200)
    args = ap.parse_args()
    if args.launches < 200:
        ap.error("--launches must be >= 200")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_step_env.py needs a CUDA device")
    import fancy_gym_b200 as fg
    gpu, power = gpu_name_and_power()
    rows = [bench_one(fg, name, dtype, B, args.launches) for B in args.sizes for name, dtype in CONFIGS]
    print(json.dumps(dict(bench="step_env", gpu=gpu, power_limit=power, hbm_datasheet_TBps=HBM_TBPS,
                          launches=args.launches, results=rows)))


if __name__ == "__main__":
    main()
