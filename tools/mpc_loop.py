#!/usr/bin/env python
"""Cost of the receding-horizon MPC loop (mpc.mpc_iteration) over the plain rollout sweep.

    python tools/mpc_loop.py [--worlds 131072] [--horizon 50] [--repeats 5] [--profile] [--out FILE]
    python -m torch.distributed.run --nproc_per_node N tools/mpc_loop.py ...

One process per GPU; every rank owns `--worlds` legged20 worlds (bench.py's c5mpc scene, seeded per
rank).  For each sweep cap K (K <= 500 with the reference's termination, and fixed K = 20) four
legs are timed with CUDA events, alternating, each from the same start state:
  a  the existing sweep: egg_restore, egg_step(n = H), rollout costs, cost allgather (bench.py c5mpc);
  c  the same with egg_step_controlled and a schedule whose every slice is the scene's f_ext;
  b  mpc_iteration with that schedule: c + host top-k selection, winner-state exchange, re-seeding
     and snapshot;
  d  egg_restore, egg_step_controlled_cost with that schedule and a representative QuadraticCost
     (running cost on p and v of every body and on every control, a per-step reference of H + 1
     rows, progress of body 0 along +x as the terminal term), cost allgather.
The physics of the four legs is identical, so c - a is the cost of the per-step slice copy, b - a
the whole overhead of the loop and d - c the cost of accumulating the configured cost on the device
(in place of the built-in terminal cost).  Then the loop runs with random time-varying schedules,
without and with the cost set, and its world-steps/s are reported.  --profile adds the device time
of the per-step kernels of one c and one d leg from torch.profiler (a separate, untimed pass).
Rank 0 prints one JSON line with the GPU name and power limit.

Memory: a schedule is H x worlds x 20 x 6 doubles, 6.3 GB per GPU at 131072 worlds and H = 50; the
script holds two (constant and random), plus the batch and one saved start state (0.4 GB).
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--worlds", type=int, default=131072, help="legged20 worlds per GPU")
    ap.add_argument("--horizon", type=int, default=50, help="steps per horizon (H)")
    ap.add_argument("--k-max", default="500,20", help="comma-separated sweep caps")
    ap.add_argument("--winners", type=int, default=16, help="k of the top-k selection")
    ap.add_argument("--repeats", type=int, default=5, help="timed repeats of each leg")
    ap.add_argument("--random-iters", type=int, default=3, help="timed loop iterations with random schedules")
    ap.add_argument("--sigma", type=float, default=0.05, help="std. dev. of the random torques (N m)")
    ap.add_argument("--profile", action="store_true", help="also record the per-step kernel times of legs c and d with torch.profiler")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    return ap.parse_args()


def gpu_info(index):
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(index)],
                           capture_output=True, text=True, timeout=30)
        name, limit = [x.strip() for x in r.stdout.strip().split(",")[:2]]
        return name, limit
    except Exception as e:  # the JSON line still names the device through torch
        return None, f"unavailable ({e})"


def spread(xs):
    xs = np.asarray(xs, dtype=np.float64)
    return {"median": float(np.median(xs)), "min": float(xs.min()), "max": float(xs.max()), "n": int(xs.size)}


def profile_legs(b, prepare, leg_c, leg_d, sync):
    """Device milliseconds of the per-step control kernels of one leg c and one leg d."""
    from torch.profiler import profile, ProfilerActivity
    out = {}
    for name, fn in (("c", leg_c), ("d", leg_d)):
        prepare(name)
        sync()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            sync()
        for e in prof.key_averages():
            kernel = re.search(r"egg_\w+", e.key)
            if kernel and ("fext_slice" in kernel.group(0) or "egg_cost" in kernel.group(0)):
                out[f"{name}: {kernel.group(0)}"] = {"calls": e.count, "ms": e.device_time_total / 1e3}
    return out


def main():
    args = parse()
    import torch
    import torch.distributed as dist
    import eggshell_b200 as E
    from eggshell_b200 import mpc

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    ws = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("mpc_loop.py needs a CUDA device: eggshell_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    if ws > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    stream = torch.cuda.current_stream(dev)
    W, H, k = args.worlds, args.horizon, args.winners
    n_total, first = W * ws, W * rank
    scene = E.scenes.legged20(W, seed=[5000, rank])
    dt, n = scene["dt"], scene["n"]
    f_ext = torch.from_numpy(scene["f_ext"]).to(dev)
    u_const = f_ext.expand(H, W, n, 6).contiguous()
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    u_rand = u_const.clone()
    u_rand[..., 3:6] += args.sigma * torch.randn(u_rand[..., 3:6].shape, generator=gen, device=dev, dtype=torch.float64)
    costs = torch.empty(W, dtype=torch.float64, device=dev)
    all_costs = torch.empty(n_total, dtype=torch.float64, device=dev)
    start = torch.empty((W, n * 18), dtype=torch.float64, device=dev)

    def representative_cost(x0):
        """x0: world 0's start rows [n, 18].  Tracks a reference that moves every body along +x at
        0.5 m/s from x0, with small velocities and small controls, and rewards progress of body 0."""
        q_run = np.zeros((n, mpc.STATE_PER_BODY))
        q_run[:, 0:3], q_run[:, 12:15] = 1.0, 0.1
        l_term = np.zeros((n, mpc.STATE_PER_BODY))
        l_term[0, 0] = -1.0
        x_ref = np.repeat(x0[None], H + 1, axis=0)
        x_ref[:, :, 0] += 0.5 * dt * np.arange(H + 1)[:, None]
        return mpc.QuadraticCost(n, q_run=q_run, u_run=1e-3, l_term=l_term, x_ref=x_ref)

    def sync():
        if ws > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn):
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        sync()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if ws > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    result = {"tool": "tools/mpc_loop.py", "scene": "legged20", "worlds_per_gpu": W, "gpus": ws, "horizon": H,
              "winners": k, "dt": dt, "device": torch.cuda.get_device_name(dev)}
    result["gpu_name"], result["power_limit"] = gpu_info(local)
    for k_max in [int(x) for x in args.k_max.split(",")]:
        b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=k_max, device=local)
        b.set_stream(stream.cuda_stream)
        b.snapshot()
        b.gather_state(np.arange(W), start.data_ptr())   # the common start of every timed leg
        cost = representative_cost(start[0].view(n, mpc.STATE_PER_BODY).cpu().numpy())

        def reset():
            b.seed_state(start.data_ptr(), W, 0)
            b.snapshot()

        def leg_a():
            b.restore()
            b.step(dt, n_steps=H)
            b.rollout_costs(costs.data_ptr())
            if ws > 1:
                dist.all_gather_into_tensor(all_costs, costs)

        def leg_c():
            b.restore()
            b.step_controlled(dt, u_const.data_ptr(), H)
            b.rollout_costs(costs.data_ptr())
            if ws > 1:
                dist.all_gather_into_tensor(all_costs, costs)

        def leg_b():
            mpc.mpc_iteration(b, u_const, dt, k, n_total, first)

        def leg_d():
            b.restore()
            b.step_controlled_cost(dt, u_const.data_ptr(), H, costs.data_ptr())
            if ws > 1:
                dist.all_gather_into_tensor(all_costs, costs)

        legs = {"a": leg_a, "c": leg_c, "b": leg_b, "d": leg_d}

        def prepare(name):   # the cost is set for leg d only (outside the timed region: set_cost synchronises)
            reset()
            b.set_cost(cost if name == "d" else None)

        for name, fn in legs.items():     # warm-up
            prepare(name)
            fn()
        t = {name: [] for name in legs}
        for _ in range(args.repeats):
            for name, fn in legs.items():
                prepare(name)
                t[name].append(timed(fn))
        a, c, bb, d = np.array(t["a"]), np.array(t["c"]), np.array(t["b"]), np.array(t["d"])
        entry = {"a_sweep_ms": spread(a), "c_controlled_sweep_ms": spread(c), "b_mpc_iteration_ms": spread(bb),
                 "d_controlled_cost_sweep_ms": spread(d),
                 "slice_copy_overhead_ms": spread(c - a), "loop_overhead_ms": spread(bb - a), "cost_overhead_ms": spread(d - c),
                 "slice_copy_overhead_pct": spread(100.0 * (c - a) / a), "loop_overhead_pct": spread(100.0 * (bb - a) / a),
                 "cost_overhead_pct": spread(100.0 * (d - c) / c)}
        if args.profile:
            entry["kernel_ms_per_horizon"] = profile_legs(b, prepare, leg_c, leg_d, sync)
        # the loop itself with random time-varying schedules (the state evolves from iteration to iteration),
        # with the built-in cost and with the configured one
        for key, qc in (("random_loop", None), ("random_loop_cost", cost)):
            reset()
            b.set_cost(qc)
            mpc.mpc_iteration(b, u_rand, dt, k, n_total, first)
            ms = timed(lambda: [mpc.mpc_iteration(b, u_rand, dt, k, n_total, first) for _ in range(args.random_iters)])
            entry[key] = {"iterations": args.random_iters, "ms_per_iteration": ms / args.random_iters,
                          "world_steps_per_s": n_total * H * args.random_iters / (ms * 1e-3)}
        st = b.status()
        entry["status_or"] = int(np.bitwise_or.reduce(st["status"]))
        result[f"k_max_{k_max}"] = entry
        b.close()
    if rank == 0:
        line = json.dumps(result)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(line + "\n")
    if ws > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
