#!/usr/bin/env python
"""Cost of the receding-horizon MPC loop (mpc.mpc_iteration) over the plain rollout sweep.

    python tools/mpc_loop.py [--worlds 131072] [--horizon 50] [--repeats 5] [--legs abcdefg] [--profile] [--out FILE]
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

Leg e times only what MPPI adds to a horizon (mpc.mppi_iteration minus the rollout), at sigma = 0 so
that the schedule is the constant one of leg c: egg_sample_controls, the allgather of the baseline,
egg_mppi_reduce, the allgather of the partials and the rank-order combine into the new nominal
schedule.  egg_sample_controls and egg_mppi_reduce are also timed alone, and their achieved GB/s
(bytes computed from the shapes) are reported against the 6555.8 GB/s copy bandwidth of BASELINE.md.
Then mppi_iteration runs with sigma > 0 on the torques and the representative cost, and its
world-steps/s are reported.  --profile adds the device time of the MPPI kernels of one leg e.

Leg f times only what CEM adds to a horizon (mpc.cem_iteration minus the rollout), at std = 0 so that
the schedule is the constant one of leg c: egg_sample_controls_std, the cost allgather with the
top-k selection, the elite schedules' gather (egg_gather_controls) and exchange, egg_control_moments
and the refit of u_nom and std.  Each of those parts is also timed on its own.  Then
egg_sample_controls_std and egg_sample_controls are timed alone, alternating in the same call, with
their GB/s against the same copy bandwidth, and cem_iteration runs with sigma > 0 on the torques and
the representative cost, and its world-steps/s are reported.
Leg g runs MPPI in joint space: a second batch of the same worlds with the 57 motors of legged20's 19
ball joints as its actuator table (scenes.legged20_motors, Batch.set_actuators), in gravity (the
actuation kernel adds m g to every body; the nominal plan starts at zero torques).  It times whole
mppi_iterations with the representative cost (its control term on the 57 motor torques), so ms per
horizon compares with the body-wrench mppi_loop_cost of leg e.  egg_sample_controls and
egg_mppi_reduce are timed alone at the row width c = 57 with their GB/s.  --profile adds the device
time of the actuation kernel (egg_actuate_kernel) per horizon against egg_fext_slice_cost_kernel of
a body-wrench rollout with the same cost.
--legs picks the legs to run (b needs a; the overheads need the legs they compare).
Rank 0 prints one JSON line with the GPU name and power limit.

Memory: a schedule is H x worlds x 20 x 6 doubles, 6.3 GB per GPU at 131072 worlds and H = 50; the
script holds three (constant, random and MPPI or CEM samples), plus the batch and one saved start state (0.4 GB).
Leg g adds a second batch and a joint-space schedule of H x worlds x 57 doubles (3.0 GB).
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
    ap.add_argument("--legs", default="abcdefg", help="legs to run (default: all)")
    ap.add_argument("--lam", type=float, default=1.0, help="MPPI temperature lambda of leg e")
    ap.add_argument("--elites", type=int, default=128, help="CEM elites of leg f (n_elite, over all GPUs)")
    ap.add_argument("--sigma-motor", type=float, default=0.5, help="std. dev. of the joint-motor torques of leg g (N m)")
    ap.add_argument("--profile", action="store_true", help="also record the kernel times of legs c, d, e and f with torch.profiler")
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


def profile_legs(prepare, legs, sync):
    """Device milliseconds of the per-step control kernels of one leg c and one leg d, and of the
    MPPI kernels of one leg e and the CEM kernels of one leg f."""
    from torch.profiler import profile, ProfilerActivity
    out = {}
    for name, fn in legs.items():
        prepare(name)
        sync()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            sync()
        for e in prof.key_averages():
            kernel = re.search(r"egg_\w+", e.key)
            if kernel and any(key in kernel.group(0) for key in ("fext_slice", "egg_actuate", "egg_cost", "egg_mppi", "egg_gather_controls",
                                                                 "egg_control_moments")):
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
    u_mppi = torch.empty_like(u_const) if ("e" in args.legs or "f" in args.legs) else None   # MPPI or CEM samples
    # MPPI planners around world 0's f_ext: sigma = 0 for the overhead of leg e, sigma on the torques for the loop
    sigma = np.zeros((n, 6))
    sigma[:, 3:6] = args.sigma
    mppi0 = mpc.MPPI(n, H, sigma=0.0, lam=args.lam, seed=11, u_nom=scene["f_ext"][0], device=dev)
    mppi1 = mpc.MPPI(n, H, sigma=sigma, lam=args.lam, seed=12, u_nom=scene["f_ext"][0], device=dev)
    # CEM planners the same way: std = 0 for the overhead of leg f, sigma on the torques for the loop
    cem0 = mpc.CEM(n, H, sigma=0.0, n_elite=args.elites, seed=13, u_nom=scene["f_ext"][0], device=dev)
    cem1 = mpc.CEM(n, H, sigma=sigma, n_elite=args.elites, seed=14, u_nom=scene["f_ext"][0], device=dev)
    motors = E.scenes.legged20_motors()
    c_joint = motors.m
    u_joint = torch.empty((H, W, c_joint), dtype=torch.float64, device=dev) if "g" in args.legs else None
    mppi_joint = mpc.MPPI(n, H, sigma=args.sigma_motor, lam=args.lam, seed=15, m=c_joint, device=dev)
    L = H * n * 6
    Lj = H * c_joint
    chunks = -(-W // 256)   # stage-1 chunks of egg_mppi_reduce
    sample_bytes = 8 * (H * W * n * 6 + L)                                  # write the samples, read u_nom
    reduce_bytes = 8 * (H * W * n * 6 + W + 2 * chunks * (L + 2) + L + 2)   # read u and J, partials out and in, result
    sample_std_bytes = 8 * (H * W * n * 6 + 2 * L)                          # write the samples, read mean and std
    sample_joint_bytes = 8 * (H * W * c_joint + Lj)                             # the same at the row width of the motors
    reduce_joint_bytes = 8 * (H * W * c_joint + W + 2 * chunks * (Lj + 2) + Lj + 2)
    costs = torch.empty(W, dtype=torch.float64, device=dev)
    all_costs = torch.empty(n_total, dtype=torch.float64, device=dev)
    start = torch.empty((W, n * 18), dtype=torch.float64, device=dev)

    def representative_cost(x0, m=None):
        """x0: world 0's start rows [n, 18].  Tracks a reference that moves every body along +x at
        0.5 m/s from x0, with small velocities and small controls, and rewards progress of body 0.
        m: the cost for a batch with an actuator table of m actuators."""
        q_run = np.zeros((n, mpc.STATE_PER_BODY))
        q_run[:, 0:3], q_run[:, 12:15] = 1.0, 0.1
        l_term = np.zeros((n, mpc.STATE_PER_BODY))
        l_term[0, 0] = -1.0
        x_ref = np.repeat(x0[None], H + 1, axis=0)
        x_ref[:, :, 0] += 0.5 * dt * np.arange(H + 1)[:, None]
        return mpc.QuadraticCost(n, q_run=q_run, u_run=1e-3, l_term=l_term, x_ref=x_ref, m=m)

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
        bj = None
        if "g" in args.legs:   # the same worlds with the joint motors as the control space
            bj = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=k_max, device=local)
            bj.set_stream(stream.cuda_stream)
            bj.set_actuators(motors)
            bj.set_cost(representative_cost(start[0].view(n, mpc.STATE_PER_BODY).cpu().numpy(), m=c_joint))
            bj.set_sampler(mppi_joint)

        def reset():
            for x in (b, bj):
                if x is not None:
                    x.seed_state(start.data_ptr(), W, 0)
                    x.snapshot()

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

        def leg_e():
            mpc.mppi_sample(b, mppi0, u_mppi, first)
            mpc.mppi_combine(b, mppi0, u_mppi, costs)

        def pack_controls(local):   # the elites' schedules of this rank, as cem_iteration fetches them
            out = torch.empty((len(local), L), dtype=torch.float64, device=dev)
            if len(local):
                b.gather_controls(u_mppi.data_ptr(), H, local, out.data_ptr())
            return out

        moments = torch.empty((2, H, n, 6), dtype=torch.float64, device=dev)

        def cem_moments(rows):
            b.control_moments(rows.data_ptr(), rows.shape[0], H, moments.data_ptr())

        def leg_f():
            mpc.cem_sample(b, cem0, u_mppi, first)
            cem_moments(mpc.cem_select(cem0, costs, n_total, pack_controls)[3])
            mpc.cem_refit(cem0, moments)

        def leg_g():
            mpc.mppi_iteration(bj, mppi_joint, dt, u_joint, first)

        legs = {name: fn for name, fn in (("a", leg_a), ("c", leg_c), ("b", leg_b), ("d", leg_d), ("e", leg_e), ("f", leg_f),
                                          ("g", leg_g)) if name in args.legs}

        def prepare(name):   # the cost is set for leg d only (outside the timed region: set_cost synchronises)
            reset()
            b.set_cost(cost if name == "d" else None)
            if name in "ef":   # the costs of a rollout of the constant schedule, which legs e and f weigh
                b.set_sampler(mppi0 if name == "e" else cem0)
                leg_c()

        for name, fn in legs.items():     # warm-up
            prepare(name)
            fn()
        t = {name: [] for name in legs}
        for _ in range(args.repeats):
            for name, fn in legs.items():
                prepare(name)
                t[name].append(timed(fn))
        t = {name: np.array(x) for name, x in t.items()}
        entry = {}
        for name, key in (("a", "a_sweep_ms"), ("c", "c_controlled_sweep_ms"), ("b", "b_mpc_iteration_ms"),
                          ("d", "d_controlled_cost_sweep_ms"), ("e", "e_mppi_additions_ms"), ("f", "f_cem_additions_ms"),
                          ("g", "g_joint_mppi_iteration_ms")):
            if name in t:
                entry[key] = spread(t[name])
        for key, hi, lo, base in (("slice_copy_overhead", "c", "a", "a"), ("loop_overhead", "b", "a", "a"),
                                  ("cost_overhead", "d", "c", "c")):
            if hi in t and lo in t:
                entry[key + "_ms"] = spread(t[hi] - t[lo])
                entry[key + "_pct"] = spread(100.0 * (t[hi] - t[lo]) / t[base])
        for name in "ef":
            if name in t and "c" in t:
                entry[f"{name}_{'mppi' if name == 'e' else 'cem'}_additions_pct_of_c"] = spread(100.0 * t[name] / t["c"])
        if "e" in t:   # the two kernels alone, and their bandwidth
            prepare("e")
            ks, kr = [], []
            ub = torch.zeros((), dtype=torch.float64, device=dev)
            part = torch.empty(L + 2, dtype=torch.float64, device=dev)
            for _ in range(args.repeats):
                ks.append(timed(lambda: b.sample_controls(mppi0.u_nom.data_ptr(), H, mppi0.seed, 0, first, u_mppi.data_ptr())))
                kr.append(timed(lambda: b.mppi_reduce(u_mppi.data_ptr(), H, costs.data_ptr(), ub.data_ptr(), args.lam, part.data_ptr())))
            ks, kr = np.array(ks), np.array(kr)
            entry["e_kernels"] = {
                "copy_bandwidth_GBps": 6555.8,
                "sample_controls": {"ms": spread(ks), "bytes": sample_bytes, "GBps": spread(sample_bytes / (ks * 1e-3) / 1e9)},
                "mppi_reduce": {"ms": spread(kr), "bytes": reduce_bytes, "GBps": spread(reduce_bytes / (kr * 1e-3) / 1e9),
                                "launches": 2, "chunks": chunks}}
        if "f" in t:   # the parts of leg f one by one, then the two samplers alone, alternating
            prepare("f")
            parts = {"sample_std": [], "cost_allgather_topk": [], "elite_gather_exchange": [], "moments": [], "update": []}
            got = {}
            for _ in range(args.repeats):
                parts["sample_std"].append(timed(lambda: mpc.cem_sample(b, cem0, u_mppi, first)))
                parts["cost_allgather_topk"].append(timed(lambda: got.update(
                    el=mpc.select_best(mpc.allgather_costs(costs), cem0.n_elite)[0])))
                parts["elite_gather_exchange"].append(timed(lambda: got.update(rows=mpc.gather_winner_states(got["el"], n_total, pack_controls))))
                parts["moments"].append(timed(lambda: cem_moments(got["rows"])))
                parts["update"].append(timed(lambda: mpc.cem_refit(cem0, moments)))
            entry["f_parts_ms"] = {key: spread(x) for key, x in parts.items()}
            kstd, kbody = [], []
            for _ in range(args.repeats):
                kstd.append(timed(lambda: b.sample_controls_std(cem0.u_nom.data_ptr(), cem0.std.data_ptr(), H, cem0.seed, 0, first,
                                                                u_mppi.data_ptr())))
                kbody.append(timed(lambda: b.sample_controls(cem0.u_nom.data_ptr(), H, cem0.seed, 0, first, u_mppi.data_ptr())))
            kstd, kbody = np.array(kstd), np.array(kbody)
            entry["f_kernels"] = {
                "copy_bandwidth_GBps": 6555.8, "elites": cem0.n_elite,
                "sample_controls_std": {"ms": spread(kstd), "bytes": sample_std_bytes, "GBps": spread(sample_std_bytes / (kstd * 1e-3) / 1e9)},
                "sample_controls": {"ms": spread(kbody), "bytes": sample_bytes, "GBps": spread(sample_bytes / (kbody * 1e-3) / 1e9)}}
        if "g" in t:   # the two MPPI kernels alone at the motors' row width, and their bandwidth
            prepare("g")
            costs.fill_(1.0)   # finite costs for the reduction (weights exp(-1 / lam))
            ks, kr = [], []
            ub = torch.zeros((), dtype=torch.float64, device=dev)
            part = torch.empty(Lj + 2, dtype=torch.float64, device=dev)
            for _ in range(args.repeats):
                ks.append(timed(lambda: bj.sample_controls(mppi_joint.u_nom.data_ptr(), H, mppi_joint.seed, 0, first, u_joint.data_ptr())))
                kr.append(timed(lambda: bj.mppi_reduce(u_joint.data_ptr(), H, costs.data_ptr(), ub.data_ptr(), args.lam, part.data_ptr())))
            ks, kr = np.array(ks), np.array(kr)
            entry["g_joint_space"] = {
                "actuators": c_joint, "sigma_motor": args.sigma_motor, "lam": args.lam, "gravity": list(b.desc.gravity),
                "ms_per_horizon": spread(t["g"]), "world_steps_per_s": spread(n_total * H / (t["g"] * 1e-3)),
                "schedule_GB": H * W * c_joint * 8 / 1e9, "body_wrench_schedule_GB": H * W * n * 6 * 8 / 1e9,
                "copy_bandwidth_GBps": 6555.8,
                "sample_controls": {"ms": spread(ks), "bytes": sample_joint_bytes, "GBps": spread(sample_joint_bytes / (ks * 1e-3) / 1e9)},
                "mppi_reduce": {"ms": spread(kr), "bytes": reduce_joint_bytes, "GBps": spread(reduce_joint_bytes / (kr * 1e-3) / 1e9),
                                "launches": 2, "chunks": chunks}}
        if args.profile:
            prof = {x: legs[x] for x in "cdefg" if x in legs}
            if "g" in legs:   # the body-wrench rollout with a cost, for egg_fext_slice_cost_kernel against egg_actuate_kernel
                prof.setdefault("d", leg_d)
            entry["kernel_ms_per_horizon"] = profile_legs(prepare, prof, sync)
        # the loop itself with random time-varying schedules (the state evolves from iteration to iteration),
        # with the built-in cost and with the configured one
        loops = [(key, qc) for key, qc, leg in (("random_loop", None, "b"), ("random_loop_cost", cost, "d")) if leg in legs]
        if "e" in legs:   # MPPI with sigma > 0 and the representative cost
            reset()
            b.set_cost(cost)
            b.set_sampler(mppi1)
            mpc.mppi_iteration(b, mppi1, dt, u_mppi, first)
            ms = timed(lambda: [mpc.mppi_iteration(b, mppi1, dt, u_mppi, first) for _ in range(args.random_iters)])
            entry["mppi_loop_cost"] = {"iterations": args.random_iters, "ms_per_iteration": ms / args.random_iters,
                                       "world_steps_per_s": n_total * H * args.random_iters / (ms * 1e-3),
                                       "sigma_torque": args.sigma, "lam": args.lam}
        if "f" in legs:   # CEM with sigma > 0 and the representative cost
            reset()
            b.set_cost(cost)
            b.set_sampler(cem1)
            mpc.cem_iteration(b, cem1, dt, u_mppi, first, n_total)
            ms = timed(lambda: [mpc.cem_iteration(b, cem1, dt, u_mppi, first, n_total) for _ in range(args.random_iters)])
            entry["cem_loop_cost"] = {"iterations": args.random_iters, "ms_per_iteration": ms / args.random_iters,
                                      "world_steps_per_s": n_total * H * args.random_iters / (ms * 1e-3),
                                      "sigma_torque": args.sigma, "elites": cem1.n_elite}
        for key, qc in loops:
            reset()
            b.set_cost(qc)
            mpc.mpc_iteration(b, u_rand, dt, k, n_total, first)
            ms = timed(lambda: [mpc.mpc_iteration(b, u_rand, dt, k, n_total, first) for _ in range(args.random_iters)])
            entry[key] = {"iterations": args.random_iters, "ms_per_iteration": ms / args.random_iters,
                          "world_steps_per_s": n_total * H * args.random_iters / (ms * 1e-3)}
        st = b.status()
        entry["status_or"] = int(np.bitwise_or.reduce(st["status"]))
        if bj is not None:
            entry["g_status_or"] = int(np.bitwise_or.reduce(bj.status()["status"]))
            bj.close()
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
