"""Cost of Coulomb-pyramid friction (egg_set_friction) against the reference's BOX friction:
`python tools/friction_bench.py [--out profiles/r3h_coulomb_friction.json] [--steps 3] [--reps 2]`.

Workloads C3 (65536 x pile64, max_contacts 1024) and C5 (131072 x legged20), each at K <= 500 and at
K = 20.  Three friction settings per batch -- BOX, Coulomb mu = 0.5, Coulomb mu uniform in [0.2, 1.0]
per world (seed 0) -- alternated in `reps` rounds inside one process.  Every timed step restores the
scene's start state first (as bench.py does), so all steps of a setting do the same work.  Reported
per setting: world-steps/s (CUDA events around restore + step), mean / max sweeps of the last step,
and the solve bucket of the step's kernel time (solve + integrate) per step and per mean sweep.  At
K = 20 nearly every world runs 20 sweeps in every setting, so the per-sweep solve time isolates the
cost of the Coulomb twins of the solve kernel."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

WORKLOADS = {"c3": ("pile64", 65536, 1024), "c5": ("legged20", 131072, 0)}


def gpu_info(torch):
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info.update(power_limit_w=float(q[0]), sm_max_mhz=float(q[1]))
    except Exception as e:   # the numbers stay valid without it; say why the limit is missing
        info["power_limit_w"] = f"unavailable: {e}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r3h_coulomb_friction.json")
    ap.add_argument("--steps", type=int, default=3, help="timed steps per setting and round")
    ap.add_argument("--reps", type=int, default=2, help="rounds over the three settings")
    ap.add_argument("--workloads", default="c3,c5")
    args = ap.parse_args()
    import torch
    import eggshell_b200 as E
    if not torch.cuda.is_available():
        raise SystemExit("friction_bench.py needs a CUDA device")
    res = {"gpu": gpu_info(torch), "steps": args.steps, "reps": args.reps, "runs": []}
    for wl in args.workloads.split(","):
        fn, W, maxc = WORKLOADS[wl]
        scene = getattr(E.scenes, fn)(W)
        settings = [("box", None), ("coulomb_0.5", 0.5), ("coulomb_U[0.2,1.0]", np.random.default_rng(0).uniform(0.2, 1.0, size=W))]
        for k_max in (500, 20):
            b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=k_max, max_contacts=maxc)
            stream = torch.cuda.current_stream()
            b.set_stream(stream.cuda_stream)
            b.snapshot()
            acc = {name: {"ms": [], "solve_ms": [], "sweeps_mean": [], "sweeps_max": []} for name, _ in settings}
            for _ in range(args.reps):
                for name, mu in settings:
                    b.set_friction(mu)
                    b.restore(); b.step(scene["dt"])   # warm-up of this instance
                    b.sync()
                    b.set_profiling(True); b.kernel_ms()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    for _ in range(args.steps):
                        b.restore()
                        b.step(scene["dt"])
                    e1.record(stream)
                    torch.cuda.synchronize()
                    kms = b.kernel_ms()
                    b.set_profiling(False)
                    st = b.status()
                    assert int(np.bitwise_or.reduce(st["status"])) == 0, (wl, k_max, name)
                    a = acc[name]
                    a["ms"].append(e0.elapsed_time(e1) / args.steps)
                    a["solve_ms"].append(kms[2] / max(kms[3], 1.0))
                    a["sweeps_mean"].append(float(st["sweeps"].mean()))
                    a["sweeps_max"].append(int(st["sweeps"].max()))
            b.close()
            for name, _ in settings:
                a = acc[name]
                ms, solve = float(np.median(a["ms"])), float(np.median(a["solve_ms"]))
                sw = float(np.mean(a["sweeps_mean"]))
                run = {"workload": wl, "scene": fn, "worlds": W, "k_max": k_max, "friction": name,
                       "world_steps_per_s": W / (ms * 1e-3), "ms_per_step": ms, "ms_per_step_rounds": a["ms"],
                       "sweeps_mean": sw, "sweeps_max": max(a["sweeps_max"]),
                       "solve_ms_per_step": solve, "solve_ms_per_step_rounds": a["solve_ms"], "solve_ms_per_sweep": solve / max(sw, 1e-9)}
                res["runs"].append(run)
                print(json.dumps(run), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
