#!/usr/bin/env python
"""bench.py — world-steps/sec of the batched rigid-body step (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3] [--dump-outputs DIR]

One "step" = one Ensemble::Step (narrowphase -> rows -> PGS -> integrate) over every world of the
rank's batch.  Default workload = BASELINE.json configs[2], the configuration the metric's target
is quoted on ("64-body contact-rich stacks"): W worlds x 64-body pile per GPU, PGS with the
reference's termination (<= 500 sweeps, residual <= 1e-9, cfm 0.01), dt = 0.005, FP64.
Weak scaling: every rank owns the same number of worlds; the only collective is one NCCL
allgather of the per-world rollout costs at the end of the timed horizon.

Prints ONE JSON line on rank 0 (see the driver contract in the task statement).
`--impl reference` times the CPU restatement of the reference step (oracle/, kind "port": the
reference itself cannot be built here — Eigen/Qt/glog are absent) on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (scene fn name, kwargs, default worlds per GPU, description)
    "c2": ("stack10", {}, 4096, "4096 worlds x 10-box stack on ground plane, contact-only PGS"),
    "c3": ("pile64", {}, 65536, "65536 worlds x 64-body random box pile, contact-rich PGS"),
    # BASELINE.json configs[3]: the dense Schur + Murty solve of lcp.cc.  The timed state is the scene
    # after SETTLE["c4"] steps: the chain has landed and rests on ~47 ground contacts (~240 rows,
    # 96 of them equality rows), ~180 Murty pivots per step.
    "c4": ("chain32", {}, 16384, "16384 worlds x 32-link articulated chain (ball joints + ground contact), dense Schur + Murty LCP"),
    "c5": ("legged20", {}, 131072, "worlds x 20-body legged ensemble (19 ball joints + foot contacts), PGS"),
    # MPC rollout sweep (BASELINE.json configs[4]): a timed "step" = one 50-step horizon from the
    # common start state (egg_restore + 50 x egg_step, state evolving inside the horizon) followed
    # by the cost kernel and the one NCCL allgather; value counts every world-step of the horizon.
    "c5mpc": ("legged20", {}, 131072, "MPC rollout sweep: worlds x 20-body legged ensemble, 50-step horizons, cost allgather"),
}
HORIZON = {"c5mpc": 50}
SETTLE = {"c4": 4}            # steps taken from the scene's start state before the snapshot that every timed step restores
DENSE = {"c4"}                # workloads on the reference's default dense solver (solver 0); the others use PGS (solver 1)
FIXED_K = 20
FLOPS_PER_ROW_UPDATE = 54.0   # SURVEY.md §8(d)
ROW_STREAM_BYTES = 208.0      # bytes of one 3-row block streamed from HBM per Gauss-Seidel pass: 176 B record + 32 B multipliers
DUMP_WORLDS = 4096            # --dump-outputs: worlds sampled (seed 0) when the batch is larger; 4096 x 64 bodies x 18 doubles = 38 MB
DUMP_MAX_BYTES = 64 << 20


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--worlds", type=int, default=0, help="worlds per GPU (0 = the workload's default)")
    ap.add_argument("--k-max", type=int, default=500)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU-baseline sample time")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fixed-k", action="store_true", help="skip the extra fixed-K (K = 20) measurement of the PGS workloads (and the strong-scaling extra of c3)")
    ap.add_argument("--no-evolving", action="store_true", help="skip the extra evolving-state measurement (the batch stepped on without restore)")
    ap.add_argument("--precision", type=int, default=64, choices=[64, 32], help="32 = opt-in FP32 constraint records (not the headline)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (body state, status, rollout cost) of a fixed "
                         "seeded sample of rank 0's worlds as DIR/<name>.npy in float64, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs is not None and (args.impl != "ours" or args.steps < 1):
        ap.error("--dump-outputs needs --impl ours and --steps >= 1")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


def scene_for(args, W, rank):
    import eggshell_b200 as E
    fn, kw, _, _ = WORKLOADS[args.workload]
    base = {"stack10": 1000, "pile64": 3000, "legged20": 5000, "chain32": 4000}[fn]
    return getattr(E.scenes, fn)(W, seed=[base, rank], **kw)


# ------------------------------------------------------------------------------------------------
# CPU reference arm (oracle port) — the only place bench.py executes oracle/.
def cpu_reference(args, cores, seconds, steps_per_sample=1):
    """Times the CPU port of Ensemble::Step on `cores` threads over a bounded sample of the same
    workload.  Returns dict(value, unit, cores, kind, sample, rows_per_s)."""
    from oracle import pyoracle as O
    from tests.helpers import oracle_world
    fn, kw, _, _ = WORKLOADS[args.workload]
    solver = 0 if args.workload in DENSE else 1
    settle = SETTLE.get(args.workload, 0)
    # calibrate with one world-step on one thread
    sc = scene_for(args, 1, 0)
    w0, _ = oracle_world(sc, 0, solver=solver, k_max=args.k_max)
    for _ in range(settle):
        w0.step(sc["dt"])
    t0 = time.perf_counter()
    w0.step(sc["dt"])
    t1 = time.perf_counter() - t0
    per_core = max(1, int(seconds / max(t1, 1e-6) / max(steps_per_sample, 1)))
    per_core = min(per_core, 4096)
    nw = per_core * cores
    sc = scene_for(args, nw, 0)
    worlds = [oracle_world(sc, w, solver=solver, k_max=args.k_max)[0] for w in range(nw)]
    if settle:                            # untimed: bring the sample to the state the GPU arm is timed on
        O.batch_step(worlds, sc["dt"], settle, cores)
    sec, rows_sweeps, rows = O.batch_step(worlds, sc["dt"], steps_per_sample, cores)
    ws = nw * steps_per_sample
    return dict(value=ws / sec, unit="world-steps/s", cores=cores, kind="port",
                sample=f"{nw} worlds x {steps_per_sample} step(s) of {WORKLOADS[args.workload][3]} on {cores} host threads "
                       f"({sec:.2f} s{', after %d untimed settling steps' % settle if settle else ''}); oracle/ = Eigen-free restatement of the reference step, g++ -O2 -march=native",
                rows_per_s=rows_sweeps / sec, seconds=sec, world_steps=ws)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import pyoracle as O
    cores = O.hardware_concurrency() or os.cpu_count() or 1
    total = args.steps + args.warmup
    per_step = max(2.0, min(20.0, 120.0 / max(total, 1)))
    # warm-up samples (untimed), then K timed samples
    hz = HORIZON.get(args.workload, 1)
    for _ in range(min(args.warmup, 1)):
        cpu_reference(args, cores, 1.0, hz)
    vals, sec, ws, rps = [], 0.0, 0, 0.0
    res = None
    for _ in range(args.steps):
        res = cpu_reference(args, cores, per_step, hz)
        sec += res["seconds"]
        ws += res["world_steps"]
        rps += res["rows_per_s"] * res["seconds"]
    value = ws / sec
    fn, kw, Wd, desc = WORKLOADS[args.workload]
    line = {
        "impl": "reference", "metric": "world-steps/sec", "value": value, "unit": "world-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sec / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {desc}", "solver": "dense-murty" if args.workload in DENSE else "pgs", "k_max": args.k_max, "tol": 1e-9, "cfm": 0.01,
                   "inputs": "bounded CPU sample of the same workload per step (same scene, same solver, same termination; fewer worlds)"},
        "cpu_baseline": {"value": value, "unit": "world-steps/s", "cores": cores, "kind": "port", "sample": res["sample"]},
        "pgs_rows_per_s": rps / sec,
        "e2e": {"value": value, "unit": "world-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def dump_outputs(path, b, st, costs):
    """Writes what a caller of the timed step receives -- egg_get_bodies (p, R, v, w), egg_get_status
    and the rollout cost of every world -- for a fixed seeded sample of the batch's worlds, as float64
    DIR/<name>.npy.  The scene is seeded, so the same arguments give the same inputs on every run."""
    W = b.W
    idx = np.arange(W) if W <= DUMP_WORLDS else np.sort(np.random.default_rng(0).choice(W, DUMP_WORLDS, replace=False))
    out = dict(zip(("p", "R", "v", "w"), b.bodies()))
    out.update(st)
    out["cost"] = costs
    out = {k: np.ascontiguousarray(a[idx], dtype=np.float64) for k, a in out.items()}
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_MAX_BYTES, f"--dump-outputs would write {total} bytes"
    os.makedirs(path, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(path, k + ".npy"), a)
    print(f"bench.py: wrote {len(out)} arrays ({total} bytes, {len(idx)} of {W} worlds) to {path}", file=sys.stderr)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                       "-i", str(self.index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.f.read().splitlines():
            c = [x.strip() for x in ln.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); power.append(float(c[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(power)),
                "samples": len(sm), "reasons": sorted(reasons)}


def run_ours(args):
    import torch
    import torch.distributed as dist
    import eggshell_b200 as E

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: eggshell_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG=VERSION prints "NCCL version ..." on stdout; rank 0's stdout must be ONE JSON line
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    fn, kw, Wd, desc = WORKLOADS[args.workload]
    W = args.worlds or Wd
    scene = scene_for(args, W, rank)
    n, nj, dt = scene["n"], scene["nj"], scene["dt"]
    maxc = {"c3": 1024}.get(args.workload, 0)
    horizon = HORIZON.get(args.workload, 1)
    dense = args.workload in DENSE
    b = E.scenes.make_batch(scene, solver=E.SOLVER_DENSE_MURTY if dense else E.SOLVER_PGS, k_max=args.k_max, max_contacts=maxc,
                            device=local, precision=args.precision)
    stream = torch.cuda.current_stream()
    b.set_stream(stream.cuda_stream)
    costs = torch.zeros(W, dtype=torch.float64, device="cuda")
    all_costs = torch.zeros(W * world, dtype=torch.float64, device="cuda") if world > 1 else costs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # Every step starts from the named scene's state (device-resident snapshot), so all K steps
    # do the same work: step = egg_restore (D2D, inside the timed region) + egg_step.
    settle = SETTLE.get(args.workload, 0)
    if settle:
        b.step(dt, n_steps=settle)
    b.snapshot()
    # ---- warm-up ----
    for _ in range(max(args.warmup, 0)):
        b.restore()
        b.step(dt, n_steps=horizon)
    b.sync()
    b.set_profiling(True)
    b.kernel_ms()
    launches0 = b.launch_count

    # ---- timed region: K steps + cost kernel + the one collective ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        b.restore()
        b.step(dt, n_steps=horizon)
        if horizon > 1:                  # MPC: one cost kernel + one allgather per horizon
            b.rollout_costs(costs.data_ptr())
            if world > 1:
                dist.all_gather_into_tensor(all_costs, costs)
    if horizon == 1:
        b.rollout_costs(costs.data_ptr())
        if world > 1:
            dist.all_gather_into_tensor(all_costs, costs)
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    launches = b.launch_count - launches0
    kms = b.kernel_ms()
    b.set_profiling(False)
    st = b.status()
    rows_last = float(st["n_rows"].astype(np.float64).sum())
    sweeps_last = float((st["n_rows"].astype(np.float64) * st["sweeps"]).sum())
    contacts_mean = float(st["n_contacts"].mean())
    status_or = int(np.bitwise_or.reduce(st["status"]))
    best = float(all_costs.min().item())
    if args.dump_outputs is not None and rank == 0:   # before the end-to-end leg below overwrites the state
        dump_outputs(args.dump_outputs, b, st, costs.cpu().numpy())

    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = W * world * args.steps * horizon / (ms_max * 1e-3)

    # ---- end-to-end: host state in pinned memory -> H2D -> step -> D2H, every step ----
    # inputs = the scene's initial state in pinned host memory; outputs land in a second pinned set
    hin = (E.pinned_empty((W, n, 3)), E.pinned_empty((W, n, 3, 3)), E.pinned_empty((W, n, 3)), E.pinned_empty((W, n, 3)))
    hout = (E.pinned_empty((W, n, 3)), E.pinned_empty((W, n, 3, 3)), E.pinned_empty((W, n, 3)), E.pinned_empty((W, n, 3)))
    b.restore()
    b.bodies(out=hin)                    # the timed state (= the scene's start state unless the workload settles first)
    h2d = d2h = sum(x.nbytes for x in hin)
    for _ in range(1):
        b.set_state(*hin); b.step(dt, n_steps=horizon); b.bodies(out=hout)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record(stream)
    for _ in range(args.e2e_steps):
        b.set_state(*hin)                # egg_set_state: pinned host -> device (+ SoA pack kernels)
        b.step(dt, n_steps=horizon)      # egg_step (x horizon for the MPC workload)
        b.bodies(out=hout)               # egg_get_bodies: device -> pinned host (syncs)
    f1.record(stream)
    barrier()
    t2 = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = W * world * args.e2e_steps * horizon / (float(t2.item()) * 1e-3)

    dense_flops = float(b.dense_work().sum()) if dense else None

    # ---- evolving state: the same batch stepped on from the timed state WITHOUT restore, so the scene
    # relaxes / spreads as it would in a rollout (the headline restores the same start state before
    # every step: fixed work per step, the worst case for the contact-rich pile) ----
    evolving = None
    if horizon == 1 and not args.no_evolving:
        b.restore()
        barrier()
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0.record(stream)
        b.step(dt, n_steps=args.steps)
        h1.record(stream)
        barrier()
        t4 = torch.tensor([h0.elapsed_time(h1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t4, op=dist.ReduceOp.MAX)
        st4 = b.status()
        evolving = {"value": W * world * args.steps / (float(t4.item()) * 1e-3), "unit": "world-steps/s", "steps": args.steps,
                    "ms_per_step": float(t4.item()) / max(args.steps, 1), "mean_contacts_last_step": float(st4["n_contacts"].mean()),
                    "mean_sweeps_last_step": float(st4["sweeps"].mean()), "status_or": int(np.bitwise_or.reduce(st4["status"])),
                    "what": "the timed state stepped on without restore (contacts and sweeps change from step to step)"}

    # ---- fixed-K line (SURVEY 7: reference termination AND fixed-K throughput): the same workload
    # with the sweep count pinned to K = 20; parity at the same K: test_pgs_fixed_k20_stepwise ----
    fixed_k = None
    if not dense and args.k_max != FIXED_K and not args.no_fixed_k:
        b.close()
        b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=FIXED_K, max_contacts=maxc, device=local, precision=args.precision)
        b.set_stream(stream.cuda_stream)
        b.snapshot()
        for _ in range(3):
            b.restore(); b.step(dt, n_steps=horizon)
        b.sync()
        b.set_profiling(True); b.kernel_ms()
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record(stream)
        for _ in range(args.steps):
            b.restore(); b.step(dt, n_steps=horizon)
            if horizon > 1:                  # MPC: one cost kernel + one allgather per horizon, as in the headline
                b.rollout_costs(costs.data_ptr())
                if world > 1:
                    dist.all_gather_into_tensor(all_costs, costs)
        g1.record(stream)
        barrier()
        t3 = torch.tensor([g0.elapsed_time(g1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t3, op=dist.ReduceOp.MAX)
        k3 = b.kernel_ms()
        b.set_profiling(False)
        st3 = b.status()
        fixed_k = {"k": FIXED_K, "value": W * world * args.steps * horizon / (float(t3.item()) * 1e-3), "unit": "world-steps/s",
                   "ms_per_step": float(t3.item()) / max(args.steps, 1), "mean_sweeps": float(st3["sweeps"].mean()),
                   "kernel_ms_per_step": {"narrowphase": k3[0] / max(k3[3], 1.0), "assembly": k3[1] / max(k3[3], 1.0), "solve_integrate": k3[2] / max(k3[3], 1.0)},
                   "status_or": int(np.bitwise_or.reduce(st3["status"])), "parity": "tests/test_gpu_parity.py::test_pgs_fixed_k20_stepwise"}

    # ---- strong-scaling extra (BASELINE.json configs[2] read as "65536 worlds on 1/2/4/8 GPUs"): the
    # workload's single-GPU world count split over the ranks, same step, device-timed max over ranks ----
    strong = None
    if world > 1 and args.workload == "c3" and not args.no_fixed_k:
        Ws = max(1, Wd // world)
        b.close()
        sub = scene_for(args, Ws, rank)
        b = E.scenes.make_batch(sub, solver=E.SOLVER_PGS, k_max=args.k_max, max_contacts=maxc, device=local, precision=args.precision)
        b.set_stream(stream.cuda_stream)
        b.snapshot()
        for _ in range(2):
            b.restore(); b.step(dt)
        barrier()
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0.record(stream)
        for _ in range(args.steps):
            b.restore(); b.step(dt)
        h1.record(stream)
        barrier()
        t4 = torch.tensor([h0.elapsed_time(h1)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t4, op=dist.ReduceOp.MAX)
        strong = {"worlds_total": Ws * world, "worlds_per_gpu": Ws, "value": Ws * world * args.steps / (float(t4.item()) * 1e-3), "unit": "world-steps/s",
                  "ms_per_step": float(t4.item()) / max(args.steps, 1), "k_max": args.k_max}

    if rank == 0:
        pk, pk_kind = peaks()
        steps_counted = max(kms[3], 1.0)
        solve_ms = kms[2] / steps_counted
        bytes_step = E.scenes.algorithmic_bytes_per_world_step(n, nj)
        nc_mean = rows_last / W / 3.0
        # Dominant kernel = PGS solve + fused integrate (egg_pgs_stream_kernel).  Gauss-Seidel visits
        # every 3-row block once per pass: 208 B per block streamed from HBM (176 B record + 32 B
        # multipliers), and the multipliers go back (32 B) after every sweep.
        # Passes per world = sweeps + 2 (x0 scatter and the final read-only residual pass; probe
        # chunks, round headers and extra exact-residual passes are NOT counted: a lower bound).
        blocks_w = st["n_rows"].astype(np.float64) / 3.0
        sweeps_w = st["sweeps"].astype(np.float64)
        row_bytes = ROW_STREAM_BYTES if args.precision == 64 else 144.0   # 112 B record + 32 B multipliers
        stream_bytes = float((blocks_w * ((sweeps_w + 2.0) * row_bytes + sweeps_w * 32.0)).sum())
        solve_bytes = W * bytes_step + stream_bytes
        achieved = solve_bytes / (solve_ms * 1e-3) / 1e9
        traffic = None
        try:   # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this kernel at this config
            tr = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")))
            key = f"{args.workload}:{W}:{args.k_max}"
            traffic = tr.get(key, {}).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
        # SURVEY.md 8(d): two bounds for the dominant kernel, the larger fraction is the roofline.
        #   HBM : algorithmic bytes = W x B_step (state in/out, static data, joints, cost) per launch
        #   FP64: algorithmic flops = 54 per PGS row update x rows x sweeps (both counted by the kernel)
        # against the measured copy bandwidth (MEASURED_PEAKS.json) and a DFMA microbenchmark of this
        # run.  The kernel's own record stream (rows re-read every sweep) is NOT algorithmic traffic:
        # it is reported separately as roofline_stream / wasted_traffic.
        try:
            fp64_peak = E.batch.fp64_peak_tflops(local)
        except Exception:
            fp64_peak = None
        flops = dense_flops if dense else FLOPS_PER_ROW_UPDATE * sweeps_last
        algo_bytes = float(W * bytes_step)
        hbm_ach = algo_bytes / (solve_ms * 1e-3) / 1e9
        f64_ach = flops / (solve_ms * 1e-3) / 1e12
        hbm_frac = hbm_ach / pk["hbm_gbs"]
        f64_frac = (f64_ach / fp64_peak) if fp64_peak else None
        share = kms[2] / max(kms[0] + kms[1] + kms[2], 1e-9)
        kname = "egg_dense_kernel (cfm decision + Schur + Murty + fused integrate)" if dense else "egg_pgs_stream_kernel (PGS solve + fused integrate)"
        roof_hbm = {"bound": "hbm", "kernel": kname, "achieved": hbm_ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": hbm_frac,
                    "peak_source": "MEASURED_PEAKS.json hbm_gbs" if pk_kind == "measured" else "fallback 6650 GB/s (MEASURED_PEAKS.json absent)",
                    "algorithmic_bytes_per_launch": algo_bytes, "definition": "W x B_step, B_step = n(2*144+128) + 56 nj + 8 (SURVEY 8d)"}
        roof_f64 = {"bound": "fp64", "kernel": kname, "achieved": f64_ach, "peak": fp64_peak, "unit": "TFLOP/s", "frac": f64_frac,
                    "peak_source": "DFMA microbenchmark of this run (egg_fp64_peak_tflops); MEASURED_PEAKS.json has no FP64 entry",
                    "algorithmic_flops_per_launch": flops,
                    "definition": ("operations of the reference algorithm counted by the kernel per world (egg_get_dense_work): cfm-decision factorisation R^3/3, "
                                   "A_ee^-1 2E^3, Schur products, and per Murty pivot LDL^T k^3/3 + solves 2k^2 + w 2k(I-k)") if dense else
                                  "54 flop x rows x sweeps (SURVEY 8d), rows and sweeps counted by the kernel"}
        roof = dict(roof_f64 if (f64_frac is not None and f64_frac >= hbm_frac) else roof_hbm)
        roof.update({"traffic": traffic, "kernel_ms": solve_ms, "kernel_share_of_step": share})
        if traffic:
            roof["wasted_traffic"] = traffic / algo_bytes
        roof_other = roof_hbm if roof["bound"] == "fp64" else roof_f64
        # efficiency of the kernel on the traffic it chose to generate (every block streamed once per pass)
        roof_stream = None if dense else {"bound": "hbm", "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": achieved / pk["hbm_gbs"],
                       "stream_bytes_per_launch": solve_bytes, "stream_over_algorithmic": solve_bytes / algo_bytes,
                       "definition": "NOT the roofline: DRAM efficiency on the kernel's own record stream, W*B_step + sum_worlds blocks*((sweeps+2)*208 + sweeps*32) bytes (FP64 records)"}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            from oracle import pyoracle as O
            cpu = cpu_reference(args, O.hardware_concurrency() or 1, args.cpu_seconds, horizon)
            cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "rows_per_s")}
        line = {
            "metric": "world-steps/sec", "value": value, "unit": "world-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64" if args.precision == 64 else "f64 arithmetic, f32 constraint records", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {desc}", "worlds_per_gpu": W, "bodies": n, "joints": nj,
                       "solver": "dense-murty" if dense else "pgs", "k_max": args.k_max, "tol": 1e-9, "cfm": 0.01, "dt": dt, "horizon": horizon, "parallelism": f"worlds sharded x{world}",
                       "step": "every timed step = egg_restore(timed state, D2D) + egg_step: all steps do the same work",
                       "timed_state": ("scene after %d settling steps" % settle) if settle else "the scene's start state",
                       "mean_pivots": float(st["pivots"].mean()) if dense else None,
                       "l2": "inputs larger than L2 (state %.0f MB + rows %.0f MB per rank)" % (W * n * 34 * 8 / 1e6, W * nc_mean * 256 / 1e6),
                       "mean_contacts_per_world": contacts_mean, "mean_rows_per_world": rows_last / W,
                       "mean_sweeps": sweeps_last / max(rows_last, 1.0), "status_or": status_or, "best_cost": best},
            "pgs_rows_per_s": sweeps_last / (solve_ms * 1e-3),
            "kernel_ms_per_step": {"narrowphase": kms[0] / steps_counted, "assembly": kms[1] / steps_counted, "solve_integrate": solve_ms},
            "roofline": roof, "roofline_other_bound": roof_other, "roofline_stream": roof_stream, "cpu_baseline": cpu, "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "world-steps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "steps": args.e2e_steps, "api": "egg_set_state + egg_step + egg_get_bodies (pinned host buffers)"},
            "gpu_launches": int(launches),
        }
        if evolving is not None:
            line["evolving"] = evolving
        if fixed_k is not None:
            line["fixed_k"] = fixed_k
        if strong is not None:
            line["strong_scaling"] = strong
        emit(line)
    b.close()
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of rank 0, written to the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    # Libraries print to stdout on their own (torch's "NCCL version ..." banner at communicator
    # creation, for one): everything written to fd 1 from here on goes to stderr, and only emit()
    # writes to the original stdout.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
