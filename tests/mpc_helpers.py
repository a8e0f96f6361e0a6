"""Helpers shared by the MPC tests: bit views, device copies, state rows, the error code of a refused
call, batches on torch's current stream, multi-rank runs, and the numpy definitions of the MPPI
noise and of the zero-gravity reaching task that the MPPI and CEM tests share."""
import os
import re
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from eggshell_b200 import SOLVER_PGS, mpc

S = mpc.STATE_PER_BODY
M32 = np.uint64(0xffffffff)


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def state_rows(b):
    """bodies() as [W, n, 18] rows (p, R row-major, v, w)."""
    p, R, v, w = b.bodies()
    W, n = p.shape[:2]
    return np.concatenate([p, R.reshape(W, n, 9), v, w], axis=-1)


def err_code(excinfo):
    """The C ABI's return code in the EggError of a refused call."""
    return int(re.search(r"failed \((-?\d+)\)", str(excinfo.value)).group(1))


def batch_on_current_stream(scene, defaults=None, **kw):
    """A batch on torch's current stream, so that torch-side buffers and the batch's kernels are
    ordered.  defaults: make_batch keywords that kw overrides."""
    import eggshell_b200 as E
    b = E.scenes.make_batch(scene, **dict(defaults or {}, **kw))
    b.set_stream(torch.cuda.current_stream().cuda_stream)
    return b


def _rank_main(target, rank, world_size, backend, port, args, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    if backend == "nccl":
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world_size, device_id=torch.device("cuda", rank))
    else:
        dist.init_process_group(backend, rank=rank, world_size=world_size)
    q.put((rank, target(rank, world_size, *args)))
    dist.barrier()
    dist.destroy_process_group()


def run_ranks(target, world_size, backend, *args, timeout):
    """target(rank, world_size, *args) in world_size spawned processes that form a `backend` process
    group (nccl: rank r on cuda:r).  target must be a module-level function, so that spawn can pickle
    it.  Returns what each rank returned, in rank order."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = free_port()
    procs = [ctx.Process(target=_rank_main, args=(target, r, world_size, backend, port, args, q)) for r in range(world_size)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=timeout) for _ in range(world_size))
    for p in procs:
        p.join(timeout=timeout)
        assert p.exitcode == 0
    return [res[r] for r in range(world_size)]


# ---- MPPI and CEM: the numpy definition of the noise, and the reaching task -----------------------
def philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al., SC'11) on arrays: ctr [4, ...], key [2, ...] of uint32 values.
    Returns the four output words as uint64 arrays holding uint32 values."""
    c = [np.asarray(x, dtype=np.uint64) & M32 for x in ctr]
    k = [np.asarray(x, dtype=np.uint64) & M32 for x in key]
    for r in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [((p1 >> np.uint64(32)) ^ c[1] ^ k[0]) & M32, p1 & M32, ((p0 >> np.uint64(32)) ^ c[3] ^ k[1]) & M32, p0 & M32]
        k = [(k[0] + np.uint64(0x9E3779B9)) & M32, (k[1] + np.uint64(0xBB67AE85)) & M32]
    return c


def _u01(lo, hi):
    x = (hi << np.uint64(32)) | lo
    return (x >> np.uint64(11)).astype(np.float64) * 2.0 ** -53 + 2.0 ** -54


def noise(H, n, g, seed, iteration):
    """eps [H, len(g), n, 6] of the global worlds g, as egg_sample_controls defines it."""
    t, w, b, p = np.meshgrid(np.arange(H), np.arange(len(g)), np.arange(n), np.arange(3), indexing="ij")
    q = ((t * n + b) * 3 + p).astype(np.uint64)
    gg = np.asarray(g, dtype=np.uint64)[w]
    c = philox4x32_10([q, gg, np.uint64(iteration & 0xffffffff), np.uint64(iteration >> 32)],
                      [np.uint64(seed & 0xffffffff), np.uint64(seed >> 32)])
    u1, u2 = _u01(c[0], c[1]), _u01(c[2], c[3])
    r = np.sqrt(-2.0 * np.log(u1))
    eps = np.stack([r * np.cos(2 * np.pi * u2), r * np.sin(2 * np.pi * u2)], axis=-1)   # [H, W, n, 3, 2]
    return eps.reshape(H, len(g), n, 6)


def clamp(v, lo, hi):
    return np.where(v < lo, lo, np.where(v > hi, hi, v))


ZERO_G_PGS = dict(solver=SOLVER_PGS, gravity=(0.0, 0.0, 0.0))   # the batch_on_current_stream defaults for boxes


def boxes(W, n, seed=0, dt=0.05):
    """n unit-mass boxes per world in zero gravity, 2 m apart and 10 m above the ground (no contacts)."""
    import eggshell_b200 as E
    s = E.scenes._base(W, n)
    rng = np.random.default_rng(seed)
    s["p"][:, :, 0] = 2.0 * np.arange(n)
    s["p"][:, :, 2] = 10.0
    s["p"] += rng.uniform(-0.1, 0.1, size=s["p"].shape)
    s.update(dt=dt, name=f"boxes{n}")
    return s


def reach_cost(x0, target):
    """Terminal cost |p - target|^2 of the single body."""
    q_term = np.zeros((1, S))
    q_term[0, 0:3] = 1.0
    x_ref = x0.copy()
    x_ref[0, 0:3] = target
    return mpc.QuadraticCost(1, q_term=q_term, x_ref=x_ref)


def costs_of(b, u, H, dt):
    c = torch.empty(b.W, dtype=torch.float64, device="cuda")
    b.restore()
    b.step_controlled_cost(dt, u.data_ptr(), H, c.data_ptr())
    return c.cpu().numpy()
