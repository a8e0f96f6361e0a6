"""Multi-GPU host logic: contiguous world shards and the one collective of the path — an allgather
of per-rollout costs followed by an identical arg-min / top-k on every rank (SURVEY.md §8e) — and
the receding-horizon loop built on it: the winners' terminal states are gathered from their owner
ranks and re-seed every world for the next horizon (`mpc_iteration`).

Worlds are independent (the reference already steps two unrelated ensembles per SimulationStep,
/root/reference/eggshell/model.cc:67-68), so there is no data-path exchange inside a horizon."""
import numpy as np

STATE_PER_BODY = 18   # p(3), R(9, row-major), v(3), w(3): a row of egg_gather_state / egg_seed_state
CONTROL_PER_BODY = 6  # f(3), tau(3): a row of egg_set_external / a control schedule slice


class QuadraticCost:
    """A quadratic running + terminal cost over a controlled horizon, shared by all worlds
    (Batch.set_cost, egg_set_cost).  With x_t [n, 18] the state before step t, x_H the state after
    the last step, u_t [n, 6] the control of step t and d_t = x_t - x_ref[t]:

        J = sum_{t<H} sum_b [ sum_c q_run[b,c] d_t[b,c]^2 + l_run[b,c] d_t[b,c] + sum_j u_run[b,j] u_t[b,j]^2 ]
          +           sum_b   sum_c q_term[b,c] d_H[b,c]^2 + l_term[b,c] d_H[b,c]

    The weights broadcast to [n, 18] ([n, 6] for u_run); x_ref broadcasts to [n, 18] (one reference
    for every step) or is [ref_steps, n, 18] with ref_steps >= H + 1 (row t for step t).  The linear
    terms express progress: l_term[0, 0] = -1 rewards body 0 for moving along +x.  Every value must
    be finite."""

    def __init__(self, n, q_run=0.0, l_run=0.0, u_run=0.0, q_term=0.0, l_term=0.0, x_ref=0.0):
        n = int(n)
        if n < 1:
            raise ValueError("QuadraticCost: n must be >= 1")
        self.n = n
        S, U = STATE_PER_BODY, CONTROL_PER_BODY
        self.q_run, self.l_run, self.q_term, self.l_term = (self._arr(a, (n, S), name) for a, name in
                                                            ((q_run, "q_run"), (l_run, "l_run"), (q_term, "q_term"), (l_term, "l_term")))
        self.u_run = self._arr(u_run, (n, U), "u_run")
        x = np.asarray(x_ref, dtype=np.float64)
        if x.ndim == 3:
            if x.shape[0] < 1:
                raise ValueError("QuadraticCost: x_ref needs ref_steps >= 1 rows")
            self.x_ref = self._arr(x, (x.shape[0], n, S), "x_ref")
        elif x.ndim <= 2:
            self.x_ref = self._arr(x, (1, n, S), "x_ref")
        else:
            raise ValueError(f"QuadraticCost: x_ref must broadcast to [{n}, {S}] or be [ref_steps, {n}, {S}]")
        self.ref_steps = self.x_ref.shape[0]

    @staticmethod
    def _arr(a, shape, name):
        a = np.asarray(a, dtype=np.float64)
        try:
            a = np.ascontiguousarray(np.broadcast_to(a, shape))
        except ValueError:
            raise ValueError(f"QuadraticCost: {name} of shape {a.shape} does not broadcast to {list(shape)}") from None
        if not np.isfinite(a).all():
            raise ValueError(f"QuadraticCost: {name} has non-finite values")
        return a

    def evaluate(self, states, u):
        """The float64 numpy reference of J: states [H + 1, W, n, 18] (x_0 ... x_H), u [H, W, n, 6].
        Returns J [W]."""
        states, u = np.asarray(states, dtype=np.float64), np.asarray(u, dtype=np.float64)
        if u.ndim != 4 or u.shape[0] < 1 or u.shape[2:] != (self.n, CONTROL_PER_BODY):
            raise ValueError(f"u must be [H >= 1, W, {self.n}, {CONTROL_PER_BODY}]")
        H, W = u.shape[:2]
        if states.shape != (H + 1, W, self.n, STATE_PER_BODY):
            raise ValueError(f"states must be [{H + 1}, {W}, {self.n}, {STATE_PER_BODY}] for a horizon of {H}")
        if 1 < self.ref_steps < H + 1:
            raise ValueError(f"the reference has {self.ref_steps} rows, fewer than H + 1 = {H + 1}")
        ref = self.x_ref[np.minimum(np.arange(H + 1), self.ref_steps - 1)]   # [H + 1, n, 18]
        d = states - ref[:, None]
        run = (self.q_run * d[:H] ** 2 + self.l_run * d[:H]).sum(axis=(0, 2, 3)) + (self.u_run * u ** 2).sum(axis=(0, 2, 3))
        return run + (self.q_term * d[H] ** 2 + self.l_term * d[H]).sum(axis=(1, 2))


def shard_range(n_worlds_total, rank, world_size):
    """Contiguous slice [lo, hi) of the global world index space owned by `rank`."""
    base, rem = divmod(int(n_worlds_total), int(world_size))
    lo = rank * base + min(rank, rem)
    hi = lo + base + (1 if rank < rem else 0)
    return lo, hi


def allgather_costs(local_costs):
    """local_costs: 1-D torch tensor (CPU/gloo or CUDA/nccl).  Returns the concatenation over ranks
    in rank order.  Uneven shards are padded to the longest one."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return local_costs.clone()
    ws = dist.get_world_size()
    n = torch.tensor([local_costs.numel()], dtype=torch.int64, device=local_costs.device)
    sizes = [torch.zeros_like(n) for _ in range(ws)]
    dist.all_gather(sizes, n)
    sizes = [int(s.item()) for s in sizes]
    m = max(sizes)
    if all(s == m for s in sizes):
        out = torch.empty(ws * m, dtype=local_costs.dtype, device=local_costs.device)
        dist.all_gather_into_tensor(out, local_costs.contiguous())
        return out
    pad = torch.full((m,), float("inf"), dtype=local_costs.dtype, device=local_costs.device)
    pad[: local_costs.numel()] = local_costs
    out = torch.empty(ws * m, dtype=local_costs.dtype, device=local_costs.device)
    dist.all_gather_into_tensor(out, pad)
    return torch.cat([out[r * m: r * m + sizes[r]] for r in range(ws)])


def select_best(all_costs, k=1):
    """Deterministic top-k (lowest cost, ties by lowest global world index) — identical on every rank."""
    c = np.asarray(all_costs.detach().cpu().numpy() if hasattr(all_costs, "detach") else all_costs, dtype=np.float64)
    order = np.lexsort((np.arange(c.size), c))
    return order[:k], c[order[:k]]


def owner_of(world_index, n_worlds_total, world_size):
    """(rank, local index) of a global world index under shard_range."""
    for r in range(world_size):
        lo, hi = shard_range(n_worlds_total, r, world_size)
        if lo <= world_index < hi:
            return r, world_index - lo
    raise IndexError(world_index)


def gather_winner_states(winners, n_total, pack):
    """Rows of the winning worlds, in `winners` order, identical on every rank: a [k, F] tensor.

    winners: global world indices (duplicates allowed), the same on every rank (select_best).
    pack(local_indices): this rank's rows for an int array of its local world indices, a [len, F]
    tensor on the device of the collective (an empty array gives a [0, F] tensor).  Each rank fills
    the slots of the winners it owns in a [world_size, k, F] buffer, one all_gather_into_tensor
    shares it, and every winner is read from its owner's slot: nothing is summed, so the rows
    (including -0.0) arrive bit for bit."""
    import torch
    import torch.distributed as dist
    winners = np.asarray(winners, dtype=np.int64).ravel()
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return pack(winners)
    rank, ws = dist.get_rank(), dist.get_world_size()
    owner = [owner_of(int(g), n_total, ws) for g in winners]
    mine = np.array([i for i, (r, _) in enumerate(owner) if r == rank], dtype=np.int64)
    rows = pack(np.array([owner[i][1] for i in mine], dtype=np.int64))
    k, F = winners.size, rows.shape[1]
    slot = torch.zeros((k, F), dtype=rows.dtype, device=rows.device)
    if mine.size:
        slot[torch.from_numpy(mine).to(rows.device)] = rows
    buf = torch.empty((ws * k, F), dtype=rows.dtype, device=rows.device)   # [world_size, k, F] (gloo wants it flat)
    dist.all_gather_into_tensor(buf, slot)
    src = torch.tensor([r for r, _ in owner], dtype=torch.int64, device=rows.device)
    return buf.view(ws, k, F)[src, torch.arange(k, device=rows.device)]


def mpc_iteration(batch, u, dt, k, n_total, first):
    """One receding-horizon iteration of a (sharded) random-shooting sweep.

    From the batch's snapshot, every world runs the control schedule u (a contiguous float64 CUDA
    tensor [H, W, n, 6] on the batch's device: slice t is the f_ext of step t); the per-world costs
    (the QuadraticCost of Batch.set_cost, accumulated over the horizon on the device, or without one
    the built-in egg_rollout_costs) are gathered over all ranks and the k best worlds win
    (select_best); their terminal states are fetched from their owner ranks; world w of this shard (global index first + w) is re-seeded from
    winner (first + w) % k and the seeded state is snapshotted as the next horizon's start.
    The batch must run on torch's current stream (Batch.set_stream), on which u is produced.
    Returns (winners, their costs, states [k, n * 18] float64 CUDA tensor)."""
    import torch
    dev = torch.device("cuda", int(batch.desc.device))
    if not (isinstance(u, torch.Tensor) and u.is_cuda and u.device == dev and u.dtype == torch.float64
            and u.is_contiguous() and u.dim() == 4 and u.shape[0] >= 1 and tuple(u.shape[1:]) == (batch.W, batch.n, 6)):
        raise ValueError(f"u must be a contiguous float64 tensor [H >= 1, {batch.W}, {batch.n}, 6] on {dev}")
    if batch.stream != torch.cuda.current_stream(dev).cuda_stream:
        raise ValueError("the batch must run on torch's current stream: Batch.set_stream(torch.cuda.current_stream().cuda_stream)")
    costs = torch.empty(batch.W, dtype=torch.float64, device=dev)
    batch.restore()
    if batch.cost is None:
        batch.step_controlled(dt, u.data_ptr(), u.shape[0])
        batch.rollout_costs(costs.data_ptr())
    else:
        batch.step_controlled_cost(dt, u.data_ptr(), u.shape[0], costs.data_ptr())
    winners, best = select_best(allgather_costs(costs), k)
    F = batch.n * STATE_PER_BODY

    def pack(local):
        out = torch.empty((len(local), F), dtype=torch.float64, device=dev)
        if len(local):
            batch.gather_state(local, out.data_ptr())
        return out

    states = gather_winner_states(winners, n_total, pack)
    batch.seed_state(states.data_ptr(), len(winners), first)
    batch.snapshot()
    return winners, best, states
