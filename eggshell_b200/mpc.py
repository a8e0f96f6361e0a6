"""Multi-GPU host logic: contiguous world shards and the one collective of the path — an allgather
of per-rollout costs followed by an identical arg-min / top-k on every rank (SURVEY.md §8e) — and
the receding-horizon loop built on it: the winners' terminal states are gathered from their owner
ranks and re-seed every world for the next horizon (`mpc_iteration`) — and an MPPI planner on top of
the same pieces (`MPPI`, `mppi_iteration`, `mppi_advance`), and a cross-entropy-method planner whose
elites' schedules are exchanged like the winners' states (`CEM`, `cem_iteration`, `cem_advance`).

Worlds are independent (the reference already steps two unrelated ensembles per SimulationStep,
/root/reference/eggshell/model.cc:67-68), so there is no data-path exchange inside a horizon."""
import numpy as np

STATE_PER_BODY = 18   # p(3), R(9, row-major), v(3), w(3): a row of egg_gather_state / egg_seed_state
CONTROL_PER_BODY = 6  # f(3), tau(3): a row of egg_set_external / a control schedule slice


def _control_shape(n, m, owner):
    """(n, 6) body wrenches for m = None, else (m,) actuator values (m >= 1)."""
    if m is None:
        return (n, CONTROL_PER_BODY)
    m = int(m)
    if m < 1:
        raise ValueError(f"{owner}: m must be >= 1")
    return (m,)


def _broadcast(a, shape, owner, name, finite=False):
    """a as a contiguous float64 array of the given shape (numpy broadcasting); the errors name the
    owner class and the argument.  finite: refuse NaN and +-inf as well."""
    a = np.asarray(a, dtype=np.float64)
    try:
        a = np.ascontiguousarray(np.broadcast_to(a, shape))
    except ValueError:
        raise ValueError(f"{owner}: {name} of shape {a.shape} does not broadcast to {list(shape)}") from None
    if finite and not np.isfinite(a).all():
        raise ValueError(f"{owner}: {name} has non-finite values")
    return a


class Actuators:
    """An actuator table (Batch.set_actuators, egg_set_actuators): the batch's control row becomes the
    m actuator values.  Actuator a applies +tau_a to body[a] and -tau_a to reaction[a] (-1: none,
    else another body), tau_a = u_a k_a with k_a = axis[a] in the world frame (frame[a] = -1) or
    rotated by R of body frame[a] (body[a] or reaction[a]) in the state before the step.  axis[a] is
    used as given (its length is the gear ratio): finite and not all zero.  Invalid tables raise
    ValueError with the rules of the C ABI."""

    def __init__(self, n, body, reaction, frame, axis):
        n = int(n)
        if n < 1:
            raise ValueError("Actuators: n must be >= 1")
        body, reaction, frame = (np.asarray(x) for x in (body, reaction, frame))
        for x, name in ((body, "body"), (reaction, "reaction"), (frame, "frame")):
            if x.ndim != 1 or not (np.issubdtype(x.dtype, np.integer) or x.size == 0):
                raise ValueError(f"Actuators: {name} must be a 1-D integer array")
        m = body.size
        if m < 1:
            raise ValueError("Actuators: m must be >= 1")
        if reaction.size != m or frame.size != m:
            raise ValueError("Actuators: body, reaction and frame must have the same length")
        axis = np.asarray(axis, dtype=np.float64)
        if axis.shape != (m, 3):
            raise ValueError(f"Actuators: axis must be [{m}, 3]")
        if ((body < 0) | (body >= n)).any():
            raise ValueError("Actuators: body out of range")
        if ((reaction < -1) | (reaction >= n) | (reaction == body)).any():
            raise ValueError("Actuators: reaction must be -1 or another body")
        if ((frame != -1) & (frame != body) & (frame != reaction)).any():
            raise ValueError("Actuators: frame must be -1, body or reaction")
        if not np.isfinite(axis).all() or (axis == 0).all(axis=1).any():
            raise ValueError("Actuators: an axis must be finite and not zero")
        self.n, self.m = n, m
        self.body, self.reaction, self.frame = (np.ascontiguousarray(x, dtype=np.int32) for x in (body, reaction, frame))
        self.axis = np.ascontiguousarray(axis)

    @classmethod
    def ball_joint_motors(cls, n, i0, i1):
        """Three motors per ball joint with unit axes x, y, z: for a joint between bodies i0 and i1 the
        torque acts on the child i1 and reacts on the parent i0, in the parent's frame; a joint anchored
        to the world (i1 = -1) gives body i0, no reaction and world axes.  Motor 3 j + k is axis k of
        joint j."""
        i0, i1 = np.asarray(i0).ravel(), np.asarray(i1).ravel()
        body = np.repeat(np.where(i1 >= 0, i1, i0), 3)
        reaction = np.repeat(np.where(i1 >= 0, i0, -1), 3)
        frame = reaction.copy()
        axis = np.tile(np.eye(3), (i0.size, 1))
        return cls(n, body, reaction, frame, axis)

    def wrench(self, states, a, mass, gravity):
        """The float64 numpy transcription of the slot egg_set_actuators defines, in the same order:
        states [..., n, 18] (the state before the step), a [..., m] (actuator values), mass [..., n],
        gravity [3].  Returns f_ext [..., n, 6]: (m_b g, the actuator torques)."""
        states, a = np.asarray(states, dtype=np.float64), np.asarray(a, dtype=np.float64)
        mass, g = np.asarray(mass, dtype=np.float64), np.asarray(gravity, dtype=np.float64)
        lead = np.broadcast_shapes(states.shape[:-2], a.shape[:-1], mass.shape[:-1])
        if states.shape[-2:] != (self.n, STATE_PER_BODY) or a.shape[-1] != self.m or mass.shape[-1] != self.n or g.shape != (3,):
            raise ValueError(f"wrench takes states [..., {self.n}, {STATE_PER_BODY}], a [..., {self.m}], mass [..., {self.n}], gravity [3]")
        f = np.zeros(lead + (self.n, 6))
        f[..., :3] = mass[..., None] * g
        tq = np.zeros(lead + (self.n, 3))
        for k in range(self.m):
            ax, fr = self.axis[k], int(self.frame[k])
            if fr >= 0:
                R = states[..., fr, 3:12].reshape(states.shape[:-2] + (3, 3))
                ax = (R[..., :, 0] * ax[0] + R[..., :, 1] * ax[1]) + R[..., :, 2] * ax[2]
            tau = a[..., k, None] * ax
            tq[..., self.body[k], :] = tq[..., self.body[k], :] + tau
            if self.reaction[k] >= 0:
                tq[..., self.reaction[k], :] = tq[..., self.reaction[k], :] - tau
        f[..., 3:] = tq
        return f


class QuadraticCost:
    """A quadratic running + terminal cost over a controlled horizon, shared by all worlds
    (Batch.set_cost, egg_set_cost).  With x_t [n, 18] the state before step t, x_H the state after
    the last step, u_t [n, 6] the control of step t and d_t = x_t - x_ref[t]:

        J = sum_{t<H} sum_b [ sum_c q_run[b,c] d_t[b,c]^2 + l_run[b,c] d_t[b,c] + sum_j u_run[b,j] u_t[b,j]^2 ]
          +           sum_b   sum_c q_term[b,c] d_H[b,c]^2 + l_term[b,c] d_H[b,c]

    The weights broadcast to [n, 18] ([n, 6] for u_run); x_ref broadcasts to [n, 18] (one reference
    for every step) or is [ref_steps, n, 18] with ref_steps >= H + 1 (row t for step t).  The linear
    terms express progress: l_term[0, 0] = -1 rewards body 0 for moving along +x.  Every value must
    be finite.  With m given the cost is for a batch with an actuator table of m actuators: u_t is the
    [m] row of actuator values and u_run broadcasts to [m] (control_shape (m,))."""

    def __init__(self, n, q_run=0.0, l_run=0.0, u_run=0.0, q_term=0.0, l_term=0.0, x_ref=0.0, m=None):
        n = int(n)
        if n < 1:
            raise ValueError("QuadraticCost: n must be >= 1")
        self.n = n
        self.control_shape = _control_shape(n, m, "QuadraticCost")
        S = STATE_PER_BODY
        self.q_run, self.l_run, self.q_term, self.l_term = (_broadcast(a, (n, S), "QuadraticCost", name, finite=True) for a, name in
                                                            ((q_run, "q_run"), (l_run, "l_run"), (q_term, "q_term"), (l_term, "l_term")))
        self.u_run = _broadcast(u_run, self.control_shape, "QuadraticCost", "u_run", finite=True)
        x = np.asarray(x_ref, dtype=np.float64)
        if x.ndim == 3:
            if x.shape[0] < 1:
                raise ValueError("QuadraticCost: x_ref needs ref_steps >= 1 rows")
            self.x_ref = _broadcast(x, (x.shape[0], n, S), "QuadraticCost", "x_ref", finite=True)
        elif x.ndim <= 2:
            self.x_ref = _broadcast(x, (1, n, S), "QuadraticCost", "x_ref", finite=True)
        else:
            raise ValueError(f"QuadraticCost: x_ref must broadcast to [{n}, {S}] or be [ref_steps, {n}, {S}]")
        self.ref_steps = self.x_ref.shape[0]

    def evaluate(self, states, u):
        """The float64 numpy reference of J: states [H + 1, W, n, 18] (x_0 ... x_H), u [H, W, n, 6]
        ([H, W, m] with an actuator table).  Returns J [W]."""
        states, u = np.asarray(states, dtype=np.float64), np.asarray(u, dtype=np.float64)
        cs = self.control_shape
        if u.ndim != 2 + len(cs) or u.shape[0] < 1 or u.shape[2:] != cs:
            raise ValueError(f"u must be [H >= 1, W, {', '.join(map(str, cs))}]")
        H, W = u.shape[:2]
        if states.shape != (H + 1, W, self.n, STATE_PER_BODY):
            raise ValueError(f"states must be [{H + 1}, {W}, {self.n}, {STATE_PER_BODY}] for a horizon of {H}")
        if 1 < self.ref_steps < H + 1:
            raise ValueError(f"the reference has {self.ref_steps} rows, fewer than H + 1 = {H + 1}")
        ref = self.x_ref[np.minimum(np.arange(H + 1), self.ref_steps - 1)]   # [H + 1, n, 18]
        d = states - ref[:, None]
        run = (self.q_run * d[:H] ** 2 + self.l_run * d[:H]).sum(axis=(0, 2, 3)) + (self.u_run * u ** 2).sum(axis=(0,) + tuple(range(2, u.ndim)))
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
    sizes = allgather_rows(torch.tensor([local_costs.numel()], dtype=torch.int64, device=local_costs.device))[:, 0].tolist()
    m = max(sizes)
    if all(s == m for s in sizes):
        return allgather_rows(local_costs).view(-1)
    pad = torch.full((m,), float("inf"), dtype=local_costs.dtype, device=local_costs.device)
    pad[: local_costs.numel()] = local_costs
    out = allgather_rows(pad)
    return torch.cat([out[r, : sizes[r]] for r in range(len(sizes))])


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


def _packer(F, device, fill):
    """A `pack` for gather_winner_states: a float64 [len(local), F] tensor on device, written by
    fill(local, out_ptr) unless local is empty."""
    import torch

    def pack(local):
        out = torch.empty((len(local), F), dtype=torch.float64, device=device)
        if len(local):
            fill(local, out.data_ptr())
        return out
    return pack


def _checked_device(batch, u=None, horizon=None):
    """The batch's CUDA device, after the checks shared by the loops and planners: u, if given, is a
    contiguous float64 schedule [horizon, W, *batch.control_shape] on that device (any H >= 1 without a
    horizon), and the batch runs on torch's current stream."""
    import torch
    dev = torch.device("cuda", int(batch.desc.device))
    cs = batch.control_shape
    if u is not None and not (isinstance(u, torch.Tensor) and u.is_cuda and u.device == dev and u.dtype == torch.float64
                              and u.is_contiguous() and u.dim() == 2 + len(cs) and tuple(u.shape[1:]) == (batch.W,) + cs
                              and (u.shape[0] >= 1 if horizon is None else u.shape[0] == horizon)):
        H = "H >= 1" if horizon is None else horizon
        raise ValueError(f"u must be a contiguous float64 tensor [{H}, {batch.W}, {', '.join(map(str, cs))}] on {dev}")
    if batch.stream != torch.cuda.current_stream(dev).cuda_stream:
        raise ValueError("the batch must run on torch's current stream: Batch.set_stream(torch.cuda.current_stream().cuda_stream)")
    return dev


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
    dev = _checked_device(batch, u)
    costs = torch.empty(batch.W, dtype=torch.float64, device=dev)
    batch.restore()
    _rollout(batch, dt, u, costs)
    winners, best = select_best(allgather_costs(costs), k)
    states = gather_winner_states(winners, n_total, _packer(batch.n * STATE_PER_BODY, dev, batch.gather_state))
    batch.seed_state(states.data_ptr(), len(winners), first)
    batch.snapshot()
    return winners, best, states


class _SamplingPlan:
    """What the sampling planners share: a nominal schedule u_nom, float64 [horizon, *control_shape] on
    `device`, the sigma and bounds of a control row handed to Batch.set_sampler, the Philox seed and the
    iteration counter.  control_shape is (n, 6), or (m,) with m given (a batch with an actuator table).
    Validated here with the rules that MPPI documents."""

    def __init__(self, n, horizon, sigma, u_lo, u_hi, seed, u_nom, device, m):
        import torch
        name = type(self).__name__
        n, horizon = int(n), int(horizon)
        if n < 1 or horizon < 1:
            raise ValueError(f"{name}: n and horizon must be >= 1")
        U = self.control_shape = _control_shape(n, m, name)
        self.n, self.horizon = n, horizon
        self.sigma = _broadcast(sigma, U, name, "sigma")
        if not np.isfinite(self.sigma).all() or (self.sigma < 0).any():
            raise ValueError(f"{name}: sigma must be finite and >= 0")
        self.u_lo = None if u_lo is None else _broadcast(u_lo, U, name, "u_lo")
        self.u_hi = None if u_hi is None else _broadcast(u_hi, U, name, "u_hi")
        for a, what in ((self.u_lo, "u_lo"), (self.u_hi, "u_hi")):
            if a is not None and np.isnan(a).any():
                raise ValueError(f"{name}: {what} has NaN values")
        lo = np.full(U, -np.inf) if self.u_lo is None else self.u_lo
        hi = np.full(U, np.inf) if self.u_hi is None else self.u_hi
        if (lo > hi).any():
            raise ValueError(f"{name}: u_lo > u_hi")
        seed = int(seed)
        if not 0 <= seed < 2 ** 64:
            raise ValueError(f"{name}: seed must be in [0, 2^64)")
        self.seed = seed
        un = np.zeros((horizon,) + U) if u_nom is None else _broadcast(
            u_nom.detach().cpu().numpy() if isinstance(u_nom, torch.Tensor) else u_nom, (horizon,) + U, name, "u_nom", finite=True)
        self.device = torch.device(device)
        self.u_nom = torch.from_numpy(un.copy()).to(self.device)   # own storage: the iterations write to it
        self.lo = torch.from_numpy(np.array(lo)).to(self.device)   # the bounds as tensors (own copies), for clamp on the device
        self.hi = torch.from_numpy(np.array(hi)).to(self.device)
        self.iteration = 0

    def clamp(self, u):
        """u clamped to [u_lo, u_hi] (broadcast over leading dimensions)."""
        import torch
        return torch.clamp(u, min=self.lo, max=self.hi)


class MPPI(_SamplingPlan):
    """Planner state of MPPI (model predictive path integral): a nominal schedule u_nom, float64
    [horizon, n, 6] on `device`, improved by mppi_iteration and executed by mppi_advance.

    sigma: the standard deviation of the noise per body and control component, broadcast to [n, 6],
    finite and >= 0.  u_lo / u_hi: bounds of every sampled and nominal control, broadcast to [n, 6]
    (None = unbounded; +-inf allowed, NaN not; u_lo <= u_hi).  lam: the temperature lambda of the
    weights exp(-(J - J_min) / lam), finite and > 0.  seed: the Philox key, in [0, 2^64).  u_nom: the
    initial nominal schedule, broadcast to [horizon, n, 6] (default zeros), finite.  Hand the planner
    to Batch.set_sampler before mppi_iteration.  With m given the planner works in the control space of
    an actuator table of m actuators: sigma, u_lo and u_hi broadcast to [m] and u_nom to [horizon, m]."""

    def __init__(self, n, horizon, sigma, lam, u_lo=None, u_hi=None, seed=0, u_nom=None, device="cuda", m=None):
        lam = float(lam)
        if not (np.isfinite(lam) and lam > 0):
            raise ValueError("MPPI: lam must be finite and > 0")
        self.lam = lam
        super().__init__(n, horizon, sigma, u_lo, u_hi, seed, u_nom, device, m)


class CEM(_SamplingPlan):
    """Planner state of the cross-entropy method: a mean schedule u_nom and a per-step standard
    deviation std, both float64 [horizon, n, 6] on `device`, refitted to the n_elite cheapest rollouts
    by cem_iteration and executed by cem_advance.

    sigma: the initial standard deviation per body and control component, broadcast to [n, 6], finite
    and >= 0; std starts as sigma in every step, and the row that cem_advance appends takes it again.
    n_elite: the number of elites, >= 1 (at most the number of worlds of the sweep).  alpha: the
    smoothing of the refit, u_nom <- clamp(alpha u_nom + (1 - alpha) mean of the elites) and
    std <- max(alpha std + (1 - alpha) std of the elites, sigma_min); 0 <= alpha < 1.  sigma_min: a
    floor on std that keeps the search from collapsing, finite and >= 0.  u_lo, u_hi, seed and u_nom
    follow the rules of MPPI.  Hand the planner to Batch.set_sampler before cem_iteration.  With m given
    the planner works in the control space of an actuator table of m actuators, as MPPI does; std is
    then [horizon, m]."""

    def __init__(self, n, horizon, sigma, n_elite, alpha=0.0, sigma_min=0.0, u_lo=None, u_hi=None, seed=0, u_nom=None,
                 device="cuda", m=None):
        import torch
        n_elite, alpha, sigma_min = int(n_elite), float(alpha), float(sigma_min)
        if n_elite < 1:
            raise ValueError("CEM: n_elite must be >= 1")
        if not 0.0 <= alpha < 1.0:
            raise ValueError("CEM: alpha must be in [0, 1)")
        if not (np.isfinite(sigma_min) and sigma_min >= 0):
            raise ValueError("CEM: sigma_min must be finite and >= 0")
        self.n_elite, self.alpha, self.sigma_min = n_elite, alpha, sigma_min
        super().__init__(n, horizon, sigma, u_lo, u_hi, seed, u_nom, device, m)
        self.std = torch.tensor(np.broadcast_to(self.sigma, (self.horizon,) + self.control_shape), device=self.device)


def allgather_rows(x):
    """x: a 1-D tensor of the same length on every rank.  Returns [world_size, len] in rank order with
    one all_gather_into_tensor (x[None] without a process group)."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return x[None]
    ws = dist.get_world_size()
    out = torch.empty(ws * x.numel(), dtype=x.dtype, device=x.device)
    dist.all_gather_into_tensor(out, x.contiguous())
    return out.view(ws, x.numel())


def allgather_rank_sum(x):
    """The sum over ranks of x, added in rank order ((x_0 + x_1) + x_2 ...), so every rank holds the
    same bits whatever the collective's own reduction order would be."""
    rows = allgather_rows(x)
    acc = rows[0].clone()
    for r in range(1, rows.shape[0]):
        acc += rows[r]
    return acc


def _plan_check(batch, plan, u, first):
    """The checks of mppi_iteration and cem_iteration for a plan (MPPI or CEM) and a schedule buffer u."""
    import torch.distributed as dist
    dev = _checked_device(batch, u, plan.horizon)
    if batch.sampler is not plan:
        raise ValueError("the batch's sampler is not this planner: call Batch.set_sampler(mppi) first")
    if plan.u_nom.device != dev:
        raise ValueError(f"the planner's u_nom must live on {dev}")
    rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
    if (first == 0) != (rank == 0):
        raise ValueError("rank 0 must own global world 0 (first = 0 exactly on rank 0)")
    return dev


def _rollout(batch, dt, u, costs):
    """Every world runs the schedule u [H, W, n, 6] from the current state; costs [W] receives J from
    the batch's QuadraticCost (step_controlled_cost), or without one from the built-in cost
    (step_controlled + rollout_costs)."""
    if batch.cost is None:
        batch.step_controlled(dt, u.data_ptr(), u.shape[0])
        batch.rollout_costs(costs.data_ptr())
    else:
        batch.step_controlled_cost(dt, u.data_ptr(), u.shape[0], costs.data_ptr())


def mppi_sample(batch, mppi, u, first):
    """Step 1 of mppi_iteration without the restore: the perturbed schedules of this iteration into u."""
    batch.sample_controls(mppi.u_nom.data_ptr(), mppi.horizon, mppi.seed, mppi.iteration, first, u.data_ptr())


def mppi_combine(batch, mppi, u, costs):
    """Steps 3 to 6 of mppi_iteration, all on the device: the baseline and nominal cost, the weighted
    sums of this shard, their rank-order sum and the candidate nominal schedule.  Returns
    (candidate [H, *control_shape], stats [nominal J, min J, sum omega, sum omega^2]) without reading
    anything back."""
    import torch
    inf = torch.tensor(float("inf"), dtype=torch.float64, device=costs.device)
    local_min = torch.where(torch.isfinite(costs), costs, inf).min()
    g = allgather_rows(torch.stack([local_min, costs[0]]))   # [world_size, 2]; costs[0] of rank 0 is global world 0
    baseline = g[:, 0].min().contiguous()
    cs = batch.control_shape
    L = mppi.horizon * int(np.prod(cs))
    part = torch.empty(L + 2, dtype=torch.float64, device=costs.device)
    batch.mppi_reduce(u.data_ptr(), mppi.horizon, costs.data_ptr(), baseline.data_ptr(), mppi.lam, part.data_ptr())
    total = allgather_rank_sum(part)
    candidate = mppi.clamp(total[:L].view((mppi.horizon,) + cs) / total[L])
    return candidate, torch.stack([g[0, 1], baseline, total[L], total[L + 1]])


def mppi_iteration(batch, mppi, dt, u, first):
    """One MPPI iteration of a (sharded) sweep.  u is the caller's schedule buffer, a contiguous float64
    CUDA tensor [H, W, n, 6] on the batch's device, overwritten with this iteration's samples; first
    is the global index of local world 0 (0 on rank 0).  The batch must run on torch's current stream
    and sample with this planner (Batch.set_sampler(mppi)).

      1. restore the snapshot; sample W perturbed copies of u_nom into u (global world 0: u_nom itself);
      2. roll them out with the batch's QuadraticCost (step_controlled_cost), or without one with the
         built-in cost (step_controlled + rollout_costs);
      3. one allgather of [finite local min J, J of global world 0]: the baseline J_min (kept on the
         device) and the nominal schedule's cost;
      4. mppi_reduce: sum_w omega_w u_w, sum omega, sum omega^2 with omega = exp(-(J - J_min) / lam);
      5. one allgather of those partials, added in rank order (identical bits on every rank);
      6. u_nom <- clamp(sum omega u / sum omega);  7. iteration += 1.

    Reads back one small tensor.  Returns {nominal_cost, min_cost, weight_sum, ess} with
    ess = (sum omega)^2 / sum omega^2 the effective number of samples.  If no rollout finished with a
    finite cost (sum omega = 0) it raises and leaves u_nom and iteration unchanged."""
    import torch
    dev = _plan_check(batch, mppi, u, first)
    costs = torch.empty(batch.W, dtype=torch.float64, device=dev)
    batch.restore()
    mppi_sample(batch, mppi, u, first)
    _rollout(batch, dt, u, costs)
    candidate, stats = mppi_combine(batch, mppi, u, costs)
    nominal, jmin, wsum, w2 = stats.cpu().numpy().tolist()
    if not wsum > 0:
        raise RuntimeError(f"mppi_iteration: the weights sum to {wsum} (no rollout finished with a finite cost); u_nom is unchanged")
    mppi.u_nom.copy_(candidate)
    mppi.iteration += 1
    return {"nominal_cost": nominal, "min_cost": jmin, "weight_sum": wsum, "ess": wsum * wsum / w2}


def mppi_advance(batch, plan, dt, n_total):
    """Executes the plan's first control (plan: an MPPI or a CEM): from the snapshot every world takes
    one step with clamp(u_nom[0]); global world 0's new state re-seeds every world of every rank and
    becomes the snapshot, the start of the next horizon; u_nom shifts by one step (the last row
    repeats).  This costs one step of the whole batch, 1/H of a horizon.  Returns (the executed control
    [*control_shape], the new start rows [n, 18]), float64 CUDA tensors."""
    dev = _checked_device(batch)
    if plan.u_nom.device != dev:
        raise ValueError(f"the planner's u_nom must live on {dev}")
    u0 = plan.clamp(plan.u_nom[0])
    batch.restore()
    batch.step_controlled(dt, u0.expand((1, batch.W) + batch.control_shape).contiguous().data_ptr(), 1)
    state = gather_winner_states([0], n_total, _packer(batch.n * STATE_PER_BODY, dev, batch.gather_state))
    batch.seed_state(state.data_ptr(), 1, 0)
    batch.snapshot()
    if plan.horizon > 1:
        plan.u_nom[:-1] = plan.u_nom[1:].clone()
    return u0, state.view(batch.n, STATE_PER_BODY)


def cem_sample(batch, cem, u, first):
    """Step 2 of cem_iteration: the schedules of this iteration, clamp(u_nom + std eps), into u."""
    batch.sample_controls_std(cem.u_nom.data_ptr(), cem.std.data_ptr(), cem.horizon, cem.seed, cem.iteration, first, u.data_ptr())


def cem_select(cem, costs, n_total, pack):
    """Steps 4 and 5 of cem_iteration: the cost allgather, the n_elite cheapest rollouts among those
    with a finite cost (select_best: ties by the lowest global world index) and their schedules from
    their owner ranks (gather_winner_states with `pack`), so every rank holds the same rows, bit for
    bit, in elite order.  Returns (all costs, elite indices, elite costs, rows [n_elite, F]).  Raises
    before the exchange if fewer than n_elite rollouts finished with a finite cost."""
    import torch
    all_costs = allgather_costs(costs)
    finite = torch.where(torch.isfinite(all_costs), all_costs, torch.full_like(all_costs, float("inf")))
    elites, ecost = select_best(finite, cem.n_elite)
    n_finite = int(np.isfinite(ecost).sum())
    if n_finite < cem.n_elite:
        raise RuntimeError(f"cem_iteration: {n_finite} rollouts finished with a finite cost, fewer than n_elite = {cem.n_elite}; "
                           "the plan is unchanged")
    return all_costs, elites, ecost, gather_winner_states(elites, n_total, pack)


def cem_refit(cem, moments):
    """Step 7 of cem_iteration without committing it: from the elites' moments [2, H, n, 6] (mean,
    population std), the candidate (clamp(alpha u_nom + (1 - alpha) mean),
    max(alpha std + (1 - alpha) std_e, sigma_min)).  Elementwise, so every rank computes the same bits."""
    import torch
    a = cem.alpha
    u_nom = cem.clamp(a * cem.u_nom + (1.0 - a) * moments[0])
    std = torch.clamp(a * cem.std + (1.0 - a) * moments[1], min=cem.sigma_min)
    return u_nom, std


def cem_iteration(batch, cem, dt, u, first, n_total):
    """One CEM iteration of a (sharded) sweep of n_total worlds.  u is the caller's schedule buffer, a
    contiguous float64 CUDA tensor [H, W, n, 6] on the batch's device, overwritten with this
    iteration's samples; first is the global index of local world 0 (0 on rank 0).  The batch must run
    on torch's current stream and sample with this planner (Batch.set_sampler(cem)).

      1. restore the snapshot;  2. sample clamp(u_nom + std eps) into u (global world 0: clamp(u_nom));
      3. roll them out with the batch's QuadraticCost, or without one with the built-in cost;
      4. allgather the costs and pick the n_elite cheapest finite ones (identical on every rank);
      5. fetch the elites' schedules from their owner ranks (gather_winner_states, one allgather);
      6. control_moments: their mean and population std, computed identically on every rank;
      7. u_nom <- clamp(alpha u_nom + (1 - alpha) mean), std <- max(alpha std + (1 - alpha) std_e,
         sigma_min);  iteration += 1.

    Every rank holds the same plan bits, whatever the sharding.  Returns {nominal_cost, min_cost,
    elite_max_cost, mean_std}: the cost of global world 0 (the plan itself), the cheapest and the most
    expensive elite, and the mean of the new std.  If fewer than n_elite rollouts finished with a finite
    cost, or the refit is not finite, it raises and leaves the plan and iteration unchanged."""
    import torch
    dev = _plan_check(batch, cem, u, first)
    if cem.std.device != dev:
        raise ValueError(f"the planner's std must live on {dev}")
    H, cs = cem.horizon, batch.control_shape
    costs = torch.empty(batch.W, dtype=torch.float64, device=dev)
    batch.restore()
    cem_sample(batch, cem, u, first)
    _rollout(batch, dt, u, costs)
    pack = _packer(H * int(np.prod(cs)), dev, lambda local, out_ptr: batch.gather_controls(u.data_ptr(), H, local, out_ptr))
    all_costs, elites, ecost, rows = cem_select(cem, costs, n_total, pack)
    moments = torch.empty((2, H) + cs, dtype=torch.float64, device=dev)
    batch.control_moments(rows.contiguous().data_ptr(), len(elites), H, moments.data_ptr())
    u_nom, std = cem_refit(cem, moments)
    ok = torch.isfinite(u_nom).all() & torch.isfinite(std).all()
    nominal, mean_std, ok = torch.stack([all_costs[0], std.mean(), ok.double()]).cpu().numpy().tolist()
    if not ok:
        raise RuntimeError("cem_iteration: the refitted plan is not finite; the plan is unchanged")
    cem.u_nom.copy_(u_nom)
    cem.std.copy_(std)
    cem.iteration += 1
    return {"nominal_cost": nominal, "min_cost": float(ecost[0]), "elite_max_cost": float(ecost[-1]), "mean_std": mean_std}


def cem_advance(batch, cem, dt, n_total):
    """Executes the plan's first control with mppi_advance (every world steps with clamp(u_nom[0]) and
    is re-seeded from global world 0, u_nom shifts by one step), then shifts std by one step; its new
    last row is the initial sigma.  Returns what mppi_advance returns."""
    import torch
    executed = mppi_advance(batch, cem, dt, n_total)
    if cem.horizon > 1:
        cem.std[:-1] = cem.std[1:].clone()
    cem.std[-1] = torch.tensor(cem.sigma, device=cem.std.device)
    return executed
