"""CEM planner: egg_sample_controls_std (the sampler of egg_sample_controls with a per-step noise
scale), egg_gather_controls (the elites' schedules), egg_control_moments (their mean and standard
deviation) and mpc.CEM, cem_iteration and cem_advance.  The first tests run on the CPU; the rest need
a CUDA device."""
import numpy as np
import pytest
import torch

from eggshell_b200 import mpc
from tests.mpc_helpers import (ZERO_G_PGS, batch_on_current_stream, bits, boxes, clamp, costs_of, cuda, err_code, noise, reach_cost,
                               run_ranks, state_rows)

gpu = pytest.mark.gpu
S, U = mpc.STATE_PER_BODY, mpc.CONTROL_PER_BODY


# ---- the numpy definitions ------------------------------------------------------------------------
def moments_numpy(rows):
    """(mean, population std) of rows [k, ...] as egg_control_moments defines them: the rows added in
    row order and divided by k, then sqrt(sum (x - mean)^2 / k) in row order, each square rounded."""
    rows = np.asarray(rows, dtype=np.float64)
    k = rows.shape[0]
    s = np.zeros(rows.shape[1:])
    for r in rows:
        s = s + r
    mean = s / k
    q = np.zeros(rows.shape[1:])
    for r in rows:
        d = r - mean
        q = q + d * d
    return mean, np.sqrt(q / k)


def refit_numpy(u_nom, std, mean, std_e, alpha, sigma_min, lo, hi):
    """The update of cem_iteration: (clamp(alpha u_nom + (1 - alpha) mean), max(alpha std + (1 - alpha) std_e, sigma_min))."""
    return clamp(alpha * u_nom + (1.0 - alpha) * mean, lo, hi), np.maximum(alpha * std + (1.0 - alpha) * std_e, sigma_min)


def _np(t):
    return t.detach().cpu().numpy()


# ---- CPU ------------------------------------------------------------------------------------------
def test_cem_validates_and_broadcasts():
    c = mpc.CEM(3, 4, sigma=[0, 0, 0, 0.1, 0.2, 0.3], n_elite=5, alpha=0.25, sigma_min=0.01, u_hi=2.0,
                seed=2 ** 64 - 1, device="cpu")
    assert c.sigma.shape == (3, U) and (c.sigma[1] == [0, 0, 0, 0.1, 0.2, 0.3]).all()
    assert c.std.shape == (4, 3, U) and c.std.dtype == torch.float64 and c.std.is_contiguous()
    assert (_np(c.std) == np.broadcast_to(c.sigma, (4, 3, U))).all()
    c.std[0, 0, 5] = 9.0   # std is its own storage, not a view of sigma
    assert c.std[1, 0, 5] == 0.3 and c.sigma[0, 5] == 0.3
    assert c.u_lo is None and c.u_hi.shape == (3, U) and (c.u_hi == 2.0).all()
    assert c.u_nom.shape == (4, 3, U) and not c.u_nom.any()
    assert c.iteration == 0 and c.n_elite == 5 and c.alpha == 0.25 and c.sigma_min == 0.01 and c.horizon == 4
    c = mpc.CEM(2, 3, sigma=1.0, n_elite=1, u_lo=-1.0, u_hi=[1, 1, 1, 2, 2, 2], u_nom=np.arange(6.0), device="cpu")
    assert c.alpha == 0.0 and c.sigma_min == 0.0 and (_np(c.u_nom[2, 1]) == np.arange(6.0)).all()
    assert torch.equal(c.clamp(torch.full((3, 2, U), 5.0, dtype=torch.float64))[0, 0], torch.tensor([1.0, 1, 1, 2, 2, 2], dtype=torch.float64))
    bad = [dict(sigma=-0.1), dict(sigma=np.nan), dict(sigma=np.inf), dict(sigma=np.ones((3, U))), dict(sigma=np.ones(5)),
           dict(n_elite=0), dict(n_elite=-3),
           dict(alpha=-0.1), dict(alpha=1.0), dict(alpha=np.nan), dict(alpha=np.inf),
           dict(sigma_min=-1e-9), dict(sigma_min=np.nan), dict(sigma_min=np.inf),
           dict(u_lo=np.nan), dict(u_hi=[0, 0, 0, 0, 0, np.nan]), dict(u_lo=1.0, u_hi=0.0), dict(u_lo=np.ones((2, 2))),
           dict(seed=-1), dict(seed=2 ** 64), dict(u_nom=np.ones((2, 2, U))), dict(u_nom=np.nan), dict(u_nom=np.ones((4, 3, 2, U)))]
    for kw in bad:
        args = dict(sigma=1.0, n_elite=4, device="cpu")
        args.update(kw)
        with pytest.raises(ValueError):
            mpc.CEM(2, 3, **args)
    for n, H in ((0, 3), (2, 0)):
        with pytest.raises(ValueError):
            mpc.CEM(n, H, sigma=1.0, n_elite=4, device="cpu")


def test_moments_definition():
    rng = np.random.default_rng(4)
    rows = rng.normal(size=(37, 5, 2, U)) * 10.0 ** rng.integers(-6, 6, size=(1, 5, 2, U)) + rng.normal(size=(1, 5, 2, U))
    mean, std = moments_numpy(rows)
    scale = np.abs(rows).max(axis=0)
    assert np.all(np.abs(mean - rows.mean(axis=0)) <= 1e-14 * scale)
    assert np.all(np.abs(std - rows.std(axis=0)) <= 1e-14 * scale)
    m1, s1 = moments_numpy(rows[:1])
    assert np.array_equal(bits(m1), bits(rows[0])) and not s1.any()   # one row: itself, and std 0
    r = rows.copy()
    r[7, 1, 0, 2] = np.nan
    m, s = moments_numpy(r)
    assert np.isnan(m[1, 0, 2]) and np.isnan(s[1, 0, 2]) and np.isnan(m).sum() == 1 and np.isnan(s).sum() == 1
    # the refit of cem_iteration on a CPU planner against its numpy definition, bit for bit
    H, n = 5, 2
    c = mpc.CEM(n, H, sigma=rng.uniform(0.1, 1.0, size=(n, U)), n_elite=37, alpha=0.3, sigma_min=0.5, u_lo=-1.0, u_hi=1.0,
                u_nom=rng.uniform(-1.0, 1.0, size=(H, n, U)), device="cpu")
    un, sd = mpc.cem_refit(c, torch.from_numpy(np.stack([mean, std])))
    eu, es = refit_numpy(_np(c.u_nom), _np(c.std), mean, std, 0.3, 0.5, -1.0, 1.0)
    assert np.array_equal(bits(_np(un)), bits(eu)) and np.array_equal(bits(_np(sd)), bits(es))
    assert (_np(un) == 1.0).any() and (_np(un) == -1.0).any() and (_np(sd) == 0.5).any()   # both bounds and the floor reached


def _pool(N=41, H=4, n=2):
    """A fixed pool of N candidate schedules [N, H n 6] and their costs, some of them not finite."""
    rng = np.random.default_rng(77)
    rows = rng.normal(size=(N, H * n * U)) * 10.0 ** rng.integers(-4, 4, size=(1, H * n * U))
    cost = rng.uniform(0.0, 1.0, size=N)
    cost[[3, 20, 40]] = [np.nan, np.inf, -np.inf]
    cost[11] = cost[30] = 0.0   # the two cheapest tie: the lower global index comes first
    return rows, cost


def _refit_on_shard(rank, ws, n_elite=9):
    """cem_select and cem_refit of this rank's shard of the pool, with the numpy moments."""
    rows, cost = _pool()
    N, F = rows.shape
    lo, hi = mpc.shard_range(N, rank, ws)
    c = mpc.CEM(2, 4, sigma=0.5, n_elite=n_elite, alpha=0.2, sigma_min=0.1, u_lo=-3.0, u_hi=3.0, u_nom=0.25, device="cpu")
    local = rows[lo:hi]
    _, elites, ecost, got = mpc.cem_select(c, torch.from_numpy(cost[lo:hi].copy()), N, lambda i: torch.from_numpy(local[i]))
    mean, std = moments_numpy(got.numpy().reshape(n_elite, 4, 2, U))
    un, sd = mpc.cem_refit(c, torch.from_numpy(np.stack([mean, std])))
    return elites, ecost, got.numpy().copy(), _np(un).copy(), _np(sd).copy()


def test_refit_on_two_gloo_ranks_matches_one_rank():
    ws = 2
    res = run_ranks(_refit_on_shard, ws, "gloo", timeout=120)
    one = _refit_on_shard(0, 1)
    rows, cost = _pool()
    order = [i for i in np.lexsort((np.arange(cost.size), cost)) if np.isfinite(cost[i])][:9]
    assert list(one[0]) == order and order[:2] == [11, 30]
    assert np.array_equal(bits(one[2]), bits(rows[order]))
    for r in range(ws):
        assert list(res[r][0]) == order
        for a, b in zip(res[r][1:], one[1:]):
            assert np.array_equal(bits(np.asarray(a)), bits(np.asarray(b)))
    # fewer finite costs than elites: raises before the exchange
    with pytest.raises(RuntimeError, match="fewer than n_elite = 39"):
        _refit_on_shard(0, 1, n_elite=39)


# ---- GPU ------------------------------------------------------------------------------------------
def _plan(n, H, seed=7, **kw):
    rng = np.random.default_rng(seed)
    args = dict(sigma=rng.uniform(0.2, 1.0, size=(n, U)), n_elite=8, seed=0x1234_5678_9abc_def0,
                u_nom=rng.normal(0.0, 1.0, size=(H, n, U)))
    args.update(kw)
    return mpc.CEM(n, H, **args)


def _sample_std(b, c, std=None, first=0, iteration=None):
    u = torch.full((c.horizon, b.W, b.n, U), np.nan, dtype=torch.float64, device="cuda")
    std = c.std if std is None else std
    b.sample_controls_std(c.u_nom.data_ptr(), std.data_ptr(), c.horizon, c.seed, c.iteration if iteration is None else iteration,
                          first, u.data_ptr())
    return u.cpu().numpy()


def _sample(b, c, first=0, iteration=None):
    u = torch.full((c.horizon, b.W, b.n, U), np.nan, dtype=torch.float64, device="cuda")
    b.sample_controls(c.u_nom.data_ptr(), c.horizon, c.seed, c.iteration if iteration is None else iteration, first, u.data_ptr())
    return u.cpu().numpy()


@gpu
def test_std_sampler_with_a_constant_std_is_the_mppi_sampler():
    W, n, H, first = 300, 3, 4, 1000
    b = batch_on_current_stream(boxes(W, n), defaults=ZERO_G_PGS)
    rng = np.random.default_rng(9)
    lo, hi = rng.uniform(-1.5, -0.5, size=(n, U)), rng.uniform(0.5, 1.5, size=(n, U))
    c = _plan(n, H, u_lo=lo, u_hi=hi)
    b.set_sampler(c)
    for f, it in ((first, 2 ** 32 + 5), (0, 3)):
        got, ref = _sample_std(b, c, first=f, iteration=it), _sample(b, c, first=f, iteration=it)
        assert np.array_equal(bits(got), bits(ref)), (f, it)
        assert (got == lo).any() and (got == hi).any()
    b.close()


@gpu
def test_std_sampler_matches_numpy():
    W, n, H, first = 300, 3, 3, 1000
    b = batch_on_current_stream(boxes(W, n), defaults=ZERO_G_PGS)
    rng = np.random.default_rng(8)
    c = _plan(n, H)
    c.iteration = 2 ** 32 + 5   # both counter words of the iteration in use
    std = rng.uniform(0.2, 2.0, size=(H, n, U))
    b.set_sampler(c)
    u = _sample_std(b, c, std=cuda(std), first=first)
    eps = noise(H, n, np.arange(first, first + W), c.seed, c.iteration)
    got = (u - c.u_nom.cpu().numpy()[:, None]) / std[:, None]
    assert np.max(np.abs(got - eps)) <= 1e-13, np.max(np.abs(got - eps))
    assert np.abs(eps).max() > 3.0
    b.close()


@gpu
def test_std_sampler_exact_cases():
    W, n, H = 256, 2, 3
    b = batch_on_current_stream(boxes(W, n), defaults=ZERO_G_PGS)
    rng = np.random.default_rng(3)
    lo, hi = rng.uniform(-1.5, -0.5, size=(n, U)), rng.uniform(0.5, 1.5, size=(n, U))
    lo[0, 0], hi[1, 5] = -np.inf, np.inf
    un = rng.normal(0.0, 1.0, size=(H, n, U))
    un[0, 0, 1] = -0.0
    c = _plan(n, H, u_nom=un, u_lo=lo, u_hi=hi, sigma=0.0)   # the sampler's sigma is not used
    std = rng.uniform(0.5, 2.0, size=(H, n, U))
    std[1, 1, 3] = 0.0   # one element without noise
    b.set_sampler(c)
    sd = cuda(std)
    u = _sample_std(b, c, std=sd)
    c_nom = clamp(un, lo, hi)
    assert np.array_equal(bits(u[:, 0]), bits(c_nom)), "global world 0 runs clamp(mean)"
    assert np.array_equal(bits(u[1, :, 1, 3]), bits(np.full(W, c_nom[1, 1, 3]))), "std = 0 keeps clamp(mean)"
    assert (u >= lo).all() and (u <= hi).all()
    at_lo, at_hi = u == lo, u == hi
    assert at_lo.sum() > 100 and at_hi.sum() > 100
    eps = noise(H, n, np.arange(W), c.seed, c.iteration)
    free = clamp(un[:, None] + std[:, None] * eps, lo, hi)
    assert np.array_equal(at_lo[:, 1:], (free == lo)[:, 1:]) and np.array_equal(at_hi[:, 1:], (free == hi)[:, 1:])
    assert np.array_equal(bits(_sample_std(b, c, std=sd)), bits(u)), "two calls"
    # std = 0 everywhere: clamp(mean) in every world, bit for bit (-0.0 included)
    zero = torch.zeros((H, n, U), dtype=torch.float64, device="cuda")
    assert np.array_equal(bits(_sample_std(b, c, std=zero)), bits(np.broadcast_to(c_nom[:, None], (H, W, n, U))))
    # one batch of W against two batches of W / 2 with first = 0 and first = W / 2
    halves = []
    for first in (0, W // 2):
        h = batch_on_current_stream(boxes(W // 2, n), defaults=ZERO_G_PGS)
        h.set_sampler(c)
        halves.append(_sample_std(h, c, std=sd, first=first))
        h.close()
    assert np.array_equal(bits(np.concatenate(halves, axis=1)), bits(u))
    b.close()


@gpu
def test_std_sampler_honours_the_per_step_std():
    W, n, H = 50000, 2, 4   # 600000 samples per step
    b = batch_on_current_stream(boxes(W, n), defaults=ZERO_G_PGS)
    c = mpc.CEM(n, H, sigma=1.0, n_elite=1, seed=99)
    b.set_sampler(c)
    std = 0.5 * (1.0 + np.arange(H))[:, None, None] * np.ones((H, n, U))
    std[:, 1, 3:] *= 3.0   # and per body and component
    x = _sample_std(b, c, std=cuda(std))[:, 1:]
    for t in range(H):
        for sl, scale in (((0, slice(None)), 0.5 * (t + 1)), ((1, slice(0, 3)), 0.5 * (t + 1)), ((1, slice(3, 6)), 1.5 * (t + 1))):
            e = x[t][:, sl[0], sl[1]] / scale
            assert abs(e.mean()) < 1.2e-2 and abs(e.std() - 1.0) < 1.2e-2, (t, sl, e.mean(), e.std())
    b.close()


@gpu
def test_gather_controls_copies_rows_bit_for_bit():
    W, n, H = 77, 3, 5
    b = batch_on_current_stream(boxes(W, n), defaults=ZERO_G_PGS)
    rng = np.random.default_rng(12)
    raw = rng.integers(0, 2 ** 63, size=(H, W, n, U), dtype=np.int64).view(np.float64)   # any bits, NaN payloads included
    raw[0, W - 1, 0, 0], raw[2, 5, 1, 1] = -0.0, np.inf
    ud = cuda(raw)
    worlds = [W - 1, 5, 0, 5, 40, W - 1]
    out = torch.full((len(worlds), H, n, U), 7.0, dtype=torch.float64, device="cuda")
    launches = b.launch_count
    b.gather_controls(ud.data_ptr(), H, worlds, out.data_ptr())
    assert b.launch_count - launches == 1
    got = out.cpu().numpy()
    assert np.array_equal(bits(got), bits(raw[:, worlds].transpose(1, 0, 2, 3)))
    # a shorter horizon reads the first steps of a [H][W][n][6] buffer with the same W
    short = torch.full((2, 2, n, U), 7.0, dtype=torch.float64, device="cuda")
    b.gather_controls(ud.data_ptr(), 2, [3, 76], short.data_ptr())
    assert np.array_equal(bits(short.cpu().numpy()), bits(raw[:2, [3, 76]].transpose(1, 0, 2, 3)))
    b.close()


@gpu
def test_control_moments_match_numpy():
    W, n, H = 64, 3, 7
    b = batch_on_current_stream(boxes(W, n), defaults=ZERO_G_PGS)
    rng = np.random.default_rng(13)
    for k in (1, 2, 37, 300):
        rows = rng.normal(size=(k, H, n, U)) * 10.0 ** rng.integers(-6, 6, size=(1, H, n, U)) + rng.normal(size=(1, H, n, U))
        rd = cuda(rows)
        out = torch.full((2, H, n, U), 7.0, dtype=torch.float64, device="cuda")
        launches = b.launch_count
        b.control_moments(rd.data_ptr(), k, H, out.data_ptr())
        assert b.launch_count - launches == 1
        got = out.cpu().numpy()
        scale = np.abs(rows).max(axis=0)
        assert np.all(np.abs(got[0] - rows.mean(axis=0)) <= 1e-14 * scale), k
        assert np.all(np.abs(got[1] - rows.std(axis=0)) <= 1e-14 * scale), k
        mean, std = moments_numpy(rows)
        assert np.array_equal(bits(got[0]), bits(mean)) and np.array_equal(bits(got[1]), bits(std)), k
        again = torch.empty_like(out)
        b.control_moments(rd.data_ptr(), k, H, again.data_ptr())
        assert np.array_equal(bits(again.cpu().numpy()), bits(got)), "two calls"
    rows[5, 2, 1, 4] = np.nan
    out = torch.empty((2, H, n, U), dtype=torch.float64, device="cuda")
    b.control_moments(cuda(rows).data_ptr(), rows.shape[0], H, out.data_ptr())
    got = out.cpu().numpy()
    assert np.isnan(got[:, 2, 1, 4]).all() and np.isfinite(got).sum() == got.size - 2
    b.close()


@gpu
def test_bad_arguments_are_refused_on_the_host():
    import eggshell_b200 as E
    from eggshell_b200.batch import EggError
    W, n, H = 64, 2, 3
    scene = boxes(W, n)
    b = batch_on_current_stream(scene, defaults=ZERO_G_PGS)
    b.step(scene["dt"])
    before = state_rows(b)
    c = _plan(n, H)
    u = torch.full((H, W, n, U), 7.0, dtype=torch.float64, device="cuda")
    out = torch.full((W * H * n * U + 2,), 7.0, dtype=torch.float64, device="cuda")
    host = np.zeros(H * W * n * U + 2)
    hp = host.ctypes.data
    mp, sp, up, op = c.u_nom.data_ptr(), c.std.data_ptr(), u.data_ptr(), out.data_ptr()
    launches = b.launch_count

    def refused(call, code, what):
        with pytest.raises(EggError) as ei:
            call()
        assert err_code(ei) == code, f"{what}: {ei.value}"

    refused(lambda: b.sample_controls_std(mp, sp, H, 1, 0, 0, up), -4, "no sampler")
    b.set_sampler(c)
    for args, what in (((hp, sp, H, 0, op), "host mean_d"), ((mp, hp, H, 0, op), "host std_d"), ((mp, sp, H, 0, hp), "host u_d"),
                       ((0, sp, H, 0, op), "NULL mean_d"), ((mp, 0, H, 0, op), "NULL std_d"), ((mp, sp, H, 0, 0), "NULL u_d"),
                       ((mp, sp, 0, 0, op), "horizon 0"), ((mp, sp, H, -1, op), "first < 0"),
                       ((mp + 8, sp, H, 0, op), "misaligned mean_d"), ((mp, sp + 8, H, 0, op), "misaligned std_d"),
                       ((mp, sp, H, 0, op + 8), "misaligned u_d")):
        m_, s_, h_, f_, u_ = args
        refused(lambda: b.sample_controls_std(m_, s_, h_, 1, 0, f_, u_), -1, what)
    for worlds, h_, u_, o_, what in (([], H, up, op, "k = 0"), (list(range(W)) + [0], H, up, op, "k > W"),
                                     ([0, -1], H, up, op, "world -1"), ([W], H, up, op, "world W"),
                                     ([0], 0, up, op, "horizon 0"), ([0], H, hp, op, "host u_d"), ([0], H, up, hp, "host out_d"),
                                     ([0], H, 0, op, "NULL u_d"), ([0], H, up, 0, "NULL out_d")):
        refused(lambda: b.gather_controls(u_, h_, worlds, o_), -1, what)
    for k, h_, r_, o_, what in ((0, H, up, op, "k = 0"), (-1, H, up, op, "k < 0"), (2, 0, up, op, "horizon 0"),
                                (2, H, hp, op, "host rows_d"), (2, H, up, hp, "host out_d"), (2, H, 0, op, "NULL rows_d")):
        refused(lambda: b.control_moments(r_, k, h_, o_), -1, what)
    assert b.launch_count == launches
    assert bool((u == 7.0).all()) and bool((out == 7.0).all())
    assert np.array_equal(bits(state_rows(b)), bits(before))
    b.close()
    # before egg_init: set_sampler is accepted, the three calls are not
    raw = E.Batch(W, n, 0, solver=E.SOLVER_PGS)
    raw.set_bodies(scene["p"], scene["R"], scene["v"], scene["w"], scene["m"], scene["I"])
    raw.set_sampler(c)
    refused(lambda: raw.sample_controls_std(mp, sp, H, 1, 0, 0, up), -4, "sample before egg_init")
    refused(lambda: raw.gather_controls(up, H, [0, 1], op), -4, "gather before egg_init")
    refused(lambda: raw.control_moments(up, 2, H, op), -4, "moments before egg_init")
    raw.close()
    assert bool((u == 7.0).all()) and bool((out == 7.0).all())


def _reach(W, seed=5):
    scene = boxes(W, 1, seed=seed)
    for key in ("p", "R", "v", "w"):
        scene[key] = np.broadcast_to(scene[key][:1], scene[key].shape).copy()
    return scene


@gpu
def test_cem_lowers_the_cost_of_a_reaching_task():
    """One box in zero gravity pushed by force controls towards a target 1.2 m away within H steps
    (the task of the MPPI test); each refit is checked against numpy from the read-back samples."""
    W, H = 1024, 10
    scene = _reach(W)
    dt = scene["dt"]
    b = batch_on_current_stream(scene, defaults=ZERO_G_PGS)
    b.snapshot()
    x0 = state_rows(b)[0]
    b.set_cost(reach_cost(x0, x0[0, 0:3] + [1.0, -0.5, 0.5]))
    c = mpc.CEM(1, H, sigma=[4.0, 4.0, 4.0, 0.0, 0.0, 0.0], n_elite=64, alpha=0.1, sigma_min=0.05, u_lo=-20.0, u_hi=20.0, seed=2024)
    b.set_sampler(c)
    u = torch.empty((H, W, 1, U), dtype=torch.float64, device="cuda")
    launches = b.launch_count
    b.step(dt)
    step_launches = b.launch_count - launches
    launches = b.launch_count
    first = mpc.cem_iteration(b, c, dt, u, 0, W)
    # the sample, H controlled steps with the running cost, the terminal cost, the gather, the moments
    assert b.launch_count - launches == 1 + H * (step_launches + 1) + 1 + 1 + 1
    assert first["nominal_cost"] == pytest.approx(1.5, rel=1e-9) and c.iteration == 1
    for _ in range(5):
        old_u, old_s = c.u_nom.cpu().numpy(), c.std.cpu().numpy()
        r = mpc.cem_iteration(b, c, dt, u, 0, W)
        ub = u.cpu().numpy()
        J = costs_of(b, u, H, dt)
        order = np.lexsort((np.arange(W), J))[:64]
        assert r["nominal_cost"] == J[0] and r["min_cost"] == J[order[0]] and r["elite_max_cost"] == J[order[-1]]
        assert np.array_equal(bits(ub[:, 0]), bits(clamp(old_u, -20.0, 20.0)))
        mean, std = moments_numpy(ub[:, order].transpose(1, 0, 2, 3))
        eu, es = refit_numpy(old_u, old_s, mean, std, 0.1, 0.05, -20.0, 20.0)
        assert np.array_equal(bits(c.u_nom.cpu().numpy()), bits(eu)) and np.array_equal(bits(c.std.cpu().numpy()), bits(es))
        assert r["mean_std"] == pytest.approx(es.mean(), rel=1e-12)
        assert (es >= 0.05).all()
    last = mpc.cem_iteration(b, c, dt, u, 0, W)
    assert last["nominal_cost"] < 0.1 * first["nominal_cost"], (first, last)
    assert c.iteration == 7
    b.close()


@gpu
def test_cem_iteration_raises_without_enough_finite_rollouts():
    W, H = 64, 3
    scene = boxes(W, 1)
    dt = scene["dt"]
    b = batch_on_current_stream(scene, defaults=ZERO_G_PGS)
    b.snapshot()
    x0 = state_rows(b)[0]
    c = _plan(1, H, alpha=0.5, sigma_min=0.1)
    b.set_sampler(c)
    u = torch.empty((H, W, 1, U), dtype=torch.float64, device="cuda")
    old_u, old_s = c.u_nom.clone(), c.std.clone()
    # every rollout overflows to inf; then finite costs, but fewer worlds than elites
    b.set_cost(mpc.QuadraticCost(1, q_term=1e308, x_ref=x0 + 10.0))
    with pytest.raises(RuntimeError, match="0 rollouts finished with a finite cost"):
        mpc.cem_iteration(b, c, dt, u, 0, W)
    assert np.isinf(costs_of(b, u, H, dt)).all()
    b.set_cost(mpc.QuadraticCost(1, q_term=1.0, x_ref=x0))
    big = _plan(1, H, n_elite=W + 1)
    b.set_sampler(big)
    with pytest.raises(RuntimeError, match=f"{W} rollouts finished with a finite cost, fewer than n_elite = {W + 1}"):
        mpc.cem_iteration(b, big, dt, u, 0, W)
    assert torch.equal(big.u_nom, _plan(1, H).u_nom) and big.iteration == 0
    b.set_sampler(c)
    assert torch.equal(c.u_nom, old_u) and torch.equal(c.std, old_s) and c.iteration == 0
    # the checks of mppi_iteration, and the planner's own
    with pytest.raises(ValueError):
        mpc.cem_iteration(b, c, dt, u[:2].contiguous(), 0, W)
    with pytest.raises(ValueError):
        mpc.cem_iteration(b, c, dt, u.cpu(), 0, W)
    with pytest.raises(ValueError):
        mpc.cem_iteration(b, _plan(1, H), dt, u, 0, W)
    with pytest.raises(ValueError):
        mpc.cem_iteration(b, c, dt, u, 5, W)
    mpc.cem_iteration(b, c, dt, u, 0, W)
    assert c.iteration == 1
    b.close()


@gpu
def test_cem_advance_steps_every_world_from_the_plan():
    import eggshell_b200 as E
    W, H = 8, 4
    scene = E.scenes.legged20(W)
    dt, n = scene["dt"], scene["n"]
    kw = dict(solver=E.SOLVER_PGS, k_max=100)
    b = E.scenes.make_batch(scene, **kw)
    b.set_stream(torch.cuda.current_stream().cuda_stream)
    b.snapshot()
    rng = np.random.default_rng(21)
    sigma = rng.uniform(0.05, 0.2, size=(n, U))
    c = mpc.CEM(n, H, sigma=sigma, n_elite=3, alpha=0.5, u_lo=-0.3, u_hi=0.3, seed=5,
                u_nom=scene["f_ext"][0] + rng.normal(0.0, 0.3, size=(H, n, U)))
    b.set_sampler(c)
    u = torch.empty((H, W, n, U), dtype=torch.float64, device="cuda")
    mpc.cem_iteration(b, c, dt, u, 0, W)
    plan, std = c.u_nom.cpu().numpy(), c.std.cpu().numpy()
    assert not np.array_equal(std[-1], sigma)
    executed, start = mpc.cem_advance(b, c, dt, W)
    c0 = clamp(plan[0], -0.3, 0.3)
    assert np.array_equal(bits(executed.cpu().numpy()), bits(c0))
    fresh = E.scenes.make_batch(scene, **kw)
    fresh.set_external(np.broadcast_to(c0, (W, n, U)))
    fresh.step(dt, 1)
    expect = state_rows(fresh)[0]
    fresh.close()
    assert np.array_equal(bits(state_rows(b)), bits(np.broadcast_to(expect, (W, n, S))))
    assert np.array_equal(bits(start.cpu().numpy()), bits(expect))
    b.restore()   # the new start is the snapshot
    assert np.array_equal(bits(state_rows(b)), bits(np.broadcast_to(expect, (W, n, S))))
    got_u, got_s = c.u_nom.cpu().numpy(), c.std.cpu().numpy()
    assert np.array_equal(bits(got_u[:-1]), bits(plan[1:])) and np.array_equal(bits(got_u[-1]), bits(plan[-1]))
    assert np.array_equal(bits(got_s[:-1]), bits(std[1:])) and np.array_equal(bits(got_s[-1]), bits(sigma))
    b.close()


def _run_planner(rank, ws, W, H, iters):
    """`iters` CEM iterations of the reaching task on this rank's shard of W worlds; returns the first
    iteration's samples of the shard and every iteration's u_nom and std."""
    lo, hi = mpc.shard_range(W, rank, ws)
    scene = _reach(W)
    for key in ("p", "R", "v", "w", "m", "I"):
        scene[key] = scene[key][lo:hi].copy()
    scene["W"] = hi - lo
    b = batch_on_current_stream(scene, defaults=ZERO_G_PGS, device=torch.cuda.current_device())
    b.snapshot()
    x0 = state_rows(b)[0]
    b.set_cost(reach_cost(x0, x0[0, 0:3] + [1.0, -0.5, 0.5]))
    c = mpc.CEM(1, H, sigma=[4.0, 4.0, 4.0, 0.0, 0.0, 0.0], n_elite=32, alpha=0.2, sigma_min=0.05, seed=77)
    b.set_sampler(c)
    u = torch.empty((H, hi - lo, 1, U), dtype=torch.float64, device=torch.device("cuda", torch.cuda.current_device()))
    plans, stds, samples = [], [], None
    for i in range(iters):
        mpc.cem_iteration(b, c, scene["dt"], u, lo, W)
        if i == 0:
            samples = u.cpu().numpy()
        plans.append(c.u_nom.cpu().numpy())
        stds.append(c.std.cpu().numpy())
    b.close()
    return samples, np.stack(plans), np.stack(stds)


@gpu
def test_one_rank_against_two_nccl_ranks():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    W, H, iters = 513, 6, 3   # uneven shards
    one = _run_planner(0, 1, W, H, iters)
    res = run_ranks(_run_planner, 2, "nccl", W, H, iters, timeout=300)
    assert np.array_equal(bits(np.concatenate([res[0][0], res[1][0]], axis=1)), bits(one[0]))
    for r in range(2):
        assert np.array_equal(bits(res[r][1]), bits(one[1])) and np.array_equal(bits(res[r][2]), bits(one[2])), r
