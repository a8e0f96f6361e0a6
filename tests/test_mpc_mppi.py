"""MPPI planner: egg_set_sampler / egg_sample_controls (Philox4x32-10 + Box-Muller noise around a
nominal schedule), egg_mppi_reduce (the cost-weighted sum) and mpc.MPPI, mppi_iteration and
mppi_advance.  The first tests run on the CPU; the rest need a CUDA device."""
import ctypes as C

import numpy as np
import pytest
import torch

from eggshell_b200 import mpc
from tests.mpc_helpers import (ZERO_G_PGS, batch_on_current_stream, bits, boxes, clamp, costs_of, cuda, err_code, noise,
                               philox4x32_10, reach_cost, run_ranks, state_rows)

gpu = pytest.mark.gpu
S, U = mpc.STATE_PER_BODY, mpc.CONTROL_PER_BODY


# ---- CPU ------------------------------------------------------------------------------------------
def test_philox_known_answers():
    """The Random123 known-answer vectors of Philox4x32-10."""
    m = 0xffffffff
    for ctr, key, expect in (((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
                             ((m, m, m, m), (m, m), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
                             ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
                              (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))):
        assert [int(x) for x in philox4x32_10(ctr, key)] == list(expect)


def test_mppi_validates_and_broadcasts():
    m = mpc.MPPI(3, 4, sigma=[0, 0, 0, 0.1, 0.2, 0.3], lam=0.5, u_hi=2.0, seed=2 ** 64 - 1, device="cpu")
    assert m.sigma.shape == (3, U) and (m.sigma[1] == [0, 0, 0, 0.1, 0.2, 0.3]).all()
    assert m.u_lo is None and m.u_hi.shape == (3, U) and (m.u_hi == 2.0).all()
    assert m.u_nom.shape == (4, 3, U) and m.u_nom.dtype == torch.float64 and not m.u_nom.any()
    assert m.iteration == 0 and m.lam == 0.5 and m.horizon == 4
    assert torch.equal(m.lo, torch.full((3, U), -np.inf, dtype=torch.float64))
    m = mpc.MPPI(2, 3, sigma=1.0, lam=1.0, u_lo=-np.inf, u_hi=np.inf, u_nom=np.arange(6.0), device="cpu")
    assert m.u_nom.shape == (3, 2, U) and (m.u_nom[2, 1].numpy() == np.arange(6.0)).all()
    assert torch.equal(m.clamp(torch.tensor([[-1e300] * 6] * 2, dtype=torch.float64)), torch.full((2, U), -1e300, dtype=torch.float64))
    b = mpc.MPPI(2, 3, sigma=1.0, lam=1.0, u_lo=-1.0, u_hi=[1, 1, 1, 2, 2, 2], device="cpu")
    assert torch.equal(b.clamp(torch.full((3, 2, U), 5.0, dtype=torch.float64))[0, 0], torch.tensor([1.0, 1, 1, 2, 2, 2], dtype=torch.float64))
    bad = [dict(sigma=-0.1), dict(sigma=np.nan), dict(sigma=np.inf), dict(sigma=np.ones((3, U))), dict(sigma=np.ones(5)),
           dict(lam=0.0), dict(lam=-1.0), dict(lam=np.nan), dict(lam=np.inf),
           dict(u_lo=np.nan), dict(u_hi=[0, 0, 0, 0, 0, np.nan]), dict(u_lo=1.0, u_hi=0.0), dict(u_lo=np.ones((2, 2))),
           dict(seed=-1), dict(seed=2 ** 64), dict(u_nom=np.ones((2, 2, U))), dict(u_nom=np.nan), dict(u_nom=np.ones((4, 3, 2, U)))]
    for kw in bad:
        args = dict(sigma=1.0, lam=1.0, device="cpu")
        args.update(kw)
        with pytest.raises(ValueError):
            mpc.MPPI(2, 3, **args)
    for n, H in ((0, 3), (2, 0)):
        with pytest.raises(ValueError):
            mpc.MPPI(n, H, sigma=1.0, lam=1.0, device="cpu")


def _partials(rank, L=37):
    """Per-rank partial sums whose rank-order sum rounds differently from other orders."""
    rng = np.random.default_rng(100 + rank)
    return rng.normal(size=L) * 10.0 ** rng.integers(-8, 8, size=L)


def _gloo_worker(rank, ws):
    return mpc.allgather_rank_sum(torch.from_numpy(_partials(rank))).numpy().copy()


def test_rank_order_combine_gloo():
    res = run_ranks(_gloo_worker, 2, "gloo", timeout=120)
    expect = _partials(0) + _partials(1)
    assert np.array_equal(bits(res[0]), bits(res[1]))
    assert np.array_equal(bits(res[0]), bits(expect))


# ---- GPU ------------------------------------------------------------------------------------------
def _sample(b, m, first=0, iteration=None, seed=None):
    u = torch.full((m.horizon, b.W, b.n, U), np.nan, dtype=torch.float64, device="cuda")
    b.sample_controls(m.u_nom.data_ptr(), m.horizon, m.seed if seed is None else seed,
                      m.iteration if iteration is None else iteration, first, u.data_ptr())
    return u.cpu().numpy()


def _planner(n, H, seed=7, **kw):
    rng = np.random.default_rng(seed)
    args = dict(sigma=rng.uniform(0.2, 1.0, size=(n, U)), lam=1.0, seed=0x1234_5678_9abc_def0,
                u_nom=rng.normal(0.0, 1.0, size=(H, n, U)))
    args.update(kw)
    return mpc.MPPI(n, H, **args)


@gpu
def test_sampler_matches_numpy():
    W, n, H, first = 300, 3, 3, 1000
    b = batch_on_current_stream(boxes(W, n), defaults=ZERO_G_PGS)
    m = _planner(n, H)
    m.iteration = 2 ** 32 + 5   # both counter words of the iteration in use
    b.set_sampler(m)
    u = _sample(b, m, first=first)
    eps = noise(H, n, np.arange(first, first + W), m.seed, m.iteration)
    un = m.u_nom.cpu().numpy()[:, None]
    got = (u - un) / m.sigma
    assert np.max(np.abs(got - eps)) <= 1e-13, np.max(np.abs(got - eps))
    assert np.abs(eps).max() > 3.0   # a real sample of the normal distribution
    b.close()


@gpu
def test_sampler_exact_cases():
    W, n, H = 256, 2, 3
    b = batch_on_current_stream(boxes(W, n), defaults=ZERO_G_PGS)
    rng = np.random.default_rng(3)
    lo, hi = rng.uniform(-1.5, -0.5, size=(n, U)), rng.uniform(0.5, 1.5, size=(n, U))
    lo[0, 0], hi[1, 5] = -np.inf, np.inf
    un = rng.normal(0.0, 1.0, size=(H, n, U))
    un[0, 0, 1] = -0.0
    m = _planner(n, H, u_nom=un, u_lo=lo, u_hi=hi, sigma=rng.uniform(0.5, 2.0, size=(n, U)))
    b.set_sampler(m)
    u = _sample(b, m)
    c_nom = clamp(un, lo, hi)
    assert np.array_equal(bits(u[:, 0]), bits(c_nom)), "global world 0 runs clamp(u_nom)"
    assert (u >= lo).all() and (u <= hi).all()
    at_lo, at_hi = u == lo, u == hi
    assert at_lo.sum() > 100 and at_hi.sum() > 100   # bounds reached, and hit exactly
    eps = noise(H, n, np.arange(W), m.seed, m.iteration)
    free = clamp(un[:, None] + m.sigma * eps, lo, hi)
    assert np.array_equal(at_lo[:, 1:], (free == lo)[:, 1:]) and np.array_equal(at_hi[:, 1:], (free == hi)[:, 1:])
    assert np.array_equal(bits(_sample(b, m)), bits(u)), "two calls"
    for kw in (dict(iteration=1), dict(seed=m.seed + 1)):
        v = _sample(b, m, **kw)
        assert np.array_equal(bits(v[:, 0]), bits(c_nom))
        inside = (u > lo) & (u < hi) & (v > lo) & (v < hi)
        inside[:, 0] = False
        assert inside.sum() > 1000 and (v[inside] != u[inside]).all(), kw
    # sigma = 0: clamp(u_nom) in every world, bit for bit (-0.0 included)
    m0 = mpc.MPPI(n, H, sigma=0.0, lam=1.0, u_nom=un, u_lo=lo, u_hi=hi)
    b.set_sampler(m0)
    assert np.array_equal(bits(_sample(b, m0)), bits(np.broadcast_to(c_nom[:, None], (H, W, n, U))))
    # one batch of W against two batches of W / 2 with first = 0 and first = W / 2
    b.set_sampler(m)
    halves = []
    for lo_w in (0, W // 2):
        h = batch_on_current_stream(boxes(W // 2, n), defaults=ZERO_G_PGS)
        h.set_sampler(m)
        halves.append(_sample(h, m, first=lo_w))
        h.close()
    assert np.array_equal(bits(np.concatenate(halves, axis=1)), bits(u))
    b.close()


@gpu
def test_noise_moments():
    W, n, H = 30000, 2, 3   # 1.08e6 samples
    b = batch_on_current_stream(boxes(W, n), defaults=ZERO_G_PGS)
    m = mpc.MPPI(n, H, sigma=1.0, lam=1.0, seed=99)
    b.set_sampler(m)
    eps = _sample(b, m)[:, 1:]
    assert abs(eps.mean()) < 5e-3 and abs(eps.std() - 1.0) < 5e-3, (eps.mean(), eps.std())
    b.close()


def _reduce(b, u, H, cost, baseline, lam):
    out = torch.full((H * b.n * U + 2,), np.nan, dtype=torch.float64, device="cuda")
    b.mppi_reduce(u.data_ptr(), H, cost.data_ptr(), baseline.data_ptr(), lam, out.data_ptr())
    return out.cpu().numpy()


def _reduce_numpy(u, cost, baseline, lam):
    """float64 numpy: (sum_w omega u [H, n, 6], sum omega, sum omega^2, sum |omega u|)."""
    om = np.where(np.isfinite(cost), np.exp(-(np.where(np.isfinite(cost), cost, 0.0) - baseline) / lam), 0.0)
    if not np.isfinite(baseline):
        om[:] = 0.0
    wu = om[None, :, None, None] * u
    return wu.sum(axis=1), om.sum(), (om * om).sum(), np.abs(wu).sum(axis=1), om


@gpu
def test_reduce_matches_numpy():
    W, n, H = 1000, 3, 4   # 4 chunks, the last one partial
    b = batch_on_current_stream(boxes(W, n), defaults=ZERO_G_PGS)
    rng = np.random.default_rng(11)
    u = rng.normal(0.0, 1.0, size=(H, W, n, U))
    cost = rng.uniform(0.0, 3.0, size=W)
    cost[[5, 17, 300, 999]] = [np.nan, np.inf, -np.inf, np.nan]
    base = np.min(cost[np.isfinite(cost)])
    ud, cd, bd = cuda(u), cuda(cost), cuda(np.array(base))
    lam = 0.7
    got = _reduce(b, ud, H, cd, bd, lam)
    s, so, so2, sabs, om = _reduce_numpy(u, cost, base, lam)
    L = H * n * U
    assert np.all(np.abs(got[:L] - s.ravel()) <= 1e-12 * sabs.ravel())
    assert abs(got[L] - so) <= 1e-12 * so and abs(got[L + 1] - so2) <= 1e-12 * so2
    assert np.array_equal(bits(_reduce(b, ud, H, cd, bd, lam)), bits(got)), "two calls"
    # the non-finite costs get weight 0: the same result as dropping those worlds' schedules
    keep = np.isfinite(cost)
    u0 = u.copy()
    u0[:, ~keep] = np.nan
    assert np.array_equal(bits(_reduce(b, cuda(u0), H, cd, bd, lam)), bits(got))
    # NaN-only costs, and a non-finite baseline: every weight is 0
    nan = cuda(np.full(W, np.nan))
    assert not _reduce(b, ud, H, nan, cuda(np.array(np.inf)), lam).any()
    assert not _reduce(b, ud, H, cd, cuda(np.array(np.nan)), lam).any()
    # a huge lambda: the plain mean; a tiny one with one clearly best world: that world's schedule
    fin = cuda(rng.uniform(0.0, 3.0, size=W))
    got = _reduce(b, ud, H, fin, cuda(np.array(0.0)), 1e300)
    assert got[L] == W and got[L + 1] == W
    assert np.all(np.abs(got[:L] / W - u.mean(axis=1).ravel()) <= 1e-12 * np.abs(u).mean(axis=1).ravel())
    one = np.ones(W)
    one[417] = 0.0
    got = _reduce(b, ud, H, cuda(one), cuda(np.array(0.0)), 1e-3)
    assert got[L] == 1.0 and np.array_equal(bits(got[:L]), bits(u[:, 417].ravel()))
    b.close()


@gpu
def test_bad_arguments_are_refused_on_the_host():
    import eggshell_b200 as E
    from eggshell_b200.batch import EggError, EggSampler, _p
    W, n, H = 64, 2, 3
    scene = boxes(W, n)
    b = batch_on_current_stream(scene, defaults=ZERO_G_PGS)
    b.step(scene["dt"])
    before = state_rows(b)
    m = _planner(n, H)
    u = torch.full((H, W, n, U), 7.0, dtype=torch.float64, device="cuda")
    out = torch.full((H * n * U + 2,), 7.0, dtype=torch.float64, device="cuda")
    cost = torch.zeros(W, dtype=torch.float64, device="cuda")
    base = torch.zeros((), dtype=torch.float64, device="cuda")
    host = np.zeros(H * W * n * U)
    hp = host.ctypes.data
    launches = b.launch_count

    def refused(call, code, what):
        with pytest.raises(EggError) as ei:
            call()
        assert err_code(ei) == code, f"{what}: {ei.value}"

    refused(lambda: b.sample_controls(m.u_nom.data_ptr(), H, 1, 0, 0, u.data_ptr()), -4, "no sampler")
    base_bytes = b.device_bytes
    b.set_sampler(m)
    assert b.device_bytes - base_bytes == 3 * n * U * 8
    refused(lambda: b.sample_controls(hp, H, 1, 0, 0, u.data_ptr()), -1, "host u_nom_d")
    refused(lambda: b.sample_controls(m.u_nom.data_ptr(), H, 1, 0, 0, hp), -1, "host u_d")
    refused(lambda: b.sample_controls(m.u_nom.data_ptr(), H, 1, 0, 0, 0), -1, "NULL u_d")
    refused(lambda: b.sample_controls(m.u_nom.data_ptr(), 0, 1, 0, 0, u.data_ptr()), -1, "horizon 0")
    refused(lambda: b.sample_controls(m.u_nom.data_ptr(), H, 1, 0, -1, u.data_ptr()), -1, "first < 0")
    for lam in (0.0, -1.0, np.nan, np.inf):
        refused(lambda: b.mppi_reduce(u.data_ptr(), H, cost.data_ptr(), base.data_ptr(), lam, out.data_ptr()), -1, f"lambda {lam}")
    refused(lambda: b.mppi_reduce(u.data_ptr(), 0, cost.data_ptr(), base.data_ptr(), 1.0, out.data_ptr()), -1, "horizon 0")
    for i in range(4):
        ptrs = [u.data_ptr(), cost.data_ptr(), base.data_ptr(), out.data_ptr()]
        ptrs[i] = hp
        refused(lambda: b.mppi_reduce(ptrs[0], H, ptrs[1], ptrs[2], 1.0, ptrs[3]), -1, f"host pointer {i}")
    # egg_set_sampler: non-finite or negative sigma, NaN bounds, u_lo > u_hi; the sampler in place stays
    one, zero = np.ones((n, U)), np.zeros((n, U))
    for sg, lo, hi in ((np.where(np.arange(U) == 2, np.nan, one), None, None), (np.where(np.arange(U) == 0, np.inf, one), None, None),
                       (-one, None, None), (one, np.where(np.arange(U) == 4, np.nan, zero), None), (one, None, np.full((n, U), np.nan)),
                       (one, one, zero)):
        s = EggSampler(_p(np.ascontiguousarray(sg)), _p(None if lo is None else np.ascontiguousarray(lo)),
                       _p(None if hi is None else np.ascontiguousarray(hi)))
        assert E.lib().egg_set_sampler(b.h, C.byref(s)) == -1
    assert b.device_bytes - base_bytes == 3 * n * U * 8
    assert b.launch_count == launches
    assert bool((u == 7.0).all()) and bool((out == 7.0).all())
    assert np.array_equal(bits(state_rows(b)), bits(before))
    ref = noise(H, n, np.arange(W), m.seed, 0)   # the sampler in place still samples with m's sigma
    got = _sample(b, m, iteration=0)
    assert np.max(np.abs((got - m.u_nom.cpu().numpy()[:, None]) / m.sigma - ref)[:, 1:]) <= 1e-13
    b.set_sampler(None)
    assert b.device_bytes == base_bytes and b.sampler is None
    b.close()
    # before egg_init: set_sampler is accepted, sampling and reducing are not
    raw = E.Batch(W, n, 0, solver=E.SOLVER_PGS)
    raw.set_bodies(scene["p"], scene["R"], scene["v"], scene["w"], scene["m"], scene["I"])
    raw.set_sampler(m)
    refused(lambda: raw.sample_controls(m.u_nom.data_ptr(), H, 1, 0, 0, u.data_ptr()), -4, "sample before egg_init")
    refused(lambda: raw.mppi_reduce(u.data_ptr(), H, cost.data_ptr(), base.data_ptr(), 1.0, out.data_ptr()), -4, "reduce before egg_init")
    raw.close()
    assert bool((u == 7.0).all()) and bool((out == 7.0).all())


@gpu
def test_mppi_lowers_the_cost_of_a_reaching_task():
    """One box in zero gravity, far from the ground, pushed by force controls towards a target 1.2 m
    away within H steps; the terminal cost is the squared distance to the target."""
    W, H = 1024, 10
    scene = boxes(W, 1, seed=5)
    for key in ("p", "R", "v", "w"):
        scene[key] = np.broadcast_to(scene[key][:1], scene[key].shape).copy()
    dt = scene["dt"]
    b = batch_on_current_stream(scene, defaults=ZERO_G_PGS)
    b.snapshot()
    x0 = state_rows(b)[0]
    b.set_cost(reach_cost(x0, x0[0, 0:3] + [1.0, -0.5, 0.5]))
    m = mpc.MPPI(1, H, sigma=[4.0, 4.0, 4.0, 0.0, 0.0, 0.0], lam=0.05, u_lo=-20.0, u_hi=20.0, seed=2024)
    b.set_sampler(m)
    u = torch.empty((H, W, 1, U), dtype=torch.float64, device="cuda")
    launches = b.launch_count
    b.step(dt)
    step_launches = b.launch_count - launches
    launches = b.launch_count
    first = mpc.mppi_iteration(b, m, dt, u, 0)
    # the sample, H controlled steps with the running cost, the terminal cost, the two reduce kernels
    assert b.launch_count - launches == 1 + H * (step_launches + 1) + 1 + 2
    assert first["nominal_cost"] == pytest.approx(1.5, rel=1e-9) and m.iteration == 1
    # the update against numpy from the read-back samples and costs
    for _ in range(5):
        old = m.u_nom.clone()
        r = mpc.mppi_iteration(b, m, dt, u, 0)
        ub = u.cpu().numpy()
        J = costs_of(b, u, H, dt)
        assert r["min_cost"] == J.min() and r["nominal_cost"] == J[0]
        assert np.array_equal(bits(ub[:, 0]), bits(m.clamp(old).cpu().numpy()))
        s, so, so2, sabs, _ = _reduce_numpy(ub, J, J.min(), m.lam)
        expect = np.clip(s / so, -20.0, 20.0)
        got = m.u_nom.cpu().numpy()
        assert np.all(np.abs(got - expect) <= 1e-12 * sabs / so + 1e-300)
        assert r["weight_sum"] == pytest.approx(so, rel=1e-12) and r["ess"] == pytest.approx(so * so / so2, rel=1e-12)
        assert 1.0 - 1e-12 <= r["ess"] <= W
    last = mpc.mppi_iteration(b, m, dt, u, 0)
    assert last["nominal_cost"] < 0.1 * first["nominal_cost"], (first, last)
    assert m.iteration == 7
    b.close()


@gpu
def test_mppi_iteration_raises_without_a_finite_rollout():
    """A cost whose every rollout overflows to inf: sum omega = 0, u_nom and iteration unchanged."""
    W, H = 64, 3
    scene = boxes(W, 1)
    dt = scene["dt"]
    b = batch_on_current_stream(scene, defaults=ZERO_G_PGS)
    b.snapshot()
    x0 = state_rows(b)[0]
    b.set_cost(mpc.QuadraticCost(1, q_term=1e308, x_ref=x0 + 10.0))
    m = _planner(1, H)
    b.set_sampler(m)
    u = torch.empty((H, W, 1, U), dtype=torch.float64, device="cuda")
    old = m.u_nom.clone()
    with pytest.raises(RuntimeError, match="weights sum to 0"):
        mpc.mppi_iteration(b, m, dt, u, 0)
    assert torch.equal(m.u_nom, old) and m.iteration == 0
    assert np.isinf(costs_of(b, u, H, dt)).all()
    # the checks of mpc_iteration, and the planner's own
    with pytest.raises(ValueError):
        mpc.mppi_iteration(b, m, dt, u[:2].contiguous(), 0)
    with pytest.raises(ValueError):
        mpc.mppi_iteration(b, m, dt, u.cpu(), 0)
    with pytest.raises(ValueError):
        mpc.mppi_iteration(b, _planner(1, H), dt, u, 0)
    with pytest.raises(ValueError):
        mpc.mppi_iteration(b, m, dt, u, 5)
    b.close()


@gpu
def test_mppi_advance_steps_every_world_from_the_plan():
    import eggshell_b200 as E
    W, H = 8, 4
    scene = E.scenes.legged20(W)
    dt, n = scene["dt"], scene["n"]
    kw = dict(solver=E.SOLVER_PGS, k_max=100)
    b = E.scenes.make_batch(scene, **kw)
    b.set_stream(torch.cuda.current_stream().cuda_stream)
    b.snapshot()
    rng = np.random.default_rng(21)
    m = mpc.MPPI(n, H, sigma=0.1, lam=1.0, u_lo=-0.3, u_hi=0.3, seed=5,
                 u_nom=scene["f_ext"][0] + rng.normal(0.0, 0.3, size=(H, n, U)))
    b.set_sampler(m)
    u = torch.empty((H, W, n, U), dtype=torch.float64, device="cuda")
    mpc.mppi_iteration(b, m, dt, u, 0)
    plan = m.u_nom.cpu().numpy()
    executed, start = mpc.mppi_advance(b, m, dt, W)
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
    got = m.u_nom.cpu().numpy()
    assert np.array_equal(bits(got[:-1]), bits(plan[1:])) and np.array_equal(bits(got[-1]), bits(plan[-1]))
    b.close()


def _run_planner(rank, ws, W, H, iters):
    """`iters` MPPI iterations of the reaching task on this rank's shard of W worlds; returns the
    first iteration's samples of the shard and every iteration's u_nom."""
    lo, hi = mpc.shard_range(W, rank, ws)
    scene = boxes(W, 1, seed=5)
    for key in ("p", "R", "v", "w", "m", "I"):
        scene[key] = np.broadcast_to(scene[key][:1], scene[key].shape)[lo:hi].copy()
    scene["W"] = hi - lo
    b = batch_on_current_stream(scene, defaults=ZERO_G_PGS, device=torch.cuda.current_device())
    b.snapshot()
    x0 = state_rows(b)[0]
    b.set_cost(reach_cost(x0, x0[0, 0:3] + [1.0, -0.5, 0.5]))
    m = mpc.MPPI(1, H, sigma=[4.0, 4.0, 4.0, 0.0, 0.0, 0.0], lam=0.05, seed=77)
    b.set_sampler(m)
    u = torch.empty((H, hi - lo, 1, U), dtype=torch.float64, device=torch.device("cuda", torch.cuda.current_device()))
    plans, samples = [], None
    for i in range(iters):
        mpc.mppi_iteration(b, m, scene["dt"], u, lo)
        if i == 0:
            samples = u.cpu().numpy()
        plans.append(m.u_nom.cpu().numpy())
    b.close()
    return samples, np.stack(plans)


@gpu
def test_one_rank_against_two_nccl_ranks():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    W, H, iters = 512, 6, 3
    one_samples, one_plans = _run_planner(0, 1, W, H, iters)
    res = run_ranks(_run_planner, 2, "nccl", W, H, iters, timeout=300)
    assert np.array_equal(bits(np.concatenate([res[0][0], res[1][0]], axis=1)), bits(one_samples))
    assert np.array_equal(bits(res[0][1]), bits(res[1][1])), "every rank holds the same plan"
    assert np.max(np.abs(res[0][1] - one_plans)) <= 1e-12 * max(1.0, np.abs(one_plans).max())
