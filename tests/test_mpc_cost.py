"""Configurable quadratic MPC cost: mpc.QuadraticCost (the numpy definition), egg_set_cost and
egg_step_controlled_cost (the running cost added on the device before every step, the terminal cost
after the last one) and mpc.mpc_iteration with a cost.  The first tests run on the CPU; the rest
need a CUDA device."""
import ctypes as C

import numpy as np
import pytest
import torch

from eggshell_b200 import mpc
from tests.mpc_helpers import batch_on_current_stream, bits, cuda, err_code, state_rows

gpu = pytest.mark.gpu
S, U = mpc.STATE_PER_BODY, mpc.CONTROL_PER_BODY
TERMS = ("q_run", "l_run", "u_run", "q_term", "l_term")


# ---- CPU ------------------------------------------------------------------------------------------
def test_quadratic_cost_validates_and_broadcasts():
    c = mpc.QuadraticCost(3, q_run=2.0, u_run=[1, 2, 3, 4, 5, 6], l_term=np.arange(18.0))
    assert c.q_run.shape == (3, S) and (c.q_run == 2.0).all()
    assert c.u_run.shape == (3, U) and (c.u_run == np.arange(1.0, 7.0)).all()
    assert c.l_term.shape == (3, S) and (c.l_term == np.arange(18.0)).all()
    assert c.l_run.shape == c.q_term.shape == (3, S) and not c.l_run.any() and not c.q_term.any()
    assert c.ref_steps == 1 and c.x_ref.shape == (1, 3, S) and not c.x_ref.any()
    assert mpc.QuadraticCost(3, x_ref=np.ones((3, S))).ref_steps == 1
    assert mpc.QuadraticCost(3, x_ref=np.ones((5, 3, S))).ref_steps == 5
    assert mpc.QuadraticCost(3, x_ref=np.ones((4, 1, S))).x_ref.shape == (4, 3, S)
    bad = [dict(q_run=np.ones((2, S))), dict(l_run=np.ones(U)), dict(u_run=np.ones((3, S))), dict(q_term=np.ones((3, 3, S))),
           dict(l_term=np.ones(7)), dict(x_ref=np.ones((3, U))), dict(x_ref=np.ones((2, 2, 3, S))), dict(x_ref=np.ones((0, 3, S))),
           dict(q_run=np.nan), dict(l_run=-np.inf), dict(u_run=[0, 0, np.inf, 0, 0, 0]), dict(q_term=np.full((3, S), np.nan)),
           dict(l_term=np.inf), dict(x_ref=np.where(np.arange(S) == 4, np.nan, 0.0))]
    for kw in bad:
        with pytest.raises(ValueError):
            mpc.QuadraticCost(3, **kw)
    with pytest.raises(ValueError):
        mpc.QuadraticCost(0)
    c = mpc.QuadraticCost(3, x_ref=np.zeros((3, 3, S)))   # a per-step reference for horizons up to 2
    assert c.evaluate(np.zeros((3, 2, 3, S)), np.zeros((2, 2, 3, U))).shape == (2,)
    assert c.evaluate(np.zeros((2, 2, 3, S)), np.zeros((1, 2, 3, U))).shape == (2,)
    for states, u in ((np.zeros((4, 2, 3, S)), np.zeros((3, 2, 3, U))),    # H = 3 needs 4 reference rows
                      (np.zeros((3, 2, 3, S)), np.zeros((3, 2, 3, U))),    # states are not H + 1
                      (np.zeros((3, 2, 3, S)), np.zeros((2, 2, 4, U))),    # another n
                      (np.zeros((1, 2, 3, S)), np.zeros((0, 2, 3, U)))):   # H = 0
        with pytest.raises(ValueError):
            c.evaluate(states, u)


def test_evaluate_by_hand():
    """2 worlds, 2 bodies, H = 2, a per-step reference; every term summed out by hand below."""
    H, W, n = 2, 2, 2
    q_run, l_run, u_run = np.zeros((n, S)), np.zeros((n, S)), np.zeros((n, U))
    q_term, l_term = np.zeros((n, S)), np.zeros((n, S))
    q_run[0, 0] = 2.0      # body 0 x
    q_run[1, 13] = 3.0     # body 1 v_y
    l_run[1, 2] = -1.0     # body 1 z
    u_run[0, 3] = 0.5      # body 0 tau_x
    u_run[1, 0] = 4.0      # body 1 f_x
    q_term[0, 2] = 10.0    # body 0 z
    l_term[0, 0] = -1.0    # body 0 x
    x_ref = np.zeros((H + 1, n, S))
    x_ref[:, 0, 0] = [0.0, 1.0, 2.0]
    x_ref[:, 1, 13] = 0.5
    x = np.zeros((H + 1, W, n, S))
    x[..., 1, 5] = 7.0     # a component without weight
    x[:, 0, 0, 0] = [0.0, 2.0, 5.0]
    x[:, 0, 0, 2] = [0.0, 0.0, 0.3]
    x[:, 0, 1, 2] = [1.0, 1.5, 2.0]
    x[:, 0, 1, 13] = [0.5, 1.5, -0.5]
    x[:, 1, 0, 0] = [1.0, 1.0, 1.0]
    x[:, 1, 0, 2] = [0.0, 0.0, -1.0]
    x[:, 1, 1, 13] = [2.0, 2.0, 2.0]
    u = np.zeros((H, W, n, U))
    u[..., 0, 5] = 9.0     # a control without weight
    u[:, 0, 0, 3] = [2.0, -2.0]
    u[:, 0, 1, 0] = [1.0, 0.0]
    u[:, 1, 0, 3] = [0.0, 4.0]
    u[:, 1, 1, 0] = [-1.0, -1.0]
    c = mpc.QuadraticCost(n, q_run=q_run, l_run=l_run, u_run=u_run, q_term=q_term, l_term=l_term, x_ref=x_ref)
    # world 0: t = 0: 2*0^2 + 3*0^2 - 1*1 + 0.5*2^2 + 4*1^2 = 5
    #          t = 1: 2*1^2 + 3*1^2 - 1*1.5 + 0.5*(-2)^2 + 4*0^2 = 5.5
    #          H:     -1*(5 - 2) + 10*0.3^2 = -2.1
    # world 1: t = 0: 2*1^2 + 3*1.5^2 - 1*0 + 0.5*0^2 + 4*(-1)^2 = 12.75
    #          t = 1: 2*0^2 + 3*1.5^2 - 1*0 + 0.5*4^2 + 4*(-1)^2 = 18.75
    #          H:     -1*(1 - 2) + 10*(-1)^2 = 11
    expect = np.array([5.0 + 5.5 - 2.1, 12.75 + 18.75 + 11.0])
    assert np.allclose(c.evaluate(x, u), expect, rtol=1e-14, atol=0)


# ---- GPU ------------------------------------------------------------------------------------------
def _scene(name, W):
    import eggshell_b200 as E
    if name == "legged20":
        return E.scenes.legged20(W), dict(solver=E.SOLVER_PGS, k_max=100), 5
    return E.scenes.chain(W, links=10, seed=3, anchor_jitter=0.1, v_jitter=0.2), dict(solver=E.SOLVER_DENSE_MURTY), 3


def _schedule(f_ext, H, seed, sigma=0.2):
    """A time-varying schedule around f_ext: random forces and torques on every body, slice by slice."""
    rng = np.random.default_rng(seed)
    u = np.broadcast_to(f_ext, (H,) + f_ext.shape).copy()
    u += rng.normal(0.0, sigma, size=u.shape)
    return u


def _host_rollout(b, u, dt):
    """x_0 ... x_H [H + 1, W, n, 18] with set_external(u[t]) + step before every step t (bit-identical to
    the controlled path, test_mpc_loop.test_time_varying_schedule_equals_host_loop)."""
    states = [state_rows(b)]
    for t in range(u.shape[0]):
        b.set_external(u[t])
        b.step(dt, 1)
        states.append(state_rows(b))
    return np.stack(states)


def _random_cost(n, states, seed, terms=TERMS, per_step=True):
    """Random nonzero weights in the listed terms; a reference near world 0's trajectory (one row per
    step, or its start only)."""
    rng = np.random.default_rng(seed)
    H = states.shape[0] - 1
    w = {t: np.zeros((n, U if t == "u_run" else S)) for t in TERMS}
    for t in terms:
        if t.startswith("q") or t == "u_run":
            w[t] = rng.uniform(0.5, 2.0, size=w[t].shape)
        else:
            w[t] = rng.normal(0.0, 1.0, size=w[t].shape)
    ref = states[:, 0] + rng.normal(0.0, 0.1, size=(H + 1, n, S))
    return mpc.QuadraticCost(n, x_ref=ref if per_step else ref[0], **w)


def _abs_terms(cost, states, u):
    """The sum of the absolute values of every term of J [W]: the scale of the rounding of the sums."""
    H = u.shape[0]
    d = np.abs(states - cost.x_ref[np.minimum(np.arange(H + 1), cost.ref_steps - 1)][:, None])
    a = np.abs
    return ((a(cost.q_run) * d[:H] ** 2 + a(cost.l_run) * d[:H]).sum(axis=(0, 2, 3)) + (a(cost.u_run) * u ** 2).sum(axis=(0, 2, 3))
            + (a(cost.q_term) * d[H] ** 2 + a(cost.l_term) * d[H]).sum(axis=(1, 2)))


def _device_cost(b, cost, ud, H, dt):
    b.set_cost(cost)
    out = torch.full((b.W,), np.nan, dtype=torch.float64, device="cuda")
    b.restore()
    b.step_controlled_cost(dt, ud.data_ptr(), H, out.data_ptr())
    return out.cpu().numpy()


def _assert_matches(got, cost, states, u, what=""):
    expect = cost.evaluate(states, u)
    tol = 1e-12 * _abs_terms(cost, states, u)
    assert np.all(np.abs(got - expect) <= tol), (what, np.max(np.abs(got - expect) / tol))


@gpu
@pytest.mark.parametrize("name,W,H", [("legged20", 64, 8), ("chain10", 8, 5)])
def test_cost_matches_numpy(name, W, H):
    scene, kw, _ = _scene(name, W)
    dt = scene["dt"]
    b = batch_on_current_stream(scene, **kw)
    b.snapshot()
    u = _schedule(b.static()[2], H, seed=51)
    states = _host_rollout(b, u, dt)
    cost = _random_cost(scene["n"], states, seed=52)
    got = _device_cost(b, cost, cuda(u), H, dt)
    assert np.array_equal(bits(state_rows(b)), bits(states[H])), "the host loop and the controlled path disagree"
    assert np.all(got != 0)
    _assert_matches(got, cost, states, u)
    b.close()


@gpu
@pytest.mark.parametrize("name", ["legged20", "chain10"])
def test_cost_path_steps_like_step_controlled(name):
    """Bodies and f_ext slot bit-identical to egg_step_controlled; H x (step launches + 1) + 1 launches."""
    W, H = 16, 6
    scene, kw, step_launches = _scene(name, W)
    dt = scene["dt"]
    b = batch_on_current_stream(scene, **kw)
    b.snapshot()
    f0 = b.static()[2]
    u = _schedule(f0, H, seed=61)
    ud = cuda(u)
    b.step_controlled(dt, ud.data_ptr(), H)
    ref_rows, ref_f = state_rows(b), b.static()[2]
    b.restore()
    b.set_external(f0)
    b.set_cost(_random_cost(scene["n"], np.stack([state_rows(b)] * (H + 1)), seed=62))
    cost = torch.empty(W, dtype=torch.float64, device="cuda")
    launches = b.launch_count
    b.step_controlled_cost(dt, ud.data_ptr(), H, cost.data_ptr())
    assert b.launch_count - launches == H * (step_launches + 1) + 1
    assert np.array_equal(bits(state_rows(b)), bits(ref_rows))
    assert np.array_equal(bits(b.static()[2]), bits(ref_f))
    assert np.array_equal(bits(ref_f), bits(u[-1]))
    b.close()


@gpu
def test_each_term_alone():
    """Only one of q_run, l_run, u_run, q_term, l_term nonzero at a time, against a per-step reference:
    a dropped term, or one evaluated at the wrong step, misses numpy by far more than the tolerance."""
    W, H = 16, 5
    scene, kw, _ = _scene("legged20", W)
    dt = scene["dt"]
    b = batch_on_current_stream(scene, **kw)
    b.snapshot()
    u = _schedule(b.static()[2], H, seed=71)
    ud = cuda(u)
    states = _host_rollout(b, u, dt)
    for i, term in enumerate(TERMS):
        cost = _random_cost(scene["n"], states, seed=72 + i, terms=(term,))
        got = _device_cost(b, cost, ud, H, dt)
        assert np.all(got != 0), term
        _assert_matches(got, cost, states, u, term)
    b.close()


@gpu
def test_constant_reference_equals_repeated_rows():
    W, H = 16, 4
    scene, kw, _ = _scene("legged20", W)
    dt, n = scene["dt"], scene["n"]
    b = batch_on_current_stream(scene, **kw)
    b.snapshot()
    ud = cuda(_schedule(b.static()[2], H, seed=81))
    one = _random_cost(n, np.stack([state_rows(b)] * (H + 1)), seed=82, per_step=False)
    rep = mpc.QuadraticCost(n, x_ref=np.repeat(one.x_ref, H + 1, axis=0), **{t: getattr(one, t) for t in TERMS})
    assert one.ref_steps == 1 and rep.ref_steps == H + 1
    base = b.device_bytes
    a = _device_cost(b, one, ud, H, dt)
    assert b.device_bytes - base == (4 * n * S + n * U + n * S) * 8
    c = _device_cost(b, rep, ud, H, dt)
    assert b.device_bytes - base == (4 * n * S + n * U + (H + 1) * n * S) * 8
    assert np.array_equal(bits(a), bits(c))
    b.set_cost(None)
    assert b.device_bytes == base and b.cost is None
    b.close()


def _shard(scene, lo, hi):
    sub = dict(scene, W=hi - lo)
    for key in ("p", "R", "v", "w", "m", "I", "c0", "c1", "f_ext"):
        sub[key] = scene[key][lo:hi].copy()
    return sub


@gpu
def test_cost_is_deterministic_and_shard_independent():
    """A world's cost has the same bits in a batch of W, in either half of a split, alone, and in a
    second run of the same batch."""
    W, H = 20, 6
    scene, kw, _ = _scene("legged20", W)
    dt, n = scene["dt"], scene["n"]
    u = _schedule(scene["f_ext"], H, seed=91)
    full = batch_on_current_stream(scene, **kw)
    full.snapshot()
    cost = _random_cost(n, np.stack([state_rows(full)] * (H + 1)), seed=92)
    ud = cuda(u)
    c_full = _device_cost(full, cost, ud, H, dt)
    rows_full = state_rows(full)
    assert np.array_equal(bits(_device_cost(full, cost, ud, H, dt)), bits(c_full)), "two runs of one batch"
    full.close()
    for lo, hi in ((0, W // 2), (W // 2, W), (13, 14)):
        part = batch_on_current_stream(_shard(scene, lo, hi), **kw)
        part.snapshot()
        c = _device_cost(part, cost, cuda(u[:, lo:hi]), H, dt)
        assert np.array_equal(bits(state_rows(part)), bits(rows_full[lo:hi])), f"physics of worlds [{lo}, {hi})"
        assert np.array_equal(bits(c), bits(c_full[lo:hi])), f"costs of worlds [{lo}, {hi})"
        part.close()


@gpu
def test_expresses_the_built_in_cost():
    """l_term[0, 0] = -1, q_term[0, 2] = 10 and x_ref = the common start state is egg_rollout_costs."""
    W, H = 16, 6
    scene, kw, _ = _scene("legged20", W)
    dt, n = scene["dt"], scene["n"]
    for key in ("p", "R", "v", "w"):
        scene[key] = np.broadcast_to(scene[key][:1], scene[key].shape).copy()
    b = batch_on_current_stream(scene, **kw)
    b.snapshot()
    x0 = state_rows(b)[0]
    l_term, q_term = np.zeros((n, S)), np.zeros((n, S))
    l_term[0, 0], q_term[0, 2] = -1.0, 10.0
    ud = cuda(_schedule(scene["f_ext"], H, seed=101))
    got = _device_cost(b, mpc.QuadraticCost(n, l_term=l_term, q_term=q_term, x_ref=x0), ud, H, dt)
    built_in = torch.empty(W, dtype=torch.float64, device="cuda")
    b.rollout_costs(built_in.data_ptr())
    expect = built_in.cpu().numpy()
    assert np.all(expect != 0) and np.unique(expect).size == W
    assert np.all(np.abs(got - expect) <= 4 * np.spacing(np.abs(expect))), np.max(np.abs(got - expect) / np.spacing(np.abs(expect)))
    b.close()


@gpu
def test_mpc_iteration_with_a_cost():
    W, H, k = 16, 4, 3
    scene, kw, step_launches = _scene("legged20", W)
    dt, n = scene["dt"], scene["n"]
    b = batch_on_current_stream(scene, **kw)
    b.snapshot()
    ud = cuda(_schedule(scene["f_ext"], H, seed=111))
    cost = _random_cost(n, np.stack([state_rows(b)] * (H + 1)), seed=112)
    configured = _device_cost(b, cost, ud, H, dt)
    launches = b.launch_count
    winners, best, states = mpc.mpc_iteration(b, ud, dt, k, W, 0)
    # H controlled steps with the running cost, the terminal cost, gather_state, seed_state
    assert b.launch_count - launches == H * (step_launches + 1) + 3
    ew, eb = mpc.select_best(configured, k)
    assert np.array_equal(winners, ew) and np.array_equal(bits(best), bits(eb))
    assert states.shape == (k, n * S)
    # cleared: the built-in cost of egg_rollout_costs again, with the launches of the old path
    b.set_cost(None)
    built_in = torch.empty(W, dtype=torch.float64, device="cuda")
    b.restore()
    b.step_controlled(dt, ud.data_ptr(), H)
    b.rollout_costs(built_in.data_ptr())
    built_in = built_in.cpu().numpy()
    launches = b.launch_count
    winners, best, _ = mpc.mpc_iteration(b, ud, dt, k, W, 0)
    assert b.launch_count - launches == H * (step_launches + 1) + 3   # controlled steps, rollout costs, gather, seed
    ew, eb = mpc.select_best(built_in, k)
    assert np.array_equal(winners, ew) and np.array_equal(bits(best), bits(eb))
    b.close()


@gpu
def test_bad_cost_arguments_are_refused_on_the_host():
    import eggshell_b200 as E
    from eggshell_b200.batch import EggCost, EggError, EXPLICIT_EULER, _p
    W, H = 8, 3
    scene, kw, _ = _scene("legged20", W)
    dt, n = scene["dt"], scene["n"]
    b = batch_on_current_stream(scene, **dict(kw, k_max=20))
    b.step(dt)
    ud = cuda(_schedule(scene["f_ext"], H, seed=121))
    before = state_rows(b)
    f_before = b.static()[2].copy()
    good = _random_cost(n, np.stack([before] * (H + 1)), seed=122)
    b.set_cost(good)
    bytes_set = b.device_bytes
    host = np.zeros(W)
    cbuf = torch.full((W,), 7.0, dtype=torch.float64, device="cuda")

    def refused(call, code, what):
        with pytest.raises(EggError) as ei:
            call()
        assert err_code(ei) == code, f"{what}: {ei.value}"

    refused(lambda: b.step_controlled_cost(dt, ud.data_ptr(), H, host.ctypes.data), -1, "host cost_d")
    refused(lambda: b.step_controlled_cost(dt, ud.data_ptr(), H, 0), -1, "NULL cost_d")
    refused(lambda: b.step_controlled_cost(dt, host.ctypes.data, H, cbuf.data_ptr()), -1, "host u_d")
    refused(lambda: b.step_controlled_cost(dt, ud.data_ptr(), 0, cbuf.data_ptr()), -1, "horizon 0")
    refused(lambda: b.step_controlled_cost(dt, ud.data_ptr(), H, cbuf.data_ptr(), integrator=EXPLICIT_EULER), -5, "integrator")
    # egg_set_cost: non-finite weights or reference values, ref_steps < 1; the cost in place stays
    ones, ref = np.ones((n, S)), np.zeros((2, n, S))
    for q, x, rs in ((np.where(np.arange(S) == 3, np.nan, ones), None, 1), (np.where(np.arange(S) == 0, np.inf, ones), None, 1),
                     (ones, np.where(np.arange(S) == 7, -np.inf, ref), 2), (ones, ref, 0)):
        c = EggCost(_p(q), None, None, None, None, _p(x), rs)
        assert E.lib().egg_set_cost(b.h, C.byref(c)) == -1
    assert b.device_bytes == bytes_set
    for R in (2, H):   # a per-step reference shorter than H + 1 rows
        b.set_cost(mpc.QuadraticCost(n, q_run=1.0, x_ref=np.zeros((R, n, S))))
        refused(lambda: b.step_controlled_cost(dt, ud.data_ptr(), H, cbuf.data_ptr()), -1, f"{R} reference rows")
    b.set_cost(None)
    refused(lambda: b.step_controlled_cost(dt, ud.data_ptr(), H, cbuf.data_ptr()), -4, "no cost")
    assert np.array_equal(bits(state_rows(b)), bits(before))
    assert np.array_equal(bits(b.static()[2]), bits(f_before))
    assert bool((cbuf == 7.0).all())
    b.set_cost(good)   # and an accepted call still runs
    b.step_controlled_cost(dt, ud.data_ptr(), H, cbuf.data_ptr())
    assert bool(torch.isfinite(cbuf).all()) and not bool((cbuf == 7.0).any())
    b.close()
    # before egg_init: set_cost is accepted, the step is not
    raw = E.Batch(W, n, scene["nj"], solver=E.SOLVER_PGS)
    raw.set_bodies(scene["p"], scene["R"], scene["v"], scene["w"], scene["m"], scene["I"])
    raw.set_cost(good)
    refused(lambda: raw.step_controlled_cost(dt, ud.data_ptr(), H, cbuf.data_ptr()), -4, "before egg_init")
    raw.close()
