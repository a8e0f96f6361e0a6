"""Actuators: a control space of m actuator values per world (egg_set_actuators, Batch.set_actuators,
mpc.Actuators), the actuation kernel of the controlled rollouts, the row-width-generic sampler,
reduction, gather and moments kernels, and the MPPI and CEM planners in joint space with gravity.
The first tests run on the CPU; the rest need a CUDA device."""
import ctypes as C

import numpy as np
import pytest
import torch

import eggshell_b200 as E
from eggshell_b200 import mpc
from tests.mpc_helpers import (ZERO_G_PGS, _u01, batch_on_current_stream, bits, boxes, clamp, cuda, err_code, philox4x32_10,
                               run_ranks, state_rows)

gpu = pytest.mark.gpu
S = mpc.STATE_PER_BODY


# ---- helpers --------------------------------------------------------------------------------------
def random_table(n, m, rng):
    """m actuators on n bodies with every kind of reaction and frame, and axes of mixed magnitudes."""
    body = rng.integers(0, n, m)
    reaction = rng.integers(-1, n, m)
    reaction = np.where(reaction == body, (body + 1) % n if n > 1 else -1, reaction)
    kind = rng.integers(0, 3, m)
    frame = np.where(kind == 0, -1, np.where(kind == 1, body, reaction))
    axis = rng.normal(size=(m, 3)) * 10.0 ** rng.uniform(-2, 2, size=(m, 1))
    return mpc.Actuators(n, body, reaction, frame, axis)


def noise_rows(H, c, g, seed, iteration):
    """eps [H, len(g), c] of the global worlds g for a control row of width c: Philox counter
    q = t ceil(c / 2) + p for the elements (2p, 2p + 1); for odd c the last second normal is dropped."""
    P = (c + 1) // 2
    t, w, p = np.meshgrid(np.arange(H), np.arange(len(g)), np.arange(P), indexing="ij")
    q = (t * P + p).astype(np.uint64)
    gg = np.asarray(g, dtype=np.uint64)[w]
    r = philox4x32_10([q, gg, np.uint64(iteration & 0xffffffff), np.uint64(iteration >> 32)],
                      [np.uint64(seed & 0xffffffff), np.uint64(seed >> 32)])
    u1, u2 = _u01(r[0], r[1]), _u01(r[2], r[3])
    rad = np.sqrt(-2.0 * np.log(u1))
    eps = np.stack([rad * np.cos(2 * np.pi * u2), rad * np.sin(2 * np.pi * u2)], axis=-1)
    return eps.reshape(H, len(g), 2 * P)[..., :c]


def moments_numpy(rows):
    """(mean, population std) of rows [k, ...] as egg_control_moments defines them."""
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


# Device arguments are held in variables until their call has been enqueued: a temporary would be
# freed at once, and the next argument's copy could reuse its memory before the kernel reads it.
def gpu_tensor(shape, fill=np.nan):
    return torch.full(shape, fill, dtype=torch.float64, device="cuda")


def actuated(scene, act, **kw):
    b = batch_on_current_stream(scene, **kw)
    b.set_actuators(act)
    return b


# ---- CPU ------------------------------------------------------------------------------------------
def test_actuators_validate():
    a = mpc.Actuators(3, [0, 2, 1], [-1, 0, 2], [-1, 2, 1], [[1, 0, 0], [0, 2.5, 0], [0, 0, -1e-3]])
    assert a.m == 3 and a.n == 3 and a.body.dtype == np.int32 and a.axis.shape == (3, 3)
    good = dict(body=[0, 1], reaction=[1, -1], frame=[1, -1], axis=[[1.0, 0, 0], [0, 0, 1.0]])
    bad = [dict(body=[0, 3]), dict(body=[-1, 1]), dict(reaction=[0, -1]), dict(reaction=[-2, -1]), dict(reaction=[3, -1]),
           dict(frame=[2, -1]), dict(frame=[1, 0]), dict(frame=[-2, -1]), dict(frame=[-1, 0]),
           dict(axis=[[0, 0, 0], [0, 0, 1.0]]), dict(axis=[[np.nan, 0, 1], [0, 0, 1.0]]), dict(axis=[[np.inf, 0, 0], [0, 0, 1.0]]),
           dict(axis=[[1.0, 0, 0]]), dict(axis=np.ones((2, 2))), dict(body=[0]), dict(frame=[1, -1, -1]),
           dict(body=[], reaction=[], frame=[], axis=np.zeros((0, 3))), dict(body=[0.0, 1.0]), dict(body=[[0, 1]])]
    mpc.Actuators(3, **good)
    for kw in bad:
        args = dict(good)
        args.update(kw)
        with pytest.raises(ValueError):
            mpc.Actuators(3, **args)
    with pytest.raises(ValueError):
        mpc.Actuators(0, **good)
    # three unit motors per ball joint: child, parent reaction, parent frame; world anchor: world axes
    j = mpc.Actuators.ball_joint_motors(4, [0, 1, 3], [1, 2, -1])
    assert j.m == 9 and list(j.body) == [1] * 3 + [2] * 3 + [3] * 3 and list(j.reaction) == [0] * 3 + [1] * 3 + [-1] * 3
    assert list(j.frame) == list(j.reaction) and np.array_equal(j.axis, np.tile(np.eye(3), (3, 1)))
    legged = E.scenes.legged20_motors()
    assert legged.m == 57 and legged.n == 20 and (legged.reaction >= 0).all() and (legged.frame == legged.reaction).all()


def _random_rows(lead, n, rng):
    q = rng.normal(size=lead + (n, 4))
    q /= np.linalg.norm(q, axis=-1, keepdims=True)
    R = E.scenes.quat_to_mat(q).reshape(lead + (n, 9))
    return np.concatenate([rng.normal(size=lead + (n, 3)), R, rng.normal(size=lead + (n, 6))], axis=-1)


def test_wrench_definition():
    rng = np.random.default_rng(1)
    n, W = 6, 5
    x = _random_rows((W,), n, rng)
    mass = rng.uniform(0.5, 2.0, size=(W, n))
    g = np.array([0.3, -0.2, -9.8])
    a = random_table(n, 11, rng)
    u = rng.normal(size=(W, a.m))
    f = a.wrench(x, u, mass, g)
    assert f.shape == (W, n, 6)
    assert np.array_equal(bits(f[..., :3]), bits(mass[..., None] * g)), "the force slots are m g"
    # one actuator with a reaction: +tau and -tau sum to exactly zero; the other bodies get nothing
    one = mpc.Actuators(n, [2], [4], [4], [rng.normal(size=3)])
    f1 = one.wrench(x, u[:, :1], mass, g)
    assert not (f1[:, 2, 3:] + f1[:, 4, 3:]).any() and f1[:, 2, 3:].any()
    assert not np.delete(f1[..., 3:], [2, 4], axis=1).any()
    # frame = -1: u axis exactly
    ax = rng.normal(size=3)
    fw = mpc.Actuators(n, [1], [-1], [-1], [ax]).wrench(x, u[:, :1], mass, g)
    assert np.array_equal(bits(fw[:, 1, 3:]), bits(u[:, :1] * ax))
    # a body frame: R k with the sums in the order of the definition
    fb = mpc.Actuators(n, [1], [3], [3], [ax]).wrench(x, u[:, :1], mass, g)
    R = x[:, 3, 3:12].reshape(W, 3, 3)
    k = (R[:, :, 0] * ax[0] + R[:, :, 1] * ax[1]) + R[:, :, 2] * ax[2]
    assert np.array_equal(bits(fb[:, 1, 3:]), bits(u[:, :1] * k))
    assert np.allclose(fb[:, 1, 3:], u[:, :1] * np.einsum("wij,j->wi", R, ax), rtol=0, atol=1e-14 * np.abs(u).max() * np.abs(ax).max())
    # the torques of a table are the sum of its actuators' torques (to rounding), and they balance
    # when every actuator has a reaction
    parts = sum(mpc.Actuators(n, a.body[i:i + 1], a.reaction[i:i + 1], a.frame[i:i + 1], a.axis[i:i + 1]).wrench(x, u[:, i:i + 1], mass, g)[..., 3:]
                for i in range(a.m))
    assert np.allclose(f[..., 3:], parts, rtol=1e-12, atol=1e-12 * np.abs(f[..., 3:]).max())
    closed = mpc.Actuators(n, a.body, np.where(a.reaction < 0, (a.body + 1) % n, a.reaction), a.frame, a.axis)
    assert np.abs(closed.wrench(x, u, mass, g)[..., 3:].sum(axis=1)).max() <= 1e-12 * np.abs(f[..., 3:]).max()
    # ball-joint motors of legged20 on its own scene
    s = E.scenes.legged20(2)
    legged = E.scenes.legged20_motors()
    xl = np.concatenate([s["p"], s["R"].reshape(2, 20, 9), s["v"], s["w"]], axis=-1)
    fl = legged.wrench(xl, np.ones((2, 57)), s["m"], [0, 0, -9.8])
    assert fl.shape == (2, 20, 6) and np.array_equal(fl[..., 2], np.full((2, 20), -9.8))
    with pytest.raises(ValueError):
        a.wrench(x, u[:, :3], mass, g)


@pytest.mark.parametrize("m", [5, 6])
def test_planner_and_cost_shapes_with_m(m):
    n, H, W = 3, 4, 2
    rng = np.random.default_rng(m)
    sig = rng.uniform(0.1, 1.0, size=m)
    p = mpc.MPPI(n, H, sigma=sig, lam=0.5, u_lo=-2.0, u_hi=np.arange(m) + 1.0, seed=3, m=m, device="cpu")
    assert p.control_shape == (m,) and p.sigma.shape == (m,) and p.u_lo.shape == (m,) and p.u_hi.shape == (m,)
    assert tuple(p.u_nom.shape) == (H, m) and not p.u_nom.any()
    assert torch.equal(p.clamp(torch.full((H, m), 100.0, dtype=torch.float64))[1], torch.arange(m, dtype=torch.float64) + 1.0)
    c = mpc.CEM(n, H, sigma=0.5, n_elite=2, u_nom=np.arange(m, dtype=float), m=m, device="cpu")
    assert c.control_shape == (m,) and tuple(c.std.shape) == (H, m) and (c.std == 0.5).all()
    assert (c.u_nom[3].numpy() == np.arange(m)).all()
    assert mpc.MPPI(n, H, sigma=1.0, lam=1.0, device="cpu").control_shape == (n, 6)
    for kw in (dict(sigma=np.ones((n, 6))), dict(sigma=np.ones(m + 1)), dict(u_nom=np.ones((H, n, 6))), dict(u_lo=np.ones(m + 1)),
               dict(m=0), dict(m=-1)):
        args = dict(sigma=1.0, lam=1.0, device="cpu", m=m)
        args.update(kw)
        with pytest.raises(ValueError):
            mpc.MPPI(n, H, **args)
    with pytest.raises(ValueError):
        mpc.CEM(n, H, sigma=np.ones(m + 1), n_elite=1, m=m, device="cpu")
    # the cost: u_run [m], evaluate(states, u [H, W, m])
    ur = rng.uniform(0.0, 1.0, size=m)
    q = mpc.QuadraticCost(n, q_term=1.0, u_run=ur, m=m)
    assert q.control_shape == (m,) and q.u_run.shape == (m,)
    states = rng.normal(size=(H + 1, W, n, S))
    u = rng.normal(size=(H, W, m))
    J = q.evaluate(states, u)
    expect = (ur * u ** 2).sum(axis=(0, 2)) + (states[H] ** 2).sum(axis=(1, 2))
    assert np.allclose(J, expect, rtol=1e-13)
    with pytest.raises(ValueError):
        q.evaluate(states, rng.normal(size=(H, W, n, 6)))
    with pytest.raises(ValueError):
        q.evaluate(states, rng.normal(size=(H, W, m + 1)))
    with pytest.raises(ValueError):
        mpc.QuadraticCost(n, u_run=np.ones(m + 1), m=m)
    with pytest.raises(ValueError):
        mpc.QuadraticCost(n, m=0)
    assert mpc.QuadraticCost(n).control_shape == (n, 6)


# ---- GPU: the actuation kernel --------------------------------------------------------------------
def _free_bodies(W, n, rng, gravity=(0.3, -0.2, -9.8)):
    """n boxes per world far apart and above the ground (no contacts) with random state and masses."""
    s = boxes(W, n)
    s["p"][:, :, 0] = 3.0 * np.arange(n)
    s["p"][:, :, 2] = 50.0
    x = _random_rows((W,), n, rng)
    s["R"] = x[..., 3:12].reshape(W, n, 3, 3)
    s["v"], s["w"] = x[..., 12:15], x[..., 15:18]
    s["m"] = rng.uniform(0.5, 2.0, size=(W, n))
    s["I"] = s["m"][..., None, None] * np.diag([0.02, 0.015, 0.01])
    return s, dict(solver=E.SOLVER_PGS, gravity=gravity)


@gpu
@pytest.mark.parametrize("m", [41, 40])
def test_slot_bits(m):
    """One actuated step on random states, random axes and all three frame kinds: the f_ext slot is
    Actuators.wrench of the state before the step, bit for bit (37 bodies: lanes take two bodies)."""
    rng = np.random.default_rng(m)
    W, n = 70, 37
    g = (0.3, -0.2, -9.8)
    scene, kw = _free_bodies(W, n, rng, g)
    act = random_table(n, m, rng)
    b = actuated(scene, act, **kw)
    x0 = state_rows(b)
    u = rng.normal(size=(1, W, m)) * 10.0 ** rng.uniform(-1, 1, size=(1, W, m))
    ud = cuda(u)
    launches = b.launch_count
    b.step(scene["dt"])
    step_launches = b.launch_count - launches
    b.set_state(scene["p"], scene["R"], scene["v"], scene["w"])
    launches = b.launch_count
    b.step_controlled(scene["dt"], ud.data_ptr(), 1)
    assert b.launch_count - launches == step_launches + 1
    f = b.static()[2]
    expect = act.wrench(x0, u[0], scene["m"], g)
    assert np.array_equal(bits(f), bits(expect))
    assert np.abs(expect[..., 3:]).max() > 1.0 and (act.frame == -1).any() and (act.frame == act.body).any() and (act.frame == act.reaction).any()
    b.close()


def _legged(W, lift=0.0, gravity=(0.0, 0.0, -9.8), v0=None):
    s = E.scenes.legged20(W)
    s["p"][..., 2] += lift
    if v0 is not None:
        s["v"][:] = v0
    del s["f_ext"]
    return s, dict(solver=E.SOLVER_PGS, k_max=100, gravity=gravity)


@gpu
def test_rollout_matches_stepwise_numpy_wrench():
    """legged20 with its 57 joint motors in gravity: an actuated rollout against a second batch stepped
    one step at a time with body wrenches, the numpy wrench of its own state; every state bit and
    status word equal.  Then the cost against QuadraticCost.evaluate, and J in batches of other W."""
    W, H = 16, 8
    scene, kw = _legged(W)
    dt, n = scene["dt"], scene["n"]
    act = E.scenes.legged20_motors()
    rng = np.random.default_rng(2)
    u = rng.normal(0.0, 2.0, size=(H, W, act.m))
    ud = cuda(u)
    a = actuated(scene, act, **kw)
    a.step_controlled(dt, ud.data_ptr(), H)
    ref = batch_on_current_stream(scene, **kw)
    states = [state_rows(ref)]
    for t in range(H):
        f = act.wrench(states[-1], u[t], scene["m"], kw["gravity"])
        dev_arg = cuda(f[None])
        ref.step_controlled(dt, dev_arg.data_ptr(), 1)
        states.append(state_rows(ref))
    states = np.stack(states)
    assert np.array_equal(bits(state_rows(a)), bits(states[H]))
    assert np.array_equal(a.status()["status"], ref.status()["status"])
    assert np.array_equal(bits(a.static()[2]), bits(ref.static()[2])), "the slot holds the last step's wrench"
    assert (ref.status()["n_contacts"] > 0).all() and np.abs(states[H] - states[0]).max() > 1e-3
    # the same rollout with a cost
    x0 = states[0, 0]
    cost = mpc.QuadraticCost(n, q_run=rng.uniform(0, 1, size=(n, S)), l_run=rng.normal(size=(n, S)), u_run=rng.uniform(0, 1, size=act.m),
                             q_term=rng.uniform(0, 1, size=(n, S)), l_term=rng.normal(size=(n, S)),
                             x_ref=x0 + rng.normal(0, 0.1, size=(H + 1, n, S)), m=act.m)
    c = actuated(scene, act, **kw)
    c.set_cost(cost)
    J = torch.empty(W, dtype=torch.float64, device="cuda")
    c.step_controlled_cost(dt, ud.data_ptr(), H, J.data_ptr())
    J = J.cpu().numpy()
    assert np.array_equal(bits(state_rows(c)), bits(states[H]))
    expect = cost.evaluate(states, u)
    assert np.all(np.abs(J - expect) <= 1e-12 * np.abs(expect)), np.abs(J / expect - 1).max()
    for Wk in (5, 1):
        sk = {k: (v[:Wk] if isinstance(v, np.ndarray) and v.ndim >= 2 and v.shape[0] == W else v) for k, v in scene.items()}
        sk["W"] = Wk
        ck = actuated(sk, act, **kw)
        ck.set_cost(cost)
        Jk = torch.empty(Wk, dtype=torch.float64, device="cuda")
        dev_arg = cuda(u[:, :Wk])
        ck.step_controlled_cost(dt, dev_arg.data_ptr(), H, Jk.data_ptr())
        assert np.array_equal(bits(Jk.cpu().numpy()), bits(J[:Wk])), Wk
        ck.close()
    for x in (a, ref, c):
        x.close()


@gpu
def test_torque_pair_physics_and_momentum():
    """Two free bodies in zero gravity, one torque pair with a world axis: I1 dw1 = tau dt = -I2 dw2.
    legged20 lifted off the ground in zero gravity under random motor torques: total momentum kept."""
    rng = np.random.default_rng(4)
    scene, kw = _free_bodies(3, 2, rng, gravity=(0.0, 0.0, 0.0))
    scene["w"][:] = 0.0   # at rest: no gyroscopic term
    dt = scene["dt"]
    axis = rng.normal(size=3)
    act = mpc.Actuators(2, [0], [1], [-1], [axis])
    b = actuated(scene, act, **kw)
    u = np.array([2.5, -0.7, 13.0])[None, :, None]
    dev_arg = cuda(u)
    b.step_controlled(dt, dev_arg.data_ptr(), 1)
    w1 = b.bodies()[3]
    for w in range(3):
        tau = u[0, w, 0] * axis * dt
        for k, sign in ((0, 1.0), (1, -1.0)):
            R = scene["R"][w, k]
            Iw = R @ scene["I"][w, k] @ R.T
            assert np.abs(Iw @ w1[w, k] - sign * tau).max() <= 1e-12 * np.abs(tau).max(), (w, k)
    b.close()
    # momentum of the legged robot in free fall without gravity
    W, H = 4, 20
    scene, kw = _legged(W, lift=1.0, gravity=(0.0, 0.0, 0.0), v0=(0.3, -0.2, 0.1))
    motors = E.scenes.legged20_motors()
    b = actuated(scene, motors, **kw)
    P0 = (scene["m"][..., None] * b.bodies()[2]).sum(axis=1)
    u = cuda(rng.normal(0.0, 1.0, size=(H, W, motors.m)))
    b.step_controlled(scene["dt"], u.data_ptr(), H)
    p, R, v, w = b.bodies()
    P = (scene["m"][..., None] * v).sum(axis=1)
    assert np.abs(P - P0).max() <= 1e-10 * np.abs(P0).max(), np.abs(P - P0).max()
    assert np.abs(w).max() > 0.1 and (p[..., 2] > 0.5).all()
    assert not b.status()["status"].any()
    b.close()


# ---- GPU: width-generic planner kernels ------------------------------------------------------------
def _table_batch(W, n, m, seed=0):
    rng = np.random.default_rng(seed)
    act = random_table(n, m, rng)
    return actuated(boxes(W, n), act, **ZERO_G_PGS), act


@gpu
@pytest.mark.parametrize("m", [7, 8])
def test_sampler_rows_match_numpy(m):
    W, n, H, first = 300, 4, 3, 1000
    b, _ = _table_batch(W, n, m)
    rng = np.random.default_rng(m)
    lo, hi = rng.uniform(-3.0, -1.5, size=m), rng.uniform(1.5, 3.0, size=m)
    p = mpc.MPPI(n, H, sigma=rng.uniform(0.2, 1.0, size=m), lam=1.0, u_lo=lo, u_hi=hi, seed=0x1234_5678_9abc_def0,
                 u_nom=rng.normal(0.0, 0.3, size=(H, m)), m=m)
    p.iteration = 2 ** 32 + 5
    b.set_sampler(p)
    u = gpu_tensor((H, W, m))
    launches = b.launch_count
    b.sample_controls(p.u_nom.data_ptr(), H, p.seed, p.iteration, first, u.data_ptr())
    assert b.launch_count - launches == 1
    un = p.u_nom.cpu().numpy()[:, None]
    got = u.cpu().numpy()
    eps = noise_rows(H, m, np.arange(first, first + W), p.seed, p.iteration)
    inside = (got > lo) & (got < hi)
    assert inside.mean() > 0.9 and (got == lo).any() and (got == hi).any()
    assert np.max(np.abs(((got - un) / p.sigma - eps)[inside])) <= 1e-13
    assert np.array_equal(got == lo, clamp(un + p.sigma * eps, lo, hi) == lo)
    # per-step std, and global world 0
    std = rng.uniform(0.2, 2.0, size=(H, m))
    dev_arg = cuda(std)
    b.sample_controls_std(p.u_nom.data_ptr(), dev_arg.data_ptr(), H, p.seed, 3, 0, u.data_ptr())
    got = u.cpu().numpy()
    assert np.array_equal(bits(got[:, 0]), bits(clamp(un[:, 0], lo, hi)))
    eps = noise_rows(H, m, np.arange(W), p.seed, 3)
    inside = (got > lo) & (got < hi)
    assert np.max(np.abs(((got - un) / std[:, None] - eps)[:, 1:][inside[:, 1:]])) <= 1e-13
    b.close()


@gpu
def test_table_of_width_6n_samples_the_body_wrench_bits():
    W, n, H, first = 200, 3, 4, 77
    rng = np.random.default_rng(6)
    sigma, lo, hi = rng.uniform(0.2, 1.0, size=(n, 6)), rng.uniform(-2.0, -1.0, size=(n, 6)), rng.uniform(1.0, 2.0, size=(n, 6))
    un = rng.normal(0.0, 0.5, size=(H, n, 6))
    body = batch_on_current_stream(boxes(W, n), defaults=ZERO_G_PGS)
    joint, _ = _table_batch(W, n, 6 * n)
    pb = mpc.MPPI(n, H, sigma=sigma, lam=1.0, u_lo=lo, u_hi=hi, seed=42, u_nom=un)
    pj = mpc.MPPI(n, H, sigma=sigma.ravel(), lam=1.0, u_lo=lo.ravel(), u_hi=hi.ravel(), seed=42, u_nom=un.reshape(H, 6 * n), m=6 * n)
    body.set_sampler(pb)
    joint.set_sampler(pj)
    std = cuda(rng.uniform(0.0, 1.5, size=(H, n, 6)))
    for it in (0, 2 ** 33 + 1):
        ub, uj = gpu_tensor((H, W, n, 6)), gpu_tensor((H, W, 6 * n))
        body.sample_controls(pb.u_nom.data_ptr(), H, 42, it, first, ub.data_ptr())
        joint.sample_controls(pj.u_nom.data_ptr(), H, 42, it, first, uj.data_ptr())
        assert np.array_equal(bits(ub.cpu().numpy().reshape(H, W, 6 * n)), bits(uj.cpu().numpy())), it
        body.sample_controls_std(pb.u_nom.data_ptr(), std.data_ptr(), H, 42, it, first, ub.data_ptr())
        joint.sample_controls_std(pj.u_nom.data_ptr(), std.data_ptr(), H, 42, it, first, uj.data_ptr())
        assert np.array_equal(bits(ub.cpu().numpy().reshape(H, W, 6 * n)), bits(uj.cpu().numpy())), it
    body.close()
    joint.close()


@gpu
@pytest.mark.parametrize("m", [7, 8])
def test_reduce_gather_moments_at_width_m(m):
    W, n, H = 1000, 4, 3   # 4 reduction chunks, the last one partial
    b, _ = _table_batch(W, n, m)
    rng = np.random.default_rng(10 + m)
    u = rng.normal(size=(H, W, m))
    ud = cuda(u)
    cost = rng.uniform(0.0, 3.0, size=W)
    cost[[5, 300]] = [np.nan, np.inf]
    base = np.min(cost[np.isfinite(cost)])
    lam = 0.7
    L = H * m
    out = gpu_tensor((L + 2,))
    launches = b.launch_count
    cd, bd = cuda(cost), cuda(np.array(base))
    b.mppi_reduce(ud.data_ptr(), H, cd.data_ptr(), bd.data_ptr(), lam, out.data_ptr())
    assert b.launch_count - launches == 2
    got = out.cpu().numpy()
    om = np.where(np.isfinite(cost), np.exp(-(np.where(np.isfinite(cost), cost, 0.0) - base) / lam), 0.0)
    s = np.einsum("w,twc->tc", om, u)
    sabs = np.einsum("w,twc->tc", om, np.abs(u))
    assert np.all(np.abs(got[:L] - s.ravel()) <= 1e-12 * sabs.ravel())
    assert abs(got[L] - om.sum()) <= 1e-12 * om.sum() and abs(got[L + 1] - (om * om).sum()) <= 1e-12 * (om * om).sum()
    worlds = [W - 1, 5, 0, 5, 417]
    g = gpu_tensor((len(worlds), H, m), 7.0)
    b.gather_controls(ud.data_ptr(), H, worlds, g.data_ptr())
    assert np.array_equal(bits(g.cpu().numpy()), bits(u[:, worlds].transpose(1, 0, 2)))
    for k in (1, 37):
        rows = rng.normal(size=(k, H, m)) * 10.0 ** rng.integers(-4, 4, size=(1, H, m))
        mo = gpu_tensor((2, H, m))
        dev_arg = cuda(rows)
        b.control_moments(dev_arg.data_ptr(), k, H, mo.data_ptr())
        mean, std = moments_numpy(rows)
        assert np.array_equal(bits(mo.cpu().numpy()), bits(np.stack([mean, std]))), k
    b.close()


# ---- GPU: state rules ------------------------------------------------------------------------------
@gpu
def test_set_actuators_state_rules():
    from eggshell_b200.batch import EggActuators, EggError, _p
    W, n, H = 32, 3, 2
    scene = boxes(W, n)
    dt = scene["dt"]
    rng = np.random.default_rng(8)
    b = batch_on_current_stream(scene, defaults=ZERO_G_PGS)
    b.snapshot()
    base_bytes = b.device_bytes
    act = random_table(n, 5, rng)
    b.set_actuators(act)
    assert b.control_shape == (5,) and b.actuators is act and b.device_bytes > base_bytes
    with_table = b.device_bytes

    def refused(call, code, what):
        with pytest.raises(EggError) as ei:
            call()
        assert err_code(ei) == code, f"{what}: {ei.value}"

    # a sampler or a cost of the wrong control shape is refused in Python; of the right one it blocks set_actuators
    with pytest.raises(ValueError):
        b.set_sampler(mpc.MPPI(n, H, sigma=1.0, lam=1.0))
    with pytest.raises(ValueError):
        b.set_cost(mpc.QuadraticCost(n))
    b.set_sampler(mpc.MPPI(n, H, sigma=1.0, lam=1.0, m=5))
    refused(lambda: b.set_actuators(None), -4, "sampler set")
    refused(lambda: b.set_actuators(random_table(n, 4, rng)), -4, "sampler set")
    b.set_sampler(None)
    b.set_cost(mpc.QuadraticCost(n, u_run=1.0, m=5))
    refused(lambda: b.set_actuators(None), -4, "cost set")
    b.set_cost(None)
    assert b.device_bytes == with_table and b.actuators is act
    # malformed tables at the C ABI: EGG_ERR_ARG, the old table stays
    L = E.lib()

    def raw(m, body, reaction, frame, axis):
        arrs = [np.ascontiguousarray(body, dtype=np.int32), np.ascontiguousarray(reaction, dtype=np.int32),
                np.ascontiguousarray(frame, dtype=np.int32), np.ascontiguousarray(axis, dtype=np.float64)]
        return L.egg_set_actuators(b.h, C.byref(EggActuators(m, *[_p(x) for x in arrs]))), arrs

    ok = ([0, 1], [1, -1], [-1, 0], [[1.0, 0, 0], [0, 1, 0]])
    for m_, bo, re, fr, ax in ((0, *ok), (2, [0, 3], *ok[1:]), (2, [0, -1], *ok[1:]), (2, ok[0], [0, -1], *ok[2:]),
                               (2, ok[0], [1, -2], *ok[2:]), (2, ok[0], [1, 3], *ok[2:]), (2, *ok[:2], [2, 0], ok[3]),
                               (2, *ok[:2], [-1, 2], ok[3]), (2, *ok[:3], [[0, 0, 0], [0, 1, 0]]), (2, *ok[:3], [[np.nan, 0, 0], [0, 1, 0]]),
                               (2, *ok[:3], [[1, 0, 0], [0, np.inf, 0]])):
        rc, _ = raw(m_, bo, re, fr, ax)
        assert rc == -1, (m_, bo, re, fr, ax)
    assert L.egg_set_actuators(b.h, C.byref(EggActuators(2, None, None, None, None))) == -1
    assert b.device_bytes == with_table
    u = rng.normal(size=(1, W, 5))
    b.restore()
    x0 = state_rows(b)
    dev_arg = cuda(u)
    b.step_controlled(dt, dev_arg.data_ptr(), 1)
    assert np.array_equal(bits(b.static()[2]), bits(act.wrench(x0, u[0], scene["m"], (0.0, 0.0, 0.0)))), "the old table is in use"
    # NULL: body wrenches again, memory released, and a body-wrench rollout bit-identical to a fresh batch's
    b.set_actuators(None)
    assert b.control_shape == (n, 6) and b.actuators is None and b.device_bytes == base_bytes
    uw = cuda(rng.normal(size=(3, W, n, 6)))
    b.restore()
    b.step_controlled(dt, uw.data_ptr(), 3)
    fresh = batch_on_current_stream(scene, defaults=ZERO_G_PGS)
    fresh.step_controlled(dt, uw.data_ptr(), 3)
    assert np.array_equal(bits(state_rows(b)), bits(state_rows(fresh)))
    assert np.array_equal(bits(b.static()[2]), bits(fresh.static()[2]))
    fresh.close()
    # a table set before egg_init works the same
    pre = E.Batch(W, n, 0, **ZERO_G_PGS)
    pre.set_stream(torch.cuda.current_stream().cuda_stream)
    pre.set_actuators(act)
    pre.set_bodies(scene["p"], scene["R"], scene["v"], scene["w"], scene["m"], scene["I"])
    pre.init()
    dev_arg = cuda(u)
    pre.step_controlled(dt, dev_arg.data_ptr(), 1)
    b.set_actuators(act)
    b.restore()
    dev_arg = cuda(u)
    b.step_controlled(dt, dev_arg.data_ptr(), 1)
    assert np.array_equal(bits(state_rows(pre)), bits(state_rows(b)))
    pre.close()
    b.close()


# ---- GPU: planners in joint space with gravity ------------------------------------------------------
ARM_TARGET = (0.5, 0.0, 1.6)   # the tip link's centre: 0.64 m from the anchor, up and to the side


def _arm(W, dt=0.02):
    """A two-link arm anchored to the world at (0, 0, 2) by a hinge about y and hinged to its second
    link about the first link's y axis, hanging in gravity; far above the ground, and the links 0.5 m
    apart so that they never touch.  Its two motors drive the two hinges; the tip is link 1's centre."""
    s = E.scenes._base(W, 2)
    s["p"][:, 0] = (0.0, 0.0, 1.75)
    s["p"][:, 1] = (0.0, 0.0, 1.25)
    js = E.scenes.hinge(0, -1, (0, 0, 0.25), (0, 0, 2.0), (0, 1, 0), (0, 1, 0))
    js += E.scenes.hinge(0, 1, (0, 0, -0.25), (0, 0, 0.25), (0, 1, 0), (0, 1, 0))
    s.update(nj=4, i0=np.array([j[0] for j in js], dtype=np.int32), i1=np.array([j[1] for j in js], dtype=np.int32),
             c0=np.tile(np.array([j[2] for j in js]), (W, 1, 1)), c1=np.tile(np.array([j[3] for j in js]), (W, 1, 1)), dt=dt, name="arm")
    act = mpc.Actuators(2, [0, 1], [-1, 0], [-1, 0], [[0, 1.0, 0], [0, 1.0, 0]])
    return s, act


def _arm_task(W, rank=0, ws=1):
    lo, hi = mpc.shard_range(W, rank, ws)
    scene, act = _arm(W)
    for key in ("p", "R", "v", "w", "m", "I", "c0", "c1"):
        scene[key] = scene[key][lo:hi].copy()
    scene["W"] = hi - lo
    b = actuated(scene, act, solver=E.SOLVER_PGS, device=torch.cuda.current_device())
    b.snapshot()
    x0 = state_rows(b)[0]
    q_term = np.zeros((2, S))
    q_term[1, 0:3] = 10.0
    x_ref = x0.copy()
    x_ref[1, 0:3] = ARM_TARGET
    b.set_cost(mpc.QuadraticCost(2, q_term=q_term, u_run=1e-4, x_ref=x_ref, m=2))
    return b, scene, lo, hi


@gpu
@pytest.mark.parametrize("planner", ["mppi", "cem"])
def test_planners_reach_with_a_hinged_arm_in_gravity(planner):
    """The arm must swing its tip to a target 0.64 m from the anchor within H steps, against gravity,
    through its two joint motors.  The nominal plan of zeros leaves it hanging (J = 10 |tip - target|^2
    = 3.7).  The threshold comes from one run on a B200: after 13 iterations MPPI's nominal plan cost
    0.020 and CEM's 0.013 of the initial cost; 0.1 leaves a margin of 5."""
    W, H, iters = 1024, 25, 12
    b, scene, _, _ = _arm_task(W)
    dt = scene["dt"]
    if planner == "mppi":
        p = mpc.MPPI(2, H, sigma=5.0, lam=0.1, u_lo=-20.0, u_hi=20.0, seed=2024, m=2)
    else:
        p = mpc.CEM(2, H, sigma=5.0, n_elite=64, alpha=0.1, sigma_min=0.1, u_lo=-20.0, u_hi=20.0, seed=2024, m=2)
    b.set_sampler(p)
    u = torch.empty((H, W, 2), dtype=torch.float64, device="cuda")
    step = mpc.mppi_iteration if planner == "mppi" else (lambda b_, p_, dt_, u_, f_: mpc.cem_iteration(b_, p_, dt_, u_, f_, W))
    costs = [step(b, p, dt, u, 0)["nominal_cost"] for _ in range(iters)]
    last = step(b, p, dt, u, 0)["nominal_cost"]
    print(planner, "nominal cost per iteration", costs + [last])
    assert costs[0] == pytest.approx(10.0 * (0.5 ** 2 + 0.35 ** 2), rel=1e-2)
    assert last < 0.1 * costs[0], costs + [last]
    assert not b.status()["status"].any()
    b.close()


@gpu
@pytest.mark.parametrize("planner", ["mppi", "cem"])
def test_advance_in_actuator_space(planner):
    W, H = 8, 4
    scene, kw = _legged(W)
    dt, n = scene["dt"], scene["n"]
    act = E.scenes.legged20_motors()
    b = actuated(scene, act, **kw)
    b.snapshot()
    rng = np.random.default_rng(21)
    sigma = rng.uniform(0.5, 2.0, size=act.m)
    common = dict(u_lo=-3.0, u_hi=3.0, seed=5, u_nom=rng.normal(0.0, 3.0, size=(H, act.m)), m=act.m)
    if planner == "mppi":
        p = mpc.MPPI(n, H, sigma=sigma, lam=1.0, **common)
    else:
        p = mpc.CEM(n, H, sigma=sigma, n_elite=3, alpha=0.5, **common)
    b.set_sampler(p)
    u = torch.empty((H, W, act.m), dtype=torch.float64, device="cuda")
    if planner == "mppi":
        mpc.mppi_iteration(b, p, dt, u, 0)
    else:
        mpc.cem_iteration(b, p, dt, u, 0, W)
    plan = p.u_nom.cpu().numpy()
    executed, start = (mpc.mppi_advance(b, p, dt, W) if planner == "mppi" else mpc.cem_advance(b, p, dt, W))
    c0 = clamp(plan[0], -3.0, 3.0)
    assert np.array_equal(bits(executed.cpu().numpy()), bits(c0))
    fresh = actuated(scene, act, **kw)
    dev_arg = cuda(np.broadcast_to(c0, (1, W, act.m)))
    fresh.step_controlled(dt, dev_arg.data_ptr(), 1)
    expect = state_rows(fresh)[0]
    fresh.close()
    assert np.array_equal(bits(state_rows(b)), bits(np.broadcast_to(expect, (W, n, S))))
    assert np.array_equal(bits(start.cpu().numpy()), bits(expect))
    got = p.u_nom.cpu().numpy()
    assert np.array_equal(bits(got[:-1]), bits(plan[1:])) and np.array_equal(bits(got[-1]), bits(plan[-1]))
    if planner == "cem":
        assert np.array_equal(bits(p.std.cpu().numpy()[-1]), bits(sigma))
    b.close()


def _run_arm(rank, ws, W, H, iters):
    b, scene, lo, hi = _arm_task(W, rank, ws)
    p = mpc.CEM(2, H, sigma=5.0, n_elite=32, alpha=0.2, sigma_min=0.1, u_lo=-20.0, u_hi=20.0, seed=77, m=2)
    b.set_sampler(p)
    u = torch.empty((H, hi - lo, 2), dtype=torch.float64, device=torch.device("cuda", torch.cuda.current_device()))
    m = mpc.MPPI(2, H, sigma=5.0, lam=0.1, u_lo=-20.0, u_hi=20.0, seed=78, m=2)
    plans = []
    for _ in range(iters):
        mpc.cem_iteration(b, p, scene["dt"], u, lo, W)
        plans += [p.u_nom.cpu().numpy(), p.std.cpu().numpy()]
    b.set_sampler(m)
    for _ in range(iters):
        mpc.mppi_iteration(b, m, scene["dt"], u, lo)
        plans.append(m.u_nom.cpu().numpy())
    b.close()
    return plans


@gpu
def test_joint_space_plans_on_one_rank_and_two_nccl_ranks():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    W, H, iters = 513, 6, 3   # uneven shards
    one = _run_arm(0, 1, W, H, iters)
    res = run_ranks(_run_arm, 2, "nccl", W, H, iters, timeout=300)
    for r in range(2):
        for a, b in zip(res[r], one):
            assert np.array_equal(bits(a), bits(b)), r
