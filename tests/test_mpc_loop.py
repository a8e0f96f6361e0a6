"""Receding-horizon MPC: per-step control schedules (egg_step_controlled), the winners' terminal
states fetched on the device (egg_gather_state, mpc.gather_winner_states) and every world re-seeded
from them (egg_seed_state, mpc.mpc_iteration).  The first test runs on CPU ranks (gloo); the rest
need a CUDA device."""
import numpy as np
import pytest
import torch

from eggshell_b200 import mpc
from tests.mpc_helpers import batch_on_current_stream, bits, cuda, err_code, run_ranks, state_rows

gpu = pytest.mark.gpu


# ---- CPU: gather_winner_states over 2 gloo ranks ---------------------------------------------------
F_FAKE = 7


def _fake_rows(g):
    """A row per global world index; every fourth element is -0.0, which a summing collective would
    turn into +0.0."""
    g = np.asarray(g, dtype=np.int64)
    j = np.arange(F_FAKE)
    r = np.sin(g[:, None] * 1.7 + j[None, :]) * 1e3
    return np.where((g[:, None] + j[None, :]) % 4 == 0, -0.0, r)


def _winner_sets(total):
    lo1 = mpc.shard_range(total, 1, 2)[0]
    return [
        [0, lo1 - 1, lo1, total - 1],                 # both ends of both shards
        [3, 1, lo1 + 2, 5, 1, total - 1, 2],          # several winners of one rank, a duplicate
        [2, 0, 2],                                    # rank 1 owns no winner
    ]


def _gather_worker(rank, ws):
    out = []
    for total in (37, 64):
        lo, _ = mpc.shard_range(total, rank, ws)
        for winners in _winner_sets(total):
            rows = mpc.gather_winner_states(np.array(winners), total, lambda local: torch.from_numpy(_fake_rows(lo + np.asarray(local))))
            out.append((total, winners, rows.numpy().copy()))
    return out


def test_gather_winner_states_gloo_bit_exact():
    res = run_ranks(_gather_worker, 2, "gloo", timeout=120)
    assert len(res[0]) == len(res[1]) == 6
    for (total, winners, a), (_, _, b) in zip(res[0], res[1]):
        expect = _fake_rows(winners)
        assert np.signbit(expect).any() and (expect == 0).any()
        assert a.shape == (len(winners), F_FAKE)
        assert np.array_equal(a.view(np.uint64), b.view(np.uint64)), f"ranks disagree ({total}, {winners})"
        assert np.array_equal(a.view(np.uint64), expect.view(np.uint64)), f"wrong rows ({total}, {winners})"


def test_gather_winner_states_single_process_calls_pack_directly():
    seen = []

    def pack(local):
        seen.append(np.asarray(local).copy())
        return torch.from_numpy(_fake_rows(local))

    rows = mpc.gather_winner_states([4, 0, 4], 8, pack)
    assert len(seen) == 1 and seen[0].tolist() == [4, 0, 4]
    assert np.array_equal(rows.numpy().view(np.uint64), _fake_rows([4, 0, 4]).view(np.uint64))


# ---- GPU ------------------------------------------------------------------------------------------
def _schedule(f_ext, H, seed, sigma=0.05):
    """A time-varying schedule around f_ext: random torques on every body, slice by slice."""
    rng = np.random.default_rng(seed)
    u = np.broadcast_to(f_ext, (H,) + f_ext.shape).copy()
    u[..., 3:6] += rng.normal(0.0, sigma, size=u[..., 3:6].shape)
    return u


@gpu
@pytest.mark.parametrize("name,W", [("pile64", 16), ("legged20", 64)])
def test_gather_state_matches_bodies(name, W):
    import eggshell_b200 as E
    scene = getattr(E.scenes, name)(W)
    b = batch_on_current_stream(scene, solver=E.SOLVER_PGS, k_max=50)
    b.step(scene["dt"], n_steps=3)
    rng = np.random.default_rng(11)
    idx = np.concatenate([[0, W - 1], rng.integers(0, W, size=9), [W - 1]])
    out = torch.full((idx.size, scene["n"] * 18), np.nan, dtype=torch.float64, device="cuda")
    b.gather_state(idx, out.data_ptr())
    rows = out.cpu().numpy().reshape(idx.size, scene["n"], 18)
    assert np.array_equal(bits(rows), bits(state_rows(b)[idx]))
    b.close()


@gpu
@pytest.mark.parametrize("k,first", [(1, 0), (1, 5), (3, 0), (3, 5)])
def test_seed_state_assigns_source_first_plus_w_mod_k(k, first):
    import eggshell_b200 as E
    W = 16
    scene = E.scenes.legged20(W)
    b = batch_on_current_stream(scene, solver=E.SOLVER_PGS, k_max=20)
    n = scene["n"]
    rng = np.random.default_rng(100 + k)
    src = rng.normal(size=(k, n, 18))
    src[:, ::3, 4] = -0.0
    b.seed_state(cuda(src).data_ptr(), k, first)
    rows = state_rows(b)
    for w in range(W):
        assert np.array_equal(bits(rows[w]), bits(src[(first + w) % k])), f"world {w}"
    b.close()


@gpu
def test_seeded_batch_steps_like_a_fresh_batch():
    """No state outside the body state survives a seed: one step of the seeded batch equals one step
    of a batch built on the host from the seeded state (same f_ext)."""
    import eggshell_b200 as E
    W = 8
    scene = E.scenes.legged20(W)
    kw = dict(solver=E.SOLVER_PGS, k_max=100)
    b = batch_on_current_stream(scene, **kw)
    b.step(scene["dt"], n_steps=4)
    winners = np.array([5, 2, 7])
    states = torch.empty((3, scene["n"] * 18), dtype=torch.float64, device="cuda")
    b.gather_state(winners, states.data_ptr())
    b.seed_state(states.data_ptr(), 3, 5)
    p, R, v, w = [x.copy() for x in b.bodies()]
    b.step(scene["dt"])
    fresh_scene = dict(scene, p=p, R=R, v=v, w=w)
    fb = batch_on_current_stream(fresh_scene, **kw)
    fb.step(scene["dt"])
    for a, c in zip(b.bodies(), fb.bodies()):
        assert np.array_equal(bits(a), bits(c))
    assert np.array_equal(b.status()["n_contacts"], fb.status()["n_contacts"])
    b.close()
    fb.close()


@gpu
@pytest.mark.parametrize("name", ["legged20", "chain10"])
def test_constant_schedule_equals_step(name):
    """A schedule whose every slice is the scene's f_ext gives the bits of egg_step(n = H)."""
    import eggshell_b200 as E
    if name == "legged20":
        scene, kw, H = E.scenes.legged20(16), dict(solver=E.SOLVER_PGS, k_max=100), 6
    else:
        scene, kw, H = E.scenes.chain(4, links=10, seed=3, anchor_jitter=0.1, v_jitter=0.2), dict(solver=E.SOLVER_DENSE_MURTY), 4
    b = batch_on_current_stream(scene, **kw)
    b.snapshot()
    b.step(scene["dt"], n_steps=H)
    ref = [x.copy() for x in b.bodies()]
    f_ext = b.static()[2]
    b.restore()
    u = cuda(np.broadcast_to(f_ext, (H,) + f_ext.shape))
    b.step_controlled(scene["dt"], u.data_ptr(), H)
    for a, c in zip(b.bodies(), ref):
        assert np.array_equal(bits(a), bits(c))
    b.close()


@gpu
def test_time_varying_schedule_equals_host_loop():
    import eggshell_b200 as E
    W, H = 16, 5
    scene = E.scenes.legged20(W)
    b = batch_on_current_stream(scene, solver=E.SOLVER_PGS, k_max=100)
    b.snapshot()
    u = _schedule(scene["f_ext"], H, seed=21)
    for t in range(H):
        b.set_external(u[t])
        b.step(scene["dt"], 1)
    ref = [x.copy() for x in b.bodies()]
    b.set_external(scene["f_ext"])
    b.restore()
    launches = b.launch_count
    ud = cuda(u)
    b.step_controlled(scene["dt"], ud.data_ptr(), H)
    step_launches = 5   # collide, three assembly kernels, solve (PGS group stream)
    assert b.launch_count - launches == H * (step_launches + 1)
    for a, c in zip(b.bodies(), ref):
        assert np.array_equal(bits(a), bits(c))
    assert np.array_equal(bits(b.static()[2]), bits(u[-1])), "the f_ext slot holds the last slice"
    b.close()


@gpu
def test_time_varying_schedule_matches_oracle():
    """Shared state before every step: the oracle adopts the GPU state and f_ext = u[t]."""
    import eggshell_b200 as E
    from tests.helpers import oracle_world, compare_step
    W, H = 4, 3
    scene = E.scenes.legged20(W)
    b = batch_on_current_stream(scene, solver=E.SOLVER_PGS, k_max=100, taps=True)
    ows = [oracle_world(scene, wi, solver=1, k_max=100)[0] for wi in range(W)]
    u = _schedule(scene["f_ext"], H, seed=31, sigma=0.2)
    ud = cuda(u)
    for t in range(H):
        p, R, v, w = b.bodies()
        for wi, ow in enumerate(ows):
            ow.set_state(p[wi], R[wi], v[wi], w[wi])
            ow.set_fext(u[t, wi])
        b.step_controlled(scene["dt"], ud[t].data_ptr(), 1)
        for ow in ows:
            ow.step(scene["dt"])
        worst = compare_step(b, ows, list(range(W)), tol=1e-9)
    print("controlled legged20 vs oracle", worst)
    b.close()


@gpu
def test_rollout_costs_match_numpy():
    import eggshell_b200 as E
    W = 64
    scene = E.scenes.legged20(W)
    b = batch_on_current_stream(scene, solver=E.SOLVER_PGS, k_max=100)
    p0 = b.bodies()[0]
    b.step_controlled(scene["dt"], cuda(_schedule(scene["f_ext"], 8, seed=41, sigma=1.0)).data_ptr(), 8)
    costs = torch.empty(W, dtype=torch.float64, device="cuda")
    b.rollout_costs(costs.data_ptr())
    c = costs.cpu().numpy()
    p = b.bodies()[0]
    dx, dz = p[:, 0, 0] - p0[:, 0, 0], p[:, 0, 2] - p0[:, 0, 2]
    expect = -dx + 10.0 * dz * dz
    assert np.all(expect != 0)
    # nvcc may contract the expression into one FMA: 2 ulp
    assert np.all(np.abs(c - expect) <= 2 * np.spacing(np.abs(expect))), np.max(np.abs(c - expect) / np.spacing(np.abs(expect)))
    b.close()


@gpu
def test_bad_arguments_are_refused_on_the_host():
    import eggshell_b200 as E
    from eggshell_b200.batch import EggError, EXPLICIT_EULER
    W = 8
    scene = E.scenes.legged20(W)
    n, dt = scene["n"], scene["dt"]
    b = batch_on_current_stream(scene, solver=E.SOLVER_PGS, k_max=20)
    b.step(dt)
    before = [x.copy() for x in b.bodies()]
    f_before = b.static()[2].copy()
    host = np.zeros((W + 1) * n * 18 * 4)
    dbuf = torch.full((W + 1, n * 18), 7.0, dtype=torch.float64, device="cuda")
    useq = cuda(np.broadcast_to(scene["f_ext"], (2, W, n, 6)))
    calls = [
        lambda: b.seed_state(host.ctypes.data, 1),
        lambda: b.gather_state([0], host.ctypes.data),
        lambda: b.step_controlled(dt, host.ctypes.data, 1),
        lambda: b.rollout_costs(host.ctypes.data),
        lambda: b.seed_state(dbuf.data_ptr(), 0),
        lambda: b.gather_state([], dbuf.data_ptr()),
        lambda: b.seed_state(dbuf.data_ptr(), W + 1),
        lambda: b.gather_state(np.arange(W + 1) % W, dbuf.data_ptr()),
        lambda: b.gather_state([0, W], dbuf.data_ptr()),
        lambda: b.gather_state([-1], dbuf.data_ptr()),
        lambda: b.seed_state(dbuf.data_ptr(), 1, -1),
        lambda: b.step_controlled(dt, useq.data_ptr(), 0),
        lambda: b.step_controlled(dt, 0, 1),
    ]
    for i, call in enumerate(calls):
        with pytest.raises(EggError) as ei:
            call()
        assert err_code(ei) == -1, f"call {i}: {ei.value}"
    with pytest.raises(EggError) as ei:
        b.step_controlled(dt, useq.data_ptr(), 1, integrator=EXPLICIT_EULER)
    assert err_code(ei) == -5
    for a, c in zip(b.bodies(), before):
        assert np.array_equal(bits(a), bits(c))
    assert np.array_equal(bits(b.static()[2]), bits(f_before))
    assert bool((dbuf == 7.0).all())
    b.close()
    # before egg_init
    raw = E.Batch(W, n, scene["nj"], solver=E.SOLVER_PGS)
    raw.set_bodies(scene["p"], scene["R"], scene["v"], scene["w"], scene["m"], scene["I"])
    for call in (lambda: raw.seed_state(dbuf.data_ptr(), 1), lambda: raw.gather_state([0], dbuf.data_ptr()),
                 lambda: raw.step_controlled(dt, useq.data_ptr(), 1)):
        with pytest.raises(EggError) as ei:
            call()
        assert err_code(ei) == -4
    raw.close()


@gpu
def test_mpc_iteration_checks_its_schedule():
    import eggshell_b200 as E
    W = 8
    scene = E.scenes.legged20(W)
    b = batch_on_current_stream(scene, solver=E.SOLVER_PGS, k_max=20)
    b.snapshot()
    good = cuda(np.broadcast_to(scene["f_ext"], (2, W, scene["n"], 6)))
    for bad in (good.float(), good.cpu(), good[:, :W - 1].contiguous(), good.transpose(0, 1), good[0]):
        with pytest.raises(ValueError):
            mpc.mpc_iteration(b, bad, scene["dt"], 2, W, 0)
    winners, costs, states = mpc.mpc_iteration(b, good, scene["dt"], 2, W, 0)
    assert len(winners) == 2 and states.shape == (2, scene["n"] * 18)
    rows = state_rows(b)
    for w in range(W):
        assert np.array_equal(bits(rows[w].ravel()), bits(states[w % 2].cpu().numpy()))
    b.close()


# ---- 1 GPU vs 2 GPUs ------------------------------------------------------------------------------
TOTAL, H2, ITERS, K2 = 8192, 4, 2, 3


def _two_gpu_inputs():
    import eggshell_b200 as E
    scene = E.scenes.legged20(TOTAL)
    rng = np.random.default_rng(77)
    u = np.broadcast_to(scene["f_ext"], (ITERS, H2) + scene["f_ext"].shape).copy()
    u[..., 3:6] += rng.normal(0.0, 0.5, size=u[..., 3:6].shape)
    return scene, u


def _shard(scene, lo, hi):
    sub = dict(scene, W=hi - lo)
    for key in ("p", "R", "v", "w", "m", "I", "c0", "c1", "f_ext"):
        sub[key] = scene[key][lo:hi].copy()
    return sub


def _run_iterations(rank, ws):
    import eggshell_b200 as E
    scene, u = _two_gpu_inputs()
    lo, hi = mpc.shard_range(TOTAL, rank, ws)
    b = batch_on_current_stream(_shard(scene, lo, hi), solver=E.SOLVER_PGS, k_max=20, device=rank)
    b.snapshot()
    out = {}
    for it in range(ITERS):
        winners, costs, _ = mpc.mpc_iteration(b, cuda(u[it, :, lo:hi]), scene["dt"], K2, TOTAL, lo)
        out[f"winners{it}"], out[f"costs{it}"] = np.asarray(winners), np.asarray(costs)
    out["state"] = state_rows(b)
    b.close()
    return out


@gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_ranks_equal_one_rank():
    ws = 2
    ranks = run_ranks(_run_iterations, ws, "nccl", timeout=600)
    one = _run_iterations(0, 1)
    for it in range(ITERS):
        for key in (f"winners{it}", f"costs{it}"):
            for r in range(ws):
                assert np.array_equal(ranks[r][key].view(np.uint64), one[key].view(np.uint64)), f"rank {r} {key}"
    state2 = np.concatenate([ranks[r]["state"] for r in range(ws)])
    assert np.array_equal(bits(state2), bits(one["state"]))
