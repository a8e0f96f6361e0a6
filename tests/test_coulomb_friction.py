"""Coulomb-pyramid friction with a per-world coefficient (egg_set_friction, INTEGRATION.md "Friction").

CPU: the oracle's Coulomb path (bounds, clamp flags, the incline physics).  GPU: the PGS stream's
Coulomb twins against the oracle one step at a time from shared state, every twin instance, the
incline in one batch, the C-ABI rules, and full-size batches.  The stepwise harness here has its own
near-tie probe: the one of tests.helpers assumes the BOX bounds [-1, 1]."""
import math

import numpy as np
import pytest

from oracle import pyoracle as O
from tests.coulomb_oracle import CoulombWorld
from tests.helpers import compare_step, oracle_world

MUS = (0.0, 0.3, 0.8, 3.0)
# Colliding heaps (pile64, the cairn's heap worlds) at K = 500 with mu = 3 do not converge (residual
# ~1e3) and the sweep amplifies rounding: the oracle built with FMA contraction moves p by up to 5e-2
# relative in one step against the oracle without it.  No implementation can meet 1e-9 there, so the
# heaps run mu = 3 at K = 20 only; at K <= 500 they take the other three values.
MUS_HEAP_K500 = (0.0, 0.3, 0.8)
# FP32 records with Coulomb friction on the colliding cairn heap stay within ~1e-3 of the FP64 oracle
# per step, not within the 1e-4 of the FP32 comparison, at K = 500 and at K = 20 alike: the bounds
# follow the normal multipliers, which carry the ~1e-7 record rounding into the tangent rows.  The
# FP32 twins are compared on legged20, which meets 1e-4; the FP64 twins on both scenes.
THETA = 0.3                          # incline angle: tan = 0.309
INCLINE_MU = (0.1, 0.2, 0.45, 1.0)   # each at least 20 % away from tan(THETA)
MASSES = (0.1, 1.0, 10.0)
STICK_V = 0.01                       # m/s after 200 steps: a sliding box moves at >= 1 m/s by then


def _with_mu(scene, mus=MUS):
    scene["mu"] = np.array([mus[w % len(mus)] for w in range(scene["W"])])
    return scene


def _oracle(scene, w, **kw):
    return CoulombWorld(oracle_world(scene, w, **kw)[0], scene["mu"][w] if "mu" in scene else None, kw.get("solver"))


def _incline(masses, mus, dt=0.005):
    """One 0.3 m cube per world resting on one face, gravity tilted by THETA about the y axis: the
    box slides down +x iff mu < tan(THETA)."""
    W = len(masses)
    m = np.asarray(masses, dtype=np.float64).reshape(W, 1)
    I = np.eye(3) * (m * 0.18 / 12)[:, :, None, None]
    sc = dict(W=W, n=1, nj=0, p=np.tile([[[0.0, 0.0, 0.15]]], (W, 1, 1)), R=np.tile(np.eye(3), (W, 1, 1, 1)),
              v=np.zeros((W, 1, 3)), w=np.zeros((W, 1, 3)), m=m, I=I, dt=dt, name="incline")
    if mus is not None:
        sc["mu"] = np.asarray(mus, dtype=np.float64)
    return sc


def _gravity():
    return (9.8 * math.sin(THETA), 0.0, -9.8 * math.cos(THETA))


# ---------------------------------------------------------------------------------------------
# Oracle (CPU)
def test_oracle_mu_zero_leaves_tangents_at_zero():
    import eggshell_b200 as E
    sc = _with_mu(E.scenes.stack10(2, seed=11), (0.0,))
    for w in range(2):
        ow = _oracle(sc, w, solver=O.SOLVER_PGS)
        for _ in range(5):
            ow.step(sc["dt"])
            lam, _, rs = ow.solution()
            assert len(lam) and np.all(lam.reshape(-1, 3)[:, :2] == 0.0)
            assert np.all(lam.reshape(-1, 3)[:, 2] >= 0.0)


@pytest.mark.parametrize("quirks", [3, 0])
def test_oracle_flags_and_bounds(quirks):
    """Every flagged tangent row equals -b or +b exactly, every free one lies in [-b, b]; normal rows
    keep [0, inf) and joints are equalities."""
    import eggshell_b200 as E
    for sc in (_with_mu(E.scenes.stack10(4, seed=12)), _with_mu(E.scenes.legged20(4, seed=13))):
        for w in range(sc["W"]):
            ow = _oracle(sc, w, solver=O.SOLVER_PGS, k_max=100, quirks=quirks)
            seen = 0
            for _ in range(3):
                ow.step(sc["dt"])
                lam, _, rs = ow.solution()
                b = ow.friction_bound()
                row = np.arange(len(lam)) % 3
                tan = (rs != 3) & (row < 2)
                cone = tan & np.isfinite(b)
                assert np.all(lam[(rs == 1) & tan] == -b[(rs == 1) & tan])
                assert np.all(lam[(rs == 2) & tan] == b[(rs == 2) & tan])
                free = cone & (rs == 0)
                assert np.all(np.abs(lam[free]) <= b[free])
                assert np.all(b[cone] >= 0) and (sc["mu"][w] > 0 or np.all(b[cone] == 0))
                assert np.all(lam[(rs != 3) & (row == 2)] >= 0)
                seen += int(cone.sum())
            assert seen > 0


def test_oracle_refuses_other_solvers_and_bad_mu():
    import eggshell_b200 as E
    sc = E.scenes.stack10(1, seed=14)
    for solver in (O.SOLVER_DENSE_MURTY, O.SOLVER_JACOBI, O.SOLVER_SOR):
        with pytest.raises(ValueError):
            CoulombWorld(oracle_world(sc, 0, solver=solver)[0], 0.5, solver)
    for bad in (-0.1, float("nan"), float("inf")):
        with pytest.raises(ValueError):
            CoulombWorld(oracle_world(sc, 0, solver=O.SOLVER_PGS)[0], bad, O.SOLVER_PGS)
    # no coefficient: the oracle's own BOX step, bit for bit
    ow = CoulombWorld(oracle_world(sc, 0, solver=O.SOLVER_PGS)[0], None, O.SOLVER_PGS)
    ref = oracle_world(sc, 0, solver=O.SOLVER_PGS)[0]
    ow.step(sc["dt"]); ref.step(sc["dt"])
    assert np.array_equal(ow.solution()[0], ref.solution()[0])


def _oracle_incline(m, mu, steps=200):
    sc = _incline([m], None if mu is None else [mu])
    ow = _oracle(sc, 0, solver=O.SOLVER_PGS, gravity=_gravity())
    vx = []
    for _ in range(steps):
        ow.step(sc["dt"])
        vx.append(ow.bodies()[2][0].copy())
    return np.array(vx)


def test_oracle_incline_stick_iff_mu_above_tan():
    """Coulomb: the box stays iff mu > tan(theta), whatever its mass; sliding, it accelerates at
    g (sin - mu cos) to a few %.  BOX friction: the outcome depends on the mass."""
    tan = math.tan(THETA)
    for mu in INCLINE_MU:
        assert abs(mu / tan - 1) >= 0.2
        for m in MASSES:
            v = _oracle_incline(m, mu)
            stuck = np.linalg.norm(v[-1]) < STICK_V
            assert stuck == (mu > tan), (m, mu, v[-1])
            if not stuck:
                a = (v[-1, 0] - v[99, 0]) / (100 * 0.005)
                expect = 9.8 * (math.sin(THETA) - mu * math.cos(THETA))
                assert abs(a / expect - 1) < 0.03, (m, mu, a, expect)
    box = [bool(np.linalg.norm(_oracle_incline(m, None)[-1]) < STICK_V) for m in MASSES]
    assert len(set(box)) == 2, box


# ---------------------------------------------------------------------------------------------
# GPU against the oracle
def coulomb_stepwise(scene, nsteps, worlds_idx, batch_kw, oracle_kw, tol=1e-9):
    """One step at a time from shared state: compare_step (narrowphase bit-exact, state and
    multipliers within tol), sweeps and row_state bit for bit, and the Coulomb near-tie probe: the
    margin of a free tangent row is its distance to the oracle's bound b (of a free normal row, its
    distance to 0); it must exceed 10x the CUDA-vs-oracle difference of the world.  Rows with b = 0
    are multipliers of exactly +-0 on both sides (their clamp flags are compared bit for bit)."""
    import eggshell_b200 as E
    b = E.scenes.make_batch(scene, taps=True, **batch_kw)
    ows = [_oracle(scene, wi, **oracle_kw) for wi in worlds_idx]
    worst_all = dict(margin_over_diff=np.inf)
    for s in range(nsteps):
        p, R, v, w = b.bodies()
        for k, wi in enumerate(worlds_idx):
            ows[k].set_state(p[wi], R[wi], v[wi], w[wi])
        b.step(scene["dt"])
        for ow in ows:
            ow.step(scene["dt"])
        worst = compare_step(b, ows, worlds_idx, tol=tol)
        st, con = b.status(), b.contacts()
        assert int(st["status"].max()) == 0
        for k, wi in enumerate(worlds_idx):
            os_ = ows[k].stats()
            assert st["sweeps"][wi] == os_["sweeps"], f"step {s} world {wi}: sweeps {st['sweeps'][wi]} != {os_['sweeps']}"
            lam, _, rs = ows[k].solution()
            assert np.array_equal(con["row_state"][wi, :len(rs)], rs), f"step {s} world {wi}: row clamp states differ"
            if os_["sweeps"] == 0 or not len(lam):
                continue
            bnd = ows[k].friction_bound()
            row = np.arange(len(lam)) % 3
            cone = np.isfinite(bnd).reshape(-1, 3)[:, :1].repeat(3, axis=1).ravel()   # blocks projected as contacts
            tan_free = cone & (row < 2) & (rs == 0) & (bnd > 0)
            nrm_free = cone & (row == 2) & (rs == 0)
            dist = np.concatenate([(bnd - np.abs(lam))[tan_free], np.abs(lam)[nrm_free]])
            if dist.size:
                diff = float(np.max(np.abs(con["lam"][wi, :len(lam)] - lam)))
                worst_all["margin_over_diff"] = min(worst_all["margin_over_diff"], float(dist.min()) / max(diff, 1e-300))
        for k_, v_ in worst.items():
            worst_all[k_] = max(worst_all.get(k_, 0.0), v_)
    b.close()
    assert worst_all["margin_over_diff"] > 10.0, f"near-tie: a free row within 10x the CUDA-vs-oracle difference of its bound ({worst_all['margin_over_diff']:.3e})"
    return worst_all


def _scenes():
    import eggshell_b200 as E
    from tests.test_pgs_instances import _cairn_mix
    pile = E.scenes.pile64(8)
    return [("stack10", E.scenes.stack10(8), list(range(8)), 4),
            ("pile64", pile, [0, 3, 6], 2),
            ("legged20", E.scenes.legged20(8), list(range(8)), 3),
            ("cairn", _cairn_mix(11), list(range(11)), 4),
            ("rounds", E.scenes.rounds(8), list(range(8)), 4)]


@pytest.mark.gpu
@pytest.mark.parametrize("quirks", [3, 0])
@pytest.mark.parametrize("k_max", [500, 20])
def test_gpu_vs_oracle(k_max, quirks):
    """mu in {0, 0.3, 0.8, 3} across the worlds of every scene (the heaps at K = 500: see MUS_HEAP_K500)."""
    import eggshell_b200 as E
    for name, sc, idx, steps in _scenes():
        _with_mu(sc, MUS_HEAP_K500 if k_max == 500 and name in ("pile64", "cairn") else MUS)
        worst = coulomb_stepwise(sc, steps, idx, dict(solver=E.SOLVER_PGS, k_max=k_max, quirks=quirks),
                                 dict(solver=O.SOLVER_PGS, k_max=k_max, quirks=quirks))
        print(f"{name} K={k_max} quirks={quirks}: " + " ".join(f"{k} {v:.1e}" for k, v in sorted(worst.items())))


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [64, 32])
@pytest.mark.parametrize("iso", [0, 1, 2])
@pytest.mark.parametrize("lpw", [1, 2, 4, 8, 16])
def test_coulomb_instance_vs_oracle(lpw, iso, prec, monkeypatch):
    """Each of the 30 Coulomb twins of egg_pgs_stream_kernel, forced through the development
    overrides as test_pgs_instances.py does: the mixed cairn (K = 500, FP64 records) and legged20
    (K = 100), every world against the oracle (FP32 records at 1e-4 with the sweep slack of
    stepwise_fp32)."""
    import eggshell_b200 as E
    import tests.helpers as H
    from tests.test_pgs_instances import OVERRIDES, _cairn_mix, _scene
    for k in OVERRIDES:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("EGG_PGS_LPW", str(lpw))
    monkeypatch.setattr(H, "oracle_world", lambda scene, w, **kw: (_oracle(scene, w, **kw), 0))
    W = 2 * (32 // lpw) + 3
    cases = [(_scene("legged20", W, iso), 2, 100, MUS)]
    if prec == 64:
        cases.insert(0, (_cairn_mix(W, iso), 4, 500, MUS_HEAP_K500))
    for sc, steps, k_max, mus in cases:
        _with_mu(sc, mus)
        kw = dict(solver=E.SOLVER_PGS, k_max=k_max)
        b = E.scenes.make_batch(sc, precision=prec, **kw)
        b.step(sc["dt"])
        cfg = b.kernel_config()
        b.close()
        assert (cfg["lpw"], cfg["iso"], cfg["precision"], cfg["rec_format"]) == (lpw, iso, prec, 1), cfg
        okw = dict(solver=O.SOLVER_PGS, k_max=k_max)
        if prec == 64:
            worst = coulomb_stepwise(sc, steps, list(range(W)), kw, okw)
        else:
            worst = H.stepwise_fp32(sc, steps, list(range(W)), kw, okw, sweep_slack=True)
        print(f"Coulomb LPW {lpw} ISO {iso} FP{prec} {sc['name']}: " + " ".join(f"{k} {v:.1e}" for k, v in sorted(worst.items())))


@pytest.mark.gpu
def test_gpu_incline_matches_oracle():
    """The incline in one batch, mu varying across the worlds: every world sticks or slides as the
    oracle's does, and as mu against tan(theta) says."""
    import eggshell_b200 as E
    ms = [m for m in MASSES for _ in INCLINE_MU]
    mus = [mu for _ in MASSES for mu in INCLINE_MU]
    sc = _incline(ms, mus)
    b = E.scenes.make_batch(sc, solver=E.SOLVER_PGS, gravity=_gravity())
    b.step(sc["dt"], n_steps=200)
    v = b.bodies()[2][:, 0]
    assert int(b.status()["status"].max()) == 0
    b.close()
    for w, (m, mu) in enumerate(zip(ms, mus)):
        stuck = np.linalg.norm(v[w]) < STICK_V
        ov = _oracle_incline(m, mu)[-1]
        assert stuck == (np.linalg.norm(ov) < STICK_V) == (mu > math.tan(THETA)), (m, mu, v[w], ov)
        assert np.max(np.abs(v[w] - ov)) < 1e-6 * max(1.0, float(np.max(np.abs(ov)))), (m, mu, v[w], ov)


# ---------------------------------------------------------------------------------------------
# C ABI
def _state(b):
    con = b.contacts()
    return [x.copy() for x in b.bodies()] + [con["lam"].copy(), con["row_state"].copy(), b.status()["sweeps"].copy()]


def _bits_equal(a, b):
    return all(np.array_equal(x.view(np.uint64) if x.dtype == np.float64 else x, y.view(np.uint64) if y.dtype == np.float64 else y)
               for x, y in zip(a, b))


@pytest.mark.gpu
def test_api_refusals_keep_the_previous_table():
    import eggshell_b200 as E
    sc = E.scenes.stack10(8)
    for solver in (E.SOLVER_DENSE_MURTY, E.SOLVER_JACOBI, E.SOLVER_SOR):
        b = E.scenes.make_batch(sc, solver=solver)
        with pytest.raises(E.EggError, match=r"\(-5\)"):
            b.set_friction(0.5)
        assert b.friction is None
        b.close()
    mu = np.linspace(0.1, 2.0, 8)
    ref = E.scenes.make_batch(sc, solver=E.SOLVER_PGS, taps=True)
    ref.set_friction(mu)
    ref.step(sc["dt"], n_steps=3)
    b = E.scenes.make_batch(sc, solver=E.SOLVER_PGS, taps=True)
    b.set_friction(mu)
    for bad in (-0.5, float("nan"), float("inf")):
        t = mu.copy()
        t[3] = bad
        with pytest.raises(E.EggError, match=r"\(-1\)"):
            b.set_friction(t)
        assert np.array_equal(b.friction, mu)
    b.step(sc["dt"], n_steps=3)
    assert _bits_equal(_state(b), _state(ref))
    b.close(); ref.close()


@pytest.mark.gpu
def test_api_device_bytes_and_clearing():
    """egg_device_bytes grows by >= 8 W bytes with a table and drops back after None; a step after
    set_friction(None) is bit-identical to a batch that never had a table, and a scalar broadcasts."""
    import eggshell_b200 as E
    sc = E.scenes.stack10(64)
    b = E.scenes.make_batch(sc, solver=E.SOLVER_PGS, taps=True)
    base = b.device_bytes
    b.set_friction(0.5)
    assert b.device_bytes - base >= 8 * 64
    assert np.array_equal(b.friction, np.full(64, 0.5))
    b.step(sc["dt"])
    b.set_friction(None)
    assert b.device_bytes == base and b.friction is None
    ref = E.scenes.make_batch(sc, solver=E.SOLVER_PGS, taps=True)
    ref.step(sc["dt"])
    b.set_state(*ref.bodies())   # the same state; the next step sees no table
    ref.set_state(*ref.bodies())
    b.step(sc["dt"]); ref.step(sc["dt"])
    assert _bits_equal(_state(b), _state(ref))
    b.close(); ref.close()


@pytest.mark.gpu
def test_api_controlled_step_equals_external_plus_step():
    import torch
    import eggshell_b200 as E
    sc = _with_mu(E.scenes.legged20(16))
    H = 3
    rng = np.random.default_rng(5)
    u = np.asarray(sc["f_ext"])[None] + rng.normal(0.0, 0.5, size=(H, 16, 20, 6))
    a = E.scenes.make_batch(sc, solver=E.SOLVER_PGS, taps=True)
    b = E.scenes.make_batch(sc, solver=E.SOLVER_PGS, taps=True)
    ud = torch.tensor(u, dtype=torch.float64, device="cuda")
    a.step_controlled(sc["dt"], ud.data_ptr(), H)
    a.sync()
    for t in range(H):
        b.set_external(u[t])
        b.step(sc["dt"])
    assert _bits_equal(_state(a), _state(b))
    a.close(); b.close()


@pytest.mark.gpu
def test_api_run_format_is_bypassed():
    import eggshell_b200 as E
    from tests.test_pgs_instances import RUNS
    sc = _with_mu(E.scenes.stack10(16))
    b = E.scenes.make_batch(sc, solver=E.SOLVER_PGS, quirks=RUNS, taps=True)
    b.step(sc["dt"])
    assert b.kernel_config()["rec_format"] == 1
    b.set_friction(None)
    b.step(sc["dt"])
    assert b.kernel_config()["rec_format"] == 2
    b.close()


# ---------------------------------------------------------------------------------------------
# Full size
@pytest.mark.gpu
@pytest.mark.parametrize("name,W", [("pile64", 65536), ("legged20", 131072)])
def test_full_size_status_and_determinism(name, W):
    """Random mu in [0.2, 1.0] per world: no status bit, and two runs of 10 steps give the same bits."""
    import eggshell_b200 as E
    sc = getattr(E.scenes, name)(W)
    sc["mu"] = np.random.default_rng(9).uniform(0.2, 1.0, size=W)
    kw = dict(solver=E.SOLVER_PGS, max_contacts=1024 if name == "pile64" else 0)
    out = []
    for _ in range(2):
        b = E.scenes.make_batch(sc, **kw)
        b.step(sc["dt"], n_steps=10)
        st = b.status()
        assert int(np.bitwise_or.reduce(st["status"])) == 0
        out.append([x.copy() for x in b.bodies()] + [st["sweeps"].copy()])
        b.close()
    assert _bits_equal(out[0], out[1])
