"""GPU parity tests proper: the CUDA path (through the C ABI) against the CPU oracle, one step at a
time from shared state.  Discrete outputs bit-exact; p, R, v, w, lambda within 1e-9 relative."""
import numpy as np
import pytest

from tests.helpers import oracle_world, compare_step, rel_err, SCALE, stepwise as _stepwise, stepwise_fp32

pytestmark = pytest.mark.gpu


def test_stack10_pgs_stepwise():
    import eggshell_b200 as E
    scene = E.scenes.stack10(8, seed=1000)
    worst = _stepwise(scene, 5, list(range(8)), dict(solver=E.SOLVER_PGS), dict(solver=1))
    print("stack10 worst", worst)


def test_pile64_pgs_stepwise():
    import eggshell_b200 as E
    scene = E.scenes.pile64(4, seed=3000)
    worst = _stepwise(scene, 2, list(range(4)), dict(solver=E.SOLVER_PGS, k_max=50), dict(solver=1, k_max=50))
    print("pile64 worst", worst)


def test_pile64_pgs_k500_stepwise():
    """The benchmarked configuration itself (C3 at the reference's termination, K <= 500 sweeps):
    4 worlds, 2 steps from shared state; sweep counts and clamp states bit-exact, state and
    multipliers within 1e-9 (every world runs all 500 sweeps on the interpenetrating lattice)."""
    import eggshell_b200 as E
    scene = E.scenes.pile64(4, seed=3000)
    worst = _stepwise(scene, 2, list(range(4)), dict(solver=E.SOLVER_PGS, k_max=500), dict(solver=1, k_max=500))
    print("pile64 K=500 worst", worst)


@pytest.mark.parametrize("name,W,steps", [("pile64", 4, 2), ("stack10", 8, 3), ("legged20", 4, 3)])
def test_pgs_fixed_k20_stepwise(name, W, steps):
    """Fixed-K mode (bench.py's `fixed_k` line, K = 20 sweeps): parity at the same K."""
    import eggshell_b200 as E
    scene = getattr(E.scenes, name)(W)
    worst = _stepwise(scene, steps, list(range(W)), dict(solver=E.SOLVER_PGS, k_max=20), dict(solver=1, k_max=20))
    print(name, "K=20 worst", worst)


def test_rounds_sphere_capsule_hinge_stepwise():
    """SURVEY row f4 / north_star (a): sphere and capsule colliders against the ground, a
    sphere-sphere pair, and a hinge (two ball joints on the axis) between two boxes, stepwise
    against the oracle (which DEFINES these contacts: the reference has boxes only -- parity
    unpinned).  Contact lists, codes (17 = sphere-sphere) and order bit-exact, state within 1e-9."""
    import eggshell_b200 as E
    scene = E.scenes.rounds(6)
    worst = _stepwise(scene, 8, list(range(6)), dict(solver=E.SOLVER_PGS, k_max=100), dict(solver=1, k_max=100), lam_tol=1e-8)
    print("rounds worst", worst)
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=100, taps=True)
    b.step(scene["dt"], n_steps=3)
    con, ph = b.contacts(), b.pair_hits()
    for wi in range(6):
        nc = con["count"][wi]
        assert (con["code"][wi, :nc] == 17).sum() == 1 and (con["i0"][wi, :nc] == -1).sum() >= 1
    assert int(np.bitwise_or.reduce(b.status()["status"])) == 0
    b.close()


def test_cairn_pgs_falling():
    import eggshell_b200 as E
    scene = E.scenes.cairn(16, rocks=4, zb=(0.2, 1.0), seed=11)
    # Multipliers at 1e-8 here (1e-9 everywhere else): the rocks land on several vertices, so the
    # contact rows of a rock are redundant (6 DOF) and lambda is fixed only by the cfm = 0.01
    # regularisation.  The solve stops at a residual of 1e-9 (constants.h:5), which leaves lambda
    # free within residual x 1/cfm: two arithmetic paths that both satisfy the reference's stopping
    # test differ by up to ~1e-7 absolute on |lambda| ~ 1e3 (tools/diag_cairn_lam.py), while the
    # quantities that do not depend on the split between redundant rows -- v, w, p, R -- agree to
    # 1e-13.
    worst = _stepwise(scene, 30, list(range(16)), dict(solver=E.SOLVER_PGS), dict(solver=1), lam_tol=1e-8)
    print("cairn worst", worst)


def test_legged_pgs_joints_and_contacts():
    import eggshell_b200 as E
    scene = E.scenes.legged20(4, seed=5000)
    worst = _stepwise(scene, 3, list(range(4)), dict(solver=E.SOLVER_PGS, k_max=100), dict(solver=1, k_max=100))
    print("legged worst", worst)


def test_pgs_general_and_mixed_inertia_paths():
    """The three M^-1 layouts of the stream kernel against the oracle: general 3x3 inverse inertia
    (anisotropic bodies), isotropic but different per body, and the EGG_OPT_EXACT_INERTIA switch."""
    import eggshell_b200 as E
    rng = np.random.default_rng(5)
    # (a) anisotropic inertia -> general kernel
    scene = E.scenes.cairn(9, rocks=5, zb=(0.1, 0.6), seed=21)
    scene["I"] = np.tile(np.diag([0.01, 0.02, 0.03]), (9, 5, 1, 1))
    worst = _stepwise(scene, 12, list(range(9)), dict(solver=E.SOLVER_PGS), dict(solver=1))
    print("anisotropic worst", worst)
    # (b) isotropic, masses and inertias differ per body -> per-body (1/m, 1/c) loads
    scene = E.scenes.cairn(9, rocks=5, zb=(0.1, 0.6), seed=22)
    scene["m"] = rng.uniform(0.5, 2.0, size=scene["m"].shape)
    scene["I"] = np.eye(3) * rng.uniform(0.05, 0.2, size=(9, 5, 1, 1))
    worst = _stepwise(scene, 12, list(range(9)), dict(solver=E.SOLVER_PGS), dict(solver=1))
    print("isotropic non-uniform worst", worst)
    # (c) uniform cubes with the inverse inertia kept exactly as computed (no snapping)
    scene = E.scenes.cairn(9, rocks=5, zb=(0.1, 0.6), seed=23)
    worst = _stepwise(scene, 12, list(range(9)), dict(solver=E.SOLVER_PGS, quirks=E.QUIRKS_REFERENCE | 4), dict(solver=1))
    print("exact inertia worst", worst)


def test_pgs_run_format_opt_in_stepwise():
    """EGG_OPT_PGS_RUNS (quirks bit 16, egg_pgs_runs.cu): a lane carries the contacts of one manifold
    through a stage and the records shrink to what cannot be rebuilt (frame quaternion, r0, 1/(D+cfm),
    rhs).  Same sweep in the same row order: contact lists, sweep counts and clamp states bit-exact,
    state and multipliers within 1e-9 of the oracle -- on stacks (runs of ground / face contacts),
    the pile at K = 50 and K = 500, joints + contacts, per-body (1/m, 1/c) and the mixed colliders."""
    import eggshell_b200 as E
    runs = E.QUIRKS_REFERENCE | 16
    for name, scene, W, steps, k in (("stack10", E.scenes.stack10(6), 6, 4, 500), ("pile64", E.scenes.pile64(3), 3, 3, 50),
                                     ("pile64 K=500", E.scenes.pile64(4, seed=3100), 4, 2, 500), ("legged20", E.scenes.legged20(4), 4, 3, 100),
                                     ("rounds", E.scenes.rounds(6), 6, 6, 100)):
        worst = _stepwise(scene, steps, list(range(W)), dict(solver=E.SOLVER_PGS, k_max=k, quirks=runs), dict(solver=1, k_max=k),
                          lam_tol=1e-8 if name == "rounds" else 1e-9)
        print("run format", name, worst)
    rng = np.random.default_rng(6)
    scene = E.scenes.cairn(9, rocks=5, zb=(0.1, 0.6), seed=22)
    scene["m"] = rng.uniform(0.5, 2.0, size=scene["m"].shape)
    scene["I"] = np.eye(3) * rng.uniform(0.05, 0.2, size=(9, 5, 1, 1))
    worst = _stepwise(scene, 12, list(range(9)), dict(solver=E.SOLVER_PGS, quirks=runs), dict(solver=1))
    print("run format, isotropic non-uniform", worst)
    # converging worlds: the probe fails, the exact residual decides; sweep counts are checked inside _stepwise
    scene = E.scenes.cairn(13, rocks=2, xb=(-1.0, 1.0), yb=(-1.0, 1.0), zb=(0.12, 0.16), seed=31)
    scene["v"] *= 0.05
    scene["w"] *= 0.05
    worst = _stepwise(scene, 6, list(range(13)), dict(solver=E.SOLVER_PGS, quirks=runs), dict(solver=1))
    print("run format, converging", worst)


def test_pgs_converging_worlds_take_the_exact_residual_path():
    """Worlds that converge before k_max: the probe lower bound fails, the exact residual decides;
    the sweep count must be the oracle's (checked inside _stepwise) and at least one world must
    actually have stopped early."""
    import eggshell_b200 as E
    scene = E.scenes.cairn(13, rocks=2, xb=(-1.0, 1.0), yb=(-1.0, 1.0), zb=(0.12, 0.16), seed=31)
    scene["v"] *= 0.05
    scene["w"] *= 0.05
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS)
    b.step(scene["dt"])
    sw = b.status()["sweeps"]
    b.close()
    assert ((sw > 0) & (sw < 500)).any(), f"no world converged early: {sw}"
    worst = _stepwise(scene, 6, list(range(13)), dict(solver=E.SOLVER_PGS), dict(solver=1))
    print("converging worst", worst, "sweeps of step 0", sw.tolist())


# ---------------------------------------------------------------------------------------------
# Against the committed golden fixtures (tests/golden/*.npz).
def _vs_golden(name, scene, nw, ns, batch_kw, tol=1e-9):
    import os
    import eggshell_b200 as E
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", name + ".npz"))
    b = E.scenes.make_batch(scene, taps=True, **batch_kw)
    for s in range(ns):
        # replay from the golden state of the previous step so that chaos cannot accumulate
        if s > 0:
            b.set_state(*[np.stack([g[f"w{wi}_s{s-1}_{k}"] for wi in range(nw)]) for k in ("p", "R", "v", "w")])
        b.step(scene["dt"])
        p, R, v, w = b.bodies()
        con = b.contacts()
        st = b.status()
        ph = b.pair_hits()
        for wi in range(nw):
            pre = f"w{wi}_s{s}_"
            nc = int(g[pre + "stats"][1])
            assert con["count"][wi] == nc
            assert st["n_contacts_raw"][wi] == g[pre + "stats"][0] and st["n_pair_hits"][wi] == g[pre + "stats"][3]
            assert st["sweeps"][wi] == g[pre + "stats"][4]
            assert np.array_equal(con["i0"][wi, :nc], g[pre + "c_i0"]) and np.array_equal(con["i1"][wi, :nc], g[pre + "c_i1"])
            assert np.array_equal(con["code"][wi, :nc], g[pre + "c_code"])
            nh = int(ph["n"][wi])
            assert np.array_equal(ph["i"][wi, :nh], g[pre + "hit_i"]) and np.array_equal(ph["j"][wi, :nh], g[pre + "hit_j"])
            assert np.array_equal(ph["code"][wi, :nh], g[pre + "hit_code"]) and np.array_equal(ph["count"][wi, :nh], g[pre + "hit_count"])
            nr = len(g[pre + "lam"])
            assert np.array_equal(con["row_state"][wi, :nr], g[pre + "row_state"])
            for key, val in (("p", p[wi]), ("R", R[wi]), ("v", v[wi]), ("w", w[wi]), ("c_pos", con["pos"][wi, :nc]),
                             ("c_nrm", con["nrm"][wi, :nc]), ("c_depth", con["depth"][wi, :nc])):
                sc = SCALE[key[2:] if key.startswith("c_") else key]
                assert rel_err(val, g[pre + key], sc) <= tol, (name, wi, s, key, rel_err(val, g[pre + key], sc))
            assert rel_err(con["lam"][wi, :nr], g[pre + "lam"], SCALE["lam"]) <= 1e-9
    b.close()


def test_golden_fixtures_pgs():
    import eggshell_b200 as E
    S = E.scenes
    _vs_golden("stack10_pgs", S.stack10(2, seed=1000), 2, 2, dict(solver=E.SOLVER_PGS))
    _vs_golden("pile64_pgs_k50", S.pile64(1, seed=3000), 1, 2, dict(solver=E.SOLVER_PGS, k_max=50))
    _vs_golden("pile64_pgs_k500", S.pile64(1, seed=3000), 1, 2, dict(solver=E.SOLVER_PGS, k_max=500))
    _vs_golden("legged20_pgs_k100", S.legged20(2, seed=5000), 2, 2, dict(solver=E.SOLVER_PGS, k_max=100))
    _vs_golden("chain32_pgs_k100", S.chain32(1, seed=4000, anchor_z=0.2), 1, 2, dict(solver=E.SOLVER_PGS, k_max=100))
    _vs_golden("cairn4_pgs", S.cairn(2, rocks=4, zb=(0.2, 0.6), seed=11), 2, 5, dict(solver=E.SOLVER_PGS))


# ---------------------------------------------------------------------------------------------
# Full BASELINE sizes: size-independent properties.
def test_full_size_c2_properties():
    """4096 worlds x 10-box stack: a world's result does not depend on the batch around it, a
    replay from the snapshot is bit-identical, and the contact list is in reference order."""
    import eggshell_b200 as E
    W = 4096
    scene = E.scenes.stack10(W, seed=1000)
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=30, taps=False)
    b.snapshot()
    b.step(scene["dt"])
    out1 = [x.copy() for x in b.bodies()]
    con = b.contacts()
    st = b.status()
    assert int(st["status"].max()) == 0
    b.restore()
    b.step(scene["dt"])
    out2 = b.bodies()
    for a, c in zip(out1, out2):
        assert np.array_equal(a, c)                       # deterministic replay
    # order: ground contacts (i0 = -1) by body, then pairs lexicographic (ensembles.cc:449-473)
    for wi in (0, 1, 17, W - 1):
        nc = con["count"][wi]
        key = con["i0"][wi, :nc].astype(np.int64) * 1000 + con["i1"][wi, :nc]
        assert np.all(np.diff(key) >= 0)
        assert np.all(con["depth"][wi, :nc] >= -1e-9)
    # independence: worlds 5..8 alone give the same bits
    sub = {k: (v[5:9] if isinstance(v, np.ndarray) and v.shape[:1] == (W,) else v) for k, v in scene.items()}
    sub["W"] = 4
    b2 = E.scenes.make_batch(sub, solver=E.SOLVER_PGS, k_max=30)
    b2.step(scene["dt"])
    for a, c in zip(out1, b2.bodies()):
        assert np.array_equal(a[5:9], c)
    # spot-check 3 worlds of the big batch against the oracle
    idx = [0, 2047, W - 1]
    ows = [oracle_world(scene, wi, solver=1, k_max=30)[0] for wi in idx]
    for ow in ows:
        ow.step(scene["dt"])
    compare_step(b, ows, idx)
    b.close(); b2.close()


def test_full_size_c3_contact_counts_and_capacity():
    """65536 worlds x 64-body pile, one step at k_max = 3: no overflow / non-finite status, contact
    statistics in the expected band, and sampled worlds bit-exact vs the oracle."""
    import eggshell_b200 as E
    W = 65536
    scene = E.scenes.pile64(W, seed=3000)
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=3, max_contacts=1024)
    b.step(scene["dt"])
    st = b.status()
    assert int(np.bitwise_or.reduce(st["status"])) == 0
    assert 400 < st["n_contacts"].mean() < 600 and st["n_contacts"].max() <= 1024
    assert 200 < st["n_pair_hits"].mean() < 320
    # sampled worlds: re-run them alone (bit-identical to their slice of the big batch) and check
    # that small batch against the oracle, contacts included
    idx = [0, 31337, W - 1]
    p, R, v, w = b.bodies()
    sub = {k: (val[idx] if isinstance(val, np.ndarray) and val.shape[:1] == (W,) else val) for k, val in scene.items()}
    sub["W"] = len(idx)
    b2 = E.scenes.make_batch(sub, solver=E.SOLVER_PGS, k_max=3, max_contacts=1024, taps=True)
    b2.step(scene["dt"])
    for big, small in zip((p, R, v, w), b2.bodies()):
        assert np.array_equal(big[idx], small)
    ows = [oracle_world(scene, wi, solver=1, k_max=3)[0] for wi in idx]
    for ow in ows:
        ow.step(scene["dt"])
    compare_step(b2, ows, list(range(len(idx))))
    b.close(); b2.close()


@pytest.mark.parametrize("name,W,k_max,steps", [("pile64", 65536, 500, 1), ("pile64", 16384, 5, 3), ("stack10", 65536, 100, 2), ("legged20", 131072, 100, 2)])
def test_full_size_pgs_runs_clean(name, W, k_max, steps):
    """Full occupancy (11 resident warps per SM, several world groups per warp), long and short
    solves: no world may end non-finite or with an internal flag, every world of a scene sees the
    same number of sweeps at these non-converging settings, and the multipliers stay bounded."""
    import eggshell_b200 as E
    scene = getattr(E.scenes, name)(W)
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=k_max, max_contacts=1024 if name == "pile64" else 0)
    for s in range(steps):
        b.step(scene["dt"])
        st = b.status()
        assert int(np.bitwise_or.reduce(st["status"])) == 0, (s, np.nonzero(st["status"])[0][:16].tolist())
        assert np.isfinite(st["residual"]).all()
    p, R, v, w = b.bodies()
    assert np.isfinite(p).all() and np.isfinite(R).all() and np.isfinite(v).all() and np.isfinite(w).all()
    assert float(np.abs(v).max()) < 1e3 and float(np.abs(w).max()) < 1e4
    b.close()


@pytest.mark.parametrize("name,W,k_max,steps", [("pile64", 4, 50, 2), ("stack10", 8, 200, 3), ("legged20", 4, 100, 3)])
def test_pgs_fp32_records_opt_in(name, W, k_max, steps):
    """precision = 32 (opt-in): constraint records of the solve stored in FP32, everything else FP64.
    Stepwise from shared state against the FP64 oracle: the narrowphase outputs stay bit-exact,
    state within 1e-4 relative (north_star's FP32 tolerance; measured ~1e-6), same sweep counts."""
    import eggshell_b200 as E
    scene = getattr(E.scenes, name)(W)
    worst_all = stepwise_fp32(scene, steps, list(range(W)), dict(solver=E.SOLVER_PGS, k_max=k_max), dict(solver=1, k_max=k_max))
    print(name, "fp32 records worst", worst_all)


@pytest.mark.parametrize("name,W,k_max,lpw,opt,prec,expect", [
    ("stack10", 65536, 10, "1", 0, 64, 1), ("stack10", 65536, 10, "", 0, 64, 1), ("pile64", 16384, 5, "", 0, 64, 8),
    ("pile64", 8192, 5, "16", 0, 64, 16), ("legged20", 131072, 10, "", 0, 64, 4), ("legged20", 65536, 10, "2", 0, 64, 2),
    ("stack10", 65536, 10, "1", 0, 32, 1), ("pile64", 16384, 5, "", 16, 64, 8), ("stack10", 65536, 10, "1", 16, 64, 1),
    ("legged20", 65536, 10, "", 16, 64, 4)])
def test_full_size_step_is_bit_reproducible(name, W, k_max, lpw, opt, prec, expect, monkeypatch):
    """The kernels are deterministic, so the same full-size step from the same state must give the
    same bits every time.  This is the test that exposes ordering bugs between the shared-memory
    loads of a stage and the TMA copy of the next one (a generic fence instead of the cross-proxy
    fence made 1-2 % of the worlds differ from run to run at 32 worlds per warp; the FP32 case runs
    there, at LPW 1).  The last three cases run the opt-in run format (EGG_OPT_PGS_RUNS), which hands
    its staging buffer back the same way.  Every case checks the lanes per world it ran at."""
    import eggshell_b200 as E
    if lpw:
        monkeypatch.setenv("EGG_PGS_LPW", lpw)
    else:
        monkeypatch.delenv("EGG_PGS_LPW", raising=False)
    scene = getattr(E.scenes, name)(W)
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=k_max, max_contacts=1024 if name == "pile64" else 0, quirks=E.QUIRKS_REFERENCE | opt,   # opt 16 = the run format
                            precision=prec)
    assert b.kernel_config()["lpw"] == expect
    b.snapshot()
    ref = None
    for r in range(3):
        b.restore()
        b.step(scene["dt"])
        out = [x.copy() for x in b.bodies()] + [b.contacts()["lam"].copy()]
        assert int(np.bitwise_or.reduce(b.status()["status"])) == 0
        if ref is None:
            ref = out
            continue
        for a, c in zip(out, ref):
            assert np.array_equal(a.view(np.uint64), c.view(np.uint64)), f"run {r} differs from run 0"
    cfg = b.kernel_config()
    assert (cfg["lpw"], cfg["precision"], cfg["rec_format"]) == (expect, prec, 2 if opt & 16 else 1), cfg
    b.close()


# ---------------------------------------------------------------------------------------------
# Dense path (what the reference ships): Schur complement + Murty principal pivoting.
def _stepwise_dense(scene, nsteps, worlds_idx, tol=1e-9, lam_tol=1e-9, oracle_kw=None, **kw):
    import eggshell_b200 as E
    b = E.scenes.make_batch(scene, solver=E.SOLVER_DENSE_MURTY, taps=True, **kw)
    ows = [oracle_world(scene, wi, solver=0, **(oracle_kw or {}))[0] for wi in worlds_idx]
    dt = scene["dt"]
    npiv = 0
    for s in range(nsteps):
        p, R, v, w = b.bodies()
        for k, wi in enumerate(worlds_idx):
            ows[k].set_state(p[wi], R[wi], v[wi], w[wi])
        b.step(dt)
        for ow in ows:
            ow.step(dt)
        worst = compare_step(b, ows, worlds_idx, tol=tol, lam_tol=lam_tol)
        st = b.status()
        con = b.contacts()
        for k, wi in enumerate(worlds_idx):
            os_ = ows[k].stats()
            assert st["pivots"][wi] == os_["pivots"], f"step {s} world {wi}: Murty pivots {st['pivots'][wi]} != {os_['pivots']}"
            assert st["cfm_applied"][wi] == os_["cfm_applied"], f"step {s} world {wi}: cfm decision differs"
            assert (st["status"][wi] & 1) == (os_["status"] & 1)
            lam, rhs, rs = ows[k].solution()
            assert np.array_equal(con["row_state"][wi, :len(rs)], rs), f"step {s} world {wi}: active set differs"
            npiv += os_["pivots"]
        assert worst["lam"] <= lam_tol, f"lambda mismatch {worst['lam']:.3e}"
    b.close()
    return npiv


def test_dense_chain10_golden():
    """C1: Chain(10,(2,2,1)) with the reference's default dense solver against the golden file,
    including steps around 400 where the chain hits the ground (contacts, cfm on, ~30 pivots)."""
    import os
    import eggshell_b200 as E
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "chain10_dense.npz"))
    scene = E.scenes.chain(1, links=10, anchor=(2.0, 2.0, 1.0))
    b = E.scenes.make_batch(scene, solver=E.SOLVER_DENSE_MURTY)
    # free swing: 2 steps from the initial state
    for s in (1, 2):
        b.step(0.001)
        p, R, v, w = b.bodies()
        for key, val in (("p", p[0]), ("R", R[0]), ("v", v[0]), ("w", w[0])):
            assert rel_err(val, g[f"s{s}_{key}"], SCALE[key]) <= 1e-9, (s, key)
        st = b.status()
        assert [st["n_contacts_raw"][0], st["n_contacts"][0], st["n_rows"][0], st["n_pair_hits"][0]] == g[f"s{s}_stats"][:4].tolist()
    # contact phase: replay golden states 399 -> 400 -> 401
    for s in (400, 401):
        b.set_state(*[g[f"s{s-1}_{k}"][None] for k in ("p", "R", "v", "w")])
        b.step(0.001)
        p, R, v, w = b.bodies()
        st = b.status()
        con = b.contacts()
        gs = g[f"s{s}_stats"]
        assert [st["n_contacts_raw"][0], st["n_contacts"][0], st["n_rows"][0], st["n_pair_hits"][0]] == gs[:4].tolist()
        assert st["pivots"][0] == gs[5] and st["cfm_applied"][0] == gs[6] and st["status"][0] == gs[7]
        nr = len(g[f"s{s}_lam"])
        assert np.array_equal(con["row_state"][0, :nr], g[f"s{s}_row_state"])
        for key, val in (("p", p[0]), ("R", R[0]), ("v", v[0]), ("w", w[0])):
            assert rel_err(val, g[f"s{s}_{key}"], SCALE[key]) <= 1e-9, (s, key)
        assert rel_err(con["lam"][0, :nr], g[f"s{s}_lam"], SCALE["lam"]) <= 1e-9
    b.close()


def test_dense_cairn_and_chain_stepwise():
    import eggshell_b200 as E
    npiv = _stepwise_dense(E.scenes.cairn(8, rocks=4, zb=(0.2, 0.5), seed=21), 25, list(range(8)))
    assert npiv > 0
    _stepwise_dense(E.scenes.chain(2, links=6, anchor=(0.0, 0.0, 0.25), seed=5, anchor_jitter=0.05), 6, [0, 1])


def test_dense_chain32_stepwise():
    """C4 (BASELINE.json configs[3]): 32-link chain landing on the ground, dense Schur + Murty
    (lcp.cc:157-336) with 96 equality rows and 90-150 contact rows.  4 worlds x 6 steps from shared
    state: pivot counts (70-300 per step), active set and cfm decision bit-exact, state and
    multipliers within 1e-9."""
    import eggshell_b200 as E
    scene = E.scenes.chain32(4, seed=4000)
    npiv = _stepwise_dense(scene, 6, [0, 1, 2, 3])
    print("chain32 dense: pivots compared", npiv)
    assert npiv > 1000


def test_dense_chain32_box_bounds():
    """The same scene with the BOX friction bounds honoured (quirk q1 off, SURVEY row f4)."""
    import eggshell_b200 as E
    q = E.QUIRK_GS_BOUNDS_SHIFT
    scene = E.scenes.chain32(2, seed=4001)
    npiv = _stepwise_dense(scene, 4, [0, 1], quirks=q, oracle_kw=dict(quirks=q))
    assert npiv > 0


def test_full_size_c4_runs_clean():
    """16384 worlds x chain32, dense solver, three steps from the scene's start (free fall, landing,
    resting contact): no world may fail its LCP, overflow the dense row capacity or go non-finite;
    sampled worlds re-run alone give the same bits and match the oracle."""
    import eggshell_b200 as E
    W = 16384
    scene = E.scenes.chain32(W, seed=4000)
    b = E.scenes.make_batch(scene, solver=E.SOLVER_DENSE_MURTY)
    for s in range(3):
        b.step(scene["dt"])
        st = b.status()
        assert int(np.bitwise_or.reduce(st["status"])) == 0, (s, np.nonzero(st["status"])[0][:16].tolist(), np.unique(st["status"]).tolist())
    assert st["n_contacts"].mean() > 20 and st["pivots"].max() < 1000 and st["pivots"].mean() > 30
    assert int(st["cfm_applied"].min()) == 1
    big = b.bodies()
    idx = [0, 7777, W - 1]
    sub = {k: (val[idx] if isinstance(val, np.ndarray) and val.shape[:1] == (W,) else val) for k, val in scene.items()}
    sub["W"] = len(idx)
    b2 = E.scenes.make_batch(sub, solver=E.SOLVER_DENSE_MURTY, taps=True)
    ows = [oracle_world(scene, wi, solver=0)[0] for wi in idx]
    for s in range(3):
        p, R, v, w = b2.bodies()
        for k in range(len(idx)):
            ows[k].set_state(p[k], R[k], v[k], w[k])
        b2.step(scene["dt"])
        for ow in ows:
            ow.step(scene["dt"])
        compare_step(b2, ows, list(range(len(idx))))
    for a, c in zip(big, b2.bodies()):
        assert np.array_equal(a[idx], c)
    b.close(); b2.close()


def test_cfm_decision_sweep():
    """ensembles.cc:513-521 adds cfm when the JacobiSVD condition number of J M^-1 J^T reaches 1e7
    (utils.cc:256-287).  The device decides from a pivoted LDL^T plus power / inverse iteration
    (egg_dense.cu).  Sweep: two separate boxes, each resting on ONE vertex (3 rows each), the second
    one heavier by a factor mu, so that cond(A) ~ mu x cond(one box); mu is bisected on the oracle
    until cond crosses 1e7 and the two decisions are compared on a ladder of relative offsets
    around the crossing.  They must agree wherever |cond / 1e7 - 1| > 1e-6; the printout shows the
    closest offsets and both decisions."""
    import eggshell_b200 as E
    from oracle import pyoracle as O
    q = np.random.default_rng(77).normal(size=(2, 4))
    q /= np.linalg.norm(q, axis=-1, keepdims=True)
    Rm = E.scenes.quat_to_mat(q)

    def scene_for(mus):
        W = len(mus)
        sc = E.scenes.cairn(W, rocks=2, seed=5)
        sc["R"][:] = Rm[None]
        sc["v"][:] = 0.0; sc["w"][:] = 0.0
        corners = np.array([[sx, sy, sz] for sx in (-.15, .15) for sy in (-.15, .15) for sz in (-.15, .15)])
        for k in range(2):
            low = np.sort((corners @ Rm[k].T)[:, 2])
            assert low[1] - low[0] > 5e-3                       # exactly one vertex below the ground
            sc["p"][:, k, :] = (2.0 * k, 0.0, -low[0] - 1e-3)
        sc["m"][:, 1] = mus
        sc["I"][:, 1] = np.eye(3)[None] * (0.1 * np.asarray(mus))[:, None, None]
        return sc

    def oracle_cond(sc, w):
        ow, _ = oracle_world(sc, w, solver=0)
        ow.update_contacts()
        assert ow.n_contacts == 2
        return O.condition_number(ow.dense_A(0.0))

    lo, hi = 1e5, 1e9
    for _ in range(60):
        mid = np.sqrt(lo * hi)
        if oracle_cond(scene_for([mid]), 0) < 1e7: lo = mid
        else: hi = mid
    mu_star = np.sqrt(lo * hi)
    offs = np.concatenate([-(10.0 ** -np.arange(1, 10)), [0.0], 10.0 ** -np.arange(9, 0, -1)])
    offs = np.concatenate([[-0.9, -0.5], offs, [0.5, 9.0, 99.0]])
    mus = mu_star * (1.0 + offs)
    sc = scene_for(mus)
    b = E.scenes.make_batch(sc, solver=E.SOLVER_DENSE_MURTY)
    b.step(sc["dt"])
    dev = b.status()["cfm_applied"].copy()
    b.close()
    rows = []
    for w, off in enumerate(offs):
        c = oracle_cond(sc, w)
        ref = int(not (c < 1e7))
        rows.append((off, c, ref, int(dev[w])))
        if abs(c / 1e7 - 1.0) > 1e-6:
            assert ref == dev[w], f"cfm decision differs at cond = {c:.9e} (offset {off:+.1e}): oracle {ref}, device {dev[w]}"
    assert {r[2] for r in rows} == {0, 1}
    print("cfm decision sweep around cond = 1e7 (offset, oracle cond, oracle decision, device decision):")
    for r in rows:
        print("  %+.1e  %.12e  %d  %d%s" % (r[0], r[1], r[2], r[3], "" if r[2] == r[3] else "   <-- differ"))


def test_post_stabilize_matches_oracle():
    """Row f1, second half: Ensemble::PostStabilize (ensembles.cc:624-657).  A hanging chain whose
    joints are broken by ~1 cm is stabilised one StepPostStabilization at a time from shared state
    (positions AND velocities move), then in one call to the end."""
    import eggshell_b200 as E
    rng = np.random.default_rng(9)
    chain = E.scenes.chain(5, links=6, anchor=(0.0, 0.0, 3.0))
    chain["p"] += rng.uniform(-0.01, 0.01, size=chain["p"].shape)
    chain["v"] = rng.uniform(-0.1, 0.1, size=chain["v"].shape)
    W = chain["W"]
    b = E.Batch(W, chain["n"], chain["nj"], solver=E.SOLVER_PGS)
    b.set_bodies(chain["p"], chain["R"], chain["v"], chain["w"], chain["m"], chain["I"])
    b.set_joints(chain["i0"], chain["i1"], chain["c0"], chain["c1"])
    b.init()                                    # BAD_INIT expected: the joints are broken on purpose
    ows = [oracle_world(chain, wi, solver=1)[0] for wi in range(W)]
    total = 0
    for it in range(6):
        p0, R0, v0, w0 = b.bodies()
        steps, e2 = b.post_stabilize(max_steps=1)
        p, R, v, w = b.bodies()
        for wi, ow in enumerate(ows):
            ow.set_state(p0[wi], R0[wi], v0[wi], w0[wi])
            osteps, oe2 = ow.post_stabilize(max_steps=1)
            assert steps[wi] == osteps
            op, oR, ov, owv = ow.bodies()
            for key, a, c in (("p", p[wi], op), ("R", R[wi], oR), ("v", v[wi], ov), ("w", w[wi], owv)):
                assert rel_err(a, c, SCALE[key]) <= 1e-9, (it, wi, key, rel_err(a, c, SCALE[key]))
            total += osteps
    assert total > 10
    steps, e2 = b.post_stabilize()
    assert np.all((e2 <= 1e-9) | (steps == 500))
    b.close()
    # with contacts: rocks resting on one vertex; both sides take one Step (which leaves the contact
    # list the loop keeps using, ensembles.cc:624-645), then stabilise one step at a time
    rocks = E.scenes.cairn(16, rocks=2, xb=(-1.0, 1.0), yb=(-1.0, 1.0), zb=(0.235, 0.255), seed=43)
    b = E.scenes.make_batch(rocks, solver=E.SOLVER_PGS)
    ows = [oracle_world(rocks, wi, solver=1)[0] for wi in range(16)]
    b.step(rocks["dt"])
    for ow in ows:
        ow.step(rocks["dt"])
    ncon = b.contacts()["count"]
    compared = 0
    for it in range(3):
        p0, R0, v0, w0 = b.bodies()
        steps, e2 = b.post_stabilize(max_steps=1)
        p, R, v, w = b.bodies()
        for wi, ow in enumerate(ows):
            if ncon[wi] != ow.n_contacts or ncon[wi] > 2:
                continue                               # > 1 contact per rock: J J^T singular, see test_init_stabilize_matches_oracle
            ow.set_state(p0[wi], R0[wi], v0[wi], w0[wi])
            osteps, oe2 = ow.post_stabilize(max_steps=1)
            assert steps[wi] == osteps
            op, oR, ov, owv = ow.bodies()
            for key, a, c in (("p", p[wi], op), ("R", R[wi], oR), ("v", v[wi], ov), ("w", w[wi], owv)):
                assert rel_err(a, c, SCALE[key]) <= 1e-8, ("rocks", it, wi, key, rel_err(a, c, SCALE[key]))
            compared += int(ncon[wi] > 0 and osteps > 0)
    assert compared > 0
    b.close()


def test_contacts_range_matches_full_readback():
    """egg_get_contacts_range: device-side transposes, any world range."""
    import eggshell_b200 as E
    scene = E.scenes.pile64(9, seed=3000)
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=5)
    b.step(scene["dt"])
    full = b.contacts()
    part = b.contacts(first=3, n_worlds=4)
    for k in full:
        assert np.array_equal(full[k][3:7], part[k]), k
    assert full["count"].min() > 300
    b.close()


def test_broadphase_cull_keeps_pair_list():
    """SURVEY row f3: the bounding-sphere cull in front of the all-pairs SAT must not change the
    colliding set: pair list (with codes and per-pair counts), contact list and geometry are
    bit-identical with and without it, on piles, stacks, chains and loose random boxes."""
    import eggshell_b200 as E
    scenes = [E.scenes.pile64(6), E.scenes.stack10(16), E.scenes.legged20(8),
              E.scenes.cairn(32, rocks=12, xb=(-0.4, 0.4), yb=(-0.4, 0.4), zb=(0.1, 0.9), seed=3)]
    for scene in scenes:
        out = []
        for quirks in (E.QUIRKS_REFERENCE, E.QUIRKS_REFERENCE | 8):
            b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=30, taps=True, quirks=quirks)
            res = []
            for s in range(3):
                b.step(scene["dt"])
                ph, con = b.pair_hits(), b.contacts()
                res.append((ph, con))
            b.close()
            out.append(res)
        nh = 0
        for (pa, ca), (pb, cb) in zip(*out):
            for k in pa:
                assert np.array_equal(pa[k], pb[k]), (scene["name"], k)
            for k in ("count", "i0", "i1", "code", "pos", "nrm", "depth"):
                assert np.array_equal(ca[k], cb[k]), (scene["name"], k)
            nh += int(np.sum(pa["n"]))
        print(scene["name"], "pair hits compared:", nh)


def test_dense_box_bounds_honoured():
    """SURVEY row f4: the dense path with the BOX friction bounds actually applied (the reference
    drops them, lcp.cc:298 = quirk q1; toolkit/lcp.cc:380-785 is its bounded Murty).  Bounded
    principal pivoting on the device against the oracle's bounded solver: same pivots, same
    active set (rows at lo / hi), state within 1e-9."""
    import eggshell_b200 as E
    q = E.QUIRK_GS_BOUNDS_SHIFT   # q1 off
    npiv = _stepwise_dense(E.scenes.cairn(8, rocks=4, zb=(0.2, 0.5), seed=21), 25, list(range(8)), quirks=q, oracle_kw=dict(quirks=q))
    assert npiv > 0


def test_cpp_host_mirror_demo():
    """The C++ mirror of model.h / ensembles.h (include/eggshell, eggshell_b200/host): the headless
    driver runs SimulationInitialization() + 25 x SimulationStep() (model.cc:33-71) and its hanging
    chain must match the oracle's Chain(10,(2,2,1)) after 25 dense steps."""
    import os
    import subprocess
    from oracle import pyoracle as O
    host = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "eggshell_b200", "host")
    subprocess.check_call(["make", "-C", host, "-s"])
    out = subprocess.run([os.path.join(host, "host_demo"), "25"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    lines = out.stdout.splitlines()
    i = lines.index("chain 10")
    got = np.array([[float(x) for x in ln.split()[1:]] for ln in lines[i + 1:i + 11]])
    W = O.World()
    W.build_chain(10, [2, 2, 1])
    W.set_params(solver=O.SOLVER_DENSE_MURTY)
    assert W.init() == 0
    for _ in range(25):
        W.step(0.001)
    p, R, v, w = W.bodies()
    assert rel_err(got[:, :3], p, SCALE["p"]) <= 1e-9 and rel_err(got[:, 3:], v, SCALE["v"]) <= 1e-9
    j = lines.index("cairn 4")
    cairn = np.array([[float(x) for x in ln.split()[1:]] for ln in lines[j + 1:j + 5]])
    assert np.all(cairn[:, 5] < 0)      # the rocks are falling


def test_host_demo_batch_dump_and_replay(tmp_path):
    """SURVEY row f2: the headless W-world driver.  host_demo steps 64 hanging chains through the C
    ABI, dumps the batch state, keeps stepping; a second process rebuilds the batch from the dump and
    must arrive at the same state bit for bit (same checksum line).  The dump's world 0 is also
    read back in text form."""
    import os
    import subprocess
    host = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "eggshell_b200", "host")
    subprocess.check_call(["make", "-C", host, "-s"])
    exe = os.path.join(host, "host_demo")
    dump = str(tmp_path / "chains.eggstate")
    a = subprocess.run([exe, "batch", "64", "8", "40", dump], capture_output=True, text=True, timeout=300)
    assert a.returncode == 0, a.stderr
    assert "status_or 0" in a.stdout
    r = subprocess.run([exe, "replay", dump, "40"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    ca = [ln for ln in a.stdout.splitlines() if ln.startswith("checksum")]
    cr = [ln for ln in r.stdout.splitlines() if ln.startswith("checksum")]
    assert ca and ca == cr, (ca, cr)
    sh = subprocess.run([exe, "show", dump, "63"], capture_output=True, text=True, timeout=60)
    assert sh.returncode == 0 and len(sh.stdout.splitlines()) == 9 and "step 40" in sh.stdout.splitlines()[0]


# ---------------------------------------------------------------------------------------------
# The other matrix-free solvers of sparse_iterations.h: Jacobi and backward SOR.
@pytest.mark.parametrize("solver,name", [(2, "jacobi"), (3, "sor")])
def test_jacobi_sor_stepwise(solver, name):
    import eggshell_b200 as E
    # Jacobi is not a contraction on these systems (the reference only runs it on diagonally
    # dominant test matrices): a few sweeps keep rounding differences from being amplified.
    km = 6 if solver == 2 else 25
    for scene, steps, kw in ((E.scenes.cairn(8, rocks=4, zb=(0.2, 0.5), seed=31), 12, dict(k_max=40 if solver == 3 else km, cfm=0.1)),
                             (E.scenes.legged20(2, seed=5000), 2, dict(k_max=km, cfm=0.1)),
                             (E.scenes.stack10(2, seed=1000), 2, dict(k_max=km, cfm=0.1))):
        idx = list(range(scene["W"]))
        b = E.scenes.make_batch(scene, solver=solver, taps=True, **kw)
        ows = [oracle_world(scene, wi, solver=solver, **kw)[0] for wi in idx]
        for s in range(steps):
            p, R, v, w = b.bodies()
            for k, wi in enumerate(idx):
                ows[k].set_state(p[wi], R[wi], v[wi], w[wi])
            b.step(scene["dt"])
            for ow in ows:
                ow.step(scene["dt"])
            worst = compare_step(b, ows, idx, tol=1e-9)
            st = b.status()
            for k, wi in enumerate(idx):
                assert st["sweeps"][wi] == ows[k].stats()["sweeps"], (name, scene["name"], s, wi)
        b.close()


def test_init_stabilize_matches_oracle():
    """Row f1: Ensemble::InitStabilize (ensembles.cc:602-622) — batched position relaxation, one
    relaxation at a time from shared state.  Scenes are chosen with a full-rank J J^T (perturbed
    joint chains; rocks touching the ground with one vertex): with redundant contacts J J^T is
    singular and -0.2 J^T (J J^T)^-1 err depends on rounding noise in the reference itself."""
    import eggshell_b200 as E
    rng = np.random.default_rng(5)
    chain = E.scenes.chain(6, links=5, anchor=(0.0, 0.0, 3.0))
    chain["p"] += rng.uniform(-0.02, 0.02, size=chain["p"].shape)       # break the joints by ~2 cm
    rocks = E.scenes.cairn(16, rocks=2, xb=(-1.0, 1.0), yb=(-1.0, 1.0), zb=(0.235, 0.255), seed=43)
    total = 0
    compared_contacts = 0
    for scene in (chain, rocks):
        b = E.Batch(scene["W"], scene["n"], scene["nj"], solver=E.SOLVER_PGS)
        b.set_bodies(scene["p"], scene["R"], scene["v"], scene["w"], scene["m"], scene["I"])
        if scene["nj"]:
            b.set_joints(scene["i0"], scene["i1"], scene["c0"], scene["c1"])
        b.init()                                                         # BAD_INIT is expected for the chain
        ows = [oracle_world(scene, wi, solver=1)[0] for wi in range(scene["W"])]
        for it in range(5):
            p0, R0, v0, w0 = b.bodies()
            steps, e2 = b.init_stabilize(max_steps=1)
            p, R, v, w = b.bodies()
            con = b.contacts()
            for wi, ow in enumerate(ows):
                ow.set_state(p0[wi], R0[wi], v0[wi], w0[wi])
                ow.update_contacts(dedupe=False)
                rows = ow.rows()
                nc_ = len(rows["i0"])
                if nc_:
                    J = np.zeros((3 * nc_, 6 * scene["n"]))
                    for k_ in range(nc_):
                        if rows["i0"][k_] >= 0:
                            J[3 * k_:3 * k_ + 3, 6 * rows["i0"][k_]:6 * rows["i0"][k_] + 6] = rows["J0"][k_]
                        if rows["i1"][k_] >= 0:
                            J[3 * k_:3 * k_ + 3, 6 * rows["i1"][k_]:6 * rows["i1"][k_] + 6] = rows["J1"][k_]
                    if np.linalg.cond(J @ J.T) > 1e8:
                        continue                                         # rank-deficient: see docstring
                    compared_contacts += ow.n_contacts
                osteps, oe2 = ow.init_stabilize(max_steps=1)
                assert steps[wi] == osteps, (scene["name"], it, wi, steps[wi], osteps)
                op, oR, _, _ = ow.bodies()
                assert rel_err(p[wi], op, SCALE["p"]) <= 1e-8 and rel_err(R[wi], oR, SCALE["R"]) <= 1e-8, (scene["name"], it, wi, rel_err(p[wi], op, SCALE["p"]), rel_err(R[wi], oR, SCALE["R"]))
                assert con["count"][wi] == ow.n_contacts
                total += osteps
        b.close()
    assert total > 10 and compared_contacts > 0
    # the full loop terminates: every world ends at err^2 <= 1e-9 or at the 100-step cap
    b = E.Batch(chain["W"], chain["n"], chain["nj"], solver=E.SOLVER_PGS)
    b.set_bodies(chain["p"], chain["R"], chain["v"], chain["w"], chain["m"], chain["I"])
    b.set_joints(chain["i0"], chain["i1"], chain["c0"], chain["c1"])
    b.init()
    steps, e2 = b.init_stabilize()
    assert np.all((e2 <= 1e-9) | (steps == 100)) and np.all(steps > 0)
    b.close()


# ---------------------------------------------------------------------------------------------
# Edge cases: empty and ragged inputs, capacity limits, API errors.
def test_edge_cases_empty_ragged_capacity_and_errors():
    """(1) Worlds without any constraint (free fall): no contacts, zero sweeps / pivots, state equal to
    the oracle's, both solvers.  (2) A ragged batch: worlds with and without contacts share a warp
    group, W is neither a multiple of the worlds per warp nor of 32; one world of one body.
    (3) Contact capacity: a world with more contacts than max_contacts drops the tail and says so
    (EGG_ST_CONTACT_OVERFLOW), the other worlds of the batch are untouched.  (4) Call-order and
    argument errors come back as error codes, never as a crash."""
    import eggshell_b200 as E
    from eggshell_b200.batch import EggError
    # (1) free fall, PGS and dense
    scene = E.scenes.cairn(5, rocks=3, zb=(5.0, 8.0), seed=41)
    scene["p"][:, :, 0] = 2.0 * np.arange(3)                            # apart from each other and far above the ground
    for kw, okw, fn in ((dict(solver=E.SOLVER_PGS), dict(solver=1), _stepwise),):
        worst = fn(scene, 3, list(range(5)), kw, okw)
        print("free fall pgs", worst)
    _stepwise_dense(scene, 3, list(range(5)))
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, taps=True)
    b.step(scene["dt"], n_steps=2)
    st = b.status()
    assert int(st["n_contacts"].max()) == 0 and int(st["sweeps"].max()) == 0 and int(st["status"].max()) == 0
    b.close()
    # (2) ragged: 7 worlds, worlds 2 and 5 lifted far above everything (no contacts), the others collide
    scene = E.scenes.cairn(7, rocks=5, zb=(0.1, 0.6), seed=43)
    for wq in (2, 5):
        scene["p"][wq, :, 2] += 50.0
        scene["p"][wq, :, 0] += 3.0 * np.arange(5)
    worst = _stepwise(scene, 6, list(range(7)), dict(solver=E.SOLVER_PGS), dict(solver=1))
    print("ragged worst", worst)
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS)
    b.step(scene["dt"])
    cnt = b.status()["n_contacts"]
    assert cnt[2] == 0 and cnt[5] == 0 and (np.delete(cnt, [2, 5]) > 0).all()
    b.close()
    _stepwise_dense(scene, 4, list(range(7)))
    one = E.scenes.cairn(1, rocks=1, zb=(0.05, 0.1), seed=44)          # one world, one body touching the ground
    worst = _stepwise(one, 5, [0], dict(solver=E.SOLVER_PGS), dict(solver=1))
    print("one body worst", worst)
    # (3) capacity: pile64 has ~500 contacts per world; with room for 64 the tail is dropped and flagged
    scene = E.scenes.pile64(3)
    scene["p"][1, :, 2] += 50.0                                         # world 1: no contacts at all
    scene["p"][1, :, 0] += 3.0 * np.arange(64)
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=10, max_contacts=64)
    b.step(scene["dt"])
    st = b.status()
    assert (st["status"][[0, 2]] & 8).all() and st["status"][1] == 0, st["status"]
    assert (st["n_contacts"][[0, 2]] == 64).all() and st["n_contacts"][1] == 0
    p, R, v, w = b.bodies()
    assert np.isfinite(p).all() and np.isfinite(v).all()
    b.close()
    # (4) errors
    b = E.Batch(2, 3, 0, solver=E.SOLVER_PGS)
    with pytest.raises(EggError):
        b.step(0.01)                                                    # egg_step before egg_init: EGG_ERR_STATE
    b.close()
    scene = E.scenes.cairn(2, rocks=2, seed=45)
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS)
    with pytest.raises(EggError):
        b.step(-1.0)                                                    # dt <= 0: EGG_ERR_ARG
    with pytest.raises(EggError):
        b.step(0.01, integrator=0)                                      # EXPLICIT_EULER: unsupported, as the reference refuses it with contacts
    b.step(0.01)                                                        # the batch is still usable
    assert int(b.status()["status"].max()) == 0
    b.close()
    with pytest.raises(EggError):
        E.Batch(0, 3, 0)                                                # no worlds
    with pytest.raises(EggError):
        E.Batch(2, 3, 0, solver=E.SOLVER_DENSE_MURTY, precision=32)     # FP32 records exist for PGS only


@pytest.mark.parametrize("name,W,k_max", [("pile64", 16384, 5), ("stack10", 65536, 10), ("legged20", 131072, 10)])
def test_full_size_worlds_are_independent_of_the_batch(name, W, k_max, monkeypatch):
    """Size-independent property that ties the full-size batches to the oracle-checked small ones: a
    world's step does not depend on which other worlds share its batch, its warp or its group stream.
    Sampled worlds of a full-occupancy batch (first / middle / last groups included) are stepped again
    in a batch of their own -- other lanes per world (forced, and checked for both batches), other
    neighbours, other stage cuts -- and must give the same bits; the small batch is then compared
    with the oracle as usual."""
    import eggshell_b200 as E
    big_lpw, small_lpw = dict(pile64=(8, 16), stack10=(1, 2), legged20=(4, 1))[name]
    monkeypatch.delenv("EGG_PGS_LPW", raising=False)
    scene = getattr(E.scenes, name)(W)
    maxc = 1024 if name == "pile64" else 0
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=k_max, max_contacts=maxc)
    assert b.kernel_config()["lpw"] == big_lpw
    b.step(scene["dt"])
    big = [x.copy() for x in b.bodies()]
    st_big = b.status()
    assert int(np.bitwise_or.reduce(st_big["status"])) == 0
    b.close()
    pick = np.array([0, 1, 5, W // 3, W // 2 + 3, W - 34, W - 2, W - 1])
    sub = dict(scene)
    for key in ("p", "R", "v", "w", "m", "I", "c0", "c1", "f_ext", "shape", "dims"):
        if key in scene and isinstance(scene[key], np.ndarray) and scene[key].shape[:1] == (W,):
            sub[key] = scene[key][pick].copy()
    sub["W"] = len(pick)
    monkeypatch.setenv("EGG_PGS_LPW", str(small_lpw))
    sb = E.scenes.make_batch(sub, solver=E.SOLVER_PGS, k_max=k_max, max_contacts=maxc, taps=True)
    assert sb.kernel_config()["lpw"] == small_lpw
    ows = [oracle_world(sub, k, solver=1, k_max=k_max)[0] for k in range(len(pick))]
    sb.step(sub["dt"])
    for ow in ows:
        ow.step(sub["dt"])
    small = sb.bodies()
    st_small = sb.status()
    for a, c in zip(small, big):
        assert np.array_equal(a.view(np.uint64), c[pick].view(np.uint64)), f"{name}: a world's step depends on its batch"
    assert np.array_equal(st_small["n_contacts"], st_big["n_contacts"][pick]) and np.array_equal(st_small["sweeps"], st_big["sweeps"][pick])
    worst = compare_step(sb, ows, list(range(len(pick))))
    print(name, "sampled worlds of the full batch vs oracle", worst)
    sb.close()


def test_full_size_dense_worlds_are_independent_of_the_batch():
    """The same property on the dense path (persistent CTAs pulling worlds from a queue, per-CTA
    scratch slabs that are reused from world to world): sampled worlds of a 4096 x chain32 batch,
    after the settling steps that bring the chain onto the ground, match a batch of their own bit
    for bit -- state, pivot counts and cfm decisions -- and that batch matches the oracle."""
    import eggshell_b200 as E
    W = 4096
    scene = E.scenes.chain32(W, seed=4000)
    b = E.scenes.make_batch(scene, solver=E.SOLVER_DENSE_MURTY)
    b.step(scene["dt"], n_steps=3)
    start = [x.copy() for x in b.bodies()]
    b.step(scene["dt"])
    big = [x.copy() for x in b.bodies()]
    st_big = b.status()
    assert int(np.bitwise_or.reduce(st_big["status"])) == 0 and int(st_big["pivots"].max()) > 0
    b.close()
    pick = np.array([0, 7, W // 2 + 1, W - 300, W - 1])
    sub = dict(scene)
    for key in ("p", "R", "v", "w", "m", "I", "c0", "c1"):
        if key in scene and isinstance(scene[key], np.ndarray) and scene[key].shape[:1] == (W,):
            sub[key] = scene[key][pick].copy()
    sub["W"] = len(pick)
    sb = E.scenes.make_batch(sub, solver=E.SOLVER_DENSE_MURTY, taps=True)
    sb.set_state(*[x[pick] for x in start])
    ows = [oracle_world(sub, k, solver=0)[0] for k in range(len(pick))]
    for k, ow in enumerate(ows):
        ow.set_state(*[x[pick][k] for x in start])
    sb.step(sub["dt"])
    for ow in ows:
        ow.step(sub["dt"])
    small = sb.bodies()
    st_small = sb.status()
    for a, c in zip(small, big):
        assert np.array_equal(a.view(np.uint64), c[pick].view(np.uint64)), "dense: a world's step depends on its batch"
    assert np.array_equal(st_small["pivots"], st_big["pivots"][pick]) and np.array_equal(st_small["cfm_applied"], st_big["cfm_applied"][pick])
    worst = compare_step(sb, ows, list(range(len(pick))))
    for k, ow in enumerate(ows):
        assert st_small["pivots"][k] == ow.stats()["pivots"] and st_small["cfm_applied"][k] == ow.stats()["cfm_applied"]
    print("dense sampled worlds of the full batch vs oracle", worst, "pivots", st_small["pivots"].tolist())
    sb.close()


def test_full_size_rollout_is_independent_of_the_batch():
    """Multi-step form of the property (an MPC horizon): twelve steps of 65536 legged worlds and the
    same twelve steps of eight of them in a batch of their own end in the same bits."""
    import eggshell_b200 as E
    W, steps = 65536, 12
    scene = E.scenes.legged20(W)
    b = E.scenes.make_batch(scene, solver=E.SOLVER_PGS, k_max=10)
    b.step(scene["dt"], n_steps=steps)
    big = [x.copy() for x in b.bodies()]
    assert int(np.bitwise_or.reduce(b.status()["status"])) == 0
    b.close()
    pick = np.array([0, 3, 9, W // 4, W // 2, W - 40, W - 2, W - 1])
    sub = dict(scene)
    for key in ("p", "R", "v", "w", "m", "I", "c0", "c1", "f_ext"):
        if key in scene and isinstance(scene[key], np.ndarray) and scene[key].shape[:1] == (W,):
            sub[key] = scene[key][pick].copy()
    sub["W"] = len(pick)
    sb = E.scenes.make_batch(sub, solver=E.SOLVER_PGS, k_max=10)
    sb.step(sub["dt"], n_steps=steps)
    for a, c in zip(sb.bodies(), big):
        assert np.array_equal(a.view(np.uint64), c[pick].view(np.uint64)), "rollout: a world's trajectory depends on its batch"
    sb.close()
